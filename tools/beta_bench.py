"""Beta node kernels on one B200, float32, seeded inputs.

Times, from ONE process and with the arms interleaved round by round:
  * latent_q_fwd / latent_q_bwd      log q(z) of the variational posterior at the latent-node shape K=50, B=1024, Z=40:
                                     z [K,B,Z] FULL, alpha and beta [B,Z] KBCAST; the backward writes dalpha and dbeta
                                     summed over K (k_kreduce_bwd_beta);
  * latent_prior_fwd / _bwd          log p(z) under the Beta prior, alpha and beta SCALAR; the backward writes dz;
  * full_fwd / full_bwd              a [50, 1024, 784] case with x, alpha and beta all FULL; the backward writes all
                                     three gradients (three psi per element);
  * sample                           zs_beta_sample at K=50, B=1024, Z=40, alpha and beta KBCAST.
Each as time per call, bytes over time (the operands read once, the results written once) and share of the HBM peak
measured in the same process (a 4 GiB device-to-device copy, read + write bytes), plus elements per second.  Records the
card name and power limit.  Writes JSON to profiles/.

Usage: python tools/beta_bench.py [--rounds 10] [--reps 20] [--out profiles/beta_bench.json]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "zhusuan-pytorch_b200"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

from zhusuan import _backend as be  # noqa: E402
from poisson_bench import card, timed, hbm_peak_gbs  # noqa: E402

K, B, Z = 50, 1024, 40
XF = 784
F, KB, SC = be.FULL, be.KBCAST, be.SCALAR
FAM = be.FAM_BETA


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "beta_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("beta_bench: needs a CUDA device (nothing is timed without one)")
    dev = torch.device("cuda")
    info = card()
    peak = hbm_peak_gbs()

    g = torch.Generator(device=dev)
    g.manual_seed(4321)

    def u(*shape, lo=0.0, hi=1.0):
        return (torch.rand(*shape, device=dev, generator=g) * (hi - lo) + lo).contiguous()

    # latent-node shape
    z = u(K, B, Z, lo=0.01, hi=0.99)
    qa, qb = u(B, Z, lo=0.5, hi=5.0), u(B, Z, lo=0.5, hi=5.0)
    pa, pb = torch.tensor([1.5], device=dev), torch.tensor([2.0], device=dev)
    gl = torch.randn(K, B, device=dev, generator=g)
    # all-FULL case
    x = u(K, B, XF, lo=0.01, hi=0.99)
    fa, fb = u(K, B, XF, lo=0.5, hi=5.0), u(K, B, XF, lo=0.5, hi=5.0)
    gf = torch.randn(K, B, device=dev, generator=g)

    arms = {
        "latent_q_fwd": lambda: be.locscale_logprob_fwd(FAM, z, F, qa, KB, qb, KB, K, B, Z),
        "latent_q_bwd": lambda: be.locscale_logprob_bwd(FAM, gl, z, F, qa, KB, qb, KB, K, B, Z, False, True, True),
        "latent_prior_fwd": lambda: be.locscale_logprob_fwd(FAM, z, F, pa, SC, pb, SC, K, B, Z),
        "latent_prior_bwd": lambda: be.locscale_logprob_bwd(FAM, gl, z, F, pa, SC, pb, SC, K, B, Z, True, False, False),
        "full_fwd": lambda: be.locscale_logprob_fwd(FAM, x, F, fa, F, fb, F, K, B, XF),
        "full_bwd": lambda: be.locscale_logprob_bwd(FAM, gf, x, F, fa, F, fb, F, K, B, XF, True, True, True),
        "sample": lambda: be.beta_sample(qa, KB, qb, KB, K, B * Z, seed=7, offset=0),
    }
    nl, nf = K * B * Z, K * B * XF
    byts = {  # float32 bytes the algorithm has to move
        "latent_q_fwd": 4.0 * (nl + 2 * B * Z + K * B),
        "latent_q_bwd": 4.0 * (nl + 2 * B * Z + K * B + 2 * B * Z),
        "latent_prior_fwd": 4.0 * (nl + K * B),
        "latent_prior_bwd": 4.0 * (nl + K * B + nl),
        "full_fwd": 4.0 * (3 * nf + K * B),
        "full_bwd": 4.0 * (3 * nf + K * B + 3 * nf),
        "sample": 4.0 * (2 * B * Z + nl),
    }
    elems = {k: (nf if k.startswith("full") else nl) for k in arms}
    for fn in arms.values():
        fn()
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, fn in arms.items():
            times[k].append(timed(fn, args.reps))

    res = {}
    for k, ts in times.items():
        ts = sorted(ts)
        us = ts[len(ts) // 2]
        gbs = byts[k] / (us * 1e-6) / 1e9
        res[k] = dict(us_median=us, us_min=ts[0], us_max=ts[-1], bytes=byts[k], gb_per_s=gbs, hbm_frac=gbs / peak,
                      elements=elems[k], gelem_per_s=elems[k] / (us * 1e-6) / 1e9)
    line = dict(tool="beta_bench", dtype="float32", K=K, B=B, Z=Z, X_full=XF, card=info, hbm_peak_gbs_measured=peak,
                hbm_peak_method="4 GiB device-to-device copy, read + write bytes, best of 3x10",
                rounds=args.rounds, reps=args.reps, results=res)
    print(json.dumps(line))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(line, f, indent=1)


if __name__ == "__main__":
    main()
