"""Poisson-likelihood importance-weighted step at K=50, B=1024, X=784 (seeded rates and counts), on one B200.

Reports, from ONE process and with the timed arms interleaved round by round:
  * fused_kernel          zs_iw_poisson_fused_loss alone (SGVB), preallocated outputs;
  * api_step_fused        the public-API step (ImportanceWeightedObjective forward + backward, Normal latent, Poisson
                          likelihood) replayed from a captured CUDA graph, fused route;
  * api_step_two_pass     the same step with zhusuan.variational.FUSED = False (log-pmf, objective, log-pmf backward);
  * bernoulli_fused_kernel zs_iw_bernoulli_fused_loss at the same shape, for comparison.
Each as time per call, bytes over time, and share of the HBM peak measured in the same process (a 4 GiB
device-to-device copy, read + write bytes).  Bytes: the [K,B,X] rate tensor read once and its gradient written once,
plus x and the [K,B] terms (kernels); the API steps are charged the fused route's bytes, so the two-pass number is the
rate it would need to reach to match.  Records the card name and power limit.  Writes JSON to profiles/.

Usage: python tools/poisson_bench.py [--rounds 10] [--reps 20] [--out profiles/poisson_bench.json]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "zhusuan-pytorch_b200"))

import torch  # noqa: E402

import zhusuan.variational  # noqa: E402
from zhusuan import _backend as be  # noqa: E402
from zhusuan.distributions import Normal, Poisson  # noqa: E402
from zhusuan.framework import BayesianNet  # noqa: E402
from zhusuan.variational import ImportanceWeightedObjective  # noqa: E402

K, B, X, Z = 50, 1024, 784, 40


def card():
    name = torch.cuda.get_device_name()
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()),
                            "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # the number is still a number; say what is missing
        q = "unavailable (%r)" % (e,)
    return dict(name=name, power_limit_and_max_sm_clock=q)


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps * 1e3  # us


def hbm_peak_gbs(reps=10):
    n = (4 << 30) // 4
    a = torch.empty(n, dtype=torch.float32, device="cuda").fill_(1.0)
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    torch.cuda.synchronize()
    best = min(timed(lambda: b.copy_(a), reps) for _ in range(3))
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * n * 4 / (best * 1e-6) / 1e9


def capture(fn, warm=3):
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    return g


class Gen(BayesianNet):
    def __init__(self, rate):
        super().__init__(device=rate.device)
        self.rate = rate

    def forward(self, observed):
        self.observe(observed)
        d = self.rate.device
        self.normal("z", mean=torch.zeros(B, Z, device=d), std=torch.ones(B, Z, device=d), n_samples=K,
                    reduce_sum_dims=[2])
        self.sn(Poisson(self.rate), name="x", reduce_sum_dims=[2])
        return self


class Var(BayesianNet):
    def __init__(self, mean, std):
        super().__init__(device=mean.device)
        self.mean, self.std = mean, std

    def forward(self, observed):
        self.observe(observed)
        self.sn(Normal(mean=self.mean, std=self.std), name="z", n_samples=K, reduce_sum_dims=[2])
        return self


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=10)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "poisson_bench.json"))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("poisson_bench: needs a CUDA device (nothing is timed without one)")
    dev = torch.device("cuda")
    info = card()
    peak = hbm_peak_gbs()

    g = torch.Generator(device=dev)
    g.manual_seed(1234)
    rate = (torch.empty(K, B, X, device=dev).exponential_(1.0, generator=g) * 2.0 + 0.05).contiguous()
    x = torch.poisson(torch.full((B, X), 1.5, device=dev), generator=g)
    probs = torch.sigmoid(2.0 * torch.randn(K, B, X, device=dev, generator=g)).contiguous()
    xb = (torch.rand(B, X, device=dev, generator=g) < 0.5).float()
    other = torch.randn(K, B, device=dev, generator=g) - 55.0
    logq = torch.randn(K, B, device=dev, generator=g) + 30.0

    outp, outb = {}, {}
    pk = lambda: be.iw_poisson_fused(be.SGVB, rate, x, other, logq, 1.0 / B, out=outp, cost_scaled=True, want_loss=True)
    bk = lambda: be.iw_bernoulli_fused(be.SGVB, probs, xb, other, logq, 1.0 / B, out=outb, cost_scaled=True,
                                       want_loss=True)
    assert pk() is not None and bk() is not None

    rate_leaf = rate.clone().requires_grad_()
    mean = (0.5 * torch.randn(B, Z, device=dev, generator=g)).requires_grad_()
    std = torch.exp(0.3 * torch.randn(B, Z, device=dev, generator=g)).requires_grad_()
    obj = ImportanceWeightedObjective(Gen(rate_leaf), Var(mean, std), axis=0, estimator="sgvb")

    def step():
        for t in (rate_leaf, mean, std):
            t.grad = None
        loss = obj({"x": x})
        loss.backward()
        return loss

    graphs = {}
    for name, fused in (("api_step_fused", True), ("api_step_two_pass", False)):
        zhusuan.variational.FUSED = fused
        try:
            graphs[name] = capture(step)
        finally:
            zhusuan.variational.FUSED = True
    arms = {"fused_kernel": pk, "bernoulli_fused_kernel": bk,
            "api_step_fused": graphs["api_step_fused"].replay, "api_step_two_pass": graphs["api_step_two_pass"].replay}
    for fn in arms.values():
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in arms}
    for _ in range(args.rounds):
        for k, fn in arms.items():
            times[k].append(timed(fn, args.reps))

    kb_bytes = 4.0 * (2 * K * B * X + B * X + 4 * K * B + B)  # rate in, drate out, x, [K,B] in/out, cost
    res = {}
    for k, ts in times.items():
        ts = sorted(ts)
        us = ts[len(ts) // 2]
        gbs = kb_bytes / (us * 1e-6) / 1e9
        res[k] = dict(us_median=us, us_min=ts[0], us_max=ts[-1], bytes=kb_bytes, gb_per_s=gbs, hbm_frac=gbs / peak)
    line = dict(tool="poisson_bench", K=K, B=B, X=X, Z=Z, card=info, hbm_peak_gbs_measured=peak,
                hbm_peak_method="4 GiB device-to-device copy, read + write bytes, best of 3x10",
                rounds=args.rounds, reps=args.reps, results=res,
                poisson_over_bernoulli_rate=res["bernoulli_fused_kernel"]["us_median"] / res["fused_kernel"]["us_median"],
                fused_over_two_pass_speedup=res["api_step_two_pass"]["us_median"] / res["api_step_fused"]["us_median"])
    print(json.dumps(line))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(line, f, indent=1)


if __name__ == "__main__":
    main()
