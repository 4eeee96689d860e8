#!/usr/bin/env python
"""Benchmark of the multi-particle stochastic-node hot path (BASELINE.json metric):
particle-samples/s for the IWAE / VIMCO objective forward+backward at K=50, plus % of HBM peak.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload iwae|vimco] [--impl reference] [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic input of config 2
(K=50 particles, B=1024 batch columns per GPU, Z=40 latent, X=784 observed; fp32):
    sample z ~ q (Philox in-kernel) with log q(z|x) and log p(z) from the same launch -> fused Bernoulli-likelihood +
    importance-weighted objective forward+backward (dprobs, dlogp, dlogq) -> backward of the two Normal
    log-densities and the pathwise backward of the sample (dmean, dstd), one launch
with the leaves at the path boundary of SURVEY.md §8(d): mean/std [B,Z], probs [K,B,X] (the decoder
output), x [B,X] and the decoder's upstream gradient dz [K,B,Z].  The MLP GEMMs are not part of the path.

  value : the PRODUCT path -- zhusuan.variational.ImportanceWeightedObjective(...)(observed); loss.backward() through
          the public Python API on device-resident tensors, replayed from a CUDA graph (the sampling launches read
          their Philox position from device memory, so every replay draws fresh noise), CUDA events, max over ranks.
          N > 1: batch columns sharded; EVERY step all-reduces (NCCL, in the timed region) the scalar objective and a
          1 346 864-float gradient buffer -- the parameter count of the example VAE -- through zhusuan.distributed.
  kernel_sequence : the same step as three raw C-ABI launches (round 1's `value`), for comparison.
  e2e   : the same step through the public Python API with PINNED HOST tensors as inputs
          (host->device and device->host copies inside the timed region).
  cpu_baseline / --impl reference : the REAL reference (baseline/_ref, see tools/vendor_reference.py) on the box's host
          cores, path-only harness and full example step; the oracle's C/OpenMP port when the reference is absent.
Rank 0 prints ONE JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

sys.dont_write_bytecode = True  # the benchmark writes nothing into the tree it runs from, which may be read-only

ROOT = os.path.dirname(os.path.abspath(__file__))
PKG = os.path.join(ROOT, "zhusuan-pytorch_b200")
REF = os.path.join(ROOT, "baseline", "_ref")

K_PART, B_COLS, Z_DIM, X_DIM = 50, 1024, 40, 784
VAE_DECODER_PARAMS = 40 * 500 + 500 + 500 * 500 + 500 + 500 * 784 + 784          # iwae.py:39-46
VAE_ENCODER_PARAMS = 784 * 500 + 500 + 500 * 500 + 500 + 2 * (500 * 40 + 40)     # iwae.py:89-97
FALLBACK_HBM_GBS = 6650.0
METRIC = "particle-samples/sec for IWAE/VIMCO fwd+bwd (K=50)"
DUMP_COLUMNS = 256  # --dump-outputs: [50, 256, 784] float32 of the likelihood gradient is 40 MB, the whole dump < 64 MB


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError("must be at least 1, got %d" % v)
    return v


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=2000,
                    help="timed steps of the measurement.  --impl reference times this many steps on the host CPU "
                         "(tens of ms each, twice over with the real reference): use a few, e.g. --steps 7")
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--workload", choices=["iwae", "vimco"], default="iwae")
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-strong", action="store_true")
    ap.add_argument("--graph", type=int, default=1, help="replay the step from a CUDA graph (1) or launch eagerly (0)")
    ap.add_argument("--batch", type=int, default=B_COLS, help="batch columns per GPU of the headline measurement")
    ap.add_argument("--port", action="store_true", help="--impl reference: time the oracle's C port, not the reference")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0: the loss and the leaves' "
                         "gradients) as DIR/<name>.npy, float32; arrays with a batch axis keep a fixed seeded "
                         "choice of %d batch columns" % DUMP_COLUMNS)
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the b200 path")
    return args


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback"


def workload_name(vimco, B=B_COLS):
    return ("vimco_bernoulli_latents" if vimco else "iwae_normal_latents") + "_K50_B%d_Z40_X784_path" % B


# --------------------------------------------------------------------------------------------- CPU arms
def cpu_port_inputs(B, vimco, seed=0):
    import numpy as np
    rng = np.random.RandomState(seed)
    K, Z, X = K_PART, Z_DIM, X_DIM
    probs = (1.0 / (1.0 + np.exp(-2.0 * rng.standard_normal((K, B, X))))).astype(np.float32)
    x = (rng.uniform(size=(B, X)) < 0.5).astype(np.float32)
    if vimco:
        pq = (1.0 / (1.0 + np.exp(-rng.standard_normal((B, Z))))).astype(np.float32)
        u = rng.uniform(size=(K, B * Z)).astype(np.float32)
        return dict(probs=probs, x=x, pq=pq, u=u)
    mean = (0.5 * rng.standard_normal((B, Z))).astype(np.float32)
    std = np.exp(0.3 * rng.standard_normal((B, Z))).astype(np.float32)
    eps = rng.standard_normal((K, B * Z)).astype(np.float32)
    dz_up = (1e-3 * rng.standard_normal((K, B, Z))).astype(np.float32)
    return dict(probs=probs, x=x, mean=mean, std=std, eps=eps, dz_up=dz_up)


def cpu_port_step(O, inp, vimco):
    """The hot path on the CPU oracle (C + OpenMP): same stages as the GPU step."""
    import numpy as np
    K, Z, X = K_PART, Z_DIM, X_DIM
    B = inp["x"].shape[0]
    if vimco:
        pq = inp["pq"]
        z = O.bernoulli_sample(pq, inp["u"], K, B * Z).reshape(K, B, Z)
        logq = O.bernoulli_logpmf_fwd(z, pq, K, B, Z)
        logpz = O.bernoulli_logpmf_fwd(z, np.full((B, Z), 0.5, np.float32), K, B, Z)
        r = O.iw_bernoulli_step(O.VIMCO, inp["probs"], inp["x"], logpz, logq)
        dpq = O.bernoulli_logpmf_bwd(r["dlogq"], z, pq, K, B, Z)
        return r["cost"].mean(), r["dprobs"], dpq
    mean, std, eps = inp["mean"], inp["std"], inp["eps"]
    z = O.normal_sample(mean, std, eps, K, B * Z).reshape(K, B, Z)
    logq = O.normal_logprob_fwd(z, mean, std, K, B, Z)
    zeros, ones = np.zeros((B, Z), np.float32), np.ones((B, Z), np.float32)
    logpz = O.normal_logprob_fwd(z, zeros, ones, K, B, Z)
    r = O.iw_bernoulli_step(O.SGVB, inp["probs"], inp["x"], logpz, logq)
    dz_p, _, _ = O.normal_logprob_bwd(r["dlogp"], z, zeros, ones, K, B, Z)
    dz_q, dm_q, ds_q = O.normal_logprob_bwd(r["dlogq"], z, mean, std, K, B, Z)
    dz = (inp["dz_up"] + dz_p + dz_q).reshape(K, B * Z)
    dm_s, ds_s = O.normal_sample_bwd(dz, eps, mean, std, K, B * Z)
    return r["cost"].mean(), r["dprobs"], dm_q + dm_s, ds_q + ds_s


def time_cpu_port(vimco, B_sample, reps, warm):
    sys.path.insert(0, ROOT)
    from oracle import zs_oracle as O
    O.build()
    cores = O.set_threads(os.cpu_count() or 1)
    inp = cpu_port_inputs(B_sample, vimco)
    for _ in range(warm):
        cpu_port_step(O, inp, vimco)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        cpu_port_step(O, inp, vimco)
        ts.append(time.perf_counter() - t0)
    ts.sort()
    med = ts[len(ts) // 2]
    return dict(value=K_PART * B_sample / med, unit="particle-samples/s", cores=cores, kind="port",
                sample="oracle C port (OpenMP, %d threads) of the same step on %d of the %d batch columns, "
                       "median of %d runs, %.1f ms each" % (cores, B_sample, B_COLS, reps, med * 1e3)), med


def time_real_reference(vimco, B_sample, reps, warm):
    """The UNMODIFIED reference (baseline/_ref/zhusuan, pure Python over torch CPU ops) on all host threads:
    (i) the path-only harness -- the same nets as the GPU arm, leaves at the path boundary -- and (ii) the full example
    step of examples/variational_autoencoder/iwae.py (its Generator / Variational MLPs + Adam), SURVEY.md §8(d)."""
    sys.path.insert(0, REF)
    import torch
    import zhusuan
    assert os.path.realpath(zhusuan.__file__).startswith(os.path.realpath(REF)), zhusuan.__file__
    from zhusuan.distributions import Bernoulli, Normal
    from zhusuan.framework.bn import BayesianNet
    from zhusuan.variational.importance_weighted_objective import ImportanceWeightedObjective
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    torch.manual_seed(0)
    K, B, Z, X = K_PART, B_sample, Z_DIM, X_DIM
    probs = torch.sigmoid(2.0 * torch.randn(K, B, X)).requires_grad_()
    x = (torch.rand(B, X) < 0.5).float()
    a = (torch.sigmoid(torch.randn(B, Z)) if vimco else 0.5 * torch.randn(B, Z)).requires_grad_()
    b = None if vimco else torch.exp(0.3 * torch.randn(B, Z)).requires_grad_()

    class Gen(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            if vimco:
                self.bernoulli("z", probs=0.5 * torch.ones(B, Z), n_samples=K, reduce_sum_dims=[2])
            else:
                self.normal("z", mean=torch.zeros(B, Z), std=torch.ones(B, Z), is_reparameterized=False, n_samples=K,
                            reduce_sum_dims=[2])
            self.sn(Bernoulli(probs=probs), name="x", reduce_sum_dims=[2])
            return self

    class Var(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            if vimco:
                self.sn(Bernoulli(probs=a), name="z", n_samples=K, reduce_sum_dims=[2])
            else:
                self.sn(Normal(mean=a, std=b), name="z", n_samples=K, reduce_sum_dims=[2])
            return self

    obj = ImportanceWeightedObjective(Gen(), Var(), axis=0, estimator="vimco" if vimco else "sgvb")
    leaves = [t for t in (probs, a, b) if t is not None]

    def path_step():
        for t in leaves:
            t.grad = None
        loss = obj({"x": x})
        loss.backward()
        return float(loss)

    def timeit(fn):
        for _ in range(warm):
            fn()
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            ts.append(time.perf_counter() - t0)
        ts.sort()
        return ts[len(ts) // 2]

    med = timeit(path_step)
    out = dict(value=K * B / med, unit="particle-samples/s", cores=cores, kind="reference",
               sample="the unmodified reference (baseline/_ref/zhusuan, torch %s CPU, %d threads), path-only harness "
                      "(leaves at the path boundary) on %d of the %d batch columns, median of %d steps, %.1f ms each"
                      % (torch.__version__, cores, B, B_COLS, reps, med * 1e3))
    # (ii) the example's own models, unmodified, with its optimiser: one full training step
    try:
        import importlib
        _stub_plot_modules()
        iwae = importlib.import_module("examples.variational_autoencoder.iwae")
        iwae.device = torch.device("cpu")
        iwae.reparameterization = not vimco
        gen, var = iwae.Generator(X, Z, K), iwae.Variational(X, Z, K)
        model = ImportanceWeightedObjective(gen, var, axis=0, estimator="vimco" if vimco else "sgvb")
        opt = torch.optim.Adam(model.parameters(), 1e-3)

        def full_step():
            loss = model({"x": x})
            opt.zero_grad()
            loss.backward()
            opt.step()

        fmed = timeit(full_step)
        out["full_example_step"] = {"value": K * B / fmed, "unit": "particle-samples/s", "ms_per_step": fmed * 1e3,
                                    "what": "examples/variational_autoencoder/iwae.py Generator + Variational + Adam, "
                                            "batch %d, K=%d" % (B, K)}
    except Exception as e:  # the path-only number stands on its own
        out["full_example_step"] = {"unavailable": repr(e)[:200]}
    return out, med


def _stub_plot_modules():
    """examples/utils.py imports PIL and matplotlib at module level (plots only); absent from this image."""
    import types
    for name in ("PIL", "PIL.Image", "matplotlib", "matplotlib.pyplot"):
        try:
            __import__(name)
        except Exception:
            m = types.ModuleType(name)
            sys.modules[name] = m
            parent, _, child = name.rpartition(".")
            if parent:
                setattr(sys.modules[parent], child, m)


def run_reference_arm(args):
    """`--impl reference`: the reference's own CPU implementation of the path on the box's host cores (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vimco = args.workload == "vimco"
    steps = args.steps
    warm = max(1, min(args.warmup, 3))
    use_real = os.path.isdir(os.path.join(REF, "zhusuan")) and not args.port
    if use_real:
        B_sample = 128
        cb, med = time_real_reference(vimco, B_sample, steps, warm)
    else:
        B_sample = 256
        cb, med = time_cpu_port(vimco, B_sample, steps, warm)
    line = {
        "impl": "reference", "metric": METRIC, "value": cb["value"],
        "unit": "particle-samples/s", "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic",
        "config": {"workload": workload_name(vimco), "K": K_PART, "B_per_step": B_sample, "Z": Z_DIM, "X": X_DIM,
                   "note": "a bounded sample of the batch columns per step (throughput is per particle-sample); "
                           "warm-up capped at 3"},
        "cpu_baseline": cb,
        "e2e": {"value": cb["value"], "unit": "particle-samples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------- clocks
class ClockSampler(object):
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for t, line in self.rows:
            if t < t0 or t > t1:
                continue
            f = [c.strip() for c in line.split(",")]
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
                for n, v in zip(names, f[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def pin_to_gpu_numa(gpu_index, rank, world):
    """Run this rank on its GPU's NUMA-local cores (its own slice of them when several ranks share a node): the
    host-buffer step moves 340 MB per step through pinned memory, and pinned pools are allocated where the thread runs."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(gpu_index)
        n = os.cpu_count() or 1
        mask = pynvml.nvmlDeviceGetCpuAffinity(h, (n + 63) // 64)
        cpus = [i for i in range(n) if (mask[i // 64] >> (i % 64)) & 1]
        allowed = sorted(os.sched_getaffinity(0))
        cpus = [c for c in cpus if c in allowed] or allowed
        if world > 1 and len(cpus) >= 2 * world:
            per = len(cpus) // world
            cpus = cpus[(rank % world) * per:(rank % world + 1) * per]
        os.sched_setaffinity(0, cpus)
        return "cpus %d-%d (%d, NUMA-local to GPU %d)" % (cpus[0], cpus[-1], len(cpus), gpu_index)
    except Exception as e:
        return "not pinned (%s)" % (repr(e)[:80],)


# --------------------------------------------------------------------------------------------- GPU arm
class KernelSequence(object):
    """Device-resident hot-path step as three raw C-ABI launches (zhusuan._backend): round 1's `value`."""

    def __init__(self, torch, be, vimco, device, seed, B=B_COLS):
        self.torch, self.be, self.vimco, self.dev, self.B = torch, be, vimco, device, B
        K, Z, X = K_PART, Z_DIM, X_DIM
        g = torch.Generator(device=device)
        g.manual_seed(seed)
        rn = lambda *s: torch.randn(*s, device=device, generator=g)
        self.probs = torch.sigmoid(2.0 * rn(K, B, X)).contiguous()
        self.x = (torch.rand(B, X, device=device, generator=g) < 0.5).float()
        self.seed = seed
        self.state = torch.zeros(2, dtype=torch.int64, device=device)  # device-side Philox position
        if vimco:
            self.pq = torch.sigmoid(rn(B, Z)).contiguous()
        else:
            self.mean = (0.5 * rn(B, Z)).contiguous()
            self.std = torch.exp(0.3 * rn(B, Z)).contiguous()
            self.dz_up = (1e-3 * rn(K, B, Z)).contiguous()
        self.launches_per_step = 0
        self.out = None

    def algorithmic_bytes(self):
        """Compulsory HBM bytes of one step with the fused design (DESIGN.md §measurement)."""
        K, B, Z, X = K_PART, self.B, Z_DIM, X_DIM
        kbx, kbz, kb, bz, bx = 4 * K * B * X, 4 * K * B * Z, 4 * K * B, 4 * B * Z, 4 * B * X
        fused = 2 * kbx + bx + 4 * kb + 4 * B          # probs R, dprobs W, x R, other/logq R, dlogp/dlogq W, cost W
        if self.vimco:
            # latent fwd: R pq, W z, its packed copy (one byte per float4 unit), logq, logp; latent bwd: R dlogq, the
            # packed sample, pq, W dpq
            small = (bz + kbz + kbz // 16 + 2 * kb) + (kb + kbz // 16 + 2 * bz)
        else:
            small = (2 * bz + kbz + 2 * kb) + (2 * kb + 2 * kbz + 4 * bz)  # fwd: R mean,std W z,logq,logp; bwd: R g's,z,dz_up
        return fused, fused + small

    def step(self):
        be = self.be
        K, B, Z = K_PART, self.B, Z_DIM
        n0 = be.launch_count
        if self.vimco:
            z, logq, logpz, zbits = be.bernoulli_latent_fwd(self.pq, be.KBCAST, K, B, Z, seed=self.seed,
                                                            rng_state=self.state, want_bits=True)
            r = be.iw_bernoulli_fused(be.VIMCO, self.probs, self.x, logpz, logq, 1.0 / B)
            dpq = be.bernoulli_latent_bwd(r["dlogq"], z, self.pq, be.KBCAST, K, B, Z, zbits=zbits)
            self.out = (r["cost"], r["dprobs"], dpq)
        else:
            z, logq, logpz = be.normal_latent_fwd(self.mean, self.std, be.KBCAST, K, B, Z, seed=self.seed,
                                                  rng_state=self.state)
            r = be.iw_bernoulli_fused(be.SGVB, self.probs, self.x, logpz, logq, 1.0 / B)
            dm, ds = be.normal_latent_bwd(r["dlogq"], r["dlogp"], self.dz_up, z, self.mean, self.std, be.KBCAST, K, B,
                                          Z, reparameterized=True)
            self.out = (r["cost"], r["dprobs"], dm, ds)
        self.launches_per_step = be.launch_count - n0
        return self.out

    def fused_only(self, other, logq, out=None):
        return self.be.iw_bernoulli_fused(self.be.VIMCO if self.vimco else self.be.SGVB, self.probs, self.x, other,
                                          logq, 1.0 / self.B, out=out)


def make_api_step(torch, vimco, leaves, device, B, world=1, bucket=None):
    """The product path: the public API on device-resident tensors.  Returns step() -> loss (0-d CUDA tensor).
    `leaves`: dict(probs, x, a[, b, dz_up]) of CUDA tensors.  The decoder is outside the path, so its two interfaces
    are stood in for: probs is a leaf (the decoder's output) and the gradient the decoder would send back to z is the
    fixed tensor dz_up, handed to autograd by _DecoderGrad (no kernel of its own)."""
    from zhusuan.distributions import Bernoulli, Normal
    from zhusuan.framework import BayesianNet
    from zhusuan.variational import ImportanceWeightedObjective
    import zhusuan.distributed as zd
    K, Z = K_PART, Z_DIM
    probs, x, a, b = leaves["probs"], leaves["x"], leaves["a"], leaves.get("b")
    dz_up = leaves.get("dz_up")
    zeros, ones = torch.zeros(B, Z, device=device), torch.ones(B, Z, device=device)
    half = torch.full((B, Z), 0.5, device=device)

    class _DecoderGrad(torch.autograd.Function):
        @staticmethod
        def forward(ctx, loss, z):
            return loss.view_as(loss)

        @staticmethod
        def backward(ctx, g):
            return g, dz_up

    class Gen(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            if vimco:
                self.bernoulli("z", probs=half, n_samples=K, reduce_sum_dims=[2])
            else:
                self.normal("z", mean=zeros, std=ones, is_reparameterized=False, n_samples=K, reduce_sum_dims=[2])
            self.sn(Bernoulli(probs=probs), name="x", reduce_sum_dims=[2])
            return self

    class Var(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            if vimco:
                self.sn(Bernoulli(probs=a), name="z", n_samples=K, reduce_sum_dims=[2])
            else:
                self.sn(Normal(mean=a, std=b), name="z", n_samples=K, reduce_sum_dims=[2])
            return self

    gen, var = Gen(device=device), Var(device=device)
    obj = ImportanceWeightedObjective(gen, var, axis=0, estimator="vimco" if vimco else "sgvb")
    grads = [t for t in (probs, a, b) if t is not None]
    if bucket is not None and len(bucket.segments) > 1:
        # the decoder's parameter gradients are complete once dprobs has gone through the decoder's backward: launch
        # their all-reduce at that point, so it overlaps the latent nodes' backward (and, in a real model, the encoder's)
        probs.register_post_accumulate_grad_hook(lambda p: bucket.reduce_segment(0))

    def step():
        for t in grads:
            t.grad = None
        if bucket is not None:
            bucket.zero_grad()
        with zd.global_batch(B * world):
            loss = obj({"x": x})
        if dz_up is not None:
            loss = _DecoderGrad.apply(loss, gen.observed["z"])
        loss.backward()
        if bucket is not None:
            bucket.finish(loss)
        return loss

    return step


def make_leaves(torch, vimco, device, B, seed):
    K, Z, X = K_PART, Z_DIM, X_DIM
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    rn = lambda *s: torch.randn(*s, device=device, generator=g)
    leaves = {"probs": torch.sigmoid(2.0 * rn(K, B, X)).contiguous().requires_grad_(),
              "x": (torch.rand(B, X, device=device, generator=g) < 0.5).float()}
    if vimco:
        leaves["a"] = torch.sigmoid(rn(B, Z)).contiguous().requires_grad_()
    else:
        leaves["a"] = (0.5 * rn(B, Z)).contiguous().requires_grad_()
        leaves["b"] = torch.exp(0.3 * rn(B, Z)).contiguous().requires_grad_()
        leaves["dz_up"] = (1e-3 * rn(K, B, Z)).contiguous()
    return leaves


_side_streams = {}


def capture(torch, fn, dev, use_graph=True, warm=3, count=None):
    """Warm `fn` up and capture it into a CUDA graph; returns (callable, "cuda-graph replay" | "eager launches",
    launches of this package's kernels in one call of fn).
    Everything, warm-up included, runs on ONE side stream: autograd remembers the stream on which a leaf's
    AccumulateGrad node was created, the nets' node caches keep the previous step's graph (and with it those nodes)
    alive, and a backward captured on another stream would have to synchronise with that stream -- which
    invalidates the capture (torch's CUDA-graph recipe warms up on the capture stream for the same reason)."""
    if not use_graph:  # eager by request (profiler runs): plain launches on the current stream
        for _ in range(warm):
            fn()
        launches = None
        if count is not None:
            n0 = count()
            fn()
            launches = count() - n0
        torch.cuda.synchronize()
        return fn, "eager launches", launches
    side = _side_streams.get(dev)
    if side is None:
        side = _side_streams[dev] = torch.cuda.Stream(device=dev)
    launches = None
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(warm):
            fn()
        if count is not None:
            n0 = count()
            fn()
            launches = count() - n0
        graph, how = None, "eager launches"
        if use_graph:
            try:
                torch.cuda.synchronize()
                graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(graph, stream=side):
                    fn()
                how = "cuda-graph replay"
            except Exception as e:  # capture unsupported: fall back to eager launches, and say so
                sys.stderr.write("CUDA graph capture failed, timing eager launches: %r\n" % (e,))
                graph, how = None, "eager launches (capture failed: %s)" % (repr(e)[:120],)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    if graph is not None:
        return graph.replay, how, launches

    def eager():  # capture failed: stay on the stream the warm-up ran on; it is joined before the closing event
        with torch.cuda.stream(side):
            fn()
        torch.cuda.current_stream().wait_stream(side)

    return eager, how, launches


def time_steps(torch, dist, run, steps, warm, world):
    """W warm-up steps, then exactly `steps` steps between CUDA events, barrier + synchronize on both sides; returns
    (ms per step as the max over ranks, per-rank list, wall-clock bounds of the timed region)."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(warm, 3)):
        run()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(steps):
        run()
    e1.record()
    barrier()
    t1 = time.perf_counter()
    ms = e0.elapsed_time(e1) / steps
    by_rank = [ms]
    if world > 1:
        allms = [torch.zeros(1, device="cuda") for _ in range(world)]
        dist.all_gather(allms, torch.tensor([ms], device="cuda"))
        by_rank = [float(t) for t in allms]
    return max(by_rank), by_rank, (t0, t1)


def step_outputs(torch, vimco, loss, leaves, B):
    """What a caller of the step holds after it -- the loss and the leaves' gradients -- as float32 numpy arrays.  The
    batch axis keeps the columns of a fixed seeded choice of DUMP_COLUMNS (all of them when B is no larger)."""
    import numpy as np
    cols = np.sort(np.random.RandomState(0).choice(B, min(B, DUMP_COLUMNS), replace=False))
    idx = torch.as_tensor(cols, device=loss.device)
    names = {"probs": "probs_grad", "a": "q_probs_grad" if vimco else "mean_grad", "b": "std_grad"}
    out = {"loss": loss.detach().float().cpu().numpy()}
    for key, name in names.items():
        if key in leaves:
            g = leaves[key].grad
            out[name] = g.index_select(1 if key == "probs" else 0, idx).float().cpu().numpy()
    return out


def measure_api(torch, dist, zd, be, vimco, dev, B, world, rank, steps, warm, use_graph, collectives, keep=False):
    """One configuration of the product path: returns dict(ms, by_rank, launch, launches_per_step, comm), and with
    `keep` also the outputs of the last timed step (step_outputs)."""
    leaves = make_leaves(torch, vimco, dev, B, seed=1234 + rank)
    bucket = None
    comm = None
    if collectives and world > 1:
        dec = torch.zeros(VAE_DECODER_PARAMS, device=dev, requires_grad=True)
        enc = torch.zeros(VAE_ENCODER_PARAMS, device=dev, requires_grad=True)
        two = os.environ.get("ZS_BENCH_SEGMENTS", "1") == "2"
        bucket = zd.GradientBucket([[dec], [enc]] if two else [[dec, enc]], backend=os.environ.get("ZS_BENCH_COMM", "auto"))
        comm = {"collectives_per_step": 2 if two else 1, "all_reduce_floats_per_step": int(bucket.flat.numel()),
                "all_reduce_bytes_per_step": int(bucket.flat.numel()) * 4, "backend": bucket.backend,
                "backend_is": "peer = zs_allreduce_sum_peer, this library's kernel over NVLink peer memory; "
                              "nccl = torch.distributed.all_reduce",
                "peer_unavailable": getattr(bucket, "_peer_error", None),
                "peer_variant": getattr(bucket._peer, "variant", None),
                "peer_variant_is": "nvls = zs_allreduce_sum_nvls (NVSwitch multicast: multimem.ld_reduce / multimem.st), "
                                   "p2p = zs_allreduce_sum_peer (peer loads / stores); the bucket times both once at "
                                   "construction and keeps the faster one for this world size",
                "peer_tuned_us": getattr(bucket._peer, "tuned_us", None),
                "what": "every step: SUM all-reduce of the example VAE's %d decoder + %d encoder parameter gradients and "
                        "the scalar objective, one bucket (what a 25 MB DDP bucket would hold), launched when backward "
                        "is done; zhusuan.distributed.GradientBucket.  ZS_BENCH_SEGMENTS=2: decoder segment launched "
                        "when dprobs is done (overlaps the latent backward), encoder segment after it"
                        % (VAE_DECODER_PARAMS, VAE_ENCODER_PARAMS)}
    step = make_api_step(torch, vimco, leaves, dev, B, world, bucket)
    last = {}

    def step_kept():  # a graph replay rewrites the loss tensor (and the gradients) recorded at capture
        last["loss"] = step()

    run, how, launches = capture(torch, step_kept, dev, use_graph, count=lambda: be.launch_count)
    ms, by_rank, wall = time_steps(torch, dist, run, steps, warm, world)
    out = dict(ms=ms, by_rank=by_rank, launch=how, launches_per_step=launches, comm=comm, wall=wall, run=run)
    if keep:
        out["outputs"] = step_outputs(torch, vimco, last["loss"], leaves, B)
    return out


def run_b200_arm(args):
    for _p in (ROOT, PKG):
        if _p not in sys.path:
            sys.path.insert(0, _p)
    import torch
    import torch.distributed as dist
    from zhusuan import _backend as be
    import zhusuan as zs
    import zhusuan.distributed as zd

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    be.require_cuda()
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    be.load()
    torch.manual_seed(0)  # the latent noise: with the same arguments every run computes the same outputs
    pinned_to = pin_to_gpu_numa(local, local, int(os.environ.get("LOCAL_WORLD_SIZE", str(world))))
    vimco = args.workload == "vimco"
    B = int(args.batch)
    use_graph = bool(args.graph)
    os.environ.setdefault("NCCL_DEBUG", "WARN")  # no version banner on stdout: rank 0 prints ONE JSON line
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29577")
        dist.init_process_group("nccl", device_id=dev)
        zd.decorrelate_rng()
    elif os.environ.get("ZS_BENCH_FORCE_PG") == "1":  # diagnosis knob: a 1-rank NCCL communicator at N = 1
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29577")
        dist.init_process_group("nccl", device_id=dev, rank=0, world_size=1)
        dist.all_reduce(torch.zeros(1, device=dev))
        torch.cuda.synchronize()

    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()

    # ---- headline: the product path (public API, device-resident, graph replay), collectives every step when N > 1
    head = measure_api(torch, dist, zd, be, vimco, dev, B, world, rank, args.steps, args.warmup, use_graph, True,
                       keep=bool(args.dump_outputs) and rank == 0)
    ms_per_step = head["ms"]
    value = world * K_PART * B / (ms_per_step * 1e-3)
    t_start, t_end = head["wall"]
    t_clock_end = t_end
    if rank == 0:  # the timed region can be shorter than nvidia-smi's sampling period: keep the step running, untimed
        while world == 1 and len([1 for t, _ in clocks.rows if t >= t_start]) < 6 and time.perf_counter() - t_end < 3.0:
            for _ in range(200):
                head["run"]()
            torch.cuda.synchronize()
            t_clock_end = time.perf_counter()
    if world > 1:
        dist.barrier()
    if rank == 0:
        clocks.stop()
    head.pop("run")
    torch.cuda.empty_cache()

    # ---- the same step as three raw C-ABI launches (round 1's headline), no collectives
    ks = KernelSequence(torch, be, vimco, dev, seed=1234 + rank, B=B)
    ks_run, ks_how, _ = capture(torch, ks.step, dev, use_graph)
    ks_ms, _, _ = time_steps(torch, dist, ks_run, min(args.steps, 500), min(args.warmup, 50), world)

    # ---- dominant kernel alone (roofline): CUDA events on the launching stream, 20 launches per graph replay so that
    # the host's launch rate is not what the events measure
    fused_bytes, step_bytes = ks.algorithmic_bytes()
    other = torch.randn(K_PART, B, device=dev) - 55.0
    logq = torch.randn(K_PART, B, device=dev) + 30.0
    outbuf = ks.fused_only(other, logq)
    per_graph = 20
    k_run, k_how, _ = capture(torch, lambda: [ks.fused_only(other, logq, out=outbuf) for _ in range(per_graph)], dev,
                              use_graph)
    reps = 10
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    k_run()
    torch.cuda.synchronize()
    k0.record()
    for _ in range(reps):
        k_run()
    k1.record()
    torch.cuda.synchronize()
    fused_ms = k0.elapsed_time(k1) / (reps * per_graph)
    peak, peak_kind = hbm_peak()
    achieved = fused_bytes / (fused_ms * 1e-3) / 1e9
    traffic = window_ms = None
    tp = os.path.join(ROOT, "profiles", "fused_traffic.json")
    if os.path.exists(tp):
        try:
            tj = json.load(open(tp))
            traffic = tj.get("dram_bytes_per_launch_" + args.workload)
            window_ms = tj.get("ncu_duration_ms_" + args.workload)
        except Exception:
            traffic = None
    del ks, outbuf, other, logq
    torch.cuda.empty_cache()

    line = {
        "metric": METRIC, "value": value, "unit": "particle-samples/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload_name(vimco, B), "K": K_PART, "B_per_gpu": B, "Z": Z_DIM, "X": X_DIM,
                   "estimator": "vimco" if vimco else "sgvb", "parallelism": "batch columns sharded x%d" % world,
                   "api": "public",
                   "api_call": "zhusuan.variational.ImportanceWeightedObjective(gen, var, axis=0)({'x': x}); "
                               "loss.backward() on CUDA tensors",
                   "l2": "inputs+outputs of a step (%.0f MB) exceed the 126 MB L2; no explicit flush" % (step_bytes / 1e6),
                   "launch": head["launch"], "rng": "device-side Philox position: every graph replay draws new latents",
                   "timed_wall_s": t_end - t_start,
                   "ms_per_step_by_rank": [round(v, 6) for v in head["by_rank"]],
                   "host_affinity": pinned_to},
        "kernel_sequence": {"ms_per_step": ks_ms, "value": world * K_PART * B / (ks_ms * 1e-3), "launch": ks_how,
                            "what": "zs_normal_latent_fwd -> zs_iw_bernoulli_fused -> zs_normal_latent_bwd through the "
                                    "ctypes binding, no collectives (round 1's headline)",
                            "api_over_kernel_sequence": ms_per_step / ks_ms},
        "comm": head["comm"],
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "kernel": "k_iw_bernoulli_boxf (zs_iw_bernoulli_fused)", "kernel_ms": fused_ms,
                     "algorithmic_bytes_per_launch": fused_bytes,
                     "peak_kind": (peak_kind + " (MEASURED_PEAKS.json)") if peak_kind == "measured"
                     else "fallback (B200_PROFILING.md)",
                     "frac_is": "back-to-back launches (a launch's deferred L2 write-back lands in the next one)",
                     "in_window_dram_gbs": (traffic / (window_ms * 1e-3) / 1e9) if traffic and window_ms else None,
                     "in_window_dram_frac": (traffic / (window_ms * 1e-3) / 1e9 / peak) if traffic and window_ms else None,
                     "in_window_is": "dram__bytes_read+write of ONE isolated launch / its ncu duration "
                                     "(profiles/fused_traffic.json)",
                     "step_algorithmic_bytes": step_bytes,
                     "step_frac": step_bytes / (ms_per_step * 1e-3) / 1e9 / peak,
                     "kernel_sequence_step_frac": step_bytes / (ks_ms * 1e-3) / 1e9 / peak,
                     "survey_bytes_per_particle_sample": 10074 if not vimco else 9911,
                     "survey_equiv_frac": (10074 if not vimco else 9911) * K_PART * B / (ms_per_step * 1e-3) / 1e9 / peak},
        "gpu_launches": head["launches_per_step"] * args.steps,
        "launches_per_step": head["launches_per_step"],
    }
    if rank == 0:
        line["clocks"] = clocks.summary(t_start, t_clock_end)

    # ---- strong scaling: the GLOBAL batch fixed (BASELINE.json configs[2]: "batch 1024, data-sharded across 2/4/8")
    if not args.no_strong:
        strong = []
        for Bg in (1024, 8192):
            if Bg % world:
                continue
            try:
                r = measure_api(torch, dist, zd, be, vimco, dev, Bg // world, world, rank, min(args.steps, 300),
                                min(args.warmup, 30), use_graph, True)
                r.pop("run")
                strong.append({"B_global": Bg, "B_per_gpu": Bg // world, "ms_per_step": r["ms"],
                               "value": K_PART * Bg / (r["ms"] * 1e-3), "launch": r["launch"]})
            except Exception as e:
                strong.append({"B_global": Bg, "error": repr(e)[:160]})
            torch.cuda.empty_cache()
        line["strong_scaling"] = strong

    # ---- configs 3, 4, 5 (the driver only runs the default invocation)
    if not args.no_secondary:
        try:
            line["secondary"] = secondary_block(torch, dist, zd, be, zs, dev, world, rank, use_graph, peak, vimco)
        except Exception as e:
            line["secondary"] = {"error": repr(e)[:300]}
        torch.cuda.empty_cache()

    # ---- e2e through the public API with pinned host buffers
    if not args.no_e2e:
        line["e2e"] = e2e_block(torch, dist, be, zs, dev, world, rank, vimco, B, max(3, args.e2e_steps))

    if rank == 0 and not args.no_cpu_baseline and world == 1:
        line["cpu_baseline"] = cpu_baseline_subprocess(args.workload)
    elif rank == 0:
        line["cpu_baseline"] = None
    if rank == 0 and args.dump_outputs:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in head["outputs"].items():
            np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if rank == 0:
        print(json.dumps(line))
    if world > 1 or dist.is_initialized():
        dist.destroy_process_group()


def cpu_baseline_subprocess(workload):
    """The reference arm in its own process (the reference's package is also called `zhusuan`), bounded sample."""
    try:
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--workload", workload,
                            "--steps", "7", "--warmup", "2"], stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True,
                           timeout=600, env={k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE")})
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith("{"):
                cb = json.loads(ln)["cpu_baseline"]
                break
        else:
            raise RuntimeError("no JSON line: %s" % (r.stderr[-300:],))
    except Exception as e:
        cb = {"error": repr(e)[:300]}
    if cb.get("kind") == "reference":  # also the stricter baseline: the oracle's C/OpenMP port of the same step
        try:
            r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--port", "--workload",
                                workload, "--steps", "7", "--warmup", "2"], stdout=subprocess.PIPE, stderr=subprocess.PIPE,
                               text=True, timeout=600)
            for ln in reversed(r.stdout.strip().splitlines()):
                if ln.startswith("{"):
                    cb["c_port"] = json.loads(ln)["cpu_baseline"]
                    break
        except Exception as e:
            cb["c_port"] = {"error": repr(e)[:200]}
    return cb


def e2e_setup(torch, vimco, B, rank=0):
    """The step of e2e_block as a callable: step() -> float(loss), every leaf and result in (pinned) host memory."""
    from zhusuan.distributions import Bernoulli, Normal
    from zhusuan.framework import BayesianNet
    from zhusuan.variational import ImportanceWeightedObjective
    K, Z, X = K_PART, Z_DIM, X_DIM
    cpu = torch.device("cpu")
    g = torch.Generator().manual_seed(99 + rank)
    pin = lambda t: t.pin_memory()
    host = {"probs": pin(torch.sigmoid(2.0 * torch.randn(K, B, X, generator=g))),
            "x": pin((torch.rand(B, X, generator=g) < 0.5).float())}
    if vimco:
        host.update(a=pin(torch.sigmoid(torch.randn(B, Z, generator=g))), prior=pin(torch.full((B, Z), 0.5)))
    else:
        host.update(a=pin(0.5 * torch.randn(B, Z, generator=g)), b=pin(torch.exp(0.3 * torch.randn(B, Z, generator=g))),
                    zeros=pin(torch.zeros(B, Z)), ones=pin(torch.ones(B, Z)))

    # persistent leaves and nets, as in a training loop; gradients are dropped at the start of a step (what
    # optimizer.zero_grad() does), which also returns the previous step's pinned gradient buffer to the pool
    probs = host["probs"].detach().requires_grad_()
    a = host["a"].detach().requires_grad_()
    b = None if vimco else host["b"].detach().requires_grad_()

    class Gen(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            if vimco:
                self.bernoulli("z", probs=host["prior"], n_samples=K, reduce_sum_dims=[2])
            else:
                self.normal("z", mean=host["zeros"], std=host["ones"], is_reparameterized=False, n_samples=K,
                            reduce_sum_dims=[2])
            self.sn(Bernoulli(probs=probs), name="x", reduce_sum_dims=[2])
            return self

    class Var(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            if vimco:
                self.sn(Bernoulli(probs=a), name="z", n_samples=K, reduce_sum_dims=[2])
            else:
                self.sn(Normal(mean=a, std=b), name="z", n_samples=K, reduce_sum_dims=[2])
            return self

    obj = ImportanceWeightedObjective(Gen(device=cpu), Var(device=cpu), axis=0, estimator="vimco" if vimco else "sgvb")
    leaves = [t for t in (probs, a, b) if t is not None]

    def step():
        for t in leaves:
            t.grad = None
        loss = obj({"x": host["x"]})
        loss.backward()
        assert probs.grad is not None and probs.grad.device.type == "cpu" and a.grad is not None
        return float(loss.detach())

    return step


def e2e_block(torch, dist, be, zs, dev, world, rank, vimco, B, n_e2e):
    """The same step through the PUBLIC Python API with pinned HOST tensors as leaves: the package uploads what the
    kernels need, runs them, and returns the loss and the gradients in host memory.  For the host-resident likelihood
    tensor the objective takes the chunk-pipelined route (zs_iw_step_host_begin)."""
    K, Z, X = K_PART, Z_DIM, X_DIM
    step = e2e_setup(torch, vimco, B, rank)
    for _ in range(3):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    n0 = be.launch_count
    t0 = time.perf_counter()
    for _ in range(n_e2e):
        step()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / n_e2e
    if world > 1:
        tt = torch.tensor([dt], device=dev)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt = float(tt)
    kbx, bx, bz = 4 * K * B * X, 4 * B * X, 4 * B * Z
    n_par = 1 if vimco else 2
    # uploads: probs, x, the variational parameters (once per step: upload_memo); downloads: dprobs, the per-column
    # costs, the parameter gradients.  The latent samples, the [K,B] log-probabilities and their gradients stay on the
    # device (draw #1 of the reference protocol is never materialised: zhusuan/_lazy.py).
    h2d = kbx + bx + n_par * bz
    d2h = kbx + 4 * B + n_par * bz
    return {"value": world * K * B / dt, "unit": "particle-samples/s", "h2d_bytes_per_step": h2d,
            "d2h_bytes_per_step": d2h, "ms_per_step": dt * 1e3,
            "api": "zhusuan.variational.ImportanceWeightedObjective(...)({'x': x}); loss.backward(), every leaf (probs, "
                   "x, parameters) and every result (loss, gradients) in host memory",
            "launches_per_step": (be.launch_count - n0) // n_e2e,
            "pcie_floor_ms": "3.3-3.5 (H2D and D2H of the 160.6 MB likelihood tensor / gradient at once, measured "
                             "93-98 GB/s aggregate)"}


def secondary_block(torch, dist, zd, be, zs, dev, world, rank, use_graph, peak, headline_is_vimco):
    """Configs 3, 4 and 5 of BASELINE.json at this run's world size (each rank works on its shard; times are the max
    over ranks; no data-path collective: batch columns / chains are independent)."""
    out = {}

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t)

    def timed(run, reps, warm=10):
        for _ in range(warm):
            run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            run()
        e1.record()
        torch.cuda.synchronize()
        return max_over_ranks(e0.elapsed_time(e1) / reps)

    def timed_kernel(fn, per_graph=10, reps=20):
        """ms per launch of a single kernel: `per_graph` launches captured into one CUDA graph (an eager ctypes launch
        costs the host ~10 us, more than these kernels run), CUDA events around `reps` replays."""
        run, how, _ = capture(torch, lambda: [fn() for _ in range(per_graph)], dev, use_graph)
        return timed(run, reps, 3) / per_graph

    # ---- config 3 (or 2, whichever is not the headline): the other estimator through the same public-API path
    other = not headline_is_vimco
    r = measure_api(torch, dist, zd, be, other, dev, B_COLS, world, rank, 300, 30, use_graph, False)
    r.pop("run")
    ksq = KernelSequence(torch, be, other, dev, 7, B_COLS)
    _, sb = ksq.algorithmic_bytes()
    del ksq
    out["vimco_K50_B1024" if other else "iwae_K50_B1024"] = {
        "value": world * K_PART * B_COLS / (r["ms"] * 1e-3), "unit": "particle-samples/s", "ms_per_step": r["ms"],
        "launches_per_step": r["launches_per_step"], "launch": r["launch"], "step_algorithmic_bytes": sb,
        "step_frac": sb / (r["ms"] * 1e-3) / 1e9 / peak, "api": "public, device-resident"}
    torch.cuda.empty_cache()

    # ---- config 4: BNN SGVB, K = 100 weight particles, layers [90, 50, 1]; y-likelihood [K, b] with a scalar logstd
    from zhusuan.framework import BayesianNet
    from zhusuan.variational import ELBO
    K4, layers = 100, [90, 50, 1]
    cfg4 = {}
    for Bg in (8192, 131072):
        b = Bg // world
        xx = torch.randn(b, 90, device=dev)
        yy = torch.randn(b, device=dev)
        ymean = torch.randn(K4, b, device=dev)
        ylogstd = torch.zeros(1, device=dev)
        ystd = torch.exp(ylogstd)
        g = torch.full((K4, 1), 1.0 / (K4 * b), device=dev)
        # (i) the y-likelihood kernels alone: normal.py:109-126 on [K, b] with the [b] observation broadcast over K
        fwd = timed_kernel(lambda: be.normal_logprob_fwd(yy, be.KBCAST, ymean, be.FULL, ystd, be.SCALAR, K4, 1, b))
        bwd = timed_kernel(lambda: be.normal_logprob_bwd(g, yy, be.KBCAST, ymean, be.FULL, ystd, be.SCALAR, K4, 1, b,
                                                         False, True, False))
        pd = K4 * b

        class Net(BayesianNet):
            def __init__(self):
                super().__init__(device=dev)
                self.y_logstd = torch.nn.Parameter(torch.zeros(1, device=dev))

            def forward(self, observed):
                self.observe(observed)
                h = self.observed["x"].unsqueeze(0).expand(K4, -1, -1)
                for i, (n_in, n_out) in enumerate(zip(layers[:-1], layers[1:])):
                    w = self.normal("w%d" % i, mean=torch.zeros(n_out, n_in + 1, device=dev),
                                    std=torch.ones(n_out, n_in + 1, device=dev), group_ndims=2, n_samples=K4,
                                    reduce_mean_dims=[0])
                    h = zs.particle_linear(w, h)
                    if i < len(layers) - 2:
                        h = torch.relu(h)
                self.normal("y", mean=h.squeeze(2), logstd=self.y_logstd, reduce_mean_dims=[0, 1], multiplier=1000000)
                return self

        class Var(BayesianNet):
            def __init__(self):
                super().__init__(device=dev)
                self.w_means = torch.nn.ParameterList([torch.nn.Parameter(torch.zeros(o, i + 1, device=dev))
                                                       for i, o in zip(layers[:-1], layers[1:])])
                self.w_logstds = torch.nn.ParameterList([torch.nn.Parameter(torch.zeros(o, i + 1, device=dev))
                                                         for i, o in zip(layers[:-1], layers[1:])])

            def forward(self, observed):
                self.observe(observed)
                for i in range(len(layers) - 1):
                    self.normal("w%d" % i, mean=self.w_means[i], logstd=self.w_logstds[i], group_ndims=2, n_samples=K4,
                                reduce_mean_dims=[0])
                return self

        model = ELBO(Net(), Var())
        params = list(model.parameters())

        def elbo_step():
            for p in params:
                p.grad = None
            model({"x": xx, "y": yy}).backward()

        full = timed(elbo_step, 20, 5)
        cfg4["B_global_%d" % Bg] = {
            "B_per_gpu": b, "y_likelihood_fwd_us": fwd * 1e3, "y_likelihood_bwd_us": bwd * 1e3,
            "y_likelihood_bytes_per_particle_datapoint": 8,
            "y_likelihood_fwd_frac": 4.0 * pd / (fwd * 1e-3) / 1e9 / peak,   # reads mean[K,b] (+ y[b])
            "y_likelihood_bwd_frac": 8.0 * pd / (bwd * 1e-3) / 1e9 / peak,   # reads mean, writes dmean
            "elbo_step_ms": full, "value": world * pd / (full * 1e-3), "unit": "particle-datapoints/s",
            "what": "ELBO(Net, Variational)(x, y).backward() through the public API, eager, incl. the two "
                    "particle_linear batched GEMMs (cuBLAS, not claimed)"}
        del xx, yy, ymean, model
        torch.cuda.empty_cache()
    out["cfg4_bnn_sgvb_K100"] = cfg4

    # ---- config 5: SG-MCMC, chains sharded over ranks, through sampler.sample()
    import zhusuan.mcmc
    cfg5 = {}
    for label, chains_global in (("chains_1024", 1024), ("chains_65536", 65536)):
        ch = chains_global // world
        for name, make in (("sgld", lambda: zhusuan.mcmc.SGLD(1e-3)),
                           ("sghmc", lambda: zhusuan.mcmc.SGHMC(1e-3, friction=0.25, n_iter_resample_v=20))):
            class Chains(BayesianNet):
                def forward(self, observed):
                    self.observe(observed)
                    self.normal("w0", mean=torch.zeros(50, 91, device=dev), std=torch.ones(50, 91, device=dev),
                                n_samples=ch, group_ndims=2, reduce_mean_dims=[0])
                    self.normal("w1", mean=torch.zeros(1, 51, device=dev), std=torch.ones(1, 51, device=dev),
                                n_samples=ch, group_ndims=2, reduce_mean_dims=[0])
                    return self

            net, sampler = Chains(device=dev), make()
            sampler.sample(net, {}, True)
            n0 = be.launch_count
            sampler.sample(net, {}, False)
            launches = be.launch_count - n0
            ms = timed(lambda: sampler.sample(net, {}, False), 30, 5)
            elems = ch * 4601
            bytes_per = 12 if name == "sgld" else 32
            cfg5["%s_%s" % (name, label)] = {
                "chains_per_gpu": ch, "ms_per_update": ms, "value": world * ch / (ms * 1e-3), "unit": "chain-steps/s",
                "element_updates_per_s": world * elems / (ms * 1e-3), "launches_per_update": launches,
                "update_kernel_algorithmic_bytes": bytes_per * elems,
                "what": "sampler.sample(net, {}) through the public API (eager: log-joint forward/backward of the "
                        "net's two Normal nodes + ONE multi-tensor update launch%s)"
                        % ("" if name == "sgld" else " before and one after the gradient")}
            del net, sampler
        torch.cuda.empty_cache()
    out["cfg5_sgmcmc"] = cfg5
    return out


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
