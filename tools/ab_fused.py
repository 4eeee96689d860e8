"""A/B timing of zs_iw_bernoulli_fused between builds of the library, interleaved in one process so
box-to-box and clock drift cancel.  Usage: ab_fused.py name=path.so [name=path.so ...]   (GPU box only)
AB_B (default 1024) and AB_K (default 50) set the shape; AB_LOGITS=1 times the logits form."""
import ctypes, os, sys
import torch

K, B, X = int(os.environ.get("AB_K", 50)), int(os.environ.get("AB_B", 1024)), 784
LOGITS = os.environ.get("AB_LOGITS", "0") == "1"
c = ctypes
vp, i64, i32, dbl = c.c_void_p, c.c_int64, c.c_int, c.c_double
libs = []
import shutil, tempfile
tmpdir = tempfile.mkdtemp()
envs = {}
for arg in sys.argv[1:]:
    # name=path.so[@ENV=V,ENV=V]: the env applies to that copy's first call (the library reads it once)
    name, path = arg.split("=", 1)
    env = {}
    if "@" in path:
        path, es = path.split("@", 1)
        env = dict(e.split("=", 1) for e in es.split(","))
    copy = os.path.join(tmpdir, name + ".so")  # a private copy: its own statics even for the same build
    shutil.copy(os.path.abspath(path), copy)
    lib = c.CDLL(copy)
    envs[name] = env
    lib.zs_iw_bernoulli_fused.restype = i32
    lib.zs_iw_bernoulli_fused.argtypes = [i32] + [vp] * 9 + [i64, i64, i64, dbl, i32, vp]
    libs.append((name, lib))
dev = "cuda"
torch.manual_seed(0)
probs = 2 * torch.randn(K, B, X, device=dev)
if not LOGITS:
    probs = torch.sigmoid(probs)
x = (torch.rand(B, X, device=dev) < 0.5).float()
other = torch.randn(K, B, device=dev) - 55
logq = torch.randn(K, B, device=dev) + 30
outs = {}
for name, lib in libs:
    outs[name] = dict(cost=torch.empty(B, device=dev), dprobs=torch.empty_like(probs),
                      dlogp=torch.empty(K, B, device=dev), dlogq=torch.empty(K, B, device=dev))
stream = torch.cuda.current_stream().cuda_stream


def set_env(name, on):
    # every variant library reads its knobs once, at its first call: the variant's environment must be in place
    # then (set_env around first_call)
    for k, v in envs[name].items():
        if on:
            os.environ[k] = v
        else:
            os.environ.pop(k, None)


def first_call(name, lib):
    set_env(name, True)
    run(lib, outs[name], 0)
    torch.cuda.synchronize()
    set_env(name, False)


def run(lib, o, est):
    rc = lib.zs_iw_bernoulli_fused(est, o["cost"].data_ptr(), o["dprobs"].data_ptr(), o["dlogp"].data_ptr(),
                                   o["dlogq"].data_ptr(), None, probs.data_ptr(), x.data_ptr(), other.data_ptr(),
                                   logq.data_ptr(), K, B, X, 1.0 / B, 2 if LOGITS else 0, stream)  # ZS_FUSED_LOGITS = 2
    assert rc == 0, rc


for name, lib in libs:
    first_call(name, lib)
for est, ename in ((0, "sgvb"), (1, "vimco")):
    res = {n: [] for n, _ in libs}
    for rnd in range(6):
        for name, lib in libs:
            set_env(name, True)
            for _ in range(5):
                run(lib, outs[name], est)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(50):
                run(lib, outs[name], est)
            e1.record()
            torch.cuda.synchronize()
            set_env(name, False)
            res[name].append(e0.elapsed_time(e1) / 50 * 1e3)
    for name, _ in libs:
        v = sorted(res[name])
        print("%-6s %-12s median %.2f us  min %.2f  max %.2f" % (ename, name, v[len(v) // 2], v[0], v[-1]))
    ref = outs[libs[0][0]]
    for name, _ in libs[1:]:
        o = outs[name]
        print("   max |diff| vs %s: dprobs %.3g cost %.3g dlogq %.3g" % (
            libs[0][0], (o["dprobs"] - ref["dprobs"]).abs().max().item(), (o["cost"] - ref["cost"]).abs().max().item(),
            (o["dlogq"] - ref["dlogq"]).abs().max().item()))
