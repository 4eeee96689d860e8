"""ctypes binding of the sm_100a C-ABI library (include/zs_b200.h).

This is the only place the Python package touches native code.  There is NO CPU fallback: if
`lib/libzs_b200.so` is missing, or no CUDA device is present, every op raises.  Tensors are passed
as raw device pointers; every launch runs with the operands' CUDA device current and goes to torch's current
stream OF THAT DEVICE, so stream / CUDA-graph semantics of the caller hold and tensors on cuda:1 work while
cuda:0 is the current device.  All operands of one call must live on one device.
"""
import ctypes
import os

import torch

_PKG_ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LIB_PATH = os.path.join(_PKG_ROOT, "lib", "libzs_b200.so")

F32, F64 = 0, 1
FULL, KBCAST, SCALAR = 0, 1, 2
SGVB, VIMCO, ELBO = 0, 1, 2
ERR_UNSUPPORTED, ERR_ALIGN = -6, -7
FUSED_ACCUMULATE_COST, FUSED_LOGITS, FUSED_COST_SCALED = 1, 2, 4
ALG_SGLD, ALG_PSGLD, ALG_SGHMC_PRE, ALG_SGHMC_POST = 0, 1, 2, 3
CHAIN_MAX_TENSORS = 32
IMPL_DEFAULT, IMPL_RING, IMPL_BOX, IMPL_BOXG = -1, 2, 3, 4
ABI_VERSION = 3

_lib = None
launch_count = 0  # kernels launched through this binding (bench.py's gpu_launches)


class BackendError(RuntimeError):
    pass


class ChainTensor(ctypes.Structure):
    """zs_chain_tensor"""
    _fields_ = [("w_out", ctypes.c_void_p), ("w", ctypes.c_void_p), ("g", ctypes.c_void_p),
                ("state", ctypes.c_void_p), ("noise", ctypes.c_void_p), ("n", ctypes.c_int64)]


def _declare(lib):
    c = ctypes
    vp, i64, u64, i32, dbl = c.c_void_p, c.c_int64, c.c_uint64, c.c_int, c.c_double
    sig = {
        "zs_abi_version": (i32, []),
        "zs_strerror": (c.c_char_p, [i32]),
        "zs_last_error": (c.c_char_p, []),
        "zs_device_info": (i32, [c.POINTER(i32)] * 3),
        "zs_rng_state_init": (i32, [vp, u64, vp]),
        "zs_philox_uniform": (i32, [i32, vp, i64, u64, u64, vp, vp]),
        "zs_philox_normal": (i32, [i32, vp, i64, dbl, dbl, u64, u64, vp, vp]),
        "zs_philox_raw": (i32, [vp, i64, u64, u64, vp, vp]),
        "zs_normal_sample": (i32, [i32, vp, vp, i32, vp, i32, vp, vp, i64, i64, u64, u64, vp, vp, vp]),
        "zs_normal_sample_bwd": (i32, [i32, vp, i32, vp, i32, vp, vp, i64, i64, u64, u64, vp, vp]),
        "zs_normal_logprob_fwd": (i32, [i32, vp, vp, i32, vp, i32, vp, i32, i64, i64, i64, vp]),
        "zs_normal_logprob_bwd": (i32, [i32, vp, vp, vp, vp, vp, i32, vp, i32, vp, i32, i64, i64, i64, vp]),
        "zs_normal_latent_fwd": (i32, [i32, vp, vp, vp, vp, i32, vp, i32, vp, vp, vp, i64, i64, i64, u64, u64, vp, vp]),
        "zs_bernoulli_latent_fwd": (i32, [i32, vp, vp, vp, vp, i32, vp, vp, i64, i64, i64, u64, u64, vp, vp, vp]),
        "zs_normal_latent_bwd": (i32, [i32, vp, vp, vp, vp, vp, vp, vp, i32, vp, i32, vp, vp, i32, i64, i64, i64, vp]),
        "zs_bernoulli_latent_bwd": (i32, [i32, vp, vp, vp, vp, i32, i64, i64, i64, vp, vp]),
        "zs_bernoulli_sample": (i32, [i32, vp, vp, i32, vp, i64, i64, u64, u64, vp, vp]),
        "zs_bernoulli_logpmf_fwd": (i32, [i32, vp, vp, i32, vp, i32, i64, i64, i64, vp]),
        "zs_bernoulli_logpmf_bwd": (i32, [i32, vp, vp, vp, vp, i32, vp, i32, i64, i64, i64, vp]),
        "zs_locscale_sample": (i32, [i32, i32, vp, vp, i32, vp, i32, vp, i64, i64, u64, u64, vp, vp, vp]),
        "zs_locscale_sample_bwd": (i32, [i32, i32, vp, i32, vp, i32, vp, vp, i64, i64, u64, u64, vp, vp]),
        "zs_locscale_logprob_fwd": (i32, [i32, i32, vp, vp, i32, vp, i32, vp, i32, i64, i64, i64, vp]),
        "zs_locscale_logprob_bwd": (i32, [i32, i32, vp, vp, vp, vp, vp, i32, vp, i32, vp, i32, i64, i64, i64, vp]),
        "zs_poisson_sample": (i32, [i32, vp, vp, i32, i64, i64, u64, u64, vp, vp]),
        "zs_beta_sample": (i32, [i32, vp, vp, i32, vp, i32, i64, i64, u64, u64, vp, vp]),
        "zs_poisson_logpmf_fwd": (i32, [i32, vp, vp, i32, vp, i32, i64, i64, i64, vp]),
        "zs_poisson_logpmf_bwd": (i32, [i32, vp, vp, vp, i32, vp, i32, i64, i64, i64, vp]),
        "zs_iw_poisson_fused": (i32, [i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, dbl, i32, vp]),
        "zs_iw_poisson_fused_loss": (i32, [i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, dbl, i32, vp]),
        "zs_bernoulli_logits_logpmf_fwd": (i32, [i32, vp, vp, i32, vp, i32, i64, i64, i64, vp]),
        "zs_bernoulli_logits_logpmf_bwd": (i32, [i32, vp, vp, vp, vp, i32, vp, i32, i64, i64, i64, vp]),
        "zs_categorical_sample": (i32, [i32, vp, vp, i32, vp, i64, i64, i64, u64, u64, vp, vp]),
        "zs_categorical_logpmf_fwd": (i32, [i32, vp, vp, i32, vp, i32, i64, i64, i64, vp]),
        "zs_categorical_logpmf_bwd": (i32, [i32, vp, vp, vp, i32, vp, i32, i64, i64, i64, vp]),
        "zs_iw_objective": (i32, [i32, i32, vp, vp, vp, vp, vp, vp, i64, i64, dbl, vp]),
        "zs_combine_sums": (i32, [i32, vp, vp, i64, dbl, vp, i64, dbl, vp]),
        "zs_log_mean_exp": (i32, [i32, vp, vp, i64, i64, vp]),
        "zs_log_mean_exp_bwd": (i32, [i32, vp, vp, vp, i64, i64, vp]),
        "zs_iw_bernoulli_fused": (i32, [i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, dbl, i32, vp]),
        "zs_iw_bernoulli_fused_loss": (i32, [i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, dbl, i32, vp]),
        "zs_scale_inplace": (i32, [i32, vp, i64, vp, i64, vp, i64, vp, vp]),
        "zs_debug_set_trace": (i32, [vp]),
        "zs_debug_set_fused_impl": (i32, [i32]),
        "zs_debug_set_latent_fwd": (i32, [i32]),
        "zs_sgld_step": (i32, [i32, vp, vp, vp, vp, i64, dbl, u64, u64, vp, vp]),
        "zs_psgld_step": (i32, [i32, vp, vp, vp, vp, vp, i64, dbl, dbl, dbl, u64, u64, vp, vp]),
        "zs_sghmc_pre": (i32, [i32, vp, vp, vp, vp, i64, dbl, i32, i32, u64, u64, vp, vp]),
        "zs_sghmc_post": (i32, [i32, vp, vp, vp, vp, vp, i64, dbl, dbl, dbl, i32, u64, u64, vp, vp]),
        "zs_sgmcmc_multi_step": (i32, [i32, i32, c.POINTER(ChainTensor), i32, dbl, dbl, dbl, i32, i32, u64, u64, vp, vp]),
        "zs_reinforce_step": (i32, [i32, vp, vp, vp, vp, vp, vp, vp, i64, dbl, dbl, vp]),
        "zs_allreduce_peer_flag_bytes": (i64, []),
        "zs_allreduce_sum_peer": (i32, [c.POINTER(vp), c.POINTER(vp), i32, i32, i64, i64, i32, i32, vp, i64, vp]),
        "zs_allreduce_sum_nvls": (i32, [vp, vp, c.POINTER(vp), i32, i32, i64, i64, i32, i32, vp, i64, vp]),
        "zs_host_step_create": (i32, [c.POINTER(vp)]),
        "zs_host_step_destroy": (i32, [vp]),
        "zs_iw_step_host_workspace": (i64, [i64, i64, i64]),
        "zs_iw_step_host": (i32, [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, dbl, vp, i64, vp]),
        "zs_iw_step_host_begin": (i32, [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, i64, i64, i64, dbl, vp, i64, i32, vp]),
        "zs_iw_step_host_wait": (i32, [vp, i32]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return sig


EXPORTS = None


def load():
    """Load the library (once).  Raises BackendError if it has not been built."""
    global _lib, EXPORTS
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise BackendError(
                "zhusuan (B200): %s not found. Build it with `python __graft_entry__.py build` "
                "(nvcc, sm_100a). There is no CPU fallback." % LIB_PATH)
        lib = ctypes.CDLL(LIB_PATH)
        EXPORTS = _declare(lib)
        if lib.zs_abi_version() != ABI_VERSION:
            raise BackendError("zhusuan (B200): %s has ABI version %d, this package needs %d; rebuild it"
                               % (LIB_PATH, lib.zs_abi_version(), ABI_VERSION))
        _lib = lib
    return _lib


def check(rc, what):
    if rc != 0:
        lib = load()
        raise BackendError("%s failed: %s (%d) %s" % (what, lib.zs_strerror(rc).decode(), rc,
                                                      lib.zs_last_error().decode()))


def require_cuda():
    if not torch.cuda.is_available():
        raise BackendError("zhusuan (B200): no CUDA device available; the hot path has no CPU fallback")


def on_compute_device(t):
    """True when `t` already lives where the kernels run (no host<->device shuttle needed)."""
    return t.is_cuda


def dtype_code(dt):
    if dt == torch.float32:
        return F32
    if dt == torch.float64:
        return F64
    raise TypeError("zhusuan (B200) kernels support float32 / float64, got %s" % dt)


def _ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _run(name, dev, *args, count=1):
    """Call entry point `name`(*args, stream) with `dev` current, on torch's current stream of `dev`.
    Returns the entry point's code (callers decide which codes mean "use another kernel")."""
    global launch_count
    fn = getattr(load(), name)
    if dev.index is None or dev.index == torch.cuda.current_device():
        rc = fn(*args, ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    else:
        with torch.cuda.device(dev):
            rc = fn(*args, ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream))
    if rc == 0:
        launch_count += count
    return rc


def _go(name, dev, *args, count=1):
    check(_run(name, dev, *args, count=count), name)


def _chk(dev, dtype, **tensors):
    """Every tensor operand: CUDA, on `dev`, contiguous, (optionally) of `dtype`."""
    for name, t in tensors.items():
        if t is None:
            continue
        if not t.is_cuda:
            raise BackendError("%s must be a CUDA tensor" % name)
        if t.device != dev:
            raise BackendError("%s lives on %s but the call's other operands are on %s; all operands of one "
                               "kernel call must share a device" % (name, t.device, dev))
        if not t.is_contiguous():
            raise BackendError("%s must be contiguous" % name)
        if dtype is not None and t.dtype != dtype:
            raise TypeError("%s has dtype %s, expected %s" % (name, t.dtype, dtype))


def _chk_state(dev, **states):
    for name, t in states.items():
        if t is None:
            continue
        if not (t.is_cuda and t.device == dev and t.dtype == torch.int64 and t.numel() >= 2 and t.is_contiguous()):
            raise BackendError("%s must be a contiguous int64[2] CUDA tensor on %s (zs_rng_state)" % (name, dev))


# ----------------------------------------------------------------------------- RNG
def rng_state_init(state, offset):
    _chk_state(state.device, rng_state=state)
    _go("zs_rng_state_init", state.device, _ptr(state), int(offset) & ((1 << 64) - 1))


def philox_raw(n, seed, offset, device, rng_state=None):
    out = torch.empty(n, dtype=torch.int32, device=device)
    _chk_state(out.device, rng_state=rng_state)
    _go("zs_philox_raw", out.device, _ptr(out), n, seed, offset, _ptr(rng_state))
    return out


def philox_uniform(n, dtype, seed, offset, device, rng_state=None):
    out = torch.empty(n, dtype=dtype, device=device)
    _chk_state(out.device, rng_state=rng_state)
    _go("zs_philox_uniform", out.device, dtype_code(dtype), _ptr(out), n, seed, offset, _ptr(rng_state))
    return out


def philox_normal(n, dtype, mean, std, seed, offset, device, rng_state=None):
    out = torch.empty(n, dtype=dtype, device=device)
    _chk_state(out.device, rng_state=rng_state)
    _go("zs_philox_normal", out.device, dtype_code(dtype), _ptr(out), n, float(mean), float(std), seed, offset,
        _ptr(rng_state))
    return out


# ----------------------------------------------------------------------------- Normal
def normal_sample(mean, mean_mode, std, std_mode, K, N, eps_in=None, eps_out=None, seed=0, offset=0, rng_state=None,
                  rng_snapshot=None):
    dt, dev = mean.dtype, mean.device
    _chk(dev, dt, mean=mean, std=std, eps_in=eps_in, eps_out=eps_out)
    _chk_state(dev, rng_state=rng_state, rng_snapshot=rng_snapshot)
    z = torch.empty((K, N), dtype=dt, device=dev)
    _go("zs_normal_sample", dev, dtype_code(dt), _ptr(z), _ptr(mean), mean_mode, _ptr(std), std_mode, _ptr(eps_in),
        _ptr(eps_out), K, N, seed, offset, _ptr(rng_state), _ptr(rng_snapshot))
    return z


def normal_sample_bwd(dz, mean_like, mean_mode, std_like, std_mode, K, N, eps=None, seed=0, offset=0,
                      need_mean=True, need_std=True, rng_state=None):
    """`rng_state`: the forward's snapshot (read, not advanced) when the noise is regenerated."""
    dt, dev = dz.dtype, dz.device
    _chk(dev, dt, dz=dz, eps=eps)
    _chk_state(dev, rng_state=rng_state)
    dmean = torch.empty_like(mean_like) if need_mean else None
    dstd = torch.empty_like(std_like) if need_std else None
    _go("zs_normal_sample_bwd", dev, dtype_code(dt), _ptr(dmean), mean_mode, _ptr(dstd), std_mode, _ptr(dz), _ptr(eps),
        K, N, seed, offset, _ptr(rng_state))
    return dmean, dstd


def normal_logprob_fwd(x, xm, mean, mm, std, sm, K, M, E):
    dt, dev = x.dtype, x.device
    _chk(dev, dt, x=x, mean=mean, std=std)
    out = torch.empty((K, M), dtype=dt, device=dev)
    _go("zs_normal_logprob_fwd", dev, dtype_code(dt), _ptr(out), _ptr(x), xm, _ptr(mean), mm, _ptr(std), sm, K, M, E)
    return out


def normal_logprob_bwd(g, x, xm, mean, mm, std, sm, K, M, E, need_x, need_mean, need_std):
    dt, dev = x.dtype, x.device
    _chk(dev, dt, g=g, x=x, mean=mean, std=std)
    dx = torch.empty_like(x) if need_x else None
    dmean = torch.empty_like(mean) if need_mean else None
    dstd = torch.empty_like(std) if need_std else None
    _go("zs_normal_logprob_bwd", dev, dtype_code(dt), _ptr(dx), _ptr(dmean), _ptr(dstd), _ptr(g), _ptr(x), xm,
        _ptr(mean), mm, _ptr(std), sm, K, M, E)
    return dx, dmean, dstd


# ----------------------------------------------------------------------------- fused latent nodes
def normal_latent_fwd(mean, std, mode, K, M, E, prior_mean=None, prior_std=None, eps_in=None, want_logq=True,
                      want_logp=True, seed=0, offset=0, rng_state=None):
    """-> (z [K,M,E], logq [K,M] | None, logp [K,M] | None), or None when the shape is not supported."""
    dt, dev = mean.dtype, mean.device
    _chk(dev, dt, mean=mean, std=std, prior_mean=prior_mean, prior_std=prior_std, eps=eps_in)
    _chk_state(dev, rng_state=rng_state)
    z = torch.empty((K, M, E), dtype=dt, device=dev)
    logq = torch.empty((K, M), dtype=dt, device=dev) if want_logq else None
    logp = torch.empty((K, M), dtype=dt, device=dev) if want_logp else None
    rc = _run("zs_normal_latent_fwd", dev, dtype_code(dt), _ptr(z), _ptr(logq), _ptr(logp), _ptr(mean), mode, _ptr(std),
              mode, _ptr(prior_mean), _ptr(prior_std), _ptr(eps_in), K, M, E, seed, offset, _ptr(rng_state))
    if rc in (ERR_UNSUPPORTED, ERR_ALIGN):
        return None
    check(rc, "zs_normal_latent_fwd")
    return z, logq, logp


def normal_latent_bwd(dlogq, dlogp, dz_up, z, mean, std, mode, K, M, E, prior_mean=None, prior_std=None,
                      reparameterized=True):
    dt, dev = z.dtype, z.device
    _chk(dev, dt, dlogq=dlogq, dlogp=dlogp, dz_up=dz_up, z=z, mean=mean, std=std, prior_mean=prior_mean,
         prior_std=prior_std)
    dmean, dstd = torch.empty_like(mean), torch.empty_like(std)
    _go("zs_normal_latent_bwd", dev, dtype_code(dt), _ptr(dmean), _ptr(dstd), _ptr(dlogq), _ptr(dlogp), _ptr(dz_up),
        _ptr(z), _ptr(mean), mode, _ptr(std), mode, _ptr(prior_mean), _ptr(prior_std), int(bool(reparameterized)), K, M, E)
    return dmean, dstd


def bernoulli_latent_fwd(probs, mode, K, M, E, prior_probs=None, u_in=None, want_logq=True, want_logp=True, seed=0,
                         offset=0, rng_state=None, want_bits=False):
    """-> (z [K,M,E], logq, logp), or None when the shape is not supported.  `want_bits=True`: a fourth element, the
    sample packed as one byte per float4 unit ([K, M, E/4] uint8; bernoulli_latent_bwd reads it instead of z), or None
    where the launch has no packed output (not float32 / KBCAST / E > 128)."""
    dt, dev = probs.dtype, probs.device
    _chk(dev, dt, probs=probs, prior_probs=prior_probs, u_in=u_in)
    _chk_state(dev, rng_state=rng_state)
    z = torch.empty((K, M, E), dtype=dt, device=dev)
    logq = torch.empty((K, M), dtype=dt, device=dev) if want_logq else None
    logp = torch.empty((K, M), dtype=dt, device=dev) if want_logp else None
    bits = None
    if want_bits and dt == torch.float32 and mode == KBCAST and E % 4 == 0 and E <= 128:
        bits = torch.empty((K, M, E // 4), dtype=torch.uint8, device=dev)
    rc = _run("zs_bernoulli_latent_fwd", dev, dtype_code(dt), _ptr(z), _ptr(logq), _ptr(logp), _ptr(probs), mode,
              _ptr(prior_probs), _ptr(u_in), K, M, E, seed, offset, _ptr(rng_state), _ptr(bits))
    if rc == ERR_UNSUPPORTED and bits is not None:  # this shape's forward kernel has no packed output
        bits = None
        rc = _run("zs_bernoulli_latent_fwd", dev, dtype_code(dt), _ptr(z), _ptr(logq), _ptr(logp), _ptr(probs), mode,
                  _ptr(prior_probs), _ptr(u_in), K, M, E, seed, offset, _ptr(rng_state), None)
    if rc in (ERR_UNSUPPORTED, ERR_ALIGN):
        return None
    check(rc, "zs_bernoulli_latent_fwd")
    return (z, logq, logp, bits) if want_bits else (z, logq, logp)


def bernoulli_latent_bwd(dlogq, z, probs, mode, K, M, E, zbits=None):
    """`zbits`: the forward's packed copy of z (bernoulli_latent_fwd(want_bits=True)); read instead of z where the
    float32 / KBCAST backward kernel runs."""
    dt, dev = z.dtype, z.device
    _chk(dev, dt, dlogq=dlogq, z=z, probs=probs)
    if zbits is not None:
        _chk(dev, torch.uint8, zbits=zbits)
        if tuple(zbits.shape) != (K, M, E // 4) or dt != torch.float32 or mode != KBCAST:
            zbits = None
    dprobs = torch.empty_like(probs)
    _go("zs_bernoulli_latent_bwd", dev, dtype_code(dt), _ptr(dprobs), _ptr(dlogq), _ptr(z), _ptr(probs), mode, K, M, E,
        _ptr(zbits))
    return dprobs


# ----------------------------------------------------------------------------- Bernoulli
def bernoulli_sample(probs, pm, K, N, u_in=None, seed=0, offset=0, rng_state=None):
    dt, dev = probs.dtype, probs.device
    _chk(dev, dt, probs=probs, u_in=u_in)
    _chk_state(dev, rng_state=rng_state)
    out = torch.empty((K, N), dtype=dt, device=dev)
    _go("zs_bernoulli_sample", dev, dtype_code(dt), _ptr(out), _ptr(probs), pm, _ptr(u_in), K, N, seed, offset,
        _ptr(rng_state))
    return out


def bernoulli_logpmf_fwd(x, xm, probs, pm, K, M, E, logits=False):
    """`logits=True`: `probs` holds logits and the sigmoid is applied in registers (zs_bernoulli_logits_logpmf_fwd)."""
    dt, dev = probs.dtype, probs.device
    _chk(dev, dt, x=x, probs=probs)
    out = torch.empty((K, M), dtype=dt, device=dev)
    name = "zs_bernoulli_logits_logpmf_fwd" if logits else "zs_bernoulli_logpmf_fwd"
    _go(name, dev, dtype_code(dt), _ptr(out), _ptr(x), xm, _ptr(probs), pm, K, M, E)
    return out


def bernoulli_logpmf_bwd(g, x, xm, probs, pm, K, M, E, need_x, need_probs, logits=False):
    dt, dev = probs.dtype, probs.device
    _chk(dev, dt, g=g, x=x, probs=probs)
    dx = torch.empty_like(x) if need_x else None
    dprobs = torch.empty_like(probs) if need_probs else None
    name = "zs_bernoulli_logits_logpmf_bwd" if logits else "zs_bernoulli_logpmf_bwd"
    _go(name, dev, dtype_code(dt), _ptr(dx), _ptr(dprobs), _ptr(g), _ptr(x), xm, _ptr(probs), pm, K, M, E)
    return dx, dprobs


# ----------------------------------------------------------------------------- Poisson
def poisson_sample(rate, rm, K, N, seed=0, offset=0, rng_state=None):
    dt, dev = rate.dtype, rate.device
    _chk(dev, dt, rate=rate)
    _chk_state(dev, rng_state=rng_state)
    out = torch.empty((K, N), dtype=dt, device=dev)
    _go("zs_poisson_sample", dev, dtype_code(dt), _ptr(out), _ptr(rate), rm, K, N, seed, offset, _ptr(rng_state))
    return out


def poisson_logpmf_fwd(x, xm, rate, rm, K, M, E):
    dt, dev = rate.dtype, rate.device
    _chk(dev, dt, x=x, rate=rate)
    out = torch.empty((K, M), dtype=dt, device=dev)
    _go("zs_poisson_logpmf_fwd", dev, dtype_code(dt), _ptr(out), _ptr(x), xm, _ptr(rate), rm, K, M, E)
    return out


def poisson_logpmf_bwd(g, x, xm, rate, rm, K, M, E):
    dt, dev = rate.dtype, rate.device
    _chk(dev, dt, g=g, x=x, rate=rate)
    drate = torch.empty_like(rate)
    _go("zs_poisson_logpmf_bwd", dev, dtype_code(dt), _ptr(drate), _ptr(g), _ptr(x), xm, _ptr(rate), rm, K, M, E)
    return drate


# ----------------------------------------------------------------------------- Beta
def beta_sample(alpha, am, beta, bm, K, N, seed=0, offset=0, rng_state=None):
    """zs_beta_sample: [K, N] Beta(alpha, beta) samples; the log-density is locscale_logprob_* with FAM_BETA."""
    dt, dev = alpha.dtype, alpha.device
    _chk(dev, dt, alpha=alpha, beta=beta)
    _chk_state(dev, rng_state=rng_state)
    out = torch.empty((K, N), dtype=dt, device=dev)
    _go("zs_beta_sample", dev, dtype_code(dt), _ptr(out), _ptr(alpha), am, _ptr(beta), bm, K, N, seed, offset,
        _ptr(rng_state))
    return out


# ----------------------------------------------------------------------------- Logistic / Laplace
# FAM_BETA: the log-density entry points only (loc = alpha, scale = beta); its sampler is beta_sample
FAM_LOGISTIC, FAM_LAPLACE, FAM_UNIFORM, FAM_BETA = 1, 2, 3, 4


def locscale_sample(family, loc, loc_mode, scale, scale_mode, K, N, u_in=None, seed=0, offset=0, rng_state=None,
                    rng_snapshot=None):
    dt, dev = loc.dtype, loc.device
    _chk(dev, dt, loc=loc, scale=scale, u_in=u_in)
    _chk_state(dev, rng_state=rng_state, rng_snapshot=rng_snapshot)
    z = torch.empty((K, N), dtype=dt, device=dev)
    _go("zs_locscale_sample", dev, dtype_code(dt), family, _ptr(z), _ptr(loc), loc_mode, _ptr(scale), scale_mode,
        _ptr(u_in), K, N, seed, offset, _ptr(rng_state), _ptr(rng_snapshot))
    return z


def locscale_sample_bwd(family, dz, loc_like, loc_mode, scale_like, scale_mode, K, N, u=None, seed=0, offset=0,
                        need_loc=True, need_scale=True, rng_state=None):
    dt, dev = dz.dtype, dz.device
    _chk(dev, dt, dz=dz, u=u)
    _chk_state(dev, rng_state=rng_state)
    dloc = torch.empty_like(loc_like) if need_loc else None
    dscale = torch.empty_like(scale_like) if need_scale else None
    _go("zs_locscale_sample_bwd", dev, dtype_code(dt), family, _ptr(dloc), loc_mode, _ptr(dscale), scale_mode, _ptr(dz),
        _ptr(u), K, N, seed, offset, _ptr(rng_state))
    return dloc, dscale


def locscale_logprob_fwd(family, x, xm, loc, lm, scale, sm, K, M, E):
    dt, dev = x.dtype, x.device
    _chk(dev, dt, x=x, loc=loc, scale=scale)
    out = torch.empty((K, M), dtype=dt, device=dev)
    _go("zs_locscale_logprob_fwd", dev, dtype_code(dt), family, _ptr(out), _ptr(x), xm, _ptr(loc), lm, _ptr(scale), sm,
        K, M, E)
    return out


def locscale_logprob_bwd(family, g, x, xm, loc, lm, scale, sm, K, M, E, need_x, need_loc, need_scale):
    dt, dev = x.dtype, x.device
    _chk(dev, dt, g=g, x=x, loc=loc, scale=scale)
    dx = torch.empty_like(x) if need_x else None
    dloc = torch.empty_like(loc) if need_loc else None
    dscale = torch.empty_like(scale) if need_scale else None
    _go("zs_locscale_logprob_bwd", dev, dtype_code(dt), family, _ptr(dx), _ptr(dloc), _ptr(dscale), _ptr(g), _ptr(x), xm,
        _ptr(loc), lm, _ptr(scale), sm, K, M, E)
    return dx, dloc, dscale


# ----------------------------------------------------------------------------- Categorical
def categorical_sample(logits, lm, K, M, C, u_in=None, seed=0, offset=0, rng_state=None):
    dt, dev = logits.dtype, logits.device
    _chk(dev, dt, logits=logits, u_in=u_in)
    _chk_state(dev, rng_state=rng_state)
    out = torch.empty((K, M), dtype=dt, device=dev)
    _go("zs_categorical_sample", dev, dtype_code(dt), _ptr(out), _ptr(logits), lm, _ptr(u_in), K, M, C, seed, offset,
        _ptr(rng_state))
    return out


def categorical_logpmf_fwd(x, xm, logits, lm, K, M, C):
    dt, dev = logits.dtype, logits.device
    _chk(dev, dt, x=x, logits=logits)
    out = torch.empty((K, M), dtype=dt, device=dev)
    _go("zs_categorical_logpmf_fwd", dev, dtype_code(dt), _ptr(out), _ptr(x), xm, _ptr(logits), lm, K, M, C)
    return out


def categorical_logpmf_bwd(g, x, xm, logits, lm, K, M, C):
    dt, dev = logits.dtype, logits.device
    _chk(dev, dt, g=g, x=x, logits=logits)
    d = torch.empty_like(logits)
    _go("zs_categorical_logpmf_bwd", dev, dtype_code(dt), _ptr(d), _ptr(g), _ptr(x), xm, _ptr(logits), lm, K, M, C)
    return d


# ----------------------------------------------------------------------------- objectives
def iw_objective(estimator, logp, logq, grad_scale, extra=None, need_grads=True):
    """logp/logq [K,B] -> (cost[B], dlogp[K,B], dlogq[K,B])."""
    dt, dev = logp.dtype, logp.device
    _chk(dev, dt, logp=logp, logq=logq, extra=extra)
    K, B = logp.shape
    cost = torch.empty(B, dtype=dt, device=dev)
    dlp = torch.empty_like(logp) if need_grads else None
    dlq = torch.empty_like(logp) if need_grads else None
    _go("zs_iw_objective", dev, dtype_code(dt), estimator, _ptr(cost), _ptr(dlp), _ptr(dlq), _ptr(logp), _ptr(logq),
        _ptr(extra), K, B, float(grad_scale))
    return cost, dlp, dlq


def combine_sums(a, scale_a, b, scale_b):
    """scale_a * a.sum() + scale_b * b.sum() as a [1] tensor, one launch (zs_combine_sums)."""
    dt, dev = a.dtype, a.device
    _chk(dev, dt, a=a, b=b)
    out = torch.empty(1, dtype=dt, device=dev)
    _go("zs_combine_sums", dev, dtype_code(dt), _ptr(out), _ptr(a), a.numel(), float(scale_a), _ptr(b), b.numel(),
        float(scale_b))
    return out


def log_mean_exp(x):
    dt, dev = x.dtype, x.device
    _chk(dev, dt, x=x)
    K, B = x.shape
    out = torch.empty(B, dtype=dt, device=dev)
    _go("zs_log_mean_exp", dev, dtype_code(dt), _ptr(out), _ptr(x), K, B)
    return out


def log_mean_exp_bwd(g, x):
    dt, dev = x.dtype, x.device
    _chk(dev, dt, g=g, x=x)
    K, B = x.shape
    dx = torch.empty_like(x)
    _go("zs_log_mean_exp_bwd", dev, dtype_code(dt), _ptr(dx), _ptr(g), _ptr(x), K, B)
    return dx


def fused_supported(K, X, dtype):
    """Shapes zs_iw_bernoulli_fused takes (the ring streams rows, so K*X need not fit anywhere)."""
    return dtype == torch.float32 and X % 4 == 0 and 1 <= K <= 4096 and X <= (1 << 20)


def fused_logits_supported(K, X, dtype):
    """Shapes the ZS_FUSED_LOGITS form takes: a fixed-geometry box kernel must be instantiated for the row
    length and a column plus one box must fit in shared memory (mirrors launch_fused_box in zs_fused_iw.cu)."""
    geo = {784: (112, 7), 128: (128, 1), 256: (256, 1), 512: (256, 2), 1024: (256, 4)}
    if dtype != torch.float32 or X not in geo or not (1 <= K <= 50):
        return False
    inner, nbox = geo[X]
    kpad = (K + 3) & ~3
    slot = (K * inner * 4 + 127) // 128 * 128
    fixed = 6 * X * 4 + 16 + 6 * kpad * 8 + 12 * kpad * 4 + 64
    return (nbox + 1) * (slot + 16) + fixed <= 227 * 1024


def fused_poisson_supported(K, X, dtype):
    """Shapes zs_iw_poisson_fused takes: the fixed-geometry box kernel, as for the logits form."""
    return fused_logits_supported(K, X, dtype)


def set_latent_fwd_impl(impl):
    """Developer hook: -1 = by shape, 0 = lane-per-unit forward, 1 = row-per-thread forward (zs_debug_set_latent_fwd)."""
    check(load().zs_debug_set_latent_fwd(int(impl)), "zs_debug_set_latent_fwd")


def set_fused_impl(impl):
    """Developer hook: IMPL_RING | IMPL_BOX | IMPL_BOXG | IMPL_DEFAULT (tests exercise every kernel variant)."""
    check(load().zs_debug_set_fused_impl(int(impl)), "zs_debug_set_fused_impl")


# zs_iw_bernoulli_fused_loss needs one zero-initialised workspace per stream that may run the launch: a small
# per-device pool, handed out by stream id (host bookkeeping only, so it also works while a graph is being captured)
_LOSS_WS_BYTES = 8 + 2 * 160 * 8  # ZS_FUSED_LOSS_WS_BYTES
_LOSS_WS_SLOTS = 64
_tickets = {}


def _ticket_ptr(dev):
    idx = dev.index if dev.index is not None else torch.cuda.current_device()
    ent = _tickets.get(idx)
    if ent is None:
        if torch.cuda.is_current_stream_capturing():
            return None  # no allocation + memset inside a capture: the caller reduces cost[B] itself this once
        ent = _tickets[idx] = (torch.zeros(_LOSS_WS_SLOTS * _LOSS_WS_BYTES // 8, dtype=torch.int64, device=dev), {})
    words, slots = ent
    sid = torch.cuda.current_stream(dev).cuda_stream
    k = slots.get(sid)
    if k is None:
        if len(slots) >= _LOSS_WS_SLOTS:
            return None
        k = slots[sid] = len(slots)
    return ctypes.c_void_p(words.data_ptr() + _LOSS_WS_BYTES * k)


def iw_bernoulli_fused(estimator, probs, x, logp_other, logq, grad_scale, need_dprobs=True, want_logpx=False,
                       out=None, logits=False, accumulate_cost=False, cost_scaled=False, want_loss=False):
    """probs [K,B,X], x [B,X], logp_other/logq [K,B] or None.  `logits=True`: `probs` holds logits and "dprobs" is
    the gradient w.r.t. them (ZS_FUSED_LOGITS).  `accumulate_cost=True` (needs out["cost"]): the per-column
    objectives are ADDED to out["cost"] (ZS_FUSED_ACCUMULATE_COST).  `cost_scaled=True`: cost[b] already carries
    grad_scale, so cost.sum() is the mean objective (ZS_FUSED_COST_SCALED).  `want_loss=True`: the launch also writes
    sum_b cost[b] into "loss" [1] (zs_iw_bernoulli_fused_loss); "loss" is None when no counter word is available.
    Returns dict(cost[B], dprobs, dlogp, dlogq, logpx, loss) or None when the shape is not supported."""
    return _iw_fused("bernoulli", estimator, probs, x, logp_other, logq, grad_scale, need_dprobs, want_logpx, out,
                     logits, accumulate_cost, cost_scaled, want_loss)


def iw_poisson_fused(estimator, rate, x, logp_other, logq, grad_scale, need_drate=True, want_logpx=False, out=None,
                     accumulate_cost=False, cost_scaled=False, want_loss=False):
    """The fused step for a Poisson likelihood (zs_iw_poisson_fused[_loss]): rate [K,B,X], counts x [B,X]; the same
    options and results as iw_bernoulli_fused, the gradient w.r.t. the rates under the key "dprobs".  None when the
    shape is not supported."""
    return _iw_fused("poisson", estimator, rate, x, logp_other, logq, grad_scale, need_drate, want_logpx, out, False,
                     accumulate_cost, cost_scaled, want_loss)


def _iw_fused(lik, estimator, probs, x, logp_other, logq, grad_scale, need_dprobs, want_logpx, out, logits,
              accumulate_cost, cost_scaled, want_loss):
    dev = probs.device
    _chk(dev, torch.float32, probs=probs, x=x, logp_other=logp_other, logq=logq)
    K, B, X = probs.shape
    o = out if out is not None else {}
    cost = o.get("cost") if "cost" in o else torch.empty(B, dtype=torch.float32, device=dev)
    dprobs = (o.get("dprobs") if "dprobs" in o else torch.empty_like(probs)) if need_dprobs else None
    dlp = o.get("dlogp") if "dlogp" in o else torch.empty((K, B), dtype=torch.float32, device=dev)
    dlq = o.get("dlogq") if "dlogq" in o else torch.empty((K, B), dtype=torch.float32, device=dev)
    lpx = (o.get("logpx") if "logpx" in o else torch.empty((K, B), dtype=torch.float32, device=dev)) if want_logpx else None
    _chk(dev, torch.float32, cost=cost, dprobs=dprobs, dlogp=dlp, dlogq=dlq, logpx=lpx)
    flags = ((FUSED_LOGITS if logits else 0) | (FUSED_ACCUMULATE_COST if accumulate_cost else 0) |
             (FUSED_COST_SCALED if cost_scaled else 0))
    ticket = _ticket_ptr(dev) if (want_loss and B >= 1 and cost is not None) else None
    loss = None
    if ticket is not None:
        loss = o.get("loss") if "loss" in o else torch.empty(1, dtype=torch.float32, device=dev)
        _chk(dev, torch.float32, loss=loss)
        name = "zs_iw_%s_fused_loss" % lik
        rc = _run(name, dev, estimator, _ptr(loss), ticket, _ptr(cost), _ptr(dprobs), _ptr(dlp), _ptr(dlq), _ptr(lpx),
                  _ptr(probs), _ptr(x), _ptr(logp_other), _ptr(logq), K, B, X, float(grad_scale), flags)
    else:
        name = "zs_iw_%s_fused" % lik
        rc = _run(name, dev, estimator, _ptr(cost), _ptr(dprobs), _ptr(dlp), _ptr(dlq), _ptr(lpx),
                  _ptr(probs), _ptr(x), _ptr(logp_other), _ptr(logq), K, B, X, float(grad_scale), flags)
    if rc in (ERR_UNSUPPORTED, ERR_ALIGN):
        return None
    check(rc, name)
    return dict(cost=cost, dprobs=dprobs, dlogp=dlp, dlogq=dlq, logpx=lpx, loss=loss)


def reinforce_step(logp, logq, moving_mean, local_step, decay, need_grads=True):
    """ELBO.reinforce with the moving-mean baseline in one launch (zs_reinforce_step).  logp / logq: same-shaped
    contiguous CUDA tensors; moving_mean [1] float32 and local_step [1] int32 CUDA buffers, updated in place.
    Returns (cost [1], dlogp, dlogq) with the gradients of the mean surrogate."""
    dt, dev = logq.dtype, logq.device
    _chk(dev, dt, logp=logp, logq=logq)
    _chk(dev, torch.float32, moving_mean=moving_mean)
    _chk(dev, torch.int32, local_step=local_step)
    n = logq.numel()
    cost = torch.empty(1, dtype=dt, device=dev)
    dlp = torch.empty_like(logq) if need_grads else None
    dlq = torch.empty_like(logq) if need_grads else None
    _go("zs_reinforce_step", dev, dtype_code(dt), _ptr(cost), _ptr(dlp), _ptr(dlq), _ptr(moving_mean), _ptr(local_step),
        _ptr(logp), _ptr(logq), n, float(decay), 1.0 / n)
    return cost, dlp, dlq


def scale_inplace(buf, scale_dev, buf1=None, buf2=None):
    """buf *= scale_dev[0] (and buf1, buf2 when given) on the device, one launch; it exits immediately when the
    scalar is 1."""
    dt, dev = buf.dtype, buf.device
    _chk(dev, dt, buf=buf, buf1=buf1, buf2=buf2, scale=scale_dev)
    n = lambda t: 0 if t is None else t.numel()
    _go("zs_scale_inplace", dev, dtype_code(dt), _ptr(buf), n(buf), _ptr(buf1), n(buf1), _ptr(buf2), n(buf2),
        _ptr(scale_dev))


# ----------------------------------------------------------------------------- SG-MCMC
def sgld_step(w, g, lr, noise=None, seed=0, offset=0, out=None, rng_state=None):
    """Returns the updated chain state (a new tensor unless `out` is given; out may be w)."""
    dt, dev = w.dtype, w.device
    _chk(dev, dt, w=w, g=g, noise=noise, out=out)
    _chk_state(dev, rng_state=rng_state)
    out = torch.empty_like(w) if out is None else out
    _go("zs_sgld_step", dev, dtype_code(dt), _ptr(out), _ptr(w), _ptr(g), _ptr(noise), w.numel(), float(lr), seed,
        offset, _ptr(rng_state))
    return out


def psgld_step(w, aux, g, lr, decay, epsilon, noise_unit=None, seed=0, offset=0, out=None, rng_state=None):
    dt, dev = w.dtype, w.device
    _chk(dev, dt, w=w, aux=aux, g=g, noise_unit=noise_unit, out=out)
    _chk_state(dev, rng_state=rng_state)
    out = torch.empty_like(w) if out is None else out
    _go("zs_psgld_step", dev, dtype_code(dt), _ptr(out), _ptr(w), _ptr(aux), _ptr(g), _ptr(noise_unit), w.numel(),
        float(lr), float(decay), float(epsilon), seed, offset, _ptr(rng_state))
    return out


def sghmc_pre(w, v, lr, resample, second_order, v_noise=None, seed=0, offset=0, out=None, rng_state=None):
    """Velocity resample (in place on v) and, for second order, the half step; returns the new w
    (w itself when no half step is taken)."""
    dt, dev = w.dtype, w.device
    _chk(dev, dt, w=w, v=v, v_noise=v_noise, out=out)
    _chk_state(dev, rng_state=rng_state)
    if not resample and not second_order:
        return w
    if second_order:
        out = torch.empty_like(w) if out is None else out
    else:
        out = w
    _go("zs_sghmc_pre", dev, dtype_code(dt), _ptr(out), _ptr(w), _ptr(v), _ptr(v_noise), w.numel(), float(lr),
        int(bool(resample)), int(bool(second_order)), seed, offset, _ptr(rng_state))
    return out


def sghmc_post(w, v, g, lr, alpha, beta, second_order, noise=None, seed=0, offset=0, out=None, rng_state=None):
    dt, dev = w.dtype, w.device
    _chk(dev, dt, w=w, v=v, g=g, noise=noise, out=out)
    _chk_state(dev, rng_state=rng_state)
    out = torch.empty_like(w) if out is None else out
    _go("zs_sghmc_post", dev, dtype_code(dt), _ptr(out), _ptr(w), _ptr(v), _ptr(g), _ptr(noise), w.numel(), float(lr),
        float(alpha), float(beta), int(bool(second_order)), seed, offset, _ptr(rng_state))
    return out


def sgmcmc_multi_step(algorithm, ws, gs=None, states=None, noises=None, outs=None, lr=0.0, a=0.0, b=0.0, resample=False,
                      second_order=False, seed=0, offset=0, rng_state=None):
    """The update of every chain-state tensor of a sampler in ONE launch (zs_sgmcmc_multi_step).
    ws / gs / states / noises / outs: equal-length lists of same-dtype contiguous CUDA tensors (entries of gs /
    states / noises may be None where the algorithm does not read them).  outs=None allocates new states
    (SGHMC_PRE without a half step returns `ws`).  Returns the list of updated chain states."""
    n = len(ws)
    if n == 0:
        return []
    if n > CHAIN_MAX_TENSORS:
        # more tensors than one parameter table holds: consecutive calls (each consumes its own stream tick)
        res = []
        for i in range(0, n, CHAIN_MAX_TENSORS):
            j = i + CHAIN_MAX_TENSORS
            sub = lambda lst: None if lst is None else lst[i:j]
            res += sgmcmc_multi_step(algorithm, ws[i:j], sub(gs), sub(states), sub(noises), sub(outs), lr, a, b,
                                     resample, second_order, seed, offset + 4 * (i // CHAIN_MAX_TENSORS), rng_state)
        return res
    dt, dev = ws[0].dtype, ws[0].device
    _chk_state(dev, rng_state=rng_state)
    gs = gs if gs is not None else [None] * n
    states = states if states is not None else [None] * n
    noises = noises if noises is not None else [None] * n
    writes = not (algorithm == ALG_SGHMC_PRE and not second_order)
    if outs is None:
        outs = [torch.empty_like(w) for w in ws] if writes else list(ws)
    table = (ChainTensor * n)()
    for i in range(n):
        _chk(dev, dt, w=ws[i], g=gs[i], state=states[i], noise=noises[i], out=outs[i])
        table[i] = ChainTensor(outs[i].data_ptr(), ws[i].data_ptr(),
                               None if gs[i] is None else gs[i].data_ptr(),
                               None if states[i] is None else states[i].data_ptr(),
                               None if noises[i] is None else noises[i].data_ptr(), ws[i].numel())
    if algorithm == ALG_SGHMC_PRE and not resample and not second_order:
        return list(ws)
    _go("zs_sgmcmc_multi_step", dev, dtype_code(dt), int(algorithm), table, n, float(lr), float(a), float(b),
        int(bool(resample)), int(bool(second_order)), seed, offset, _ptr(rng_state))
    return outs


# ----------------------------------------------------------------------------- peer-memory all-reduce
MAX_PEERS, PEER_FLAG_SETS = 8, 4


def allreduce_peer_flag_bytes():
    return int(load().zs_allreduce_peer_flag_bytes())


def allreduce_sum_peer(buf_ptrs, flag_ptrs, rank, first, count, flag_set, device, ctas=0, extra=None, extra_index=0):
    """SUM-all-reduce floats [first, first + count) of the ranks' peer-mapped buffers (zs_allreduce_sum_peer) on
    torch's current stream of `device`.  buf_ptrs / flag_ptrs: per-rank base addresses (ints) as mapped here.
    `extra` (a 1-element float32 CUDA tensor) is stored at float index `extra_index` of this rank's buffer first."""
    world = len(buf_ptrs)
    bufs = (ctypes.c_void_p * world)(*[ctypes.c_void_p(int(p)) for p in buf_ptrs])
    flags = (ctypes.c_void_p * world)(*[ctypes.c_void_p(int(p)) for p in flag_ptrs])
    _go("zs_allreduce_sum_peer", device, bufs, flags, int(rank), world, int(first), int(count), int(flag_set), int(ctas),
        _ptr(extra), int(extra_index))


def allreduce_sum_nvls(mc_ptr, local_ptr, flag_ptrs, rank, first, count, flag_set, device, ctas=0, extra=None,
                       extra_index=0):
    """The same exchange through the NVSwitch multicast mapping `mc_ptr` of the buffer (zs_allreduce_sum_nvls)."""
    world = len(flag_ptrs)
    flags = (ctypes.c_void_p * world)(*[ctypes.c_void_p(int(p)) for p in flag_ptrs])
    _go("zs_allreduce_sum_nvls", device, ctypes.c_void_p(int(mc_ptr)), ctypes.c_void_p(int(local_ptr)), flags, int(rank),
        world, int(first), int(count), int(flag_set), int(ctas), _ptr(extra), int(extra_index))


# ----------------------------------------------------------------------------- host-buffer step (e2e)
class HostStep(object):
    """Owner of one zs_host_step handle (streams, events, "a step is in flight") on a CUDA device."""

    def __init__(self, device):
        self.device = device
        h = ctypes.c_void_p()
        with torch.cuda.device(device):
            check(load().zs_host_step_create(ctypes.byref(h)), "zs_host_step_create")
        self.handle = h

    def __del__(self):
        h, self.handle = getattr(self, "handle", None), None
        if h and _lib is not None:
            try:
                _lib.zs_host_step_destroy(h)
            except Exception:
                pass


def iw_step_host_workspace(K, B, X):
    return int(load().zs_iw_step_host_workspace(K, B, X))


def _hp(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def iw_step_host(hs, estimator, cost_h, dprobs_h, dlogp_h, dlogq_h, probs_h, x_h, other_h, logq_h, K, B, X, grad_scale,
                 ws):
    """All *_h are pinned CPU tensors (or None); ws is a device uint8 workspace.  Synchronises."""
    _go("zs_iw_step_host", ws.device, hs.handle, estimator, _hp(cost_h), _hp(dprobs_h), _hp(dlogp_h), _hp(dlogq_h),
        _hp(probs_h), _hp(x_h), _hp(other_h), _hp(logq_h), K, B, X, float(grad_scale), _ptr(ws), ws.numel())


def iw_step_host_begin(hs, estimator, cost_h, dprobs_h, dlogp, dlogq, probs_h, x_h, other, logq, K, B, X, grad_scale,
                       ws, scalars_on_device):
    """Enqueue the host-buffer step and return.  cost_h / dprobs_h / probs_h / x_h are pinned CPU tensors;
    other / logq / dlogp / dlogq are CUDA tensors [K,B] when `scalars_on_device` else pinned CPU tensors.
    Follow with iw_step_host_wait(hs, 0) (cost and every kernel done) and iw_step_host_wait(hs, 1) (dprobs landed)."""
    global launch_count
    fn = load().zs_iw_step_host_begin
    with torch.cuda.device(ws.device):
        rc = fn(hs.handle, estimator, _hp(cost_h), _hp(dprobs_h), _hp(dlogp), _hp(dlogq), _hp(probs_h), _hp(x_h),
                _hp(other), _hp(logq), K, B, X, float(grad_scale), _ptr(ws), ws.numel(), 1 if scalars_on_device else 0,
                ctypes.c_void_p(torch.cuda.current_stream(ws.device).cuda_stream))
    check(rc, "zs_iw_step_host_begin")
    launch_count += 1


def iw_step_host_wait(hs, what):
    check(load().zs_iw_step_host_wait(hs.handle, int(what)), "zs_iw_step_host_wait")
