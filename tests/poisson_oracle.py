"""CPU restatement of the Poisson node (tests/poisson_oracle.c) and the backend stand-ins that let the oracle mode of
tests/test_poisson.py run the package's host logic without a GPU -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The shared library is compiled on first use into the temporary directory (the tree may be read-only), keyed by the
source's hash.  `install(monkeypatch)` installs tests/oracle_backend.py's stand-ins plus the Poisson ones below.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import torch

from oracle import zs_oracle as O

_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "poisson_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), "zs_poisson_oracle_%d_%s.so" % (os.getuid(), tag))
        if not os.path.exists(path):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
            tmp = path + ".%d.tmp" % os.getpid()
            subprocess.check_call([cc, "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-std=c11",
                                   "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, path)
        _lib = ctypes.CDLL(path)
    return _lib


def _sfx(dt):
    return {np.float32: "f32", np.float64: "f64"}[dt]


def _p(a):
    return a.ctypes.data_as(ctypes.c_void_p)


def _i64(v):
    return ctypes.c_int64(int(v))


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def poisson_sample(rate, mode, K, N, seed, offset):
    """rate: numpy array laid out for `mode` (FULL [K*N], KBCAST [N], SCALAR [1]) -> [K, N] counts."""
    dt = rate.dtype.type
    rate = _c(rate, dt)
    out = np.empty(K * N, dt)
    getattr(lib(), "orc_poisson_sample_" + _sfx(dt))(_p(out), _p(rate), ctypes.c_int(mode), _i64(K), _i64(N),
                                                      ctypes.c_uint64(seed), ctypes.c_uint64(offset))
    return out.reshape(K, N)


def poisson_logpmf_fwd(x, xm, rate, rm, K, M, E):
    dt = rate.dtype.type
    x, rate = _c(x, dt), _c(rate, dt)
    out = np.empty(K * M, dt)
    getattr(lib(), "orc_poisson_logpmf_fwd_" + _sfx(dt))(_p(out), _p(x), ctypes.c_int(xm), _p(rate), ctypes.c_int(rm),
                                                          _i64(K), _i64(M), _i64(E))
    return out.reshape(K, M)


def poisson_logpmf_bwd(g, x, xm, rate, rm, K, M, E):
    dt = rate.dtype.type
    g, x, rate = _c(g, dt), _c(x, dt), _c(rate, dt)
    drate = np.empty(rate.size, dt)
    getattr(lib(), "orc_poisson_logpmf_bwd_" + _sfx(dt))(_p(drate), _p(g), _p(x), ctypes.c_int(xm), _p(rate),
                                                          ctypes.c_int(rm), _i64(K), _i64(M), _i64(E))
    return drate.reshape(rate.shape)


def iw_poisson_step(estimator, rate, x, logp_other, logq, grad_scale, need_drate=True):
    """The fused Poisson step restated: log-pmf -> IW objective (oracle/zs_oracle.py) -> rate gradient."""
    K, B, X = rate.shape
    lpx = poisson_logpmf_fwd(x, 1, rate, 0, K, B, X)
    lp = lpx if logp_other is None else lpx + logp_other
    lq = np.zeros_like(lpx) if logq is None else logq
    cost, dlp, dlq = O.iw_objective(estimator, lp, lq, grad_scale)
    drate = poisson_logpmf_bwd(dlp, x, 1, rate, 0, K, B, X) if need_drate else None
    return dict(cost=cost, drate=drate, dlogp=dlp, dlogq=dlq, logpx=lpx)


# ---- backend stand-ins (signatures of zhusuan._backend) ------------------------------------------------------
def _np(t):
    return None if t is None else t.detach().cpu().numpy()


def _t(a, like):
    return torch.from_numpy(np.ascontiguousarray(a)).to(like.dtype)


def be_poisson_sample(rate, rm, K, N, seed=0, offset=0, rng_state=None):
    return _t(poisson_sample(_np(rate), rm, K, N, seed, offset), rate)


def be_poisson_logpmf_fwd(x, xm, rate, rm, K, M, E):
    return _t(poisson_logpmf_fwd(_np(x), xm, _np(rate), rm, K, M, E), rate)


def be_poisson_logpmf_bwd(g, x, xm, rate, rm, K, M, E):
    return _t(poisson_logpmf_bwd(_np(g), _np(x), xm, _np(rate), rm, K, M, E), rate)


def be_iw_poisson_fused(estimator, rate, x, logp_other, logq, grad_scale, need_drate=True, want_logpx=False, out=None,
                        accumulate_cost=False, cost_scaled=False, want_loss=False):
    r = iw_poisson_step(estimator, _np(rate), _np(x), _np(logp_other), _np(logq), grad_scale, need_drate)
    cost = r["cost"] * (np.float32(grad_scale) if cost_scaled else np.float32(1.0))
    return dict(cost=_t(cost, rate), dprobs=_t(r["drate"], rate) if need_drate else None,
                dlogp=_t(r["dlogp"], rate), dlogq=_t(r["dlogq"], rate),
                logpx=_t(r["logpx"], rate) if want_logpx else None)


def install(monkeypatch):
    import oracle_backend
    from zhusuan import _backend
    oracle_backend.install(monkeypatch)
    for name in ("poisson_sample", "poisson_logpmf_fwd", "poisson_logpmf_bwd", "iw_poisson_fused"):
        monkeypatch.setattr(_backend, name, globals()["be_" + name])
