"""CPU restatement of the Beta node (tests/beta_oracle.c) and the backend stand-ins that let the oracle mode of
tests/test_beta.py run the package's host logic without a GPU -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The shared library is compiled on first use into the temporary directory (the tree may be read-only), keyed by the
source's hash.  `install(monkeypatch)` installs tests/oracle_backend.py's stand-ins plus the Beta ones below; the
log-density stand-ins take family 4 (Beta) and hand every other family to oracle_backend.
"""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import torch

FAM_BETA = 4
_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "beta_oracle.c")
_lib = None


def lib():
    global _lib
    if _lib is None:
        src = open(_SRC, "rb").read()
        tag = hashlib.sha256(src).hexdigest()[:16]
        path = os.path.join(tempfile.gettempdir(), "zs_beta_oracle_%d_%s.so" % (os.getuid(), tag))
        if not os.path.exists(path):
            cc = "/usr/bin/gcc" if os.path.exists("/usr/bin/gcc") else "gcc"
            tmp = path + ".%d.tmp" % os.getpid()
            subprocess.check_call([cc, "-O2", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-std=c11",
                                   "-o", tmp, _SRC, "-lm"])
            os.replace(tmp, path)
        _lib = ctypes.CDLL(path)
        for sfx in ("f32", "f64"):
            f = getattr(_lib, "orc_digamma_" + sfx)
            f.restype, f.argtypes = ctypes.c_double, [ctypes.c_double]
    return _lib


def _sfx(dt):
    return {np.float32: "f32", np.float64: "f64"}[dt]


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _i64(v):
    return ctypes.c_int64(int(v))


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def digamma(x, dtype=np.float64):
    f = getattr(lib(), "orc_digamma_" + _sfx(dtype))
    return np.array([f(float(v)) for v in np.ravel(x)], dtype).reshape(np.shape(x))


def beta_sample(alpha, am, beta, bm, K, N, seed, offset):
    """alpha / beta: numpy arrays laid out for their modes (FULL [K*N], KBCAST [N], SCALAR [1]) -> [K, N] samples."""
    dt = alpha.dtype.type
    alpha, beta = _c(alpha, dt), _c(beta, dt)
    out = np.empty(K * N, dt)
    getattr(lib(), "orc_beta_sample_" + _sfx(dt))(_p(out), _p(alpha), ctypes.c_int(am), _p(beta), ctypes.c_int(bm),
                                                   _i64(K), _i64(N), ctypes.c_uint64(seed), ctypes.c_uint64(offset))
    return out.reshape(K, N)


def beta_logprob_fwd(x, xm, a, am, b, bm, K, M, E):
    dt = a.dtype.type
    x, a, b = _c(x, dt), _c(a, dt), _c(b, dt)
    out = np.empty(K * M, dt)
    getattr(lib(), "orc_beta_logprob_fwd_" + _sfx(dt))(_p(out), _p(x), ctypes.c_int(xm), _p(a), ctypes.c_int(am),
                                                        _p(b), ctypes.c_int(bm), _i64(K), _i64(M), _i64(E))
    return out.reshape(K, M)


def beta_logprob_bwd(g, x, xm, a, am, b, bm, K, M, E, need=(True, True, True)):
    """(dx, da, db), each with the layout of its operand (None where not needed)."""
    dt = a.dtype.type
    g, x, a, b = _c(g, dt), _c(x, dt), _c(a, dt), _c(b, dt)
    outs = [np.empty(v.size, dt) if n else None for v, n in zip((x, a, b), need)]
    getattr(lib(), "orc_beta_logprob_bwd_" + _sfx(dt))(*[_p(o) for o in outs], _p(g), _p(x), ctypes.c_int(xm), _p(a),
                                                        ctypes.c_int(am), _p(b), ctypes.c_int(bm), _i64(K), _i64(M),
                                                        _i64(E))
    return tuple(None if o is None else o.reshape(v.shape) for o, v in zip(outs, (x, a, b)))


# ---- backend stand-ins (signatures of zhusuan._backend) ------------------------------------------------------
def _np(t):
    return None if t is None else t.detach().cpu().numpy()


def _t(a, like):
    return torch.from_numpy(np.ascontiguousarray(a)).to(like.dtype)


def install(monkeypatch):
    import oracle_backend
    from zhusuan import _backend
    oracle_backend.install(monkeypatch)
    other_fwd, other_bwd = _backend.locscale_logprob_fwd, _backend.locscale_logprob_bwd

    def be_locscale_logprob_fwd(family, x, xm, loc, lm, scale, sm, K, M, E):
        if family != FAM_BETA:
            return other_fwd(family, x, xm, loc, lm, scale, sm, K, M, E)
        return _t(beta_logprob_fwd(_np(x), xm, _np(loc), lm, _np(scale), sm, K, M, E), x)

    def be_locscale_logprob_bwd(family, g, x, xm, loc, lm, scale, sm, K, M, E, need_x, need_loc, need_scale):
        if family != FAM_BETA:
            return other_bwd(family, g, x, xm, loc, lm, scale, sm, K, M, E, need_x, need_loc, need_scale)
        outs = beta_logprob_bwd(_np(g), _np(x), xm, _np(loc), lm, _np(scale), sm, K, M, E,
                                need=(need_x, need_loc, need_scale))
        return tuple(None if o is None else _t(o, x) for o in outs)

    def be_beta_sample(alpha, am, beta, bm, K, N, seed=0, offset=0, rng_state=None):
        return _t(beta_sample(_np(alpha), am, _np(beta), bm, K, N, seed, offset), alpha)

    monkeypatch.setattr(_backend, "locscale_logprob_fwd", be_locscale_logprob_fwd)
    monkeypatch.setattr(_backend, "locscale_logprob_bwd", be_locscale_logprob_bwd)
    monkeypatch.setattr(_backend, "beta_sample", be_beta_sample)
