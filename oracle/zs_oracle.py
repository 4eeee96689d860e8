"""ctypes/numpy front-end of the CPU oracle — TEST INFRASTRUCTURE, NOT PRODUCT CODE.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs import
this module.  The product package (zhusuan-pytorch_b200/zhusuan) never does, and fails loudly
when its CUDA library is missing instead of falling back to anything here.

Every function takes and returns numpy arrays (float32 or float64, chosen by the inputs) and
follows the reference formula cited in oracle/zs_oracle_impl.h.
"""
import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libzs_oracle.so")

FULL, KBCAST, SCALAR = 0, 1, 2
SGVB, VIMCO = 0, 1


def build(force=False):
    """Compile oracle/libzs_oracle.so with the committed Makefile (gcc, OpenMP)."""
    src_m = max(os.path.getmtime(os.path.join(_HERE, f)) for f in ("zs_oracle.c", "zs_oracle_impl.h", "Makefile"))
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < src_m:
        env = dict(os.environ)
        env.pop("CC", None)
        subprocess.check_call(["make", "-C", _HERE, "-B", "libzs_oracle.so"], env=env,
                              stdout=subprocess.DEVNULL)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(_LIB_PATH):
            build()
        _lib = ctypes.CDLL(_LIB_PATH)
        _lib.orc_set_threads.restype = ctypes.c_int
    return _lib


def set_threads(n):
    """Set (n>0) / query the OpenMP thread count used by the oracle's parallel loops."""
    return int(lib().orc_set_threads(int(n)))


def _sfx(dt):
    if dt == np.float32:
        return "_f32"
    if dt == np.float64:
        return "_f64"
    raise TypeError("oracle supports float32 / float64, got %r" % (dt,))


def _c(a, dt):
    return np.ascontiguousarray(a, dtype=dt)


def _p(a):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def _mode(a, K, per_particle):
    """Layout mode of operand `a` for a [K, per_particle] problem."""
    n = a.size
    if n == K * per_particle and not (K == 1 and False):
        if n == per_particle and K == 1:
            return FULL
        return FULL
    if n == per_particle:
        return KBCAST
    if n == 1:
        return SCALAR
    raise ValueError("operand of size %d fits neither [K*N]=%d, [N]=%d nor [1]" % (n, K * per_particle, per_particle))


def _i64(v):
    return ctypes.c_int64(int(v))


def _call(name, dt, *args):
    getattr(lib(), name + _sfx(dt))(*args)


# --------------------------------------------------------------------------- Normal
def normal_sample(mean, std, eps, K, N):
    dt = eps.dtype.type
    mean, std, eps = _c(mean, dt), _c(std, dt), _c(eps, dt)
    z = np.empty(K * N, dt)
    _call("orc_normal_sample", dt, _p(z), _p(mean), _mode(mean, K, N), _p(std), _mode(std, K, N), _p(eps), _i64(K),
          _i64(N))
    return z.reshape(K, N)


def normal_sample_bwd(dz, eps, mean_like, std_like, K, N):
    dt = dz.dtype.type
    dz, eps = _c(dz, dt), _c(eps, dt)
    mm, sm = _mode(mean_like, K, N), _mode(std_like, K, N)
    dmean = np.zeros(mean_like.size, dt)
    dstd = np.zeros(std_like.size, dt)
    _call("orc_normal_sample_bwd", dt, _p(dmean), mm, _p(dstd), sm, _p(dz), _p(eps), _i64(K), _i64(N))
    return dmean.reshape(mean_like.shape), dstd.reshape(std_like.shape)


def normal_logprob_fwd(x, mean, std, K, M, E):
    dt = np.result_type(x, mean, std).type
    x, mean, std = _c(x, dt), _c(mean, dt), _c(std, dt)
    out = np.empty(K * M, dt)
    _call("orc_normal_logprob_fwd", dt, _p(out), _p(x), _mode(x, K, M * E), _p(mean), _mode(mean, K, M * E), _p(std),
          _mode(std, K, M * E), _i64(K), _i64(M), _i64(E))
    return out.reshape(K, M)


def normal_logprob_bwd(g, x, mean, std, K, M, E):
    dt = np.result_type(x, mean, std).type
    g, x, mean, std = _c(g, dt), _c(x, dt), _c(mean, dt), _c(std, dt)
    dx, dmean, dstd = np.zeros(x.size, dt), np.zeros(mean.size, dt), np.zeros(std.size, dt)
    _call("orc_normal_logprob_bwd", dt, _p(dx), _p(dmean), _p(dstd), _p(g), _p(x), _mode(x, K, M * E), _p(mean),
          _mode(mean, K, M * E), _p(std), _mode(std, K, M * E), _i64(K), _i64(M), _i64(E))
    return dx.reshape(x.shape), dmean.reshape(mean.shape), dstd.reshape(std.shape)


# --------------------------------------------------------------------------- Bernoulli
def bernoulli_sample(probs, u, K, N):
    dt = u.dtype.type
    probs, u = _c(probs, dt), _c(u, dt)
    out = np.empty(K * N, dt)
    _call("orc_bernoulli_sample", dt, _p(out), _p(probs), _mode(probs, K, N), _p(u), _i64(K), _i64(N))
    return out.reshape(K, N)


def bernoulli_logpmf_fwd(x, probs, K, M, E):
    dt = np.result_type(x, probs).type
    x, probs = _c(x, dt), _c(probs, dt)
    out = np.empty(K * M, dt)
    _call("orc_bernoulli_logpmf_fwd", dt, _p(out), _p(x), _mode(x, K, M * E), _p(probs), _mode(probs, K, M * E),
          _i64(K), _i64(M), _i64(E))
    return out.reshape(K, M)


def bernoulli_logpmf_bwd(g, x, probs, K, M, E, need_dx=False):
    dt = np.result_type(x, probs).type
    g, x, probs = _c(g, dt), _c(x, dt), _c(probs, dt)
    dx = np.zeros(x.size, dt) if need_dx else None
    dprobs = np.zeros(probs.size, dt)
    _call("orc_bernoulli_logpmf_bwd", dt, _p(dx), _p(dprobs), _p(g), _p(x), _mode(x, K, M * E), _p(probs),
          _mode(probs, K, M * E), _i64(K), _i64(M), _i64(E))
    if need_dx:
        return dx.reshape(x.shape), dprobs.reshape(probs.shape)
    return dprobs.reshape(probs.shape)


# Bernoulli given by logits: the reference forms probs = torch.sigmoid(logits) in the operand dtype
# (zhusuan/distributions/bernoulli.py:47-50) and evaluates the log-pmf above (:84-95); autograd of torch.sigmoid
# is grad * (1 - p) * p.  Restated in numpy on top of the C functions above.
def sigmoid(logits):
    dt = logits.dtype.type
    return (dt(1) / (dt(1) + np.exp(-logits))).astype(dt)


def bernoulli_logits_logpmf_fwd(x, logits, K, M, E):
    return bernoulli_logpmf_fwd(x, sigmoid(np.asarray(logits)), K, M, E)


def bernoulli_logits_logpmf_bwd(g, x, logits, K, M, E, need_dx=False):
    p = sigmoid(np.asarray(logits))
    r = bernoulli_logpmf_bwd(g, x, p, K, M, E, need_dx=need_dx)
    dx, dp = r if need_dx else (None, r)
    dl = (dp * ((1 - p) * p)).astype(p.dtype)
    return (dx, dl) if need_dx else dl


def iw_bernoulli_logits_step(estimator, logits, x, logp_other, logq, grad_scale=None, need_dprobs=True):
    """iw_bernoulli_step for a likelihood given by logits; "dprobs" of the result is the gradient w.r.t. the logits."""
    p = sigmoid(np.asarray(logits))
    r = iw_bernoulli_step(estimator, p, x, logp_other, logq, grad_scale, need_dprobs)
    if need_dprobs:
        r["dprobs"] = (r["dprobs"] * ((1 - p) * p)).astype(p.dtype)
    return r


# --------------------------------------------------------------------------- Logistic / Laplace (numpy restatement)
LOGISTIC, LAPLACE, UNIFORM = 1, 2, 3


def locscale_noise(family, u):
    """eps of z = loc + scale * eps.  Logistic: log u - log(1 - u), u ~ U(0,1) (zhusuan/distributions/logistic.py:66-67);
    Laplace: -sign(u) log1p(-|u|), u ~ U(-1,1) (torch.distributions.Laplace.sample, called by laplace.py:74)."""
    u = np.asarray(u)
    if family == UNIFORM:  # Uniform draws u ~ U[0,1) itself (torch.rand; zhusuan/distributions/uniform.py:63-66)
        return u
    if family == LOGISTIC:
        return (np.log(u) - np.log(1 - u)).astype(u.dtype)
    return (-np.sign(u) * np.log1p(-np.abs(u))).astype(u.dtype)


def locscale_sample(family, loc, scale, u, K, N):
    eps = locscale_noise(family, np.asarray(u).reshape(K, N))
    loc, scale = np.asarray(loc).reshape(-1, N), np.asarray(scale).reshape(-1, N)
    return (loc + scale * eps).astype(eps.dtype)                      # logistic.py:68 / Laplace.rsample


def locscale_sample_bwd(family, dz, u, K, N, full=False):
    """Pathwise gradient of the sample: (dloc, dscale), summed over K unless `full`."""
    eps = locscale_noise(family, np.asarray(u).reshape(K, N))
    dz = np.asarray(dz).reshape(K, N)
    if full:
        return dz.copy(), (dz * eps).astype(dz.dtype)
    return dz.sum(0).astype(dz.dtype), (dz * eps).sum(0).astype(dz.dtype)


def _softplus(v):
    return np.where(v > 20, v, np.log1p(np.exp(np.minimum(v, 20))))   # torch.nn.Softplus (threshold 20)


def locscale_logprob_fwd(family, x, loc, scale, K, M, E):
    dt = np.result_type(x, loc, scale).type
    x, loc, scale = (np.broadcast_to(np.asarray(a, dt).reshape((-1, M, E)), (K, M, E)) for a in (x, loc, scale))
    if family == UNIFORM:  # loc = low, scale = high: torch.distributions.Uniform.log_prob (uniform.py:81)
        with np.errstate(divide="ignore"):
            lp = np.log(((loc <= x) & (x < scale)).astype(dt)) - np.log(scale - loc)
    elif family == LOGISTIC:
        z = (x - loc) / scale                                          # logistic.py:81
        lp = -z - 2 * _softplus(-z) - np.log(scale)                    # logistic.py:82
    else:
        lp = -np.log(2 * scale) - np.abs(x - loc) / scale              # torch Laplace.log_prob (laplace.py:92)
    return lp.astype(dt).sum(-1).astype(dt)


def locscale_logprob_bwd(family, g, x, loc, scale, K, M, E):
    """Autograd of the expressions above for upstream g[K,M]: (dx, dloc, dscale), each reduced to its operand's
    shape ([K,M,E] or [M,E])."""
    dt = np.result_type(x, loc, scale).type
    shapes = [np.asarray(a).reshape((-1, M, E)).shape for a in (x, loc, scale)]
    x, loc, scale = (np.broadcast_to(np.asarray(a, dt).reshape((-1, M, E)), (K, M, E)) for a in (x, loc, scale))
    g = np.asarray(g, dt).reshape(K, M, 1)
    if family == UNIFORM:  # autograd sees only -log(high - low): (dx, dlow, dhigh) = (0, g/(high-low), -g/(high-low))
        r = (g / (scale - loc)).astype(dt)
        outs = []
        for grad, shp in zip((np.zeros_like(r), r, -r), shapes):
            outs.append(grad if shp[0] == K and K > 1 or shp == (K, M, E) else grad.sum(0, keepdims=True).astype(dt))
        return tuple(o.reshape(s_) for o, s_ in zip(outs, shapes))
    if family == LOGISTIC:
        z = (x - loc) / scale
        with np.errstate(over="ignore"):
            sgm = np.where(-z > 20, 1.0, 1.0 / (1.0 + np.exp(z)))
        dz = g * (-1 + 2 * sgm)
        dx = dz / scale
        dscale = -(dz * z) / scale - g / scale
    else:
        d = x - loc
        dx = -(g * np.sign(d)) / scale
        dscale = -g / scale + (g * np.abs(d)) / (scale * scale)
    outs = []
    for grad, shp in zip((dx, -dx, dscale), shapes):
        grad = grad.astype(dt)
        outs.append(grad if shp[0] == K and K > 1 or shp == (K, M, E) else grad.sum(0, keepdims=True).astype(dt))
    return tuple(o.reshape(s) for o, s in zip(outs, shapes))


# --------------------------------------------------------------------------- Categorical (parity unpinned)
def categorical_logpmf_fwd(x, logits, K, M, C):
    dt = logits.dtype.type
    x, logits = _c(x, dt), _c(logits, dt)
    out = np.empty(K * M, dt)
    lm = FULL if logits.size == K * M * C else KBCAST
    _call("orc_categorical_logpmf_fwd", dt, _p(out), _p(x), _mode(x, K, M), _p(logits), lm, _i64(K), _i64(M), _i64(C))
    return out.reshape(K, M)


def categorical_logpmf_bwd(g, x, logits, K, M, C):
    dt = logits.dtype.type
    g, x, logits = _c(g, dt), _c(x, dt), _c(logits, dt)
    lm = FULL if logits.size == K * M * C else KBCAST
    d = np.zeros(logits.size, dt)
    _call("orc_categorical_logpmf_bwd", dt, _p(d), _p(g), _p(x), _mode(x, K, M), _p(logits), lm, _i64(K), _i64(M),
          _i64(C))
    return d.reshape(logits.shape)


def categorical_sample(logits, u, K, M, C):
    dt = logits.dtype.type
    logits, u = _c(logits, dt), _c(u, dt)
    lm = FULL if logits.size == K * M * C else KBCAST
    out = np.empty(K * M, dt)
    _call("orc_categorical_sample", dt, _p(out), _p(logits), lm, _p(u), _i64(K), _i64(M), _i64(C))
    return out.reshape(K, M)


# --------------------------------------------------------------------------- Poisson (explicit operand modes)
def poisson_sample(rate, mode, K, N, seed, offset):
    """rate: numpy array laid out for `mode` (FULL [K*N], KBCAST [N], SCALAR [1]) -> [K, N] counts."""
    dt = rate.dtype.type
    rate = _c(rate, dt)
    out = np.empty(K * N, dt)
    _call("orc_poisson_sample", dt, _p(out), _p(rate), mode, _i64(K), _i64(N), ctypes.c_uint64(seed),
          ctypes.c_uint64(offset))
    return out.reshape(K, N)


def poisson_logpmf_fwd(x, xm, rate, rm, K, M, E):
    dt = rate.dtype.type
    x, rate = _c(x, dt), _c(rate, dt)
    out = np.empty(K * M, dt)
    _call("orc_poisson_logpmf_fwd", dt, _p(out), _p(x), xm, _p(rate), rm, _i64(K), _i64(M), _i64(E))
    return out.reshape(K, M)


def poisson_logpmf_bwd(g, x, xm, rate, rm, K, M, E):
    dt = rate.dtype.type
    g, x, rate = _c(g, dt), _c(x, dt), _c(rate, dt)
    drate = np.empty(rate.size, dt)
    _call("orc_poisson_logpmf_bwd", dt, _p(drate), _p(g), _p(x), xm, _p(rate), rm, _i64(K), _i64(M), _i64(E))
    return drate.reshape(rate.shape)


def iw_poisson_step(estimator, rate, x, logp_other, logq, grad_scale, need_drate=True):
    """The fused Poisson step restated: log-pmf -> IW objective -> rate gradient.
    rate [K,B,X], x [B,X], logp_other/logq [K,B] or None.  Returns dict(cost, drate, dlogp, dlogq, logpx)."""
    K, B, X = rate.shape
    lpx = poisson_logpmf_fwd(x, KBCAST, rate, FULL, K, B, X)
    lp = lpx if logp_other is None else lpx + logp_other
    lq = np.zeros_like(lpx) if logq is None else logq
    cost, dlp, dlq = iw_objective(estimator, lp, lq, grad_scale)
    drate = poisson_logpmf_bwd(dlp, x, KBCAST, rate, FULL, K, B, X) if need_drate else None
    return dict(cost=cost, drate=drate, dlogp=dlp, dlogq=dlq, logpx=lpx)


# --------------------------------------------------------------------------- Beta (explicit operand modes)
def digamma(x, dtype=np.float64):
    """psi as the Beta gradients evaluate it, elementwise in `dtype`."""
    f = getattr(lib(), "orc_digamma" + _sfx(dtype))
    f.restype, f.argtypes = ctypes.c_double, [ctypes.c_double]
    return np.array([f(float(v)) for v in np.ravel(x)], dtype).reshape(np.shape(x))


def beta_sample(alpha, am, beta, bm, K, N, seed, offset):
    """alpha / beta: numpy arrays laid out for their modes (FULL [K*N], KBCAST [N], SCALAR [1]) -> [K, N] samples."""
    dt = alpha.dtype.type
    alpha, beta = _c(alpha, dt), _c(beta, dt)
    out = np.empty(K * N, dt)
    _call("orc_beta_sample", dt, _p(out), _p(alpha), am, _p(beta), bm, _i64(K), _i64(N), ctypes.c_uint64(seed),
          ctypes.c_uint64(offset))
    return out.reshape(K, N)


def beta_logprob_fwd(x, xm, a, am, b, bm, K, M, E):
    dt = a.dtype.type
    x, a, b = _c(x, dt), _c(a, dt), _c(b, dt)
    out = np.empty(K * M, dt)
    _call("orc_beta_logprob_fwd", dt, _p(out), _p(x), xm, _p(a), am, _p(b), bm, _i64(K), _i64(M), _i64(E))
    return out.reshape(K, M)


def beta_logprob_bwd(g, x, xm, a, am, b, bm, K, M, E, need=(True, True, True)):
    """(dx, da, db), each with the layout of its operand (None where not needed)."""
    dt = a.dtype.type
    g, x, a, b = _c(g, dt), _c(x, dt), _c(a, dt), _c(b, dt)
    outs = [np.empty(v.size, dt) if n else None for v, n in zip((x, a, b), need)]
    _call("orc_beta_logprob_bwd", dt, *[_p(o) for o in outs], _p(g), _p(x), xm, _p(a), am, _p(b), bm, _i64(K),
          _i64(M), _i64(E))
    return tuple(None if o is None else o.reshape(v.shape) for o, v in zip(outs, (x, a, b)))


# --------------------------------------------------------------------------- objectives
def log_mean_exp(x):
    """axis-0 log_mean_exp of [K,B] (zhusuan/utils.py:6-21)."""
    dt = x.dtype.type
    x = _c(x, dt)
    K, B = x.shape
    out = np.empty(B, dt)
    _call("orc_log_mean_exp", dt, _p(out), _p(x), _i64(K), _i64(B))
    return out


def iw_objective(estimator, logp, logq, grad_scale=None):
    """Returns (cost[B], dlogp[K,B], dlogq[K,B]); gradients are of sum_b cost_b * grad_scale
    (default 1/B, i.e. of the reference's `.mean()` loss)."""
    dt = np.result_type(logp, logq).type
    logp, logq = _c(logp, dt), _c(logq, dt)
    if logp.ndim == 1:
        logp, logq = logp[:, None], logq[:, None]
    K, B = logp.shape
    gs = (1.0 / B) if grad_scale is None else grad_scale
    cost, dlp, dlq = np.empty(B, dt), np.empty((K, B), dt), np.empty((K, B), dt)
    name = "orc_iw_sgvb" if estimator == SGVB else "orc_iw_vimco"
    gs_c = ctypes.c_float(gs) if dt == np.float32 else ctypes.c_double(gs)
    _call(name, dt, _p(cost), _p(dlp), _p(dlq), _p(logp), _p(logq), _i64(K), _i64(B), gs_c)
    return cost, dlp, dlq


def iw_bernoulli_step(estimator, probs, x, logp_other, logq, grad_scale=None, need_dprobs=True):
    """One importance-weighted step of the Bernoulli-likelihood path (the bench workload).
    probs [K,B,X], x [B,X], logp_other/logq [K,B] or None.
    Returns dict(cost, dprobs, dlogp, dlogq, logpx)."""
    dt = probs.dtype.type
    probs, x = _c(probs, dt), _c(x, dt)
    K, B, X = probs.shape
    lo = None if logp_other is None else _c(logp_other, dt)
    lq = None if logq is None else _c(logq, dt)
    gs = (1.0 / B) if grad_scale is None else grad_scale
    cost, dlp, dlq, lpx = np.empty(B, dt), np.empty((K, B), dt), np.empty((K, B), dt), np.empty((K, B), dt)
    dprobs = np.empty((K, B, X), dt) if need_dprobs else None
    gs_c = ctypes.c_float(gs) if dt == np.float32 else ctypes.c_double(gs)
    _call("orc_iw_bernoulli_step", dt, ctypes.c_int(estimator), _p(cost), _p(dprobs), _p(dlp), _p(dlq), _p(lpx),
          _p(probs), _p(x), _p(lo), _p(lq), _i64(K), _i64(B), _i64(X), gs_c)
    return dict(cost=cost, dprobs=dprobs, dlogp=dlp, dlogq=dlq, logpx=lpx)


def reinforce_step(logp, logq, moving_mean, local_step, decay=0.8, grad_scale=None):
    """ELBO.reinforce with the moving-mean baseline (elbo.py:200-238).  Returns (cost, dlogp, dlogq,
    new moving_mean (float32), new local_step)."""
    dt = np.result_type(logp, logq).type
    shape = np.shape(logp)
    logp, logq = _c(logp, dt).reshape(-1), _c(logq, dt).reshape(-1)
    n = logp.size
    gs = (1.0 / n) if grad_scale is None else grad_scale
    cost, dlp, dlq = np.empty(1, dt), np.empty(n, dt), np.empty(n, dt)
    mm = np.array([moving_mean], np.float32).reshape(1)
    ls = np.array([local_step], np.int32).reshape(1)
    gs_c = ctypes.c_float(gs) if dt == np.float32 else ctypes.c_double(gs)
    _call("orc_reinforce_step", dt, _p(cost), _p(dlp), _p(dlq), _p(mm), _p(ls), _p(logp), _p(logq), _i64(n),
          ctypes.c_double(decay), gs_c)
    return cost[0], dlp.reshape(shape), dlq.reshape(shape), mm[0], int(ls[0])


# --------------------------------------------------------------------------- SG-MCMC (in place on copies)
def sgld_step(w, g, noise, lr):
    dt = w.dtype.type
    w = np.array(w, dtype=dt, copy=True)
    _call("orc_sgld_step", dt, _p(w), _p(_c(g, dt)), _p(_c(noise, dt)), _i64(w.size), ctypes.c_double(lr))
    return w


def psgld_step(w, aux, g, unit, lr, decay=0.9, epsilon=1e-3):
    dt = w.dtype.type
    w, aux = np.array(w, dtype=dt, copy=True), np.array(aux, dtype=dt, copy=True)
    _call("orc_psgld_step", dt, _p(w), _p(aux), _p(_c(g, dt)), _p(_c(unit, dt)), _i64(w.size), ctypes.c_double(lr),
          ctypes.c_double(decay), ctypes.c_double(epsilon))
    return w, aux


def sghmc_pre(w, v, v_noise, resample, second_order):
    dt = w.dtype.type
    w, v = np.array(w, dtype=dt, copy=True), np.array(v, dtype=dt, copy=True)
    vn = _c(v_noise if v_noise is not None else np.zeros_like(v), dt)
    _call("orc_sghmc_pre", dt, _p(w), _p(v), _p(vn), _i64(w.size), ctypes.c_int(int(resample)),
          ctypes.c_int(int(second_order)))
    return w, v


def sghmc_post(w, v, g, noise, lr, alpha, second_order):
    dt = w.dtype.type
    w, v = np.array(w, dtype=dt, copy=True), np.array(v, dtype=dt, copy=True)
    _call("orc_sghmc_post", dt, _p(w), _p(v), _p(_c(g, dt)), _p(_c(noise, dt)), _i64(w.size), ctypes.c_double(lr),
          ctypes.c_double(alpha), ctypes.c_int(int(second_order)))
    return w, v


# --------------------------------------------------------------------------- Philox
def philox_kat(ctr, key):
    c = (ctypes.c_uint32 * 4)(*ctr)
    k = (ctypes.c_uint32 * 2)(*key)
    o = (ctypes.c_uint32 * 4)()
    lib().orc_philox_kat(o, c, k)
    return [int(v) for v in o]


def philox_raw(n, seed, offset):
    out = np.empty(n, np.uint32)
    lib().orc_philox_raw(_p(out), _i64(n), ctypes.c_uint64(seed), ctypes.c_uint64(offset))
    return out


def philox_uniform(n, seed, offset):
    out = np.empty(n, np.float32)
    lib().orc_philox_uniform_f32(_p(out), _i64(n), ctypes.c_uint64(seed), ctypes.c_uint64(offset))
    return out


def philox_uniform_open(n, seed, offset):
    out = np.empty(n, np.float32)
    lib().orc_philox_uniform_open_f32(_p(out), _i64(n), ctypes.c_uint64(seed), ctypes.c_uint64(offset))
    return out


def philox_normal(n, seed, offset, mean=0.0, std=1.0):
    out = np.empty(n, np.float32)
    lib().orc_philox_normal_f32(_p(out), _i64(n), ctypes.c_float(mean), ctypes.c_float(std), ctypes.c_uint64(seed),
                                ctypes.c_uint64(offset))
    return out
