"""TEST-ONLY stand-in for zhusuan._backend built on the CPU oracle.

`install(monkeypatch)` replaces the ctypes entry points of the product's backend with oracle-based
implementations on CPU tensors, so the host logic of the package (layouts, autograd wiring,
StochasticTensor / BayesianNet semantics, objective assembly, sampler state machines) can be tested in
the CPU container.  The product never imports this module; `-m gpu` tests run the same scenarios
against the real kernels.
"""
import numpy as np
import torch

from oracle import zs_oracle as O

FULL, KBCAST, SCALAR = 0, 1, 2


def _np(t):
    return None if t is None else t.detach().cpu().numpy()


def _t(a, like):
    return torch.from_numpy(np.ascontiguousarray(a)).to(like.dtype)


def normal_sample(mean, mean_mode, std, std_mode, K, N, eps_in=None, eps_out=None, seed=0, offset=0, rng_state=None,
                  rng_snapshot=None):
    if eps_in is None:
        eps = O.philox_normal(K * N, seed, offset).astype(_np(mean).dtype).reshape(K, N)
    else:
        eps = _np(eps_in).reshape(K, N)
    if eps_out is not None:
        eps_out.copy_(_t(eps, mean))
    return _t(O.normal_sample(_np(mean), _np(std), eps, K, N), mean)


def normal_sample_bwd(dz, mean_like, mean_mode, std_like, std_mode, K, N, eps=None, seed=0, offset=0,
                      need_mean=True, need_std=True, rng_state=None):
    e = O.philox_normal(K * N, seed, offset).astype(_np(dz).dtype).reshape(K, N) if eps is None else _np(eps).reshape(K, N)
    dm, ds = O.normal_sample_bwd(_np(dz).reshape(K, N), e, _np(mean_like), _np(std_like), K, N)
    return (_t(dm, dz) if need_mean else None), (_t(ds, dz) if need_std else None)


def normal_logprob_fwd(x, xm, mean, mm, std, sm, K, M, E):
    return _t(O.normal_logprob_fwd(_np(x), _np(mean), _np(std), K, M, E), x)


def normal_logprob_bwd(g, x, xm, mean, mm, std, sm, K, M, E, need_x, need_mean, need_std):
    dx, dm, ds = O.normal_logprob_bwd(_np(g), _np(x), _np(mean), _np(std), K, M, E)
    return (_t(dx, x) if need_x else None, _t(dm, x) if need_mean else None, _t(ds, x) if need_std else None)


def normal_latent_fwd(mean, std, mode, K, M, E, prior_mean=None, prior_std=None, eps_in=None, want_logq=True,
                      want_logp=True, seed=0, offset=0, rng_state=None):
    dt = _np(mean).dtype
    eps = (O.philox_normal(K * M * E, seed, offset).astype(dt) if eps_in is None else _np(eps_in)).reshape(K, M * E)
    z = O.normal_sample(_np(mean), _np(std), eps, K, M * E).reshape(K, M, E)
    logq = O.normal_logprob_fwd(z, _np(mean), _np(std), K, M, E) if want_logq else None
    logp = None
    if want_logp:
        pm_ = np.zeros((M, E), dt) if prior_mean is None else _np(prior_mean)
        ps_ = np.ones((M, E), dt) if prior_std is None else _np(prior_std)
        logp = O.normal_logprob_fwd(z, pm_, ps_, K, M, E)
    return _t(z, mean), None if logq is None else _t(logq, mean), None if logp is None else _t(logp, mean)


def normal_latent_bwd(dlogq, dlogp, dz_up, z, mean, std, mode, K, M, E, prior_mean=None, prior_std=None,
                      reparameterized=True):
    dt = _np(z).dtype
    zz, m, sd = _np(z).reshape(K, M, E), _np(mean), _np(std)
    gq = np.zeros((K, M), dt) if dlogq is None else _np(dlogq).reshape(K, M)
    dz_q, dm, ds = O.normal_logprob_bwd(gq, zz, m, sd, K, M, E)
    dzt = dz_q.reshape(K, M, E).copy()
    if dlogp is not None:
        pm_ = np.zeros((M, E), dt) if prior_mean is None else _np(prior_mean)
        ps_ = np.ones((M, E), dt) if prior_std is None else _np(prior_std)
        dz_p, _, _ = O.normal_logprob_bwd(_np(dlogp).reshape(K, M), zz, pm_, ps_, K, M, E)
        dzt = dzt + dz_p.reshape(K, M, E)
    if dz_up is not None:
        dzt = dzt + _np(dz_up).reshape(K, M, E)
    dm, ds = dm.reshape(m.shape).astype(dt), ds.reshape(sd.shape).astype(dt)
    if reparameterized:
        eps = ((zz - m.reshape((-1, M, E))) / sd.reshape((-1, M, E))).astype(dt)
        sm, ss = O.normal_sample_bwd(dzt.reshape(K, M * E), eps.reshape(K, M * E), m, sd, K, M * E)
        dm, ds = dm + sm.reshape(m.shape), ds + ss.reshape(sd.shape)
    return _t(dm, z), _t(ds, z)


def _pack_bits(z):
    """[K,M,E] 0/1 -> [K,M,E/4] uint8, bit q of a byte = element 4j+q (the kernels' packed-sample layout)."""
    K, M, E = z.shape
    b = (z.reshape(K, M, E // 4, 4) != 0).astype(np.uint8)
    return (b[..., 0] | (b[..., 1] << 1) | (b[..., 2] << 2) | (b[..., 3] << 3)).astype(np.uint8)


def bernoulli_latent_fwd(probs, mode, K, M, E, prior_probs=None, u_in=None, want_logq=True, want_logp=True, seed=0,
                         offset=0, rng_state=None, want_bits=False):
    dt = _np(probs).dtype
    u = (O.philox_uniform(K * M * E, seed, offset).astype(dt) if u_in is None else _np(u_in)).reshape(K, M * E)
    z = O.bernoulli_sample(_np(probs), u, K, M * E).reshape(K, M, E)
    logq = O.bernoulli_logpmf_fwd(z, _np(probs), K, M, E) if want_logq else None
    logp = None
    if want_logp:
        pp = np.full((M, E), 0.5, dt) if prior_probs is None else _np(prior_probs)
        logp = O.bernoulli_logpmf_fwd(z, pp, K, M, E)
    out = (_t(z, probs), None if logq is None else _t(logq, probs), None if logp is None else _t(logp, probs))
    if want_bits:
        ok = dt == np.float32 and mode == KBCAST and E % 4 == 0 and E <= 128
        out = out + ((torch.from_numpy(_pack_bits(z)) if ok else None),)
    return out


def bernoulli_latent_bwd(dlogq, z, probs, mode, K, M, E, zbits=None):
    dp = O.bernoulli_logpmf_bwd(_np(dlogq).reshape(K, M), _np(z).reshape(K, M, E), _np(probs), K, M, E)
    return _t(dp.reshape(probs.shape), probs)


def bernoulli_sample(probs, pm, K, N, u_in=None, seed=0, offset=0, rng_state=None):
    u = O.philox_uniform(K * N, seed, offset).astype(_np(probs).dtype).reshape(K, N) if u_in is None else _np(u_in)
    return _t(O.bernoulli_sample(_np(probs), u.reshape(K, N), K, N), probs)


def bernoulli_logpmf_fwd(x, xm, probs, pm, K, M, E, logits=False):
    f = O.bernoulli_logits_logpmf_fwd if logits else O.bernoulli_logpmf_fwd
    return _t(f(_np(x), _np(probs), K, M, E), probs)


def bernoulli_logpmf_bwd(g, x, xm, probs, pm, K, M, E, need_x, need_probs, logits=False):
    f = O.bernoulli_logits_logpmf_bwd if logits else O.bernoulli_logpmf_bwd
    dx, dp = f(_np(g), _np(x), _np(probs), K, M, E, need_dx=True)
    return (_t(dx, probs) if need_x else None, _t(dp, probs) if need_probs else None)


def poisson_sample(rate, rm, K, N, seed=0, offset=0, rng_state=None):
    return _t(O.poisson_sample(_np(rate), rm, K, N, seed, offset), rate)


def poisson_logpmf_fwd(x, xm, rate, rm, K, M, E):
    return _t(O.poisson_logpmf_fwd(_np(x), xm, _np(rate), rm, K, M, E), rate)


def poisson_logpmf_bwd(g, x, xm, rate, rm, K, M, E):
    return _t(O.poisson_logpmf_bwd(_np(g), _np(x), xm, _np(rate), rm, K, M, E), rate)


def beta_sample(alpha, am, beta, bm, K, N, seed=0, offset=0, rng_state=None):
    return _t(O.beta_sample(_np(alpha), am, _np(beta), bm, K, N, seed, offset), alpha)


FAM_LOGISTIC, FAM_LAPLACE, FAM_BETA = 1, 2, 4


def _locscale_u(family, K, N, dtype, u_in, seed, offset):
    if u_in is not None:
        return _np(u_in).reshape(K, N)
    u = O.philox_uniform_open(K * N, seed, offset).astype(dtype).reshape(K, N)
    return (2 * u - 1).astype(dtype) if family == FAM_LAPLACE else u


def locscale_sample(family, loc, loc_mode, scale, scale_mode, K, N, u_in=None, seed=0, offset=0, rng_state=None,
                    rng_snapshot=None):
    u = _locscale_u(family, K, N, _np(loc).dtype, u_in, seed, offset)
    return _t(O.locscale_sample(family, _np(loc), _np(scale), u, K, N), loc)


def locscale_sample_bwd(family, dz, loc_like, loc_mode, scale_like, scale_mode, K, N, u=None, seed=0, offset=0,
                        need_loc=True, need_scale=True, rng_state=None):
    uu = _locscale_u(family, K, N, _np(dz).dtype, u, seed, offset)
    dl, ds = O.locscale_sample_bwd(family, _np(dz), uu, K, N, full=(loc_mode == FULL and K > 1))
    return (_t(dl.reshape(loc_like.shape), dz) if need_loc else None,
            _t(ds.reshape(scale_like.shape), dz) if need_scale else None)


def locscale_logprob_fwd(family, x, xm, loc, lm, scale, sm, K, M, E):
    if family == FAM_BETA:  # loc = alpha, scale = beta
        return _t(O.beta_logprob_fwd(_np(x), xm, _np(loc), lm, _np(scale), sm, K, M, E), x)
    return _t(O.locscale_logprob_fwd(family, _np(x), _np(loc), _np(scale), K, M, E), x)


def locscale_logprob_bwd(family, g, x, xm, loc, lm, scale, sm, K, M, E, need_x, need_loc, need_scale):
    if family == FAM_BETA:
        outs = O.beta_logprob_bwd(_np(g), _np(x), xm, _np(loc), lm, _np(scale), sm, K, M, E,
                                  need=(need_x, need_loc, need_scale))
        return tuple(None if o is None else _t(o, x) for o in outs)
    dx, dl, ds = O.locscale_logprob_bwd(family, _np(g), _np(x), _np(loc), _np(scale), K, M, E)
    return (_t(dx.reshape(x.shape), x) if need_x else None, _t(dl.reshape(loc.shape), x) if need_loc else None,
            _t(ds.reshape(scale.shape), x) if need_scale else None)


def categorical_sample(logits, lm, K, M, C, u_in=None, seed=0, offset=0, rng_state=None):
    u = O.philox_uniform(K * M, seed, offset).astype(_np(logits).dtype) if u_in is None else _np(u_in)
    return _t(O.categorical_sample(_np(logits), u.reshape(K, M), K, M, C), logits)


def categorical_logpmf_fwd(x, xm, logits, lm, K, M, C):
    return _t(O.categorical_logpmf_fwd(_np(x), _np(logits), K, M, C), logits)


def categorical_logpmf_bwd(g, x, xm, logits, lm, K, M, C):
    return _t(O.categorical_logpmf_bwd(_np(g), _np(x), _np(logits), K, M, C), logits)


def iw_objective(estimator, logp, logq, grad_scale, extra=None, need_grads=True):
    lp = _np(logp) + (0 if extra is None else _np(extra))
    K, B = lp.shape
    if estimator == 2:  # ELBO
        x = lp.astype(np.float64) - _np(logq)
        cost = (-x.mean(0)).astype(lp.dtype)
        g = np.full((K, B), grad_scale / K, lp.dtype)
        return _t(cost, logp), _t(-g, logp), _t(g, logp)
    cost, dlp, dlq = O.iw_objective(estimator, lp, _np(logq), grad_scale)
    return _t(cost, logp), _t(dlp, logp), _t(dlq, logp)


def combine_sums(a, scale_a, b, scale_b):
    v = scale_a * _np(a).astype(np.float64).sum() + scale_b * _np(b).astype(np.float64).sum()
    return torch.tensor([v], dtype=a.dtype)


def log_mean_exp(x):
    return _t(O.log_mean_exp(_np(x)), x)


def log_mean_exp_bwd(g, x):
    xn = _np(x).astype(np.float64)
    w = np.exp(xn - xn.max(0, keepdims=True))
    return _t(_np(g)[None, :] * w / w.sum(0, keepdims=True), x)


def fused_supported(K, X, dtype):
    return dtype == torch.float32 and X % 4 == 0 and 1 <= K <= 4096


def iw_bernoulli_fused(estimator, probs, x, logp_other, logq, grad_scale, need_dprobs=True, want_logpx=False, out=None,
                       logits=False, accumulate_cost=False, cost_scaled=False, want_loss=False):
    f = O.iw_bernoulli_logits_step if logits else O.iw_bernoulli_step
    r = f(estimator, _np(probs), _np(x), _np(logp_other), _np(logq), grad_scale, need_dprobs=need_dprobs)
    cost = r["cost"] * (np.float32(grad_scale) if cost_scaled else np.float32(1.0))
    return dict(cost=_t(cost, probs), dprobs=_t(r["dprobs"], probs) if need_dprobs else None,
                dlogp=_t(r["dlogp"], probs), dlogq=_t(r["dlogq"], probs),
                logpx=_t(r["logpx"], probs) if want_logpx else None)


def iw_poisson_fused(estimator, rate, x, logp_other, logq, grad_scale, need_drate=True, want_logpx=False, out=None,
                     accumulate_cost=False, cost_scaled=False, want_loss=False):
    r = O.iw_poisson_step(estimator, _np(rate), _np(x), _np(logp_other), _np(logq), grad_scale, need_drate)
    cost = r["cost"] * (np.float32(grad_scale) if cost_scaled else np.float32(1.0))
    return dict(cost=_t(cost, rate), dprobs=_t(r["drate"], rate) if need_drate else None,
                dlogp=_t(r["dlogp"], rate), dlogq=_t(r["dlogq"], rate),
                logpx=_t(r["logpx"], rate) if want_logpx else None)


def reinforce_step(logp, logq, moving_mean, local_step, decay, need_grads=True):
    cost, dlp, dlq, mm, ls = O.reinforce_step(_np(logp), _np(logq), float(moving_mean), int(local_step), decay)
    moving_mean.fill_(float(mm))
    local_step.fill_(int(ls))
    return (torch.tensor([cost], dtype=logq.dtype), _t(dlp, logq) if need_grads else None,
            _t(dlq, logq) if need_grads else None)


def scale_inplace(buf, scale_dev, buf1=None, buf2=None):
    if float(scale_dev) != 1.0:
        for b in (buf, buf1, buf2):
            if b is not None:
                b.mul_(scale_dev)


def philox_normal(n, dtype, mean, std, seed, offset, device, rng_state=None):
    return torch.from_numpy(O.philox_normal(n, seed, offset, mean, std)).to(dtype)


def sgld_step(w, g, lr, noise=None, seed=0, offset=0, out=None, rng_state=None):
    if noise is None:
        noise = philox_normal(w.numel(), w.dtype, 0.0, float(np.float32(np.sqrt(np.float64(np.float32(lr))))), seed,
                              offset, None).reshape(w.shape)
    return _t(O.sgld_step(_np(w), _np(g), _np(noise), lr), w)


def psgld_step(w, aux, g, lr, decay, epsilon, noise_unit=None, seed=0, offset=0, out=None, rng_state=None):
    if noise_unit is None:
        noise_unit = philox_normal(w.numel(), w.dtype, 0.0, 1.0, seed, offset, None).reshape(w.shape)
    nw, na = O.psgld_step(_np(w), _np(aux), _np(g), _np(noise_unit), lr, decay, epsilon)
    aux.copy_(_t(na, w))
    return _t(nw, w)


def sghmc_pre(w, v, lr, resample, second_order, v_noise=None, seed=0, offset=0, out=None, rng_state=None):
    if not resample and not second_order:
        return w
    if resample and v_noise is None:
        v_noise = philox_normal(w.numel(), w.dtype, 0.0, float(np.float32(np.sqrt(lr))), seed, offset, None).reshape(w.shape)
    nw, nv = O.sghmc_pre(_np(w), _np(v), _np(v_noise), resample, second_order)
    v.copy_(_t(nv, w))
    return _t(nw, w) if second_order else w


def sghmc_post(w, v, g, lr, alpha, beta, second_order, noise=None, seed=0, offset=0, out=None, rng_state=None):
    if noise is None:
        std = float(np.float32(np.sqrt(2.0 * (alpha - beta) * lr)))
        noise = philox_normal(w.numel(), w.dtype, 0.0, std, seed, offset, None).reshape(w.shape)
    nw, nv = O.sghmc_post(_np(w), _np(v), _np(g), _np(noise), lr, alpha, second_order)
    v.copy_(_t(nv, w))
    return _t(nw, w)


ALG_SGLD, ALG_PSGLD, ALG_SGHMC_PRE, ALG_SGHMC_POST = 0, 1, 2, 3


def sgmcmc_multi_step(algorithm, ws, gs=None, states=None, noises=None, outs=None, lr=0.0, a=0.0, b=0.0, resample=False,
                      second_order=False, seed=0, offset=0, rng_state=None):
    """Stand-in of zs_sgmcmc_multi_step: tensor t draws its noise from the quads [q_t, q_t + ceil(n_t/4)) of ONE
    Philox stream position, exactly as the kernel does."""
    n = len(ws)
    gs = gs if gs is not None else [None] * n
    states = states if states is not None else [None] * n
    noises = noises if noises is not None else [None] * n
    total_q = sum((w.numel() + 3) // 4 for w in ws)
    unit = None

    def unit_noise(q0, cnt):
        nonlocal unit
        if unit is None:
            unit = O.philox_normal(4 * total_q, seed, offset, 0.0, 1.0)
        return unit[4 * q0:4 * q0 + cnt]

    res, q0 = [], 0
    for i, w in enumerate(ws):
        cnt = w.numel()
        dt = _np(w).dtype

        def scaled(std):
            return _t((np.float32(std) * unit_noise(q0, cnt)).astype(dt).reshape(w.shape), w)

        if algorithm == ALG_SGLD:
            nz = noises[i] if noises[i] is not None else scaled(np.float32(np.sqrt(np.float64(np.float32(lr)))))
            res.append(sgld_step(w, gs[i], lr, noise=nz))
        elif algorithm == ALG_PSGLD:
            nz = noises[i] if noises[i] is not None else scaled(1.0)
            res.append(psgld_step(w, states[i], gs[i], lr, a, b, noise_unit=nz))
        elif algorithm == ALG_SGHMC_PRE:
            nz = noises[i]
            if resample and nz is None:
                nz = scaled(np.float32(np.sqrt(lr)))
            res.append(sghmc_pre(w, states[i], lr, resample, second_order, v_noise=nz))
        else:
            nz = noises[i] if noises[i] is not None else scaled(np.float32(np.sqrt(2.0 * (a - b) * lr)))
            res.append(sghmc_post(w, states[i], gs[i], lr, a, b, second_order, noise=nz))
        q0 += (cnt + 3) // 4
    return res


_counter = {"off": 0}


def _next_philox(device):
    _counter["off"] += 4
    return 1234, _counter["off"]


def _draw_args(device):
    seed, offset = _next_philox(device)
    return dict(seed=seed, offset=offset, rng_state=None)


def install(monkeypatch):
    """Patch the product's backend / device helpers with the CPU stand-ins above."""
    from zhusuan import _backend, _ops, _rng
    for name in ("normal_sample", "normal_sample_bwd", "normal_logprob_fwd", "normal_logprob_bwd", "normal_latent_fwd", "normal_latent_bwd",
                 "bernoulli_latent_fwd", "bernoulli_latent_bwd", "bernoulli_sample",
                 "bernoulli_logpmf_fwd", "bernoulli_logpmf_bwd", "poisson_sample", "poisson_logpmf_fwd",
                 "poisson_logpmf_bwd", "beta_sample", "locscale_sample", "locscale_sample_bwd",
                 "locscale_logprob_fwd", "locscale_logprob_bwd", "categorical_sample", "categorical_logpmf_fwd",
                 "categorical_logpmf_bwd", "iw_objective", "combine_sums", "log_mean_exp", "log_mean_exp_bwd", "fused_supported",
                 "iw_bernoulli_fused", "iw_poisson_fused", "reinforce_step", "scale_inplace", "philox_normal", "sgld_step", "psgld_step", "sghmc_pre",
                 "sghmc_post", "sgmcmc_multi_step"):
        monkeypatch.setattr(_backend, name, globals()[name])
    monkeypatch.setattr(_backend, "require_cuda", lambda: None)
    monkeypatch.setattr(_backend, "on_compute_device", lambda t: True)
    monkeypatch.setattr(_ops, "to_compute", lambda t: t)
    monkeypatch.setattr(_ops, "compute_device", lambda: torch.device("cpu"))
    monkeypatch.setattr(_rng, "next_philox", _next_philox)
    monkeypatch.setattr(_rng, "draw_args", _draw_args)
    _counter["off"] = 0
