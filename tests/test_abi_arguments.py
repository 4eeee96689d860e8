"""CPU: the C ABI's argument validation.  Every call here is rejected (or found to have nothing to do) before any CUDA
call, so the exact return code of each entry point, and the order in which its checks run, is pinned without a
device.  Pointers are small fake addresses: A is 16-byte aligned, U is not; nothing is ever dereferenced."""
import os

import pytest

OK, ARG, DTYPE, UNSUPPORTED, ALIGN = 0, -1, -2, -6, -7
F32, F64, BAD = 0, 1, 7
FULL, KBCAST, SCALAR = 0, 1, 2
SGVB, VIMCO, ELBO = 0, 1, 2
LOGISTIC, LAPLACE, UNIFORM, BETA = 1, 2, 3, 4
ACCUMULATE, LOGITS, COST_SCALED = 1, 2, 4
SGLD, PSGLD, SGHMC_PRE, SGHMC_POST = 0, 1, 2, 3
A, U = 16, 20

CASES = []


def case(expect, fn, args):
    CASES.append(pytest.param(fn, args, expect, id="%s-%d" % (fn, sum(1 for c in CASES if c.values[0] == fn))))


# ---- row log-density entry points: (spec name, family or None, parameters) ------------------------------------
ROWS = [("normal_logprob", None, 2), ("bernoulli_logpmf", None, 1), ("bernoulli_logits_logpmf", None, 1),
        ("poisson_logpmf", None, 1)] + [("locscale_logprob", f, 2) for f in (LOGISTIC, LAPLACE, UNIFORM, BETA)]


def rows_fwd(name, fam, npar, dtype=F32, out=A, x=A, xm=FULL, a=A, am=FULL, b=A, bm=FULL, K=1, M=1, E=1):
    head = [dtype] + ([] if fam is None else [fam]) + [out, x, xm, a, am]
    return "zs_%s_fwd" % name, head + ([b, bm] if npar == 2 else []) + [K, M, E]


def rows_bwd(name, fam, npar, dtype=F32, dx=None, da=A, db=None, g=A, x=A, xm=FULL, a=A, am=FULL, b=A, bm=FULL, K=1,
             M=1, E=1):
    grads = {"normal_logprob": [dx, da, db], "locscale_logprob": [dx, da, db], "poisson_logpmf": [da]}.get(name, [dx, da])
    head = [dtype] + ([] if fam is None else [fam]) + grads + [g, x, xm, a, am]
    return "zs_%s_bwd" % name, head + ([b, bm] if npar == 2 else []) + [K, M, E]


for spec in ROWS:
    name, fam, npar = spec
    case(ARG, *rows_fwd(*spec, out=None))
    case(ARG, *rows_fwd(*spec, x=None))
    case(ARG, *rows_fwd(*spec, a=None))
    case(ARG, *rows_fwd(*spec, K=-1))
    case(ARG, *rows_fwd(*spec, M=-1))
    case(ARG, *rows_fwd(*spec, E=0))
    case(ARG, *rows_fwd(*spec, xm=7))
    case(ARG, *rows_fwd(*spec, am=-1))
    case(DTYPE, *rows_fwd(*spec, dtype=BAD))
    case(DTYPE, *rows_fwd(*spec, dtype=BAD, K=0))  # the dtype is checked before the empty shape
    case(ARG, *rows_bwd(*spec, g=None))
    case(ARG, *rows_bwd(*spec, x=None))
    case(ARG, *rows_bwd(*spec, a=None))
    case(ARG, *rows_bwd(*spec, M=-1))
    case(ARG, *rows_bwd(*spec, E=0))
    case(ARG, *rows_bwd(*spec, am=3))
    case(DTYPE, *rows_bwd(*spec, dtype=BAD))
    case(DTYPE, *rows_bwd(*spec, dtype=BAD, K=0))
    case(OK, *rows_bwd(*spec, dtype=BAD, da=None))  # no gradient requested: nothing to do, whatever the dtype
    case(UNSUPPORTED, *rows_bwd(*spec, am=SCALAR))
    case(OK, *rows_bwd(*spec, am=SCALAR, M=0))
    if npar == 2:
        case(ARG, *rows_fwd(*spec, b=None))
        case(ARG, *rows_fwd(*spec, bm=7))
        case(ARG, *rows_bwd(*spec, b=None))
        case(ARG, *rows_bwd(*spec, bm=7))
        case(UNSUPPORTED, *rows_bwd(*spec, db=A, bm=SCALAR))
    if name != "poisson_logpmf":
        case(UNSUPPORTED, *rows_bwd(*spec, dx=A, xm=SCALAR))
for fam in (0, 5):
    case(ARG, *rows_fwd("locscale_logprob", fam, 2))
    case(ARG, *rows_fwd("locscale_logprob", fam, 2, dtype=BAD))
    case(ARG, *rows_bwd("locscale_logprob", fam, 2))
    case(ARG, *rows_bwd("locscale_logprob", fam, 2, da=None))  # the family is checked before "no gradient requested"


# ---- location-scale samplers -----------------------------------------------------------------------------------
def ls_sample(dtype=F32, fam=LOGISTIC, z=A, loc=A, lm=FULL, scale=A, sm=FULL, u=None, K=1, N=1):
    return "zs_locscale_sample", [dtype, fam, z, loc, lm, scale, sm, u, K, N, 0, 0, None, None]


def ls_sample_bwd(dtype=F32, fam=LOGISTIC, dloc=A, lm=FULL, dscale=None, sm=FULL, dz=A, u=None, K=1, N=1):
    return "zs_locscale_sample_bwd", [dtype, fam, dloc, lm, dscale, sm, dz, u, K, N, 0, 0, None]


for kw, expect in [(dict(z=None), ARG), (dict(scale=None), ARG), (dict(N=-1), ARG), (dict(lm=7), ARG),
                   (dict(fam=0), ARG), (dict(fam=BETA), ARG), (dict(fam=0, K=0), ARG), (dict(dtype=BAD, K=0), OK)]:
    case(expect, *ls_sample(**kw))
for kw, expect in [(dict(dz=None), ARG), (dict(K=-1), ARG), (dict(sm=7), ARG), (dict(fam=BETA), ARG),
                   (dict(fam=0, dloc=None), ARG), (dict(lm=SCALAR), UNSUPPORTED), (dict(dscale=A, sm=SCALAR), UNSUPPORTED),
                   (dict(dtype=BAD, K=0), OK), (dict(dtype=BAD, dloc=None), OK), (dict(dtype=BAD), DTYPE),
                   (dict(dtype=BAD, fam=UNIFORM), DTYPE)]:
    case(expect, *ls_sample_bwd(**kw))


# ---- fused latent nodes ----------------------------------------------------------------------------------------
def n_lat_fwd(dtype=F32, z=A, mean=A, mm=KBCAST, std=A, sm=KBCAST, pmean=None, pstd=None, eps=None, K=1, M=1, E=4):
    return "zs_normal_latent_fwd", [dtype, z, A, A, mean, mm, std, sm, pmean, pstd, eps, K, M, E, 0, 0, None]


def b_lat_fwd(dtype=F32, z=A, probs=A, pm=KBCAST, prior=None, u=None, K=1, M=1, E=4, zbits=None):
    return "zs_bernoulli_latent_fwd", [dtype, z, A, A, probs, pm, prior, u, K, M, E, 0, 0, None, zbits]


def n_lat_bwd(dtype=F32, dmean=A, dstd=A, z=A, mean=A, mm=KBCAST, std=A, sm=KBCAST, K=1, M=1, E=4):
    return "zs_normal_latent_bwd", [dtype, dmean, dstd, A, A, A, z, mean, mm, std, sm, None, None, 1, K, M, E]


def b_lat_bwd(dtype=F32, dprobs=A, dlogq=A, z=A, probs=A, pm=KBCAST, K=1, M=1, E=4, zbits=None):
    return "zs_bernoulli_latent_bwd", [dtype, dprobs, dlogq, z, probs, pm, K, M, E, zbits]


for kw, expect in [(dict(z=None), ARG), (dict(std=None), ARG), (dict(M=-1), ARG), (dict(E=0), ARG),
                   (dict(E=6), UNSUPPORTED), (dict(E=6, z=U), UNSUPPORTED), (dict(mm=FULL), UNSUPPORTED),
                   (dict(mm=SCALAR, sm=SCALAR), UNSUPPORTED), (dict(mm=7, sm=7), UNSUPPORTED), (dict(mean=U), ALIGN),
                   (dict(eps=U), ALIGN), (dict(pstd=U), ALIGN), (dict(dtype=BAD), DTYPE), (dict(dtype=BAD, K=0), OK)]:
    case(expect, *n_lat_fwd(**kw))
for kw, expect in [(dict(probs=None), ARG), (dict(K=-1), ARG), (dict(zbits=A, dtype=F64), UNSUPPORTED),
                   (dict(zbits=A, dtype=BAD), UNSUPPORTED), (dict(E=2), UNSUPPORTED), (dict(pm=SCALAR), UNSUPPORTED),
                   (dict(u=U), ALIGN), (dict(prior=U), ALIGN), (dict(dtype=BAD), DTYPE), (dict(dtype=BAD, K=0), OK)]:
    case(expect, *b_lat_fwd(**kw))
for kw, expect in [(dict(z=None), ARG), (dict(K=-1), ARG), (dict(E=6), UNSUPPORTED), (dict(sm=FULL), UNSUPPORTED),
                   (dict(dmean=U), ALIGN), (dict(E=10, dmean=U), UNSUPPORTED), (dict(dtype=BAD), DTYPE),
                   (dict(dtype=BAD, dmean=None, dstd=None), OK), (dict(dtype=BAD, M=0), OK)]:
    case(expect, *n_lat_bwd(**kw))
for kw, expect in [(dict(dprobs=None), ARG), (dict(dlogq=None), ARG), (dict(E=5), UNSUPPORTED),
                   (dict(pm=SCALAR), UNSUPPORTED), (dict(z=U), ALIGN), (dict(dtype=BAD), DTYPE),
                   (dict(dtype=BAD, K=0), OK)]:
    case(expect, *b_lat_bwd(**kw))


# ---- fused importance-weighted step ----------------------------------------------------------------------------
def fused(lik, est=SGVB, probs=A, x=A, dprobs=A, logq=A, K=2, B=1, X=4, flags=0):
    return "zs_iw_%s_fused" % lik, [est, A, dprobs, A, A, None, probs, x, A, logq, K, B, X, 1.0, flags]


def fused_loss(lik, est=SGVB, loss=A, ws=A, cost=A, probs=A, x=A, logq=A, K=2, B=1, X=4, flags=0):
    return "zs_iw_%s_fused_loss" % lik, [est, loss, ws, cost, A, A, A, None, probs, x, A, logq, K, B, X, 1.0, flags]


COMMON_FUSED = [(dict(probs=None), ARG), (dict(x=None), ARG), (dict(K=0), ARG), (dict(X=0), ARG), (dict(est=ELBO), ARG),
                (dict(est=7), ARG), (dict(est=VIMCO, K=1), ARG), (dict(est=VIMCO, logq=None), ARG), (dict(flags=8), ARG),
                (dict(flags=ACCUMULATE | 16), ARG)]
for lik in ("bernoulli", "poisson"):
    for kw, expect in COMMON_FUSED + [
            (dict(B=-1), ARG), (dict(B=0), OK), (dict(B=0, est=VIMCO), OK), (dict(B=0, est=ELBO), ARG),
            (dict(B=0, flags=ACCUMULATE | COST_SCALED), OK), (dict(X=6), UNSUPPORTED), (dict(X=6, probs=U), UNSUPPORTED),
            (dict(probs=U), ALIGN), (dict(x=U), ALIGN), (dict(dprobs=U), ALIGN),
            (dict(B=0, flags=LOGITS), OK if lik == "bernoulli" else ARG)]:
        case(expect, *fused(lik, **kw))
    for kw, expect in COMMON_FUSED + [(dict(loss=None), ARG), (dict(ws=None), ARG), (dict(cost=None), ARG),
                                      (dict(B=0), ARG), (dict(B=-1), ARG)]:
        case(expect, *fused_loss(lik, **kw))
case(ARG, *fused("poisson", flags=LOGITS))
case(ARG, *fused_loss("poisson", flags=LOGITS))
case(ARG, *fused_loss("poisson", flags=LOGITS | ACCUMULATE))


# ---- SG-MCMC ---------------------------------------------------------------------------------------------------
def sgld(dtype=F32, w_out=A, w=A, g=A, n=4, lr=0.1):
    return "zs_sgld_step", [dtype, w_out, w, g, None, n, lr, 0, 0, None]


def psgld(dtype=F32, aux=A, n=4, lr=0.1):
    return "zs_psgld_step", [dtype, A, A, aux, A, None, n, lr, 0.9, 1e-5, 0, 0, None]


def sghmc_pre(dtype=F32, v=A, n=4, lr=0.1, resample=1, second=0):
    return "zs_sghmc_pre", [dtype, A, A, v, None, n, lr, resample, second, 0, 0, None]


def sghmc_post(dtype=F32, g=A, n=4, lr=0.1, alpha=0.2, beta=0.1):
    return "zs_sghmc_post", [dtype, A, A, A, g, None, n, lr, alpha, beta, 0, 0, 0, None]


for kw, expect in [(dict(w_out=None), ARG), (dict(g=None), ARG), (dict(n=-1), ARG), (dict(lr=-1.0), ARG),
                   (dict(dtype=BAD), DTYPE), (dict(dtype=BAD, n=0), DTYPE)]:
    case(expect, *sgld(**kw))
for kw, expect in [(dict(aux=None), ARG), (dict(n=-1), ARG), (dict(dtype=BAD), DTYPE), (dict(dtype=BAD, n=0), DTYPE)]:
    case(expect, *psgld(**kw))
for kw, expect in [(dict(v=None), ARG), (dict(lr=-1.0), ARG), (dict(dtype=BAD, resample=0), OK),
                   (dict(dtype=BAD), DTYPE), (dict(dtype=BAD, resample=0, second=1), DTYPE)]:
    case(expect, *sghmc_pre(**kw))
for kw, expect in [(dict(g=None), ARG), (dict(n=-1), ARG), (dict(alpha=0.1, beta=0.2), ARG), (dict(dtype=BAD), DTYPE)]:
    case(expect, *sghmc_post(**kw))


# ---- objectives ------------------------------------------------------------------------------------------------
def iw_obj(dtype=F32, est=SGVB, logp=A, logq=A, K=2, B=1):
    return "zs_iw_objective", [dtype, est, A, A, A, logp, logq, None, K, B, 1.0]


for kw, expect in [(dict(logp=None), ARG), (dict(logq=None), ARG), (dict(K=0), ARG), (dict(B=-1), ARG),
                   (dict(est=5), ARG), (dict(est=VIMCO, K=1), ARG), (dict(dtype=BAD, B=0), OK),
                   (dict(dtype=BAD), DTYPE), (dict(dtype=BAD, est=VIMCO), DTYPE), (dict(dtype=BAD, est=ELBO), DTYPE)]:
    case(expect, *iw_obj(**kw))
case(ARG, "zs_log_mean_exp", [F32, None, A, 2, 3])
case(ARG, "zs_log_mean_exp", [F32, A, A, 0, 3])
case(OK, "zs_log_mean_exp", [BAD, A, A, 2, 0])
case(DTYPE, "zs_log_mean_exp", [BAD, A, A, 2, 3])
case(ARG, "zs_log_mean_exp_bwd", [F32, A, None, A, 2, 3])
case(ARG, "zs_log_mean_exp_bwd", [F32, None, A, A, 2, 3])
case(DTYPE, "zs_log_mean_exp_bwd", [BAD, A, A, A, 2, 3])
case(ARG, "zs_combine_sums", [F32, None, A, 2, 1.0, A, 2, 1.0])
case(ARG, "zs_combine_sums", [F32, A, None, 2, 1.0, A, 2, 1.0])
case(ARG, "zs_combine_sums", [F32, A, A, -1, 1.0, A, 2, 1.0])
case(DTYPE, "zs_combine_sums", [BAD, A, A, 2, 1.0, None, 0, 1.0])
case(ARG, "zs_scale_inplace", [F32, None, 4, None, 0, None, 0, A])
case(ARG, "zs_scale_inplace", [F32, A, -4, None, 0, None, 0, A])
case(ALIGN, "zs_scale_inplace", [F32, A, 4, U, 4, None, 0, A])
case(OK, "zs_scale_inplace", [BAD, A, 0, None, 0, None, 0, A])
case(ARG, "zs_reinforce_step", [F32, A, A, A, A, None, A, A, 4, 0.9, 0.25])
case(ARG, "zs_reinforce_step", [F32, A, A, A, A, A, A, A, 0, 0.9, 0.25])
case(DTYPE, "zs_reinforce_step", [BAD, A, A, A, A, A, A, A, 4, 0.9, 0.25])

# ---- Categorical -----------------------------------------------------------------------------------------------
case(ARG, "zs_categorical_sample", [F32, None, A, FULL, None, 1, 1, 3, 0, 0, None])
case(ARG, "zs_categorical_sample", [F32, A, A, FULL, None, 1, 1, 0, 0, 0, None])
case(ARG, "zs_categorical_sample", [F32, A, A, SCALAR, None, 1, 1, 3, 0, 0, None])
case(OK, "zs_categorical_sample", [BAD, A, A, KBCAST, None, 0, 1, 3, 0, 0, None])
for C in (3, 40):
    case(ARG, "zs_categorical_logpmf_fwd", [F32, A, None, FULL, A, FULL, 1, 1, C])
    case(ARG, "zs_categorical_logpmf_fwd", [F32, A, A, 7, A, FULL, 1, 1, C])
    case(ARG, "zs_categorical_logpmf_fwd", [F32, A, A, FULL, A, SCALAR, 1, 1, C])
    case(OK, "zs_categorical_logpmf_fwd", [BAD, A, A, FULL, A, FULL, 1, 0, C])
    case(DTYPE, "zs_categorical_logpmf_fwd", [BAD, A, A, FULL, A, FULL, 1, 1, C])
    case(ARG, "zs_categorical_logpmf_bwd", [F32, None, A, A, FULL, A, FULL, 1, 1, C])
    case(ARG, "zs_categorical_logpmf_bwd", [F32, A, A, A, FULL, A, SCALAR, 1, 1, C])
    case(OK, "zs_categorical_logpmf_bwd", [BAD, A, A, A, FULL, A, KBCAST, 0, 1, C])
    case(DTYPE, "zs_categorical_logpmf_bwd", [BAD, A, A, A, FULL, A, KBCAST, 1, 1, C])
case(ARG, "zs_categorical_logpmf_fwd", [F32, A, A, FULL, A, FULL, 1, 1, 0])


@pytest.fixture(scope="module")
def lib():
    from zhusuan import _backend
    if not os.path.exists(_backend.LIB_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _backend.load()


@pytest.mark.parametrize("fn, args, expect", CASES)
def test_rejected_before_any_cuda_call(lib, fn, args, expect):
    rc = getattr(lib, fn)(*args, None)
    assert rc == expect, (rc, lib.zs_last_error())


def _chain_table(count, **fields):
    from zhusuan import _backend
    table = (_backend.ChainTensor * count)()
    for t in table:
        t.w_out = t.w = t.g = t.state = A
        t.n = 4
        for k, v in fields.items():
            setattr(t, k, v)
    return table


@pytest.mark.parametrize("dtype, alg, n_tensors, table, lr, a, b, resample, expect", [
    (F32, SGLD, -1, None, 0.1, 0.0, 0.0, 0, ARG),
    (F32, SGLD, 1, None, 0.1, 0.0, 0.0, 0, ARG),
    (F32, SGLD, 1, {}, -0.1, 0.0, 0.0, 0, ARG),
    (BAD, SGLD, 0, None, 0.1, 0.0, 0.0, 0, OK),
    (BAD, SGLD, 1, {}, 0.1, 0.0, 0.0, 0, DTYPE),
    (BAD, 9, 1, {}, 0.1, 0.0, 0.0, 0, DTYPE),
    (F32, 9, 1, {}, 0.1, 0.0, 0.0, 0, ARG),
    (F64, 9, 1, {}, 0.1, 0.0, 0.0, 0, ARG),
    (F32, SGHMC_POST, 1, {}, 0.1, 0.1, 0.2, 0, ARG),
    (F32, SGHMC_PRE, 1, {}, 0.1, 0.0, 0.0, 0, OK),
    (F64, SGLD, 33, {}, 0.1, 0.0, 0.0, 0, UNSUPPORTED),
    (F32, PSGLD, 33, {}, 0.1, 0.9, 1e-5, 0, UNSUPPORTED),
    (F32, SGLD, 1, {"w": None}, 0.1, 0.0, 0.0, 0, ARG),
    (F64, PSGLD, 2, {"state": None}, 0.1, 0.9, 1e-5, 0, ARG),
    (F32, SGHMC_PRE, 1, {"n": -1}, 0.1, 0.0, 0.0, 1, ARG),
    (F64, SGHMC_POST, 1, {"g": None}, 0.1, 0.2, 0.1, 0, ARG),
])
def test_sgmcmc_multi_step_rejected_before_any_cuda_call(lib, dtype, alg, n_tensors, table, lr, a, b, resample, expect):
    tab = None if table is None else _chain_table(max(n_tensors, 1), **table)
    rc = lib.zs_sgmcmc_multi_step(dtype, alg, tab, n_tensors, lr, a, b, resample, 0, 0, 0, None, None)
    assert rc == expect, (rc, lib.zs_last_error())
