"""The Poisson node: log-pmf and rate gradient (every layout mode, fp32 / fp64, event and StochasticTensor reductions),
the sampler, BayesianNet registration and the fused Poisson-likelihood importance-weighted step.

Modes as in tests/test_api.py: `oracle` (CPU; the ctypes backend replaced by the CPU oracle, with the Poisson node
restated in tests/poisson_oracle.c), `cuda` (B200 kernels, CUDA tensors) and `cuda-host` (CPU tensors in and out).
The anchor is torch.distributions.Poisson, the function the reference's Poisson delegates to, cross-checked with scipy.
Parity rule (DESIGN.md §4): within 1e-5 normwise of float32 torch, or no farther from float64 torch than float32 torch is.
"""
import math

import numpy as np
import pytest
import torch
from scipy import stats

import zhusuan
import zhusuan.variational
from zhusuan import _backend, _rng
from zhusuan.distributions import Normal, Poisson
from zhusuan.framework import BayesianNet, StochasticTensor
from zhusuan.variational import ImportanceWeightedObjective

MODES = [pytest.param("oracle"), pytest.param("cuda", marks=pytest.mark.gpu),
         pytest.param("cuda-host", marks=pytest.mark.gpu)]


@pytest.fixture(params=MODES)
def dev(request, monkeypatch):
    mode = request.param
    if mode == "oracle":
        import poisson_oracle
        poisson_oracle.install(monkeypatch)
        return torch.device("cpu")
    return torch.device("cuda") if mode == "cuda" else torch.device("cpu")


def T(a, dev, dtype=torch.float32, grad=False):
    t = torch.tensor(np.asarray(a), dtype=dtype, device=dev)
    t.requires_grad_(grad)
    return t


def _np64(t):
    return t.detach().cpu().double().numpy() if torch.is_tensor(t) else np.asarray(t, np.float64)


def parity(got, x, rate, fn, dtype):
    """`fn(x, rate)` is the torch restatement; compare `got` with it in float64 (and scipy), under the parity rule."""
    ref64 = _np64(fn(torch.tensor(_np64(x)), torch.tensor(_np64(rate))))
    g = _np64(got)
    assert g.shape == ref64.shape
    fin = np.isfinite(ref64)
    np.testing.assert_array_equal(g[~fin], ref64[~fin])  # -inf where rate == 0 < x, identically
    err = np.linalg.norm(g[fin] - ref64[fin])
    nrm = max(np.linalg.norm(ref64[fin]), 1e-30)
    if dtype == torch.float64:
        assert err <= 1e-12 * nrm, err / nrm
        return
    ref32 = _np64(fn(torch.tensor(_np64(x), dtype=torch.float32), torch.tensor(_np64(rate), dtype=torch.float32)))
    assert err <= max(1e-5 * nrm, np.linalg.norm(ref32[fin] - ref64[fin])), err / nrm


def _counts(rng, shape, rate):
    return rng.poisson(np.broadcast_to(rate, shape)).astype(np.float64)


def _torch_logpmf(x, rate):
    return torch.distributions.Poisson(rate, validate_args=False).log_prob(x)


# ============================================================================ values and gradients
# (x shape, rate shape): both FULL; rate broadcast over particles (KBCAST); x broadcast (KBCAST); a scalar rate
LAYOUTS = [((5, 4, 6), (5, 4, 6)), ((5, 4, 6), (4, 6)), ((4, 6), (5, 4, 6)), ((5, 4, 6), ())]


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("xs,rs", LAYOUTS)
@pytest.mark.parametrize("group_ndims", [0, 1, 2])
def test_log_prob_values(dev, dtype, xs, rs, group_ndims):
    rng = np.random.RandomState(11)
    rate = rng.gamma(1.5, 3.0, size=rs) + 0.05
    if rs:
        rate.reshape(-1)[::7] = 0.0  # rate == 0: 0 at x == 0, -inf at x > 0
    shape = np.broadcast_shapes(xs, rs)
    x = _counts(rng, xs, np.broadcast_to(rate, shape)[(0,) * (len(shape) - len(xs))] if len(xs) < len(shape) else rate)
    x.reshape(-1)[1::5] += 1.0  # some counts where rate == 0
    p = Poisson(T(rate, dev, dtype), group_ndims=group_ndims)
    got = p.log_prob(T(x, dev, dtype))
    assert got.dtype == dtype and got.device.type == dev.type

    def fn(xx, rr):
        lp = _torch_logpmf(xx, rr)
        return lp.sum(list(range(-group_ndims, 0))) if group_ndims else lp

    parity(got, x, rate, fn, dtype)
    if group_ndims == 0:  # scipy cross-check of the anchor itself
        sp = stats.poisson.logpmf(np.broadcast_to(x, shape), np.broadcast_to(rate, shape))
        np.testing.assert_allclose(_np64(fn(torch.tensor(x), torch.tensor(rate))), sp, rtol=1e-10, atol=1e-10)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("xs,rs", LAYOUTS[:3])
def test_rate_gradient(dev, dtype, xs, rs):
    rng = np.random.RandomState(12)
    rate = rng.gamma(2.0, 2.0, size=rs) + 0.1
    shape = np.broadcast_shapes(xs, rs)
    x = rng.poisson(3.0, size=xs).astype(np.float64)
    w = rng.standard_normal(shape[:-1])
    r = T(rate, dev, dtype, grad=True)
    lp = Poisson(r, group_ndims=1).log_prob(T(x, dev, dtype))
    (g,) = torch.autograd.grad((lp * T(w, dev, dtype)).sum(), [r])

    def fn(xx, rr):
        rr = rr.clone().requires_grad_()
        out = (_torch_logpmf(xx, rr).sum(-1) * torch.tensor(w, dtype=rr.dtype)).sum()
        return torch.autograd.grad(out, [rr])[0]

    parity(g, x, rate, fn, dtype)


def test_counts_carry_no_gradient(dev):
    x = T([1.0, 2.0], dev, grad=True)
    with pytest.raises(ValueError, match="counts have no gradient"):
        Poisson(T([1.0, 3.0], dev)).log_prob(x)


@pytest.mark.parametrize("plan", [
    dict(group_ndims=0, reduce_mean_dims=None, reduce_sum_dims=[2]),
    dict(group_ndims=1, reduce_mean_dims=[0], reduce_sum_dims=None),
    dict(group_ndims=0, reduce_mean_dims=[1], reduce_sum_dims=[0]),
    dict(group_ndims=2, reduce_mean_dims=None, reduce_sum_dims=None, multiplier=3),
])
def test_stochastic_tensor_reductions(dev, plan):
    rng = np.random.RandomState(13)
    rate = rng.gamma(2.0, 1.5, size=(4, 6)) + 0.1
    x = rng.poisson(rate, size=(5, 4, 6)).astype(np.float64)
    net = BayesianNet(device=dev)
    net.observe({"n": T(x, dev)})
    kw = {k: v for k, v in plan.items() if k != "group_ndims"}
    net.poisson("n", rate=T(rate, dev), group_ndims=plan["group_ndims"], n_samples=5, **kw)
    got = net.nodes["n"].log_prob()
    ref = torch.tensor(stats.poisson.logpmf(x, rate))
    g = plan["group_ndims"]
    if g:
        ref = ref.sum(list(range(-g, 0)))
    dims = []
    if plan.get("reduce_mean_dims"):
        ref = ref.mean(plan["reduce_mean_dims"], keepdim=True)
        dims += plan["reduce_mean_dims"]
    if plan.get("reduce_sum_dims"):
        ref = ref.sum(plan["reduce_sum_dims"], keepdim=True)
        dims += plan["reduce_sum_dims"]
    for d in sorted(dims, reverse=True):
        ref = ref.squeeze(d)
    if plan.get("multiplier"):
        ref = ref * plan["multiplier"]
    assert tuple(got.shape) == tuple(ref.shape)
    r = _np64(ref)
    assert np.linalg.norm(_np64(got) - r) <= 1e-5 * np.linalg.norm(r)


# ============================================================================ distribution and framework surface
def test_distribution_surface(dev):
    rate = T([[0.5, 2.0, 7.0]], dev)
    p = Poisson(rate, check_numerics=True, some_unknown_kwarg=1)  # unknown kwargs are swallowed
    assert p.dtype == torch.float32 and not p.is_continuous and not p.is_reparameterized
    assert tuple(p.batch_shape) == (1, 3) and p.rate is not None
    assert torch.allclose(p.lograte.cpu(), torch.log(rate.cpu()))
    assert tuple(p.sample().shape) == (1, 3) and tuple(p.sample(1).shape) == (1, 3)  # Q3: no particle axis
    s = p.sample(4)
    assert tuple(s.shape) == (4, 1, 3) and s.dtype == torch.float32 and s.device.type == dev.type
    assert p.sample_cache is s
    assert torch.equal(p.log_prob(None), p.log_prob(s))  # Q2: log_prob(None) is taken at the cached sample
    s = s.cpu().numpy()
    assert np.all(s == np.round(s)) and np.all(s >= 0)
    assert Poisson(T([1.0], dev, torch.float64)).sample(3).dtype == torch.float64
    assert Poisson(torch.tensor([1.0, 2.0]), dtype=torch.float64).dtype == torch.float64
    with pytest.raises(TypeError, match="must have a dtype in"):
        Poisson(torch.tensor([1, 2], dtype=torch.int32))


def test_bayesian_net_registration(dev):
    net = BayesianNet(device=dev)
    a = net.sn("Poisson", "a", rate=T([1.0, 4.0], dev), n_samples=3)
    b = net.poisson("b", rate=T([2.0, 5.0], dev))
    assert tuple(a.shape) == (3, 2) and tuple(b.shape) == (2,)
    assert isinstance(net.nodes["a"], StochasticTensor) and isinstance(net.nodes["a"].dist, Poisson)
    assert tuple(net.nodes["a"].log_prob().shape) == (3, 2)
    net.observe({"c": T([3.0, 0.0], dev)})
    net.poisson("c", rate=T([3.0, 0.5], dev), group_ndims=1)
    np.testing.assert_allclose(_np64(net.nodes["c"].log_prob()), stats.poisson.logpmf([3, 0], [3.0, 0.5]).sum(),
                               rtol=1e-6)
    with pytest.raises(NotImplementedError):
        net.stochastic_node("Gamma", "g", alpha=1., beta=1.)
    with pytest.raises(ValueError):
        net.poisson(3, rate=1.0)


# ============================================================================ sampler
@pytest.mark.parametrize("lam", [0.1, 3.0, 9.9, 10.0, 40.0, 1e4])
def test_sampler_distribution(dev, lam):
    """Chi-square against the pmf and the first two moments, on both sides of the Knuth / PTRS switch at 10."""
    n = 60000
    s = Poisson(torch.full((n,), lam, device=dev)).sample().cpu().double().numpy()
    assert np.all(s == np.round(s)) and s.min() >= 0
    assert abs(s.mean() - lam) < 5 * math.sqrt(lam / n)
    assert abs(s.var() / lam - 1) < 0.04
    lo, hi = stats.poisson.ppf(1e-4, lam), stats.poisson.ppf(1 - 1e-4, lam)
    if hi - lo > 60:  # bin wide distributions into ~60 equiprobable-ish cells
        edges = np.unique(stats.poisson.ppf(np.linspace(1e-4, 1 - 1e-4, 61), lam))
    else:
        edges = np.arange(lo, hi + 1)
    edges = np.concatenate([[-0.5], edges[1:] - 0.5, [np.inf]])
    obs = np.histogram(s, edges)[0]
    cdf = stats.poisson.cdf(np.floor(edges[1:] - 0.5 + 1e-9), lam)
    exp = np.diff(np.concatenate([[0.0], cdf])) * n
    exp[-1] = n - exp[:-1].sum()
    keep = exp >= 5
    if keep.sum() >= 2:
        chi2 = ((obs[keep] - exp[keep]) ** 2 / exp[keep]).sum() + (obs[~keep].sum() - exp[~keep].sum()) ** 2 / max(
            exp[~keep].sum(), 5.0)
        assert stats.chi2.sf(chi2, keep.sum()) > 1e-4, chi2


def test_sampler_rate_zero_and_broadcast(dev):
    rate = T([[0.0, 2.0, 25.0]], dev)
    s = Poisson(rate).sample(2000).cpu().numpy()
    assert tuple(s.shape) == (2000, 1, 3)
    assert np.all(s[:, 0, 0] == 0)
    assert abs(s[:, 0, 1].mean() - 2.0) < 0.2 and abs(s[:, 0, 2].mean() - 25.0) < 1.0


# the kernel and the C restatement agree except where libm and CUDA math tip an accept / reject decision of PTRS
DISAGREE_MAX = 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_sampler_matches_oracle_and_geometry(dtype):
    import poisson_oracle
    rng = np.random.RandomState(14)
    n = 200000
    rate = np.concatenate([rng.uniform(0, 10, n // 2), rng.uniform(10, 500, n // 2)])
    r = torch.tensor(rate, dtype=dtype, device="cuda")
    big = _backend.poisson_sample(r, _backend.FULL, 1, n, seed=77, offset=8)
    small = _backend.poisson_sample(r[:1000].contiguous(), _backend.FULL, 1, 1000, seed=77, offset=8)
    assert torch.equal(big[0, :1000], small[0])  # a 1000-element grid draws what a 200000-element grid drew
    kb = _backend.poisson_sample(r[:500].contiguous(), _backend.KBCAST, 4, 500, seed=77, offset=8)
    ref_kb = poisson_oracle.poisson_sample(rate[:500].astype(_np_dtype(dtype)), _backend.KBCAST, 4, 500, 77, 8)
    ref = poisson_oracle.poisson_sample(rate.astype(_np_dtype(dtype)), _backend.FULL, 1, n, 77, 8)
    assert np.mean(big.cpu().numpy() != ref) <= DISAGREE_MAX
    assert np.mean(kb.cpu().numpy() != ref_kb) <= DISAGREE_MAX
    other = _backend.poisson_sample(r, _backend.FULL, 1, n, seed=77, offset=12)  # the next stream position
    assert np.mean(other.cpu().numpy() == big.cpu().numpy()) < 0.5


def _np_dtype(dtype):
    return np.float32 if dtype == torch.float32 else np.float64


@pytest.mark.gpu
def test_sampler_graph_replay_draws_fresh_samples():
    rate = torch.full((4096,), 6.0, device="cuda")
    p = Poisson(rate)
    p.sample(2)  # first draw outside capture initialises the device-side stream position
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            out = p.sample(2)
    torch.cuda.current_stream().wait_stream(s)
    g.replay()
    a = out.clone()
    g.replay()
    b = out.clone()
    assert not torch.equal(a, b)
    assert abs(a.mean().item() - 6.0) < 0.2 and abs(b.mean().item() - 6.0) < 0.2


# ============================================================================ fused Poisson-likelihood IW step
class _Gen(BayesianNet):
    def __init__(self, rate, K):
        super().__init__(device=rate.device)
        self.rate, self.K = rate, K

    def forward(self, observed):
        self.observe(observed)
        B, Z = self.observed["z"].shape[1:]
        dt, d = self.rate.dtype, self.rate.device
        self.normal("z", mean=torch.zeros([B, Z], dtype=dt, device=d), std=torch.ones([B, Z], dtype=dt, device=d),
                    is_reparameterized=False, n_samples=self.K, reduce_sum_dims=[2])
        self.sn(Poisson(self.rate), name="x", reduce_sum_dims=[2])
        return self


class _Var(BayesianNet):
    def __init__(self, mean, logstd, K, reparam):
        super().__init__(device=mean.device)
        self.mean, self.logstd, self.K, self.reparam = mean, logstd, K, reparam

    def forward(self, observed):
        self.observe(observed)
        self.sn(Normal(mean=self.mean, logstd=self.logstd, is_reparameterized=self.reparam), name="z",
                n_samples=self.K, reduce_sum_dims=[2])
        return self


def _iw_step(dev, est, K, B, X, Z, fused, seed=21, dtype=torch.float32):
    """Loss and boundary gradients (rate, mean, logstd) through the public API, plus what the reference
    restatement needs: the counts, the rates, the latent sample and its log-densities."""
    rng = np.random.RandomState(seed)
    x = T(rng.poisson(2.0, size=(B, X)).astype(np.float64), dev, dtype)
    rate = T(rng.gamma(2.0, 1.0, size=(K, B, X)) + 0.05, dev, dtype, grad=True)
    mean = T(0.3 * rng.standard_normal((B, Z)), dev, dtype, grad=True)
    logstd = T(0.1 * rng.standard_normal((B, Z)), dev, dtype, grad=True)
    eps = T(rng.standard_normal((K, B, Z)), dev, dtype)
    zhusuan.variational.FUSED = fused
    try:
        gen, var = _Gen(rate, K), _Var(mean, logstd, K, est == "sgvb")
        obj = ImportanceWeightedObjective(gen, var, axis=0, estimator=est)
        with _rng.inject(normal=[eps, eps]):
            loss = obj({"x": x})
        (loss * 2.0).backward()  # a non-unit upstream gradient exercises the in-place scaling
    finally:
        zhusuan.variational.FUSED = True
    z = var.nodes["z"].dist.sample_cache.detach()  # the sample the step used (`.tensor` would draw a new one)
    logq = var.nodes["z"].log_prob().detach()
    return dict(loss=loss.detach(), drate=rate.grad, dmean=mean.grad, dlogstd=logstd.grad, x=x, rate=rate.detach(),
                z=z, logq=logq, gen=gen)


def _restate(r, dtype):
    """torch restatement of the Poisson-likelihood step on the latent sample the step used, in `dtype`: the SGVB loss
    and d/drate (d cost / d log p(x|z) is -w / B for both estimators; the VIMCO control variate acts on log q only)."""
    x, rate = r["x"].cpu().to(dtype), r["rate"].cpu().to(dtype).requires_grad_()
    z = r["z"].cpu().to(dtype)
    logpx = torch.distributions.Poisson(rate, validate_args=False).log_prob(x.unsqueeze(0)).sum(-1)
    logpz = torch.distributions.Normal(torch.zeros((), dtype=dtype), torch.ones((), dtype=dtype)).log_prob(z).sum(-1)
    logw = logpx + logpz - r["logq"].cpu().to(dtype)
    w = torch.softmax(logw, 0).detach()
    surrogate = -(w * logw).sum(0).mean()
    (drate,) = torch.autograd.grad(surrogate, [rate])
    return surrogate.detach(), drate


def _check_step(fz, tp, est):
    """Parity rule for the step.  Its float32 log-weights are about -1.3e3 here, so the rounding of a log-weight (one
    float32 ulp is 1.2e-4) moves every weight and gradient by ~1e-4 relative: float32 torch itself is that far from
    float64.  Both routes must stay within max(2e-5, twice float32 torch's distance) of float64 torch, and within
    twice that of each other for the gradients the restatement does not cover."""
    loss64, drate64 = _restate(fz, torch.float64)
    loss32, drate32 = _restate(fz, torch.float32)
    tol = max(2e-5, 2 * _normwise(drate32, drate64), 2 * _normwise(loss32, loss64))
    for r in (fz, tp):
        assert _normwise(r["drate"] / 2.0, drate64) < tol
        if est == "sgvb":  # the VIMCO surrogate adds a control-variate term in log q
            assert _normwise(r["loss"], loss64) < tol
    for k in ("loss", "drate", "dmean", "dlogstd"):
        assert _normwise(fz[k], tp[k]) < 2 * tol, k


def _normwise(a, b):
    a, b = _np64(a), _np64(b)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


@pytest.mark.parametrize("est", ["sgvb", "vimco"])
def test_fused_step_matches_two_pass_and_reference(dev, est):
    """K = 50, X = 784: the fixed-geometry Poisson kernel (on CUDA) against the two-pass route and a float64 torch
    restatement, in loss and every boundary gradient."""
    if dev.type == "cpu" and torch.cuda.is_available():
        pytest.skip("the fused route needs device-resident rates (host-resident ones take the generic path)")
    K, B, X, Z = 50, 6, 784, 4
    fz = _iw_step(dev, est, K, B, X, Z, fused=True)
    tp = _iw_step(dev, est, K, B, X, Z, fused=False)
    assert torch.equal(fz["z"], tp["z"])
    _check_step(fz, tp, est)


@pytest.mark.gpu
@pytest.mark.parametrize("est", ["sgvb", "vimco"])
def test_fused_step_full_size(est):
    """B = 1024 (the 160 MB rate tensor): fused against the two-pass route and the float64 restatement, normwise."""
    dev = torch.device("cuda")
    K, B, X, Z = 50, 1024, 784, 8
    fz = _iw_step(dev, est, K, B, X, Z, fused=True, seed=22)
    assert _backend.fused_poisson_supported(K, X, torch.float32)
    tp = _iw_step(dev, est, K, B, X, Z, fused=False, seed=22)
    _check_step(fz, tp, est)


@pytest.mark.gpu
def test_fused_kernel_dispatch_and_fallback():
    """X = 100 has no fixed-geometry instantiation: the entry point refuses, the public API falls back silently to the
    two-pass route and gives the same numbers as with FUSED = False."""
    dev = torch.device("cuda")
    rate = torch.rand(8, 3, 100, device=dev) + 0.1
    x = torch.randint(0, 4, (3, 100), device=dev).float()
    assert _backend.iw_poisson_fused(_backend.SGVB, rate, x, None, None, 1.0 / 3) is None
    ok = _backend.iw_poisson_fused(_backend.SGVB, torch.rand(8, 3, 128, device=dev) + 0.1,
                                   torch.randint(0, 4, (3, 128), device=dev).float(), None, None, 1.0 / 3)
    assert ok is not None
    a = _iw_step(dev, "sgvb", 8, 3, 100, 2, fused=True, seed=23)
    b = _iw_step(dev, "sgvb", 8, 3, 100, 2, fused=False, seed=23)
    for k in ("loss", "drate", "dmean", "dlogstd"):
        assert torch.equal(a[k], b[k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("est", [_backend.SGVB, _backend.VIMCO])
def test_fused_kernel_entry_point_against_restatement(est):
    """zs_iw_poisson_fused at each instantiated row length (K = 50 and K = 7), against the oracle restatement; with
    counts that are mostly zero and rates of at least 0.01 (zero and subnormal rates: tests/test_fused_box_columns.py)."""
    import poisson_oracle
    rng = np.random.RandomState(24)
    for X, K in ((128, 50), (256, 7), (512, 50), (784, 50), (1024, 33)):
        B = 5
        rate = (rng.gamma(1.0, 2.0, size=(K, B, X)) + 0.01).astype(np.float32)
        x = (rng.poisson(0.3, size=(B, X))).astype(np.float32)
        lo = rng.standard_normal((K, B)).astype(np.float32)
        lq = rng.standard_normal((K, B)).astype(np.float32)
        t = lambda a: torch.tensor(a, device="cuda")
        r = _backend.iw_poisson_fused(est, t(rate), t(x), t(lo), t(lq), 1.0 / B, want_logpx=True)
        ref = poisson_oracle.iw_poisson_step(est, rate.astype(np.float64), x.astype(np.float64), lo.astype(np.float64),
                                             lq.astype(np.float64), 1.0 / B)
        assert _normwise(r["logpx"], ref["logpx"]) < 1e-6, X
        assert _normwise(r["cost"], ref["cost"]) < 2e-5, X
        assert _normwise(r["dlogp"], ref["dlogp"]) < 2e-5, X
        assert _normwise(r["dlogq"], ref["dlogq"]) < 2e-5, X
        assert _normwise(r["dprobs"], ref["drate"]) < 2e-5, X
