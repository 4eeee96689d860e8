"""The Beta node: log-density and its gradients w.r.t. x, alpha and beta (every layout mode, fp32 / fp64, event and
StochasticTensor reductions, every row-kernel path), the sampler, BayesianNet registration and a Beta-Bernoulli model
under the two estimators for non-reparameterised latents.

Modes as in tests/test_poisson.py: `oracle` (CPU; the ctypes backend replaced by the CPU oracle, with the Beta node
restated in oracle/zs_oracle_impl.h), `cuda` (B200 kernels, CUDA tensors) and `cuda-host` (CPU tensors in and out).
The anchor is torch.distributions.Beta in float64, the function the reference's Beta delegates to, cross-checked with
scipy.  Parity rule (DESIGN.md §4): float64 within 1e-12 normwise; float32 within 1e-5 normwise of float64 torch, or
no farther from it than float32 torch is.  Non-finite entries must match float64 torch exactly.
"""
import math
import zlib

import numpy as np
import pytest
import torch
from scipy import special, stats

import zhusuan.variational
from zhusuan import _backend
from zhusuan.distributions import Beta, Bernoulli
from zhusuan.framework import BayesianNet, StochasticTensor
from zhusuan.variational import ELBO, ImportanceWeightedObjective

MODES = [pytest.param("oracle"), pytest.param("cuda", marks=pytest.mark.gpu),
         pytest.param("cuda-host", marks=pytest.mark.gpu)]
FULL, KBCAST, SCALAR = _backend.FULL, _backend.KBCAST, _backend.SCALAR


@pytest.fixture(params=MODES)
def dev(request, monkeypatch):
    mode = request.param
    if mode == "oracle":
        import oracle_backend
        request.getfixturevalue("oracle")  # rebuilds the oracle library if its sources changed
        oracle_backend.install(monkeypatch)
        return torch.device("cpu")
    return torch.device("cuda") if mode == "cuda" else torch.device("cpu")


def T(a, dev, dtype=torch.float32, grad=False):
    t = torch.tensor(np.asarray(a), dtype=dtype, device=dev)
    t.requires_grad_(grad)
    return t


def _np64(t):
    return t.detach().cpu().double().numpy() if torch.is_tensor(t) else np.asarray(t, np.float64)


def _np_dtype(dtype):
    return np.float32 if dtype == torch.float32 else np.float64


def _torch_logpdf(x, a, b):
    return torch.distributions.Beta(a, b, validate_args=False).log_prob(x)


def parity(got, args, fn, dtype):
    """`fn(*args)` is the torch restatement; compare `got` with it in float64 under the parity rule.  `args` are the
    values the kernel saw (already rounded to `dtype`)."""
    ref64 = _np64(fn(*[torch.tensor(_np64(v)) for v in args]))
    g = _np64(got)
    assert g.shape == ref64.shape
    fin = np.isfinite(ref64)
    np.testing.assert_array_equal(g[~fin], ref64[~fin])
    assert np.all(np.isfinite(g[fin]))
    err = np.linalg.norm(g[fin] - ref64[fin])
    nrm = max(np.linalg.norm(ref64[fin]), 1e-30)
    if dtype == torch.float64:
        assert err <= 1e-12 * nrm, err / nrm
        return
    ref32 = _np64(fn(*[torch.tensor(_np64(v), dtype=torch.float32) for v in args]))
    assert err <= max(1e-5 * nrm, np.linalg.norm(ref32[fin] - ref64[fin])), err / nrm


# ============================================================================ values and gradients
# (x shape, alpha shape, beta shape): all FULL; alpha and beta broadcast over particles (KBCAST); x broadcast (KBCAST);
# alpha and beta both SCALAR; alpha SCALAR with beta FULL
LAYOUTS = [((5, 4, 6), (5, 4, 6), (5, 4, 6)), ((5, 4, 6), (4, 6), (4, 6)), ((4, 6), (5, 4, 6), (5, 4, 6)),
           ((5, 4, 6), (), ()), ((5, 4, 6), (), (5, 4, 6))]
LAYOUT_IDS = ["full", "params_kbcast", "x_kbcast", "params_scalar", "alpha_scalar"]
# edges, at full-shape positions: x = 0 with alpha = 1 (finite value, dx = NaN), x = 0 with alpha < 1 (+inf),
# x = 1 with beta < 1 (+inf), x = 1 with beta = 1
EDGES = [((0, 0, 0), 0.0, 1.0, None), ((1, 1, 1), 0.0, 0.5, None), ((2, 2, 2), 1.0, None, 0.5),
         ((3, 3, 3), 1.0, None, 1.0)]


def _plant(arr, pos, v):
    if arr.ndim == 0 or v is None:
        return
    arr[tuple(pos[len(pos) - arr.ndim:])] = v


def _inputs(xs, as_, bs, seed, edges=True):
    """x mostly inside (0, 1) with the EDGES planted; parameters from a mix of < 1, == 1, moderate and 500."""
    rng = np.random.RandomState(seed)

    def param(shape):
        if not shape:  # the SCALAR layouts: alpha = 1 meets the x = 0 edge
            return np.array(1.0)
        p = rng.choice([0.3, 0.7, 1.0, 2.5, 6.0, 40.0, 500.0], size=shape) * rng.uniform(0.9, 1.1, size=shape)
        p.reshape(-1)[::9] = 1.0
        return p

    a, b = param(as_), param(bs)
    if not bs:
        b = np.array(0.5)
    x = rng.uniform(0.02, 0.98, size=xs)
    if edges:
        for pos, xv, av, bv in EDGES:
            _plant(x, pos, xv)
            _plant(a, pos, av)
            _plant(b, pos, bv)
    return x, a, b


def _rounded(v, dtype):
    return np.asarray(v, _np_dtype(dtype)).astype(np.float64)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("shapes", LAYOUTS, ids=LAYOUT_IDS)
@pytest.mark.parametrize("group_ndims", [0, 1, 2])
def test_log_prob_values(dev, dtype, shapes, group_ndims):
    x, a, b = [_rounded(v, dtype) for v in _inputs(*shapes, seed=31)]
    d = Beta(T(a, dev, dtype), T(b, dev, dtype), group_ndims=group_ndims)
    got = d.log_prob(T(x, dev, dtype))
    assert got.dtype == dtype and got.device.type == dev.type

    def fn(xx, aa, bb):
        lp = _torch_logpdf(xx, aa, bb)
        return lp.sum(list(range(-group_ndims, 0))) if group_ndims else lp

    parity(got, (x, a, b), fn, dtype)
    if group_ndims == 0:  # scipy cross-check of the anchor itself, away from the edges
        shape = np.broadcast_shapes(*shapes)
        xb, ab, bb = [np.broadcast_to(v, shape) for v in (x, a, b)]
        inner = (xb > 0) & (xb < 1)
        ref = _np64(fn(torch.tensor(x), torch.tensor(a), torch.tensor(b)))
        np.testing.assert_allclose(ref[inner], stats.beta.logpdf(xb[inner], ab[inner], bb[inner]), rtol=1e-9,
                                   atol=1e-9)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("shapes", LAYOUTS, ids=LAYOUT_IDS)
def test_gradients(dev, dtype, shapes):
    """d/dx, d/dalpha, d/dbeta against torch float64 autograd, with the edge patterns (NaN / inf) included."""
    x, a, b = [_rounded(v, dtype) for v in _inputs(*shapes, seed=32)]
    shape = np.broadcast_shapes(*shapes)
    w = _rounded(np.random.RandomState(33).standard_normal(shape[:-1]), dtype)
    tx, ta, tb = T(x, dev, dtype, True), T(a, dev, dtype, True), T(b, dev, dtype, True)
    lp = Beta(ta, tb, group_ndims=1).log_prob(tx)
    got = torch.autograd.grad((lp * T(w, dev, dtype)).sum(), [tx, ta, tb])

    for i in range(3):
        def fn(xx, aa, bb, i=i):
            ins = [v.clone().requires_grad_() for v in (xx, aa, bb)]
            out = (_torch_logpdf(*ins).sum(-1) * torch.tensor(w, dtype=xx.dtype)).sum()
            return torch.autograd.grad(out, [ins[i]])[0]

        parity(got[i], (x, a, b), fn, dtype)


def test_edge_patterns_come_from_torch(dev):
    """The inf / NaN pattern of the edges, read from torch float64 and matched exactly in both dtypes."""
    x = np.array([0.0, 0.0, 1.0, 1.0, 0.0])
    a = np.array([1.0, 0.5, 2.0, 3.0, 2.0])
    b = np.array([2.0, 2.0, 0.5, 1.0, 1.0])
    for dtype in (torch.float32, torch.float64):
        tx, ta, tb = T(x, dev, dtype, True), T(a, dev, dtype, True), T(b, dev, dtype, True)
        lp = Beta(ta, tb).log_prob(tx)
        got = torch.autograd.grad(lp.sum(), [tx, ta, tb])
        rx, ra, rb = [torch.tensor(v, requires_grad=True) for v in (x, a, b)]
        ref = _torch_logpdf(rx, ra, rb)
        refg = torch.autograd.grad(ref.sum(), [rx, ra, rb])
        for g_, r_ in zip((lp,) + tuple(got), (ref,) + tuple(refg)):
            g_, r_ = _np64(g_), _np64(r_)
            fin = np.isfinite(r_)
            np.testing.assert_array_equal(g_[~fin], r_[~fin])
            np.testing.assert_allclose(g_[fin], r_[fin], rtol=1e-5, atol=1e-6)


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_digamma_accuracy(dev, dtype):
    """dalpha at x = 0.5 and g = 1 is log 0.5 - psi(alpha) + psi(alpha + beta): psi over alpha in [1e-3, 1e4]
    against scipy.special.digamma, element by element against the sum of the terms' magnitudes."""
    alpha = _rounded(np.logspace(-3, 4, 200), dtype)
    beta = _rounded(np.full(200, 0.7), dtype)
    ta = T(alpha, dev, dtype, True)
    lp = Beta(ta, T(beta, dev, dtype)).log_prob(T(np.full(200, 0.5), dev, dtype))
    (da,) = torch.autograd.grad(lp.sum(), [ta])
    ab = _rounded(alpha + beta, dtype)  # the kernel adds in the operand dtype
    pa, pab = special.digamma(alpha), special.digamma(ab)
    ref = math.log(0.5) - pa + pab
    mag = abs(math.log(0.5)) + np.abs(pa) + np.abs(pab)
    tol = 1e-13 if dtype == torch.float64 else 64 * 2.0 ** -24  # the recurrence's rounding, relative to the terms
    err = np.abs(_np64(da) - ref) / mag
    assert err.max() <= tol, (err.max(), alpha[err.argmax()])


@pytest.mark.parametrize("plan", [
    dict(group_ndims=0, reduce_mean_dims=None, reduce_sum_dims=[2]),
    dict(group_ndims=1, reduce_mean_dims=[0], reduce_sum_dims=None),
    dict(group_ndims=0, reduce_mean_dims=[1], reduce_sum_dims=[0]),
    dict(group_ndims=2, reduce_mean_dims=None, reduce_sum_dims=None, multiplier=3),
])
def test_stochastic_tensor_reductions(dev, plan):
    rng = np.random.RandomState(34)
    a, b = rng.uniform(0.5, 4.0, size=(4, 6)), rng.uniform(0.5, 4.0, size=(4, 6))
    x = rng.beta(a, b, size=(5, 4, 6)).clip(1e-6, 1 - 1e-6)
    net = BayesianNet(device=dev)
    net.observe({"p": T(x, dev, torch.float64)})
    kw = {k: v for k, v in plan.items() if k != "group_ndims"}
    net.beta("p", alpha=T(a, dev, torch.float64), beta=T(b, dev, torch.float64), group_ndims=plan["group_ndims"],
             n_samples=5, **kw)
    got = net.nodes["p"].log_prob()
    ref = torch.tensor(stats.beta.logpdf(x, a, b))
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
    assert np.linalg.norm(_np64(got) - r) <= 1e-9 * np.linalg.norm(r)


# ============================================================================ distribution and framework surface
def test_distribution_surface(dev):
    alpha, beta = T([[0.5, 2.0, 7.0]], dev), T([1.5], dev)
    d = Beta(alpha, beta, check_numerics=True, some_unknown_kwarg=1)  # unknown kwargs are swallowed
    assert d.dtype == torch.float32 and d.is_continuous and not d.is_reparameterized
    assert tuple(d.batch_shape) == (1, 3) and d.alpha is not None and d.beta is not None
    assert tuple(d.sample().shape) == (1, 3) and tuple(d.sample(1).shape) == (1, 3)  # no particle axis for 1
    s = d.sample(4)
    assert tuple(s.shape) == (4, 1, 3) and s.dtype == torch.float32 and s.device.type == dev.type
    assert d.sample_cache is s
    assert torch.equal(d.log_prob(None), d.log_prob(s))  # log_prob(None) is taken at the cached sample
    assert np.all(np.isfinite(_np64(d.log_prob(s))))
    sn = s.cpu().numpy()
    assert np.all(sn > 0) and np.all(sn < 1)
    a_req = T([2.0, 3.0], dev, grad=True)
    assert not Beta(a_req, T([1.0, 1.0], dev)).sample(2).requires_grad  # no pathwise gradient
    assert Beta(T([1.0], dev, torch.float64), T([2.0], dev, torch.float64)).sample(3).dtype == torch.float64
    assert Beta(torch.tensor([1.0, 2.0]), 1.0, dtype=torch.float64).dtype == torch.float64
    with pytest.raises(TypeError, match="must have a dtype in"):
        Beta(torch.tensor([1, 2], dtype=torch.int32), torch.tensor([1, 2], dtype=torch.int32))
    np.testing.assert_allclose(_np64(d.prob(T([[0.5, 0.5, 0.5]], dev))),
                               stats.beta.pdf(0.5, [[0.5, 2.0, 7.0]], 1.5), rtol=1e-5)


def test_bayesian_net_registration(dev):
    net = BayesianNet(device=dev)
    a = net.sn("Beta", "a", alpha=T([1.0, 4.0], dev), beta=T([2.0, 0.5], dev), n_samples=3)
    b = net.beta("b", alpha=T([2.0, 5.0], dev), beta=T([1.0, 1.0], dev))
    c = net.sn(Beta(T([0.5, 3.0], dev), T([0.5, 3.0], dev)), "c", n_samples=2)
    assert tuple(a.shape) == (3, 2) and tuple(b.shape) == (2,) and tuple(c.shape) == (2, 2)
    for name in ("a", "b", "c"):
        assert isinstance(net.nodes[name], StochasticTensor) and isinstance(net.nodes[name].dist, Beta)
    assert tuple(net.nodes["a"].log_prob().shape) == (3, 2)
    net.observe({"o": T([0.25, 0.75], dev)})
    net.beta("o", alpha=T([3.0, 0.5], dev), beta=T([2.0, 1.5], dev), group_ndims=1)
    np.testing.assert_allclose(_np64(net.nodes["o"].log_prob()),
                               stats.beta.logpdf([0.25, 0.75], [3.0, 0.5], [2.0, 1.5]).sum(), rtol=1e-5)
    for name, kw in (("Gamma", dict(alpha=1., beta=1.)), ("Exponential", dict(rate=1.)),
                     ("StudentT", dict(df=3., loc=0., scale=1.))):
        with pytest.raises(NotImplementedError):
            net.stochastic_node(name, "g", **kw)
    with pytest.raises(ValueError):
        net.beta(3, alpha=1.0, beta=1.0)


# ============================================================================ sampler
def _ks_pvalue(s, a, b):
    """Kolmogorov-Smirnov p-value against scipy.stats.beta, with the statistic taken over the samples below 1 - 1e-9:
    above that the dtype cannot represent the distribution (Beta(0.1, 0.1) puts 1.3% of its mass beyond 1 - 2^-53,
    which the sampler's clamp, like torch's, returns as nextafter(1, 0))."""
    s = np.sort(s)
    n = s.size
    F = stats.beta.cdf(s, a, b)
    i = np.arange(1, n + 1)
    inner = s < 1 - 1e-9
    d = max(np.max((i / n - F)[inner]), np.max((F - (i - 1) / n)[inner]))
    return stats.kstwo.sf(d, n)


@pytest.mark.parametrize("ab", [(0.1, 0.1), (0.5, 3.0), (1.0, 1.0), (2.0, 5.0), (30.0, 0.7), (200.0, 50.0)])
def test_sampler_distribution(dev, ab):
    """Kolmogorov-Smirnov against scipy.stats.beta, and the first two moments."""
    a, b = ab
    n = 50000
    s = Beta(torch.full((n,), a, dtype=torch.float64, device=dev), torch.full((n,), b, dtype=torch.float64,
                                                                            device=dev)).sample()
    s = s.cpu().numpy()
    assert np.all(s > 0) and np.all(s < 1)
    assert _ks_pvalue(s, a, b) > 1e-4
    mean = a / (a + b)
    var = a * b / ((a + b) ** 2 * (a + b + 1))
    assert abs(s.mean() - mean) < 5 * math.sqrt(var / n)
    assert abs(s.var() / var - 1) < 0.05


@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_sampler_tiny_parameters_stay_in_range(dev, dtype):
    """alpha = beta = 1e-3: most gamma draws underflow, yet no sample is NaN, 0 or 1, and log_prob stays finite."""
    n = 100000
    d = Beta(torch.full((n,), 1e-3, dtype=dtype, device=dev), torch.full((n,), 1e-3, dtype=dtype, device=dev))
    s = d.sample()
    sn = s.cpu().numpy()
    fi = np.finfo(_np_dtype(dtype))
    assert not np.any(np.isnan(sn))
    assert sn.min() >= fi.tiny and sn.max() <= np.nextafter(_np_dtype(dtype)(1), _np_dtype(dtype)(0))
    assert np.all(np.isfinite(_np64(d.log_prob(s))))
    assert 0.3 < np.mean(sn < 0.5) < 0.7  # U-shaped: mass at both ends


def test_sampler_broadcast_modes(dev):
    """alpha [3] with a scalar beta: the particles read alpha KBCAST; per-column means."""
    alpha = T([0.5, 2.0, 20.0], dev)
    s = Beta(alpha, 2.0).sample(4000).cpu().numpy()
    assert tuple(s.shape) == (4000, 3)
    for j, a in enumerate([0.5, 2.0, 20.0]):
        m, v = a / (a + 2.0), a * 2.0 / ((a + 2.0) ** 2 * (a + 3.0))
        assert abs(s[:, j].mean() - m) < 5 * math.sqrt(v / 4000)


def test_sampler_invalid_parameters_give_nan(dev):
    alpha = T([0.0, -1.0, float("nan"), float("inf"), 2.0], dev)
    s = Beta(alpha, T([1.0, 1.0, 1.0, 1.0, 0.0], dev)).sample().cpu().numpy()
    assert np.all(np.isnan(s))


# the kernel and the C restatement agree except where libm and CUDA math tip an accept / reject decision
DISAGREE_MAX = 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_sampler_matches_oracle_geometry_and_modes(oracle, dtype):
    rng = np.random.RandomState(35)
    n = 200000
    a = np.exp(rng.uniform(-4, 6, n)).astype(_np_dtype(dtype))
    b = np.exp(rng.uniform(-4, 6, n)).astype(_np_dtype(dtype))
    ta, tb = torch.tensor(a, device="cuda"), torch.tensor(b, device="cuda")
    big = _backend.beta_sample(ta, FULL, tb, FULL, 1, n, seed=91, offset=8)
    small = _backend.beta_sample(ta[:1000].contiguous(), FULL, tb[:1000].contiguous(), FULL, 1, 1000, seed=91,
                                 offset=8)
    assert torch.equal(big[0, :1000], small[0])  # a 1000-element launch draws what a 200000-element launch drew
    ref = oracle.beta_sample(a, FULL, b, FULL, 1, n, 91, 8)
    assert np.mean(~np.isclose(big.cpu().numpy(), ref, rtol=1e-6, atol=0)) <= DISAGREE_MAX
    # KBCAST and SCALAR parameters draw what the same values expanded to FULL draw
    K, N = 4, 500
    kb = _backend.beta_sample(ta[:N].contiguous(), KBCAST, tb[:N].contiguous(), KBCAST, K, N, seed=91, offset=8)
    full = _backend.beta_sample(ta[:N].repeat(K).contiguous(), FULL, tb[:N].repeat(K).contiguous(), FULL, K, N,
                                seed=91, offset=8)
    assert torch.equal(kb, full)
    ref_kb = oracle.beta_sample(a[:N], KBCAST, b[:N], KBCAST, K, N, 91, 8)
    assert np.mean(~np.isclose(kb.cpu().numpy(), ref_kb, rtol=1e-6, atol=0)) <= DISAGREE_MAX
    sc = _backend.beta_sample(ta[:1].contiguous(), SCALAR, tb[:1].contiguous(), SCALAR, K, N, seed=91, offset=8)
    sc_full = _backend.beta_sample(ta[:1].expand(K * N).contiguous(), FULL, tb[:1].expand(K * N).contiguous(), FULL,
                                   K, N, seed=91, offset=8)
    assert torch.equal(sc, sc_full)
    other = _backend.beta_sample(ta, FULL, tb, FULL, 1, n, seed=91, offset=12)  # the next stream position
    o, bg = other.cpu().numpy(), big.cpu().numpy()
    fi = np.finfo(_np_dtype(dtype))
    inner = (bg > fi.tiny) & (bg < 1 - fi.epsneg)  # clamped samples coincide at any position
    assert np.mean(o[inner] == bg[inner]) < 0.01


@pytest.mark.gpu
def test_sampler_graph_replay_draws_fresh_samples():
    d = Beta(torch.full((4096,), 2.0, device="cuda"), torch.full((4096,), 3.0, device="cuda"))
    d.sample(2)  # first draw outside capture initialises the device-side stream position
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            out = d.sample(2)
    torch.cuda.current_stream().wait_stream(s)
    g.replay()
    a = out.clone()
    g.replay()
    b = out.clone()
    assert not torch.equal(a, b)
    assert abs(a.mean().item() - 0.4) < 0.02 and abs(b.mean().item() - 0.4) < 0.02


# ============================================================================ row-kernel paths (GPU)
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _path_shape(path):
    """(K, M, E) selecting each path of dispatch_rows_fwd / dispatch_bwd (see tests/test_row_kernel_paths.py)."""
    if path == "lpr1":
        return (7, 300, 2)
    if path == "lpr8":
        return (9, 70, 48)
    if path == "lpr32":
        return (50, 64, 784)
    if path == "cluster_split":  # E >= 2048 and few rows: cluster forward, split (or 256-lane) backward
        K, M = 2, 1
        assert K * M * 32 < _sms() * 1024
        return (K, M, 8192)
    raise AssertionError(path)


PATHS = ["lpr1", "lpr8", "lpr32", "cluster_split"]


def _path_inputs(K, M, E, modes, dtype, seed):
    rng = np.random.RandomState(seed)
    shp = {FULL: (K, M, E), KBCAST: (M, E), SCALAR: (1,)}
    x = rng.uniform(0.01, 0.99, size=shp[modes[0]])
    a = np.exp(rng.uniform(-1.5, 3.0, size=shp[modes[1]]))
    b = np.exp(rng.uniform(-1.5, 3.0, size=shp[modes[2]]))
    return [torch.tensor(v, dtype=dtype, device="cuda") for v in (x, a, b)]


def _full(t, mode, K, M, E):
    if mode == FULL:
        return t
    return t.reshape(1, M, E).expand(K, M, E) if mode == KBCAST else t.reshape(1, 1, 1).expand(K, M, E)


def _ref_fwd_bwd(x, a, b, modes, K, M, E, g):
    """torch in the dtype of x: row sums [K, M] and the gradients of sum(g * rows) in the operands' layouts."""
    ins = [_full(v.cpu(), m, K, M, E).clone().requires_grad_() for v, m in zip((x, a, b), modes)]
    rows = _torch_logpdf(*ins).sum(-1)
    grads = torch.autograd.grad((rows * g.cpu().to(x.dtype)).sum(), ins)
    out = []
    for gr, m in zip(grads, modes):
        out.append(gr if m == FULL else (gr.sum(0) if m == KBCAST else None))
    return rows, out


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("path", PATHS)
@pytest.mark.parametrize("layout", ["full", "latent", "likelihood", "prior"])
def test_row_paths(dtype, path, layout):
    """Every row-kernel path in the layouts a Beta node runs in: all FULL, the variational posterior (alpha, beta
    KBCAST; the backward takes k_kreduce_bwd), x broadcast (k_kreduce_bwd for dx) and the prior (alpha, beta SCALAR)."""
    K, M, E = _path_shape(path)
    modes = {"full": (FULL, FULL, FULL), "latent": (FULL, KBCAST, KBCAST), "likelihood": (KBCAST, FULL, FULL),
             "prior": (FULL, SCALAR, SCALAR)}[layout]
    x, a, b = _path_inputs(K, M, E, modes, dtype, seed=zlib.crc32(repr((path, layout)).encode()) % 10000)
    g = torch.randn(K, M, dtype=dtype, device="cuda")
    fam = _backend.FAM_BETA
    rows = _backend.locscale_logprob_fwd(fam, x, modes[0], a, modes[1], b, modes[2], K, M, E)
    need = [True, modes[1] != SCALAR, modes[2] != SCALAR]
    grads = _backend.locscale_logprob_bwd(fam, g, x, modes[0], a, modes[1], b, modes[2], K, M, E, *need)
    args = [v.double().cpu() for v in (x, a, b)]

    def fwd(xx, aa, bb):
        ins = [_full(v, m, K, M, E) for v, m in zip((xx, aa, bb), modes)]
        return _torch_logpdf(*ins).sum(-1)

    parity(rows, args, fwd, dtype)
    for i in range(3):
        if not need[i]:
            continue

        def bwd(xx, aa, bb, i=i):
            return _ref_fwd_bwd(xx, aa, bb, modes, K, M, E, g)[1][i]

        parity(grads[i], args, bwd, dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
@pytest.mark.parametrize("path", PATHS)
def test_scalar_parameters_bit_identical_to_full(dtype, path):
    """SCALAR alpha and beta (the hoisted lgamma / psi terms) give the bits of the same values expanded to FULL:
    forward, and the backward w.r.t. x."""
    K, M, E = _path_shape(path)
    x, a, b = _path_inputs(K, M, E, (FULL, SCALAR, SCALAR), dtype, seed=36)
    af, bf = a.expand(K * M * E).contiguous(), b.expand(K * M * E).contiguous()
    g = torch.randn(K, M, dtype=dtype, device="cuda")
    fam = _backend.FAM_BETA
    r_s = _backend.locscale_logprob_fwd(fam, x, FULL, a, SCALAR, b, SCALAR, K, M, E)
    r_f = _backend.locscale_logprob_fwd(fam, x, FULL, af, FULL, bf, FULL, K, M, E)
    assert torch.equal(r_s, r_f)
    dx_s = _backend.locscale_logprob_bwd(fam, g, x, FULL, a, SCALAR, b, SCALAR, K, M, E, True, False, False)[0]
    dx_f = _backend.locscale_logprob_bwd(fam, g, x, FULL, af, FULL, bf, FULL, K, M, E, True, False, False)[0]
    assert torch.equal(dx_s, dx_f)


@pytest.mark.gpu
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_kbcast_backward_is_full_backward_summed(dtype):
    """alpha, beta KBCAST (the hoisted psi values of k_kreduce_bwd_beta): the FULL backward summed over K in float64,
    under the parity rule."""
    K, M, E = 50, 64, 784
    x, a, b = _path_inputs(K, M, E, (FULL, KBCAST, KBCAST), dtype, seed=37)
    af, bf = a.expand(K, M, E).contiguous(), b.expand(K, M, E).contiguous()
    g = torch.randn(K, M, dtype=dtype, device="cuda")
    fam = _backend.FAM_BETA
    _, da, db = _backend.locscale_logprob_bwd(fam, g, x, FULL, a, KBCAST, b, KBCAST, K, M, E, False, True, True)
    _, daf, dbf = _backend.locscale_logprob_bwd(fam, g, x, FULL, af, FULL, bf, FULL, K, M, E, False, True, True)
    for got, full in ((da, daf), (db, dbf)):
        ref = full.double().sum(0)
        err = np.linalg.norm(_np64(got) - _np64(ref))
        nrm = np.linalg.norm(_np64(ref))
        assert err <= (1e-12 if dtype == torch.float64 else 1e-5) * nrm, err / nrm


# ============================================================================ Beta-Bernoulli model end to end
class _Gen(BayesianNet):
    def __init__(self, dev, dtype, K):
        super().__init__(device=dev)
        self.dt, self.K = dtype, K

    def forward(self, observed):
        self.observe(observed)
        d = self.device
        self.beta("z", alpha=torch.tensor(1.5, dtype=self.dt, device=d), beta=torch.tensor(2.0, dtype=self.dt, device=d),
                  n_samples=self.K, reduce_sum_dims=[2])
        self.sn(Bernoulli(probs=self.observed["z"]), name="x", reduce_sum_dims=[2])
        return self


class _Var(BayesianNet):
    def __init__(self, alpha, beta, K):
        super().__init__(device=alpha.device)
        self.alpha, self.beta_, self.K = alpha, beta, K

    def forward(self, observed):
        self.observe(observed)
        self.sn(Beta(alpha=self.alpha, beta=self.beta_), name="z", n_samples=self.K, reduce_sum_dims=[2])
        return self


def _model_step(dev, est, dtype, K=16, B=6, Z=5, seed=38):
    rng = np.random.RandomState(seed)
    x = T((rng.uniform(size=(B, Z)) < 0.4).astype(np.float64), dev, dtype)
    alpha = T(rng.uniform(0.8, 3.0, size=(B, Z)), dev, dtype, grad=True)
    beta = T(rng.uniform(0.8, 3.0, size=(B, Z)), dev, dtype, grad=True)
    gen, var = _Gen(dev, dtype, K), _Var(alpha, beta, K)
    if est == "vimco":
        obj = ImportanceWeightedObjective(gen, var, axis=0, estimator="vimco")
    else:
        obj = ELBO(gen, var, estimator="reinforce")
    loss = obj({"x": x})
    loss.backward()
    z = var.nodes["z"].dist.sample_cache.detach()
    mm = float(obj.moving_mean.item()) if est == "reinforce" else None
    return dict(loss=loss.detach(), dalpha=alpha.grad, dbeta=beta.grad, x=x, alpha=alpha.detach(), beta=beta.detach(),
                z=z, mm=mm)


def _restate(r, est, dtype):
    """torch restatement of the step on the latent sample it drew, in `dtype`: the surrogate loss and its gradients
    w.r.t. alpha and beta (the sample itself carries no gradient)."""
    x, z = r["x"].cpu().to(dtype), r["z"].cpu().to(dtype)
    alpha = r["alpha"].cpu().to(dtype).requires_grad_()
    beta = r["beta"].cpu().to(dtype).requires_grad_()
    prior = torch.distributions.Beta(torch.tensor(1.5, dtype=dtype), torch.tensor(2.0, dtype=dtype),
                                     validate_args=False)
    logpz = prior.log_prob(z).sum(-1)
    logpx = (x * torch.log(z + 1e-8) + (1 - x) * torch.log((1 - z) + 1e-8)).sum(-1)  # the package's Bernoulli
    lp = logpz + logpx
    lq = torch.distributions.Beta(alpha, beta, validate_args=False).log_prob(z).sum(-1)
    K = lp.shape[0]
    if est == "vimco":
        lw = lp - lq
        others = (lw.sum(0, keepdim=True) - lw) / (K - 1)  # each particle's log-weight replaced by the others' mean
        rep = lw.unsqueeze(0).repeat(K, 1, 1)
        idx = torch.arange(K)
        rep[idx, idx] = others
        lme = torch.logsumexp(lw, 0) - math.log(K)
        control = torch.logsumexp(rep, 1) - math.log(K)
        signal = (lme.unsqueeze(0) - control).detach()
        w = torch.softmax(lw, 0).detach()  # the reference's surrogate: -sum_k log q_k signal_k - sum_k w_k log w_k
        loss = (-(lq * signal).sum(0) - (w * lw).sum(0)).mean()
    else:
        signal = (lp - lq).detach() - torch.tensor(r["mm"], dtype=torch.float32).to(dtype)
        loss = (-(lp + signal * lq)).mean()
    da, db = torch.autograd.grad(loss, [alpha, beta])
    return loss.detach(), da, db


def _normwise(a, b):
    a, b = _np64(a), _np64(b)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30)


@pytest.mark.parametrize("est", ["vimco", "reinforce"])
@pytest.mark.parametrize("dtype", [torch.float32, torch.float64])
def test_beta_bernoulli_model(dev, est, dtype):
    """Prior Beta(1.5, 2) (SCALAR parameters), q = Beta(alpha[B,Z], beta[B,Z]) over K = 16 particles, x ~ Bernoulli(z):
    loss and the gradients of alpha and beta against a float64 torch restatement on the sample the step drew."""
    r = _model_step(dev, est, dtype)
    zn = _np64(r["z"])
    assert zn.shape == (16, 6, 5) and np.all((zn > 0) & (zn < 1))
    l64, da64, db64 = _restate(r, est, torch.float64)
    if dtype == torch.float64:
        tol = 1e-10
    else:
        l32, da32, db32 = _restate(r, est, torch.float32)
        tol = max(2e-5, 2 * _normwise(l32, l64), 2 * _normwise(da32, da64), 2 * _normwise(db32, db64))
    assert _normwise(r["loss"], l64) < tol
    assert _normwise(r["dalpha"], da64) < tol
    assert _normwise(r["dbeta"], db64) < tol
