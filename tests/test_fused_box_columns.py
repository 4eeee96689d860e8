"""The fixed-geometry box kernels (k_iw_bernoulli_boxf, k_iw_poisson_boxf) with many columns per CTA.

These kernels are persistent (at most one CTA per SM), and every CTA rotates per-column state: a 3-slot x / C_b
staging ring, a 4-slot ring of the [K, B] scalars and `nslot` tensor-copy slots (2 at X = 128 and X = 256).  State read
from the wrong column only shows once a CTA takes >= 4 columns, so B = 4 G + 3 here (G = the SM count): every CTA
takes at least 4 columns and the grid does not divide B.  Neighbouring columns differ strongly (counts, binary or
fractional x, logp_other, logq), so a wrong slot moves log p(x | z) or the cost by tens of nats.

References: oracle.iw_bernoulli_step, oracle.iw_bernoulli_logits_step and oracle.iw_poisson_step in
float64 for log p(x | z) and the cost; the gradients staged as in test_gpu_kernels.test_fused_vs_oracle (the oracle
fed the kernel's own log p(x | z), since the weights see exp() of float32 log-weights).  Every comparison is
elementwise, with the scale of the element's own column or row.
"""
import numpy as np
import pytest
import torch

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

from zhusuan import _backend as be  # noqa: E402

XS = [128, 256, 512, 784, 1024]
FORMS = ["probs", "logits", "poisson"]
# K = 1 (SGVB only); 25: one row per warp; 26 and 50: two rows per warp; 27: the last warp without its second row
CASES = [("sgvb", 1), ("sgvb", 26), ("sgvb", 50), ("vimco", 25), ("vimco", 27), ("vimco", 50)]


def _B():
    return 4 * torch.cuda.get_device_properties(0).multi_processor_count + 3


def _inputs(form, K, B, X, seed):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    col = torch.arange(B, device="cuda", dtype=torch.float32)
    n = lambda *s: torch.randn(*s, generator=g, device="cuda")  # noqa: E731
    if form == "poisson":
        p = torch.exp(0.5 * n(K, B, X)) + 0.05
        x = torch.poisson((0.5 + col % 5)[:, None].expand(B, X).contiguous(), generator=g)
    else:
        p = torch.sigmoid(2 * n(K, B, X)) if form == "probs" else torch.clamp(2 * n(K, B, X), -7, 7)
        u = torch.rand(B, X, generator=g, device="cuda")
        x = torch.where((col % 3 == 1)[:, None], u, (u < 0.5).float())  # every third column fractional (not binary)
    other = -55 + 5 * n(K, B) + 40 * (col % 4)
    logq = 30 + 4 * n(K, B) - 25 * (col % 3)
    return p.contiguous(), x.contiguous(), other.contiguous(), logq.contiguous()


def _launch(form, est, p, x, other, logq, **kw):
    B = x.shape[0]
    if form == "poisson":
        return be.iw_poisson_fused(est, p, x, other, logq, 1.0 / B, **kw)
    need = kw.pop("need_drate", True)
    return be.iw_bernoulli_fused(est, p, x, other, logq, 1.0 / B, need_dprobs=need, logits=form == "logits", **kw)


def _nan_out(K, B, X, need_grad=True):
    nan = lambda *s: torch.full(s, float("nan"), device="cuda")  # noqa: E731
    o = {"cost": nan(B), "dlogp": nan(K, B), "dlogq": nan(K, B), "logpx": nan(K, B)}
    if need_grad:
        o["dprobs"] = nan(K, B, X)
    return o


def _np(t):
    return t.detach().cpu().double().numpy()


def _oracle_step(oracle, form, est, p, x, other, logq):
    code = oracle.SGVB if est == be.SGVB else oracle.VIMCO
    args = (code, _np(p), _np(x), _np(other), _np(logq))
    if form == "poisson":
        return oracle.iw_poisson_step(*args, 1.0 / x.shape[0], need_drate=False)
    step = oracle.iw_bernoulli_logits_step if form == "logits" else oracle.iw_bernoulli_step
    return step(*args, need_dprobs=False)


def _oracle_bwd(oracle, form, g, p, x):
    K, B, X = p.shape
    if form == "poisson":
        return oracle.poisson_logpmf_bwd(g, _np(x), oracle.KBCAST, _np(p), oracle.FULL, K, B, X)
    if form == "logits":
        return oracle.bernoulli_logits_logpmf_bwd(g, _np(x), _np(p), K, B, X)
    return oracle.bernoulli_logpmf_bwd(g, _np(x), _np(p), K, B, X)


def _logpx_mag(form, p, x):
    """sum_x |sub-term| of log p(x | z) per (k, b), float64 (the Bernoulli terms are all <= 0: |log p| itself)."""
    p, x = p.double(), x.double()[None]
    if form == "poisson":
        return (torch.xlogy(x, p).abs() + p + torch.lgamma(x + 1)).sum(-1).cpu().numpy()
    q = torch.sigmoid(p) if form == "logits" else p
    return (x * torch.log(q + 1e-8) + (1 - x) * torch.log((1 - q) + 1e-8)).abs().sum(-1).cpu().numpy()


def _close(got, ref, scale, rtol, what):
    """|got - ref| <= rtol * scale elementwise (scale broadcast against ref)."""
    got = np.asarray(got, np.float64)
    tol = rtol * np.broadcast_to(scale, ref.shape) + 1e-30
    bad = ~(np.abs(got - ref) <= tol)
    if bad.any():
        i = np.unravel_index(np.argmax(bad), ref.shape)
        raise AssertionError("%s: %d of %d elements out of tolerance; first at %s: got %r want %r tol %r"
                             % (what, bad.sum(), bad.size, i, got[i], ref[i], tol[i]))


def _check_step(oracle, form, est, p, x, other, logq, r):
    K, B, X = p.shape
    o = _oracle_step(oracle, form, est, p, x, other, logq)
    mag = _logpx_mag(form, p, x)
    lpx = _np(r["logpx"])
    _close(lpx, o["logpx"], mag, 4e-6, "logpx")
    lw = o["logpx"] + _np(other) - _np(logq)
    col = np.abs(lw).max(0) + mag.max(0)  # the column's log-weight scale
    _close(_np(r["cost"]), o["cost"], col, 1e-5, "cost against the float64 step")
    # staged: the float64 objective of the kernel's own log p(x | z)
    code = oracle.SGVB if est == be.SGVB else oracle.VIMCO
    oc, olp, olq = oracle.iw_objective(code, lpx + _np(other), _np(logq), 1.0 / B)
    _close(_np(r["cost"]), oc, col, 1e-5, "cost")
    _close(_np(r["dlogp"]), olp, np.abs(olp).max(0), 1e-5, "dlogp")
    _close(_np(r["dlogq"]), olq, np.abs(olq).max(0), 1e-5, "dlogq")
    odp = _oracle_bwd(oracle, form, olp, p, x)
    _close(_np(r["dprobs"]), odp, np.abs(odp).max(-1, keepdims=True), 1e-5, "dprobs")


@pytest.mark.parametrize("est,K", CASES, ids=["%s-K%d" % c for c in CASES])
@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("X", XS)
def test_box_many_columns_per_cta(oracle, X, form, est, K):
    B = _B()
    code = be.SGVB if est == "sgvb" else be.VIMCO
    while not be.fused_poisson_supported(K, X, torch.float32):  # X = 1024 fits K <= 39: 38 keeps two rows per warp
        K -= 2
    p, x, other, logq = _inputs(form, K, B, X, seed=X + K)
    r = _launch(form, code, p, x, other, logq, want_logpx=True, out=_nan_out(K, B, X))
    assert r is not None
    _check_step(oracle, form, code, p, x, other, logq, r)


@pytest.mark.parametrize("X", [128, 784])
@pytest.mark.parametrize("est", [be.SGVB, be.VIMCO], ids=["sgvb", "vimco"])
def test_poisson_flags_leave_other_outputs_unchanged(X, est):
    """ZS_FUSED_ACCUMULATE_COST, ZS_FUSED_COST_SCALED, the in-launch loss, the forward-only launch and absent
    logp_other / logq, at B = 4 G + 3: each changes only what it is meant to change."""
    K, B = 50, _B()
    p, x, other, logq = _inputs("poisson", K, B, X, seed=7)
    base = _launch("poisson", est, p, x, other, logq, want_logpx=True, out=_nan_out(K, B, X))
    same = lambda r, keys: all(torch.equal(r[k], base[k]) for k in keys)  # noqa: E731
    acc = torch.zeros(B, device="cuda")
    for _ in range(3):
        o = _nan_out(K, B, X)
        o["cost"] = acc
        r = _launch("poisson", est, p, x, other, logq, want_logpx=True, out=o, accumulate_cost=True)
        assert same(r, ("dprobs", "dlogp", "dlogq", "logpx"))
    torch.testing.assert_close(acc, 3 * base["cost"], rtol=1e-6, atol=0)
    r = _launch("poisson", est, p, x, other, logq, want_logpx=True, out=_nan_out(K, B, X), cost_scaled=True)
    assert same(r, ("dprobs", "dlogp", "dlogq", "logpx"))
    torch.testing.assert_close(r["cost"], base["cost"] * (1.0 / B), rtol=1e-6, atol=0)
    seen = []
    for _ in range(4):
        r = _launch("poisson", est, p, x, other, logq, want_logpx=True, out=_nan_out(K, B, X), want_loss=True)
        assert r["loss"] is not None and same(r, ("cost", "dprobs", "dlogp", "dlogq", "logpx"))
        want = _np(r["cost"]).sum()
        assert abs(float(r["loss"]) - want) <= 1.5e-7 * abs(want), (float(r["loss"]), want)
        seen.append(float(r["loss"]))
    assert len(set(seen)) == 1
    r = _launch("poisson", est, p, x, other, logq, want_logpx=True, out=_nan_out(K, B, X, need_grad=False),
                need_drate=False)
    assert r["dprobs"] is None and same(r, ("cost", "dlogp", "dlogq", "logpx"))
    if est == be.SGVB:
        zero = torch.zeros_like(other)
        z = _launch("poisson", est, p, x, zero, zero, want_logpx=True, out=_nan_out(K, B, X))
        r = _launch("poisson", est, p, x, None, None, want_logpx=True, out=_nan_out(K, B, X))
        assert all(torch.equal(r[k], z[k]) for k in ("cost", "dprobs", "dlogp", "dlogq", "logpx"))


def _two_pass(est, p, x, other, logq):
    """The route the public API takes without the fused kernel: log-pmf rows -> IW objective -> rate gradient."""
    K, B, X = p.shape
    lpx = be.poisson_logpmf_fwd(x, be.KBCAST, p, be.FULL, K, B, X)
    cost, dlp, dlq = be.iw_objective(est, lpx, logq, 1.0 / B, extra=other)
    drate = be.poisson_logpmf_bwd(dlp, x, be.KBCAST, p, be.FULL, K, B, X)
    return dict(cost=cost, dprobs=drate, dlogp=dlp, dlogq=dlq, logpx=lpx)


@pytest.mark.parametrize("X", [128, 784])
def test_poisson_edge_values(oracle, X):
    """Counts >= 32 (lgammaf rather than the table) and non-integer counts; rate = 0 where x = 0 (contributes 0); one
    particle with rate = 0 where x > 0 (log-weight -inf, weight 0; the reference's surrogate cost of that column is
    0 * -inf = NaN, on both routes); subnormal rates with
    x > 0 in every particle of a column (finite x log r, as torch and the two-pass route give).  Fused against the
    two-pass route and float64 torch.  At rate = 0, x = 0 d/drate is g (0/0 - 1) = NaN in torch: both routes give NaN.
    """
    K, B = 50, _B()
    est = be.SGVB
    p, x, other, logq = _inputs("poisson", K, B, X, seed=11)
    x[0::7] += 40.0                 # counts >= 32
    x[1::7] += 0.5                  # non-integer counts
    x[2::7, 5] = 0.0
    p[:, 2::7, 5] = 0.0             # rate = 0 where x = 0
    x[3::7, 9] = 4.0
    p[3, 3::7, 9] = 0.0             # particle 3: rate = 0 < x
    x[4::7, 17] = 2.0
    p[:, 4::7, 17] = 1e-40          # subnormal rates, x > 0, every particle of the column
    assert (p[:, 4::7, 17] > 0).all()
    fz = _launch("poisson", est, p, x, other, logq, want_logpx=True, out=_nan_out(K, B, X))
    tp = _two_pass(est, p, x, other, logq)

    lpx64 = torch.distributions.Poisson(p.double(), validate_args=False).log_prob(x.double()[None]).sum(-1)
    lpx64 = lpx64.cpu().numpy()
    fin = np.isfinite(lpx64)
    assert (~fin).sum() == len(range(3, B, 7)) and np.all(lpx64[3, 3::7] == -np.inf)
    mag = _logpx_mag("poisson", p, x)
    for r, name in ((fz, "fused"), (tp, "two-pass")):
        lpx = _np(r["logpx"])
        assert np.array_equal(lpx[~fin], lpx64[~fin]), name
        _close(lpx[fin], lpx64[fin], mag[fin], 4e-6, name + " logpx")
        assert np.all(_np(r["dlogp"])[3, 3::7] == 0), name  # weight 0
        d = _np(r["dprobs"])
        assert np.all(d[3, 3::7, 9] != d[3, 3::7, 9]) and np.all(d[:, 2::7, 5] != d[:, 2::7, 5]), name  # NaN
    # the reference's SGVB surrogate -sum_k w_k log w_k is NaN (0 * -inf) in a column with a -inf log-weight, and
    # finite in every other column
    lw64 = lpx64 + _np(other) - _np(logq)
    with np.errstate(invalid="ignore"):
        w64 = np.exp(lw64 - lw64.max(0))
        w64 /= w64.sum(0)
        cost64 = -(w64 * lw64).sum(0)
    assert np.array_equal(np.isnan(cost64), np.isin(np.arange(B) % 7, [3]))
    _, dlp64, _ = oracle.iw_objective(oracle.SGVB, np.where(fin, lpx64, -1e30) + _np(other), _np(logq), 1.0 / B)
    col = np.abs(np.where(fin, lw64, 0)).max(0) + mag.max(0)
    for r, name in ((fz, "fused"), (tp, "two-pass")):
        c = _np(r["cost"])
        assert np.array_equal(np.isnan(c), np.isnan(cost64)), name
        ok = ~np.isnan(cost64)
        _close(c[ok], cost64[ok], col[ok], 1e-5, name + " cost against float64 torch")
    # at r = 1e-40 < x, 1 / r overflows float32 on both routes: d/drate is g inf, NaN where the weight is 0
    a, b = _np(fz["dprobs"]), _np(tp["dprobs"])
    assert not np.isfinite(a[:, 4::7, 17]).any() and not np.isfinite(b[:, 4::7, 17]).any()
    # the same non-finite pattern as the two-pass route, and close to it elsewhere
    assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[np.isinf(b)], b[np.isinf(b)])
    ok = np.isfinite(b)
    # scale: the column's largest gradient (a particle of weight 1e-20 carries the float32 log-weight noise of both
    # routes, ~1e-2 relative at these |log w| of several thousand)
    colmax = np.abs(np.where(ok, b, 0)).max(axis=(0, 2))[None, :, None]
    _close(a[ok], b[ok], np.broadcast_to(colmax, b.shape)[ok], 1e-3, "drate against two-pass")
    _close(_np(fz["dlogp"]), dlp64, np.abs(dlp64).max(0), 1e-3, "dlogp against float64 torch")
