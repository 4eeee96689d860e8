"""Every dispatch path of the log-density row kernels (zs_nodes.cu: dispatch_rows_fwd, dispatch_bwd) for all seven ops,
against float64 torch, row by row and element by element.

The kernel and its lane count are chosen from E, the row count against the SM count, operand alignment and the layout
modes.  The shapes below select each of them (computed from the device's SM count), and test_dispatch_selects_each_path
checks under torch.profiler that they still do.  Outputs are NaN-filled before every launch, so an element a kernel
fails to write cannot pass by holding an earlier call's answer.

Tolerances, per row of the forward and per element of every gradient, where `mag` is the sum of the absolute values of
the op's additive sub-terms (for a KBCAST gradient: of every particle's contribution, sum_k |.|):
  float64: 1e-12 * mag;
  float32: max(2 |ref32 - ref64|, C * 2^-24 * mag) with C per op (C_F32), ref32 being torch's own float32
  evaluation (DESIGN.md §4: no farther from float64 than float32 torch is).
Non-finite reference values (-inf rows, inf / NaN gradients) must be matched exactly.
"""
import re
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = [pytest.mark.gpu, pytest.mark.skipif(not torch.cuda.is_available(), reason="needs a CUDA device")]

from zhusuan import _backend as be  # noqa: E402

DEV = "cuda"
FULL, KBCAST, SCALAR = be.FULL, be.KBCAST, be.SCALAR
# C_F32 per op: the largest float32 error measured over this file on a B200 (1000 W power limit), in units of
# 2^-24 * mag where 2 |ref32 - ref64| does not already cover it, with a margin of 2.5-3.  Normal 4.7; Bernoulli 43 (a
# one-element row: the SFU log2's absolute error of 2^-22 against a term near 0); Bernoulli-logits 1673 (the SFU
# sigmoid is a few ulp of p, which 1 - p amplifies near |l| = 7); the other four ops pass at 32.
C_F32 = {"bernoulli": 128, "logits": 4096}
C_F32_DEFAULT = 32
OPS = ["normal", "bernoulli", "logits", "logistic", "laplace", "uniform", "poisson"]
TWO_PARAM = ("normal", "logistic", "laplace", "uniform")
FAM = {"logistic": be.FAM_LOGISTIC, "laplace": be.FAM_LAPLACE, "uniform": be.FAM_UNIFORM}
DTYPES = [torch.float32, torch.float64]
# operand modes (x, a, b): every parameter FULL, the latent shape, the likelihood shape, a SCALAR second parameter
MODES = {"full": (FULL, FULL, FULL), "latent": (FULL, KBCAST, KBCAST), "likelihood": (KBCAST, FULL, FULL),
         "scalar_b": (FULL, FULL, SCALAR)}
ROWC, SPLIT_MAX = 8, 256  # CTAs per row of k_rows_fwd_cluster; most virtual rows of the split backward


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _vn(dtype):
    return 4 if dtype == torch.float32 else 2


def _few_rows(K, M, E):
    return E >= 2048 and K * M * 32 < _sms() * 1024


def _split(K, M, E, dtype):
    """dispatch_bwd's cut of a long row into S virtual rows."""
    S, vn = 1, _vn(dtype)
    while S < SPLIT_MAX and E % (2 * S * vn) == 0 and E // (2 * S) >= 1024 and K * M * S * 32 < _sms() * 2048:
        S *= 2
    return S


def _shape(path, i):
    """(K, M, E) of the i-th case of `path`; None where this device cannot select the path."""
    G = _sms()
    if path == "lpr1":
        return [(7, 300, 1), (5, 130, 2)][i]
    if path == "lpr8":
        return [(9, 70, 3), (4, 33, 48)][i]
    if path == "lpr32":
        return [(50, 64, 784), (3, 40, 52), (50, 64, 785)][i]
    if path == "cluster":
        if i < 2:
            return [(3, 2, 8192), (3, 2, 8195)][i]
        M = min(60, (32 * G - 1) // 50)  # more rows than the 2048 a launch keeps in flight: the row loop runs twice
        return (50, M, 2048) if 50 * M > 2048 else None
    if path == "split":
        return [(2, 1, 8192), (3, 2, 16384)][i]
    if path == "lanes256":
        return (3, 2, 4601)
    raise AssertionError(path)


PATH_CASES = [("lpr1", 0), ("lpr1", 1), ("lpr8", 0), ("lpr8", 1), ("lpr32", 0), ("lpr32", 1), ("lpr32", 2),
              ("cluster", 0), ("cluster", 1), ("cluster", 2), ("split", 0), ("split", 1), ("lanes256", 0)]


# ----------------------------------------------------------------------------- inputs
def _seed(*key):
    return zlib.crc32(repr(key).encode()) % 10000


def _draw(op, role, shape, rng):
    if role == "x":
        if op in ("bernoulli", "logits"):
            return (rng.uniform(size=shape) < 0.5).astype(np.float64)
        if op == "uniform":
            return rng.uniform(-0.9, 0.9, size=shape)
        if op == "poisson":
            return rng.poisson(2.0, size=shape).astype(np.float64)
        return 1.5 * rng.standard_normal(shape)
    if role == "a":
        if op == "bernoulli":
            return rng.uniform(0.02, 0.98, size=shape)
        if op == "logits":
            return np.clip(2.0 * rng.standard_normal(shape), -7.0, 7.0)
        if op == "uniform":
            return -1.0 - rng.uniform(size=shape)
        if op == "poisson":
            return rng.gamma(2.0, 1.0, size=shape) + 0.05
        return rng.standard_normal(shape)
    if op == "uniform":
        return 1.0 + rng.uniform(size=shape)
    return np.exp(0.3 * rng.standard_normal(shape))


def _op_shape(mode, K, M, E):
    return {FULL: (K, M, E), KBCAST: (M, E), SCALAR: (1,)}[mode]


def _put(arr, mode, k, m, e, v):
    if mode == FULL:
        arr[k, m, e] = v
    elif mode == KBCAST:
        arr[m, e] = v
    return mode != SCALAR


def _get(arr, mode, k, m, e):
    return arr[k, m, e] if mode == FULL else (arr[m, e] if mode == KBCAST else arr[0])


def _positions(K, M, E, dtype):
    """Where a path bug lands: the last element, the cluster CTAs' segment boundaries and the S-slice boundaries."""
    vn = _vn(dtype)
    per = -(-E // (ROWC * vn)) * vn
    pos = {E - 1}
    for j in range(1, ROWC):
        pos |= {per * j - 1, per * j}
    S = _split(K, M, E, dtype) if E >= 2048 else 1
    for j in range(1, S):
        pos |= {j * E // S - 1, j * E // S}
    return sorted(p for p in pos if 0 <= p < E)


def _sentinels(op, arrs, modes, K, M, E, dtype):
    """Values that cannot be confused, in every third row only (the other rows keep finite values to compare): the
    finite kinds at every boundary position of the row, one -inf kind at one position (rotating over the rows)."""
    x, a, b = arrs
    xm, am, bm = modes
    pos = _positions(K, M, E, dtype)
    rows = [r for r in range(K * M) if r % 3 == 1] or [K * M - 1]
    for i, r in enumerate(rows):
        k, m = divmod(r, M)
        for j, e in enumerate(pos):
            if op == "bernoulli":
                _put(a, am, k, m, e, float(j % 2))  # p in {0, 1}
            elif op == "logistic":  # |z| > 20 on both sides
                if not _put(x, xm, k, m, e, 1e3 if j % 2 else -1e3):
                    _put(a, am, k, m, e, -1e3 if j % 2 else 1e3)
            elif op == "laplace":  # x == loc: zero gradient in x and loc
                if am == FULL:
                    _put(a, am, k, m, e, _get(x, xm, k, m, e))
                else:
                    _put(x, xm, k, m, e, _get(a, am, k, m, e))
            elif op == "poisson" and am != SCALAR:  # rate = 0 where x = 0: contributes 0
                _put(a, am, k, m, e, 0.0)
                if am == KBCAST and xm == FULL:
                    x[:, m, e] = 0.0
                else:
                    _put(x, xm, k, m, e, 0.0)
        e = pos[i % len(pos)]
        if op == "uniform":  # outside the support: -inf
            _put(x, xm, k, m, e, 5.0)
        elif op == "poisson" and am != SCALAR:  # rate = 0 < x: -inf
            _put(a, am, k, m, e, 0.0)
            if am == KBCAST and xm == FULL:
                x[:, m, e] = 3.0
            else:
                _put(x, xm, k, m, e, 3.0)


def _inputs(op, modes, K, M, E, dtype, seed, sentinels=True):
    rng = np.random.RandomState(seed)
    roles = ("x", "a", "b") if op in TWO_PARAM else ("x", "a")
    arrs = [_draw(op, role, _op_shape(mode, K, M, E), rng) for role, mode in zip(roles, modes)]
    if len(arrs) == 2:
        arrs.append(None)
    if sentinels:
        _sentinels(op, arrs, modes, K, M, E, dtype)
    # the float64 reference sees exactly the values the kernel sees
    return [None if v is None else torch.tensor(v, dtype=dtype).double() for v in arrs]


def _device(t, dtype, misalign):
    """On the GPU in `dtype`; `misalign`: a contiguous slice one element into its storage (not 16-byte aligned), which
    keeps the vectorised kernels away."""
    if t is None:
        return None
    if not misalign:
        return t.to(dtype).to(DEV).contiguous()
    buf = torch.empty(t.numel() + 1, dtype=dtype, device=DEV)
    buf[1:] = t.reshape(-1).to(dtype)
    v = buf[1:].view(t.shape)
    assert v.is_contiguous() and v.data_ptr() % 16 != 0
    return v


# ----------------------------------------------------------------------------- kernels through the C ABI
def _nan(shape, dtype):
    return torch.full(shape, float("nan"), dtype=dtype, device=DEV)


def _fwd(op, x, xm, a, am, b, bm, K, M, E):
    P, dc, d = be._ptr, be.dtype_code(x.dtype), x.device
    out = _nan((K, M), x.dtype)
    if op == "normal":
        be._go("zs_normal_logprob_fwd", d, dc, P(out), P(x), xm, P(a), am, P(b), bm, K, M, E)
    elif op in ("bernoulli", "logits"):
        name = "zs_bernoulli_logits_logpmf_fwd" if op == "logits" else "zs_bernoulli_logpmf_fwd"
        be._go(name, d, dc, P(out), P(x), xm, P(a), am, K, M, E)
    elif op == "poisson":
        be._go("zs_poisson_logpmf_fwd", d, dc, P(out), P(x), xm, P(a), am, K, M, E)
    else:
        be._go("zs_locscale_logprob_fwd", d, dc, FAM[op], P(out), P(x), xm, P(a), am, P(b), bm, K, M, E)
    return out


def _bwd(op, g, x, xm, a, am, b, bm, K, M, E, want):
    """Gradients named in `want` (subset of "xab"), NaN-filled before the launch."""
    P, dc, d = be._ptr, be.dtype_code(x.dtype), x.device
    dx, da, db = (_nan(t.shape, t.dtype) if n in want else None
                  for n, t in (("x", x), ("a", a), ("b", b if b is not None else a)))
    if op == "normal":
        be._go("zs_normal_logprob_bwd", d, dc, P(dx), P(da), P(db), P(g), P(x), xm, P(a), am, P(b), bm, K, M, E)
    elif op in ("bernoulli", "logits"):
        name = "zs_bernoulli_logits_logpmf_bwd" if op == "logits" else "zs_bernoulli_logpmf_bwd"
        be._go(name, d, dc, P(dx), P(da), P(g), P(x), xm, P(a), am, K, M, E)
    elif op == "poisson":
        be._go("zs_poisson_logpmf_bwd", d, dc, P(da), P(g), P(x), xm, P(a), am, K, M, E)
    else:
        be._go("zs_locscale_logprob_bwd", d, dc, FAM[op], P(dx), P(da), P(db), P(g), P(x), xm, P(a), am, P(b), bm,
               K, M, E)
    return {"x": dx, "a": da, "b": db}


# ----------------------------------------------------------------------------- float64 references
def _terms(op, x, a, b):
    """The op's log-density as additive sub-terms (their absolute values set the tolerance scale)."""
    if op == "normal":
        logstd = torch.log(b)
        c = torch.full_like(x * a, -0.9189385332046727)  # normal.py:122, rounded to the operand dtype
        return [c, -logstd, -(0.5 * torch.exp(-2 * logstd)) * (x - a) ** 2]
    if op in ("bernoulli", "logits"):
        p = torch.sigmoid(a) if op == "logits" else a
        return [x * torch.log(p + 1e-8), (1 - x) * torch.log((1 - p) + 1e-8)]
    if op == "logistic":
        z = (x - a) / b
        return [-z, -2 * F.softplus(-z), -torch.log(b)]
    if op == "laplace":
        return [-torch.log(2 * b), -torch.abs(x - a) / b]
    if op == "uniform":
        return [-torch.log(b - a)]
    return [torch.xlogy(x, a), -a, -torch.lgamma(x + 1)]


def _logp(op, x, a, b):
    """The reference's log-density, elementwise: the formula as the reference writes it, or torch.distributions where
    the reference delegates to it."""
    D = torch.distributions
    if op == "laplace":
        return D.Laplace(a, b, validate_args=False).log_prob(x)
    if op == "uniform":
        return D.Uniform(a, b, validate_args=False).log_prob(x)
    if op == "poisson":
        return D.Poisson(a, validate_args=False).log_prob(x)
    return sum(_terms(op, x, a, b))


def _reference(op, ops, modes, g, want, dtype, K, M, E):
    """In `dtype` (torch's own evaluation): the row sums [K, M] and the gradients of sum(g * rows) w.r.t. the operands
    in `want`, reduced to the operand's shape (summed over K for KBCAST); plus, in float64, their magnitudes."""
    full = [None if t is None else t.to(DEV, dtype).expand(K, M, E).clone().requires_grad_() for t in ops]
    lp = _logp(op, *full)
    rows = lp.sum(-1)
    gd = g.to(DEV, dtype)
    leaves = {n: full[i] for i, n in enumerate("xab") if n in want}
    grads = {}
    if leaves:  # an operand the op ignores (Uniform's x) has a zero gradient
        gs = torch.autograd.grad((rows * gd).sum(), list(leaves.values()), allow_unused=True)
        grads = {n: torch.zeros_like(leaves[n]) if t is None else t for n, t in zip(leaves, gs)}
    red = lambda n, t: t.sum(0) if modes["xab".index(n)] == KBCAST else t  # noqa: E731
    out = {"rows": rows.detach(), **{n: red(n, t) for n, t in grads.items()}}
    if dtype != torch.float64:
        return out
    terms = _terms(op, *full)
    out["rows_mag"] = sum(t.detach().abs() for t in terms).nan_to_num(0.0, 0.0, 0.0).sum(-1)
    for n, leaf in leaves.items():
        mag = torch.zeros_like(leaf)
        for t in terms:
            if t.requires_grad:
                (gt,) = torch.autograd.grad((t * gd[..., None]).sum(), [leaf], retain_graph=True, allow_unused=True)
                if gt is not None:
                    mag += gt.abs().nan_to_num(0.0, 0.0, 0.0)
        out[n + "_mag"] = red(n, mag)
    return out


def _check(got, ref64, ref32, mag, dtype, what, c32=C_F32_DEFAULT):
    got, ref64, mag = (t.detach().to(DEV, torch.float64) for t in (got, ref64, mag))
    fin = torch.isfinite(ref64)
    assert torch.equal(torch.isnan(got), torch.isnan(ref64)), "%s: NaN pattern" % what
    assert torch.equal(got[~fin & ~torch.isnan(ref64)], ref64[~fin & ~torch.isnan(ref64)]), "%s: inf pattern" % what
    assert torch.isfinite(got[fin]).all(), "%s: non-finite where the reference is finite" % what
    err = (got - ref64).abs()[fin]
    if dtype == torch.float64:
        tol = 1e-12 * mag[fin]
    else:
        d32 = (ref32.detach().to(DEV, torch.float64) - ref64).abs().nan_to_num(0.0, 0.0, 0.0)[fin]
        tol = torch.maximum(2 * d32, c32 * 2.0 ** -24 * mag[fin])
    bad = err > tol
    if bad.any():
        i = int(torch.nonzero(bad)[0])
        raise AssertionError("%s: %d of %d elements out of tolerance; first: got %r want %r tol %r"
                             % (what, int(bad.sum()), bad.numel(), float(got[fin][i]), float(ref64[fin][i]),
                                float(tol[i])))


def _grad_sets(op, modes):
    """Gradient requests: every operand that has one, then (when that mixes KBCAST and FULL operands, which sends the
    whole call to k_kreduce_bwd) the FULL ones alone, which take the row backward."""
    names = [n for n, md in zip("xab", modes) if md != SCALAR and (n != "b" or op in TWO_PARAM)]
    if op == "poisson":
        names = [n for n in names if n == "a"]  # the count carries no gradient
    sets = [names] if names else []
    full_only = [n for n in names if modes["xab".index(n)] == FULL]
    if full_only and full_only != names:
        sets.append(full_only)
    return sets


def _run_case(op, dtype, mode_name, K, M, E, misalign=False, seed=0, sentinels=True):
    modes = MODES[mode_name]
    ops = _inputs(op, modes, K, M, E, dtype, seed, sentinels)
    dev = [None if t is None else _device(t, dtype, misalign and i == 0) for i, t in enumerate(ops)]
    xm, am, bm = modes
    if op not in TWO_PARAM:
        bm = SCALAR
    tag = "%s %s %s K=%d M=%d E=%d%s" % (op, dtype, mode_name, K, M, E, " misaligned" if misalign else "")
    g = torch.tensor(np.random.RandomState(seed + 1).standard_normal((K, M)), dtype=dtype)
    got = _fwd(op, dev[0], xm, dev[1], am, dev[2], bm, K, M, E)
    sets = _grad_sets(op, modes)
    want_all = set().union(*sets) if sets else set()
    r64 = _reference(op, ops, modes, g.double(), want_all, torch.float64, K, M, E)
    r32 = _reference(op, ops, modes, g, want_all, torch.float32, K, M, E) if dtype == torch.float32 else r64
    c32 = C_F32.get(op, C_F32_DEFAULT)
    _check(got, r64["rows"], r32["rows"], r64["rows_mag"], dtype, tag + " fwd", c32)
    for want in sets:
        gr = _bwd(op, g.to(DEV), dev[0], xm, dev[1], am, dev[2], bm, K, M, E, want)
        for n in want:
            _check(gr[n], r64[n], r32[n], r64[n + "_mag"], dtype, "%s d%s (requested %s)" % (tag, n, "".join(want)),
                   c32)
    return dev, got


# ----------------------------------------------------------------------------- tests
@pytest.mark.parametrize("path,i", PATH_CASES, ids=["%s-%d" % c for c in PATH_CASES])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("op", OPS)
def test_row_paths(op, dtype, path, i):
    """Each op on each forward / backward path, in every layout mode; aligned shapes also with a misaligned operand
    (the scalar variants of the same path)."""
    shape = _shape(path, i)
    if shape is None:
        pytest.skip("too few SMs for more rows than a cluster launch keeps in flight")
    K, M, E = shape
    for mode_name in MODES:
        if mode_name == "scalar_b" and op not in TWO_PARAM:
            continue
        _run_case(op, dtype, mode_name, K, M, E, seed=_seed(op, path, i, mode_name))
        if E % _vn(dtype) == 0 and E > 48:
            _run_case(op, dtype, mode_name, K, M, E, misalign=True, seed=_seed(op, path, i, mode_name) + 7)


KREDUCE_KS = [1, 7, 8, 9, 100]
KREDUCE_ME = [(1, 31), (3, 11), (5, 2048)]  # M * E = 31, 33, 10240


@pytest.mark.parametrize("K", KREDUCE_KS)
@pytest.mark.parametrize("M,E", KREDUCE_ME)
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("op", OPS)
def test_kreduce_paths(op, dtype, K, M, E):
    """k_kreduce_bwd: gradients of KBCAST operands summed over K in 8 particle slices of a 32-element block; K around
    and far above the slice count, M * E around the block width."""
    for mode_name in ("latent", "likelihood"):
        _run_case(op, dtype, mode_name, K, M, E, seed=K * 31 + E)


@pytest.mark.parametrize("E", [50, 785, 2050, 8195])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
@pytest.mark.parametrize("op", OPS)
def test_all_scalar_forward(op, dtype, E):
    """Every operand SCALAR (allowed by zs_b200.h for every operand) with E not a multiple of the pack width: each row
    is E times the same term, whichever kernel runs (LPR 32 at E < 2048, the cluster kernel at E >= 2048)."""
    K, M = 3, 2
    vals = {"normal": (0.7, -0.2, 1.3), "bernoulli": (1.0, 0.3, None), "logits": (0.0, 1.5, None),
            "logistic": (0.4, 0.1, 0.8), "laplace": (0.4, 0.1, 0.8), "uniform": (0.2, -1.0, 1.5),
            "poisson": (2.0, 3.5, None)}[op]
    ops = [None if v is None else torch.tensor([v], dtype=dtype) for v in vals]
    dev = [None if t is None else t.to(DEV) for t in ops]
    got = _fwd(op, dev[0], SCALAR, dev[1], SCALAR, dev[2], SCALAR, K, M, E)
    full = [None if t is None else t.double().expand(K, M, E) for t in ops]
    ref64 = _logp(op, *full).sum(-1)
    ref32 = _logp(op, *[None if t is None else t.expand(K, M, E) for t in ops]).sum(-1)
    mag = sum(t.abs() for t in _terms(op, *full)).sum(-1)
    _check(got, ref64, ref32, mag, dtype, "%s all-SCALAR E=%d" % (op, E), C_F32.get(op, C_F32_DEFAULT))


@pytest.mark.parametrize("path,i", PATH_CASES, ids=["%s-%d" % c for c in PATH_CASES])
@pytest.mark.parametrize("dtype", DTYPES, ids=["f32", "f64"])
def test_normal_scalar_std_bit_identical(dtype, path, i):
    """ScalarB<NormalOp> hoists log(std), exp(-2 log std) out of the element loop with the same expressions in the same
    order: a SCALAR std gives bit-identical log-densities and x / mean gradients to the same std expanded to FULL."""
    shape = _shape(path, i)
    if shape is None:
        pytest.skip("too few SMs for more rows than a cluster launch keeps in flight")
    K, M, E = shape
    x, mean, std = _inputs("normal", MODES["scalar_b"], K, M, E, dtype, seed=5)
    x, mean, std = x.to(dtype).to(DEV), mean.to(dtype).to(DEV), std.to(dtype).to(DEV)
    std_full = std.expand(K, M, E).contiguous()
    g = torch.randn(K, M, dtype=dtype, device=DEV)
    a = _fwd("normal", x, FULL, mean, FULL, std, SCALAR, K, M, E)
    b = _fwd("normal", x, FULL, mean, FULL, std_full, FULL, K, M, E)
    assert torch.equal(a, b)
    ga = _bwd("normal", g, x, FULL, mean, FULL, std, SCALAR, K, M, E, "xa")
    gb = _bwd("normal", g, x, FULL, mean, FULL, std_full, FULL, K, M, E, "xa")
    assert torch.equal(ga["x"], gb["x"]) and torch.equal(ga["a"], gb["a"])
    # the latent shape: mean KBCAST, so the mean gradient goes through k_kreduce_bwd
    mk = mean[0].contiguous()
    ga = _bwd("normal", g, x, FULL, mk, KBCAST, std, SCALAR, K, M, E, "xa")
    gb = _bwd("normal", g, x, FULL, mk, KBCAST, std_full, FULL, K, M, E, "xa")
    assert torch.equal(ga["x"], gb["x"]) and torch.equal(ga["a"], gb["a"])


# (path, dtype, misalign, fwd kernel pattern, bwd kernel pattern); the backward requests the gradient of the FULL mean
DISPATCH = [
    ("lpr1", 0, torch.float32, False, r"k_rows_fwd<float, zs::NormalOp<float>, 1, false>",
     r"k_rows_bwd<float, zs::NormalOp<float>, 1, false>"),
    ("lpr8", 1, torch.float64, False, r"k_rows_fwd<double, zs::NormalOp<double>, 8, false>",
     r"k_rows_bwd<double, zs::NormalOp<double>, 8, false>"),
    ("lpr32", 0, torch.float32, False, r"k_rows_fwd<float, zs::NormalOp<float>, 32, true>",
     r"k_rows_bwd<float, zs::NormalOp<float>, 32, true>"),
    ("lpr32", 0, torch.float32, True, r"k_rows_fwd<float, zs::NormalOp<float>, 32, false>",
     r"k_rows_bwd<float, zs::NormalOp<float>, 32, false>"),
    ("lpr32", 2, torch.float64, False, r"k_rows_fwd<double, zs::NormalOp<double>, 32, false>",
     r"k_rows_bwd<double, zs::NormalOp<double>, 32, false>"),
    ("cluster", 0, torch.float32, False, r"k_rows_fwd_cluster<float, zs::NormalOp<float>, true>",
     r"k_rows_bwd<float, zs::NormalOp<float>, 32, true>"),
    ("cluster", 1, torch.float32, False, r"k_rows_fwd_cluster<float, zs::NormalOp<float>, false>",
     r"k_rows_bwd<float, zs::NormalOp<float>, 256, false>"),
    ("split", 0, torch.float64, False, r"k_rows_fwd_cluster<double, zs::NormalOp<double>, true>",
     r"k_rows_bwd<double, zs::NormalOp<double>, 32, true>"),
    ("lanes256", 0, torch.float32, False, r"k_rows_fwd_cluster<float, zs::NormalOp<float>, false>",
     r"k_rows_bwd<float, zs::NormalOp<float>, 256, false>"),
]


def test_dispatch_selects_each_path():
    """The shapes above select the kernels they are meant to: the launched kernel's name carries the expected
    template arguments (cluster or not, lanes per row, vectorised or not; k_kreduce_bwd for a KBCAST gradient)."""
    from torch.profiler import ProfilerActivity, profile

    def launched(fn):
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return [e.name for e in prof.events() if "zs::" in e.name]

    for path, i, dtype, misalign, fwd_pat, bwd_pat in DISPATCH:
        K, M, E = _shape(path, i)
        x, mean, std = (_device(t, dtype, misalign and j == 0) for j, t in
                        enumerate(_inputs("normal", MODES["full"], K, M, E, dtype, seed=3)))
        g = torch.randn(K, M, dtype=dtype, device=DEV)
        names = launched(lambda: _fwd("normal", x, FULL, mean, FULL, std, FULL, K, M, E))
        assert len(names) == 1 and re.search(fwd_pat, names[0]), (path, i, names)
        names = launched(lambda: _bwd("normal", g, x, FULL, mean, FULL, std, FULL, K, M, E, "a"))
        assert len(names) == 1 and re.search(bwd_pat, names[0]), (path, i, names)
    if _shape("cluster", 2) is not None:
        K, M, E = _shape("cluster", 2)
        assert K * M > 2048 and _few_rows(K, M, E)
    assert _split(2, 1, 8192, torch.float32) == 8 and _split(3, 2, 16384, torch.float64) == 16
    assert _split(3, 2, 4601, torch.float32) == 1 and _few_rows(3, 2, 4601)
    K, M, E = 9, 1, 31
    x, mean, std = (t.float().to(DEV) for t in _inputs("normal", MODES["latent"], K, M, E, torch.float32, seed=4))
    g = torch.randn(K, M, device=DEV)
    names = launched(lambda: _bwd("normal", g, x, FULL, mean, KBCAST, std, KBCAST, K, M, E, "xab"))
    assert len(names) == 1 and re.search(r"k_kreduce_bwd<float, zs::NormalOp<float>\s*>", names[0]), names
