"""Host-side glue between the reference-shaped Python API and the C-ABI kernels.

Responsibilities (all host logic, no math):
  * view a broadcast problem as the [K, M, E] particle-row layout of include/zs_b200.h and classify
    every operand as FULL / KBCAST / SCALAR (what the reference does with `.repeat`, normal.py:94-95,
    115-116; bernoulli.py:75,90);
  * wrap each kernel pair in a torch.autograd.Function so the reference's autograd contract holds;
  * move CPU tensors to the current CUDA device and results back to the caller's device (the
    reference's tests feed CPU tensors); there is no CPU implementation to fall back to.
"""
import weakref

import torch
from ._shapes import broadcast_shapes as _bshapes

from . import _backend as be
from . import _rng
from ._lazy import LazyDraw, lazy_first_draws, lazy_active  # noqa: F401  (re-exported)

FULL, KBCAST, SCALAR = be.FULL, be.KBCAST, be.SCALAR


def _prod(xs):
    p = 1
    for v in xs:
        p *= int(v)
    return p


def compute_device():
    be.require_cuda()
    return torch.device("cuda", torch.cuda.current_device())


_upload_memo = [None]


class upload_memo(object):
    """Within this context a host tensor is uploaded once, however many nodes read it (an objective step reads the
    variational parameters three times: two draws, one log-density), and its gradient comes back with one copy."""

    def __enter__(self):
        self.owner = _upload_memo[0] is None
        if self.owner:
            _upload_memo[0] = {}
        return self

    def __exit__(self, *exc):
        if self.owner:
            _upload_memo[0] = None
        return False


def to_compute(t):
    """Differentiable move to the CUDA device the kernels run on.  A CPU tensor that this package
    itself produced (see back_home) still has its device original attached: reuse it instead of
    uploading the bytes again -- unless the CPU tensor takes part in autograd itself (a user may ask for the gradient
    w.r.t. it, or hook it): then the op must stay connected to the CPU tensor."""
    if isinstance(t, LazyDraw):
        dev_twin = getattr(t, "_zs_dev", None)
        if dev_twin is not None:  # a result this package parked on the device (lazy_host_results): no copy at all
            return dev_twin
        t = t._zs_materialize()
    if t.is_cuda:
        return t
    twin = getattr(t, "_zs_twin", None)
    if twin is not None and twin[1] == t._version and not t.requires_grad:
        return twin[0]
    memo = _upload_memo[0]
    if memo is None:
        return t.to(compute_device())
    key = (id(t), t._version)
    hit = memo.get(key)
    if hit is not None and hit[0] is t:
        return hit[1]
    d = t.to(compute_device())
    memo[key] = (t, d)  # holding `t` keeps its id unique for the life of the memo
    return d


# Pinned host buffers are slow to allocate (cudaHostAlloc of the 160 MB gradient takes tens of ms), so they are
# pooled.  A buffer is handed out again only when NOTHING else uses its storage: the pool's own tensor is then the
# storage's single owner (use count 2 = that tensor + the temporary storage handle of the query).  Views, detach()ed
# aliases, autograd's saved tensors and `.grad` attributes all hold the storage, so results a caller still looks at
# are never overwritten (a weak reference to the tensor object handed out does not see those aliases).
_pin_pool = {}


def _storage_in_use(buf):
    return torch._C._storage_Use_Count(buf.untyped_storage()._cdata) > 2


def pinned_like_pool(shape, dtype, key=None):
    shape = tuple(int(v) for v in shape)
    k = (key, shape, dtype)
    entries = _pin_pool.setdefault(k, [])
    for buf in entries:
        if not _storage_in_use(buf):
            return buf.view(shape)
    buf = torch.empty(shape, dtype=dtype, pin_memory=True)
    entries.append(buf)
    return buf.view(shape)


class _ToHostPinned(torch.autograd.Function):
    """Device -> host copy through pinned memory, ~10x the rate of a copy into pageable memory; the gradient goes
    back with a plain upload."""

    @staticmethod
    def forward(ctx, t):
        ctx.dev = t.device
        out = pinned_like_pool(t.shape, t.dtype)
        out.copy_(t, non_blocking=True)
        torch.cuda.current_stream(t.device).synchronize()
        return out

    @staticmethod
    def backward(ctx, g):
        return g.to(ctx.dev)


_keep_on_device = [0]

# data-parallel runs: the number of batch columns of the GLOBAL batch (zhusuan.distributed.global_batch), or None
_global_batch = [None]


def _mean_scale(B):
    """1 / (columns the mean objective averages over): the local batch, or the global batch of a data-parallel step
    (each rank then returns its additive share of the global mean and of its gradient)."""
    n = _global_batch[0]
    return 1.0 / float(n if n else B)


def _mean_cost(cost, B):
    n = _global_batch[0]
    return cost.mean() if not n else cost.sum() * (1.0 / float(n))


class device_results(object):
    """Inside this context ops return their results on the compute device instead of the caller's
    device.  The objectives use it for intermediate [K,B] log-probabilities that only they consume, so a
    host-resident model does not pay a device->host->device round trip (and two synchronisations) per node."""

    def __enter__(self):
        _keep_on_device[0] += 1
        return self

    def __exit__(self, *exc):
        _keep_on_device[0] -= 1
        return False


_lazy_host = [0]


class lazy_host_results(object):
    """Inside this context a LARGE result that belongs on the host (a latent sample of a host-resident model: 8 MB at
    config 2) is handed back as a LazyDraw standing for the host copy: the device->host transfer and its
    synchronisation happen only if host code actually touches the values (a CPU decoder does; a model whose only
    consumers are this package's nodes never does).  Ops of this package recognise the object and read the device
    original.  The objectives enter it for the duration of a step."""

    def __enter__(self):
        _lazy_host[0] += 1
        return self

    def __exit__(self, *exc):
        _lazy_host[0] -= 1
        return False


def back_home(t, home):
    """Return `t` on the caller's device; remember the device original for later ops."""
    if t.device == home or _keep_on_device[0]:
        return t
    big = home.type == "cpu" and t.is_cuda and t.numel() * t.element_size() >= (1 << 16)
    if big and _lazy_host[0] and not _rng.has_injected():
        lazy = LazyDraw(lambda self, t=t: _host_copy(t), t.shape, t.dtype, home)
        lazy._zs_dev = t
        return lazy
    if big:
        out = _ToHostPinned.apply(t)
    else:
        out = t.to(home)
    try:
        out._zs_twin = (t, out._version)
    except Exception:
        pass
    return out


def _host_copy(t):
    out = _ToHostPinned.apply(t)
    try:
        out._zs_twin = (t, out._version)
    except Exception:
        pass
    return out


# --------------------------------------------------------------------------------------------
# layout
# --------------------------------------------------------------------------------------------
class Layout(object):
    """[K, M, E] view of the broadcast of `shapes` with the last `n_event` axes summed."""

    def __init__(self, shapes, n_event):
        S = tuple(_bshapes(*shapes))
        if n_event > len(S):
            raise ValueError("cannot reduce %d event axes of a %d-d value" % (n_event, len(S)))
        self.S = S
        self.lead = S[:len(S) - n_event]
        self.E = _prod(S[len(S) - n_event:])
        self.k_axis = len(self.lead) > 0
        self.K = int(self.lead[0]) if self.k_axis else 1
        self.M = _prod(self.lead[1:]) if self.k_axis else 1

    def canon(self, t):
        """Return (contiguous tensor, mode) for an operand broadcastable to S.  Differentiable."""
        S = self.S
        if t.numel() == 1 and _prod(S) != 1 and not t.requires_grad:
            return t.reshape(1).contiguous(), SCALAR
        pad = (1,) * (len(S) - t.dim()) + tuple(t.shape)
        if pad == S:
            return t.contiguous(), FULL
        if self.k_axis and self.K > 1 and pad[0] == 1:
            # broadcast over particles; any further broadcasting inside a particle is materialised
            return t.reshape(pad[1:]).expand(S[1:]).contiguous(), KBCAST
        return t.expand(S).contiguous(), FULL


# --------------------------------------------------------------------------------------------
# Normal
# --------------------------------------------------------------------------------------------
class _NormalLogProb(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, mean, std, modes, K, M, E):
        out = be.normal_logprob_fwd(x, modes[0], mean, modes[1], std, modes[2], K, M, E)
        ctx.save_for_backward(x, mean, std)
        ctx.cfg = (modes, K, M, E)
        return out

    @staticmethod
    def backward(ctx, g):
        x, mean, std = ctx.saved_tensors
        modes, K, M, E = ctx.cfg
        nx, nm, ns = ctx.needs_input_grad[:3]
        dx, dmean, dstd = be.normal_logprob_bwd(g.contiguous(), x, modes[0], mean, modes[1], std, modes[2], K, M, E,
                                                nx, nm, ns)
        return dx, dmean, dstd, None, None, None, None


def normal_log_prob(x, mean, std, n_event):
    """sum over the last n_event axes of the Normal log-density (normal.py:109-126 + base.py:175-176)."""
    home = x.device
    x, mean, std = to_compute(x), to_compute(mean), to_compute(std)
    L = Layout([x.shape, mean.shape, std.shape], n_event)
    if _prod(L.S) == 0:
        return back_home(torch.zeros(L.lead, dtype=x.dtype, device=x.device), home)
    (xc, xm), (mc, mm), (sc, sm) = L.canon(x), L.canon(mean), L.canon(std)
    out = _NormalLogProb.apply(xc, mc, sc, (xm, mm, sm), L.K, L.M, L.E)
    return back_home(out.reshape(L.lead), home)


def _draw_kwargs(dev, injected, want_snapshot=False):
    """(kwargs of the sampling launch, kwargs of a backward that regenerates its noise)."""
    if injected is not None:
        return dict(seed=0, offset=0), dict(seed=0, offset=0)
    kw = _rng.draw_args(dev)
    if kw.get("rng_state") is None:
        return kw, dict(seed=kw["seed"], offset=kw["offset"])
    if not want_snapshot:
        return kw, None
    snap = _rng.snapshot_buffer(dev)
    kw = dict(kw, rng_snapshot=snap)
    # the snapshot holds the absolute position the forward used: the backward adds nothing to it
    return kw, dict(seed=kw["seed"], offset=0, rng_state=snap)


class _NormalSample(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mean, std, modes, K, N, eps_in):
        fwd_kw, bwd_kw = _draw_kwargs(mean.device, eps_in, want_snapshot=True)
        z = be.normal_sample(mean, modes[0], std, modes[1], K, N, eps_in=eps_in, **fwd_kw)
        ctx.save_for_backward(mean, std, eps_in)
        ctx.cfg = (modes, K, N, bwd_kw)
        return z

    @staticmethod
    def backward(ctx, dz):
        mean, std, eps = ctx.saved_tensors
        modes, K, N, bwd_kw = ctx.cfg
        nm, ns = ctx.needs_input_grad[:2]
        dmean, dstd = be.normal_sample_bwd(dz.contiguous(), mean, modes[0], std, modes[1], K, N, eps=eps,
                                           need_mean=nm, need_std=ns, **bwd_kw)
        return dmean, dstd, None, None, None, None


def normal_sample(mean, std, n_samples, reparameterized):
    """Normal._sample (normal.py:89-107): [n_samples] + mean.shape (no leading axis for n_samples 1).

    The noise has the shape of `mean` (as in the reference, :90-104); injected noise, when present,
    replaces it (see _rng.inject)."""
    home = mean.device
    mean, std = to_compute(mean), to_compute(std)
    K = int(n_samples)
    base = tuple(mean.shape)
    out_shape = ((K,) if K > 1 else ()) + base
    N = _prod(base)
    eps_in = _rng.take_injected("normal")
    if eps_in is not None:
        eps_in = to_compute(eps_in).to(mean.dtype).reshape(K, N).contiguous()
    fits = tuple(_bshapes(base, std.shape)) == base
    if not fits or N == 0:
        # std broadcasts the mean (e.g. mean [1,3], std [2,1]): rare, composed from a noise draw
        if eps_in is None:
            eps_in = be.philox_normal(K * N, mean.dtype, 0.0, 1.0, device=mean.device, **_rng.draw_args(mean.device))
        eps = eps_in.reshape(out_shape)
        z = (mean.unsqueeze(0) + std.unsqueeze(0) * eps) if K > 1 else (mean + std * eps)
        z = z if reparameterized else z.detach()
        return back_home(z, home)
    L = Layout([out_shape], 0)
    L.k_axis, L.K, L.M = K > 1, K, N  # the particle axis is the sample axis
    L.S = out_shape
    (mc, mm), (sc, sm) = L.canon(mean), L.canon(std)
    if K == 1:
        mm = FULL if mm != SCALAR else mm
    if reparameterized:
        z = _NormalSample.apply(mc, sc, (mm, sm), K, N, eps_in)
    else:
        with torch.no_grad():
            z = _NormalSample.apply(mc.detach(), sc.detach(), (mm, sm), K, N, eps_in)
    return back_home(z.reshape(out_shape), home)


# --------------------------------------------------------------------------------------------
# Latent nodes: sample AND log q(sample) from one launch (zs_*_latent_fwd), joint backward (zs_*_latent_bwd)
# --------------------------------------------------------------------------------------------
class _NormalLatent(torch.autograd.Function):
    """(mean, std) -> (z [K,M,E], log q(z) [K,M], log N(z; 0, 1) [K,M]).  The third output is the log-density of the
    sample under the STANDARD Normal prior, produced by the same launch because it costs two FMAs per element there
    and a launch plus a pass over z anywhere else; a generator whose prior node is a standard Normal picks it up
    (std_prior_logp), any other prior ignores it.  backward receives the gradients reaching z (decoder, a non-standard
    prior node), log q and the standard-prior term and returns d/dmean, d/dstd from ONE launch: the density terms,
    the pathwise term through z = mean + std*eps when reparameterised (eps recovered from the sample), summed over
    particles."""

    @staticmethod
    def forward(ctx, mean, std, mode, K, M, E, eps_in, reparameterized):
        fwd_kw, _ = _draw_kwargs(mean.device, eps_in)
        r = be.normal_latent_fwd(mean, std, mode, K, M, E, eps_in=eps_in, want_logp=True, **fwd_kw)
        if r is None:
            raise be.BackendError("latent kernel refused a shape latent_supported() accepted")
        z, logq, logp = r
        ctx.save_for_backward(z, mean, std)
        ctx.cfg = (mode, K, M, E, reparameterized)
        ctx.set_materialize_grads(False)  # an output nobody differentiates arrives as None, not as a zero-filled tensor
        if not reparameterized:
            ctx.mark_non_differentiable(z)
        return z, logq, logp

    @staticmethod
    def backward(ctx, dz, dlogq, dlogp):
        z, mean, std = ctx.saved_tensors
        mode, K, M, E, reparam = ctx.cfg
        dz = dz.contiguous() if (dz is not None and reparam) else None
        dlogq = None if dlogq is None else dlogq.contiguous()
        # the prior term depends on the parameters only through the sample
        dlogp = dlogp.contiguous() if (dlogp is not None and reparam) else None
        dmean, dstd = be.normal_latent_bwd(dlogq, dlogp, dz, z, mean, std, mode, K, M, E, reparameterized=reparam)
        return dmean, dstd, None, None, None, None, None, None


class _BernoulliLatent(torch.autograd.Function):
    """probs -> (z, log q(z), log Bernoulli(z; 0.5)); samples carry no gradient, log q's gradient reaches probs in
    one launch (the prior term is constant in probs)."""

    @staticmethod
    def forward(ctx, probs, mode, K, M, E, u_in):
        fwd_kw, _ = _draw_kwargs(probs.device, u_in)
        r = be.bernoulli_latent_fwd(probs, mode, K, M, E, u_in=u_in, want_logp=True, want_bits=True, **fwd_kw)
        if r is None:
            raise be.BackendError("latent kernel refused a shape latent_supported() accepted")
        z, logq, logp, bits = r
        ctx.bits = bits  # the sample packed as bits (or None): what the backward reads instead of the 16x larger z
        ctx.save_for_backward(z, probs)
        ctx.cfg = (mode, K, M, E)
        ctx.mark_non_differentiable(z, logp)
        # without this autograd hands backward zero-filled [K,M,E] / [K,M] tensors for z and log p: two fill launches
        # (8 MB at config 3) per step for gradients that are never read
        ctx.set_materialize_grads(False)
        return z, logq, logp

    @staticmethod
    def backward(ctx, dz, dlogq, dlogp):
        z, probs = ctx.saved_tensors
        mode, K, M, E = ctx.cfg
        if dlogq is None:
            return torch.zeros_like(probs), None, None, None, None, None
        return (be.bernoulli_latent_bwd(dlogq.contiguous(), z, probs, mode, K, M, E, zbits=ctx.bits), None, None, None,
                None, None)


# log-density of a fused draw under the standard prior of its family, keyed by the identity of the sample tensor the
# caller holds: {id(z): (weakref(z), family, n_event, logp)}.  Entries die with the sample.
_std_logp = {}


def _remember_std_logp(z, family, n_event, logp):
    key = id(z)

    def _gone(_ref, key=key):
        _std_logp.pop(key, None)

    _std_logp[key] = (weakref.ref(z, _gone), family, n_event, logp)


STD_PRIOR_FOLD = True  # set False to always evaluate a prior node with its own launch


def std_prior_logp(given, family, n_event):
    """log p(given) under the family's standard prior (Normal(0, 1) / Bernoulli(0.5)) summed over the last n_event
    axes, if `given` is a sample whose fused draw already produced it; else None."""
    if not STD_PRIOR_FOLD:
        return None
    e = _std_logp.get(id(given))
    if e is None or e[0]() is not given or e[1] != family or e[2] != n_event:
        return None
    return e[3]


# "is this prior parameter tensor all equal to c?" without synchronising (or re-scanning) on the hot path: Python
# numbers are known, tensors are checked ONCE per tensor object and version (for a CUDA tensor one synchronisation at
# first sight, never during stream capture; for a host tensor one pass over it: 0.1 ms per [1024, 40] prior parameter,
# twice per step of a host-resident model before this memo).
_const_memo = {}


def is_constant(t, c):
    if not torch.is_tensor(t):
        return float(t) == c
    if t.numel() == 0 or t.requires_grad:
        return False
    key = (id(t), float(c))
    hit = _const_memo.get(key)
    if hit is not None and hit[0]() is t and hit[1] == t._version:
        return hit[2]
    if t.is_cuda and torch.cuda.is_current_stream_capturing():
        return False
    val = bool((t == c).all())
    if len(_const_memo) > 256:
        _const_memo.clear()

    def _gone(_ref, key=key):
        _const_memo.pop(key, None)

    _const_memo[key] = (weakref.ref(t, _gone), t._version, val)
    return val


def _aligned(t):
    """Contiguous and 16-byte aligned (a view into the middle of a buffer may not be); differentiable."""
    t = t.contiguous()
    return t.clone() if t.data_ptr() % 16 else t


def latent_supported(base_shape, n_event, dtype, *params):
    """Shapes the fused latent kernels take: the last n_event axes form an event row of E % 4 == 0 elements, every
    parameter has exactly the batch shape (no inner broadcasting), float32 / float64."""
    if n_event < 1 or n_event > len(base_shape) or dtype not in (torch.float32, torch.float64):
        return False
    E = _prod(base_shape[len(base_shape) - n_event:])
    if E == 0 or E % 4 != 0 or _prod(base_shape) == 0:
        return False
    return all(tuple(p.shape) == tuple(base_shape) for p in params)


def normal_sample_logq(mean, std, n_samples, reparameterized, n_event):
    """Normal._sample (normal.py:89-107) and the node's log q at that sample (normal.py:109-126 + the event sums) from
    one launch.  Returns (z, logq): z like normal_sample(), logq of shape ([K] +) batch_shape[:-n_event]."""
    home = mean.device
    mean, std = to_compute(mean), to_compute(std)
    K = int(n_samples)
    base = tuple(mean.shape)
    E = _prod(base[len(base) - n_event:])
    M = _prod(base[:len(base) - n_event])
    out_shape = ((K,) if K > 1 else ()) + base
    lead = ((K,) if K > 1 else ()) + base[:len(base) - n_event]
    eps_in = _rng.take_injected("normal")
    if eps_in is not None:
        eps_in = to_compute(eps_in).to(mean.dtype).reshape(K, M, E).contiguous()
    mode = KBCAST if K > 1 else FULL
    mc, sc = _aligned(mean.reshape(M, E)), _aligned(std.reshape(M, E))
    z, logq, logp = _NormalLatent.apply(mc, sc, mode, K, M, E, eps_in, bool(reparameterized))
    z = back_home(z.reshape(out_shape), home)
    _remember_std_logp(z, "normal", n_event, logp.reshape(lead))
    return z, logq.reshape(lead)


def bernoulli_sample_logq(probs, n_samples, n_event):
    home = probs.device
    probs = to_compute(probs)
    K = int(n_samples)
    base = tuple(probs.shape)
    E = _prod(base[len(base) - n_event:])
    M = _prod(base[:len(base) - n_event])
    out_shape = ((K,) if K > 1 else ()) + base
    lead = ((K,) if K > 1 else ()) + base[:len(base) - n_event]
    u_in = _rng.take_injected("uniform")
    if u_in is not None:
        u_in = to_compute(u_in).to(probs.dtype).reshape(K, M, E).contiguous()
    mode = KBCAST if K > 1 else FULL
    z, logq, logp = _BernoulliLatent.apply(_aligned(probs.reshape(M, E)), mode, K, M, E, u_in)
    z = back_home(z.reshape(out_shape), home)
    _remember_std_logp(z, "bernoulli", n_event, logp.reshape(lead))
    return z, logq.reshape(lead)


# --------------------------------------------------------------------------------------------
# Logistic / Laplace: the Normal node's kernel templates with another noise transform / log-density
# --------------------------------------------------------------------------------------------
class _LocScaleLogProb(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, loc, scale, family, modes, K, M, E):
        out = be.locscale_logprob_fwd(family, x, modes[0], loc, modes[1], scale, modes[2], K, M, E)
        ctx.save_for_backward(x, loc, scale)
        ctx.cfg = (family, modes, K, M, E)
        return out

    @staticmethod
    def backward(ctx, g):
        x, loc, scale = ctx.saved_tensors
        family, modes, K, M, E = ctx.cfg
        nx, nl, ns = ctx.needs_input_grad[:3]
        dx, dloc, dscale = be.locscale_logprob_bwd(family, g.contiguous(), x, modes[0], loc, modes[1], scale, modes[2],
                                                   K, M, E, nx, nl, ns)
        return dx, dloc, dscale, None, None, None, None, None


def locscale_log_prob(family, x, loc, scale, n_event):
    """Sum over the last n_event axes of the Logistic (logistic.py:72-83) / Laplace (laplace.py:78-92) log-density."""
    home = x.device
    x, loc, scale = to_compute(x), to_compute(loc), to_compute(scale)
    L = Layout([x.shape, loc.shape, scale.shape], n_event)
    if _prod(L.S) == 0:
        return back_home(torch.zeros(L.lead, dtype=x.dtype, device=x.device), home)
    (xc, xm), (lc, lm), (sc, sm) = L.canon(x), L.canon(loc), L.canon(scale)
    out = _LocScaleLogProb.apply(xc, lc, sc, family, (xm, lm, sm), L.K, L.M, L.E)
    return back_home(out.reshape(L.lead), home)


class _LocScaleSample(torch.autograd.Function):
    @staticmethod
    def forward(ctx, loc, scale, family, modes, K, N, u_in):
        fwd_kw, bwd_kw = _draw_kwargs(loc.device, u_in, want_snapshot=True)
        z = be.locscale_sample(family, loc, modes[0], scale, modes[1], K, N, u_in=u_in, **fwd_kw)
        ctx.save_for_backward(loc, scale, u_in)
        ctx.cfg = (family, modes, K, N, bwd_kw)
        return z

    @staticmethod
    def backward(ctx, dz):
        loc, scale, u = ctx.saved_tensors
        family, modes, K, N, bwd_kw = ctx.cfg
        nl, ns = ctx.needs_input_grad[:2]
        dloc, dscale = be.locscale_sample_bwd(family, dz.contiguous(), loc, modes[0], scale, modes[1], K, N, u=u,
                                              need_loc=nl, need_scale=ns, **bwd_kw)
        return dloc, dscale, None, None, None, None, None


def locscale_sample(family, loc, scale, n_samples, reparameterized):
    """Logistic._sample (logistic.py:56-70) / Laplace._sample (laplace.py:60-76): [n_samples] + batch shape, noise
    from in-kernel Philox uniforms (or injected uniforms, _rng.inject(uniform=...))."""
    home = loc.device
    loc, scale = to_compute(loc), to_compute(scale)
    base = tuple(_bshapes(loc.shape, scale.shape))
    loc, scale = loc.expand(base).contiguous(), scale.expand(base).contiguous()
    K = int(n_samples)
    out_shape = ((K,) if K > 1 else ()) + base
    N = _prod(base)
    if N == 0:
        return back_home(torch.zeros(out_shape, dtype=loc.dtype, device=loc.device), home)
    u_in = _rng.take_injected("uniform")
    if u_in is not None:
        u_in = to_compute(u_in).to(loc.dtype).reshape(K, N).contiguous()
    mode = KBCAST if K > 1 else FULL
    if reparameterized:
        z = _LocScaleSample.apply(loc, scale, family, (mode, mode), K, N, u_in)
    else:
        with torch.no_grad():
            z = _LocScaleSample.apply(loc.detach(), scale.detach(), family, (mode, mode), K, N, u_in)
    return back_home(z.reshape(out_shape), home)


# --------------------------------------------------------------------------------------------
# Bernoulli
# --------------------------------------------------------------------------------------------
class _BernoulliLogPmf(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, probs, modes, K, M, E, logits=False):
        out = be.bernoulli_logpmf_fwd(x, modes[0], probs, modes[1], K, M, E, logits=logits)
        ctx.save_for_backward(x, probs)
        ctx.cfg = (modes, K, M, E, logits)
        return out

    @staticmethod
    def backward(ctx, g):
        x, probs = ctx.saved_tensors
        modes, K, M, E, logits = ctx.cfg
        nx, np_ = ctx.needs_input_grad[:2]
        dx, dprobs = be.bernoulli_logpmf_bwd(g.contiguous(), x, modes[0], probs, modes[1], K, M, E, nx, np_,
                                             logits=logits)
        return dx, dprobs, None, None, None, None, None


def bernoulli_log_prob(x, probs, n_event, logits=False):
    """sum over the last n_event axes of x*log(p+1e-8) + (1-x)*log(1-p+1e-8) (bernoulli.py:84-95).
    `logits=True`: `probs` holds logits, p = sigmoid(logits) is formed inside the kernel (bernoulli.py:47-50)
    and the gradient flows to the logits."""
    home = probs.device
    x, probs = to_compute(x), to_compute(probs)
    L = Layout([x.shape, probs.shape], n_event)
    if _prod(L.S) == 0:
        return back_home(torch.zeros(L.lead, dtype=probs.dtype, device=probs.device), home)
    (xc, xm), (pc, pm) = L.canon(x), L.canon(probs)
    if pm == SCALAR:  # the kernels take probs as FULL / KBCAST only when it needs no gradient either way
        pc, pm = probs.expand(L.S).contiguous(), FULL
    out = _BernoulliLogPmf.apply(xc, pc, (xm, pm), L.K, L.M, L.E, bool(logits))
    return back_home(out.reshape(L.lead), home)


def bernoulli_sample(probs, n_samples):
    """Bernoulli._sample (bernoulli.py:72-82): float samples, [n_samples] + probs.shape."""
    home = probs.device
    probs = to_compute(probs).detach()
    K = int(n_samples)
    base = tuple(probs.shape)
    out_shape = ((K,) if K > 1 else ()) + base
    N = _prod(base)
    if N == 0:
        return back_home(torch.zeros(out_shape, dtype=probs.dtype, device=probs.device), home)
    u_in = _rng.take_injected("uniform")
    if u_in is not None:
        u_in = to_compute(u_in).to(probs.dtype).reshape(K, N).contiguous()
    kw, _ = _draw_kwargs(probs.device, u_in)
    out = be.bernoulli_sample(probs.contiguous(), KBCAST if K > 1 else FULL, K, N, u_in=u_in, **kw)
    return back_home(out.reshape(out_shape), home)


# --------------------------------------------------------------------------------------------
# Poisson
# --------------------------------------------------------------------------------------------
class _PoissonLogPmf(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, rate, modes, K, M, E):
        out = be.poisson_logpmf_fwd(x, modes[0], rate, modes[1], K, M, E)
        ctx.save_for_backward(x, rate)
        ctx.cfg = (modes, K, M, E)
        return out

    @staticmethod
    def backward(ctx, g):
        x, rate = ctx.saved_tensors
        modes, K, M, E = ctx.cfg
        drate = be.poisson_logpmf_bwd(g.contiguous(), x, modes[0], rate, modes[1], K, M, E) if ctx.needs_input_grad[1] \
            else None
        return None, drate, None, None, None, None


def _no_count_grad(x):
    if torch.is_tensor(x) and x.requires_grad:
        raise ValueError("Poisson.log_prob: the counts have no gradient (the log-pmf is defined at integers); "
                         "pass a tensor that does not require grad (e.g. x.detach())")


def poisson_log_prob(x, rate, n_event):
    """sum over the last n_event axes of xlogy(x, rate) - rate - lgamma(x + 1) (the reference's poisson.py:75,
    torch.distributions.Poisson.log_prob); the gradient reaches `rate` only."""
    _no_count_grad(x)
    home = rate.device
    x, rate = to_compute(x), to_compute(rate)
    L = Layout([x.shape, rate.shape], n_event)
    if _prod(L.S) == 0:
        return back_home(torch.zeros(L.lead, dtype=rate.dtype, device=rate.device), home)
    (xc, xm), (rc, rm) = L.canon(x), L.canon(rate)
    if rm == SCALAR:  # as for Bernoulli: a gradient w.r.t. a SCALAR operand is the host's job, so expand it
        rc, rm = rate.expand(L.S).contiguous(), FULL
    out = _PoissonLogPmf.apply(xc, rc, (xm, rm), L.K, L.M, L.E)
    return back_home(out.reshape(L.lead), home)


def poisson_sample(rate, n_samples):
    """Poisson._sample (the reference's poisson.py:61): float counts, [n_samples] + rate.shape (no leading axis
    for n_samples 1), drawn in-kernel from Philox uniforms; no gradient."""
    home = rate.device
    rate = to_compute(rate).detach()
    K = int(n_samples)
    base = tuple(rate.shape)
    out_shape = ((K,) if K > 1 else ()) + base
    N = _prod(base)
    if N == 0:
        return back_home(torch.zeros(out_shape, dtype=rate.dtype, device=rate.device), home)
    kw, _ = _draw_kwargs(rate.device, None)
    out = be.poisson_sample(rate.contiguous(), KBCAST if K > 1 else FULL, K, N, **kw)
    return back_home(out.reshape(out_shape), home)


# --------------------------------------------------------------------------------------------
# Beta (log-density: locscale_log_prob with FAM_BETA)
# --------------------------------------------------------------------------------------------
def beta_sample(alpha, beta, n_samples):
    """Beta._sample (torch.distributions.Beta.sample, which the reference's beta.py calls): [n_samples] + the
    broadcast shape of alpha and beta (no leading axis for n_samples 1), drawn in-kernel; no gradient."""
    home = alpha.device
    # uploaded outside no_grad: a memoised upload is reused by the log-density, which needs its autograd edge
    alpha, beta = to_compute(alpha).detach(), to_compute(beta).detach()
    with torch.no_grad():
        base = tuple(_bshapes(alpha.shape, beta.shape))
        alpha, beta = alpha.expand(base).contiguous(), beta.expand(base).contiguous()
        K = int(n_samples)
        out_shape = ((K,) if K > 1 else ()) + base
        N = _prod(base)
        if N == 0:
            return back_home(torch.zeros(out_shape, dtype=alpha.dtype, device=alpha.device), home)
        kw, _ = _draw_kwargs(alpha.device, None)
        mode = KBCAST if K > 1 else FULL
        out = be.beta_sample(alpha, mode, beta, mode, K, N, **kw)
    return back_home(out.reshape(out_shape), home)


# --------------------------------------------------------------------------------------------
# Categorical (not in the reference; see distributions/categorical.py)
# --------------------------------------------------------------------------------------------
class _CategoricalLogPmf(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, logits, modes, K, M, C):
        out = be.categorical_logpmf_fwd(x, modes[0], logits, modes[1], K, M, C)
        ctx.save_for_backward(x, logits)
        ctx.cfg = (modes, K, M, C)
        return out

    @staticmethod
    def backward(ctx, g):
        x, logits = ctx.saved_tensors
        modes, K, M, C = ctx.cfg
        d = be.categorical_logpmf_bwd(g.contiguous(), x, modes[0], logits, modes[1], K, M, C)
        return None, d, None, None, None, None


def categorical_log_prob(x, logits):
    """log_softmax(logits)[x]; x has shape (...,) + logits.shape[:-1] (or broadcastable to it)."""
    home = logits.device
    x, logits = to_compute(x), to_compute(logits)
    C = int(logits.shape[-1])
    L = Layout([x.shape, logits.shape[:-1]], 0)
    if _prod(L.S) == 0:
        return back_home(torch.zeros(L.S, dtype=logits.dtype, device=logits.device), home)
    xc, xm = L.canon(x.to(logits.dtype))
    lpad = (1,) * (len(L.S) - (logits.dim() - 1)) + tuple(logits.shape[:-1])
    if lpad == L.S:
        lc, lm = logits.contiguous(), FULL
    elif L.K > 1 and lpad[0] == 1:
        lc, lm = logits.reshape(lpad[1:] + (C,)).expand(L.S[1:] + (C,)).contiguous(), KBCAST
    else:
        lc, lm = logits.expand(L.S + (C,)).contiguous(), FULL
    out = _CategoricalLogPmf.apply(xc, lc, (xm, lm), L.K, L.M, C)
    return back_home(out.reshape(L.S), home)


def categorical_sample(logits, n_samples):
    home = logits.device
    logits = to_compute(logits).detach().contiguous()
    K = int(n_samples)
    base = tuple(logits.shape[:-1])
    C = int(logits.shape[-1])
    out_shape = ((K,) if K > 1 else ()) + base
    M = _prod(base)
    if M == 0:
        return back_home(torch.zeros(out_shape, dtype=logits.dtype, device=logits.device), home)
    u_in = _rng.take_injected("uniform")
    if u_in is not None:
        u_in = to_compute(u_in).to(logits.dtype).reshape(K, M).contiguous()
    kw, _ = _draw_kwargs(logits.device, u_in)
    out = be.categorical_sample(logits, KBCAST if K > 1 else FULL, K, M, C, u_in=u_in, **kw)
    return back_home(out.reshape(out_shape), home)


# --------------------------------------------------------------------------------------------
# objectives
# --------------------------------------------------------------------------------------------
class _IWObjective(torch.autograd.Function):
    """cost (scalar mean or per column) of the IW-SGVB / VIMCO surrogate with its gradient computed in
    the same launch (importance_weighted_objective.py:16-25,102-191)."""

    @staticmethod
    def forward(ctx, logp, logq, estimator, reduce_mean):
        K, B = logp.shape
        need = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        cost, dlp, dlq = be.iw_objective(estimator, logp, logq, _mean_scale(B) if reduce_mean else 1.0, need_grads=need)
        ctx.save_for_backward(dlp, dlq)
        ctx.reduce_mean = reduce_mean
        return _mean_cost(cost, B) if reduce_mean else cost

    @staticmethod
    def backward(ctx, g):
        dlp, dlq = ctx.saved_tensors
        if not ctx.reduce_mean:
            g = g.reshape(1, -1)
        return (dlp * g if ctx.needs_input_grad[0] else None, dlq * g if ctx.needs_input_grad[1] else None, None, None)


def iw_objective(logp, logq, axis, estimator, reduce_mean):
    """logp/logq: same-shaped tensors; `axis` is the particle axis.  Returns the surrogate cost
    (0-d if reduce_mean else the shape of logp without `axis`)."""
    home = logp.device
    logp, logq = torch.broadcast_tensors(to_compute(logp), to_compute(logq))
    nd = logp.dim()
    ax = axis % nd if nd > 0 else 0
    lp = logp.movedim(ax, 0) if nd > 0 else logp.reshape(1)
    lq = logq.movedim(ax, 0) if nd > 0 else logq.reshape(1)
    rest = tuple(lp.shape[1:])
    K = int(lp.shape[0])
    lp2, lq2 = lp.reshape(K, -1).contiguous(), lq.reshape(K, -1).contiguous()
    out = _IWObjective.apply(lp2, lq2, estimator, bool(reduce_mean))
    if not reduce_mean:
        out = out.reshape(rest)
    return back_home(out, home)


class _ElboWithLogDet(torch.autograd.Function):
    """ELBO.sgvb with a flow (elbo.py:155-161): -mean_{k,b}(logp - logq) - sum(log_det) from ONE objective launch (the
    per-column costs and both gradients) and ONE reduction launch that folds the log-determinants in."""

    @staticmethod
    def forward(ctx, logp, logq, log_det):
        K, B = logp.shape
        need = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        cost, dlp, dlq = be.iw_objective(be.ELBO, logp, logq, _mean_scale(B), need_grads=need)
        ctx.save_for_backward(dlp, dlq)
        ctx.ld_shape = log_det.shape
        return be.combine_sums(cost, _mean_scale(B), log_det.reshape(-1), -1.0).reshape(())

    @staticmethod
    def backward(ctx, g):
        dlp, dlq = ctx.saved_tensors
        return (dlp * g if ctx.needs_input_grad[0] else None, dlq * g if ctx.needs_input_grad[1] else None,
                (-g).expand(ctx.ld_shape) if ctx.needs_input_grad[2] else None)


def elbo_with_log_det(logp, logq, log_det):
    """logp / logq [K, ...] broadcastable, log_det any shape -> the scalar ELBO cost with the flow term."""
    home = logq.device
    lp, lq = torch.broadcast_tensors(to_compute(logp), to_compute(logq))
    K = int(lp.shape[0])
    ld = to_compute(log_det).to(lq.dtype).contiguous()
    out = _ElboWithLogDet.apply(lp.reshape(K, -1).contiguous(), lq.reshape(K, -1).contiguous(), ld)
    return back_home(out, home)


class _Reinforce(torch.autograd.Function):
    """ELBO.reinforce, moving-mean baseline, mean over all elements: surrogate cost, both gradients and the in-place
    update of the float32 state in ONE launch (elbo.py:200-238)."""

    @staticmethod
    def forward(ctx, logp, logq, moving_mean, local_step, decay):
        need = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        cost, dlp, dlq = be.reinforce_step(logp, logq, moving_mean, local_step, decay, need_grads=need)
        ctx.save_for_backward(dlp, dlq)
        return cost.reshape(())

    @staticmethod
    def backward(ctx, g):
        dlp, dlq = ctx.saved_tensors
        return (dlp * g if ctx.needs_input_grad[0] else None, dlq * g if ctx.needs_input_grad[1] else None, None, None,
                None)


def reinforce(logp, logq, moving_mean, local_step, decay):
    """logp / logq broadcastable tensors; moving_mean [1] float32 / local_step [1] int32 module buffers (any device:
    they are moved to the compute device for the launch and written back)."""
    home = logq.device
    lp, lq = torch.broadcast_tensors(to_compute(logp), to_compute(logq))
    lp, lq = lp.contiguous(), lq.contiguous()
    mm = moving_mean if be.on_compute_device(moving_mean) else to_compute(moving_mean.detach()).clone()
    ls = local_step if be.on_compute_device(local_step) else to_compute(local_step.detach()).clone()
    out = _Reinforce.apply(lp, lq, mm, ls, float(decay))
    if mm is not moving_mean:
        with torch.no_grad():
            moving_mean.copy_(mm)
            local_step.copy_(ls)
    return back_home(out, home)


class _LogMeanExp(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x):
        ctx.save_for_backward(x)
        return be.log_mean_exp(x)

    @staticmethod
    def backward(ctx, g):
        (x,) = ctx.saved_tensors
        return be.log_mean_exp_bwd(g.contiguous(), x)


def log_mean_exp(x, dim, keepdims):
    home = x.device
    x = to_compute(x)
    nd = x.dim()
    ax = dim % nd
    xm = x.movedim(ax, 0)
    rest = tuple(xm.shape[1:])
    out = _LogMeanExp.apply(xm.reshape(xm.shape[0], -1).contiguous()).reshape(rest)
    if keepdims:
        out = out.unsqueeze(ax)
    return back_home(out, home)


class _IWBernoulliFused(torch.autograd.Function):
    """Bernoulli likelihood + IW objective, forward and backward in ONE launch (zs_fused_iw.cu).
    The gradients are computed for a unit upstream gradient; backward applies the actual upstream
    scalar with zs_scale_inplace, which is a no-op launch for the usual loss.backward()."""

    @staticmethod
    def forward(ctx, probs, x, logp_other, logq, estimator, logits=False):
        K, B, X = probs.shape
        # per-column costs come out already scaled by 1 / (columns of the local or global batch): the mean objective
        # is ONE reduction over them
        # ... which the launch does itself (zs_iw_bernoulli_fused_loss): no reduction kernel after it
        r = be.iw_bernoulli_fused(estimator, probs, x, logp_other, logq, _mean_scale(B),
                                  need_dprobs=ctx.needs_input_grad[0], logits=logits, cost_scaled=True, want_loss=True)
        if r is None:
            raise be.BackendError("fused IW kernel refused a shape fused_supported() accepted")
        ctx.grads = (r["dprobs"], r["dlogp"], r["dlogq"])
        loss = r.get("loss")
        return loss.reshape(()) if loss is not None else r["cost"].sum()

    @staticmethod
    def backward(ctx, g):
        if ctx.grads is None:
            raise RuntimeError("the fused IW objective hands its gradient buffers to autograd and can be "
                               "back-propagated once; set zhusuan.variational.FUSED = False for retain_graph")
        dprobs, dlp, dlq = ctx.grads
        ctx.grads = None
        g1 = g.reshape(1).contiguous()
        # one launch applies the upstream scalar to all three gradient buffers (a no-op for loss.backward())
        if dprobs is not None:
            be.scale_inplace(dprobs, g1, dlp, dlq)
        else:
            be.scale_inplace(dlp, g1, dlq)
        return (dprobs, None, dlp if ctx.needs_input_grad[2] else None, dlq if ctx.needs_input_grad[3] else None,
                None, None)


def iw_bernoulli_fused(probs, x, logp_other, logq, estimator, logits=False):
    """probs [K,B,X] (CUDA, float32; logits when `logits=True`), x [B,X], logp_other / logq [K,B] or None
    -> scalar loss."""
    probs = _aligned(probs)
    x = _aligned(x.to(probs.dtype))
    lo = None if logp_other is None else logp_other.contiguous()
    lq = None if logq is None else logq.contiguous()
    return _IWBernoulliFused.apply(probs, x, lo, lq, estimator, bool(logits))


class _IWPoissonFused(torch.autograd.Function):
    """Poisson likelihood + IW objective, forward and backward in ONE launch (zs_iw_poisson_fused_loss); the
    upstream scalar is applied in backward exactly as for _IWBernoulliFused."""

    @staticmethod
    def forward(ctx, rate, x, logp_other, logq, estimator):
        K, B, X = rate.shape
        r = be.iw_poisson_fused(estimator, rate, x, logp_other, logq, _mean_scale(B), need_drate=ctx.needs_input_grad[0],
                                cost_scaled=True, want_loss=True)
        if r is None:
            raise be.BackendError("fused Poisson IW kernel refused a shape fused_poisson_supported() accepted")
        ctx.grads = (r["dprobs"], r["dlogp"], r["dlogq"])
        loss = r.get("loss")
        return loss.reshape(()) if loss is not None else r["cost"].sum()

    @staticmethod
    def backward(ctx, g):
        return _IWBernoulliFused.backward(ctx, g)[:5]  # same gradient buffers; one input (`logits`) fewer


def iw_poisson_fused(rate, x, logp_other, logq, estimator):
    """rate [K,B,X] (CUDA, float32), counts x [B,X], logp_other / logq [K,B] or None -> scalar loss."""
    rate = _aligned(rate)
    x = _aligned(x.to(rate.dtype))
    lo = None if logp_other is None else logp_other.contiguous()
    lq = None if logq is None else logq.contiguous()
    return _IWPoissonFused.apply(rate, x, lo, lq, estimator)


# --------------------------------------------------------------------------------------------
# host-buffer route: probs / x live in (pinned) host memory
# --------------------------------------------------------------------------------------------
_host_pool = {}


def _pinned(shape, key):
    return pinned_like_pool(shape, torch.float32, key)


def _workspace(nbytes):
    ws = _host_pool.get("ws")
    if ws is None or ws.numel() < nbytes or ws.device != compute_device():
        ws = torch.empty(nbytes, dtype=torch.uint8, device=compute_device())
        _host_pool["ws"] = ws
    return ws


def _host_step_handle(dev):
    """One zs_host_step handle per (thread's) compute device: the library keeps no global state for these calls."""
    key = ("hs", dev.index)
    hs = _host_pool.get(key)
    if hs is None:
        hs = be.HostStep(dev)
        _host_pool[key] = hs
    return hs


class _IWBernoulliFusedHost(torch.autograd.Function):
    """The fused likelihood + objective step for HOST-resident probs / x: zs_iw_step_host_begin pipelines
    H2D copies, the fused kernel and D2H copies over column chunks.  The [K,B] log-weight terms and their
    gradients stay on the device (they come from / go to the latent nodes' kernels); forward returns as soon
    as the per-column costs have landed, while the tail of dprobs is still on its way to pinned host memory.

    backward must hand autograd a gradient that HAS landed whenever anything may read it during the backward pass:
    a CPU decoder upstream of `probs` (its backward nodes run on the CPU thread right away), or an existing
    `probs.grad` (AccumulateGrad adds into it).  Only when `probs` is a leaf without a gradient -- AccumulateGrad
    then just stores the tensor -- the wait is deferred to an end-of-backward callback so the latent nodes'
    backward overlaps the transfer (`defer_ok`, decided by the caller who sees the real tensor)."""

    @staticmethod
    def forward(ctx, probs, x, logp_other, logq, estimator, defer_ok):
        K, B, X = probs.shape
        dev = compute_device()
        hs = _host_step_handle(dev)
        cost = _pinned((B,), "cost")
        dprobs = _pinned((K, B, X), "dprobs") if ctx.needs_input_grad[0] else None
        dlp = torch.empty((K, B), dtype=torch.float32, device=dev)
        dlq = torch.empty((K, B), dtype=torch.float32, device=dev)
        ws = _workspace(be.iw_step_host_workspace(K, B, X))
        be.iw_step_host_begin(hs, estimator, cost, dprobs, dlp, dlq, probs, x, logp_other, logq, K, B, X,
                              _mean_scale(B), ws, True)
        be.iw_step_host_wait(hs, 0)
        ctx.grads = (dprobs, dlp, dlq)
        ctx.hs = hs
        ctx.defer_ok = bool(defer_ok)
        return _mean_cost(cost, B)

    @staticmethod
    def backward(ctx, g):
        if ctx.grads is None:
            raise RuntimeError("the fused IW objective hands its gradient buffers to autograd and can be "
                               "back-propagated once; set zhusuan.variational.FUSED = False for retain_graph")
        dprobs, dlp, dlq = ctx.grads
        ctx.grads = None
        hs = ctx.hs
        gv = float(g)
        if dprobs is not None:
            if gv != 1.0 or not ctx.defer_ok:
                be.iw_step_host_wait(hs, 1)
                if gv != 1.0:
                    dprobs = dprobs * gv
            else:
                # dprobs may still be landing: the engine runs this after the whole backward pass, before
                # loss.backward() / autograd.grad() return to the caller
                torch.autograd.Variable._execution_engine.queue_callback(lambda: be.iw_step_host_wait(hs, 1))
        return (dprobs, None, dlp * gv if ctx.needs_input_grad[2] else None,
                dlq * gv if ctx.needs_input_grad[3] else None, None, None)


def iw_bernoulli_fused_host(probs, x, logp_other, logq, estimator):
    """probs [K,B,X] / x [B,X] float32 CPU tensors (pinned for full PCIe speed), logp_other / logq
    [K,B] tensors (any device; moved to the compute device) or None -> scalar CPU loss."""
    be.require_cuda()
    f = lambda t: None if t is None else to_compute(t).to(torch.float32).contiguous()
    # the deferred wait is only safe when autograd will merely STORE the gradient (see the class docstring)
    defer_ok = probs.is_leaf and probs.grad is None and probs.is_contiguous()
    return _IWBernoulliFusedHost.apply(probs.contiguous(), x.to(torch.float32).contiguous(), f(logp_other), f(logq),
                                       estimator, defer_ok)
