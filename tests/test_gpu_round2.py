"""GPU tests of what round 2 added to the boundary and the product path:
graph-safe device-side Philox state, multi-tensor SG-MCMC launch, the prior's log-density folded into the latent launch,
deferred first draws, a CUDA-graph capturable public-API step, pinned-pool / host-route / device-guard fixes."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from zhusuan import _backend as be  # noqa: E402
from zhusuan import _ops, _rng  # noqa: E402

DEV = "cuda"
KBCAST = be.KBCAST


def host(t):
    return t.detach().cpu().numpy()


def _state(offset=0):
    st = torch.zeros(2, dtype=torch.int64, device=DEV)
    be.rng_state_init(st, offset)
    return st


# ----------------------------------------------------------------------------- device-side stream position
def test_rng_state_advances_one_tick_per_launch(oracle):
    """A launch with a device state draws from offset + state and advances the state by ZS_RNG_TICK once: a sequence of
    launches equals by-value launches at base, base + 4, base + 8 ... bit for bit, whatever the grid size."""
    base, seed = 1000, 77
    st = _state(base)
    for i, n in enumerate([64, 4096, 1 << 20, 4]):  # 1 CTA ... grid capped below the work
        got = host(be.philox_raw(n, seed, 12, DEV, rng_state=st)).view(np.uint32)
        assert np.array_equal(got, oracle.philox_raw(n, seed, base + 12 + 4 * i))
        assert host(st).tolist() == [base + 4 * (i + 1), 0]  # offset advanced, arrival counter back to zero


def test_rng_state_in_every_sampler():
    """Each sampling entry point honours the state: equal to the by-value call at the state's position, and advances."""
    K, N, seed = 6, 1000, 5
    mean, std = torch.randn(N, device=DEV), torch.rand(N, device=DEV) + 0.5
    p = torch.rand(N, device=DEV)
    cases = [
        lambda **kw: be.normal_sample(mean, KBCAST, std, KBCAST, K, N, **kw),
        lambda **kw: be.bernoulli_sample(p, KBCAST, K, N, **kw),
        lambda **kw: be.locscale_sample(be.FAM_LOGISTIC, mean, KBCAST, std, KBCAST, K, N, **kw),
        lambda **kw: be.categorical_sample(torch.arange(10 * 7, device=DEV, dtype=torch.float32).reshape(10, 7).sin(), KBCAST, K, 10, 7, **kw),
        lambda **kw: be.normal_latent_fwd(mean.reshape(25, 40), std.reshape(25, 40), KBCAST, K, 25, 40, **kw)[0],
        lambda **kw: be.bernoulli_latent_fwd(p.reshape(25, 40), KBCAST, K, 25, 40, **kw)[0],
        lambda **kw: be.sgld_step(mean, std, 1e-2, **kw),
        lambda **kw: be.psgld_step(mean, torch.ones_like(mean), std, 1e-2, 0.9, 1e-3, **kw),
        lambda **kw: be.sghmc_post(mean, torch.zeros_like(mean), std, 1e-2, 0.3, 0.02, True, **kw),
        lambda **kw: be.philox_normal(N, torch.float32, 0.0, 1.0, device=DEV, **kw),
        lambda **kw: be.philox_uniform(N, torch.float32, device=DEV, **kw),
    ]
    for f in cases:
        st = _state(40)
        a = f(seed=seed, offset=8, rng_state=st)
        b = f(seed=seed, offset=8, rng_state=st)
        assert torch.equal(a, f(seed=seed, offset=48))
        assert torch.equal(b, f(seed=seed, offset=52))
        assert not torch.equal(a, b)
        assert host(st).tolist() == [48, 0]


def test_rng_state_untouched_by_injected_noise():
    N = 256
    mean, std = torch.zeros(N, device=DEV), torch.ones(N, device=DEV)
    st = _state(8)
    be.normal_sample(mean, KBCAST, std, KBCAST, 2, N, eps_in=torch.randn(2, N, device=DEV), rng_state=st)
    be.sgld_step(mean, std, 1e-2, noise=torch.randn(N, device=DEV), rng_state=st)
    assert host(st).tolist() == [8, 0]


def test_sample_backward_regenerates_from_snapshot():
    """Forward under a device state records the position it used; the backward regenerates exactly that noise."""
    K, N = 7, 333
    mean, std = torch.randn(N, device=DEV), torch.rand(N, device=DEV) + 0.5
    st, snap = _state(100), torch.zeros(2, dtype=torch.int64, device=DEV)
    eps = torch.empty(K, N, device=DEV)
    be.normal_sample(mean, KBCAST, std, KBCAST, K, N, eps_out=eps, seed=3, offset=4, rng_state=st, rng_snapshot=snap)
    assert host(snap).tolist() == [104, 0]
    be.normal_sample(mean, KBCAST, std, KBCAST, K, N, seed=3, offset=4, rng_state=st)  # the stream moves on
    dz = torch.randn(K, N, device=DEV)
    dm, ds = be.normal_sample_bwd(dz, mean, KBCAST, std, KBCAST, K, N, seed=3, offset=0, rng_state=snap)
    dm_ref, ds_ref = be.normal_sample_bwd(dz, mean, KBCAST, std, KBCAST, K, N, eps=eps)
    assert torch.equal(dm, dm_ref) and torch.equal(ds, ds_ref)
    assert host(snap).tolist() == [104, 0]  # a snapshot is read, never advanced


def test_graph_replays_draw_fresh_noise():
    """The point of the device-side state: a captured sampling launch draws new noise on every replay."""
    K, M, E, seed = 50, 64, 40, 9
    mean, std = torch.randn(M, E, device=DEV), torch.rand(M, E, device=DEV) + 0.5
    st = _state(0)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        be.normal_latent_fwd(mean, std, KBCAST, K, M, E, seed=seed, rng_state=st)  # warm-up, tick 0
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            z, lq, lp = be.normal_latent_fwd(mean, std, KBCAST, K, M, E, seed=seed, rng_state=st)
    torch.cuda.current_stream().wait_stream(s)
    seen = []
    for _ in range(3):
        g.replay()
        torch.cuda.synchronize()
        seen.append(z.clone())
    assert not torch.equal(seen[0], seen[1]) and not torch.equal(seen[1], seen[2])
    for i, zi in enumerate(seen):  # replay i is the launch at tick i + 1 of the stream
        ref, _, _ = be.normal_latent_fwd(mean, std, KBCAST, K, M, E, seed=seed, offset=4 * (i + 1))
        assert torch.equal(zi, ref)
    # the by-value form is what round 1 had: every replay repeats the same draw
    g2 = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g2, stream=s):
            z2, _, _ = be.normal_latent_fwd(mean, std, KBCAST, K, M, E, seed=seed, offset=4)
    g2.replay(); a = z2.clone(); g2.replay(); torch.cuda.synchronize()
    assert torch.equal(a, z2)


def test_public_api_uses_device_state_and_reseeds():
    from zhusuan.distributions import Normal
    mean, std = torch.zeros(8, 40, device=DEV), torch.ones(8, 40, device=DEV)
    torch.manual_seed(123)
    a = Normal(mean=mean, std=std).sample(5)
    b = Normal(mean=mean, std=std).sample(5)
    torch.manual_seed(123)
    a2 = Normal(mean=mean, std=std).sample(5)
    torch.rand(3, device=DEV)  # torch's own generator use in between moves our stream to a fresh block, never back
    b2 = Normal(mean=mean, std=std).sample(5)
    assert torch.equal(a, a2) and not torch.equal(a, b) and not torch.equal(b2, a) and not torch.equal(b2, b)


# ----------------------------------------------------------------------------- multi-tensor SG-MCMC
@pytest.mark.parametrize("dt", [torch.float32, torch.float64])
def test_sgmcmc_multi_step_equals_single_tensor_calls(dt):
    """One launch over several tensors == per-tensor launches fed the noise of the shared stream position: tensor t
    owns quads [q_t, q_t + ceil(n_t/4)), element i word i%4 of counter q_t + i/4."""
    sizes = [4550, 51, 3, 128, 1]  # odd sizes, an unaligned tail, a sub-quad tensor
    seed, off, lr = 21, 64, 1e-2
    ws = [torch.randn(n, device=DEV, dtype=dt) for n in sizes]
    gs = [torch.randn(n, device=DEV, dtype=dt) for n in sizes]
    quads = [(n + 3) // 4 for n in sizes]
    unit = be.philox_normal(4 * sum(quads), torch.float32, 0.0, 1.0, seed, off, DEV)
    q0 = np.concatenate([[0], np.cumsum(quads)])
    noise = lambda t, std: (np.float32(std) * unit[4 * q0[t]:4 * q0[t] + sizes[t]]).to(dt)

    new = be.sgmcmc_multi_step(be.ALG_SGLD, ws, gs, lr=lr, seed=seed, offset=off)
    for t in range(len(sizes)):
        ref = be.sgld_step(ws[t], gs[t], lr, noise=noise(t, np.sqrt(np.float64(np.float32(lr)))))
        torch.testing.assert_close(new[t], ref, rtol=1e-6 if dt == torch.float32 else 1e-7, atol=1e-7)
    # one tensor: bit-identical to the single-tensor entry point
    assert torch.equal(be.sgmcmc_multi_step(be.ALG_SGLD, ws[:1], gs[:1], lr=lr, seed=seed, offset=off)[0],
                       be.sgld_step(ws[0], gs[0], lr, seed=seed, offset=off))

    aux = [torch.rand(n, device=DEV, dtype=dt) for n in sizes]
    aux2 = [a.clone() for a in aux]
    new = be.sgmcmc_multi_step(be.ALG_PSGLD, ws, gs, aux, lr=lr, a=0.9, b=1e-3, seed=seed, offset=off)
    for t in range(len(sizes)):
        ref = be.psgld_step(ws[t], aux2[t], gs[t], lr, 0.9, 1e-3, noise_unit=noise(t, 1.0))
        torch.testing.assert_close(new[t], ref, rtol=1e-5, atol=1e-6)
        torch.testing.assert_close(aux[t], aux2[t])

    for second in (False, True):
        v = [torch.randn(n, device=DEV, dtype=dt) for n in sizes]
        v2 = [a.clone() for a in v]
        half = be.sgmcmc_multi_step(be.ALG_SGHMC_PRE, ws, None, v, lr=lr, resample=True, second_order=second, seed=seed,
                                    offset=off)
        for t in range(len(sizes)):
            ref = be.sghmc_pre(ws[t], v2[t], lr, True, second, v_noise=noise(t, np.sqrt(lr)))
            torch.testing.assert_close(half[t], ref)
            torch.testing.assert_close(v[t], v2[t])
        new = be.sgmcmc_multi_step(be.ALG_SGHMC_POST, half, gs, v, lr=lr, a=0.3, b=0.02, second_order=second, seed=seed,
                                   offset=off + 4)
        unit2 = be.philox_normal(4 * sum(quads), torch.float32, 0.0, 1.0, seed, off + 4, DEV)
        for t in range(len(sizes)):
            nz = (np.float32(np.sqrt(2.0 * (0.3 - 0.02) * lr)) * unit2[4 * q0[t]:4 * q0[t] + sizes[t]]).to(dt)
            ref = be.sghmc_post(half[t], v2[t], gs[t], lr, 0.3, 0.02, second, noise=nz)
            torch.testing.assert_close(new[t], ref, rtol=1e-6, atol=1e-7)
            torch.testing.assert_close(v[t], v2[t], rtol=1e-6, atol=1e-7)


def test_sgmcmc_multi_step_more_tensors_than_one_table():
    n = be.CHAIN_MAX_TENSORS + 5
    ws = [torch.randn(17, device=DEV) for _ in range(n)]
    gs = [torch.randn(17, device=DEV) for _ in range(n)]
    new = be.sgmcmc_multi_step(be.ALG_SGLD, ws, gs, lr=1e-2, seed=1, offset=0)
    assert len(new) == n and all(torch.isfinite(t).all() and not torch.equal(t, w) for t, w in zip(new, ws))


def test_sampler_update_is_one_launch_for_all_latents():
    """SGLD over two differently shaped latents (the BNN of bnn_sgmcmc.py): one kernel launch of ours per update."""
    import zhusuan
    import zhusuan.mcmc
    from zhusuan.framework import BayesianNet

    class Net(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            self.normal("w0", mean=torch.zeros(50, 91, device=DEV), std=torch.ones(50, 91, device=DEV), n_samples=8,
                        group_ndims=2, reduce_mean_dims=[0])
            self.normal("w1", mean=torch.zeros(1, 51, device=DEV), std=torch.ones(1, 51, device=DEV), n_samples=8,
                        group_ndims=2, reduce_mean_dims=[0])
            return self

    net = Net(device=torch.device(DEV))
    sgld = zhusuan.mcmc.SGLD(learning_rate=1e-3)
    s0 = sgld.sample(net, {}, True)
    w0 = {k: v.clone() for k, v in s0.items()}
    n0 = be.launch_count
    s1 = sgld.sample(net, {}, False)
    launches = be.launch_count - n0
    # two log-density forward + two backward launches of the net's nodes, ONE update launch
    assert launches == 5, launches
    assert all(not torch.equal(s1[k], w0[k]) and s1[k].requires_grad and s1[k].is_leaf for k in s1)


# ----------------------------------------------------------------------------- product path: <= 4 launches, capturable
def _iwae_nets(K, B, Z, X, mean, std, probs, prior="cuda", vimco=False, use_first_draw=False):
    from zhusuan.distributions import Bernoulli, Normal
    from zhusuan.framework import BayesianNet
    d = torch.device(DEV)
    if prior == "cuda":
        pm, ps = torch.zeros(B, Z, device=DEV), torch.ones(B, Z, device=DEV)
    elif prior == "cpu":  # what examples/variational_autoencoder/iwae.py:60-61 builds every step
        pm, ps = torch.zeros(B, Z), torch.ones(B, Z)
    else:
        pm, ps = 0.0, 1.0
    half = torch.full((B, Z), 0.5, device=DEV)
    seen = {}

    class Gen(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            if vimco:
                self.bernoulli("z", probs=half, n_samples=K, reduce_sum_dims=[2])
            else:
                self.normal("z", mean=pm, std=ps, is_reparameterized=False, n_samples=K, reduce_sum_dims=[2])
            self.sn(Bernoulli(probs=probs), name="x", reduce_sum_dims=[2])
            return self

    class Var(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            if vimco:
                z = self.sn(Bernoulli(probs=mean), name="z", n_samples=K, reduce_sum_dims=[2])
            else:
                z = self.sn(Normal(mean=mean, std=std), name="z", n_samples=K, reduce_sum_dims=[2])
            seen["first"] = z
            if use_first_draw:
                seen["used"] = z * 2.0
            return self

    return Gen(device=d), Var(device=d), seen


def _leaves(K, B, Z, X, vimco=False, seed=0):
    g = torch.Generator(device=DEV).manual_seed(seed)
    rn = lambda *s: torch.randn(*s, device=DEV, generator=g)
    probs = torch.sigmoid(2 * rn(K, B, X)).requires_grad_()
    x = (torch.rand(B, X, device=DEV, generator=g) < 0.5).float()
    if vimco:
        return torch.sigmoid(rn(B, Z)).requires_grad_(), None, probs, x
    return (0.5 * rn(B, Z)).requires_grad_(), torch.exp(0.3 * rn(B, Z)).requires_grad_(), probs, x


@pytest.mark.parametrize("prior", ["cuda", "cpu", "scalar"])
@pytest.mark.parametrize("vimco", [False, True])
def test_api_step_is_at_most_four_launches(prior, vimco):
    """ImportanceWeightedObjective forward + backward through the public API on CUDA tensors: the draw with log q AND
    the standard prior's log p (one launch), the fused likelihood + objective (one), its upstream-gradient scaling
    (a no-op launch), the latent backward (one).  Draw #1 is never materialised; the prior node launches nothing."""
    from zhusuan.variational import ImportanceWeightedObjective
    K, B, Z, X = 50, 32, 40, 784
    mean, std, probs, x = _leaves(K, B, Z, X, vimco)
    gen, var, seen = _iwae_nets(K, B, Z, X, mean, std, probs, prior, vimco)
    obj = ImportanceWeightedObjective(gen, var, axis=0, estimator="vimco" if vimco else "sgvb")
    obj({"x": x}).backward()  # first sight of the prior tensors (one-time check of the CUDA ones)
    n0 = be.launch_count
    loss = obj({"x": x})
    loss.backward()
    assert be.launch_count - n0 <= 4, be.launch_count - n0
    assert isinstance(seen["first"], _ops.LazyDraw) and not seen["first"].materialized
    assert torch.isfinite(loss) and torch.isfinite(mean.grad).all() and torch.isfinite(probs.grad).all()


@pytest.mark.parametrize("vimco", [False, True])
def test_folded_prior_equals_separate_prior_launch(vimco):
    """Same injected noise, standard prior picked up from the latent launch vs evaluated by its own kernels: loss and
    every boundary gradient agree to float32 round-off of the two evaluation orders."""
    from zhusuan.variational import ImportanceWeightedObjective
    K, B, Z, X = 10, 16, 40, 128
    res = []
    for fold in (True, False):
        mean, std, probs, x = _leaves(K, B, Z, X, vimco, seed=3)
        gen, var, _ = _iwae_nets(K, B, Z, X, mean, std, probs, "cpu", vimco)
        obj = ImportanceWeightedObjective(gen, var, axis=0, estimator="vimco" if vimco else "sgvb")
        g = torch.Generator(device=DEV).manual_seed(11)
        noise = [torch.rand(K, B, Z, device=DEV, generator=g) if vimco else torch.randn(K, B, Z, device=DEV, generator=g)
                 for _ in range(2)]
        _ops.STD_PRIOR_FOLD = fold
        try:
            n0 = be.launch_count
            with _rng.inject(uniform=noise) if vimco else _rng.inject(normal=noise):
                loss = obj({"x": x})
            loss.backward()
            n = be.launch_count - n0
        finally:
            _ops.STD_PRIOR_FOLD = True
        res.append((loss.detach(), mean.grad.clone(), None if std is None else std.grad.clone(), probs.grad.clone(), n))
    (l1, m1, s1, p1, n1), (l2, m2, s2, p2, n2) = res
    assert n2 > n1  # the unfolded run pays for the prior node
    torch.testing.assert_close(l1, l2, rtol=1e-6, atol=0)
    torch.testing.assert_close(p1, p2, rtol=1e-5, atol=1e-5 * float(p2.abs().max()))
    torch.testing.assert_close(m1, m2, rtol=1e-5, atol=1e-5 * float(m2.abs().max()))
    if s1 is not None:
        torch.testing.assert_close(s1, s2, rtol=1e-5, atol=1e-5 * float(s2.abs().max()))


def test_nonstandard_prior_is_not_folded():
    from zhusuan.variational import ImportanceWeightedObjective
    from zhusuan.distributions import Bernoulli, Normal
    from zhusuan.framework import BayesianNet
    K, B, Z, X = 6, 8, 40, 128
    mean, std, probs, x = _leaves(K, B, Z, X)
    pm = torch.full((B, Z), 0.25, device=DEV)

    class Gen(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            self.normal("z", mean=pm, std=torch.ones(B, Z, device=DEV), n_samples=K, reduce_sum_dims=[2])
            self.sn(Bernoulli(probs=probs), name="x", reduce_sum_dims=[2])
            return self

    class Var(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            self.sn(Normal(mean=mean, std=std), name="z", n_samples=K, reduce_sum_dims=[2])
            return self

    obj = ImportanceWeightedObjective(Gen(device=torch.device(DEV)), Var(device=torch.device(DEV)), axis=0)
    eps = torch.randn(K, B, Z, device=DEV)
    with _rng.inject(normal=[eps, eps]):
        loss = obj({"x": x})
    z = mean.detach() + std.detach() * eps
    logp = torch.distributions.Normal(pm, 1.0).log_prob(z).sum(-1)
    logq = torch.distributions.Normal(mean.detach(), std.detach()).log_prob(z).sum(-1)
    p = probs.detach()
    logpx = (x * torch.log(p + 1e-8) + (1 - x) * torch.log(1 - p + 1e-8)).sum(-1)
    lw = logpx + logp - logq
    w = torch.softmax(lw, 0)
    torch.testing.assert_close(loss, -(w * lw).sum(0).mean(), rtol=1e-5, atol=0)


def test_first_draw_materialises_only_when_used():
    from zhusuan.variational import ImportanceWeightedObjective
    K, B, Z, X = 6, 8, 40, 128
    mean, std, probs, x = _leaves(K, B, Z, X)
    gen, var, seen = _iwae_nets(K, B, Z, X, mean, std, probs, use_first_draw=True)
    obj = ImportanceWeightedObjective(gen, var, axis=0)
    loss = obj({"x": x})
    first = seen["first"]
    assert isinstance(first, _ops.LazyDraw) and first.materialized
    assert seen["used"].shape == (K, B, Z) and seen["used"].is_cuda and not isinstance(seen["used"], _ops.LazyDraw)
    # draw #2 (what the objective used) is a different sample and stays the distribution's current value
    z2 = var.nodes["z"].dist.sample_cache
    assert not isinstance(z2, _ops.LazyDraw) and not torch.equal(z2, first._zs_real)
    loss.backward()
    # outside an objective, stochastic_node returns an ordinary tensor
    z = var({"x": x}).nodes["z"]
    assert not isinstance(seen["first"], _ops.LazyDraw)


@pytest.mark.parametrize("vimco", [False, True])
def test_public_api_step_captured_in_a_cuda_graph(vimco):
    """The whole public-API step (objective forward + loss.backward()) is capturable; replays draw new latents and
    reproduce the eager step's numbers for the same stream position."""
    from zhusuan.variational import ImportanceWeightedObjective
    K, B, Z, X = 50, 64, 40, 784
    mean, std, probs, x = _leaves(K, B, Z, X, vimco)
    gen, var, _ = _iwae_nets(K, B, Z, X, mean, std, probs, "cuda", vimco)
    obj = ImportanceWeightedObjective(gen, var, axis=0, estimator="vimco" if vimco else "sgvb")
    leaves = [t for t in (mean, std, probs) if t is not None]
    torch.manual_seed(5)

    def step():
        for t in leaves:
            t.grad = None
        loss = obj({"x": x})
        loss.backward()
        return loss

    # Everything runs on ONE side stream, as torch's CUDA-graph recipe does with its warm-up: autograd binds a leaf's
    # AccumulateGrad node to the stream it was first used on, the nets' node caches keep the previous step's graph
    # alive, and a backward captured on a different stream would have to synchronise with it (invalid during capture).
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        eager = []
        for _ in range(3):  # tick 0, 1, 2 of a freshly seeded stream
            loss = step()
            eager.append((loss.detach().clone(), mean.grad.clone(), var.nodes["z"].dist.sample_cache.detach().clone()))
        torch.manual_seed(5)
        step()  # warm-up outside capture: tick 0 (also re-initialises the device state from the generator)
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        n0 = be.launch_count
        with torch.cuda.graph(g, stream=s):
            loss = step()
        launches = be.launch_count - n0
    torch.cuda.current_stream().wait_stream(s)
    assert launches <= 4, launches
    z_static = var.nodes["z"].dist.sample_cache
    for i in (1, 2):
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(z_static, eager[i][2])
        torch.testing.assert_close(loss, eager[i][0], rtol=1e-6, atol=0)
        torch.testing.assert_close(mean.grad, eager[i][1], rtol=1e-5, atol=1e-6 * float(eager[i][1].abs().max()))


# ----------------------------------------------------------------------------- host-resident callers
def test_pinned_pool_never_hands_out_a_buffer_somebody_still_uses():
    a = _ops.pinned_like_pool((1 << 16,), torch.float32, "t")
    alias = a.view(256, 256)[3]  # a view keeps only the STORAGE alive
    del a
    b = _ops.pinned_like_pool((1 << 16,), torch.float32, "t")
    assert b.data_ptr() != alias.untyped_storage().data_ptr()
    del alias
    c = _ops.pinned_like_pool((1 << 16,), torch.float32, "t")  # now one of the two buffers is free again
    assert c.data_ptr() != b.data_ptr()


def test_host_resident_sgld_states_do_not_alias():
    """Two equal-shaped host-resident latents (>= 64 KB: the pooled pinned route) keep distinct storage across updates,
    and earlier returned samples are not overwritten by later steps (ADVICE round 1, high)."""
    import zhusuan
    import zhusuan.mcmc
    from zhusuan.framework import BayesianNet

    class Net(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            self.normal("a", mean=torch.zeros(128, 160), std=torch.ones(128, 160), n_samples=2, group_ndims=2,
                        reduce_mean_dims=[0])
            self.normal("b", mean=torch.ones(128, 160), std=torch.ones(128, 160), n_samples=2, group_ndims=2,
                        reduce_mean_dims=[0])
            return self

    net = Net()
    sgld = zhusuan.mcmc.SGLD(learning_rate=1e-4)
    sgld.sample(net, {}, True)
    s1 = sgld.sample(net, {}, False)
    a1, b1 = s1["a"], s1["b"]
    assert a1.device.type == "cpu" and a1.untyped_storage().data_ptr() != b1.untyped_storage().data_ptr()
    assert abs(float(a1.mean())) < 0.1 and abs(float(b1.mean()) - 1.0) < 0.1  # b did not overwrite a
    keep = a1.detach().clone()
    for _ in range(3):
        s = sgld.sample(net, {}, False)
    assert torch.equal(a1.detach(), keep)  # a collected posterior sample stays what it was
    assert not torch.equal(s["a"].detach(), keep)


def test_host_route_gradient_is_complete_when_a_cpu_decoder_reads_it():
    """probs produced by a CPU decoder: SigmoidBackward / AddmmBackward read dprobs DURING backward, so the host route
    must have landed it by then (ADVICE round 1, high).  Compared with the same model on the device."""
    from zhusuan.distributions import Bernoulli, Normal
    from zhusuan.framework import BayesianNet
    from zhusuan.variational import ImportanceWeightedObjective
    K, B, Z, X = 50, 256, 40, 784
    torch.manual_seed(0)
    lin = torch.nn.Linear(Z, X)
    x = (torch.rand(B, X) < 0.5).float()
    mean, std = 0.3 * torch.randn(B, Z), torch.exp(0.2 * torch.randn(B, Z))
    eps = torch.randn(K, B, Z)

    def run(device):
        d = torch.device(device)
        l = torch.nn.Linear(Z, X).to(d)
        l.load_state_dict(lin.state_dict())
        m, s_, xx = mean.to(d), std.to(d), x.to(d)

        class Gen(BayesianNet):
            def forward(self, observed):
                self.observe(observed)
                z = self.normal("z", mean=torch.zeros(B, Z, device=d), std=torch.ones(B, Z, device=d), n_samples=K,
                                is_reparameterized=False, reduce_sum_dims=[2])
                self.sn(Bernoulli(probs=torch.sigmoid(l(z))), name="x", reduce_sum_dims=[2])
                return self

        class Var(BayesianNet):
            def forward(self, observed):
                self.observe(observed)
                self.sn(Normal(mean=m, std=s_), name="z", n_samples=K, reduce_sum_dims=[2])
                return self

        obj = ImportanceWeightedObjective(Gen(device=d), Var(device=d), axis=0)
        out = []
        for _ in range(3):  # repeated steps: a pooled buffer would hold the previous step's gradient
            l.zero_grad()
            with _rng.inject(normal=[eps.to(d), eps.to(d)]):
                loss = obj({"x": xx})
            loss.backward()
            out.append((float(loss), l.weight.grad.detach().cpu().clone()))
        return out

    ref, got = run("cuda"), run("cpu")
    for (lr_, gr), (lg, gg) in zip(ref, got):
        assert abs(lr_ - lg) <= 1e-5 * abs(lr_)
        torch.testing.assert_close(gg, gr, rtol=2e-4, atol=2e-4 * float(gr.abs().max()))


def test_cpu_sample_keeps_its_autograd_connection():
    """ADVICE round 1 (low): a reparameterised sample returned on the CPU stays a differentiable input of later ops."""
    from zhusuan.distributions import Normal
    mean = torch.zeros(64, 512, requires_grad=True)  # 128 KB: the pinned return route
    q = Normal(mean=mean, std=torch.ones(64, 512))
    z = q.sample(2)
    lp = Normal(mean=torch.zeros(64, 512), std=torch.ones(64, 512)).log_prob(z)
    (gz,) = torch.autograd.grad(lp.sum(), z)
    torch.testing.assert_close(gz, -z.detach())


def test_gradient_bucket_zeroing_in_line_and_overlapped():
    """GradientBucket on one GPU (no process group: the collectives are local no-ops): `.grad` tensors are views of the
    flat buffer, zero_grad() in line and zero_grad(overlap=True) (memset on the side stream, joined by the parameters'
    tensor hook before the first accumulation) both leave exactly this step's gradients in the buffer, step after step;
    finish(loss) puts the objective into the bucket's last slot."""
    import zhusuan.distributed as zd
    torch.manual_seed(3)
    lin = torch.nn.Sequential(torch.nn.Linear(64, 48), torch.nn.Tanh(), torch.nn.Linear(48, 7)).to(DEV)
    bucket = zd.GradientBucket([lin.parameters()])
    assert bucket.backend == "local"
    assert all(p.grad.untyped_storage().data_ptr() == bucket.flat.untyped_storage().data_ptr() for p in lin.parameters())
    for step, overlap in enumerate((True, False, True, True)):
        x = torch.randn(16, 64, device=DEV)
        bucket.zero_grad(overlap=overlap)
        loss = lin(x).square().mean()
        loss.backward()
        bucket.finish(loss)
        torch.cuda.synchronize()
        ref = torch.autograd.grad(lin(x).square().mean(), list(lin.parameters()))
        for p, r in zip(lin.parameters(), ref):
            torch.testing.assert_close(p.grad, r, rtol=1e-5, atol=1e-7)
        torch.testing.assert_close(bucket.loss(), loss.detach(), rtol=0, atol=0)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_operands_on_a_non_current_device():
    """ADVICE round 1 (medium): tensors on cuda:1 while cuda:0 is current launch on cuda:1's stream."""
    from zhusuan.distributions import Normal
    torch.cuda.set_device(0)
    d1 = torch.device("cuda", 1)
    mean, std = torch.zeros(16, 40, device=d1), torch.ones(16, 40, device=d1)
    z = Normal(mean=mean, std=std).sample(4)
    assert z.device == d1 and torch.isfinite(z).all() and torch.cuda.current_device() == 0
    lp = Normal(mean=mean, std=std, group_ndims=1).log_prob(z)
    ref = torch.distributions.Normal(mean, std).log_prob(z).sum(-1)
    torch.testing.assert_close(lp, ref, rtol=1e-5, atol=1e-4)
    with pytest.raises(be.BackendError):
        be.normal_logprob_fwd(z.reshape(4, -1), be.FULL, mean.to("cuda:0").reshape(-1), KBCAST, std.reshape(-1), KBCAST,
                              4, 16, 40)


def test_fused_objective_takes_an_unaligned_view():
    """ADVICE round 1 (low): a contiguous but not 16-byte aligned probs view is realigned, not refused."""
    from zhusuan import _backend
    K, B, X = 8, 4, 128
    buf = torch.rand(K * B * X + 1, device=DEV) * 0.9 + 0.05
    probs = buf[1:].view(K, B, X).requires_grad_()
    assert probs.data_ptr() % 16 != 0
    x = (torch.rand(B, X, device=DEV) < 0.5).float()
    loss = _ops.iw_bernoulli_fused(probs, x, None, None, _backend.SGVB)
    loss.backward()
    ref = _ops.iw_bernoulli_fused(probs.detach().clone(), x, None, None, _backend.SGVB)
    torch.testing.assert_close(loss, ref)


# ----------------------------------------------------------------------------- parity at benchmark row sizes
def _bench_size_case(cname, est, latent, use_logits, dtype=torch.float32):
    """Run one case of tests/golden/bench_size.npz through the PUBLIC API on CUDA; returns dict(loss, dbig, da, db)."""
    import importlib.util
    import os
    from zhusuan.distributions import Bernoulli, Normal
    from zhusuan.framework import BayesianNet
    from zhusuan.variational import ImportanceWeightedObjective
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "make_golden_bench.py")
    spec = importlib.util.spec_from_file_location("make_golden_bench", here)
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    inp = mg.inputs()
    K, B, Z, X = mg.K, mg.B, mg.Z, mg.X
    t = lambda a, grad=False: torch.tensor(a, dtype=dtype, device=DEV).requires_grad_(grad)
    big = t(inp["logits"] if use_logits else inp["probs"], True)
    a = t(inp["mean"] if latent == "normal" else inp["probs_q"], True)
    b = t(inp["logstd"], True) if latent == "normal" else None
    x = t(inp["x"])
    d = torch.device(DEV)

    class Gen(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            if latent == "normal":
                self.normal("z", mean=torch.zeros(B, Z, dtype=dtype), std=torch.ones(B, Z, dtype=dtype),
                            is_reparameterized=False, n_samples=K, reduce_sum_dims=[2])
            else:
                self.bernoulli("z", probs=0.5 * torch.ones(B, Z, dtype=dtype), n_samples=K, reduce_sum_dims=[2])
            self.sn(Bernoulli(logits=big) if use_logits else Bernoulli(probs=big), name="x", reduce_sum_dims=[2])
            return self

    class Var(BayesianNet):
        def forward(self, observed):
            self.observe(observed)
            if latent == "normal":
                self.sn(Normal(mean=a, logstd=b, is_reparameterized=(est == "sgvb")), name="z", n_samples=K,
                        reduce_sum_dims=[2])
            else:
                self.sn(Bernoulli(probs=a), name="z", n_samples=K, reduce_sum_dims=[2])
            return self

    obj = ImportanceWeightedObjective(Gen(device=d), Var(device=d), axis=0, estimator=est)
    eps, u = t(inp["eps"]), t(inp["u"])
    # the reference protocol consumes two draws per step; both replay the recorded noise
    with _rng.inject(normal=[eps, eps], uniform=[u, u]):
        n0 = be.launch_count
        loss = obj({"x": x})
    grads = torch.autograd.grad(loss, [big, a] + ([b] if b is not None else []))
    return dict(loss=loss.detach(), dbig=grads[0], da=grads[1], db=grads[2] if b is not None else None,
                launches=be.launch_count - n0, F64_COLS=mg.F64_COLS, dbig_mask=mg.dbig_mask)


def _dist(a, ref):
    a, ref = np.asarray(a, np.float64), np.asarray(ref, np.float64)
    return (float(np.abs(a - ref).max() / max(np.abs(ref).max(), 1e-300)),
            float(np.linalg.norm(a - ref) / max(np.linalg.norm(ref), 1e-300)))


def _dbig_vs_fixture(r, g, p):
    """Distances of the big gradient r["dbig"] [K, B, X] from the fixture's samples of the reference's float32 run and
    of the first F64_COLS batch columns of its float64 run (tests/golden/make_golden_bench.py)."""
    got = host(r["dbig"])
    out = []
    for tag, a in (("f32_dbig", got), ("f64_dbig_cols", got[:, :r["F64_COLS"]])):
        out.append(_dist(a[r["dbig_mask"](a.shape, g[p + tag + "_rows"])], g[p + tag + "_sample"]))
    return out


@pytest.mark.parametrize("cname,est,latent,use_logits", [("sgvb_normal", "sgvb", "normal", False),
                                                         ("vimco_bernoulli", "vimco", "bernoulli", False),
                                                         ("sgvb_normal_logits", "sgvb", "normal", True)])
def test_reference_fixture_at_benchmark_row_sizes(golden, cname, est, latent, use_logits):
    """K = 50, X = 784: the shipped default kernel (boxf<., 28, 7, .>) through the public API against the REAL
    reference.  Values: 1e-5 relative.  Gradients: north_star's 1e-5 normwise against the reference's float32 run where
    float32 allows it; in any case no farther from the reference's float64 run than 3x the distance of the reference's
    OWN float32 run from it (the recorded budget), i.e. inside the reference's float32 noise.  The big gradient is
    compared on the fixture's sample of it: the particle rows that carry it and a seeded sixteenth of the others."""
    g = golden("bench_size")
    r = _bench_size_case(cname, est, latent, use_logits)
    p = cname + "_"
    assert abs(float(r["loss"]) - float(g[p + "f32_loss"])) <= 1e-5 * abs(float(g[p + "f32_loss"]))
    assert abs(float(r["loss"]) - float(g[p + "f64_loss"])) <= 1e-5 * abs(float(g[p + "f64_loss"]))
    for key, got, f64 in (("dbig", r["dbig"], None), ("da", r["da"], g[p + "f64_da"]),
                          ("db", r["db"], g[p + "f64_db"] if p + "f64_db" in g.files else None)):
        if got is None:
            continue
        if key == "dbig":
            vs32, vs64 = _dbig_vs_fixture(r, g, p)
        else:
            got = host(got)
            vs32, vs64 = _dist(got, g[p + "f32_" + key]), _dist(got, f64)
        budget = g["budget_" + p + key]
        assert vs32[0] <= 4e-5, (key, "vs reference float32, max-norm", vs32)
        assert vs64[0] <= max(3.0 * float(budget[0]), 1e-5), (key, "vs reference float64", vs64, "budget", budget)
        assert vs64[1] <= max(3.0 * float(budget[1]), 1e-5), (key, "vs reference float64 rel-L2", vs64, "budget", budget)
