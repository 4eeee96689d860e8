"""Importance-weighted objective (IWAE bound) with the SGVB and VIMCO estimators — drop-in for
zhusuan/variational/importance_weighted_objective.py of the reference.

Both estimators run as ONE kernel over the [K,B] log-weights that produces the surrogate cost and
its gradient (the reference launches ~40 aten kernels and, for VIMCO, materialises a [B,K,K] tensor,
:164-191).  When the generator's likelihood is a Bernoulli node over [K,B,X] probabilities, the
likelihood log-pmf, the objective and the likelihood's backward are fused further into the
resident-column kernel (zs_iw_bernoulli_fused): probs is read from HBM once, dprobs written once.  A Poisson
likelihood over [K,B,X] rates takes the same kernel's Poisson form (zs_iw_poisson_fused).
"""
import torch
from zhusuan._shapes import broadcast_shapes as _bshapes
import torch.nn as nn

from zhusuan.framework.stochastic_tensor import StochasticTensor
from zhusuan.distributions.bernoulli import Bernoulli
from zhusuan.distributions.poisson import Poisson
from zhusuan import _ops
from zhusuan import _backend as _be

__all__ = [
    'iw_objective',
    'ImportanceWeightedObjective',
    'compute_iw_term',
]


def compute_iw_term(x, axis):
    """sum_k wt_k * x_k with wt = softmax(x, axis) detached (reference :16-25): its value is the
    self-normalised average of log w and its gradient the IWAE gradient."""
    x = torch.as_tensor(x)
    return -_ops.iw_objective(x, torch.zeros_like(x), axis, _be.SGVB, False)


class ImportanceWeightedObjective(nn.Module):
    def __init__(self, generator, variational, axis=None, estimator='sgvb'):
        super().__init__()
        self.generator = generator
        self.variational = variational
        if axis is None:
            raise ValueError("ImportanceWeightedObjective is a multi-sample objective, "
                             "the `axis` argument must be specified.")
        self._axis = axis
        if estimator not in ('sgvb', 'vimco'):
            raise NotImplementedError()
        self.estimator = estimator

    def log_joint(self, nodes):
        """Sum of `node.log_prob()` over `nodes`; a term that cannot be added in place replaces the
        running sum, as in the reference (:66-77)."""
        total = None
        for name in nodes.keys():
            lp = nodes[name].log_prob()
            try:
                total = total + lp
            except Exception:
                total = lp
        return total

    # -- fused path -----------------------------------------------------------------------------
    def _fusable_likelihood(self, nodes_p):
        """Name of a generator node that is an observed Bernoulli likelihood over [K,B,X] probabilities, or an observed
        Poisson likelihood over device-resident [K,B,X] rates, whose only reduction is the sum over X — the shape the
        fused kernel handles — else None."""
        from zhusuan import variational as _v
        if not _v.FUSED or self._axis != 0:
            return None
        best, best_numel = None, 0
        for name, node in nodes_p.items():
            if not isinstance(node, StochasticTensor) or not isinstance(node.dist, (Bernoulli, Poisson)):
                continue
            poisson = isinstance(node.dist, Poisson)
            logits = None if poisson else node.dist.from_logits
            probs = node.dist.rate if poisson else (node.dist.probs if logits is None else logits)  # [K,B,X] operand
            x = node._observed_value()
            if x is None or not torch.is_tensor(x) or probs.dim() != 3:
                continue
            if not _be.on_compute_device(probs) and not (probs.device.type == 'cpu' and torch.cuda.is_available()):
                continue
            if tuple(x.shape) != tuple(probs.shape[1:]) or x.requires_grad or node._multiplier:
                continue
            n_event, mean_dims, sum_dims = node.reduction_plan(x.shape)
            if n_event != 1 or mean_dims or sum_dims:
                continue
            if poisson:
                # device-resident rates only (host-resident ones take the generic path), instantiated row lengths
                if not _be.on_compute_device(probs) or not _be.fused_poisson_supported(
                        int(probs.shape[0]), int(probs.shape[2]), probs.dtype):
                    continue
            elif logits is not None:
                # the logits form exists on the device-resident route, for the instantiated row lengths
                if not _be.on_compute_device(probs) or not _be.fused_logits_supported(
                        int(probs.shape[0]), int(probs.shape[2]), probs.dtype):
                    continue
            elif not _be.fused_supported(int(probs.shape[0]), int(probs.shape[2]), probs.dtype):
                continue
            if best is None or probs.numel() > best_numel:
                best, best_numel = name, probs.numel()
        return best

    def _forward_fused(self, nodes_p, nodes_q, lik):
        node = nodes_p[lik]
        poisson = isinstance(node.dist, Poisson)
        logits = None if poisson else node.dist.from_logits
        probs = node.dist.rate if poisson else (node.dist.probs if logits is None else logits)
        K, B = int(probs.shape[0]), int(probs.shape[1])
        x = node._observed_value()
        node.dist.sample_cache = x

        def kb_sum(nodes, skip=None):
            total = None
            for name in nodes.keys():
                if name == skip:
                    continue
                lp = nodes[name].log_prob()
                if not torch.is_tensor(lp) or tuple(lp.shape) != (K, B):
                    return False
                total = lp if total is None else total + lp
            return total

        host_route = not _be.on_compute_device(probs)
        if host_route:
            # the [K,B] terms are consumed by the kernel only: keep them (and their gradients) on the device
            with _ops.device_results():
                logp_other = kb_sum(nodes_p, skip=lik)
                logq = kb_sum(nodes_q)
        else:
            logp_other = kb_sum(nodes_p, skip=lik)
            logq = kb_sum(nodes_q)
        if logp_other is False or logq is False:
            return None
        if self.estimator == 'vimco' and logq is None:
            return None
        est = _be.SGVB if self.estimator == 'sgvb' else _be.VIMCO
        dev = probs.device
        if host_route:
            # host-resident likelihood tensor: chunk-pipelined H2D / kernel / D2H (zs_iw_step_host_begin)
            return _ops.iw_bernoulli_fused_host(probs, x.to(dev), logp_other, logq, est)
        lo = None if logp_other is None else logp_other.to(dev, probs.dtype)
        lq = None if logq is None else logq.to(dev, probs.dtype)
        if poisson:
            return _ops.iw_poisson_fused(probs, x.to(dev), lo, lq, est)
        return _ops.iw_bernoulli_fused(probs, x.to(dev), lo, lq, est, logits=logits is not None)

    # -- reference protocol ---------------------------------------------------------------------
    def forward(self, observed, reduce_mean=True):
        # host-resident parameters cross PCIe once per step; large host-bound results (the latent samples of a
        # host-resident model) are copied back only if host code reads them
        with _ops.upload_memo(), _ops.lazy_host_results():
            return self._forward(observed, reduce_mean)

    def _forward(self, observed, reduce_mean=True):
        # draw #1 of every latent (what stochastic_node returns to the variational net's forward) is deferred until
        # that forward uses it; the draw both nets see is the `.tensor` read below, as in the reference (:85)
        with _ops.lazy_first_draws():
            self.variational(observed)
        nodes_q = self.variational.nodes
        latents = {}
        for k, v in nodes_q.items():
            latents[k] = v.tensor
            if self.estimator == "vimco" and isinstance(v, StochasticTensor) and v.dist.is_reparameterized:
                raise ValueError("with vimco estimator, the is_reparameterized must be false")
        nodes_p = self.generator({**latents, **observed}).nodes

        # VIMCO always averages over the batch (:190-191); SGVB only with reduce_mean
        if reduce_mean or self.estimator == 'vimco':
            lik = self._fusable_likelihood(nodes_p)
            if lik is not None:
                loss = self._forward_fused(nodes_p, nodes_q, lik)
                if loss is not None:
                    return loss

        logpxz = self.log_joint(nodes_p)
        logqz = self.log_joint(nodes_q)
        if self.estimator == 'sgvb':
            return self.sgvb(logpxz, logqz, reduce_mean)
        return self.vimco(logpxz, logqz, reduce_mean)

    def sgvb(self, logpxz, logqz, reduce_mean=True):
        """IWAE bound with the pathwise gradient: mean_b( -sum_k wt_kb log w_kb ) (:102-132)."""
        logpxz, logqz = _as_pair(logpxz, logqz)
        return _ops.iw_objective(logpxz, logqz, self._axis, _be.SGVB, reduce_mean)

    def vimco(self, logpxz, logqz, reduce_mean=True):
        """VIMCO (Mnih & Rezende 2016): score-function gradient with the leave-one-out control
        variate whose baseline replaces particle k by the geometric mean of the others (:134-191).
        `reduce_mean` is ignored — the reference always returns the batch mean (:191)."""
        logpxz, logqz = _as_pair(logpxz, logqz)
        err_msg = "VIMCO is a multi-sample gradient estimator, size along " \
                  "`axis` in the objective should be larger than 1."
        shape = tuple(_bshapes(logpxz.shape, logqz.shape))
        try:
            if shape[self._axis] < 2:
                raise ValueError(err_msg)
        except IndexError:
            raise ValueError(err_msg)
        return _ops.iw_objective(logpxz, logqz, self._axis, _be.VIMCO, True)


def _as_pair(logpxz, logqz):
    logqz = torch.as_tensor(logqz)
    logpxz = torch.as_tensor(logpxz, dtype=logqz.dtype if not torch.is_tensor(logpxz) else None)
    if logpxz.dtype != logqz.dtype:
        dt = torch.promote_types(logpxz.dtype, logqz.dtype)
        logpxz, logqz = logpxz.to(dt), logqz.to(dt)
    if logpxz.device != logqz.device:
        logqz = logqz.to(logpxz.device)
    return logpxz, logqz


iw_objective = 'ImportanceWeightedObjective',
