"""Univariate Beta — drop-in for zhusuan/distributions/beta.py of the reference.

The reference wraps torch.distributions.Beta (sample, log_prob).  Here log_prob is
xlogy(alpha - 1, x) + xlogy(beta - 1, 1 - x) + lgamma(alpha + beta) - (lgamma(alpha) + lgamma(beta)) with the
event-axis sum fused into one kernel (the location-scale log-density entry points with alpha as loc and beta as
scale), and samples are drawn in-kernel as torch's CPU Dirichlet sampler draws them: two Marsaglia-Tsang gamma
variates, G_alpha / (G_alpha + G_beta), clamped into (0, 1).  Never reparameterised: like the reference's `.sample()`,
a sample carries no gradient.  Gradients of log_prob reach x, alpha and beta.

Nothing is validated on the device: torch.distributions with validate_args rejects non-positive parameters and values
outside [0, 1], which would need a host synchronisation here (DESIGN.md §1).
"""
import torch

from zhusuan._shapes import broadcast_shapes as _bshapes
from zhusuan.distributions.base import Distribution, DEFAULT_DEVICE, resolve_device
from zhusuan.distributions.utils import assert_same_log_float_dtype, check_broadcast
from zhusuan import _ops, _backend as _be

__all__ = ['Beta']


class Beta(Distribution):
    """Beta(alpha, beta) on (0, 1); `batch_shape` is the broadcast shape of `alpha` and `beta`."""

    def __init__(self, alpha, beta, dtype=None, is_continuous=True, group_ndims=0, device=DEFAULT_DEVICE, **kwargs):
        device = resolve_device(device, alpha, beta)
        self._alpha = torch.as_tensor(alpha, dtype=dtype).to(device)
        self._beta = torch.as_tensor(beta, dtype=dtype).to(device)
        check_broadcast(self._alpha, self._beta)
        dtype = assert_same_log_float_dtype([(self._alpha, "Beta.alpha"), (self._beta, "Beta.beta")])
        super(Beta, self).__init__(dtype, is_continuous, is_reparameterized=False, group_ndims=group_ndims,
                                   device=device, **kwargs)

    @property
    def alpha(self):
        return self._alpha

    @property
    def beta(self):
        return self._beta

    def _batch_shape(self):
        return _bshapes(self._alpha.shape, self._beta.shape)

    def sample_device(self):
        return self._alpha.device

    def _sample(self, n_samples=1, **kwargs):
        s = _ops.beta_sample(self._alpha, self._beta, n_samples)
        self.sample_cache = s
        return s

    def _log_prob_event(self, given, n_event):
        return _ops.locscale_log_prob(_be.FAM_BETA, self._given(given), self._alpha, self._beta, n_event)

    def _log_prob(self, sample=None):
        return self._log_prob_event(sample, 0)

    def _prob(self, given):
        return torch.exp(self._log_prob(given))
