"""Univariate Poisson — drop-in for zhusuan/distributions/poisson.py of the reference.

The reference wraps torch.distributions.Poisson (:61 sample, :75 log_prob).  Here log_prob is
xlogy(x, rate) - rate - lgamma(x + 1) with the event-axis sum fused into one kernel, and samples are
float counts drawn in-kernel from Philox uniforms (Knuth below rate 10, transformed rejection above, as
torch's CPU sampler).  Never reparameterised; the counts carry no gradient.

Nothing is validated on the device: torch.distributions with validate_args rejects negative rates and
non-integer counts, which would need a host synchronisation here (DESIGN.md §1).
"""
import torch

from zhusuan.distributions.base import Distribution, DEFAULT_DEVICE, resolve_device
from zhusuan.distributions.utils import assert_same_log_float_dtype
from zhusuan import _ops

__all__ = ['Poisson']


class Poisson(Distribution):
    """Poisson(rate): counts with mean and variance `rate`; `batch_shape == rate.shape`."""

    def __init__(self, rate, dtype=None, is_continuous=False, group_ndims=0, device=DEFAULT_DEVICE, **kwargs):
        device = resolve_device(device, rate)
        self._rate = torch.as_tensor(rate, dtype=dtype).to(device)
        dtype = assert_same_log_float_dtype([(self._rate, "Poisson.rate")])
        self._lograte = None  # built on first use: nothing on the hot path reads it
        super(Poisson, self).__init__(dtype, is_continuous, is_reparameterized=False, group_ndims=group_ndims,
                                      device=device, **kwargs)

    @property
    def rate(self):
        return self._rate

    @property
    def lograte(self):
        if self._lograte is None:
            self._lograte = torch.log(self._rate)
        return self._lograte

    def _batch_shape(self):
        return self._rate.shape

    def sample_device(self):
        return self._rate.device

    def _sample(self, n_samples=1, **kwargs):
        s = _ops.poisson_sample(self._rate, n_samples)
        self.sample_cache = s
        return s

    def _log_prob_event(self, given, n_event):
        return _ops.poisson_log_prob(self._given(given), self._rate, n_event)

    def _log_prob(self, sample=None):
        return self._log_prob_event(sample, 0)

    def _prob(self, given):
        return torch.exp(self._log_prob(given))
