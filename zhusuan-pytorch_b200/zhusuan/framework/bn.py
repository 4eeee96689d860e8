"""BayesianNet — the node registry users subclass (drop-in for zhusuan/framework/bn.py).

Same attributes (`_nodes`, `_cache`, `_observed`, `_device`), properties and methods as the
reference (:72-240): `observe`, `stochastic_node` / `sn` / `snode`, the per-distribution aliases of
the hot-path distributions, `log_joint` / `_log_joint`.  Normal, Bernoulli, Categorical, Logistic, Laplace,
Uniform, Poisson and Beta are registered: the other aliases of the reference (gamma, exponential, studentT) wrap
torch.distributions and are outside the accelerated path.
"""
import torch
import torch.nn as nn

from zhusuan.framework.stochastic_tensor import StochasticTensor
from zhusuan.distributions import Distribution, Normal, Bernoulli, Categorical, Logistic, Laplace, Uniform, Poisson, Beta

__all__ = ['BayesianNet']

name_mapping = {
    "Normal": Normal,
    "Bernoulli": Bernoulli,
    "Categorical": Categorical,
    "Logistic": Logistic,
    "Laplace": Laplace,
    "Uniform": Uniform,
    "Poisson": Poisson,
    "Beta": Beta,
}

_OUT_OF_SCOPE = ("Exponential", "Gamma", "StudentT")


class BayesianNet(nn.Module):
    def __init__(self, observed=None, device=torch.device('cpu')):
        super(BayesianNet, self).__init__()
        self._nodes = {}
        self._cache = {}
        self._observed = observed if observed else {}
        self._device = device

    # -- registries -----------------------------------------------------------------------------
    @property
    def nodes(self):
        return self._nodes

    @property
    def cache(self):
        return self._cache

    @property
    def observed(self):
        return self._observed

    @property
    def device(self):
        """Device of the module's parameters, else the device given at construction / `.to()`."""
        for p in self.parameters():
            return p.device
        return self._device

    def to(self, device):
        self._device = device
        return super().to(device)

    def observe(self, observed):
        self._observed = {}
        for k, v in observed.items():
            self._observed[k] = v
        return self

    # -- node construction ----------------------------------------------------------------------
    def _register(self, name, distribution, n_samples, kwargs):
        if not isinstance(name, str):
            raise ValueError("name of stochastic_node must be str")
        self._nodes[name] = StochasticTensor(self, name, distribution, n_samples=n_samples, **kwargs)
        return self._nodes[name].first_draw()

    def stochastic_node(self, distribution, name, n_samples=None, **kwargs):
        """Add node `name` following `distribution` (a registered name or a Distribution instance)
        and return its value: the observation if `name` is observed, else a fresh sample."""
        if isinstance(distribution, str):
            if distribution not in name_mapping:
                if distribution in _OUT_OF_SCOPE:
                    raise NotImplementedError("%s is outside the B200 hot path (registered: %s)"
                                              % (distribution, ", ".join(name_mapping)))
                raise KeyError(distribution)
            dist = name_mapping[distribution](device=self.device, **kwargs)
        elif isinstance(distribution, Distribution):
            distribution._device = self.device
            dist = distribution
        else:
            raise ValueError('distribution must be name of sub class of Distribution or an instance of Distribution')
        return self._register(name, dist, n_samples, kwargs)

    def sn(self, dist, name, n_samples=None, **kwargs):
        return self.stochastic_node(dist, name, n_samples, **kwargs)

    def snode(self, *args, **kwargs):
        return self.stochastic_node(*args, **kwargs)

    def normal(self, name, mean=0., std=None, logstd=None, dtype=None, is_continuous=True, is_reparameterized=True,
               group_ndims=0, n_samples=None, **kwargs):
        if not isinstance(name, str):
            raise ValueError("name of stochastic_node must be str")
        dist = Normal(mean=mean, std=std, logstd=logstd, dtype=dtype, is_continuous=is_continuous,
                      is_reparameterized=is_reparameterized, group_ndims=group_ndims, device=self.device, **kwargs)
        return self._register(name, dist, n_samples, kwargs)

    def bernoulli(self, name, logits=None, probs=None, dtype=None, is_continuous=False, group_ndims=0,
                  n_samples=None, **kwargs):
        if not isinstance(name, str):
            raise ValueError("name of stochastic_node must be str")
        dist = Bernoulli(logits=logits, probs=probs, dtype=dtype, is_continuous=is_continuous,
                         group_ndims=group_ndims, device=self.device, **kwargs)
        return self._register(name, dist, n_samples, kwargs)

    def categorical(self, name, logits=None, probs=None, dtype=None, is_continuous=False, group_ndims=0,
                    n_samples=None, **kwargs):
        if not isinstance(name, str):
            raise ValueError("name of stochastic_node must be str")
        dist = Categorical(logits=logits, probs=probs, dtype=dtype, is_continuous=is_continuous,
                           group_ndims=group_ndims, device=self.device, **kwargs)
        return self._register(name, dist, n_samples, kwargs)

    def poisson(self, name, rate, dtype=None, is_continuous=False, group_ndims=0, n_samples=None, **kwargs):
        if not isinstance(name, str):
            raise ValueError("name of stochastic_node must be str")
        dist = Poisson(rate=rate, dtype=dtype, is_continuous=is_continuous, group_ndims=group_ndims,
                       device=self.device, **kwargs)
        return self._register(name, dist, n_samples, kwargs)

    def beta(self, name, alpha, beta, dtype=None, is_continuous=True, group_ndims=0, n_samples=None, **kwargs):
        if not isinstance(name, str):
            raise ValueError("name of stochastic_node must be str")
        dist = Beta(alpha=alpha, beta=beta, dtype=dtype, is_continuous=is_continuous, group_ndims=group_ndims,
                    device=self.device, **kwargs)
        return self._register(name, dist, n_samples, kwargs)

    def laplace(self, name, loc, scale, dtype=None, is_continuous=True, group_ndims=0, n_samples=None, **kwargs):
        if not isinstance(name, str):
            raise ValueError("name of stochastic_node must be str")
        dist = Laplace(loc=loc, scale=scale, dtype=dtype, is_continuous=is_continuous, group_ndims=group_ndims,
                       device=self.device, **kwargs)
        return self._register(name, dist, n_samples, kwargs)

    def uniform(self, name, low, high, dtype=None, is_continuous=True, is_reparameterized=True, group_ndims=0,
                n_samples=None, **kwargs):
        if not isinstance(name, str):
            raise ValueError("name of stochastic_node must be str")
        dist = Uniform(low=low, high=high, dtype=dtype, is_continuous=is_continuous,
                       is_reparameterized=is_reparameterized, group_ndims=group_ndims, device=self.device, **kwargs)
        return self._register(name, dist, n_samples, kwargs)

    def logistic(self, name, loc, scale, dtype=None, is_continuous=True, group_ndims=0, n_samples=None, **kwargs):
        """As in the reference, `bn.logistic` builds a LAPLACE node (framework/bn.py:336-352 constructs
        `Laplace(...)`; SURVEY Q16).  Use `bn.sn(Logistic(...), name)` for a Logistic node."""
        if not isinstance(name, str):
            raise ValueError("name of stochastic_node must be str")
        dist = Laplace(loc=loc, scale=scale, dtype=dtype, is_continuous=is_continuous, group_ndims=group_ndims,
                       device=self.device, **kwargs)
        return self._register(name, dist, n_samples, kwargs)

    # -- log joint ------------------------------------------------------------------------------
    def _log_joint(self):
        """Sum of the conditional log-probabilities of all StochasticTensor nodes at their current
        values.  Users may override this (test/mcmc/test_mcmc.py:33-37 of the reference does)."""
        total = 0
        for node in self._nodes.values():
            if isinstance(node, StochasticTensor):
                lp = node.log_prob()
                try:
                    total = total + lp
                except Exception:
                    total = lp
        return total

    def log_joint(self, use_cache=False):
        if use_cache:
            if not hasattr(self, '_log_joint_cache'):
                self._log_joint_cache = self._log_joint()
        else:
            self._log_joint_cache = self._log_joint()
        return self._log_joint_cache
