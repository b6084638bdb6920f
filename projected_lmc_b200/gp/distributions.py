"""Minimal distribution objects returned by the model (no gpytorch dependency)."""
from __future__ import annotations

import torch

from . import settings


class Distribution:
    pass


class MultivariateNormal(Distribution):
    """Train-mode handle returned by ``model(X)``: the batched latent prior N(0, K_l).

    Like gpytorch's lazy ``MultivariateNormal(mean, LazyEvaluatedKernelTensor)`` it
    computes nothing; the MLL hands it to the CUDA engine (projected_lmc.py:1130-1131)."""

    def __init__(self, model, x, noise_likelihood=None):
        self.model = model
        self.x = x
        self.noise_likelihood = noise_likelihood

    def with_noise(self, likelihood):
        return MultivariateNormal(self.model, self.x, likelihood)

    @property
    def batch_shape(self):
        return torch.Size([self.model.n_latents])

    @property
    def event_shape(self):
        return torch.Size([self.x.shape[-2]])

    @property
    def mean(self):
        return torch.zeros(self.model.n_latents, self.x.shape[-2], dtype=self.x.dtype, device=self.x.device)

    def log_prob(self, value):
        if self.noise_likelihood is None:
            raise RuntimeError("log_prob of the noise-free latent prior is not defined; call likelihood(dist) first")
        return self.model._latent_log_prob(value)


class MultitaskMultivariateNormal(Distribution):
    """Eval-mode result: task means [n*, p] and marginal variances [n*, p], computed eagerly.

    The reference builds the full (n* p) x (n* p) covariance as a dense Kronecker sum
    (projected_lmc.py:1149-1155).  Here everything joint is lazy: ``covariance_matrix``,
    ``rsample`` / ``sample`` and ``log_prob`` are computed on first use from the latent
    structure (``joint``: the model's _JointPosterior for these test points) with the
    task-level noise ``task_noise`` [p, p] (eps I, + F F^T after full_likelihood)."""

    def __init__(self, mean, variance, joint=None, task_noise=None):
        self._mean = mean
        self._var = variance
        self._joint = joint
        self._task_noise = task_noise
        self._covar = None

    @property
    def mean(self):
        return self._mean

    @property
    def variance(self):
        return self._var.clamp_min(settings.min_variance.value())

    @property
    def stddev(self):
        return self.variance.sqrt()

    def confidence_region(self):
        s2 = self.stddev * 2
        return self.mean - s2, self.mean + s2

    def add_task_noise(self, task_covar):
        """The posterior with I (x) task_covar [p, p] added to its covariance."""
        noise = None
        if self._task_noise is not None:
            noise = self._task_noise + task_covar.detach().to(self._task_noise.dtype)
        return MultitaskMultivariateNormal(self._mean, self._var + task_covar.diagonal()[None, :], self._joint, noise)

    def _joint_or_raise(self):
        if self._joint is None:
            raise NotImplementedError("this distribution carries marginal variances only")
        return self._joint

    @property
    def covariance_matrix(self):
        """Dense [n* p, n* p] covariance, point-major / task-minor (computed on first access)."""
        if self._covar is None:
            self._covar = self._joint_or_raise().task_covariance(self._task_noise)
        return self._covar

    def rsample(self, sample_shape=torch.Size(), base_samples=None):
        """Posterior draws [*sample_shape, n*, p]; the normals come from torch's CUDA generator."""
        if base_samples is not None:
            raise NotImplementedError("base_samples is not supported: draws are taken through the latent structure "
                                      "(q n* + n* p normals per sample), not through a root of the dense covariance")
        return self._joint_or_raise().rsample(torch.Size(sample_shape), self._task_noise)

    def sample(self, sample_shape=torch.Size(), base_samples=None):
        with torch.no_grad():
            return self.rsample(sample_shape, base_samples)

    def log_prob(self, value):
        """Joint log-density of value [..., n*, p]: shape [...]."""
        return self._joint_or_raise().log_prob(value, self._task_noise)
