"""Likelihood stand-ins: the batched latent GaussianLikelihood (projected noise
Sigma_P) and the task-level likelihood returned by ``full_likelihood()``."""
from __future__ import annotations

import torch

from .constraints import GreaterThan


class Likelihood(torch.nn.Module):
    pass


class HomoskedasticNoise(torch.nn.Module):
    def __init__(self, noise_constraint=None, batch_shape=torch.Size()):
        super().__init__()
        self.register_parameter("raw_noise", torch.nn.Parameter(torch.zeros(*batch_shape, 1)))
        self.raw_noise_constraint = noise_constraint if noise_constraint is not None else GreaterThan(1e-4)

    @property
    def noise(self):
        return self.raw_noise_constraint.transform(self.raw_noise)


class _GaussianLikelihoodBase(Likelihood):
    pass


class GaussianLikelihood(_GaussianLikelihoodBase):
    """gpytorch.likelihoods.GaussianLikelihood(batch_shape=[q]): noise = softplus(raw)+lb, raw init 0."""

    def __init__(self, noise_constraint=None, batch_shape=torch.Size(), **kwargs):
        super().__init__()
        self.batch_shape = torch.Size(batch_shape)
        self.noise_covar = HomoskedasticNoise(noise_constraint=noise_constraint, batch_shape=self.batch_shape)

    @property
    def noise(self) -> torch.Tensor:
        return self.noise_covar.noise

    @noise.setter
    def noise(self, value):
        nc = self.noise_covar
        value = torch.as_tensor(value, dtype=nc.raw_noise.dtype, device=nc.raw_noise.device)
        with torch.no_grad():
            nc.raw_noise.copy_(nc.raw_noise_constraint.inverse_transform(value.expand_as(nc.raw_noise)))

    def forward(self, dist, *params, **kwargs):
        return dist.with_noise(self)

    def __call__(self, dist, *params, **kwargs):
        return self.forward(dist, *params, **kwargs)


class MultitaskGaussianLikelihood(Likelihood):
    """Task-noise likelihood built by ``ProjectedGPModel.full_likelihood`` (projected_lmc.py:1023-1074):
    rank = num_tasks, no global noise; marginal adds I (x) F F^T."""

    def __init__(self, num_tasks, rank=0, has_global_noise=False, dtype=None, device=None, **kwargs):
        super().__init__()
        if has_global_noise:
            raise NotImplementedError("global noise is not used by the projected model")
        self.num_tasks = num_tasks
        self.rank = rank
        self.register_parameter(
            "task_noise_covar_factor", torch.nn.Parameter(torch.randn(num_tasks, max(rank, 1), dtype=dtype, device=device))
        )

    @property
    def task_noise_covar(self) -> torch.Tensor:
        Fm = self.task_noise_covar_factor
        return Fm @ Fm.transpose(-1, -2)

    def forward(self, dist, *params, **kwargs):
        return dist.add_task_noise(self.task_noise_covar)

    def __call__(self, dist, *params, **kwargs):
        return self.forward(dist, *params, **kwargs)
