"""Stationary ARD kernels: parameter holders with gpytorch's names and constraints.

The Gram matrices themselves are never evaluated in Python: ``kernel_id`` selects
the fused CUDA epilogue (csrc/gram.cu).  Semantics: gpytorch 1.11 RBFKernel /
MaternKernel / RQKernel / ScaleKernel as instantiated by handle_covar_ (projected_lmc.py:107-181).
"""
from __future__ import annotations

import torch

from .constraints import Positive


class Kernel(torch.nn.Module):
    has_lengthscale = True
    kernel_id = None

    def __init__(self, ard_num_dims=None, batch_shape=torch.Size(), active_dims=None, lengthscale_prior=None,
                 lengthscale_constraint=None, **kwargs):
        super().__init__()
        self.ard_num_dims = ard_num_dims
        self.batch_shape = torch.Size(batch_shape)
        self.active_dims = None if active_dims is None else tuple(active_dims)
        d = 1 if ard_num_dims is None else ard_num_dims
        self.register_parameter("raw_lengthscale", torch.nn.Parameter(torch.zeros(*self.batch_shape, 1, d)))
        self.raw_lengthscale_constraint = lengthscale_constraint if lengthscale_constraint is not None else Positive()
        # gpytorch: register_prior("lengthscale_prior", prior, lambda m: m.lengthscale, ...): the log-density of the
        # constrained lengthscale is added to the MLL by ExactMarginalLogLikelihood._add_other_terms
        self.lengthscale_prior = lengthscale_prior

    def named_priors(self, prefix=""):
        if self.lengthscale_prior is not None:
            yield prefix + "lengthscale_prior", self, self.lengthscale_prior, (lambda m: m.lengthscale)

    def __add__(self, other):
        return AdditiveKernel(*_flatten(self), *_flatten(other))

    @property
    def lengthscale(self) -> torch.Tensor:
        return self.raw_lengthscale_constraint.transform(self.raw_lengthscale)

    @lengthscale.setter
    def lengthscale(self, value):
        value = torch.as_tensor(value, dtype=self.raw_lengthscale.dtype, device=self.raw_lengthscale.device)
        raw = self.raw_lengthscale_constraint.inverse_transform(value.expand_as(self.raw_lengthscale))
        with torch.no_grad():
            self.raw_lengthscale.copy_(raw)


class RBFKernel(Kernel):
    kernel_id = 0


class MaternKernel(Kernel):
    def __init__(self, nu=2.5, **kwargs):
        if nu not in (0.5, 1.5, 2.5):
            raise RuntimeError("nu expected to be 0.5, 1.5, or 2.5")
        super().__init__(**kwargs)
        self.nu = nu

    @property
    def kernel_id(self):
        return {2.5: 1, 1.5: 2, 0.5: 3}[self.nu]


class RQKernel(Kernel):
    """gpytorch.kernels.RQKernel: k = (1 + s / (2 alpha))^-alpha on the squared scaled distance s (the RBF input path:
    centred expansion, clamp_min 0).  ``raw_alpha`` [*batch_shape, 1], initialised to 0, under ``alpha_constraint``
    (default Positive(), so alpha starts at ln 2); the reference puts no prior on it."""
    kernel_id = 4

    def __init__(self, alpha_constraint=None, **kwargs):
        super().__init__(**kwargs)
        self.register_parameter("raw_alpha", torch.nn.Parameter(torch.zeros(*self.batch_shape, 1)))
        self.raw_alpha_constraint = alpha_constraint if alpha_constraint is not None else Positive()

    @property
    def alpha(self) -> torch.Tensor:
        return self.raw_alpha_constraint.transform(self.raw_alpha)

    @alpha.setter
    def alpha(self, value):
        value = torch.as_tensor(value, dtype=self.raw_alpha.dtype, device=self.raw_alpha.device)
        raw = self.raw_alpha_constraint.inverse_transform(value.expand_as(self.raw_alpha))
        with torch.no_grad():
            self.raw_alpha.copy_(raw)


class ScaleKernel(torch.nn.Module):
    def __init__(self, base_kernel, batch_shape=torch.Size(), outputscale_constraint=None, **kwargs):
        super().__init__()
        self.base_kernel = base_kernel
        self.batch_shape = torch.Size(batch_shape)
        self.register_parameter("raw_outputscale", torch.nn.Parameter(torch.zeros(*self.batch_shape)))
        self.raw_outputscale_constraint = outputscale_constraint if outputscale_constraint is not None else Positive()

    @property
    def outputscale(self) -> torch.Tensor:
        return self.raw_outputscale_constraint.transform(self.raw_outputscale)

    @outputscale.setter
    def outputscale(self, value):
        value = torch.as_tensor(value, dtype=self.raw_outputscale.dtype, device=self.raw_outputscale.device)
        with torch.no_grad():
            self.raw_outputscale.copy_(self.raw_outputscale_constraint.inverse_transform(value.expand_as(self.raw_outputscale)))

    @property
    def kernel_id(self):
        return self.base_kernel.kernel_id

    @property
    def active_dims(self):
        return self.base_kernel.active_dims

    def named_priors(self, prefix=""):
        yield from self.base_kernel.named_priors(prefix + "base_kernel.")

    def __add__(self, other):
        return AdditiveKernel(*_flatten(self), *_flatten(other))


class InducingPointKernel(torch.nn.Module):
    """gpytorch.kernels.InducingPointKernel(base_kernel, inducing_points, likelihood): parameter holder
    (``inducing_points`` [m, d], shared by the latents); the SGPR arithmetic lives in projected_lmc_b200/sgpr.py."""

    def __init__(self, base_kernel, inducing_points, likelihood, **kwargs):
        super().__init__()
        self.base_kernel = base_kernel
        self.likelihood = likelihood
        if inducing_points.dim() == 1:
            inducing_points = inducing_points.unsqueeze(-1)
        self.register_parameter("inducing_points", torch.nn.Parameter(inducing_points))

    def named_priors(self, prefix=""):
        yield from self.base_kernel.named_priors(prefix + "base_kernel.")


def _flatten(k):
    return list(k.kernels) if isinstance(k, AdditiveKernel) else [k]


class AdditiveKernel(torch.nn.Module):
    """k(x, x') = sum_g k_g(x, x'): what ``covar_module += ScaleKernel(...)`` builds in handle_covar_
    (projected_lmc.py:159-162).  ``kernels`` is a ModuleList like gpytorch's, so parameter names match
    (``covar_module.kernels.<g>.base_kernel.raw_lengthscale`` ...)."""

    def __init__(self, *kernels):
        super().__init__()
        self.kernels = torch.nn.ModuleList(kernels)

    def named_priors(self, prefix=""):
        for i, k in enumerate(self.kernels):
            yield from k.named_priors(f"{prefix}kernels.{i}.")

    def __add__(self, other):
        return AdditiveKernel(*_flatten(self), *_flatten(other))
