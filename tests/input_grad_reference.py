"""Closed form of the gradient of the eval-mode predictive means and variances w.r.t. the test inputs, restated in
torch on top of the unchanged oracle (the reference gets it from autograd through gpytorch's exact_prediction).

Per latent l and additive component g, with z = x / ell_{l,g} (the centring cancels in the distances),
s_ij = |z_i - z*_j|^2, K*_l = sum_g o_{l,g} k_g(s), alpha_l = K_l^-1 TY_l and beta_l = K_l^-1 K*_l, and task-level
cotangents g_mean, g_var [n*, p]:
  gm_l[j] = sum_t g_mean[j,t] H[l,t],  gv_l[j] = sum_t g_var[j,t] H[l,t]^2         (mixing adjoint)
  w[i,j] = gm_l[j] alpha_l[i] - 2 gv_l[j] beta_l[i,j],   A[i,j] = w[i,j] o_{l,g} k_g'(s_ij)
  d/dx*_{jk} += sum_l (2 / ell_{l,g,k}) (z*_{jk} sum_i A[i,j] - sum_i A[i,j] z_{ik})   for k in the dims of g.
The prior variance k(x*, x*) is constant for these stationary kernels and contributes nothing.  RQ needs
rq_reference.rq_kernels around the call (as for the oracle) and its alpha per component in ``alphas``.
"""
import math
import warnings
from unittest import mock

import torch

from oracle import plmc_oracle as O
from projected_lmc_b200 import ProjectedGPModel, gp

from . import helpers


def dk_ds(kind, s, alpha=None):
    """dk/ds of the kernel profiles of csrc/kernel_math.cuh (Matern-1/2: 0 at s = 0, where it is not differentiable)."""
    if kind == "rbf":
        return -0.5 * torch.exp(-0.5 * s)
    if kind == "rq":
        a = alpha.reshape(-1, 1, 1)
        b = 1 + s / (2 * a)
        return -0.5 * b.pow(-a) / b
    r = s.clamp_min(1e-30).sqrt()
    if kind == "matern52":
        return -(5.0 / 6.0) * (1 + math.sqrt(5) * r) * torch.exp(-math.sqrt(5) * r)
    if kind == "matern32":
        return -1.5 * torch.exp(-math.sqrt(3) * r)
    return torch.where(s > 1e-30, -0.5 * torch.exp(-r) / r, torch.zeros_like(s))


def components(p, d, alphas=None):
    """[(dims, ell [q, d_g], os [q] | None, alpha [q] | None)] of the oracle parameters."""
    alphas = alphas or [None]
    if p.components is None:
        return [(list(range(d)), O.lengthscale(p).reshape(p.q, -1), O.outputscale(p), alphas[0])]
    return [(list(c.dims), O.softplus(c.raw_lengthscale).reshape(p.q, -1),
             None if c.raw_outputscale is None else O.softplus(c.raw_outputscale), alphas[i % len(alphas)])
            for i, c in enumerate(p.components)]


def mixing_adjoint(H, g_mean, g_var):
    """Latent cotangents [q, n*] (None where the task-level one is None)."""
    gm = None if g_mean is None else (g_mean @ H.T).T
    gv = None if g_var is None else (g_var @ H.pow(2).T).T
    return gm, gv


def latent_predict(p, X, Y, Xs):
    """Latent posterior means / variances [q, n*] of the exact model (as oracle.predict, before the mixing)."""
    n = X.shape[0]
    TY = O.project_data(p, Y)
    K = O.gram(p, X, training=False) + torch.diag_embed(O.noise(p)[:, None].expand(-1, n))
    L = O.psd_safe_cholesky(K)
    alpha = torch.cholesky_solve(TY.unsqueeze(-1), L).squeeze(-1)
    Ks = O.gram(p, X, Xs, training=False)
    V = torch.linalg.solve_triangular(L, Ks, upper=False)
    kss = sum((torch.ones(p.q, dtype=X.dtype) if os_ is None else os_)
              for _, _, os_, _ in components(p, X.shape[1]))[:, None]
    return (Ks * alpha[:, :, None]).sum(1), kss - V.pow(2).sum(1)


def latent_input_grad(p, X, Y, Xs, gm, gv, alphas=None):
    """d/dXs of sum_lj gm[l,j] mu_l(j) + gv[l,j] v_l(j) by the closed form: [n*, d]."""
    with torch.no_grad():
        n = X.shape[0]
        TY = O.project_data(p, Y)
        K = O.gram(p, X, training=False) + torch.diag_embed(O.noise(p)[:, None].expand(-1, n))
        L = O.psd_safe_cholesky(K)
        alpha = torch.cholesky_solve(TY.unsqueeze(-1), L).squeeze(-1)
        w = torch.zeros((p.q, n, Xs.shape[0]), dtype=X.dtype)
        if gm is not None:
            w = w + gm[:, None, :] * alpha[:, :, None]
        if gv is not None:
            beta = torch.cholesky_solve(O.gram(p, X, Xs, training=False), L)
            w = w - 2 * gv[:, None, :] * beta
        out = torch.zeros_like(Xs)
        for dims, ell, os_, a in components(p, X.shape[1], alphas):
            z = X[:, dims] / ell[:, None, :]
            zs = Xs[:, dims] / ell[:, None, :]
            s = (z[:, :, None, :] - zs[:, None, :, :]).pow(2).sum(-1)
            A = w * dk_ds(p.kernel, s, a)
            if os_ is not None:
                A = A * os_[:, None, None]
            term = zs * A.sum(1)[:, :, None] - A.transpose(1, 2) @ z
            out[:, dims] += (2.0 / ell[:, None, :] * term).sum(0)
    return out


def input_grad(p, X, Y, Xs, g_mean, g_var, alphas=None):
    """d/dXs of sum(mean * g_mean + var_f * g_var) of oracle.predict by the closed form: [n*, d]."""
    gm, gv = mixing_adjoint(O.lmc_coefficients(p).detach(), g_mean, g_var)
    return latent_input_grad(p, X, Y, Xs, gm, gv, alphas)


def autograd_input_grad(p, X, Y, Xs, g_mean, g_var, which=1):
    """The same through torch autograd of oracle.predict (which = 1: var_f, 2: var_y)."""
    xs = Xs.detach().clone().requires_grad_(True)
    out = O.predict(p, X, Y, xs)
    f = 0.0
    if g_mean is not None:
        f = f + (out[0] * g_mean).sum()
    if g_var is not None:
        f = f + (out[which] * g_var).sum()
    (g,) = torch.autograd.grad(f, xs)
    return g


def rq_model(X, Y, q, outputscales=False, seed=0, variant="PLMC", **extra):
    """An RQ-kernel model, parameters moved off their symmetric init (as helpers.make_model)."""
    torch.manual_seed(seed)
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        m = ProjectedGPModel(X, Y, Y.shape[1], q, mean_type=gp.means.ZeroMean, kernel_type=gp.kernels.RQKernel,
                             init_lmc_coeffs=True, outputscales=outputscales, **dict(helpers.VARIANTS[variant]),
                             **extra)
    g = torch.Generator().manual_seed(seed + 1)
    with torch.no_grad():
        for name, prm in m.named_parameters():
            if "Q_plus" not in name:
                prm.add_(0.1 * torch.randn(prm.shape, generator=g, dtype=prm.dtype))
    return m


def oracle_params_and_alphas(m_cpu):
    """(helpers.oracle_params, the raw_alpha of every component for rq_reference.rq_kernels, or None without RQ)."""
    if m_cpu._base_kernel().kernel_id != 4:
        return helpers.oracle_params(m_cpu), None
    with mock.patch.dict(helpers.KNAMES, {4: "rq"}):
        p = helpers.oracle_params(m_cpu)
    cov = m_cpu._covar()
    kers = list(cov.kernels) if hasattr(cov, "kernels") else [cov]
    return p, [(k.base_kernel if hasattr(k, "base_kernel") else k).raw_alpha for k in kers]
