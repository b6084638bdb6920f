"""Model classes of the projected-LMC path with the reference's API surface.

Mirrors (same class names, constructor arguments, helper methods, parameter and
buffer names, error behaviour) of ``projectedlmc/projected_lmc.py``:
  handle_covar_ (:107-181), init_lmc_coefficients (:183-201), ExactGPModel (:264-436,
  constructor / lscales / outputscale), ProjectedGPModel (:893-1155).
The arithmetic of the path runs in libplmc_b200 (CUDA, sm_100a) through
``engine.LatentEngine``; small p x p / q x q algebra (QR of the mixing matrix, the
task-noise matrix) stays in torch on the same device so autograd reaches H, M, B.
"""
from __future__ import annotations

import warnings
from functools import reduce
from typing import List, Optional, Union

import numpy as np
import torch
from torch import Tensor
from torch.autograd.function import once_differentiable

from . import gp, ops
from .engine import LatentEngine
from .functions import LatentLogProb, ProjectData, ops_components
from .mixing import (LMCMixingMatrix, LowerTriangularParam, PositiveDiagonalParam, ScalarParam,
                     UpperTriangularParam)


def handle_covar_(kernel, dim: int, decomp: Optional[List[List[int]]] = None, n_funcs: int = 1,
                  prior_scales: Optional[Tensor] = None, prior_width: Optional[Tensor] = None,
                  outputscales: bool = True, ker_kwargs: Optional[dict] = None):
    """Kernel factory (drop-in for handle_covar_, projected_lmc.py:107-181): ARD kernels with batch shape
    [n_funcs].  ``decomp`` = groups of input dimensions, one sub-kernel per group, each wrapped in a ScaleKernel and
    summed (``decomp = [[0,1],[1,2]]`` -> k1(x0,x1) + k2(x1,x2)); ``prior_scales`` / ``prior_width`` put a Normal
    (one dimension) or MultivariateNormal (several; covariance diag(scale*width) exactly as the reference writes it)
    prior on each group's lengthscales and initialise them at the prior mean."""
    ker_kwargs = {} if ker_kwargs is None else ker_kwargs
    if decomp is None:
        decomp = [list(range(dim))]
    l_priors = [None] * len(decomp)
    if prior_scales is not None:
        if prior_width is None:
            raise ValueError('A prior width should be provided if a prior mean is')
        if type(prior_scales) is not list:   # an array with one length per variable, or a list with one array per kernel
            prior_scales = [prior_scales[idx_list] for idx_list in decomp]
        if type(prior_width) is not list:
            prior_width = [prior_width[idx_list] for idx_list in decomp]
        for i_ker, idx_list in enumerate(decomp):
            if len(idx_list) > 1:
                l_priors[i_ker] = gp.priors.MultivariateNormalPrior(
                    loc=prior_scales[i_ker], covariance_matrix=torch.diag_embed(prior_scales[i_ker] * prior_width[i_ker]))
            else:
                l_priors[i_ker] = gp.priors.NormalPrior(loc=prior_scales[i_ker],
                                                        scale=prior_scales[i_ker] * prior_width[i_ker])
    kernels = [kernel(ard_num_dims=len(idx_list), active_dims=idx_list, lengthscale_prior=l_priors[i_ker],
                      batch_shape=torch.Size([n_funcs]), **ker_kwargs) for i_ker, idx_list in enumerate(decomp)]
    if len(decomp) > 1:
        covar_module = gp.kernels.ScaleKernel(kernels[0], batch_shape=torch.Size([n_funcs]))
        for ker in kernels[1:]:
            covar_module += gp.kernels.ScaleKernel(ker, batch_shape=torch.Size([n_funcs]))
    elif outputscales:
        covar_module = gp.kernels.ScaleKernel(kernels[0], batch_shape=torch.Size([n_funcs]))
    else:
        covar_module = kernels[0]
    if prior_scales is not None and kernels[0].has_lengthscale:
        try:
            for i_ker in range(len(kernels)):
                kernels[i_ker].lengthscale = l_priors[i_ker].mean
        except Exception:
            raise ValueError('Provided prior scales were of the wrong shape')
    return covar_module


def init_lmc_coefficients(train_y: Tensor, n_latents: int, QR_form: bool = False):
    """Data-driven initial mixing matrix: truncated SVD of Y^T (sklearn randomized_svd,
    random_state=0) or, with fewer points than latents, a complete QR."""
    from sklearn.utils.extmath import randomized_svd

    n_data, _ = train_y.shape
    Yt = train_y.cpu().numpy().T
    kw = dict(device=train_y.device, dtype=train_y.dtype)
    if n_data >= n_latents:
        U, S, _ = randomized_svd(Yt, n_components=n_latents, random_state=0)
        U, S = torch.as_tensor(U, **kw), torch.as_tensor(S, **kw)
    else:
        Qc, Rc = np.linalg.qr(Yt, mode='complete')
        S = 1e-3 * torch.ones(n_latents, **kw)
        S[:n_data] = torch.as_tensor(np.diag(Rc).copy(), **kw)
        U = torch.as_tensor(Qc[:, :n_latents], **kw)
    if QR_form:
        return U, S
    return (U * S / np.sqrt(n_data - 1)).T


class ExactGPModel(torch.nn.Module):
    """Batched exact-GP parameter holder (constructor, ``lscales``, ``outputscale``).

    Only the pieces the projected model inherits are implemented; a stand-alone batched
    exact GP is outside the hot-path scope."""

    def __init__(self, train_x: Tensor, train_y: Tensor, likelihood, n_tasks: int = 1,
                 prior_scales: Optional[Tensor] = None, prior_width: Optional[Tensor] = None,
                 mean_type=gp.means.ConstantMean, decomp: Optional[List[List[int]]] = None,
                 outputscales: bool = False, kernel_type=gp.kernels.RBFKernel, ker_kwargs: Optional[dict] = None,
                 n_inducing_points: Optional[int] = None, **kwargs):
        super().__init__()
        if train_x.dim() == 1:
            train_x = train_x.unsqueeze(-1)
        self.train_inputs = (train_x,)
        self.train_targets = train_y
        self.likelihood = likelihood
        ker_kwargs = {} if ker_kwargs is None else ker_kwargs
        self.dim = train_x.shape[1]
        self.n_tasks = n_tasks
        self.batch_lik = isinstance(likelihood, gp.likelihoods.GaussianLikelihood)
        self.mean_module = mean_type(input_size=self.dim, batch_shape=torch.Size([n_tasks]))
        self.covar_module = handle_covar_(_resolve_kernel(kernel_type), dim=self.dim, decomp=decomp,
                                          prior_scales=prior_scales, prior_width=prior_width,
                                          outputscales=outputscales, n_funcs=n_tasks, ker_kwargs=ker_kwargs)
        if n_inducing_points is not None:
            self.covar_module = gp.kernels.InducingPointKernel(self.covar_module,
                                                              torch.randn(n_inducing_points, self.dim), likelihood)

    # gpytorch.models.ExactGP moves its training data together with the module
    def _apply(self, fn, *args, **kwargs):
        self.train_inputs = tuple(fn(t) for t in self.train_inputs)
        self.train_targets = fn(self.train_targets)
        out = super()._apply(fn, *args, **kwargs)
        eng = getattr(self, "_engine", None)
        if eng is not None:      # .float() / .double(): the arithmetic grade follows the model's dtype
            eng.grade = "fp32" if self.train_inputs[0].dtype == torch.float32 else "fp64"
        return out

    def named_priors(self):
        """(name, module, prior, closure) of every registered prior (gpytorch Module.named_priors)."""
        yield from self.covar_module.named_priors("covar_module.")

    def _inducing(self):
        """The inducing-point kernel wrapper, or None for the exact model."""
        cm = self.covar_module
        return cm if isinstance(cm, gp.kernels.InducingPointKernel) else None

    def _covar(self):
        """The kernel proper (under the inducing-point wrapper, if any)."""
        cm = self.covar_module
        return cm.base_kernel if isinstance(cm, gp.kernels.InducingPointKernel) else cm

    def added_loss_terms(self):
        """gpytorch Module.added_loss_terms: the inducing-point kernel registers one during the training-mode
        forward; it is evaluated together with the latent log-probabilities and handed out here."""
        if self._inducing() is not None and getattr(self, "_sgpr_added", None) is not None:
            yield _StoredLoss(self._sgpr_added)

    def _base_kernel(self):
        """The (first) ARD kernel under the optional ScaleKernel / sum."""
        cm = self._covar()
        if hasattr(cm, 'kernels'):
            cm = cm.kernels[0]
        return cm.base_kernel if hasattr(cm, 'base_kernel') else cm

    def _kernel_components(self):
        """[(kernel_id, active dims, lengthscale [q, d_g], outputscale [q] | None)] of the additive kernel
        (ops.Component: a shape parameter such as RQKernel's alpha [q] rides along as ``.shape_param``)."""
        cm = self._covar()
        out = []
        for ker in (cm.kernels if hasattr(cm, 'kernels') else [cm]):
            base = ker.base_kernel if hasattr(ker, 'base_kernel') else ker
            dims = tuple(range(self.dim)) if base.active_dims is None else tuple(base.active_dims)
            out.append(ops.Component(base.kernel_id, dims, base.lengthscale.squeeze(-2),
                                     ker.outputscale if hasattr(ker, 'base_kernel') else None,
                                     base.alpha.squeeze(-1) if hasattr(base, 'raw_alpha') else None))
        return out

    def lscales(self, unpacked: bool = True) -> Union[List[Tensor], Tensor]:
        """Learned lengthscales: one n_funcs x n_dims tensor per sub-kernel (a single tensor for a non-composite
        kernel when ``unpacked``), as projected_lmc.py:324-346."""
        if hasattr(self._covar(), 'kernels'):
            return [(k.base_kernel if hasattr(k, 'base_kernel') else k).lengthscale.data.squeeze()
                    for k in self._covar().kernels]
        scales = self._base_kernel().lengthscale.data.squeeze()
        return scales if unpacked else [scales]

    def outputscale(self, unpacked: bool = False) -> Tensor:
        """Learned outputscales, n_funcs x n_kernels; raises when the model has none (projected_lmc.py:348-365)."""
        cm = self._covar()
        n_kernels = len(cm.kernels) if hasattr(cm, 'kernels') else 1
        n_funcs = self.n_latents if hasattr(self, 'n_latents') else self.n_tasks
        res = torch.zeros((n_funcs, n_kernels))
        if n_kernels > 1:
            for i_ker in range(n_kernels):
                res[:, i_ker] = cm.kernels[i_ker].outputscale.data.squeeze()
        else:
            res[:, 0] = cm.outputscale.data.squeeze()
        return res.squeeze() if (n_kernels == 1 and unpacked) else res


def _resolve_kernel(kernel_type):
    """Accept our own kernel classes, or gpytorch's by class name."""
    if isinstance(kernel_type, type) and issubclass(kernel_type, gp.kernels.Kernel):
        return kernel_type
    name = getattr(kernel_type, "__name__", str(kernel_type))
    if hasattr(gp.kernels, name):
        return getattr(gp.kernels, name)
    raise NotImplementedError(f"kernel {name} is not supported on the B200 path (RBFKernel, MaternKernel, RQKernel)")


class ProjectedGPModel(ExactGPModel):
    """The projected LMC model (drop-in for projected_lmc.py:893-1155)."""

    def __init__(self, train_x: Tensor, train_y: Tensor, n_tasks: int, n_latents: int, proj_likelihood=None,
                 init_lmc_coeffs: bool = False, BDN: bool = True, diagonal_B: bool = False, scalar_B: bool = False,
                 diagonal_R: bool = False, mean_type=gp.means.ConstantMean, ortho_param='matrix_exp', bulk=True,
                 noise_thresh: float = -9., noise_init: float = 1e-2, outputscales: bool = False, eps=1e-3,
                 **kwargs):
        if proj_likelihood is None or proj_likelihood.noise.shape[0] != n_latents:
            warnings.warn("In projected GP model the dimension of the likelihood is the number of latent processes. "
                          "Provided likelihood was the wrong shape or None, so it was replaced by a fresh one")
            proj_likelihood = gp.likelihoods.GaussianLikelihood(
                batch_shape=torch.Size([n_latents]),
                noise_constraint=gp.constraints.GreaterThan(np.exp(noise_thresh)))

        super().__init__(train_x, torch.zeros_like(train_y), proj_likelihood, n_tasks=n_latents,
                         mean_type=gp.means.ZeroMean, outputscales=outputscales, **kwargs)
        self.register_buffer('train_y', train_y)
        if mean_type is not gp.means.ZeroMean and getattr(mean_type, "__name__", "") != "ZeroMean":
            raise ValueError('Projected GP model does not support non-zero output-wise means for now !')

        n_data, n_tasks = train_y.shape
        fast = scalar_B and BDN
        if init_lmc_coeffs:
            if fast:
                Q_plus, R = init_lmc_coefficients(train_y, n_latents=n_latents, QR_form=True)
            else:
                Q_plus, R_padded = init_lmc_coefficients(train_y, n_latents=n_tasks, QR_form=True)
                R = R_padded[:n_latents]
        else:
            Q_plus, R_padded, _ = torch.linalg.svd(torch.randn(n_tasks, n_latents))
            R = R_padded[:n_latents]
            if fast:
                Q_plus = Q_plus[:, :n_latents]
        R = torch.diag_embed(R) / np.sqrt(n_data - 1)
        lmc = LMCMixingMatrix(Q_plus, R, bulk=bulk)
        if not bulk:
            lmc = torch.nn.utils.parametrizations.orthogonal(
                lmc, name="Q_plus", orthogonal_map=ortho_param, use_trivialization=(ortho_param != 'householder'))
            torch.nn.utils.parametrize.register_parametrization(
                lmc, "R", PositiveDiagonalParam() if diagonal_R else UpperTriangularParam())
        self.lmc_coefficients = lmc

        n_disc = n_tasks - n_latents
        if scalar_B:
            diagonal_B = True
            self.register_parameter("log_B_tilde", torch.nn.Parameter(np.log(noise_init) * torch.ones(n_disc)))
            torch.nn.utils.parametrize.register_parametrization(
                self, "log_B_tilde", ScalarParam(bounds=(noise_thresh, -noise_thresh)))
            if BDN:
                self.register_buffer('Y_squared_norm', (train_y ** 2).sum())
        elif diagonal_B:
            self.register_parameter("log_B_tilde", torch.nn.Parameter(np.log(noise_init) * torch.ones(n_disc)))
            # registered but never applied, as in the reference (:981)
            self.log_B_tilde_constraint = gp.constraints.GreaterThan(noise_thresh)
        else:
            self.register_parameter("B_tilde_inv_chol", torch.nn.Parameter(
                torch.diag_embed(np.log(1 / noise_init) * torch.ones(n_disc))))
            torch.nn.utils.parametrize.register_parametrization(
                self, "B_tilde_inv_chol", LowerTriangularParam(bounds=(noise_thresh, -noise_thresh)))
        self.diagonal_B, self.scalar_B = diagonal_B, scalar_B
        if not BDN:
            self.register_parameter("M", torch.nn.Parameter(torch.zeros((n_latents, n_disc))))

        self.n_tasks = n_tasks
        self.n_latents = n_latents
        self.latent_dim = -1
        self.eps = eps

        self._engine = LatentEngine()
        self._engine.grade = "fp32" if train_x.dtype == torch.float32 else "fp64"
        self._latent_range = (0, n_latents)   # latents owned by this process (distributed.shard_latents)
        self._dist_group = None
        self._pred_cache = None
        self._pred_key = None

    # ---- small helpers -------------------------------------------------------------
    def projected_noise(self) -> Tensor:
        """Modeled noises of the latent processes (diagonal of Sigma_P), size n_latents."""
        return self.likelihood.noise.squeeze(-1)

    def projection_matrix(self) -> Tensor:
        """T [n_tasks, n_latents] with  Y T = projected data."""
        Q, R, Q_orth = self.lmc_coefficients.QR()
        T = torch.linalg.solve_triangular(R.T, Q, upper=False, left=False)
        if hasattr(self, "M"):
            T = T + Q_orth @ self.M.T * self.projected_noise()[None, :]
        return T

    def project_data(self, data: Tensor) -> Tensor:
        """T^T data^T, shape n_latents x n_points (CUDA kernel 1; T is formed on the host)."""
        T = self.projection_matrix()
        return ProjectData.apply(T, _as_f64(data).contiguous()).to(T.dtype)

    def B_tilde(self) -> Tensor:
        """Discarded-noise factor, symmetric (or diagonal) of size n_tasks - n_latents."""
        if self.diagonal_B:
            return torch.diag_embed(torch.exp(self.log_B_tilde))
        k = self.n_tasks - self.n_latents
        L_inv = torch.linalg.solve_triangular(self.B_tilde_inv_chol, torch.eye(
            k, dtype=self.B_tilde_inv_chol.dtype, device=self.B_tilde_inv_chol.device), upper=False)
        return L_inv.T @ L_inv

    def _B_tilde_root(self) -> Tensor:
        if self.diagonal_B:
            return torch.diag_embed(torch.exp(self.log_B_tilde / 2))
        k = self.n_tasks - self.n_latents
        eye = torch.eye(k, dtype=self.B_tilde_inv_chol.dtype, device=self.B_tilde_inv_chol.device)
        return torch.linalg.solve_triangular(self.B_tilde_inv_chol, eye, upper=False).T

    def task_noise_covar(self) -> Tensor:
        """Sigma [p, p]: the task-level noise implied by (H, Sigma_P, M, B_tilde)."""
        Q, R, Q_orth = self.lmc_coefficients.QR()
        QR = Q @ R
        sigma_p = self.projected_noise()
        if hasattr(self, "M"):
            B = self._B_tilde_root()
            B = B @ B.T
            SM = sigma_p[:, None] * self.M
            cross = -QR @ SM @ B @ Q_orth.T
            D_rot = torch.diag_embed(sigma_p) + SM @ B @ SM.T
            return QR @ D_rot @ QR.T + cross + cross.T + Q_orth @ B @ Q_orth.T
        if self.scalar_B:
            if self.log_B_tilde.numel() > 0:
                eye = torch.eye(self.n_tasks, dtype=QR.dtype, device=QR.device)
                B_term = torch.exp(self.log_B_tilde[0]) * (eye - Q @ Q.T)
            else:
                B_term = 0.
        else:
            Br = Q_orth @ self._B_tilde_root()
            B_term = Br @ Br.T
        Dr = QR * torch.sqrt(sigma_p)[None, :]
        return Dr @ Dr.T + B_term

    def full_likelihood(self):
        """Task-level likelihood: MultitaskGaussianLikelihood whose factor is
        chol(Sigma + jitter), jitter from 1e-6 growing x10 while below ``self.eps``."""
        sigma_p = self.projected_noise()
        res = gp.likelihoods.MultitaskGaussianLikelihood(num_tasks=self.n_tasks, rank=self.n_tasks,
                                                         has_global_noise=False, dtype=sigma_p.dtype,
                                                         device=sigma_p.device)
        with torch.no_grad():
            Sigma = self.task_noise_covar()
            eye = torch.eye(self.n_tasks, dtype=Sigma.dtype, device=Sigma.device)
            jitter, done = 1e-6, False
            while jitter < self.eps:
                F, info = torch.linalg.cholesky_ex(Sigma + jitter * eye)
                if int(info) == 0:
                    res.task_noise_covar_factor.data = F
                    done = True
                    break
                jitter *= 10
                warnings.warn("Cholesky of the full noise covariance failed. Trying again with jitter {0} ...".format(jitter))
            if not done:
                warnings.warn("full noise covariance is not positive definite up to eps; the likelihood keeps its "
                              "random initial factor (reference behaviour)")
        return res

    # ---- CUDA path -----------------------------------------------------------------
    def _local_components(self, detach=False):
        """(spec, tensors) of the kernel for the latents owned by this process: spec = ((kernel id, dims, has
        outputscale, has shape parameter), ...), tensors = [ell_0, (os_0), (alpha_0), ell_1, ...] as contiguous
        float64."""
        lo, hi = self._latent_range
        spec, tensors = [], []
        for comp in self._kernel_components():
            kid, dims, ell, os_ = comp
            shape = ops.shape_of(comp)
            spec.append((kid, dims, os_ is not None, shape is not None))
            tensors.append(_as_f64(ell)[lo:hi])
            if os_ is not None:
                tensors.append(_as_f64(os_)[lo:hi])
            if shape is not None:
                tensors.append(_as_f64(shape)[lo:hi])
        if detach:
            tensors = [t.detach().contiguous() for t in tensors]
        return tuple(spec), tensors

    def _latent_log_prob(self, proj_target: Tensor) -> Tensor:
        """log N(TY_l; 0, K_l + noise_l I) for the latents owned by this process."""
        X = _as_f64(self.train_inputs[0])
        lo, hi = self._latent_range
        spec, tensors = self._local_components()
        ind = self._inducing()
        if ind is not None:     # SGPR: low-rank covariance K_fu K_uu^-1 K_uf + noise, plus the added loss term
            from . import sgpr
            self._engine.xmean(X)
            lp, added = sgpr.latent_log_prob(self._engine, X, _as_f64(proj_target)[lo:hi].contiguous(),
                                             _as_f64(ind.inducing_points), ops_components(spec, tensors),
                                             _as_f64(self.projected_noise())[lo:hi])
            self._sgpr_added = added
            return lp.to(proj_target.dtype)
        lp = LatentLogProb.apply(self._engine, X, spec, _as_f64(proj_target)[lo:hi],
                                 _as_f64(self.projected_noise())[lo:hi], *tensors)
        return lp.to(proj_target.dtype)

    def forward(self, x: Tensor):
        """Latent prior handle (nothing is evaluated yet, like gpytorch's lazy MVN)."""
        return gp.distributions.MultivariateNormal(self, x)

    def _check_train_inputs(self, x: Tensor):
        tx = self.train_inputs[0]
        if x is tx:
            return
        if x.dim() == 1:
            x = x.unsqueeze(-1)
        if x.shape != tx.shape or not torch.equal(x, tx):
            raise RuntimeError("You must train on the training inputs!")

    def _parameter_key(self):
        """Changes whenever a parameter, train_y or the owned latent range changes."""
        return tuple((id(p), p._version) for p in self.parameters()) + (self.train_y._version, self._latent_range)

    def _prediction_state(self):
        key = self._parameter_key()
        # the factor lives in the engine's shared workspace: compute_loo / kernel_cond / a training-mode handle
        # rewrite it, so the cache is also checked against the engine's workspace generation
        stale = self._inducing() is None and not self._engine.state_is_current(self._pred_cache)
        if self._pred_cache is None or self._pred_key != key or stale:
            with torch.no_grad():
                X = _as_f64(self.train_inputs[0])
                lo, hi = self._latent_range
                spec, tensors = self._local_components(detach=True)
                TY = _as_f64(self.project_data(self.train_y))[lo:hi].contiguous()
                noise = _as_f64(self.projected_noise())[lo:hi].contiguous()
                if self._inducing() is not None:
                    from . import sgpr
                    self._engine.xmean(X)
                    self._pred_cache = sgpr.prediction_state(
                        self._engine, X, TY, _as_f64(self._inducing().inducing_points).detach().contiguous(),
                        ops_components(spec, tensors), noise)
                else:
                    self._pred_cache = self._engine.factorize(X, TY, ops_components(spec, tensors), noise)
                self._pred_key = key
        return self._pred_cache

    def _predict_latents(self, st, xs):
        if self._inducing() is not None:
            from . import sgpr
            return sgpr.predict_latents(self._engine, st, _as_f64(self.train_inputs[0]), xs)
        return self._engine.predict_latents(st, xs)

    def train(self, mode: bool = True):
        if mode:
            self._pred_cache, self._pred_key = None, None
        return super().train(mode)

    def compute_latent_distrib(self, x: Tensor, **kwargs):
        """Latent processes at ``x``: prior handle in training mode, posterior mean/variance
        ([n_latents, n_points]) in eval mode."""
        if self.training:
            self._check_train_inputs(x)
            return self.forward(x)
        if self._input_grad(x):
            xs = _as_f64(x if x.dim() > 1 else x.unsqueeze(-1)).contiguous()
            m, v = _LatentPrediction.apply(self, xs, False)
            return LatentPosterior(m.to(x.dtype), v.to(x.dtype), _JointPosterior(self, xs.detach(), x.dtype))
        with torch.no_grad():
            st = self._prediction_state()
            xs = _as_f64(x if x.dim() > 1 else x.unsqueeze(-1)).contiguous()
            m, v = self._predict_latents(st, xs)
        return LatentPosterior(m.to(x.dtype), v.to(x.dtype), _JointPosterior(self, xs, x.dtype))

    def _input_grad(self, x: Tensor) -> bool:
        """Eval-mode predictions are differentiable w.r.t. the test inputs when grad is enabled and x requires it
        (not for latent-sharded models, whose outputs stay detached)."""
        return torch.is_grad_enabled() and x.requires_grad and self._dist_group is None and \
            self._latent_range == (0, self.n_latents)

    def _full_components(self):
        """The kernel components of all latents as contiguous float64 (no autograd)."""
        def f64(t):
            return None if t is None else _as_f64(t).contiguous()
        out = []
        for c in self._kernel_components():
            kid, dims, ell, os_ = c
            out.append(ops.Component(kid, dims, f64(ell), f64(os_), f64(ops.shape_of(c))))
        return out

    def kernel_cond(self):
        """Condition numbers of the noisy latent train covariances K_l + s_l I (dense SVD: small n)."""
        with torch.no_grad():
            X = _as_f64(self.train_inputs[0])
            comps = self._full_components()
            K = self._engine.dense_gram(X, comps, _as_f64(self.projected_noise()).contiguous())
            return torch.linalg.cond(K)

    def compute_loo(self, output=None):
        """Leave-one-out predictive variances and residuals of the latent GPs,
        both n_points x n_latents (by-product of K^-1 and alpha)."""
        with torch.no_grad():
            X = _as_f64(self.train_inputs[0])
            comps = self._full_components()
            TY = _as_f64(self.project_data(self.train_y)).contiguous()
            s2, r = self._engine.loo(X, TY, comps, _as_f64(self.projected_noise()).contiguous())
        dt = self.train_y.dtype
        return s2.T.to(dt), r.T.to(dt)

    def __call__(self, x: Tensor, **kwargs):
        """Training mode: latent prior handle.  Eval mode: task-level posterior with
        ``.mean`` / ``.variance`` of shape n_points x n_tasks."""
        if self.training:
            self._check_train_inputs(x)
            return self.forward(x)
        if self._input_grad(x):
            return self._differentiable_call(x)
        with torch.no_grad():
            st = self._prediction_state()
            xs = _as_f64(x if x.dim() > 1 else x.unsqueeze(-1)).contiguous()
            joint = _JointPosterior(self, xs, x.dtype)
            # a non-finite test point gives NaN predictions for that point in the reference; the integer tensor
            # path of the solve would not propagate it, so such rows are computed at 0 and overwritten below
            bad_rows = ~torch.isfinite(xs).all(dim=1)
            has_bad = bool(bad_rows.any())
            if has_bad:
                xs = xs.clone()
                xs[bad_rows] = 0.0
            lat_mean, lat_var = self._predict_latents(st, xs)
            lo, hi = self._latent_range
            Ht = _as_f64(self.lmc_coefficients())[lo:hi].contiguous()
            ns = xs.shape[0]
            mean = torch.empty((ns, self.n_tasks), dtype=torch.float64, device=xs.device)
            var = torch.empty_like(mean)
            var_add = torch.full((self.n_tasks,), float(self.eps) if lo == 0 else 0.0, dtype=torch.float64,
                                 device=xs.device)
            ops.mix_tasks(lat_mean, lat_var, Ht, var_add, mean, var, ns)
            if self._dist_group is not None:
                import torch.distributed as dist
                both = torch.stack((mean, var))          # one collective for the two [n*, p] tiles
                dist.all_reduce(both, group=self._dist_group)
                mean, var = both[0], both[1]
            if has_bad:
                mean[bad_rows] = float("nan")
                var[bad_rows] = float("nan")
            joint.task_mean = mean
            task_noise = float(self.eps) * torch.eye(self.n_tasks, dtype=torch.float64, device=xs.device)
        return gp.distributions.MultitaskMultivariateNormal(mean.to(x.dtype), var.to(x.dtype), joint, task_noise)

    def _differentiable_call(self, x: Tensor):
        """The eval branch of __call__ with .mean / .variance differentiable w.r.t. x (same values, bit for bit).
        Model parameters receive no gradient through predictions; the joint quantities (covariance_matrix, rsample,
        log_prob) stay detached."""
        xs = _as_f64(x if x.dim() > 1 else x.unsqueeze(-1)).contiguous()
        joint = _JointPosterior(self, xs.detach(), x.dtype)
        bad_rows = ~torch.isfinite(xs.detach()).all(dim=1)
        lat_mean, lat_var = _LatentPrediction.apply(self, xs, True)
        with torch.no_grad():
            Ht = _as_f64(self.lmc_coefficients()).contiguous()
            var_add = torch.full((self.n_tasks,), float(self.eps), dtype=torch.float64, device=xs.device)
        mean, var = _MixTasks.apply(lat_mean, lat_var, Ht, var_add)
        if bool(bad_rows.any()):
            mean = mean.masked_fill(bad_rows[:, None], float("nan"))
            var = var.masked_fill(bad_rows[:, None], float("nan"))
        joint.task_mean = mean.detach()
        task_noise = float(self.eps) * torch.eye(self.n_tasks, dtype=torch.float64, device=xs.device)
        return gp.distributions.MultitaskMultivariateNormal(mean.to(x.dtype), var.to(x.dtype), joint, task_noise)


class _LatentPrediction(torch.autograd.Function):
    """Latent posterior means / variances [q, n*] at the float64 test points xs [n*, d] of an eval-mode model, with
    their gradient w.r.t. xs.  The forward is the model's no-grad prediction (``zero_bad``: non-finite rows are
    predicted at 0, as ProjectedGPModel.__call__ does).  The backward keeps nothing of size n x n* from the forward:
    the exact model recomputes each tile in LatentEngine.predict_latents_grad, the inducing-point model runs torch
    autograd through its cross block with the test points as rows.  A parameter or train_y changed since the forward
    is an error; a rewritten engine workspace (compute_loo, a training step) is re-factorised.  Rows of non-finite
    test points get NaN gradients.  Not twice differentiable."""

    @staticmethod
    def forward(ctx, model, xs, zero_bad):
        xin = xs
        bad_rows = ~torch.isfinite(xs).all(dim=1)
        if zero_bad and bool(bad_rows.any()):
            xin = xs.clone()
            xin[bad_rows] = 0.0
        st = model._prediction_state()
        m, v = model._predict_latents(st, xin)
        ctx.model, ctx.key = model, model._parameter_key()
        ctx.save_for_backward(xs)
        ctx.set_materialize_grads(False)
        return m, v

    @staticmethod
    @once_differentiable
    def backward(ctx, g_mean, g_var):
        model = ctx.model
        (xs,) = ctx.saved_tensors
        if g_mean is None and g_var is None:
            return None, None, None
        if model._parameter_key() != ctx.key:
            raise RuntimeError("the model's parameters or train_y changed after this prediction was made; "
                               "call the model again before backpropagating to the test inputs")
        bad_rows = ~torch.isfinite(xs).all(dim=1)
        has_bad = bool(bad_rows.any())
        x0 = xs.masked_fill(bad_rows[:, None], 0.0) if has_bad else xs
        st = model._prediction_state()
        if model._inducing() is not None:
            from . import sgpr
            with torch.enable_grad():
                xr = x0.detach().requires_grad_(True)
                m, v = sgpr.predict_latents(model._engine, st, _as_f64(model.train_inputs[0]), xr, test_rows=True)
                outs = [(o, g) for o, g in ((m, g_mean), (v, g_var)) if g is not None]
                (g,) = torch.autograd.grad([o for o, _ in outs], (xr,), [g for _, g in outs])
        else:
            g = model._engine.predict_latents_grad(st, x0, g_mean, g_var)
        if has_bad:
            g[bad_rows] = float("nan")
        return None, g, None


class _MixTasks(torch.autograd.Function):
    """Task-level means / marginal variances [n*, p] from the latent ones (ops.mix_tasks), differentiable w.r.t. the
    latent means and variances (ops.mix_tasks_bwd); H and var_add receive no gradient."""

    @staticmethod
    def forward(ctx, lat_mean, lat_var, H, var_add):
        ns = lat_mean.shape[1]
        mean = torch.empty((ns, H.shape[1]), dtype=torch.float64, device=lat_mean.device)
        var = torch.empty_like(mean)
        ops.mix_tasks(lat_mean, lat_var, H, var_add, mean, var, ns)
        ctx.H = H
        ctx.set_materialize_grads(False)
        return mean, var

    @staticmethod
    @once_differentiable
    def backward(ctx, g_mean, g_var):
        if g_mean is None and g_var is None:
            return None, None, None, None
        g_lm, g_lv = ops.mix_tasks_bwd(ctx.H, None if g_mean is None else g_mean.contiguous(),
                                       None if g_var is None else g_var.contiguous())
        return g_lm, g_lv, None, None


class _StoredLoss:
    def __init__(self, value):
        self.value = value

    def loss(self, *params):
        return self.value


class LatentPosterior:
    def __init__(self, mean, variance, joint=None):
        self.mean, self.variance = mean, variance
        self._joint = joint
        self._covar = None

    @property
    def stddev(self):
        return self.variance.clamp_min(0).sqrt()

    @property
    def covariance_matrix(self):
        """Latent posterior covariances [q, n*, n*] (the reference's batched latent MVN; computed on first access)."""
        if self._covar is None:
            self._covar = self._joint.latent_covariance()
        return self._covar


class _JointPosterior:
    """The joint quantities of one eval-mode prediction, computed on demand: the latent posterior covariances
    C_l = K**_l - V_l^T V_l, the task-level covariance, posterior draws and the joint log-density.  It keeps its own
    copy of the test inputs and the parameter key of the prediction: a parameter or train_y changed since then is
    an error, a rewritten engine workspace (compute_loo, a training step) only means the factor is recomputed."""

    def __init__(self, model, xs, dtype):
        self.model = model
        self.xs = xs.clone()
        self.bad_rows = ~torch.isfinite(self.xs).all(dim=1)
        self.has_bad = bool(self.bad_rows.any())
        if self.has_bad:        # computed at 0, reported as NaN (as the marginal variances)
            self.xs[self.bad_rows] = 0.0
        self.dtype = dtype
        self.key = model._parameter_key()
        self.task_mean = None    # [n*, p] float64, set by the task-level prediction
        self._lat = None
        self._factor = None

    def _latent(self):
        m = self.model
        if m._inducing() is not None:
            raise NotImplementedError("joint posterior quantities (covariance_matrix, rsample, log_prob) are not "
                                      "implemented for the inducing-point (SGPR) model")
        if m._latent_range != (0, m.n_latents) or m._dist_group is not None:
            raise NotImplementedError("joint posterior quantities (covariance_matrix, rsample, log_prob) are not "
                                      "implemented for latent-sharded models (distributed.shard_latents)")
        if m._parameter_key() != self.key:
            raise RuntimeError("the model's parameters or train_y changed after this prediction was made; "
                               "call the model again for the joint posterior")
        if self._lat is None:
            with torch.no_grad():
                self._lat = m._engine.latent_covariance(m._prediction_state(), self.xs)
        return self._lat

    def _no_nan_inputs(self):
        if self.has_bad:
            from .engine import NanError
            raise NanError("cholesky: the posterior covariance contains NaN (non-finite test inputs)")

    def _mixing(self):
        return _as_f64(self.model.lmc_coefficients()).detach().contiguous()

    def latent_covariance(self):
        _, C = self._latent()
        ns = self.xs.shape[0]
        Cn = C[:, :ns, :ns]
        out = torch.tril(Cn) + torch.tril(Cn, -1).transpose(1, 2)
        if self.has_bad:
            out[:, self.bad_rows, :] = float("nan")
            out[:, :, self.bad_rows] = float("nan")
        return out.to(self.dtype)

    def task_covariance(self, task_noise):
        _, C = self._latent()
        ns, p = self.xs.shape[0], self.model.n_tasks
        with torch.no_grad():
            S = (0.5 * (task_noise + task_noise.T)).contiguous()     # exactly symmetric, so is the result
            T = ops.task_covariance(C, self._mixing(), S, ns)
            if self.has_bad:
                T4 = T.view(ns, p, ns, p)
                T4[self.bad_rows] = float("nan")
                T4[:, :, self.bad_rows] = float("nan")
        return T.to(self.dtype)

    def rsample(self, sample_shape, task_noise):
        self._no_nan_inputs()
        lat_mean, C = self._latent()
        ns, p, q = self.xs.shape[0], self.model.n_tasks, C.shape[0]
        eng = self.model._engine
        with torch.no_grad():
            if self._factor is None:
                self._factor = eng.factor_covariance(C, ns)
            S = int(torch.Size(sample_shape).numel())
            dev = C.device
            eps = torch.randn((q, ns, S), dtype=torch.float64, device=dev)
            E = torch.randn((S, ns, p), dtype=torch.float64, device=dev)
            R = torch.linalg.cholesky(0.5 * (task_noise + task_noise.T)).contiguous()
            G = eng.latent_draws(*self._factor, eps)
            out = ops.mix_samples(self.task_mean, G, self._mixing(), E, R, ns, S)
        return out.reshape(*sample_shape, ns, p).to(self.dtype)

    def sample_latents(self, normals):
        """Latent draws mean_l + chol(C_l) normals_l for given normals [q, n*, S] (deterministic)."""
        self._no_nan_inputs()
        lat_mean, C = self._latent()
        eng = self.model._engine
        with torch.no_grad():
            if self._factor is None:
                self._factor = eng.factor_covariance(C, self.xs.shape[0])
            return eng.sample_latents(lat_mean, *self._factor, _as_f64(normals).contiguous())

    def log_prob(self, value, task_noise):
        self._no_nan_inputs()
        _, C = self._latent()
        ns, p = self.xs.shape[0], self.model.n_tasks
        if value.shape[-2:] != (ns, p):
            raise ValueError(f"log_prob expects values of shape [..., {ns}, {p}], got {tuple(value.shape)}")
        batch = value.shape[:-2]
        with torch.no_grad():
            vals = _as_f64(value).reshape(-1, ns, p)
            S = (0.5 * (task_noise + task_noise.T)).contiguous()
            lp = self.model._engine.joint_log_prob(C, self._mixing(), S, self.task_mean, vals)
        return lp.reshape(batch).to(value.dtype)


def _as_f64(t: Tensor) -> Tensor:
    return t if t.dtype == torch.float64 else t.to(torch.float64)
