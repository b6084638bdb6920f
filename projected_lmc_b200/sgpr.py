"""Inducing-point (SGPR, Titsias 2009) latent GPs: ``ExactGPModel(..., n_inducing_points=m)`` wraps the kernel in
gpytorch's ``InducingPointKernel`` (projected_lmc.py:302-303; used with m = 500 for the ship / SARCOS runs,
realdata_experiments.py:398,505).  Semantics restated from gpytorch 1.11:

  training:  covar = Q_ff = K_fu K_uu^-1 K_uf  (low rank), likelihood adds sigma^2 I;
             log N(y; 0, Q_ff + sigma^2 I)  +  added loss term  -1/2 sum_i (k_ii - q_ii) / sigma^2
  eval:      the train block gains the diagonal correction diag(k_ii - q_ii) (clamped at 0), the test diagonal too;
             exact-GP prediction under that covariance.

Everything is O(n m^2): the kernel blocks K_uf / K_uu and their adjoints run in libplmc_b200 (csrc/gram.cu forward,
csrc/sgpr.cu backward -- no dK/dtheta is materialised); the m x m Cholesky factors, the two n x m triangular solves
and the Gram product are plain library calls in torch (autograd handles them), in float64."""
from __future__ import annotations

import math
import warnings

import torch

from . import ops
from ._cabi import npad as _npad
from .gp import settings


class CrossGram(torch.autograd.Function):
    """K[l, i, j] = os_l k(|(u_i - x_j) / ell_l|^2): rows = points U [m, d] (differentiable), columns = data X [n, d].
    ``symmetric``: X is U itself (K_uu); the adjoint then accounts for both roles of U.  ``shape``: the kernel's
    shape parameter [q] (RQ alpha), None for kernels without one."""

    @staticmethod
    def forward(ctx, U, X, xmean, kid, ell, os_, symmetric, shape=None):
        m, n = U.shape[0], X.shape[0]
        Ud, ed = U.detach().contiguous(), ell.detach().contiguous()
        od = None if os_ is None else os_.detach().contiguous()
        ad = None if shape is None else shape.detach().contiguous()
        mp, np_ = _npad(m), _npad(n)
        Zr, znr = ops.scale_inputs(Ud, xmean, ed, mp)
        Zc, znc = (Zr, znr) if symmetric else ops.scale_inputs(X.detach().contiguous(), xmean, ed, np_)
        Kx = torch.empty((ed.shape[0], mp, np_), dtype=torch.float64, device=U.device)
        ops.cross_gram(Zr, znr, Zc, znc, kid, od, Kx, m, np_, shape=ad)
        empty = torch.empty(0, device=U.device)
        ctx.save_for_backward(Zr, Zc, ed, od if od is not None else empty, ad if ad is not None else empty)
        ctx.meta = (kid, m, n, od is not None, symmetric, ad is not None)
        return Kx[:, :m, :n]

    @staticmethod
    def backward(ctx, G):
        Zr, Zc, ell, os_, shape = ctx.saved_tensors
        kid, m, n, has_os, symmetric, has_shape = ctx.meta
        G = G.contiguous()
        if symmetric:
            G = G + G.transpose(1, 2)
        g = ops.cross_gram_bwd(Zr, Zc, G, kid, os_ if has_os else None, ell, m, n,
                               shape=shape if has_shape else None)
        g_ell, g_os, g_rows = g[0], g[1], g[2]
        g_shape = g[3] if has_shape else None
        if symmetric:   # each unordered pair was counted twice in the lengthscale / outputscale / shape sums
            g_ell, g_os = 0.5 * g_ell, 0.5 * g_os
            g_shape = None if g_shape is None else 0.5 * g_shape
        return g_rows, None, None, None, g_ell, (g_os if has_os else None), None, g_shape


def _chol_safe(A: torch.Tensor, max_tries: int):
    """linear_operator psd_safe_cholesky: plain factorisation first, then jitter 1e-8 * 10^i on failing members."""
    L, info = torch.linalg.cholesky_ex(A)
    if not bool(info.any()):
        return L
    base = settings.cholesky_jitter.value()
    eye = torch.eye(A.shape[-1], dtype=A.dtype, device=A.device)
    Ap, prev = A, 0.0
    for i in range(max_tries):
        new = base * (10 ** i)
        Ap = Ap + ((info > 0).to(A.dtype) * (new - prev))[:, None, None] * eye
        prev = new
        warnings.warn(f"A not p.d., added jitter of {new:.1e} to the diagonal", RuntimeWarning)
        L, info = torch.linalg.cholesky_ex(Ap)
        if not bool(info.any()):
            return L
    raise RuntimeError(f"Matrix not positive definite after repeatedly adding jitter up to {new:.1e}.")


def _blocks(engine, X, U, comps):
    """(K_uu [q, m, m], K_uf [q, m, n], prior variance [q]) of the additive kernel."""
    Kuu = Kuf = kss = None
    for c in comps:
        kid, dims, ell, os_ = c
        Xg, xm = engine._sub_inputs(X, dims)
        Ug = U if len(dims) == U.shape[1] and tuple(dims) == tuple(range(U.shape[1])) else U[:, list(dims)]
        a = CrossGram.apply(Ug, Ug, xm, kid, ell, os_, True, ops.shape_of(c))
        b = CrossGram.apply(Ug, Xg, xm, kid, ell, os_, False, ops.shape_of(c))
        v = torch.ones(ell.shape[0], dtype=torch.float64, device=X.device) if os_ is None else os_
        Kuu, Kuf, kss = (a, b, v) if Kuu is None else (Kuu + a, Kuf + b, kss + v)
    return Kuu, Kuf, kss


def latent_log_prob(engine, X, TY, U, comps, noise, max_tries=None):
    """(lp [q], added loss [q]): log N(TY_l; 0, Q_l + noise_l I) and -1/2 sum_i (k_ii - q_ii) / noise_l."""
    if max_tries is None:
        max_tries = settings.cholesky_max_tries.value()
    n = X.shape[0]
    Kuu, Kuf, kss = _blocks(engine, X, U, comps)
    Luu = _chol_safe(Kuu, max_tries)
    A = torch.linalg.solve_triangular(Luu, Kuf, upper=False)                       # L_uu^-1 K_uf   [q, m, n]
    s2 = noise
    eye = torch.eye(A.shape[1], dtype=A.dtype, device=A.device)
    B = eye + (A @ A.transpose(1, 2)) / s2[:, None, None]
    LB = torch.linalg.cholesky(B)
    Ay = (A @ TY.unsqueeze(-1))                                                     # [q, m, 1]
    c = torch.linalg.solve_triangular(LB, Ay, upper=False).squeeze(-1)
    quad = (TY ** 2).sum(-1) / s2 - (c ** 2).sum(-1) / s2 ** 2
    logdet = n * torch.log(s2) + 2.0 * torch.log(torch.diagonal(LB, dim1=1, dim2=2)).sum(-1)
    lp = -0.5 * (quad + logdet + n * math.log(2 * math.pi))
    added = -0.5 * (n * kss - (A ** 2).sum((1, 2))) / s2
    return lp, added


def prediction_state(engine, X, TY, U, comps, noise, max_tries=None):
    if max_tries is None:
        max_tries = settings.cholesky_max_tries.value()
    Kuu, Kuf, kss = _blocks(engine, X, U, comps)
    Luu = _chol_safe(Kuu, max_tries)
    A = torch.linalg.solve_triangular(Luu, Kuf, upper=False)
    D = (kss[:, None] - (A ** 2).sum(1)).clamp_min(0.0) + noise[:, None]            # diagonal correction + noise  [q, n]
    AD = A / D[:, None, :]
    eye = torch.eye(A.shape[1], dtype=A.dtype, device=A.device)
    LB = _chol_safe(eye + AD @ A.transpose(1, 2), max_tries)
    w = torch.cholesky_solve(AD @ TY.unsqueeze(-1), LB)                              # B_d^-1 A D^-1 y   [q, m, 1]
    return dict(Luu=Luu, LB=LB, w=w, kss=kss, U=U, comps=comps)


def predict_latents(engine, st, X, Xs, tile=65536, test_rows=False):
    """Latent posterior means / variances at Xs under the eval-mode SGPR covariance: ([q, n*], [q, n*]).
    ``test_rows``: the cross block is built with the test points as the rows of CrossGram (and transposed), so that
    torch autograd reaches Xs through the block's adjoint."""
    q = st["kss"].shape[0]
    ns = Xs.shape[0]
    mean = torch.empty((q, ns), dtype=torch.float64, device=Xs.device)
    var = torch.empty((q, ns), dtype=torch.float64, device=Xs.device)
    U = st["U"]
    for s0 in range(0, ns, tile):
        xs = Xs[s0:s0 + tile]
        Kus = None
        for c in st["comps"]:
            kid, dims, ell, os_ = c
            _, xm = engine._sub_inputs(X, dims)
            full = len(dims) == U.shape[1] and tuple(dims) == tuple(range(U.shape[1]))
            Ug, xg = (U, xs) if full else (U[:, list(dims)], xs[:, list(dims)].contiguous())
            if test_rows:
                b = CrossGram.apply(xg, Ug, xm, kid, ell, os_, False, ops.shape_of(c)).transpose(1, 2)
            else:
                b = CrossGram.apply(Ug, xg, xm, kid, ell, os_, False, ops.shape_of(c))
            Kus = b if Kus is None else Kus + b
        As = torch.linalg.solve_triangular(st["Luu"], Kus, upper=False)                      # [q, m, t]
        mean[:, s0:s0 + tile] = (As * st["w"]).sum(1)
        V = torch.linalg.solve_triangular(st["LB"], As, upper=False)
        qss = (As ** 2).sum(1)
        kstar = torch.maximum(st["kss"][:, None], qss)                                       # clamp(k** - q**, 0) + q**
        var[:, s0:s0 + tile] = kstar - qss + (V ** 2).sum(1)
    return mean, var
