"""torch.autograd glue around the CUDA engine (no arithmetic of its own)."""
from __future__ import annotations

import torch

from . import ops


def ops_components(spec, tensors):
    """[ops.Component (kernel id, dims, ell, os | None; shape parameter | None)] from the flat (spec, tensors) form
    used across the autograd boundary.  A spec entry is (kid, dims, has_os) or (kid, dims, has_os, has_shape)."""
    out, i = [], 0
    for kid, dims, has_os, *rest in spec:
        ell = tensors[i]
        i += 1
        os_ = shape = None
        if has_os:
            os_ = tensors[i]
            i += 1
        if rest and rest[0]:
            shape = tensors[i]
            i += 1
        out.append(ops.Component(kid, dims, ell, os_, shape))
    return out


class ProjectData(torch.autograd.Function):
    """TY = T^T Y^T  (kernel 1).  Gradient flows to T only (Y is data)."""

    @staticmethod
    def forward(ctx, T: torch.Tensor, Y: torch.Tensor) -> torch.Tensor:
        T64 = T.detach().to(torch.float64).contiguous()
        ctx.Y = Y
        ctx.in_dtype = T.dtype
        return ops.project_fwd(Y, T64)

    @staticmethod
    def backward(ctx, G: torch.Tensor):
        dT = ops.project_bwd(ctx.Y, G.contiguous())
        return dT.to(ctx.in_dtype), None


class LatentLogProb(torch.autograd.Function):
    """lp_l = log N(TY_l; 0, sum_g o_gl k_gl(X,X) + noise_l I), batched over latents (kernels 2-4).

    ``spec`` = ((kernel id, active dims, has outputscale, has shape parameter), ...) describes the additive kernel;
    ``tensors`` are its parameters in order (ell_0 [q, d_0], os_0 [q] if any, alpha_0 [q] if any (RQ), ell_1, ...).  The backward quantities are produced
    eagerly in forward (K -> L -> K^-1 is done in place in one cached workspace, so nothing of size n^2 is saved
    for backward)."""

    @staticmethod
    def forward(ctx, engine, X, spec, TY, noise, *tensors):
        need = any(t is not None and t.requires_grad for t in (TY, noise, *tensors))
        comps = ops_components(spec, [t.detach().contiguous() for t in tensors])
        lp, grads = engine.log_prob_and_grads(X, TY.detach().contiguous(), comps, noise.detach().contiguous(), need)
        ctx.grads = grads
        return lp

    @staticmethod
    def backward(ctx, go):
        if ctx.grads is None:
            raise RuntimeError("LatentLogProb.backward called but no input required grad in forward")
        g_ty, g_noise, g_tensors = ctx.grads
        ctx.grads = None
        out = [(g * go[:, None]) if g.dim() == 2 else (g * go) for g in g_tensors]
        return (None, None, None, g_ty * go[:, None], g_noise * go, *out)
