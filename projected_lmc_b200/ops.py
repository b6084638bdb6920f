"""Thin torch-tensor wrappers over the C ABI (one Python function per entry point).

Every wrapper takes CUDA float64 tensors, launches on the current stream of the device that owns
them and returns immediately (no synchronisation).  Shapes follow include/plmc_b200.h.
"""
from __future__ import annotations

import ctypes
import functools

import torch

from . import _cabi
from ._cabi import (GEMM_FLAG_SINGLE_CTA, GEMM_FP64, GEMM_INT8_DIGITS, GEMM_INT8_RNS, GemmCfg, PlmcError, check, lib,
                    npad, ptr, stream)

KERNEL_IDS = {"rbf": 0, "matern52": 1, "matern32": 2, "matern12": 3, "rq": 4}
KERNEL_RQ = 4
# kernels with a shape parameter (one value per latent): the ...2 entry points carry it
SHAPED_KERNELS = frozenset({KERNEL_RQ})


class Component(tuple):
    """One additive kernel component, (kernel id, dims, ell [q, d_g], os [q] | None), with the kernel's shape
    parameter [q] (RQ: alpha) as ``.shape_param``.  It unpacks as the plain 4-tuple of the kernels without one,
    which callers may keep using."""

    def __new__(cls, kid, dims, ell, os_, shape_param=None):
        self = super().__new__(cls, (kid, dims, ell, os_))
        self.shape_param = shape_param
        return self


def shape_of(comp):
    """The shape parameter of a component (None for a plain 4-tuple or a kernel without one)."""
    return getattr(comp, "shape_param", None)

# layout codes of plmc_gemm: bit1 -> A(m,k) m-contiguous, bit0 -> B(k,n) n-contiguous
A_KC_B_KC, A_KC_B_NC, A_MC_B_KC, A_MC_B_NC = 0, 1, 2, 3


def _on_device(fn):
    """Run the wrapped call with the device of its tensor arguments current (the library launches on the
    current device and its current stream); tensors on different devices are an error."""

    @functools.wraps(fn)
    def wrapper(*args, **kwargs):
        dev = None
        for a in args:
            if isinstance(a, torch.Tensor):
                if not a.is_cuda:
                    raise PlmcError("libplmc_b200 was handed a non-CUDA tensor; there is no CPU fallback")
                if dev is None:
                    dev = a.device
                elif a.device != dev:
                    raise PlmcError(f"libplmc_b200 call with tensors on different devices: {dev} and {a.device}")
        if dev is None or dev.index == torch.cuda.current_device():
            return fn(*args, **kwargs)
        with torch.cuda.device(dev):
            return fn(*args, **kwargs)

    return wrapper


def gemm_cfg(ws, mode: int, precision: int, min_dim: int = 512, flags: int = 0, alt_precision: int = 0,
             rns_min_k: int = 0, rns_min_mnk: int = 0, min_mnk: int = 0):
    """plmc_gemm_cfg for the factorisation calls (None = pure FP64).  The struct keeps its scratch tensor alive."""
    if ws is None or mode == GEMM_FP64 or precision <= 0:
        return None
    cfg = GemmCfg(ptr(ws), ws.numel() * ws.element_size(), int(mode), int(precision), max(128, int(min_dim)),
                  int(flags), int(alt_precision), int(rns_min_k), int(rns_min_mnk), int(min_mnk))
    cfg._keepalive = ws
    return cfg


def _cfgp(cfg):
    return None if cfg is None else ctypes.byref(cfg)


def _bstride(t: torch.Tensor) -> int:
    return t.stride(0) if t.dim() == 3 else 0


@_on_device
def gemm(layout, A, B, C, M, N, K, alpha=1.0, beta=0.0, lower=False, triA=False, triB=False):
    """C[b] = alpha * op(A[b]) op(B[b]) + beta * C[b]; A, B, C are [batch, rows, ld] views."""
    batch = C.shape[0]
    check(
        lib().plmc_gemm(
            layout, ptr(A), A.stride(-2), _bstride(A), ptr(B), B.stride(-2), _bstride(B), ptr(C), C.stride(-2),
            _bstride(C), M, N, K, float(alpha), float(beta), int(lower), int(triA), int(triB), batch, stream(),
        ),
        "plmc_gemm",
    )
    return C


def alloc_dinv(np_: int, batch: int, device) -> torch.Tensor:
    """Side buffer of the factorisation calls: [batch, plmc_dinv_bytes / 8] (leaf inverses + dense-block scratch)."""
    per = _cabi.load().plmc_dinv_bytes(np_, 1) // 8
    return torch.empty((batch, per), dtype=torch.float64, device=device)


@_on_device
def potrf(K: torch.Tensor, dinv: torch.Tensor, info: torch.Tensor, cfg=None):
    """In-place lower Cholesky of K [batch, npad, ld]; info int32 [batch]."""
    b, np_, _ = K.shape
    check(lib().plmc_potrf_batched(ptr(K), K.stride(1), K.stride(0), np_, b, ptr(dinv), ptr(info), _cfgp(cfg),
                                   stream()), "potrf")


@_on_device
def trsm(op: int, L, dinv, B, alpha=1.0, cfg=None):
    """op 0: X L^T = aB | 1: X L = aB (B [batch, m, npad]) | 2: L X = aB | 3: L^T X = aB (B [batch, npad, m])."""
    b, np_, _ = L.shape
    m = B.shape[1] if op in (0, 1) else B.shape[2]
    check(
        lib().plmc_trsm_batched(
            op, ptr(L), L.stride(1), L.stride(0), np_, b, ptr(dinv), ptr(B), B.stride(1), B.stride(0), m,
            float(alpha), _cfgp(cfg), stream(),
        ),
        "trsm",
    )


@_on_device
def trmm(op: int, X, dinv, B, alpha=1.0, cfg=None):
    """In place, X lower triangular [batch, npad, npad] (e.g. inv(L) from trtri): op 1 B := a B X (B [batch, m, npad]),
    op 2 B := a X B, op 3 B := X^T B (B [batch, npad, m]); the dense-block scratch part of dinv is overwritten."""
    b, np_, _ = X.shape
    check(
        lib().plmc_trmm_batched(
            op, ptr(X), X.stride(1), X.stride(0), np_, b, ptr(dinv), ptr(B), B.stride(1), B.stride(0),
            B.shape[1] if op == 1 else B.shape[2],
            float(alpha), _cfgp(cfg), stream(),
        ),
        "trmm",
    )


@_on_device
def solve_logdet(L, dinv, y, n, rhs=None):
    """z = L^-1 y, alpha = L^-T z, |z|^2, 2 sum log L_ii for y [batch, >=n]."""
    b, np_, _ = L.shape
    dev = L.device
    if rhs is None:
        rhs = torch.empty((b, np_, 128), dtype=torch.float64, device=dev)
    z = torch.empty((b, n), dtype=torch.float64, device=dev)
    alpha = torch.empty((b, n), dtype=torch.float64, device=dev)
    quad = torch.empty((b,), dtype=torch.float64, device=dev)
    logdet = torch.empty((b,), dtype=torch.float64, device=dev)
    check(
        lib().plmc_solve_logdet(
            ptr(L), L.stride(1), L.stride(0), n, np_, b, ptr(dinv), ptr(y), y.stride(0), ptr(rhs), ptr(z), ptr(alpha),
            n, ptr(quad), ptr(logdet), stream(),
        ),
        "solve_logdet",
    )
    return z, alpha, quad, logdet


@_on_device
def trtri(L, dinv, cfg=None):
    b, np_, _ = L.shape
    check(lib().plmc_trtri_batched(ptr(L), L.stride(1), L.stride(0), np_, b, ptr(dinv), _cfgp(cfg), stream()), "trtri")


@_on_device
def lauum(L, dinv, cfg=None):
    b, np_, _ = L.shape
    check(lib().plmc_lauum_batched(ptr(L), L.stride(1), L.stride(0), np_, b, ptr(dinv), _cfgp(cfg), stream()), "lauum")


@_on_device
def potri(L, dinv, cfg=None):
    b, np_, _ = L.shape
    check(lib().plmc_potri_batched(ptr(L), L.stride(1), L.stride(0), np_, b, ptr(dinv), _cfgp(cfg), stream()), "potri")


@_on_device
def project_fwd(Y: torch.Tensor, T: torch.Tensor) -> torch.Tensor:
    n, p = Y.shape
    q = T.shape[1]
    TY = torch.empty((q, n), dtype=torch.float64, device=Y.device)
    check(lib().plmc_project_fwd(ptr(Y), ptr(T), ptr(TY), n, p, q, n, stream()), "project_fwd")
    return TY


@_on_device
def project_bwd(Y: torch.Tensor, G: torch.Tensor) -> torch.Tensor:
    n, p = Y.shape
    q = G.shape[0]
    ws = torch.empty((lib().plmc_project_bwd_ws(n, p, q) // 8,), dtype=torch.float64, device=Y.device)
    dT = torch.empty((p, q), dtype=torch.float64, device=Y.device)
    check(lib().plmc_project_bwd(ptr(Y), ptr(G), G.stride(0), ptr(dT), ptr(ws), n, p, q, stream()), "project_bwd")
    return dT


def dpad_of(d: int) -> int:
    return ((d + 3) // 4) * 4


@_on_device
def col_mean(X: torch.Tensor) -> torch.Tensor:
    n, d = X.shape
    out = torch.empty((d,), dtype=torch.float64, device=X.device)
    check(lib().plmc_col_mean(ptr(X), n, d, ptr(out), stream()), "col_mean")
    return out


@_on_device
def scale_inputs(X, xmean, ell, rows_pad):
    """Z [q, rows_pad, dpad], zn [q, rows_pad]."""
    n, d = X.shape
    q = ell.shape[0]
    dp = dpad_of(d)
    Z = torch.empty((q, rows_pad, dp), dtype=torch.float64, device=X.device)
    zn = torch.empty((q, rows_pad), dtype=torch.float64, device=X.device)
    check(lib().plmc_scale_inputs(ptr(X), ptr(xmean), ptr(ell), ptr(Z), ptr(zn), n, d, dp, rows_pad, q, stream()),
          "scale_inputs")
    return Z, zn


def _check_shape(kernel_id, shape):
    if (kernel_id in SHAPED_KERNELS) != (shape is not None):
        raise PlmcError(f"kernel {kernel_id}: a shape parameter is required by the rational quadratic kernel and "
                        "refused by the others")


@_on_device
def gram(Z, zn, kernel_id, os_, diag_add, K, n, accumulate=False, *, shape=None):
    """shape: the kernel's shape parameter [q] (RQ alpha), None for kernels without one."""
    _check_shape(kernel_id, shape)
    q, np_, dp = Z.shape
    check(
        lib().plmc_gram2(ptr(Z), ptr(zn), kernel_id, ptr(os_), ptr(shape), ptr(diag_add), ptr(K), K.stride(1),
                         K.stride(0), n, np_, dp, q, int(accumulate), stream()),
        "gram",
    )


@_on_device
def cross_gram(Ztr, zntr, Zte, znte, kernel_id, os_, Kx, n, mt, accumulate=False, *, shape=None):
    _check_shape(kernel_id, shape)
    q, np_, dp = Ztr.shape
    check(
        lib().plmc_cross_gram2(ptr(Ztr), ptr(zntr), ptr(Zte), ptr(znte), kernel_id, ptr(os_), ptr(shape), ptr(Kx),
                               Kx.stride(1), Kx.stride(0), n, np_, Zte.shape[1], mt, dp, q, int(accumulate), stream()),
        "cross_gram",
    )


@_on_device
def cross_gram_bwd(Zr, Zc, G, kernel_id, os_, ell, nr, nc, *, shape=None):
    """Adjoint of K[l,i,j] = os[l] k(|zr_i - zc_j|^2) for the cotangent G [q, nr, >=nc]:
    (g_ell [q, d], g_os [q], g_rows [nr, d] summed over latents, w.r.t. the unscaled row points), and g_shape [q]
    appended when the kernel has a shape parameter."""
    _check_shape(kernel_id, shape)
    q, rpr, dp = Zr.shape
    rpc = Zc.shape[1]
    d = ell.shape[1]
    dev = G.device
    ws = torch.empty((lib().plmc_cross_gram_bwd_ws2(nr, nc, d, q, kernel_id) // 8,), dtype=torch.float64, device=dev)
    g_ell = torch.empty((q, d), dtype=torch.float64, device=dev)
    g_os = torch.empty((q,), dtype=torch.float64, device=dev)
    g_rows = torch.empty((nr, d), dtype=torch.float64, device=dev)
    g_shape = None if shape is None else torch.empty((q,), dtype=torch.float64, device=dev)
    check(
        lib().plmc_cross_gram_bwd2(ptr(Zr), rpr, ptr(Zc), rpc, ptr(G), G.stride(1), G.stride(0), kernel_id, ptr(os_),
                                   ptr(shape), ptr(ell), ptr(g_ell), ptr(g_os), ptr(g_shape), ptr(g_rows), ptr(ws), nr,
                                   nc, d, dp, q, stream()),
        "cross_gram_bwd",
    )
    return (g_ell, g_os, g_rows) if shape is None else (g_ell, g_os, g_rows, g_shape)


@_on_device
def grad_sweep(Kinv, alpha, Z, zn, ell, kernel_id, os_, n, *, shape=None):
    """(g_ell, g_os, g_noise), and g_shape [q] appended when the kernel has a shape parameter."""
    _check_shape(kernel_id, shape)
    q, np_, dp = Z.shape
    d = ell.shape[1]
    dev = Kinv.device
    ws = torch.empty((lib().plmc_grad_ws2(np_, d, q, kernel_id) // 8,), dtype=torch.float64, device=dev)
    g_ell = torch.empty((q, d), dtype=torch.float64, device=dev)
    g_os = torch.empty((q,), dtype=torch.float64, device=dev)
    g_noise = torch.empty((q,), dtype=torch.float64, device=dev)
    g_shape = None if shape is None else torch.empty((q,), dtype=torch.float64, device=dev)
    check(
        lib().plmc_grad_sweep2(ptr(Kinv), Kinv.stride(1), Kinv.stride(0), ptr(alpha), alpha.stride(0), ptr(Z), ptr(zn),
                               ptr(ell), kernel_id, ptr(os_), ptr(shape), ptr(g_ell), ptr(g_os), ptr(g_noise),
                               ptr(g_shape), ptr(ws), n, np_, d, dp, q, stream()),
        "grad_sweep",
    )
    return (g_ell, g_os, g_noise) if shape is None else (g_ell, g_os, g_noise, g_shape)


@_on_device
def latent_mean(Kx, alpha, n, mt):
    q = Kx.shape[0]
    out = torch.empty((q, mt), dtype=torch.float64, device=Kx.device)
    check(lib().plmc_latent_mean(ptr(Kx), Kx.stride(1), Kx.stride(0), ptr(alpha), alpha.stride(0), ptr(out), mt, n, mt,
                                 q, stream()), "latent_mean")
    return out


@_on_device
def latent_var(V, os_, mt):
    q, np_, _ = V.shape
    out = torch.empty((q, mt), dtype=torch.float64, device=V.device)
    check(lib().plmc_latent_var(ptr(V), V.stride(1), V.stride(0), ptr(os_), ptr(out), mt, np_, mt, q, stream()),
          "latent_var")
    return out


@_on_device
def mix_tasks(lat_mean, lat_var, H, var_add, mean, var, mt, accumulate=False):
    q, p = H.shape
    check(lib().plmc_mix_tasks(ptr(lat_mean), ptr(lat_var), lat_mean.stride(0), ptr(H), ptr(var_add), ptr(mean),
                               ptr(var), mt, p, q, int(accumulate), stream()), "mix_tasks")


@_on_device
def syrk(A, C, alpha=1.0, beta=0.0, cfg=None):
    """lower(C[b]) = alpha A[b]^T A[b] + beta C[b] for A [batch, k, >=n], C [batch, n, ld] (n, k multiples of 128)."""
    b, n, _ = C.shape
    check(lib().plmc_syrk_batched(ptr(A), A.stride(1), A.stride(0), ptr(C), C.stride(1), C.stride(0), n, A.shape[1],
                                  float(alpha), float(beta), b, _cfgp(cfg), stream()), "syrk")


@_on_device
def task_covariance(C, H, S, ns, tiled=False):
    """Task-level covariance from the lower tiles of C [q, m, m]: dense [ns p, ns p], or (tiled) the lower 128-tiles of
    a [1, npad(ns p), npad(ns p)] matrix with identity padding."""
    q, p = H.shape
    N = ns * p
    T = torch.empty((1, npad(N), npad(N)) if tiled else (N, N), dtype=torch.float64, device=C.device)
    check(lib().plmc_task_covariance(ptr(C), C.stride(1), C.stride(0), ptr(H), ptr(S), ptr(T), T.stride(-2), ns, p, q,
                                     int(tiled), stream()), "task_covariance")
    return T


@_on_device
def mix_samples(mean, G, H, E, R, ns, S):
    """out [S, ns, p] = mean + (latent draws G [q, >=ns, >=S] mixed by H) + E R^T."""
    q, p = H.shape
    out = torch.empty((S, ns, p), dtype=torch.float64, device=G.device)
    check(lib().plmc_mix_samples(ptr(mean), ptr(G), G.stride(1), G.stride(0), ptr(H), ptr(E), ptr(R), ptr(out), ns, S,
                                 p, q, stream()), "mix_samples")
    return out


@_on_device
def peak_dmma(blocks, threads, iters, scratch):
    check(lib().plmc_peak_dmma(blocks, threads, iters, ptr(scratch), stream()), "peak_dmma")
    return blocks * (threads // 32) * iters * 16 * 512


@_on_device
def peak_dfma(blocks, threads, iters, scratch):
    check(lib().plmc_peak_dfma(blocks, threads, iters, ptr(scratch), stream()), "peak_dfma")
    return blocks * threads * iters * 16 * 2


@_on_device
def peak_copy(src, dst):
    n = src.numel()
    check(lib().plmc_peak_copy(ptr(src), ptr(dst), n, stream()), "peak_copy")
    return 16 * n


@_on_device
def peak_i8(iters, scratch, cta_group=2):
    """Shared-memory-resident tcgen05.mma.kind::i8 loop on every SM: returns the INT8 operations issued."""
    ops_ = ctypes.c_double(0.0)
    check(lib().plmc_peak_i8(int(iters), int(cta_group), ptr(scratch), ctypes.byref(ops_), stream()), "peak_i8")
    return ops_.value


def stats_reset():
    check(_cabi.load().plmc_stats_reset(), "stats_reset")


def stats_add(launches: int):
    check(_cabi.load().plmc_stats_add(int(launches)), "stats_add")


def sweep_debug(direct: bool):
    """Diagnostics: force the direct-difference gradient sweep (the kernel for d > 24) for every input dimension."""
    check(_cabi.load().plmc_sweep_debug(int(bool(direct))), "sweep_debug")


def trace_enable(on: bool):
    """Per-shape CUDA-event timing of every GEMM of the factorisation layer (diagnostics)."""
    check(_cabi.load().plmc_trace_enable(int(bool(on))), "trace_enable")


def trace_report():
    check(_cabi.load().plmc_trace_report(), "trace_report")


def stats_get():
    """(kernel launches, GEMM launches, GEMM algorithmic FLOPs) since the last reset."""
    a, b, c = ctypes.c_longlong(0), ctypes.c_longlong(0), ctypes.c_double(0.0)
    check(_cabi.load().plmc_stats_get(ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)), "stats_get")
    return a.value, b.value, c.value


@_on_device
def ozaki_gemm(layout, A, B, C, M, N, K, alpha=1.0, beta=0.0, lower=False, slices=7, same_operand=False, ws=None):
    """C = alpha op(A) op(B) + beta C (2-D views) on the tcgen05 INT8 path (FP64 via 8-bit digit planes)."""
    need = lib().plmc_ozaki_ws_bytes(M, N, K, slices, int(same_operand))
    if ws is None or ws.numel() < need:
        ws = torch.empty((need,), dtype=torch.uint8, device=C.device)
    check(
        lib().plmc_ozaki_gemm(layout, ptr(A), A.stride(-2), ptr(B), B.stride(-2), ptr(C), C.stride(-2), M, N, K,
                              float(alpha), float(beta), int(lower), slices, int(same_operand), ptr(ws), ws.numel(),
                              stream()),
        "ozaki_gemm",
    )
    return C


def rns_bits(moduli: int, K: int) -> int:
    return int(_cabi.load().plmc_rns_bits(int(moduli), int(K)))


@_on_device
def rns_gemm(layout, A, B, C, M, N, K, alpha=1.0, beta=0.0, lower=False, moduli=16, same_operand=False, ws=None,
             flags=0):
    """C = alpha op(A) op(B) + beta C (2-D views) on the tcgen05 INT8 path, residue-number-system scheme."""
    if ws is None:
        need = lib().plmc_rns_ws_bytes(M, N, K, moduli, int(same_operand), int(lower))
        ws = torch.empty((need,), dtype=torch.uint8, device=C.device)
    check(
        lib().plmc_rns_gemm(layout, ptr(A), A.stride(-2), ptr(B), B.stride(-2), ptr(C), C.stride(-2), M, N, K,
                            float(alpha), float(beta), int(lower), int(moduli), int(same_operand), ptr(ws), ws.numel(),
                            int(flags), stream()),
        "rns_gemm",
    )
    return C
