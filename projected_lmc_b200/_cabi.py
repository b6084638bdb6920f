"""ctypes binding of libplmc_b200.so (the C ABI declared in include/plmc_b200.h).

There is no CPU fallback: if the shared library is missing or a tensor is not a
CUDA tensor the call raises.  PyTorch is used only for device memory and the
current stream.
"""
from __future__ import annotations

import ctypes
from ctypes import c_double, c_int, c_longlong, c_void_p
from pathlib import Path

import torch

_LIB_PATH = Path(__file__).resolve().parent / "libplmc_b200.so"
_lib = None
_inited_devices = set()

P, LL, I, D = c_void_p, c_longlong, c_int, c_double

GEMM_FP64, GEMM_INT8_DIGITS, GEMM_INT8_RNS = 0, 1, 2
GEMM_FLAG_SINGLE_CTA = 1


class GemmCfg(ctypes.Structure):
    """plmc_gemm_cfg (include/plmc_b200.h): per-call arithmetic of the large GEMMs of the factorisation layer."""
    _fields_ = [("ws", c_void_p), ("ws_bytes", c_longlong), ("mode", c_int), ("precision", c_int),
                ("min_dim", c_int), ("flags", c_int), ("alt_precision", c_int), ("rns_min_k", c_int),
                ("rns_min_mnk", c_longlong), ("min_mnk", c_longlong)]


CFG = ctypes.POINTER(GemmCfg)

# name -> argtypes (restype is int unless listed in _RET_LL)
_SIGNATURES = {
    "plmc_version": [],
    "plmc_init": [],
    "plmc_stats_reset": [],
    "plmc_stats_add": [LL],
    "plmc_trace_enable": [I],
    "plmc_ozaki_debug": [P],
    "plmc_trace_report": [],
    "plmc_stats_get": [P, P, P],
    "plmc_npad": [LL],
    "plmc_dinv_bytes": [LL, I],
    "plmc_project_fwd": [P, P, P, LL, I, I, LL, P],
    "plmc_project_bwd_ws": [LL, I, I],
    "plmc_project_bwd": [P, P, LL, P, P, LL, I, I, P],
    "plmc_kernel_profile_host": [I, P, LL, P, P],
    "plmc_kernel_profile2_host": [I, P, P, LL, P, P, P],
    "plmc_log1p_host": [P, LL, P],
    "plmc_sqrt_reciprocal_host": [P, LL, P, P],
    "plmc_col_mean": [P, LL, I, P, P],
    "plmc_scale_inputs": [P, P, P, P, P, LL, I, I, LL, I, P],
    "plmc_gram": [P, P, I, P, P, P, LL, LL, LL, LL, I, I, I, P],
    "plmc_cross_gram": [P, P, P, P, I, P, P, LL, LL, LL, LL, LL, LL, I, I, I, P],
    "plmc_cross_gram_bwd_ws": [LL, LL, I, I],
    "plmc_cross_gram_bwd": [P, LL, P, LL, P, LL, LL, I, P, P, P, P, P, P, LL, LL, I, I, I, P],
    "plmc_gram2": [P, P, I, P, P, P, P, LL, LL, LL, LL, I, I, I, P],
    "plmc_cross_gram2": [P, P, P, P, I, P, P, P, LL, LL, LL, LL, LL, LL, I, I, I, P],
    "plmc_cross_gram_bwd_ws2": [LL, LL, I, I, I],
    "plmc_cross_gram_bwd2": [P, LL, P, LL, P, LL, LL, I, P, P, P, P, P, P, P, P, LL, LL, I, I, I, P],
    "plmc_potrf_batched": [P, LL, LL, LL, I, P, P, CFG, P],
    "plmc_trsm_batched": [I, P, LL, LL, LL, I, P, P, LL, LL, LL, D, CFG, P],
    "plmc_trmm_batched": [I, P, LL, LL, LL, I, P, P, LL, LL, LL, D, CFG, P],
    "plmc_solve_logdet": [P, LL, LL, LL, LL, I, P, P, LL, P, P, P, LL, P, P, P],
    "plmc_trtri_batched": [P, LL, LL, LL, I, P, CFG, P],
    "plmc_lauum_batched": [P, LL, LL, LL, I, P, CFG, P],
    "plmc_potri_batched": [P, LL, LL, LL, I, P, CFG, P],
    "plmc_grad_ws": [LL, I, I],
    "plmc_sweep_debug": [I],
    "plmc_grad_sweep": [P, LL, LL, P, LL, P, P, P, I, P, P, P, P, P, LL, LL, I, I, I, P],
    "plmc_grad_ws2": [LL, I, I, I],
    "plmc_grad_sweep2": [P, LL, LL, P, LL, P, P, P, I, P, P, P, P, P, P, P, LL, LL, I, I, I, P],
    "plmc_latent_mean": [P, LL, LL, P, LL, P, LL, LL, LL, I, P],
    "plmc_latent_var": [P, LL, LL, P, P, LL, LL, LL, I, P],
    "plmc_mix_tasks": [P, P, LL, P, P, P, P, LL, I, I, I, P],
    "plmc_syrk_batched": [P, LL, LL, P, LL, LL, LL, LL, D, D, I, CFG, P],
    "plmc_task_covariance": [P, LL, LL, P, P, P, LL, LL, I, I, I, P],
    "plmc_mix_samples": [P, P, LL, LL, P, P, P, P, LL, LL, I, I, P],
    "plmc_gemm": [I, P, LL, LL, P, LL, LL, P, LL, LL, I, I, I, D, D, I, I, I, I, P],
    "plmc_ozaki_ws_bytes": [I, I, I, I, I],
    "plmc_rns_bits": [I, I],
    "plmc_rns_ws_bytes": [I, I, I, I, I, I],
    "plmc_rns_constants": [I, I, P, P, P, P, P],
    "plmc_peak_i8": [LL, I, P, P, P],
    "plmc_rns_gemm": [I, P, LL, P, LL, P, LL, I, I, I, D, D, I, I, I, P, LL, I, P],
    "plmc_ozaki_gemm": [I, P, LL, P, LL, P, LL, I, I, I, D, D, I, I, I, P, LL, P],
    "plmc_peak_dmma": [I, I, LL, P, P],
    "plmc_peak_dfma": [I, I, LL, P, P],
    "plmc_peak_copy": [P, P, LL, P],
    "plmc_peak_mixed": [I, I, LL, LL, P, P],
}
_RET_LL = {"plmc_npad", "plmc_dinv_bytes", "plmc_project_bwd_ws", "plmc_grad_ws", "plmc_ozaki_ws_bytes",
           "plmc_rns_ws_bytes", "plmc_cross_gram_bwd_ws", "plmc_grad_ws2", "plmc_cross_gram_bwd_ws2"}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class PlmcError(RuntimeError):
    pass


def lib_path() -> Path:
    return _LIB_PATH


def load():
    """Load the shared library (no device work).  Raises if it is not built."""
    global _lib
    if _lib is None:
        if not _LIB_PATH.exists():
            raise PlmcError(
                f"{_LIB_PATH} not found: build it with `python -m projected_lmc_b200.build` "
                "(there is no CPU fallback for the projected-LMC hot path)"
            )
        lib = ctypes.CDLL(str(_LIB_PATH))
        for name, argtypes in _SIGNATURES.items():
            try:
                fn = getattr(lib, name)
            except AttributeError as e:  # an incomplete build must not be usable
                raise PlmcError(f"{_LIB_PATH} does not export {name}; rebuild it") from e
            fn.argtypes = argtypes
            fn.restype = LL if name in _RET_LL else I
        _lib = lib
    return _lib


def lib():
    """Library handle ready for device calls (function attributes are set lazily per device inside the library)."""
    l = load()
    if not torch.cuda.is_available():
        raise PlmcError("projected_lmc_b200 needs a CUDA device (sm_100a); no CPU fallback exists")
    return l


def device_of(*tensors):
    """Context manager making the device of the given tensors current for the duration of a library call
    (the library launches on the current device; a tensor on another GPU would otherwise be launched on the
    wrong device's stream)."""
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise PlmcError("libplmc_b200 was handed a non-CUDA tensor; there is no CPU fallback")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise PlmcError(f"libplmc_b200 call with tensors on different devices: {dev} and {t.device}")
    return torch.cuda.device(dev)


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        raise PlmcError(f"libplmc_b200 call {what} failed with code {rc}")


def ptr(t) -> c_void_p:
    if t is None:
        return c_void_p(0)
    if not t.is_cuda:
        raise PlmcError("libplmc_b200 was handed a non-CUDA tensor; there is no CPU fallback")
    if t.dtype not in (torch.float64, torch.int32, torch.uint8):
        raise PlmcError(f"libplmc_b200 works on float64 / int32 buffers, got {t.dtype}")
    return c_void_p(t.data_ptr())


def stream() -> c_void_p:
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def npad(n: int) -> int:
    return ((int(n) + 127) // 128) * 128
