"""ctypes binding of the C-ABI library (include/movae_b200.h).  There is NO fallback: if the
shared library is missing or a call fails, a RuntimeError is raised (its text contains "CUDA" for
device-side failures so the reference's filter at /root/reference/main.py:197-208 still matches)."""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int64, c_size_t, c_void_p

import torch

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", "libmovae_b200.so")
ABI_VERSION = 2
MAX_K = 8
DIAG_DOUBLES = 8
DIAG_SIMILARITY, DIAG_COUNT, DIAG_GAMMA, DIAG_RANK, DIAG_STATUS, DIAG_RESIDUAL, DIAG_TRACE = range(7)
MGDA_NORM = {"none": 0, "l2": 1, "loss": 2, "loss+": 3}
AMTL_SCALE = {"min": 0, "median": 1, "rmse": 2}
UPGRAD_NORM = {"trace": 0, "min_l2": 1, "l2": 2, "draw": 3}

SOLVE_CONSTANT, SOLVE_UPGRAD, SOLVE_MGDA, SOLVE_ALIGNED_MTL, SOLVE_DUALPROJ, SOLVE_COMFORT, SOLVE_PCGRAD, SOLVE_IMTLG = range(8)
VQ_AUTO, VQ_EXACT, VQ_TENSOR = range(3)


MAX_WORLD = 8


class P2PCtx(ctypes.Structure):
    """mirror of `movae_p2p_ctx` (include/movae_b200.h)"""
    _fields_ = [("rank", ctypes.c_int32), ("world", ctypes.c_int32), ("peers", c_void_p * MAX_WORLD)]


MAX_SEGMENTS = 32


class JacSegments(ctypes.Structure):
    """mirror of `movae_jac_segments` (include/movae_b200.h)"""
    _fields_ = [("n_segments", ctypes.c_int32), ("k", ctypes.c_int32), ("n", c_int64 * MAX_SEGMENTS),
                ("out_off", c_int64 * MAX_SEGMENTS), ("rows", (c_void_p * 8) * MAX_SEGMENTS)]


class SolveSpec(ctypes.Structure):
    """mirror of `movae_solve_spec` (include/movae_b200.h)"""
    _fields_ = [("kind", ctypes.c_int32), ("mode", ctypes.c_int32), ("max_iters", ctypes.c_int32),
                ("stable", ctypes.c_int32), ("value", c_float), ("norm_eps", c_float), ("reg_eps", c_float),
                ("epsilon", c_float), ("min_eigenvalue_eps", c_float)]


class OptimSpec(ctypes.Structure):
    """mirror of `movae_optim_spec` (include/movae_b200.h)"""
    _fields_ = [("kind", ctypes.c_int32), ("hold_step", ctypes.c_int32), ("lr", c_double), ("beta1", c_double),
                ("beta2", c_double), ("eps", c_double), ("weight_decay", c_double), ("max_grad_norm", c_double)]


OPT_SGD, OPT_ADAM, OPT_ADAMW, OPT_RMSPROP = range(4)

_SIGNATURES = {
    "movae_abi_version": (c_int, []),
    "movae_last_error": (c_char_p, []),
    "movae_device_info": (c_int, [POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "movae_gram_workspace_bytes": (c_size_t, [c_int]),
    "movae_gram_f32": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "movae_solve_constant": (c_int, [c_void_p, c_int, c_float, c_void_p, c_void_p, c_void_p]),
    "movae_solve_upgrad": (c_int, [c_void_p, c_int, c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p]),
    "movae_solve_nupgrad": (c_int, [c_void_p, c_int, c_void_p, c_float, c_float, c_int, c_void_p, c_void_p, c_void_p]),
    "movae_solve_dualproj": (c_int, [c_void_p, c_int, c_void_p, c_float, c_float, c_void_p, c_void_p, c_void_p]),
    "movae_solve_mgda": (c_int, [c_void_p, c_int, c_int, c_void_p, c_float, c_int, c_int, c_float, c_void_p,
                                 c_void_p, c_void_p]),
    "movae_solve_aligned_mtl": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "movae_recombine_f32": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_int, c_void_p]),
    "movae_solve": (c_int, [c_void_p, c_int, POINTER(SolveSpec), c_void_p, c_void_p, c_void_p, c_void_p]),
    "movae_solve_aux": (c_int, [c_void_p, c_int, POINTER(SolveSpec), c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "movae_aggregate_f32": (c_int, [c_void_p, c_int, c_int64, c_int64, POINTER(SolveSpec), c_void_p, c_void_p, c_void_p, c_int,
                                    c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, POINTER(P2PCtx), c_void_p]),
    "movae_aggregate_segments_f32": (c_int, [POINTER(JacSegments), POINTER(SolveSpec), c_void_p, c_void_p, c_void_p, c_int, c_void_p,
                                             c_void_p, c_void_p, c_void_p, c_size_t, POINTER(P2PCtx), c_void_p]),
    "movae_aggregate_timestamps": (c_int, [c_void_p, POINTER(ctypes.c_uint64 * 6), c_void_p]),
    "movae_host_gram_f32": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p, c_size_t,
                                    c_int64, c_void_p, c_void_p]),
    "movae_host_recombine_f32": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int64,
                                         c_void_p, c_void_p]),
    "movae_host_recombine_async_f32": (c_int, [c_void_p, c_int, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_int64,
                                               c_void_p, c_void_p]),
    "movae_p2p_exchange_bytes": (c_size_t, []),
    "movae_p2p_alloc": (c_int, [c_size_t, POINTER(c_void_p), ctypes.c_char_p]),
    "movae_p2p_open": (c_int, [ctypes.c_char_p, POINTER(c_void_p)]),
    "movae_p2p_close": (c_int, [c_void_p]),
    "movae_p2p_free": (c_int, [c_void_p]),
    "movae_p2p_barrier": (c_int, [POINTER(P2PCtx), c_void_p, c_void_p]),
    "movae_vq_tensor_path_supported": (c_int, [c_int, c_int]),
    "movae_vq_workspace_bytes": (c_size_t, [c_int64, c_int, c_int]),
    "movae_vq_argmin_f32": (c_int, [c_void_p, c_int64, c_int, c_int64, c_void_p, c_int, c_void_p, c_int, c_void_p,
                                    c_void_p, c_size_t, c_void_p]),
    "movae_vq_gather_f32": (c_int, [c_void_p, c_int64, c_int, c_int64, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_size_t, c_void_p]),
    "movae_vq_forward_f32": (c_int, [c_void_p, c_int64, c_int, c_int64, c_void_p, c_int, c_void_p, c_void_p, c_void_p,
                                     c_void_p, c_int, c_void_p, c_size_t, c_void_p]),
    "movae_vq_backward_workspace_bytes": (c_size_t, [c_int64, c_int, c_int]),
    "movae_vq_backward_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int, c_int64, c_void_p, c_int,
                                      c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "movae_vq_usage": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_size_t, c_void_p]),
    "movae_vq_pack_codes": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "movae_vq_bitmap_count": (c_int, [c_void_p, c_int, c_void_p, c_void_p]),
    "movae_optim_state_bytes": (c_size_t, []),
    "movae_optim_step_f32": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int64, POINTER(OptimSpec), c_void_p, c_void_p,
                                     c_void_p, c_void_p]),
}

_lib = None


def exported_symbols():
    """Names include/movae_b200.h declares (kept in sync by tests/test_abi.py)."""
    return tuple(_SIGNATURES)


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"movae_b200: CUDA library {LIB_PATH} is missing -- build it with "
                f"`python mo-vae_b200/build.py` (there is no CPU fallback)")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        got = handle.movae_abi_version()
        if got != ABI_VERSION:
            raise RuntimeError(f"movae_b200: ABI version mismatch (library {got}, binding {ABI_VERSION})")
        _lib = handle
    return _lib


def check(status: int, what: str) -> None:
    if status != 0:
        msg = lib().movae_last_error().decode("utf-8", "replace")
        if status == 1:
            raise ValueError(f"movae_b200.{what}: {msg}")
        raise RuntimeError(f"movae_b200.{what} failed (status {status}): {msg}")


def ptr(t) -> int:
    return 0 if t is None else t.data_ptr()


def stream_of(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def require_cuda(t: torch.Tensor, name: str) -> None:
    if not t.is_cuda:
        raise RuntimeError(
            f"movae_b200: `{name}` must be a CUDA tensor (got device {t.device}); this path is CUDA-only, "
            f"there is no CPU fallback")
