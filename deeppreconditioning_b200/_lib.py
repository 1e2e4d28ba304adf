"""ctypes binding of ``libdpcg.so`` (the C ABI declared in ``include/dpcg.h``).

There is deliberately **no fallback**: if the shared object is missing or a call fails, the product path raises.
"""

from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

import torch

# DPCG_LIB selects another build of the same library (tuning variants made by `build.build_variant`).
LIB_PATH = Path(os.environ.get("DPCG_LIB") or Path(__file__).resolve().parent / "lib" / "libdpcg.so")

DP_OK = 0
DP_ERR_STRUCTURE = 5
DP_ERR_TIMEOUT = 6

PRECOND_IDENTITY, PRECOND_JACOBI, PRECOND_MULTIPLY, PRECOND_SOLVE, PRECOND_CSR = range(5)
ENGINE_FUSED, ENGINE_STEPPED = 0, 1
ASSEMBLE_TRIL, ASSEMBLE_TRIL_T, ASSEMBLE_SYMMETRISE = 0, 1, 2

_p = C.c_void_p
_i32 = C.c_int32
_i64 = C.c_int64


class PcgSystem(C.Structure):
    """``dp_pcg_system_t``."""

    _fields_ = [(name, _i32) for name in (
        "n", "precond", "a_nnz", "m_nnz", "mt_nnz", "fwd_nchunks", "bwd_nchunks",
        "fwd_max_level_chunks", "bwd_max_level_chunks", "solve_algorithm")] + [(name, _p) for name in (
            "a_rowptr", "a_col", "a_val", "m_rowptr", "m_col", "m_val", "mt_rowptr", "mt_col", "mt_val",
            "dinv", "fwd_plan", "bwd_plan",
            "fwd_ls_rowptr", "fwd_ls_col", "fwd_ls_val", "fwd_ls_perm", "fwd_ls_level",
            "bwd_ls_rowptr", "bwd_ls_col", "bwd_ls_val", "bwd_ls_perm", "bwd_ls_level",
            "b", "x", "work", "iters_out", "res_out", "history", "coef",
            "a_col16", "a_val32", "a_tile_base", "m_col16", "m_val32", "m_tile_base",
            "mt_col16", "mt_val32", "mt_tile_base")]


class TrsvSystem(C.Structure):
    """``dp_trsv_system_t``."""

    _fields_ = [("n", _i32), ("upper", _i32), ("max_level_chunks", _i32), ("reserved", _i32), ("nchunks", _i64)] + [
        (name, _p) for name in ("rowptr", "col", "val", "plan", "b", "x")]


class TrsvLsSystem(C.Structure):
    """``dp_trsv_ls_system_t``."""

    _fields_ = [("n", _i32), ("nnz", _i32), ("upper", _i32), ("flags", _i32)] + [
        (name, _p) for name in ("rowptr_p", "col_p", "val_p", "perm", "level_sorted", "b", "x")]


class PcgParams(C.Structure):
    """``dp_pcg_params_t``."""

    _fields_ = [("rtol", C.c_double), ("max_iter", _i32), ("engine", _i32), ("check_every", _i32), ("reserved", _i32)]


class SpconvLayer(C.Structure):
    """``dp_spconv_layer_t``."""

    _fields_ = [("nout", _i64), ("ntaps", _i32), ("cin", _i32), ("cout", _i32), ("reserved", _i32)] + [
        (name, _p) for name in ("src", "in_", "weight", "bias", "slope", "head_weight", "head_bias", "indices", "out")]


class SpconvGrad(C.Structure):
    """``dp_spconv_grad_t``."""

    _fields_ = [("nout", _i64), ("ntaps", _i32), ("cin", _i32), ("cout", _i32), ("reserved", _i32)] + [
        (name, _p) for name in ("src", "in_", "grad_out", "pre", "slope", "tail_indices", "grad_pre", "grad_weight",
                                "grad_bias", "grad_slope")]


class DpcgError(RuntimeError):
    pass


_SIGNATURES = {
    "dp_version": (C.c_int, []),
    "dp_status_string": (C.c_char_p, [C.c_int]),
    "dp_last_cuda_error": (C.c_char_p, []),
    "dp_device_info": (C.c_int, [C.POINTER(C.c_int)] * 3),
    "dp_csr_from_coo_workspace_bytes": (C.c_size_t, [_i32, _i64]),
    "dp_csr_from_coo": (C.c_int, [_p, _p, _i64, _i32, _i32, _i32, _p, _p, _p, _p, _p, _p, C.c_size_t, _p]),
    "dp_csr_transpose_workspace_bytes": (C.c_size_t, [_i32, _i32]),
    "dp_csr_transpose": (C.c_int, [_i32, _i32, _p, _p, _p, _p, _p, _p, _p, C.c_size_t, _p]),
    "dp_csr_inv_diagonal": (C.c_int, [_i32, _p, _p, _p, _p, _p, _p]),
    "dp_csr_aat_nnz": (C.c_int, [_i32, _p, _p, _p, _p, _p, _p]),
    "dp_spmv_csr_f64": (C.c_int, [_i32, _i32, _p, _p, _p, _p, _p, _p]),
    "dp_csr_pack_tile_rows": (_i32, []),
    "dp_csr_pack": (C.c_int, [_i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p]),
    "dp_spmv_csr_packed_f64": (C.c_int, [_i32, _i32, _p, _p, _p, _p, _p, _p, _p]),
    "dp_coo_spmv_batch_f32": (C.c_int, [_p, _p, _i64, _i32, _i32, _p, _i32, _p, _p]),
    "dp_sptrsv_analyse_workspace_bytes": (C.c_size_t, [_i32]),
    "dp_sptrsv_analyse": (C.c_int, [_i32, _p, _p, _i32, _p, _p, _p, _p, _p, _p, C.c_size_t, _p]),
    "dp_sptrsv_plan_chunks": (_i64, [_i32, _p]),
    "dp_sptrsv_plan_sizes_workspace_bytes": (C.c_size_t, [_i32]),
    "dp_sptrsv_plan_sizes": (C.c_int, [_i32, _p, _p, _p, _p, _p, C.c_size_t, _p]),
    "dp_sptrsv_plan_build": (C.c_int, [_i32, _i32, _p, _p, _p, _p, _i64, _p]),
    "dp_sptrsv_workspace_bytes": (C.c_size_t, []),
    "dp_sptrsv_solve_f64": (C.c_int, [_i32, _p, _p, _p, _i32, _p, _i64, _i32, _p, _p, _p, _p, C.c_size_t, _p]),
    "dp_sptrsv_batch_workspace_bytes": (C.c_size_t, [_i32]),
    "dp_sptrsv_solve_batch_f64": (C.c_int, [C.POINTER(TrsvSystem), _i32, _p, _p, C.c_size_t, _p]),
    "dp_sptrsv_permute_workspace_bytes": (C.c_size_t, [_i32]),
    "dp_sptrsv_permute": (C.c_int, [_i32, _i32, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, _p, C.c_size_t, _p]),
    "dp_sptrsv_ls_limits": (None, [_p]),
    "dp_sptrsv_ls_workspace_bytes": (C.c_size_t, [_i32]),
    "dp_sptrsv_ls_solve_batch_f64": (C.c_int, [C.POINTER(TrsvLsSystem), _i32, _p, C.c_size_t, _p]),
    "dp_sptrsv_ls_prepare": (C.c_int, [C.POINTER(TrsvLsSystem), _i32, _p, C.c_size_t, _p]),
    "dp_sptrsv_ls_launch": (C.c_int, [_i32, _p, C.c_size_t, _p]),
    "dp_sptrsv_ts_prepare": (C.c_int, [C.POINTER(TrsvLsSystem), _i32, _p, C.c_size_t, _p]),
    "dp_sptrsv_ts_launch": (C.c_int, [_i32, _i32, _i32, _i32, _i32, _p, _p, _p]),
    "dp_sptrsv_ts_limits": (None, [_p]),
    "dp_sptrsv_ts_workspace_bytes": (C.c_size_t, [C.POINTER(TrsvLsSystem), _i32]),
    "dp_sptrsv_ts_solve_batch_f64": (C.c_int, [C.POINTER(TrsvLsSystem), _i32, _p, _p, C.c_size_t, _p]),
    "dp_ic0_f64": (C.c_int, [_i32, _p, _p, _p, _p, _p, _i64, _i32, _p, _p, C.c_size_t, _p]),
    "dp_icholt_host": (C.c_int, [_i32, _p, _p, _p, _i32, C.c_double, _p, _p, _p, _i64, _p]),
    "dp_spconv_sort_workspace_bytes": (C.c_size_t, [_i32, _i32]),
    "dp_spconv_sort_sites": (C.c_int, [_p, _i64, _i32, _i32, _i32, _p, _p, _p, _p, _p, C.c_size_t, _p]),
    "dp_spconv_rules_workspace_bytes": (C.c_size_t, [_i32, _i32, _i32]),
    "dp_spconv_rules_count": (C.c_int, [_p, _p, _i32, _i32, _i32, _i32, _i32, _p, _p, C.c_size_t, _p]),
    "dp_spconv_rules_fill": (C.c_int, [_p, _p, _p, _i32, _i32, _i32, _i32, _i32, _p, _p, _p, _p, _p]),
    "dp_spconv_layer_f32": (C.c_int, [C.POINTER(SpconvLayer), _p]),
    "dp_spconv_layer_train_f32": (C.c_int, [C.POINTER(SpconvLayer), _p, _p, _p, _p]),
    "dp_spconv_rules_invert": (C.c_int, [_p, _i64, _i32, _i64, _p, _p, _p]),
    "dp_spconv_wgrad_chunk_sites": (_i32, []),
    "dp_spconv_wgrad_workspace_bytes": (C.c_size_t, [_i64, _i32, _i32, _i32]),
    "dp_spconv_wgrad_f32": (C.c_int, [C.POINTER(SpconvGrad), _p, C.c_size_t, _p]),
    "dp_pcg_work_doubles": (_i64, [_i32]),
    "dp_pcg_workspace_bytes": (C.c_size_t, [_i32]),
    "dp_debug_pcg_trace": (C.c_int, [_p, _i32, _p, _i32]),
    "dp_debug_pipe_trace": (C.c_int, [_p, _i32, _i32]),
    "dp_pcg_solve_f64": (C.c_int, [C.POINTER(PcgSystem), _i32, C.POINTER(PcgParams), _p, _p, C.c_size_t, _p]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def lib() -> C.CDLL:
    """Load ``libdpcg.so`` (once). Raises if it has not been built — there is no CPU path behind this package."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise DpcgError(
                f"{LIB_PATH} is missing: build it with `python -m deeppreconditioning_b200.build` "
                "(nvcc, sm_100a). deeppreconditioning_b200 has no CPU fallback."
            )
        handle = C.CDLL(str(LIB_PATH))
        for name, (restype, argtypes) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = restype, argtypes
        _lib = handle
    return _lib


def check(status: int, what: str = "") -> None:
    if status != DP_OK:
        l = lib()
        msg = l.dp_status_string(status).decode()
        if status == 4:
            msg += f" ({l.dp_last_cuda_error().decode()})"
        raise DpcgError(f"libdpcg {what}: {msg}")


def ptr(t: torch.Tensor | None) -> int | None:
    """Device pointer of a CUDA tensor (``None`` -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise DpcgError("libdpcg takes device pointers: got a CPU tensor (no CPU fallback)")
    if not t.is_contiguous():
        raise DpcgError("libdpcg needs contiguous tensors")
    return t.data_ptr()


def stream_ptr(device=None) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def device_info() -> dict:
    sm, ctas, l2 = C.c_int(), C.c_int(), C.c_int()
    check(lib().dp_device_info(C.byref(sm), C.byref(ctas), C.byref(l2)), "dp_device_info")
    return {"sm_count": sm.value, "pcg_ctas_per_sm": ctas.value, "l2_bytes": l2.value}


def raise_on_flag(flag: torch.Tensor, what: str) -> None:
    """Check a device status word (synchronises)."""
    value = int(flag.item())
    if value:
        raise DpcgError(f"libdpcg {what}: device flag {value} ({lib().dp_status_string(value).decode()})")
