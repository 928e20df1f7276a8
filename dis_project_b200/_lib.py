"""ctypes binding of ``liblfm_b200.so`` (the C-ABI declared in ``include/lfm_b200.h``).

The library is built in-tree by ``__graft_entry__.build()`` /
``make -C dis_project_b200/csrc``.  There is NO CPU fallback: if the shared
object is missing or no sm_100 GPU is visible, every compute entry point raises.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "liblfm_b200.so")

LFM_OK = 0
STATUS = {0: "LFM_OK", -1: "LFM_ERR_INVALID", -2: "LFM_ERR_CUDA", -3: "LFM_ERR_UNSUPPORTED",
          -4: "LFM_ERR_WORKSPACE", -5: "LFM_ERR_NO_DEVICE", -6: "LFM_ERR_COMM"}


class LfmError(RuntimeError):
    def __init__(self, status: int, where: str):
        self.status = status
        msg = STATUS.get(status, str(status))
        try:
            msg += ": " + lib().lfm_status_string(status).decode()
        except Exception:  # pragma: no cover
            pass
        super().__init__(f"{where} failed with {msg}")


_lib: Optional[C.CDLL] = None

_i64, _int, _dbl, _ptr, _sz = C.c_int64, C.c_int, C.c_double, C.c_void_p, C.c_size_t


class GemmDesc(C.Structure):
    """lfm_gemm_desc of include/lfm_b200.h (lfm_debug_dgemm)."""
    _fields_ = [("transA", _int), ("transB", _int), ("M", _i64), ("N", _i64), ("K", _i64),
                ("A", _ptr), ("lda", _i64), ("B", _ptr), ("ldb", _i64), ("C", _ptr), ("ldc", _i64),
                ("alpha", _dbl), ("beta", _dbl), ("lower_only", _int), ("kmode", _int), ("batch", _int),
                ("strideA", _i64), ("strideB", _i64), ("strideC", _i64), ("tile", _int), ("tri_skip", _int),
                ("k_split", _i64), ("k_lo", _i64), ("k_hi", _i64)]

# name -> (restype, argtypes); mirrors include/lfm_b200.h one to one
SIGNATURES = {
    "lfm_abi_version": (_int, []),
    "lfm_status_string": (C.c_char_p, [_int]),
    "lfm_device_check": (_int, []),
    "lfm_cross_covariance": (_int, [_ptr, _i64, _i64, _ptr, _ptr, _int, _ptr, _ptr, _i64]),
    "lfm_gram": (_int, [_ptr, _i64, _ptr, _int, _ptr, _ptr, _i64]),
    "lfm_h": (_int, [_ptr, _i64, _ptr, _ptr, _ptr, _ptr, _int, _ptr, _ptr]),
    "lfm_mean_function": (_int, [_ptr, _i64, _ptr, _int, _ptr, _ptr]),
    "lfm_constrain": (_int, [_ptr, _i64, _int, _ptr, _ptr]),
    "lfm_unconstrain": (_int, [_ptr, _i64, _int, _ptr, _ptr]),
    "lfm_count_distinct_times": (_i64, [_i64, _ptr]),
    "lfm_plan_launch": (_int, [_ptr, _ptr]),
    "lfm_plan_destroy": (_int, [_ptr]),
    "lfm_nlml_workspace_bytes_tg": (_sz, [_i64, _int, _i64]),
    "lfm_nlml_het_tg": (_int, [_ptr, _i64, _int, _ptr, _ptr, _ptr, _ptr, _dbl, _i64, _ptr, _sz, _ptr, _ptr]),
    "lfm_nlml_grad_het_tg": (_int, [_ptr, _i64, _int, _ptr, _ptr, _ptr, _ptr, _dbl, _i64, _ptr, _sz, _ptr, _ptr]),
    "lfm_nlml_grad_unc_het_tg": (_int, [_ptr, _i64, _int, _ptr, _ptr, _ptr, _ptr, _dbl, _i64, _ptr, _sz, _ptr, _ptr]),
    "lfm_nlml_grad_plan_create_het": (_int, [C.POINTER(C.c_void_p), _i64, _int, _ptr, _ptr, _ptr, _ptr, _dbl, _i64, _int,
                                             _ptr, _sz, _ptr, _ptr]),
    "lfm_nlml_grad_het_host": (_int, [_ptr, _i64, _int, _ptr, _ptr, _ptr, _ptr, _dbl, _int, _ptr, _ptr]),
    "lfm_latent_posterior_workspace_bytes": (_sz, [_i64, _int, _i64]),
    "lfm_latent_posterior": (_int, [_ptr, _i64, _int, _ptr, _ptr, _ptr, _ptr, _dbl, _i64, _ptr, _ptr, _sz,
                                    _ptr, _ptr, _ptr]),
    "lfm_gene_posterior_workspace_bytes": (_sz, [_i64, _int, _i64]),
    "lfm_gene_posterior": (_int, [_ptr, _i64, _int, _ptr, _ptr, _ptr, _ptr, _dbl, _i64, _ptr, _ptr, _sz,
                                  _ptr, _ptr, _ptr, _ptr]),
    "lfm_count_unique_rows": (_int, [_i64, _ptr]),
    "lfm_batched_fit_init": (_int, [_ptr, _i64, _int, _ptr, _ptr, _ptr, _ptr, _i64, _ptr, _ptr, _i64]),
    "lfm_batched_queue_bytes": (_sz, [_i64, _int, _int]),
    "lfm_batched_nlml_grad_unc_het": (_int, [_ptr, _i64, _i64, _int, _ptr, _ptr, _i64, _ptr, _i64, _ptr, _dbl, _int, _int,
                                             _ptr, _ptr, _ptr]),
    "lfm_batched_fit_het": (_int, [_ptr, _i64, _i64, _int, _ptr, _ptr, _i64, _ptr, _i64, _ptr, _ptr, _dbl, _dbl, _dbl, _dbl,
                                   _dbl, _int, _int, _int, _int, _int, _int, _int, _ptr, _i64, _ptr, _ptr, _ptr, _ptr, _ptr,
                                   _int, _ptr, _sz]),
    "lfm_batched_posterior_workspace_bytes": (_sz, [_i64, _i64, _int, _i64, _int, _int]),
    "lfm_batched_latent_posterior": (_int, [_ptr, _i64, _i64, _int, _ptr, _ptr, _i64, _ptr, _i64, _ptr, _dbl, _i64, _ptr,
                                            _int, _ptr, _sz, _ptr, _ptr, _ptr]),
    "lfm_batched_gene_posterior": (_int, [_ptr, _i64, _i64, _int, _ptr, _ptr, _i64, _ptr, _i64, _ptr, _dbl, _i64, _ptr,
                                          _int, _ptr, _sz, _ptr, _ptr, _ptr, _ptr]),
    "lfm_batched_structure_bytes": (_sz, [_i64, _int, _int, _int]),
    "lfm_batched_team_size": (_int, [_i64, _i64, _int, _int, _int]),
    "lfm_batched_best": (_int, [_ptr, _i64, _int, _ptr, _i64, _i64, _ptr, _dbl, _ptr]),
    "lfm_comm_available": (_int, []),
    "lfm_comm_unique_id": (_int, [_ptr]),
    "lfm_comm_create": (_int, [C.POINTER(_ptr), _int, _int, _ptr]),
    "lfm_comm_world": (_int, [_ptr]),
    "lfm_comm_rank": (_int, [_ptr]),
    "lfm_comm_allreduce_min_i64": (_int, [_ptr, _ptr, _sz, _ptr]),
    "lfm_comm_allgather_f64": (_int, [_ptr, _ptr, _ptr, _sz, _ptr]),
    "lfm_comm_destroy": (_int, [_ptr]),
    "lfm_handle_create": (_int, [C.POINTER(_ptr)]),
    "lfm_handle_destroy": (_int, [_ptr]),
    "lfm_nlml_grad_host": (_int, [_ptr, _i64, _int, _ptr, _ptr, _ptr, _dbl, _int, _ptr, _ptr]),
    "lfm_latent_posterior_host": (_int, [_ptr, _i64, _int, _ptr, _ptr, _ptr, _ptr, _dbl, _i64, _ptr, _ptr,
                                         _ptr, _ptr]),
    "lfm_batched_fit_het_host": (_int, [_ptr, _i64, _i64, _int, _ptr, _ptr, _ptr, _ptr, _dbl, _dbl, _dbl, _dbl, _dbl,
                                        _int, _int, _int, _ptr, _ptr, _ptr]),
    "lfm_debug_leaf_profile": (_int, [_ptr, _ptr, _ptr, _ptr, _ptr]),
    "lfm_debug_launch_count": (C.c_ulonglong, []),
    "lfm_debug_batched_stamps": (_int, [_ptr, _i64, _i64, _int, _ptr, _ptr, _ptr, _ptr, _dbl, _int, _int, _int, _ptr, _ptr,
                                        _ptr]),
    "lfm_debug_profile_begin": (_int, []),
    "lfm_debug_profile_end": (_int, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "lfm_debug_profile_sum_ms": (C.c_double, []),
    "lfm_debug_profile_variants": (_sz, [C.c_char_p, _sz]),
    "lfm_debug_profile_chain": (_int, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_longlong)]),
    "lfm_debug_dgemm_nt": (_int, [_ptr, _i64, _i64, _i64, _ptr, _ptr, _ptr]),
    "lfm_debug_dgemm": (_int, [_ptr, _ptr, C.POINTER(_int)]),
    "lfm_debug_potrf_potri": (_int, [_ptr, _i64, _ptr, _ptr, _ptr, _ptr]),
    "lfm_debug_potrf_potri_eval": (_int, [_ptr, _i64, _ptr, _ptr, _ptr, _int, C.POINTER(_int), _ptr]),
    "lfm_debug_syrk": (_int, [_ptr, _i64, _i64, _ptr, _i64, _ptr, _i64]),
    "lfm_debug_syrk_stamps": (_int, [_ptr, _i64, _i64, _ptr, _i64, _ptr, _i64, _ptr]),
}


def lib() -> C.CDLL:
    """Load the shared library (once).  Raises if it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C dis_project_b200/csrc`.  There is no CPU fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(status: int, where: str) -> None:
    if status != LFM_OK:
        raise LfmError(status, where)


_device_ok = False


def require_device() -> None:
    """Fail loudly unless an sm_100 GPU is usable (no silent fallback).  The positive answer is cached:
    cudaGetDeviceProperties costs milliseconds."""
    global _device_ok
    if _device_ok:
        return
    import torch

    if not torch.cuda.is_available():
        raise RuntimeError("dis_project_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    check(lib().lfm_device_check(), "lfm_device_check")
    _device_ok = True
