"""Loader for the C-ABI shared library (include/ace_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C additivecausalexpansion_b200/csrc``
with nvcc for sm_100a.  There is no CPU fallback: if the library is missing, importing the compute API
raises, and with no CUDA device every compute entry point returns ACE_ERR_NO_DEVICE.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# ACE_B200_LIB: load another build of the library (tuning experiments: make OUT=... EXTRA=...)
SO_PATH = os.environ.get("ACE_B200_LIB") or os.path.join(_HERE, "libace_b200.so")
CSRC = os.path.join(_HERE, "csrc")
HEADER = os.path.join(os.path.dirname(_HERE), "include", "ace_b200.h")

c_double_p = C.POINTER(C.c_double)
c_int_p = C.POINTER(C.c_int)


class AceGemmDesc(C.Structure):
    """struct ace_gemm_desc (include/ace_b200.h): every field of the DMMA GEMM's launch descriptor."""

    _fields_ = ([(f"buf_{x}", C.c_int) for x in ("A", "B", "C", "Ct", "Adiag", "Bdiag")]
                + [(f"off_{x}", C.c_longlong) for x in ("A", "B", "C", "Ct", "Adiag", "Bdiag")]
                + [(x, C.c_longlong) for x in ("lda", "ldb", "ldc", "ldct")]
                + [(x, C.c_int) for x in ("M", "N", "K", "a_tri", "b_tri", "lower_only")]
                + [("alpha", C.c_double), ("beta", C.c_double)]
                + [(x, C.c_int) for x in ("tile_first", "tile_stride", "a_row_off", "s_row_off", "batch", "m_dec",
                                          "ksplit", "klen")]
                + [(x, C.c_longlong) for x in ("sA", "sB", "sC", "sCt", "sAdiag", "sBdiag")])


class AceFitConfig(C.Structure):
    """struct ace_fit_config (include/ace_b200.h)."""

    _fields_ = [
        ("kernel", C.c_int),
        ("optimizer", C.c_int),
        ("learning_rate", C.c_double),
        ("beta1", C.c_double),
        ("beta2", C.c_double),
        ("momentum", C.c_double),
        ("norm_clip", C.c_int),
        ("clip_at", C.c_double),
        ("std_y", C.c_double),
        ("device", C.c_int),
        ("use_graph", C.c_int),
    ]


def build(force: bool = False, verbose: bool = False) -> str:
    """Compile csrc/*.cu into libace_b200.so (nvcc cross-compiles without a GPU; objects build in parallel)."""
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cu", ".cuh", ".inl"))] + [HEADER]
    stale = (not os.path.exists(SO_PATH)) or any(os.path.getmtime(s) > os.path.getmtime(SO_PATH) for s in srcs)
    if force or stale:
        cmd = ["make", "-j", str(min(8, os.cpu_count() or 1)), "-C", CSRC, "../libace_b200.so"] + (["-B"] if force else [])
        subprocess.check_call(cmd, stdout=None if verbose else subprocess.DEVNULL)
    return SO_PATH


_LIB = None

# name -> (restype, argtypes); every symbol include/ace_b200.h declares
_d, _i, _p, _ip = C.c_double, C.c_int, c_double_p, c_int_p
_vp = C.c_void_p
SIGNATURES = {
    "ace_last_error": (C.c_char_p, []),
    "ace_version": (C.c_char_p, []),
    "ace_device_count": (_i, []),
    "ace_set_device": (_i, [_i]),
    "ace_kernmat_SE_cpp": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "ace_kernmat_Matern32_cpp": (_i, [_p, _p, _p, _p, _i, _i, _i, _i, _p, _p, _p]),
    "ace_kernmat_SE_symmetric_cpp": (_i, [_p, _p, _i, _i, _i, _p, _p, _p]),
    "ace_kernmat_Matern32_symmetric_cpp": (_i, [_p, _p, _i, _i, _i, _p, _p, _p]),
    "ace_invkernel_cpp": (_i, [_p, _i, _d, _p, _p]),
    "ace_grad_SE_cpp": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, C.c_uint, _d, _i, _i, _p]),
    "ace_grad_Matern_cpp": (_i, [_p, _p, _p, _p, _p, _p, _p, _p, _p, C.c_uint, _d, _i, _i, _p]),
    "ace_stats_cpp": (_i, [_p, _p, _p, _p, _d, _d, _i, _p]),
    "ace_mu_solution_cpp": (_i, [_p, _p, _i, _p]),
    "ace_pred_cpp": (_i, [_p, _d, _d, _p, _p, _p, _d, _d, _i, _i, _p, _p, _p]),
    "ace_pred_marginal_cpp": (_i, [_p, _p, _d, _d, _p, _p, _p, _d, _d, _d, _i, _i, _i, _i, _p, _p, _p, _p]),
    "ace_norm_clip_cpp": (None, [_i, _p, _i, _d]),
    "ace_Nesterov_cpp": (_i, [_d, _d, _p, _p, _p, _i]),
    "ace_Nadam_cpp": (_i, [_d, _d, _d, _d, _d, _p, _p, _p, _p, _i]),
    "ace_Adam_cpp": (_i, [_d, _d, _d, _d, _d, _p, _p, _p, _p, _i]),
    "ace_fit_default_config": (None, [C.POINTER(AceFitConfig)]),
    "ace_fit_create": (_i, [C.POINTER(_vp), _p, _p, _p, _i, _i, _i, _p, C.POINTER(AceFitConfig)]),
    "ace_fit_destroy": (_i, [_vp]),
    "ace_fit_para_update": (_i, [_vp, _i, _p, _p]),
    "ace_fit_run": (_i, [_vp, _i, _i, _d, _d, _p, _ip]),
    "ace_fit_get_train_stats": (_i, [_vp, _p]),
    "ace_comm_unique_id": (_i, [C.c_char_p]),
    "ace_shard_plan": (_i, [_i, _i, _i, _ip, _ip]),
    "ace_fit_shard": (_i, [_vp, C.c_char_p, _i, _i]),
    "ace_fit_shard_emulate": (_i, [_vp, _i]),
    "ace_dbg_shard_trace_dump": (_i, [_i]),
    "ace_fit_upload_data": (_i, [_vp, _p, _p, _p]),
    "ace_fit_kernel_launches": (_i, [_vp, _ip]),
    "ace_fit_timer_start": (_i, [_vp]),
    "ace_fit_timer_stop": (_i, [_vp, _p]),
    "ace_fit_get_parameters": (_i, [_vp, _p]),
    "ace_fit_set_parameters": (_i, [_vp, _p]),
    "ace_fit_get_gradients": (_i, [_vp, _p]),
    "ace_fit_get_optimizer_state": (_i, [_vp, _p, _p]),
    "ace_fit_get_invKmatn": (_i, [_vp, _p]),
    "ace_fit_get_alpha": (_i, [_vp, _p]),
    "ace_fit_dims": (_i, [_vp, _ip, _ip, _ip, _ip]),
    "ace_fit_last_timing": (_i, [_vp, _p]),
    "ace_fit_predict": (_i, [_vp, _p, _p, _i, _d, _d, _p, _p, _p]),
    "ace_fit_predict_marginal": (_i, [_vp, _p, _p, _p, _i, _d, _d, _d, _i, _p, _p, _p, _p]),
    "ace_fit_predict_marginal_batch": (_i, [_vp, _p, _p, _p, _i, _d, _d, _d, C.POINTER(C.c_ubyte), _i, _p, _p, _p, _p, _ip]),
    "ace_fit_batch_create": (_i, [C.POINTER(_vp), _i, _p, C.c_long, _p, C.c_long, _p, C.c_long, _i, _i, _i, _p,
                                  C.POINTER(AceFitConfig)]),
    "ace_fit_batch_destroy": (_i, [_vp]),
    "ace_fit_batch_dims": (_i, [_vp, _ip, _ip, _ip, _ip, _ip]),
    "ace_fit_batch_set_std_y": (_i, [_vp, _p]),
    "ace_fit_batch_para_update": (_i, [_vp, _i, _p, _ip]),
    "ace_fit_batch_run": (_i, [_vp, _i, _d, _p, _ip, _ip]),
    "ace_fit_batch_status": (_i, [_vp, _ip, _ip]),
    "ace_fit_batch_get_train_stats": (_i, [_vp, _p, _ip]),
    "ace_fit_batch_get_parameters": (_i, [_vp, _p]),
    "ace_fit_batch_get_gradients": (_i, [_vp, _p]),
    "ace_fit_batch_get_optimizer_state": (_i, [_vp, _p, _p]),
    "ace_fit_batch_get_alpha": (_i, [_vp, _p]),
    "ace_fit_batch_get_invKmatn": (_i, [_vp, _i, _p]),
    "ace_fit_batch_last_timing": (_i, [_vp, _p]),
    "ace_fit_batch_extract": (_i, [_vp, _i, C.POINTER(_vp)]),
    "ace_dbg_gemm_nt": (_i, [_p, _p, _p, _i, _i, _i, _d, _d, _i]),
    "ace_dbg_gemm_nt_desc": (_i, [C.POINTER(AceGemmDesc), C.POINTER(_p), C.POINTER(C.c_longlong), _i]),
    "ace_dbg_spd_inverse_lowrank": (_i, [_p, _p, _i, _i, _i, _ip, _i, _p, _p, _p]),
    "ace_dbg_spd_inverse": (_i, [_p, _i, _p, _p, _p, _p]),
    "ace_dbg_spd_inverse_fused": (_i, [_p, _i, _p, _p]),
    "ace_dbg_diag_block": (_i, [_p, _i, _p, _p, _p, _p]),
    "ace_dbg_diag_block_timeline": (_i, [C.POINTER(C.c_longlong), _i]),
    "ace_dbg_diag_block_batch": (_i, [_p, _i, _i, _p, _p, _p, _p]),
    "ace_bench_dense": (_i, [_i, _i, _p]),
    "ace_dbg_set_trtri_max_h": (_i, [_i]),
    "ace_dbg_trtri_raw": (_i, [_p, _i, _p, _p, _p, _p]),
    "ace_dbg_uut_engines": (_i, [_p, _i, C.POINTER(C.c_int), _i, _p, _p, _p]),
    "ace_dbg_fit_set_uut_engine": (_i, [_vp, _i]),
    "ace_dbg_uut_i8_direct": (_i, [_p, _i, _i, _p, _p]),
    "ace_dbg_uut_crt_params": (_i, [_i, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]),
    "ace_dbg_trtri_engines": (_i, [_p, _i, C.POINTER(C.c_int), _i, _p, _p]),
    "ace_dbg_oz_nt": (_i, [_p, _i, _p, _i, _i, _i, _i, _p, _p]),
    "ace_dbg_kernel_plan": (_i, [_i, _i, _i, _i, C.c_char_p, _i, C.c_char_p, _i]),
    "ace_ncs_basis": (_i, [_p, _i, _p, _i, _p]),
    "ace_ncs_basis_deriv": (_i, [_p, _i, _p, _i, _p]),
    "ace_normalize_train": (_i, [_p, _p, _p, _i, _i, _i, _p]),
    "ace_normalize_test": (_i, [_p, _p, _i, _i, _i, _p]),
    "ace_normalize_train_gpu": (_i, [_p, _p, _p, _i, _i, _i, _p]),
    "ace_normalize_test_gpu": (_i, [_p, _p, _i, _i, _i, _p]),
}


def lib():
    """The loaded library with typed signatures.  Raises if it has not been built."""
    global _LIB
    if _LIB is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                f"{SO_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                "(there is no CPU fallback for the ACE hot path)")
        L = C.CDLL(SO_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _LIB = L
    return _LIB


class AceError(RuntimeError):
    def __init__(self, status: int, where: str):
        self.status = status
        msg = lib().ace_last_error()
        super().__init__(f"{where}: status {status}: {msg.decode() if msg else ''}")


class NotFiniteError(AceError, FloatingPointError):
    """The reference's stop("Some gradients are not finite, NaN, or NA. ...")."""


ACE_ERR_NOT_FINITE = 1073741824


def check(status: int, where: str) -> None:
    if status == 0:
        return
    if status == ACE_ERR_NOT_FINITE:
        raise NotFiniteError(status, where)
    raise AceError(status, where)
