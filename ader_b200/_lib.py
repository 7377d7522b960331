"""ctypes binding of libader_b200.so (the C ABI declared in include/ader_b200.h).

There is no CPU fallback: if the shared library is missing it is built with nvcc, and if that
fails the import raises.  Every entry point returns an int status; non-zero raises
``AderError`` carrying ``ader_last_error()``.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

ABI_VERSION = 2


class AderError(RuntimeError):
    pass


class AderModel(C.Structure):
    _fields_ = [("v_tab", C.c_int32), ("d", C.c_int32), ("maxlen", C.c_int32),
                ("num_blocks", C.c_int32), ("num_heads", C.c_int32)]


class AderLossArgs(C.Structure):
    _fields_ = [("M", C.c_int32), ("n_train", C.c_int32), ("n_ex", C.c_int32), ("V", C.c_int32),
                ("V_prev", C.c_int32), ("mode", C.c_int32), ("lambda_", C.c_float),
                ("pos", C.c_void_p), ("ex_pos", C.c_void_p), ("teacher", C.c_void_p),
                ("teacher_row", C.c_void_p), ("teacher_ld", C.c_int64),
                ("n_train_global", C.c_int32), ("n_ex_global", C.c_int32),
                ("teacher_rep", C.c_void_p), ("teacher_table", C.c_void_p), ("teacher_table16", C.c_void_p)]


class AderAdamArgs(C.Structure):
    _fields_ = [("lr", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float), ("eps", C.c_float),
                ("V", C.c_int32), ("ewc_lambda", C.c_float), ("fisher", C.c_void_p),
                ("theta_star", C.c_void_p)]


DP_MAX_RANKS = 16
DP_FLAG_WORDS = 64


class AderDpComm(C.Structure):
    _fields_ = [("rank", C.c_int32), ("world", C.c_int32), ("separate_arrive", C.c_int32), ("reserved", C.c_int32),
                ("theta", C.c_void_p * DP_MAX_RANKS),
                ("grad", C.c_void_p * DP_MAX_RANKS), ("flags", C.c_void_p * DP_MAX_RANKS),
                ("mc_theta", C.c_void_p), ("mc_grad", C.c_void_p)]


_P = C.c_void_p
_MP = C.POINTER(AderModel)
_CP = C.POINTER(AderDpComm)

# name -> (restype, argtypes); mirrors include/ader_b200.h one to one (tests/test_abi.py checks
# that every symbol declared in the header is exported and listed here).
SIGNATURES = {
    "ader_abi_version": (C.c_int32, []),
    "ader_last_error": (C.c_char_p, []),
    "ader_param_count": (C.c_int64, [_MP]),
    "ader_param_offset": (C.c_int64, [_MP, C.c_int32]),
    "ader_dense_count": (C.c_int64, [_MP]),
    "ader_path_check": (C.c_int32, [_MP, C.c_int32]),
    "ader_encoder_ws_bytes": (C.c_size_t, [_MP, C.c_int32, C.c_int32]),
    "ader_encoder_bwd_ws_bytes": (C.c_size_t, [_MP, C.c_int32, C.c_int32]),
    "ader_encoder_ws_slot": (C.c_int64, [_MP, C.c_int32, C.c_int32, C.c_int32, C.c_int32]),
    "ader_encoder_fwd": (C.c_int32, [_MP, _P, _P, C.c_int32, C.c_int32, _P, _P, C.c_float, C.c_uint64, _P]),
    "ader_encoder_bwd": (C.c_int32, [_MP, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, C.c_float, C.c_uint64, _P]),
    "ader_encoder_fwd_tc": (C.c_int32, [_MP, _P, _P, C.c_int32, C.c_int32, _P, _P, C.c_float, C.c_uint64, _P, _P]),
    "ader_encoder_bwd_tc": (C.c_int32, [_MP, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P, C.c_float, C.c_uint64, _P, _P]),
    "ader_loss_ws_bytes": (C.c_size_t, [_MP, C.POINTER(AderLossArgs)]),
    "ader_loss_fwd_bwd": (C.c_int32, [_MP, _P, _P, C.POINTER(AderLossArgs), _P, _P, _P, _P, _P, _P]),
    "ader_loss_tc_ws_bytes": (C.c_size_t, [_MP, C.POINTER(AderLossArgs)]),
    "ader_loss_fwd_bwd_tc": (C.c_int32, [_MP, _P, _P, C.POINTER(AderLossArgs), _P, _P, _P, _P, _P, _P]),
    "ader_debug_loss_tc_kernels": (C.c_int32, [_MP, _P, C.POINTER(AderLossArgs), _P, _P, _P]),
    "ader_loss_tc_vp_ws_bytes": (C.c_size_t, [_MP, C.POINTER(AderLossArgs), C.c_int32, C.c_int32]),
    "ader_loss_tc_vp_fwd": (C.c_int32, [_MP, _P, _P, C.POINTER(AderLossArgs), C.c_int32, C.c_int32, _P, _P, _P]),
    "ader_loss_tc_vp_bwd": (C.c_int32, [_MP, _P, _P, C.POINTER(AderLossArgs), C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "ader_train_fwd_bwd_tc": (C.c_int32, [_MP, _P, _P, C.c_int32, C.c_int32, C.POINTER(AderLossArgs), _P, _P, _P, _P, _P, _P, _P,
                                          _P, C.c_float, C.c_uint64, _P, C.c_int32, _P]),
    "ader_train_step_tc": (C.c_int32, [_MP, _P, _P, C.c_int32, C.c_int32, C.POINTER(AderLossArgs), _P, _P, _P, _P, _P, _P, _P,
                                       _P, C.c_float, C.c_uint64, _P, _P, _P, _P, C.POINTER(AderAdamArgs), C.c_int32, _P]),
    "ader_table16_ws_bytes": (C.c_size_t, [_MP, C.c_int32]),
    "ader_pack_table16": (C.c_int32, [_MP, _P, C.c_int32, _P, _P]),
    "ader_logits": (C.c_int32, [_MP, _P, _P, C.c_int32, C.c_int32, _P, C.c_int64, _P]),
    "ader_adam_step": (C.c_int32, [_MP, _P, _P, _P, _P, _P, C.POINTER(AderAdamArgs), _P]),
    "ader_eval_ws_bytes": (C.c_size_t, [_MP, C.c_int32, C.c_int32]),
    "ader_eval_rank_topk": (C.c_int32, [_MP, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "ader_eval_rank_tc_ws_bytes": (C.c_size_t, [_MP, C.c_int32, C.c_int32]),
    "ader_eval_rank_tc": (C.c_int32, [_MP, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "ader_eval_topk_chunks": (C.c_int32, [_MP, C.c_int32, C.c_int32]),
    "ader_eval_rank_topk_tc": (C.c_int32, [_MP, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "ader_recommend_topk": (C.c_int32, [_MP, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "ader_recommend_tc_ws_bytes": (C.c_size_t, [_MP, C.c_int32, C.c_int32]),
    "ader_recommend_topk_tc": (C.c_int32, [_MP, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "ader_logsumexp": (C.c_int32, [_MP, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "ader_logsumexp_tc_ws_bytes": (C.c_size_t, [_MP, C.c_int32, C.c_int32]),
    "ader_logsumexp_tc": (C.c_int32, [_MP, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "ader_herding_ws_bytes": (C.c_size_t, [_MP, C.c_int32]),
    "ader_herding_segmented": (C.c_int32, [_MP, _P, C.c_int32, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P]),
    "ader_fisher_accumulate": (C.c_int32, [_MP, _P, _P, C.c_int32, _P]),
    "ader_fisher_finalize": (C.c_int32, [_MP, _P, _P, C.c_int32, C.c_int32, _P]),
    "ader_fisher_batched_ws_bytes": (C.c_size_t, [_MP, C.c_int32, C.c_int32]),
    "ader_fisher_batched": (C.c_int32, [_MP, _P, _P, _P, C.c_int32, C.c_int32, C.c_int32, _P, _P, _P, _P, _P]),
    "ader_dp_wait": (C.c_int32, [_CP, _P]),
    "ader_dp_adam_step": (C.c_int32, [_MP, _CP, _P, _P, _P, C.POINTER(AderAdamArgs), _P]),
    "ader_dp_status": (C.c_int32, [_CP, C.POINTER(C.c_int32), C.POINTER(C.c_uint32)]),
    "ader_ipc_export": (C.c_int32, [_P, _P, C.POINTER(C.c_int64)]),
    "ader_ipc_open": (C.c_int32, [_P, C.POINTER(C.c_void_p)]),
    "ader_ipc_close": (C.c_int32, [_P]),
    "ader_gather_rows_i32": (C.c_int32, [_P, _P, C.c_int32, C.c_int32, _P, _P]),
    "ader_gather_batch_q": (C.c_int32, [_P, _P, C.c_int32, _P, _P, C.c_int32, _P, _P, _P, C.c_int32, _P, _P, _P, _P]),
    "ader_queue_advance": (C.c_int32, [_P, _P]),
    "ader_gather_batch": (C.c_int32, [_P, _P, _P, C.c_int32, _P, _P, _P, C.c_int32, C.c_int32, _P, _P, _P, _P]),
}

_lib = None


def lib_path() -> str:
    return _build.LIB_PATH


def load() -> C.CDLL:
    """Load (building first if needed) the shared library; raises if that is impossible."""
    global _lib
    if _lib is not None:
        return _lib
    # build() returns at once when the .so is newer than every source / header (mtime check), so a pulled kernel change
    # can never run against a stale library; a box without nvcc (or a read-only tree) uses the shipped .so as it is
    path = _build.LIB_PATH
    alt = os.environ.get("ADER_B200_LIB")       # debug builds (python -m ader_b200.build --timeline): use that file as it is
    if alt:
        if not os.path.exists(alt):
            raise AderError("ADER_B200_LIB=%s does not exist" % alt)
        path = alt
    else:
        try:
            path = _build.build(force=os.environ.get("ADER_B200_REBUILD") == "1")
        except Exception:
            if not os.path.exists(path):
                raise
    lib = C.CDLL(path)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is missing: fail loudly
        fn.restype = res
        fn.argtypes = args
    if lib.ader_abi_version() != ABI_VERSION:
        raise AderError("libader_b200.so ABI %d != binding ABI %d" % (lib.ader_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = load().ader_last_error().decode("utf-8", "replace")
        raise AderError("%s failed (%d): %s" % (what or "libader_b200 call", rc, msg))
