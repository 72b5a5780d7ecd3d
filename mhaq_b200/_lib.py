"""ctypes binding of the C ABI declared in ``include/mhaq_fq.h``.

The shared library ``mhaq_b200/csrc/libmhaq_fq.so`` is built in-tree by
``__graft_entry__.build()`` (or ``make -C mhaq_b200/csrc``).  There is no CPU
or PyTorch fallback: if the library is missing, importing this module raises.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_float, c_int, c_int64, c_uint64, c_void_p, c_char_p

_HERE = os.path.dirname(os.path.abspath(__file__))
# MHAQ_FQ_LIB: experiment knob to load an alternative build of the same ABI
LIB_PATH = os.environ.get("MHAQ_FQ_LIB") or os.path.join(_HERE, "csrc", "libmhaq_fq.so")

ABI_VERSION = 7
NPART = 8  # MHAQ_FQ_NPART

class WRowFwdDesc(ctypes.Structure):
    """mhaq_fq_wrow_fwd_desc"""
    _fields_ = [(n, c_void_p) for n in ("w", "log_scale", "wq", "row_min", "row_max", "log_range")] + [
        ("n_rows", c_int64), ("n_inner", c_int64)]


class WRowBwdDesc(ctypes.Structure):
    """mhaq_fq_wrow_bwd_desc"""
    _fields_ = [(n, c_void_p) for n in ("g_wq", "w", "log_scale", "row_min", "row_max", "g_log_range",
                                        "g_row_min", "g_row_max", "r", "g_w", "g_log_scale")] + [
        ("n_rows", c_int64), ("n_inner", c_int64), ("g_log_scale_acc", c_void_p)]


class IConvEpilogue(ctypes.Structure):
    """mhaq_fq_iconv_epilogue"""
    _fields_ = [("residual", c_void_p), ("activation", c_int), ("negative_slope", c_float), ("y", c_void_p),
                ("codes", c_void_p), ("code_scale", c_void_p), ("code_zero_point", c_void_p),
                ("code_max_val", c_void_p)]


ACT_NONE, ACT_RELU, ACT_LEAKY_RELU = 0, 1, 2  # MHAQ_FQ_ACT_*


class IConvGeometry(ctypes.Structure):
    """mhaq_fq_iconv_geometry"""
    _fields_ = [(n, c_int) for n in ("kernel_h", "kernel_w", "stride_h", "stride_w", "pad_h", "pad_w",
                                     "dilation_h", "dilation_w", "groups")]

# name -> (restype, argtypes); mirrors include/mhaq_fq.h one to one
_P = c_void_p
_SIGNATURES = {
    "mhaq_fq_abi_version": (c_int, []),
    "mhaq_fq_build_info": (c_char_p, []),
    "mhaq_fq_num_tasks": (c_int64, [c_int64, c_int64]),
    "mhaq_fq_workspace_bytes": (c_int64, [c_int64, c_int64]),
    "mhaq_fq_ticket_count": (c_int64, [c_int64, c_int64, c_int64]),
    "mhaq_fq_stream_capture_id": (c_uint64, [_P]),
    "mhaq_fq_fwd_f32": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                c_int64, c_int64, c_int64, _P, _P]),
    "mhaq_fq_minmax_finalize": (c_int, [_P, c_int64, c_int64, _P, _P]),
    "mhaq_fq_bwd_f32": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                c_int64, c_int64, c_int64, c_int, c_int, _P, c_uint64, c_uint64,
                                _P, _P, _P, _P]),
    "mhaq_fq_bwd_finalize_f32": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                         c_int64, c_int64, c_int64, _P, _P, _P, _P, _P]),
    "mhaq_fq_bwd_fused_f32": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                      c_int64, c_int64, c_int64, c_int, c_int, _P, c_uint64, c_uint64,
                                      _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mhaq_fq_bwd_fused_acc_f32": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                          c_int64, c_int64, c_int64, c_int, c_int, _P, c_uint64, c_uint64,
                                          _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mhaq_fq_bwd_single_launch": (c_int, [c_int64, c_int64, c_int64, c_int, c_int]),
    "mhaq_fq_aewgs_stats_f32": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                        c_int64, c_int64, c_int64, c_int, _P, _P]),
    "mhaq_fq_aewgs_stats_finalize_f32": (c_int, [_P, c_int64, c_int64, c_int64, _P, _P]),
    "mhaq_fq_wrow_fwd_f32": (c_int, [_P, _P, _P, c_int64, c_int64, _P, _P, _P, _P]),
    "mhaq_fq_wrow_bwd_f32": (c_int, [_P, _P, _P, _P, _P, _P, _P, _P, c_int64, c_int64, c_int, _P,
                                     c_uint64, c_uint64, _P, _P, _P, _P]),
    "mhaq_fq_rowstat_f32": (c_int, [_P, c_int64, c_int64, _P, _P, _P, _P, _P]),
    "mhaq_fq_rowstat_bwd_f32": (c_int, [_P, _P, c_int64, c_int64, _P, _P, _P, _P, _P, _P, _P, _P]),
    "mhaq_fq_wrow_multi_fwd_f32": (c_int, [_P, c_int, _P]),
    "mhaq_fq_wrow_multi_aewgs_stats_f32": (c_int, [_P, c_int, _P, c_int64, _P]),
    "mhaq_fq_wrow_multi_bwd_f32": (c_int, [_P, c_int, c_int, c_uint64, c_uint64, _P, _P, c_int64, _P]),
    "mhaq_fq_potential_loss_fwd_f32": (c_int, [_P, _P, c_int64, _P, _P, c_int64, _P, _P, _P, c_float, c_float,
                                               c_float, c_float, c_int, c_int, _P, _P]),
    "mhaq_fq_potential_loss_bwd_f32": (c_int, [_P, _P, c_int64, _P, _P, c_int64, _P, _P, c_float, c_float,
                                               c_float, _P, _P, _P, _P, _P, _P]),
    "mhaq_fq_noise_f32": (c_int, [_P, c_int64, c_int64, c_uint64, c_uint64, _P, _P]),
    "mhaq_fq_packed_row_bytes": (c_int64, [c_int64, c_int]),
    "mhaq_fq_pack_f32": (c_int, [_P, _P, c_int, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int,
                                 c_int64, c_int64, c_int64, _P, _P]),
    "mhaq_fq_unpack_f32": (c_int, [_P, c_int, _P, _P, _P, c_int, c_int, c_int, c_int64, c_int64, c_int64, _P]),
    "mhaq_fq_iconv_weight_bytes": (c_int64, [c_int64, c_int64, _P, _P, _P, _P]),
    "mhaq_fq_act_codes_f32": (c_int, [_P, _P, _P, _P, _P, c_int64, c_int64, c_int64, _P, _P]),
    "mhaq_fq_iconv_u8": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, _P, c_int64, c_int64, c_int64, c_int64,
                                 c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P]),
    "mhaq_fq_iconv_fused_u8": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_int64, c_int64, c_int64, c_int64,
                                       c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "mhaq_fq_iconv_grouped_weight_bytes": (c_int64, [c_int64, c_int64, _P, _P, _P, _P, _P, _P, _P]),
    "mhaq_fq_iconv_grouped_u8": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_int64, c_int64, c_int64, c_int64,
                                         c_int64, _P, c_int, c_int, _P, _P]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


class MhaqLibraryError(ImportError):
    pass


def _load() -> ctypes.CDLL:
    if not os.path.exists(LIB_PATH):
        raise MhaqLibraryError(
            f"{LIB_PATH} not found: the sm_100a CUDA library has not been built. "
            "Run `python -c 'import __graft_entry__ as g; g.build()'` or "
            "`make -C mhaq_b200/csrc`. There is no CPU fallback."
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in _SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:  # pragma: no cover - build/header mismatch
            raise MhaqLibraryError(f"{LIB_PATH} does not export {name}") from exc
        fn.restype = res
        fn.argtypes = args
    got = lib.mhaq_fq_abi_version()
    if got != ABI_VERSION:
        raise MhaqLibraryError(f"ABI mismatch: library {got}, binding {ABI_VERSION}")
    return lib


lib = _load()


def check(rc: int, what: str) -> None:
    """Turn a C-ABI return code into a RuntimeError (no exceptions cross the ABI)."""
    if rc == 0:
        return
    if rc < 0:
        names = {-1: "MHAQ_FQ_EINVAL (bad shape/stride/method)", -2: "MHAQ_FQ_ENULL (null pointer)"}
        raise RuntimeError(f"{what}: {names.get(rc, rc)}")
    raise RuntimeError(f"{what}: CUDA error {rc}")
