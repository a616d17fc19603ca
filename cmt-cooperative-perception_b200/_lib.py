"""ctypes loader for ``libcmtcoop_b200.so`` (the C-ABI drop-in boundary, ``include/cmtcoop_b200.h``).

There is no fallback: if the shared library is missing, or the device is not sm_100, every
operator raises.  Nothing here imports ``oracle/``.
"""
from __future__ import annotations

import ctypes
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcmtcoop_b200.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "cmtcoop_b200.h")

CMT_F32, CMT_BF16, CMT_F16, CMT_BF16_SIMT = 0, 1, 2, 3
GEMM_RELU, GEMM_BIAS_PER_ROW, GEMM_FORCE_SIMT, GEMM_TRANSPOSE_OUT = 1, 2, 4, 8
LN_X_ROW_BROADCAST = 1

_c = ctypes
_vp, _i, _i64, _f, _sz = _c.c_void_p, _c.c_int, _c.c_int64, _c.c_float, _c.c_size_t

# name -> (restype, argtypes); mirrors include/cmtcoop_b200.h declaration by declaration.
SIGNATURES = {
    "cmt_version": (_i, []),
    "cmt_last_error_string": (_c.c_char_p, []),
    "cmt_check_device": (_i, [_i]),
    "cmt_ray_pe": (_i, [_vp, _vp, _i, _i, _i, _i, _f, _f, _vp, _i, _vp]),
    "cmt_ray_query_pe": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _f, _vp, _i, _vp]),
    "cmt_masked_view_sum": (_i, [_vp, _vp, _vp, _i64, _vp, _i, _i, _i, _i, _i, _vp, _vp]),
    "cmt_pos2embed": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "cmt_gather_tokens": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _i, _vp, _vp]),
    "cmt_sensor_key_keep": (_i, [_vp, _vp, _i, _i, _i, _i, _vp]),
    "cmt_gemm_bias_act": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i64, _i64, _i64, _i64, _i64, _i,
                               _i64, _i64, _i64, _f, _i, _i, _i, _vp, _vp]),
    "cmt_gemm_segmented": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _vp, _i, _i64, _i, _i64, _i64, _i64, _i, _i64, _i64, _i,
                                _i64, _f, _i, _i, _vp]),
    "cmt_nchw_to_padded_nhwc": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, _vp]),
    "cmt_shared_conv_tokens": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i64, _i, _i, _vp, _i]),
    "cmt_cross_attn_workspace_bytes": (_sz, [_i, _i, _i, _i]),
    "cmt_cross_attn_fwd": (_i, [_vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i64, _i64, _i64,
                                _i64, _i64, _i64, _vp, _vp, _vp, _i64, _i, _i, _vp, _sz, _vp]),
    "cmt_lse_merge": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i64, _i64, _i, _vp]),
    "cmt_lse_merge_peer": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _i, _vp]),
    "cmt_coop_max": (_i, [_vp, _vp, _vp, _i64, _vp]),
    "cmt_add_layernorm": (_i, [_vp, _vp, _vp, _vp, _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp]),
    "cmt_task_head_tail": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _i, _i, _i, _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "cmt_split3_bf16": (_i, [_vp, _vp, _vp, _vp, _i64, _i, _i, _i, _i64, _vp, _vp]),
    "cmt_bbox_topk_decode": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _vp, _f, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _i]),
    "cmt_debug_attn_timing": (_i, [_vp]),
}

_lib = None


class CmtLibraryError(RuntimeError):
    pass


def header_symbols(path: str = HEADER_PATH):
    """Names of every function the public header declares."""
    text = open(path).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(cmt_[a-z0-9_]+)\s*\(", text)))


def load():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise CmtLibraryError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(or `make -C cmt-cooperative-perception_b200/csrc`). There is no fallback implementation.")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return load().cmt_last_error_string().decode("utf-8", "replace")


def check(rc: int, what: str):
    if rc != 0:
        raise CmtLibraryError(f"{what} failed (code {rc}): {last_error()}")
