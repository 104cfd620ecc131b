"""ctypes binding of libdvd_b200.so (include/dvd_b200.h).

The product path has NO fallback: if the shared library is missing or a call fails, a
RuntimeError is raised.  Build with ``python -m dvd_b200.build`` (or ``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DVD_LIB", os.path.join(_HERE, "libdvd_b200.so"))      # DVD_LIB: instrumented build (tools/gemm_trace.py)

PREC_FP32 = 0
PREC_BF16 = 1
PREC_BF16X3 = 2
TABLE_ROW = 384 + 2304 + 3072

_vp = C.c_void_p


class Mat(C.Structure):
    _fields_ = [("f32", _vp), ("bf16", _vp), ("bf16_lo", _vp), ("n", C.c_int32), ("k", C.c_int32)]


class DecLayer(C.Structure):
    _fields_ = [("n1_w", _vp), ("n1_b", _vp), ("qkv", Mat), ("fc", Mat), ("n2_w", _vp), ("n2_b", _vp),
                ("conv1", Mat), ("bn1_scale", _vp), ("bn1_shift", _vp), ("dw_w", _vp), ("bn2_scale", _vp),
                ("bn2_shift", _vp), ("conv2", Mat), ("bn3_scale", _vp), ("bn3_shift", _vp),
                ("qkv_ln", Mat), ("qkv_colsum", _vp), ("qkv_cvec", _vp), ("conv1_ln", Mat), ("conv1_colsum", _vp), ("conv1_cvec", _vp)]


class Weights(C.Structure):
    _fields_ = [("pos", _vp), ("pyr", Mat * 7), ("pyr_b", _vp * 7), ("emb", Mat * 5), ("emb_b", _vp * 5),
                ("t_mlp0", Mat), ("t_mlp2", Mat), ("t_mlp0_b", _vp), ("t_mlp2_b", _vp),
                ("blk_ada", Mat), ("blk_ada_b", _vp), ("xattn_in", Mat), ("xattn_in_b", _vp),
                ("xattn_out", Mat), ("xattn_out_b", _vp), ("blk_qkv", Mat), ("blk_qkv_b", _vp),
                ("blk_proj", Mat), ("blk_proj_b", _vp), ("blk_fc1", Mat), ("blk_fc1_b", _vp),
                ("blk_fc2", Mat), ("blk_fc2_b", _vp), ("dec_hpe", _vp), ("dec_wpe", _vp),
                ("h_scale0", Mat), ("h_scale2", Mat), ("w_scale0", Mat), ("w_scale2", Mat),
                ("h_scale0_b", _vp), ("h_scale2_b", _vp), ("w_scale0_b", _vp), ("w_scale2_b", _vp),
                ("dec", DecLayer * 6), ("dec_ln_w", _vp), ("dec_ln_b", _vp), ("fin", Mat), ("fin_b", _vp),
                ("fin_ada", Mat), ("fin_ada_b", _vp), ("pyr_h", Mat * 7)]


class UnwarpDoc(C.Structure):
    _fields_ = [("photo", _vp), ("out", _vp), ("H", C.c_int32), ("W", C.c_int32)]


# name -> (restype, argtypes); mirrors include/dvd_b200.h one to one
_i, _f, _sz = C.c_int, C.c_float, C.c_size_t
_WP = C.POINTER(Weights)
_FP = C.POINTER(C.c_float)
SIGNATURES = {
    "dvd_version": (_i, []),
    "dvd_last_error": (C.c_char_p, []),
    "dvd_check_device": (_i, []),
    "dvd_unwarp_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "dvd_unwarp_u8": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "dvd_unwarp_f32_u8": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _f, _vp]),
    "dvd_unwarp_table_bytes": (_sz, [_i]),
    "dvd_unwarp_u8_plan": (_i, [C.POINTER(UnwarpDoc), _i, _i, _i, _i, _f, _vp, _sz, C.POINTER(C.c_longlong)]),
    "dvd_unwarp_u8_mixed": (_i, [_vp, _i, _vp, _vp]),
    "dvd_grid_sample_f32": (_i, [_vp, _vp, _vp, _i, _i, _i, _i, _i, _i, _vp]),
    "dvd_fullres_grid_f32": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _f, _vp]),
    "dvd_workspace_bytes": (_sz, [_i, _i, _i]),
    "dvd_tables_init": (_i, [_WP, _FP, _i, _vp, _vp]),
    "dvd_static_forward": (_i, [_WP, _vp, _sz, _i, _i, _i, _vp, _vp, _vp, _vp, _vp]),
    "dvd_denoise_step": (_i, [_WP, _vp, _sz, _i, _i, _i, _vp, _vp, _vp, _i, _vp, _f, _f, _vp, _vp, _vp]),
    "dvd_hyp_mean_clamp": (_i, [_vp, _vp, _i, _i, _vp]),
    "dvd_sample": (_i, [_WP, _vp, _sz, _i, _i, _i, _vp, _vp, _vp, _FP, _FP, _FP, _i, _vp, _vp, _vp]),
    "dvd_workspace_feat": (_vp, [_vp, _i, _i, _i]),
    "dvd_workspace_tensor": (_vp, [_vp, _i, _i, _i, C.c_char_p, C.POINTER(C.c_longlong)]),
    "dvd_test_gemm": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp, _sz, _vp]),
    "dvd_test_attention": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _f, _i, _vp, _sz, _vp]),
    "dvd_test_dwconv": (_i, [_vp, _vp, _vp, _vp, _vp, _vp, _vp, _i, _i, _vp]),
    "dvd_gemm_bf16": (_i, [_vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "dvd_gemm_tune": (_i, [_vp, _vp, _i, _vp, _vp, _i, _vp, _vp, _vp, _i, _vp, _vp, _vp, _vp, _i, _i, _i, _vp]),
    "dvd_debug_stop_after": (_i, [_i]),
    "dvd_profile_begin": (_i, []),
    "dvd_profile_end": (_i, [C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(C.c_longlong), C.POINTER(C.c_double)]),
    "dvd_launch_count": (C.c_longlong, [_i]),
}

_lib = None


def lib() -> C.CDLL:
    """Loads the shared library (once).  Raises loudly when it is missing: there is no CPU path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"{LIB_PATH} not found: the CUDA extension has not been built "
                               "(run `python -m dvd_b200.build`). dvd_b200 has no CPU fallback.")
        l = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(l, name)          # AttributeError if the .so is stale
            fn.restype = res
            fn.argtypes = args
        _lib = l
    return _lib


def check(rc: int, what: str = ""):
    if rc != 0:
        msg = lib().dvd_last_error().decode(errors="replace")
        raise RuntimeError(f"libdvd_b200 {what} failed (code {rc}): {msg}")


def ptr(t):
    """data_ptr of a tensor as c_void_p (None -> NULL)."""
    return None if t is None else _vp(t.data_ptr())


def stream_ptr():
    import torch
    return _vp(torch.cuda.current_stream().cuda_stream)
