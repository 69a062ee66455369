"""ctypes binding of libsvit_sm100.so (the C ABI declared in include/svit_b200.h).

There is no CPU fallback and no torch-op fallback: if the shared library is missing the import of
any compute path fails loudly with instructions to build it (``python -m svit_b200.build`` or
``__graft_entry__.build()``).
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
# SVIT_LIB selects an instrumented build of the same library (tools/*_timeline.py); never a different implementation
LIB_PATH = os.environ.get("SVIT_LIB") or os.path.join(HERE, "libsvit_sm100.so")

F32, BF16 = 0, 1
IMPL_AUTO, IMPL_SIMT, IMPL_TC = 0, 1, 2

vp, i32, i64, f32 = C.c_void_p, C.c_int32, C.c_int64, C.c_float


class GemmArgs(C.Structure):
    _fields_ = [
        ("A", vp), ("B", vp), ("C", vp),
        ("M", i64), ("N", i64), ("K", i64), ("lda", i64), ("ldb", i64), ("ldc", i64),
        ("transA", i32), ("transB", i32),
        ("bias", vp), ("residual", vp), ("ldr", i64),
        ("sample_scale", vp), ("rows_per_sample", i64),
        ("gelu_pre", vp), ("ldg", i64),
        ("pre_out", vp), ("ldp", i64),
        ("act", i32),
        ("rows_in", i64), ("rows_out", i64), ("row_off", i64),
        ("dtype", i32), ("out_dtype", i32), ("impl", i32),
        ("batch", i64), ("strideA", i64), ("strideB", i64), ("strideC", i64), ("b_inner", i64), ("strideB_inner", i64),
        ("a_inner", i64), ("strideA_inner", i64), ("alpha", f32),
        ("ln_stats", vp), ("ln_colsum", vp),
    ]


class AttnArgs(C.Structure):
    _fields_ = [
        ("q", vp), ("k", vp), ("v", vp), ("rel_h", vp), ("rel_w", vp), ("rel_t", vp), ("out", vp), ("lse", vp),
        ("B", i32), ("h", i32), ("qt", i32), ("qh", i32), ("qw", i32), ("kt", i32), ("kh", i32), ("kw", i32),
        ("O", i32), ("scale", f32), ("dtype", i32), ("impl", i32),
        ("dout", vp), ("dq", vp), ("dk", vp), ("dv", vp), ("d_rel_h", vp), ("d_rel_w", vp), ("d_rel_t", vp),
        ("ws_e", vp), ("ws_de", vp), ("ws_delta", vp),
        ("rel_tab", vp), ("idx_h", vp), ("idx_w", vp), ("idx_t", vp), ("key_cols", vp),
        ("ntab_h", i32), ("ntab_w", i32), ("ntab_t", i32),
        ("sel_tab", vp), ("sel_cols", i32),
        ("ws_s", vp), ("ws_dp", vp), ("ws_p", vp), ("ws_ds", vp), ("ws_dq", vp), ("sel_bwd", vp), ("nep", i32),
        ("d_rel_tab", vp), ("ws_etab", vp),
    ]


# name -> argtypes; every function returns int.  Mirrors include/svit_b200.h one to one
# (tests/test_abi_symbols.py checks that the two lists agree).
PROTOTYPES = {
    "svit_abi_version": [],
    "svit_destroy": [],
    "svit_row_stats": [vp, vp, i64, C.c_int, f32, C.c_int, vp],
    "svit_mlp_fused_supported": [i64, C.c_int, C.c_int, C.c_int],
    "svit_mlp_fused": [vp, vp, vp, vp, vp, vp, vp, i64, C.c_int, C.c_int, C.c_int, vp, vp, f32, vp],
    "svit_layernorm_fwd": [vp, vp, vp, vp, vp, vp, i64, C.c_int, f32, C.c_int, vp],
    "svit_layernorm_bwd": [vp, vp, vp, vp, vp, vp, vp, vp, i64, C.c_int, C.c_int, vp],
    "svit_pool_ln_fwd": [vp, i64, i64, i64, vp, vp, vp, vp, vp] + [C.c_int] * 7 + [f32, C.c_int, vp],
    "svit_pool_ln_fwd_save": [vp, i64, i64, i64, vp, vp, vp, vp, vp, vp] + [C.c_int] * 7 + [f32, C.c_int, vp],
    "svit_pool_ln_bwd_saved": [vp, i64, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp] + [C.c_int] * 7 + [f32, C.c_int, vp],
    "svit_pool_ln_bwd": [vp, i64, i64, i64, vp, vp, vp, vp, vp, vp, vp, vp, vp] + [C.c_int] * 7 + [f32, C.c_int, vp],
    "svit_skip_maxpool_fwd": [vp, vp] + [C.c_int] * 8 + [vp],
    "svit_skip_maxpool_bwd": [vp, vp, vp] + [C.c_int] * 8 + [vp],
    "svit_skip_maxpool_fwd_idx": [vp, vp, vp] + [C.c_int] * 8 + [vp],
    "svit_skip_maxpool_bwd_idx": [vp, vp, vp] + [C.c_int] * 8 + [vp],
    "svit_gemm": [C.POINTER(GemmArgs), vp],
    "svit_colsum": [vp, vp, i64, C.c_int, i64, C.c_int, vp],
    "svit_scale_rows": [vp, vp, vp, i64, C.c_int, i64, C.c_int, vp],
    "svit_attn_fwd": [C.POINTER(AttnArgs), vp],
    "svit_attn_bwd": [C.POINTER(AttnArgs), vp],
    "svit_assemble_tokens_fwd": [vp, vp, vp, vp, C.c_int, i64, C.c_int, C.c_int, C.c_int, C.c_int, vp],
    "svit_assemble_tokens_bwd": [vp, vp, vp, vp, C.c_int, i64, C.c_int, C.c_int, C.c_int, C.c_int, vp],
    "svit_im2col3d": [vp, vp] + [C.c_int] * 17 + [vp],
    "svit_col2im3d": [vp, vp] + [C.c_int] * 17 + [vp],
    "svit_gather_cls_obj_fwd": [vp, vp, C.c_int, i64, C.c_int, C.c_int, C.c_int, vp],
    "svit_gather_cls_obj_bwd": [vp, vp, C.c_int, i64, C.c_int, C.c_int, C.c_int, vp],
    "svit_roi_tokens_fwd": [vp, i64, vp, vp, i64, vp, C.c_int, vp] + [C.c_int] * 8 + [f32, C.c_int, C.c_int, vp],
    "svit_roi_tokens_bwd": [vp, i64, vp, vp, vp] + [C.c_int] * 8 + [f32, C.c_int, C.c_int, vp],
    "svit_roi_align_fwd": [vp, vp, vp] + [C.c_int] * 6 + [f32, C.c_int, C.c_int, C.c_int, vp],
    "svit_match_haog": [vp, vp, i64, vp],
    "svit_zero_empty_boxes": [vp, i64, f32, vp],
    "svit_normalize_u8": [vp, vp] + [C.c_int] * 4 + [f32] * 6 + [C.c_int, vp],
    "svit_s2d_clip": [vp, vp] + [C.c_int] * 9 + [f32] * 6 + [vp],
    "svit_patch_embed_s2d_supported": [C.c_int] * 11,
    "svit_patch_embed_s2d": [vp, vp, vp, vp, i64, C.c_int] + [C.c_int] * 15 + [vp],
    "svit_patch_embed_s2d_dgrad_supported": [C.c_int] * 11,
    "svit_patch_embed_s2d_dgrad": [vp, i64, C.c_int, vp, vp] + [C.c_int] * 15 + [vp],
    "svit_d2s_clip": [vp, vp] + [C.c_int] * 9 + [vp],
    "svit_crop_flip_normalize_u8": [vp, vp, vp, vp, vp] + [C.c_int] * 6 + [f32] * 6 + [C.c_int, vp],
    "svit_boxes_crop_flip": [vp, vp, vp, vp, vp, C.c_int, i64, C.c_int, C.c_int, f32, vp],
    "svit_head_fwd": [vp] * 14 + [C.c_int] * 8 + [vp],
    "svit_haog_loss": [vp, vp, C.c_int, i64, vp, vp, i64, vp, vp, vp, vp, vp, vp],
    "svit_grad_sqnorm": [vp, vp, vp, C.c_int, C.c_int, vp, vp],
    "svit_adamw_step": [vp, vp, vp, C.c_int, C.c_int, f32, f32, f32, f32, C.c_int, f32, vp, vp],
    "svit_adamw_step_dev": [vp, vp, vp, C.c_int, C.c_int, vp, f32, f32, f32, f32, vp, vp],
}

_lib = None


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found. The svit_b200 compute path is CUDA only (no fallback); build it with "
                "`python -m svit_b200.build` (needs nvcc, cross-compiles sm_100a without a GPU).")
        L = C.CDLL(LIB_PATH)
        for name, argt in PROTOTYPES.items():
            fn = getattr(L, name)  # AttributeError if the library does not export it
            fn.argtypes = argt
            fn.restype = C.c_int
        _lib = L
    return _lib


def check(rc: int, what: str):
    if rc == 0:
        return
    if rc < 0:
        msg = {-1: "invalid argument", -2: "unsupported configuration"}.get(rc, "argument error")
        raise RuntimeError(f"{what}: {msg} (svit error {rc})")
    raise RuntimeError(f"{what}: CUDA error {rc}")
