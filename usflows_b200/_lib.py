"""ctypes binding of libusflows_b200.so -- the only route from the Python host code to the CUDA kernels.

There is no fallback: if the library is missing it is (re)built with nvcc when possible, otherwise importing
the compute path raises.  Every wrapper raises RuntimeError with `usf_last_error()` on a non-zero status.
"""
from __future__ import annotations

import ctypes as C
import os
import shutil

from . import build as _build

_lib = None

c_f32p = C.c_void_p  # device pointers travel as integers
c_i64 = C.c_int64
c_i32 = C.c_int32


class LinearArgs(C.Structure):
    """Mirror of `usf_linear_args` (include/usflows_b200.h)."""

    _fields_ = [
        ("M", C.c_int64), ("N", C.c_int32), ("K", C.c_int32), ("engine", C.c_int32), ("trans_w", C.c_int32),
        ("a", C.c_void_p), ("a_lo", C.c_void_p), ("lda", C.c_int64),
        ("w", C.c_void_p), ("w_lo", C.c_void_p), ("ldw", C.c_int64),
        ("bias", C.c_void_p), ("relu", C.c_int32), ("resid_sign", C.c_float),
        ("resid", C.c_void_p), ("resid_lo", C.c_void_p), ("ldr", C.c_int64),
        ("colscale", C.c_void_p), ("postsub", C.c_void_p),
        ("out_f32", C.c_void_p), ("ld_f32", C.c_int64),
        ("out_hi", C.c_void_p), ("out_lo", C.c_void_p), ("ld_split", C.c_int64),
        ("out_bf16", C.c_void_p), ("ld_bf16", C.c_int64),
        ("resid_h16", C.c_void_p), ("resid_l16", C.c_void_p), ("ldr_16", C.c_int64),
        ("out_h16", C.c_void_p), ("out_l16", C.c_void_p), ("ld_16", C.c_int64),
        ("overflow_flag", C.c_void_p),
        ("split_k", C.c_int32), ("reserved0", C.c_int32),
    ]


class ConvPixArgs(C.Structure):
    """Mirror of `usf_conv_pix_args` (include/usflows_b200.h)."""

    _fields_ = [
        ("a16", C.c_void_p), ("n_images", C.c_int64),
        ("h", C.c_int32), ("w", C.c_int32), ("ksize", C.c_int32), ("dilation", C.c_int32),
        ("w1", C.c_void_p), ("bias1", C.c_void_p),
        ("n1", C.c_int32), ("relu1", C.c_int32), ("gated", C.c_int32), ("post_relu", C.c_int32),
        ("w2", C.c_void_p), ("bias2", C.c_void_p), ("gamma", C.c_void_p), ("beta", C.c_void_p),
        ("eps", C.c_float), ("sign", C.c_float),
        ("out_f32", C.c_void_p), ("ld_f32", C.c_int64), ("out16", C.c_void_p),
        ("relu_planes", C.c_int32), ("c_x", C.c_int32),
        ("x", C.c_void_p), ("ldx", C.c_int64), ("inv_mask", C.c_void_p), ("overflow_flag", C.c_void_p),
    ]


class GlueArgs(C.Structure):
    """Mirror of `usf_glue_args` (include/usflows_b200.h)."""

    _fields_ = [
        ("h", C.c_void_p), ("l", C.c_void_p), ("ld", C.c_int64),
        ("src_f32", C.c_void_p), ("ld_src", C.c_int64),
        ("rows", C.c_int64), ("n", C.c_int32), ("reserved0", C.c_int32),
        ("mask_h", C.c_void_p), ("ld_mask", C.c_int64),
        ("sign", C.c_float), ("reserved1", C.c_int32),
        ("out_h", C.c_void_p), ("out_l", C.c_void_p), ("ld_out", C.c_int64),
        ("t_h", C.c_void_p), ("t_l", C.c_void_p), ("ld_t", C.c_int64),
        ("colsum", C.c_void_p),
        ("mul", C.c_void_p), ("ld_mul", C.c_int64),
        ("colsum2", C.c_void_p),
        ("overflow_flag", C.c_void_p),
    ]


class PlanLinear(C.Structure):
    """Mirror of `usf_plan_linear` (include/usflows_b200.h)."""

    _fields_ = [
        ("N", C.c_int32), ("K", C.c_int32), ("engine", C.c_int32), ("relu", C.c_int32),
        ("w", C.c_void_p), ("w_lo", C.c_void_p), ("ldw", C.c_int64),
        ("bias", C.c_void_p),
        ("src", C.c_int32), ("dst", C.c_int32),
        ("in_col0", C.c_int32), ("in_width", C.c_int32),
        ("out_col0", C.c_int32), ("resid_sign", C.c_float),
    ]


class Dequant(C.Structure):
    """Mirror of `usf_dequant` (include/usflows_b200.h)."""

    _fields_ = [
        ("mode", C.c_int32), ("reserved0", C.c_int32), ("seed", C.c_uint64), ("row0", C.c_int64), ("dev_params", C.c_void_p),
    ]


class Draw(C.Structure):
    """Mirror of `usf_draw` (include/usflows_b200.h)."""

    _fields_ = [("seed", C.c_uint64), ("offset", C.c_uint64), ("row0", C.c_int64), ("dev_params", C.c_void_p)]


DEQUANT_UNIFORM, DEQUANT_MIDPOINT = 0, 1
MODE_CODES = {"fp32": 0, "fp32_tf32": 1, "fp32_simt": 2, "tf32": 3, "bf16": 4}
PLAN_SRC_STREAM, PLAN_SRC_HIDDEN = 0, 1
PLAN_DST_STREAM, PLAN_DST_HIDDEN, PLAN_DST_SEGMENT = 0, 1, 2


class Planes(C.Structure):
    """Mirror of `usf_planes` (include/usflows_b200.h)."""

    _fields_ = [
        ("f32", C.c_void_p), ("ld_f32", C.c_int64),
        ("hi", C.c_void_p), ("lo", C.c_void_p), ("ld_split", C.c_int64),
        ("bf16", C.c_void_p), ("ld_bf16", C.c_int64),
        ("h16", C.c_void_p), ("l16", C.c_void_p), ("ld_16", C.c_int64),
    ]


ENGINE_SIMT, ENGINE_TC_3XTF32, ENGINE_TC_TF32, ENGINE_TC_BF16, ENGINE_TC_3XF16 = 0, 1, 2, 3, 4
BASE_LAPLACE, BASE_NORMAL = 0, 1
LP_INF, LP_1, LP_2 = 0, 1, 2
NORM_LOGNORMAL, NORM_GAMMA_MIXTURE, NORM_GENGAMMA_MIXTURE, NORM_LOGNORMAL_MIXTURE = 0, 1, 2, 3
TRI_NONE, TRI_LOWER_UPPER, TRI_UPPER_LOWER = 0, 1, 2

_P, _I64, _I32, _F, _U64 = C.c_void_p, C.c_int64, C.c_int32, C.c_float, C.c_uint64

# name -> (restype, argtypes); must list every symbol declared in include/usflows_b200.h
SIGNATURES = {
    "usf_last_error": (C.c_char_p, []),
    "usf_abi_version": (C.c_int, []),
    "usf_device_info": (C.c_int, [C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int64)]),
    "usf_linear": (C.c_int, [C.POINTER(LinearArgs), _P]),
    "usf_ingest": (C.c_int, [_P, _I64, _I64, _I32, _P, _P, _P, _P, _I64, _P, _P, _I64, _P, _I64, _P]),
    "usf_ingest_f16": (C.c_int, [_P, _I64, _I64, _I32, _P, _P, _P, _P, _P, _I64, _P, _P]),
    "usf_ingest_u8": (C.c_int, [_P, _I64, _I64, _I32, C.POINTER(Dequant), _P, _P, _P, C.POINTER(Planes), _P, _P]),
    "usf_layout_transpose_u8": (C.c_int, [_P, _I64, _I32, _I32, C.POINTER(Dequant), _P, _I32, _P, _P]),
    "usf_flow_logprob_u8": (C.c_int, [_P, _P, _I64, _I64, C.POINTER(Dequant), _P, _P, _P]),
    "usf_split_f16": (C.c_int, [_P, _I64, _I32, _I64, _P, _P, _I64, _P, _P]),
    "usf_base_logprob": (C.c_int, [_P, _P, _I64, _I64, _I32, _P, _P, _I32, _F, _P, _P]),
    "usf_flow_small": (C.c_int, [_P, _I64, _I64, _I32, _P, _I32, _P, _I32, _I32, _I32, _P, _I64, _P]),
    "usf_base_sample": (C.c_int, [_I64, _I32, _P, _P, _I32, _U64, _U64, _P, _I64, _P, _P, _I64, _P, _I64, _P]),
    "usf_base_sample_at": (C.c_int, [_I64, _I32, _P, _P, _I32, C.POINTER(Draw), _P, _I64, _P, _P, _I64, _P, _I64, _P]),
    "usf_quantize_u8": (C.c_int, [_P, _I64, _I64, _I32, _P, _I64, _P]),
    "usf_affine_couple": (C.c_int, [_P, _I64, _I64, _I32, _P, _I64, _P, _P, _I64, _P, _I64, _P, _P, _I64, _P, _F, _F, _F, _P, _P]),
    "usf_sub_rows": (C.c_int, [_P, _P, _I64, _P]),
    "usf_radial_logprob": (C.c_int, [_P, _P, _I64, _I64, _I32, _P, _I32, _I32, _P, _I32, _F, _F, _P, _P]),
    "usf_radial_sample": (C.c_int, [_I64, _I32, _P, _I32, _I32, _P, _I32, _U64, _U64, _P, _I64, _P]),
    "usf_radial_sample_at": (C.c_int, [_I64, _I32, _P, _I32, _I32, _P, _I32, C.POINTER(Draw), _P, _I64, _P]),
    "usf_layout_transpose": (C.c_int, [_P, _I64, _I32, _I32, _P, _I32, _I32, _P, _P]),
    "usf_layout_transpose_to_u8": (C.c_int, [_P, _I64, _I32, _I32, _P, _I32, _P, _P]),
    "usf_im2col": (C.c_int, [_P, _I64, _I64, _I32, _I32, _I32, _I32, _I32, _P, _I32, C.POINTER(Planes), _P, _P]),
    "usf_conv2d_rows": (C.c_int, [C.POINTER(LinearArgs), _P, _I64, _I64, _I32, _I32, _I32, _I32, _I32, _P, _I32, _P]),
    "usf_masked_add": (C.c_int, [_P, _I64, _P, _I64, _I64, _I32, _I32, _P, _F, _P]),
    "usf_pix_encode": (C.c_int, [_P, _I64, _I64, _I32, _I32, _P, _I32, _P, _P, _P]),
    "usf_conv2d_pix": (C.c_int, [C.POINTER(ConvPixArgs), _P]),
    "usf_gate_norm": (C.c_int, [_P, _I64, _P, _I64, _I64, _I32, _I32, _I32, _P, _P, _F, _P, _I64, C.POINTER(Planes), _I32,
                                C.POINTER(Planes), _P, _P]),
    "usf_leaky_relu": (C.c_int, [_P, _I64, _I64, _I32, _F, _P, _I64, _P, _P]),
    "usf_permute": (C.c_int, [_P, _I64, _I64, _I32, _P, _P, _I64, _P]),
    "usf_lu_assemble": (C.c_int, [_P, _P, _I32, _I64, _P, _P, _I64, _I32, _P]),
    "usf_lu_logabsdet": (C.c_int, [_P, _I32, _I64, _P, _P]),
    "usf_vec_logabs": (C.c_int, [_P, _I64, _P, _P]),
    "usf_tri_inverse_work_floats": (C.c_int64, [_I32]),
    "usf_tri_inverse": (C.c_int, [_P, _I32, _I64, _I32, _I32, _P, _I64, _P, _P]),
    "usf_transpose": (C.c_int, [_P, _I32, _I32, _I64, _P, _I64, _P]),
    "usf_scale_rows_cols": (C.c_int, [_P, _I32, _I32, _I64, _P, _P, _P, _I64, _P]),
    "usf_split_tf32": (C.c_int, [_P, _I64, _I32, _I64, _P, _P, _I64, _P]),
    "usf_to_bf16": (C.c_int, [_P, _I64, _I32, _I64, _P, _I64, _P]),
    "usf_householder_right": (C.c_int, [_P, _I32, _I64, _P, _P, _P]),
    "usf_softplus": (C.c_int, [_P, _I64, _P, _P]),
    "usf_matmul_f64": (C.c_int, [_P, _I64, _P, _I64, _P, _I64, _I32, _I32, _I32, _P]),
    "usf_matmul_f64_tri": (C.c_int, [_P, _I64, _P, _I64, _P, _I64, _I32, _I32, _P]),
    "usf_plan_create": (C.c_int, [C.POINTER(_P), _I32, _I32, _I64]),
    "usf_plan_add_linear": (C.c_int, [_P, C.POINTER(PlanLinear)]),
    "usf_plan_set_base": (C.c_int, [_P, _I32, _P, _P, _F]),
    "usf_plan_finalize": (C.c_int, [_P]),
    "usf_plan_workspace_bytes": (C.c_int64, [_P]),
    "usf_flow_apply": (C.c_int, [_P, _P, _I64, _I64, _P, _I64, _P, _P]),
    "usf_flow_logprob": (C.c_int, [_P, _P, _I64, _I64, _P, _P, _P]),
    "usf_plan_destroy": (C.c_int, [_P]),
    "usf_planes_glue": (C.c_int, [C.POINTER(GlueArgs), _P]),
    "usf_base_backward": (C.c_int, [_P, _I64, _I64, _I32, _P, _P, _I32, _P, _P, _I64, _P, _P, _I64, _P, _P, _P]),
    "usf_mat_prep": (C.c_int, [_P, _I64, _I32, _I32, _I32, _P, _P, _F, _P, _I64, _P, _P, _I64, _P, _P, _I64, _P, _P]),
    "usf_rowdot": (C.c_int, [_P, _I64, _I32, _I32, _P, _P, _F, _P, _P]),
    "usf_colcomb": (C.c_int, [_P, _I64, _I32, _I32, _P, _F, _P, _P]),
    "usf_rank1": (C.c_int, [_P, _I64, _I32, _I32, _P, _P, _F, _P]),
    "usf_tri_mask": (C.c_int, [_P, _I64, _I32, _I32, _F, _P, _I64, _F, _P, _I64, _P]),
    "usf_tri_inverse_batched": (C.c_int, [_P, _P, _P, _I32, _I64, _I64, _I32, C.c_uint32, _P]),
    "usf_debug_set_block_n": (C.c_int, [C.c_int]),
    "usf_debug_set_pdl": (C.c_int, [C.c_int]),
    "usf_debug_set_store_path": (C.c_int, [C.c_int]),
}


def library_path() -> str:
    return _build.LIB


def load():
    """Load (building first if the sources changed and nvcc exists).  Raises if impossible."""
    global _lib
    if _lib is not None:
        return _lib
    if _build.needs_build():
        nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
        if os.path.exists(nvcc) or shutil.which("nvcc"):
            _build.build()
        elif not os.path.exists(_build.LIB):
            raise RuntimeError(
                "usflows_b200: libusflows_b200.so is not built and nvcc is unavailable; run "
                "`python -m usflows_b200.build` (there is no CPU fallback)")
    lib = C.CDLL(_build.LIB)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the ABI and this table disagree
        fn.restype = res
        fn.argtypes = args
    if lib.usf_abi_version() != 10:
        raise RuntimeError("usflows_b200: ABI version mismatch between _lib.py and the shared library")
    _lib = lib
    return lib


def check(status: int) -> None:
    if status != 0:
        msg = load().usf_last_error().decode(errors="replace")
        raise RuntimeError(f"usflows_b200 [{status}]: {msg}")
