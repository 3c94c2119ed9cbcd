"""Typed Python wrappers over the C ABI: torch CUDA tensors in, kernels launched on the current stream.

torch is used here for device memory and stream handles only.  Non-CUDA tensors raise: there is no CPU
path in this package (the CPU oracle lives in oracle/ and is test infrastructure).
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Optional

import torch

from . import _lib
from ._lib import (BASE_LAPLACE, BASE_NORMAL, ENGINE_SIMT, ENGINE_TC_3XF16, ENGINE_TC_3XTF32,  # noqa: F401
                   ENGINE_TC_BF16, ENGINE_TC_TF32, LP_1, LP_2, LP_INF, NORM_GAMMA_MIXTURE, NORM_GENGAMMA_MIXTURE, NORM_LOGNORMAL_MIXTURE,
                   NORM_LOGNORMAL, TRI_LOWER_UPPER, TRI_NONE, TRI_UPPER_LOWER, LinearArgs, Planes, check)


LAUNCHES = 0     # kernels launched through this module since the caller last reset it (bench.py `gpu_launches`)


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


class on_device:
    """Makes the device of `t` the current CUDA device for the duration of the block.  The C ABI launches on the
    stream it is handed and has no device argument: `_stream()` is the current stream of the CURRENT device, so every
    public entry point (Flow.log_prob / sample / ..., the layer and distribution methods) runs its launches inside
    this guard -- a flow living on cuda:1 works while cuda:0 is current, as it does in the reference's plain PyTorch."""

    def __init__(self, t):
        dev = t.device if isinstance(t, torch.Tensor) else torch.device(t)
        self._guard = torch.cuda.device(dev) if dev.type == "cuda" and torch.cuda.is_available() else None

    def __enter__(self):
        if self._guard is not None:
            self._guard.__enter__()
        return self

    def __exit__(self, *exc):
        if self._guard is not None:
            self._guard.__exit__(*exc)
        return False


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def require_cuda(t: torch.Tensor, name: str = "tensor", dtype=torch.float32) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"usflows_b200: {name} must be a CUDA tensor (no CPU fallback exists)")
    if dtype is not None and t.dtype != dtype:
        raise RuntimeError(f"usflows_b200: {name} must have dtype {dtype}, got {t.dtype}")
    return t


def _ld(t: torch.Tensor) -> int:
    """Leading dimension of a 2-D row-major view (last dim contiguous)."""
    if t.dim() == 1:
        return t.shape[0]
    assert t.dim() == 2 and (t.stride(1) == 1 or t.shape[1] == 1), "row-major 2-D view expected"
    return t.stride(0) if t.shape[0] > 1 else max(t.stride(0), t.shape[1])


def pad4(n: int, mult: int = 8) -> int:
    return (n + mult - 1) // mult * mult


@dataclass
class Act:
    """One activation matrix [rows, width] in up to three storage planes (views into workspaces)."""

    rows: int
    width: int
    f32: Optional[torch.Tensor] = None      # full fp32 values
    hi: Optional[torch.Tensor] = None       # tf32-representable high part  (value = hi + lo)
    lo: Optional[torch.Tensor] = None
    bf16: Optional[torch.Tensor] = None
    h16: Optional[torch.Tensor] = None      # fp16 split planes: value = h16 + l16 * 2^-11
    l16: Optional[torch.Tensor] = None

    def resid_planes(self):
        if self.f32 is not None:
            return self.f32, None
        if self.hi is not None:
            return self.hi, self.lo
        raise RuntimeError("activation has no fp32-accurate plane to use as a residual")


# the planes of an Act each contraction engine's operands are prepared in (what `linear` reads as A)
ENGINE_PLANES = {ENGINE_SIMT: ("f32",), ENGINE_TC_TF32: ("f32",), ENGINE_TC_3XF16: ("h16", "l16"),
                 ENGINE_TC_3XTF32: ("hi", "lo"), ENGINE_TC_BF16: ("bf16",)}


def linear(engine: int, a: Act, w, w_lo, N: int, K: int, *, bias=None, relu=False, resid: Optional[Act] = None,
           resid_sign: float = 1.0, colscale=None, postsub=None, out: Act, trans_w: bool = False,
           overflow_flag: Optional[torch.Tensor] = None) -> None:
    """out = epilogue(a . w^T); see usf_linear in include/usflows_b200.h."""
    args = LinearArgs()
    args.M, args.N, args.K = a.rows, N, K
    args.engine, args.trans_w = engine, int(trans_w)
    if engine == ENGINE_TC_3XF16:
        args.a, args.a_lo, args.lda = _ptr(a.h16), _ptr(a.l16), _ld(a.h16)
    elif engine == ENGINE_TC_BF16:
        args.a, args.a_lo, args.lda = _ptr(a.bf16), None, _ld(a.bf16)
    elif engine == ENGINE_TC_3XTF32:
        args.a, args.a_lo, args.lda = _ptr(a.hi), _ptr(a.lo), _ld(a.hi)
    elif a.f32 is not None:
        args.a, args.a_lo, args.lda = _ptr(a.f32), None, _ld(a.f32)
    else:  # SIMT / TF32 reading split planes (SIMT adds lo; TF32 uses the hi plane)
        args.a, args.a_lo, args.lda = _ptr(a.hi), (_ptr(a.lo) if engine == ENGINE_SIMT else None), _ld(a.hi)
    args.w, args.w_lo, args.ldw = _ptr(w), _ptr(w_lo), _ld(w)
    args.bias, args.relu, args.resid_sign = _ptr(bias), int(relu), float(resid_sign)
    if resid is not None:
        if resid.f32 is None and resid.hi is None and resid.h16 is not None:
            args.resid_h16, args.resid_l16, args.ldr_16 = _ptr(resid.h16), _ptr(resid.l16), _ld(resid.h16)
        else:
            r, rl = resid.resid_planes()
            args.resid, args.resid_lo, args.ldr = _ptr(r), _ptr(rl), _ld(r)
    args.colscale, args.postsub = _ptr(colscale), _ptr(postsub)
    if out.f32 is not None:
        args.out_f32, args.ld_f32 = _ptr(out.f32), _ld(out.f32)
    if out.hi is not None:
        args.out_hi, args.out_lo, args.ld_split = _ptr(out.hi), _ptr(out.lo), _ld(out.hi)
    if out.bf16 is not None:
        args.out_bf16, args.ld_bf16 = _ptr(out.bf16), _ld(out.bf16)
    if out.h16 is not None:
        args.out_h16, args.out_l16, args.ld_16 = _ptr(out.h16), _ptr(out.l16), _ld(out.h16)
        args.overflow_flag = _ptr(overflow_flag)
    global LAUNCHES
    LAUNCHES += 1
    check(_lib.load().usf_linear(C.byref(args), _stream()))


def ingest(x: torch.Tensor, out: Act, *, div=None, mul=None, sub=None,
           overflow_flag: Optional[torch.Tensor] = None) -> None:
    global LAUNCHES
    LAUNCHES += 1
    rows, d = x.shape
    if out.h16 is not None:
        check(_lib.load().usf_ingest_f16(_ptr(x), _ld(x), rows, d, _ptr(div), _ptr(mul), _ptr(sub), _ptr(out.h16),
                                         _ptr(out.l16), _ld(out.h16), _ptr(overflow_flag), _stream()))
        return
    check(_lib.load().usf_ingest(
        _ptr(x), _ld(x), rows, d, _ptr(div), _ptr(mul), _ptr(sub),
        _ptr(out.f32), _ld(out.f32) if out.f32 is not None else 0,
        _ptr(out.hi), _ptr(out.lo), _ld(out.hi) if out.hi is not None else 0,
        _ptr(out.bf16), _ld(out.bf16) if out.bf16 is not None else 0, _stream()))


# ---- 8-bit inputs ---------------------------------------------------------------------------------------------------------
DEQUANT_MODES = {"uniform": _lib.DEQUANT_UNIFORM, "midpoint": _lib.DEQUANT_MIDPOINT}


@dataclass(frozen=True)
class Dequant:
    """How 8-bit rows become fp32 (usf_dequant): `mode` ("uniform" / "midpoint"), the Philox key `seed`, the global row of
    local row 0 `row0`, and optionally `params`, a device int64 [2] tensor {seed, row base} read at run time (seed replaced,
    row base added to row0) so that one captured graph serves every call."""

    mode: str
    seed: int
    row0: int = 0
    params: Optional[torch.Tensor] = None

    def shifted(self, rows: int) -> "Dequant":
        return Dequant(self.mode, self.seed, self.row0 + int(rows), self.params)

    def struct(self):
        s = _lib.Dequant()
        s.mode, s.seed, s.row0 = DEQUANT_MODES[self.mode], self.seed & (2**64 - 1), self.row0
        s.dev_params = _ptr(self.params)
        return s


def draw_seed() -> int:
    """One 63-bit dequantisation seed from torch.default_generator (`torch.manual_seed` reproduces it)."""
    return int(torch.empty((), dtype=torch.int64).random_(0, 2**63 - 1, generator=torch.default_generator))


def dequant_spec(x, mode, seed=None, row0: int = 0) -> Optional[Dequant]:
    """Validates a `dequantize=` argument against the input; None when `mode` is None (fp32 input)."""
    if mode is None:
        return None
    if mode not in DEQUANT_MODES:
        raise ValueError(f"usflows_b200: unknown dequantize mode {mode!r}; choose from {tuple(DEQUANT_MODES)}")
    if not isinstance(x, torch.Tensor) or x.dtype != torch.uint8:
        raise ValueError(f"usflows_b200: dequantize={mode!r} takes a uint8 input, got "
                         f"{x.dtype if isinstance(x, torch.Tensor) else type(x).__name__}")
    return Dequant(mode, draw_seed() if seed is None else int(seed), int(row0))


def ingest_u8(x: torch.Tensor, dq: Dequant, out: Act, *, div=None, mul=None, sub=None,
              overflow_flag: Optional[torch.Tensor] = None) -> None:
    """`ingest` reading 8-bit rows x [rows, d] (uint8), dequantised as `dq` says; see usf_ingest_u8."""
    global LAUNCHES
    LAUNCHES += 1
    rows, d = x.shape
    p, s = _planes_struct(out), dq.struct()
    check(_lib.load().usf_ingest_u8(_ptr(x), _ld(x), rows, d, C.byref(s), _ptr(div), _ptr(mul), _ptr(sub), C.byref(p),
                                    _ptr(overflow_flag), _stream()))


def dequantize(x_u8: torch.Tensor, mode: str = "uniform", seed: Optional[int] = None, row_offset: int = 0) -> torch.Tensor:
    """fp32 values of the 8-bit CUDA tensor `x_u8` [rows, *event] (a 1-D tensor is one row): element j (flat index within
    the row) of row r becomes (k + u) / 256 with Philox noise u keyed by (seed, row_offset + r, j) ("uniform", the
    reference's DequantizedDataset), or (k + 0.5) / 256 ("midpoint").  `seed=None` draws one from torch.default_generator.
    The values are exactly those `Flow.log_prob(x_u8, dequantize=mode, seed=seed)` evaluates."""
    dq = dequant_spec(x_u8, mode, seed, row_offset)
    require_cuda(x_u8, "x_u8", torch.uint8)
    x2 = x_u8.reshape(1, -1) if x_u8.dim() <= 1 else x_u8.reshape(x_u8.shape[0], math.prod(x_u8.shape[1:]))
    if x2.shape[1] > 0 and x2.stride(1) != 1:
        x2 = x2.contiguous()
    out = torch.empty(x2.shape, dtype=torch.float32, device=x_u8.device)
    if out.numel():
        with on_device(x_u8):
            ingest_u8(x2, dq, Act(x2.shape[0], x2.shape[1], f32=out))
    return out.reshape(x_u8.shape)


def base_logprob(z: Act, loc, scale, kind: int, add_const: float, out: torch.Tensor) -> None:
    global LAUNCHES
    LAUNCHES += 1
    p, pl = z.resid_planes()
    check(_lib.load().usf_base_logprob(_ptr(p), _ptr(pl), _ld(p), z.rows, z.width, _ptr(loc), _ptr(scale), kind,
                                       float(add_const), _ptr(out), _stream()))


def base_sample(out: Act, loc, scale, kind: int, seed: int, offset: int) -> None:
    check(_lib.load().usf_base_sample(
        out.rows, out.width, _ptr(loc), _ptr(scale), kind, seed & (2**64 - 1), offset & (2**64 - 1),
        _ptr(out.f32), _ld(out.f32) if out.f32 is not None else 0,
        _ptr(out.hi), _ptr(out.lo), _ld(out.hi) if out.hi is not None else 0,
        _ptr(out.bf16), _ld(out.bf16) if out.bf16 is not None else 0, _stream()))


@dataclass(frozen=True)
class Draw:
    """Which Philox draws a sampling call makes (usf_draw): key `seed`, sub-stream `offset`, the global row of local row 0
    `row0`, and optionally `params`, a device int64 [2] tensor {seed, row base} read at run time (seed replaced, row base
    added to row0) so that one captured graph serves every chunk.  Rows [r0, r1) of a call are the call `shifted(r0)` over
    r1 - r0 rows."""

    seed: int
    row0: int = 0
    params: Optional[torch.Tensor] = None
    offset: int = 0

    def shifted(self, rows: int) -> "Draw":
        return Draw(self.seed, self.row0 + int(rows), self.params, self.offset)

    @property
    def plain(self) -> bool:
        """The draws of the row0 = 0 entries (usf_base_sample / usf_radial_sample)."""
        return self.row0 == 0 and self.params is None

    def struct(self):
        s = _lib.Draw()
        s.seed, s.offset, s.row0 = self.seed & (2**64 - 1), self.offset & (2**64 - 1), self.row0
        s.dev_params = _ptr(self.params)
        return s


def base_sample_at(out: Act, loc, scale, kind: int, draw: Draw) -> None:
    """`base_sample` drawing the global rows draw.row0 .. draw.row0 + out.rows - 1; see usf_base_sample_at."""
    s = draw.struct()
    check(_lib.load().usf_base_sample_at(
        out.rows, out.width, _ptr(loc), _ptr(scale), kind, C.byref(s),
        _ptr(out.f32), _ld(out.f32) if out.f32 is not None else 0,
        _ptr(out.hi), _ptr(out.lo), _ld(out.hi) if out.hi is not None else 0,
        _ptr(out.bf16), _ld(out.bf16) if out.bf16 is not None else 0, _stream()))


def quantize_u8(y: torch.Tensor, out: torch.Tensor) -> None:
    """out [rows, d] uint8 = min(255, max(0, floor(256 y))), NaN -> 0, from fp32 y [rows, d]; see usf_quantize_u8."""
    global LAUNCHES
    LAUNCHES += 1
    rows, d = y.shape
    check(_lib.load().usf_quantize_u8(_ptr(y), _ld(y), rows, d, _ptr(out), _ld(out), _stream()))


def quantize(y: torch.Tensor) -> torch.Tensor:
    """8-bit values of the fp32 CUDA tensor `y` [rows, *event] (a 1-D tensor is one row): min(255, max(0, floor(256 y))),
    NaN -> 0 -- the inverse of `dequantize` in both modes, and the pixels `Flow.sample(..., quantize=True)` returns."""
    require_cuda(y, "y")
    y2 = y.reshape(1, -1) if y.dim() <= 1 else y.reshape(y.shape[0], math.prod(y.shape[1:]))
    if y2.shape[1] > 0 and y2.stride(1) != 1:
        y2 = y2.contiguous()
    out = torch.empty(y2.shape, dtype=torch.uint8, device=y.device)
    if out.numel():
        with on_device(y):
            quantize_u8(y2, out)
    return out.reshape(y.shape)


def flow_small(x: torch.Tensor, prog_i32: torch.Tensor, blob: torch.Tensor, n_ops: int, D: int, H: int,
               out: torch.Tensor) -> None:
    """Whole layer stack in one launch (d <= 8, conditioner width <= 64); see usf_flow_small."""
    global LAUNCHES
    LAUNCHES += 1
    rows, d = x.shape
    check(_lib.load().usf_flow_small(_ptr(x), _ld(x), rows, d, _ptr(prog_i32), n_ops, _ptr(blob), blob.numel(), D, H,
                                     _ptr(out), _ld(out), _stream()))


def affine_couple(st: torch.Tensor, x: Act, direction: float, s_min: float, s_max: float,
                  row_ladj: Optional[torch.Tensor] = None, overflow_flag: Optional[torch.Tensor] = None) -> None:
    """In-place affine coupling update of the planes of `x` [rows, h] from st [rows, 2h]; see usf_affine_couple."""
    global LAUNCHES
    LAUNCHES += 1
    check(_lib.load().usf_affine_couple(
        _ptr(st), _ld(st), x.rows, x.width,
        _ptr(x.f32), _ld(x.f32) if x.f32 is not None else 0,
        _ptr(x.hi), _ptr(x.lo), _ld(x.hi) if x.hi is not None else 0,
        _ptr(x.bf16), _ld(x.bf16) if x.bf16 is not None else 0,
        _ptr(x.h16), _ptr(x.l16), _ld(x.h16) if x.h16 is not None else 0,
        _ptr(overflow_flag), float(direction), float(s_min), float(s_max), _ptr(row_ladj), _stream()))


def radial_logprob(z: Act, loc, p_kind: int, norm_kind: int, norm_params: torch.Tensor, n_comp: int, dv_const: float,
                   add_const: float, out: torch.Tensor) -> None:
    """Lp-radial base density of the rows of z; see usf_radial_logprob."""
    global LAUNCHES
    LAUNCHES += 1
    p, pl = z.resid_planes()
    check(_lib.load().usf_radial_logprob(_ptr(p), _ptr(pl), _ld(p), z.rows, z.width, _ptr(loc), p_kind, norm_kind,
                                         _ptr(norm_params), n_comp, float(dv_const), float(add_const), _ptr(out),
                                         _stream()))


def radial_sample(out: torch.Tensor, loc, p_kind: int, norm_kind: int, norm_params: torch.Tensor, n_comp: int,
                  seed: int, offset: int) -> None:
    rows, d = out.shape
    check(_lib.load().usf_radial_sample(rows, d, _ptr(loc), p_kind, norm_kind, _ptr(norm_params), n_comp,
                                        seed & (2**64 - 1), offset & (2**64 - 1), _ptr(out), _ld(out), _stream()))


def radial_sample_at(out: torch.Tensor, loc, p_kind: int, norm_kind: int, norm_params: torch.Tensor, n_comp: int,
                     draw: Draw) -> None:
    """`radial_sample` drawing the global rows draw.row0 .. draw.row0 + rows - 1; see usf_radial_sample_at."""
    rows, d = out.shape
    s = draw.struct()
    check(_lib.load().usf_radial_sample_at(rows, d, _ptr(loc), p_kind, norm_kind, _ptr(norm_params), n_comp, C.byref(s),
                                           _ptr(out), _ld(out), _stream()))


def _planes_struct(a: Optional[Act]):
    if a is None:
        return None
    p = Planes()
    if a.f32 is not None:
        p.f32, p.ld_f32 = _ptr(a.f32), _ld(a.f32)
    if a.hi is not None:
        p.hi, p.lo, p.ld_split = _ptr(a.hi), _ptr(a.lo), _ld(a.hi)
    if a.bf16 is not None:
        p.bf16, p.ld_bf16 = _ptr(a.bf16), _ld(a.bf16)
    if a.h16 is not None:
        p.h16, p.l16, p.ld_16 = _ptr(a.h16), _ptr(a.l16), _ld(a.h16)
    return p


def gate_norm(o: torch.Tensor, n: int, *, xres: Optional[torch.Tensor] = None, gated: bool = False, gamma=None, beta=None,
              eps: float = 1e-5, y_f32: Optional[torch.Tensor] = None, act: Optional[Act] = None, act_relu: bool = False,
              raw: Optional[Act] = None, overflow_flag: Optional[torch.Tensor] = None, pre_relu: bool = False) -> None:
    """GatedMLP gate + LayerNormVector + re-encoding between two contractions of a ConvNet conditioner; see usf_gate_norm."""
    global LAUNCHES
    LAUNCHES += 1
    pa, pr = _planes_struct(act), _planes_struct(raw)
    check(_lib.load().usf_gate_norm(
        _ptr(o), _ld(o), _ptr(xres), _ld(xres) if xres is not None else 0, o.shape[0], n, int(gated), int(pre_relu), _ptr(gamma),
        _ptr(beta), float(eps), _ptr(y_f32), _ld(y_f32) if y_f32 is not None else 0,
        C.byref(pa) if pa is not None else None, int(act_relu), C.byref(pr) if pr is not None else None,
        _ptr(overflow_flag), _stream()))


def layout_transpose(x: torch.Tensor, n: int, a: int, b: int, out: torch.Tensor, scale=None, scale_mode: int = 0,
                     scale_on_input: bool = True) -> None:
    """out[n, b, a] = in[n, a, b] (x| /) scale; see usf_layout_transpose."""
    global LAUNCHES
    LAUNCHES += 1
    check(_lib.load().usf_layout_transpose(_ptr(x), n, a, b, _ptr(scale), scale_mode if scale is not None else 0,
                                           int(scale_on_input), _ptr(out), _stream()))


def layout_transpose_u8(x: torch.Tensor, dq: Dequant, n: int, c: int, hw: int, out: torch.Tensor, scale=None,
                        scale_mode: int = 0) -> None:
    """8-bit NCHW images x [n, c*hw] -> dequantised channels-last fp32 out (x| /) scale; see usf_layout_transpose_u8."""
    global LAUNCHES
    LAUNCHES += 1
    s = dq.struct()
    check(_lib.load().usf_layout_transpose_u8(_ptr(x), n, c, hw, C.byref(s), _ptr(scale), scale_mode if scale is not None else 0,
                                              _ptr(out), _stream()))


def layout_transpose_to_u8(x: torch.Tensor, n: int, a: int, b: int, out: torch.Tensor, scale=None, scale_mode: int = 0) -> None:
    """Channels-last fp32 x [n, a*b] -> 8-bit NCHW out[n, b, a] (x| /) scale, quantised; see usf_layout_transpose_to_u8."""
    global LAUNCHES
    LAUNCHES += 1
    check(_lib.load().usf_layout_transpose_to_u8(_ptr(x), n, a, b, _ptr(scale), scale_mode if scale is not None else 0,
                                                 _ptr(out), _stream()))


def im2col(x: torch.Tensor, n_images: int, h: int, w: int, c: int, k: int, dilation: int, out: Act, *, mask=None,
           relu: bool = False, overflow_flag: Optional[torch.Tensor] = None) -> None:
    """Operand rows [n*h*w, k*k*c] of a k x k 'same' convolution over channels-last rows; see usf_im2col."""
    global LAUNCHES
    LAUNCHES += 1
    p = _planes_struct(out)
    check(_lib.load().usf_im2col(_ptr(x), _ld(x), n_images, h, w, c, k, dilation, _ptr(mask), int(relu), C.byref(p),
                                 _ptr(overflow_flag), _stream()))


CONV_TC_SMEM_LIMIT = 227 * 1024


def conv2d_rows_supported(N: int, K: int, c_in: int) -> bool:
    """Whether usf_conv2d_rows serves this shape (N <= 64, C % 16 == 0, whole weight resident in shared memory)."""
    bn = 32 if N <= 32 else 64
    return N <= 64 and c_in % 16 == 0 and 3 * 32768 + ((K + 31) // 32) * 2 * bn * 128 + 1280 <= CONV_TC_SMEM_LIMIT


def conv2d_rows(x: torch.Tensor, n_images: int, h: int, w: int, c: int, k: int, dilation: int, w_hi, w_lo, N: int, *,
                bias=None, relu: bool = False, out: Act, mask=None, relu_in: bool = False,
                overflow_flag: Optional[torch.Tensor] = None) -> None:
    """k x k 'same' convolution over channels-last rows as an implicit GEMM on tcgen05; see usf_conv2d_rows."""
    global LAUNCHES
    LAUNCHES += 1
    args = LinearArgs()
    args.M, args.N, args.K = n_images * h * w, N, k * k * c
    args.engine = ENGINE_TC_3XTF32
    args.w, args.w_lo, args.ldw = _ptr(w_hi), _ptr(w_lo), _ld(w_hi)
    args.bias, args.relu, args.resid_sign = _ptr(bias), int(relu), 1.0
    if out.f32 is not None:
        args.out_f32, args.ld_f32 = _ptr(out.f32), _ld(out.f32)
    if out.hi is not None:
        args.out_hi, args.out_lo, args.ld_split = _ptr(out.hi), _ptr(out.lo), _ld(out.hi)
    if out.bf16 is not None:
        args.out_bf16, args.ld_bf16 = _ptr(out.bf16), _ld(out.bf16)
    if out.h16 is not None:
        args.out_h16, args.out_l16, args.ld_16 = _ptr(out.h16), _ptr(out.l16), _ld(out.h16)
        args.overflow_flag = _ptr(overflow_flag)
    check(_lib.load().usf_conv2d_rows(C.byref(args), _ptr(x), _ld(x), n_images, h, w, c, k, dilation, _ptr(mask),
                                      int(relu_in), _stream()))


PIX_SMEM_LIMIT = 227 * 1024


def conv2d_pix_supported(h: int, w: int, k: int, gated: bool = True) -> bool:
    """Whether usf_conv2d_pix serves this image / kernel size (rows <= 256 pixels wide; the k*k*4 KB weight next to at least
    two 32 KB pipeline stages -- and the gate's operand tile -- in shared memory)."""
    fixed = k * k * 4096 + (8192 if gated else 0) + 32768 + 7168
    return w <= 256 and k % 2 == 1 and (PIX_SMEM_LIMIT - fixed) // 32768 >= 2


def pix_encode(x: torch.Tensor, hw: int, out16: torch.Tensor, *, mask=None, relu: bool = False,
               overflow_flag: Optional[torch.Tensor] = None) -> None:
    """fp32 channels-last rows [rows, c <= 32] -> pixel planes [rows, 64] fp16 (32 hi | 32 lo'); see usf_pix_encode."""
    global LAUNCHES
    LAUNCHES += 1
    rows, c = x.shape
    check(_lib.load().usf_pix_encode(_ptr(x), _ld(x), rows, c, hw, _ptr(mask), int(relu), _ptr(out16), _ptr(overflow_flag),
                                     _stream()))


def conv2d_pix(a16: torch.Tensor, n_images: int, h: int, w: int, k: int, dilation: int, w1: torch.Tensor, bias1: torch.Tensor,
               n1: int, *, relu1: bool = False, gated: bool = False, post_relu: bool = False, w2=None, bias2=None, gamma=None,
               beta=None, eps: float = 0.0, out_f32=None, out16=None, relu_planes: bool = False, x=None, inv_mask=None,
               sign: float = 1.0, overflow_flag: Optional[torch.Tensor] = None) -> None:
    """k x k 'same' convolution over pixel planes (one 4-D TMA box per tap), plain or as a whole GatedConv block; see
    usf_conv2d_pix."""
    global LAUNCHES
    LAUNCHES += 1
    a = _lib.ConvPixArgs()
    a.a16, a.n_images, a.h, a.w, a.ksize, a.dilation = _ptr(a16), n_images, h, w, k, dilation
    a.w1, a.bias1, a.n1, a.relu1 = _ptr(w1), _ptr(bias1), n1, int(relu1)
    a.gated, a.post_relu, a.w2, a.bias2 = int(gated), int(post_relu), _ptr(w2), _ptr(bias2)
    a.gamma, a.beta, a.eps, a.sign = _ptr(gamma), _ptr(beta), float(eps), float(sign)
    if out_f32 is not None:
        a.out_f32, a.ld_f32 = _ptr(out_f32), _ld(out_f32)
    a.out16, a.relu_planes = _ptr(out16), int(relu_planes)
    if x is not None:
        a.x, a.ldx, a.inv_mask, a.c_x = _ptr(x), _ld(x), _ptr(inv_mask), x.shape[1]
    a.overflow_flag = _ptr(overflow_flag)
    check(_lib.load().usf_conv2d_pix(C.byref(a), _stream()))


def masked_add(x: torch.Tensor, t: torch.Tensor, hw: int, g: torch.Tensor, sign: float) -> None:
    global LAUNCHES
    LAUNCHES += 1
    check(_lib.load().usf_masked_add(_ptr(x), _ld(x), _ptr(t), _ld(t), x.shape[0], x.shape[1], hw, _ptr(g), float(sign),
                                     _stream()))


def sub_rows(out: torch.Tensor, v: torch.Tensor) -> None:
    check(_lib.load().usf_sub_rows(_ptr(out), _ptr(v), out.numel(), _stream()))


def leaky_relu(x: torch.Tensor, slope: float, y: torch.Tensor, neg_count: Optional[torch.Tensor] = None) -> None:
    rows, d = x.shape
    check(_lib.load().usf_leaky_relu(_ptr(x), _ld(x), rows, d, float(slope), _ptr(y), _ld(y), _ptr(neg_count), _stream()))


def permute(x: torch.Tensor, perm_i32: torch.Tensor, y: torch.Tensor) -> None:
    rows, d = x.shape
    check(_lib.load().usf_permute(_ptr(x), _ld(x), rows, d, _ptr(perm_i32), _ptr(y), _ld(y), _stream()))


# ---- weight preparation --------------------------------------------------------------------------
def lu_assemble(L_raw, U_raw, L=None, U=None, transpose_u=False) -> None:
    d = (L_raw if L_raw is not None else U_raw).shape[0]
    ref = L if L is not None else U
    check(_lib.load().usf_lu_assemble(_ptr(L_raw), _ptr(U_raw), d, _ld(L_raw if L_raw is not None else U_raw),
                                      _ptr(L), _ptr(U), _ld(ref), int(transpose_u), _stream()))


def lu_logabsdet(U_raw, out2) -> None:
    check(_lib.load().usf_lu_logabsdet(_ptr(U_raw), U_raw.shape[0], _ld(U_raw), _ptr(out2), _stream()))


def vec_logabs(v, out2) -> None:
    check(_lib.load().usf_vec_logabs(_ptr(v), v.numel(), _ptr(out2), _stream()))


def tri_inverse(T, lower: bool, unit_diag: bool, X) -> None:
    d = T.shape[0]
    n = _lib.load().usf_tri_inverse_work_floats(d)
    work = torch.empty(n, dtype=torch.float32, device=T.device)
    check(_lib.load().usf_tri_inverse(_ptr(T), d, _ld(T), int(lower), int(unit_diag), _ptr(X), _ld(X), _ptr(work), _stream()))


def transpose(a, out) -> None:
    check(_lib.load().usf_transpose(_ptr(a), a.shape[0], a.shape[1], _ld(a), _ptr(out), _ld(out), _stream()))


def scale_rows_cols(a, out, rowf=None, colf=None) -> None:
    check(_lib.load().usf_scale_rows_cols(_ptr(a), a.shape[0], a.shape[1], _ld(a), _ptr(rowf), _ptr(colf), _ptr(out), _ld(out), _stream()))


def split_tf32(a, hi, lo) -> None:
    check(_lib.load().usf_split_tf32(_ptr(a), a.shape[0], a.shape[1], _ld(a), _ptr(hi), _ptr(lo), _ld(hi), _stream()))


def split_f16(a, hi, lo, overflow_flag=None) -> None:
    check(_lib.load().usf_split_f16(_ptr(a), a.shape[0], a.shape[1], _ld(a), _ptr(hi), _ptr(lo), _ld(hi),
                                    _ptr(overflow_flag), _stream()))


def to_bf16(a, out) -> None:
    check(_lib.load().usf_to_bf16(_ptr(a), a.shape[0], a.shape[1], _ld(a), _ptr(out), _ld(out), _stream()))


def householder_right(W, v, work) -> None:
    check(_lib.load().usf_householder_right(_ptr(W), W.shape[0], _ld(W), _ptr(v), _ptr(work), _stream()))


def softplus(a, out) -> None:
    check(_lib.load().usf_softplus(_ptr(a), a.numel(), _ptr(out), _stream()))


def matmul_f32(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor, bias=None) -> None:
    """out = a @ b (+ bias) in fp32 on CUDA cores (weight preparation); b is [K, N] row-major."""
    M, K = a.shape
    N = b.shape[1]
    linear(ENGINE_SIMT, Act(M, K, f32=a), b, None, N, K, bias=bias, out=Act(M, N, f32=out), trans_w=True)


def matmul_f64(a: torch.Tensor, b: torch.Tensor, out: torch.Tensor, tri: int = 0) -> None:
    """out = a @ b in fp64 (weight composition, once per weight version).  `tri`: TRI_LOWER_UPPER (a lower, b upper
    triangular) / TRI_UPPER_LOWER -- square factors stored dense; the product skips the k range where one of them is zero."""
    M, K = a.shape
    N = b.shape[1]
    assert a.dtype == b.dtype == out.dtype == torch.float64 and b.shape[0] == K and out.shape == (M, N)
    if tri:
        assert M == N == K
        check(_lib.load().usf_matmul_f64_tri(_ptr(a), _ld(a), _ptr(b), _ld(b), _ptr(out), _ld(out), M, tri, _stream()))
    else:
        check(_lib.load().usf_matmul_f64(_ptr(a), _ld(a), _ptr(b), _ld(b), _ptr(out), _ld(out), M, N, K, _stream()))


# ---- training step (see include/usflows_b200.h, "Training step") -------------------------------------------------------
def linear_splitk(engine: int, a_t: Act, w_t: Act, N: int, K: int, out: torch.Tensor, split_k: int) -> None:
    """out[M, N] (fp32) = a_t[M, K] . w_t[N, K]^T with the contraction cut into `split_k` pieces (dW = dY^T . X: a_t and w_t are
    the TRANSPOSED planes of dY and X, K = batch rows).  The library zero-fills `out`."""
    args = LinearArgs()
    args.M, args.N, args.K = a_t.rows, N, K
    args.engine = engine
    if engine == ENGINE_TC_3XF16:
        args.a, args.a_lo, args.lda = _ptr(a_t.h16), _ptr(a_t.l16), _ld(a_t.h16)
        args.w, args.w_lo, args.ldw = _ptr(w_t.h16), _ptr(w_t.l16), _ld(w_t.h16)
    else:
        raise RuntimeError("usflows_b200: linear_splitk runs on the fp16-split tcgen05 engine")
    args.resid_sign = 1.0
    args.out_f32, args.ld_f32 = _ptr(out), _ld(out)
    args.split_k = int(split_k)
    global LAUNCHES
    LAUNCHES += 1
    check(_lib.load().usf_linear(C.byref(args), _stream()))


def planes_glue(src, *, rows: int, n: int, mask_h=None, sign: float = 1.0, out: Optional[Act] = None, t: Optional[Act] = None,
                colsum=None, mul=None, colsum2=None, overflow_flag=None) -> None:
    """One pass between two contractions of the training step; `src` is an Act with fp16 split planes or an fp32 tensor."""
    from ._lib import GlueArgs
    g = GlueArgs()
    if isinstance(src, Act):
        g.h, g.l, g.ld = _ptr(src.h16), _ptr(src.l16), _ld(src.h16)
    else:
        g.src_f32, g.ld_src = _ptr(src), _ld(src)
    g.rows, g.n, g.sign = rows, n, float(sign)
    if mask_h is not None:
        g.mask_h, g.ld_mask = _ptr(mask_h), _ld(mask_h)
    if out is not None:
        g.out_h, g.out_l, g.ld_out = _ptr(out.h16), _ptr(out.l16), _ld(out.h16)
    if t is not None:
        g.t_h, g.t_l, g.ld_t = _ptr(t.h16), _ptr(t.l16), _ld(t.h16)
    g.colsum = _ptr(colsum)
    if colsum2 is not None:
        g.mul, g.ld_mul, g.colsum2 = _ptr(mul), _ld(mul), _ptr(colsum2)
    g.overflow_flag = _ptr(overflow_flag)
    global LAUNCHES
    LAUNCHES += 1
    check(_lib.load().usf_planes_glue(C.byref(g), _stream()))


def base_backward(z: torch.Tensor, loc, scale, kind: int, g: Act, t: Optional[Act], dloc, dscale) -> None:
    """d(-log p)/dz of the Laplace / Normal base as planes (+ transposed planes) and the column sums for loc / scale."""
    global LAUNCHES
    LAUNCHES += 1
    rows, d = z.shape
    check(_lib.load().usf_base_backward(_ptr(z), _ld(z), rows, d, _ptr(loc), _ptr(scale), kind, _ptr(g.h16), _ptr(g.l16),
                                        _ld(g.h16), _ptr(t.h16) if t is not None else None,
                                        _ptr(t.l16) if t is not None else None, _ld(t.h16) if t is not None else 0,
                                        _ptr(dloc), _ptr(dscale), _stream()))


def mat_prep(src: torch.Tensor, *, transpose: bool = False, row_idx=None, col_idx=None, scale: float = 1.0,
             out_f32: Optional[torch.Tensor] = None, out: Optional[Act] = None, out_t: Optional[Act] = None,
             overflow_flag=None) -> None:
    """Weight-side copy / transpose / gather / split of an fp32 matrix; the output shape decides rows x cols (`out_t`
    receives the transposed planes [cols, rows] of the same result)."""
    if out_f32 is not None:
        rows, cols = out_f32.shape
    elif out is not None:
        rows, cols = out.h16.shape
    else:
        cols, rows = out_t.h16.shape
    global LAUNCHES
    LAUNCHES += 1
    check(_lib.load().usf_mat_prep(_ptr(src), _ld(src), rows, cols, int(transpose), _ptr(row_idx), _ptr(col_idx), float(scale),
                                   _ptr(out_f32), _ld(out_f32) if out_f32 is not None else 0,
                                   _ptr(out.h16) if out is not None else None, _ptr(out.l16) if out is not None else None,
                                   _ld(out.h16) if out is not None else 0,
                                   _ptr(out_t.h16) if out_t is not None else None, _ptr(out_t.l16) if out_t is not None else None,
                                   _ld(out_t.h16) if out_t is not None else 0, _ptr(overflow_flag), _stream()))


def rowdot(W: torch.Tensor, v: torch.Tensor, alpha: float, out: torch.Tensor, row_idx=None) -> None:
    """out[i] = alpha * W[row_idx[i] or i, :] . v"""
    check(_lib.load().usf_rowdot(_ptr(W), _ld(W), out.numel(), W.shape[1], _ptr(row_idx), _ptr(v), float(alpha), _ptr(out),
                                 _stream()))


def colcomb(W: torch.Tensor, v: torch.Tensor, alpha: float, out: torch.Tensor) -> None:
    """out[j] += alpha * sum_i v[i] W[i, j]"""
    check(_lib.load().usf_colcomb(_ptr(W), _ld(W), W.shape[0], W.shape[1], _ptr(v), float(alpha), _ptr(out), _stream()))


def rank1(A: torch.Tensor, u: torch.Tensor, v: torch.Tensor, alpha: float) -> None:
    """A[i, j] += alpha * u[i] v[j]"""
    check(_lib.load().usf_rank1(_ptr(A), _ld(A), A.shape[0], A.shape[1], _ptr(u), _ptr(v), float(alpha), _stream()))


def tri_mask(src: torch.Tensor, mode: int, scale: float, out: torch.Tensor, diag_src=None, coef: float = 0.0) -> None:
    d = src.shape[0]
    check(_lib.load().usf_tri_mask(_ptr(src), _ld(src), d, mode, float(scale), _ptr(diag_src),
                                   _ld(diag_src) if diag_src is not None else 0, float(coef), _ptr(out), _ld(out), _stream()))


def tri_inverse_batched(T: torch.Tensor, X: torch.Tensor, tmp: torch.Tensor, unit_mask: int) -> None:
    """Inverses of the lower-triangular matrices T[m] (stack [n_mats, d, d], contiguous) into X[m]."""
    n_mats, d, _ = T.shape
    check(_lib.load().usf_tri_inverse_batched(_ptr(T), _ptr(X), _ptr(tmp), d, T.stride(1), T.stride(0), n_mats,
                                              unit_mask & 0xFFFFFFFF, _stream()))
