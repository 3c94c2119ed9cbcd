"""Execution of flows over image-shaped events (`in_dims = [C, H, W]`): the reference's 1x1-convolution mode of
`BlockAffineTransform` (transforms.py:904-962), `MaskedCoupling` with masks over [C, H, W] (flows.py:494-536) and
`networks.ConvNet2D` conditioners (networks.py:405-510), `ScaleTransform` over [C, H, W] (transforms.py:105-125).

Inside the layer stack a batch lives channels-last as a row matrix [N*H*W, C] (csrc/image.cuh):
  BlockAffineTransform    -> usf_linear over N*H*W rows with the C x C matrix (the same contraction as the flat case)
  k x k convolution       -> usf_im2col (zero padding 'same'; fused with the coupling's `x * mask` and the ReLU in front
                             of the convolution) + usf_linear with K = k*k*C_in
  1 x 1 convolution       -> usf_linear (bias / ReLU in the epilogue)
  gate, ReLU, LayerNormChannels -> usf_gate_norm (one pass over the row)
  x +- (1 - mask) * t     -> usf_masked_add
  ScaleTransform and the NCHW <-> channels-last conversion -> usf_layout_transpose at the two ends of a pass
  base density            -> the flat kernels on the same memory viewed as [N, H*W*C], loc / scale permuted once.
The stream is kept in fp32; every contraction reads operand planes of the engine `engine._engine_for` picks for its
shape (tcgen05 split engines for widths >= 32, the SIMT engine below that -- e.g. the 16-channel MNIST squeeze).
"""
from __future__ import annotations

import math
from typing import List, Optional

import torch

from . import engine, ops
from .engine import Prim, _engine_for, _operand, _workspace
from .ops import Act, ENGINE_TC_3XF16, ENGINE_TC_3XTF32
IMPLICIT_CONV = True                # k x k convolutions as implicit GEMMs (usf_conv2d_rows) where the shape allows it
PIX_CONV = True                     # ... and the whole ConvNet2D on pixel planes (usf_conv2d_pix) where its widths allow it
PIX_CH = 32                         # channels of a pixel-plane row
PIX_MODES = ("fp32", "tf32", "bf16")  # the reduced-precision modes take the pixel-plane route too: it is fp32-accurate AND
                                    # 3x faster than their own gather / implicit-GEMM routes (0.40-0.48 M images/s)
IMAGE_CHUNK_ROWS = 1 << 19          # channels-last rows (N*H*W) per chunk: bounds the im2col workspace (rows x k*k*C)
IMAGE_CHUNK_ROWS_PIX = 1 << 21      # ... when every conditioner runs on pixel planes (~0.6 KB of workspace per row): fewer,
                                    # longer launches win over L2 residency (tools/img_chunk_probe.py: 16 384 images as
                                    # 2^17 / 2^18 / 2^19 / 2^20-row chunks 16.9 / 15.2 / 13.1 / 12.3 ms)


def _act(dev, name: str, rows: int, width: int, eng: int) -> Act:
    a = Act(rows, width)
    for pl in ops.ENGINE_PLANES[eng]:
        setattr(a, pl, _workspace.planes(dev, name, rows, width, pl))
    return a


def _dense(dev, name: str, rows: int, width: int) -> torch.Tensor:
    """Dense fp32 [rows, width] workspace (no row padding: the layout kernel writes whole images contiguously)."""
    return _workspace.planes(dev, name, 1, rows * width, "f32").view(rows, width)


class _Gemm:
    """One contraction out = A . W^T + b with its weight in the operand format of the engine chosen for its shape."""

    def __init__(self, mode: str, w: torch.Tensor, b: Optional[torch.Tensor], wflag, pad_n: bool = False,
                 conv_cin: int = 0):
        self.n_true = w.shape[0]
        if pad_n and mode != "fp32_simt" and w.shape[0] < engine.TC_MIN_DIM <= w.shape[1]:
            # a narrow output (the c_in channels of the conditioner's last convolution) would fall to the SIMT engine:
            # zero rows up to the tensor-core minimum width cost nothing there (the caller reads the first n_true columns)
            extra = engine.TC_MIN_DIM - w.shape[0]
            w = torch.cat([w, torch.zeros(extra, w.shape[1], dtype=w.dtype, device=w.device)])
            if b is not None:
                b = torch.cat([b, torch.zeros(extra, dtype=b.dtype, device=b.device)])
        self.N, self.K = w.shape
        self.engine = _engine_for(mode, self.N, self.K)
        self.w, self.w_lo = _operand(w, mode, self.engine, wflag if self.engine == ENGINE_TC_3XF16 else None)
        self.bias = None if b is None else b.to(torch.float32).contiguous()
        # implicit-GEMM convolution: tf32 hi / lo planes of the same weight (the kernel computes in the 3-term tf32 split)
        self.conv_w = None
        if conv_cin and IMPLICIT_CONV and mode in ("fp32", "fp32_tf32") and ops.conv2d_rows_supported(self.N, self.K, conv_cin):
            self.conv_w = _operand(w, "fp32_tf32", ENGINE_TC_3XTF32)

    def __call__(self, a: Act, out: Act, relu: bool = False, flag=None) -> None:
        ops.linear(self.engine, a, self.w, self.w_lo, self.N, self.K, bias=self.bias, relu=relu, out=out,
                   overflow_flag=flag)


def _pix_weight(w: torch.Tensor, taps: int, cin: int, n_pad: int, wflag) -> torch.Tensor:
    """Contraction weight [N, taps * cin] (usf_im2col column order) -> [n_pad, taps * 64] fp16 for usf_conv2d_pix: per tap
    32 high halves | 32 low halves' of the input channels, channels >= cin and rows >= N zero."""
    n = w.shape[0]
    w3 = torch.zeros(n_pad, taps, PIX_CH, dtype=torch.float32, device=w.device)
    w3[:n, :, :cin] = w.to(torch.float32).reshape(n, taps, cin)
    hi, lo = _operand(w3.reshape(n_pad, taps * PIX_CH), "fp32", ENGINE_TC_3XF16, wflag)
    return torch.cat([hi.reshape(n_pad, taps, PIX_CH), lo.reshape(n_pad, taps, PIX_CH)], dim=2).reshape(n_pad, taps * 64).contiguous()


def _pad_vec(b: torch.Tensor, n: int) -> torch.Tensor:
    out = torch.zeros(n, dtype=torch.float32, device=b.device)
    out[:b.shape[0]] = b.to(torch.float32)
    return out


def _conv_weight(conv) -> torch.Tensor:
    """nn.Conv2d weight [C_out, C_in, kh, kw] -> contraction weight [C_out, (kh, kw, C_in)] (the usf_im2col column order)."""
    w = conv.weight.detach()
    return w.permute(0, 2, 3, 1).reshape(w.shape[0], -1).contiguous()


class _ConvNet2DPlan:
    """Launch plan of a ConvNet2D (networks.py:405-510) over channels-last rows."""

    def __init__(self, net, mode: str, wflag, H: int, W: int):
        d = net._describe()
        for prm in net.parameters():
            ops.require_cuda(prm, "conditioner parameter")
        self.k, self.dil, self.H, self.W = d["k"], d["dilation"], H, W
        self.c_in = d["first"].weight.shape[1]
        kk = self.k * self.k
        cin = lambda conv: conv.weight.shape[1] if kk > 1 else 0      # noqa: E731  (1x1 convolutions are plain contractions)
        self.first = _Gemm(mode, _conv_weight(d["first"]), d["first"].bias.detach(), wflag, conv_cin=cin(d["first"]))
        self.blocks = []
        for b in d["blocks"]:
            ln = None if b["ln"] is None else (b["ln"].gamma.detach().reshape(-1).contiguous(),
                                               b["ln"].beta.detach().reshape(-1).contiguous(), float(b["ln"].eps))
            g1 = _Gemm(mode, _conv_weight(b["conv1"]), b["conv1"].bias.detach(), wflag, conv_cin=cin(b["conv1"]))
            g2 = None if not b["gated"] else _Gemm(mode, _conv_weight(b["conv2"]), b["conv2"].bias.detach(), wflag)
            gp = None if b.get("proj") is None else _Gemm(mode, _conv_weight(b["proj"]), b["proj"].bias.detach(), wflag)
            self.blocks.append((b["gated"], g1, g2, ln, gp))
        self.last = _Gemm(mode, _conv_weight(d["last"]), d["last"].bias.detach(), wflag, pad_n=True, conv_cin=cin(d["last"]))
        self.gemms = [self.first, self.last] + [g for b in self.blocks for g in (b[1], b[2], b[4]) if g is not None]
        self.pix = None
        if self._pix_ok(mode, d, H, W):
            self._prepare_pix(d, wflag)

    # ---- the whole network on pixel planes (usf_conv2d_pix): 2 + num_layers launches + usf_pix_encode -------------------
    def _pix_ok(self, mode: str, d: dict, H: int, W: int) -> bool:
        if not (PIX_CONV and IMPLICIT_CONV and mode in PIX_MODES and self.k > 1):
            return False
        gated_any = any(b["gated"] for b in d["blocks"])
        if not ops.conv2d_pix_supported(H, W, self.k, gated_any):
            return False
        widths = [d["first"].weight.shape[1] <= PIX_CH, d["first"].weight.shape[0] == PIX_CH,
                  d["last"].weight.shape[1] == PIX_CH, d["last"].weight.shape[0] <= PIX_CH, d["last"].weight.shape[0] % 4 == 0]
        for b in d["blocks"]:
            widths += [tuple(b["conv1"].weight.shape[:2]) == (PIX_CH, PIX_CH), b.get("proj") is None]
            if b["gated"]:
                widths += [tuple(b["conv2"].weight.shape[:2]) == (2 * PIX_CH, PIX_CH)]
        return all(widths)

    def _prepare_pix(self, d: dict, wflag) -> None:
        taps = self.k * self.k
        pw = lambda conv, n_pad, t: _pix_weight(_conv_weight(conv), t, conv.weight.shape[1], n_pad, wflag)   # noqa: E731
        blocks = []
        for b in d["blocks"]:
            ln = None if b["ln"] is None else (b["ln"].gamma.detach().reshape(-1).float().contiguous(),
                                               b["ln"].beta.detach().reshape(-1).float().contiguous(), float(b["ln"].eps))
            blk = dict(gated=b["gated"], w1=pw(b["conv1"], PIX_CH, taps), b1=_pad_vec(b["conv1"].bias.detach(), PIX_CH), ln=ln)
            if b["gated"]:
                blk.update(w2=pw(b["conv2"], 2 * PIX_CH, 1), b2=_pad_vec(b["conv2"].bias.detach(), 2 * PIX_CH))
            blocks.append(blk)
        self.pix = dict(first=(pw(d["first"], PIX_CH, taps), _pad_vec(d["first"].bias.detach(), PIX_CH)), blocks=blocks,
                        last=(pw(d["last"], PIX_CH, taps), _pad_vec(d["last"].bias.detach(), PIX_CH)),
                        n_out=d["last"].weight.shape[0])

    def run_pix(self, x_rows: torch.Tensor, n_images: int, mask_cl, flag, *, update=None) -> Optional[torch.Tensor]:
        """t = net(x * mask) on pixel planes.  `update` = (x, inv_mask, sign): the last convolution applies the coupling
        update x += sign * (1 - mask) * t itself and nothing is returned; else t comes back as fp32 rows [n*H*W, c_out]."""
        dev, rows = x_rows.device, x_rows.shape[0]
        H, W, k, dil, px = self.H, self.W, self.k, self.dil, self.pix
        bufs = [_workspace.planes(dev, "pix_a", rows, 64, "pix"), _workspace.planes(dev, "pix_b", rows, 64, "pix")]
        y = _workspace.planes(dev, "img_y", rows, PIX_CH, "f32")
        blocks = px["blocks"]
        relu_for = lambda i: i < len(blocks) and blocks[i]["gated"]     # noqa: E731  (GatedConv starts with a ReLU)
        ops.pix_encode(x_rows, H * W, bufs[0], mask=mask_cl, overflow_flag=flag)
        cur = 0
        ops.conv2d_pix(bufs[cur], n_images, H, W, k, dil, px["first"][0], px["first"][1], PIX_CH, out_f32=y,
                       out16=bufs[cur ^ 1], relu_planes=relu_for(0), overflow_flag=flag)
        cur ^= 1
        for i, b in enumerate(blocks):
            gamma, beta, eps = b["ln"] if b["ln"] is not None else (None, None, 0.0)
            if b["gated"]:      # GatedConv (networks.py:100-121) -> ReLU -> LayerNormChannels: one launch
                ops.conv2d_pix(bufs[cur], n_images, H, W, k, dil, b["w1"], b["b1"], PIX_CH, gated=True, post_relu=True,
                               w2=b["w2"], bias2=b["b2"], gamma=gamma, beta=beta, eps=eps, out_f32=y, out16=bufs[cur ^ 1],
                               relu_planes=relu_for(i + 1), overflow_flag=flag)
            else:               # Conv k x k -> ReLU -> LayerNormChannels
                ops.conv2d_pix(bufs[cur], n_images, H, W, k, dil, b["w1"], b["b1"], PIX_CH, relu1=True, gamma=gamma, beta=beta,
                               eps=eps, out_f32=y, out16=bufs[cur ^ 1], relu_planes=relu_for(i + 1), overflow_flag=flag)
            cur ^= 1
        if update is not None:
            xs, inv_mask, sign = update
            ops.conv2d_pix(bufs[cur], n_images, H, W, k, dil, px["last"][0], px["last"][1], px["n_out"], x=xs,
                           inv_mask=inv_mask, sign=sign, overflow_flag=flag)
            return None
        t = _workspace.planes(dev, "img_t", rows, px["n_out"], "f32")
        ops.conv2d_pix(bufs[cur], n_images, H, W, k, dil, px["last"][0], px["last"][1], px["n_out"], out_f32=t,
                       overflow_flag=flag)
        return t

    def run(self, x_rows: torch.Tensor, n_images: int, mask_cl: Optional[torch.Tensor], flag) -> torch.Tensor:
        """t = net(x * mask) as fp32 rows [n*H*W, c_out] (a workspace buffer)."""
        if self.pix is not None:
            return self.run_pix(x_rows, n_images, mask_cl, flag)
        dev, rows = x_rows.device, x_rows.shape[0]
        H, W, k, dil = self.H, self.W, self.k, self.dil

        def conv(src: torch.Tensor, c: int, g: _Gemm, out: Act, *, mask=None, relu_in=False, relu_out=False):
            if g.conv_w is not None and src.stride(0) % 4 == 0:        # no gathered copy in memory: implicit GEMM
                ops.conv2d_rows(src, n_images, H, W, c, k, dil, g.conv_w[0], g.conv_w[1], g.N, bias=g.bias, relu=relu_out,
                                out=out, mask=mask, relu_in=relu_in, overflow_flag=flag)
                return
            if k == 1:
                cols = _act(dev, "img_cols", rows, c, g.engine)
                ops.im2col(src, n_images, H, W, c, 1, 1, cols, mask=mask, relu=relu_in, overflow_flag=flag)
            else:
                cols = _act(dev, "img_cols", rows, k * k * c, g.engine)
                ops.im2col(src, n_images, H, W, c, k, dil, cols, mask=mask, relu=relu_in, overflow_flag=flag)
            g(cols, out, relu=relu_out, flag=flag)

        f32 = lambda name, width: Act(rows, width, f32=_workspace.planes(dev, name, rows, width, "f32"))   # noqa: E731
        y = f32("img_y", self.first.N)                       # residual stream of the conditioner
        conv(x_rows, self.c_in, self.first, y, mask=mask_cl)
        for gated, g1, g2, ln, gp in self.blocks:
            gamma, beta, eps = ln if ln is not None else (None, None, 0.0)
            if gated:                                        # GatedConv (networks.py:100-121) -> ReLU -> LayerNormChannels
                hid = _act(dev, "img_h", rows, g1.N, g2.engine)
                conv(y.f32, g1.K // (k * k), g1, hid, relu_in=True, relu_out=True)
                vg = f32("img_st", g2.N)
                g2(hid, vg, flag=flag)
                n = g2.n_true // 2                           # block width: c_in of a GatedConv, c_out of a GatedConvND
                if gp is not None:                           # GatedConvND whose width changes: residual = proj(x), a 1x1
                    cols = _act(dev, "img_cols", rows, gp.K, gp.engine)            # convolution (networks.py:186-201)
                    ops.im2col(y.f32, n_images, H, W, gp.K, 1, 1, cols, overflow_flag=flag)
                    res = f32("img_r", gp.N)
                    gp(cols, res, flag=flag)
                    y = f32("img_y", n)                      # the old residual stream has been consumed (conv1, proj)
                    ops.gate_norm(vg.f32, n, xres=res.f32, gated=True, pre_relu=True, gamma=gamma, beta=beta, eps=eps,
                                  y_f32=y.f32)
                    continue
                ops.gate_norm(vg.f32, n, xres=y.f32, gated=True, pre_relu=True, gamma=gamma, beta=beta,
                              eps=eps, y_f32=y.f32)
            else:                                            # Conv k x k -> ReLU -> LayerNormChannels
                o = f32("img_st", g1.N)
                conv(y.f32, g1.K // (k * k), g1, o)
                y2 = f32("img_y", g1.N)
                ops.gate_norm(o.f32, g1.N, gated=False, pre_relu=True, gamma=gamma, beta=beta, eps=eps, y_f32=y2.f32)
                y = y2
        t = f32("img_t", self.last.N)
        conv(y.f32, self.last.K // (k * k), self.last, t)
        return t.f32[:, :self.last.n_true]


class ImageProgram(engine.ProgramCore):
    """Launch program of one direction of a layer stack over image-shaped events, for one mode and weight version."""

    small = None
    has_row_ladj = False
    fp16_weight_modes = PIX_MODES      # the pixel-plane conditioners take fp16 split weights in these modes

    def __init__(self, layers, direction: str, mode: Optional[str], in_dims):
        self.C, self.H, self.W = (int(v) for v in in_dims)
        self.HW = self.H * self.W
        super().__init__(layers, direction, mode)

    def _in_mode(self, mode: str) -> "ImageProgram":
        return ImageProgram(self.layers, self.direction, mode, (self.C, self.H, self.W))

    def _build(self, prims: List[Prim]) -> None:
        self.entry_scale = self.exit_scale = None            # (vector in NCHW order, mode 1 = multiply / 2 = divide)
        if prims and prims[0].kind in ("mul", "div"):
            self.entry_scale = (prims[0].v.contiguous(), 1 if prims[0].kind == "mul" else 2)
            prims = prims[1:]
        if prims and prims[-1].kind in ("mul", "div"):
            self.exit_scale = (prims[-1].v.contiguous(), 1 if prims[-1].kind == "mul" else 2)
            prims = prims[:-1]
        if engine.MERGE_AFFINE:                              # consecutive 1x1 convolutions (the inverse of one block's affine
            merged: List[Prim] = []                          # conjugation, the next block's) are ONE C x C map, composed in fp64
            for p in prims:
                if p.kind == "aff" and merged and merged[-1].kind == "aff":
                    merged[-1] = engine._compose_run([merged[-1], p])
                else:
                    merged.append(p)
            prims = merged
        self.ops = []
        for p in prims:
            if p.kind == "aff":                              # 1x1 convolution with the C x C matrix (transforms.py:904-962)
                dev = p.W.device
                self.ops.append(("aff", _Gemm(self.mode, p.W, p.c, self._weight_flag(dev))))
            elif p.kind == "coupling" and p.prep.get("net") == "convnet2d":
                dev = p.prep["mask"].device
                m = p.prep["mask"].reshape(self.C, self.HW).t().contiguous()          # channels-last order
                plan = _ConvNet2DPlan(p.prep["module"], self.mode, self._weight_flag(dev), self.H, self.W)
                self.ops.append(("coupling", plan, m.reshape(-1), (1 - m).reshape(-1).contiguous(), p.sign))
            else:
                raise NotImplementedError(f"usflows_b200: no image-shaped kernel path for a '{p.kind}' step here "
                                          "(ScaleTransform is supported at either end of the stack)")
        # fp16 split planes are in play (fp32 mode everywhere; tf32 / bf16 modes inside pixel-plane conditioners): chunks carry
        # a device flag and are re-run on the tf32-split program when a value leaves the fp16 range
        self.uses_range_flag = self.mode == "fp32" or (self.mode in PIX_MODES and any(
            op[0] == "coupling" and op[1].pix is not None for op in self.ops))

    def out_width(self, d_in: int) -> int:
        if d_in != self.C * self.HW:
            raise RuntimeError("usflows_b200: event shape mismatch")
        return d_in

    def plan_able(self) -> bool:                             # the whole-stack C entry covers flat events only
        return False

    def final_buffer(self, device, name: str, rows: int, d_in: int) -> torch.Tensor:
        """The workspace buffer [rows, d_in] a channels-last chunk result is written to when it is handed on."""
        return _dense(device, "img_" + name, rows, d_in)

    # ----------------------------------------------------------------------------------------------
    def _run_chunk(self, x: torch.Tensor, out: torch.Tensor, flag, dq: Optional[ops.Dequant] = None, *,
                   nchw_out: bool = False, quantize: bool = False) -> None:
        """x [n, C*H*W] (NCHW, read-only) -> out [n, C*H*W]: channels-last ([n, H*W*C]), or NCHW when `nchw_out`.  With
        `dq`, x is uint8 and the NCHW -> channels-last conversion dequantises it.  With `quantize` (NCHW only), out is uint8
        and the channels-last -> NCHW conversion writes the quantised pixels (ops.quantize)."""
        dev, n = x.device, x.shape[0]
        rows, C, HW = n * self.HW, self.C, self.HW
        nchw_out = nchw_out or quantize
        direct = not nchw_out and self.exit_scale is None    # the channels-last stream itself is the result
        bufs = [_dense(dev, "img_x0", rows, C), _dense(dev, "img_x1", rows, C)]
        which, cur = 0, bufs[0]
        es = self.entry_scale
        if dq is not None:
            ops.layout_transpose_u8(x, dq, n, C, HW, cur, scale=None if es is None else es[0], scale_mode=0 if es is None else es[1])
        else:
            ops.layout_transpose(x, n, C, HW, cur, scale=None if es is None else es[0], scale_mode=0 if es is None else es[1],
                                 scale_on_input=True)
        for idx, op in enumerate(self.ops):
            if op[0] == "aff":
                g = op[1]
                a = Act(rows, C, f32=cur)
                if ops.ENGINE_PLANES[g.engine] != ("f32",):      # tensor-core engine: re-encode the fp32 stream into its planes
                    a = _act(dev, "img_a", rows, C, g.engine)
                    ops.ingest(cur, a, overflow_flag=flag)
                if direct and idx == len(self.ops) - 1:
                    dst = out.view(rows, C)
                else:
                    which ^= 1
                    dst = bufs[which]
                g(a, Act(rows, C, f32=dst), flag=flag)
                cur = dst
            else:
                _, plan, mask_cl, inv_cl, sign = op
                if plan.pix is not None and plan.pix["n_out"] == C:     # the last convolution updates x itself
                    plan.run_pix(cur, n, mask_cl, flag, update=(cur, inv_cl, sign))
                else:
                    t = plan.run(cur, n, mask_cl, flag)
                    ops.masked_add(cur, t, HW, inv_cl, sign)
        if direct:
            if cur.data_ptr() != out.data_ptr():
                out.view(rows, C).copy_(cur)
            return
        xs = self.exit_scale
        if quantize:
            ops.layout_transpose_to_u8(cur, n, HW, C, out, scale=None if xs is None else xs[0], scale_mode=0 if xs is None else xs[1])
        elif nchw_out:
            ops.layout_transpose(cur, n, HW, C, out, scale=None if xs is None else xs[0], scale_mode=0 if xs is None else xs[1],
                                 scale_on_input=False)
        else:                                                # channels-last result with a trailing scale: two conversions
            tmp = _dense(dev, "img_tmp", n, C * HW)
            ops.layout_transpose(cur, n, HW, C, tmp, scale=xs[0], scale_mode=xs[1], scale_on_input=False)
            ops.layout_transpose(tmp, n, C, HW, out)

    def _chunk_bounds(self, rows: int, chunk_rows: Optional[int]):
        """Whole images, IMAGE_CHUNK_ROWS* channels-last rows per chunk."""
        all_pix = all(op[0] != "coupling" or op[1].pix is not None for op in self.ops)
        per = max(1, (chunk_rows or (IMAGE_CHUNK_ROWS_PIX if all_pix else IMAGE_CHUNK_ROWS)) // self.HW)
        return [(r0, min(rows, r0 + per)) for r0 in range(0, rows, per)]

    def _chunk(self, x, out, flag, dq, ladj_rows, to_caller: bool) -> None:
        self._run_chunk(x, out, flag, dq, nchw_out=to_caller)      # the caller's output is NCHW, a sink's channels-last


def channels_last_index(C: int, HW: int, device) -> torch.Tensor:
    """perm with flat_channels_last[j] = flat_nchw[perm[j]]."""
    return torch.arange(C * HW, device=device).reshape(C, HW).t().reshape(-1)


def run_convnet2d(net, x: torch.Tensor, mode: Optional[str] = None) -> torch.Tensor:
    """Plain evaluation of a `nn.ConvNet2D` on x [N, C, H, W] through the kernels a coupling uses."""
    ops.require_cuda(x, "input")
    N, C, H, W = x.shape
    mode = mode or engine.get_precision()
    with torch.no_grad():
        plan = _ConvNet2DPlan(net, mode, None, H, W)
        rows = N * H * W
        cur = torch.empty(rows, C, dtype=torch.float32, device=x.device)
        if N == 0:
            return torch.empty(0, plan.last.n_true, H, W, dtype=torch.float32, device=x.device)
        ops.layout_transpose(x.contiguous(), N, C, H * W, cur)
        t = plan.run(cur, N, None, None)
        out = torch.empty(N, t.shape[1], H, W, dtype=torch.float32, device=x.device)
        ops.layout_transpose(t.contiguous() if t.stride(0) != t.shape[1] else t, N, H * W, t.shape[1], out)
    return out
