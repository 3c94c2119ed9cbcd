"""Host-side execution engine: compiles a stack of transform layers into a launch program of fused
kernels and runs it chunk by chunk over the batch rows.

  data -> latent ("backward", `Flow.log_prob`, reference flows.py:225-245) and
  latent -> data ("forward", `Flow.sample` / `_forward`, flows.py:247-265, 45-55).

Planning folds every per-feature vector op into a neighbouring kernel:
  ScaleTransform.backward + the first affine layer's `y - b`  -> the ingest kernel
  `y - b` of later affine layers                              -> `postsub` of the producing contraction
  ScaleTransform.forward                                      -> `colscale` of the last contraction
  bias / ReLU / coupling mask / residual add-sub              -> contraction epilogue
so a USFlow evaluation is one ingest, 5B+1 contractions and (for log_prob) one base-density reduction.

Precision modes (`set_precision`, or `Flow(precision=...)`):
  "fp32"       fp32-level accuracy on tensor cores (default): tcgen05 kind::f16 on fp16 split planes
               (x = hi + lo' 2^-11, 3 products); a chunk whose activations leave the fp16 range (|x| > 65000,
               reported by a device flag) is re-run with "fp32_tf32"
  "fp32_tf32"  tcgen05 kind::tf32 with the 3-term tf32 split -- fp32-level accuracy at half the rate of "fp32"
  "fp32_simt"  CUDA-core FFMA contraction (cross-check engine; also used for tiny / unaligned layers)
  "tf32"       tcgen05 kind::tf32 single pass
  "bf16"       tcgen05 kind::f16 with bf16 operands, fp32 accumulate and fp32 residual stream
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import List, Optional, Tuple

import torch

from . import ops
from .ops import Act, ENGINE_SIMT, ENGINE_TC_3XF16, ENGINE_TC_3XTF32, ENGINE_TC_BF16, ENGINE_TC_TF32, pad4

PRECISIONS = ("fp32", "fp32_tf32", "fp32_simt", "tf32", "bf16")
_default_precision = "fp32"
_default_chunk_rows = 65536
TC_MIN_DIM = 32          # contractions narrower than this run on the SIMT engine
MERGE_AFFINE = False     # compose NEIGHBOURING dense affine layers (Aff_i^-1 . Aff_{i+1}) into one operator.  Off by
                         # default: the merged matrix is rounded as a whole, and its rounding error is amplified by
                         # the condition numbers of BOTH layers (the chained form only by one) -- measured 3-4x
                         # further from the fp64 evaluation than the reference on the ill-conditioned fixtures
COMPRESS_MASK = True     # run couplings on contiguous column halves when the mask allows it
FUSE_SMALL = True        # d <= 8 and conditioner width <= 64: the whole layer stack in ONE launch (usf_flow_small)


def set_precision(mode: str) -> None:
    global _default_precision
    if mode not in PRECISIONS:
        raise ValueError(f"unknown precision {mode!r}; choose from {PRECISIONS}")
    _default_precision = mode


def get_precision() -> str:
    return _default_precision


def set_chunk_rows(rows: int) -> None:
    global _default_chunk_rows
    _default_chunk_rows = int(rows)


def chunk_bounds(rows: int, cap: int) -> List[Tuple[int, int]]:
    """(r0, r1) of each chunk of a `rows`-row batch: ceil(rows / cap) near-equal chunks, each rounded up to whole 256-row
    tiles (the last chunk takes the rest)."""
    if rows <= 0:
        return []
    n_chunks = (rows + cap - 1) // cap
    chunk = min(rows, ((rows + n_chunks - 1) // n_chunks + 255) // 256 * 256)
    return [(r0, min(rows, r0 + chunk)) for r0 in range(0, rows, chunk)]


def run_chunks(bounds, device, guarded: bool, first, again, shared_flags=(), ladj_rows=None) -> None:
    """first(i, r0, r1, flag) for every chunk (r0, r1) of `bounds`, in order.  `guarded`: the program runs on fp16 split
    planes, so every chunk gets its own int32 range flag (else `flag` is None); after ONE device->host read, again(i, r0, r1)
    recomputes each chunk whose flag is set, in order, with the tf32-split program (same accuracy class, no range limit).
    Every chunk is recomputed when one of `shared_flags` (the flag of a captured graph replayed for several chunks) is set.
    `ladj_rows[r0:r1]` (per-row log-determinants the abandoned pass has already added to) is zeroed before again(i, r0, r1)."""
    if not guarded:
        for i, (r0, r1) in enumerate(bounds):
            first(i, r0, r1, None)
        return
    flags = torch.zeros(len(bounds), dtype=torch.int32, device=device)
    for i, (r0, r1) in enumerate(bounds):
        first(i, r0, r1, flags[i:i + 1])
    redo = torch.nonzero(torch.cat([flags, *shared_flags]) if shared_flags else flags).reshape(-1).tolist()
    if redo and redo[-1] >= len(bounds):
        redo = range(len(bounds))
    for i in redo:
        r0, r1 = bounds[i]
        if ladj_rows is not None:
            ladj_rows[r0:r1].zero_()
        again(i, r0, r1)


# --------------------------------------------------------------------------------------------------
# lowering: layers -> primitive ops -> composed affine runs -> launch steps
# --------------------------------------------------------------------------------------------------
def _engine_for(mode: str, N: int, K: int) -> int:
    if mode == "fp32_simt" or min(N, K) < TC_MIN_DIM:
        return ENGINE_SIMT
    return {"fp32": ENGINE_TC_3XF16, "fp32_tf32": ENGINE_TC_3XTF32, "tf32": ENGINE_TC_TF32, "bf16": ENGINE_TC_BF16}[mode]


def _planes(mode: str) -> tuple:
    """The operand planes of a mode: those of the engine its contractions of tensor-core width run on."""
    return ops.ENGINE_PLANES[_engine_for(mode, TC_MIN_DIM, TC_MIN_DIM)]


@dataclass
class Prim:
    """One primitive op of the lowered layer stack (direction already applied)."""
    kind: str                                   # "aff" | "mul" | "div" | "perm" | "coupling" | "leaky"
    W: Optional[torch.Tensor] = None            # aff: fp64 [dout, din]
    c: Optional[torch.Tensor] = None            # aff: fp64 [dout] (y = x W^T + c)
    v: Optional[torch.Tensor] = None            # mul / div: fp32 [d] ; perm: int64 [d]
    prep: Optional[dict] = None                 # coupling: raw conditioner weights / biases / mask
    sign: float = 1.0
    slope: float = 1.0


def _lower_layer(layer, direction: str, out: List[Prim]) -> None:
    from . import transforms as T
    fwd = direction == "forward"
    if isinstance(layer, T.InverseTransform):
        _lower_layer(layer.transform, "backward" if fwd else "forward", out)
        return
    if isinstance(layer, T.BlockAffineTransform):
        layer = layer.block_transform
    if isinstance(layer, (T.AffineTransform, T.Bijective1x1Conv2d)):    # Bijective1x1Conv2d: the C x C map of a 1x1 convolution
        p = layer._prepared()
        if fwd:    # x @ W^T + b                     (transforms.py:913-934)
            out.append(Prim("aff", W=p["matrix64"], c=p["bias"].double()))
        else:      # (y - b) @ Winv^T = y Winv^T - Winv b   (transforms.py:936-962)
            out.append(Prim("aff", W=p["inverse64"], c=-_matvec64(p["inverse64"], p["bias"].double())))
        return
    if isinstance(layer, T.MaskedCoupling):
        out.append(Prim("coupling", prep=layer._raw(), sign=1.0 if fwd else -1.0))
        return
    if isinstance(layer, T.ScaleTransform):
        s = layer.scale.detach().reshape(-1)
        ops.require_cuda(s, "ScaleTransform.scale")
        out.append(Prim("mul" if fwd else "div", v=s))
        return
    if isinstance(layer, T.LeakyReLUTransform):
        out.append(Prim("leaky", slope=layer.alpha if fwd else 1.0 / layer.alpha))
        return
    if isinstance(layer, T.Permute):
        out.append(Prim("perm", v=(layer.permutation if fwd else layer.inv_permutation).long()))
        return
    raise NotImplementedError(f"usflows_b200: no kernel path for layer type {type(layer).__name__}")


def _matmul64(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    out = torch.empty(a.shape[0], b.shape[1], dtype=torch.float64, device=a.device)
    ops.matmul_f64(a.contiguous(), b.contiguous(), out)
    return out


def _matvec64(W: torch.Tensor, v: torch.Tensor) -> torch.Tensor:
    return _matmul64(W, v.reshape(-1, 1)).reshape(-1)


def _compose_run(run: List[Prim]) -> Prim:
    """Fold a run of affine / diagonal / permutation maps (applied left to right) into one dense (W, c) in fp64:
    (W2, c2) o (W1, c1) = (W2 W1, W2 c1 + c2)."""
    W = c = None
    pend: List[Prim] = []                     # diagonal / permutation maps seen before the first dense one

    def apply_left(W, c, p):                  # (W, c) followed by p
        if p.kind == "mul":
            v = p.v.double()
            return W * v[:, None], None if c is None else c * v
        if p.kind == "div":
            v = 1.0 / p.v.double()
            return W * v[:, None], None if c is None else c * v
        if p.kind == "perm":                  # y = x[:, idx]
            return W[p.v], None if c is None else c[p.v]
        W2 = _matmul64(p.W, W)
        c2 = p.c if c is None else (_matvec64(p.W, c) + (p.c if p.c is not None else 0))
        return W2, c2

    for p in run:
        if W is None:
            if p.kind != "aff":
                pend.append(p)
                continue
            W, c = p.W, p.c
            for q in reversed(pend):          # q happened BEFORE the dense map: fold into its columns
                if q.kind == "mul":
                    W = W * q.v.double()[None, :]
                elif q.kind == "div":
                    W = W * (1.0 / q.v.double())[None, :]
                else:                          # x' = x[:, idx]; y = x' W^T  ->  W_new[:, idx[j]] = W[:, j]
                    Wn = torch.zeros_like(W)
                    Wn[:, q.v] = W
                    W = Wn
            continue
        W, c = apply_left(W, c, p)
    return Prim("aff", W=W, c=c)


@dataclass
class Step:
    kind: str                                  # "mm" | "leaky" | "permute" | "vec" | "affine" (affine coupling update)
                                               # | "gate" (ConvNet conditioner: gate + LayerNorm + re-encoding)
    src: str = "x"                             # "x" (stream), "h" (conditioner hidden) or "hr" (its un-rectified copy)
    dst: str = "x"                             # "x", "h", "st" (fp32 scratch) or "r" (fp32 residual of the conditioner)
    w: Optional[torch.Tensor] = None           # operand-format weight [N, K] (hi plane / fp32 / bf16)
    w_lo: Optional[torch.Tensor] = None
    N: int = 0
    K: int = 0
    engine: int = ENGINE_SIMT
    bias: Optional[torch.Tensor] = None
    relu: bool = False
    resid: bool = False                        # out = x + sign * value (in place on the stream segment `out_seg`)
    sign: float = 1.0
    in_seg: Optional[tuple] = None             # (col0, width) of the stream read as A (None = whole stream)
    out_seg: Optional[tuple] = None            # (col0, width) of the stream written (None = whole / new buffer)
    vec_div: Optional[torch.Tensor] = None     # "vec" steps: ((x / div) * mul)
    vec_mul: Optional[torch.Tensor] = None
    slope: float = 1.0
    perm: Optional[torch.Tensor] = None
    final: bool = False                        # writes the program's fp32 result
    clip: Optional[tuple] = None               # "affine" steps: (log-scale min, max)
    gated: bool = False                        # "gate" steps: x + val * sigmoid(gate) (else: pass the scratch through)
    ln: Optional[tuple] = None                 #   (gamma, beta, eps) of the LayerNormVector that follows, or None
    keep_f32: bool = False                     #   keep the result as the fp32 residual of the next gated block
    want_raw: bool = False                     #   also write un-rectified operand planes (input of the next block's proj)


def _operand(w64_or_32: torch.Tensor, mode: str, engine: int, overflow_flag: Optional[torch.Tensor] = None):
    """fp32/fp64 weight [N, K] -> operand planes of the engine (ops.ENGINE_PLANES), zero-filled, pitch padded to a 16-byte
    multiple: (plane, None), or (hi, lo) of a split format, two planes of ONE allocation with hi first."""
    w = w64_or_32.to(torch.float32)
    rows, cols = w.shape
    ld = pad4(cols)
    src = torch.zeros(rows, ld, dtype=torch.float32, device=w.device)[:, :cols]
    src.copy_(w)
    if ops.ENGINE_PLANES[engine] == ("f32",):
        return src, None
    dtype = {ENGINE_TC_3XF16: torch.float16, ENGINE_TC_3XTF32: torch.float32, ENGINE_TC_BF16: torch.bfloat16}[engine]
    buf = torch.zeros(len(ops.ENGINE_PLANES[engine]), rows, ld, dtype=dtype, device=w.device)[:, :, :cols]
    if engine == ENGINE_TC_3XF16:
        ops.split_f16(src, buf[0], buf[1], overflow_flag)
    elif engine == ENGINE_TC_3XTF32:
        ops.split_tf32(src, buf[0], buf[1])
    else:
        ops.to_bf16(src, buf[0])
    return buf[0], buf[1] if len(buf) == 2 else None


def convnet_steps(mode: str, desc: dict, first_w, first_b, last_w, last_b, wflag=None, *, in_seg=None, out_seg=None,
                  resid: bool = False, sign: float = 1.0) -> List[Step]:
    """Launch steps of a `nn.ConvNet` vector conditioner (networks.py:287-307): every Linear is one contraction, the
    GatedMLP gate (networks.py:237-245), the LayerNormVector and the ReLU / re-encoding in front of the next Linear are
    one `gate` step.  `desc` = dict(first, blocks, last) of detached (weight, bias) tensors; `first_*` / `last_*` are the
    outer Linears as the caller wants them run (mask folded / compressed)."""
    steps: List[Step] = []

    def mm(w, b, **kw):
        N, K = w.shape
        eng = _engine_for(mode, N, K)
        wo, wl = _operand(w, mode, eng, wflag)
        steps.append(Step("mm", w=wo, w_lo=wl, N=N, K=K, engine=eng, bias=b.to(torch.float32).contiguous(), **kw))

    blocks = desc["blocks"]

    def gate(n, blk, nxt):
        steps.append(Step("gate", src="st", dst="h", N=n, gated=bool(blk and blk["gated"]), ln=blk["ln"] if blk else None,
                          relu=nxt is not None, keep_f32=nxt is not None and nxt["gated"] and nxt["proj"] is None,
                          want_raw=nxt is not None and nxt["proj"] is not None))

    mm(first_w, first_b, src="x", dst="st", in_seg=in_seg)
    gate(first_w.shape[0], None, blocks[0] if blocks else None)
    for i, blk in enumerate(blocks):
        nxt = blocks[i + 1] if i + 1 < len(blocks) else None
        if blk["gated"]:
            mm(*blk["lin1"], src="h", dst="h", relu=True)              # relu(Linear(relu(x)))
            if blk["proj"] is not None:
                mm(*blk["proj"], src="hr", dst="r")                    # residual = proj(x)
            mm(*blk["lin2"], src="h", dst="st")                        # [val | gate]
        else:
            mm(*blk["lin1"], src="h", dst="st")                        # Linear(relu(x))
        gate(blk["lin1"][0].shape[0], blk, nxt)
    mm(last_w, last_b, src="h", dst="x", resid=resid, sign=sign, out_seg=out_seg)
    return steps


class ProgramCore:
    """What the launch programs of flat (Program) and image-shaped (image_engine.ImageProgram) events share: the lowering of
    the layer stack, the fp16-range policy for weights, the tf32-split fallback and the chunked `run`.  A subclass supplies
      _build(prims)          its launches from the lowered stack, and `uses_range_flag`
      _in_mode(mode)         the same program in another precision mode (the tf32-split fallback)
      _chunk_bounds(rows, chunk_rows) -> [(r0, r1), ...]
      _chunk(x, out, flag, dq, ladj_rows, to_caller)   one chunk into `out`: the caller's output when `to_caller`, else
                             the `final_buffer` handed to a sink
      out_width(d_in)"""

    fp16_weight_modes = ("fp32",)      # the modes whose weight preparation writes fp16 split planes

    def __init__(self, layers, direction: str, mode: Optional[str]):
        self.mode = mode or _default_precision
        self.layers, self.direction = list(layers), direction
        self._fallback_prog: Optional["ProgramCore"] = None
        self._wflag: Optional[torch.Tensor] = None          # set by weight preparation if a weight leaves fp16 range
        prims: List[Prim] = []
        for layer in (self.layers if direction == "forward" else self.layers[::-1]):
            _lower_layer(layer, direction, prims)
        self._build(prims)
        # a weight does not fit fp16: always run the tf32-split program
        self.force_fallback = self._wflag is not None and int(self._wflag.item()) != 0

    def _weight_flag(self, device) -> Optional[torch.Tensor]:
        """The device flag weight preparation sets when a weight leaves the fp16 range (None in modes without fp16 weights)."""
        if self.mode not in self.fp16_weight_modes:
            return None
        if self._wflag is None:
            self._wflag = torch.zeros(1, dtype=torch.int32, device=device)
        return self._wflag

    def _fallback(self) -> "ProgramCore":
        """The same program in "fp32_tf32" mode: the same accuracy class without the fp16 range limit."""
        if self._fallback_prog is None:
            self._fallback_prog = self._in_mode("fp32_tf32")
        return self._fallback_prog

    @property
    def guarded(self) -> bool:
        """Chunks run launch by launch on fp16 split planes under a range flag (the single-launch program has none, the
        always-tf32-split one needs none)."""
        return self.uses_range_flag and self.small is None and not self.force_fallback

    def run(self, x: torch.Tensor, *, out: Optional[torch.Tensor] = None, sink=None, chunk_rows: Optional[int] = None,
            ladj_rows: Optional[torch.Tensor] = None, dq: Optional[ops.Dequant] = None) -> Optional[torch.Tensor]:
        """Evaluate the program on x [rows, d] chunk by chunk into `out` (allocated when None).  With `sink`, the result of
        each chunk is handed to `sink(chunk_f32 [r, width], r0, r1)` from a reused workspace buffer (`final_buffer`)
        instead.  With `dq`, x is uint8 and its first ingest dequantises it (ops.Dequant).  `ladj_rows` [rows]: per-row
        log-determinants the affine couplings add to."""
        ops.require_cuda(x, "input", torch.float32 if dq is None else torch.uint8)
        if x.dim() != 2:
            raise RuntimeError("usflows_b200: expected a [rows, d] input")
        x = x.contiguous()
        rows, width = x.shape[0], self.out_width(x.shape[1])         # out_width also rejects a wrong event width
        if sink is None and out is None:
            out = torch.empty(rows, width, dtype=torch.float32, device=x.device)
        if rows == 0:                       # empty batch: nothing to launch
            return None if sink is not None else out
        if self.force_fallback:
            return self._fallback().run(x, out=out, sink=sink, chunk_rows=chunk_rows, ladj_rows=ladj_rows, dq=dq)

        def chunk(prog, r0, r1, flag):
            fin = out[r0:r1] if sink is None else self.final_buffer(x.device, "final", r1 - r0, x.shape[1])
            prog._chunk(x[r0:r1], fin, flag, None if dq is None else dq.shifted(r0),
                        None if ladj_rows is None else ladj_rows[r0:r1], sink is None)
            if sink is not None:
                sink(fin, r0, r1)

        run_chunks(self._chunk_bounds(rows, chunk_rows), x.device, self.uses_range_flag,
                   lambda i, r0, r1, flag: chunk(self, r0, r1, flag),
                   lambda i, r0, r1: chunk(self._fallback(), r0, r1, None), ladj_rows=ladj_rows)
        return None if sink is not None else out


class Program(ProgramCore):
    """Launch program of one direction of a layer stack for one precision mode and weight version."""

    def __init__(self, layers, direction: str, mode: Optional[str] = None, build=None):
        """`build(mode)` -> the launch steps of a program that evaluates one conditioner network alone (`layers` is then
        empty)."""
        self.build = build
        super().__init__(layers, direction, mode)

    def _in_mode(self, mode: str) -> "Program":
        return Program(self.layers, self.direction, mode, self.build)

    def _build(self, prims: List[Prim]) -> None:
        # 1. compose maximal runs of affine-like maps that contain at least one dense matrix
        items: List[Prim] = []
        run: List[Prim] = []

        def flush():
            if not run:
                return
            if not any(p.kind == "aff" for p in run):
                items.extend(run)
            elif MERGE_AFFINE:
                items.append(_compose_run(run))
            else:
                # one contraction per dense layer (as the reference); diagonal / permutation maps are folded into
                # the nearest dense layer -- that is exact up to one rounding of the scaled weight
                dense = [i for i, p in enumerate(run) if p.kind == "aff"]
                for n, i in enumerate(dense):      # leading maps join the first dense layer, others the earlier one
                    lo = 0 if n == 0 else i
                    hi = dense[n + 1] if n + 1 < len(dense) else len(run)
                    items.append(_compose_run(run[lo:hi]))
            run.clear()

        for p in prims:
            if p.kind in ("aff", "mul", "div", "perm"):
                run.append(p)
            else:
                flush()
                items.append(p)
        flush()
        self.items = items
        self.has_row_ladj = any(p.kind == "coupling" and p.prep.get("affine") for p in items)
        self.small = self._pack_small(items) if FUSE_SMALL else None
        # 2. widths, engine choice (tiny problems run the whole program on the SIMT engine)
        dims = []
        for p in items:
            if p.kind == "aff":
                dims += list(p.W.shape)
            elif p.kind == "coupling":
                for w in p.prep["weights"]:
                    dims += list(w.shape)
        compress = self._compression_plan(items)
        if compress is not None:
            dims += [compress["h1"], compress["h0"]]
        if dims and min(dims) < TC_MIN_DIM and self.mode != "fp32_simt":
            self.mode = "fp32_simt"
            compress = self._compression_plan(items)
        self.compress = compress
        self.steps = self._emit(items, compress) if self.build is None else self.build(self.mode)
        self.uses_range_flag = self.mode == "fp32"              # fp16 split planes: chunks carry a range flag

    # -- tiny event sizes: pack every layer into one weight blob + op list for the whole-flow kernel
    @staticmethod
    def _pack_small(items):
        if not items or any(p.kind not in ("aff", "coupling") for p in items):
            return None
        d = None
        hidden = 0
        for p in items:
            if p.kind == "aff":
                if p.W.shape[0] != p.W.shape[1]:
                    return None
                dd = p.W.shape[0]
            else:
                ws = p.prep["weights"]
                if len(ws) < 2 or p.prep.get("affine") or p.prep.get("net"):
                    return None
                dd = ws[0].shape[1]
                if ws[-1].shape[0] != dd:
                    return None
                hidden = max([hidden] + [w.shape[0] for w in ws[:-1]])
            if d is None:
                d = dd
            if dd != d:
                return None
        if d is None or d > 8 or hidden > 64:
            return None
        D = 2 if d <= 2 else 4 if d <= 4 else 8
        H = 32 if hidden <= 32 else 64
        dev = (items[0].W if items[0].kind == "aff" else items[0].prep["weights"][0]).device
        prog, blocks, off = [], [], 0

        def pad2(t, r, c):
            o = torch.zeros(r, c, dtype=torch.float32, device=dev)
            o[:t.shape[0], :t.shape[1]] = t.to(torch.float32)
            return o

        def pad1(t, n):
            o = torch.zeros(n, dtype=torch.float32, device=dev)
            o[:t.shape[0]] = t.to(torch.float32)
            return o

        for p in items:
            parts = []
            if p.kind == "aff":
                W = torch.eye(D, dtype=torch.float32, device=dev)
                W[:d, :d] = p.W.to(torch.float32)
                c = pad1(p.c if p.c is not None else torch.zeros(d, device=dev), D)
                parts = [W.reshape(-1), c]
                code = 0
            else:
                ws, bs, m = p.prep["weights"], p.prep["biases"], p.prep["mask"].reshape(-1).to(torch.float32)
                parts.append(pad2(ws[0] * m[None, :], H, D).reshape(-1))
                parts.append(pad1(bs[0], H))
                for w, b in zip(ws[1:-1], bs[1:-1]):
                    parts.append(pad2(w, H, H).reshape(-1))
                    parts.append(pad1(b, H))
                g = float(p.sign) * (1 - m)
                parts.append(pad2(ws[-1] * g[:, None], D, H).reshape(-1))
                parts.append(pad1(bs[-1] * g, D))
                code = 1 | ((len(ws) - 2) << 8)
            blk = torch.cat(parts)
            if blk.numel() % 4:
                blk = torch.cat([blk, torch.zeros(4 - blk.numel() % 4, dtype=torch.float32, device=dev)])
            prog += [code, off]
            off += blk.numel()
            blocks.append(blk)
        if off * 4 > 200 * 1024:
            return None
        return dict(prog=torch.tensor(prog, dtype=torch.int32, device=dev), blob=torch.cat(blocks).contiguous(),
                    n_ops=len(items), D=D, H=H, d=d)

    # -- mask compression: run the couplings in a feature order that makes "conditioner inputs" and "updated
    #    features" two contiguous column segments, so the first / last conditioner GEMMs shrink to half size
    def _compression_plan(self, items):
        coups = [i for i, p in enumerate(items) if p.kind == "coupling"]
        if not coups or not COMPRESS_MASK:
            return None
        part = items[coups[0]].prep["mask"]
        for i in coups:
            m = items[i].prep["mask"]
            if m.shape != part.shape or not (torch.equal(m, part) or torch.equal(m, 1 - part)):
                return None
            # every block of consecutive couplings must be bounded by dense affine steps on both sides
            j = i
            while j >= 0 and items[j].kind == "coupling":
                j -= 1
            k = i
            while k < len(items) and items[k].kind == "coupling":
                k += 1
            if j < 0 or k >= len(items) or items[j].kind != "aff" or items[k].kind != "aff":
                return None
        idx1 = torch.nonzero(part > 0.5).reshape(-1)
        idx0 = torch.nonzero(part <= 0.5).reshape(-1)
        h1, h0 = int(idx1.numel()), int(idx0.numel())
        if h1 == 0 or h0 == 0:
            return None
        if self.mode != "fp32_simt" and (h1 % 8 or h0 % 8):
            return None
        return dict(part=part, idx1=idx1, idx0=idx0, order=torch.cat([idx1, idx0]), h1=h1, h0=h0)

    @staticmethod
    def _coupling_io(mask, compress, ws, bs, affine: bool = False):
        """(in_seg, out_seg) of a coupling's conditioner, whose Linear weights / biases `ws` / `bs` (first to last) are
        adapted in place.  With mask compression the conditioner reads the column segment in_seg and updates out_seg, and
        its first / last Linear keep only those columns / rows; else both segments are None and the mask is folded into
        the first / last Linear.  `affine`: the last Linear's rows are [log-scale | shift], both halves are re-indexed."""
        if compress is None:
            m = mask.reshape(-1).to(torch.float32)
            g = torch.cat([1 - m, 1 - m]) if affine else 1 - m
            ws[0] = ws[0] * m[None, :]
            ws[-1], bs[-1] = ws[-1] * g[:, None], bs[-1] * g
            return None, None
        first = torch.equal(mask, compress["part"])                 # the conditioner reads the idx1 features
        idx_in = compress["idx1"] if first else compress["idx0"]
        idx_out = compress["idx0"] if first else compress["idx1"]
        if affine:                                                  # rows [0, d): log-scale, [d, 2d): shift
            idx_out = torch.cat([idx_out, mask.numel() + idx_out])
        ws[0] = ws[0][:, idx_in]
        ws[-1], bs[-1] = ws[-1][idx_out], bs[-1][idx_out]
        h1, h0 = compress["h1"], compress["h0"]
        return ((0, h1), (h1, h0)) if first else ((h1, h0), (0, h1))

    def _emit(self, items, compress) -> List[Step]:
        mode = self.mode
        steps: List[Step] = []
        n = len(items)
        for i, p in enumerate(items):
            if p.kind == "aff":
                W, c = p.W, p.c
                if compress is not None:
                    if i > 0 and items[i - 1].kind == "coupling":
                        W = W[:, compress["order"]]
                    if i + 1 < n and items[i + 1].kind == "coupling":
                        W = W[compress["order"]]
                        c = None if c is None else c[compress["order"]]
                N, K = W.shape
                eng = _engine_for(mode, N, K)
                w, w_lo = _operand(W, mode, eng, self._weight_flag(W.device))
                bias = None if c is None else c.to(torch.float32).contiguous()
                steps.append(Step("mm", w=w, w_lo=w_lo, N=N, K=K, engine=eng, bias=bias))
            elif p.kind == "coupling" and p.prep.get("net") == "convnet":
                desc = p.prep["desc"]
                ws, bs = [desc["first"][0], desc["last"][0]], [desc["first"][1], desc["last"][1]]
                in_seg, out_seg = self._coupling_io(p.prep["mask"], compress, ws, bs)
                steps += convnet_steps(mode, desc, ws[0], bs[0], ws[1], bs[1], self._weight_flag(ws[0].device),
                                       in_seg=in_seg, out_seg=out_seg, resid=True, sign=p.sign)
            elif p.kind == "coupling":
                ws, bs = list(p.prep["weights"]), list(p.prep["biases"])
                nl = len(ws)
                affine = bool(p.prep.get("affine"))
                in_seg, out_seg = self._coupling_io(p.prep["mask"], compress, ws, bs, affine)
                for j in range(nl):
                    last = j == nl - 1
                    N, K = ws[j].shape
                    eng = _engine_for(mode, N, K)
                    w, w_lo = _operand(ws[j], mode, eng, self._weight_flag(ws[j].device))
                    if last and affine:
                        steps.append(Step("mm", src="x" if j == 0 else "h", dst="st", w=w, w_lo=w_lo, N=N, K=K, engine=eng,
                                          bias=bs[j].to(torch.float32).contiguous(), in_seg=in_seg if j == 0 else None))
                        steps.append(Step("affine", sign=p.sign, out_seg=out_seg, N=N // 2, clip=tuple(p.prep["clip"])))
                        continue
                    steps.append(Step("mm", src="x" if j == 0 else "h", dst="x" if last else "h", w=w, w_lo=w_lo,
                                      N=N, K=K, engine=eng, bias=bs[j].to(torch.float32).contiguous(), relu=not last,
                                      resid=last, sign=p.sign, in_seg=in_seg if j == 0 else None,
                                      out_seg=out_seg if last else None))
            elif p.kind == "mul":
                steps.append(Step("vec", vec_mul=p.v))
            elif p.kind == "div":
                steps.append(Step("vec", vec_div=p.v))
            elif p.kind == "perm":
                steps.append(Step("permute", perm=p.v.to(torch.int32)))
            elif p.kind == "leaky":
                steps.append(Step("leaky", slope=p.slope))
        if not steps:
            steps.append(Step("vec"))
        last_x = max(i for i, st in enumerate(steps) if st.dst == "x")
        if steps[last_x].kind == "affine":
            raise NotImplementedError("usflows_b200: a flow ending in an affine coupling needs a following layer "
                                      "(USFlow ends in an LU layer and a scale)")
        steps[last_x].final = True
        return steps

    # ----------------------------------------------------------------------------------------------
    def out_width(self, d_in: int) -> int:
        w = d_in
        for st in self.steps:
            if st.kind == "mm" and st.dst == "x" and st.out_seg is None:
                w = st.N
        return w

    def n_launches(self) -> int:
        return len(self.steps)

    def run(self, x: torch.Tensor, *, out: Optional[torch.Tensor] = None, sink=None, chunk_rows: Optional[int] = None,
            ladj_rows: Optional[torch.Tensor] = None, dq: Optional[ops.Dequant] = None) -> Optional[torch.Tensor]:
        sm = self.small
        if sm is not None and x.dim() == 2 and x.shape[0] and x.shape[1] == sm["d"]:    # one launch for the whole stack
            ops.require_cuda(x, "input", torch.float32 if dq is None else torch.uint8)
            x = x.contiguous() if dq is None else _dequantized(x.contiguous(), dq)        # it reads fp32
            res = out if (out is not None and sink is None) else torch.empty(x.shape, dtype=torch.float32, device=x.device)
            ops.flow_small(x, sm["prog"], sm["blob"], sm["n_ops"], sm["D"], sm["H"], res)
            if sink is not None:
                sink(res, 0, x.shape[0])
                return None
            return res
        return super().run(x, out=out, sink=sink, chunk_rows=chunk_rows, ladj_rows=ladj_rows, dq=dq)

    def _chunk_bounds(self, rows: int, chunk_rows: Optional[int]):
        return chunk_bounds(rows, chunk_rows or _default_chunk_rows)

    def _chunk(self, x, out, flag, dq, ladj_rows, to_caller: bool) -> None:
        self._run_chunk(x, out, flag, dq, ladj_rows=ladj_rows)

    def final_buffer(self, device, name: str, rows: int, d_in: int) -> torch.Tensor:
        """The workspace buffer [rows, out_width(d_in)] a chunk's result is written to when it is handed on."""
        return _workspace.planes(device, name, rows, self.out_width(d_in), "f32")

    def _run_chunk(self, x: torch.Tensor, final_out: torch.Tensor, flag: Optional[torch.Tensor] = None,
                   dq: Optional[ops.Dequant] = None, *, ladj_rows: Optional[torch.Tensor] = None) -> None:
        """One chunk x [rows, d]; with `dq`, x is uint8 and is dequantised by the first kernel that reads it."""
        dev, rows = x.device, x.shape[0]
        steps = self.steps
        hidden = _planes(self.mode)                                       # conditioner hidden and contraction operands
        stream = hidden + ("f32",) if self.mode == "bf16" else hidden      # bf16: the residual stream stays fp32 too
        flip = {"x": 0, "h": 0}
        cur: Optional[Act] = None               # stream
        hid: Optional[Act] = None               # conditioner hidden
        hid_raw: Optional[Act] = None           # ConvNet conditioner: un-rectified planes of the hidden (input of a proj)
        res_buf: Optional[torch.Tensor] = None  # ConvNet conditioner: fp32 residual stream of the gated blocks
        st_buf: Optional[torch.Tensor] = None   # fp32 scratch: affine coupling [log-scale | shift], ConvNet [val | gate]

        def new_act(slot: str, width: int, planes: tuple) -> Act:
            flip[slot] ^= 1
            a = Act(rows, width)
            for pl in planes:
                setattr(a, pl, _workspace.planes(dev, f"{slot}{flip[slot]}", rows, width, pl))
            return a

        def seg_view(a: Act, seg) -> Act:
            if seg is None:
                return a
            c0, w = seg
            v = Act(a.rows, w)
            for pl in ("f32", "hi", "lo", "bf16", "h16", "l16"):
                t = getattr(a, pl)
                if t is not None:
                    setattr(v, pl, t[:, c0:c0 + w])
            return v

        def ingest(src: Act, out: Act, **kw) -> None:
            if src is src_f32 and dq is not None:
                ops.ingest_u8(x, dq, out, **kw)
            else:
                ops.ingest(src.f32, out, **kw)

        # the user's tensor: read-only.  8-bit rows have no plane a consumer could read: the first step ingests them
        src_f32 = Act(rows, x.shape[1], f32=x if dq is None else None)
        cur = src_f32
        if dq is not None and steps and steps[0].kind in ("leaky", "permute"):    # kernels that read fp32 only
            cur = new_act("x", x.shape[1], ("f32",))
            ingest(src_f32, cur)
        for i, st in enumerate(steps):
            nxt = steps[i + 1] if i + 1 < len(steps) else None
            if st.kind == "mm":
                if st.src == "x":
                    in_coupling = st.dst in ("h", "st") or st.resid
                    need = stream if in_coupling else hidden
                    direct_ok = st.engine == ENGINE_SIMT or (x.data_ptr() % 16 == 0 and x.stride(0) % 4 == 0)
                    if not all(getattr(cur, pl) is not None for pl in need) or (cur is src_f32 and not direct_ok):
                        if cur.f32 is None and not (cur is src_f32 and dq is not None):
                            raise RuntimeError("internal: activation has no fp32 plane to re-encode from")
                        b = new_act("x", cur.width, need)
                        ingest(cur, b, overflow_flag=flag)
                        cur = b
                    a = seg_view(cur, st.in_seg)
                else:
                    a = hid_raw if st.src == "hr" else hid
                if st.dst in ("st", "r"):                             # fp32 scratch (affine coupling's [s | t], ConvNet)
                    out = Act(rows, st.N, f32=_workspace.planes(dev, st.dst, rows, st.N, "f32"))
                    resid = None
                elif st.dst == "h":
                    out = new_act("h", st.N, hidden)
                    resid = None
                elif st.resid:                                         # coupling output
                    if st.out_seg is not None:                         # in place on the updated column segment
                        out = seg_view(cur, st.out_seg)
                        resid = out
                        full_out = cur
                    else:
                        resid = cur
                        out = new_act("x", st.N, stream)
                        full_out = out
                    if st.final:
                        if st.out_seg is not None:
                            raise RuntimeError("internal: a compressed coupling cannot be the final step")
                        out = Act(rows, st.N, f32=final_out)
                        full_out = out
                    elif nxt is not None and nxt.kind in ("leaky", "permute", "vec") and full_out.f32 is None:
                        out.f32 = _workspace.planes(dev, "xf", rows, st.N, "f32")
                else:                                                  # affine step
                    resid = None
                    if st.final:
                        out = Act(rows, st.N, f32=final_out)
                    else:
                        elementwise_next = nxt is not None and nxt.kind in ("leaky", "permute", "vec")
                        out = new_act("x", st.N, ("f32",) if elementwise_next else stream)
                    full_out = out
                ops.linear(st.engine, a, st.w, st.w_lo, st.N, st.K, bias=st.bias, relu=st.relu, resid=resid,
                           resid_sign=st.sign, out=out, overflow_flag=flag)
                if st.dst == "st":
                    st_buf = out.f32
                elif st.dst == "r":
                    res_buf = out.f32
                elif st.dst == "h":
                    hid = out
                else:
                    cur = full_out
            elif st.kind == "gate":                                    # ConvNet conditioner glue between two contractions
                act = new_act("h", st.N, hidden)
                raw = None
                if st.want_raw:
                    raw = Act(rows, st.N)
                    for pl in hidden:
                        setattr(raw, pl, _workspace.planes(dev, "hr", rows, st.N, pl))
                y = None
                if st.keep_f32:                                        # gated: in place on the residual stream
                    y = res_buf if st.gated else _workspace.planes(dev, "r", rows, st.N, "f32")
                gamma, beta, eps = st.ln if st.ln is not None else (None, None, 0.0)
                ops.gate_norm(st_buf, st.N, xres=res_buf if st.gated else None, gated=st.gated, gamma=gamma, beta=beta,
                              eps=eps, y_f32=y, act=act, act_relu=st.relu, raw=raw, overflow_flag=flag)
                hid, hid_raw = act, raw
                if y is not None:
                    res_buf = y
            elif st.kind == "affine":                                  # x_seg <- x_seg * exp(s) + t  (or the inverse), in place
                if cur is src_f32:                                     # never update the caller's tensor
                    b = new_act("x", cur.width, stream)
                    ingest(cur, b, overflow_flag=flag)
                    cur = b
                target = seg_view(cur, st.out_seg)
                ops.affine_couple(st_buf, target, st.sign, st.clip[0], st.clip[1], row_ladj=ladj_rows, overflow_flag=flag)
                if nxt is not None and nxt.kind in ("leaky", "permute", "vec") and cur.f32 is None:
                    raise NotImplementedError("usflows_b200: an elementwise layer directly after an affine coupling is not built")
            else:                                                      # elementwise kernels on the fp32 plane
                if cur.f32 is None and not (st.kind == "vec" and cur is src_f32 and dq is not None):
                    raise RuntimeError("internal: elementwise step needs an fp32 stream plane")
                out = Act(rows, cur.width, f32=final_out) if st.final else new_act("x", cur.width, ("f32",))
                if st.kind == "vec":
                    ingest(cur, out, div=st.vec_div, mul=st.vec_mul)
                elif st.kind == "leaky":
                    ops.leaky_relu(cur.f32, st.slope, out.f32)
                else:
                    ops.permute(cur.f32, st.perm, out.f32)
                cur = out

    # -- whole-stack C entry (usf_plan_* / usf_flow_*): one call per chunk instead of one per launch --------------------
    def plan_able(self) -> bool:
        return (self.small is None and not self.force_fallback and not self.has_row_ladj and bool(self.steps)
                and all(st.kind == "mm" and st.dst in ("x", "h") and st.src in ("x", "h")
                        and (not st.resid or st.out_seg is not None) for st in self.steps)
                and self.steps[-1].dst == "x" and self.steps[-1].out_seg is None)

    def c_plan(self, d_in: int, max_rows: int, base=None, add_const: float = 0.0) -> "CPlan":
        """The launch program as a library-owned plan (None when a step kind is outside its scope).  Cached per
        (input width, rows capacity, base parameters)."""
        if not self.plan_able():
            return None
        key = (d_in, max_rows, None if base is None else tuple(t.data_ptr() for t in base._prepared()), float(add_const))
        cache = self.__dict__.setdefault("_c_plans", {})
        if key not in cache:
            if len(cache) >= 4:
                cache.pop(next(iter(cache))).close()
            cache[key] = CPlan(self, d_in, max_rows, base, add_const)
        return cache[key]

class CPlan:
    """Owner of one `usf_plan` (include/usflows_b200.h, "Whole-stack evaluation"): keeps the Program (whose operand planes
    the plan points into) and the base parameters alive, destroys the plan with itself."""

    def __init__(self, prog: "Program", d_in: int, max_rows: int, base=None, add_const: float = 0.0):
        import ctypes as C
        from . import _lib
        lib = _lib.load()
        self._lib, self.prog, self.base, self.max_rows, self.d_in = lib, prog, base, int(max_rows), int(d_in)
        handle = C.c_void_p()
        CPlan._drain_parked()
        _lib.check(lib.usf_plan_create(C.byref(handle), d_in, _lib.MODE_CODES[prog.mode], int(max_rows)))
        self.handle = handle
        self._keep = []
        try:
            for st in prog.steps:
                s = _lib.PlanLinear()
                s.N, s.K, s.engine, s.relu = st.N, st.K, st.engine, int(st.relu)
                s.w, s.w_lo, s.ldw = st.w.data_ptr(), (None if st.w_lo is None else st.w_lo.data_ptr()), ops._ld(st.w)
                s.bias = None if st.bias is None else st.bias.data_ptr()
                s.src = _lib.PLAN_SRC_STREAM if st.src == "x" else _lib.PLAN_SRC_HIDDEN
                if st.dst == "h":
                    s.dst = _lib.PLAN_DST_HIDDEN
                elif st.resid:
                    if st.out_seg is None:
                        raise NotImplementedError("coupling outputs on the whole stream are not in the plan's scope")
                    s.dst, s.out_col0 = _lib.PLAN_DST_SEGMENT, st.out_seg[0]
                else:
                    s.dst = _lib.PLAN_DST_STREAM
                if st.in_seg is not None:
                    s.in_col0, s.in_width = st.in_seg
                s.resid_sign = float(st.sign)
                _lib.check(lib.usf_plan_add_linear(handle, C.byref(s)))
            if base is not None:
                loc, scale = base._prepared()
                self._keep += [loc, scale]
                _lib.check(lib.usf_plan_set_base(handle, base.base_kind, loc.data_ptr(), scale.data_ptr(), float(add_const)))
            with ops.on_device(prog.steps[0].w):
                _lib.check(lib.usf_plan_finalize(handle))
        except Exception:
            self.close()
            raise
        self.out_width = prog.out_width(d_in)

    # A plan owns device memory that usf_plan_destroy releases with cudaFree, and the garbage collector may run a plan's
    # __del__ at ANY point -- also while a CUDA graph is being captured on this thread, where cudaFree is not permitted
    # and invalidates the capture (seen: a plan of an earlier weight version collected inside `_log_prob_small_batch`'s
    # capture).  Destruction under a capture is therefore parked and carried out by the next close / create outside one.
    _parked: List[tuple] = []

    @staticmethod
    def _capturing() -> bool:
        try:
            return torch.cuda.is_available() and torch.cuda.is_current_stream_capturing()
        except Exception:                      # noqa: BLE001
            return False

    @classmethod
    def _drain_parked(cls) -> None:
        while cls._parked and not cls._capturing():
            lib, handle = cls._parked.pop()
            lib.usf_plan_destroy(handle)

    def close(self) -> None:
        if getattr(self, "handle", None) is not None:
            handle, self.handle = self.handle, None
            if self._capturing():
                CPlan._parked.append((self._lib, handle))
            else:
                self._lib.usf_plan_destroy(handle)
                CPlan._drain_parked()

    def __del__(self):
        try:
            self.close()
        except Exception:                      # noqa: BLE001  (interpreter shutdown)
            pass

    def log_prob(self, x: torch.Tensor, out: torch.Tensor, flag: Optional[torch.Tensor] = None,
                 dq: Optional[ops.Dequant] = None) -> None:
        """out[r] = log p(x[r]) for r < rows <= max_rows on the current stream; with `dq`, x is uint8 (usf_flow_logprob_u8)."""
        ops.LAUNCHES += len(self.prog.steps) + 2
        from . import _lib
        fl = None if flag is None else flag.data_ptr()
        if dq is not None:
            import ctypes as C
            s = dq.struct()
            _lib.check(self._lib.usf_flow_logprob_u8(self.handle, x.data_ptr(), ops._ld(x), x.shape[0], C.byref(s),
                                                     out.data_ptr(), fl, ops._stream()))
            return
        _lib.check(self._lib.usf_flow_logprob(self.handle, x.data_ptr(), ops._ld(x), x.shape[0], out.data_ptr(), fl,
                                              ops._stream()))

    def apply(self, x: torch.Tensor, z: torch.Tensor, flag: Optional[torch.Tensor] = None) -> None:
        ops.LAUNCHES += len(self.prog.steps) + 1
        from . import _lib
        _lib.check(self._lib.usf_flow_apply(self.handle, x.data_ptr(), ops._ld(x), x.shape[0], z.data_ptr(), ops._ld(z),
                                            None if flag is None else flag.data_ptr(), ops._stream()))


# --------------------------------------------------------------------------------------------------
# workspace
# --------------------------------------------------------------------------------------------------
class _Workspace:
    """Reusable device buffers keyed by (device, slot name, plane)."""

    def __init__(self):
        self._bufs = {}
        self.generation = 0          # bumped whenever a buffer is (re)allocated: captured CUDA graphs go stale

    _PAIR = {"h16": ("p16", 0), "l16": ("p16", 1), "hi": ("p32", 0), "lo": ("p32", 1)}

    def planes(self, device, name: str, rows: int, width: int, fmt: str) -> torch.Tensor:
        ld = pad4(width)
        need = rows * ld
        dtype = torch.bfloat16 if fmt == "bf16" else torch.float16 if fmt in ("h16", "l16", "pix") else torch.float32
        pair = self._PAIR.get(fmt)
        if pair is not None:
            # the two planes of a split format live in ONE allocation, hi first: the contraction kernel then fetches both
            # with one 3-D TMA operation per tile (plane = third tensor dimension; needs lo - hi > 0)
            key = (device, name, pair[0])
            buf = self._bufs.get(key)
            if buf is None or buf.shape[1] < need:
                buf = torch.empty(2, max(need, 8), dtype=dtype, device=device)
                self._bufs[key] = buf
                self.generation += 1
            return buf[pair[1], :need].view(rows, ld)[:, :width]
        key = (device, name, fmt)
        buf = self._bufs.get(key)
        if buf is None or buf.numel() < need:
            buf = torch.empty(max(need, 1), dtype=dtype, device=device)
            self._bufs[key] = buf
            self.generation += 1
        return buf[:need].view(rows, ld)[:, :width]


_workspace = _Workspace()


# --------------------------------------------------------------------------------------------------
# public helpers used by the layer / flow classes
# --------------------------------------------------------------------------------------------------
def _dequantized(x: torch.Tensor, dq: ops.Dequant) -> torch.Tensor:
    """fp32 copy of the 8-bit rows x [rows, d] (for the routes that read fp32 only)."""
    out = torch.empty(x.shape, dtype=torch.float32, device=x.device)
    if x.numel():
        ops.ingest_u8(x, dq, Act(x.shape[0], x.shape[1], f32=out))
    return out


def _flatten_rows(x: torch.Tensor, event_ndim: int = 1, dtype=torch.float32):
    ops.require_cuda(x, "input", dtype)
    batch_shape = x.shape[:x.dim() - event_ndim]
    return x.reshape(math.prod(batch_shape), math.prod(x.shape[x.dim() - event_ndim:])), batch_shape


def run_layers(layers, direction: str, x: torch.Tensor, mode: Optional[str] = None,
               chunk_rows: Optional[int] = None) -> torch.Tensor:
    x2, batch_shape = _flatten_rows(x)
    with torch.no_grad(), ops.on_device(x2):
        y = Program(layers, direction, mode).run(x2, chunk_rows=chunk_rows)
    return y.reshape(*batch_shape, y.shape[-1]) if x.dim() != 2 else y


def run_mlp(net, x: torch.Tensor, mode: Optional[str] = None) -> torch.Tensor:
    """Plain evaluation of a DenseNN (no mask, no residual) through the contraction kernels."""
    lin = list(net.layers)                   # DenseNN, or an _MLPView of a ConditionalDenseNN without its context layer

    def build(mode):
        steps = []
        for j, l in enumerate(lin):
            last = j == len(lin) - 1
            N, K = l.weight.shape
            eng = _engine_for(mode, N, K)
            w, w_lo = _operand(l.weight.detach(), mode, eng)
            steps.append(Step("mm", src="x" if j == 0 else "h", dst="x" if last else "h", w=w, w_lo=w_lo, N=N, K=K,
                              engine=eng, bias=l.bias.detach().contiguous(), relu=not last, final=last))
        return steps
    return _run_net(x, mode, [l.weight for l in lin], build)


def _run_net(x: torch.Tensor, mode: Optional[str], weights, build) -> torch.Tensor:
    """x [..., d] through a network with weight matrices `weights` whose launch steps are `build(mode)`; the whole network
    runs on the SIMT engine when one of its contractions is narrower than TC_MIN_DIM."""
    with ops.on_device(x):
        x2, batch_shape = _flatten_rows(x)
        mode = mode or _default_precision
        if min(min(w.shape) for w in weights) < TC_MIN_DIM:
            mode = "fp32_simt"
        with torch.no_grad():
            y = Program([], "forward", mode, build).run(x2)
    return y.reshape(*batch_shape, y.shape[-1]) if x.dim() != 2 else y


def total_ladj(layers) -> float:
    """Sum of the forward log|det J| of all layers -- a model constant for a USFlow (every layer's log-det
    is data independent).  One device->host read per weight version (callers cache)."""
    parts = [l._ladj_device() for l in layers]
    parts = [p for p in parts if p is not None]
    if not parts:
        return 0.0, 0
    tot = torch.stack(parts).double().sum(0).cpu()
    return float(tot[0]), int(tot[1])


def base_log_prob(base, z: torch.Tensor, add_const: float = 0.0) -> torch.Tensor:
    d = math.prod(base.event_shape)
    z2, batch_shape = _flatten_rows(z, len(base.event_shape))
    if z2.shape[1] != d:
        raise RuntimeError("usflows_b200: event shape mismatch in base log_prob")
    z2 = z2.contiguous()
    out = torch.empty(z2.shape[0], dtype=torch.float32, device=z2.device)
    if z2.shape[0]:                                             # empty batch: nothing to launch
        with ops.on_device(z2):
            base._density_into(Act(z2.shape[0], d, f32=z2), add_const, out)
    return out.reshape(batch_shape)


def base_sample(base, sample_shape=None) -> torch.Tensor:
    if sample_shape is None:
        sample_shape = []
    shape = [int(s) for s in sample_shape]
    rows = max(1, math.prod(shape))
    d = math.prod(base.event_shape)
    out = torch.empty(rows, d, dtype=torch.float32, device=base._prepared()[0].device)
    seed, offset = philox_call_stream(out.device)
    with ops.on_device(out):
        base._sample_into(out, ops.Draw(seed, offset=offset))
    return out.reshape(*shape, *base.event_shape)


class _Salt(__import__("threading").local):
    value = 0


philox_salt = _Salt()            # thread-local: the row-shard driver (parallel.py) gives every device its own stream family
PHILOX_CALL_STRIDE = 0x1000      # the kernels derive sub-streams at offset + [0, 0x200): calls must not overlap there
_philox_calls = 0                # fallback call counter (non-CUDA devices: the emulated backend of the CPU tests)


def philox_call_stream(device) -> tuple:
    """(seed, offset) of the Philox stream of ONE sampling call.  Taken from torch's CUDA generator of the device so that
    `torch.manual_seed(s)` reproduces samples and every call in the process -- of any flow / distribution object --
    draws from its own stream: the generator's offset advances by 4 per call (it is a process-global, monotonically
    increasing counter that a re-seed resets), and the call index is spread by PHILOX_CALL_STRIDE because the kernels
    use offset + small constants for their sub-streams (radius, rejection rounds, extremal coordinate)."""
    global _philox_calls
    device = torch.device(device)
    if device.type == "cuda":
        gen = torch.cuda.default_generators[device.index if device.index is not None else torch.cuda.current_device()]
        seed, off = int(gen.initial_seed()), int(gen.get_offset())
        gen.set_offset(off + 4)
        call = off // 4
    else:
        seed, call = int(torch.initial_seed()), _philox_calls
        _philox_calls += 1
    if philox_salt.value:
        seed = (seed ^ (philox_salt.value * 0x9E3779B97F4A7C15)) & ((1 << 64) - 1)
    return seed, (call * PHILOX_CALL_STRIDE) & ((1 << 62) - 1)


def leaky_relu_ladj(x: torch.Tensor, alpha: float) -> torch.Tensor:
    x2, batch_shape = _flatten_rows(x)
    x2 = x2.contiguous()
    y = torch.empty_like(x2)
    cnt = torch.empty(x2.shape[0], dtype=torch.float32, device=x2.device)
    ops.leaky_relu(x2, alpha, y, cnt)
    out = cnt * math.log(alpha)
    return out.reshape(batch_shape) if x.dim() > 1 else out.reshape(())


def profile_step(fn) -> dict:
    """Run `fn` once with CUDA events around every hot-path kernel launch; returns milliseconds summed per
    kernel class ("linear NxK", "ingest", "base_logprob") plus "_names" (launch order) and "_total"."""
    records = []
    originals = {name: getattr(ops, name) for name in ("linear", "ingest", "base_logprob", "flow_small", "gate_norm", "radial_logprob",
                                                         "affine_couple", "im2col", "conv2d_rows", "layout_transpose",
                                                         "masked_add", "pix_encode", "conv2d_pix")}

    def wrap(name, f):
        def inner(*a, **k):
            if name == "linear":
                label = f"linear {a[4]}x{a[5]}"
            else:
                label = name
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            f(*a, **k)
            e1.record()
            records.append((label, e0, e1))
        return inner

    from . import flows
    use_plan = flows.USE_C_PLAN
    try:
        flows.USE_C_PLAN = False               # launch by launch from Python, so that every launch can be bracketed
        for name, f in originals.items():
            setattr(ops, name, wrap(name, f))
        torch.cuda.synchronize()
        fn()
        torch.cuda.synchronize()
    finally:
        flows.USE_C_PLAN = use_plan
        for name, f in originals.items():
            setattr(ops, name, f)
    out = {}
    for label, e0, e1 in records:
        out[label] = out.get(label, 0.0) + e0.elapsed_time(e1)
    out["_total"] = sum(v for k, v in out.items() if not k.startswith("_"))
    out["_names"] = [r[0] for r in records]
    return out


def _convnet_desc(net) -> dict:
    """(weight, bias) tensors of a `nn.ConvNet` in the structure `convnet_steps` reads."""
    d = net._describe()
    for prm in net.parameters():
        ops.require_cuda(prm, "conditioner parameter")

    def wb(lin):
        return None if lin is None else (lin.weight.detach(), lin.bias.detach())

    blocks = [dict(gated=b["gated"], lin1=wb(b["lin1"]), lin2=wb(b["lin2"]), proj=wb(b["proj"]),
                   ln=None if b["ln"] is None else (b["ln"].weight.detach().contiguous(), b["ln"].bias.detach().contiguous(),
                                                   float(b["ln"].eps))) for b in d["blocks"]]
    return dict(first=wb(d["first"]), blocks=blocks, last=wb(d["last"]))


def _convnet_weights(desc: dict) -> list:
    ws = [desc["first"][0], desc["last"][0]]
    for b in desc["blocks"]:
        ws += [t[0] for t in (b["lin1"], b["lin2"], b["proj"]) if t is not None]
    return ws


def run_conditioner(net, x: torch.Tensor, mode: Optional[str] = None) -> torch.Tensor:
    """Plain evaluation of a `nn.ConvNet` (no mask, no residual) through the same kernels a coupling uses."""
    desc = _convnet_desc(net)

    def build(mode):
        steps = convnet_steps(mode, desc, *desc["first"], *desc["last"])
        steps[-1].final = True
        return steps
    return _run_net(x, mode, _convnet_weights(desc), build)
