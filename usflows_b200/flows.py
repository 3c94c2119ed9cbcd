"""`Flow` and `USFlow` -- drop-in mirrors of the reference's model API (src/usflows/flows.py:22-605).

Same constructor signatures, attributes (`layers`, `trainable_layers`, `base_distribution`, `device`,
`export`), state-dict layout and methods (`log_prob`, `sample`, `_forward`, `backward`, `forward`, `to`,
`is_feasible`, `add_jitter`, `log_prior`).  Evaluation runs through `engine.Program`: fused sm_100a kernels
behind the C ABI, prepared weights cached per weight version, the total log|det J| (a model constant for
every USFlow layer, SURVEY section 0.4) computed once per weight version.  CUDA tensors only.
"""
from __future__ import annotations

import math
import threading
from typing import Any, Dict, Iterable, List, Literal, Optional, Type

import torch

from . import engine, image_engine, ops
from .distributions import DistributionModule, Independent, _FrozenBase
from .transforms import MaskedAffineCoupling
from .transforms import (BaseTransform, Bijective1x1Conv2d, BlockAffineTransform, HouseholderTransform, InverseTransform, LUTransform,
                         MaskedCoupling, ScaleTransform, SequentialAffineTransform)


SMALL_BATCH_GRAPH_ROWS = 4096   # `log_prob` on at most this many rows replays one captured CUDA graph (0 = off)
SMALL_BATCH_GRAPH_IMAGES = 1024 # the same for image-shaped events (one chunk; ~15 us of host time per launch otherwise)
USE_C_PLAN = True             # device-resident `log_prob` / `backward` / `_forward`: ONE C call per chunk (usf_flow_logprob /
                              # usf_flow_apply on a library-owned plan) where the program is contractions only
HOST_CUDA_GRAPHS = True       # `log_prob_host`: replay one captured CUDA graph per full-size chunk
HOST_CHUNK_ROWS = 16384      # rows per H2D copy / kernel batch of `log_prob_host` (copy i+1 overlaps compute i)
HOST_CHUNK_UNITS = (1, 1, 2, 3)   # `log_prob_host` chunk sizes in wave-aligned units (the last entry repeats).  Only the first
                             # copy is exposed, later chunks may grow as fast as the copy stays ahead of the kernels: a C2
                             # row copies 1.4x faster than it computes, so chunk k may hold ~1.4x the rows of chunk k-1.
                             # Measured on C2 (65 536 rows, B200): uniform 7.11 ms, (1, 2, 2, ..) 6.68 ms, (1, 2, 4, ..) 7.0 ms
HOST_STAGE_BYTES = 1 << 30   # the whole batch is staged on the device when it fits (copies run back to back); else a 2-buffer ring
HOST_MAX_STAGE_SLICES = 8    # ... and when it needs at most this many chunks (one captured graph + result buffer per slice)


_capture_lock = threading.Lock()     # one graph capture at a time per process (the launch-mode switch below is global)
_capture_streams: Dict[int, Any] = {}


def capture_stream(device) -> "torch.cuda.Stream":
    """The side stream graph captures of `device` run on.  torch.cuda.graph's default is ONE process-wide stream created on
    whichever device captured first; a capture for another device would then launch on the wrong device (peer access, or an
    illegal address), which is what the row-shard driver (parallel.py) hit with two GPUs in one process."""
    device = torch.device(device)
    idx = device.index if device.index is not None else torch.cuda.current_device()
    s = _capture_streams.get(idx)
    if s is None:
        s = _capture_streams[idx] = torch.cuda.Stream(device=idx)
    return s


class _plain_stream_order:
    """Kernels captured into a CUDA graph are launched without programmatic dependent launch: inside a graph the
    programmatic edges bought nothing and cost 4% on the chunked host path (measured); on a plain stream they hide the
    launch latency and the next kernel's prologue (-1.7% per step).  Holds the process-wide capture lock: the row-shard
    driver (parallel.py) warms several devices up from several threads.

    Also keeps the cyclic garbage collector off for the duration of the capture: a collection that starts inside it may
    finalise CUDA graphs and plans of an earlier weight version, and `cudaGraphExecDestroy` / `cudaFree` issued by the
    capturing thread invalidate a thread-local capture ("operation not permitted when stream is capturing"; torch >= 2.9
    no longer collects before a capture by itself).  The garbage is collected after the capture instead."""

    def __enter__(self):
        import gc
        from . import _lib
        _capture_lock.acquire()
        self._gc_was_on = gc.isenabled()
        gc.disable()
        _lib.check(_lib.load().usf_debug_set_pdl(0))

    def __exit__(self, *exc):
        import gc
        from . import _lib
        try:
            _lib.check(_lib.load().usf_debug_set_pdl(1))
        finally:
            if self._gc_was_on:
                gc.enable()
            _capture_lock.release()
        return False


def _capture(dev, body) -> "torch.cuda.CUDAGraph":
    """`body()` captured into a CUDA graph on `dev`, after one eager pass that sizes every workspace buffer it uses."""
    body()
    torch.cuda.synchronize(dev)
    graph = torch.cuda.CUDAGraph()
    with _plain_stream_order(), torch.cuda.graph(graph, stream=capture_stream(dev), capture_error_mode="thread_local"):
        body()
    return graph


def _wave_aligned_chunk_rows(prog, device) -> int:
    """Rows per H2D copy / kernel batch of `log_prob_host`: the smallest multiple of 256-row tile rows >= HOST_CHUNK_ROWS / 2
    for which the widest layer's tile count is a whole number of waves of the persistent CTA-pair kernel (one tile per
    SM pair and wave).  A small first copy keeps the pipeline fill short (the copy of chunk i+1 hides under the kernels
    of chunk i); whole waves keep the tail of every launch full."""
    import ctypes
    from . import _lib
    if prog.small is not None:                                   # one launch per chunk: copy granularity only
        return max(HOST_CHUNK_ROWS, (32 << 20) // (4 * prog.small["d"]))
    widest = max([st.N for st in prog.steps if st.kind == "mm"] or [0])
    if widest < 32:
        return HOST_CHUNK_ROWS
    sm = ctypes.c_int(0)
    _lib.check(_lib.load().usf_device_info(ctypes.byref(sm), None, None, None))
    pairs = max(1, sm.value // 2)
    n_blocks = -(-widest // 256) if widest % 256 == 0 else -(-widest // 208)
    unit = pairs // math.gcd(pairs, n_blocks)                 # tile rows (of 256 rows) per whole number of waves
    k = max(1, -(-(HOST_CHUNK_ROWS // 2) // (256 * unit)))
    return 256 * unit * k


def _uniform_bounds(n: int, step: int):
    """Chunks of `step` rows from the start; the last one takes the rest."""
    return [(r0, min(n, r0 + step)) for r0 in range(0, n, step)]


def growing_bounds(n: int, unit: int, units):
    """Chunks of `log_prob_host`: `units` (the last entry repeats) in multiples of `unit` rows from the start.  Its H2D copy
    of chunk i+1 hides under the kernels of chunk i (a row copies faster than it computes), so only the FIRST copy is
    exposed: start with the smallest wave-aligned chunk and let the later ones grow (fewer kernel boundaries, fuller
    tails).  Fewer than unit // 2 rows left join the last chunk instead of making a launch sequence of their own."""
    bounds, r0 = [], 0
    while r0 < n:
        take = min(unit * units[min(len(bounds), len(units) - 1)], n - r0)
        if n - r0 - take < unit // 2:
            take = n - r0
        bounds.append((r0, r0 + take))
        r0 += take
    return bounds


def sample_host_bounds(n: int, unit: int, uniform: bool = False):
    """Chunks of `sample_host`.  There the LAST device-to-host copy is the exposed one, so the chunks are those of
    `log_prob_host` mirrored: they shrink towards the end, and the first chunk takes the remainder.  `uniform`: chunks of
    `unit` rows from the start."""
    if uniform:
        return _uniform_bounds(n, unit)
    return [(n - r1, n - r0) for r0, r1 in reversed(growing_bounds(n, unit, HOST_CHUNK_UNITS))]


def _cached_graph(prog, key, build) -> dict:
    """The graph entry of `key` = (route, slot, staging buffer data_ptr, rows, variant) from `build()` (the graph, its range
    `flag` and the buffers a replay uses), unless one captured since the last workspace reallocation (`gen`) is cached.  On
    insert, stale entries and those of the same (route, slot, variant) over another buffer go; at most 8 stay per (route,
    slot).  The cache lives ON the Program (one per weight version and mode): graphs point into its operand planes and die
    with it instead of surviving under a recycled id()."""
    cache = prog.__dict__.setdefault("_graphs", {})
    ent = cache.get(key)
    if ent is not None and ent["gen"] == engine._workspace.generation:
        return ent
    ent = build()
    ent["gen"] = engine._workspace.generation
    for k in [k for k, e in cache.items() if e["gen"] != ent["gen"] or (k[:2] == key[:2] and k[4] == key[4] and k[2] != key[2])]:
        del cache[k]
    while sum(1 for k in cache if k[:2] == key[:2]) >= 8:        # a few row counts per staging slot; drop the oldest
        del cache[next(k for k in cache if k[:2] == key[:2])]
    cache[key] = ent
    return ent


def _capture_chunks(bounds, n_slots: int, unit: int, capture) -> dict:
    """{(slot, rows): capture(slot, rows)} for every chunk i of `bounds` of at least unit // 2 rows, with slot = i % n_slots.
    Largest first, so that the shared workspaces are sized once; a second pass recaptures what a workspace that grew
    meanwhile invalidated.  The flags are zeroed at the end: the eager pass of a capture may have set them."""
    sizes = [r1 - r0 for r0, r1 in bounds]
    graphs = {}
    for _ in range(2):
        for i in sorted(range(len(sizes)), key=lambda j: -sizes[j]):
            if sizes[i] >= unit // 2:
                graphs[(i % n_slots, sizes[i])] = capture(i % n_slots, sizes[i])
        if all(g["gen"] == engine._workspace.generation for g in graphs.values()):
            break
    for g in graphs.values():
        if g["flag"] is not None:
            g["flag"].zero_()
    return graphs


class Flow(torch.nn.Module):
    """Base flow: a list of bijective layers over a base distribution (flows.py:22-292)."""

    export_modes = Literal["log_prob", "sample", "forward", "backward"]
    export: str = "log_prob"
    device = "cpu"
    _context_needs_soft_training = False

    def __init__(self, base_distribution, layers, soft_training: bool = False, training_noise_prior=None,
                 device: str = "cpu", precision: Optional[str] = None, *args, **kwargs) -> None:
        super().__init__(*args, **kwargs)
        if training_noise_prior is None:                           # flows.py:79-80
            training_noise_prior = torch.distributions.Uniform(0, 1e-6)
        self.soft_training = soft_training
        self.training_noise_prior = training_noise_prior
        self.layers = layers
        self.trainable_layers = torch.nn.ModuleList([l for l in layers if isinstance(l, torch.nn.Module)])
        if isinstance(base_distribution, torch.distributions.Distribution):      # a plain torch Laplace / Normal object
            base_distribution = _FrozenBase(base_distribution)
        self.base_distribution = base_distribution
        # ConditionalDenseNN conditioners tell "no context" (its context layer is skipped: `backward` / `_forward`,
        # flows.py:45-67) from the zero context that a soft-training USFlow substitutes in `log_prob` / `sample`
        # (flows.py:559-565, 580-590: the context layer's bias stays) -- two launch programs per direction
        self._cond_dense_nets = []
        self._layer_route = False             # a conditioner without a fused lowering (networks.BottleneckConv)
        for l in layers:
            while isinstance(l, InverseTransform):
                l = l.transform
            if isinstance(l, MaskedCoupling) and hasattr(l.conditioner, "zero_context_default"):
                self._cond_dense_nets.append(l.conditioner)
            if isinstance(l, MaskedCoupling) and getattr(l.conditioner, "layer_route_only", False):
                self._layer_route = True
        self._zero_ctx = bool(soft_training and self._context_needs_soft_training)
        self.precision = precision
        self.to(device)
        self.device = device
        batch_shape = self.base_distribution.batch_shape
        if len(batch_shape) > 0:                                   # flows.py:97-101
            self.base_distribution = Independent(self.base_distribution, len(batch_shape))
        self._programs: Dict[str, Any] = {}
        ev = tuple(self._event_shape())
        if len(ev) == 3:                    # a Bijective1x1Conv2d's log|det| counts the pixels of the event (its own
            for l in layers:                # forward sees them on the tensor; the launch program needs them up front)
                while isinstance(l, InverseTransform):
                    l = l.transform
                if isinstance(l, Bijective1x1Conv2d) and l.n_blocks is None:
                    l.n_blocks = ev[1] * ev[2]

    # -- reference API ---------------------------------------------------------------------------
    def simplify(self) -> "Flow":
        """The same flow with every LU / Householder / sequential affine layer replaced by its plain matrix form
        (`PlaneBijectiveLinearTransform`, `Bijective1x1Conv2d` for image-shaped events): flows.py:600-606.  The result
        stays on this flow's device and keeps its precision mode (the reference's lands on its default device)."""
        return Flow(self.base_distribution, [l.simplify() for l in self.layers], device=self.device,
                    precision=self.precision)

    def forward(self, x: torch.Tensor):
        """Export-mode dispatch (flows.py:30-43)."""
        if self.export == "log_prob":
            return self.log_prob(x)
        if self.export == "sample":
            return self.sample()
        if self.export == "forward":
            return self._forward(x)
        if self.export == "backward":
            return self.backward(x)
        raise ValueError(f"Unknown export mode {self.export}")

    def reference_module(self, export_mode: str = "log_prob") -> torch.nn.Module:
        """Frozen pure-PyTorch module with the reference's semantics of this flow (for ONNX export / inspection on any
        device; never used by `log_prob` / `sample`, which run on the CUDA kernels only)."""
        from .export import ReferenceSemantics
        return ReferenceSemantics(self, export_mode)

    def to_onnx(self, path: str, export_mode: str = "log_prob", **export_kwargs) -> None:
        """Saves the model as an ONNX file (flows.py:212-223); `export_mode` as `Flow.export`."""
        from .export import to_onnx
        to_onnx(self, path, export_mode, **export_kwargs)

    def _forward(self, x: torch.Tensor) -> torch.Tensor:
        """latent -> data through every layer's `forward` (flows.py:45-55)."""
        return self._run("forward", x)

    def backward(self, x: torch.Tensor) -> torch.Tensor:
        """data -> latent through every layer's `backward` in reverse order (flows.py:57-67)."""
        return self._run("backward", x)

    def log_prob(self, x: torch.Tensor, context: Optional[torch.Tensor] = None, *, dequantize: Optional[str] = None,
                 seed: Optional[int] = None) -> torch.Tensor:
        """log p(x) = base.log_prob(z) - sum_k log|det J_k|  (flows.py:225-245).

        With `dequantize` ("uniform" or "midpoint"), x is a uint8 batch [*batch, *event] of 8-bit values that the first kernel
        reading it dequantises, exactly as `usflows_b200.dequantize(x.reshape(-1, *event), dequantize, seed)` would (the
        reference's DequantizedDataset for "uniform"); `seed=None` draws a fresh seed from torch.default_generator."""
        return self._log_prob_any(x, context, ops.dequant_spec(x, dequantize, seed))

    def _log_prob_any(self, x: torch.Tensor, context, dq: Optional[ops.Dequant]) -> torch.Tensor:
        if self.soft_training:
            self._require_conditional()
        elif self._context_needs_soft_training:
            context = None                    # USFlow.log_prob drops the context unless soft_training (flows.py:559-567)
        if context is not None or self._layer_route:
            if dq is not None:                # the layer-by-layer route reads fp32
                x2, _ = engine._flatten_rows(x, len(self._event_shape()), torch.uint8)
                with ops.on_device(x):
                    x = engine._dequantized(x2.contiguous(), dq).reshape(x.shape)
            return self._with_context("log_prob", x, context)
        with ops.on_device(x):                # no context = context 0 (flows.py:559-565): the conditional conditioners
            return self._log_prob(x, dq)      # are lowered without their context input, which is exact

    def _require_conditional(self) -> None:
        """Soft training hands a context to every coupling's conditioner (transforms.py:284-289), which only the
        conditional networks accept: the reference fails with a TypeError on the first call otherwise (SURVEY Q6)."""
        for l in self.layers:
            while isinstance(l, InverseTransform):
                l = l.transform
            if isinstance(l, MaskedCoupling) and not getattr(l.conditioner, "context_channels", 0):
                raise TypeError(f"soft_training passes a context to the conditioner; {type(l.conditioner).__name__} takes "
                                "none (use ConditionalDenseNN / CondConvNet / CondConvNet2D)")

    def _with_context(self, what: str, x: torch.Tensor, context: torch.Tensor) -> torch.Tensor:
        """Evaluation with an explicit context (flows.py:235-238, 257-263): the context channel of the conditional
        conditioners is data, so this runs the layer-by-layer route of the training pass (training.py: every contraction
        on the library's kernels, no gradient bookkeeping)."""
        from . import training
        ops.require_cuda(x, "input")
        ev = len(self._event_shape())
        batch_shape = x.shape[:x.dim() - ev]
        x2 = x.reshape(-1, *x.shape[x.dim() - ev:])
        if context is not None:
            context = torch.as_tensor(context, dtype=torch.float32, device=x.device)
        with torch.no_grad(), ops.on_device(x):
            if what == "log_prob":
                return training.log_prob_autograd(self, x2, context).reshape(batch_shape)
            return training.apply_autograd(self, x2, what, context).reshape(*batch_shape, *x2.shape[1:])

    def _log_prob(self, x: torch.Tensor, dq: Optional[ops.Dequant] = None) -> torch.Tensor:
        """`dq`: x is uint8 (ops.Dequant); every route below reaches the same result as on the dequantised fp32 rows."""
        prog, ladj = self._program("backward", self._zero_ctx)
        base = self._base_module()
        base._prepared()                  # parameter-side work happens here, outside any graph capture
        x2, batch_shape = engine._flatten_rows(x, len(self._event_shape()), torch.float32 if dq is None else torch.uint8)
        if dq is not None:
            x2 = x2.contiguous()
        rows, d = x2.shape
        images = isinstance(prog, image_engine.ImageProgram)
        perm = self._channels_last_perm(x2.device) if images else None      # image-shaped events: the latent is channels-last
        if x2.is_cuda and 0 < rows <= (SMALL_BATCH_GRAPH_IMAGES if images else SMALL_BATCH_GRAPH_ROWS) and prog.small is None \
                and not prog.force_fallback and not prog.has_row_ladj and not torch.cuda.is_current_stream_capturing():
            lp = self._log_prob_small_batch(prog, ladj, x2 if dq is None else engine._dequantized(x2, dq), perm)
            if lp is not None:
                return lp.reshape(batch_shape)
        if USE_C_PLAN and x2.is_cuda and rows > 0 and prog.plan_able() and getattr(base, "base_kind", -1) >= 0 \
                and not torch.cuda.is_current_stream_capturing():
            return self._log_prob_plan(prog, base, ladj, x2, dq).reshape(batch_shape)
        out = torch.empty(rows, dtype=torch.float32, device=x2.device)
        # affine couplings: per-row log-determinants next to the model constant
        row_ladj = torch.zeros(rows, dtype=torch.float32, device=x2.device) if prog.has_row_ladj else None
        with torch.no_grad():
            prog.run(x2, sink=lambda z, r0, r1: base._density_into(ops.Act(r1 - r0, d, f32=z), -ladj, out[r0:r1], perm=perm),
                     ladj_rows=row_ladj, dq=dq)
            if row_ladj is not None and rows:
                ops.sub_rows(out, row_ladj)
        return out.reshape(batch_shape)

    @staticmethod
    def _plan_chunks(rows: int):
        """(chunk bounds, plan capacity) as `Program.run` would cut the batch; the capacity is rounded up so that a few plans
        serve every batch size."""
        cap = engine._default_chunk_rows
        bounds = engine.chunk_bounds(rows, cap)
        chunk = bounds[0][1]
        size = 4096
        while size < chunk:
            size *= 2
        return bounds, min(size, max(cap, chunk))

    def _log_prob_plan(self, prog, base, ladj: float, x2: torch.Tensor, dq: Optional[ops.Dequant] = None) -> torch.Tensor:
        """`log_prob` through the whole-stack C entry: one `usf_flow_logprob` call per chunk (ingest, every contraction and
        the base density are launched by the library).  Same kernels, same order, same bits as the launch-by-launch route."""
        rows, d = x2.shape
        x2 = x2.contiguous()
        bounds, capacity = self._plan_chunks(rows)
        shifted = lambda r0: None if dq is None else dq.shifted(r0)        # noqa: E731
        with torch.no_grad():
            plan = prog.c_plan(d, capacity, base, -ladj)
            out = torch.empty(rows, dtype=torch.float32, device=x2.device)
            engine.run_chunks(
                bounds, x2.device, prog.uses_range_flag,
                lambda i, r0, r1, flag: plan.log_prob(x2[r0:r1], out[r0:r1], flag, shifted(r0)),
                lambda i, r0, r1: prog._fallback().run(x2[r0:r1], sink=lambda z, a, b: base._density_into(
                    ops.Act(b - a, z.shape[1], f32=z), -ladj, out[r0 + a:r0 + b]), dq=shifted(r0)))
        return out

    def _log_prob_small_batch(self, prog, ladj: float, x2: torch.Tensor, perm: Optional[torch.Tensor]):
        """Small batches are bound by the host-side cost of ~23 kernel launches (~40 us each through ctypes + tensor-map
        encoding), not by the kernels: the launch program + base density of a given row count is captured ONCE into a CUDA
        graph over fixed staging buffers and replayed (input copied in, result cloned out).  Returns None when a value
        left the fp16 range (the caller then takes the launch-by-launch route, which handles the tf32-split re-run)."""
        rows, d = x2.shape
        dev = x2.device

        def build():
            base = self._base_module()
            base._prepared()                  # parameter-side work happens here, outside any graph capture
            xin = torch.empty(rows, d, dtype=torch.float32, device=dev)
            out = torch.empty(rows, dtype=torch.float32, device=dev)
            flag = torch.zeros(1, dtype=torch.int32, device=dev) if prog.uses_range_flag else None
            fin = prog.final_buffer(dev, "final_small", rows, d)

            def body():
                prog._run_chunk(xin, fin, flag)
                base._density_into(ops.Act(rows, fin.shape[1], f32=fin), -ladj, out, perm=perm)
            xin.copy_(x2)
            return dict(graph=_capture(dev, body), x=xin, out=out, flag=flag)
        with torch.no_grad():
            ent = _cached_graph(prog, ("small", None, None, rows, None), build)
            ent["x"].copy_(x2)
            if ent["flag"] is not None:
                ent["flag"].zero_()
            ent["graph"].replay()
            if ent["flag"] is not None and int(ent["flag"].item()) != 0:
                return None
            return ent["out"].clone()

    def _staging(self, name: str, rows: int, width: int, dtype: torch.dtype, dev) -> torch.Tensor:
        """The device buffer [>= rows, width] this flow keeps for `name` and `dtype` (fp32 and 8-bit calls in turn keep their
        own buffers, and the graphs captured over them); reallocated when it has too few rows, another width or device."""
        bufs = self.__dict__.setdefault("_stage", {})
        buf = bufs.get((name, dtype))
        if buf is None or buf.shape[0] < rows or buf.shape[1] != width or buf.device != dev:
            buf = bufs[(name, dtype)] = torch.empty(rows, width, dtype=dtype, device=dev)
        return buf

    def _side_stream(self, dev) -> "torch.cuda.Stream":
        """The stream the host copies of `log_prob_host` / `sample_host` run on, under the kernels of the next chunk."""
        s = self.__dict__.get("_side")
        if s is None or s.device != dev:
            s = self._side = torch.cuda.Stream(device=dev)
        return s

    def log_prob_host(self, x_host: torch.Tensor, out_host: Optional[torch.Tensor] = None,
                      chunk_rows: Optional[int] = None, *, dequantize: Optional[str] = None, seed: Optional[int] = None,
                      row_offset: int = 0) -> torch.Tensor:
        """`log_prob` for rows living in HOST memory (pinned for full copy speed): the batch is streamed
        through the device in chunks -- H2D copy of chunk i+1 on a side stream overlaps the kernels of
        chunk i -- and the log-probs are copied back into `out_host`.  Returns `out_host`.

        With `dequantize` (see `log_prob`), x_host is a uint8 batch: a quarter of the bytes cross to the device, and the
        ingest kernels dequantise.  Row r of x_host is global row `row_offset + r` of the noise (a caller that splits one
        batch over several calls passes each part's offset and one seed to get the noise of a single call)."""
        if x_host.is_cuda:
            raise RuntimeError("log_prob_host expects a host tensor; use log_prob for device tensors")
        dq = ops.dequant_spec(x_host, dequantize, seed, row_offset)
        with ops.on_device(next(self.parameters())):
            return self._log_prob_host(x_host, out_host, chunk_rows, dq)

    def _log_prob_host(self, x_host, out_host, chunk_rows, dq: Optional[ops.Dequant] = None):
        dev = next(self.parameters()).device
        if self._layer_route:                 # no launch program to overlap the copies with: plain chunks
            out = torch.empty(x_host.shape[0], dtype=torch.float32) if out_host is None else out_host
            step = max(1, chunk_rows or 8192)
            for r0 in range(0, x_host.shape[0], step):
                out[r0:r0 + step].copy_(self._log_prob_any(x_host[r0:r0 + step].to(dev), None,
                                                           None if dq is None else dq.shifted(r0)))
            return out
        prog, ladj = self._program("backward", self._zero_ctx)
        prog = prog._fallback() if prog.force_fallback else prog
        base = self._base_module()
        base._prepared()                  # parameter-side work happens here, outside any graph capture
        x2 = x_host.reshape(-1, math.prod(self._event_shape()))
        rows, d = x2.shape
        if out_host is None:
            out_host = torch.empty(rows, dtype=torch.float32, pin_memory=True)
        sdt = torch.float32 if dq is None else torch.uint8      # 8-bit rows are staged as they are (a quarter of the bytes)
        images = len(self._event_shape()) == 3
        if images:
            # image-shaped events: uniform chunks in two staging buffers in turn, each through `_log_prob` (whose routes
            # guard their own chunks); the H2D copy of chunk i + 1 is issued before chunk i is enqueued
            bounds = _uniform_bounds(rows, max(1, chunk_rows or HOST_CHUNK_ROWS))
            whole, ahead = False, 1
        else:
            # an explicit `chunk_rows` gives uniform chunks
            unit = min(chunk_rows or _wave_aligned_chunk_rows(prog, dev), max(rows, 1))
            bounds = growing_bounds(rows, unit, (1,) if chunk_rows else HOST_CHUNK_UNITS)
            # staging: one device buffer per chunk (slices of one allocation holding the whole batch) when that fits -- the
            # copies then run back to back on the copy stream, independent of the kernels --, else two buffers used in turn
            whole = rows * d * sdt.itemsize <= HOST_STAGE_BYTES and len(bounds) <= HOST_MAX_STAGE_SLICES
            ahead = 0
        chunk = max([r1 - r0 for r0, r1 in bounds], default=1)
        stage = self._staging("host", max(rows, 1) if whole else 2 * chunk, d, sdt, dev)
        if whole:
            bufs = [stage[r0:r1] for r0, r1 in bounds] or [stage[:0]]
        else:
            bufs = [stage[:chunk], stage[chunk:2 * chunk]]
        n_buf = len(bufs)
        out_dev = self._staging("out", rows, 1, torch.float32, dev).view(-1)[:rows]
        side = self._side_stream(dev)
        main = torch.cuda.current_stream(dev)
        copied = [torch.cuda.Event() for _ in range(n_buf)]
        consumed = [torch.cuda.Event() for _ in range(n_buf)]
        guarded = not images and prog.guarded
        row_ladj = torch.zeros(rows, dtype=torch.float32, device=dev) if prog.has_row_ladj else None
        lr = lambda r0, r1: None if row_ladj is None else row_ladj[r0:r1]     # noqa: E731
        shifted = lambda r0: None if dq is None else dq.shifted(r0)           # noqa: E731

        def sink_at(r0):
            return lambda z, a, b: base._density_into(ops.Act(b - a, d, f32=z), -ladj, out_dev[r0 + a:r0 + b])

        def issue_copy(i):
            r0, r1 = bounds[i]
            slot = i % n_buf
            with torch.cuda.stream(side):
                if i >= n_buf:
                    side.wait_event(consumed[slot])
                bufs[slot][:r1 - r0].copy_(x2[r0:r1], non_blocking=True)
                copied[slot].record(side)

        def capture(slot, size):
            """The launch program of one chunk reading staging buffer `slot`.  With `dq`, the buffer holds 8-bit rows; the
            graph reads their {seed, global row} from its `params` tensor, written before every replay."""
            buf = bufs[slot][:size]

            def build():
                flag = torch.zeros(1, dtype=torch.int32, device=dev) if prog.uses_range_flag else None
                fin = prog.final_buffer(dev, f"final_host{slot}", size, d)
                params = None if dq is None else torch.zeros(2, dtype=torch.int64, device=dev)
                dqg = None if dq is None else ops.Dequant(dq.mode, 0, 0, params)
                return dict(graph=_capture(dev, lambda: prog._run_chunk(buf, fin, flag, dqg)), fin=fin, flag=flag, params=params)
            return _cached_graph(prog, ("host", slot, buf.data_ptr(), size, None if dq is None else dq.mode), build)

        def first(i, r0, r1, flag):
            if i + ahead < len(bounds):
                issue_copy(i + ahead)
            slot = i % n_buf
            buf = bufs[slot][:r1 - r0]
            g = graphs.get((slot, r1 - r0))
            main.wait_event(copied[slot])
            if images:
                out_dev[r0:r1] = self._log_prob(buf.reshape(r1 - r0, *self._event_shape()), shifted(r0))
            elif g is not None:
                # one graph launch replaces the ~23 kernel launches of the chunk: the host-side launch cost
                # (~40 us per launch through ctypes + tensor-map encoding) is what bounds small chunks otherwise
                if g["params"] is not None:
                    g["params"].copy_(params[i])
                g["graph"].replay()
                sink_at(r0)(g["fin"], 0, r1 - r0)
            elif guarded:
                fin = prog.final_buffer(dev, "final", r1 - r0, d)
                prog._run_chunk(buf, fin, flag, shifted(r0), ladj_rows=lr(r0, r1))
                sink_at(r0)(fin, 0, r1 - r0)
            else:
                prog.run(buf, chunk_rows=chunk, sink=sink_at(r0), ladj_rows=lr(r0, r1), dq=shifted(r0))
            consumed[slot].record(main)

        def again(i, r0, r1):
            buf = bufs[i % n_buf][:r1 - r0]
            if n_buf < len(bounds):                       # staging buffers in turn: the slot may hold another chunk's rows
                buf.copy_(x2[r0:r1])
            prog._fallback().run(buf, chunk_rows=chunk, sink=sink_at(r0), ladj_rows=lr(r0, r1), dq=shifted(r0))

        with torch.no_grad():
            graphs = {}
            if not images and HOST_CUDA_GRAPHS and rows >= unit and prog.small is None and not prog.has_row_ladj:
                graphs = _capture_chunks(bounds, n_buf, unit, capture)
            if graphs and dq is not None:                 # {seed, global row} of every chunk, read by the graphs' ingest
                params = torch.tensor([[dq.seed, dq.row0 + r0] for r0, _ in bounds], dtype=torch.int64).to(dev)
            side.wait_stream(main)
            if ahead and bounds:
                issue_copy(0)
            # a graph's flag is not per chunk: when one is set, every chunk is recomputed
            engine.run_chunks(bounds, dev, guarded, first, again, shared_flags=[g["flag"] for g in graphs.values()],
                              ladj_rows=row_ladj)
            if row_ladj is not None and rows:
                ops.sub_rows(out_dev, row_ladj)
            out_host.reshape(-1)[:rows].copy_(out_dev, non_blocking=True)
            main.synchronize()
        return out_host

    def sample(self, sample_shape: Iterable[int] = None, context: Optional[torch.Tensor] = None, *, seed: Optional[int] = None,
               quantize: bool = False) -> torch.Tensor:
        """Draw from the base and push through the layers (flows.py:247-265).

        With `seed`, the base draws are keyed by (seed, global row) alone (ops.Draw): the result does not depend on
        `torch.manual_seed`, and row r equals row r of `sample_host(n, seed=seed)`.  With `quantize`, the result is uint8
        `[*sample_shape, *event]`: the 8-bit pixels `usflows_b200.quantize` makes of the samples."""
        if sample_shape is None:
            sample_shape = [1]
        shape = [int(s) for s in sample_shape]
        with ops.on_device(next(self.parameters())):
            ev = len(self._event_shape())
            if seed is None:
                z = self.base_distribution.sample(shape)
                z = z.reshape(-1, *z.shape[z.dim() - ev:])
            else:
                rows = math.prod(shape)
                z = self._draw(rows, ops.Draw(int(seed))).reshape(rows, *self._event_shape())
            y = self._run("forward", z, self._zero_ctx) if context is None else self._with_context("forward", z, context)
            if quantize:
                y = ops.quantize(y)
        return y.reshape(*shape, *y.shape[1:])

    def _draw(self, rows: int, draw: ops.Draw, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Base draws [rows, d] of the global rows draw.row0 .. draw.row0 + rows - 1, into `out` when given."""
        if out is None:
            out = torch.empty(rows, math.prod(self._event_shape()), dtype=torch.float32, device=next(self.parameters()).device)
        if rows:
            with torch.no_grad():
                self._base_module()._sample_into(out, draw)
        return out

    def sample_host(self, n: int, out_host: Optional[torch.Tensor] = None, *, seed: Optional[int] = None,
                    quantize: bool = False, row_offset: int = 0, chunk_rows: Optional[int] = None) -> torch.Tensor:
        """`n` samples [n, *event] streamed into HOST memory (`out_host`, allocated pinned when None) in chunks, returned.
        The device holds two chunks of output whatever `n` is, and the device-to-host copy of chunk i runs on a side stream
        under the kernels of the next chunk.  Row r is global row `row_offset + r` of the stream of `seed` (the rows
        `sample(seed=seed)` draws from 0 on), so a caller that splits one draw over several calls or devices passes each
        part's offset and one seed; `seed=None` draws one from torch.default_generator.  With `quantize`, the result is
        uint8 pixels (see `sample`): a quarter of the bytes cross to the host.  `chunk_rows` gives uniform chunks."""
        n, row_offset = int(n), int(row_offset)
        if n < 0 or row_offset < 0:
            raise ValueError(f"usflows_b200: sample_host needs n >= 0 and row_offset >= 0, got {n}, {row_offset}")
        ev = tuple(self._event_shape())
        dtype = torch.uint8 if quantize else torch.float32
        if out_host is None:
            out_host = torch.empty(n, *ev, dtype=dtype, pin_memory=torch.cuda.is_available())
        elif out_host.is_cuda:
            raise RuntimeError("sample_host writes host memory; use sample for device tensors")
        elif out_host.dtype != dtype or tuple(out_host.shape) != (n, *ev) or not out_host.is_contiguous():
            raise ValueError(f"usflows_b200: out_host must be a contiguous {dtype} tensor of shape {(n, *ev)}, got "
                             f"{out_host.dtype} {tuple(out_host.shape)}")
        draw = ops.Draw(ops.draw_seed() if seed is None else int(seed), row_offset)
        if n:
            with ops.on_device(next(self.parameters())), torch.no_grad():
                self._sample_host(out_host.view(n, -1), draw, quantize, chunk_rows)
        return out_host

    def _sample_host(self, flat: torch.Tensor, draw: ops.Draw, quantize: bool, chunk_rows: Optional[int]) -> None:
        dev = next(self.parameters()).device
        cuda = dev.type == "cuda"
        n, d = flat.shape
        base = self._base_module()
        base._prepared()                  # parameter-side work happens here, outside any graph capture
        prog = None if self._layer_route else self._program("forward", self._zero_ctx)[0]
        if prog is not None and prog.force_fallback:
            prog = prog._fallback()
        images = isinstance(prog, image_engine.ImageProgram)
        launch = prog is not None and not images and prog.small is None       # the flat launch program, chunk by chunk
        if launch:
            unit = min(chunk_rows or _wave_aligned_chunk_rows(prog, dev), n)
            bounds = sample_host_bounds(n, unit, uniform=bool(chunk_rows))
        else:                             # images: eager chunks; single-launch and layer-route flows: plain chunks
            bounds = _uniform_bounds(n, chunk_rows or (prog._chunk_bounds(n, None)[0][1] if images else HOST_CHUNK_ROWS))
        chunk = max(r1 - r0 for r0, r1 in bounds)
        # two output buffers used in turn; fp32 and uint8 calls in turn keep their own buffers and captured graphs
        stage = self._staging("sample", 2 * chunk, d, flat.dtype, dev)
        half = stage.shape[0] // 2
        bufs = [stage[:half], stage[half:2 * half]]
        main = torch.cuda.current_stream(dev) if cuda else None
        side = self._side_stream(dev) if cuda else None
        ready = [torch.cuda.Event() for _ in range(2)] if cuda else None
        copied = [torch.cuda.Event() for _ in range(2)] if cuda else None
        issued = [0]

        def emit(r0, r1, run):
            """run(buf) fills an output buffer with rows [r0, r1); its D2H copy follows on the side stream, and the buffer's
            next use waits for that copy."""
            slot = issued[0] % 2
            issued[0] += 1
            buf = bufs[slot][:r1 - r0]
            if not cuda:
                run(buf)
                flat[r0:r1].copy_(buf)
                return
            main.wait_event(copied[slot])
            run(buf)
            ready[slot].record(main)
            with torch.cuda.stream(side):
                side.wait_event(ready[slot])
                flat[r0:r1].copy_(buf, non_blocking=True)
                copied[slot].record(side)

        def compute(p, buf, r0, r1, flag):
            rows, dr = r1 - r0, draw.shifted(r0)
            if p is None or p.small is not None:          # what `sample` runs
                z = self._draw(rows, dr).reshape(rows, *self._event_shape())
                y = self._run("forward", z, self._zero_ctx).reshape(rows, d)
                if quantize:
                    ops.quantize_u8(y, buf)
                else:
                    buf.copy_(y)
                return
            z = engine._workspace.planes(dev, "sample_z", 1, rows * d, "f32").view(rows, d)
            base._sample_into(z, dr)
            if images:
                p._run_chunk(z, buf, flag, nchw_out=True, quantize=quantize)
                return
            fin = p.final_buffer(dev, "final_q", rows, d) if quantize else buf
            p._run_chunk(z, fin, flag)
            if quantize:
                ops.quantize_u8(fin, buf)

        def capture(slot, rows):
            """One chunk writing output buffer `slot`: the base draws at the {seed, row base} read from its `params` tensor
            (written before every replay), the launch program, the quantisation."""
            buf = bufs[slot][:rows]

            def build():
                flag = torch.zeros(1, dtype=torch.int32, device=dev) if prog.uses_range_flag else None
                params = torch.zeros(2, dtype=torch.int64, device=dev)
                z = engine._workspace.planes(dev, f"sample_z{slot}", 1, rows * d, "f32").view(rows, d)
                fin = prog.final_buffer(dev, f"final_q{slot}", rows, d) if quantize else buf
                dr = ops.Draw(0, 0, params)

                def body():
                    base._sample_into(z, dr)
                    prog._run_chunk(z, fin, flag)
                    if quantize:
                        ops.quantize_u8(fin, buf)
                return dict(graph=_capture(dev, body), flag=flag, params=params)
            return _cached_graph(prog, ("sample", slot, buf.data_ptr(), rows, quantize), build)

        graphs = {}
        if cuda and launch and HOST_CUDA_GRAPHS and n >= unit:
            graphs = _capture_chunks(bounds, 2, unit, capture)
            wrap = lambda v: (v + 2**63) % 2**64 - 2**63                     # noqa: E731  (uint64 bits as int64)
            params = torch.tensor([[wrap(draw.seed), draw.row0 + r0] for r0, _ in bounds], dtype=torch.int64).to(dev)

        def first(i, r0, r1, flag):
            g = graphs.get((i % 2, r1 - r0))
            if g is None:
                emit(r0, r1, lambda buf: compute(prog, buf, r0, r1, flag))
                return

            def replay(buf):
                g["params"].copy_(params[i])
                g["graph"].replay()
            emit(r0, r1, replay)

        def again(i, r0, r1):                             # the same rows of the noise on the tf32-split program
            emit(r0, r1, lambda buf: compute(prog._fallback(), buf, r0, r1, None))

        if cuda:
            side.wait_stream(main)
        # a graph's flag is not per chunk: when one is set, every chunk is recomputed
        engine.run_chunks(bounds, dev, prog is not None and prog.guarded, first, again,
                          shared_flags=[g["flag"] for g in graphs.values()])
        if cuda:
            side.synchronize()

    def fit(self, data_train, optim=None, optim_params: Optional[Dict[str, Any]] = None, batch_size: int = 32,
            shuffle: bool = True, gradient_clip: Optional[float] = None, device=None, epochs: int = 1, **kw):
        """Maximum-likelihood training loop with the reference's signature (flows.py:113-210); returns the epoch
        losses.  Default optimiser: `usflows_b200.optim.SophiaG`.  Under an initialised `torch.distributed`
        process group the batch is sharded over the ranks and the gradients are all-reduced (see training.py)."""
        from . import training
        return training.fit(self, data_train, optim=optim, optim_params=optim_params, batch_size=batch_size,
                            shuffle=shuffle, gradient_clip=gradient_clip, device=device, epochs=epochs, **kw)

    def to(self, device):
        self.device = device
        self.trainable_layers = torch.nn.ModuleList([l.to(device) for l in self.trainable_layers])
        for l in self.layers:                                    # plain-attribute tensors (masks)
            if isinstance(l, BaseTransform):
                l.to(device)
        self._distribution_to(device)
        self._programs = {}
        return super().to(device)

    def is_feasible(self) -> bool:
        return all(l.is_feasible() for l in self.layers if isinstance(l, BaseTransform))

    def add_jitter(self, jitter: float = 1e-6) -> None:
        for l in self.layers:
            if isinstance(l, BaseTransform) and not l.is_feasible():
                l.add_jitter(jitter)

    def log_prior(self):
        return 0

    def _distribution_to(self, device) -> None:
        pass

    # -- engine glue -----------------------------------------------------------------------------
    def _base_module(self) -> DistributionModule:
        b = self.base_distribution
        return b.base_dist if isinstance(b, Independent) else b

    def _event_shape(self):
        return self.base_distribution.event_shape

    def _channels_last_perm(self, device) -> torch.Tensor:
        C, H, W = self._event_shape()
        key = (C, H, W, str(device))
        if getattr(self, "_cl_perm_key", None) != key:
            self._cl_perm, self._cl_perm_key = image_engine.channels_last_index(C, H * W, device), key
        return self._cl_perm

    def _weights_key(self):
        return tuple((p.data_ptr(), p._version) for p in self.parameters())

    def _program(self, direction: str, zero_ctx: bool = False):
        """(Program, total forward log|det J|) for the current weight version; `zero_ctx`: lowered for the zero context of a
        soft-training `log_prob` / `sample` (only ConditionalDenseNN conditioners tell it from no context)."""
        mode = self.precision or engine.get_precision()
        key = (mode,) + self._weights_key()
        slot = direction
        if self._cond_dense_nets:
            slot = (direction, bool(zero_ctx))
        hit = self._programs.get(slot)
        if hit is None or hit[0] != key:
            for net in self._cond_dense_nets:
                net.zero_context_default = bool(zero_ctx)
            with torch.no_grad():
                ev = tuple(self._event_shape())
                if len(ev) == 3:
                    prog = image_engine.ImageProgram(self.layers, direction, mode, ev)
                elif len(ev) == 1:
                    prog = engine.Program(self.layers, direction, mode)
                else:
                    raise NotImplementedError("usflows_b200: events of shape [d] and [C, H, W] are built")
            ladj, n_bad = engine.total_ladj(self.layers)
            hit = (key, prog, ladj, n_bad)
            self._programs[slot] = hit
        return hit[1], hit[2]

    def _apply_plan(self, prog, x2: torch.Tensor) -> torch.Tensor:
        rows, d = x2.shape
        x2 = x2.contiguous()
        bounds, capacity = self._plan_chunks(rows)
        plan = prog.c_plan(d, capacity)
        y = torch.empty(rows, prog.out_width(d), dtype=torch.float32, device=x2.device)
        engine.run_chunks(bounds, x2.device, prog.uses_range_flag,
                          lambda i, r0, r1, flag: plan.apply(x2[r0:r1], y[r0:r1], flag),
                          lambda i, r0, r1: prog._fallback().run(x2[r0:r1], out=y[r0:r1]))
        return y

    def _run(self, direction: str, x: torch.Tensor, zero_ctx: bool = False) -> torch.Tensor:
        if self._layer_route:
            return self._with_context(direction, x, None)
        x2, batch_shape = engine._flatten_rows(x, len(self._event_shape()))
        with torch.no_grad(), ops.on_device(x2):
            prog, _ = self._program(direction, zero_ctx)
            if USE_C_PLAN and x2.is_cuda and x2.shape[0] > 0 and prog.plan_able() and not torch.cuda.is_current_stream_capturing():
                y = self._apply_plan(prog, x2)
            else:
                y = prog.run(x2)
        return y.reshape(*batch_shape, *self._event_shape())


class USFlow(Flow):
    """Uniformly scaling flow: [BlockAffine(LU..[, Householder]) -> additive MaskedCoupling
    [-> BlockAffine^-1]] x coupling_blocks -> BlockAffine(LU) -> Scale  (flows.py:380-491)."""

    MASKTYPE = Literal["checkerboard", "channel"]

    _context_needs_soft_training = True

    def __init__(self, base_distribution, in_dims: List[int], coupling_blocks: int,
                 conditioner_cls: Type[torch.nn.Module], conditioner_args: Dict[str, Any], soft_training=False,
                 prior_scale: Optional[float] = None, training_noise_prior=None, affine_conjugation: bool = False,
                 nonlinearity: Optional[torch.nn.Module] = None, lu_transform: int = 1, householder: int = 1,
                 masktype: str = "checkerboard", *args, **kwargs):
        self.coupling_blocks = coupling_blocks
        self.in_dims = in_dims
        self.conditioner_cls = conditioner_cls
        self.conditioner_args = conditioner_args
        self.prior_scale = prior_scale
        if masktype == "checkerboard":
            self.mask_Generator = USFlow.create_checkerboard_mask
        elif masktype == "channel":
            self.mask_Generator = USFlow.create_channel_mask
        else:
            raise ValueError(f"Unknown mask type {masktype}")
        if lu_transform < 0:
            raise ValueError("Number of LU transforms must be non-negative")
        if householder < 0:
            raise ValueError("Number of Householder vectors transforms must be non-negative")
        self.lu_transform = lu_transform
        self.householder = householder
        # EXTENSION (not in the reference, whose coupling is additive only): coupling="affine" builds scale-and-shift
        # couplings; the conditioner then has to emit 2*d values (DenseNN: param_dims=[d, d])
        coupling = kwargs.pop("coupling", "additive")
        if coupling not in ("additive", "affine"):
            raise ValueError(f"Unknown coupling type {coupling}")
        self.coupling = coupling

        layers = []
        mask = self.mask_Generator(in_dims)
        for _ in range(coupling_blocks):
            affine_layers = [LUTransform(in_dims[0], prior_scale) for _ in range(lu_transform)]
            if householder > 0:
                affine_layers.append(HouseholderTransform(dim=in_dims[0], nvs=householder))
            block_affine_layer = None
            if affine_layers:
                block_affine_layer = BlockAffineTransform(in_dims, SequentialAffineTransform(affine_layers))
                layers.append(block_affine_layer)
            coupling_cls = MaskedAffineCoupling if coupling == "affine" else MaskedCoupling
            layers.append(coupling_cls(mask, conditioner_cls(**conditioner_args)))
            if affine_conjugation and block_affine_layer is not None:
                layers.append(InverseTransform(block_affine_layer))   # shares parameters (flows.py:469-470)
            mask = 1 - mask
        layers.append(BlockAffineTransform(in_dims, LUTransform(in_dims[0], prior_scale)))
        layers.append(ScaleTransform(in_dims))
        super().__init__(base_distribution, layers, soft_training=soft_training,
                         training_noise_prior=training_noise_prior, *args, **kwargs)

    @classmethod
    def create_checkerboard_mask(cls, in_dims, invert: bool = False) -> torch.Tensor:
        """(sum of index coordinates) mod 2, float32, shape (1, *in_dims)  (flows.py:494-514)."""
        axes = [torch.arange(d, dtype=torch.int32) for d in in_dims]
        idx = torch.stack(torch.meshgrid(*axes, indexing="ij"))
        mask = torch.fmod(idx.sum(dim=0), 2).to(torch.float32).view(1, *in_dims)
        return 1 - mask if invert else mask

    @classmethod
    def create_channel_mask(cls, in_dims, invert: bool = False) -> torch.Tensor:
        """(first index coordinate) mod 2  (flows.py:516-536)."""
        axes = [torch.arange(d, dtype=torch.int32) for d in in_dims]
        idx = torch.stack(torch.meshgrid(*axes, indexing="ij"))
        mask = torch.fmod(idx[0], 2).to(torch.float32).view(1, *in_dims)
        return 1 - mask if invert else mask

    def log_prior(self):
        """Sum of the top-level layers' log_prior -- identically 0 in the reference because
        BlockAffineTransform does not forward to its LU layer (flows.py:538-549, SURVEY Q3)."""
        if self.prior_scale is not None:
            return sum(l.log_prior() for l in self.layers)
        return 0

    def load_state_dict(self, state_dict, strict: bool = True, **kw):
        """Accepts reference checkpoints: InverseTransform layers alias block i's parameters and appear a
        second time under `trainable_layers.{i+2}.transform...` (SURVEY 8b) -- both copies are accepted."""
        return super().load_state_dict(state_dict, strict=strict, **kw)
