"""Row-sharded evaluation of one flow on several GPUs of a box from ONE process (SURVEY 7 step 9 / 8e).

`log_prob`, `sample`, `backward`, `_forward` are independent per row (no batch statistics anywhere in the layer stack), so
the batch is cut into contiguous row blocks, one per device; the weights (<= 0.5 GB) are replicated, every device owns its
prepared-weight cache, launch program, CUDA graphs, staging buffers and copy stream, and there is NO data-path collective.
The per-device work is issued from one host thread per device (the launches release the GIL), each ending in its own
stream synchronisation; rows come from / results go to HOST memory (pin it for full copy speed), which is where a
caller that feeds several GPUs from one process has them.

    from usflows_b200 import parallel
    lp = parallel.log_prob_sharded(flow, x_host)                    # all visible GPUs
    sf = parallel.ShardedFlow(flow, devices=[0, 1, 2, 3]); lp = sf.log_prob(x_host); y = sf.sample(1 << 20)

The multi-process form (one rank per GPU under torchrun, as `bench.py --gpus N` and `Flow.fit` use) needs nothing from this
module: every rank calls `flow.log_prob_host` on its own rows.
"""
from __future__ import annotations

import copy
import math
import threading
from concurrent.futures import ThreadPoolExecutor
from typing import List, Optional, Sequence

import torch

from . import engine, ops

_UNCOPIED = ("_programs", "_stage", "_side", "_cl_perm", "_cl_perm_key", "_sharded")


def shard_bounds(n: int, rank: int, world: int):
    """Contiguous, near-equal slice [lo, hi) of n rows for `rank` of `world` (same rule as training.shard_bounds)."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def replicate(flow, device):
    """A copy of `flow` on `device` that shares nothing with it (parameters copied; caches, staging buffers, streams and
    captured graphs are per replica and are rebuilt on first use)."""
    stash = {k: flow.__dict__.pop(k) for k in _UNCOPIED if k in flow.__dict__}
    try:
        rep = copy.deepcopy(flow)
    finally:
        flow.__dict__.update(stash)
    rep._programs = {}
    return rep.to(device)


class ShardedFlow:
    """`flow` replicated over `devices` (default: every visible CUDA device); see the module docstring."""

    def __init__(self, flow, devices: Optional[Sequence] = None):
        if devices is None:
            devices = list(range(torch.cuda.device_count()))
        devs = [torch.device("cuda", d) if isinstance(d, int) else torch.device(d) for d in devices]
        if not devs:
            raise RuntimeError("usflows_b200.parallel: no CUDA device (there is no CPU fallback)")
        if len({d.index for d in devs}) != len(devs):
            raise ValueError("usflows_b200.parallel: every device may appear once (the workspaces are per device)")
        self.flow, self.devices = flow, devs
        home = next(flow.parameters()).device
        self.replicas = [flow if d == home else replicate(flow, d) for d in devs]
        self._synced = flow._weights_key()
        self._pool = ThreadPoolExecutor(max_workers=len(devs), thread_name_prefix="usf-shard")

    def close(self) -> None:
        self._pool.shutdown(wait=True)

    def sync_weights(self) -> None:
        """Copy the source flow's parameters into the replicas if they changed since the last call (device-to-device
        copies; the replicas then re-prepare their weights on first use, once per weight version as everywhere)."""
        key = self.flow._weights_key()
        if key == self._synced:
            return
        src = dict(self.flow.named_parameters())
        with torch.no_grad():
            for rep in self.replicas:
                if rep is self.flow:
                    continue
                for name, p in rep.named_parameters():
                    p.copy_(src[name], non_blocking=True)
        for d in self.devices:
            torch.cuda.synchronize(d)
        self._synced = key

    def _map(self, fn, n_rows: int):
        bounds = [shard_bounds(n_rows, i, len(self.devices)) for i in range(len(self.devices))]
        futs = [self._pool.submit(fn, i, rep, lo, hi) for i, (rep, (lo, hi)) in enumerate(zip(self.replicas, bounds))]
        return [f.result() for f in futs]            # re-raises a worker's exception here

    def log_prob(self, x_host: torch.Tensor, out_host: Optional[torch.Tensor] = None, *, dequantize: Optional[str] = None,
                 seed: Optional[int] = None) -> torch.Tensor:
        """log p of the rows of `x_host` [rows, *event] (host memory) -> `out_host` [rows] (host memory).  With `dequantize`
        (see Flow.log_prob), x_host is uint8; one seed serves all devices and every block keeps its global row numbers, so
        the result does not depend on the number of devices."""
        if x_host.is_cuda:
            raise RuntimeError("usflows_b200.parallel: expects host rows (each device copies its own block)")
        if dequantize is not None:
            seed = ops.dequant_spec(x_host, dequantize, seed).seed
        self.sync_weights()
        ev = math.prod(self.flow._event_shape())
        x2 = x_host.reshape(-1, ev)
        rows = x2.shape[0]
        if out_host is None:
            out_host = torch.empty(rows, dtype=torch.float32, pin_memory=True)
        flat = out_host.reshape(-1)

        def work(i, rep, lo, hi):
            if hi > lo:
                if dequantize is None:
                    rep.log_prob_host(x2[lo:hi], flat[lo:hi])
                else:
                    rep.log_prob_host(x2[lo:hi], flat[lo:hi], dequantize=dequantize, seed=seed, row_offset=lo)
        self._map(work, rows)
        return out_host

    def sample(self, n: int, out_host: Optional[torch.Tensor] = None, *, seed: Optional[int] = None,
               quantize: bool = False) -> torch.Tensor:
        """`n` samples [n, *event] in host memory; every device draws from its own Philox stream.  With `seed` or
        `quantize` (see Flow.sample_host), one seed serves all devices and device i streams its block [lo, hi) as global
        rows lo .. hi - 1 of that seed's stream, so the result does not depend on the number of devices."""
        if seed is not None or quantize:
            return self._sample_stream(n, out_host, ops.draw_seed() if seed is None else int(seed), quantize)
        self.sync_weights()
        ev = tuple(self.flow._event_shape())
        if out_host is None:
            out_host = torch.empty(n, *ev, dtype=torch.float32, pin_memory=True)

        def work(i, rep, lo, hi):
            if hi > lo:
                engine.philox_salt.value = i + 1
                try:
                    y = rep.sample([hi - lo])
                finally:
                    engine.philox_salt.value = 0
                out_host[lo:hi].copy_(y, non_blocking=True)
                torch.cuda.current_stream(self.devices[i]).synchronize()
        self._map(work, n)
        return out_host

    def _sample_stream(self, n: int, out_host: Optional[torch.Tensor], seed: int, quantize: bool) -> torch.Tensor:
        if n < 0:
            raise ValueError("usflows_b200: the number of samples must be >= 0")
        self.sync_weights()
        if out_host is None:
            out_host = torch.empty(n, *self.flow._event_shape(), dtype=torch.uint8 if quantize else torch.float32,
                                   pin_memory=True)

        def work(i, rep, lo, hi):
            if hi > lo:
                rep.sample_host(hi - lo, out_host[lo:hi], seed=seed, quantize=quantize, row_offset=lo)
        self._map(work, n)
        return out_host

    def backward(self, x_host: torch.Tensor, out_host: Optional[torch.Tensor] = None) -> torch.Tensor:
        return self._rows("backward", x_host, out_host)

    def _forward(self, z_host: torch.Tensor, out_host: Optional[torch.Tensor] = None) -> torch.Tensor:
        return self._rows("forward", z_host, out_host)

    def _rows(self, direction: str, x_host, out_host):
        self.sync_weights()
        ev = tuple(self.flow._event_shape())
        x2 = x_host.reshape(-1, *ev)
        if out_host is None:
            out_host = torch.empty(x2.shape, dtype=torch.float32, pin_memory=True)

        def work(i, rep, lo, hi):
            if hi > lo:
                dev = self.devices[i]
                y = rep._run(direction, x2[lo:hi].to(dev, non_blocking=True))
                out_host[lo:hi].copy_(y, non_blocking=True)
                torch.cuda.current_stream(dev).synchronize()
        self._map(work, x2.shape[0])
        return out_host


_lock = threading.Lock()


def _sharded(flow, devices) -> ShardedFlow:
    key = None if devices is None else tuple(str(d) for d in devices)
    with _lock:
        cache = flow.__dict__.setdefault("_sharded", {})
        if key not in cache:
            cache[key] = ShardedFlow(flow, devices)
        return cache[key]


def log_prob_sharded(flow, x_host: torch.Tensor, devices: Optional[Sequence] = None,
                     out_host: Optional[torch.Tensor] = None, *, dequantize: Optional[str] = None,
                     seed: Optional[int] = None) -> torch.Tensor:
    """`flow.log_prob` of host rows on `devices` (default: all visible GPUs), rows split into contiguous blocks; uint8 rows
    with `dequantize` as in ShardedFlow.log_prob."""
    return _sharded(flow, devices).log_prob(x_host, out_host, dequantize=dequantize, seed=seed)


def sample_sharded(flow, n: int, devices: Optional[Sequence] = None, out_host: Optional[torch.Tensor] = None, *,
                   seed: Optional[int] = None, quantize: bool = False) -> torch.Tensor:
    """`n` samples of `flow` in host memory, drawn on `devices` (default: all visible GPUs); `seed` / `quantize` as in
    ShardedFlow.sample."""
    return _sharded(flow, devices).sample(n, out_host, seed=seed, quantize=quantize)
