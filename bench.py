#!/usr/bin/env python
"""Benchmark of the USFlows hot path on B200:  `log_prob` throughput (samples/s) of a flat USFlow.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c4|c5|c1|c2cn|mnist_img] [--precision fp32|tf32|bf16]
    python bench.py --impl reference ...      # the reference algorithm's CPU path (oracle port) on host cores
    python bench.py --workload c5 --sweep-full   # the 1 K - 64 M point sweep of BASELINE config 5 on its own
    python bench.py --dump-outputs DIR ...       # also write the log-probs of the last timed step to DIR/log_prob.npy

Contract (one JSON line on stdout, printed by rank 0): metric/value/unit/n_gpus/steps/warmup/ms_per_step/
higher_is_better/scaling/vs_baseline/dtype/data/config + roofline, cpu_baseline, e2e, clocks, gpu_launches.

A "step" is one `log_prob` pass over one batch of synthetic rows per GPU (weak scaling: every rank evaluates
its own `rows` rows, no data-path collective).  `value` is measured with the batch resident in HBM; `e2e` goes
through `Flow.log_prob_host` with pinned HOST buffers (H2D of the batch and D2H of the log-probs inside the
timed region).  Workloads follow BASELINE.json / SURVEY 8d:
  c2: d=784,  B=4, MLP [1024,1024], Laplace base, 65536 rows   <- the configuration the metric is quoted on
  c4: d=3072, B=8, MLP [1024,1024], Normal base,  32768 rows
  c5: d=3072, B=4, MLP [1024,1024], Laplace base, 32768 rows
  c1: d=2,    B=10, MLP [32,32],    Laplace base, 1048576 rows
Inputs are larger than L2 (c2: 205 MB per batch vs 126 MB), so no explicit L2 flush is needed between steps.

Besides the headline numbers the default line carries, so that the driver's N = 1, 2, 4, 8 runs record them:
  train    C3: the MLE training step (8192 rows per GPU, NCCL gradient all-reduce overlapped with the backward pass)
  configs  C4 (fp32 and bf16 modes, log_prob and sample) and the C5 batch sweep (total points split over the ranks)
  h2d      the host -> device copy bandwidth of one rank alone and of all ranks at once (what bounds `e2e` at N > 1)
`--no-extra` drops `configs`, `--no-train` drops `train`.
"""
from __future__ import annotations

import argparse
import atexit
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "c2": dict(spec=dict(in_dims=[784], coupling_blocks=4, hidden_dims=[1024, 1024], affine_conjugation=True,
                         lu_transform=1, householder=0, base="laplace"), rows=65536, cpu_rows=8192,
               name="C2 MNIST-shaped 784-D USFlow (B=4, MLP 1024x1024, Laplace) batch log_prob"),
    "c4": dict(spec=dict(in_dims=[3072], coupling_blocks=8, hidden_dims=[1024, 1024], affine_conjugation=True,
                         lu_transform=1, householder=0, base="normal"), rows=32768, cpu_rows=1024,
               name="C4 CIFAR-shaped 3072-D USFlow (B=8, MLP 1024x1024, Normal) batch log_prob"),
    "c5": dict(spec=dict(in_dims=[3072], coupling_blocks=4, hidden_dims=[1024, 1024], affine_conjugation=True,
                         lu_transform=1, householder=0, base="laplace"), rows=32768, cpu_rows=2048,
               name="C5 3072-D USFlow (B=4, MLP 1024x1024, Laplace) batch log_prob"),
    # C2's shape with the reference's own MLP-style conditioner (networks.ConvNet, vector branch: 2 gated blocks of width
    # 1024 with LayerNorm) and the base of its live MNIST configuration (experiments/mnist/mnist.yaml:79-92: L1-radial,
    # LogNormal radius) -- SURVEY 8f rows 2 and 4
    "c2cn": dict(spec=dict(in_dims=[784], coupling_blocks=4, conditioner="convnet", c_hidden=[1024, 1024], gating=True,
                           normalize_layers=True, affine_conjugation=True, lu_transform=1, householder=0, base="radial",
                           p=1, norm="lognormal"), rows=65536, cpu_rows=4096,
                 name="C2-shaped 784-D USFlow (B=4, ConvNet conditioner 2 gated blocks x 1024 + LayerNorm, L1-radial "
                      "LogNormal base) batch log_prob"),
    # the reference's live MNIST configuration (experiments/mnist/mnist.yaml:44-92): 28x28 images squeezed to [16, 7, 7],
    # 15 coupling blocks, ConvNet2D conditioner (32 hidden channels, 3 gated 3x3 blocks, LayerNormChannels), conjugated
    # 1x1-convolution LU layers, L1-radial LogNormal base -- SURVEY 8f row 3
    "mnist_img": dict(spec=dict(in_dims=[16, 7, 7], coupling_blocks=15, conditioner="convnet2d", c_hidden=32, num_layers=3,
                                kernel_size=3, gating=True, normalize_layers=True, affine_conjugation=True, lu_transform=1,
                                householder=0, base="radial", p=1, norm="lognormal"), rows=16384, cpu_rows=256,
                      name="MNIST [16,7,7] USFlow (B=15, ConvNet2D 32 ch x 3 gated 3x3 blocks + LayerNorm, 1x1-conv LU, "
                           "L1-radial LogNormal base) batch log_prob"),
    "c1": dict(spec=dict(in_dims=[2], coupling_blocks=10, hidden_dims=[32, 32], affine_conjugation=True,
                         lu_transform=1, householder=0, base="laplace"), rows=1 << 20, cpu_rows=65536,
               name="C1 2-D USFlow (B=10, MLP 32x32, Laplace) batch log_prob"),
}

MODE_PRODUCTS = {"fp32": 3.0, "fp32_tf32": 6.0, "tf32": 2.0, "bf16": 1.0}   # tensor-pipe cost per algorithmic MAC in
#                                                                             units of one bf16/fp16 MMA (tf32 runs at 1/2)
SWEEP_POINTS = [1 << 10, 1 << 13, 1 << 16, 1 << 19, 1 << 22, 1 << 26]      # C5: total points of one pass (all ranks)
SWEEP_BLOCK = 1 << 16                                                       # rows generated on the device at a time
SWEEP_DEFAULT_MAX_PER_GPU = 1 << 23                                         # default line: skip points above this per rank
DUMP_MAX_BYTES = 64 << 20                                                   # --dump-outputs: all files together


def dump_outputs(directory: str, arrays: dict) -> None:
    """Writes each output as `directory/<name>.npy` in float32, so that two builds can be compared output for output.
    An output too large for the budget is cut to a fixed, seeded sample of its rows; the chosen row indices go to
    `<name>_rows.npy` (float64, exact for any row count that fits in memory)."""
    import numpy as np
    import torch
    os.makedirs(directory, exist_ok=True)
    budget = DUMP_MAX_BYTES // max(1, len(arrays))
    for name, t in arrays.items():
        a = t.detach().float().cpu()
        if a.numel() * 4 > budget:
            keep = budget // (a[0].numel() * 4 + 8)           # every kept row also stores its float64 index
            rows = torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
            a = a[rows]
            np.save(os.path.join(directory, name + "_rows.npy"), rows.numpy().astype(np.float64))
        np.save(os.path.join(directory, name + ".npy"), a.numpy())


def algorithmic_flops_per_sample(spec) -> float:
    """SURVEY 8d: (2B+1) * 2 d^2 + B * 2 (d H + H^2 + H d) with conjugation (B+1 affine layers without)."""
    d, B = spec["in_dims"][0], spec["coupling_blocks"]
    if spec.get("conditioner") == "convnet2d":     # per pixel: 1x1-conv affine layers 2 C^2; k x k convolutions 2 k^2 Cin Cout
        C, hw = spec["in_dims"][0], spec["in_dims"][1] * spec["in_dims"][2]
        ch, kk, L = spec["c_hidden"], spec.get("kernel_size", 3) ** 2, spec["num_layers"]
        per_block = 2 * kk * ch * ch + (2 * ch * 2 * ch if spec.get("gating", True) else 0)
        cond = 2 * kk * C * ch + L * per_block + 2 * kk * ch * C
        n_aff = 2 * B + 1 if spec.get("affine_conjugation") else B + 1
        return hw * (n_aff * 2 * C * C + B * cond)
    if spec.get("conditioner") == "convnet":       # Linear(d,h0) + per block [h_in h + h 2h (+ proj)] + Linear(h_last, d)
        ch = list(spec["c_hidden"])
        mlp = 2 * d * ch[0] + 2 * ch[-1] * d
        for i, oc in enumerate(ch):
            ic = ch[i - 1] if i > 0 else ch[0]
            mlp += 2 * ic * oc + (2 * oc * 2 * oc if spec.get("gating", True) else 0) + (2 * ic * oc if ic != oc else 0)
    else:
        dims = [d] + list(spec["hidden_dims"]) + [d]
        mlp = sum(2 * dims[i] * dims[i + 1] for i in range(len(dims) - 1))
    n_aff = 2 * B + 1 if spec.get("affine_conjugation") else B + 1
    return n_aff * 2 * d * d + B * mlp


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), "measured"
    # MEASURED_PEAKS.json is driver-written; when it is absent use the fallback /opt/skills/guides/B200_PROFILING.md
    # states (6.65 TB/s, 1.59 PFLOP/s burst, ~1.4 PFLOP/s sustained under the power cap) and say so
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


def committed_traffic(workload: str, precision: str):
    """DRAM traffic of the dominant kernel from the committed `ncu --set full` capture of this workload (profiles/):
    dram__bytes_read.sum + dram__bytes_write.sum, as the mean per launch and summed over the launches of one step.
    ncu cannot run inside a timed bench, so this is the one figure of the line that is read, not measured live."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        path = os.path.join(ROOT, "profiles", name)
        if os.path.exists(path):
            with open(path) as f:
                t = json.load(f)
            if t.get("workload", "c2") == workload and t.get("precision", "fp32") == precision:
                return t.get("dram_bytes_per_launch"), t.get("dram_bytes_per_step"), "profiles/" + name
    return None, None, None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.idx, self.proc, self.lines = gpu_index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.idx)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
            atexit.register(self._end)            # a run that fails before stop() leaves no sampler behind
        except OSError:
            self.proc = None

    def _end(self):
        if self.proc.poll() is None:
            self.proc.terminate()
        self.proc.wait()

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self._end()
        sm, smax, reasons, power = [], None, set(), []
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax = float(f[2]); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "power_w_max": max(power) if power else None, "samples": len(sm)}


def bind_to_gpu_numa_node(local_rank: int, world: int) -> dict:
    """Pin this rank's host threads (and with them, by first touch, its pinned staging buffers) to the CPUs of its GPU's
    NUMA node, and give every rank of the node its own slice of those CPUs so that the copy-issuing threads of N ranks
    do not share cores.  Reads sysfs only; a box that exposes one node / no topology leaves the affinity as it is."""
    info = {"numa_node": None, "cpus": None}
    try:
        import torch
        prop = torch.cuda.get_device_properties(local_rank)
        bus = f"{getattr(prop, 'pci_domain_id', 0):04x}:{prop.pci_bus_id:02x}:{prop.pci_device_id:02x}.0"
        node_path = f"/sys/bus/pci/devices/{bus}/numa_node"
        node = int(open(node_path).read().strip()) if os.path.exists(node_path) else -1
        info["pci"] = bus
        info["numa_node"] = node
        allowed = sorted(os.sched_getaffinity(0))
        cpus = allowed
        if node >= 0 and os.path.exists(f"/sys/devices/system/node/node{node}/cpulist"):
            ids = []
            for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
                a, _, b = part.partition("-")
                ids += list(range(int(a), int(b or a) + 1))
            local = [c for c in allowed if c in set(ids)]
            if local:
                cpus = local
        if world > 1 and len(cpus) >= 2 * world:          # one slice per rank (ranks of one box share the node list)
            per = len(cpus) // world
            cpus = cpus[local_rank * per:(local_rank + 1) * per]
        os.sched_setaffinity(0, cpus)
        info["cpus"] = f"{cpus[0]}-{cpus[-1]} ({len(cpus)})"
    except Exception as e:                                # noqa: BLE001  (topology is advisory)
        info["error"] = repr(e)[:120]
    return info


# ------------------------------------------------------------------------------------------------
def cpu_reference_run(wl, steps: int, warmup: int, rows: int):
    """The reference algorithm's own CPU path (oracle port = same ATen ops in the same order, including the
    per-call weight re-preparation) on all host cores.  Returns (as-is samples/s, amortised samples/s, cores)."""
    import torch
    from oracle import flow_oracle as O
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    spec = wl["spec"]
    params = O.random_params(spec, 0)
    g = torch.Generator().manual_seed(1)
    x = torch.rand(rows, *spec["in_dims"], generator=g)
    with torch.no_grad():
        for _ in range(warmup):
            O.flow_log_prob(x, spec, params)
        t0 = time.perf_counter()
        for _ in range(steps):
            O.flow_log_prob(x, spec, params)
        t_asis = (time.perf_counter() - t0) / steps
        _, prepared = O.flow_log_prob_amortised(x, spec, params)
        t0 = time.perf_counter()
        for _ in range(steps):
            O.flow_log_prob_amortised(x, spec, params, prepared=prepared)
        t_am = (time.perf_counter() - t0) / steps
    return rows / t_asis, rows / t_am, cores, t_asis


class Harness:
    """Process-group plumbing shared by every leg: barrier + device events, max over ranks."""

    def __init__(self, torch, dist, dev, world, rank):
        self.torch, self.dist, self.dev, self.world, self.rank = torch, dist, dev, world, rank

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def timed(self, fn, steps):
        torch = self.torch
        self.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        self.barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(ms, op=self.dist.ReduceOp.MAX)
        return float(ms) / steps

    def gather_floats(self, v: float):
        t = self.torch.tensor([v], device=self.dev, dtype=self.torch.float64)
        if self.world == 1:
            return [float(v)]
        out = [self.torch.zeros_like(t) for _ in range(self.world)]
        self.dist.all_gather(out, t)
        return [float(o) for o in out]


def measure_tf32_peak(torch, dev):
    """cuBLAS TF32 8192^3 back to back (the denominator of the tf32 mode; SURVEY 8d says measure it, not assume 1/2)."""
    old = torch.backends.cuda.matmul.allow_tf32
    try:
        torch.backends.cuda.matmul.allow_tf32 = True
        a = torch.randn(8192, 8192, device=dev)
        b = torch.randn(8192, 8192, device=dev)
        for _ in range(3):
            a @ b
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        n = 20
        for _ in range(n):
            a @ b
        e1.record()
        torch.cuda.synchronize()
        return 2 * 8192 ** 3 * n / (e0.elapsed_time(e1) * 1e-3) / 1e12
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old


def h2d_probe(h: Harness, x_host, x_dev):
    """Host -> device bandwidth of this workload's pinned batch: rank 0 alone, then all ranks at the same time."""
    torch = h.torch
    nbytes = x_host.numel() * 4

    def copy():
        x_dev.copy_(x_host, non_blocking=True)
    alone = None
    for r in range(min(h.world, 1)):                      # rank 0 alone (the others wait at the barrier)
        h.barrier()
        if h.rank == r:
            copy(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); copy(); copy(); copy(); e1.record(); torch.cuda.synchronize()
            alone = 3 * nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9
        h.barrier()
    copy(); torch.cuda.synchronize()
    h.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); copy(); copy(); copy(); e1.record(); torch.cuda.synchronize()
    mine = 3 * nbytes / (e0.elapsed_time(e1) * 1e-3) / 1e9
    per_rank = h.gather_floats(mine)
    alone0 = h.gather_floats(alone if alone is not None else 0.0)[0]
    return dict(rank0_alone_gbs=alone0, per_rank_concurrent_gbs=per_rank, aggregate_concurrent_gbs=sum(per_rank),
                bytes=nbytes, note="pinned host -> device copies of one batch; concurrent = all ranks copying at once")


def run_c4(h: Harness, U, O, build_flow, steps, peaks):
    """BASELINE config 4 (CIFAR-shaped 3072-D deep stack): log_prob and sample, fp32 and bf16 modes, weak scaling."""
    torch = h.torch
    wl = WORKLOADS["c4"]
    spec, rows = wl["spec"], wl["rows"]
    fps = algorithmic_flops_per_sample(spec)
    params = O.random_params(spec, 0)
    x = torch.rand(rows, 3072, device=h.dev, generator=torch.Generator(device=h.dev).manual_seed(2 + h.rank))
    out = dict(workload=wl["name"], rows_per_gpu_per_step=rows, flops_per_sample=fps, modes={})
    ref_lp = None
    for mode in ("fp32", "bf16"):
        flow = build_flow(spec, params, device=h.dev, precision=mode)
        lp = flow.log_prob(x[:256])
        if ref_lp is None:
            ref_lp = lp.double().cpu()
        err = float(((lp.double().cpu() - ref_lp).abs() / ref_lp.abs().clamp(min=1)).max())
        for _ in range(2):
            flow.log_prob(x)
        ms_lp = h.timed(lambda: flow.log_prob(x), steps)
        flow.sample([rows])
        ms_s = h.timed(lambda: flow.sample([rows]), max(2, steps // 2))
        tf = rows * fps / (ms_lp * 1e-3) / 1e12
        out["modes"][mode] = dict(log_prob_samples_per_sec=h.world * rows / (ms_lp * 1e-3), log_prob_ms=ms_lp,
                                  sample_samples_per_sec=h.world * rows / (ms_s * 1e-3), sample_ms=ms_s,
                                  tflops_per_gpu=tf, frac=tf / peaks["bf16_tflops_sustained"],
                                  frac_of_mode_ceiling=tf / (peaks["bf16_tflops_sustained"] / MODE_PRODUCTS[mode]),
                                  max_rel_diff_vs_fp32_mode=err)
        del flow
    return out


def run_c5_sweep(h: Harness, U, O, build_flow, peaks, full: bool, modes=("fp32", "bf16")):
    """BASELINE config 5: batch sweep 1 K - 64 M synthetic points through the 3072-D flow, log_prob and sample.  The
    TOTAL point count of a sweep entry is split evenly over the ranks (rows are independent; no collective); rows are
    generated on the device in blocks of 65 536 (64 M x 3072 floats = 805 GB does not exist anywhere at once) and every
    block is evaluated exactly once per pass, so an entry's time is the time of the whole pass, max over ranks."""
    torch = h.torch
    wl = WORKLOADS["c5"]
    spec = wl["spec"]
    fps = algorithmic_flops_per_sample(spec)
    params = O.random_params(spec, 0)
    gen = torch.Generator(device=h.dev).manual_seed(3 + h.rank)
    block = torch.rand(SWEEP_BLOCK, 3072, device=h.dev, generator=gen)
    entries = []
    for mode in modes:
        flow = build_flow(spec, params, device=h.dev, precision=mode)
        flow.log_prob(block[:256])
        flow.log_prob(block)
        flow.sample([SWEEP_BLOCK])
        for total in SWEEP_POINTS:
            per = -(-total // h.world)
            if per > SWEEP_DEFAULT_MAX_PER_GPU and not full:
                entries.append(dict(points=total, precision=mode, skipped=f"{per} rows per GPU: run with --sweep-full"))
                continue

            def lp_pass():
                left = per
                while left > 0:
                    n = min(left, SWEEP_BLOCK)
                    torch.rand(n, 3072, device=h.dev, generator=gen, out=block[:n])    # fresh synthetic points
                    flow.log_prob(block[:n])
                    left -= n

            def s_pass():
                left = per
                while left > 0:
                    n = min(left, SWEEP_BLOCK)
                    flow.sample([n])
                    left -= n
            reps = 3 if per <= (1 << 16) else 1
            if per <= (1 << 16):                      # small entries: one untimed pass first (graph capture, workspaces)
                lp_pass()
                s_pass()
            ms_lp = h.timed(lp_pass, reps)
            ms_s = h.timed(s_pass, reps)
            tf = per * fps / (ms_lp * 1e-3) / 1e12
            entries.append(dict(points=total, rows_per_gpu=per, precision=mode,
                                log_prob_samples_per_sec=h.world * per / (ms_lp * 1e-3), log_prob_ms=ms_lp,
                                sample_samples_per_sec=h.world * per / (ms_s * 1e-3), sample_ms=ms_s,
                                tflops_per_gpu=tf, frac=tf / peaks["bf16_tflops_sustained"],
                                frac_of_mode_ceiling=tf / (peaks["bf16_tflops_sustained"] / MODE_PRODUCTS[mode])))
        del flow
    return dict(workload=wl["name"], flops_per_sample=fps, block_rows=SWEEP_BLOCK, scaling="strong (total points split over ranks)",
                note="log_prob passes include the on-device generation of the points (torch.rand, 4 d B written per row)",
                entries=entries)


def run_train(h: Harness, U, O, build_flow, spec, steps):
    """BASELINE config 3: Fashion-MNIST-shaped MLE training, weak scaling: 8192 rows per GPU per step, gradient
    all-reduce over NCCL (bucketed, overlapped with the backward pass: usflows_b200/training.py), SophiaG lr=1e-3 wd=0
    as the reference's config (experiments/fashion/fashionclasses_veriflow.yaml:37-42)."""
    torch = h.torch
    from usflows_b200 import training
    per_gpu = 8192
    d = spec["in_dims"][0]
    flow = build_flow(spec, O.random_params(spec, 0), device=h.dev, precision="fp32")
    opt = U.SophiaG(list(flow.parameters()), lr=1e-3, weight_decay=0.0)
    ts = training.TrainStep(flow, opt, distributed=h.world > 1)
    gt = torch.Generator().manual_seed(100 + h.rank)
    xt = torch.rand(per_gpu, d, generator=gt).to(h.dev)
    losses = []
    for _ in range(3):
        losses.append(ts.step(xt))
    ms = h.timed(lambda: losses.append(ts.step(xt)), max(3, steps))
    # the exchange alone (all buckets, nothing to overlap with), for the share it would take unhidden
    ar_ms = None
    if ts.reducer is not None:
        def exchange():
            ts.reducer.begin()
            ts.reducer.finish()
        exchange()
        ar_ms = h.timed(exchange, 5)
    bad = float(ts.infeasible)
    l0, l1 = float(losses[0]) * h.world, float(losses[-1]) * h.world
    ts.close()
    return dict(metric="train_samples_per_sec", value=h.world * per_gpu / (ms * 1e-3), unit="samples/s",
                ms_per_step=ms, global_batch=per_gpu * h.world, rows_per_gpu=per_gpu,
                grad_floats=sum(p.numel() for p in flow.parameters()),
                allreduce_bytes_per_step=ts.allreduce_bytes, allreduce_ms_alone=ar_ms,
                allreduce="NCCL all-reduce(sum), bucketed, launched from gradient hooks during the backward pass"
                if h.world > 1 else "none (1 GPU)",
                engine=getattr(training, "TRAIN_ENGINE_NOTE", None),
                loss_first=l0, loss_last=l1, infeasible_entries=bad,
                note="zero_grad + density pass + backward + gradient all-reduce + SophiaG step + device-side "
                     "invertibility check, all inside the timed region")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="usflows_b200", choices=["usflows_b200", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--precision", default="fp32", choices=["fp32", "fp32_tf32", "fp32_simt", "tf32", "bf16"])
    ap.add_argument("--rows", type=int, default=0, help="rows per GPU per step (default: the workload's)")
    ap.add_argument("--chunk-rows", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-modes", action="store_true", help="skip the extra tf32 / bf16 mode measurements")
    ap.add_argument("--only-logprob", action="store_true",
                    help="profiling aid: warm-up + timed log_prob steps only, then exit (no JSON line)")
    ap.add_argument("--train", action="store_true", help="(default now) kept for compatibility")
    ap.add_argument("--no-train", action="store_true", help="skip the C3 training leg")
    ap.add_argument("--no-extra", action="store_true", help="skip the C4 lines and the C5 sweep")
    ap.add_argument("--sweep-full", action="store_true", help="C5 sweep: run every point (64 M on one GPU takes ~2 min)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the log-probs of the last timed step (rank 0) to DIR/log_prob.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    wl = WORKLOADS[args.workload]
    spec = wl["spec"]
    d = 1
    for v in spec["in_dims"]:
        d *= v
    flops_per_sample = algorithmic_flops_per_sample(spec)

    base_line = dict(metric="log_prob_samples_per_sec", unit="samples/s", n_gpus=args.gpus, steps=args.steps,
                     warmup=args.warmup, higher_is_better=True, scaling="weak", vs_baseline=None,
                     data="synthetic")

    # ---------------------------------------------------------------- reference arm (CPU, rank 0 only)
    if args.impl == "reference":
        if rank != 0:
            return
        rows = args.rows or wl["cpu_rows"]
        v_asis, v_am, cores, t = cpu_reference_run(wl, max(1, args.steps), max(1, min(args.warmup, 1)), rows)
        line = dict(base_line, impl="reference", value=v_asis, ms_per_step=t * 1e3, dtype="f32",
                    config=dict(workload=wl["name"], rows_per_step=rows, d=d, hidden=spec.get("hidden_dims", spec.get("c_hidden")),
                                coupling_blocks=spec["coupling_blocks"], engine="torch CPU (oracle port of the reference)"),
                    cpu_baseline=dict(value=v_asis, unit="samples/s", cores=cores, kind="port",
                                      sample=f"{rows} rows x {max(1, args.steps)} steps of the same workload; "
                                             f"as-is (per-call weight re-preparation, as the reference does); "
                                             f"amortised = {v_am:.1f} samples/s", amortised_value=v_am),
                    e2e=dict(value=v_asis, unit="samples/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0))
        print(json.dumps(line), flush=True)
        return

    # ---------------------------------------------------------------- B200 arm
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    affinity = bind_to_gpu_numa_node(local_rank, world)       # before any pinned allocation (first touch)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    h = Harness(torch, dist, dev, world, rank)

    import usflows_b200 as U
    from usflows_b200 import engine, ops
    from usflows_b200.builders import build_flow
    from oracle import flow_oracle as O      # parameters only (deterministic synthetic model); timed code is ours

    if args.chunk_rows:
        U.set_chunk_rows(args.chunk_rows)
        if len(spec["in_dims"]) > 1:                 # image-shaped events: channels-last rows (N*H*W) per chunk
            from usflows_b200 import image_engine
            image_engine.IMAGE_CHUNK_ROWS = image_engine.IMAGE_CHUNK_ROWS_PIX = args.chunk_rows
    rows = args.rows or wl["rows"]
    params = O.random_params(spec, 0)
    flow = build_flow(spec, params, device=dev, precision=args.precision)
    g = torch.Generator().manual_seed(1 + rank)
    x_host = torch.rand(rows, *spec["in_dims"], generator=g).pin_memory()
    x = x_host.to(dev)
    out_host = torch.empty(rows, dtype=torch.float32).pin_memory()
    timed = h.timed

    # the first call (library load, module load of the kernels, weight preparation, launch program) and, separately, what
    # a weight update costs the next log_prob: every parameter's version bumped in place (values unchanged), then one
    # 256-row call against the same call with the weights left alone -- weight preparation + program rebuild
    t0 = time.perf_counter()
    lp = flow.log_prob(x[:256])
    torch.cuda.synchronize()
    first_call_ms = (time.perf_counter() - t0) * 1e3
    reprep = []
    for _ in range(3):
        with torch.no_grad():
            for p in flow.parameters():
                p.mul_(1.0)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        flow.log_prob(x[:256])
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        flow.log_prob(x[:256])
        torch.cuda.synchronize()
        reprep.append(((t1 - t0) - (time.perf_counter() - t1)) * 1e3)
    prep_ms = sorted(reprep)[1]

    last = {}

    def step():
        last["log_prob"] = flow.log_prob(x)
    for _ in range(args.warmup):
        step()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ops.LAUNCHES = 0
    ranged = bool(os.environ.get("USF_PROFILE_RANGE"))          # ncu --profile-from-start off: the timed steps only
    if ranged:
        torch.cuda.profiler.start()
    ms_step = timed(step, args.steps)
    if ranged:
        torch.cuda.profiler.stop()
    launches = ops.LAUNCHES
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last)
    if args.only_logprob:
        if rank == 0:
            sampler.stop()
            print(f"log_prob: {ms_step:.3f} ms/step, {launches} launches in {args.steps} steps", flush=True)
        return
    value = world * rows / (ms_step * 1e-3)

    # the sampling pass (latent -> data) of the same model and batch size: base draws + forward layer stack
    sample_step = lambda: flow.sample([rows])          # noqa: E731
    for _ in range(max(1, args.warmup // 2)):
        sample_step()
    ms_sample = timed(sample_step, max(2, args.steps // 2))

    # end to end: pinned host rows in, host log-probs out, copies inside the timed region
    e2e_step = lambda: flow.log_prob_host(x_host, out_host)   # noqa: E731
    for _ in range(max(1, args.warmup // 2)):
        e2e_step()
    ms_e2e = timed(e2e_step, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    h2d = h2d_probe(h, x_host, x)

    # kernel-class breakdown of one step (events around every launch; after the timed region)
    breakdown = engine.profile_step(lambda: flow.log_prob(x))
    gemm_ms = sum(v for k, v in breakdown.items() if k.startswith("linear"))
    conv_names = ("im2col", "conv2d_rows", "pix_encode", "conv2d_pix")
    if len(spec["in_dims"]) > 1:            # image path: the convolutions (pixel planes, implicit GEMM, or gather + contraction)
        gemm_ms += sum(breakdown.get(k, 0.0) for k in conv_names)
    peaks, peak_kind = measured_peaks()
    traffic, traffic_step, traffic_src = committed_traffic(args.workload, args.precision)
    achieved_tf = rows * flops_per_sample / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    peak_tf = peaks["bf16_tflops_sustained"]
    n_gemm = sum(1 for k in breakdown.get("_names", []) if k.startswith("linear") or
                 (len(spec["in_dims"]) > 1 and k in conv_names)) or 1

    extra_modes = {}
    tf32_peak = None
    if not args.no_modes and world == 1:
        tf32_peak = measure_tf32_peak(torch, dev)
        for mode in ("fp32_tf32", "tf32", "bf16"):
            if mode == args.precision:
                continue
            f2 = build_flow(spec, params, device=dev, precision=mode)
            f2.log_prob(x[:256])
            for _ in range(2):
                f2.log_prob(x)
            ms = timed(lambda: f2.log_prob(x), max(3, args.steps // 2))
            ref = lp.double().cpu()
            err = float(((f2.log_prob(x[:256]).double().cpu() - ref).abs() / ref.abs().clamp(min=1)).max())
            bd = engine.profile_step(lambda: f2.log_prob(x))
            g_ms = sum(v for k, v in bd.items() if k.startswith("linear"))
            tf_k = rows * flops_per_sample / (g_ms * 1e-3) / 1e12 if g_ms > 0 else 0.0
            mode_peak = tf32_peak if mode == "tf32" else tf32_peak / 3.0 if mode == "fp32_tf32" else peak_tf
            extra_modes[mode] = dict(value=rows / (ms * 1e-3), ms_per_step=ms,
                                     tflops=rows * flops_per_sample / (ms * 1e-3) / 1e12,
                                     kernel_ms_per_step=g_ms, kernel_tflops=tf_k, frac=tf_k / peak_tf,
                                     frac_of_mode_peak=tf_k / mode_peak,
                                     mode_peak_tflops=mode_peak,
                                     mode_peak_source="cuBLAS tf32 8192^3 measured in this run" + (" / 3 products" if mode == "fp32_tf32" else "")
                                     if mode != "bf16" else f"bf16_tflops_sustained, of {peak_kind}",
                                     max_rel_diff_vs_fp32_mode=err)
            del f2

    train = None
    if not args.no_train and len(spec["in_dims"]) == 1 and spec.get("hidden_dims") and args.workload == "c2":
        train = run_train(h, U, O, build_flow, spec, args.steps)

    configs = None
    if not args.no_extra and args.workload == "c2":
        configs = dict(c4=run_c4(h, U, O, build_flow, max(3, args.steps // 2), peaks),
                       c5_sweep=run_c5_sweep(h, U, O, build_flow, peaks, args.sweep_full))
    elif args.workload == "c5" and args.sweep_full:
        configs = dict(c5_sweep=run_c5_sweep(h, U, O, build_flow, peaks, True))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    cpu = None
    if not args.no_cpu_baseline and world == 1:
        v_asis, v_am, cores, _ = cpu_reference_run(wl, 3, 1, wl["cpu_rows"])
        cpu = dict(value=v_asis, unit="samples/s", cores=cores, kind="port",
                   sample=f"{wl['cpu_rows']} rows x 3 steps of the same workload through the oracle port of the "
                          f"reference (torch CPU, per-call weight re-preparation as the reference does)",
                   amortised_value=v_am)

    roofline = dict(bound="tensor", achieved=achieved_tf, peak=peak_tf, unit="TFLOP/s",
                    frac=achieved_tf / peak_tf, traffic=traffic, traffic_per_step=traffic_step,
                    traffic_note=None if traffic is None else
                    f"dram__bytes_read.sum + dram__bytes_write.sum from the committed ncu --set full capture ({traffic_src}): "
                    f"`traffic` = mean PER LAUNCH of the dominant kernel, `traffic_per_step` = sum over its launches of one step",
                    peak_source=f"bf16_tflops_sustained, of {peak_kind}",
                    kernel="tc2::gemm_tc2_kernel (CTA-pair tcgen05, all launches of one step)" if len(spec["in_dims"]) == 1
                    else "convpix::conv_pix_kernel (ConvNet2D conditioners on pixel planes: TMA-box taps, tcgen05 kind::f16 x3; "
                         "convtc::conv_tc_kernel for other widths / modes) + pix_encode + the 1x1-convolution contractions, "
                         "all launches of one step",
                    kernel_ms_per_step=gemm_ms,
                    launches_per_step=n_gemm,
                    algorithmic_bytes_per_step=rows * (4 * d + 4),
                    note="algorithmic fp32 FLOPs over the summed CUDA-event time of the GEMM launches of one step; "
                         "the fp32 mode spends 3 fp16 MMAs per algorithmic MAC (fp16 runs at the bf16 rate), so its "
                         "ceiling is 1/3 of this peak (1/6 for fp32_tf32)",
                    frac_of_mode_ceiling=(achieved_tf / (peak_tf / MODE_PRODUCTS[args.precision]))
                    if args.precision in MODE_PRODUCTS else None,
                    tf32_peak_measured=tf32_peak)
    if breakdown.get("flow_small"):
        # tiny event size: the whole stack is one FP32-FMA bound launch (usf_flow_small); neither HBM nor the tensor pipe
        # bounds it, so the figure is set against the nominal FP32 FMA rate of the part (stated, not measured)
        sm_count = torch.cuda.get_device_properties(dev).multi_processor_count
        fma_peak = sm_count * 128 * 2 * 1.965e9 / 1e12
        ach = rows * flops_per_sample / (breakdown["flow_small"] * 1e-3) / 1e12
        roofline = dict(bound="fp32_fma", achieved=ach, peak=fma_peak, unit="TFLOP/s", frac=ach / fma_peak, traffic=None,
                        peak_source="nominal: SMs x 128 FMA lanes x 2 x 1965 MHz", kernel="flow_small_kernel",
                        kernel_ms_per_step=breakdown["flow_small"], launches_per_step=1,
                        hbm_gbs_for_context=rows * (4 * d + 4) / (breakdown["flow_small"] * 1e-3) / 1e9)

    line = dict(
        base_line, impl="usflows_b200", value=value, ms_per_step=ms_step,
        dtype={"fp32": "f32 (fp16-split x3 on tcgen05 kind::f16, fp32 accumulate/promote; tf32-split fallback)",
               "fp32_tf32": "f32 (tf32-split x3 on tcgen05 kind::tf32)", "fp32_simt": "f32", "tf32": "tf32",
               "bf16": "bf16"}[args.precision],
        config=dict(workload=wl["name"], rows_per_gpu_per_step=rows, d=d, hidden=spec.get("hidden_dims", spec.get("c_hidden")),
                    coupling_blocks=spec["coupling_blocks"], precision=args.precision,
                    chunk_rows=engine._default_chunk_rows if len(spec["in_dims"]) == 1 else
                    f"{__import__('usflows_b200.image_engine', fromlist=['x']).IMAGE_CHUNK_ROWS_PIX} channels-last rows "
                    f"(pixel-plane route; {__import__('usflows_b200.image_engine', fromlist=['x']).IMAGE_CHUNK_ROWS} on the others)",
                    l2="inputs larger than L2, no flush",
                    flops_per_sample=flops_per_sample, prep_ms_once_per_weight_version=prep_ms, first_call_ms=first_call_ms,
                    host_affinity=affinity),
        roofline=roofline,
        cpu_baseline=cpu,
        e2e=dict(value=world * rows / (ms_e2e * 1e-3), unit="samples/s", ms_per_step=ms_e2e,
                 h2d_bytes_per_step=rows * d * 4, d2h_bytes_per_step=rows * 4,
                 h2d_gbs_needed_per_rank=rows * d * 4 / (ms_e2e * 1e-3) / 1e9),
        h2d=h2d,
        sample=dict(metric="sample_samples_per_sec", value=world * rows / (ms_sample * 1e-3), unit="samples/s",
                    ms_per_step=ms_sample, tflops=rows * flops_per_sample / (ms_sample * 1e-3) / 1e12,
                    note="Flow.sample([rows]): Philox base draws + forward pass; same algorithmic FLOPs per sample"),
        train=train, configs=configs, gpu_launches=launches, clocks=clocks, modes=extra_modes,
        breakdown_ms={k: v for k, v in breakdown.items() if not k.startswith("_")})
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
