"""Samples to host memory on the B200: `sample([n], seed=s).cpu()` (what a caller does without the host path) against
`sample_host(n, seed=s)` in fp32 and `sample_host(n, seed=s, quantize=True)`, for C2 (fp32 and bf16 modes) and mnist_img.

    python tools/sample_probe.py --out DIR [--reps N] [--warmup W]

The three ways are timed alternately (N times each) after warm-up, every call ending in a device synchronise; the median
per call is reported with rows/s, next to the device-resident `sample` alone (CUDA events).  Before timing, both host
results are checked to equal the device samples bit for bit.  Also measured: the device-to-host copy rate alone (the fp32
output of one call into pinned memory) and the usf_quantize_u8 pass over one default chunk as a share of that chunk's
device-resident sampling time.  The GPU name and power limit (read-only nvidia-smi query) are recorded next to the
numbers; the JSON goes to DIR/sample_host_probe.json."""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import WORKLOADS  # noqa: E402
from tools.u8_probe import gpu_info  # noqa: E402


def wall_ms(fns, reps):
    """Alternating median wall time per call (ms) of each of fns; every call ends in a device synchronise."""
    acc = [[] for _ in fns]
    for _ in range(reps):
        for fn, a in zip(fns, acc):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            a.append((time.perf_counter() - t0) * 1e3)
    return [statistics.median(a) for a in acc], acc


def event_ms(fn, reps):
    ts = []
    for _ in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        ts.append(s.elapsed_time(e))
    return statistics.median(ts)


def probe(name, precision, reps, warmup):
    from usflows_b200 import flows, ops
    from usflows_b200.builders import build_flow
    from oracle import flow_oracle as O
    wl = WORKLOADS[name]
    spec, rows = wl["spec"], wl["rows"]
    dev = torch.device("cuda", 0)
    flow = build_flow(spec, O.random_params(spec, 0), device=dev, precision=precision)
    ev = tuple(spec["in_dims"])
    d = 1
    for v in ev:
        d *= v
    seed = 12345
    res = {"workload": name, "precision": precision, "rows": rows, "d": d}
    ref = flow.sample([rows], seed=seed)
    out_f = torch.empty(rows, *ev, dtype=torch.float32).pin_memory()
    out_u = torch.empty(rows, *ev, dtype=torch.uint8).pin_memory()
    res["equal_fp32"] = bool(torch.equal(flow.sample_host(rows, out_f, seed=seed), ref.cpu()))
    res["equal_uint8"] = bool(torch.equal(flow.sample_host(rows, out_u, seed=seed, quantize=True), ops.quantize(ref).cpu()))

    def device_then_copy():
        flow.sample([rows], seed=seed).cpu()

    def host_f():
        flow.sample_host(rows, out_f, seed=seed)

    def host_u():
        flow.sample_host(rows, out_u, seed=seed, quantize=True)
    for fn in (device_then_copy, host_f, host_u):
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    med, alls = wall_ms([device_then_copy, host_f, host_u], reps)
    res["ms"] = {"sample_then_cpu": med[0], "sample_host_fp32": med[1], "sample_host_uint8": med[2]}
    res["ms_all"] = {"sample_then_cpu": alls[0], "sample_host_fp32": alls[1], "sample_host_uint8": alls[2]}
    res["device_sample_ms"] = event_ms(lambda: flow.sample([rows], seed=seed), reps)
    res["rows_per_s"] = {k: rows / (v * 1e-3) for k, v in res["ms"].items()}
    res["d2h_bytes_per_call"] = {"fp32": rows * d * 4, "uint8": rows * d}
    # the device-to-host copy alone: one call's fp32 output into pinned memory
    copy_ms = event_ms(lambda: out_f.copy_(ref, non_blocking=True), reps)
    res["d2h_copy_ms"] = copy_ms
    res["d2h_GB_per_s"] = rows * d * 4 / (copy_ms * 1e-3) / 1e9
    # usf_quantize_u8 over one default chunk against that chunk's device-resident sampling
    prog = flow._program("forward")[0]
    chunk = min(rows, flows._wave_aligned_chunk_rows(prog, dev) if len(ev) == 1 else rows)
    y = ref.reshape(rows, d)[:chunk].contiguous()
    q = torch.empty(chunk, d, dtype=torch.uint8, device=dev)
    res["chunk_rows"] = chunk
    res["quantize_chunk_ms"] = event_ms(lambda: ops.quantize_u8(y, q), reps)
    res["sample_chunk_ms"] = event_ms(lambda: flow.sample([chunk], seed=seed), reps)
    res["quantize_share_of_chunk"] = res["quantize_chunk_ms"] / res["sample_chunk_ms"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory that receives sample_host_probe.json")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sample_probe: no CUDA device")
    results = {"gpu": gpu_info(), "runs": []}
    for name, precision in (("c2", "fp32"), ("c2", "bf16"), ("mnist_img", "fp32")):
        r = probe(name, precision, args.reps, args.warmup)
        results["runs"].append(r)
        print(json.dumps({k: (round(v, 4) if isinstance(v, float) else v) for k, v in r.items() if k not in ("ms_all", "ms")}
                         | {"ms": {k: round(v, 3) for k, v in r["ms"].items()}}), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "sample_host_probe.json"), "w") as f:
        json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
