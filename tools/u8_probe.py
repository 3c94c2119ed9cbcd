"""8-bit input vs fp32 input on the B200: device-resident log_prob, log_prob_host from pinned memory and the row-shard
driver over every visible GPU, for C2 (65 536 rows; fp32 and bf16 modes) and mnist_img (16 384 images).

    python tools/u8_probe.py --out DIR [--reps N] [--warmup W]

Each pair is timed alternately (fp32 input, then uint8 input, N times) with CUDA events after warm-up; the median per call
is reported with rows/s and the host-to-device bytes of one call.  Before timing, the uint8 result is checked to equal
`log_prob(dequantize(x_u8, seed=s))` at the timed size.  The GPU name and power limit (read-only nvidia-smi query) are
recorded next to the numbers; the JSON goes to DIR/u8_probe.json."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from bench import WORKLOADS  # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
    except (OSError, subprocess.SubprocessError):
        q = []
    return {"nvidia_smi": q, "torch_name": torch.cuda.get_device_name(0), "device_count": torch.cuda.device_count()}


def timed_pair(fa, fb, reps, sync_devices):
    """Alternating median wall time per call (ms) of fa and fb; every call ends in a device synchronise."""
    ta, tb = [], []
    for _ in range(reps):
        for fn, acc in ((fa, ta), (fb, tb)):
            for d in sync_devices:
                torch.cuda.synchronize(d)
            t0 = time.perf_counter()
            fn()
            for d in sync_devices:
                torch.cuda.synchronize(d)
            acc.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ta), statistics.median(tb), ta, tb


def event_pair(fa, fb, reps):
    """Alternating median device time per call (ms, CUDA events on the current stream)."""
    ta, tb = [], []
    for _ in range(reps):
        for fn, acc in ((fa, ta), (fb, tb)):
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            fn()
            e.record()
            e.synchronize()
            acc.append(s.elapsed_time(e))
    return statistics.median(ta), statistics.median(tb), ta, tb


def probe(name, precision, reps, warmup):
    import usflows_b200 as U
    from usflows_b200 import parallel
    from usflows_b200.builders import build_flow
    from oracle import flow_oracle as O
    wl = WORKLOADS[name]
    spec, rows = wl["spec"], wl["rows"]
    dev = torch.device("cuda", 0)
    flow = build_flow(spec, O.random_params(spec, 0), device=dev, precision=precision)
    g = torch.Generator().manual_seed(1)
    xu_host = torch.randint(0, 256, (rows, *spec["in_dims"]), generator=g, dtype=torch.uint8).pin_memory()
    xu = xu_host.to(dev)
    seed = 12345
    xf = U.dequantize(xu, "uniform", seed=seed)
    xf_host = xf.cpu().pin_memory()
    d = xf[0].numel()
    res = {"workload": name, "precision": precision, "rows": rows, "d": d}

    lp_f = flow.log_prob(xf)
    lp_u = flow.log_prob(xu, dequantize="uniform", seed=seed)
    res["equal_device"] = bool(torch.equal(lp_f, lp_u))
    res["equal_host"] = bool(torch.equal(flow.log_prob_host(xu_host, dequantize="uniform", seed=seed), lp_f.cpu()))
    devices = list(range(torch.cuda.device_count()))
    res["equal_sharded"] = bool(torch.equal(parallel.log_prob_sharded(flow, xu_host, dequantize="uniform", seed=seed),
                                            lp_f.cpu()))

    def dev_f():
        flow.log_prob(xf)

    def dev_u():
        flow.log_prob(xu, dequantize="uniform", seed=seed)
    out_host = torch.empty(rows, dtype=torch.float32).pin_memory()

    def host_f():
        flow.log_prob_host(xf_host, out_host)

    def host_u():
        flow.log_prob_host(xu_host, out_host, dequantize="uniform", seed=seed)

    def sh_f():
        parallel.log_prob_sharded(flow, xf_host, out_host=out_host)

    def sh_u():
        parallel.log_prob_sharded(flow, xu_host, out_host=out_host, dequantize="uniform", seed=seed)
    for fn in (dev_f, dev_u, host_f, host_u, sh_f, sh_u):
        for _ in range(warmup):
            fn()
    torch.cuda.synchronize()
    a, b, ra, rb = event_pair(dev_f, dev_u, reps)
    res["device_ms"] = {"fp32": a, "uint8": b, "fp32_all": ra, "uint8_all": rb}
    a, b, ra, rb = timed_pair(host_f, host_u, reps, [dev])
    res["host_ms"] = {"fp32": a, "uint8": b, "fp32_all": ra, "uint8_all": rb}
    a, b, ra, rb = timed_pair(sh_f, sh_u, reps, [torch.device("cuda", i) for i in devices])
    res["sharded_ms"] = {"fp32": a, "uint8": b, "gpus": len(devices), "fp32_all": ra, "uint8_all": rb}
    res["h2d_bytes_per_call"] = {"fp32": rows * d * 4, "uint8": rows * d}
    res["rows_per_s"] = {k: {m: rows / (res[k][m] * 1e-3) for m in ("fp32", "uint8")}
                         for k in ("device_ms", "host_ms", "sharded_ms")}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory that receives u8_probe.json")
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("u8_probe: no CUDA device")
    results = {"gpu": gpu_info(), "runs": []}
    for name, precision in (("c2", "fp32"), ("c2", "bf16"), ("mnist_img", "fp32")):
        r = probe(name, precision, args.reps, args.warmup)
        results["runs"].append(r)
        print(json.dumps({k: v for k, v in r.items() if k not in ("device_ms", "host_ms", "sharded_ms")}
                         | {k: {m: round(r[k][m], 3) for m in ("fp32", "uint8")} for k in ("device_ms", "host_ms", "sharded_ms")}),
              flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "u8_probe.json"), "w") as f:
        json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
