"""H2D bandwidth and host-buffer log_prob (e2e) timing probe (run on the B200 box)."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch
from usflows_b200.builders import build_flow
from oracle import flow_oracle as O
import bench

spec = bench.WORKLOADS["c2"]["spec"]
flow = build_flow(spec, O.random_params(spec, 0), device="cuda", precision="fp32")
rows, d = 65536, 784
x_host = torch.rand(rows, d).pin_memory()
out_host = torch.empty(rows).pin_memory()
x = torch.empty(rows, d, device="cuda")
def timed(fn, n=10):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n): fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / n * 1e3
ms = timed(lambda: x.copy_(x_host, non_blocking=True))
print(f"raw H2D {rows*d*4/1e6:.0f} MB: {ms:.2f} ms = {rows*d*4/ms/1e6:.1f} GB/s")
ms = timed(lambda: flow.log_prob(x))
print(f"device log_prob: {ms:.2f} ms")
for chunk in (None, 9472, 18944, 16384):
    ms = timed(lambda: flow.log_prob_host(x_host, out_host, chunk_rows=chunk))
    print(f"log_prob_host chunk {chunk}: {ms:.2f} ms = {rows/ms/1e3:.2f} M rows/s")
from usflows_b200 import _lib
for pdl in (0, 1):
    _lib.load().usf_debug_set_pdl(pdl)
    flow._program("backward")[0]._graphs.clear()            # re-capture with / without programmatic edges
    ms_dev = timed(lambda: flow.log_prob(x))
    ms = timed(lambda: flow.log_prob_host(x_host, out_host))
    print(f"pdl={pdl}: device log_prob {ms_dev:.3f} ms, log_prob_host {ms:.3f} ms = {rows/ms/1e3:.2f} M rows/s")
