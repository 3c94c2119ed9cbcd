"""First-contact diagnostics on a B200: exercises every kernel family and prints errors instead of asserting.
Usage (GPU box):  python tools/gpu_probe.py [--quick]"""
import json
import os
import sys
import time
import traceback

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

import usflows_b200 as U  # noqa: E402
from usflows_b200 import _lib, ops  # noqa: E402
from usflows_b200.ops import Act  # noqa: E402
from helpers import build_flow, load_case, rel_err, SMALL_CASES, LARGE_CASES  # noqa: E402

RESULTS = {}


def section(name):
    def deco(fn):
        t = time.time()
        try:
            out = fn()
            RESULTS[name] = out
            print(f"[{name}] {json.dumps(out)}  ({time.time() - t:.1f}s)", flush=True)
        except Exception as e:  # noqa: BLE001
            RESULTS[name] = {"error": repr(e)}
            print(f"[{name}] ERROR {e!r}", flush=True)
            traceback.print_exc()
        return fn
    return deco


def gemm_case(engine, M, N, K, bn=0, seed=0, epi=False):
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    bias = torch.randn(N, generator=g)
    ref = a.double() @ w.double().T
    if epi:
        ref = torch.relu(ref + bias.double())
    dev = "cuda"
    ld = ops.pad4(K)
    out = torch.zeros(M, ops.pad4(N), device=dev)[:, :N]
    _lib.load().usf_debug_set_block_n(bn)
    if engine == ops.ENGINE_TC_BF16:
        ab = torch.zeros(M, ld, dtype=torch.bfloat16, device=dev)[:, :K]; ab.copy_(a)
        wb = torch.zeros(N, ld, dtype=torch.bfloat16, device=dev)[:, :K]; wb.copy_(w)
        act, wt, wl = Act(M, K, bf16=ab), wb, None
        ref = ab.double().cpu() @ wb.double().cpu().T
        if epi:
            ref = torch.relu(ref + bias.double())
    elif engine == ops.ENGINE_TC_3XTF32:
        af = torch.zeros(M, ld, device=dev)[:, :K]; af.copy_(a)
        wf = torch.zeros(N, ld, device=dev)[:, :K]; wf.copy_(w)
        ah, al = torch.zeros(2, M, ld, device=dev)[:, :, :K]
        wh, wl = torch.zeros(2, N, ld, device=dev)[:, :, :K]
        ops.split_tf32(af, ah, al); ops.split_tf32(wf, wh, wl)
        act, wt = Act(M, K, hi=ah, lo=al), wh
    else:
        af = torch.zeros(M, ld, device=dev)[:, :K]; af.copy_(a)
        wf = torch.zeros(N, ld, device=dev)[:, :K]; wf.copy_(w)
        act, wt, wl = Act(M, K, f32=af), wf, None
    ops.linear(engine, act, wt, wl, N, K, bias=bias.to(dev) if epi else None, relu=epi, out=Act(M, N, f32=out))
    torch.cuda.synchronize()
    _lib.load().usf_debug_set_block_n(0)
    return rel_err(out, ref)


quick = "--quick" in sys.argv
print(torch.cuda.get_device_name(0), torch.version.cuda, flush=True)

if "--tc-smoke" in sys.argv:      # run under a short `timeout`: catches protocol deadlocks cheaply
    for eng in (ops.ENGINE_TC_3XTF32, ops.ENGINE_TC_TF32, ops.ENGINE_TC_BF16):
        for bn in (32, 128, 208, 256):
            print("tc-smoke", eng, bn, gemm_case(eng, 300, 520, 256, bn=bn, epi=True), flush=True)
    sys.exit(0)


@section("simt_gemm")
def _():
    return {f"{M}x{N}x{K}": gemm_case(ops.ENGINE_SIMT, M, N, K, epi=True) for M, N, K in [(5, 3, 2), (130, 70, 33), (256, 784, 1024)]}


for eng_name, eng in [("tf32", ops.ENGINE_TC_TF32), ("3xtf32", ops.ENGINE_TC_3XTF32), ("bf16", ops.ENGINE_TC_BF16)]:
    @section(f"tc_{eng_name}_basic")
    def _(eng=eng):
        return {"128x128x32_bn128": gemm_case(eng, 128, 128, 32 if eng != ops.ENGINE_TC_BF16 else 64, bn=128)}

    @section(f"tc_{eng_name}_shapes")
    def _(eng=eng):
        out = {}
        for (M, N, K, bn) in [(128, 256, 256, 256), (256, 784, 1024, 0), (300, 1024, 784, 0), (1000, 3072, 1000, 0),
                              (77, 100, 50, 0), (4096, 784, 784, 208), (4096, 784, 784, 224), (512, 96, 96, 96),
                              (512, 64, 160, 64), (512, 160, 64, 160), (512, 192, 40, 192), (333, 32, 36, 32)]:
            out[f"{M}x{N}x{K}_bn{bn}"] = gemm_case(eng, M, N, K, bn=bn, epi=True)
        return out


@section("tri_inverse")
def _():
    out = {}
    for d in [5, 64, 100, 784]:
        g = torch.Generator().manual_seed(d)
        L = (torch.rand(d, d, generator=g) * 0.1).tril(-1) + torch.eye(d)
        Uu = (torch.rand(d, d, generator=g) * 0.1).triu(1) + torch.diag(torch.rand(d, generator=g) + 0.5)
        X = torch.empty(d, d, device="cuda")
        ops.tri_inverse(L.cuda(), True, True, X)
        out[f"L{d}"] = rel_err(X, torch.inverse(L.double()))
        ops.tri_inverse(Uu.cuda(), False, False, X)
        out[f"U{d}"] = rel_err(X, torch.inverse(Uu.double()))
    return out


def flow_case(name, mode):
    spec, params, arr = load_case(name)
    flow = build_flow(spec, params, precision=mode)
    x, z0 = arr["x"].cuda(), arr["z0"].cuda()
    lp = flow.log_prob(x)
    z = flow.backward(x)
    y = flow._forward(z0)
    torch.cuda.synchronize()
    return dict(lp_vs_ref32=rel_err(lp, arr["lp32"]), lp_vs_f64=rel_err(lp, arr["lp64"]), ref32_vs_f64=rel_err(arr["lp32"], arr["lp64"]),
                z_vs_ref32=rel_err(z, arr["z32"]), z_vs_f64=rel_err(z, arr["z64"]), zref_vs_f64=rel_err(arr["z32"], arr["z64"]),
                y_vs_ref32=rel_err(y, arr["y32"]), y_vs_f64=rel_err(y, arr["y64"]), yref_vs_f64=rel_err(arr["y32"], arr["y64"]))


def time_gemm(engine, M, N, K, bn, iters=10):
    dev = "cuda"
    lib = _lib.load()
    lib.usf_debug_set_block_n(bn)
    ld = ops.pad4(K)
    if engine == ops.ENGINE_TC_BF16:
        a = Act(M, K, bf16=torch.randn(M, ld, device=dev).to(torch.bfloat16)[:, :K])
        w, wl = torch.randn(N, ld, device=dev).to(torch.bfloat16)[:, :K], None
        out = Act(M, N, bf16=torch.empty(M, ops.pad4(N), device=dev, dtype=torch.bfloat16)[:, :N])
    elif engine == ops.ENGINE_TC_3XTF32:
        a = Act(M, K, hi=torch.randn(M, ld, device=dev)[:, :K], lo=torch.randn(M, ld, device=dev)[:, :K] * 1e-4)
        w, wl = torch.randn(N, ld, device=dev)[:, :K], torch.randn(N, ld, device=dev)[:, :K] * 1e-4
        out = Act(M, N, hi=torch.empty(M, ops.pad4(N), device=dev)[:, :N], lo=torch.empty(M, ops.pad4(N), device=dev)[:, :N])
    else:
        a = Act(M, K, f32=torch.randn(M, ld, device=dev)[:, :K])
        w, wl = torch.randn(N, ld, device=dev)[:, :K], None
        out = Act(M, N, f32=torch.empty(M, ops.pad4(N), device=dev)[:, :N])
    bias = torch.randn(N, device=dev)
    run = lambda: ops.linear(engine, a, w, wl, N, K, bias=bias, relu=True, out=out)  # noqa: E731
    for _ in range(3):
        run()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        run()
    e1.record()
    torch.cuda.synchronize()
    lib.usf_debug_set_block_n(0)
    ms = e0.elapsed_time(e1) / iters
    return round(2.0 * M * N * K / (ms * 1e-3) / 1e12, 1)


if "--perf" in sys.argv:
    for eng_name, eng in [("3xtf32", ops.ENGINE_TC_3XTF32), ("tf32", ops.ENGINE_TC_TF32), ("bf16", ops.ENGINE_TC_BF16), ("simt", ops.ENGINE_SIMT)]:
        @section(f"perf_{eng_name}_TFLOPs")
        def _(eng=eng, eng_name=eng_name):
            out = {}
            for (M, N, K) in [(16384, 1024, 1024), (16384, 784, 784), (16384, 1024, 784), (16384, 784, 1024), (16384, 3072, 3072), (65536, 1024, 1024)]:
                if eng == ops.ENGINE_SIMT:
                    out[f"{M}x{N}x{K}"] = time_gemm(eng, M, N, K, 0, iters=3)
                    continue
                for bn in ([256, 208, 128] if N != 1024 and N != 3072 else [256, 128]):
                    out[f"{M}x{N}x{K}_bn{bn}"] = time_gemm(eng, M, N, K, bn)
            return out

modes = ["fp32"] if "--fp32-only" in sys.argv else ["fp32_simt", "fp32", "tf32", "bf16"]
for mode in modes:
    for name in SMALL_CASES + ([] if quick else LARGE_CASES):
        section(f"flow_{mode}_{name}")(lambda name=name, mode=mode: flow_case(name, mode))

os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
with open(os.path.join(ROOT, "gpurun_out", "probe.json"), "w") as f:
    json.dump(RESULTS, f, indent=1)
print("done")
