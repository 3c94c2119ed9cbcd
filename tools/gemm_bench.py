"""GEMM micro-benchmark / checker for the tcgen05 contraction kernels (run on the B200 box).

    python tools/gemm_bench.py [--engines 3xtf32,tf32,bf16] [--shapes 16384x784x784,...] [--bn 0] [--check]
                               [--iters 20] [--flags 0]

Prints one JSON line per (engine, shape): time, MMA-level TFLOP/s (counting every tensor-core pass), and the
error against an fp64 product when --check is given.
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

from usflows_b200 import _lib, ops  # noqa: E402
from usflows_b200.ops import Act  # noqa: E402

ENG = {"simt": ops.ENGINE_SIMT, "3xtf32": ops.ENGINE_TC_3XTF32, "tf32": ops.ENGINE_TC_TF32, "bf16": ops.ENGINE_TC_BF16,
       "3xf16": ops.ENGINE_TC_3XF16}
PASSES = {"simt": 1, "3xtf32": 3, "tf32": 1, "bf16": 1, "3xf16": 3}


def make_case(engine, M, N, K, seed, epi, dev="cuda"):
    g = torch.Generator().manual_seed(seed)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    bias = torch.randn(N, generator=g).to(dev) if epi else None
    ldk, ldn = ops.pad4(K), ops.pad4(N)
    af = torch.zeros(M, ldk, device=dev)[:, :K]; af.copy_(a)
    wf = torch.zeros(N, ldk, device=dev)[:, :K]; wf.copy_(w)
    out = Act(M, N)
    if engine == "bf16":
        ab = torch.zeros(M, ldk, dtype=torch.bfloat16, device=dev)[:, :K]; ab.copy_(a)
        wb = torch.zeros(N, ldk, dtype=torch.bfloat16, device=dev)[:, :K]; wb.copy_(w)
        act, wt, wl = Act(M, K, bf16=ab), wb, None
        ref_a, ref_w = ab.double(), wb.double()
        out.bf16 = torch.zeros(M, ldn, dtype=torch.bfloat16, device=dev)[:, :N]
        out.f32 = torch.zeros(M, ldn, device=dev)[:, :N]
    elif engine == "3xf16":
        ah, al = torch.zeros(2, M, ldk, dtype=torch.float16, device=dev)[:, :, :K]
        wh, wl = torch.zeros(2, N, ldk, dtype=torch.float16, device=dev)[:, :, :K]
        ops.split_f16(af, ah, al); ops.split_f16(wf, wh, wl)
        act, wt = Act(M, K, h16=ah, l16=al), wh
        ref_a, ref_w = af.double(), wf.double()
        out.h16, out.l16 = torch.zeros(2, M, ldn, dtype=torch.float16, device=dev)[:, :, :N]
    elif engine == "3xtf32":
        ah, al = torch.zeros(2, M, ldk, device=dev)[:, :, :K]
        wh, wl = torch.zeros(2, N, ldk, device=dev)[:, :, :K]
        ops.split_tf32(af, ah, al); ops.split_tf32(wf, wh, wl)
        act, wt = Act(M, K, hi=ah, lo=al), wh
        ref_a, ref_w = af.double(), wf.double()
        out.hi, out.lo = torch.zeros(2, M, ldn, device=dev)[:, :, :N]
    else:
        act, wt, wl = Act(M, K, f32=af), wf, None
        ref_a, ref_w = af.double(), wf.double()
        out.f32 = torch.zeros(M, ldn, device=dev)[:, :N]
    return act, wt, wl, bias, out, ref_a, ref_w


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--engines", default="3xf16,3xtf32,tf32,bf16")
    ap.add_argument("--shapes", default="16384x784x784,16384x1024x784,16384x1024x1024,16384x784x1024,16384x3072x3072")
    ap.add_argument("--bn", type=int, default=0)
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--check", action="store_true")
    ap.add_argument("--epi", action="store_true", help="bias + relu epilogue")
    ap.add_argument("--resid", action="store_true", help="3xf16: in-place coupling residual (out = out - (a.w^T + bias))")
    ap.add_argument("--flags", type=int, default=0,
                    help="usf_debug_set_store_path flags (4 = register/patch store, 32 = no TMA stores, 256 = residual without the in-box)")
    args = ap.parse_args()
    lib = _lib.load()
    lib.usf_debug_set_block_n(args.bn)
    _lib.check(lib.usf_debug_set_store_path(args.flags))
    print(torch.cuda.get_device_name(0), flush=True)
    for eng in args.engines.split(","):
        for shp in args.shapes.split(","):
            M, N, K = (int(v) for v in shp.split("x"))
            act, wt, wl, bias, out, ref_a, ref_w = make_case(eng, M, N, K, 0, args.epi)

            def run():
                if args.resid and eng == "3xf16":
                    ops.linear(ENG[eng], act, wt, wl, N, K, bias=bias, resid=out, resid_sign=-1.0, out=out)
                else:
                    ops.linear(ENG[eng], act, wt, wl, N, K, bias=bias, relu=args.epi, out=out)
            rec = dict(engine=eng, M=M, N=N, K=K, bn=args.bn, flags=args.flags)
            try:
                for _ in range(3):
                    run()
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(args.iters):
                    run()
                e1.record()
                torch.cuda.synchronize()
                us = e0.elapsed_time(e1) * 1e3 / args.iters
                rec.update(us=round(us, 1), alg_tflops=round(2 * M * N * K / us / 1e6, 1),
                           mma_tflops=round(PASSES[eng] * 2 * M * N * K / us / 1e6, 1))
                if args.check:
                    rows = min(M, 2048)
                    ref = ref_a[:rows] @ ref_w.T
                    if args.epi:
                        ref = torch.relu(ref + bias.double())
                    got = out.f32 if out.f32 is not None else (out.hi + out.lo) if out.hi is not None else \
                        (out.h16.float() + out.l16.float() / 2048.0)
                    err = float((got[:rows].double() - ref).abs().max() / ref.abs().max())
                    rec["max_err_rel"] = err
                    tail = ref_a[M - 300:] @ ref_w.T
                    if args.epi:
                        tail = torch.relu(tail + bias.double())
                    rec["tail_err_rel"] = float((got[M - 300:].double() - tail).abs().max() / tail.abs().max())
            except Exception as e:  # noqa: BLE001
                rec["error"] = repr(e)
            print(json.dumps(rec), flush=True)


if __name__ == "__main__":
    main()
