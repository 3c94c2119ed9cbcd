"""Unit tests of individual C-ABI kernels against fp64 torch-CPU arithmetic (run with -m gpu on the B200)."""
import pytest
import torch

from helpers import rel_err

pytestmark = pytest.mark.gpu


def _planes(t, kind):
    from usflows_b200 import ops
    from usflows_b200.ops import Act
    M, K = t.shape
    ld = ops.pad4(K)
    dev = "cuda"
    if kind == "bf16":
        b = torch.zeros(M, ld, dtype=torch.bfloat16, device=dev)[:, :K]
        b.copy_(t)
        return Act(M, K, bf16=b), b.float().cpu()
    f = torch.zeros(M, ld, device=dev)[:, :K]
    f.copy_(t)
    if kind == "split":
        hi, lo = torch.zeros(2, M, ld, device=dev)[:, :, :K]
        ops.split_tf32(f, hi, lo)
        return Act(M, K, hi=hi, lo=lo), (hi.double() + lo.double()).cpu()
    return Act(M, K, f32=f), t


ENGINES = [("simt", 0, "f32", 3e-6), ("3xtf32", 1, "split", 3e-6), ("tf32", 2, "f32", 2e-3), ("bf16", 3, "bf16", 3e-6)]


@pytest.mark.parametrize("eng_name,eng,fmt,tol", ENGINES)
@pytest.mark.parametrize("M,N,K", [(1, 40, 40), (128, 128, 32), (300, 784, 1024), (1000, 1024, 784), (257, 3072, 520),
                                   (513, 100, 50), (64, 33, 47), (300, 784, 784), (1000, 1024, 392), (515, 392, 1024),
                                   (257, 208, 72), (64, 48, 40)])
def test_linear_all_engines_full_epilogue(eng_name, eng, fmt, tol, M, N, K):
    from usflows_b200 import ops
    from usflows_b200.ops import Act
    if eng != 0 and min(N, K) < 32:
        pytest.skip("tcgen05 engines are used for N, K >= 32")
    g = torch.Generator().manual_seed(M * 7 + N)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    bias, colscale, postsub = (torch.randn(N, generator=g) for _ in range(3))
    resid = torch.randn(M, N, generator=g)
    act, a_used = _planes(a, fmt)
    wact, w_used = _planes(w, fmt)
    racc, r_used = _planes(resid, "split" if fmt == "split" else "f32")
    w_hi = wact.bf16 if fmt == "bf16" else (wact.hi if fmt == "split" else wact.f32)
    out = Act(M, N, f32=torch.zeros(M, ops.pad4(N), device="cuda")[:, :N],
              hi=torch.zeros(M, ops.pad4(N), device="cuda")[:, :N], lo=torch.zeros(M, ops.pad4(N), device="cuda")[:, :N],
              bf16=torch.zeros(M, ops.pad4(N), device="cuda", dtype=torch.bfloat16)[:, :N])
    ops.linear(eng, act, w_hi, wact.lo, N, K, bias=bias.cuda(), relu=True, resid=racc, resid_sign=-1.0,
               colscale=colscale.cuda(), postsub=postsub.cuda(), out=out)
    ref = torch.relu(a_used.double() @ w_used.double().T + bias.double())
    ref = (r_used.double() - ref) * colscale.double() - postsub.double()
    assert rel_err(out.f32, ref) <= tol
    assert rel_err(out.hi.double() + out.lo.double(), out.f32) <= 1e-6          # split planes reconstruct the value
    assert rel_err(out.bf16.float(), out.f32) <= 1e-2


@pytest.mark.parametrize("M,N,K", [(4096, 16, 16), (50000, 16, 16), (7001, 10, 7), (4100, 3, 16), (9000, 16, 5)])
def test_narrow_rows_kernel_full_epilogue(M, N, K):
    """The SIMT engine's narrow fast path (N, K <= 16, many rows: the 16 x 16 1x1-convolution affine layers of the image
    flows): the same full epilogue as the tiled kernel, against fp64."""
    from usflows_b200 import ops
    from usflows_b200.ops import Act
    g = torch.Generator().manual_seed(M + N + K)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    bias, colscale, postsub = (torch.randn(N, generator=g) for _ in range(3))
    resid = torch.randn(M, N, generator=g)
    act, _ = _planes(a, "f32")
    wact, _ = _planes(w, "f32")
    racc, _ = _planes(resid, "f32")
    out = Act(M, N, f32=torch.zeros(M, ops.pad4(N), device="cuda")[:, :N],
              hi=torch.zeros(M, ops.pad4(N), device="cuda")[:, :N], lo=torch.zeros(M, ops.pad4(N), device="cuda")[:, :N])
    ops.linear(0, act, wact.f32, None, N, K, bias=bias.cuda(), relu=True, resid=racc, resid_sign=-1.0,
               colscale=colscale.cuda(), postsub=postsub.cuda(), out=out)
    ref = torch.relu(a.double() @ w.double().T + bias.double())
    ref = (resid.double() - ref) * colscale.double() - postsub.double()
    assert rel_err(out.f32, ref) <= 3e-6
    assert rel_err(out.hi.double() + out.lo.double(), out.f32) <= 1e-6
    plain = torch.empty(M, N, device="cuda")                       # dense output, no epilogue terms
    ops.linear(0, act, wact.f32, None, N, K, out=Act(M, N, f32=plain))
    assert rel_err(plain, a.double() @ w.double().T) <= 3e-6


@pytest.mark.parametrize("bn", [32, 64, 128, 208, 256])
def test_tile_widths(bn):
    """Every tcgen05 tile width on the 3xTF32 engine (several accumulation chains per tile) against fp64."""
    from usflows_b200 import _lib, ops
    from usflows_b200.ops import Act
    M, N, K = 400, 600, 500
    g = torch.Generator().manual_seed(bn)
    a, w = torch.randn(M, K, generator=g), torch.randn(N, K, generator=g) / K ** 0.5
    act, a_used = _planes(a, "split")
    wact, w_used = _planes(w, "split")
    out = Act(M, N, f32=torch.zeros(M, ops.pad4(N), device="cuda")[:, :N])
    lib = _lib.load()
    lib.usf_debug_set_block_n(bn)
    try:
        ops.linear(1, act, wact.hi, wact.lo, N, K, out=out)
        torch.cuda.synchronize()
    finally:
        lib.usf_debug_set_block_n(0)
    assert rel_err(out.f32, a_used.double() @ w_used.double().T) <= 3e-6


def test_simt_transposed_weight_and_unaligned():
    from usflows_b200 import ops
    g = torch.Generator().manual_seed(0)
    a, b = torch.randn(37, 53, generator=g), torch.randn(53, 29, generator=g)
    out = torch.empty(37, 29, device="cuda")
    ops.matmul_f32(a.cuda(), b.cuda(), out)
    assert rel_err(out, a.double() @ b.double()) <= 2e-6


def test_ingest_and_base_logprob():
    from usflows_b200 import ops
    from usflows_b200.ops import Act
    g = torch.Generator().manual_seed(1)
    for rows, d in [(7, 5), (300, 784), (129, 3072)]:
        x = torch.rand(rows, d, generator=g)
        div, sub = torch.rand(d, generator=g) + 0.5, torch.randn(d, generator=g)
        out = Act(rows, d, f32=torch.empty(rows, d, device="cuda"),
                  hi=torch.zeros(rows, ops.pad4(d), device="cuda")[:, :d], lo=torch.zeros(rows, ops.pad4(d), device="cuda")[:, :d])
        ops.ingest(x.cuda(), out, div=div.cuda(), sub=sub.cuda())
        ref = x / div - sub
        assert torch.equal(out.f32.cpu(), ref)                                   # same fp32 ops, bit exact
        assert rel_err(out.hi.double() + out.lo.double(), ref) <= 3e-7
        loc, scale = torch.randn(d, generator=g), torch.rand(d, generator=g) + 0.5
        res = torch.empty(rows, device="cuda")
        for kind, dist in ((ops.BASE_LAPLACE, torch.distributions.Laplace), (ops.BASE_NORMAL, torch.distributions.Normal)):
            ops.base_logprob(Act(rows, d, f32=out.f32), loc.cuda(), scale.cuda(), kind, 1.25, res)
            want = dist(loc.double(), scale.double()).log_prob(ref.double()).sum(-1) + 1.25
            assert rel_err(res, want) <= 2e-6


@pytest.mark.parametrize("d", [1, 5, 64, 100, 784, 1500])
def test_triangular_inverse_and_lu_prep(d):
    from usflows_b200 import ops
    g = torch.Generator().manual_seed(d)
    L_raw = torch.randn(d, d, generator=g) * (0.6 / d ** 0.5)
    U_raw = torch.randn(d, d, generator=g) * (0.6 / d ** 0.5)
    U_raw = U_raw.triu(1) + torch.diag(torch.sign(torch.randn(d, generator=g)) * torch.exp(torch.randn(d, generator=g) * 0.1))
    L, U = torch.empty(d, d, device="cuda"), torch.empty(d, d, device="cuda")
    ops.lu_assemble(L_raw.cuda(), U_raw.cuda(), L, U)
    assert torch.equal(L.cpu(), L_raw.tril(-1) + torch.eye(d)) and torch.equal(U.cpu(), U_raw.triu())
    X = torch.empty(d, d, device="cuda")
    ops.tri_inverse(L, True, True, X)
    assert rel_err(X, torch.inverse(L.double().cpu())) <= 2e-6
    ops.tri_inverse(U, False, False, X)
    assert rel_err(X, torch.inverse(U.double().cpu())) <= 2e-6
    out2 = torch.empty(2, device="cuda")
    ops.lu_logabsdet(U_raw.cuda(), out2)
    assert abs(float(out2[0]) - float(U_raw.diag().abs().log().double().sum())) <= 1e-5 * max(1.0, d ** 0.5)
    assert float(out2[1]) == 0


def test_reference_known_answer_triangular_solve():
    """The reference's own triangular-solve test (tests/veriflow/linalg_test.py:7-20: all-ones lower / upper triangular
    10 x 10 systems, 10 random right-hand sides, tolerance 1e-5), through the kernels that replace the triangular
    solves on this path: X = T^-1 by usf_tri_inverse, then x = X y as a contraction."""
    from usflows_b200 import ops
    torch.manual_seed(0)
    x = torch.stack([torch.rand(10) for _ in range(10)])
    for lower in (True, False):
        M = torch.tril(torch.ones(10, 10)) if lower else torch.triu(torch.ones(10, 10))
        y = torch.stack([M @ xi for xi in x])
        X = torch.empty(10, 10, device="cuda")
        ops.tri_inverse(M.cuda(), lower, False, X)
        got = torch.empty(10, 10, device="cuda")
        ops.linear(ops.ENGINE_SIMT, ops.Act(10, 10, f32=y.cuda()), X, None, 10, 10, out=ops.Act(10, 10, f32=got))
        assert bool(((got.cpu() - x).abs() < 1e-5).all())


def test_householder_and_transpose():
    from usflows_b200 import ops
    g = torch.Generator().manual_seed(3)
    d = 130
    W = torch.randn(d, d, generator=g)
    v = torch.randn(d, generator=g)
    Wd = W.cuda().clone()
    ops.householder_right(Wd, v.cuda(), torch.empty(d, device="cuda"))
    ref = W.double() @ (torch.eye(d, dtype=torch.float64) - 2 * torch.outer(v.double(), v.double()) / v.double().dot(v.double()))
    assert rel_err(Wd, ref) <= 2e-6
    Wt = torch.empty(d, d, device="cuda")
    ops.transpose(Wd, Wt)
    assert torch.equal(Wt.cpu(), Wd.cpu().T)


def test_errors_are_loud():
    from usflows_b200 import ops
    from usflows_b200.ops import Act
    with pytest.raises(RuntimeError, match="usflows_b200"):
        a = Act(4, 40, f32=torch.zeros(4, 41, device="cuda")[:, 1:])      # misaligned operand for a tcgen05 engine
        ops.linear(2, a, torch.zeros(40, 40, device="cuda"), None, 40, 40, out=Act(4, 40, f32=torch.zeros(4, 40, device="cuda")))


def _f16_planes(t):
    from usflows_b200 import ops
    from usflows_b200.ops import Act
    M, K = t.shape
    ld = ops.pad4(K)
    f = torch.zeros(M, ld, device="cuda")[:, :K]
    f.copy_(t)
    h, l = torch.zeros(2, M, ld, dtype=torch.float16, device="cuda")[:, :, :K]
    ops.split_f16(f, h, l)
    return Act(M, K, h16=h, l16=l), (h.double() + l.double() / 2048.0).cpu()


@pytest.mark.parametrize("M,N,K", [(1, 40, 40), (300, 784, 1024), (1000, 392, 784), (777, 1024, 392), (257, 3072, 520),
                                   (513, 100, 56), (2048, 224, 72), (640, 432, 1000), (300, 784, 784), (1000, 1024, 392),
                                   (515, 392, 1024), (257, 208, 72), (64, 48, 40)])
def test_fp16_split_engine_full_epilogue(M, N, K):
    """3 x fp16 tensor-core products with the fp16-split residual and output planes (the default fp32 mode)."""
    from usflows_b200 import ops
    from usflows_b200.ops import Act
    g = torch.Generator().manual_seed(M + 3 * N + K)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    bias, colscale, postsub = (torch.randn(N, generator=g) for _ in range(3))
    resid = torch.randn(M, N, generator=g)
    act, a_used = _f16_planes(a)
    wact, w_used = _f16_planes(w)
    racc, r_used = _f16_planes(resid)
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    out = Act(M, N, f32=torch.zeros(M, ops.pad4(N), device="cuda")[:, :N])
    out.h16, out.l16 = torch.zeros(2, M, ops.pad4(N), dtype=torch.float16, device="cuda")[:, :, :N]
    ops.linear(ops.ENGINE_TC_3XF16, act, wact.h16, wact.l16, N, K, bias=bias.cuda(), relu=True, resid=racc, resid_sign=-1.0,
               colscale=colscale.cuda(), postsub=postsub.cuda(), out=out, overflow_flag=flag)
    ref = torch.relu(a_used @ w_used.T + bias.double())
    ref = (r_used - ref) * colscale.double() - postsub.double()
    assert rel_err(out.f32, ref) <= 3e-6
    assert rel_err(out.h16.double() + out.l16.double() / 2048.0, out.f32) <= 1e-6
    assert int(flag) == 0


@pytest.mark.parametrize("eng_name,eng,fmt", [("3xtf32", 1, "split"), ("tf32", 2, "f32"), ("bf16", 3, "bf16"), ("3xf16", 4, "f16")])
@pytest.mark.parametrize("M,N,K", [(300, 784, 392), (515, 392, 1024), (130, 600, 72), (64, 48, 40), (513, 100, 56)])
def test_forced_store_paths_equal_the_staged_store(eng_name, eng, fmt, M, N, K):
    """The staged coalesced-store epilogue and the generic register/patch epilogue produce identical bits."""
    from usflows_b200 import _lib, ops
    from usflows_b200.ops import Act
    g = torch.Generator().manual_seed(M + N + K)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    bias = torch.randn(N, generator=g).cuda()
    act, _ = _f16_planes(a) if fmt == "f16" else _planes(a, fmt)
    wact, _ = _f16_planes(w) if fmt == "f16" else _planes(w, fmt)
    w_hi = wact.h16 if fmt == "f16" else wact.bf16 if fmt == "bf16" else (wact.hi if fmt == "split" else wact.f32)
    w_lo = wact.l16 if fmt == "f16" else wact.lo
    lib = _lib.load()
    results = []
    for flags in (0, 4, 32):
        out = Act(M, N, f32=torch.zeros(M, ops.pad4(N), device="cuda")[:, :N],
                  hi=torch.zeros(M, ops.pad4(N), device="cuda")[:, :N], lo=torch.zeros(M, ops.pad4(N), device="cuda")[:, :N],
                  bf16=torch.zeros(M, ops.pad4(N), device="cuda", dtype=torch.bfloat16)[:, :N])
        out.h16, out.l16 = torch.zeros(2, M, ops.pad4(N), dtype=torch.float16, device="cuda")[:, :, :N]
        lib.usf_debug_set_store_path(flags)
        try:
            ops.linear(eng, act, w_hi, w_lo, N, K, bias=bias, relu=True, out=out)
            torch.cuda.synchronize()
        finally:
            lib.usf_debug_set_store_path(0)
        results.append(out)
    p = results[0]
    for q in results[1:]:
        for name in ("f32", "hi", "lo", "bf16", "h16", "l16"):
            assert torch.equal(getattr(p, name), getattr(q, name)), name
    # padding columns beyond N stay untouched
    if ops.pad4(N) != N:
        assert float(p.f32._base[:, N:].abs().max()) == 0.0 and float(p.h16._base[..., N:].abs().max()) == 0.0


@pytest.mark.parametrize("M,N,K", [(300, 784, 392), (70000, 1024, 128), (515, 400, 1024), (130, 608, 72), (64, 48, 40),
                                   (1000, 392, 1024), (257, 112, 64)])
def test_forced_residual_and_store_paths_equal_the_tma_store(M, N, K):
    """fp16-split planes only (the hot configuration): boxes stored by TMA == stored by the epilogue warps themselves,
    including the in-place coupling form (residual read from the planes that are written)."""
    from usflows_b200 import _lib, ops
    from usflows_b200.ops import Act
    g = torch.Generator().manual_seed(M + N + K)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    bias = torch.randn(N, generator=g).cuda()
    x0 = torch.randn(M, N, generator=g)
    act, _ = _f16_planes(a)
    wact, _ = _f16_planes(w)
    lib = _lib.load()
    outs = []
    for flags in (0, 256, 32, 4):                         # 256: residual read lane-per-row instead of through the in-box
        stream, _ = _f16_planes(x0)                       # fresh copy of the stream for the in-place update
        lib.usf_debug_set_store_path(flags)
        try:
            ops.linear(ops.ENGINE_TC_3XF16, act, wact.h16, wact.l16, N, K, bias=bias, resid=stream, resid_sign=-1.0,
                       out=Act(M, N, h16=stream.h16, l16=stream.l16))
            torch.cuda.synchronize()
        finally:
            lib.usf_debug_set_store_path(0)
        outs.append(stream)
    for q in outs[1:]:
        assert torch.equal(outs[0].h16, q.h16) and torch.equal(outs[0].l16, q.l16)
    ref = x0.double() - (a.double() @ w.double().T + bias.double().cpu())
    assert rel_err(outs[0].h16.double() + outs[0].l16.double() / 2048.0, ref) <= 2e-5


# ---- training-step kernels (ABI 4) -----------------------------------------------------------------------------------
def _f16_planes(t):
    from usflows_b200 import ops
    from usflows_b200.ops import Act
    M, K = t.shape
    buf = torch.zeros(2, M, ops.pad4(K), dtype=torch.float16, device="cuda")
    a = Act(M, K, h16=buf[0, :, :K], l16=buf[1, :, :K])
    src = torch.zeros(M, ops.pad4(K), device="cuda")[:, :K]
    src.copy_(t)
    ops.split_f16(src, a.h16, a.l16)
    return a, (a.h16.double() + a.l16.double() / 2048.0).cpu()


@pytest.mark.parametrize("n_out,k_out,rows,split", [(784, 784, 8192, 8), (1024, 392, 4096, 16), (392, 1024, 1000, 5),
                                                    (64, 48, 300, 3), (256, 256, 77, 4), (784, 784, 8192, 1)])
def test_split_k_weight_gradient_contraction(n_out, k_out, rows, split):
    """dW[n, k] = sum_r dY[r, n] X[r, k] as usf_linear on the TRANSPOSED planes with the batch rows as K, cut into split_k
    pieces that meet in fp32 memory (red.global.add.v4.f32)."""
    from usflows_b200 import ops
    g = torch.Generator().manual_seed(rows + n_out)
    dy = torch.randn(rows, n_out, generator=g)
    x = torch.randn(rows, k_out, generator=g)
    dyT, dy_used = _f16_planes(dy.t().contiguous())
    xT, x_used = _f16_planes(x.t().contiguous())
    out = torch.full((n_out, ops.pad4(k_out, 4)), 7.0, device="cuda")[:, :k_out]        # stale content must not survive
    ops.linear_splitk(ops.ENGINE_TC_3XF16, dyT, xT, k_out, rows, out, split)
    ref = dy_used @ x_used.t()
    assert rel_err(out, ref) <= 3e-6
    ops.linear_splitk(ops.ENGINE_TC_3XF16, dyT, xT, k_out, rows, out, split)           # same result on a second call
    assert rel_err(out, ref) <= 3e-6


@pytest.mark.parametrize("rows,n", [(8192, 784), (300, 392), (65, 64), (1000, 1024), (7, 40)])
def test_planes_glue_mask_transpose_colsum(rows, n):
    from usflows_b200 import ops
    from usflows_b200.ops import Act
    g = torch.Generator().manual_seed(rows + n)
    v = torch.randn(rows, n, generator=g)
    act = torch.relu(torch.randn(rows, n, generator=g))
    mul = torch.randn(rows, n, generator=g)
    src, v_used = _f16_planes(v)
    mask, _ = _f16_planes(act)
    new = lambda r, c: Act(r, c, h16=torch.zeros(r, ops.pad4(c), dtype=torch.float16, device="cuda")[:, :c],   # noqa: E731
                           l16=torch.zeros(r, ops.pad4(c), dtype=torch.float16, device="cuda")[:, :c])
    out, t = new(rows, n), new(n, rows)
    cs, cs2 = torch.ones(n, device="cuda"), torch.zeros(n, device="cuda")
    mulp = torch.zeros(rows, ops.pad4(n, 4), device="cuda")[:, :n]
    mulp.copy_(mul)
    ops.planes_glue(src, rows=rows, n=n, mask_h=mask.h16, sign=-1.0, out=out, t=t, colsum=cs, mul=mulp, colsum2=cs2)
    want = -(v_used * (act > 0))
    got = out.h16.double().cpu() + out.l16.double().cpu() / 2048.0
    assert torch.equal(got, want)                                            # mask / sign are exact on the planes
    got_t = t.h16.double().cpu() + t.l16.double().cpu() / 2048.0
    assert torch.equal(got_t, want.t())
    assert rel_err(cs, 1.0 + want.sum(0)) <= 1e-5                            # accumulates onto the existing content
    assert rel_err(cs2, (want * mul.double()).sum(0)) <= 1e-5
    # fp32 input, in place on planes, transposed only
    t2 = new(n, rows)
    vp = torch.zeros(rows, ops.pad4(n, 4), device="cuda")[:, :n]
    vp.copy_(v)
    ops.planes_glue(vp, rows=rows, n=n, t=t2)
    assert torch.equal(t2.h16.double().cpu() + t2.l16.double().cpu() / 2048.0, v_used.t())


@pytest.mark.parametrize("kind", [0, 1])
def test_base_backward_matches_autograd(kind):
    from usflows_b200 import ops
    from usflows_b200.ops import Act
    rows, d = 500, 96
    g = torch.Generator().manual_seed(kind)
    z = torch.randn(rows, d, generator=g) * 2
    loc = torch.randn(d, generator=g) * 0.3
    scale = torch.rand(d, generator=g) + 0.5
    zz, ll, ss = z.double().requires_grad_(), loc.double().requires_grad_(), scale.double().requires_grad_()
    dist = torch.distributions.Laplace(ll, ss) if kind == 0 else torch.distributions.Normal(ll, ss)
    (-dist.log_prob(zz).sum()).backward()
    new = lambda r, c: Act(r, c, h16=torch.zeros(r, ops.pad4(c), dtype=torch.float16, device="cuda")[:, :c],   # noqa: E731
                           l16=torch.zeros(r, ops.pad4(c), dtype=torch.float16, device="cuda")[:, :c])
    gp, tp = new(rows, d), new(d, rows)
    dloc, dscale = torch.zeros(d, device="cuda"), torch.zeros(d, device="cuda")
    zp = torch.zeros(rows, ops.pad4(d, 4), device="cuda")[:, :d]
    zp.copy_(z)
    ops.base_backward(zp, loc.cuda(), scale.cuda(), kind, gp, tp, dloc, dscale)
    got = gp.h16.double().cpu() + gp.l16.double().cpu() / 2048.0
    assert rel_err(got, zz.grad) <= 1e-6
    assert torch.equal(tp.h16.cpu(), gp.h16.cpu().t()) and torch.equal(tp.l16.cpu(), gp.l16.cpu().t())
    assert rel_err(dloc, ll.grad) <= 1e-5 and rel_err(dscale, ss.grad) <= 1e-5


@pytest.mark.parametrize("d", [40, 64, 200, 784])
def test_batched_triangular_inverse(d):
    from usflows_b200 import ops
    g = torch.Generator().manual_seed(d)
    n = 6
    T = torch.randn(n, d, d, generator=g).tril() / d ** 0.5
    for m in range(n):
        T[m].diagonal().copy_(torch.where(torch.rand(d, generator=g) < 0.5, -1.0, 1.0) * (0.5 + torch.rand(d, generator=g)))
    junk = torch.randn(n, d, d, generator=g).triu(1)                   # content above the diagonal is ignored
    Td = (T + junk).cuda()
    X, tmp = torch.full_like(Td, 3.0), torch.zeros_like(Td)
    unit_mask = 0b010101
    ops.tri_inverse_batched(Td, X, tmp, unit_mask)
    for m in range(n):
        t = T[m].double()
        if (unit_mask >> m) & 1:
            t = t.tril(-1) + torch.eye(d, dtype=torch.float64)
        want = torch.linalg.solve_triangular(t, torch.eye(d, dtype=torch.float64), upper=False)
        assert rel_err(X[m], want) <= 1e-4 * max(1.0, float(torch.linalg.cond(t)) * 1e-3), m
        assert float(X[m].triu(1).abs().max()) == 0.0


def test_mat_prep_and_tri_mask():
    from usflows_b200 import ops
    from usflows_b200.ops import Act
    g = torch.Generator().manual_seed(2)
    src = torch.randn(50, 72, generator=g).cuda()
    ri = torch.randperm(72, generator=g).to(torch.int32).cuda()
    ci = torch.randperm(50, generator=g).to(torch.int32).cuda()
    out = torch.zeros(72, 52, device="cuda")[:, :50]
    pl = Act(72, 50, h16=torch.zeros(72, 56, dtype=torch.float16, device="cuda")[:, :50],
             l16=torch.zeros(72, 56, dtype=torch.float16, device="cuda")[:, :50])
    plt = Act(50, 72, h16=torch.zeros(50, 72, dtype=torch.float16, device="cuda"),
              l16=torch.zeros(50, 72, dtype=torch.float16, device="cuda"))
    ops.mat_prep(src, transpose=True, row_idx=ri, col_idx=ci, scale=-2.0, out_f32=out, out=pl, out_t=plt)
    want = -2.0 * src.t()[ri.long()][:, ci.long()]
    assert torch.equal(out, want)
    assert rel_err(pl.h16.double() + pl.l16.double() / 2048.0, want) <= 1e-6
    assert torch.equal(plt.h16, pl.h16.t()) and torch.equal(plt.l16, pl.l16.t())
    # the bias path of an inverse affine layer: row dots (gathered rows), column combination, rank-1 update
    W = torch.randn(40, 56, generator=g).cuda()
    v, u = torch.randn(56, generator=g).cuda(), torch.randn(40, generator=g).cuda()
    rows_i = torch.randperm(40, generator=g).to(torch.int32).cuda()
    o = torch.zeros(40, device="cuda")
    ops.rowdot(W, v, -1.0, o, row_idx=rows_i)
    assert rel_err(o, -(W[rows_i.long()].double() @ v.double())) <= 1e-6
    acc = torch.ones(56, device="cuda")
    ops.colcomb(W, u, 0.5, acc)
    assert rel_err(acc, 1.0 + 0.5 * (u.double() @ W.double())) <= 1e-6
    A = W.clone()
    ops.rank1(A, u, v, -2.0)
    assert rel_err(A, W.double() - 2.0 * torch.outer(u.double(), v.double())) <= 1e-6
    sq = torch.randn(40, 40, generator=g).cuda()
    diag_src = (torch.randn(40, 40, generator=g) + 3 * torch.eye(40)).cuda()
    o0, o1 = torch.zeros(40, 40, device="cuda"), torch.zeros(40, 40, device="cuda")
    ops.tri_mask(sq, 0, 0.5, o0)
    ops.tri_mask(sq, 1, 0.5, o1, diag_src=diag_src, coef=2.0)
    assert torch.equal(o0, 0.5 * sq.tril(-1))
    assert rel_err(o1, 0.5 * sq.triu() + torch.diag(2.0 / diag_src.diagonal())) <= 1e-6


@pytest.mark.parametrize("eng_name,eng,fmt", [("tf32", 2, "f32"), ("bf16", 3, "bf16"), ("3xf16", 4, "f16")])
@pytest.mark.parametrize("planes", ["bf16", "bf16+f32+resid", "f32", "f32+resid"])
@pytest.mark.parametrize("M,N,K", [(300, 784, 392), (70000, 1024, 64), (515, 392, 1024), (130, 600, 72), (64, 48, 40), (257, 112, 64)])
def test_forced_store_paths_equal_the_tma_store_of_bf16_and_fp32_planes(eng_name, eng, fmt, planes, M, N, K):
    """Mode 2 of the asynchronous store path (bf16 plane and / or fp32 plane leave through TMA tensor stores: the bf16 and
    tf32 precision modes, and every fp32 result of the fp16-split engine) == the epilogue warps storing themselves (flag 32)
    == the generic register path (flag 4), including the in-place coupling form with an fp32 residual stream."""
    from usflows_b200 import _lib, ops
    from usflows_b200.ops import Act
    g = torch.Generator().manual_seed(M + N + K)
    a = torch.randn(M, K, generator=g)
    w = torch.randn(N, K, generator=g) / K ** 0.5
    bias = torch.randn(N, generator=g).cuda()
    x0 = torch.randn(M, N, generator=g)
    act, a_used = _f16_planes(a) if fmt == "f16" else _planes(a, fmt)
    wact, w_used = _f16_planes(w) if fmt == "f16" else _planes(w, fmt)
    w_hi = wact.h16 if fmt == "f16" else wact.bf16 if fmt == "bf16" else wact.f32
    w_lo = wact.l16 if fmt == "f16" else None
    lib = _lib.load()
    results = []
    for flags in (0, 32, 4):
        out = Act(M, N)
        if "f32" in planes:
            out.f32 = torch.zeros(M, ops.pad4(N), device="cuda")[:, :N]
            out.f32.copy_(x0)
        if "bf16" in planes:
            out.bf16 = torch.zeros(M, ops.pad4(N), device="cuda", dtype=torch.bfloat16)[:, :N]
        resid = Act(M, N, f32=out.f32) if "resid" in planes else None           # in place on the fp32 stream
        lib.usf_debug_set_store_path(flags)
        try:
            ops.linear(eng, act, w_hi, w_lo, N, K, bias=bias, relu="resid" not in planes, resid=resid, resid_sign=-1.0, out=out)
            torch.cuda.synchronize()
        finally:
            lib.usf_debug_set_store_path(0)
        results.append(out)
    p = results[0]
    for q in results[1:]:
        for name in ("f32", "bf16"):
            if getattr(p, name) is not None:
                assert torch.equal(getattr(p, name), getattr(q, name)), name
    ref = a_used.double() @ w_used.double().T + bias.double().cpu()
    ref = x0.double() - ref if "resid" in planes else torch.relu(ref)
    tol = {"tf32": 3e-3, "bf16": 3e-6, "3xf16": 3e-6}[eng_name]
    got = p.f32 if p.f32 is not None else p.bf16.float()
    assert rel_err(got, ref) <= (tol if p.f32 is not None else 1e-2)
    for name in ("f32", "bf16"):                      # padding columns beyond N stay untouched
        t = getattr(p, name)
        if t is not None and ops.pad4(N) != N and "f32" not in planes:
            assert float(t._base[:, N:].abs().float().max()) == 0.0


@pytest.mark.parametrize("M,N,K", [(1, 1, 1), (5, 3, 7), (64, 64, 16), (130, 70, 33), (784, 784, 784), (100, 784, 50),
                                   (1000, 1, 9), (2600, 2500, 130)])
def test_matmul_f64_tensor_core_tiles(M, N, K):
    """`usf_matmul_f64` (fp64 MMA tiles, 64 x 64 and -- once the grid fills the SMs twice -- 128 x 128) against torch's CPU
    fp64 product: ragged edges in M, N and K, leading dimensions that are not the widths, exact small-integer products."""
    from usflows_b200 import ops
    g = torch.Generator().manual_seed(M * 7 + N * 3 + K)
    a = torch.randn(M, K, generator=g, dtype=torch.float64)
    b = torch.randn(K, N, generator=g, dtype=torch.float64)
    ad = torch.zeros(M, K + 3, dtype=torch.float64, device="cuda")[:, 1:K + 1]
    bd = torch.zeros(K, N + 5, dtype=torch.float64, device="cuda")[:, 2:N + 2]
    ad.copy_(a)
    bd.copy_(b)
    out = torch.full((M, N + 1), float("nan"), dtype=torch.float64, device="cuda")[:, :N]
    ops.matmul_f64(ad, bd, out)
    want = a @ b
    assert float((out.cpu() - want).abs().max()) <= 1e-13 * max(1.0, float(want.abs().max())) * max(1, K) ** 0.5
    ai = torch.randint(-8, 9, (M, K), generator=g).double()
    bi = torch.randint(-8, 9, (K, N), generator=g).double()
    oi = torch.empty(M, N, dtype=torch.float64, device="cuda")
    ops.matmul_f64(ai.cuda(), bi.cuda(), oi)
    assert torch.equal(oi.cpu(), ai @ bi)               # integers: every product and partial sum is exact in fp64


@pytest.mark.parametrize("d", [1, 17, 64, 200, 784, 2600])
def test_matmul_f64_triangular_factors(d):
    """`usf_matmul_f64_tri`: L . U and U^-1 . L^-1 shaped products (factors stored dense) equal the dense product bit for
    bit on integer factors, and to fp64 rounding on random ones -- the skipped k ranges only ever held zeros."""
    from usflows_b200 import ops
    g = torch.Generator().manual_seed(d)
    for exact in (True, False):
        a = (torch.randint(-4, 5, (d, d), generator=g).double() if exact else torch.randn(d, d, generator=g, dtype=torch.float64))
        b = (torch.randint(-4, 5, (d, d), generator=g).double() if exact else torch.randn(d, d, generator=g, dtype=torch.float64))
        for tri, A, B in ((ops.TRI_LOWER_UPPER, a.tril(), b.triu()), (ops.TRI_UPPER_LOWER, a.triu(), b.tril())):
            out = torch.full((d, d), float("nan"), dtype=torch.float64, device="cuda")
            ops.matmul_f64(A.cuda(), B.cuda(), out, tri)
            dense = torch.empty(d, d, dtype=torch.float64, device="cuda")
            ops.matmul_f64(A.cuda(), B.cuda(), dense)
            want = A @ B
            if exact:
                assert torch.equal(out.cpu(), want) and torch.equal(dense.cpu(), want)
            else:
                assert float((out.cpu() - want).abs().max()) <= 1e-13 * max(1.0, float(want.abs().max())) * d ** 0.5
    with pytest.raises(RuntimeError):
        ops.check(ops._lib.load().usf_matmul_f64_tri(1, 4, 1, 4, 1, 4, 4, 7, None))
