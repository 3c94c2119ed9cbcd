"""TEST-ONLY stand-in for the C ABI: emulates every `usflows_b200.ops` entry point with torch CPU ops so the
host logic (layer planning, fusion, plane bookkeeping, weight-preparation order, caching, state-dict
compatibility) can be tested without a GPU.  Installed by the `fake_ops` fixture through monkeypatching;
never importable from the product package."""
import torch

from usflows_b200 import ops as real_ops
from usflows_b200.ops import Act, ENGINE_SIMT, ENGINE_TC_3XF16, ENGINE_TC_3XTF32, ENGINE_TC_BF16, ENGINE_TC_TF32

CALLS = []
real_conv2d_rows_supported = real_ops.conv2d_rows_supported
real_ops_conv2d_pix_supported = real_ops.conv2d_pix_supported


def tf32_round(x: torch.Tensor) -> torch.Tensor:
    i = x.contiguous().view(torch.int32)
    i = (i + 0x1000) & ~0x1FFF
    return i.view(torch.float32)


def f16_split(v: torch.Tensor):
    h = v.to(torch.float16)
    l = ((v - h.float()) * 2048.0).to(torch.float16)
    return h, l


def f16_join(h, l):
    return h.float() + l.float() / 2048.0


def _store(out: Act, v: torch.Tensor, flag=None):
    if out.h16 is not None:
        h, l = f16_split(v)
        out.h16.copy_(h)
        out.l16.copy_(l)
        if flag is not None and bool((~(v.abs() <= 65000.0)).any()):
            flag.fill_(1)
    if out.f32 is not None:
        out.f32.copy_(v)
    if out.hi is not None:
        h = tf32_round(v)
        out.hi.copy_(h)
        out.lo.copy_(tf32_round(v - h))
    if out.bf16 is not None:
        out.bf16.copy_(v.to(torch.bfloat16))


def linear(engine, a, w, w_lo, N, K, *, bias=None, relu=False, resid=None, resid_sign=1.0, colscale=None,
           postsub=None, out=None, trans_w=False, overflow_flag=None):
    CALLS.append(("linear", engine, a.rows, N, K))
    if engine == ENGINE_TC_3XF16:
        assert a.h16 is not None and w.dtype == torch.float16 and w_lo is not None
        A, W = f16_join(a.h16, a.l16), f16_join(w, w_lo)
    elif engine == ENGINE_TC_BF16:
        A = a.bf16.float()
        W = w.float()
    elif engine == ENGINE_TC_3XTF32:
        assert a.hi is not None and a.lo is not None and w_lo is not None
        A, W = a.hi + a.lo, w + w_lo
    elif engine == ENGINE_TC_TF32:
        A = a.f32 if a.f32 is not None else a.hi
        W = w
    else:
        A = a.f32 if a.f32 is not None else a.hi + a.lo
        W = w if w_lo is None else w + w_lo
    assert A.shape == (a.rows, K), (A.shape, a.rows, K)
    v = A @ (W if trans_w else W.T)
    assert v.shape[1] == N
    if bias is not None:
        v = v + bias
    if relu:
        v = torch.relu(v)
    if resid is not None:
        if resid.f32 is None and resid.hi is None and resid.h16 is not None:
            r = f16_join(resid.h16, resid.l16)
        else:
            r, rl = resid.resid_planes()
            r = r if rl is None else r + rl
        v = r + resid_sign * v
    if colscale is not None:
        v = v * colscale
    if postsub is not None:
        v = v - postsub
    _store(out, v, overflow_flag)


def ingest(x, out, *, div=None, mul=None, sub=None, overflow_flag=None):
    CALLS.append(("ingest",))
    v = x
    if div is not None:
        v = v / div
    if mul is not None:
        v = v * mul
    if sub is not None:
        v = v - sub
    _store(out, v, overflow_flag)


def base_logprob(z, loc, scale, kind, add_const, out):
    CALLS.append(("base_logprob",))
    p, pl = z.resid_planes()
    v = p if pl is None else p + pl
    if kind == real_ops.BASE_LAPLACE:
        lp = -torch.log(2 * scale) - (v - loc).abs() / scale
    else:
        lp = -((v - loc) ** 2) / (2 * scale ** 2) - scale.log() - 0.9189385332046727
    out.copy_(lp.sum(-1) + add_const)


def base_sample(out, loc, scale, kind, seed, offset):
    """The device's draws: the fp64 restatement of base_sample_kernel, rounded to fp32."""
    from philox_ref import ref_base_sample
    v = ref_base_sample(out.rows, out.width, loc.double().numpy(), scale.double().numpy(), kind, seed, offset)
    _store(out, torch.from_numpy(v).to(torch.float32))


def flow_small(x, prog_i32, blob, n_ops, D, H, out):
    """The op-list semantics of usf_flow_small (include/usflows_b200.h), row by row in torch."""
    CALLS.append(("flow_small", n_ops, D, H))
    rows, d = x.shape
    v = torch.zeros(rows, D)
    v[:, :d] = x
    prog = prog_i32.tolist()
    for op in range(n_ops):
        code, off = prog[2 * op], prog[2 * op + 1]
        w = blob[off:]
        if code & 0xff == 0:
            W, c = w[:D * D].reshape(D, D), w[D * D:D * D + D]
            v = v @ W.T + c
        else:
            n_mid = code >> 8
            W0, b0 = w[:H * D].reshape(H, D), w[H * D:H * D + H]
            h = torch.relu(v @ W0.T + b0)
            w = w[H * D + H:]
            for _ in range(n_mid):
                Wm, bm = w[:H * H].reshape(H, H), w[H * H:H * H + H]
                h = torch.relu(h @ Wm.T + bm)
                w = w[H * H + H:]
            Wl, bl = w[:D * H].reshape(D, H), w[D * H:D * H + D]
            v = v + (h @ Wl.T + bl)
    out.copy_(v[:, :d])


def affine_couple(st, x, direction, s_min, s_max, row_ladj=None, overflow_flag=None):
    CALLS.append(("affine_couple", direction))
    h = x.width
    s = st[:, :h].clamp(s_min, s_max)
    t = st[:, h:2 * h]
    if x.f32 is not None:
        v = x.f32
    elif x.h16 is not None:
        v = f16_join(x.h16, x.l16)
    elif x.hi is not None:
        v = x.hi + x.lo
    else:
        v = x.bf16.float()
    new = v * torch.exp(s) + t if direction > 0 else (v - t) * torch.exp(-s)
    _store(x, new, overflow_flag)
    if row_ladj is not None:
        row_ladj += s.sum(-1)


def _radial_norm_logpdf(r, norm_kind, params, K):
    logr = r.log()
    if norm_kind == real_ops.NORM_LOGNORMAL:
        mu, sg = params[0], params[1]
        return -((logr - mu) ** 2) / (2 * sg ** 2) - sg.log() - 0.9189385332046727 - logr
    logw, a, b = torch.log_softmax(params[:K], 0), params[K:2 * K], params[2 * K:3 * K]
    if norm_kind == real_ops.NORM_LOGNORMAL_MIXTURE:      # a = mu, b = sigma
        t = logw - ((logr[:, None] - a) ** 2) / (2 * b ** 2) - b.log() - 0.9189385332046727
        return torch.logsumexp(t, -1) - logr
    t = logw + a * b.log() - torch.lgamma(a)
    if norm_kind == real_ops.NORM_GENGAMMA_MIXTURE:       # R = scale S^(1 / power)
        sc, q = params[3 * K:4 * K], params[4 * K:5 * K]
        lu = logr[:, None] - sc.log()
        t = t + q.log() - sc.log() + (a * q - 1) * lu - b * torch.exp(q * lu)
    else:
        t = t + torch.xlogy(a - 1, r[:, None]) - b * r[:, None]
    return torch.logsumexp(t, -1)


def radial_logprob(z, loc, p_kind, norm_kind, norm_params, n_comp, dv_const, add_const, out):
    CALLS.append(("radial_logprob", p_kind, norm_kind))
    p, pl = z.resid_planes()
    v = (p if pl is None else p + pl) - loc
    r = v.abs().sum(-1) if p_kind == real_ops.LP_1 else v.pow(2).sum(-1).sqrt() if p_kind == real_ops.LP_2 \
        else v.abs().max(-1).values
    out.copy_(_radial_norm_logpdf(r, norm_kind, norm_params, n_comp) - (dv_const + (z.width - 1) * r.log()) + add_const)


def radial_sample(out, loc, p_kind, norm_kind, norm_params, n_comp, seed, offset):
    g = torch.Generator().manual_seed((seed + offset) % (2 ** 63))
    rows, d = out.shape
    if norm_kind == real_ops.NORM_LOGNORMAL:
        r = torch.exp(norm_params[0] + norm_params[1] * torch.randn(rows, generator=g))
    else:
        K = n_comp
        k = torch.multinomial(torch.softmax(norm_params[:K], 0), rows, replacement=True, generator=g)
        if norm_kind == real_ops.NORM_LOGNORMAL_MIXTURE:
            r = torch.exp(norm_params[K:2 * K][k] + norm_params[2 * K:3 * K][k] * torch.randn(rows, generator=g))
        else:
            r = torch.distributions.Gamma(norm_params[K:2 * K][k], norm_params[2 * K:3 * K][k]).sample()
        if norm_kind == real_ops.NORM_GENGAMMA_MIXTURE:
            r = norm_params[3 * K:4 * K][k] * r ** (1.0 / norm_params[4 * K:5 * K][k])
    if p_kind == real_ops.LP_2:
        u = torch.randn(rows, d, generator=g)
        u = u / u.norm(dim=-1, keepdim=True)
    elif p_kind == real_ops.LP_1:
        e = -torch.log(torch.rand(rows, d, generator=g))
        u = e / e.sum(-1, keepdim=True) * (torch.randint(0, 2, (rows, d), generator=g) * 2 - 1)
    else:
        u = torch.rand(rows, d, generator=g) * 2 - 1
        u[torch.arange(rows), torch.randint(0, d, (rows,), generator=g)] = 1.0
    out.copy_(loc + r[:, None] * u)


def gate_norm(o, n, *, xres=None, gated=False, gamma=None, beta=None, eps=1e-5, y_f32=None, act=None, act_relu=False,
              raw=None, overflow_flag=None, pre_relu=False):
    CALLS.append(("gate_norm", n, bool(gated), gamma is not None, bool(act_relu), raw is not None, y_f32 is not None))
    v = o[:, :n]
    if gated:
        assert o.shape[1] == 2 * n and xres is not None and xres.shape[1] == n
        v = xres + v * torch.sigmoid(o[:, n:2 * n])
    else:
        assert o.shape[1] == n
    if pre_relu:
        v = torch.relu(v)
    if gamma is not None:
        v = torch.nn.functional.layer_norm(v, (n,), gamma, beta, eps)
    v = v.clone()
    if y_f32 is not None:
        y_f32.copy_(v)
    if raw is not None:
        _store(raw, v, overflow_flag)
    if act is not None:
        _store(act, torch.relu(v) if act_relu else v, overflow_flag)


def layout_transpose(x, n, a, b, out, scale=None, scale_mode=0, scale_on_input=True):
    CALLS.append(("layout_transpose", a, b, scale_mode if scale is not None else 0))
    v = x.reshape(n, a, b)
    if scale is not None and scale_mode:
        s = scale.reshape(a, b) if scale_on_input else scale.reshape(b, a).T
        v = v * s if scale_mode == 1 else v / s
    out.reshape(n, b, a).copy_(v.transpose(1, 2))


def im2col(x, n_images, h, w, c, k, dilation, out, *, mask=None, relu=False, overflow_flag=None):
    CALLS.append(("im2col", c, k, mask is not None, bool(relu)))
    v = x.reshape(n_images, h, w, c)
    if mask is not None:
        v = v * mask.reshape(h, w, c)
    if relu:
        v = torch.relu(v)
    pad = (k // 2) * dilation
    vp = torch.nn.functional.pad(v, (0, 0, pad, pad, pad, pad))
    cols = [vp[:, kh * dilation:kh * dilation + h, kw * dilation:kw * dilation + w, :] for kh in range(k) for kw in range(k)]
    _store(out, torch.cat(cols, dim=-1).reshape(n_images * h * w, k * k * c), overflow_flag)


def conv2d_rows(x, n_images, h, w, c, k, dilation, w_hi, w_lo, N, *, bias=None, relu=False, out=None, mask=None,
                relu_in=False, overflow_flag=None):
    CALLS.append(("conv2d_rows", c, k, N, mask is not None, bool(relu_in), bool(relu)))
    cols = Act(n_images * h * w, k * k * c, f32=torch.empty(n_images * h * w, k * k * c))
    im2col(x, n_images, h, w, c, k, dilation, cols, mask=mask, relu=relu_in)
    CALLS.pop()
    v = cols.f32 @ (w_hi + w_lo).T
    if bias is not None:
        v = v + bias
    if relu:
        v = torch.relu(v)
    _store(out, v, overflow_flag)


def conv2d_rows_supported(N, K, c_in):
    return real_conv2d_rows_supported(N, K, c_in)


def _pix_decode(p16):
    return f16_join(p16[:, :32], p16[:, 32:64])


def _pix_store(out16, v, relu, flag):
    v = torch.relu(v) if relu else v
    full = torch.zeros(v.shape[0], 32)
    full[:, :v.shape[1]] = v
    h, l = f16_split(full)
    out16[:, :32].copy_(h)
    out16[:, 32:64].copy_(l)
    if flag is not None and bool((~(full.abs() <= 65000.0)).any()):
        flag.fill_(1)


def pix_encode(x, hw, out16, *, mask=None, relu=False, overflow_flag=None):
    CALLS.append(("pix_encode", x.shape[1], mask is not None, bool(relu)))
    v = x
    if mask is not None:
        v = v * mask.reshape(hw, x.shape[1]).repeat(x.shape[0] // hw, 1)
    _pix_store(out16, v, relu, overflow_flag)


def conv2d_pix_supported(h, w, k, gated=True):
    return real_ops_conv2d_pix_supported(h, w, k, gated)


def conv2d_pix(a16, n_images, h, w, k, dilation, w1, bias1, n1, *, relu1=False, gated=False, post_relu=False, w2=None,
               bias2=None, gamma=None, beta=None, eps=0.0, out_f32=None, out16=None, relu_planes=False, x=None, inv_mask=None,
               sign=1.0, overflow_flag=None):
    CALLS.append(("conv2d_pix", k, n1, bool(gated), gamma is not None, out16 is not None, x is not None))
    taps = k * k
    a = _pix_decode(a16)                                           # [rows, 32]
    cols = Act(a.shape[0], taps * 32, f32=torch.empty(a.shape[0], taps * 32))
    im2col(a, n_images, h, w, 32, k, dilation, cols)
    CALLS.pop()
    wt = w1.reshape(32, taps, 64)
    wf = f16_join(wt[:, :, :32], wt[:, :, 32:]).reshape(32, taps * 32)
    v = cols.f32 @ wf.T + bias1
    if gated:
        u = torch.relu(v)
        uh, ul = f16_split(u)
        if overflow_flag is not None and bool((~(u.abs() <= 65000.0)).any()):
            overflow_flag.fill_(1)
        vg = f16_join(uh, ul) @ f16_join(w2[:, :32], w2[:, 32:]).T + bias2
        v = out_f32[:, :32] + vg[:, :32] * torch.sigmoid(vg[:, 32:])
        if post_relu:
            v = torch.relu(v)
    elif relu1:
        v = torch.relu(v)
    v = v[:, :n1]
    if gamma is not None:
        v = torch.nn.functional.layer_norm(v, (n1,), gamma, beta, eps)
    v = v.clone()
    if x is not None:
        c = x.shape[1]
        x += sign * inv_mask.reshape(h * w, c).repeat(x.shape[0] // (h * w), 1) * v[:, :c]
    if out_f32 is not None:
        out_f32[:, :n1].copy_(v)
    if out16 is not None:
        _pix_store(out16, v, relu_planes, overflow_flag)


def masked_add(x, t, hw, g, sign):
    CALLS.append(("masked_add", sign))
    rows, c = x.shape
    x += sign * g.reshape(hw, c).repeat(rows // hw, 1) * t


def sub_rows(out, v):
    out -= v


def leaky_relu(x, slope, y, neg_count=None):
    y.copy_(torch.where(x >= 0, x, x * slope))
    if neg_count is not None:
        neg_count.copy_((x < 0).float().sum(-1))


def permute(x, perm_i32, y):
    y.copy_(x.index_select(-1, perm_i32.long()))


def lu_assemble(L_raw, U_raw, L=None, U=None, transpose_u=False):
    if L is not None:
        L.copy_(L_raw.tril(-1) + torch.eye(L_raw.shape[0]))
    if U is not None:
        U.copy_(U_raw.triu().T if transpose_u else U_raw.triu())


def lu_logabsdet(U_raw, out2):
    d = U_raw.diag()
    out2[0] = d.abs().log().double().sum().float()
    out2[1] = float((d == 0).sum())


def vec_logabs(v, out2):
    out2[0] = v.abs().log().double().sum().float()
    out2[1] = float((v == 0).sum())


def tri_inverse(T, lower, unit_diag, X):
    Tm = T.tril() if lower else T.triu()
    if unit_diag:
        Tm = Tm - torch.diag(Tm.diag()) + torch.eye(T.shape[0])
    X.copy_(torch.inverse(Tm.double()).float())


def transpose(a, out):
    out.copy_(a.T)


def scale_rows_cols(a, out, rowf=None, colf=None):
    v = a
    if rowf is not None:
        v = v * rowf[:, None]
    if colf is not None:
        v = v * colf[None, :]
    out.copy_(v)


def split_tf32(a, hi, lo):
    h = tf32_round(a)
    hi.copy_(h)
    if lo is not None:
        lo.copy_(tf32_round(a - h))


def split_f16(a, hi, lo, overflow_flag=None):
    h, l = f16_split(a)
    hi.copy_(h)
    lo.copy_(l)
    if overflow_flag is not None and bool((~(a.abs() <= 65000.0)).any()):
        overflow_flag.fill_(1)


def to_bf16(a, out):
    out.copy_(a.to(torch.bfloat16))


def householder_right(W, v, work):
    W.copy_(W - torch.outer(W @ v, v) * (2.0 / torch.dot(v, v)))


def softplus(a, out):
    out.copy_(torch.nn.functional.softplus(a))


def matmul_f32(a, b, out, bias=None):
    v = a @ b
    out.copy_(v if bias is None else v + bias)


def matmul_f64(a, b, out, tri=0):
    if tri == real_ops.TRI_LOWER_UPPER:           # the kind is a promise about the zeros of the factors
        assert not a.triu(1).any() and not b.tril(-1).any()
    elif tri == real_ops.TRI_UPPER_LOWER:
        assert not a.tril(-1).any() and not b.triu(1).any()
    out.copy_(a @ b)


# ---- training step (emulation of the "Training step" entries of include/usflows_b200.h) -------------------------------
def linear_splitk(engine, a_t, w_t, N, K, out, split_k):
    CALLS.append(("linear_splitk", a_t.rows, N, K, split_k))
    assert engine == ENGINE_TC_3XF16 and a_t.h16.shape == (a_t.rows, K) and w_t.h16.shape == (N, K)
    A, W = f16_join(a_t.h16, a_t.l16), f16_join(w_t.h16, w_t.l16)
    out.copy_(A @ W.T)


def planes_glue(src, *, rows, n, mask_h=None, sign=1.0, out=None, t=None, colsum=None, mul=None, colsum2=None,
                overflow_flag=None):
    CALLS.append(("planes_glue", rows, n))
    if isinstance(src, Act):
        h, l = src.h16.clone(), src.l16.clone()
    else:
        h, l = f16_split(src)
        if overflow_flag is not None and bool((~(src.abs() <= 65000.0)).any()):
            overflow_flag.fill_(1)
    assert h.shape == (rows, n)
    if mask_h is not None:
        keep = mask_h.float() > 0
        h, l = h * keep, l * keep
    if sign < 0:
        h, l = -h, -l
    if out is not None:
        out.h16.copy_(h)
        out.l16.copy_(l)
    if t is not None:
        t.h16.copy_(h.t())
        t.l16.copy_(l.t())
    v = f16_join(h, l)
    if colsum is not None:
        colsum.add_(v.sum(0))
    if colsum2 is not None:
        colsum2.add_((v * mul).sum(0))


def base_backward(z, loc, scale, kind, g, t, dloc, dscale):
    CALLS.append(("base_backward",))
    zz = z - loc
    if kind == real_ops.BASE_LAPLACE:
        gv = zz.sign() / scale
        ds = 1 / scale - zz.abs() / scale ** 2
    else:
        gv = zz / scale ** 2
        ds = 1 / scale - zz ** 2 / scale ** 3
    h, l = f16_split(gv)
    g.h16.copy_(h)
    g.l16.copy_(l)
    if t is not None:
        t.h16.copy_(h.t())
        t.l16.copy_(l.t())
    if dloc is not None:
        dloc.add_(-gv.sum(0))
    if dscale is not None:
        dscale.add_(ds.sum(0))


def mat_prep(src, *, transpose=False, row_idx=None, col_idx=None, scale=1.0, out_f32=None, out=None, out_t=None,
             overflow_flag=None):
    v = src.t() if transpose else src
    if row_idx is not None:
        v = v[row_idx.long()]
    if col_idx is not None:
        v = v[:, col_idx.long()]
    v = scale * v
    shape = out_f32.shape if out_f32 is not None else out.h16.shape if out is not None else out_t.h16.shape[::-1]
    v = v[:shape[0], :shape[1]]
    if out_f32 is not None:
        out_f32.copy_(v)
    h, l = f16_split(v)
    if out is not None:
        out.h16.copy_(h)
        out.l16.copy_(l)
    if out_t is not None:
        out_t.h16.copy_(h.t())
        out_t.l16.copy_(l.t())


def rowdot(W, v, alpha, out, row_idx=None):
    Wr = W if row_idx is None else W[row_idx.long()]
    out.copy_(alpha * (Wr[:out.numel()] @ v))


def colcomb(W, v, alpha, out):
    out.add_(alpha * (v @ W))


def rank1(A, u, v, alpha):
    A.add_(alpha * torch.outer(u, v))


def tri_mask(src, mode, scale, out, diag_src=None, coef=0.0):
    v = scale * (src.tril(-1) if mode == 0 else src.triu())
    if diag_src is not None and mode == 1:
        v = v + torch.diag(coef / diag_src.diagonal())
    out.copy_(v)


def tri_inverse_batched(T, X, tmp, unit_mask):
    for m in range(T.shape[0]):
        t = T[m].tril()
        if (unit_mask >> m) & 1:
            t = t.tril(-1) + torch.eye(t.shape[0])
        X[m].copy_(torch.linalg.solve_triangular(t, torch.eye(t.shape[0]), upper=False))


def require_cuda(t, name="tensor", dtype=torch.float32):
    return t


def install(monkeypatch):
    CALLS.clear()
    for name in ["conv2d_rows", "pix_encode", "conv2d_pix", "conv2d_pix_supported", "layout_transpose", "im2col", "masked_add", "radial_logprob", "radial_sample", "gate_norm", "affine_couple", "sub_rows", "flow_small", "linear", "ingest", "base_logprob", "base_sample", "leaky_relu", "permute", "lu_assemble",
                 "lu_logabsdet", "vec_logabs", "tri_inverse", "transpose", "scale_rows_cols", "split_tf32", "split_f16", "to_bf16",
                 "householder_right", "softplus", "matmul_f32", "matmul_f64", "require_cuda", "linear_splitk", "planes_glue",
                 "base_backward", "mat_prep", "tri_mask", "tri_inverse_batched", "rowdot", "colcomb", "rank1"]:
        monkeypatch.setattr(real_ops, name, globals()[name])
