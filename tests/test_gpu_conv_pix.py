"""usf_pix_encode / usf_conv2d_pix (csrc/conv_pix.cuh): the ConvNet2D conditioner on pixel planes -- k x k convolution taps as
4-D TMA boxes, the GatedConv block (networks.py:100-121) + ReLU + LayerNormChannels (networks.py:40-58) in one launch, the
masked coupling update (transforms.py:284-290) in the last convolution's epilogue -- against fp64 torch on the SAME encoded
inputs, through the C ABI.  Tolerance: fp32 accuracy of the 3-product fp16 split (2e-6 of the output scale per contraction).
"""
import pytest
import torch
import torch.nn.functional as F

from helpers import build_flow, load_case, rel_err

pytestmark = pytest.mark.gpu


def _decode(p16):
    return p16[:, :32].double() + p16[:, 32:64].double() / 2048.0


def _encode_input(n, C, H, W, seed, mask=True, relu=False):
    from usflows_b200 import ops
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(n, C, H, W, generator=g)
    m = (torch.rand(C, H, W, generator=g) > 0.5).float() if mask else None
    rows = n * H * W
    x_cl = x.permute(0, 2, 3, 1).reshape(rows, C).contiguous().cuda()
    m_cl = None if m is None else m.permute(1, 2, 0).reshape(-1).contiguous().cuda()
    a16 = torch.full((rows, 64), float("nan"), dtype=torch.float16, device="cuda")
    ops.pix_encode(x_cl, H * W, a16, mask=m_cl, relu=relu)
    v = x if m is None else x * m
    v = torch.relu(v) if relu else v
    return a16, v, x_cl, m


def _weight(N, C, k, seed):
    from usflows_b200 import image_engine
    g = torch.Generator().manual_seed(seed)
    w = torch.randn(N, C, k, k, generator=g) / (k * C ** 0.5)
    b = torch.randn(N, generator=g)
    w_im2col = w.permute(0, 2, 3, 1).reshape(N, -1).cuda()
    n_pad = 64 if N == 64 else 32
    return w, b, image_engine._pix_weight(w_im2col, k * k, C, n_pad, None), image_engine._pad_vec(b.cuda(), n_pad)


def _as_image(p_rows, n, H, W):
    return p_rows.reshape(n, H, W, -1).permute(0, 3, 1, 2)


def _decoded_weight(w16, N, C, k):
    """The fp16-split weight the kernel actually multiplies with, as an fp64 conv weight [N, C, k, k]."""
    t = w16.reshape(w16.shape[0], k * k, 64)
    wf = t[:, :, :32].double() + t[:, :, 32:].double() / 2048.0
    return wf[:N, :, :C].reshape(N, k, k, C).permute(0, 3, 1, 2).cpu()


@pytest.mark.parametrize("n,C,H,W", [(3, 16, 7, 7), (1, 32, 4, 4), (2, 5, 20, 13), (300, 9, 3, 2)])
@pytest.mark.parametrize("relu", [False, True])
def test_pix_encode(n, C, H, W, relu):
    a16, v, _, _ = _encode_input(n, C, H, W, seed=n + C, relu=relu)
    want = torch.zeros(n * H * W, 32, dtype=torch.float64)
    want[:, :C] = v.permute(0, 2, 3, 1).reshape(-1, C).double()
    got = _decode(a16).cpu()
    assert torch.isfinite(got).all()
    assert float((got - want).abs().max()) <= 2.0 ** -21 * float(want.abs().max())
    assert float(a16[:, C:32].abs().max()) == 0.0 if C < 32 else True


GEOMS = [(5, 7, 7, 16, 32, 3, 1), (1, 7, 7, 32, 32, 3, 1), (37, 7, 7, 32, 32, 3, 1), (2000, 7, 7, 32, 32, 3, 1),
         (70, 4, 4, 32, 16, 3, 1), (3, 20, 20, 8, 32, 3, 1), (2, 23, 11, 32, 12, 3, 2), (4, 6, 6, 16, 32, 5, 1),
         (6, 5, 3, 32, 32, 1, 1), (1, 1, 1, 4, 4, 3, 1), (2, 40, 256, 32, 32, 3, 1)]


@pytest.mark.parametrize("geom", GEOMS)
def test_plain_convolution_matches_conv2d(geom):
    """conv + bias (+ ReLU) on pixel planes == F.conv2d(padding='same') in fp64 on the decoded planes: whole-image tiles
    (several images per tile, ragged last tile), image-row tiles (H*W > 256), borders, dilation, 1x1 / 5x5 kernels."""
    from usflows_b200 import ops
    n, H, W, C, N, k, dil = geom
    assert ops.conv2d_pix_supported(H, W, k, False)
    a16, _, _, _ = _encode_input(n, C, H, W, seed=H * W + C + N)
    w, b, w16, b32 = _weight(N, C, k, seed=N + k)
    rows = n * H * W
    xin = _as_image(_decode(a16).cpu()[:, :C], n, H, W)
    wd = _decoded_weight(w16, N, C, k)
    want = F.conv2d(xin, wd, b.double(), padding="same", dilation=dil).permute(0, 2, 3, 1).reshape(rows, N)
    out = torch.full((rows, N), float("nan"), device="cuda")
    p16 = torch.full((rows, 64), float("nan"), dtype=torch.float16, device="cuda")
    ops.conv2d_pix(a16, n, H, W, k, dil, w16, b32, N, out_f32=out, out16=p16, relu_planes=True)
    scale = float(want.abs().max())
    assert float((out.cpu().double() - want).abs().max()) <= 2e-6 * scale
    assert float((_decode(p16).cpu()[:, :N] - torch.relu(want)).abs().max()) <= 3e-6 * scale
    if N < 32:
        assert float(p16[:, N:32].abs().max()) == 0.0 and float(p16[:, 32 + N:].abs().max()) == 0.0
    # ReLU + LayerNorm in the epilogue (the non-gated ConvNet2D block: Conv -> ReLU -> LayerNormChannels)
    g = torch.Generator().manual_seed(7)
    gamma, beta = torch.rand(N, generator=g) + 0.5, torch.randn(N, generator=g)
    out2 = torch.full((rows, N), float("nan"), device="cuda")
    ops.conv2d_pix(a16, n, H, W, k, dil, w16, b32, N, relu1=True, gamma=gamma.cuda(), beta=beta.cuda(), eps=1e-5, out_f32=out2)
    want2 = F.layer_norm(torch.relu(want), (N,), gamma.double(), beta.double(), 1e-5)
    assert float((out2.cpu().double() - want2).abs().max()) <= 2e-5 * max(1.0, float(want2.abs().max()))


@pytest.mark.parametrize("n,H,W,c_x", [(5, 7, 7, 16), (64, 7, 7, 16), (3, 18, 18, 32), (11, 4, 4, 8)])
@pytest.mark.parametrize("sign", [1.0, -1.0])
def test_last_convolution_applies_the_coupling_update(n, H, W, c_x, sign):
    from usflows_b200 import ops
    a16, _, x_cl, m = _encode_input(n, c_x, H, W, seed=n + H)
    w, b, w16, b32 = _weight(c_x, 32, 3, seed=5)
    a16h, _, _, _ = _encode_input(n, 32, H, W, seed=99, mask=False)          # a hidden activation with 32 channels
    rows = n * H * W
    t = F.conv2d(_as_image(_decode(a16h).cpu(), n, H, W), _decoded_weight(w16, c_x, 32, 3), b.double(), padding="same")
    t = t.permute(0, 2, 3, 1).reshape(rows, c_x)
    inv = (1 - m).permute(1, 2, 0).reshape(H * W, c_x)
    want = x_cl.cpu().double() + sign * inv.repeat(n, 1).double() * t
    x = x_cl.clone()
    ops.conv2d_pix(a16h, n, H, W, 3, 1, w16, b32, c_x, x=x, inv_mask=inv.reshape(-1).contiguous().cuda(), sign=sign)
    assert float((x.cpu().double() - want).abs().max()) <= 2e-6 * float(want.abs().max())


@pytest.mark.parametrize("n,H,W", [(5, 7, 7), (1, 7, 7), (333, 7, 7), (33, 4, 4), (2, 20, 20), (1, 3, 70), (3001, 7, 7), (40, 30, 30)])
@pytest.mark.parametrize("ln,relu_planes", [(True, True), (False, False)])
def test_gated_block_in_one_launch(n, H, W, ln, relu_planes):
    """y <- LN(relu(y + val * sigmoid(gate))), [val | gate] = Conv1x1(relu(Conv3x3(planes))) (networks.py:100-121 + the ReLU
    and LayerNormChannels of ConvNet2D, networks.py:469-481) against fp64 torch on the decoded inputs."""
    from usflows_b200 import ops
    rows = n * H * W
    a16, _, _, _ = _encode_input(n, 32, H, W, seed=n * H, mask=False, relu=True)
    w1, b1, w16_1, b32_1 = _weight(32, 32, 3, seed=11)
    w2, b2, w16_2, b32_2 = _weight(64, 32, 1, seed=12)
    g = torch.Generator().manual_seed(3)
    y0 = torch.randn(rows, 32, generator=g)
    gamma, beta = torch.rand(32, generator=g) + 0.5, torch.randn(32, generator=g)
    u = torch.relu(F.conv2d(_as_image(_decode(a16).cpu(), n, H, W), _decoded_weight(w16_1, 32, 32, 3), b1.double(), padding="same"))
    vg = F.conv2d(u, _decoded_weight(w16_2, 64, 32, 1), b2.double()).permute(0, 2, 3, 1).reshape(rows, 64)
    want = torch.relu(y0.double() + vg[:, :32] * torch.sigmoid(vg[:, 32:]))
    if ln:
        want = F.layer_norm(want, (32,), gamma.double(), beta.double(), 1e-5)
    y = y0.cuda()
    p16 = torch.full((rows, 64), float("nan"), dtype=torch.float16, device="cuda")
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    ops.conv2d_pix(a16, n, H, W, 3, 1, w16_1, b32_1, 32, gated=True, post_relu=True, w2=w16_2, bias2=b32_2,
                   gamma=gamma.cuda() if ln else None, beta=beta.cuda() if ln else None, eps=1e-5, out_f32=y, out16=p16,
                   relu_planes=relu_planes, overflow_flag=flag)
    tol = 1e-5 * max(1.0, float(want.abs().max()))
    assert float((y.cpu().double() - want).abs().max()) <= tol
    wp = torch.relu(want) if relu_planes else want
    assert float((_decode(p16).cpu() - wp).abs().max()) <= tol
    assert int(flag.item()) == 0


def test_overflow_flag_and_multi_tile_gated_block():
    from usflows_b200 import ops
    n, H, W = 9, 7, 7
    a16, _, _, _ = _encode_input(n, 32, H, W, seed=1, mask=False)
    w, b, w16, b32 = _weight(32, 32, 3, seed=2)
    rows = n * H * W
    # the gated block with several tiles per CTA (the gate contraction of tile i is issued among the chains of tile i + 1)
    # against fp64 torch on the decoded inputs, as test_gated_block_in_one_launch
    n2 = 4000
    rows2 = n2 * H * W
    a2, _, _, _ = _encode_input(n2, 32, H, W, seed=4, mask=False, relu=True)
    w2_, b2_, w16_2, b32_2 = _weight(64, 32, 1, seed=6)
    y0 = torch.randn(rows2, 32, generator=torch.Generator().manual_seed(8))
    u = torch.relu(F.conv2d(_as_image(_decode(a2).cpu(), n2, H, W), _decoded_weight(w16, 32, 32, 3), b.double(), padding="same"))
    vg = F.conv2d(u, _decoded_weight(w16_2, 64, 32, 1), b2_.double()).permute(0, 2, 3, 1).reshape(rows2, 64)
    want = torch.relu(y0.double() + vg[:, :32] * torch.sigmoid(vg[:, 32:]))
    y = y0.cuda()
    ops.conv2d_pix(a2, n2, H, W, 3, 1, w16, b32, 32, gated=True, post_relu=True, w2=w16_2, bias2=b32_2, out_f32=y)
    assert float((y.cpu().double() - want).abs().max()) <= 1e-5 * max(1.0, float(want.abs().max()))
    flag = torch.zeros(1, dtype=torch.int32, device="cuda")
    p16 = torch.empty(rows, 64, dtype=torch.float16, device="cuda")
    ops.conv2d_pix(a16, n, H, W, 3, 1, w16, (b32 + 1e5).contiguous(), 32, out16=p16, overflow_flag=flag)
    assert int(flag.item()) == 1


def test_pixel_plane_route_equals_the_implicit_gemm_route_on_flows():
    from usflows_b200 import image_engine
    for name in ("img_mnist_16x7x7", "img_c32_4x4_noln"):
        spec, params, arr = load_case(name)
        x = arr["x"].cuda()
        flow = build_flow(spec, params)
        lp, z = flow.log_prob(x), flow.backward(x)
        image_engine.PIX_CONV = False
        try:
            f2 = build_flow(spec, params)
            lp_rows, z_rows = f2.log_prob(x), f2.backward(x)
        finally:
            image_engine.PIX_CONV = True
        assert rel_err(lp, arr["lp32"]) <= 1e-5 and rel_err(lp_rows, arr["lp32"]) <= 1e-5
        assert rel_err(lp, lp_rows) <= 3e-6 and rel_err(z, z_rows) <= 3e-6
        assert rel_err(flow._forward(z), x) <= 1e-4


def test_image_flow_outside_the_fp16_range_falls_back_per_chunk():
    """Pixel planes are fp16 split planes: a chunk whose activations leave the fp16 range raises the device flag and is re-run
    by the tf32-split program (usf_conv2d_rows route), as in the flat path; the other chunks keep the fast route."""
    from usflows_b200 import image_engine
    spec, params, arr = load_case("img_mnist_16x7x7")
    x = arr["x"].cuda().clone()
    x[5] *= 1e6                                            # one image of the second chunk leaves the range
    old = image_engine.IMAGE_CHUNK_ROWS, image_engine.IMAGE_CHUNK_ROWS_PIX
    image_engine.IMAGE_CHUNK_ROWS = image_engine.IMAGE_CHUNK_ROWS_PIX = 49 * 4
    try:
        z = build_flow(spec, params, precision="fp32").backward(x)
        z_ref = build_flow(spec, params, precision="fp32_tf32").backward(x)
    finally:
        image_engine.IMAGE_CHUNK_ROWS, image_engine.IMAGE_CHUNK_ROWS_PIX = old
    assert bool(torch.isfinite(z).all())
    assert torch.equal(z[4:8], z_ref[4:8])                 # the flagged chunk: exactly the fallback program's result
    assert rel_err(z[:4], z_ref[:4]) <= 3e-6 and not torch.equal(z[:4], z_ref[:4])     # the others: the fp16-split engine


def test_small_image_batches_replay_one_cached_graph():
    """`log_prob` of an image-shaped flow on a small batch: the ~100 launches of the step are captured once per batch size
    and replayed; same bits as the launch-by-launch route, follows new inputs and new weights, and a batch outside the
    fp16 range falls through to the launch-by-launch route (which re-runs the chunk on the tf32-split program)."""
    from usflows_b200 import flows
    spec, params, arr = load_case("img_mnist_16x7x7")
    x = arr["x"].cuda()
    flow = build_flow(spec, params)
    old = flows.SMALL_BATCH_GRAPH_IMAGES
    flows.SMALL_BATCH_GRAPH_IMAGES = 0
    try:
        want = flow.log_prob(x)
        want2 = flow.log_prob(x.flip(0))
    finally:
        flows.SMALL_BATCH_GRAPH_IMAGES = old
    prog, _ = flow._program("backward")
    assert torch.equal(flow.log_prob(x), want) and sum(k[0] == "small" for k in prog.__dict__.get("_graphs", {})) == 1
    assert torch.equal(flow.log_prob(x.flip(0)), want2)                 # replay on new inputs
    assert torch.equal(flow.log_prob(x[:7]), want[:7]) and sum(k[0] == "small" for k in prog._graphs) == 2
    big = x.clone()
    big[3] *= 1e6
    lp_big = flow.log_prob(big)
    assert bool(torch.isfinite(lp_big[:3]).all()) and torch.equal(lp_big[:3], want[:3])
    with torch.no_grad():
        for p_ in flow.parameters():
            p_.mul_(1.001)
    lp_new = flow.log_prob(x)
    assert not torch.equal(lp_new, want) and rel_err(lp_new, want) < 0.5    # the graph followed the new weight version
