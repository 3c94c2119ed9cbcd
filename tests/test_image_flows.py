"""SURVEY 8f row 3: flows over image-shaped events `in_dims = [C, H, W]` -- BlockAffineTransform's 1x1-convolution mode
(transforms.py:904-962), masks over [C, H, W] (flows.py:494-536), `networks.ConvNet2D` conditioners (networks.py:405-510),
ScaleTransform over [C, H, W] -- run channels-last as row matrices (usflows_b200/image_engine.py, csrc/image.cuh).

Flow-level parity against the golden fixtures of the real reference: test_gpu_parity.py / test_host_logic.py (IMG_CASES).
Here: the launch plan on the emulated backend, the conditioner module, and (-m gpu) the three layout kernels against
torch, the reference's live MNIST configuration against the oracle on fresh inputs, sampling, host-row path.
"""
import pytest
import torch
import torch.nn.functional as F

from helpers import IMG_CASES, build_flow, load_case, rel_err
from oracle import flow_oracle as O

MNIST_SPEC = dict(in_dims=[16, 7, 7], coupling_blocks=3, conditioner="convnet2d", c_hidden=32, num_layers=3, kernel_size=3,
                  gating=True, normalize_layers=True, affine_conjugation=True, lu_transform=1, householder=0, base="radial",
                  p=1, norm="lognormal")     # experiments/mnist/mnist.yaml:55-92 with fewer coupling blocks


# ---------------------------------------------------------------------------------------------------------------------
def test_image_launch_plan(fake_ops):
    spec, params, arr = load_case("img_mnist_16x7x7")
    flow = build_flow(spec, params, device="cpu", precision="fp32")
    fake_ops.CALLS.clear()
    lp = flow.log_prob(arr["x"])
    assert lp.shape == (arr["x"].shape[0],)
    names = [c[0] for c in fake_ops.CALLS]
    B, L = spec["coupling_blocks"], spec["num_layers"]
    assert names.count("layout_transpose") == 1                       # NCHW -> channels-last, fused with x / scale
    assert [c for c in fake_ops.CALLS if c[0] == "layout_transpose"][0][1:] == (16, 49, 2)
    # the whole ConvNet2D on pixel planes: encode + first + one launch per gated block + last (which updates x itself)
    assert names.count("pix_encode") == B and names.count("conv2d_pix") == B * (2 + L)
    assert names.count("conv2d_rows") == 0 and names.count("im2col") == 0
    assert names.count("gate_norm") == 0 and names.count("masked_add") == 0
    assert names.count("linear") == 2 * B + 1                          # the 1x1-convolution affine layers
    assert names.count("radial_logprob") == 1                          # on the channels-last memory, loc permuted
    pix = [c for c in fake_ops.CALLS if c[0] == "conv2d_pix"]
    assert pix[0][1:] == (3, 32, False, False, True, False)            # first: planes out
    assert pix[1][1:] == (3, 32, True, True, True, False)              # GatedConv + ReLU + LayerNormChannels in one launch
    assert pix[1 + L][1:] == (3, 16, False, False, False, True)        # last: the coupling update
    assert [c for c in fake_ops.CALLS if c[0] == "pix_encode"][0][1:] == (16, True, False)   # x * mask fused into the encoding
    from usflows_b200 import image_engine
    image_engine.PIX_CONV = False                                      # the implicit-GEMM route (one launch per k x k conv)
    try:
        fake_ops.CALLS.clear()
        lp1 = build_flow(spec, params, device="cpu", precision="fp32").log_prob(arr["x"])
        names1 = [c[0] for c in fake_ops.CALLS]
        calls1 = list(fake_ops.CALLS)
    finally:
        image_engine.PIX_CONV = True
    assert rel_err(lp1, lp) < 1e-5
    assert names1.count("conv2d_rows") == B * (2 + L) and names1.count("im2col") == 0
    assert names1.count("gate_norm") == B * L and names1.count("masked_add") == B
    assert names1.count("linear") == (2 * B + 1) + B * L              # 1x1-conv affine layers + the 1x1 gate convolutions
    first = [c for c in calls1 if c[0] == "conv2d_rows"][0]
    assert first[1:] == (16, 3, 32, True, False, False)                # coupling mask fused into the first gather
    from usflows_b200 import image_engine
    image_engine.IMPLICIT_CONV = False                                 # the gather + contraction route
    try:
        fake_ops.CALLS.clear()
        lp2 = build_flow(spec, params, device="cpu", precision="fp32").log_prob(arr["x"])
        names2 = [c[0] for c in fake_ops.CALLS]
    finally:
        image_engine.IMPLICIT_CONV = True
    assert names2.count("im2col") == B * (2 + L) and names2.count("conv2d_rows") == 0
    assert names2.count("linear") == (2 * B + 1) + B * (2 + 2 * L)
    assert rel_err(lp2, lp) < 1e-5
    # rows of the contractions: N * H * W
    assert {c[2] for c in fake_ops.CALLS if c[0] == "linear"} == {arr["x"].shape[0] * 49}


def test_image_program_merges_neighbouring_affine_maps_on_request(fake_ops):
    """engine.MERGE_AFFINE (off by default, see engine.py): the inverse 1x1 convolution of one block's affine conjugation
    and the next block's are one C x C map."""
    from usflows_b200 import engine
    spec, params, arr = load_case("img_mnist_16x7x7")
    lp = build_flow(spec, params, device="cpu", precision="fp32").log_prob(arr["x"])
    n_plain = [c[0] for c in fake_ops.CALLS].count("linear")
    engine.MERGE_AFFINE = True
    try:
        fake_ops.CALLS.clear()
        lp_m = build_flow(spec, params, device="cpu", precision="fp32").log_prob(arr["x"])
        n_merged = [c[0] for c in fake_ops.CALLS].count("linear")
    finally:
        engine.MERGE_AFFINE = False
    B = spec["coupling_blocks"]
    assert n_merged == B + 1 and n_merged < n_plain
    assert rel_err(lp_m, lp) < 1e-5


def test_pixel_plane_route_is_taken_only_where_the_widths_fit(fake_ops):
    """<= 32 input channels and 32 hidden channels (usf_conv2d_pix's operand row); other conditioners keep the round-1 routes;
    the tf32-split mode (the fp16-range fallback) never uses fp16 planes."""
    for name, mode, want in (("img_mnist_16x7x7", "fp32", True), ("img_c32_4x4_noln", "fp32", True), ("img_c4_4x4", "fp32", False),
                             ("img_c6_5x3_plain_channel", "fp32", False), ("img_mnist_16x7x7", "bf16", True),
                             ("img_mnist_16x7x7", "fp32_tf32", False), ("img_mnist_16x7x7", "fp32_simt", False)):
        spec, params, arr = load_case(name)
        fake_ops.CALLS.clear()
        build_flow(spec, params, device="cpu", precision=mode).log_prob(arr["x"][:4])
        names = {c[0] for c in fake_ops.CALLS}
        assert ("conv2d_pix" in names) == want, (name, mode)
        assert ("pix_encode" in names) == want


def test_image_flow_api_shapes(fake_ops):
    spec, params, arr = load_case("img_c4_4x4")
    flow = build_flow(spec, params, device="cpu")
    x = arr["x"]
    z = flow.backward(x)
    assert z.shape == x.shape
    assert rel_err(flow._forward(z), x) < 1e-4
    assert flow.log_prob(x[:6].reshape(2, 3, 4, 4, 4)).shape == (2, 3)
    s = flow.sample([5])
    assert s.shape == (5, 4, 4, 4)
    assert flow.log_prob(x[:0]).shape == (0,)
    # state-dict names are the reference's (the fixture's parameter keys loaded strictly); masks alternate per block
    m0, m1 = flow.layers[1].mask, flow.layers[4].mask
    assert m0.shape == (1, 4, 4, 4) and torch.equal(m0 + m1, torch.ones_like(m0))
    per_layer = torch.stack([torch.as_tensor(l.log_abs_det_jacobian(None, None), dtype=torch.float32).reshape(())
                             for l in flow.layers])
    assert rel_err(per_layer, arr["ladj32"]) <= 2e-6                   # BlockAffine: inner x H*W (transforms.py:964-980)


def test_image_program_rejects_a_wrong_event_width(fake_ops):
    """The event width is checked before any kernel reads the rows, also where no output is allocated: `log_prob` hands
    each chunk to a sink, `run(out=...)` writes into the caller's buffer."""
    spec, params, arr = load_case("img_mnist_16x7x7")
    flow = build_flow(spec, params, device="cpu")
    x = arr["x"][:20, :, :, :6].contiguous()                          # [20, 16, 7, 6]: one column short
    fake_ops.CALLS.clear()
    with pytest.raises(RuntimeError, match="event shape mismatch"):
        flow.log_prob(x)
    prog, _ = flow._program("backward")
    with pytest.raises(RuntimeError, match="event shape mismatch"):
        prog.run(x.reshape(20, -1), out=torch.empty(20, 16 * 7 * 7))
    assert fake_ops.CALLS == []


def test_convnet2d_module_matches_oracle(fake_ops):
    import usflows_b200 as U
    spec, params, _ = load_case("img_mnist_16x7x7")
    net = U.ConvNet2D(c_in=16, c_hidden=32, num_layers=3, padding="same", kernel_size=3)
    prefix = "trainable_layers.1.conditioner."
    net.load_state_dict({k[len(prefix):]: v for k, v in params.items() if k.startswith(prefix)}, strict=True)
    x = torch.randn(5, 16, 7, 7, generator=torch.Generator().manual_seed(2))
    assert rel_err(net(x), O.convnet2d(x, prefix, params, spec)) < 1e-5
    with pytest.raises(NotImplementedError):
        U.ConvNet2D(c_in=4, c_hidden=8, padding=0)                     # not shape preserving


@pytest.mark.parametrize("name", ["img_c4_4x4", "img_c6_5x3_plain_channel", "img_mnist_16x7x7"])
def test_image_training_pass_matches_oracle_gradients(fake_ops, name):
    """`Flow.fit`'s autograd pass (flows.py:195-199) for image-shaped flows: loss and every parameter gradient against
    autograd through the oracle (= the reference's own ops)."""
    from usflows_b200 import training
    spec, params, arr = load_case(name)
    flow = build_flow(spec, params, device="cpu")
    x = arr["x"][:12]
    loss = -training.log_prob_autograd(flow, x).mean()
    loss.backward()
    p = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in params.items()}
    want_loss = -O.flow_log_prob(x, spec, p).mean()
    want_loss.backward()
    assert abs(float(loss.detach()) - float(want_loss.detach())) <= 2e-5 * max(1.0, abs(float(want_loss.detach())))
    got = dict(flow.named_parameters())
    checked = 0
    for key in got:
        if "conditioner" in key or key.startswith("base_distribution") or key.endswith("scale"):
            g, w = got[key].grad, p[key].grad
            assert g is not None and w is not None, key
            assert float((g - w).abs().max()) <= 3e-4 * max(1.0, float(w.abs().max())), key
            checked += 1
    assert checked >= 8


# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("shape", [(3, 16, 49), (5, 49, 16), (2, 3, 1024), (1, 100, 70), (7, 1, 5)])
@pytest.mark.parametrize("mode", [0, 1, 2])
def test_layout_transpose_kernel(shape, mode):
    from usflows_b200 import ops
    n, a, b = shape
    g = torch.Generator().manual_seed(a * b)
    x = torch.randn(n, a, b, generator=g).cuda()
    s = (0.5 + torch.rand(a * b, generator=g)).cuda()
    for on_input in (True, False):
        out = torch.empty(n, b, a, device="cuda")
        ops.layout_transpose(x, n, a, b, out, scale=s if mode else None, scale_mode=mode, scale_on_input=on_input)
        want = x
        if mode:
            sv = s.reshape(a, b) if on_input else s.reshape(b, a).t()
            want = x * sv if mode == 1 else x / sv
        assert torch.equal(out, want.transpose(1, 2).contiguous())


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["f32", "h16", "tf32", "bf16"])
@pytest.mark.parametrize("geom", [(3, 7, 7, 16, 3, 1), (2, 5, 3, 6, 3, 1), (2, 8, 8, 4, 5, 1), (2, 9, 6, 8, 3, 2), (4, 4, 4, 3, 1, 1)])
def test_im2col_kernel_matches_conv(geom, fmt):
    """gather + contraction == F.conv2d(padding='same') on the same (masked, rectified) input."""
    from test_radial_convnet import _join, _planes
    from usflows_b200 import ops
    n, H, W, C, k, dil = geom
    g = torch.Generator().manual_seed(H * W + C)
    x = torch.randn(n, C, H, W, generator=g)
    mask = (torch.rand(C, H, W, generator=g) > 0.5).float()
    w = torch.randn(5, C, k, k, generator=g)
    rows = n * H * W
    x_cl = x.permute(0, 2, 3, 1).reshape(rows, C).contiguous().cuda()
    m_cl = mask.permute(1, 2, 0).reshape(-1).contiguous().cuda()
    cols = _planes(rows, k * k * C, fmt)
    ops.im2col(x_cl, n, H, W, C, k, dil, cols, mask=m_cl, relu=True)
    got = _join(cols).cpu() @ w.permute(0, 2, 3, 1).reshape(5, -1).t()
    want = F.conv2d(torch.relu(x * mask), w, padding="same", dilation=dil).permute(0, 2, 3, 1).reshape(rows, 5)
    assert rel_err(got, want) <= (3e-2 if fmt == "bf16" else 1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["f32", "h16", "tf32"])
@pytest.mark.parametrize("geom", [(300, 7, 7, 32, 32, 3, 1), (64, 7, 7, 16, 32, 3, 1), (17, 5, 3, 16, 20, 3, 1), (9, 8, 8, 16, 64, 3, 1),
                                  (11, 9, 6, 32, 12, 3, 2), (5, 4, 4, 32, 16, 3, 1), (2000, 7, 7, 32, 32, 3, 1), (3, 6, 5, 64, 8, 1, 1), (4, 6, 6, 16, 16, 5, 1)])
def test_implicit_gemm_convolution_matches_conv2d(geom, fmt):
    """usf_conv2d_rows (A tiles gathered into shared memory, tcgen05 tf32 split) == F.conv2d(padding='same') in fp64 on
    the same (masked, rectified) input, with bias and ReLU in the epilogue; ragged last tile, K tails, border pixels."""
    from test_radial_convnet import _join, _planes
    from usflows_b200 import engine, ops
    n, H, W, C, N, k, dil = geom
    assert ops.conv2d_rows_supported(N, k * k * C, C)
    g = torch.Generator().manual_seed(H * W + C + N)
    x = torch.randn(n, C, H, W, generator=g)
    mask = (torch.rand(C, H, W, generator=g) > 0.5).float()
    w = torch.randn(N, C, k, k, generator=g) / (k * C ** 0.5)
    b = torch.randn(N, generator=g)
    rows = n * H * W
    x_cl = x.permute(0, 2, 3, 1).reshape(rows, C).contiguous().cuda()
    m_cl = mask.permute(1, 2, 0).reshape(-1).contiguous().cuda()
    w_hi, w_lo = engine._operand(w.permute(0, 2, 3, 1).reshape(N, -1).cuda(), "fp32_tf32", ops.ENGINE_TC_3XTF32)
    out = _planes(rows, N, fmt)
    ops.conv2d_rows(x_cl, n, H, W, C, k, dil, w_hi, w_lo, N, bias=b.cuda(), relu=True, out=out, mask=m_cl, relu_in=True)
    want = torch.relu(F.conv2d(torch.relu(x * mask).double(), w.double(), b.double(), padding="same", dilation=dil))
    want = want.permute(0, 2, 3, 1).reshape(rows, N)
    assert rel_err(_join(out), want) <= 2e-6
    # without mask / ReLUs, against the gather + contraction route
    out2 = _planes(rows, N, "f32")
    ops.conv2d_rows(x_cl, n, H, W, C, k, dil, w_hi, w_lo, N, out=out2)
    want2 = F.conv2d(x.double(), w.double(), padding="same", dilation=dil).permute(0, 2, 3, 1).reshape(rows, N)
    assert rel_err(out2.f32, want2) <= 2e-6


@pytest.mark.gpu
def test_implicit_and_gathered_convolution_paths_agree_on_a_flow():
    from usflows_b200 import image_engine
    spec, params, arr = load_case("img_mnist_16x7x7")
    x = arr["x"].cuda()
    lp = build_flow(spec, params).log_prob(x)
    image_engine.IMPLICIT_CONV = False
    try:
        lp_gather = build_flow(spec, params).log_prob(x)
    finally:
        image_engine.IMPLICIT_CONV = True
    assert rel_err(lp, arr["lp32"]) <= 1e-5 and rel_err(lp_gather, arr["lp32"]) <= 1e-5
    assert rel_err(lp, lp_gather) <= 2e-6


@pytest.mark.gpu
def test_masked_add_kernel():
    from usflows_b200 import ops
    g = torch.Generator().manual_seed(1)
    n, HW, C = 6, 15, 6
    x = torch.randn(n * HW, C, generator=g).cuda()
    t = torch.randn(n * HW, C, generator=g).cuda()
    gmask = (torch.rand(HW, C, generator=g) > 0.5).float().cuda()
    want = x - gmask.repeat(n, 1) * t
    ops.masked_add(x, t, HW, gmask.reshape(-1), -1.0)
    assert torch.equal(x, want)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "fp32_tf32", "fp32_simt"])
def test_mnist_config_against_oracle_on_fresh_inputs(mode):
    spec = MNIST_SPEC
    params = O.random_params(spec, 31)
    x = torch.rand(600, 16, 7, 7, generator=torch.Generator().manual_seed(4))
    flow = build_flow(spec, params, precision=mode)
    lp64 = O.flow_log_prob(x, spec, params, dtype=torch.float64)
    z64 = O.flow_backward(x, spec, params, dtype=torch.float64)
    e_lp = rel_err(O.flow_log_prob(x, spec, params), lp64)
    e_z = rel_err(O.flow_backward(x, spec, params), z64)
    lp = flow.log_prob(x.cuda())
    z = flow.backward(x.cuda())
    assert rel_err(lp, lp64) <= 3 * e_lp + 1e-5
    assert rel_err(z, z64) <= 3 * e_z + 3e-5
    e_rt = rel_err(O.flow_forward(O.flow_backward(x, spec, params), spec, params), x)
    assert rel_err(flow._forward(z), x) <= 3 * e_rt + 1e-4
    # chunking over images does not change a bit; neither does the host-rows path
    from usflows_b200 import image_engine
    old = image_engine.IMAGE_CHUNK_ROWS, image_engine.IMAGE_CHUNK_ROWS_PIX
    image_engine.IMAGE_CHUNK_ROWS = image_engine.IMAGE_CHUNK_ROWS_PIX = 49 * 100
    try:
        assert torch.equal(flow.log_prob(x.cuda()), lp)
    finally:
        image_engine.IMAGE_CHUNK_ROWS, image_engine.IMAGE_CHUNK_ROWS_PIX = old
    assert torch.equal(flow.log_prob_host(x.pin_memory()).cuda(), lp)
    s = flow.sample([32])
    assert s.shape == (32, 16, 7, 7) and bool(torch.isfinite(s).all())


@pytest.mark.gpu
def test_mnist_config_full_batch_properties():
    """65 536 images (3.2 M channels-last rows): determinism, round trip, log_prob == base(z) - sum ladj."""
    spec = dict(MNIST_SPEC, coupling_blocks=2)
    params = O.random_params(spec, 5)
    flow = build_flow(spec, params)
    x = torch.rand(65536, 16, 7, 7, generator=torch.Generator().manual_seed(6)).cuda()
    lp = flow.log_prob(x)
    assert bool(torch.isfinite(lp).all()) and torch.equal(lp, flow.log_prob(x))
    z = flow.backward(x)
    assert rel_err(flow._forward(z), x) <= 2e-4
    total = float(sum(torch.as_tensor(l.log_abs_det_jacobian(None, None)).double() for l in flow.layers))
    assert rel_err(flow.base_distribution.log_prob(z) - total, lp) <= 1e-5
    want = O.flow_log_prob(x[:64].cpu(), spec, params, dtype=torch.float64)
    assert rel_err(lp[:64], want) <= 1e-5


@pytest.mark.gpu
def test_image_flow_fit_runs_and_lowers_the_loss():
    spec, params, arr = load_case("img_mnist_16x7x7")
    flow = build_flow(spec, params)
    losses = flow.fit(arr["x"].cuda(), optim=torch.optim.Adam, optim_params=dict(lr=1e-3), batch_size=24, epochs=6,
                      shuffle=False)
    assert all(torch.isfinite(torch.as_tensor(float(l))) for l in losses)
    assert float(losses[-1]) < float(losses[0])
    assert bool(torch.isfinite(flow.log_prob(arr["x"].cuda())).all())     # the kernels follow the updated weights


@pytest.mark.gpu
@pytest.mark.parametrize("name", IMG_CASES)
def test_image_cases_sampling_path(name):
    spec, params, arr = load_case(name)
    flow = build_flow(spec, params)
    y = flow._forward(arr["z0"].cuda())
    assert rel_err(y, arr["y32"]) <= 3e-5
    assert flow.sample([3, 2]).shape == (3, 2, *spec["in_dims"])
