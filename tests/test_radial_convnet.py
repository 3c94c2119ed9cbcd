"""SURVEY 8f rows 2 and 4: the reference's own MLP-style conditioner (`networks.ConvNet`, vector branch:
networks.py:205-245, 287-307) and the Lp-radial base family (`RadialDistribution` with `LogNormal` / `GammaMM` radius
distributions, distributions.py:181-197, 327-372, 478-549, 674-707).

CPU part (fake backend): planning of the ConvNet conditioner, autograd parity of the training pass, state-dict layout.
GPU part (`-m gpu`, through the C ABI): `usf_gate_norm` and `usf_radial_logprob` against torch / the oracle on seeded
inputs, size-independent properties of `usf_radial_sample`, full-size rows (65 536 x 784) against the oracle's formula.
Flow-level parity against the golden fixtures of the real reference lives in test_gpu_parity.py (EXT_CASES).
"""
import math

import pytest
import torch

from helpers import EXT_CASES, build_flow, load_case, rel_err
from oracle import flow_oracle as O


# ---------------------------------------------------------------------------------------------------------------------
# host logic on the emulated backend
# ---------------------------------------------------------------------------------------------------------------------
def test_convnet_coupling_launch_program(fake_ops):
    """A gated block is 2 contractions + 1 glue launch; first / last Linear 1 each (+ the first glue launch)."""
    spec, params, arr = load_case("d64_convnet")
    flow = build_flow(spec, params, device="cpu", precision="fp32")
    fake_ops.CALLS.clear()
    flow.log_prob(arr["x"])
    lin = [c for c in fake_ops.CALLS if c[0] == "linear"]
    glue = [c for c in fake_ops.CALLS if c[0] == "gate_norm"]
    B, nblk = spec["coupling_blocks"], len(spec["c_hidden"])
    assert len(lin) == (2 * B + 1) + B * (2 + 2 * nblk)
    assert len(glue) == B * (1 + nblk)
    # mask compression: the outer conditioner contractions run on half the features
    assert sorted({c[4] for c in lin if c[3] == 128 and c[4] != 128}) == [32]
    # glue launches: first one passes the scratch through (no gate, no LayerNorm) and keeps the fp32 residual
    assert glue[0][1:] == (128, False, False, True, False, True)
    assert glue[1][1:] == (128, True, True, True, False, True)
    assert glue[2][1:] == (128, True, True, False, False, False)      # last block: un-rectified, no residual kept


def test_convnet_projection_block_uses_raw_planes(fake_ops):
    spec, params, arr = load_case("d64_convnet_proj_radial2")
    flow = build_flow(spec, params, device="cpu", precision="fp32")
    fake_ops.CALLS.clear()
    lp = flow.log_prob(arr["x"])
    glue = [c for c in fake_ops.CALLS if c[0] == "gate_norm"]
    assert glue[1][1:] == (128, True, True, True, True, False)         # next block projects 128 -> 64: raw planes, no y_f32
    assert any(c[0] == "radial_logprob" for c in fake_ops.CALLS)
    assert rel_err(lp, arr["lp32"]) < 2e-5


def test_convnet_module_forward_matches_oracle(fake_ops):
    import usflows_b200 as U
    spec, params, _ = load_case("d64_convnet_proj_radial2")
    net = U.ConvNet(in_dims=[64], c_hidden=spec["c_hidden"])
    prefix = "trainable_layers.1.conditioner."
    net.load_state_dict({k[len(prefix):]: v for k, v in params.items() if k.startswith(prefix)}, strict=True)
    x = torch.randn(17, 64, generator=torch.Generator().manual_seed(3))
    want = O.convnet_vector(x, prefix, params, spec)
    assert rel_err(net(x), want) < 1e-5


def test_convnet_state_dict_names_are_the_reference_names():
    import usflows_b200 as U
    net = U.ConvNet(in_dims=[10], c_hidden=[12, 8], gating=True)
    assert sorted(net.state_dict()) == sorted(
        ["nn.0.weight", "nn.0.bias", "nn.1.net1.1.weight", "nn.1.net1.1.bias", "nn.1.net1.3.weight", "nn.1.net1.3.bias",
         "nn.2.layernorm.weight", "nn.2.layernorm.bias", "nn.3.net1.1.weight", "nn.3.net1.1.bias", "nn.3.net1.3.weight",
         "nn.3.net1.3.bias", "nn.3.proj.weight", "nn.3.proj.bias", "nn.4.layernorm.weight", "nn.4.layernorm.bias",
         "nn.5.weight", "nn.5.bias"])
    plain = U.ConvNet(in_dims=[10], c_hidden=[12], gating=False, normalize_layers=False)
    assert sorted(plain.state_dict()) == sorted(["nn.0.weight", "nn.0.bias", "nn.1.1.weight", "nn.1.1.bias",
                                                 "nn.2.weight", "nn.2.bias"])
    # the convolutional branch (networks.py:308-377): GatedConvND with a projected residual where the width changes
    spatial = U.ConvNet(in_dims=[16, 7, 7], c_hidden=[32, 24], gating=True)
    assert sorted(spatial.state_dict()) == sorted(
        ["nn.0.weight", "nn.0.bias", "nn.1.net.1.weight", "nn.1.net.1.bias", "nn.1.net.3.weight", "nn.1.net.3.bias",
         "nn.3.gamma", "nn.3.beta", "nn.4.net.1.weight", "nn.4.net.1.bias", "nn.4.net.3.weight", "nn.4.net.3.bias",
         "nn.4.proj.weight", "nn.4.proj.bias", "nn.6.gamma", "nn.6.beta", "nn.7.weight", "nn.7.bias"])
    assert tuple(spatial.nn[4].proj.weight.shape) == (24, 32, 1, 1) and tuple(spatial.nn[7].weight.shape) == (16, 24, 3, 3)
    with pytest.raises(NotImplementedError):
        U.ConvNet(in_dims=[16, 7], c_hidden=[32])               # 1-D / 3-D convolutions are not built


def test_radial_constructor_contract():
    import usflows_b200 as U
    nd = U.LogNormal(torch.ones(1), torch.ones(1))
    with pytest.raises(ValueError):
        U.RadialDistribution(torch.zeros(4), nd, p=2)            # p must be a float (distributions.py:355-356)
    with pytest.raises(ValueError):
        U.RadialDistribution(torch.zeros(4), nd, p=-1.0)
    with pytest.raises(ValueError):
        U.RadialDistribution(torch.zeros(4), nd, p=3.0)
    r = U.RadialDistribution(torch.zeros(6), nd, p=1.0)
    assert tuple(r.event_shape) == (6,) and tuple(r.batch_shape) == () and r.dim == 6
    assert sorted(r.state_dict()) == ["loc", "norm_distribution.loc", "norm_distribution.scale_unconstrained"]
    g = U.GammaMM(torch.ones(5), torch.ones(5), torch.ones(5) / 5)
    assert sorted(g.state_dict()) == ["concentration_unconstrained", "mixture_logits", "rate_unconstrained"]
    assert sorted(U.Gamma(torch.ones(1), torch.ones(1)).state_dict()) == ["concentration_unconstrained", "rate_unconstrained"]
    # the reference's Chi and torch's Chi2 / HalfNormal carry no parameters: only `loc` is in the state dict
    for nd0 in (U.Chi(6, 1.5), torch.distributions.Chi2(torch.tensor(6.0)), torch.distributions.HalfNormal(torch.tensor(2.0))):
        assert sorted(U.RadialDistribution(torch.zeros(6), nd0, p=2.0).state_dict()) == ["loc"]
    with pytest.raises(NotImplementedError):
        U.RadialDistribution(torch.zeros(6), torch.distributions.Pareto(torch.tensor(1.0), torch.tensor(1.0)), p=2.0)
    for nd0 in (torch.distributions.Weibull(torch.tensor(1.0), torch.tensor(2.0)), torch.distributions.Exponential(torch.tensor(1.0)),
                torch.distributions.LogNormal(torch.tensor(0.0), torch.tensor(1.0)), torch.distributions.Gamma(torch.tensor(2.0), torch.tensor(1.0))):
        assert sorted(U.RadialDistribution(torch.zeros(6), nd0, p=1.0).state_dict()) == ["loc"]
    # the reference's MixtureModel layout (distributions.py:730-795): a ParameterList + the logits
    for cls in (U.WeibullMM, U.LogNormalMM):
        m = cls(torch.ones(3), 2 * torch.ones(3), torch.zeros(3))
        assert list(m.state_dict()) == ["mixture_logits", "unconstrained_params.0", "unconstrained_params.1"]
    assert torch.allclose(torch.nn.functional.softplus(U.WeibullMM(torch.ones(3), 2 * torch.ones(3), torch.zeros(3))
                                                       .unconstrained_params[1]), 2 * torch.ones(3))
    assert torch.equal(U.LogNormalMM(torch.ones(3), 2 * torch.ones(3), torch.zeros(3)).unconstrained_params[0], torch.ones(3))
    with pytest.raises(ValueError):
        U.Chi(-1.0)
    # r-independent part of the differential volume against the oracle's formula at r = 1
    for p in (1.0, 2.0, math.inf):
        rd = U.RadialDistribution(torch.zeros(9), nd, p=p)
        want = float(O.radial_log_delta_volume(p, torch.ones((), dtype=torch.float64), 9))
        assert abs(rd.log_delta_volume_const() - want) < 1e-12


@pytest.mark.parametrize("name", ["d64_convnet_proj_radial2", "d40_convnet_plain_gmm1", "d64_convnet_noln",
                                  "d32_radial2_chi", "img_c4_4x4_radial2_gamma", "d28_radialinf_weibullmm",
                                  "d30_radial2_lognormalmm"])
def test_training_pass_matches_oracle_gradients(fake_ops, name):
    from usflows_b200 import training
    spec, params, arr = load_case(name)
    flow = build_flow(spec, params, device="cpu")
    x = arr["x"][:24]
    loss = -training.log_prob_autograd(flow, x).mean()
    loss.backward()
    p = {k: v.clone().requires_grad_(v.is_floating_point()) for k, v in params.items()}
    # the oracle runs in float64: its float32 run can round a first-layer weight gradient off by ~1e-3 on its own, more
    # than the tolerance below, depending on the CPU kernels of the torch build
    want_loss = -O.flow_log_prob(x, spec, p, torch.float64).mean()
    want_loss.backward()
    assert abs(float(loss) - float(want_loss)) <= 2e-5 * max(1.0, abs(float(want_loss)))
    got = dict(flow.named_parameters())
    checked = 0
    for key in got:
        if "conditioner" in key or key.startswith("base_distribution"):
            g, w = got[key].grad, p[key].grad
            assert g is not None and w is not None, key
            assert float((g - w).abs().max()) <= 2e-4 * max(1.0, float(w.abs().max())), key
            checked += 1
    assert checked >= 8


# ---------------------------------------------------------------------------------------------------------------------
# kernels through the C ABI
# ---------------------------------------------------------------------------------------------------------------------
ALL_NORMS = ["lognormal", "gammamm", "gamma", "chi", "chi2", "halfnormal", "weibull", "exponential", "torchlognormal",
             "weibullmm", "lognormalmm"]


def _radial_spec(p, norm, d, K=20):
    # df / chi_scale: the Chi-family radius distributions (a `chi_scale`-scaled standard normal in `df` dimensions)
    return dict(in_dims=[d], coupling_blocks=1, hidden_dims=[8], base="radial", p=p, norm=norm, n_comp=K,
                df=max(1, d // 2) + 0.5, chi_scale=1.75, w_scale=1.5 * math.sqrt(d), w_conc=2.5, rate=2.0 / math.sqrt(d),
                ln_loc=0.4 * math.log(d), ln_scale=0.3)


def _radial_module(spec, params):
    import usflows_b200 as U
    q = "base_distribution.norm_distribution."
    sp = torch.nn.functional.softplus
    if spec["norm"] == "lognormal":
        nd = U.LogNormal(params[q + "loc"].clone(), sp(params[q + "scale_unconstrained"]))
    elif spec["norm"] == "gamma":
        nd = U.Gamma(sp(params[q + "concentration_unconstrained"]), sp(params[q + "rate_unconstrained"]))
    elif spec["norm"] == "chi":
        nd = U.Chi(spec["df"], spec["chi_scale"])
    elif spec["norm"] == "chi2":                  # torch objects go straight in, as in the reference's configurations
        nd = torch.distributions.Chi2(torch.tensor(float(spec["df"])))
    elif spec["norm"] == "halfnormal":
        nd = torch.distributions.HalfNormal(torch.tensor(float(spec["chi_scale"])))
    elif spec["norm"] == "weibull":
        nd = torch.distributions.Weibull(torch.tensor(float(spec["w_scale"])), torch.tensor(float(spec["w_conc"])))
    elif spec["norm"] == "exponential":
        nd = torch.distributions.Exponential(torch.tensor(float(spec["rate"])))
    elif spec["norm"] == "torchlognormal":
        nd = torch.distributions.LogNormal(torch.tensor(float(spec["ln_loc"])), torch.tensor(float(spec["ln_scale"])))
    elif spec["norm"] == "weibullmm":
        nd = U.WeibullMM(sp(params[q + "unconstrained_params.0"]), sp(params[q + "unconstrained_params.1"]),
                         params[q + "mixture_logits"].clone())
    elif spec["norm"] == "lognormalmm":
        nd = U.LogNormalMM(params[q + "unconstrained_params.0"].clone(), sp(params[q + "unconstrained_params.1"]),
                           params[q + "mixture_logits"].clone())
    else:
        nd = U.GammaMM(sp(params[q + "concentration_unconstrained"]), sp(params[q + "rate_unconstrained"]),
                       params[q + "mixture_logits"].clone())
    p = math.inf if spec["p"] == "inf" else float(spec["p"])
    return U.RadialDistribution(params["base_distribution.loc"].clone(), nd, p=p).to("cuda")


@pytest.mark.gpu
@pytest.mark.parametrize("d", [3, 32, 785, 3072])
@pytest.mark.parametrize("norm", ALL_NORMS)
@pytest.mark.parametrize("p", [1, 2, "inf"])
def test_radial_logprob_kernel_matches_oracle(p, norm, d):
    spec = _radial_spec(p, norm, d)
    params = O.random_params(spec, 21)
    base = _radial_module(spec, params)
    g = torch.Generator().manual_seed(d)
    z = torch.randn(257, d, generator=g) * (0.05 + 3 * torch.rand(257, 1, generator=g))
    want = O.radial_log_prob(z.double(), spec, O._cast(params, torch.float64))
    got = base.log_prob(z.cuda())
    assert got.shape == (257,)
    assert rel_err(got, want) <= 1e-5
    # the reference's own fp32 evaluation is no closer to the fp64 value
    ref32 = O.radial_log_prob(z, spec, params)
    assert rel_err(got, want) <= 3 * rel_err(ref32, want) + 2e-6


@pytest.mark.gpu
def test_radial_logprob_full_size_rows_and_batch_shapes():
    spec = _radial_spec(1, "lognormal", 784)
    params = O.random_params(spec, 4)
    base = _radial_module(spec, params)
    z = torch.randn(65536, 784, generator=torch.Generator().manual_seed(0))
    got = base.log_prob(z.cuda())
    want = O.radial_log_prob(z, spec, params)
    assert rel_err(got, want) <= 1e-5
    assert base.log_prob(z[:6].reshape(2, 3, 784).cuda()).shape == (2, 3)
    assert base.log_prob(z[:0].cuda()).shape == (0,)


@pytest.mark.gpu
@pytest.mark.parametrize("norm", ALL_NORMS)
@pytest.mark.parametrize("p", [1, 2, "inf"])
def test_radial_sample_properties(p, norm):
    """x - loc = R u with ||u||_p = 1 exactly up to rounding, so the radius of a sample IS its Lp norm: its empirical
    distribution must follow the radius distribution (mean of log R for LogNormal; mean / variance for the mixture),
    the direction must be sign-symmetric, and sampling must be reproducible under torch.manual_seed."""
    d, n = 48, 200000
    spec = _radial_spec(p, norm, d, K=6)
    params = O.random_params(spec, 33)
    base = _radial_module(spec, params)
    torch.manual_seed(1234)
    x = base.sample([n])
    assert x.shape == (n, d) and bool(torch.isfinite(x).all())
    v = (x - base.loc.detach()).double().cpu()
    pp = math.inf if p == "inf" else float(p)
    r = v.norm(p=pp, dim=-1)
    q = "base_distribution.norm_distribution."
    sp = torch.nn.functional.softplus
    if norm == "torchlognormal":
        mu, sg = spec["ln_loc"], spec["ln_scale"]
        assert abs(float(r.log().mean()) - mu) < 5 * sg / math.sqrt(n) + 1e-4
        assert abs(float(r.log().std()) - sg) < 0.01 * sg
    elif norm == "lognormal":
        mu, sg = float(params[q + "loc"]), float(sp(params[q + "scale_unconstrained"]))
        assert abs(float(r.log().mean()) - mu) < 5 * sg / math.sqrt(n) + 1e-4
        assert abs(float(r.log().std()) - sg) < 0.01 * sg
    elif norm not in ("gamma", "gammamm"):           # moments of the torch / reference distribution object itself
        nd = O.radial_norm_distribution(spec, O._cast(params, torch.float64))
        rs = nd.sample((400000,)).double()
        mean, second = float(rs.mean()), float((rs ** 2).mean())
        sd = math.sqrt(max(second - mean ** 2, 0.0))
        assert abs(float(r.mean()) - mean) < 8 * sd / math.sqrt(n)
        assert abs(float((r ** 2).mean()) - second) < 0.03 * second
    else:
        a, b = sp(params[q + "concentration_unconstrained"]).double(), sp(params[q + "rate_unconstrained"]).double()
        w = torch.softmax(params[q + "mixture_logits"].double(), 0) if norm == "gammamm" else torch.ones(1, dtype=torch.float64)
        mean = float((w * a / b).sum())
        second = float((w * (a * (a + 1) / b ** 2)).sum())
        sd = math.sqrt(second - mean ** 2)
        assert abs(float(r.mean()) - mean) < 6 * sd / math.sqrt(n)
        assert abs(float((r ** 2).mean()) - second) < 0.02 * second
    if p == "inf":                                   # one coordinate pinned to +1 (distributions.py:303-314)
        assert bool(((v / r[:, None]).max(-1).values - 1).abs().max() < 1e-5)
    else:
        assert abs(float((v > 0).double().mean()) - 0.5) < 0.002
    x_next = base.sample([n])                        # the next call draws from another Philox stream ...
    assert not torch.equal(x_next, x)
    other = _radial_module(spec, params)             # ... and so does another object in the same process (ADVICE r1)
    assert not torch.equal(other.sample([n]), x) and not torch.equal(other.sample([n]), x_next)
    torch.manual_seed(1234)                          # re-seeding reproduces the sequence of calls
    assert torch.equal(base.sample([n]), x)
    assert torch.equal(other.sample([n]), x_next)
    assert base.sample().shape == (d,)               # sample_shape=None peels the sample dim (distributions.py:480-497)
    # log_prob of its own samples is finite and consistent with the oracle
    lp = base.log_prob(x[:512])
    want = O.radial_log_prob(x[:512].cpu().double(), spec, O._cast(params, torch.float64))
    assert rel_err(lp, want) <= 1e-5


def _planes(rows, n, fmt):
    from usflows_b200.ops import Act
    a = Act(rows, n)
    if fmt == "f32":
        a.f32 = torch.empty(rows, n, device="cuda")
    elif fmt == "h16":
        a.h16 = torch.empty(rows, n, dtype=torch.float16, device="cuda")
        a.l16 = torch.empty(rows, n, dtype=torch.float16, device="cuda")
    elif fmt == "tf32":
        a.hi = torch.empty(rows, n, device="cuda")
        a.lo = torch.empty(rows, n, device="cuda")
    else:
        a.bf16 = torch.empty(rows, n, dtype=torch.bfloat16, device="cuda")
    return a


def _join(a):
    if a.f32 is not None:
        return a.f32
    if a.h16 is not None:
        return a.h16.float() + a.l16.float() / 2048.0
    if a.hi is not None:
        return a.hi + a.lo
    return a.bf16.float()


@pytest.mark.gpu
@pytest.mark.parametrize("fmt", ["f32", "h16", "tf32", "bf16"])
@pytest.mark.parametrize("n", [8, 50, 128, 1024])
@pytest.mark.parametrize("gated,norm", [(True, True), (True, False), (False, True), (False, False)])
def test_gate_norm_kernel_matches_torch(gated, norm, n, fmt):
    """torch fp32 reference of the same op (GatedMLP gate networks.py:241-245 + nn.LayerNorm), evaluated in fp64."""
    from usflows_b200 import ops
    rows = 333
    g = torch.Generator().manual_seed(n)
    o = torch.randn(rows, 2 * n if gated else n, generator=g).cuda()
    xres = torch.randn(rows, n, generator=g).cuda()
    gamma = (1 + 0.3 * torch.randn(n, generator=g)).cuda()
    beta = (0.3 * torch.randn(n, generator=g)).cuda()
    v = o.double()[:, :n]
    if gated:
        v = xres.double() + v * torch.sigmoid(o.double()[:, n:])
    if norm:
        v = torch.nn.functional.layer_norm(v, (n,), gamma.double(), beta.double(), 1e-5)
    act, raw = _planes(rows, n, fmt), _planes(rows, n, fmt)
    y = xres.clone()                                 # in place on the residual stream, as the engine runs it
    ops.gate_norm(o, n, xres=y if gated else None, gated=gated, gamma=gamma if norm else None,
                  beta=beta if norm else None, eps=1e-5, y_f32=y, act=act, act_relu=True, raw=raw)
    tol = 1e-2 if fmt == "bf16" else 2e-6
    assert rel_err(y, v) <= 2e-6
    assert rel_err(_join(raw), v) <= tol
    assert rel_err(_join(act), torch.relu(v)) <= tol


@pytest.mark.gpu
def test_gate_norm_rejects_bad_arguments():
    from usflows_b200 import ops
    o = torch.zeros(4, 16, device="cuda")
    with pytest.raises(RuntimeError):
        ops.gate_norm(o, 8, gated=True, y_f32=torch.zeros(4, 8, device="cuda"))      # gated without a residual
    with pytest.raises(RuntimeError):
        ops.gate_norm(o, 16)                                                           # no output at all


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["fp32", "fp32_tf32", "fp32_simt"])
def test_convnet_flow_against_oracle_on_fresh_seeded_inputs(mode):
    """C2-shaped width (d = 784 is the reference's flat MNIST size) with the ConvNet conditioner and the radial base the
    live MNIST configuration uses (experiments/mnist/mnist.yaml:79-92: p = 1, LogNormal radius)."""
    spec = dict(in_dims=[784], coupling_blocks=2, conditioner="convnet", c_hidden=[256, 256], gating=True,
                normalize_layers=True, affine_conjugation=True, lu_transform=1, householder=0, base="radial", p=1,
                norm="lognormal")
    params = O.random_params(spec, 77)
    x = torch.rand(2000, 784, generator=torch.Generator().manual_seed(8))
    flow = build_flow(spec, params, precision=mode)
    lp64 = O.flow_log_prob(x, spec, params, dtype=torch.float64)
    z64 = O.flow_backward(x, spec, params, dtype=torch.float64)
    e_lp = rel_err(O.flow_log_prob(x, spec, params), lp64)
    e_z = rel_err(O.flow_backward(x, spec, params), z64)
    assert rel_err(flow.log_prob(x.cuda()), lp64) <= 3 * e_lp + 1e-5
    z = flow.backward(x.cuda())
    assert rel_err(z, z64) <= 3 * e_z + 3e-5
    # round trip, against the oracle's own fp32 round trip (latents of size ~40 through a scale layer with |s| >= 0.1)
    e_rt = rel_err(O.flow_forward(O.flow_backward(x, spec, params), spec, params), x)
    assert rel_err(flow._forward(z), x) <= 3 * e_rt + 1e-4
    # chunking does not change a single bit
    import usflows_b200 as U
    a = flow.log_prob(x.cuda())
    U.set_chunk_rows(512)
    try:
        b = flow.log_prob(x.cuda())
    finally:
        U.set_chunk_rows(65536)
    assert torch.equal(a, b)
    s = flow.sample([64])
    assert s.shape == (64, 784) and bool(torch.isfinite(s).all())


@pytest.mark.gpu
def test_convnet_radial_training_step_runs_and_lowers_the_loss():
    spec, params, arr = load_case("d64_convnet_proj_radial2")
    flow = build_flow(spec, params)
    x = arr["x"].cuda()
    losses = flow.fit(x, optim=torch.optim.Adam, optim_params=dict(lr=1e-3), batch_size=40, epochs=6, shuffle=False)
    assert all(math.isfinite(float(l)) for l in losses)
    assert float(losses[-1]) < float(losses[0])


@pytest.mark.gpu
@pytest.mark.parametrize("name", EXT_CASES)
def test_ext_cases_host_rows_path(name):
    """`log_prob_host` (pinned host rows in, host log-probs out: the bench's e2e path) for the new components."""
    spec, params, arr = load_case(name)
    flow = build_flow(spec, params)
    out = flow.log_prob_host(arr["x"].pin_memory())
    assert rel_err(out, arr["lp32"]) <= 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("norm", ALL_NORMS)
def test_radius_distribution_on_its_own(norm):
    """`norm_distribution.log_prob(r)` / `.sample(shape)` outside a RadialDistribution (the reference's DistributionModule
    surface, distributions.py:147-151): the radial kernels on a one-dimensional event."""
    spec = _radial_spec(2, norm, 24, K=5)
    params = O.random_params(spec, 17)
    nd = _radial_module(spec, params).norm_distribution
    ref = O.radial_norm_distribution(spec, O._cast(params, torch.float64))
    r = torch.rand(1000, 1, dtype=torch.float64, generator=torch.Generator().manual_seed(23)) * 12 + 0.05
    want = ref.log_prob(r)
    want = want[:, 0] if want.dim() == 2 else want
    got = nd.log_prob(r.float().cuda())
    assert got.shape == (1000,) and rel_err(got, want) <= 1e-5
    torch.manual_seed(5)
    s = nd.sample([100000])
    assert s.shape == (100000, 1) and bool((s > 0).all()) and bool(torch.isfinite(s).all())
    rs = ref.sample((200000,)).double().reshape(-1)
    sd = float(rs.std())
    assert abs(float(s.double().mean()) - float(rs.mean())) < 8 * sd / math.sqrt(100000)
