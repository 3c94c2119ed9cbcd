"""The sampling half of the hot path, draw by draw, and every configuration of the tiny-event whole-flow kernel.

The samplers are deterministic functions of Philox4x32-10 words, so moments are the wrong yardstick: a shared counter, a
repeated grid-stride pass, a parameter taken from the wrong column, or a sub-stream read from the wrong tag all leave every
marginal moment intact.  tests/philox_ref.py restates each sampler in fp64 on top of a Philox restatement that is checked
against the Random123 known answers (test_dequant_u8.py); here

- the restatements themselves are checked against scipy's distributions (CPU, no GPU needed);
- usf_base_sample and usf_radial_sample are compared with them element by element (GPU);
- the device samples are tested for goodness of fit independently of the restatements (GPU);
- `Flow.sample`, `_RadiusDistribution.sample` and the row-shard driver are tied to the base draws they came from (GPU);
- every (D, H) instantiation of usf_flow_small runs, at row counts that reach its odd-row tail and grid-stride loop (GPU).
"""
import math

import numpy as np
import pytest
import torch
from scipy import special, stats

import fake_backend
from helpers import build_flow, elementwise_err, load_case, rel_err
from oracle import flow_oracle as O
from philox_ref import mixture_cdf, ref_base_eps, ref_base_sample, ref_radial_sample, unpack_norm_params
from usflows_b200 import engine, ops

EPS32 = 2.0 ** -23
P_MIN = 1e-6                   # every goodness-of-fit check: p-value above this (fixed seeds: a failure is reproducible)
OFFSETS = [0, 5 * engine.PHILOX_CALL_STRIDE, (1 << 62) - engine.PHILOX_CALL_STRIDE]


def _sms() -> int:
    return torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count


# ---------------------------------------------------------------------------------------------------------------------
# exact distribution functions of the radius (fp64, scipy)
# ---------------------------------------------------------------------------------------------------------------------
def radius_cdf(kind, K, params, r):
    P = unpack_norm_params(kind, K, params)
    r = np.asarray(r, dtype=np.float64)
    if kind == ops.NORM_LOGNORMAL:
        return stats.norm.cdf((np.log(r) - P["mu"][0]) / P["sigma"][0])
    w = np.diff(np.concatenate([[0.0], mixture_cdf(P["logits"])]))
    if kind == ops.NORM_LOGNORMAL_MIXTURE:
        t = stats.norm.cdf((np.log(r)[:, None] - P["a"][None, :]) / P["b"][None, :])
    elif kind == ops.NORM_GENGAMMA_MIXTURE:          # R = s S^(1/q): P(R <= r) = P(S <= (r / s)^q)
        t = special.gammainc(P["a"][None, :], P["b"][None, :] * (r[:, None] / P["scale"][None, :]) ** P["power"][None, :])
    else:
        t = special.gammainc(P["a"][None, :], P["b"][None, :] * r[:, None])
    return t @ w


def _pack(logits, a, b, scale=None, power=None):
    parts = [logits, a, b] + ([] if scale is None else [scale, power])
    return np.concatenate([np.asarray(p, dtype=np.float32).reshape(-1) for p in parts])


def _radius_configs():
    """Hand-packed parameters of every radius family the library builds (layout of USF_NORM_*), in the regimes of the
    sampler: Marsaglia-Tsang with a >= 1, the a < 1 boost, q == 2 and q != 2 powers, K = 1 and mixtures."""
    g = np.random.default_rng(7)
    K = 6
    return {
        "lognormal": (ops.NORM_LOGNORMAL, 1, np.array([2.0, 0.35], dtype=np.float32)),
        "torchlognormal": (ops.NORM_LOGNORMAL, 1, np.array([0.5, 1.2], dtype=np.float32)),
        "lognormalmm": (ops.NORM_LOGNORMAL_MIXTURE, K, _pack(g.random(K), 1 + g.random(K), 0.2 + 0.3 * g.random(K))),
        "gammamm": (ops.NORM_GAMMA_MIXTURE, K, _pack(g.random(K), [0.3, 0.5, 1.0, 2.5, 7.0, 400.0], 0.5 + g.random(K))),
        "gamma": (ops.NORM_GAMMA_MIXTURE, 1, _pack([0.0], [0.3], [1.5])),
        "exponential": (ops.NORM_GAMMA_MIXTURE, 1, _pack([0.0], [1.0], [2.0])),
        "chi2": (ops.NORM_GAMMA_MIXTURE, 1, _pack([0.0], [3.25], [0.5])),
        "chi": (ops.NORM_GENGAMMA_MIXTURE, 1, _pack([0.0], [3.25], [0.5], [1.75], [2.0])),
        "halfnormal": (ops.NORM_GENGAMMA_MIXTURE, 1, _pack([0.0], [0.5], [0.5], [2.0], [2.0])),
        "weibull": (ops.NORM_GENGAMMA_MIXTURE, 1, _pack([0.0], [1.0], [1.0], [1.5], [2.5])),
        "weibullmm": (ops.NORM_GENGAMMA_MIXTURE, 4, _pack(g.random(4), np.ones(4), np.ones(4), 1 + 3 * g.random(4),
                                                         1.5 + 2 * g.random(4))),
    }


RADIUS_CONFIGS = _radius_configs()


# ---------------------------------------------------------------------------------------------------------------------
# 1. the restatements against scipy (CPU)
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", [ops.BASE_LAPLACE, ops.BASE_NORMAL])
def test_base_restatement_follows_its_distribution(kind):
    e = ref_base_eps(25000, 4, kind, seed=0x1234_5678_9ABC, offset=3 * engine.PHILOX_CALL_STRIDE)
    dist = stats.laplace if kind == ops.BASE_LAPLACE else stats.norm
    for j in range(4):                                   # each word of a Philox call, both Box-Muller outputs
        assert stats.kstest(e[:, j], dist.cdf).pvalue > P_MIN, j
    assert stats.kstest(e.reshape(-1), dist.cdf).pvalue > P_MIN
    # loc / scale per column; a different offset is a different stream
    loc, scale = np.arange(4) - 1.5, np.arange(1, 5) * 0.5
    x = ref_base_sample(25000, 4, loc, scale, kind, seed=0x1234_5678_9ABC, offset=3 * engine.PHILOX_CALL_STRIDE)
    assert np.allclose(x, loc + scale * e, rtol=0, atol=1e-12)
    other = ref_base_eps(25000, 4, kind, seed=0x1234_5678_9ABC, offset=4 * engine.PHILOX_CALL_STRIDE)
    assert abs(np.corrcoef(e.reshape(-1), other.reshape(-1))[0, 1]) < 5 / math.sqrt(e.size)


@pytest.mark.parametrize("name", sorted(RADIUS_CONFIGS))
def test_radial_restatement_radius_follows_its_distribution(name):
    kind, K, params = RADIUS_CONFIGS[name]
    n = 100000
    s = ref_radial_sample(n, 1, [0.0], ops.LP_INF, kind, params, K, seed=99, offset=7 * engine.PHILOX_CALL_STRIDE)
    assert np.array_equal(s.x[:, 0], s.radius)           # d = 1, p = inf: the direction is +1
    assert stats.kstest(s.radius, lambda r: radius_cdf(kind, K, params, r)).pvalue > P_MIN
    assert s.fragile.mean() <= 1e-3


@pytest.mark.parametrize("p_kind", [ops.LP_1, ops.LP_2, ops.LP_INF])
def test_radial_restatement_direction_lies_on_the_unit_sphere(p_kind):
    kind, K, params = RADIUS_CONFIGS["gammamm"]
    d = 5
    s = ref_radial_sample(40000, d, np.zeros(d), p_kind, kind, params, K, seed=3, offset=0)
    u = s.x / s.radius[:, None]
    norm = {ops.LP_1: np.abs(u).sum(1), ops.LP_2: np.sqrt((u * u).sum(1)), ops.LP_INF: np.abs(u).max(1)}[p_kind]
    assert np.allclose(norm, 1.0, rtol=1e-12, atol=0)
    _check_direction(u, s.radius, p_kind)


# ---------------------------------------------------------------------------------------------------------------------
# 2. usf_base_sample against the restatement, element by element
# ---------------------------------------------------------------------------------------------------------------------
def _column_params(d, seed):
    g = torch.Generator().manual_seed(seed)
    loc = (torch.rand(d, generator=g) * 6 - 3).cuda()
    scale = (0.1 + 2 * torch.rand(d, generator=g)).cuda()
    return loc, scale


def _planes(rows, d, ld, with_split=False):
    f32 = torch.full((rows, ld), float("nan"), device="cuda")[:, :d]
    act = ops.Act(rows, d, f32=f32)
    if with_split:
        ld8 = (ld + 7) // 8 * 8
        act.hi = torch.full((rows, ld8), float("nan"), device="cuda")[:, :d]
        act.lo = torch.full((rows, ld8), float("nan"), device="cuda")[:, :d]
        act.bf16 = torch.full((rows, ld8), float("nan"), device="cuda", dtype=torch.bfloat16)[:, :d]
    return act


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 3, 4, 5, 7, 8, 33, 784])
@pytest.mark.parametrize("kind", [ops.BASE_LAPLACE, ops.BASE_NORMAL])
def test_base_sample_matches_the_restatement(kind, d):
    """|got - want| <= 1e-6 (|loc_j| + scale_j max(|e|, 1)), every element, f32 output on the vector path (leading
    dimension a multiple of 4) and on the scalar path (one that is not).  The tf32 split planes and the bf16 plane must
    be the roundings of the f32 result, bit for bit.  Measured on a B200 (1000 W limit): at most 0.21 of the bound."""
    loc, scale = _column_params(d, 100 + d + 7 * kind)
    cap = 8 * _sms() * 256                                # ew_grid's cap on work items per pass (8 blocks / SM)
    d4 = (d + 3) // 4
    big = cap // d4 + 7                                   # rows * ceil(d / 4) > cap: the grid strides
    assert big * d4 > cap
    worst = 0.0
    for rows in (1, 3, 1000, big):
        for off in OFFSETS:
            seed = 0xC0FFEE + rows
            e = torch.from_numpy(ref_base_eps(rows, d, kind, seed, off))
            want = loc.double().cpu() + scale.double().cpu() * e
            bound = 1e-6 * (loc.double().cpu().abs() + scale.double().cpu() * e.abs().clamp(min=1.0))
            ld_vec = (d + 3) // 4 * 4
            a_vec = _planes(rows, d, ld_vec, with_split=True)
            ops.base_sample(a_vec, loc, scale, kind, seed, off)
            a_sc = _planes(rows, d, ld_vec + 1)
            ops.base_sample(a_sc, loc, scale, kind, seed, off)
            got = a_vec.f32.cpu()
            err = (got.double() - want).abs()
            worst = max(worst, float((err / bound).max()))
            assert bool((err <= bound).all()), (rows, off, float((err / bound).max()))
            assert torch.equal(a_sc.f32.cpu(), got), (rows, off)
            hi = a_vec.hi.cpu()
            assert torch.equal(hi, fake_backend.tf32_round(got)), (rows, off)
            assert torch.equal(a_vec.lo.cpu(), fake_backend.tf32_round(got - hi)), (rows, off)
            assert torch.equal(a_vec.bf16.cpu(), got.to(torch.bfloat16)), (rows, off)
    print(f"base_sample kind={kind} d={d}: max |err| / bound = {worst:.3f}")


# ---------------------------------------------------------------------------------------------------------------------
# 3. usf_radial_sample against the restatement
# ---------------------------------------------------------------------------------------------------------------------
def _radial_tolerance(ref, loc, d):
    """fp32 error model of one sample x = loc + (R / n) e: the radius to a few ulp (growing with |ln R| through the
    exp / pow of its last step), the p-norm n of the raw draws as an fp32 sum of d terms (growing with sqrt d), the raw
    draw e to a few ulp of max(|e|, 1), and the final fma."""
    mul = ref.radius / ref.nrm
    e = (ref.x - loc[None, :]) / mul[:, None]
    rel = 32 + 4 * np.abs(np.log(ref.radius)) + 2 * math.sqrt(d)
    return EPS32 * (2 * np.abs(loc)[None, :] + np.abs(mul)[:, None] * np.maximum(np.abs(e), 1.0) * rel[:, None])


def _compare_radial(got, ref, loc, d, what):
    """Non-fragile rows element by element within `_radial_tolerance`; fragile rows at most 1e-3 of all.  Measured on a
    B200 (1000 W limit) over every case of this file: at most 0.47 of the tolerance, fragile rows at most 5.3e-4 (the
    K = 128 log-normal mixture)."""
    ok = ~ref.fragile
    frac = float(ref.fragile.mean())
    assert frac <= 1e-3, (what, frac)
    tol = _radial_tolerance(ref, loc, d)
    err = np.abs(got.astype(np.float64) - ref.x)
    ratio = err[ok] / tol[ok]
    worst = float(ratio.max()) if ratio.size else 0.0
    assert worst <= 1.0, (what, worst, np.argwhere(err > tol)[:5].tolist())
    print(f"radial_sample {what}: max |err| / bound = {worst:.3f}, fragile rows {frac:.2e}")
    return worst, frac


def _stride_rows():
    return 8 * _sms() * 8 + 37          # ew_grid(rows * 32, 256) caps at 8 blocks of 8 warps per SM: the grid strides


RADIAL_D = [1, 3, 5, 48, 130, 784]
ALL_NORMS = ["lognormal", "gammamm", "gamma", "chi", "chi2", "halfnormal", "weibull", "exponential", "torchlognormal",
             "weibullmm", "lognormalmm"]


@pytest.mark.gpu
@pytest.mark.parametrize("p", [1, 2, "inf"])
@pytest.mark.parametrize("norm", ALL_NORMS)
def test_radial_sample_matches_the_restatement(norm, p):
    from test_radial_convnet import _radial_module, _radial_spec
    d = RADIAL_D[(ALL_NORMS.index(norm) * 3 + [1, 2, "inf"].index(p)) % len(RADIAL_D)]
    spec = _radial_spec(p, norm, d, K=6)
    params = O.random_params(spec, 40 + d)
    base = _radial_module(spec, params)
    kind, K, packed = base.norm_distribution._norm_params()
    loc = base.loc.detach().reshape(-1).contiguous()
    rows = _stride_rows() if d < 784 else 2048
    seed, off = 0x5EED_0000 + d, 3 * engine.PHILOX_CALL_STRIDE
    out = torch.empty(rows, d, device="cuda")
    ops.radial_sample(out, loc, base._p_kind, kind, packed, K, seed, off)
    ref = ref_radial_sample(rows, d, loc.cpu().numpy(), base._p_kind, kind, packed.cpu().numpy(), K, seed, off)
    _compare_radial(out.cpu().numpy(), ref, loc.double().cpu().numpy(), d, f"{norm} p={p} d={d}")


def _gamma_mix_params(K, seed):
    """Packed Gamma-mixture parameters with every concentration regime of the sampler: the a < 1 boost (0.3, 0.5),
    a = 1, 2.5, and ~400.  Packed by hand: `GammaMM` stores log(exp(a) - 1), as the reference does, which overflows in
    fp32 above a ~ 88."""
    g = torch.Generator().manual_seed(seed)
    conc = torch.tensor([0.3, 0.5, 1.0, 2.5, 397.0]).repeat(K)[:K]
    rate = conc / (1.0 + torch.rand(K, generator=g))
    return torch.cat([torch.rand(K, generator=g), conc, rate]).cuda()


@pytest.mark.gpu
@pytest.mark.parametrize("p_kind,d", [(ops.LP_2, 130), (ops.LP_1, 48), (ops.LP_INF, 5)])
@pytest.mark.parametrize("K", [1, 6, 33, 128])
def test_radial_mixture_components_and_concentrations(K, p_kind, d):
    """K = 33 crosses the 32-lane loop of gamma_mix_prepare, 128 is RAD_MAX_COMP; the concentrations run both the
    Marsaglia-Tsang rounds and the boost; at d = 130 a row has 33 column groups, more than the 32 lanes."""
    import usflows_b200 as U
    mixes = [("gammamm", (ops.NORM_GAMMA_MIXTURE, K, _gamma_mix_params(K, K)))]
    if K > 1:
        g = torch.Generator().manual_seed(K)
        nd = U.LogNormalMM(torch.rand(K, generator=g) * 2, 0.1 + 0.5 * torch.rand(K, generator=g),
                           torch.rand(K, generator=g)).to("cuda")
        mixes.append(("lognormalmm", nd._norm_params()))
    loc = torch.linspace(-1, 1, d, device="cuda")
    rows = _stride_rows()
    for name, (kind, KK, packed) in mixes:
        assert KK == K
        seed, off = 777 + K, (1 << 62) - engine.PHILOX_CALL_STRIDE
        out = torch.empty(rows, d, device="cuda")
        ops.radial_sample(out, loc, p_kind, kind, packed, K, seed, off)
        ref = ref_radial_sample(rows, d, loc.cpu().numpy(), p_kind, kind, packed.cpu().numpy(), K, seed, off)
        _compare_radial(out.cpu().numpy(), ref, loc.double().cpu().numpy(), d, f"{name} K={K} p={p_kind} d={d}")


@pytest.mark.gpu
def test_radial_sample_rejects_too_many_components():
    out = torch.empty(4, 3, device="cuda")
    params = torch.ones(3 * 129, device="cuda")
    with pytest.raises(RuntimeError, match="mixture components"):
        ops.radial_sample(out, torch.zeros(3, device="cuda"), ops.LP_2, ops.NORM_GAMMA_MIXTURE, params, 129, 1, 0)
    ops.radial_sample(out, torch.zeros(3, device="cuda"), ops.LP_2, ops.NORM_GAMMA_MIXTURE, params[:3 * 128], 128, 1, 0)
    assert bool(torch.isfinite(out).all())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["gammamm", "weibull", "lognormal"])
def test_radius_distribution_sample_is_the_restatement(name):
    """`_RadiusDistribution.sample`: the radial kernel on a one-dimensional event, stream (torch seed, call 0)."""
    import usflows_b200 as U
    nd = {"gammamm": lambda: U.GammaMM(torch.tensor([0.3, 0.5, 1.0, 2.5, 60.0, 7.0]), torch.tensor([0.5, 1, 1, 2, 50, 3.0]),
                                       torch.rand(6, generator=torch.Generator().manual_seed(2))).to("cuda"),
          "weibull": lambda: U.WeibullMM(torch.full((1,), 1.5), torch.full((1,), 2.5),
                                                                            torch.zeros(1)).to("cuda"),
          "lognormal": lambda: U.LogNormal(torch.full((1,), 0.7), torch.full((1,), 0.4)).to("cuda")}[name]()
    kind, K, packed = nd._norm_params()
    torch.manual_seed(4321)
    got = nd.sample([3000])
    assert got.shape == (3000, 1)
    ref = ref_radial_sample(3000, 1, [0.0], ops.LP_INF, kind, packed.cpu().numpy(), K, 4321, 0)
    _compare_radial(got.cpu().numpy(), ref, np.zeros(1), 1, f"radius {name}")


# ---------------------------------------------------------------------------------------------------------------------
# 4. goodness of fit of the device samples (independent of the restatement)
# ---------------------------------------------------------------------------------------------------------------------
def _corr_p(a, b):
    """Two-sided p-value of the sample correlation of a and b being zero (normal approximation, n large)."""
    a, b = a - a.mean(), b - b.mean()
    rho = float((a * b).sum() / math.sqrt(float((a * a).sum()) * float((b * b).sum())))
    return 2 * stats.norm.sf(abs(rho) * math.sqrt(a.size))


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [ops.BASE_LAPLACE, ops.BASE_NORMAL])
def test_base_sample_goodness_of_fit(kind):
    d, rows = 8, 1 << 17                                   # 2^20 draws
    loc, scale = _column_params(d, 5 + kind)
    dist = stats.laplace if kind == ops.BASE_LAPLACE else stats.norm
    x = torch.empty(rows, d, device="cuda")
    ops.base_sample(ops.Act(rows, d, f32=x), loc, scale, kind, 2024, 0)
    x2 = torch.empty(rows, d, device="cuda")
    ops.base_sample(ops.Act(rows, d, f32=x2), loc, scale, kind, 2024, engine.PHILOX_CALL_STRIDE)
    z = ((x - loc) / scale).double().cpu().numpy()
    z2 = ((x2 - loc) / scale).double().cpu().numpy()
    for j in range(d):                                     # each column standardised by its own loc and scale
        assert stats.kstest(z[:, j], dist.cdf).pvalue > P_MIN, j
    for f in (lambda t: t, lambda t: t * t):
        for i in range(d):
            for j in range(i + 1, d):                      # every pair of columns, within and across column groups
                assert _corr_p(f(z[:, i]), f(z[:, j])) > P_MIN, (i, j)
        assert _corr_p(f(z[:-1]).reshape(-1), f(z[1:]).reshape(-1)) > P_MIN          # rows r and r + 1
        assert _corr_p(f(z).reshape(-1), f(z2).reshape(-1)) > P_MIN                  # two consecutive calls


def _check_direction(u, radius, p_kind):
    """Goodness of fit of the direction u = (x - loc) / R on the unit Lp sphere of dimension d."""
    n, d = u.shape
    if p_kind == ops.LP_2:
        assert stats.kstest(u[:, 0] ** 2, stats.beta(0.5, (d - 1) / 2).cdf).pvalue > P_MIN
    elif p_kind == ops.LP_1:
        assert stats.kstest(np.abs(u[:, 0]), stats.beta(1, d - 1).cdf).pvalue > P_MIN
    else:
        pinned = np.abs(u).argmax(1)
        assert np.allclose(u[np.arange(n), pinned], 1.0, rtol=0, atol=1e-6)
        assert stats.chisquare(np.bincount(pinned, minlength=d)).pvalue > P_MIN
        others = u.copy()
        others[np.arange(n), pinned] = np.nan
        assert stats.kstest(others[~np.isnan(others)], stats.uniform(-1, 2).cdf).pvalue > P_MIN
    if p_kind != ops.LP_INF:
        signs = (u > 0).sum()
        assert stats.binomtest(int(signs), u.size).pvalue > P_MIN
    assert _corr_p(np.log(radius), np.abs(u[:, 0])) > P_MIN          # radius and direction are independent


@pytest.mark.gpu
@pytest.mark.parametrize("name", sorted(RADIUS_CONFIGS))
def test_radial_sample_goodness_of_fit(name):
    """||x - loc||_p of 2^20 device samples against the exact radius CDF, and the direction (x - loc) / R against the
    uniform distribution on the unit Lp sphere."""
    kind, K, params = RADIUS_CONFIGS[name]
    i = sorted(RADIUS_CONFIGS).index(name)
    p_kind = [ops.LP_1, ops.LP_2, ops.LP_INF][i % 3]
    d, rows = 5, 1 << 20
    # loc = 0: an fp32 sample x = loc + R u carries the rounding of |loc|, which would swamp the tiny radii of the
    # a < 1 Gammas (per-column loc is checked element by element above)
    loc = torch.zeros(d, device="cuda")
    out = torch.empty(rows, d, device="cuda")
    ops.radial_sample(out, loc, p_kind, kind, torch.from_numpy(params).cuda(), K, 31 + i, 0)
    v = (out.double() - loc.double()).cpu().numpy()
    r = {ops.LP_1: np.abs(v).sum(1), ops.LP_2: np.sqrt((v * v).sum(1)), ops.LP_INF: np.abs(v).max(1)}[p_kind]
    assert stats.kstest(r, lambda t: radius_cdf(kind, K, params, t)).pvalue > P_MIN
    _check_direction(v / r[:, None], r, p_kind)


# ---------------------------------------------------------------------------------------------------------------------
# 5. Flow.sample end to end
# ---------------------------------------------------------------------------------------------------------------------
SAMPLE_CASES = ["c1_d2_laplace", "d6_hh_normal", "d32_h64", "img_c4_4x4", "img_mnist_16x7x7", "d784_radial1_lognormal"]


def _perturbed_case(name):
    """A golden case with the base's loc and scale different in every element, so that a draw landing in the wrong
    element (NCHW / channels-last, a shifted column) changes the value."""
    spec, params, _ = load_case(name)
    params = dict(params)
    g = torch.Generator().manual_seed(len(name))
    shape = params["base_distribution.loc"].shape
    params["base_distribution.loc"] = 0.3 * (torch.rand(shape, generator=g) * 2 - 1)
    if "base_distribution.scale_unconstrained" in params:
        params["base_distribution.scale_unconstrained"] = O.inv_softplus(0.5 + torch.rand(shape, generator=g))
    return spec, params


def _base_draws(flow, spec, n, seed, offset):
    """fp64 base draws of one sampling call at (seed, offset) and the fragile-row mask."""
    base = flow.base_distribution
    ev = list(spec["in_dims"])
    d = math.prod(ev)
    if spec.get("base") == "radial":
        kind, K, packed = base.norm_distribution._norm_params()
        ref = ref_radial_sample(n, d, base.loc.detach().cpu().numpy(), base._p_kind, kind, packed.cpu().numpy(), K,
                                seed, offset)
        z, fragile = ref.x, ref.fragile
    else:
        loc, scale = base._prepared()
        z = ref_base_sample(n, d, loc.cpu().numpy(), scale.cpu().numpy(), base.base_kind, seed, offset)
        fragile = np.zeros(n, dtype=bool)
    return torch.from_numpy(z).reshape(n, *ev), torch.from_numpy(fragile)


def _check_forward(got, z64, fragile, spec, params, what):
    keep = ~fragile
    want = O.flow_forward(z64[keep], spec, params, torch.float64)
    e_ref = rel_err(O.flow_forward(z64[keep].float(), spec, params), want)
    err = rel_err(got.cpu()[keep], want)
    assert err <= 3 * e_ref + 3e-5, (what, err, e_ref)
    return err


@pytest.mark.gpu
@pytest.mark.parametrize("name", SAMPLE_CASES)
def test_flow_sample_is_the_forward_pass_of_the_restated_draws(name):
    spec, params = _perturbed_case(name)
    flow = build_flow(spec, params)
    n = 256 if math.prod(spec["in_dims"]) >= 784 else 512
    seed = 1000 + len(name)
    torch.manual_seed(seed)
    y = flow.sample([n])
    y2 = flow.sample([n])                                  # the next call: offset PHILOX_CALL_STRIDE
    assert y.shape == (n, *spec["in_dims"])
    for got, off in ((y, 0), (y2, engine.PHILOX_CALL_STRIDE)):
        z64, fragile = _base_draws(flow, spec, n, seed, off)
        assert float(fragile.double().mean()) <= 1e-2
        _check_forward(got, z64, fragile, spec, params, (name, off))


@pytest.mark.gpu
def test_sharded_sample_uses_the_salted_stream():
    from usflows_b200 import parallel
    spec, params = _perturbed_case("d6_hh_normal")
    flow = build_flow(spec, params)
    n, seed = 600, 77
    torch.manual_seed(seed)
    got = parallel.sample_sharded(flow, n, devices=[torch.cuda.current_device()])
    salted = (seed ^ 0x9E3779B97F4A7C15) & ((1 << 64) - 1)       # device 0 of the driver: salt 1
    z64, fragile = _base_draws(flow, spec, n, salted, 0)
    _check_forward(got, z64, fragile, spec, params, "sharded")


# ---------------------------------------------------------------------------------------------------------------------
# 6. every usf_flow_small instantiation
# ---------------------------------------------------------------------------------------------------------------------
def _small_spec(d, hidden, conj, blocks=2, base="laplace"):
    return dict(in_dims=[d], coupling_blocks=blocks, hidden_dims=hidden, affine_conjugation=conj, lu_transform=1,
                householder=0, base=base)


# (spec, expected (D, H) or None for the layer route, blob bound)
SMALL_CASES = {
    "d2_h32_nmid0": (_small_spec(2, [32], True), (2, 32), None),
    "d2_h32_nmid1": (_small_spec(2, [24, 32], False, 3, "normal"), (2, 32), None),
    "d3_h32_nmid2": (_small_spec(3, [32, 32, 32], False), (4, 32), None),
    "d4_h20": (_small_spec(4, [20, 20], True), (4, 32), None),
    "d8_h32": (_small_spec(8, [32, 32], False, 2, "normal"), (8, 32), None),
    "d5_h48": (_small_spec(5, [48], True), (8, 64), None),
    "d2_h64_big_blob": (_small_spec(2, [64, 64, 64], True, 2), (2, 64), "above48k"),
    "d4_h40": (_small_spec(4, [40, 33], False, 2, "normal"), (4, 64), None),
    "d8_h64": (_small_spec(8, [64, 64], True), (8, 64), None),
    "d8_h64_layer_route": (_small_spec(8, [64, 64, 64], True, 6), None, "above200k"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(SMALL_CASES))
def test_flow_small_every_instantiation(case, monkeypatch):
    spec, want_route, blob = SMALL_CASES[case]
    d = spec["in_dims"][0]
    params = O.random_params(spec, 60 + len(case))
    calls = []
    real = ops.flow_small

    def recording(x, prog, blob_t, n_ops, D, H, out):
        calls.append((D, H, blob_t.numel() * 4))
        return real(x, prog, blob_t, n_ops, D, H, out)
    monkeypatch.setattr(ops, "flow_small", recording)

    flow = build_flow(spec, params)
    sms = _sms()
    big = 8 * sms * 128 * 2 + 1001                         # past the grid-stride start of the R = 2 and R = 1 kernels
    g = torch.Generator().manual_seed(len(case))
    x_all = torch.rand(big, d, generator=g)
    z_all = torch.randn(big, d, generator=g)
    sub = torch.cat([torch.arange(0, 64), torch.arange(big // 2, big // 2 + 31), torch.arange(big - 65, big)])
    results = {}
    for rows in (1, 2, 3, 255, big):
        x, z = x_all[:rows].cuda(), z_all[:rows].cuda()
        calls.clear()
        results[rows] = (flow.log_prob(x), flow.backward(x), flow._forward(z))
        if want_route is None:
            assert calls == [], calls
        else:
            assert len(calls) == 3 and all(c[:2] == want_route for c in calls), calls
        idx = sub[sub < rows]
        xs, zs = x_all[idx], z_all[idx]
        lp, zz, yy = (t.cpu()[idx] for t in results[rows])
        want_lp = O.flow_log_prob(xs, spec, params, torch.float64)
        want_z = O.flow_backward(xs, spec, params, torch.float64)
        want_y = O.flow_forward(zs, spec, params, torch.float64)
        assert rel_err(lp, want_lp) <= 3 * rel_err(O.flow_log_prob(xs, spec, params), want_lp) + 1e-5, (case, rows)
        assert rel_err(zz, want_z) <= 3 * rel_err(O.flow_backward(xs, spec, params), want_z) + 3e-5, (case, rows)
        assert rel_err(yy, want_y) <= 3 * rel_err(O.flow_forward(zs, spec, params), want_y) + 3e-5, (case, rows)
    if blob == "above48k":
        assert calls[0][2] > 48 * 1024
    if want_route is not None:
        # sample through the fused route, tied to its base draws
        seed = 4242
        torch.manual_seed(seed)
        calls.clear()
        s = flow.sample([big])
        assert len(calls) == 1 and calls[0][:2] == want_route
        z64, _ = _base_draws(flow, spec, big, seed, 0)
        _check_forward(s[sub], z64[sub], torch.zeros(sub.numel(), dtype=torch.bool), spec, params, (case, "sample"))
        # 8-bit rows: the fused route dequantises exactly as ops.dequantize
        x_u8 = torch.randint(0, 256, (big, d), generator=g, dtype=torch.uint8).cuda()
        calls.clear()
        lp_u8 = flow.log_prob(x_u8, dequantize="uniform", seed=99)
        assert calls and calls[-1][:2] == want_route
        assert torch.equal(lp_u8, flow.log_prob(ops.dequantize(x_u8, "uniform", seed=99)))
    # every row against the layer-by-layer route of the same flow, and both against the fp64 oracle.  Two fp32 routes
    # that sum in different orders differ by up to 3.5e-5 element-wise over these 300 k rows (measured on a B200,
    # d = 8); the oracle's own fp32 run is off by up to 5.7e-5 on the latents of the same rows, so the bound is
    # scaled by the oracle's fp32 error, element-wise, over all rows.
    monkeypatch.setattr(engine, "FUSE_SMALL", False)
    layered = build_flow(spec, params)
    calls.clear()
    x, z = x_all.cuda(), z_all.cuda()
    others = (layered.log_prob(x), layered.backward(x), layered._forward(z))
    assert calls == []
    oracle = ((O.flow_log_prob, x_all), (O.flow_backward, x_all), (O.flow_forward, z_all))
    for got, other, (fn, inp) in zip(results[big], others, oracle):
        want = fn(inp, spec, params, torch.float64)
        bound = 3 * elementwise_err(fn(inp, spec, params), want)[0] + 1e-5
        assert elementwise_err(got, want)[0] <= bound, (case, fn.__name__)
        assert elementwise_err(got, other)[0] <= bound, (case, fn.__name__)
