"""Sampling to host memory: the row-keyed draws (usf_base_sample_at / usf_radial_sample_at, usf_draw), the 8-bit output
(usf_quantize_u8 / usf_layout_transpose_to_u8, `usflows_b200.quantize`), `Flow.sample(seed=, quantize=)`,
`Flow.sample_host` and the seeded row-shard driver.

The contract every route relies on: with a seed, global row r of the samples draws from Philox counters keyed by
(seed, offset 0, r) only, so chunking, graph replay and sharding cannot change a bit; q = min(255, max(0, floor(256 y))),
NaN -> 0, which is the exact inverse of the dequantisation in both modes.  `np_quantize` restates it in numpy."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import fake_backend
from helpers import build_flow, load_case, rel_err
from philox_ref import ref_base_sample
from test_dequant_u8 import GPU_CASES, np_dequant

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def np_quantize(y):
    """uint8 values of the fp32 array y: floor(256 y) clamped to [0, 255], NaN -> 0."""
    t = np.floor(np.asarray(y, dtype=np.float32) * np.float32(256.0))
    return np.where(np.isnan(t), 0, np.clip(t, 0, 255)).astype(np.uint8)


# ---- quantisation -----------------------------------------------------------------------------------------------------
def test_quantize_inverts_the_dequantisation():
    k = np.arange(256, dtype=np.uint8).reshape(32, 8)
    for mode in ("uniform", "midpoint"):
        for seed in (0, 7, 2 ** 62 + 5):
            assert np.array_equal(np_quantize(np_dequant(k, mode, seed)), k)
            assert np.array_equal(np_quantize(np_dequant(k, mode, seed, row0=1000)), k)


def test_quantize_edge_values():
    y = np.array([-0.0, -1e-30, -3.0, 0.0, 1.0 / 256, 0.5, 255.5 / 256, 1.0 - 2 ** -24, 1.0, 7.0, np.inf, -np.inf, np.nan],
                 dtype=np.float32)
    assert np_quantize(y).tolist() == [0, 0, 0, 0, 1, 128, 255, 255, 255, 255, 255, 0, 0]


# ---- emulated backend -------------------------------------------------------------------------------------------------
def _fake_base_sample_at(out, loc, scale, kind, draw):
    fake_backend.CALLS.append(("sample_at", draw.seed, draw.row0, out.rows))
    assert draw.params is None and draw.offset == 0
    v = ref_base_sample(draw.row0 + out.rows, out.width, loc.double().numpy(), scale.double().numpy(), kind, draw.seed, 0)
    fake_backend._store(out, torch.from_numpy(v[draw.row0:]).to(torch.float32))


def _fake_quantize_u8(y, out):
    out.copy_(torch.from_numpy(np_quantize(y.numpy())))


def _fake_layout_transpose_to_u8(x, n, a, b, out, scale=None, scale_mode=0):
    tmp = torch.empty(out.shape, dtype=torch.float32)
    fake_backend.layout_transpose(x, n, a, b, tmp, scale=scale, scale_mode=scale_mode, scale_on_input=False)
    _fake_quantize_u8(tmp, out)


@pytest.fixture
def fake_sample(fake_ops, monkeypatch):
    from usflows_b200 import flows, ops
    monkeypatch.setattr(ops, "base_sample_at", _fake_base_sample_at)
    monkeypatch.setattr(ops, "quantize_u8", _fake_quantize_u8)
    monkeypatch.setattr(ops, "quantize", lambda y: torch.from_numpy(np_quantize(y.numpy())))
    monkeypatch.setattr(ops, "layout_transpose_to_u8", _fake_layout_transpose_to_u8)
    monkeypatch.setattr(flows, "_wave_aligned_chunk_rows", lambda prog, dev: 256)
    return fake_ops


# ---- chunking ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 255, 256, 700, 1000, 5000, 12345])
def test_chunk_schedule_covers_the_rows_and_shrinks_at_the_end(n):
    from usflows_b200 import flows
    unit = 256
    bounds = flows.sample_host_bounds(n, min(unit, n))
    assert bounds[0][0] == 0 and bounds[-1][1] == n
    assert all(a[1] == b[0] for a, b in zip(bounds, bounds[1:]))
    sizes = [r1 - r0 for r0, r1 in bounds]
    assert all(s > 0 for s in sizes)
    if len(sizes) > 1:
        assert all(s % unit == 0 for s in sizes[1:]) and sizes[-1] == unit          # wave-aligned, smallest last
        assert all(a >= b for a, b in zip(sizes[1:], sizes[2:]))
    assert flows.sample_host_bounds(n, 777, uniform=True) == [(r0, min(n, r0 + 777)) for r0 in range(0, n, 777)]


@pytest.mark.parametrize("name", ["d100_h50_hh", "img_c4_4x4", "c1_d2_laplace", "img_bottleneck_c4_5x4"])
@pytest.mark.parametrize("quantize", [False, True])
def test_every_chunk_draws_its_global_rows(fake_sample, name, quantize):
    spec, params, _ = load_case(name)
    flow = build_flow(spec, params, device="cpu", precision="fp32")
    image = len(spec["in_dims"]) == 3
    n, off, step = (23, 5, 7) if image else (1000, 40, None if name == "d100_h50_hh" else 300)     # the last: plain chunks
    fake_backend.CALLS.clear()
    got = flow.sample_host(n, seed=9, quantize=quantize, row_offset=off, chunk_rows=step)
    draws = [c for c in fake_backend.CALLS if c[0] == "sample_at"]
    assert {c[1] for c in draws} == {9}
    assert sorted((c[2], c[2] + c[3]) for c in draws)[0][0] == off and len(draws) > 1
    spans = sorted((c[2], c[2] + c[3]) for c in draws)
    assert all(a[1] == b[0] for a, b in zip(spans, spans[1:])) and spans[-1][1] == off + n
    want = flow.sample([off + n], seed=9)[off:]
    assert got.shape == (n, *spec["in_dims"]) and got.dtype == (torch.uint8 if quantize else torch.float32)
    if quantize:
        assert (got.int() - torch.from_numpy(np_quantize(want.numpy())).int()).abs().max() <= 1
        assert torch.equal(flow.sample([off + n], seed=9, quantize=True)[off:], torch.from_numpy(np_quantize(want.numpy())))
    else:
        assert rel_err(got, want) <= 1e-6


def test_fp16_range_rerun_redraws_the_same_rows(fake_sample, monkeypatch):
    """Every chunk's ingest raises the range flag: the tf32-split re-run must draw the same rows of the noise."""
    from usflows_b200 import ops
    spec, params, _ = load_case("d100_h50_hh")
    f16 = build_flow(spec, params, device="cpu", precision="fp32")
    tf = build_flow(spec, params, device="cpu", precision="fp32_tf32")
    want = tf.sample_host(700, seed=5, row_offset=3)

    def tripping(x, out, *, overflow_flag=None, **kw):
        fake_backend.ingest(x, out, overflow_flag=overflow_flag, **kw)
        if overflow_flag is not None:
            overflow_flag.fill_(1)
    monkeypatch.setattr(ops, "ingest", tripping)
    fake_backend.CALLS.clear()
    got = f16.sample_host(700, seed=5, row_offset=3)
    assert ops.ENGINE_TC_3XTF32 in {c[1] for c in fake_backend.CALLS if c[0] == "linear"}
    draws = [c[2] for c in fake_backend.CALLS if c[0] == "sample_at"]
    assert len(draws) == 2 * len(set(draws)) and min(draws) == 3
    assert torch.equal(got, want)


# ---- sharding ---------------------------------------------------------------------------------------------------------
def _two_shards(flow):
    from concurrent.futures import ThreadPoolExecutor
    from usflows_b200 import parallel
    sf = parallel.ShardedFlow.__new__(parallel.ShardedFlow)
    sf.flow, sf.devices, sf.replicas, sf._synced = flow, ["a", "b"], [flow, flow], flow._weights_key()
    sf._pool = ThreadPoolExecutor(max_workers=1)
    return sf


def test_row_shard_driver_streams_each_block_at_its_global_rows(fake_sample):
    spec, params, _ = load_case("d6_hh_normal")
    flow = build_flow(spec, params, device="cpu", precision="fp32")
    seen = []

    def host(n, out_host=None, *, seed=None, quantize=False, row_offset=0, chunk_rows=None):
        seen.append((n, seed, row_offset, quantize))
        out_host.copy_(flow.sample([11], seed=seed, quantize=quantize)[row_offset:row_offset + n])
        return out_host
    sf = _two_shards(flow)
    flow.sample_host = host
    try:
        out = torch.empty(11, 6)
        sf.sample(11, out, seed=31)
        q = torch.empty(11, 6, dtype=torch.uint8)
        sf.sample(11, q, quantize=True, seed=32)
    finally:
        sf.close()
        del flow.sample_host
    assert sorted(seen) == [(5, 31, 6, False), (5, 32, 6, True), (6, 31, 0, False), (6, 32, 0, True)]
    assert torch.equal(out, flow.sample([11], seed=31)) and torch.equal(q, flow.sample([11], seed=32, quantize=True))


def test_row_shard_driver_without_keywords_keeps_the_salted_streams(fake_sample, monkeypatch):
    from types import SimpleNamespace
    from usflows_b200 import engine
    monkeypatch.setattr(torch.cuda, "current_stream", lambda device=None: SimpleNamespace(synchronize=lambda: None))
    spec, params, _ = load_case("d6_hh_normal")
    flow = build_flow(spec, params, device="cpu", precision="fp32")
    salts = []

    def sample(shape, context=None, **kw):
        assert not kw
        salts.append((shape[0], engine.philox_salt.value))
        return torch.zeros(shape[0], 6)
    sf = _two_shards(flow)
    flow.sample = sample
    flow.sample_host = None                                       # the streaming path must not be taken
    try:
        sf.sample(11, torch.empty(11, 6))
    finally:
        sf.close()
        del flow.sample, flow.sample_host
    assert sorted(salts) == [(5, 2), (6, 1)]


# ---- errors and ABI ---------------------------------------------------------------------------------------------------
def test_argument_errors(fake_sample):
    spec, params, _ = load_case("d6_hh_normal")
    flow = build_flow(spec, params, device="cpu", precision="fp32")
    with pytest.raises(ValueError, match="n >= 0"):
        flow.sample_host(-1)
    with pytest.raises(ValueError, match="n >= 0"):
        flow.sample_host(4, row_offset=-2)
    with pytest.raises(ValueError, match="out_host"):
        flow.sample_host(4, torch.empty(4, 6, dtype=torch.float64))
    with pytest.raises(ValueError, match="out_host"):
        flow.sample_host(4, torch.empty(4, 6), quantize=True)
    with pytest.raises(ValueError, match="out_host"):
        flow.sample_host(4, torch.empty(5, 6))
    with pytest.raises(ValueError, match="out_host"):
        flow.sample_host(4, torch.empty(6, 4).t())
    assert flow.sample_host(0).shape == (0, 6)


def test_seed_none_draws_from_the_default_generator(fake_sample):
    spec, params, _ = load_case("d6_hh_normal")
    flow = build_flow(spec, params, device="cpu", precision="fp32")
    torch.manual_seed(17)
    a = flow.sample_host(300)
    torch.manual_seed(17)
    assert torch.equal(a, flow.sample_host(300)) and not torch.equal(a, flow.sample_host(300))


def test_c_entries_reject_bad_arguments_without_gpu():
    from usflows_b200 import _lib
    lib = _lib.load()
    dr = _lib.Draw()
    buf = ctypes.c_void_p(16)
    assert lib.usf_base_sample_at(4, 4, buf, buf, 0, None, buf, 4, None, None, 0, None, 0, None) == -1
    assert b"bad draw" in lib.usf_last_error()
    dr.row0 = -1
    assert lib.usf_base_sample_at(4, 4, buf, buf, 0, ctypes.byref(dr), buf, 4, None, None, 0, None, 0, None) == -1
    dr.row0 = 0
    assert lib.usf_base_sample_at(4, 4, buf, buf, 9, ctypes.byref(dr), buf, 4, None, None, 0, None, 0, None) == -1
    assert lib.usf_base_sample_at(4, 0, buf, buf, 0, ctypes.byref(dr), buf, 4, None, None, 0, None, 0, None) == -1
    assert lib.usf_radial_sample_at(4, 4, buf, 2, 0, buf, 1, None, buf, 4, None) == -1
    assert b"bad draw" in lib.usf_last_error()
    assert lib.usf_radial_sample_at(4, 4, buf, 5, 0, buf, 1, ctypes.byref(dr), buf, 4, None) == -1
    assert lib.usf_radial_sample_at(4, 8, buf, 2, 0, buf, 1, ctypes.byref(dr), buf, 4, None) == -1      # ldo < d
    assert lib.usf_quantize_u8(None, 4, 1, 4, buf, 4, None) == -1
    assert lib.usf_quantize_u8(buf, 4, 1, 4, None, 4, None) == -1
    assert lib.usf_quantize_u8(buf, 4, 1, 4, buf, 3, None) == -1                                    # ldo < d
    assert lib.usf_quantize_u8(buf, 4, -1, 4, buf, 4, None) == -1
    assert lib.usf_layout_transpose_to_u8(None, 1, 16, 4, None, 0, buf, None) == -1
    assert lib.usf_layout_transpose_to_u8(buf, 1, 16, 4, None, 1, buf, None) == -1                   # scale missing
    assert lib.usf_layout_transpose_to_u8(buf, 1, 16, 4, buf, 3, buf, None) == -1


def test_draw_struct_layout_matches_header():
    from usflows_b200 import _lib
    with open(os.path.join(ROOT, "include", "usflows_b200.h")) as f:
        text = f.read()
    body = re.search(r"typedef struct usf_draw \{(.*?)\} usf_draw;", text, flags=re.S).group(1)
    names = re.findall(r"\*?(\w+);", body)
    assert names == [f[0] for f in _lib.Draw._fields_] == ["seed", "offset", "row0", "dev_params"]
    assert ctypes.sizeof(_lib.Draw) == 32
    assert [getattr(_lib.Draw, f).offset for f in names] == [0, 8, 16, 24]


# ---- B200 ---------------------------------------------------------------------------------------------------------------
def _radial_params(kind):
    from usflows_b200 import ops
    if kind == ops.NORM_LOGNORMAL:
        return torch.tensor([0.3, 0.4]), 1
    logits, a, b = [0.1, -0.4, 0.7], [0.6, 2.5, 7.0], [1.0, 2.0, 3.5]
    if kind == ops.NORM_GAMMA_MIXTURE:
        return torch.tensor(logits + a + b), 3
    if kind == ops.NORM_GENGAMMA_MIXTURE:
        return torch.tensor(logits + a + b + [0.5, 1.0, 2.0] + [2.0, 1.5, 0.7]), 3
    return torch.tensor(logits + [0.0, 0.5, 1.0] + [0.2, 0.3, 0.5]), 3


@pytest.mark.gpu
@pytest.mark.parametrize("d", [5, 7, 100, 784])
@pytest.mark.parametrize("kind", [0, 1])
def test_base_draws_at_global_rows(kind, d):
    from usflows_b200 import ops
    dev = "cuda"
    loc, scale = torch.randn(d, device=dev), torch.rand(d, device=dev) + 0.5
    rows, seed, off = 1000, 0x1234_5678_9ABC, 3 * 0x1000

    def draw(rows, dr):
        out = torch.empty(rows, d, device=dev)
        ops.base_sample_at(ops.Act(rows, d, f32=out), loc, scale, kind, dr)
        return out
    old = torch.empty(rows, d, device=dev)
    ops.base_sample(ops.Act(rows, d, f32=old), loc, scale, kind, seed, off)
    assert torch.equal(draw(rows, ops.Draw(seed, 0, None, off)), old)
    assert torch.equal(draw(300, ops.Draw(seed, 0, None, off).shifted(450)), old[450:750])
    params = torch.tensor([seed, 450], dtype=torch.int64, device=dev)
    assert torch.equal(draw(300, ops.Draw(0, 0, params, off)), old[450:750])
    assert torch.equal(draw(300, ops.Draw(0, 100, params, off)), old[550:850])
    ref = ref_base_sample(760, d, loc.cpu().double().numpy(), scale.cpu().double().numpy(), kind, seed, off)[700:]
    got = draw(60, ops.Draw(seed, 700, None, off)).cpu().double().numpy()
    assert np.abs(got - ref).max() <= 1e-4 * (1 + np.abs(ref).max())


@pytest.mark.gpu
@pytest.mark.parametrize("norm_kind", [0, 1, 2, 3])
@pytest.mark.parametrize("p_kind", [0, 1, 2])
def test_radial_draws_at_global_rows(p_kind, norm_kind):
    from usflows_b200 import ops
    dev = "cuda"
    d, rows, seed, off = 13, 900, 77, 0x2000
    loc = torch.randn(d, device=dev)
    params, K = _radial_params(norm_kind)
    params = params.to(dev)

    def draw(rows, dr):
        out = torch.empty(rows, d, device=dev)
        ops.radial_sample_at(out, loc, p_kind, norm_kind, params, K, dr)
        return out
    old = torch.empty(rows, d, device=dev)
    ops.radial_sample(old, loc, p_kind, norm_kind, params, K, seed, off)
    assert torch.equal(draw(rows, ops.Draw(seed, 0, None, off)), old)
    assert torch.equal(draw(200, ops.Draw(seed, 0, None, off).shifted(333)), old[333:533])
    dp = torch.tensor([seed, 333], dtype=torch.int64, device=dev)
    assert torch.equal(draw(200, ops.Draw(0, 0, dp, off)), old[333:533])


@pytest.mark.gpu
@pytest.mark.parametrize("d", [3, 8, 100, 784])
def test_quantize_is_bit_identical_to_the_restatement(d):
    import usflows_b200 as U
    g = torch.Generator().manual_seed(d)
    y = torch.rand(513, d, generator=g) * 1.2 - 0.1
    y[0, : min(d, 8)] = torch.tensor([-0.0, float("nan"), 1.0, 255.5 / 256, float("inf"), -float("inf"), -3.0, 0.5])[: min(d, 8)]
    got = U.quantize(y.cuda())
    assert got.dtype == torch.uint8 and torch.equal(got.cpu(), torch.from_numpy(np_quantize(y.numpy())))
    wide = y.cuda()[:, : d - 1] if d > 1 else y.cuda()                  # strided rows
    assert torch.equal(U.quantize(wide).cpu(), torch.from_numpy(np_quantize(wide.cpu().numpy())))
    k = torch.randint(0, 256, (300, d), generator=g, dtype=torch.uint8).cuda()
    for mode in ("uniform", "midpoint"):
        assert torch.equal(U.quantize(U.dequantize(k, mode, seed=d)), k)


def _n_rows(spec):
    return 700 if len(spec["in_dims"]) == 3 else 5000


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
@pytest.mark.parametrize("name", GPU_CASES + ["c1_d2_laplace", "img_bottleneck_c4_5x4"])
def test_every_route_streams_the_samples_of_its_seed(name, precision):
    import usflows_b200 as U
    from usflows_b200 import parallel
    spec, params, _ = load_case(name)
    flow = build_flow(spec, params, precision=precision)
    n = _n_rows(spec)
    ref = flow.sample([n], seed=11)
    torch.manual_seed(1)
    assert torch.equal(flow.sample([n], seed=11), ref)                  # reproducible, whatever torch's generator says
    ref = ref.cpu()
    assert ref.shape == (n, *spec["in_dims"]) and torch.isfinite(ref).all()
    got = flow.sample_host(n, seed=11)
    assert got.is_pinned() and torch.equal(got, ref)
    assert torch.equal(flow.sample_host(n, seed=11, chunk_rows=777), ref)
    U.set_chunk_rows(1024)
    try:
        assert torch.equal(flow.sample([n], seed=11).cpu(), ref)
        assert torch.equal(flow.sample_host(n, seed=11), ref)
    finally:
        U.set_chunk_rows(65536)
    q = flow.sample_host(n, seed=11, quantize=True)
    assert q.dtype == torch.uint8 and torch.equal(q, torch.from_numpy(np_quantize(ref.numpy())))
    assert torch.equal(flow.sample([n], seed=11, quantize=True).cpu(), q)
    assert torch.equal(U.quantize(flow.sample([n], seed=11)).cpu(), q)
    # one draw split over two calls, and over the visible devices
    n1 = n // 3
    a, b = flow.sample_host(n1, seed=11), flow.sample_host(n - n1, seed=11, row_offset=n1)
    assert torch.equal(torch.cat([a, b]), ref)
    assert torch.equal(parallel.sample_sharded(flow, n, seed=11), ref)
    assert torch.equal(parallel.sample_sharded(flow, n, seed=11, quantize=True), q)
    assert not torch.equal(flow.sample_host(n, seed=12), ref)


@pytest.mark.gpu
def test_fp16_range_guard_when_sampling():
    """A huge base scale pushes the ingested draws past the fp16 range: the chunks are recomputed on the tf32 split."""
    spec, params, _ = load_case("c2_d784")
    f16 = build_flow(spec, params, precision="fp32")
    tf = build_flow(spec, params, precision="fp32_tf32")
    for f in (f16, tf):
        with torch.no_grad():
            f._base_module().scale_unconstrained.fill_(1e6)
    want = tf.sample_host(5000, seed=2)
    assert torch.equal(f16.sample_host(5000, seed=2), want)
    assert torch.equal(f16.sample_host(5000, seed=2, chunk_rows=777), want)
    assert torch.equal(f16.sample([5000], seed=2).cpu(), want)


@pytest.mark.gpu
def test_streaming_memory_is_bounded_by_the_chunks():
    spec, params, _ = load_case("c2_d784")
    flow = build_flow(spec, params, precision="fp32")
    chunk, d = 2048, 784
    flow.sample_host(2 * chunk, seed=1, chunk_rows=chunk)              # workspaces, buffers and graphs of this chunk size
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    out = flow.sample_host(20 * chunk, seed=1, chunk_rows=chunk)
    torch.cuda.synchronize()
    assert torch.cuda.max_memory_allocated() - before <= 4 * chunk * d * 4
    assert torch.equal(out[:2 * chunk], flow.sample_host(2 * chunk, seed=1, chunk_rows=chunk))
    with pytest.raises(RuntimeError, match="host memory"):
        flow.sample_host(4, torch.empty(4, d, device="cuda"))


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["d100_h50_hh", "c2_d784"])
def test_seeded_samples_against_the_oracle(name):
    from oracle import flow_oracle as O
    spec, params, _ = load_case(name)
    flow = build_flow(spec, params, precision="fp32")
    y = flow.sample([64], seed=0xABCDEF).cpu()
    base = flow._base_module()
    loc, scale = base._prepared()
    d = loc.numel()
    z = torch.from_numpy(ref_base_sample(64, d, loc.cpu().double().numpy(), scale.cpu().double().numpy(), base.base_kind,
                                         0xABCDEF, 0))
    want = O.flow_forward(z, spec, params, dtype=torch.float64)
    assert rel_err(y, want) <= 3 * rel_err(O.flow_forward(z.float(), spec, params), want) + 1e-5
