"""8-bit inputs: dequantisation fused into the ingest kernels (usf_ingest_u8 / usf_layout_transpose_u8 / usf_flow_logprob_u8)
and the `dequantize=` argument of log_prob, log_prob_host and the row-shard driver.

The contract every route relies on (include/usflows_b200.h, usf_dequant): value k at flat event index j of global row r
becomes ((k << 16) | low) / 2^24 with low = 2 (Philox4x32-10(seed, (r, j >> 2))[j & 3] >> 17) + 1 ("uniform") or 0x8000
("midpoint").  `np_dequant` restates it in numpy; the emulated backend's 8-bit ops are built on that restatement."""
import ctypes

import numpy as np
import pytest
import torch

import fake_backend
from helpers import build_flow, load_case, rel_err
from philox_ref import MASK, np_philox4x32_10


def np_dequant(x, mode, seed, row0=0):
    """fp32 values of the uint8 rows x [rows, d] (numpy), global rows row0 .. row0 + rows - 1."""
    x = np.asarray(x, dtype=np.uint8)
    rows, d = x.shape
    k = x.astype(np.uint64)
    if mode == "midpoint":
        low = np.full(x.shape, 0x8000, dtype=np.uint64)
    else:
        r = (np.uint64(row0) + np.arange(rows, dtype=np.uint64))[:, None] * np.ones((1, d), dtype=np.uint64)
        j = np.ones((rows, 1), dtype=np.uint64) * np.arange(d, dtype=np.uint64)[None, :]
        hi = j >> np.uint64(2)
        seed = np.uint64(seed)
        out = np_philox4x32_10((r & MASK, r >> np.uint64(32), hi & MASK, hi >> np.uint64(32)), (seed & MASK, seed >> np.uint64(32)))
        word = np.choose((j & np.uint64(3)).astype(np.int64), out)
        low = ((word >> np.uint64(17)) << np.uint64(1)) | np.uint64(1)
    return ((k << np.uint64(16)) | low).astype(np.float32) * np.float32(2.0 ** -24)


def _hex(words):
    return [f"{int(w):08x}" for w in words]


def test_philox_restatement_reproduces_the_random123_known_answers():
    assert _hex(np_philox4x32_10((0, 0, 0, 0), (0, 0))) == ["6627e8d5", "e169c58d", "bc57ac4c", "9b00dbd8"]
    ones = 0xFFFFFFFF
    assert _hex(np_philox4x32_10((ones,) * 4, (ones, ones))) == ["408f276d", "41c83b0e", "a20bc7c6", "6d5451fd"]
    assert _hex(np_philox4x32_10((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0))) == \
        ["d16cfe09", "94fdcceb", "5001e420", "24126ea1"]


def test_dequantised_values_stay_inside_their_bin_and_are_exact():
    x = np.arange(256, dtype=np.uint8).reshape(32, 8)
    for mode in ("uniform", "midpoint"):
        v = np_dequant(x, mode, seed=12345).astype(np.float64)
        k = x.astype(np.float64)
        assert (v > k / 256).all() and (v < (k + 1) / 256).all()
        assert np.array_equal(v * 2 ** 24, np.round(v * 2 ** 24))
    assert np.array_equal(np_dequant(x, "midpoint", 0), (x.astype(np.float32) + 0.5) / 256)
    # noise depends on (seed, global row, j) only
    assert np.array_equal(np_dequant(x, "uniform", 7)[5:], np_dequant(x[5:], "uniform", 7, row0=5))
    assert not np.array_equal(np_dequant(x, "uniform", 7), np_dequant(x, "uniform", 8))


# ---- emulated backend ------------------------------------------------------------------------------------------------
def _fake_ingest_u8(x, dq, out, *, div=None, mul=None, sub=None, overflow_flag=None):
    fake_backend.CALLS.append(("ingest_u8", dq.row0))
    assert dq.params is None
    v = torch.from_numpy(np_dequant(x.numpy(), dq.mode, dq.seed, dq.row0))
    fake_backend.ingest(v, out, div=div, mul=mul, sub=sub, overflow_flag=overflow_flag)


def _fake_layout_transpose_u8(x, dq, n, c, hw, out, scale=None, scale_mode=0):
    fake_backend.CALLS.append(("layout_transpose_u8", dq.row0))
    v = torch.from_numpy(np_dequant(x.numpy(), dq.mode, dq.seed, dq.row0))
    fake_backend.layout_transpose(v, n, c, hw, out, scale=scale, scale_mode=scale_mode, scale_on_input=True)


@pytest.fixture
def fake_u8(fake_ops, monkeypatch):
    from usflows_b200 import ops
    monkeypatch.setattr(ops, "ingest_u8", _fake_ingest_u8)
    monkeypatch.setattr(ops, "layout_transpose_u8", _fake_layout_transpose_u8)
    return fake_ops


def _u8_batch(rows, ev, seed=0):
    g = torch.Generator().manual_seed(seed)
    return torch.randint(0, 256, (rows, *ev), generator=g, dtype=torch.uint8)


def _deq(x, mode, seed, row0=0):
    return torch.from_numpy(np_dequant(x.reshape(x.shape[0], -1).numpy(), mode, seed, row0)).reshape(x.shape)


@pytest.mark.parametrize("mode", ["uniform", "midpoint"])
@pytest.mark.parametrize("name", ["d100_h50_hh", "d36_conddense_nocontext", "d64_convnet_proj_radial2", "img_c4_4x4"])
def test_chunked_log_prob_passes_global_rows(fake_u8, monkeypatch, name, mode):
    from usflows_b200 import engine, image_engine
    spec, params, _ = load_case(name)
    flow = build_flow(spec, params, device="cpu", precision="fp32")
    x = _u8_batch(23 if len(spec["in_dims"]) == 3 else 600, spec["in_dims"])     # chunks: 5 images / 256 rows
    want = flow.log_prob(_deq(x, mode, 99))
    monkeypatch.setattr(engine, "_default_chunk_rows", 256)
    monkeypatch.setattr(image_engine, "IMAGE_CHUNK_ROWS", 5 * 16)
    monkeypatch.setattr(image_engine, "IMAGE_CHUNK_ROWS_PIX", 5 * 16)
    fake_backend.CALLS.clear()
    got = flow.log_prob(x, dequantize=mode, seed=99)
    rows0 = sorted({c[1] for c in fake_backend.CALLS if c[0] in ("ingest_u8", "layout_transpose_u8")})
    assert len(rows0) > 1 and rows0[0] == 0
    assert rel_err(got, want) <= 1e-6
    assert torch.equal(flow.log_prob(_deq(x, mode, 99)), flow.log_prob(x, dequantize=mode, seed=99))


def test_fp16_range_rerun_keeps_the_global_rows(fake_u8, monkeypatch):
    """Every chunk's ingest raises the range flag: the tf32-split re-run must read the same rows of the noise."""
    from usflows_b200 import engine
    spec, params, _ = load_case("d100_h50_hh")
    f16 = build_flow(spec, params, device="cpu", precision="fp32")
    tf = build_flow(spec, params, device="cpu", precision="fp32_tf32")
    x = _u8_batch(600, spec["in_dims"], seed=3)
    monkeypatch.setattr(engine, "_default_chunk_rows", 256)

    def tripping(x, dq, out, *, overflow_flag=None, **kw):
        _fake_ingest_u8(x, dq, out, overflow_flag=overflow_flag, **kw)
        if overflow_flag is not None:
            overflow_flag.fill_(1)
    from usflows_b200 import ops
    monkeypatch.setattr(ops, "ingest_u8", tripping)
    fake_backend.CALLS.clear()
    got = f16.log_prob(x, dequantize="uniform", seed=5)
    assert ops.ENGINE_TC_3XTF32 in {c[1] for c in fake_backend.CALLS if c[0] == "linear"}
    assert torch.equal(got, tf.log_prob(_deq(x, "uniform", 5)))


def test_row_shard_driver_gives_each_block_its_global_rows(fake_u8):
    """Two emulated shards: one seed for both, block i starts at its global row."""
    from usflows_b200 import ops, parallel
    spec, params, _ = load_case("d6_hh_normal")
    flow = build_flow(spec, params, device="cpu", precision="fp32")
    x = _u8_batch(11, spec["in_dims"], seed=4)
    seen = []

    def host(x_host, out_host=None, chunk_rows=None, *, dequantize=None, seed=None, row_offset=0):
        seen.append((x_host.shape[0], seed, row_offset))
        out_host.copy_(flow._log_prob_any(x_host, None, ops.Dequant(dequantize, seed, row_offset)))
        return out_host

    sf = parallel.ShardedFlow.__new__(parallel.ShardedFlow)
    sf.flow, sf.devices, sf.replicas, sf._synced = flow, ["a", "b"], [flow, flow], flow._weights_key()
    from concurrent.futures import ThreadPoolExecutor
    sf._pool = ThreadPoolExecutor(max_workers=1)
    flow.log_prob_host = host
    try:
        out = torch.empty(11)
        sf.log_prob(x, out, dequantize="uniform", seed=31)
    finally:
        sf.close()
        del flow.log_prob_host
    assert sorted(seen) == [(5, 31, 6), (6, 31, 0)]
    full = _deq(x, "uniform", 31)
    assert torch.equal(out[:6], flow.log_prob(full[:6])) and torch.equal(out[6:], flow.log_prob(full[6:]))


def test_argument_errors(fake_u8):
    import usflows_b200 as U
    spec, params, arr = load_case("d6_hh_normal")
    flow = build_flow(spec, params, device="cpu", precision="fp32")
    x = _u8_batch(4, spec["in_dims"])
    with pytest.raises(ValueError, match="uint8"):
        flow.log_prob(arr["x"], dequantize="uniform")
    with pytest.raises(ValueError, match="unknown dequantize mode"):
        flow.log_prob(x, dequantize="floor")
    with pytest.raises(ValueError, match="uint8"):
        flow.log_prob_host(arr["x"], dequantize="midpoint")
    with pytest.raises(ValueError, match="unknown dequantize mode"):
        U.dequantize(x, "nearest")
    from usflows_b200 import parallel
    with pytest.raises(ValueError, match="uint8"):
        parallel.ShardedFlow.log_prob(parallel.ShardedFlow.__new__(parallel.ShardedFlow), arr["x"], dequantize="uniform")


def test_seed_none_draws_from_the_default_generator():
    from usflows_b200 import ops
    x = torch.zeros(2, 3, dtype=torch.uint8)
    torch.manual_seed(17)
    a, b = ops.dequant_spec(x, "uniform").seed, ops.dequant_spec(x, "uniform").seed
    torch.manual_seed(17)
    assert ops.dequant_spec(x, "uniform").seed == a and a != b and 0 <= a < 2 ** 63


def test_c_entries_reject_bad_arguments_without_gpu():
    from usflows_b200 import _lib
    lib = _lib.load()
    dq = _lib.Dequant()
    planes = _lib.Planes()
    buf = ctypes.c_void_p(16)
    assert lib.usf_ingest_u8(None, 4, 1, 4, ctypes.byref(dq), None, None, None, ctypes.byref(planes), None, None) == -1
    assert b"bad input" in lib.usf_last_error()
    assert lib.usf_ingest_u8(buf, 4, 1, 4, None, None, None, None, ctypes.byref(planes), None, None) == -1
    assert b"dequantisation" in lib.usf_last_error()
    dq.mode = 7
    assert lib.usf_ingest_u8(buf, 4, 1, 4, ctypes.byref(dq), None, None, None, ctypes.byref(planes), None, None) == -1
    dq.mode = _lib.DEQUANT_UNIFORM
    assert lib.usf_ingest_u8(buf, 4, 1, 4, ctypes.byref(dq), None, None, None, ctypes.byref(planes), None, None) == -1
    assert b"output plane" in lib.usf_last_error()
    assert lib.usf_ingest_u8(buf, 2, 1, 4, ctypes.byref(dq), None, None, None, ctypes.byref(planes), None, None) == -1
    assert lib.usf_layout_transpose_u8(None, 1, 4, 16, ctypes.byref(dq), None, 0, buf, None) == -1
    assert lib.usf_layout_transpose_u8(buf, 1, 4, 16, None, None, 0, buf, None) == -1
    assert lib.usf_layout_transpose_u8(buf, 1, 4, 16, ctypes.byref(dq), None, 1, buf, None) == -1     # scale missing
    h = ctypes.c_void_p()
    assert lib.usf_plan_create(ctypes.byref(h), 8, 0, 16) == 0
    try:
        assert lib.usf_flow_logprob_u8(h, buf, 8, 1, ctypes.byref(dq), buf, None, None) == -1      # not finalized
        assert lib.usf_flow_logprob_u8(None, buf, 8, 1, ctypes.byref(dq), buf, None, None) == -1
    finally:
        assert lib.usf_plan_destroy(h) == 0
    # the header's struct and the ctypes mirror agree
    assert ctypes.sizeof(_lib.Dequant) == 4 + 4 + 8 + 8 + 8


# ---- B200 ---------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["uniform", "midpoint"])
@pytest.mark.parametrize("d", [5, 100, 784])
def test_dequantize_is_bit_identical_to_the_restatement(d, mode):
    import usflows_b200 as U
    x = _u8_batch(777, (d,), seed=d)
    got = U.dequantize(x.cuda(), mode, seed=0x1234_5678_9ABC_DEF, row_offset=40)
    assert torch.equal(got.cpu(), _deq(x, mode, 0x1234_5678_9ABC_DEF, 40))
    wide = _u8_batch(777, (d + 13,), seed=1).cuda()                 # strided rows (ld = d + 13)
    assert torch.equal(U.dequantize(wide[:, :d], mode, seed=3).cpu(), _deq(wide[:, :d].cpu(), mode, 3))
    img = _u8_batch(9, (4, 5, 7), seed=2)
    assert torch.equal(U.dequantize(img.cuda(), mode, seed=11).cpu(), _deq(img, mode, 11))
    torch.manual_seed(5)
    a = U.dequantize(x.cuda(), mode)
    torch.manual_seed(5)
    assert torch.equal(a, U.dequantize(x.cuda(), mode))


GPU_CASES = ["d100_h50_hh", "c2_d784", "d64_convnet_proj_radial2", "d36_conddense_nocontext", "img_mnist_16x7x7", "img_c4_4x4",
             "img_c6_5x3_plain_channel"]


@pytest.mark.gpu
@pytest.mark.parametrize("precision", ["fp32", "fp32_tf32", "fp32_simt", "tf32", "bf16"])
@pytest.mark.parametrize("name", GPU_CASES)
def test_every_route_reaches_the_result_of_the_dequantised_rows(name, precision):
    import usflows_b200 as U
    from usflows_b200 import parallel
    from oracle import flow_oracle as O
    spec, params, _ = load_case(name)
    flow = build_flow(spec, params, precision=precision)
    image = len(spec["in_dims"]) == 3
    rows = 1500 if image else 5000                                     # past the small-batch graph path
    x = _u8_batch(rows, spec["in_dims"], seed=7)
    xd = x.cuda()
    for mode, seed in (("uniform", 123), ("midpoint", 0)):
        ref = flow.log_prob(U.dequantize(xd, mode, seed=seed))
        assert torch.equal(flow.log_prob(xd, dequantize=mode, seed=seed), ref)
        U.set_chunk_rows(1024)
        try:
            assert torch.equal(flow.log_prob(xd, dequantize=mode, seed=seed),
                               flow.log_prob(U.dequantize(xd, mode, seed=seed)))
        finally:
            U.set_chunk_rows(65536)
        small = flow.log_prob(xd[:100], dequantize=mode, seed=seed)    # small-batch graph path
        assert torch.equal(small, flow.log_prob(U.dequantize(xd[:100], mode, seed=seed)))
    # host path: growing chunk schedule with graph replay, two seeds in turn, uniform chunks, the row-shard driver
    xh = x.pin_memory()
    for seed in (5, 6):
        ref = flow.log_prob(U.dequantize(xd, "uniform", seed=seed)).cpu()
        assert torch.equal(flow.log_prob_host(xh, dequantize="uniform", seed=seed), ref)
    assert not torch.equal(ref, flow.log_prob(U.dequantize(xd, "uniform", seed=5)).cpu())
    ref = flow.log_prob(U.dequantize(xd, "uniform", seed=8)).cpu()
    assert torch.equal(flow.log_prob_host(xh, chunk_rows=777, dequantize="uniform", seed=8), ref)
    assert torch.equal(parallel.log_prob_sharded(flow, xh, dequantize="uniform", seed=8), ref)
    # the dequantised rows against the fp64 oracle (DESIGN section 2 bounds: 1e-5 for the fp32-accurate modes)
    if precision in ("fp32", "fp32_tf32", "fp32_simt"):
        xs = U.dequantize(xd[:64], "uniform", seed=8).cpu()
        lp = flow.log_prob(xd[:64], dequantize="uniform", seed=8).cpu()
        assert rel_err(lp, O.flow_log_prob(xs, spec, params, dtype=torch.float64)) <= \
            3 * rel_err(O.flow_log_prob(xs, spec, params), O.flow_log_prob(xs, spec, params, dtype=torch.float64)) + 1e-5


@pytest.mark.gpu
def test_uint8_without_dequantize_keeps_the_dtype_error():
    spec, params, _ = load_case("d6_hh_normal")
    flow = build_flow(spec, params)
    with pytest.raises(RuntimeError, match="dtype"):
        flow.log_prob(_u8_batch(4, spec["in_dims"]).cuda())


@pytest.mark.gpu
def test_fp16_range_guard_with_uint8_input():
    """A tiny ScaleTransform pushes the ingested values past the fp16 range: the chunk is recomputed on the tf32 split."""
    import usflows_b200 as U
    spec, params, _ = load_case("d100_h50_hh")
    f16 = build_flow(spec, params, precision="fp32")
    tf = build_flow(spec, params, precision="fp32_tf32")
    for f in (f16, tf):
        with torch.no_grad():
            f.layers[-1].scale.mul_(1e-6)
    x = _u8_batch(5000, spec["in_dims"], seed=1)
    want = tf.log_prob(U.dequantize(x.cuda(), "uniform", seed=2))
    assert torch.equal(f16.log_prob(x.cuda(), dequantize="uniform", seed=2), want)
    assert torch.equal(f16.log_prob_host(x.pin_memory(), dequantize="uniform", seed=2), want.cpu())


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["c2_d784", "img_mnist_16x7x7"])
def test_dequantisation_adds_no_kernel(name):
    """fp32 mode, C-plan and image-program routes: a uint8 call launches as many CUDA kernels as an fp32 call."""
    import usflows_b200 as U
    from torch.profiler import ProfilerActivity, profile
    spec, params, _ = load_case(name)
    flow = build_flow(spec, params, precision="fp32")
    rows = 2048 if len(spec["in_dims"]) == 3 else 8192
    x = _u8_batch(rows, spec["in_dims"], seed=2).cuda()
    xf = U.dequantize(x, "uniform", seed=1)
    flow.log_prob(xf)
    flow.log_prob(x, dequantize="uniform", seed=1)
    torch.cuda.synchronize()

    def kernels(fn):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            fn()
            torch.cuda.synchronize()
        return sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA
                   and "memcpy" not in e.name.lower() and "memset" not in e.name.lower())
    assert kernels(lambda: flow.log_prob(x, dequantize="uniform", seed=1)) == kernels(lambda: flow.log_prob(xf))
