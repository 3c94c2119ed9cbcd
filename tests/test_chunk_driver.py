"""The chunk driver every evaluation route runs through (engine.chunk_bounds / engine.run_chunks): how a batch is cut, and
the fp16-range re-run of the "fp32" mode -- a chunk whose activations leave the fp16 range raises its device flag and is
recomputed with the tf32-split program; the other chunks keep the fp16-split result.  Chunks are tripped on purpose: their
rows must equal the "fp32_tf32" flow's, every other row the "fp32" flow's on the same rows.  On the emulated backend the two
programs may agree on a row, so which chunks were re-run is counted from the tf32-split launches there; on the B200 the
results of the two programs differ, and the rows alone tell."""
import pytest
import torch

import fake_backend
from helpers import build_flow, load_case
from oracle import flow_oracle as O
from test_dequant_u8 import _deq, _fake_ingest_u8, _u8_batch, fake_u8  # noqa: F401  (fake_u8 is a fixture)

AFFINE_D64 = dict(in_dims=[64], coupling_blocks=2, hidden_dims=[64, 64], affine_conjugation=True, lu_transform=1,
                  householder=0, base="laplace", coupling="affine")     # every width >= TC_MIN_DIM: the "fp32" engine
ADDITIVE_D64 = dict(AFFINE_D64, coupling="additive")                   # ... and the whole-stack C entry covers it


def _case(name):
    if name in ("affine_d64", "additive_d64"):
        spec = AFFINE_D64 if name == "affine_d64" else ADDITIVE_D64
        params = O.random_params(spec, 11)
        for k, v in params.items():     # well-conditioned LU factors and scales near 1: inputs in [0, 1) stay in the fp16 range
            if k.endswith(("L_raw", "U_raw")):
                params[k] = 0.1 * v
            elif k.endswith(".scale"):
                params[k] = 1 + 0.1 * v
        return spec, params
    spec, params, _ = load_case(name)
    return spec, params


def _flows(name, device):
    spec, params = _case(name)
    return spec, build_flow(spec, params, device=device, precision="fp32"), \
        build_flow(spec, params, device=device, precision="fp32_tf32")


def _rows(n, d, chunks, scale, seed=1):
    """n rows and a copy whose rows [r0, r1) of each of `chunks` are scaled out of the fp16 range."""
    x = torch.rand(n, *d, generator=torch.Generator().manual_seed(seed))
    big = x.clone()
    for r0, r1 in chunks:
        big[r0:r1] *= scale
    return x, big


def _check_rerun(got, want16, want_tf, chunks, distinct=False):
    """Rows of `chunks` equal the tf32-split program's, every other row the fp16-split program's.  `distinct`: the two
    programs' results differ on those other rows too, so a re-run of every chunk would not pass."""
    rerun = torch.zeros(got.shape[0], dtype=torch.bool)
    for r0, r1 in chunks:
        rerun[r0:r1] = True
    assert torch.equal(got[rerun], want_tf[rerun]) and torch.equal(got[~rerun], want16[~rerun])
    assert not distinct or not torch.equal(want16[~rerun], want_tf[~rerun])


def _tf32_split_calls():
    """Launches of the tf32-split program: its contractions, and its implicit-GEMM convolutions (image conditioners)."""
    return [c for c in fake_backend.CALLS
            if (c[0] == "linear" and c[1] == fake_backend.ENGINE_TC_3XTF32) or c[0] == "conv2d_rows"]


# ---- emulated backend ------------------------------------------------------------------------------------------------
def test_chunk_bounds_cut_as_before():
    from usflows_b200 import engine

    def inline(rows, cap):                                  # the cut Program.run made before chunk_bounds existed
        if rows == 0:
            return []
        n_chunks = (rows + cap - 1) // cap
        chunk = min(rows, ((rows + n_chunks - 1) // n_chunks + 255) // 256 * 256)
        return [(r0, min(rows, r0 + chunk)) for r0 in range(0, rows, chunk)]

    for cap in (1, 100, 256, 1000, 4096, 65536):
        for rows in sorted({0, 1, 255, 256, 257, 600, cap - 1, cap, cap + 1, 3 * cap + 7, 10 * cap}):
            got = engine.chunk_bounds(rows, cap)
            assert got == inline(rows, cap), (rows, cap)
            assert [r for b in got for r in b] == sorted(r for b in got for r in b) and sum(r1 - r0 for r0, r1 in got) == rows


def test_run_chunks_rereads_every_chunk_when_a_shared_flag_is_set():
    from usflows_b200 import engine
    bounds = [(0, 4), (4, 8), (8, 10)]
    ladj = torch.ones(10)
    seen, redo = [], []

    def first(i, r0, r1, flag):
        seen.append((i, r0, r1, flag is None))
        if flag is not None and i == 1:
            flag.fill_(1)

    engine.run_chunks(bounds, "cpu", True, first, lambda i, r0, r1: redo.append(i), ladj_rows=ladj)
    assert seen == [(0, 0, 4, False), (1, 4, 8, False), (2, 8, 10, False)] and redo == [1]
    assert torch.equal(ladj, torch.tensor([1.0] * 4 + [0.0] * 4 + [1.0] * 2))
    redo.clear()
    engine.run_chunks(bounds, "cpu", True, lambda *a: None, lambda i, r0, r1: redo.append(i),
                      shared_flags=[torch.zeros(1, dtype=torch.int32), torch.ones(1, dtype=torch.int32)])
    assert redo == [0, 1, 2]
    seen.clear()
    engine.run_chunks(bounds, "cpu", False, first, None)     # unguarded: no flag, nothing re-run
    assert [s[3] for s in seen] == [True, True, True]


@pytest.mark.parametrize("what", ["log_prob", "backward"])
@pytest.mark.parametrize("name", ["d100_h50_hh", "affine_d64", "additive_d64"])
def test_only_the_flagged_chunk_is_rerun(fake_ops, monkeypatch, name, what):
    """600 rows at 256-row chunks: (0, 256), (256, 512), (512, 600); chunk 1 leaves the fp16 range.  The affine couplings
    add per-row log-determinants: the re-run chunk must not keep those of the abandoned pass."""
    from usflows_b200 import engine
    spec, f16, tf = _flows(name, "cpu")
    monkeypatch.setattr(engine, "_default_chunk_rows", 256)
    x, big = _rows(600, spec["in_dims"], [(256, 512)], 3e5)
    want16, want_tf = getattr(f16, what)(x), getattr(tf, what)(big)
    fake_backend.CALLS.clear()
    getattr(tf, what)(big[256:512])
    per_chunk = len(_tf32_split_calls())
    fake_backend.CALLS.clear()
    got = getattr(f16, what)(big)
    calls = _tf32_split_calls()
    assert per_chunk > 0 and len(calls) == per_chunk and {c[2] for c in calls} == {256}
    _check_rerun(got, want16, want_tf, [(256, 512)])


def test_only_the_flagged_chunk_is_rerun_on_8bit_rows(fake_u8, monkeypatch):
    """The tf32-split re-run of chunk 1 dequantises the same global rows 256.. as its first pass."""
    from usflows_b200 import engine, ops
    _, f16, tf = _flows("d100_h50_hh", "cpu")
    monkeypatch.setattr(engine, "_default_chunk_rows", 256)
    x = _u8_batch(600, [100], seed=3)

    def tripping(x, dq, out, *, overflow_flag=None, **kw):
        _fake_ingest_u8(x, dq, out, overflow_flag=overflow_flag, **kw)
        if overflow_flag is not None and dq.row0 == 256:
            overflow_flag.fill_(1)
    monkeypatch.setattr(ops, "ingest_u8", tripping)
    xf = _deq(x, "uniform", 5)
    want16, want_tf = f16.log_prob(xf), tf.log_prob(xf)
    fake_backend.CALLS.clear()
    got = f16.log_prob(x, dequantize="uniform", seed=5)
    assert {c[2] for c in _tf32_split_calls()} == {256}
    _check_rerun(got, want16, want_tf, [(256, 512)])


@pytest.mark.parametrize("what", ["log_prob", "backward"])
def test_only_the_flagged_image_chunk_is_rerun(fake_ops, monkeypatch, what):
    """Chunks of 4 images; image 5 (chunk 1) leaves the fp16 range of the pixel planes."""
    from usflows_b200 import image_engine
    spec, f16, tf = _flows("img_mnist_16x7x7", "cpu")
    monkeypatch.setattr(image_engine, "IMAGE_CHUNK_ROWS", 49 * 4)
    monkeypatch.setattr(image_engine, "IMAGE_CHUNK_ROWS_PIX", 49 * 4)
    x, big = _rows(12, spec["in_dims"], [(5, 6)], 1e6)
    want16, want_tf = getattr(f16, what)(x), getattr(tf, what)(big)
    fake_backend.CALLS.clear()
    getattr(tf, what)(big[4:8])
    per_chunk = len(_tf32_split_calls())
    fake_backend.CALLS.clear()
    got = getattr(f16, what)(big)
    assert per_chunk > 0 and len(_tf32_split_calls()) == per_chunk
    _check_rerun(got, want16, want_tf, [(4, 8)])


def test_only_the_flagged_chunk_of_a_network_run_alone_is_rerun(fake_ops, monkeypatch):
    """nn.DenseNN / nn.ConvNet called on their own (engine.run_mlp / run_conditioner): chunk 1 leaves the fp16 range and is
    recomputed with the network's own tf32-split launches."""
    from usflows_b200 import engine, nn
    monkeypatch.setattr(engine, "_default_chunk_rows", 256)
    torch.manual_seed(0)
    x, big = _rows(600, [64], [(256, 512)], 3e5)
    for run, net in ((engine.run_mlp, nn.DenseNN(64, [64, 64], [64])), (engine.run_conditioner, nn.ConvNet([64], [64, 64]))):
        want16, want_tf = run(net, x, "fp32"), run(net, big, "fp32_tf32")
        fake_backend.CALLS.clear()
        got = run(net, big, "fp32")
        assert {c[2] for c in _tf32_split_calls()} == {256}
        _check_rerun(got, want16, want_tf, [(256, 512)])


# ---- B200 ------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("what", ["log_prob", "backward"])
def test_gpu_whole_stack_plan_reruns_only_the_flagged_chunk(monkeypatch, what):
    """`log_prob` / `backward` through the whole-stack C entry (one call per chunk), chunk 1 re-run launch by launch."""
    from usflows_b200 import engine, flows
    spec, f16, tf = _flows("additive_d64", "cuda")
    monkeypatch.setattr(engine, "_default_chunk_rows", 256)
    monkeypatch.setattr(flows, "SMALL_BATCH_GRAPH_ROWS", 0)
    x, big = _rows(800, spec["in_dims"], [(256, 512)], 3e5)
    x, big = x.cuda(), big.cuda()
    want16, want_tf = getattr(f16, what)(x), getattr(tf, what)(big)
    got = getattr(f16, what)(big)
    prog, _ = f16._program("backward")                        # data -> latent: both calls
    assert prog.plan_able() and prog.__dict__.get("_c_plans")
    _check_rerun(got, want16, want_tf, [(256, 512)], distinct=True)


def _host_staging(monkeypatch, staging):
    """"whole": the batch staged on the device at once, one buffer per chunk; "ring": two staging buffers in turn, so a
    re-run has to stage its rows again."""
    from usflows_b200 import flows
    monkeypatch.setattr(flows, "HOST_MAX_STAGE_SLICES", 8 if staging == "whole" else 1)


@pytest.mark.gpu
@pytest.mark.parametrize("staging", ["whole", "ring"])
def test_gpu_host_path_reruns_only_the_flagged_chunks(monkeypatch, staging):
    """`log_prob_host` at chunk_rows=256 over 800 rows: (0, 256), (256, 512), (512, 800), launch by launch; chunks 0 and 2
    leave the fp16 range."""
    from usflows_b200 import flows
    spec, f16, tf = _flows("d100_h50_hh", "cuda")
    monkeypatch.setattr(flows, "HOST_CUDA_GRAPHS", False)
    _host_staging(monkeypatch, staging)
    x, big = _rows(800, spec["in_dims"], [(0, 256), (512, 800)], 3e5)
    x, big = x.pin_memory(), big.pin_memory()
    want16, want_tf = f16.log_prob_host(x, chunk_rows=256), tf.log_prob_host(big, chunk_rows=256)
    _check_rerun(f16.log_prob_host(big, chunk_rows=256), want16, want_tf, [(0, 256), (512, 800)], distinct=True)


@pytest.mark.gpu
@pytest.mark.parametrize("staging", ["whole", "ring"])
def test_gpu_host_chunk_graphs_rerun_every_chunk(monkeypatch, staging):
    """With captured chunk graphs a flag belongs to a graph, not to a chunk: one tripped chunk re-runs them all."""
    from usflows_b200 import flows
    spec, f16, tf = _flows("d100_h50_hh", "cuda")
    _host_staging(monkeypatch, staging)
    x, big = _rows(800, spec["in_dims"], [(256, 512)], 3e5)
    x, big = x.pin_memory(), big.pin_memory()
    monkeypatch.setattr(flows, "HOST_CUDA_GRAPHS", False)
    want16, want_tf = f16.log_prob_host(x, chunk_rows=256), tf.log_prob_host(big, chunk_rows=256)
    monkeypatch.setattr(flows, "HOST_CUDA_GRAPHS", True)
    got = f16.log_prob_host(big, chunk_rows=256)
    prog, _ = f16._program("backward")
    assert any(k[0] == "host" for k in prog.__dict__.get("_graphs", {}))
    assert torch.equal(got, want_tf) and not torch.equal(want16[:256], want_tf[:256])


@pytest.mark.gpu
def test_gpu_host_path_reruns_only_the_flagged_image_chunk():
    """Image events on the host path: chunks of 4 images, each through `log_prob`; image 5 leaves the fp16 range."""
    spec, f16, tf = _flows("img_mnist_16x7x7", "cuda")
    x, big = _rows(12, spec["in_dims"], [(5, 6)], 1e6)
    x, big = x.pin_memory(), big.pin_memory()
    want16, want_tf = f16.log_prob_host(x, chunk_rows=4), tf.log_prob_host(big, chunk_rows=4)
    _check_rerun(f16.log_prob_host(big, chunk_rows=4), want16, want_tf, [(4, 8)])
