"""GPU: the CUDA path (through the C ABI) reproduces the reference outputs in
tests/golden/ and agrees with the oracle on the same inputs.  Bit-exact for
integer/bool outputs, rtol 1e-5 for floats (see tests/_cases.py)."""
import numpy as np
import pytest

from tests._cases import assert_matches, case_names, load_case, uses_blas

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def rt():
    import torch

    from aesara_b200.runtime import lib
    from aesara_b200.runtime.vm import ProgramExecutor

    lib.check(lib.load().ab_init(0))
    torch.cuda.set_device(0)
    return ProgramExecutor


# fixtures whose whole program is int64 shape arithmetic (SURVEY a9): nothing to launch
PURE_METADATA = ()
_LAUNCHES = {}


@pytest.mark.parametrize("name", case_names())
def test_cuda_matches_reference_and_oracle(rt, name):
    from oracle.program_np import run_program

    from aesara_b200.runtime import lib

    prog, ins, want = load_case(name)
    ex = rt(prog)
    before = lib.load().ab_launch_count()
    got = ex(*[np.array(a) for a in ins])
    launched = lib.load().ab_launch_count() - before
    _LAUNCHES[name] = launched
    # every fixture must reach CUDA: tensor arguments are uploaded whatever their size
    # (runtime/vm.py host_needed_vars); only programs that are shape arithmetic from end to
    # end may finish without a launch
    assert launched > 0 or name in PURE_METADATA, f"{name}: no kernel of libaesara_b200.so ran"
    oracle = run_program(prog, [np.array(a) for a in ins])
    blas = uses_blas(prog)
    for k, (g, w, o) in enumerate(zip(got, want, oracle)):
        assert_matches(g, w, blas=blas, what=f"{name} output {k} vs reference")
        assert_matches(g, o, blas=blas, what=f"{name} output {k} vs oracle")


@pytest.mark.parametrize("name", ["cfg2_fused", "cfg3_mlp", "cfg5_logreg"])
def test_device_resident_call(rt, name):
    """Inputs given as DeviceArrays, outputs left on the device."""
    from aesara_b200.runtime.device import DeviceArray

    prog, ins, want = load_case(name)
    ex = rt(prog, host_outputs=False)
    dins = [DeviceArray.from_numpy(a) if np.ndim(a) > 0 else a for a in ins]
    got = ex(*dins)
    for k, (g, w) in enumerate(zip(got, want)):
        assert isinstance(g, DeviceArray) or np.ndim(g) == 0
        assert_matches(np.asarray(g), w, blas=uses_blas(prog), what=f"{name} out {k}")


@pytest.mark.parametrize("name", ["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"])
def test_baseline_calls_match_the_c_linker(rt, name):
    """The five BASELINE graphs as the linker lowers them (the committed programs), at the
    sizes and on the seeded inputs of tests/test_gpu_function.py, against the outputs the
    reference C-linker computed for the same calls (stored, sampled where large)."""
    from aesara_b200 import graphs as G
    from aesara_b200.runtime import lib
    from tests._cases import BASELINE_CALLS, assert_matches_c_linker

    program, _, inputs = BASELINE_CALLS[name]
    prog, _, _ = load_case(program)
    ex = rt(prog)
    before = lib.load().ab_launch_count()
    got = ex(*[np.array(a) for a in inputs(G)])
    assert lib.load().ab_launch_count() > before, "no kernel of libaesara_b200.so ran"
    assert_matches_c_linker(name, got)
    if name == "cfg4":
        scan = [st["runner"] for st in ex._state if "runner" in st][0]
        assert scan.used_fast_path, "the persistent Scan kernel did not run"


def test_host_api_pinned_uploads_overlap_and_results_are_not_recycled(rt):
    """Page-locked arguments go through the asynchronous copy stream, pageable ones
    through the synchronous path; both give the same bits.  Large outputs come back in
    page-locked blocks that the caller owns (a later call must not overwrite them)."""
    import torch

    prog, _, _ = load_case("cfg2_fused")
    n = 1 << 20
    rng = np.random.default_rng(3)
    ins = [rng.standard_normal(n).astype("float32") for _ in range(3)]
    pinned = []
    for a in ins:
        t = torch.empty(a.shape, dtype=torch.float32, pin_memory=True)
        t.numpy()[:] = a
        pinned.append(t)
    ex = rt(prog)
    (r_pageable,) = ex(*ins)
    (r_pinned,) = ex(*[t.numpy() for t in pinned])
    assert np.array_equal(r_pageable, r_pinned)
    keep = r_pinned.copy()
    (r_other,) = ex(*[-a for a in ins])
    assert np.array_equal(r_pinned, keep), "an earlier result was overwritten by a later call"
    assert not np.array_equal(r_other, keep)
    assert len(ex._inflight) == 0  # the last call had pageable arguments only
    (r_again,) = ex(*[t.numpy() for t in pinned])
    assert len(ex._inflight) == 3 and np.array_equal(r_again, keep)


@pytest.mark.parametrize("n", [1, 3, 1023, 1 << 20, (1 << 22) + 5])
def test_fused_elemwise_sizes(rt, n):
    """cfg2 graph at ragged sizes, incl. misaligned views (scalar fallback path)."""
    from oracle.program_np import run_program
    from aesara_b200.runtime.device import DeviceArray

    prog, _, _ = load_case("cfg2_fused")
    rng = np.random.default_rng(n)
    ins = [rng.standard_normal(n + 1).astype("float32") for _ in range(3)]
    ex = rt(prog)
    want = run_program(prog, [a[:n] for a in ins])[0]
    got = ex(*[a[:n] for a in ins])[0]
    assert_matches(got, want, what="aligned")
    dins = [DeviceArray.from_numpy(a).index((slice(1, None),)) for a in ins]  # 4-byte offset views
    got2 = ex(*dins)[0]
    want2 = run_program(prog, [a[1:] for a in ins])[0]
    assert_matches(got2, want2, what="misaligned")


def test_empty_inputs(rt):
    prog, _, _ = load_case("cfg2_fused")
    ex = rt(prog)
    z = np.zeros(0, "float32")
    assert ex(z, z, z)[0].shape == (0,)


def test_shape_mismatch_raises(rt):
    prog, _, _ = load_case("cfg2_fused")
    ex = rt(prog)
    a = np.zeros(8, "float32")
    b = np.zeros(9, "float32")
    with pytest.raises(Exception, match="dimension mismatch"):
        ex(a, b, a)


def test_full_size_properties(rt):
    """cfg2 at 2^26 elements: linearity in z and agreement of two launch geometries."""
    import torch

    from aesara_b200.runtime.device import DeviceArray

    prog, _, _ = load_case("cfg2_fused")
    ex = rt(prog, host_outputs=False)
    n = 1 << 26
    g = torch.Generator(device="cuda").manual_seed(0)
    x, y, z = (torch.randn(n, device="cuda", generator=g) for _ in range(3))
    o1 = ex(DeviceArray.from_torch(x), DeviceArray.from_torch(y), DeviceArray.from_torch(z))[0]
    o2 = ex(DeviceArray.from_torch(x), DeviceArray.from_torch(y), DeviceArray.from_torch(2 * z))[0]
    t1 = torch.frombuffer(o1.owner, dtype=torch.float32) if False else o1.owner.view(torch.float32)
    t2 = o2.owner.view(torch.float32)
    assert torch.equal(t2[:n], 2 * t1[:n])  # exact: scaling by 2 commutes with rounding
    ref = (torch.nn.functional.softplus(torch.tanh(x.double()) + y.double()) * z.double())
    err = ((t1[:n].double() - ref).abs() / (ref.abs() + 1e-6)).max().item()
    assert err < 1e-5


def test_logreg_full_size_fused_vs_node_by_node(rt):
    """cfg5 at 2^22 rows x 512 (no CPU truth at this size): the single-pass row-region
    kernel agrees with the node-by-node device execution, and doubling a duplicated batch
    leaves the mean cost and gradients unchanged (a checksum of checksums)."""
    import os

    import torch

    from aesara_b200.runtime.device import DeviceArray

    prog, _, _ = load_case("cfg5_logreg")
    N, D = 1 << 22, 512
    g = torch.Generator(device="cuda").manual_seed(1)
    X = torch.randn(N, D, device="cuda", generator=g)
    y = (torch.rand(N, device="cuda", generator=g) < 0.5).float()
    w = torch.randn(D, device="cuda", generator=g) * 0.01
    ins = [DeviceArray.from_torch(X), DeviceArray.from_torch(y), DeviceArray.from_torch(w), np.float32(0.1)]
    ex = rt(prog, host_outputs=False)
    fused = [np.asarray(o) for o in ex(*ins)]
    assert ex.fused_regions_run == 1
    os.environ["AB_NO_ROWFUSE"] = "1"
    try:
        plain = [np.asarray(o) for o in rt(prog, host_outputs=False)(*ins)]
    finally:
        del os.environ["AB_NO_ROWFUSE"]
    for k, (a, b) in enumerate(zip(fused, plain)):
        assert_matches(a, b, blas=True, what=f"full-size logreg out {k}: fused vs node-by-node")
    half = [DeviceArray.from_torch(X[: N // 2]), DeviceArray.from_torch(y[: N // 2]), ins[2], ins[3]]
    X2 = torch.cat([X[: N // 2], X[: N // 2]])
    y2 = torch.cat([y[: N // 2], y[: N // 2]])
    dup = [DeviceArray.from_torch(X2), DeviceArray.from_torch(y2), ins[2], ins[3]]
    a = [np.asarray(o) for o in ex(*half)]
    b = [np.asarray(o) for o in ex(*dup)]
    for k, (u, v) in enumerate(zip(a, b)):
        assert_matches(v, u, blas=True, what=f"duplicated batch out {k}")


def test_output_combiner_device_path_single_rank(rt):
    """shard.OutputCombiner on the device (NCCL, world_size 1): pack -> all_gather ->
    weighted sum by the backend's own Elemwise/CAReduce kernels == identity."""
    import os
    import socket

    import torch.distributed as dist

    from aesara_b200.runtime.device import DeviceArray
    from aesara_b200.shard import OutputCombiner

    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("nccl", rank=0, world_size=1)
    try:
        rng = np.random.default_rng(0)
        outs = [rng.standard_normal(()).astype("float32"), rng.standard_normal((7, 5)).astype("float32"),
                rng.standard_normal(33).astype("float32")]
        comb = OutputCombiner(1, mode="mean")
        got = comb([DeviceArray.from_numpy(o) for o in outs])
        for g, w in zip(got, outs):
            np.testing.assert_allclose(g.to_numpy(), w, rtol=1e-6)
        # the large-payload plan: weight the local buffer, one in-place all_reduce
        comb2 = OutputCombiner(1, mode="mean", plan="allreduce")
        got2 = comb2([DeviceArray.from_numpy(o) for o in outs])
        for g, w in zip(got2, outs):
            np.testing.assert_allclose(g.to_numpy(), w, rtol=1e-6)
    finally:
        dist.destroy_process_group()


def test_mlp_medium_size_fp32_faithful_vs_oracle(rt):
    """cfg3 graph at B=4096, H=512 (tensor-core path engaged for every GEMM).  With 4096-term
    fp32 dot products the fp32 CPU path (oracle = what the reference's sgemm path computes)
    is itself only ~1e-5..1e-4 accurate on cancellation-prone gradient entries (SURVEY H3),
    so the bar is stated against a float64 ground truth: the fp32-faithful (3xTF32) device
    result is at least as close to it as the fp32 CPU path (within 2x), and both agree
    norm-wise to 5e-5; the bf16 compute policy stays within its stated 2e-2."""
    from oracle.program_np import run_program

    prog, _, _ = load_case("cfg3_mlp")
    rng = np.random.default_rng(42)
    B, H = 4096, 512
    ins = [rng.standard_normal((B, H)).astype("float32"), rng.standard_normal((B, H)).astype("float32"),
           (rng.standard_normal((H, H)) / np.sqrt(H)).astype("float32"), np.zeros(H, "float32"),
           (rng.standard_normal((H, H)) / np.sqrt(H)).astype("float32"), np.zeros(H, "float32")]
    cpu32 = run_program(prog, [np.array(a) for a in ins])
    X, Y, W1, b1, W2, b2 = [a.astype(np.float64) for a in ins]
    h = np.tanh(X @ W1 + b1)
    diff = h @ W2 + b2 - Y
    dout = 2.0 * diff / diff.size
    dpre = (dout @ W2.T) * (1.0 - h * h)
    truth = [np.mean(diff ** 2), X.T @ dpre, dpre.sum(0), h.T @ dout, dout.sum(0)]

    def nerr(a, t):
        return float(np.max(np.abs(np.asarray(a, np.float64) - t)) / max(np.max(np.abs(t)), 1e-300))

    got = rt(prog, precision=0)(*ins)
    for k, (g, c, t) in enumerate(zip(got, cpu32, truth)):
        e_dev, e_cpu = nerr(g, t), nerr(c, t)
        assert e_dev <= max(2.0 * e_cpu, 1e-5), f"out {k}: device {e_dev:.2e} vs fp32 CPU {e_cpu:.2e}"
        assert_matches(g, c, blas=True, rtol=5e-5, what=f"fp32-faithful out {k} vs fp32 CPU path")
    got_bf16 = rt(prog, precision=2)(*ins)
    for k, (g, t) in enumerate(zip(got_bf16, truth)):
        assert nerr(g, t) < 2e-2, f"bf16 policy out {k}"


def lib_launches():
    from aesara_b200.runtime import lib

    return lib.load().ab_launch_count()


def _fused_vs_plain(fused, plain, what, exact_sums=True):
    """cfg3 outputs [loss, dW1, db1, dW2, db2]: the products see identical operands (the
    epilogue evaluates the same scalar expressions on the same fp32 values; a bf16 plane written
    by the epilogue equals the separate pack), so the weight gradients are BIT-identical.  Loss
    and bias gradients, fp32-faithful policy: float64(-equivalent) sums of identical float32
    terms in a different (still deterministic) order: equal to the last float32 bit or one ulp.
    tf32 / bf16 policies (``exact_sums=False``): the epilogue adds 8 / 32 terms at a time as a
    float32 tree before the float64 stage -- a few 2^-24 of the sum of magnitudes, checked
    norm-wise at 2e-6 (the terms themselves carry 2^-8 from the bf16 operands)."""
    for k, (a, b) in enumerate(zip(fused, plain)):
        if np.ndim(a) == 2:
            np.testing.assert_array_equal(a, b, err_msg=f"{what} output {k}: fused vs node-by-node")
        elif exact_sums:
            np.testing.assert_allclose(a, b, rtol=3e-7, atol=0, err_msg=f"{what} output {k}: fused vs node-by-node")
        else:
            np.testing.assert_allclose(a, b, rtol=0, atol=2e-6 * float(np.max(np.abs(b))),
                                       err_msg=f"{what} output {k}: fused vs node-by-node")


@pytest.mark.parametrize("precision", [0, 2])
def test_mlp_gemm_epilogue_fusion_matches_node_by_node(rt, precision, monkeypatch):
    """cfg3 graph, B=1024, H=512: the three Gemm/Dot22 -> Elemwise pairs run as fused
    tcgen05 kernels (runtime/gemmfuse.py) and give the node-by-node result (the epilogue
    evaluates the same scalar expression on the same fp32 values; the bf16 shadow plane it
    writes equals the separate pack, so even the bf16 policy is bit-identical)."""
    import os

    prog, _, _ = load_case("cfg3_mlp")
    if precision == 0:
        # off by default under the fp32-faithful policy (slower than node by node there)
        assert not any(type(f).__name__ == "GemmEpilogueFusion" for f in rt(prog, precision=0)._fusions)
        monkeypatch.setenv("AB_GEMM_FUSE_FP32", "1")
    rng = np.random.default_rng(21)
    B, H = 1024, 512
    ins = [rng.standard_normal((B, H)).astype("float32"), rng.standard_normal((B, H)).astype("float32"),
           (rng.standard_normal((H, H)) / np.sqrt(H)).astype("float32"), (rng.standard_normal(H) * 0.1).astype("float32"),
           (rng.standard_normal((H, H)) / np.sqrt(H)).astype("float32"), (rng.standard_normal(H) * 0.1).astype("float32")]
    ex = rt(prog, precision=precision)
    n_gemm_fusions = sum(type(f).__name__ == "GemmEpilogueFusion" for f in ex._fusions)
    assert n_gemm_fusions == 3 and len(ex._fusions) == 3  # Sqr -> Sum (the loss) is inside region 2
    before = lib_launches()
    fused = ex(*ins)
    n_fused_launches = lib_launches() - before
    assert ex.fused_regions_run == 3
    assert not any(f.broken for f in ex._fusions)
    # under the bf16 policy dout and dpre exist as bf16 operand planes only
    assert sum(f.f32_skipped for f in ex._fusions) == (2 if precision == 2 else 0)
    os.environ["AB_NO_GEMM_FUSE"] = os.environ["AB_NO_RED_FUSE"] = "1"
    try:
        ex_plain = rt(prog, precision=precision)
    finally:
        del os.environ["AB_NO_GEMM_FUSE"], os.environ["AB_NO_RED_FUSE"]
    assert not ex_plain._fusions
    before = lib_launches()
    plain = ex_plain(*ins)
    assert n_fused_launches < lib_launches() - before
    _fused_vs_plain(fused, plain, f"precision {precision}", exact_sums=precision == 0)
    # the round-1 regions (one Elemwise per product) still give the same bits
    os.environ["AB_GEMM_FUSE_SINGLE"] = "1"
    try:
        single = rt(prog, precision=precision)(*ins)
    finally:
        del os.environ["AB_GEMM_FUSE_SINGLE"]
    _fused_vs_plain(single, plain, f"precision {precision}, single-node regions", exact_sums=precision == 0)


@pytest.mark.parametrize("precision", [0, 2])
@pytest.mark.parametrize("B", [1000, 777, 4099])
def test_mlp_gemm_epilogue_fusion_ragged_batch(rt, precision, B, monkeypatch):
    """cfg3 graph with a batch that is not a multiple of the 32-row chunks / 128-row tiles of the
    fused epilogue (last warp partly outside, last tile partly outside, odd K of the weight
    gradients; B=4099 takes the 2-CTA kernel): staged row stores, column sums over partly
    empty 32-row blocks and the transposed bf16 plane's ragged rows give the node-by-node
    result."""
    import os

    prog, _, _ = load_case("cfg3_mlp")
    if precision == 0:
        monkeypatch.setenv("AB_GEMM_FUSE_FP32", "1")
    rng = np.random.default_rng(B)
    H = 256
    ins = [rng.standard_normal((B, H)).astype("float32"), rng.standard_normal((B, H)).astype("float32"),
           (rng.standard_normal((H, H)) / np.sqrt(H)).astype("float32"), (rng.standard_normal(H) * 0.1).astype("float32"),
           (rng.standard_normal((H, H)) / np.sqrt(H)).astype("float32"), (rng.standard_normal(H) * 0.1).astype("float32")]
    ex = rt(prog, precision=precision)
    fused = ex(*ins)
    assert ex.fused_regions_run == 3 and not any(f.broken for f in ex._fusions)
    os.environ["AB_NO_GEMM_FUSE"] = os.environ["AB_NO_RED_FUSE"] = "1"
    try:
        plain = rt(prog, precision=precision)(*ins)
    finally:
        del os.environ["AB_NO_GEMM_FUSE"], os.environ["AB_NO_RED_FUSE"]
    _fused_vs_plain(fused, plain, f"precision {precision}, B={B}", exact_sums=precision == 0)


@pytest.mark.parametrize("T,B,H", [(12, 256, 128), (5, 384, 192), (4, 200, 64)])
def test_lstm_medium_size_vs_oracle_and_graph_replay(rt, T, B, H):
    """cfg4 graph at medium sizes (a full 2-CTA tile, a ragged second 2-CTA tile, and a
    batch below 256 that takes the 1-CTA kernel): eager device loop == oracle; the
    CUDA-graph replay of the whole evaluation returns bit-identical results."""
    from oracle.program_np import run_program
    from aesara_b200.runtime.device import DeviceArray
    from aesara_b200.runtime.graph import GraphReplay

    prog, _, _ = load_case("cfg4_lstm")
    rng = np.random.default_rng(3)
    ins = [rng.standard_normal((T, B, 4 * H)).astype("float32"), np.zeros((B, H), "float32"),
           np.zeros((B, H), "float32"), (rng.standard_normal((H, 4 * H)) / np.sqrt(H)).astype("float32")]
    want = run_program(prog, [np.array(a) for a in ins])
    ex = rt(prog, host_outputs=False)
    dins = [DeviceArray.from_numpy(a) for a in ins]
    eager = [o.to_numpy() for o in ex(*dins)]
    for k, (g, w) in enumerate(zip(eager, want)):
        assert_matches(g, w, blas=True, rtol=1e-5, what=f"lstm out {k}")
    scan_idx = [i for i, n in enumerate(prog.nodes) if n.op == "Scan"][0]
    assert ex._state[scan_idx]["runner"].used_fast_path  # the persistent LSTM kernel ran
    # the general device loop (per-step launches) gives the same answer
    import os

    os.environ["AB_SCAN_NO_FAST"] = "1"
    try:
        ex_gen = rt(prog, host_outputs=False)
        general = [o.to_numpy() for o in ex_gen(*dins)]
    finally:
        del os.environ["AB_SCAN_NO_FAST"]
    assert not ex_gen._state[scan_idx]["runner"].used_fast_path
    for k, (g, e) in enumerate(zip(general, eager)):
        assert_matches(g, e, blas=True, rtol=1e-5, what=f"general loop vs fast path out {k}")
    replay = GraphReplay(ex)
    for _ in range(3):
        outs = replay(*dins)
    assert replay.replays >= 2
    for g, e in zip(outs, eager):
        np.testing.assert_array_equal(g.to_numpy(), e)


@pytest.mark.parametrize("N,D,fused", [(1000, 48, True), (4099, 512, True), (257, 36, True), (3000, 1024, True),
                                       (333, 128, True), (500, 1100, False), (500, 30, False)])
def test_logreg_row_region_fusion(rt, N, D, fused):
    """cfg5 graph: the Gemv -> Elemwise -> Sum / Gemv(X.T) region runs as one pass over X
    (runtime/rowfuse.py) and matches both the node-by-node device execution and the
    oracle; operands the fused kernel does not take (D > 1024, D % 4 != 0) fall back to the
    node-by-node path."""
    import os

    from oracle.program_np import run_program

    prog, _, _ = load_case("cfg5_logreg")
    rng = np.random.default_rng(N + D)
    ins = [rng.standard_normal((N, D)).astype("float32"), (rng.random(N) < 0.5).astype("float32"),
           (rng.standard_normal(D) * 0.05).astype("float32"), np.float32(0.25)]
    want = run_program(prog, [np.array(a) for a in ins])
    ex = rt(prog)
    assert len(ex._fusions) == 1
    got = ex(*ins)
    assert ex.fused_regions_run == (1 if fused else 0)
    os.environ["AB_NO_ROWFUSE"] = "1"
    try:
        ex_plain = rt(prog)
    finally:
        del os.environ["AB_NO_ROWFUSE"]
    assert not ex_plain._fusions
    plain = ex_plain(*ins)
    for k, (g, p, w) in enumerate(zip(got, plain, want)):
        assert_matches(g, w, blas=True, what=f"fused logreg out {k} vs oracle")
        assert_matches(g, p, blas=True, what=f"fused logreg out {k} vs node-by-node")


def test_logreg_row_region_fusion_strided_and_device_scalars(rt):
    """X as a column slice of a wider matrix (row stride > D), y as a strided view, the
    bias as a 1-element device array."""
    from aesara_b200.runtime.device import DeviceArray
    from oracle.program_np import run_program

    prog, _, _ = load_case("cfg5_logreg")
    rng = np.random.default_rng(7)
    N, D = 2000, 256
    big = rng.standard_normal((N, D + 64)).astype("float32")
    y2 = (rng.random(2 * N) < 0.5).astype("float32")
    w = (rng.standard_normal(D) * 0.05).astype("float32")
    b = np.float32(-0.5)
    want = run_program(prog, [np.ascontiguousarray(big[:, 32 : 32 + D]), y2[::2].copy(), w, b])
    Xd = DeviceArray.from_numpy(big).index((slice(None), slice(32, 32 + D)))
    yd = DeviceArray.from_numpy(y2).index((slice(None, None, 2),))
    ex = rt(prog)
    got = ex(Xd, yd, DeviceArray.from_numpy(w), DeviceArray.from_numpy(np.asarray(b)))
    assert ex.fused_regions_run == 1
    for k, (g, wv) in enumerate(zip(got, want)):
        assert_matches(g, wv, blas=True, what=f"strided fused logreg out {k}")


def test_mlp_full_size_fused_equals_node_by_node(rt):
    """BASELINE cfg3 size (B=65536, H=4096; no CPU truth at this size): the fused
    execution (3 GEMM epilogues + Sqr->Sum) is bit-identical to node-by-node execution
    under the bf16 policy, and row-permuting the batch leaves loss and gradients unchanged
    up to summation order."""
    import os

    import torch

    from aesara_b200.runtime.device import DeviceArray

    prog, _, _ = load_case("cfg3_mlp")
    B, H = 65536, 4096
    g = torch.Generator(device="cuda").manual_seed(5)
    X = torch.randn(B, H, device="cuda", generator=g)
    Y = torch.randn(B, H, device="cuda", generator=g)
    W1 = torch.randn(H, H, device="cuda", generator=g) / H ** 0.5
    W2 = torch.randn(H, H, device="cuda", generator=g) / H ** 0.5
    b1 = torch.randn(H, device="cuda", generator=g) * 0.1
    b2 = torch.randn(H, device="cuda", generator=g) * 0.1

    def run(ex, Xt, Yt):
        outs = ex(*[DeviceArray.from_torch(t) for t in (Xt, Yt, W1, b1, W2, b2)])
        return [np.asarray(o) for o in outs]

    ex = rt(prog, precision=2, host_outputs=False)
    fused = run(ex, X, Y)
    assert ex.fused_regions_run == 3
    os.environ["AB_NO_GEMM_FUSE"] = os.environ["AB_NO_RED_FUSE"] = "1"
    try:
        plain = run(rt(prog, precision=2, host_outputs=False), X, Y)
    finally:
        del os.environ["AB_NO_GEMM_FUSE"], os.environ["AB_NO_RED_FUSE"]
    _fused_vs_plain(fused, plain, "full-size MLP", exact_sums=False)
    perm = torch.randperm(B, device="cuda", generator=g)
    shuffled = run(ex, X[perm].contiguous(), Y[perm].contiguous())
    for k, (a, b) in enumerate(zip(shuffled, fused)):
        assert_matches(a, b, blas=True, rtol=2e-5, what=f"full-size MLP output {k} under a batch permutation")


def test_lstm_full_size_fast_path_vs_general_loop(rt):
    """BASELINE cfg4 size (T=128, B=8192, H=1024): the persistent kernel and the general
    per-step device loop agree on h_T, c_T (both fp32-faithful; different summation order)."""
    import os

    import torch

    from aesara_b200.runtime.device import DeviceArray

    prog, _, _ = load_case("cfg4_lstm")
    T, B, H = 128, 8192, 1024
    g = torch.Generator(device="cuda").manual_seed(9)
    x = torch.randn(T, B, 4 * H, device="cuda", generator=g)
    U = torch.randn(H, 4 * H, device="cuda", generator=g) / H ** 0.5
    z = torch.zeros(B, H, device="cuda")
    ins = [DeviceArray.from_torch(t) for t in (x, z, z.clone(), U)]
    ex = rt(prog, host_outputs=False)
    fast = [np.asarray(o) for o in ex(*ins)]
    scan_idx = [i for i, n in enumerate(prog.nodes) if n.op == "Scan"][0]
    assert ex._state[scan_idx]["runner"].used_fast_path
    os.environ["AB_SCAN_NO_FAST"] = "1"
    try:
        general = [np.asarray(o) for o in rt(prog, host_outputs=False)(*ins)]
    finally:
        del os.environ["AB_SCAN_NO_FAST"]
    for k, (a, b) in enumerate(zip(fast, general)):
        assert np.isfinite(a).all()
        assert_matches(a, b, blas=True, rtol=2e-5, what=f"full-size LSTM output {k}: persistent kernel vs general loop")


def test_gemm_full_size_tile_independence(rt):
    """BASELINE-size GEMM property (no CPU truth at this size): rows of a
    [16384, 4096] x [4096, 4096] product equal the product of the row subset, for
    both the 2-CTA and the ragged-tail tile paths; bf16 result is within 2e-2 of the
    fp32-faithful one."""
    import torch

    from aesara_b200.runtime import kernels as K
    from aesara_b200.runtime.device import DeviceArray

    g = torch.Generator(device="cuda").manual_seed(5)
    M, N, Kd = 16384, 4096, 4096
    a = torch.randn(M, Kd, device="cuda", generator=g)
    b = torch.randn(Kd, N, device="cuda", generator=g) / 64.0
    A, Bm = DeviceArray.from_torch(a), DeviceArray.from_torch(b)
    full = DeviceArray.empty((M, N), "float32")
    K.gemm(full, 1.0, A, Bm, 0.0, precision=0)
    sub_rows = slice(5000, 5000 + 777)
    sub = DeviceArray.empty((777, N), "float32")
    K.gemm(sub, 1.0, A.index((sub_rows,)), Bm, 0.0, precision=0)
    f = full.owner.view(torch.float32).view(M, N)[sub_rows]
    s = sub.owner.view(torch.float32)[: 777 * N].view(777, N)
    assert torch.equal(f, s)  # identical arithmetic per output element, whatever the tiling
    lo = DeviceArray.empty((M, N), "float32")
    K.gemm(lo, 1.0, A, Bm, 0.0, precision=2)
    l = lo.owner.view(torch.float32).view(M, N)
    rel = ((l - full.owner.view(torch.float32).view(M, N)).abs().max() / f.abs().max()).item()
    assert rel < 2e-2


@pytest.mark.parametrize("name,gates", [("scan_rnn_tanh_cell", 1), ("scan_gated_unit_cell", 3)])
def test_scan_cell_family_runs_as_one_persistent_kernel(rt, name, gates):
    """Scan inner graphs "one Gemm(x_t, 1, h, U, 1) + Elemwise on its column slices" other than
    the LSTM get a generated cell in the persistent kernel (runtime/scan_cell.py): reference
    outputs reproduced, the general per-step loop agrees, and far fewer launches."""
    import os

    from aesara_b200.runtime import lib
    from oracle.program_np import run_program

    prog, ins, want = load_case(name)
    ex = rt(prog)
    before = lib.load().ab_launch_count()
    got = ex(*[np.array(a) for a in ins])
    fast_launches = lib.load().ab_launch_count() - before
    scan = [st["runner"] for st in ex._state if "runner" in st][0]
    assert scan.used_fast_path and scan.fast_path_kind == "jit"
    for k, (g, w) in enumerate(zip(got, want)):
        assert_matches(g, w, blas=True, what=f"{name} output {k} vs the reference")
    os.environ["AB_SCAN_NO_FAST"] = "1"
    try:
        ex_gen = rt(prog)
        before = lib.load().ab_launch_count()
        general = ex_gen(*[np.array(a) for a in ins])
        slow_launches = lib.load().ab_launch_count() - before
    finally:
        del os.environ["AB_SCAN_NO_FAST"]
    assert not [st["runner"] for st in ex_gen._state if "runner" in st][0].used_fast_path
    for k, (g, e) in enumerate(zip(got, general)):
        assert_matches(g, e, blas=True, what=f"{name} output {k}: persistent kernel vs general loop")
    assert fast_launches < slow_launches
    # larger, ragged shapes against the oracle (second 2-CTA tile partly empty; 1-CTA kernel)
    rng = np.random.default_rng(gates)
    for T, B, H in ((9, 384, 128), (4, 200, 64)):
        vals = [rng.standard_normal((T, B, gates * H)).astype("float32"),
                (rng.standard_normal((B, H)) * 0.1).astype("float32"),
                (rng.standard_normal((H, gates * H)) / np.sqrt(H)).astype("float32")]
        o = run_program(prog, [np.array(a) for a in vals])
        g = rt(prog)(*vals)
        for k, (a, b) in enumerate(zip(g, o)):
            assert_matches(a, b, blas=True, what=f"{name} at T={T}, B={B}, H={H} output {k} vs oracle")


def test_lstm_generated_cell_equals_the_ahead_of_time_cell(rt):
    """The LSTM through the generated-cell path (AB_SCAN_JIT) is BIT-identical to the
    ahead-of-time kernel: same skeleton, the cell emitted from the inner graph's expressions."""
    import os

    prog, _, _ = load_case("cfg4_lstm")
    rng = np.random.default_rng(8)
    T, B, H = 7, 512, 128
    ins = [rng.standard_normal((T, B, 4 * H)).astype("float32"), np.zeros((B, H), "float32"),
           np.zeros((B, H), "float32"), (rng.standard_normal((H, 4 * H)) / np.sqrt(H)).astype("float32")]
    ex = rt(prog)
    aot = ex(*ins)
    assert [st["runner"] for st in ex._state if "runner" in st][0].fast_path_kind == "lstm"
    os.environ["AB_SCAN_JIT"] = "1"
    try:
        ex2 = rt(prog)
        jit = ex2(*ins)
    finally:
        del os.environ["AB_SCAN_JIT"]
    assert [st["runner"] for st in ex2._state if "runner" in st][0].fast_path_kind == "jit"
    for a, b in zip(aot, jit):
        np.testing.assert_array_equal(a, b)


@pytest.mark.parametrize("shape", [(1000, 777), (64, 4099), (33, 17), (5, 300, 130)])
def test_elemwise_transposed_operands_take_the_tiled_kernel(rt, shape):
    """An expression over a matrix and DimShuffle{1,0} views of others (`a.T * b + c.T > 0`):
    the tiled kernel (csrc/ab_elemwise.cuh ab_ew_tile: row-contiguous inputs turned through
    shared memory) gives the bits of the index-arithmetic kernel (AB_EW_NO_TILE), on float32,
    float64, int and bool operands, ragged tile edges and a batched (3-D) case."""
    import os

    from aesara_b200.runtime import kernels as K
    from aesara_b200.runtime.device import DeviceArray

    rng = np.random.default_rng(sum(shape))
    tshape = shape[:-2] + (shape[-1], shape[-2])
    perm = list(range(len(shape) - 2)) + [len(shape) - 1, len(shape) - 2]
    for dts in (("float32", "float32", "float32"), ("float64", "float32", "int32"), ("int16", "bool", "int64")):
        a = (rng.standard_normal(tshape) * 3).astype(dts[0])
        b = (rng.standard_normal(shape) * 3).astype(dts[1])
        c = (rng.standard_normal(tshape) * 3).astype(dts[2])
        out_dt = np.result_type(*dts).name if "bool" not in dts else "int64"
        expr = {"inputs": list(dts), "out_dtypes": [out_dt, "bool"], "outputs": ["t2", "t3"], "name": "tiled_probe",
                "stmts": [{"op": "cast", "args": ["i0"], "dtype": out_dt, "in_dtypes": [dts[0]]},
                          {"op": "cast", "args": ["i1"], "dtype": out_dt, "in_dtypes": [dts[1]]},
                          {"op": "add", "args": ["t0", "t1"], "dtype": out_dt, "in_dtypes": [out_dt, out_dt]},
                          {"op": "gt", "args": ["i2", {"const": 0, "dtype": dts[2]}], "dtype": "bool", "in_dtypes": [dts[2], dts[2]]}]}
        kern = K.ElemwiseKernel.get(expr)
        ins = [DeviceArray.from_numpy(a).dimshuffle(perm), DeviceArray.from_numpy(b),
               DeviceArray.from_numpy(c).dimshuffle(perm)]
        res = []
        for no_tile in (False, True):
            if no_tile:
                os.environ["AB_EW_NO_TILE"] = "1"
            try:
                outs = [DeviceArray.empty(shape, out_dt), DeviceArray.empty(shape, "bool")]
                kern.launch(shape, ins, outs)
                res.append([o.to_numpy() for o in outs])
            finally:
                os.environ.pop("AB_EW_NO_TILE", None)
        at_, ct_ = np.transpose(a, perm), np.transpose(c, perm)
        want0 = at_.astype(out_dt) + b.astype(out_dt)
        np.testing.assert_array_equal(res[0][0], res[1][0])
        np.testing.assert_array_equal(res[0][1], res[1][1])
        np.testing.assert_array_equal(res[0][0], want0)
        np.testing.assert_array_equal(res[0][1], ct_ > 0)


def test_zz_launch_counts_are_recorded():
    """Writes the per-fixture launch counts next to the run (gpurun_out/) for the record."""
    import json
    import os

    if not _LAUNCHES:
        pytest.skip("parity matrix did not run in this session")
    d = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out")
    os.makedirs(d, exist_ok=True)
    with open(os.path.join(d, "golden_launch_counts.json"), "w") as f:
        json.dump(_LAUNCHES, f, indent=1, sort_keys=True)
    assert all(v > 0 for k, v in _LAUNCHES.items() if k not in PURE_METADATA)
