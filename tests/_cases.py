"""Shared helpers: load golden fixtures, compare with the tolerances stated here.

Tolerance policy (BASELINE north star; the reference's own test tolerances are
aesara/tensor/math.py:85-96: f32 rtol=atol=1e-5, f64 rtol=1e-5/atol=1e-8):
  * integer / bool outputs: bit-exact;
  * float outputs of element-wise / reduction graphs: rtol 1e-5 (+ atol 1e-6 f32, 1e-10 f64);
  * float outputs downstream of a dot product: rtol 1e-5 relative to the
    largest magnitude of the output (norm-wise), because the summation order
    differs between BLAS, NumPy and the device kernels.
"""
import glob
import os

import numpy as np

from aesara_b200.ir import Program

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
BLAS_OPS = {"Dot22", "Dot22Scalar", "Gemm", "Gemv", "Ger", "Dot", "Scan"}

# The five BASELINE graphs at the sizes tests/test_gpu_function.py calls them with: committed
# program, graph builder in aesara_b200.graphs, seeded inputs.  c_linker_baseline.npz holds the
# reference C-linker's outputs for these calls (tests/golden/make_golden.py --c-linker), so that
# the comparison also runs where the Aesara front-end is not installed.
BASELINE_CALLS = {
    "cfg1": ("cfg1_readme", "cfg1_readme", lambda G: G.cfg1_inputs(300)),
    "cfg2": ("cfg2_fused", "cfg2_fused_elemwise", lambda G: G.cfg2_inputs(100003, yscale=12.0)),
    "cfg3": ("cfg3_mlp", "cfg3_mlp", lambda G: G.cfg3_inputs(384, 256)),
    "cfg4": ("cfg4_lstm", "cfg4_lstm_scan", lambda G: G.cfg4_inputs(6, 256, 64)),
    "cfg5": ("cfg5_logreg", "cfg5_logreg", lambda G: G.cfg5_inputs(5000, 128)),
}
C_LINKER_GOLDEN = os.path.join(GOLDEN, "c_linker_baseline.npz")
C_LINKER_SAMPLE = 8192  # outputs larger than this are stored at a fixed, seeded sample of positions


def sample_positions(size):
    """Flat positions stored of an output with ``size`` elements (None: all of them)."""
    if size <= C_LINKER_SAMPLE:
        return None
    return np.sort(np.random.default_rng(size).choice(size, C_LINKER_SAMPLE, replace=False))


def assert_matches_c_linker(name, got):
    """``got`` (the outputs of BASELINE_CALLS[name]) against the stored C-linker outputs, at the
    stored positions; ``cfg2`` is the only graph without a dot product."""
    z = np.load(C_LINKER_GOLDEN)
    n = sum(1 for f in z.files if f.startswith(f"{name}_out_"))
    assert len(got) == n, f"{name}: {len(got)} outputs, {n} stored"
    for k, g in enumerate(got):
        g = np.asarray(g)
        if f"{name}_pos_{k}" in z.files:
            g = g.reshape(-1)[z[f"{name}_pos_{k}"]]
        assert_matches(g, z[f"{name}_out_{k}"], blas=name != "cfg2", what=f"{name} output {k} vs the C-linker")


def shardplan_mixed_graph(at):
    """Inputs and outputs of the hand-built graph of tests/test_shardplan.py, on the front-end's
    ``aesara.tensor`` module ``at``; lowered (``FAST_COMPILE``) it is golden/programs/
    shardplan_mixed_outputs.json."""
    X, w = at.fmatrix("X"), at.fvector("w")
    z = at.tanh(X @ w)
    return [X, w], [(z ** 2).sum(), at.dot(X.T, z), z * 2, w * 3, (X ** 2).sum(axis=0) / X.shape[0]]


def case_names():
    return sorted(os.path.basename(p)[:-5] for p in glob.glob(os.path.join(GOLDEN, "*.json")))


def load_case(name):
    prog = Program.load(os.path.join(GOLDEN, name + ".json"))
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    ins = [z[f"in_{k}"] for k in range(len(prog.inputs))]
    outs = [z[f"out_{k}"] for k in range(len(prog.outputs))]
    return prog, ins, outs


def uses_blas(prog):
    return any(n.op in BLAS_OPS for n in prog.nodes)


def assert_matches(got, want, blas=False, rtol=1e-5, what=""):
    got = np.asarray(got)
    want = np.asarray(want)
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    assert got.dtype == want.dtype, f"{what}: dtype {got.dtype} != {want.dtype}"
    if want.dtype.kind in "biu":
        np.testing.assert_array_equal(got, want, err_msg=what)
        return
    if blas:
        scale = float(np.max(np.abs(want))) if want.size else 1.0
        atol = rtol * max(scale, 1e-30)
        np.testing.assert_allclose(got, want, rtol=rtol, atol=atol, err_msg=what)
    else:
        atol = 1e-6 if want.dtype == np.float32 else 1e-10
        np.testing.assert_allclose(got, want, rtol=rtol, atol=atol, equal_nan=True, err_msg=what)
