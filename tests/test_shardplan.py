"""CPU: the shardability analysis (aesara_b200/shardplan.py, SURVEY 8e's general rule).

For every fixture graph the analysis accepts, the claim it makes — "these inputs split along
this axis, and the outputs combine as sum / mean / concat" — is checked NUMERICALLY: the oracle
evaluates the program on three unequal row blocks, the results are combined exactly as the plan
says, and must equal the oracle's evaluation of the whole batch.  Graphs that are not batch maps
must be refused with ReplicasOnly."""
import os

import numpy as np
import pytest

from aesara_b200 import shardplan as S
from tests._cases import load_case


def _split(n, parts=(0.5, 0.2, 0.3)):
    cuts = [0]
    for p in parts[:-1]:
        cuts.append(cuts[-1] + max(1, int(round(n * p))))
    cuts.append(n)
    return list(zip(cuts[:-1], cuts[1:]))


def _check_numerically(prog, ins, plan, rtol=2e-5):
    from oracle.program_np import run_program

    axes = plan.sharded_inputs
    extents = {np.shape(a)[ax] for a, ax in zip(ins, axes) if ax is not None}
    if len(extents) != 1 or min(extents) < 3:
        pytest.skip("the fixture's sharded inputs do not share one row count (run-time broadcasting)")
    full = run_program(prog, [np.array(a) for a in ins])
    n = extents.pop()
    blocks = _split(n)
    shard_outs = []
    for s, e in blocks:
        local = []
        for a, ax in zip(ins, axes):
            if ax is None:
                local.append(np.array(a))
            else:
                sl = [slice(None)] * np.ndim(a)
                sl[ax] = slice(s, e)
                local.append(np.array(np.asarray(a)[tuple(sl)]))
        shard_outs.append(run_program(prog, local))
    rows = [e - s for s, e in blocks]
    for k, mode in enumerate(plan.outputs):
        parts = [np.asarray(o[k], np.float64) if np.asarray(o[k]).dtype.kind == "f" else np.asarray(o[k])
                 for o in shard_outs]
        if mode[0] == "sum":
            got = sum(parts)
        elif mode[0] == "mean":
            got = sum(p * (r / float(n)) for p, r in zip(parts, rows))
        elif mode[0] == "concat":
            got = np.concatenate(parts, axis=mode[1])
        else:
            got = parts[0]
        want = np.asarray(full[k])
        assert np.shape(got) == want.shape, (k, mode)
        scale = max(float(np.max(np.abs(want))) if want.size else 1.0, 1e-30)
        np.testing.assert_allclose(got, want, rtol=rtol, atol=rtol * scale, err_msg=f"output {k} combined as {mode}")


@pytest.mark.parametrize("name,expect_inputs,expect_modes", [
    ("cfg3_mlp", [0, 0, None, None, None, None], ["mean"] * 5),
    ("cfg5_logreg", [0, 0, None, None], ["mean"] * 3),
    ("cfg2_fused", [0, 0, 0], ["concat"]),
    ("cfg1_readme", [None, None, 0], ["concat"]),
    ("softmax_classifier", [0, 0, None], ["mean", "mean", "concat", "concat", "concat"]),
])
def test_inferred_plan_is_numerically_right(name, expect_inputs, expect_modes):
    prog, ins, _ = load_case(name)
    plan = S.infer_sharded_inputs(prog)
    assert plan.sharded_inputs == expect_inputs
    assert [m[0] for m in plan.outputs] == expect_modes
    _check_numerically(prog, ins, plan)


def test_scan_batch_axis():
    """cfg4: the sequence is [T, B, 4H] — the batch is axis 1; states [B, H] axis 0; U replicated."""
    prog, ins, _ = load_case("cfg4_lstm")
    plan = S.analyse(prog, [1, 0, 0, None])
    assert plan.outputs == [("concat", 0), ("concat", 0)]
    _check_numerically(prog, ins, plan)
    with pytest.raises(S.ReplicasOnly):
        S.analyse(prog, [0, 0, 0, None])      # time is not a batch axis
    with pytest.raises(S.ReplicasOnly):
        S.analyse(prog, [1, 0, 0, 0])         # U meets the batch on the K axis


def test_sum_outputs_and_mixed_graph():
    """A hand-built program, ``z = tanh(X @ w)`` -> ``[(z ** 2).sum(), X.T @ z, z * 2, w * 3,
    (X ** 2).sum(axis=0) / X.shape[0]]`` as the front-end lowers it (``FAST_COMPILE``, stored by
    tests/golden/make_golden.py --shardplan-program): unnormalised sums combine as `sum`, per-row
    values as `concat`, and parameters as `rep`.  Where a front-end is available, the program it
    lowers now is checked too."""
    from aesara_b200.compat import bootstrap
    from aesara_b200.ir import Program
    from tests._cases import GOLDEN, shardplan_mixed_graph

    prog = Program.load(os.path.join(GOLDEN, "programs", "shardplan_mixed_outputs.json"))
    plan = S.infer_sharded_inputs(prog)
    assert plan.sharded_inputs == [0, None]
    assert [m[0] for m in plan.outputs] == ["sum", "sum", "concat", "rep", "mean"]
    if bootstrap.available():
        aesara = bootstrap.load_aesara()
        import aesara.tensor as at

        from aesara_b200.lower import lower_fgraph

        f = aesara.function(*shardplan_mixed_graph(at), mode="FAST_COMPILE")
        live = lower_fgraph(f.maker.fgraph)
        assert [n.op for n in live.nodes] == [n.op for n in prog.nodes]
        live_plan = S.infer_sharded_inputs(live)
        assert live_plan.sharded_inputs == plan.sharded_inputs and live_plan.outputs == plan.outputs
    rng = np.random.default_rng(0)
    _check_numerically(prog, [rng.standard_normal((50, 7)).astype("float32"),
                              rng.standard_normal(7).astype("float32")], plan)


def _shardable_fixtures():
    from tests._cases import case_names

    return case_names()


@pytest.mark.parametrize("name", _shardable_fixtures())
def test_every_plan_the_analysis_accepts_is_numerically_right(name):
    """The whole fixture table: whatever the analysis accepts must combine to the unsharded
    result (the label algebra is validated by arithmetic, not by inspection)."""
    prog, ins, _ = load_case(name)
    try:
        plan = S.infer_sharded_inputs(prog)
    except S.ReplicasOnly:
        pytest.skip("replicas only")
    _check_numerically(prog, ins, plan)


@pytest.mark.parametrize("name", ["careduce_big_1d", "views_negative_steps", "cumsum_cumprod", "join_split_reshape",
                                  "reshape_flatten_noncontig", "indexing_embedding"])
def test_graphs_that_are_not_batch_maps_are_refused(name):
    prog, _, _ = load_case(name)
    with pytest.raises(S.ReplicasOnly, match="replicas only"):
        S.infer_sharded_inputs(prog)


def test_label_algebra_of_means():
    """x.shape[0] of a sharded x is a local row count: dividing a batch sum by it gives a
    per-shard mean (weights n_r / N); dividing twice is refused as an output."""
    sc, rows, part = ("scal", 1), ("rows", 0, 0), ("part", 0)
    node = type("N", (), {"label": "t", "op": "t"})()
    assert S._div(part, sc, node) == ("part", 1)
    assert S._div(rows, sc, node) == ("rows", 0, 1)
    assert S._mul(("rows", 0, 1), sc, node) == rows
    assert S._matmul(("rows", 1, 0), ("rows", 0, 1), node) == ("part", 1)
    with pytest.raises(S.ReplicasOnly):
        S._add([part, S.REP], node)
    with pytest.raises(S.ReplicasOnly):
        S._matmul(("rows", 0, 0), ("rows", 0, 0), node)
