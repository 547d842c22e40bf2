"""Generate the golden fixtures under tests/golden/ with the REFERENCE itself.

Run in the build container only (it imports /root/reference through the
overlay in aesara_b200.compat):

    PYTHONPATH=. python tests/golden/make_golden.py

For every case it
  1. builds the symbolic graph with the reference front-end,
  2. lets the reference rewriter optimise it (``fast_run``) and compiles it with
     the reference C linker (``Mode("cvm")`` = g++-compiled thunks driven by the C VM),
  3. lowers the *same* optimised graph with ``aesara_b200.lower`` → ``<case>.json``,
  4. evaluates the reference function on seeded inputs → ``<case>.npz``
     (``in_<k>`` arrays in program-input order, ``out_<k>`` reference outputs).

The fixtures pin both the oracle (tests/test_oracle.py, CPU) and the CUDA path
(tests/test_gpu_parity.py, ``-m gpu``).  The reference publishes no golden
vectors of its own for this path (SURVEY.md §8c), so these are "outputs of the
reference itself run here".
"""

import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
warnings.simplefilter("ignore")

from oracle import ref as _ref  # noqa: E402

_ref.materialise()
_ref.activate()
from aesara_b200 import graphs as G  # noqa: E402
from aesara_b200.compat.bootstrap import load_aesara  # noqa: E402

aesara = load_aesara()
import aesara.tensor as at  # noqa: E402

RNG = np.random.default_rng(666)  # the reference's unittests__rseed (configdefaults.py:1197)
CASES = {}


def case(name):
    def deco(fn):
        CASES[name] = fn
        return fn

    return deco


def rnd(shape, dtype="float32", lo=-3.0, hi=3.0):
    dt = np.dtype(dtype)
    if dt.kind == "f":
        return (RNG.random(shape) * (hi - lo) + lo).astype(dt)
    if dt.kind == "b":
        return RNG.random(shape) < 0.5
    info = np.iinfo(dt)
    return RNG.integers(max(info.min, -50), min(info.max, 50), size=shape, endpoint=True).astype(dt)


# ---------------------------------------------------------------- BASELINE configs
@case("cfg1_readme")
def _():
    i, o = G.cfg1_readme()
    return i, o, G.cfg1_inputs(96, seed=1)


@case("cfg2_fused")
def _():
    i, o = G.cfg2_fused_elemwise()
    return i, o, G.cfg2_inputs(4099, seed=2)


@case("cfg2_fused_allbranches")
def _():
    i, o = G.cfg2_fused_elemwise()
    return i, o, G.cfg2_inputs(4096, seed=3, yscale=20.0)


@case("cfg3_mlp")
def _():
    i, o = G.cfg3_mlp()
    return i, o, G.cfg3_inputs(256, 128, seed=4)


@case("cfg4_lstm")
def _():
    i, o = G.cfg4_lstm_scan()
    return i, o, G.cfg4_inputs(6, 64, 32, seed=5)


@case("cfg5_logreg")
def _():
    i, o = G.cfg5_logreg()
    return i, o, G.cfg5_inputs(1000, 48, seed=6)


# ---------------------------------------------------------------- Elemwise tables
# shapes follow tests/tensor/test_elemwise.py:214-229 (TestBroadcast)
@case("ew_broadcast_f64")
def _():
    a, b = at.dmatrix("a"), at.dmatrix("b")
    c, d = at.dtensor4("c"), at.dtensor4("d")
    outs = [a + b, a * b - a, c / (d * d + 1.0), at.exp(a) + at.sqrt(abs(b))]
    return [a, b, c, d], outs, [rnd((3, 5), "float64"), rnd((1, 5), "float64"),
                                rnd((2, 3, 4, 5), "float64"), rnd((1, 3, 1, 5), "float64")]


@case("ew_outer_broadcast")
def _():
    a, b = at.fmatrix("a"), at.fmatrix("b")
    return [a, b], [a + b, at.maximum(a, b) * 2], [rnd((1, 7)), rnd((5, 1))]


@case("ew_transposed_views")
def _():
    a, b = at.fmatrix("a"), at.fmatrix("b")
    t = at.tensor3("t", dtype="float32")
    outs = [a.T * b + 1, at.tanh(t.dimshuffle(2, 0, 1)) - t.dimshuffle(2, 0, 1) ** 2,
            (a.T + b)[::-1, ::2]]
    return [a, b, t], outs, [rnd((6, 4)), rnd((4, 6)), rnd((3, 4, 5))]


@case("ew_int_arith")
def _():
    x, y = at.ivector("x"), at.ivector("y")
    b8 = at.bvector("b8")
    outs = [x + y, x * y - x, x // y, x % y, abs(x), -x, at.sgn(x), x & y, x | y, x ^ y, ~x,
            at.maximum(x, y), at.minimum(x, y), b8 + b8, b8 * b8, at.cast(x, "int8"),
            at.cast(x * 1000, "int16"), x / y, at.switch(x > y, x, y), at.clip(x, -5, 5)]
    xv = rnd(257, "int32")
    yv = rnd(257, "int32")
    yv[yv == 0] = 7
    return [x, y, b8], outs, [xv, yv, rnd(257, "int8")]


@case("ew_uint_bool")
def _():
    u, v = at.vector("u", dtype="uint8"), at.vector("v", dtype="uint16")
    p, q = at.vector("p", dtype="bool"), at.vector("q", dtype="bool")
    outs = [u + u, u * u, v - v // 3, u // 3, u % 7, p & q, p | q, p ^ q, ~p, at.eq(u, 3),
            at.neq(v, u), at.lt(u, v), at.cast(p, "float32") + 1, at.switch(p, u, 9),
            at.cast(v, "uint8"), at.cast(u, "int64") - 200]
    return [u, v, p, q], outs, [rnd(130, "uint8"), rnd(130, "uint16"), rnd(130, "bool"), rnd(130, "bool")]


@case("ew_int64_mixed")
def _():
    x, y = at.lvector("x"), at.wvector("y")
    f = at.fvector("f")
    outs = [x * y, x // (abs(y) + 1), x % (abs(y) + 1), x + f, at.cast(f * 10, "int64") + x,
            at.floor(f), at.ceil(f), at.round(f), at.trunc(f), at.cast(f, "int32"),
            at.int_div(f, at.cast(abs(y) + 1, "float32")), at.mod(f, 1.5)]
    return [x, y, f], outs, [rnd(100, "int64"), rnd(100, "int16"), rnd(100, "float32", -9.5, 9.5)]


@case("ew_math_f32")
def _():
    x = at.fvector("x")
    px = abs(x) + 0.1
    outs = [at.exp(x), at.log(px), at.log1p(px), at.expm1(x), at.sqrt(px), at.sin(x), at.cos(x),
            at.tan(x * 0.4), at.tanh(x), at.sinh(x), at.cosh(x), at.arctan(x), at.arcsinh(x),
            at.sigmoid(x), at.softplus(x * 15), at.erf(x), at.erfc(x), at.log2(px), at.log10(px),
            at.exp2(x), at.sqr(x), at.reciprocal(px), at.arctan2(x, px), at.pow(px, x * 0.5),
            at.log1mexp(-px), at.isnan(x / (x - x)), at.deg2rad(x)]
    return [x], outs, [rnd(513, "float32", -4.0, 4.0)]


@case("ew_math_f64")
def _():
    x = at.dvector("x")
    px = abs(x) + 0.1
    outs = [at.exp(x), at.log(px), at.log1p(px), at.tanh(x), at.sigmoid(x), at.softplus(x * 15),
            at.erf(x), at.sqrt(px), at.sin(x) * at.cos(x), at.pow(px, x), at.arccosh(px + 1),
            at.arctanh(at.tanh(x) * 0.9), at.arcsin(at.sin(x)), at.arccos(at.cos(x))]
    return [x], outs, [rnd(300, "float64", -4.0, 4.0)]


@case("ew_fusion_multi")
def _():
    # a few rows in the spirit of tests/tensor/rewriting/test_elemwise.py:300-903
    x, y, z = at.fmatrix("x"), at.fmatrix("y"), at.fmatrix("z")
    iv = at.imatrix("iv")
    outs = [x + y + z, x * y * z - (x + y), (x + y) / (abs(z) + 1), at.exp(x + y + z),
            x + at.cast(iv, "float32") * y, at.switch(at.gt(x, y), x * 2, y / 2),
            at.sqr(x) + at.sqr(y) + at.sqr(z), at.eq(iv, 2) * x]
    return [x, y, z, iv], outs, [rnd((17, 9)), rnd((17, 9)), rnd((17, 9)), rnd((17, 9), "int32")]


@case("ew_scalar_0d")
def _():
    a, b = at.fscalar("a"), at.dscalar("b")
    x = at.fvector("x")
    return [a, b, x], [a * x + a, at.exp(b) * b, a + b, x.sum() * a], [np.float32(1.5), np.float64(-0.25), rnd(33)]


# ---------------------------------------------------------------- random Elemwise graphs
# Seeded random compositions over mixed dtypes: the reference's type promotion, fusion and
# in-place passes decide the Composite bodies; values stay in domains where C and CUDA are
# both defined (non-zero integer divisors, bounded float -> int casts).
def _fuzz_graph(seed, n_outs=7, n_elems=193):
    r = np.random.default_rng(seed)
    f32, f64 = at.fvector("f32"), at.dvector("f64")
    i32, i64, i8, u8 = at.ivector("i32"), at.lvector("i64"), at.bvector("i8"), at.vector("u8", dtype="uint8")
    bo = at.vector("bo", dtype="bool")
    floats, ints = [f32, f64], [i32, i64, i8, u8]
    pool_f, pool_i, pool_b = list(floats), list(ints), [bo]

    def pick(pool):
        return pool[int(r.integers(len(pool)))]

    unary_f = [at.tanh, at.sigmoid, abs, at.neg, at.sqr, at.floor, at.ceil, lambda t: at.exp(at.tanh(t)),
               lambda t: at.log(abs(t) + 1), lambda t: at.sqrt(abs(t)), at.sgn, lambda t: at.softplus(t),
               lambda t: at.log1p(abs(t)), lambda t: at.expm1(at.tanh(t)), at.sin, at.cos, at.arctan,
               lambda t: at.round(t)]
    binary_f = [lambda a, b: a + b, lambda a, b: a - b, lambda a, b: a * b, lambda a, b: a / (abs(b) + 0.5),
                at.maximum, at.minimum, lambda a, b: a // (abs(b) + 1), lambda a, b: a % (abs(b) + 1),
                lambda a, b: at.switch(at.gt(a, b), a, b * 2), lambda a, b: at.arctan2(a, abs(b) + 0.1),
                lambda a, b: abs(a) ** at.tanh(b)]
    binary_i = [lambda a, b: a + b, lambda a, b: a - b, lambda a, b: a * b, lambda a, b: a // (abs(b) + 1),
                lambda a, b: a % (abs(b) + 1), lambda a, b: a & b, lambda a, b: a | b, lambda a, b: a ^ b,
                at.maximum, at.minimum, lambda a, b: at.switch(at.lt(a, b), a, b)]
    unary_i = [abs, at.neg, lambda t: ~t, at.sgn, lambda t: at.cast(t, "int8"), lambda t: at.cast(t, "int64"),
               lambda t: at.cast(t, "uint8"), lambda t: at.cast(t, "int16"), lambda t: at.cast(t, "float32")]
    cmp_ops = [at.lt, at.gt, at.le, at.ge, at.eq, at.neq]
    for _ in range(int(r.integers(14, 22))):
        kind = r.random()
        if kind < 0.40:
            a = pick(pool_f)
            b = pick(pool_f + pool_i) if r.random() < 0.4 else pick(pool_f)
            pool_f.append(pick(binary_f)(a, b))
        elif kind < 0.58:
            pool_f.append(pick(unary_f)(pick(pool_f)))
        elif kind < 0.74:
            pool_i.append(pick(binary_i)(pick(pool_i), pick(pool_i)))
        elif kind < 0.84:
            v = pick(unary_i)(pick(pool_i))
            (pool_f if "float" in v.dtype else pool_i).append(v)
        elif kind < 0.92:
            a, b = (pick(pool_f), pick(pool_f)) if r.random() < 0.5 else (pick(pool_i), pick(pool_i))
            pool_b.append(pick(cmp_ops)(a, b))
        elif kind < 0.96:
            pool_b.append(pick([lambda a, b: a & b, lambda a, b: a | b, lambda a, b: a ^ b])(pick(pool_b), pick(pool_b)))
        else:
            # bounded float -> int cast, then back into the integer pool
            pool_i.append(at.cast(at.floor(at.tanh(pick(pool_f)) * 100), pick(["int32", "int64", "int16"])))
    cands = pool_f[2:] + pool_i[4:] + pool_b[1:]
    idx = r.permutation(len(cands))[:n_outs]
    outs = [cands[int(k)] for k in idx]
    vals = [rnd(n_elems, "float32"), rnd(n_elems, "float64"), rnd(n_elems, "int32"), rnd(n_elems, "int64"),
            rnd(n_elems, "int8"), rnd(n_elems, "uint8"), rnd(n_elems, "bool")]
    return [f32, f64, i32, i64, i8, u8, bo], outs, vals


for _seed in range(8):
    def _make(seed=_seed):
        return _fuzz_graph(1000 + seed)

    CASES[f"ew_fuzz_{_seed}"] = _make


# ---------------------------------------------------------------- CAReduce tables
# axes table of tests/tensor/test_elemwise.py:412-428 (TestCAReduce)
@case("careduce_sum_axes")
def _():
    x = at.ftensor3("x")
    m = at.fmatrix("m")
    outs = [x.sum(), x.sum(axis=0), x.sum(axis=1), x.sum(axis=2), x.sum(axis=(0, 2)),
            x.sum(axis=(1, 2)), x.sum(axis=(0, 1)), m.sum(axis=0), m.sum(axis=1), m.T.sum(axis=0),
            m.mean(), x.mean(axis=1)]
    return [x, m], outs, [rnd((5, 67, 9)), rnd((300, 130))]


@case("careduce_ops_dtypes")
def _():
    f = at.fmatrix("f")
    d = at.dmatrix("d")
    i8 = at.bmatrix("i8")
    i32 = at.imatrix("i32")
    bo = at.matrix("bo", dtype="bool")
    u8 = at.matrix("u8", dtype="uint8")
    outs = [f.max(), f.max(axis=0), f.min(axis=1), d.prod(axis=0), d.sum(), i8.sum(), i8.sum(axis=0),
            i8.max(axis=1), i8.min(), i32.prod(axis=1), i32.sum(axis=0), bo.all(), bo.any(axis=0),
            bo.all(axis=1), bo.sum(), u8.sum(axis=1), u8.max(), at.max(i32, axis=0), d.max(axis=1)]
    return [f, d, i8, i32, bo, u8], outs, [rnd((33, 65)), rnd((20, 11), "float64", 0.5, 1.5),
                                           rnd((40, 33), "int8"), rnd((9, 6), "int32"),
                                           rnd((12, 40), "bool"), rnd((30, 70), "uint8")]


@case("prod_grad_without_zeros")
def _():
    x = at.fmatrix("x")
    d = at.dvector("d")
    outs = [aesara.grad(x.prod(), x), aesara.grad(x.prod(axis=1).sum(), x), aesara.grad(d.prod() * 2, d),
            at.math.ProdWithoutZeros(axis=0)(x), at.math.ProdWithoutZeros()(d)]
    xv = rnd((5, 6), "float32", 0.5, 1.5)
    xv[1, 2] = 0.0
    xv[3, 0] = 0.0
    xv[3, 4] = 0.0
    dv = rnd(9, "float64", 0.5, 1.5)
    dv[4] = 0.0
    return [x, d], outs, [xv, dv]


@case("careduce_big_1d")
def _():
    x = at.fvector("x")
    return [x], [x.sum(), x.max(), (x * x).sum(), x.mean()], [rnd(300001)]


@case("careduce_nan")
def _():
    x = at.fmatrix("x")
    xv = rnd((8, 9))
    xv[2, 3] = np.nan
    return [x], [x.max(axis=0), x.min(axis=1), x.sum(axis=0), x.max()], [xv]


# ---------------------------------------------------------------- BLAS family
@case("blas_dot22_layouts")
def _():
    a, b, c = at.fmatrix("a"), at.fmatrix("b"), at.fmatrix("c")
    outs = [at.dot(a, b), at.dot(a.T, c), at.dot(b.T, a.T), at.dot(a, b) * 0.5]
    return [a, b, c], outs, [rnd((130, 70)), rnd((70, 96)), rnd((130, 40))]


@case("blas_gemm_alpha_beta")
def _():
    z, x, y = at.fmatrix("z"), at.fmatrix("x"), at.fmatrix("y")
    a, b = at.fscalar("a"), at.fscalar("b")
    outs = [b * z + a * at.dot(x, y), z - at.dot(x, y), z + 2.0 * at.dot(x, y)]
    return [z, x, y, a, b], outs, [rnd((150, 200)), rnd((150, 64)), rnd((64, 200)), np.float32(0.8), np.float32(0.4)]


@case("blas_gemm_f64")
def _():
    z, x, y = at.dmatrix("z"), at.dmatrix("x"), at.dmatrix("y")
    outs = [0.4 * z + 0.8 * at.dot(x, y), at.dot(x.T, z)]
    return [z, x, y], outs, [rnd((50, 60), "float64"), rnd((50, 33), "float64"), rnd((33, 60), "float64")]


@case("blas_gemv_ger")
def _():
    A, x, y = at.fmatrix("A"), at.fvector("x"), at.fvector("y")
    outs = [at.dot(A, x), at.dot(A.T, y), y + 0.5 * at.dot(A, x), A + at.outer(y, x) * 2.0,
            at.dot(y, A), at.dot(x, x)]
    return [A, x, y], outs, [rnd((300, 129)), rnd(129), rnd(300)]


@case("blas_gemv_f64")
def _():
    A, x, y = at.dmatrix("A"), at.dvector("x"), at.dvector("y")
    return [A, x, y], [at.dot(A, x) * 2 + y, at.dot(A.T, y)], [rnd((77, 50), "float64"), rnd(50, "float64"), rnd(77, "float64")]


# ---------------------------------------------------------------- views / layout edge cases
@case("views_negative_steps")
def _():
    x = at.fmatrix("x")
    v = at.fvector("v")
    t = at.ftensor3("t")
    outs = [x[::-1] * 2, x[5:1:-2, ::3] + 1, x[:, -1], x[-2], x[1:-1, 2:-2].sum(axis=0),
            at.dot(x[::-1], v), at.dot(x[:, ::-1], v[::-1]), at.dot(x[::2].T, x[::2]),
            t[::-1, :, ::-2].sum(axis=1), t[1][::-1].T + 0.5, v[::-3].max(), at.exp(v[None, :] + v[:, None])[::4, 1::5],
            x[2:2].sum(), x[:, 3:1].shape[1] + x[:0].sum(axis=0)]
    return [x, v, t], outs, [rnd((12, 10)), rnd(10), rnd((4, 5, 6))]


@case("incsubtensor_variants")
def _():
    x = at.fmatrix("x")
    v = at.fvector("v")
    s = at.fscalar("s")
    outs = [at.set_subtensor(x[1:4], 0.5), at.inc_subtensor(x[::2, 1::3], s), at.set_subtensor(x[:, 2], v[:x.shape[0]]),
            at.inc_subtensor(x[-1], v[:x.shape[1]] * 2), at.set_subtensor(x[2:5, 1:3], x[0:3, 4:6] + 1),
            at.inc_subtensor(v[::-1][:3], 10.0), at.set_subtensor(x[3, 4], s * s), at.inc_subtensor(x[1:1], 7.0)]
    return [x, v, s], outs, [rnd((7, 9)), rnd(9), np.float32(1.25)]


@case("reshape_flatten_noncontig")
def _():
    x = at.fmatrix("x")
    t = at.ftensor3("t")
    n = at.lscalar("n")
    outs = [x.T.reshape((-1,)), x.reshape((n, -1)) * 2, t.dimshuffle(2, 0, 1).reshape((6, -1)).sum(axis=1),
            x.flatten() + 1, t.flatten(2), x[::2].reshape((3, 2, -1)).max(axis=2), x.T.flatten()[::5],
            at.shape_padleft(x.sum(axis=0), 2) + t[:1, :1, :1].reshape((1, 1, 1)),
            x.reshape((1, -1))[0, 3:9], at.reshape(x.sum(), ())]
    return [x, t, n], outs, [rnd((6, 10)), rnd((4, 5, 6)), np.int64(4)]


@case("nan_inf_semantics_f32")
def _():
    x, y = at.fvector("x"), at.fvector("y")
    outs = [at.maximum(x, y), at.minimum(x, y), at.lt(x, y), at.ge(x, y), at.eq(x, x), at.neq(x, y),
            at.switch(at.isnan(x), y, x), x / y, x // y, x % y, at.sqrt(x), at.log(abs(x)), at.exp(x * 40),
            at.isinf(x / y), at.sgn(x), abs(x), at.clip(x, y, y + 2), at.floor(x), at.tanh(x * 1e6),
            at.sigmoid(x * 200), at.softplus(x * 200), at.log1p(x), at.true_div(1.0, x) * 0.0, at.pow(x, y)]
    xv = np.array([0.0, -0.0, 1.5, -2.5, np.nan, np.inf, -np.inf, 3.0, -3.0, 1e-30, 7.25, -7.25, 0.5, 2.0, -1.0, 9.0], "float32")
    yv = np.array([0.0, 2.0, -2.0, 0.0, 1.0, np.inf, 2.0, np.nan, -0.0, 1e30, 2.0, 2.0, -np.inf, 0.5, 0.5, -3.0], "float32")
    return [x, y], outs, [xv, yv]


@case("alloc_and_shape_ops")
def _():
    x = at.fmatrix("x")
    v = at.fvector("v")
    n = at.lscalar("n")
    outs = [at.zeros((n, 3)) + v[:3], at.ones_like(x) * v[:x.shape[1]], at.alloc(v, n, v.shape[0]) * 2,
            at.fill(x, 2.5) + x, x.shape[0] * 2 + x.shape[1], at.zeros_like(x, dtype="int32") + n,
            at.alloc(np.float32(1.5), n), at.prod(x.shape) + at.cast(n, "int64"),
            at.tile(v[:2], (3, 2)), at.repeat(v[:3], 2), at.stack([v, v * 2]).T.sum(axis=1),
            at.full_like(x, 4.0)[1:, :2] - x[1:, :2]]
    return [x, v, n], outs, [rnd((4, 6)), rnd(6), np.int64(5)]


@case("blas_edge_shapes")
def _():
    a, b, c = at.fmatrix("a"), at.fmatrix("b"), at.fmatrix("c")
    v = at.fvector("v")
    z = at.fmatrix("z")
    outs = [at.dot(a[:1], b), at.dot(a, b[:, :1]), at.dot(a[:, :1], b[:1]), at.dot(a[:0], b), at.dot(a, b[:, :0]),
            at.dot(a[:1], v[:a.shape[1]]), at.dot(v[:a.shape[0]], a), z + 0.5 * at.dot(a, b), at.dot(c, c.T) - at.dot(c.T, c)[:4, :4].sum(),
            at.dot(a, b).T + at.dot(b.T, a.T), at.outer(v, v)[:3] + 1, at.dot(v, v) * v]
    return [a, b, c, v, z], outs, [rnd((5, 7)), rnd((7, 6)), rnd((4, 9)), rnd(8), rnd((5, 6))]


# ---------------------------------------------------------------- Scan
@case("scan_cumsum_allsteps")
def _():
    x = at.fmatrix("x")
    s0 = at.fvector("s0")
    res, _ = aesara.scan(lambda x_t, s: s * 0.5 + x_t, sequences=[x], outputs_info=[s0])
    return [x, s0], [res, res[-1]], [rnd((7, 40)), rnd(40)]


@case("scan_two_taps_nitsot")
def _():
    x = at.fvector("x")
    init = at.fvector("init")  # two initial values

    def step(x_t, f_tm2, f_tm1):
        f = f_tm1 + f_tm2 * 0.5 + x_t
        return f, f * 2

    (f, g), _ = aesara.scan(step, sequences=[x], outputs_info=[dict(initial=init, taps=[-2, -1]), None])
    return [x, init], [f, g], [rnd(9), rnd(2)]


# Scan gradients / while loops (§8f N2): reversed Scan with mit-mot accumulators
# (scan/op.py:2379-3129), nit-sot outputs, `until` conditions
@case("scan_grad_rnn")
def _():
    x = at.fmatrix("x")           # [T, n]
    h0 = at.fvector("h0")
    W = at.fmatrix("W")           # [n, n]

    def step(x_t, h_tm1, W_):
        return at.tanh(at.dot(h_tm1, W_) + x_t)

    hs, _ = aesara.scan(step, sequences=[x], outputs_info=[h0], non_sequences=[W])
    loss = (hs ** 2).sum() + hs[-1].sum()
    gW, gx, gh0 = aesara.grad(loss, [W, x, h0])
    return [x, h0, W], [loss, gW, gx, gh0], [rnd((6, 12), "float32", -1, 1), rnd(12, "float32", -1, 1),
                                              rnd((12, 12), "float32", -0.4, 0.4)]


@case("scan_grad_lstm")
def _():
    i, o = G.cfg4_lstm_scan()
    x, h0, c0, U = i
    loss = (o[0] ** 2).sum() + o[1].sum()
    gU, gx = aesara.grad(loss, [U, x])
    T, B, H = 5, 6, 8
    r = np.random.default_rng(11)
    vals = [r.standard_normal((T, B, 4 * H)).astype("float32"),
            (r.standard_normal((B, H)) * 0.1).astype("float32"),
            (r.standard_normal((B, H)) * 0.1).astype("float32"),
            (r.standard_normal((H, 4 * H)) / np.sqrt(H)).astype("float32")]
    return i, [loss, gU, gx], vals


@case("scan_while_until")
def _():
    from aesara.scan.utils import until

    x0 = at.fvector("x0")
    limit = at.fscalar("limit")

    def step(v, lim):
        nv = v * 1.5 + 1.0
        return nv, until(nv.sum() > lim)

    vs, _ = aesara.scan(step, outputs_info=[x0], non_sequences=[limit], n_steps=40)
    return [x0, limit], [vs, vs[-1], vs.shape[0]], [rnd(5, "float32", 0, 1), np.float32(300.0)]


@case("scan_seq_taps_shared_nsteps")
def _():
    x = at.fvector("x")
    k = at.lscalar("k")

    def step(x_tm1, x_t, x_tp1, acc):
        return acc + x_tm1 * x_tp1 - x_t

    out, _ = aesara.scan(step, sequences=[dict(input=x, taps=[-1, 0, 1])], outputs_info=[at.zeros((), "float32")],
                         n_steps=k)
    return [x, k], [out, out[-1] * 2], [rnd(11), np.int64(7)]


# ---------------------------------------------------------------- Softmax family (§8f N1)
@case("softmax_classifier")
def _():
    from aesara.tensor.special import log_softmax, softmax

    x, t, W = at.fmatrix("x"), at.fmatrix("t"), at.fmatrix("W")
    logits = x @ W
    loss = -(t * log_softmax(logits, axis=1)).sum(axis=1).mean()
    g = aesara.grad(loss, W)
    outs = [loss, g, softmax(logits, axis=1), at.argmax(logits, axis=1), logits.max(axis=1)]
    tv = np.eye(37, dtype="float32")[RNG.integers(0, 37, size=300)]
    return [x, t, W], outs, [rnd((300, 64)), tv, rnd((64, 37), "float32", -0.5, 0.5)]


@case("softmax_axes")
def _():
    from aesara.tensor.special import log_softmax, softmax

    x3 = at.ftensor3("x3")
    d = at.dmatrix("d")
    big = at.fmatrix("big")
    sm = softmax(x3, axis=1)
    outs = [softmax(x3, axis=0), sm, softmax(x3, axis=2), softmax(x3, axis=None),
            log_softmax(d, axis=-1), log_softmax(d, axis=0), softmax(big, axis=1),
            aesara.grad((sm * sm).sum(), x3)]
    return [x3, d, big], outs, [rnd((5, 7, 9)), rnd((11, 13), "float64"), rnd((3, 2500))]


@case("max_and_argmax")
def _():
    x = at.ftensor3("x")
    i = at.imatrix("i")
    outs = [at.argmax(x, axis=0), at.argmax(x, axis=2), at.argmax(x), at.max_and_argmax(x, axis=1)[0],
            at.max_and_argmax(x, axis=1)[1], at.argmax(i, axis=1), at.argmax(x, axis=[0, 2]),
            at.argmin(x, axis=1)]
    xv = rnd((6, 50, 8))
    xv[2, 10, 3] = xv[2, 40, 3] = 9.0  # ties: first occurrence wins
    return [x, i], outs, [xv, rnd((9, 300), "int32")]


# ---------------------------------------------------------------- indexing / layout (§8f N3)
@case("indexing_embedding")
def _():
    E = at.fmatrix("E")           # embedding table
    idx = at.lvector("idx")
    i32 = at.ivector("i32")
    T3 = at.ftensor3("T3")
    iv = at.lvector("iv")         # int64 values, for the bit-exact integer scatter
    emb = E[idx]
    loss = (emb * emb).sum()
    gE = aesara.grad(loss, E)     # AdvancedIncSubtensor1 with duplicate indices
    outs = [emb, gE, E[i32], T3[idx[:4]], at.inc_subtensor(E[i32], 1.5),
            at.set_subtensor(E[idx[:3]], 0.0), at.inc_subtensor(at.zeros_like(iv)[idx % 5], iv[idx % 7])]
    idxv = np.array([3, 0, 7, 3, -1, 3, 2, 0, 9, -10], dtype="int64")
    return [E, idx, i32, T3, iv], outs, [rnd((10, 24)), idxv, np.array([1, 1, -2, 5], "int32"),
                                         rnd((10, 3, 5)), rnd(12, "int64")]


@case("classifier_int_labels")
def _():
    from aesara.tensor.special import log_softmax

    x, W = at.fmatrix("x"), at.fmatrix("W")
    y = at.lvector("y")
    logits = x @ W
    lp = log_softmax(logits, axis=1)
    loss = -at.mean(lp[at.arange(y.shape[0]), y])          # ARange + AdvancedSubtensor
    g = aesara.grad(loss, W)                               # AdvancedIncSubtensor in the backward pass
    acc = at.mean(at.eq(at.argmax(logits, axis=1), y))
    return [x, W, y], [loss, g, acc], [rnd((200, 48)), rnd((48, 10), "float32", -0.5, 0.5),
                                       RNG.integers(0, 10, size=200).astype("int64")]


@case("adv_index_pairs")
def _():
    x = at.fmatrix("x")
    t = at.ftensor3("t")
    i, j = at.lvector("i"), at.lvector("j")
    k32 = at.ivector("k32")
    v = at.fvector("v")
    n = at.lscalar("n")
    outs = [x[i, j], t[i, j], t[i, j][:, ::2] * 2, at.inc_subtensor(x[i, j], v), at.set_subtensor(x[i, j], 0.5),
            at.inc_subtensor(t[i, j], 1.0), at.inc_subtensor(x[k32, k32], v[:k32.shape[0]] * 2),
            at.arange(n) * 2, at.arange(2, n, 3), at.arange(0, n, 1, dtype="float32") / 4, at.arange(n)[::-1] + i[:1],
            x[at.arange(x.shape[0]), at.argmax(x, axis=1)], at.arange(300, dtype="int32").sum() + n]
    iv = np.array([0, 3, 3, -1, 2, 0, 3], "int64")
    jv = np.array([1, 4, 4, -2, 0, 1, 4], "int64")
    return [x, t, i, j, k32, v, n], outs, [rnd((4, 5)), rnd((4, 5, 6)), iv, jv, np.array([1, 1, 2], "int32"),
                                           rnd(7), np.int64(11)]


@case("batched_dot_ifelse")
def _():
    from aesara.ifelse import ifelse

    a, b = at.ftensor3("a"), at.ftensor3("b")
    m = at.fmatrix("m")
    c = at.iscalar("c")
    bd = at.batched_dot(a, b)
    outs = [bd, at.batched_dot(a, m[: a.shape[0], : a.shape[2]]), at.batched_dot(m[: a.shape[0], : a.shape[1]], a),
            ifelse(c, bd * 2, bd - 1), ifelse(at.gt(m.sum(), 1e6), m + 1, m * 3), aesara.grad((bd ** 2).sum(), a)]
    return [a, b, m, c], outs, [rnd((4, 5, 6)), rnd((4, 6, 3)), rnd((7, 9)), np.int32(1)]


@case("cumsum_cumprod")
def _():
    x = at.fmatrix("x")
    t = at.dtensor3("t")
    v = at.fvector("v")
    iv = at.lvector("iv")
    outs = [at.cumsum(x, axis=0), at.cumsum(x, axis=1), at.cumsum(x), at.cumprod(t * 0.5, axis=1), at.cumsum(t, axis=2),
            at.cumsum(v), at.cumprod(v * 0.01 + 1), at.cumsum(iv), at.cumsum(x.T, axis=0)[::2], at.cumsum(x[:0], axis=0),
            aesara.grad(at.cumsum(v).sum() + (at.cumsum(x, axis=1) ** 2).sum(), [v, x])[1]]
    return [x, t, v, iv], outs, [rnd((9, 14)), rnd((3, 5, 4), "float64"), rnd(5000), rnd(700, "int64")]


@case("diag_eye")
def _():
    x = at.fmatrix("x")
    t = at.ftensor3("t")
    n = at.lscalar("n")
    outs = [at.diag(x) * 2, x.diagonal(1) + 1, x.diagonal(-2), t.diagonal(0, 0, 2).sum(axis=1), at.diag(x).sum(),
            at.eye(n) * 3, at.eye(n, n + 4, 2) + 1, at.eye(n + 9, n, -3, dtype="int32"), x + at.eye(x.shape[0], x.shape[1]),
            aesara.grad(at.diag(x).sum() * 2, x), at.tril(x), at.triu(x, 1) * 2, at.tri(n, n + 3, -1, dtype="int32"),
            at.tril(at.ones((n, n)), 2).sum(axis=0)]
    return [x, t, n], outs, [rnd((9, 12)), rnd((5, 4, 6)), np.int64(11)]


@case("join_split_reshape")
def _():
    a, b, c = at.fmatrix("a"), at.fmatrix("b"), at.fmatrix("c")
    v = at.lvector("v")
    j0 = at.join(0, a, b)
    j1 = at.join(1, a, c)
    s = at.split(j1, [2, 5], n_splits=2, axis=1)
    outs = [j0, j1 * 2, s[0] + 1, s[1] - 1, at.join(0, v, v * 2), j0.reshape((-1, 2)),
            at.concatenate([a.T, b.T], axis=1), at.stack([a, a * 3], axis=0)]
    return [a, b, c, v], outs, [rnd((4, 6)), rnd((3, 6)), rnd((4, 1)), rnd(5, "int64")]


# ---------------------------------------------------------------- device-sized twins
# Round-1 review: fixtures with a few dozen elements say little about a launch geometry.  The
# cases below repeat the small tables above at >= 1000 elements per tensor (several CTAs, the
# vectorised and the ragged tail paths), and add device-sized Join / Split / Shape, NaN / inf /
# IntDiv, outer-broadcast and 3-D transposed-view cases.
@case("ew_outer_broadcast_big")
def _():
    a, b = at.fmatrix("a"), at.fmatrix("b")
    return [a, b], [a + b, at.maximum(a, b) * 2, a * b - at.minimum(a, b)], [rnd((1, 1501)), rnd((1103, 1))]


@case("ew_transposed_views_big")
def _():
    a, b = at.fmatrix("a"), at.fmatrix("b")
    t = at.tensor3("t", dtype="float32")
    outs = [a.T * b + 1, at.tanh(t.dimshuffle(2, 0, 1)) - t.dimshuffle(2, 0, 1) ** 2,
            (a.T + b)[::-1, ::2], t.dimshuffle(1, 2, 0) * 2 + t.dimshuffle(1, 2, 0)[::-1],
            at.exp(t.dimshuffle(0, 2, 1))[:, ::3, 1:] * 0.5]
    return [a, b, t], outs, [rnd((67, 45)), rnd((45, 67)), rnd((31, 42, 53))]


@case("nan_inf_semantics_f32_big")
def _():
    x, y = at.fvector("x"), at.fvector("y")
    outs = [at.maximum(x, y), at.minimum(x, y), at.lt(x, y), at.ge(x, y), at.eq(x, x), at.neq(x, y),
            at.switch(at.isnan(x), y, x), x / y, x // y, x % y, at.sqrt(x), at.log(abs(x)), at.exp(x * 40),
            at.isinf(x / y), at.sgn(x), abs(x), at.clip(x, y, y + 2), at.floor(x), at.tanh(x * 1e6),
            at.sigmoid(x * 200), at.softplus(x * 200), at.log1p(x), at.true_div(1.0, x) * 0.0, at.pow(x, y),
            at.int_div(x, y) * 2 + at.mod(x, y), at.ceil(x), at.trunc(y), at.round(x)]
    sp = np.array([0.0, -0.0, 1.5, -2.5, np.nan, np.inf, -np.inf, 3.0, -3.0, 1e-30, 7.25, -7.25, 0.5, 2.0,
                   -1.0, 9.0, 1e30, -1e30, 2.5, -0.5], "float32")
    # every special value against every special value, then ordinary values
    xs, ys = np.meshgrid(sp, sp, indexing="ij")
    xv = np.concatenate([xs.ravel(), rnd(1000, "float32", -9.5, 9.5)]).astype("float32")
    yv = np.concatenate([ys.ravel(), rnd(1000, "float32", -4.0, 4.0)]).astype("float32")
    return [x, y], outs, [xv, yv]


@case("incsubtensor_variants_big")
def _():
    x = at.fmatrix("x")
    v = at.fvector("v")
    s = at.fscalar("s")
    outs = [at.set_subtensor(x[1:40], 0.5), at.inc_subtensor(x[::2, 1::3], s), at.set_subtensor(x[:, 2], v[:x.shape[0]]),
            at.inc_subtensor(x[-1], v[:x.shape[1]] * 2), at.set_subtensor(x[20:50, 10:30], x[0:30, 40:60] + 1),
            at.inc_subtensor(v[::-1][:300], 10.0), at.set_subtensor(x[3, 4], s * s), at.inc_subtensor(x[1:1], 7.0),
            at.inc_subtensor(x[::-3, ::-2], x[::-3, ::-2] * 2), at.set_subtensor(x.T[5:25], v[:x.shape[0]])]
    return [x, v, s], outs, [rnd((71, 93)), rnd(1200), np.float32(1.25)]


@case("join_split_shape_big")
def _():
    a, b, c = at.fmatrix("a"), at.fmatrix("b"), at.fmatrix("c")
    v = at.lvector("v")
    t = at.ftensor3("t")
    j0 = at.join(0, a, b)
    j1 = at.join(1, a, c)
    s = at.split(j1, [20, 47], n_splits=2, axis=1)
    s3 = at.split(t, [5, 0, 12], n_splits=3, axis=1)
    outs = [j0, j1 * 2, s[0] + 1, s[1] - 1, at.join(0, v, v * 2), j0.reshape((-1, 2)),
            at.concatenate([a.T, b.T], axis=1), at.stack([a, a * 3], axis=0),
            at.join(2, t, t[:, :, ::-1] * 2), s3[0] * 2, s3[1].shape[1] + s3[2].sum(axis=1),
            at.join(0, a[::2], b[::-1], a[:0]), j0.shape[0] * 1000 + j1.shape[1], at.shape(at.join(1, t, t))[1:],
            at.join(-2, a.T, c.T)]
    return [a, b, c, v, t], outs, [rnd((41, 60)), rnd((33, 60)), rnd((41, 7)), rnd(1500, "int64"), rnd((9, 17, 23))]


@case("alloc_and_shape_ops_big")
def _():
    x = at.fmatrix("x")
    v = at.fvector("v")
    n = at.lscalar("n")
    outs = [at.zeros((n, 30)) + v[:30], at.ones_like(x) * v[:x.shape[1]], at.alloc(v, n, v.shape[0]) * 2,
            at.fill(x, 2.5) + x, x.shape[0] * 2 + x.shape[1], at.zeros_like(x, dtype="int32") + n,
            at.alloc(np.float32(1.5), n * 30), at.prod(x.shape) + at.cast(n, "int64"),
            at.tile(v[:20], (30, 2)), at.repeat(v[:300], 4), at.stack([v, v * 2]).T.sum(axis=1),
            at.full_like(x, 4.0)[1:, :2] - x[1:, :2], at.shape(x * 2)[::-1] + at.shape(v)[0]]
    return [x, v, n], outs, [rnd((44, 61)), rnd(61 * 20), np.int64(50)]


@case("prod_grad_without_zeros_big")
def _():
    x = at.fmatrix("x")
    d = at.dvector("d")
    outs = [aesara.grad(x.prod(), x), aesara.grad(x.prod(axis=1).sum(), x), aesara.grad(d.prod() * 2, d),
            at.math.ProdWithoutZeros(axis=0)(x), at.math.ProdWithoutZeros()(d)]
    xv = rnd((40, 50), "float32", 0.97, 1.03)
    xv[1, 2] = 0.0
    xv[3, 0] = 0.0
    xv[3, 4] = 0.0
    xv[30, 44] = 0.0
    dv = rnd(1100, "float64", 0.99, 1.01)
    dv[400] = 0.0
    return [x, d], outs, [xv, dv]


@case("blas_edge_shapes_big")
def _():
    a, b, c = at.fmatrix("a"), at.fmatrix("b"), at.fmatrix("c")
    v = at.fvector("v")
    z = at.fmatrix("z")
    outs = [at.dot(a[:1], b), at.dot(a, b[:, :1]), at.dot(a[:, :1], b[:1]), at.dot(a[:0], b), at.dot(a, b[:, :0]),
            at.dot(a[:1], v[:a.shape[1]]), at.dot(v[:a.shape[0]], a), z + 0.5 * at.dot(a, b), at.dot(c, c.T) - at.dot(c.T, c)[:4, :4].sum(),
            at.dot(a, b).T + at.dot(b.T, a.T), at.outer(v, v)[:3] + 1, at.dot(v, v) * v]
    return [a, b, c, v, z], outs, [rnd((50, 70)), rnd((70, 60)), rnd((40, 90)), rnd(1080), rnd((50, 60))]


@case("ew_scalar_0d_big")
def _():
    a, b = at.fscalar("a"), at.dscalar("b")
    x = at.fvector("x")
    return [a, b, x], [a * x + a, at.exp(b) * b, a + b, x.sum() * a, x * at.cast(b, "float32") - a],\
        [np.float32(1.5), np.float64(-0.25), rnd(3301)]


@case("scan_cumsum_allsteps_big")
def _():
    x = at.fmatrix("x")
    s0 = at.fvector("s0")
    res, _ = aesara.scan(lambda x_t, s: s * 0.5 + x_t, sequences=[x], outputs_info=[s0])
    return [x, s0], [res, res[-1]], [rnd((9, 1400)), rnd(1400)]


@case("scan_two_taps_nitsot_big")
def _():
    x = at.fmatrix("x")
    init = at.fmatrix("init")  # two initial rows

    def step(x_t, f_tm2, f_tm1):
        f = f_tm1 + f_tm2 * 0.5 + x_t
        return f, at.tanh(f) * 2

    (f, g), _ = aesara.scan(step, sequences=[x], outputs_info=[dict(initial=init, taps=[-2, -1]), None])
    return [x, init], [f, g, g[-1].sum()], [rnd((9, 1200), "float32", -1, 1), rnd((2, 1200), "float32", -1, 1)]


@case("scan_seq_taps_shared_nsteps_big")
def _():
    x = at.fmatrix("x")
    k = at.lscalar("k")

    def step(x_tm1, x_t, x_tp1, acc):
        return acc + x_tm1 * x_tp1 - x_t

    out, _ = aesara.scan(step, sequences=[dict(input=x, taps=[-1, 0, 1])],
                         outputs_info=[at.zeros_like(x[0])], n_steps=k)
    return [x, k], [out, out[-1] * 2], [rnd((11, 1300)), np.int64(7)]


@case("scan_while_until_big")
def _():
    from aesara.scan.utils import until

    x0 = at.fvector("x0")
    limit = at.fscalar("limit")

    def step(v, lim):
        nv = v * 1.25 + 0.5
        return nv, until(nv.mean() > lim)

    vs, _ = aesara.scan(step, outputs_info=[x0], non_sequences=[limit], n_steps=60)
    return [x0, limit], [vs, vs[-1], vs.shape[0]], [rnd(2000, "float32", 0, 1), np.float32(300.0)]


# ---------------------------------------------------------------- Scan cell family (one Gemm + Elemwise)
@case("scan_rnn_tanh_cell")
def _():
    """tanh-RNN with pre-projected inputs: h_t = tanh(x_t + h_{t-1} @ U): 1 gate, 1 state."""
    x = at.ftensor3("x")
    h0, U = at.fmatrix("h0"), at.fmatrix("U")
    hs, _ = aesara.scan(lambda x_t, h, U_: at.tanh(x_t + at.dot(h, U_)), sequences=[x], outputs_info=[h0],
                        non_sequences=[U])
    T, B, H = 5, 256, 64
    r = np.random.default_rng(21)
    return [x, h0, U], [hs[-1], hs.sum(axis=0)], [r.standard_normal((T, B, H)).astype("float32"),
                                                  (r.standard_normal((B, H)) * 0.1).astype("float32"),
                                                  (r.standard_normal((H, H)) / np.sqrt(H)).astype("float32")]


@case("scan_gated_unit_cell")
def _():
    """A minimal gated unit on one product (3 gates, 1 state):
    pre = x_t + h @ U;  z = sigmoid(pre_0), r = sigmoid(pre_1), n = tanh(pre_2 * r);  h' = (1 - z) * h + z * n."""
    x = at.ftensor3("x")
    h0, U = at.fmatrix("h0"), at.fmatrix("U")

    def step(x_t, h, U_):
        H = h.shape[1]
        pre = x_t + at.dot(h, U_)
        z = at.sigmoid(pre[:, :H])
        r = at.sigmoid(pre[:, H : 2 * H])
        n = at.tanh(pre[:, 2 * H :] * r)
        return (1.0 - z) * h + z * n

    hs, _ = aesara.scan(step, sequences=[x], outputs_info=[h0], non_sequences=[U])
    T, B, H = 6, 256, 64
    r = np.random.default_rng(22)
    return [x, h0, U], [hs[-1], hs], [r.standard_normal((T, B, 3 * H)).astype("float32"),
                                      (r.standard_normal((B, H)) * 0.1).astype("float32"),
                                      (r.standard_normal((H, 3 * H)) / np.sqrt(H)).astype("float32")]


PY_LINKER_CASES = {"indexing_embedding", "adv_index_pairs", "classifier_int_labels", "cumsum_cumprod", "batched_dot_ifelse"}


def main(names):
    from aesara_b200.graphs import optimized_program

    for name in names:
        ins, outs, values = CASES[name]()
        # AdvancedIncSubtensor1's C code needs NumPy-1 PyArrayMapIter (gone in NumPy 2) and
        # CumOp's passes NPY_MAXDIMS as the "flatten" axis (NumPy 2 wants NPY_RAVEL_AXIS):
        # those cases run the reference's Python `perform` implementations instead
        linker = "py" if name in PY_LINKER_CASES else "cvm"
        prog, f = optimized_program(ins, outs, name=name, linker=linker)
        ref = f(*values)
        prog.save(os.path.join(HERE, name + ".json"))
        blob = {}
        for k, v in enumerate(values):
            blob[f"in_{k}"] = np.asarray(v)
        for k, v in enumerate(ref):
            blob[f"out_{k}"] = np.asarray(v)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **blob)
        print(f"{name}: {len(prog.nodes)} nodes {prog.op_counts()}")


def c_linker_baseline():
    """The reference C-linker's outputs of the BASELINE calls of tests/_cases.py (sampled where
    large) -> c_linker_baseline.npz."""
    from aesara.compile.mode import Mode

    from tests._cases import BASELINE_CALLS, C_LINKER_GOLDEN, sample_positions

    blob = {}
    for name, (_, graph, inputs) in BASELINE_CALLS.items():
        i, o = getattr(G, graph)()
        f = aesara.function(i, o, mode=Mode("cvm", "fast_run"), on_unused_input="ignore")
        for k, v in enumerate(f(*inputs(G))):
            v = np.asarray(v)
            pos = sample_positions(v.size)
            if pos is None:
                blob[f"{name}_out_{k}"] = v
            else:
                blob[f"{name}_pos_{k}"] = pos
                blob[f"{name}_out_{k}"] = v.reshape(-1)[pos]
        print(f"{name}: {len(o)} outputs")
    np.savez_compressed(C_LINKER_GOLDEN, **blob)


def shardplan_mixed_program():
    """The hand-built graph of tests/test_shardplan.py::test_sum_outputs_and_mixed_graph as the
    front-end lowers it -> programs/shardplan_mixed_outputs.json."""
    from aesara_b200.lower import lower_fgraph
    from tests._cases import shardplan_mixed_graph

    f = aesara.function(*shardplan_mixed_graph(at), mode="FAST_COMPILE")
    os.makedirs(os.path.join(HERE, "programs"), exist_ok=True)
    lower_fgraph(f.maker.fgraph).save(os.path.join(HERE, "programs", "shardplan_mixed_outputs.json"))


if __name__ == "__main__":
    if sys.argv[1:] == ["--c-linker"]:
        c_linker_baseline()
    elif sys.argv[1:] == ["--shardplan-program"]:
        shardplan_mixed_program()
    else:
        main(sys.argv[1:] or list(CASES))
