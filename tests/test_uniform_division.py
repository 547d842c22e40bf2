"""Division by a launch-uniform [1, 1] operand in the fused GEMM epilogue (ab_div_uniform in
codegen/gemm_epilogue.py): for d = +-2^k whose reciprocal is a normal float, x * (1/d) is the
same float32 as x / d for every x.  Restated on the host with IEEE float32 arithmetic."""

import numpy as np

from aesara_b200.codegen.gemm_epilogue import gemm_region_source
from aesara_b200.codegen.scalar_cuda import emit_body


def _uniform_rcp(d):
    """The device rule (ab_uniform_rcp): 1/d for d = +-2^k with a normal reciprocal, else 0."""
    b = int(np.float32(d).view(np.uint32))
    e = (b >> 23) & 0xFF
    if (b & 0x7FFFFF) == 0 and 1 <= e <= 253:
        return np.float32(1.0) / np.float32(d)
    return np.float32(0.0)


def _xs():
    rng = np.random.default_rng(0)
    f = np.finfo(np.float32)
    special = [0.0, -0.0, np.inf, -np.inf, np.nan, f.tiny, -f.tiny, f.smallest_subnormal, -f.smallest_subnormal,
               f.max, -f.max, 1.0, -1.0, 3.0, 0.1, 2.0 ** -140, 2.0 ** -127 * 1.5]
    bits = rng.integers(0, 2 ** 32, size=200_000, dtype=np.uint64).astype(np.uint32)
    return np.concatenate([np.array(special, dtype=np.float32), bits.view(np.float32)])


def test_multiply_by_exact_reciprocal_equals_division():
    x = _xs()
    ks = list(range(-126, 127)) + [127, -127, -149]
    checked = 0
    with np.errstate(all="ignore"):
        for k in ks:
            for sign in (1.0, -1.0):
                d = np.float32(sign * 2.0 ** k)
                r = _uniform_rcp(d)
                if r == 0:
                    # 2^127 (subnormal reciprocal) and the subnormal divisors keep the division
                    assert k in (127, -127, -149)
                    continue
                q_div = x / d
                q_mul = x * r
                both_nan = np.isnan(q_div) & np.isnan(q_mul)
                assert np.array_equal(q_div.view(np.uint32)[~both_nan], q_mul.view(np.uint32)[~both_nan]), k
                assert np.array_equal(np.isnan(q_div), np.isnan(q_mul))
                checked += 1
        # the quotients above include subnormal results (x tiny, k > 0) and overflow (k < 0)
        assert np.any((np.abs(x / np.float32(2.0 ** 20)) < np.finfo(np.float32).tiny) & (x != 0))
    assert checked == 2 * 253


def test_other_divisors_keep_the_division():
    for d in (3.0, 0.1, 0.0, -0.0, np.inf, -np.inf, np.nan, 2.0 ** -149, 2.0 ** 127, 2.0 ** 28 + 2.0 ** 5):
        assert _uniform_rcp(np.float32(d)) == 0
    assert _uniform_rcp(np.float32(2.0 ** 28)) == np.float32(2.0 ** -28)  # B * H of cfg3


def test_region_source_divides_by_the_scalar_operand():
    """(i0 * i1) / i2 with i2 a statically [1, 1] operand: the generated body takes its
    reciprocal and the kernel is built with the multiply variant; the Elemwise emitter (no
    uniform divisors) still writes the plain division."""
    expr = {"inputs": ["float32"] * 3, "out_dtypes": ["float32"], "outputs": ["t1"], "name": "div",
            "stmts": [{"op": "mul", "args": ["i0", "i1"], "in_dtypes": ["float32", "float32"], "dtype": "float32"},
                      {"op": "true_divide", "args": ["t0", "i2"], "in_dtypes": ["float32", "float32"],
                       "dtype": "float32"}]}
    assert "(t0 / i2)" in emit_body(expr)
    src = gemm_region_source(expr, 2, cin=False, scalar_mask=0b10)
    assert "ab_div_uniform(t0, i2, r2, udiv)" in src
    assert "#define AB_EP_UDIV 1" in src and "#define AB_EP_SCALARMASK 2" in src
    src = gemm_region_source(expr, 2, cin=False, scalar_mask=0b01)  # the divisor is not uniform
    assert "(t0 / i2)" in src and "#define AB_EP_UDIV 0" in src
