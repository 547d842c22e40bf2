"""CUDA source of a tcgen05 GEMM whose epilogue runs the Elemwise / Sum nodes that consume
the product.

The reference runs ``Dot22``/``Gemm`` and the following ``Elemwise`` nodes (``tanh(x @ W +
b)``, ``g * (1 - h**2)``, ``2*(h @ W2 - Y + b2)/n`` ...) and their ``Sum`` consumers as
separate thunks: every [M, N] intermediate goes to memory and comes straight back
(``tensor/blas.py:872/1659`` then ``tensor/elemwise.py:835`` / ``:1221``).  Here the scalar
expressions of those Elemwise nodes are merged into ONE scalar program, emitted as
``ab_ep_body`` (same emitter as the Elemwise kernels) in front of
``csrc/ab_gemm_tcgen05_kernel.cuh`` compiled with ``AB_EPILOGUE``: the epilogue warps apply it
to ``v = alpha*acc + beta*C_in`` while the values are in registers, store only the values
somebody outside the region reads (float32 and / or the bf16 plane the next GEMM wants as its
operand), and accumulate column sums / the total of one value each in float64.
"""

from __future__ import annotations

import os

from .scalar_cuda import emit_body

_CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "csrc")
MAX_OPERANDS = 4
MAX_OUTPUTS = 3


def _read(name):
    with open(os.path.join(_CSRC, name)) as f:
        text = f.read()
    keep = []
    for line in text.split("\n"):
        if line.startswith('#include "') or line.strip() == "#pragma once":
            continue
        keep.append(line)
    return "\n".join(keep)


def merge_exprs(steps, n_operands, outputs, name="region"):
    """Merge the scalar expressions of a chain / DAG of Elemwise nodes into one expression.

    ``steps``: list of ``(expr, arg_refs)`` in evaluation order; ``arg_refs[k]`` says where
    input ``k`` of that node's expression comes from: ``("acc",)`` the GEMM result,
    ``("op", j)`` memory operand ``j``, ``("val", s)`` the output of step ``s``.
    ``outputs``: list of ``("acc",)`` / ``("val", s)`` — the values the program yields.
    The merged expression has inputs ``[acc, operand 0, ...]`` (all float32)."""
    stmts, val_ref = [], {}

    def src(ref):
        if ref[0] == "acc":
            return "i0"
        if ref[0] == "op":
            return f"i{1 + ref[1]}"
        return val_ref[ref[1]]

    for s, (expr, arg_refs) in enumerate(steps):
        if len(expr["out_dtypes"]) != 1 or expr["out_dtypes"][0] != "float32":
            raise NotImplementedError("fused epilogue: one float32 output per node")
        if any(dt != "float32" for dt in expr["inputs"]):
            raise NotImplementedError("fused epilogue: float32 operands")
        base = len(stmts)

        def remap(r):
            if isinstance(r, dict):
                return r
            if r[0] == "i":
                return src(arg_refs[int(r[1:])])
            return f"t{base + int(r[1:])}"

        for st in expr["stmts"]:
            new = dict(st)
            new["args"] = [remap(r) for r in st["args"]]
            stmts.append(new)
        val_ref[s] = remap(expr["outputs"][0])
    outs = [src(o) for o in outputs]
    return {"inputs": ["float32"] * (1 + n_operands), "out_dtypes": ["float32"] * len(outs),
            "outputs": outs, "stmts": stmts, "name": name}


_UNIFORM_DIV = """\
// x / d for a d that is the same for every element of the launch (codegen/scalar_cuda.py
// emit_body).  r = ab_uniform_rcp(d) is 1 / d when d = +-2^k and 2^-k is a normal float, else
// 0.  For such a d, x * r is the same correctly rounded value as x / d for every x (subnormal
// results, zeros, infinities, NaN).  `fast` is a compile-time constant at every call: the
// kernel checks r != 0 once and runs the chunk loop built for that case.
__device__ __forceinline__ float ab_uniform_rcp(float d) {
  const unsigned e = (__float_as_uint(d) >> 23) & 0xffu;
  return ((__float_as_uint(d) & 0x7fffffu) == 0u && e >= 1u && e <= 253u) ? 1.0f / d : 0.0f;
}
__device__ __forceinline__ float ab_div_uniform(float x, float d, float r, bool fast) {
  return fast ? x * r : x / d;
}"""


def gemm_region_source(merged, n_operands, colsum=-1, fullsum=-1, cin=True, pre_op=-1, tplane=-1,
                       exact_sums=True, row_mask=0, scalar_mask=0):
    """``merged``: expression from :func:`merge_exprs` (input 0 = the accumulator value).
    ``colsum`` / ``fullsum``: index of the value whose column sums / total the epilogue
    accumulates in float64 (-1: none).  ``cin``: the product has a beta*C term read from memory
    (a ``Gemm``) — read a chunk ahead; ``pre_op``: the memory operand that is a full [M, N]
    matrix with unit column stride (the launch checks it), read a chunk ahead as well (-1:
    none).  ``tplane``: index of the value that can also be written as a transposed bf16
    operand plane (-1: none; must equal ``colsum`` when both are given -- the kernel keeps one
    value per chunk in registers for both).
    ``exact_sums``: the sums inside a warp are kept as float pairs (float64-equivalent, the
    fp32-faithful policy); otherwise 8 / 32 addends at a time are added as a float32 tree (the
    tf32 / bf16 policies, whose addends carry a larger error than that already).
    ``row_mask``: bit k set = memory operand k is statically a [1, N] row (a bias).
    ``scalar_mask``: bit k set = memory operand k is statically [1, 1]: read once per kernel,
    and a division by it is decided once per kernel (``ab_div_uniform``)."""
    if tplane >= 0 and colsum >= 0 and tplane != colsum:
        raise NotImplementedError("fused epilogue: transposed plane and column sums of different values")
    n_out = len(merged["out_dtypes"])
    if not 1 <= n_out <= MAX_OUTPUTS:
        raise NotImplementedError("fused epilogue: 1..3 values")
    if n_operands > MAX_OPERANDS:
        raise NotImplementedError("fused epilogue: at most 4 memory operands")
    scalars = [k for k in range(n_operands) if (scalar_mask >> k) & 1]
    args = ["(V)"] + [f"(E)[{k}][(T)]" for k in range(n_operands)] + [f"(O)[{k}][(T)]" for k in range(n_out)]
    body = emit_body(merged, fn_name="ab_ep_body", uniform_divisors=[1 + k for k in scalars])
    udiv = "ab_div_uniform(" in body
    args += [f"(R)[{k}]" for k in scalars] + (["(F)"] if scalars else [])
    gen = [
        "// generated by aesara_b200.codegen.gemm_epilogue — " + merged.get("name", ""),
        "#define AB_EPILOGUE 1",
        f"#define AB_EP_NOPS {n_operands}",
        f"#define AB_EP_NOUT {n_out}",
        f"#define AB_EP_COLSUM ({colsum})",
        f"#define AB_EP_FULLSUM ({fullsum})",
        f"#define AB_EP_CIN {1 if cin else 0}",
        f"#define AB_EP_PRE_OP ({pre_op})",
        f"#define AB_EP_TPLANE ({tplane})",
        f"#define AB_EP_EXACT_SUMS {1 if exact_sums else 0}",
        f"#define AB_EP_ROWMASK {int(row_mask)}",
        f"#define AB_EP_SCALARMASK {int(scalar_mask)}",
        f"#define AB_EP_UDIV {1 if udiv else 0}",  # the program divides by a [1, 1] operand
        # the stored / reduced / transposed value leaves through shared memory (coalesced
        # stores, shuffle-free transposes); AB_EP_NO_STAGING=1 keeps the register-only epilogue
        f"#define AB_EP_STAGED {0 if os.environ.get('AB_EP_NO_STAGING') else 1}",
        _UNIFORM_DIV,
        body,
        "#define AB_EP_EVAL(V, E, T, O, R, F) ab_ep_body(" + ", ".join(args) + ")",
        "namespace ab { namespace tc {} }",
    ]
    return "\n".join([
        _read("ab_types.cuh"),
        _read("ab_tcgen05.cuh"),
        "\n".join(gen),
        "using namespace ab::tc;",
        _read("ab_gemm_tcgen05_kernel.cuh"),
    ])


def gemm_epilogue_source(expr, acc_input, operand_inputs):
    """Single consumer node (kept for callers that fuse exactly one Elemwise): ``expr`` is its
    scalar expression, ``acc_input`` the input fed by the GEMM result, ``operand_inputs`` the
    inputs read from memory in ``ep_ptr`` order."""
    n_in = len(expr["inputs"])
    if sorted([acc_input] + list(operand_inputs)) != list(range(n_in)):
        raise NotImplementedError("fused epilogue: operand list does not cover the expression inputs")
    refs = [("acc",) if k == acc_input else ("op", list(operand_inputs).index(k)) for k in range(n_in)]
    merged = merge_exprs([(expr, refs)], len(operand_inputs), [("val", 0)], name=expr.get("name", ""))
    return gemm_region_source(merged, len(operand_inputs))
