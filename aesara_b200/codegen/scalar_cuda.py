"""IR scalar expression -> CUDA C++ (`ab_body`).

One table entry per scalar Op, transcribing the semantics of the reference's
``c_code`` (``aesara/scalar/basic.py`` — line numbers next to each entry — and
``aesara/scalar/math.py:1110-1258``): the reference casts the argument to the
*output* C type and calls the libm function of that name; temporaries are
typed with the output dtype, so arithmetic follows C promotion rules.
"""

from __future__ import annotations

import math

from ..ir import CTYPE

FLOATS = ("float32", "float64")
INTS = ("int8", "int16", "int32", "int64")
UINTS = ("uint8", "uint16", "uint32", "uint64")


class UnsupportedScalar(NotImplementedError):
    pass


def ctype(dt):
    try:
        return CTYPE[dt]
    except KeyError:
        raise UnsupportedScalar(f"dtype {dt} has no device representation") from None


def literal(value, dtype):
    """A C literal of the given dtype."""
    ct = ctype(dtype)
    if dtype == "bool":
        return f"(({ct}){1 if value else 0})"
    if dtype in INTS:
        v = int(value)
        if v == -(2**63):
            return f"(({ct})(-9223372036854775807LL - 1LL))"
        return f"(({ct}){v}LL)"
    if dtype in UINTS:
        return f"(({ct}){int(value)}ULL)"
    v = float(value)
    if dtype == "float32":
        if math.isnan(v):
            return "AB_NAN_F"
        if math.isinf(v):
            return "AB_INF_F" if v > 0 else "(-AB_INF_F)"
        import numpy as np

        return repr(float(np.float32(v))) + "f"
    if dtype == "float64":
        if math.isnan(v):
            return "AB_NAN_D"
        if math.isinf(v):
            return "AB_INF_D" if v > 0 else "(-AB_INF_D)"
        return repr(v)
    raise UnsupportedScalar(f"constant of dtype {dtype}")


def _f(name, dt):
    """libm function name for the float type (C++ overloads would do the same)."""
    return name + ("f" if dt == "float32" else "")


def _kind(dt):
    if dt in FLOATS:
        return "f"
    if dt in INTS:
        return "i"
    if dt in UINTS:
        return "u"
    if dt == "bool":
        return "b"
    raise UnsupportedScalar(f"dtype {dt} is not supported on device")


def _upcast(dts):
    import numpy as np

    return np.result_type(*[np.dtype(d) for d in dts]).name


def _unary_float(name):
    # e.g. basic.py:3102-3109 Exp: z = exp((T_out)x)
    def gen(a, idt, odt, st):
        if odt not in FLOATS:
            raise UnsupportedScalar(f"{name} with output dtype {odt}")
        return f"{_f(name, odt)}(({ctype(odt)}){a[0]})"

    return gen


def _cmp(sym):  # basic.py:1360-1461
    return lambda a, idt, odt, st: f"({a[0]} {sym} {a[1]})"


def _add(a, idt, odt, st):  # basic.py:1829-1837
    return "(" + (" || " if odt == "bool" else " + ").join(a) + ")"


def _mul(a, idt, odt, st):  # basic.py:1897-1907
    return "(" + (" && " if odt == "bool" else " * ").join(a) + ")"


def _true_divide(a, idt, odt, st):  # basic.py:1997-2011
    if _kind(idt[0]) in "biu" and _kind(idt[1]) in "biu":
        return f"(((double){a[0]}) / {a[1]})"
    return f"({a[0]} / {a[1]})"


def _int_div(a, idt, odt, st):  # basic.py:2055-2127
    t = _upcast(idt)
    ct = ctype(t)
    k = _kind(t)
    if k == "f":
        return f"ab_floordiv_f(({ct}){a[0]}, ({ct}){a[1]})"
    fn = "ab_floordiv_uint" if k in "ub" else "ab_floordiv_int"
    return f"{fn}<{ct}>(({ct}){a[0]}, ({ct}){a[1]})"


def _mod(a, idt, odt, st):  # basic.py:2165-2240
    t = _upcast(idt)
    ct = ctype(t)
    k = _kind(t)
    if k == "f":
        return f"ab_mod_f(({ct}){a[0]}, ({ct}){a[1]})"
    fn = "ab_mod_uint" if k in "ub" else "ab_mod_int"
    return f"{fn}<{ct}>(({ct}){a[0]}, ({ct}){a[1]})"


def _pow(a, idt, odt, st):  # basic.py:2263: pow(x, y) under C++ overloading
    t = _upcast(idt)
    if t == "float32":
        return f"powf((float){a[0]}, (float){a[1]})"
    return f"pow((double){a[0]}, (double){a[1]})"


def _maximum(a, idt, odt, st):  # basic.py:1745-1752
    t = _upcast(idt)
    if _kind(t) == "f":
        return f"ab_max_f(({ctype(t)}){a[0]}, ({ctype(t)}){a[1]})"
    return f"ab_max_int<{ctype(t)}>(({ctype(t)}){a[0]}, ({ctype(t)}){a[1]})"


def _minimum(a, idt, odt, st):  # basic.py:1788-1793
    t = _upcast(idt)
    if _kind(t) == "f":
        return f"ab_min_f(({ctype(t)}){a[0]}, ({ctype(t)}){a[1]})"
    return f"ab_min_int<{ctype(t)}>(({ctype(t)}){a[0]}, ({ctype(t)}){a[1]})"


def _cast(a, idt, odt, st):  # basic.py:2466-2470
    if odt == "bool":
        return f"(({a[0]}) ? 1 : 0)"
    return f"(({ctype(odt)}){a[0]})"


def _abs(a, idt, odt, st):  # basic.py:2570-2585
    k = _kind(idt[0])
    if k == "f":
        return f"{_f('fabs', idt[0])}({a[0]})"
    if k == "i":
        return f"(({a[0]}) < 0 ? -({a[0]}) : ({a[0]}))"
    return f"({a[0]})"


def _sgn(a, idt, odt, st):  # basic.py:2614-2630
    k = _kind(idt[0])
    if k == "f":
        return f"ab_sgn_f({a[0]})"
    if k == "i":
        return f"(({a[0]}) >= 0 ? (({a[0]}) == 0 ? 0 : 1) : -1)"
    return f"(({a[0]}) == 0 ? 0 : 1)"


def _isnan(a, idt, odt, st):  # basic.py:1478-1489
    return f"(isnan({a[0]}) ? 1 : 0)" if _kind(idt[0]) == "f" else "0"


def _isinf(a, idt, odt, st):  # basic.py:1505-1518
    return f"(isinf({a[0]}) ? 1 : 0)" if _kind(idt[0]) == "f" else "0"


def _invert(a, idt, odt, st):  # basic.py:1720-1725
    return f"(!{a[0]})" if odt == "bool" else f"(~{a[0]})"


def _trunc(a, idt, odt, st):  # basic.py:2702
    fl = _f("floor", odt)
    return f"(({a[0]}) >= 0 ? {fl}({a[0]}) : -{fl}(-({a[0]})))"


def _float_only(fn_name):
    def gen(a, idt, odt, st):
        if odt not in FLOATS:
            raise UnsupportedScalar(f"{fn_name} needs a float output, got {odt}")
        return f"{fn_name}(({ctype(odt)}){a[0]})"

    return gen


def _inrange(a, idt, odt, st):  # basic.py:1545-1553
    c1 = ">" if st.get("openlow") else ">="
    c2 = "<" if st.get("openhi") else "<="
    return f"(({a[0]} {c1} {a[1]}) && ({a[0]} {c2} {a[2]}))"


def _mean(a, idt, odt, st):  # basic.py:1871-1876
    return f"(({' + '.join(a)}) / ((double){len(a)}))"


TABLE = {
    "lt": _cmp("<"), "gt": _cmp(">"), "le": _cmp("<="), "ge": _cmp(">="),
    "eq": _cmp("=="), "neq": _cmp("!="),
    "isnan": _isnan, "isinf": _isinf, "inrange": _inrange,
    "switch": lambda a, i, o, s: f"(({a[0]}) ? ({a[1]}) : ({a[2]}))",  # :1586
    "or": lambda a, i, o, s: f"({a[0]} | {a[1]})",  # :1665
    "xor": lambda a, i, o, s: f"({a[0]} ^ {a[1]})",  # :1683
    "and": lambda a, i, o, s: f"({a[0]} & {a[1]})",  # :1701
    "invert": _invert,
    "maximum": _maximum, "minimum": _minimum,
    "add": _add, "mul": _mul, "mean": _mean,
    "sub": lambda a, i, o, s: f"({a[0]} - {a[1]})",  # :1955
    "true_divide": _true_divide, "int_div": _int_div, "mod": _mod, "pow": _pow,
    "clip": lambda a, i, o, s: (  # :2355
        f"(({a[0]}) < ({a[1]}) ? ({a[1]}) : (({a[0]}) > ({a[2]}) ? ({a[2]}) : ({a[0]})))"
    ),
    "second": lambda a, i, o, s: f"({a[1]})",  # :2385
    "identity": lambda a, i, o, s: f"({a[0]})",  # :2417
    "cast": _cast, "abs": _abs, "sgn": _sgn,
    "ceil": _unary_float("ceil"), "floor": _unary_float("floor"),  # :2655 / :2681
    "trunc": _trunc,
    "round_half_to_even": lambda a, i, o, s: f"{_f('rint', o)}({a[0]})",  # :2738 (npy_rint)
    "round_half_away_from_zero": lambda a, i, o, s: f"{_f('round', o)}({a[0]})",  # :2821
    "neg": lambda a, i, o, s: f"(-{a[0]})",  # :2853
    "reciprocal": lambda a, i, o, s: f"(1.0 / {a[0]})",  # :2892
    "log": _unary_float("log"), "log2": _unary_float("log2"),
    "log10": _unary_float("log10"), "log1p": _unary_float("log1p"),
    "exp": _unary_float("exp"), "exp2": _unary_float("exp2"),
    "expm1": _unary_float("expm1"),
    "sqr": lambda a, i, o, s: f"({a[0]} * {a[0]})",  # :3208
    "sqrt": _unary_float("sqrt"),
    "deg2rad": lambda a, i, o, s: f"({a[0]} * (3.14159265358979323846 / 180.0))",  # :3277
    "rad2deg": lambda a, i, o, s: f"({a[0]} * (180.0 / 3.14159265358979323846))",  # :3312
    "cos": _unary_float("cos"), "arccos": _unary_float("acos"),
    "sin": _unary_float("sin"), "arcsin": _unary_float("asin"),
    "tan": _unary_float("tan"), "arctan": _unary_float("atan"),
    "arctan2": lambda a, i, o, s: f"{_f('atan2', o)}(({ctype(o)}){a[0]}, ({ctype(o)}){a[1]})",
    "cosh": _unary_float("cosh"), "arccosh": _unary_float("acosh"),
    "sinh": _unary_float("sinh"), "arcsinh": _unary_float("asinh"),
    "tanh": _unary_float("tanh"), "arctanh": _unary_float("atanh"),
    "sigmoid": _float_only("ab_sigmoid"),  # math.py:1110
    "softplus": _float_only("ab_softplus"),  # math.py:1172
    "log1mexp": _float_only("ab_log1mexp"),  # math.py:1248
    "erf": _unary_float("erf"), "erfc": _unary_float("erfc"),
    "erfinv": _unary_float("erfinv"), "erfcinv": _unary_float("erfcinv"),
    "erfcx": _unary_float("erfcx"),
    "gamma": _unary_float("tgamma"), "gammaln": _unary_float("lgamma"),
}


def emit_body(expr, fn_name="ab_body", uniform_divisors=()):
    """Return CUDA source of ``__device__ void ab_body(in..., out&...)``.

    ``uniform_divisors``: indices k of float32 inputs that hold the same value for every element
    of a launch.  The function then takes one more parameter ``r<k>`` per such input, ``1/i<k>``
    when that is an exact power of two with a normal reciprocal, and a last ``bool udiv``: true
    when the caller has checked, once, that every ``r<k>`` is such a reciprocal.  A float32
    division by ``i<k>`` becomes ``ab_div_uniform(x, i<k>, r<k>, udiv)``: ``x * r<k>`` under
    ``udiv`` (the same bits as the IEEE division, without its per-element refinement and
    slow-path branch), the IEEE division otherwise."""
    in_dts = expr["inputs"]
    out_dts = expr["out_dtypes"]
    params = [f"const {ctype(dt)} i{k}" for k, dt in enumerate(in_dts)]
    params += [f"{ctype(dt)}& o{k}" for k, dt in enumerate(out_dts)]
    udiv = {f"i{k}": f"r{k}" for k in uniform_divisors if in_dts[k] == "float32"}
    params += [f"const float {r}" for r in udiv.values()] + (["const bool udiv"] if udiv else [])
    lines = [f"__device__ __forceinline__ void {fn_name}({', '.join(params)}) {{"]

    def ref(r):
        if isinstance(r, dict):
            return literal(r["const"], r["dtype"])
        return r

    for k, st in enumerate(expr["stmts"]):
        gen = TABLE.get(st["op"])
        if gen is None:
            raise UnsupportedScalar(f"scalar op {st['op']} has no device expression")
        args = [ref(r) for r in st["args"]]
        idt = st.get("in_dtypes")
        if idt is None:
            raise UnsupportedScalar("statement without in_dtypes")
        for dt in list(idt) + [st["dtype"]]:
            _kind(dt)
        if (st["op"] == "true_divide" and st["dtype"] == "float32" and list(idt) == ["float32", "float32"]
                and args[1] in udiv):
            rhs = f"ab_div_uniform({args[0]}, {args[1]}, {udiv[args[1]]}, udiv)"
        else:
            rhs = gen(args, idt, st["dtype"], st)
        lines.append(f"  const {ctype(st['dtype'])} t{k} = {rhs};")
    for k, r in enumerate(expr["outputs"]):
        lines.append(f"  o{k} = {ref(r)};")
    lines.append("}")
    return "\n".join(lines)
