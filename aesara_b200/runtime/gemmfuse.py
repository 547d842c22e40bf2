"""GEMM-epilogue regions: ``Dot22``/``Gemm``/``Dot22Scalar`` followed by the ``Elemwise`` nodes
that consume the product — and the ``Sum`` nodes that consume *those* — run as a single
tcgen05 kernel whose epilogue evaluates the merged scalar program of the Elemwise nodes
(``codegen/gemm_epilogue.py``, ``csrc/ab_gemm_tcgen05_kernel.cuh``).

In BASELINE config 3 (SURVEY App. A.3) the regions are

* ``Dot22(X, W1)`` -> ``tanh(. + b1)``                                             (h)
* ``Gemm(Y, 1, h, W2, -1)`` -> ``. + b2`` (diff) -> ``2*diff/n`` (dout), ``Sqr(diff)`` ->
  ``Sum`` (loss), ``Sum{axis=0}(dout)`` (db2)
* ``Dot22(dout, W2.T)`` -> ``. * (1 - h**2)`` (dpre) -> ``Sum{axis=0}(dpre)`` (db1)

i.e. every [B, H] intermediate between a product and the next one, which the reference's
node-by-node execution writes and re-reads (``tensor/blas.py:872/1659`` then
``tensor/elemwise.py:835`` and ``:1221``).  A value nobody outside the region reads (diff) is
never stored; a value only the next products read (dout, dpre under the bf16 policy) is stored
as the bf16 operand plane alone; column sums and totals are accumulated in float64 per
32-row block inside the epilogue and added up by a second, deterministic pass of the ordinary
CAReduce kernel.

Like ``rowfuse.RowFusion`` this is an executor-level region: the lowered program is not
changed.  The member nodes are skipped and the region runs at its *anchor* — the first member
position at which every operand the region reads exists (a later member's operand may be
produced after the GEMM node, e.g. the ``1/n`` factor of the loss gradient); every reader
outside the region comes after the anchor.  Anything the fused kernel does not take (problem
too small for the tensor-core path, operands that do not broadcast over the [M, N] result,
misaligned operands) runs node by node as before.
"""

from __future__ import annotations

import os

import numpy as np

from ..codegen.gemm_epilogue import MAX_OPERANDS, MAX_OUTPUTS, gemm_region_source, merge_exprs
from . import lib as _lib
from .device import DeviceArray

GEMM_OPS = ("Dot22", "Gemm", "Dot22Scalar")


class EpilogueRequest:
    """What ``kernels.gemm`` needs to launch the fused variant (set on the executor by
    ``GemmEpilogueFusion.run`` for exactly one ``K.gemm`` call)."""

    def __init__(self, fusion, operands, out_plan, colsum, fullsum):
        self.fusion = fusion
        self.operands = operands          # DeviceArrays (2-D, broadcastable over [M, N])
        self.out_plan = out_plan          # per value: (store float32, write the bf16 plane, write the transposed plane)
        self.colsum = colsum              # the module accumulates column sums / a total
        self.fullsum = fullsum
        self.applied = False
        self.arrays = None                # per value: DeviceArray [M, N] (written iff stored)
        self.shadows = None               # per value: (torch buffer, pitch) or None
        self.tshadows = None              # per value: (torch buffer, pitch) of the TRANSPOSED plane or None
        self.colsum_ws = None             # DeviceArray float64 [row_blocks, N]
        self.fullsum_ws = None            # DeviceArray float64 [row_blocks * cols]


def _gemm_operands(node):
    return (node.inputs[2], node.inputs[3]) if node.op == "Gemm" else (node.inputs[0], node.inputs[1])


def _plane_users(program, v):
    """How tensor-core products read the row-major matrix ``v``: ``(natural, transposed)`` lists
    of GEMM node indices.  *natural*: the contraction runs along the columns of ``v`` (``v`` as
    the left operand, ``v.T`` as the right one) -- its bf16 plane is K-major as written.
    *transposed*: the contraction runs along the ROWS of ``v`` (``v`` as the right operand,
    ``v.T`` as the left one: both operands of a weight gradient ``X.T @ G``) -- K-major only
    in the transposed plane."""
    cons = getattr(program, "_ab_consumers", None)
    if cons is None:
        cons = {}
        for i, n in enumerate(program.nodes):
            for w in n.inputs:
                cons.setdefault(w, []).append(i)
        program._ab_consumers = cons
    nodes = program.nodes
    nat, tr = [], []
    for c in cons.get(v, []):
        cn = nodes[c]
        if cn.op in GEMM_OPS:
            xv, yv = _gemm_operands(cn)
            if xv == v:
                nat.append(c)
            if yv == v:
                tr.append(c)
        elif cn.op == "DimShuffle" and list(cn.params.get("new_order", [])) == [1, 0]:
            t = cn.outputs[0]
            for c2 in cons.get(t, []):
                n2 = nodes[c2]
                if n2.op in GEMM_OPS:
                    xv, yv = _gemm_operands(n2)
                    if xv == t:
                        tr.append(c2)
                    if yv == t:
                        nat.append(c2)
    return nat, tr


class GemmEpilogueFusion:
    def __init__(self, program, g, ew, reds, steps, operand_vars, out_values, out_vars, anchor,
                 consumers):
        self.program = program
        self.g = g
        self.e = ew[0]
        self.ew = ew                          # Elemwise members, evaluation order
        self.reds = reds                      # [(node index, "col" | "full", value index)]
        self.members = sorted([g] + ew + [r for r, _, _ in reds])
        self.first, self.last = g, self.members[-1]
        self.anchor = anchor
        self.steps = steps
        self.operand_vars = operand_vars      # memory operands of the merged program, ep_ptr order
        self.out_values = out_values          # refs ("val", s) of the values the program yields
        self.out_vars = out_vars              # their variable ids (None: reduction source only)
        self._consumers = consumers           # var -> external consumer node indices
        self.colsum = next((k for _, kind, k in reds if kind == "col"), -1)
        self.fullsum = next((k for _, kind, k in reds if kind == "full"), -1)
        self.shadow_consumer = any(v is not None and self._gemm_consumers(v) for v in out_vars)
        # the one value whose transposed bf16 plane the module can write (shares its registers
        # with the column sums, so it has to be that value when the region has column sums)
        cand = [k for k, v in enumerate(out_vars) if v is not None and _plane_users(program, v)[1]]
        if os.environ.get("AB_EP_NO_TPLANE") or (self.fullsum >= 0 and os.environ.get("AB_EP_TPLANE_NO_FULLSUM")):
            cand = []
        self.tplane = (self.colsum if self.colsum in cand else -1) if self.colsum >= 0 else (cand[0] if cand else -1)
        self.exact_sums = True                # set by the executor: float-pair sums (fp32-faithful policy)
        self.planes = True                    # set by the executor: bf16 operand planes exist (bf16 policy)
        self.broken = False
        self.f32_skipped = 0                  # values kept as a bf16 plane only (last run)
        self._src = None
        self._pre_op = -1
        self._handle = None

    # ------------------------------------------------------------------ analysis
    @staticmethod
    def detect(program, destroys, taken=()):
        if os.environ.get("AB_NO_GEMM_FUSE"):
            return []
        nodes = program.nodes
        consumers = {}
        for i, n in enumerate(nodes):
            for v in n.inputs:
                consumers.setdefault(v, []).append(i)
        producer = {v: i for i, n in enumerate(nodes) for v in n.outputs}
        wide = not os.environ.get("AB_GEMM_FUSE_SINGLE")
        found, used = [], set(taken)
        for g, n in enumerate(nodes):
            if n.op not in GEMM_OPS or g in used:
                continue
            f = GemmEpilogueFusion._grow(program, g, consumers, producer, destroys, used, wide)
            if f is not None:
                found.append(f)
                used.update(f.members)
        return found

    @staticmethod
    def _grow(program, g, consumers, producer, destroys, used, wide):
        nodes = program.nodes
        z = nodes[g].outputs[0]
        zv = program.vars[z]
        if zv.dtype != "float32" or zv.ndim != 2 or z in program.outputs:
            return None
        # candidate members in schedule order (producers precede consumers)
        cand = []
        vals = {z}
        for c in range(g + 1, len(nodes)):
            cn = nodes[c]
            if c in used or not any(v in vals for v in cn.inputs):
                continue
            if cn.op == "Elemwise" and GemmEpilogueFusion._absorbable(program, cn, vals):
                cand.append(c)
                vals.add(cn.outputs[0])
            elif cn.op == "CAReduce" and wide and GemmEpilogueFusion._reducible(program, cn):
                cand.append(c)
            if not wide and cand:
                break
        # largest prefix of the candidates that forms a legal region
        while cand:
            f = GemmEpilogueFusion._build(program, g, cand, consumers, producer, destroys)
            if f is not None:
                return f
            cand.pop()
        return None

    @staticmethod
    def _absorbable(program, en, vals):
        if len(en.outputs) != 1:
            return False
        expr = en.params["expr"]
        ov = program.vars[en.outputs[0]]
        if ov.dtype != "float32" or ov.ndim != 2 or any(dt != "float32" for dt in expr["inputs"]):
            return False
        return all(program.vars[v].kind == "tensor" and program.vars[v].ndim == 2 for v in en.inputs)

    @staticmethod
    def _reducible(program, rn):
        p = rn.params
        if p.get("scalar_op") != "add" or p.get("in_dtype") != "float32" or p.get("acc_dtype") != "float64":
            return False
        return sorted(p.get("axis") or []) in ([0], [0, 1])

    @staticmethod
    def _build(program, g, cand, consumers, producer, destroys):
        nodes = program.nodes
        z = nodes[g].outputs[0]
        ew = [c for c in cand if nodes[c].op == "Elemwise"]
        if not ew:
            return None
        # merged program: steps + operand list
        val_of = {z: ("acc",)}
        steps, operand_vars = [], []
        for s, c in enumerate(ew):
            cn = nodes[c]
            refs = []
            for v in cn.inputs:
                if v in val_of:
                    refs.append(val_of[v])
                else:
                    if v not in operand_vars:
                        operand_vars.append(v)
                    refs.append(("op", operand_vars.index(v)))
            steps.append((cn.params["expr"], refs))
            val_of[cn.outputs[0]] = ("val", s)
        if len(operand_vars) > MAX_OPERANDS:
            return None
        member_set = set([g] + cand)
        # reductions: at most one per kind, source must be a region value (not the raw product)
        reds, red_src = [], {}
        for c in cand:
            cn = nodes[c]
            if cn.op != "CAReduce":
                continue
            src = cn.inputs[0]
            if val_of.get(src, ("acc",))[0] != "val":
                return None
            kind = "col" if sorted(cn.params["axis"]) == [0] else "full"
            if kind in red_src:
                return None
            red_src[kind] = (c, src)
        ext = {}
        for v in val_of:
            ext[v] = [c for c in consumers.get(v, []) if c not in member_set]
        if ext[z]:
            return None  # the raw product is read outside the region
        out_values, out_vars = [], []
        for v, ref in val_of.items():
            if ref[0] == "val" and (ext[v] or v in program.outputs):
                out_values.append(ref)
                out_vars.append(v)
        for kind, (c, src) in red_src.items():
            ref = val_of[src]
            if ref not in out_values:
                out_values.append(ref)
                out_vars.append(None)
            reds.append((c, kind, out_values.index(ref)))
        if not 1 <= len(out_values) <= MAX_OUTPUTS:
            return None
        # every Elemwise member's value must be used by somebody (inside or outside)
        # anchor: first member after the last producer of an external input
        ext_inputs = [v for v in nodes[g].inputs] + list(operand_vars)
        lo = max([producer.get(v, -1) for v in ext_inputs] + [-1])
        later = [m for m in sorted(member_set) if m > lo]
        if not later:
            return None
        anchor = later[0]
        if anchor < g:
            return None
        readers = [c for v in val_of for c in ext[v]]
        for c, _kind, _k in reds:
            readers += [r for r in consumers.get(nodes[c].outputs[0], []) if r not in member_set]
        if any(r <= anchor for r in readers):
            return None
        # the GEMM is deferred to the anchor: nothing outside the region may rewrite memory in between
        if any(destroys[i] for i in range(g + 1, anchor) if i not in member_set):
            return None
        return GemmEpilogueFusion(program, g, ew, reds, steps, operand_vars, out_values, out_vars,
                                  anchor, ext)

    # ------------------------------------------------------------------ helpers
    def _gemm_consumers(self, v):
        """External GEMM nodes that read value ``v`` as a matrix operand (directly or through a
        DimShuffle{1,0} view)."""
        nodes = self.program.nodes
        out = []
        for c in self._consumers.get(v, []):
            cn = nodes[c]
            if cn.op in GEMM_OPS and v in _gemm_operands(cn):
                out.append(c)
        return out

    def _plane_only_ok(self, ex, env, v, shape):
        """True when every reader of ``v`` outside the region is a tensor-core product that takes
        the bf16 operand plane (so the float32 matrix need not be written)."""
        prog = self.program
        nodes = prog.nodes
        if v in prog.outputs or ex.trace is not None or os.environ.get("AB_EP_KEEP_F32"):
            return False
        lib = _lib.load()
        for c in self._consumers.get(v, []):
            cn = nodes[c]
            if cn.op not in GEMM_OPS:
                return False
            xv, yv = _gemm_operands(cn)
            if cn.inputs.count(v) != (xv == v) + (yv == v):
                return False  # also read as the z of a Gemm
            shapes = []
            for w in (xv, yv):
                if w == v:
                    shapes.append(tuple(shape))
                else:
                    a = env.get(w)
                    if not isinstance(a, DeviceArray) or a.ndim != 2 or a.dtype != np.float32:
                        return False
                    shapes.append(a.shape)
            (m, k), (k2, n) = shapes
            if k != k2 or not lib.ab_gemm_tensorcore_eligible(m, n, k):
                return False
        return True

    # ------------------------------------------------------------------ execution
    def source(self):
        if self._src is None:
            names = "+".join(st[0].get("name", "?") for st in self.steps)
            merged = merge_exprs(self.steps, len(self.operand_vars), self.out_values, name=names)
            prog = self.program
            # the operand that is a whole matrix (not known to broadcast along rows): read ahead
            pre_op = -1
            for k, v in enumerate(self.operand_vars):
                ss = prog.vars[v].static_shape
                c = prog.vars[v].const
                if c is None and not (ss is not None and len(ss) == 2 and ss[0] == 1):
                    pre_op = k
                    break
            self._src = gemm_region_source(merged, len(self.operand_vars), self.colsum, self.fullsum,
                                           cin=prog.nodes[self.g].op == "Gemm", pre_op=pre_op,
                                           tplane=self.tplane if self.planes else -1,
                                           exact_sums=self.exact_sums, row_mask=self._kind_mask("row"),
                                           scalar_mask=self._kind_mask("scalar"))
            self._pre_op = pre_op
        return self._src

    def _kind_mask(self, kind):
        """Operands whose shape is known statically: ``row`` = [1, N] with N unknown or > 1 (a
        bias), ``scalar`` = [1, 1]."""
        mask = 0
        for k, v in enumerate(self.operand_vars):
            ss = self.program.vars[v].static_shape
            if ss is not None and len(ss) == 2 and ss[0] == 1 and (ss[1] == 1) == (kind == "scalar"):
                mask |= 1 << k
        return mask

    def _operands_fit(self, ops, M, N):
        """The module was generated for these operand shapes: the read-ahead matrix is [M, N]
        and the row operands are [1, N], both with unit column stride."""
        self.source()
        rows = self._kind_mask("row")
        for k, a in enumerate(ops):
            want = (M, N) if k == self._pre_op else ((1, N) if (rows >> k) & 1 else None)
            if want is not None and (a.shape != want or (N > 1 and a.strides[1] != 1)):
                return False
        return True

    def compile_all(self):
        _lib.compile_cubin(self.source(), "gemm_ep")
        return 1

    def handle(self):
        if self._handle is None:
            self._handle = _lib.load_module(self.source(), "gemm_ep")
        return self._handle

    def run(self, ex, env):
        from . import kernels as K
        from .vm import _EXEC, _as_dev_inputs
        from ..ir import Node

        if self.broken:
            return False
        prog = self.program
        nodes = prog.nodes
        gn = nodes[self.g]
        gargs = [env[v] for v in gn.inputs]
        x, y = (gargs[0], gargs[1]) if gn.op != "Gemm" else (gargs[2], gargs[3])
        if not (isinstance(x, DeviceArray) and isinstance(y, DeviceArray)):
            return False
        M, N = x.shape[0], y.shape[1]
        ops = _as_dev_inputs(ex, self.anchor, Node("Elemwise", list(self.operand_vars), []),
                             [env[v] for v in self.operand_vars])
        for a in ops:
            if a.dtype != np.float32 or a.ndim != 2 or a.shape[0] not in (1, M) or a.shape[1] not in (1, N):
                return False
        if not self._operands_fit(ops, M, N):
            return False
        plan = []
        for k, v in enumerate(self.out_vars):
            if v is None:
                plan.append((False, False, False))  # reduction source only
                continue
            planes = self.planes and ex.precision == 2 and N % 8 == 0
            nat_users, t_users = _plane_users(prog, v)
            tshadow = planes and k == self.tplane and bool(t_users)
            # products that contract over the rows of v and find no transposed plane read the
            # natural one as an MN-major operand
            shadow = planes and (bool(nat_users) or (bool(t_users) and not tshadow))
            store = not ((shadow or tshadow) and self._plane_only_ok(ex, env, v, (M, N)))
            plan.append((store, shadow, tshadow))
        req = EpilogueRequest(self, ops, plan, self.colsum >= 0, self.fullsum >= 0)
        ex._gemm_epilogue = req
        try:
            out = _EXEC[gn.op](ex, self.g, gn, gargs)
        except _lib.AbError:
            # the fused launch was refused (alignment, driver limits): never try again here
            self.broken = True
            ex._gemm_epilogue = None
            return False
        finally:
            ex._gemm_epilogue = None
        if not req.applied:
            # the product took another path (SIMT / too small): finish node by node
            env[gn.outputs[0]] = out
            ex._run_nodes([m for m in self.members if m != self.g], env)
            return True
        self.f32_skipped = 0
        for k, v in enumerate(self.out_vars):
            if v is None:
                continue
            env[v] = req.arrays[k]
            if req.shadows[k] is not None:
                ex.pack_cache.adopt(req.arrays[k], *req.shadows[k])
            if req.tshadows[k] is not None:
                ex.pack_cache.adopt(req.arrays[k], *req.tshadows[k], transposed=True)
            if not plan[k][0]:
                self.f32_skipped += 1
                ex.pack_cache.never_stored(req.arrays[k])
        for c, kind, _k in self.reds:
            rn = nodes[c]
            ws = req.colsum_ws if kind == "col" else req.fullsum_ws
            kern = K.CAReduceKernel.get("add", "float64", "float64", rn.params["out_dtype"])
            res = kern.launch(ws, (0,))
            if kind == "full":
                res = res.reshape_view(()) if res.ndim else res
            env[rn.outputs[0]] = res
        return True
