#!/usr/bin/env python
"""Benchmark of the hot path (BASELINE.json metric): graph-evals/s of an optimised
Aesara graph executed by the B200 backend, measured THROUGH THE DROP-IN BOUNDARY
(``aesara.function(..., mode=B200)`` -> ``Function.__call__`` -> ``B200VM`` -> C ABI -> CUDA),
with the roofline of its dominant kernels and the reference's own C-linker timed beside it.

    python bench.py --gpus 1 --steps 10 --warmup 3                 # headline: cfg3 MLP fwd+grad
    python bench.py --workload elemwise|lstm|logreg|readme          # the other BASELINE configs
    python bench.py --impl reference                                # the reference C-linker on the host
    torchrun --nproc-per-node N bench.py --gpus N ...               # weak scaling over batch rows

A "step" is one call of the compiled function on one batch of synthetic inputs.
``value``: device-resident inputs (``trust_input``), outputs left on the device, the
evaluation replayed as one CUDA graph.  ``device_ms`` / ``roofline``: a second timed region
of the same K steps launched eagerly with CUDA events around every node.  ``e2e``: the call a
user makes -- page-locked host ndarrays in, host ndarrays out, copies inside the timed region.
The front-end the plugin sits behind (graph builder + rewriter) is whichever ``aesara`` is
importable; on the GPU box that is the travelling copy of the reference (``oracle/_ref``),
used as the host of the plugin and as the CPU arm, never as a compute fallback.
"""

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
PRECISIONS = {"fp32": 0, "tf32": 1, "bf16": 2}
TOLERANCE = {"fp32": 1e-5, "tf32": 2e-3, "bf16": 2e-2}
E2E_CHUNKS = int(os.environ.get("AB_E2E_CHUNKS", "8"))


# ----------------------------------------------------------------------------- workloads
def workload_spec(name, batch=0, hidden=0, n=0, steps_t=0):
    if name == "mlp":
        B, H = batch or 65536, hidden or 4096
        return dict(
            name="mlp", program="cfg3_mlp", graph="cfg3_mlp", B=B, H=H, rows="B",
            desc=f"cfg3: 2-layer tanh MLP fwd+grad (MSE), batch {B} x hidden {H}, f32 graph",
            gemm_flops=5 * 2.0 * B * H * H,            # SURVEY 8d: 5 GEMMs x 2BH^2
            n_gemm=5, shard_inputs=(0, 1), outputs=("loss", "dW1", "db1", "dW2", "db2"),
        )
    if name == "elemwise":
        n = n or (1 << 28)
        return dict(
            name="elemwise", program="cfg2_fused", graph="cfg2_fused_elemwise", n=n, rows="n",
            desc=f"cfg2: fused Elemwise softplus(tanh(x)+y)*z on 3x{n} f32",
            gemm_flops=0.0, n_gemm=0, shard_inputs=(0, 1, 2), outputs=("out",),
        )
    if name == "lstm":
        T, B, H = steps_t or 128, batch or 8192, hidden or 1024
        return dict(
            name="lstm", program="cfg4_lstm", graph="cfg4_lstm_scan", T=T, B=B, H=H, rows="B",
            desc=f"cfg4: Scan LSTM cell, T={T} steps, batch {B}, hidden {H}, f32",
            gemm_flops=2.0 * T * B * H * 4 * H, n_gemm=T,      # SURVEY 8d: 8.80 TFLOP
            ideal_bytes=(T * B * 4 * H + 4 * B * H + H * 4 * H) * 4.0,  # 17.33 GB (x read once)
            outputs=("h_T", "c_T"),
        )
    if name == "logreg":
        N, D = n or (1 << 24), hidden or 512
        return dict(
            name="logreg", program="cfg5_logreg", graph="cfg5_logreg", N=N, D=D, rows="N",
            desc=f"cfg5: logistic-regression cost+grad, {N} rows x {D} f32 per GPU",
            gemm_flops=0.0, n_gemm=0, shard_inputs=(0, 1),
            graph_bytes=(2.0 * N * D + 12.0 * N) * 4,      # SURVEY 8d graph-as-optimised
            # single-pass row-region fusion (runtime/rowfuse.py): X once, y read by `1 - y` and
            # by the fused kernel, `1 - y` written and read back
            fused_bytes=(1.0 * N * D + 4.0 * N) * 4, outputs=("cost", "grad_w", "grad_b"),
        )
    if name == "readme":
        n = n or 1000
        return dict(
            name="readme", program="cfg1_readme", graph="cfg1_readme", n=n, rows=None,
            desc=f"cfg1: README a/a + (M+a).dot(v), {n}x{n} f64",
            gemm_flops=0.0, n_gemm=0, outputs=("d",),
        )
    raise SystemExit(f"unknown workload {name}")


def make_inputs_numpy(spec, rng, rows=None):
    """Seeded host inputs (SURVEY 8d definitions); ``rows`` replaces the batch extent."""
    if spec["name"] == "lstm":
        T, H = spec["T"], spec["H"]
        B = rows or spec["B"]
        x = rng.standard_normal((T, B, 4 * H), dtype=np.float32)
        U = (rng.standard_normal((H, 4 * H), dtype=np.float32) / np.sqrt(H)).astype(np.float32)
        return [x, np.zeros((B, H), np.float32), np.zeros((B, H), np.float32), U]
    if spec["name"] == "logreg":
        N, D = rows or spec["N"], spec["D"]
        X = rng.standard_normal((N, D), dtype=np.float32)
        y = (rng.random(N) < 0.5).astype(np.float32)
        w = (rng.standard_normal(D) * 0.01).astype(np.float32)
        return [X, y, w, np.float32(0.0)]
    if spec["name"] == "readme":
        n = spec["n"]
        return [np.float64(1.5), rng.standard_normal(n), rng.standard_normal((n, n))]
    if spec["name"] == "mlp":
        B, H = rows or spec["B"], spec["H"]
        X = rng.standard_normal((B, H), dtype=np.float32)
        Y = rng.standard_normal((B, H), dtype=np.float32)
        W1 = (rng.standard_normal((H, H), dtype=np.float32) / np.sqrt(H)).astype(np.float32)
        W2 = (rng.standard_normal((H, H), dtype=np.float32) / np.sqrt(H)).astype(np.float32)
        return [X, Y, W1, np.zeros(H, np.float32), W2, np.zeros(H, np.float32)]
    n = rows or spec["n"]
    return [rng.standard_normal(n, dtype=np.float32) for _ in range(3)]


def make_inputs_device(spec, seed, shared_seed=1234):
    """Synthetic inputs generated on the device.  Batch data is seeded per rank, parameters
    (weights) with ``shared_seed`` so that every rank holds the same replica."""
    import torch

    from aesara_b200.runtime.device import DeviceArray

    g = torch.Generator(device="cuda").manual_seed(seed)
    gp = torch.Generator(device="cuda").manual_seed(shared_seed)
    if spec["name"] == "mlp":
        B, H = spec["B"], spec["H"]
        X = torch.randn(B, H, device="cuda", generator=g)
        Y = torch.randn(B, H, device="cuda", generator=g)
        W1 = torch.randn(H, H, device="cuda", generator=gp) / H ** 0.5
        W2 = torch.randn(H, H, device="cuda", generator=gp) / H ** 0.5
        ts = [X, Y, W1, torch.zeros(H, device="cuda"), W2, torch.zeros(H, device="cuda")]
    elif spec["name"] == "lstm":
        T, B, H = spec["T"], spec["B"], spec["H"]
        x = torch.randn(T, B, 4 * H, device="cuda", generator=g)
        U = torch.randn(H, 4 * H, device="cuda", generator=gp) / H ** 0.5
        ts = [x, torch.zeros(B, H, device="cuda"), torch.zeros(B, H, device="cuda"), U]
    elif spec["name"] == "logreg":
        N, D = spec["N"], spec["D"]
        X = torch.randn(N, D, device="cuda", generator=g)
        y = (torch.rand(N, device="cuda", generator=g) < 0.5).float()
        w = torch.randn(D, device="cuda", generator=gp) * 0.01
        ts = [X, y, w]
        return [DeviceArray.from_torch(t) for t in ts] + [np.float32(0.0)], ts
    elif spec["name"] == "readme":
        n = spec["n"]
        v = torch.randn(n, device="cuda", generator=g, dtype=torch.float64)
        M = torch.randn(n, n, device="cuda", generator=g, dtype=torch.float64)
        ts = [v, M]
        return [np.float64(1.5)] + [DeviceArray.from_torch(t) for t in ts], ts
    else:
        ts = [torch.randn(spec["n"], device="cuda", generator=g) for _ in range(3)]
    return [DeviceArray.from_torch(t) for t in ts], ts


# ----------------------------------------------------------------------------- front-end
def front_end():
    """``aesara`` as the plugin sees it: an installed package, ``$AESARA_B200_REFERENCE``, or
    the travelling copy of the reference (oracle/_ref).  Returns the module or None."""
    from aesara_b200.compat import bootstrap

    if not bootstrap.available():
        from oracle import ref

        ref.activate()
    if not bootstrap.available():
        return None
    return bootstrap.load_aesara()


def graph_of(spec):
    from aesara_b200 import graphs as G

    return getattr(G, spec["graph"])()


class ProgramCallable:
    """Fallback when no front-end is importable: the committed lowered program run by the
    executor directly (what round 1 measured).  ``boundary`` in the JSON line says which."""

    def __init__(self, spec, precision, device_outputs, cuda_graph):
        from aesara_b200.ir import Program
        from aesara_b200.runtime.vm import ProgramExecutor

        prog = Program.load(os.path.join(GOLDEN, spec["program"] + ".json"))
        self.executor = ProgramExecutor(prog, precision=precision, host_outputs=not device_outputs)
        self.replay = None
        if cuda_graph:
            from aesara_b200.runtime.graph import GraphReplay

            self.replay = GraphReplay(self.executor)

    def __call__(self, *args):
        return (self.replay or self.executor)(*args)


def compile_b200(spec, precision, device_outputs, cuda_graph, shard=None, host_chunks=0):
    """-> (callable, executor, boundary).  The callable is an ``aesara`` ``Function`` linked
    by ``B200Linker`` when a front-end is available."""
    aesara = front_end()
    if aesara is None:
        pc = ProgramCallable(spec, PRECISIONS[precision], device_outputs, cuda_graph)
        if shard is not None:
            from aesara_b200 import shardplan
            from aesara_b200.shard import ShardedExecutor

            pc.executor = ShardedExecutor(pc.executor, shardplan.infer_sharded_inputs(pc.executor.program))
        return pc, pc.executor, "lowered program (no front-end importable)"
    import aesara_b200.linker as L

    i, o = graph_of(spec)
    kw = {}
    if shard is not None:
        kw["shard"] = shard
    if host_chunks:
        kw["host_chunks"] = host_chunks
    f = aesara.function(i, o, mode=L.mode(precision=precision, device_outputs=device_outputs,
                                          cuda_graph=cuda_graph, **kw), on_unused_input="ignore")
    if device_outputs:
        f.trust_input = True
    return f, f.vm.executor, "aesara.function(mode=B200) -> Function.__call__"


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nme, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def ncu_traffic(summary, kernel_substr):
    """DRAM bytes per launch (dram__bytes_read.sum + dram__bytes_write.sum) of the kernel from
    a committed ``ncu --set full`` summary under profiles/ (None if it is not there)."""
    path = os.path.join(ROOT, "profiles", summary)
    if not os.path.exists(path):
        return None
    unit = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    total, inside, seen = 0.0, False, 0
    for line in open(path):
        if line.startswith("kernel:"):
            if inside and seen == 2:
                break
            inside, total, seen = kernel_substr in line, 0.0, 0
        elif inside and ("dram__bytes_read.sum " in line or "dram__bytes_write.sum " in line):
            parts = line.split()
            total += float(parts[1]) * unit.get(parts[2], 1.0)
            seen += 1
    return total if seen == 2 else None


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return dict(hbm=d["hbm_gbs"], bf16=d.get("bf16_tflops_sustained", d["bf16_tflops"]),
                    bf16_burst=d["bf16_tflops"], src="measured (MEASURED_PEAKS.json)")
    return dict(hbm=6650.0, bf16=1400.0, bf16_burst=1590.0, src="fallback (B200_PROFILING.md)")


# ----------------------------------------------------------------------------- CPU arm
def _host_threads():
    n = os.cpu_count() or 1
    try:  # torchrun pins OMP_NUM_THREADS=1: give the BLAS under NumPy every host core back
        from threadpoolctl import threadpool_limits

        threadpool_limits(limits=n)
    except Exception:
        pass
    return n


def reference_leg(spec, budget_s, want_steps=None):
    """The reference's OWN CPU implementation of the path: the same symbolic graph compiled by
    the unmodified reference (oracle/_ref) with its C-linker, ``Mode("cvm", "fast_run")``
    (aesara/link/vm.py:1057-1174, link/c/c_code/lazylinker_c.c), timed on the host cores with
    both OpenMP settings (BASELINE.md 3).  Full-size evaluations when they fit ``budget_s``,
    otherwise a stated row sample scaled per row.  Falls back to the NumPy oracle port when no
    reference copy travelled."""
    from oracle import ref

    cores = _host_threads()
    if ref.activate() is None:
        return port_leg(spec, budget_s)
    from aesara_b200.compat.bootstrap import load_aesara

    aesara = load_aesara()
    from aesara.compile.mode import Mode

    fns = {}
    for omp in (False, True):
        with aesara.config.change_flags(openmp=omp):
            i, o = graph_of(spec)
            f = aesara.function(i, o, mode=Mode("cvm", "fast_run"), on_unused_input="ignore")
        f.trust_input = True
        fns[omp] = f
    rng = np.random.default_rng(0)
    rows_key = spec["rows"]
    full = spec[rows_key] if rows_key else None

    def timed(f, ins, reps):
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            f(*ins)
            ts.append(time.perf_counter() - t0)
        return ts

    def prep(ins):
        # trust_input skips TensorType.filter: scalars must already be 0-d arrays
        return [np.asarray(a) for a in ins]

    t_start = time.perf_counter()
    if full is None:
        ins = prep(make_inputs_numpy(spec, rng))
        cal = {omp: min(timed(f, ins, 3)) for omp, f in fns.items()}
        best = min(cal, key=cal.get)
        n = want_steps or 20
        ts = timed(fns[best], ins, n)
        t = float(np.median(ts))
        return {"value": 1.0 / t, "unit": "graph-evals/s", "cores": cores, "kind": "reference",
                "sample": "full size", "steps_timed": n, "ms_per_eval": t * 1e3, "openmp": best,
                "openmp_false_ms": cal[False] * 1e3, "openmp_true_ms": cal[True] * 1e3,
                "linker": 'Mode("cvm", "fast_run")'}
    # calibrate on full/64 rows (at least 256), both OpenMP settings
    cal_rows = max(min(full, 256), full // 64)
    ins = prep(make_inputs_numpy(spec, rng, rows=cal_rows))
    cal = {}
    for omp, f in fns.items():
        f(*ins)
        cal[omp] = min(timed(f, ins, 2))
    best = min(cal, key=cal.get)
    f = fns[best]
    est_full = cal[best] * full / cal_rows
    left = budget_s - (time.perf_counter() - t_start)
    if est_full * 2.2 <= left:
        rows = full
    else:
        rows = cal_rows
        while rows * 2 <= full and est_full * (rows * 2 / full) * 3.2 <= left:
            rows *= 2
    if rows != cal_rows:
        ins = None
        ins = prep(make_inputs_numpy(spec, rng, rows=rows))
        f(*ins)  # warm-up at this size (allocations, page faults)
    per = est_full * rows / full
    left = budget_s - (time.perf_counter() - t_start)
    n = int(max(1, min(want_steps or 3, left / max(per, 1e-9))))
    ts = timed(f, ins, n)
    t = float(np.median(ts))
    scale = full / rows
    out = {"value": 1.0 / (t * scale), "unit": "graph-evals/s", "cores": cores, "kind": "reference",
           "sample": ("full size, un-extrapolated" if rows == full else
                      f"{rows} of {full} rows per evaluation; time scaled by {full}/{rows}"),
           "steps_timed": n, "ms_per_eval": t * scale * 1e3, "ms_per_eval_measured": t * 1e3,
           "openmp": best, "linker": 'Mode("cvm", "fast_run")',
           "calibration": {"rows": cal_rows, "openmp_false_ms": cal[False] * 1e3,
                           "openmp_true_ms": cal[True] * 1e3}}
    return out


def port_leg(spec, budget_s):
    """NumPy oracle port on a bounded row sample (used only when the reference copy is absent)."""
    from aesara_b200.ir import Program
    from oracle.program_np import run_program

    cores = _host_threads()
    prog = Program.load(os.path.join(GOLDEN, spec["program"] + ".json"))
    rng = np.random.default_rng(0)
    rows_key = spec["rows"]
    full = spec[rows_key] if rows_key else None
    rows = None if full is None else max(min(full, 256), full // 64)
    ins = make_inputs_numpy(spec, rng, rows=rows)
    run_program(prog, ins)
    ts = []
    t_end = time.perf_counter() + budget_s
    while len(ts) < 2 or (time.perf_counter() < t_end and len(ts) < 8):
        t0 = time.perf_counter()
        run_program(prog, ins)
        ts.append(time.perf_counter() - t0)
    scale = (full / rows) if rows else 1.0
    t = float(np.median(ts)) * scale
    return {"value": 1.0 / t, "unit": "graph-evals/s", "cores": cores, "kind": "port",
            "sample": "full size" if not rows else f"{rows} of {full} rows; time scaled by {full}/{rows}",
            "steps_timed": len(ts), "ms_per_eval": t * 1e3}


def run_reference_arm(args, spec, rank):
    if rank != 0:
        return
    # before libgomp is loaded by the first compiled module (torchrun exports OMP_NUM_THREADS=1)
    os.environ["OMP_NUM_THREADS"] = str(os.cpu_count() or 1)
    t0 = time.perf_counter()
    cb = reference_leg(spec, budget_s=150.0, want_steps=args.steps)
    v = cb["value"]
    line = {
        "impl": "reference", "metric": "graph-evals/s", "value": v, "unit": "graph-evals/s",
        "n_gpus": args.gpus, "steps": cb["steps_timed"], "steps_requested": args.steps,
        "warmup": 1, "ms_per_step": cb.get("ms_per_eval_measured", cb["ms_per_eval"]),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32" if spec["name"] != "readme" else "f64", "data": "synthetic",
        "config": {"workload": spec["desc"],
                   "note": ("the unmodified reference (oracle/_ref) through aesara.function with its "
                            "C-linker on the host cores; each step is " + cb["sample"])
                   if cb["kind"] == "reference" else
                   "oracle port (NumPy restatement); no reference copy travelled"},
        "cpu_baseline": cb, "wall_s": time.perf_counter() - t0,
        "e2e": {"value": v, "unit": "graph-evals/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ----------------------------------------------------------------------------- GPU arm
GEMM_OPS = ("Dot22", "Gemm", "Dot22Scalar", "Scan", "Dot", "BatchedDot")
HBM_OPS = ("Elemwise", "CAReduce", "Gemv", "Ger", "Softmax", "MaxAndArgmax")


def truth_check(spec, precision, outs, keep):
    """Measured error of THIS run's outputs against a float64 evaluation of the same inputs
    (tests/_truth.py: torch.float64 on the GPU, a checker outside every timed region)."""
    import torch

    from tests._truth import logreg_truth, mlp_truth, nerr

    outs = outs if isinstance(outs, (list, tuple)) else [outs]
    host = [np.asarray(o.to_numpy() if hasattr(o, "to_numpy") else o) for o in outs]
    if spec["name"] == "mlp":
        H = spec["H"]
        blocks = [(0, 0), (H // 2, max(H // 2 - 128, 0))] if H >= 256 else []
        t = mlp_truth(*keep, blocks)
        loss, dW1, db1, dW2, db2 = host
        err = {"loss": abs(float(loss) - float(t["loss"])) / abs(float(t["loss"])),
               "db1": nerr(db1, t["db1"]), "db2": nerr(db2, t["db2"])}
        for nm, dev, tr in (("dW1", dW1, t["dW1"]), ("dW2", dW2, t["dW2"])):
            scale = float(np.max(np.abs(dev)))
            err[nm + "_blocks"] = max([float(np.max(np.abs(dev[r:r + 128, c:c + 128].astype(np.float64) - b.cpu().numpy()))) / scale
                                       for (r, c), b in zip(blocks, tr)] or [0.0])
        tol = TOLERANCE[precision]
    else:
        X, y, w = keep
        t = logreg_truth(X, y, w, 0.0)
        cost, gw, gb = host
        err = {"cost": abs(float(cost) - float(t["cost"])) / abs(float(t["cost"])), "grad_w": nerr(gw, t["grad_w"]),
               "grad_b": abs(float(gb) - float(t["grad_b"])) / max(abs(float(t["grad_b"])), float(t["grad_w"].abs().max()))}
        tol = 1e-5
    torch.cuda.synchronize()
    return {"vs": "float64 evaluation of the same inputs (torch.float64 checker, tests/_truth.py); norm-wise",
            "err": err, "max_err": max(err.values()), "stated_tolerance": tol, "within": max(err.values()) <= tol}


DUMP_BUDGET = 64 * 10 ** 6  # bytes of all files together, .npy headers included
NPY_HEADER_MAX = 4096       # np.save writes a header of at most this many bytes per file


def dump_outputs(outs, names, d):
    """Write the outputs of one step as ``d/<name>.npy`` (float32 / float64).  An output larger
    than its even share of DUMP_BUDGET (after the headers) is written as the flat elements at
    sorted positions drawn with ``np.random.default_rng(0)``, the same on every run."""
    from aesara_b200.runtime.device import DeviceArray

    outs = outs if isinstance(outs, (list, tuple)) else [outs]
    assert len(outs) == len(names), (len(outs), names)
    os.makedirs(d, exist_ok=True)
    share = (DUMP_BUDGET - NPY_HEADER_MAX * len(outs)) // len(outs)
    for name, o in zip(names, outs):
        a = np.asarray(o.to_numpy() if isinstance(o, DeviceArray) else o)
        if a.dtype not in (np.float32, np.float64):
            a = a.astype(np.float64)
        if a.nbytes > share:
            flat = a.reshape(-1)
            a = flat[np.sort(np.random.default_rng(0).integers(0, flat.size, share // flat.itemsize))]
        np.save(os.path.join(d, name + ".npy"), a)


def measure(spec, precision, steps, warmup, rank=0, world=1, dist=None, use_graph=True,
            node_region=True, e2e_steps=0, seed=1234, check_truth=False, dump_dir=None):
    """One workload on this rank's GPU.  Returns a dict of measurements (see main()).  With
    ``dump_dir`` the outputs of the last timed step are written there (dump_outputs)."""
    import torch

    from aesara_b200.runtime import lib
    from aesara_b200.runtime.device import DeviceArray

    L = lib.load()
    # N > 1: the row sharding and the combination of the outputs are the linker's
    # (mode(shard="rows")): derived from the graph, one process per GPU, NCCL all-reduces
    f, ex, boundary = compile_b200(spec, precision, device_outputs=True,
                                   cuda_graph=use_graph and (world == 1 or os.environ.get("AB_SHARD_GRAPH", "1") != "0"),
                                   shard="rows" if world > 1 else None)
    dev_in, keep = make_inputs_device(spec, seed=seed + rank)

    def step():
        return f(*dev_in)

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    last = None

    def timed_region(n):
        nonlocal last
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        e0.record()
        for _ in range(n):
            last = step()
        e1.record()
        barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device="cuda")
        if dist is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item() / n

    res = {"boundary": boundary}
    if check_truth and world == 1 and spec["name"] in ("mlp", "logreg"):
        res["parity"] = truth_check(spec, precision, step(), keep)
    if world > 1:
        plan = getattr(ex, "plan", None)
        res["shard_plan"] = None if plan is None else {
            "sharded_inputs": plan.sharded_inputs, "outputs": [list(o) for o in plan.outputs]}
    for _ in range(max(warmup, 3)):
        step()
    barrier()
    clocks = ClockSampler(torch.cuda.current_device())
    clocks.start()
    l0 = L.ab_launch_count()
    ms_step = timed_region(steps)
    launches = L.ab_launch_count() - l0
    if dump_dir is not None:
        # before the next call: a replayed graph writes every step into the same output buffers
        dump_outputs(last, spec["outputs"], dump_dir)
    last = None
    replay = getattr(getattr(f, "vm", None), "_replay", None) or getattr(f, "replay", None)
    replayed = bool(replay is not None and replay.replays)
    res.update(ms_per_step=ms_step, executor="cuda-graph replay" if replayed else "eager launches")

    # second timed region: the same K steps launched eagerly with CUDA events around every node
    per_node = {}
    ms_eager = None
    if node_region:
        vm = getattr(f, "vm", None)
        saved = None
        if vm is not None:
            saved, vm._replay = vm._replay, None
        elif hasattr(f, "replay"):
            saved, f.replay = f.replay, None
        ex.time_nodes = True
        step()
        stats_runs = []
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        l1 = L.ab_launch_count()
        e0.record()
        for _ in range(steps):
            step()
            stats_runs.append(ex.node_events)
        e1.record()
        barrier()
        launches_eager = L.ab_launch_count() - l1
        ms_eager = e0.elapsed_time(e1) / steps
        for evs in stats_runs:
            for i, a, b, nb in evs:
                d = per_node.setdefault(i, {"ms": [], "bytes": nb})
                d["ms"].append(a.elapsed_time(b))
        ex.time_nodes = False
        if vm is not None:
            vm._replay = saved
        elif hasattr(f, "replay"):
            f.replay = saved
        if replayed:
            launches = launches_eager  # a replayed graph re-issues the kernels captured once
    clk = clocks.stop()
    res.update(ms_per_step_eager=ms_eager, gpu_launches=int(launches), clocks=clk,
               fused_regions_run=ex.fused_regions_run)
    if world > 1:
        res["exchange"] = {"collectives_per_step": getattr(ex, "exchanges", None),
                           "issued_before_the_evaluation_finished": getattr(ex, "early_issued", None)}
        ex = getattr(ex, "ex", ex)  # the wrapped ProgramExecutor for the per-node statistics

    # per-kind device time and per-kernel HBM fractions from the per-node events
    prog = ex.program
    fused_gemm = {getattr(fu, "anchor", fu.last) for fu in ex._fusions
                  if type(fu).__name__ == "GemmEpilogueFusion" and not fu.broken}
    fused_any = {getattr(fu, "anchor", fu.last): fu for fu in ex._fusions}
    gemm_ms = hbm_ms = other_ms = 0.0
    hbm_nodes, gemm_nodes = [], []
    for i, d in sorted(per_node.items()):
        op = "Gemm" if i in fused_gemm else prog.nodes[i].op
        t = float(np.mean(d["ms"]))
        if op in GEMM_OPS:
            gemm_ms += t
            gemm_nodes.append({"node": i, "label": (prog.nodes[i].label or prog.nodes[i].op)[:60],
                               "fused_members": len(fused_any[i].members) if i in fused_any else 1,
                               "ms": round(t, 4)})
        elif op in HBM_OPS:
            hbm_ms += t
            label = prog.nodes[i].label or prog.nodes[i].op
            if i in fused_any:
                label = type(fused_any[i]).__name__ + ": " + label
            if t > 0.02:  # >20 us: a bandwidth figure means something
                hbm_nodes.append({"node": i, "label": label[:80], "ms": round(t, 4), "bytes": d["bytes"],
                                  "gbs": d["bytes"] / (t * 1e-3) / 1e9})
        else:
            other_ms += t
    res.update(device_ms={"gemm": gemm_ms, "elemwise_careduce": hbm_ms, "other": other_ms}, hbm_nodes=hbm_nodes,
               gemm_nodes=gemm_nodes)

    # end to end through the public call: pinned host inputs, H2D + eval + D2H of every output
    if e2e_steps and world == 1:
        host_in, h2d = [], 0
        for t in keep:
            h = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            h.copy_(t)
            host_in.append(h)
            h2d += h.numel() * h.element_size()
        template = [None if isinstance(a, DeviceArray) else a for a in dev_in]
        del keep[:]
        del dev_in[:]
        f = ex = None
        import gc

        gc.collect()
        torch.cuda.empty_cache()
        f2, ex2, _ = compile_b200(spec, precision, device_outputs=False, cuda_graph=False,
                                  host_chunks=E2E_CHUNKS)
        it = iter(host_in)
        host_args = [slot if slot is not None else next(it).numpy() for slot in template]

        def e2e_step():
            r = f2(*host_args)
            r = r if isinstance(r, (list, tuple)) else [r]
            return sum(np.asarray(a).nbytes for a in r)

        d2h = e2e_step()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(e2e_steps):
            e2e_step()
        b.record()
        torch.cuda.synchronize()
        e2e_ms = a.elapsed_time(b) / e2e_steps
        res["e2e"] = {"value": 1e3 / e2e_ms, "unit": "graph-evals/s", "h2d_bytes_per_step": h2d,
                      "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "steps": e2e_steps,
                      "call": "Function.__call__ with page-locked host ndarrays in, host ndarrays out",
                      "row_chunks": getattr(ex2, "chunks_run", 1),
                      "pipeline": ("mode(host_chunks=%d): rows uploaded and evaluated in blocks, the upload of one "
                                   "overlapping the evaluation of the previous (batch map proven by shardplan)"
                                   % E2E_CHUNKS) if getattr(ex2, "chunks_run", 1) > 1 else "whole batch"}
        del ex2
        del f2, host_args, host_in
    else:
        del keep[:]
        del dev_in[:]
        f = ex = None
    import gc

    gc.collect()
    torch.cuda.empty_cache()
    return res


def sharded_parity(spec, precision, rank, world, dist, rows_per_rank=2048):
    """Pre-flight of an N-GPU run: the combined outputs of the row-sharded function equal ONE
    GPU's evaluation of the concatenated batch (rank 0 gathers the shards and evaluates the
    unsharded function).  Reduced row count, full width.  Returns the worst norm-wise error."""
    import copy

    import torch

    from aesara_b200.runtime.device import DeviceArray

    small = copy.deepcopy(spec)
    if spec["rows"] is None:
        return None
    small[spec["rows"]] = rows_per_rank
    fs, exs, _ = compile_b200(small, precision, device_outputs=True, cuda_graph=False, shard="rows")
    dev_in, keep = make_inputs_device(small, seed=777 + rank)
    outs = fs(*dev_in)
    outs = outs if isinstance(outs, (list, tuple)) else [outs]
    plan = exs.plan
    # gather every rank's sharded inputs on every rank (small), concatenate along the axis
    full_in = []
    ti = iter(keep)
    for a, ax in zip(dev_in, plan.sharded_inputs):
        if not isinstance(a, DeviceArray):
            full_in.append(a)
            continue
        t = next(ti)
        if ax is None:
            full_in.append(a)
            continue
        parts = [torch.empty_like(t) for _ in range(world)]
        dist.all_gather(parts, t.contiguous())
        full_in.append(DeviceArray.from_torch(torch.cat(parts, dim=ax).contiguous()))
    err, checked = 0.0, 0
    if rank == 0:
        f1, _, _ = compile_b200(small, precision, device_outputs=True, cuda_graph=False)
        want = f1(*full_in)
        want = want if isinstance(want, (list, tuple)) else [want]
        for k, (g, w_, m) in enumerate(zip(outs, want, plan.outputs)):
            if m[0] not in ("sum", "mean", "rep"):
                continue
            g = np.asarray(g.to_numpy() if isinstance(g, DeviceArray) else g, np.float64)
            w_ = np.asarray(w_.to_numpy() if isinstance(w_, DeviceArray) else w_, np.float64)
            err = max(err, float(np.max(np.abs(g - w_)) / max(np.max(np.abs(w_)), 1e-30)))
            checked += 1
    t = torch.tensor([err], device="cuda", dtype=torch.float64)
    dist.broadcast(t, src=0)
    torch.cuda.synchronize()
    return {"vs": f"one GPU evaluating the concatenated batch ({rows_per_rank} rows per rank x {world})",
            "normwise_err": float(t.item()), "outputs_checked": checked,
            "tolerance": TOLERANCE[precision] if spec["n_gemm"] else 1e-5,
            "combine": [list(o) for o in plan.outputs]}


def roofline_of(spec, precision, m, peaks):
    """The roofline object of the dominant kernel family from one measure() result."""
    dm = m["device_ms"]
    if spec["n_gemm"]:
        t = dm["gemm"] if dm["gemm"] else m["ms_per_step"]
        ach = spec["gemm_flops"] / (t * 1e-3) / 1e12
        peak = peaks["bf16"] if precision == "bf16" else peaks["bf16"] / 2.0
        r = {"bound": "tensor",
             "kernel": ("ab_lstm_scan (persistent 2-CTA tcgen05 Scan kernel)" if spec["name"] == "lstm" else
                        "tcgen05 GEMM launches (+operand packs) of the Gemm/Dot22 nodes, consumer Elemwise fused in"),
             "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak,
             "peak_source": peaks["src"] + (" sustained bf16" if precision == "bf16"
                                            else "; tf32 = bf16/2 (nominal ratio)"),
             "traffic": None, "ms_per_step": t,
             "timed": "CUDA events around every node over the eager timed region"}
        if precision == "fp32":
            # fp32-faithful products issue three TF32 MMAs each
            r["mma_per_product"] = 3
            r["ceiling_3xtf32"] = peak / 3.0
            r["frac_of_3xtf32_ceiling"] = ach / (peak / 3.0)
        if spec["name"] == "lstm":
            r["hbm_ideal_gbs"] = spec["ideal_bytes"] / (t * 1e-3) / 1e9
        return r
    if spec["name"] == "readme":
        return {"bound": "hbm", "kernel": "launch-latency bound (24 MB working set in L2)", "achieved": None,
                "peak": peaks["hbm"], "unit": "GB/s", "frac": None, "traffic": None}
    t = dm["elemwise_careduce"] or m["ms_per_step"]
    single_pass = bool(spec.get("fused_bytes")) and m["fused_regions_run"] > 0
    if spec["name"] == "logreg":
        nbytes = spec["fused_bytes"] if single_pass else spec["graph_bytes"]
        kern = "ab_rowfused (single pass over X)" if single_pass else "Gemv + Elemwise + Sum, node by node"
    else:
        nbytes = sum(n["bytes"] for n in m["hbm_nodes"]) or 16.0 * spec["n"]
        kern = "ab_ew_flat_vec (generated fused Elemwise)"
    ach = nbytes / (t * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": kern, "achieved": ach, "peak": peaks["hbm"], "unit": "GB/s",
            "frac": ach / peaks["hbm"], "peak_source": peaks["src"], "traffic": None, "ms_per_step": t,
            "algorithmic_bytes": nbytes}


def private_caches():
    """Where the tree cannot be written, point the caches the benchmark fills at run time at a
    temporary directory: the JIT kernel cache becomes links to the cubins the build left in
    aesara_b200/_kcache (kernels compiled now are added beside them), and the front-end's
    C-linker compiles into an empty directory instead of oracle/_ref/compiledir.  A writable
    tree keeps both caches in place; they are git-ignored."""
    import atexit
    import shutil
    import tempfile

    def writable(p):
        while not os.path.exists(p):
            p = os.path.dirname(p)
        return os.access(p, os.W_OK)

    kcache = os.path.join(ROOT, "aesara_b200", "_kcache")
    compiledir = os.path.join(ROOT, "oracle", "_ref", "compiledir")
    move_k = not os.environ.get("AESARA_B200_CACHE") and not writable(kcache)
    move_c = (not os.environ.get("AESARA_B200_COMPILEDIR") and os.path.isdir(os.path.dirname(compiledir))
              and not writable(compiledir))
    if not (move_k or move_c):
        return
    d = tempfile.mkdtemp(prefix="aesara_b200_bench_")
    atexit.register(shutil.rmtree, d, True)
    if move_k:
        kc = os.path.join(d, "kernels")
        os.makedirs(kc)
        if os.path.isdir(kcache):
            for name in os.listdir(kcache):
                if name.endswith(".cubin"):
                    os.symlink(os.path.join(kcache, name), os.path.join(kc, name))
        os.environ["AESARA_B200_CACHE"] = kc
    if move_c:
        os.environ["AESARA_B200_COMPILEDIR"] = os.path.join(d, "compiledir")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps; with --impl reference at most this many, within a 150 s budget")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="mlp", choices=["mlp", "elemwise", "lstm", "logreg", "readme"])
    ap.add_argument("--steps-t", type=int, default=0, help="Scan length for --workload lstm")
    ap.add_argument("--graph", type=int, default=1, help="1/0: replay the evaluation as a CUDA graph for `value`")
    ap.add_argument("--precision", default=None, choices=list(PRECISIONS),
                    help="GEMM compute policy; default: bf16 for mlp (BASELINE cfg3), fp32 (3xTF32) otherwise")
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--hidden", type=int, default=0)
    ap.add_argument("--n", type=int, default=0)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-also", action="store_true", help="skip the one-liners of the other configs")
    ap.add_argument("--no-truth", action="store_true", help="skip the float64 parity check of the headline run")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32/float64, "
                         "64 MB in all: large outputs as a fixed sample of elements); not with --impl reference")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what the device path computed; --impl reference has no such outputs")
    private_caches()
    spec = workload_spec(args.workload, args.batch, args.hidden, args.n, args.steps_t)
    if args.precision is None:
        args.precision = "bf16" if args.workload == "mlp" else "fp32"
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference_arm(args, spec, rank)
        return

    import torch

    from aesara_b200.runtime import lib

    torch.cuda.set_device(local_rank)
    lib.check(lib.load().ab_init(local_rank))
    dist = None
    if world > 1:
        import torch.distributed as dist

        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    peaks = measured_peaks()
    parity = None
    if world > 1:
        parity = sharded_parity(spec, args.precision, rank, world, dist)
        if parity is not None and not parity["normwise_err"] <= 4 * parity["tolerance"]:
            raise SystemExit(f"sharded evaluation disagrees with the single-GPU one: {parity}")
    m = measure(spec, args.precision, args.steps, args.warmup, rank, world, dist,
                use_graph=bool(args.graph), e2e_steps=0 if args.no_e2e else args.steps,
                check_truth=not args.no_truth, dump_dir=args.dump_outputs if rank == 0 else None)
    ms_step = m["ms_per_step"]
    value = world * 1e3 / ms_step  # every rank evaluates its shard once per step
    roofline = roofline_of(spec, args.precision, m, peaks)

    # DRAM traffic of the dominant kernel, per launch, from the committed ncu --set full summary
    tsrc = None
    if spec["name"] == "mlp" and args.precision == "bf16":
        tsrc = ("r02_bench_step_ncu_v4.txt", "ab_gemm_ep_2cta_f16")  # first launch of the capture: region 3
    elif spec["name"] == "logreg" and m["fused_regions_run"] > 0:
        tsrc = ("r01_rowfused_logreg.txt", "ab_rowfused")
    elif spec["name"] == "elemwise":
        tsrc = ("r01_elemwise_cfg2_v2_unroll1.txt", "ab_ew_flat_vec")
    if tsrc is not None:
        roofline["traffic"] = ncu_traffic(*tsrc)
        roofline["traffic_source"] = f"profiles/{tsrc[0]} ({tsrc[1]}, dram__bytes_read.sum + dram__bytes_write.sum per launch)"

    also = None
    if rank == 0 and world == 1 and not args.no_also and args.workload == "mlp":
        # the other BASELINE configs and the fp32-faithful policy, a few steps each, so that the
        # driver's record carries them (value, ms, roofline fraction)
        also = {}
        todo = [("mlp_fp32_faithful", workload_spec("mlp", args.batch, args.hidden), "fp32", 3),
                ("elemwise_cfg2", workload_spec("elemwise"), "fp32", 10),
                ("lstm_cfg4", workload_spec("lstm"), "fp32", 3),
                ("logreg_cfg5", workload_spec("logreg"), "fp32", 10),
                ("readme_cfg1", workload_spec("readme"), "fp32", 50)]
        for key, sp, prec, k in todo:
            try:
                mm = measure(sp, prec, k, 3, use_graph=True, check_truth=not args.no_truth)
                rr = roofline_of(sp, prec, mm, peaks)
                also[key] = {"workload": sp["desc"], "ms_per_step": mm["ms_per_step"],
                             "value": 1e3 / mm["ms_per_step"], "steps": k, "executor": mm["executor"],
                             "bound": rr["bound"], "achieved": rr["achieved"], "unit": rr["unit"],
                             "frac": rr.get("frac"), "kernel": rr["kernel"],
                             "frac_of_3xtf32_ceiling": rr.get("frac_of_3xtf32_ceiling"),
                             "gpu_launches": mm["gpu_launches"],
                             "parity_max_err": (mm.get("parity") or {}).get("max_err")}
            except Exception as e:  # an auxiliary line must not take the headline down
                also[key] = {"error": f"{type(e).__name__}: {e}"[:300]}

    if rank == 0:
        cb = None if args.no_cpu else reference_leg(spec, budget_s=30.0)
        if world == 1:
            par = "single"
        else:
            par = (f"dp{world} (batch rows sharded; outputs combined by one NCCL collective over the "
                   "packed outputs: all-reduce when large, all-gather + local weighted sum when small)")
        line = {
            "metric": "graph-evals/s", "value": value, "unit": "graph-evals/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"bf16": "bf16", "tf32": "tf32", "fp32": "f32 (3xTF32)"}[args.precision]
            if spec["n_gemm"] else ("f64" if spec["name"] == "readme" else "f32"),
            "data": "synthetic",
            "config": {"workload": spec["desc"], "parallelism": par, "boundary": m["boundary"],
                       "l2": ("working set fits L2: launch-latency bound, reported as evals/s only"
                              if spec["name"] == "readme" else "inputs >> 126 MB L2, no flush needed"),
                       "executor": m["executor"],
                       "gemm_precision": args.precision if spec["n_gemm"] else None,
                       "stated_tolerance": (f"norm-wise rtol {TOLERANCE[args.precision]} vs the reference "
                                            "C-linker (tests/test_gpu_parity.py, tests/test_gpu_function.py)")
                       if spec["n_gemm"] else "rtol 1e-5 vs the reference C-linker",
                       "per_gpu": {k: spec[k] for k in ("B", "H", "n", "N", "D", "T") if k in spec}},
            "roofline": roofline,
            "hbm_kernels": [dict(n, frac=n["gbs"] / peaks["hbm"]) for n in m["hbm_nodes"]],
            "gemm_nodes": m["gemm_nodes"],
            "device_ms": m["device_ms"], "ms_per_step_eager": m["ms_per_step_eager"],
            "cpu_baseline": cb, "e2e": m.get("e2e"), "gpu_launches": m["gpu_launches"],
            "clocks": m["clocks"], "parity": m.get("parity"), "also": also,
        }
        if world > 1:
            line["parity_sharded"] = parity
            line["shard_plan"] = m.get("shard_plan")
            line["exchange"] = m.get("exchange")
        print(json.dumps(line))
    if dist is not None:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
