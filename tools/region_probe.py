#!/usr/bin/env python
"""The three fused GEMM-epilogue regions of cfg3 (bf16 policy, B = 65536, H = 4096) against the
plain tcgen05 GEMM of each region's shape, which is the floor a region's epilogue can hide under.

    python tools/region_probe.py [--iters N]   # B200: ms per launch, one JSON line
    python tools/region_probe.py --sass        # no GPU: SASS instructions of each region's chunk loop

GPU mode runs one eager step of the cfg3 program, keeps the arguments of the three fused
``K.gemm`` calls, then launches each of them and each plain product back to back, ``--iters`` times
between CUDA events, three interleaved rounds, best round.  The fused time includes only the
GEMM launch, not the second pass that adds up the column sums.  The JSON line also has the card's
name, power limit and SM clock, read in the same process.  The working set, about 1.5 GB per
launch, is much larger than L2.

``--sass`` compiles the regions' NVRTC modules, as ``build()`` does, and disassembles
``ab_gemm_ep_2cta_f16`` with ``cuobjdump``.  A chunk loop is a backward branch whose body holds
the ``LDTM`` (tcgen05.ld) of the chunk.  These are static counts that show progress, not timings.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

KERNEL = "ab_gemm_ep_2cta_f16"  # the fused kernel cfg3 launches (2-CTA pairs, bf16 operands)


def regions(precision=2):
    from aesara_b200.ir import Program
    from aesara_b200.runtime.vm import ProgramExecutor

    prog = Program.load(os.path.join(ROOT, "tests", "golden", "cfg3_mlp.json"))
    ex = ProgramExecutor(prog, precision=precision)
    fus = sorted((f for f in ex._fusions if type(f).__name__ == "GemmEpilogueFusion"), key=lambda f: f.g)
    return prog, ex, fus


def chunk_loops(sass):
    """[(first, last, instructions)] of the innermost backward-branch loops around an LDTM."""
    ins = []  # (offset, text)
    for line in sass.splitlines():
        m = re.match(r"\s*/\*([0-9a-f]{4,})\*/\s+(.*?)\s*;", line)
        if m:
            ins.append((int(m.group(1), 16), m.group(2)))
    off_idx = {o: i for i, (o, _) in enumerate(ins)}
    ldtm = [i for i, (_, t) in enumerate(ins) if re.search(r"\bLDTM\b", t)]
    loops = []
    for i, (o, t) in enumerate(ins):
        m = re.search(r"\bBRA\b.*?`?\(?\.L_x_\d+\)?|\bBRA\b\s+(0x[0-9a-f]+)", t)
        if not m:
            continue
        tgt = re.search(r"0x([0-9a-f]+)", t.split("BRA", 1)[1])
        if not tgt:
            continue
        j = off_idx.get(int(tgt.group(1), 16))
        if j is None or j > i:
            continue
        if any(j <= k <= i for k in ldtm):
            loops.append((j, i))
    inner = [(a, b) for a, b in loops if not any(a <= c and d <= b and (c, d) != (a, b) for c, d in loops)]
    out = []
    for a, b in sorted(set(inner)):
        body = [t for _, t in ins[a:b + 1]]
        out.append({"instructions": len(body), "per_element": round(len(body) / 32.0, 2),
                    "BRA": sum(1 for t in body if re.search(r"\bBRA\b", t)),
                    "LDC": sum(1 for t in body if re.search(r"\bLDCU?\b", t)),
                    "MUFU": sum(1 for t in body if "MUFU" in t),
                    "local": sum(1 for t in body if re.search(r"\b(LDL|STL)\b", t))})
    return out


def sass_counts():
    from aesara_b200.runtime import lib

    lib.load()
    res = {}
    for k, f in enumerate(regions()[2]):
        cubin = lib.compile_cubin(f.source(), "gemm_ep")
        with tempfile.NamedTemporaryFile(suffix=".cubin") as tf:
            tf.write(cubin)
            tf.flush()
            sass = subprocess.run(["cuobjdump", "-sass", "-fun", KERNEL, tf.name], capture_output=True,
                                  text=True, check=True).stdout
            usage = subprocess.run(["cuobjdump", "-res-usage", tf.name], capture_output=True, text=True).stdout
        m = re.search(rf"Function {KERNEL}:\s*\n\s*REG:(\d+) STACK:(\d+)", usage)
        res[f"region{k + 1}"] = {"kernel": KERNEL, "chunk_loops": chunk_loops(sass),
                                 "reg": int(m.group(1)) if m else None, "stack": int(m.group(2)) if m else None}
    return res


def gpu_info():
    import torch

    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm,clocks_throttle_reasons.active",
                            "--format=csv,noheader", "-i", "0"], capture_output=True, text=True, timeout=30).stdout
        info["nvidia_smi"] = q.strip()
    except (OSError, subprocess.SubprocessError) as e:
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def gpu_probe(iters, B=65536, H=4096):
    import torch

    from aesara_b200.runtime import kernels as K
    from aesara_b200.runtime import lib
    from aesara_b200.runtime.device import DeviceArray

    lib.check(lib.load().ab_init(0))
    torch.cuda.set_device(0)
    prog, ex, fus = regions()
    g = torch.Generator(device="cuda").manual_seed(1234)
    ts = [torch.randn(B, H, device="cuda", generator=g), torch.randn(B, H, device="cuda", generator=g),
          torch.randn(H, H, device="cuda", generator=g) / H ** 0.5, torch.zeros(H, device="cuda"),
          torch.randn(H, H, device="cuda", generator=g) / H ** 0.5, torch.zeros(H, device="cuda")]
    ins = [DeviceArray.from_torch(t) for t in ts]
    calls = []
    real_gemm = K.gemm

    def spy(*a, **kw):
        if kw.get("epilogue") is not None:
            calls.append((a, dict(kw)))
        return real_gemm(*a, **kw)

    K.gemm = spy
    try:
        ex(*ins)
    finally:
        K.gemm = real_gemm
    torch.cuda.synchronize()
    assert len(calls) == len(fus) == 3, f"expected the three cfg3 regions, saw {len(calls)} fused launches"

    def fused(i):
        a, kw = calls[i]
        return lambda: K.gemm(*a, **kw)

    X, D, W = ts[0], ts[1], ts[2]
    dX, dD, dW = DeviceArray.from_torch(X), DeviceArray.from_torch(D), DeviceArray.from_torch(W)
    C = DeviceArray.empty((B, H), "float32")
    cache = K.PackCache()
    plain = {
        "fwd  X[B,H] @ W[H,H]  (regions 1, 2)": lambda: K.gemm(C, 1.0, dX, dW, 0.0, precision=2, cache=cache),
        "dh   D[B,H] @ W.T     (region 3)": lambda: K.gemm(C, 1.0, dD, dW.dimshuffle([1, 0]), 0.0, precision=2,
                                                            cache=cache),
    }
    runs = {"region1 X@W1 -> tanh(.+b1)": fused(0), "region2 h@W2 -> +b2-Y, 2d/n, loss, db2": fused(1),
            "region3 g@W2.T -> g*(1-h^2), db1": fused(2), **plain}

    def time(fn):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(iters):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / iters

    info0 = gpu_info()
    best = {}
    names = list(runs)
    for rnd in range(3):
        for name in names[rnd:] + names[:rnd]:  # no launch is always first
            best[name] = min(best.get(name, 1e9), time(runs[name]))
    info1 = gpu_info()
    return {"probe": "region_probe", "B": B, "H": H, "iters": iters, "ms_per_launch": {k: round(v, 4) for k, v in best.items()},
            "gpu": info0["name"], "nvidia_smi_before": info0["nvidia_smi"], "nvidia_smi_after": info1["nvidia_smi"]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sass", action="store_true", help="static SASS counts of the chunk loops (no GPU)")
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    res = sass_counts() if args.sass else gpu_probe(args.iters)
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
