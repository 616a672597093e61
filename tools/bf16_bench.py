#!/usr/bin/env python
"""bf16 and fp16 features against fp32 features on the headline graph (BASELINE.json configs[4], bench.gen_rows):
50M nodes, ~976M stored entries, d = 128, 10 classes, Y = D^-1/2 (A+I) D^-1/2 X with the degree scale on the fly.

    python tools/bf16_bench.py [--reps 10] [--warmup 3] [--out profiles/f16_r06.json]

X is drawn in fp32 by the generator and cast to bf16 and to fp16 once; the fp32 arm reads Xb.float().  Timed in one
process with CUDA events, the arms alternating within every repetition:
    spmm_f32         fp32 X -> fp32 Y                          (wdgh_spmm_csr)
    spmm_bf16_f32    bf16 X -> fp32 Y                          (wdgh_spmm_csr_bf16)
    spmm_bf16_bf16   bf16 X -> bf16 Y
    spmm_f16_f32     fp16 X -> fp32 Y                          (wdgh_spmm_csr_f16)
    spmm_f16_f16     fp16 X -> fp16 Y
    step_bf16        degree scale + bf16 -> fp32 SpMM + label pass (the step bench.py times, with bf16 features)
    step_f32         the same step with fp32 features: bench.py's step (its spmm_structure_fused is wdgh_spmm_csr followed
                     by wdgh_structure_counts on one stream, the two launches made here; it has no bf16 form)
Per arm: median ms, GEdges/s (stored entries / time) and the algorithmic-bytes roofline fraction (bytes below, peak as
bench.py takes it).  After the timing, on the full graph: Y of the bf16 arms must be torch.equal to the fp32 call on
Xb.float() (fp32 output) and to its rounding to bf16 (bf16 output), Y of the fp16 arms likewise to the fp32 call on
Xh.float() and its rounding to fp16.  Prints one JSON line and writes it to --out.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "when-do-gnns-help_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

import bench  # noqa: E402


def spmm_bytes(nnz, n, d, x_bytes, y_bytes):
    """Algorithmic bytes of one aggregation (DESIGN.md section 4): per stored entry a 4 B column id, a 4 B scale gather
    and one feature row; per row 8 B rowptr, a 4 B scale, the self-loop feature row and the output row."""
    return nnz * (4 + 4 + x_bytes * d) + n * (8 + 4 + x_bytes * d + y_bytes * d)


def label_bytes(nnz, n):
    """the label pass as bench.time_label_pass counts it"""
    return nnz * 4 + n * (8 + 4 + 1 + 1 + 4 + 4)


def hbm_peak():
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        return float(mp["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def card(device):
    """name, power limit and max SM clock of the GPU the numbers were taken on (read-only query)"""
    try:
        uuid = str(torch.cuda.get_device_properties(device).uuid)
        sel = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
        out = subprocess.run(["nvidia-smi", "-i", sel, "--query-gpu=name,power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [v.strip() for v in out.split(",")]
        return {"name": name, "power_limit": power, "sm_max_clock": clock}
    except Exception as e:  # the numbers stay valid, the card is then unknown
        return {"name": torch.cuda.get_device_name(device), "power_limit": None, "error": str(e)}


def equal_rows(a, b, to=None, block=1 << 21):
    """torch.equal(a, b.to(to)) over row blocks (no full-size temporary)"""
    for r in range(0, a.shape[0], block):
        bb = b[r:r + block]
        if not torch.equal(a[r:r + block], bb if to is None else bb.to(to)):
            return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=50_000_000)
    ap.add_argument("--avg-degree", type=float, default=20.0)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--classes", type=int, default=10)
    ap.add_argument("--homophily", type=float, default=0.3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "f16_r06.json"))
    args = ap.parse_args()

    import wdgh_b200 as W
    from wdgh_b200 import graph as G

    W._lib.require_device()
    device = torch.device("cuda", torch.cuda.current_device())
    n, d, C = args.nodes, args.dim, args.classes
    rowptr, col, x, labels = bench.gen_rows(0, n, n, args.avg_degree, C, args.homophily, d, device)
    xb = x.to(torch.bfloat16)
    xh = x.to(torch.float16)
    del x
    x32 = xb.float()
    torch.cuda.empty_cache()
    nnz = int(col.shape[0])
    g = G.CSRGraph(rowptr, col, None, n)
    _ = g.plan
    dinv, _, code = g.degree_scale(W.NORM_SYM, True)
    # one fp32 and one 2-byte output buffer serve every half arm (the checks re-run each arm after the timing), so that
    # the five matrices of the full graph fit next to the three feature matrices
    y32 = torch.empty((n, d), dtype=torch.float32, device=device)
    yh32 = torch.empty((n, d), dtype=torch.float32, device=device)
    ybb = torch.empty((n, d), dtype=torch.bfloat16, device=device)
    yhh = ybb.view(torch.float16)
    ystep = yh32
    scratch = [None]

    def step(xx):
        g._dinv.clear()
        dv, _, cd = g.degree_scale(W.NORM_SYM, True)
        G.spmm(g, xx, W.NORM_SYM, True, out=ystep, dinv=dv, deg_code=cd)
        scratch[0] = G.structure_counts_raw(g, labels, C, scratch[0])

    arms = {
        "spmm_f32": lambda: G.spmm(g, x32, W.NORM_SYM, True, out=y32, dinv=dinv, deg_code=code),
        "spmm_bf16_f32": lambda: G.spmm(g, xb, W.NORM_SYM, True, out=yh32, dinv=dinv, deg_code=code),
        "spmm_bf16_bf16": lambda: G.spmm(g, xb, W.NORM_SYM, True, out=ybb, dinv=dinv, deg_code=code),
        "spmm_f16_f32": lambda: G.spmm(g, xh, W.NORM_SYM, True, out=yh32, dinv=dinv, deg_code=code),
        "spmm_f16_f16": lambda: G.spmm(g, xh, W.NORM_SYM, True, out=yhh, dinv=dinv, deg_code=code),
        "step_bf16": lambda: step(xb),
        "step_f32": lambda: step(x32),
    }
    for _ in range(args.warmup):
        for fn in arms.values():
            fn()
    torch.cuda.synchronize()
    ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.reps)]
          for k in arms}
    for r in range(args.reps):
        for k, fn in arms.items():
            ev[k][r][0].record()
            fn()
            ev[k][r][1].record()
    torch.cuda.synchronize()

    # every half arm once more against the fp32 call on the same values: bf16 first, then fp16 (x32 <- Xh.float())
    def check(arm16_f32, arm16_16, y16, dtype):
        arms["spmm_f32"]()
        arms[arm16_f32]()
        eq32 = equal_rows(yh32, y32)
        arms[arm16_16]()
        torch.cuda.synchronize()
        return eq32, equal_rows(y16, y32, to=dtype)

    eq_f32, eq_bf16 = check("spmm_bf16_f32", "spmm_bf16_bf16", ybb, torch.bfloat16)
    for r in range(0, n, 1 << 22):
        x32[r:r + (1 << 22)].copy_(xh[r:r + (1 << 22)])
    eq_f16_f32, eq_f16 = check("spmm_f16_f32", "spmm_f16_f16", yhh, torch.float16)

    peak, peak_src = hbm_peak()
    alg = {"spmm_f32": spmm_bytes(nnz, n, d, 4, 4), "spmm_bf16_f32": spmm_bytes(nnz, n, d, 2, 4),
           "spmm_bf16_bf16": spmm_bytes(nnz, n, d, 2, 2), "spmm_f16_f32": spmm_bytes(nnz, n, d, 2, 4),
           "spmm_f16_f16": spmm_bytes(nnz, n, d, 2, 2)}
    alg["step_bf16"] = alg["spmm_bf16_f32"] + label_bytes(nnz, n)
    alg["step_f32"] = alg["spmm_f32"] + label_bytes(nnz, n)
    res = {}
    for k in arms:
        times = [a.elapsed_time(b) for a, b in ev[k]]
        ms = statistics.median(times)
        res[k] = {"ms": ms, "ms_min": min(times), "ms_max": max(times), "gedges_s": nnz / (ms * 1e-3) / 1e9,
                  "algorithmic_bytes": alg[k], "achieved_gbs": alg[k] / (ms * 1e-3) / 1e9,
                  "frac": alg[k] / (ms * 1e-3) / 1e9 / peak}
    line = {"tool": "tools/bf16_bench.py", "nodes": n, "stored_entries": nnz, "dim": d, "classes": C,
            "norm": "sym D^-1/2 (A+I) D^-1/2 on the fly", "reps": args.reps, "warmup": args.warmup,
            "arms": res, "speedup_spmm_bf16_f32": res["spmm_f32"]["ms"] / res["spmm_bf16_f32"]["ms"],
            "speedup_spmm_bf16_bf16": res["spmm_f32"]["ms"] / res["spmm_bf16_bf16"]["ms"],
            "speedup_spmm_f16_f32": res["spmm_f32"]["ms"] / res["spmm_f16_f32"]["ms"],
            "speedup_spmm_f16_f16": res["spmm_f32"]["ms"] / res["spmm_f16_f16"]["ms"],
            "f16_f32_over_bf16_f32": res["spmm_f16_f32"]["ms"] / res["spmm_bf16_f32"]["ms"],
            "speedup_step": res["step_f32"]["ms"] / res["step_bf16"]["ms"],
            "equal_bf16_f32_vs_f32": eq_f32, "equal_bf16_bf16_vs_f32_rounded": eq_bf16,
            "equal_f16_f32_vs_f32": eq_f16_f32, "equal_f16_f16_vs_f32_rounded": eq_f16,
            "peak_gbs": peak, "peak_source": peak_src, "card": card(device)}
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    if not (eq_f32 and eq_bf16 and eq_f16_f32 and eq_f16):
        sys.exit(3)


if __name__ == "__main__":
    main()
