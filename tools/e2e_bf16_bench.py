#!/usr/bin/env python
"""Host-buffer pipeline (the e2e path) with bf16 and fp16 features against fp32 features on the headline graph
(BASELINE.json configs[4], bench.gen_rows): 50M nodes, ~976M stored entries, d = 128, 10 classes,
Y = D^-1/2 (A+I) D^-1/2 X.

    python tools/e2e_bf16_bench.py [--reps 5] [--warmup 1] [--out profiles/e2e_f16_r06.json]

X is drawn in fp32 by the generator and cast to bf16 and to fp16 once; the fp32 arms read Xb.float().  All inputs and
outputs live in pinned host memory (about 95 GB at full size; the bf16 and fp16 Y share one buffer).  Timed in one
process with a host clock around the synchronous call, the arms alternating within every repetition:
    e2e_f32          wdgh_pipeline_host, fp32 X, fp32 Y back          (what bench.py's e2e times)
    e2e_bf16_f32y    wdgh_pipeline_host_bf16, bf16 X, fp32 Y back
    e2e_bf16_bf16y   wdgh_pipeline_host_bf16, bf16 X, bf16 Y back
    e2e_f16_f32y     wdgh_pipeline_host_f16, fp16 X, fp32 Y back
    e2e_f16_f16y     wdgh_pipeline_host_f16, fp16 X, fp16 Y back
    counters_f32     wdgh_pipeline_host, fp32 X, counters only (y_host = NULL)
    counters_bf16    wdgh_pipeline_host_bf16, bf16 X, counters only
    counters_f16     wdgh_pipeline_host_f16, fp16 X, counters only
Per arm: median ms and spread, GEdges/s, H2D / D2H bytes and the effective link rate ((H2D + D2H) / time).
Checks in the same run: the counters of every arm are identical; on a seeded sample of rows, the fp32 Y of the half
features equals the fp32 Y of e2e_f32 on the same values (Xb.float(), then Xh.float()) exactly (every feature type
takes the same copy / compute form, whose phases are bit-identical), and the half Y equals the fp32 Y of the same
features rounded to nearest even.  Prints one JSON line, writes it to --out and exits non-zero when a check fails.
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "when-do-gnns-help_b200"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

import bench  # noqa: E402
from bf16_bench import card  # noqa: E402

HEADLINE_NODES = 50_000_000


def column_blocks(d):
    """True when the Y-returning arms copy X in 64-column blocks (csrc/pipeline_host.cu, schedule)"""
    return d % 64 == 0 and 2 <= d // 64 <= 64


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=HEADLINE_NODES)
    ap.add_argument("--avg-degree", type=float, default=20.0)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--classes", type=int, default=10)
    ap.add_argument("--homophily", type=float, default=0.3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--sample-rows", type=int, default=1 << 20)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "e2e_f16_r06.json"))
    args = ap.parse_args()

    import wdgh_b200 as W
    from wdgh_b200 import graph as G

    W._lib.require_device()
    device = torch.device("cuda", torch.cuda.current_device())
    n, d, C = args.nodes, args.dim, args.classes
    rowptr, col, x, labels = bench.gen_rows(0, n, n, args.avg_degree, C, args.homophily, d, device)
    nnz = int(col.shape[0])
    xb = x.to(torch.bfloat16)
    xh = x.to(torch.float16)
    del x

    def pinned(t, dtype=None):
        h = torch.empty(t.shape, dtype=dtype or t.dtype, pin_memory=True)
        for r in range(0, t.shape[0], 1 << 22):   # row blocks: no full-size device temporary for the fp32 copy
            h[r:r + (1 << 22)].copy_(t[r:r + (1 << 22)])
        return h

    try:
        rowptr_h, col_h = pinned(rowptr), pinned(col)
        lab_h = pinned(labels, torch.int32)
        xb_h, xh_h, x32_h = pinned(xb), pinned(xh), pinned(xb, torch.float32)
        y32_h = torch.empty((n, d), dtype=torch.float32, pin_memory=True)
        ybf_h = torch.empty((n, d), dtype=torch.bfloat16, pin_memory=True)
        yh_h = ybf_h.view(torch.float16)
    except RuntimeError as e:
        print(json.dumps({"tool": "tools/e2e_bf16_bench.py", "nodes": n,
                          "error": f"pinning the host buffers failed ({str(e)[:120]}); run again with a smaller --nodes"}),
              flush=True)
        sys.exit(2)
    del rowptr, col, labels, xb, xh
    torch.cuda.empty_cache()

    n_cnt = W._lib.sc_words(C)
    small_d2h = n_cnt * 8 + 16
    graph_h2d = (n + 1) * 8 + nnz * 4 + n * 4
    counters = {}

    def run(k, x_h, y_h):
        counters[k] = G.pipeline_host(rowptr_h, col_h, x_h, lab_h, C, W.NORM_SYM, True, y=y_h)

    arms = {
        "e2e_f32": (x32_h, y32_h),
        "e2e_bf16_f32y": (xb_h, y32_h),
        "e2e_bf16_bf16y": (xb_h, ybf_h),
        "e2e_f16_f32y": (xh_h, y32_h),
        "e2e_f16_f16y": (xh_h, yh_h),
        "counters_f32": (x32_h, None),
        "counters_bf16": (xb_h, None),
        "counters_f16": (xh_h, None),
    }
    for _ in range(args.warmup):
        for k, (xh, yh) in arms.items():
            run(k, xh, yh)
    times = {k: [] for k in arms}
    for _ in range(args.reps):
        for k, (xh, yh) in arms.items():
            t0 = time.perf_counter()
            run(k, xh, yh)
            times[k].append(time.perf_counter() - t0)

    # checks: counters of the last timed call of every arm; Y on a seeded row sample of one more call per Y arm
    ref_c, ref_s = counters["e2e_f32"]
    counters_equal = all((c == ref_c).all() and (s == ref_s).all() for c, s in counters.values())
    gen = torch.Generator().manual_seed(7)
    rows = torch.randint(0, n, (min(args.sample_rows, n),), generator=gen)

    def check(arm_f32y, arm_halfy, x_h, y_half_h):
        """(max abs error and equality of the half features' fp32 Y against e2e_f32 on x32_h, the half Y is its
        rounding, max |Y|) on the sample rows"""
        run("e2e_f32", x32_h, y32_h)
        y_f32 = y32_h[rows].clone()
        run(arm_f32y, x_h, y32_h)
        y_h32 = y32_h[rows].clone()
        run(arm_halfy, x_h, y_half_h)
        y_hh = y_half_h[rows].clone()
        return ((y_h32 - y_f32).abs().max().item(), torch.equal(y_h32, y_f32),
                torch.equal(y_hh, y_h32.to(y_half_h.dtype)), y_f32.abs().max().item())

    err, y_ok, bf16_ok, scale = check("e2e_bf16_f32y", "e2e_bf16_bf16y", xb_h, ybf_h)
    for r in range(0, n, 1 << 22):               # the fp32 arm on the fp16 values
        x32_h[r:r + (1 << 22)].copy_(xh_h[r:r + (1 << 22)])
    err16, y16_ok, f16_ok, _ = check("e2e_f16_f32y", "e2e_f16_f16y", xh_h, yh_h)
    W._lib.lib.wdgh_pipeline_host_release()

    x_bytes = {"e2e_f32": 4, "e2e_bf16_f32y": 2, "e2e_bf16_bf16y": 2, "e2e_f16_f32y": 2, "e2e_f16_f16y": 2,
               "counters_f32": 4, "counters_bf16": 2, "counters_f16": 2}
    y_bytes = {"e2e_f32": 4, "e2e_bf16_f32y": 4, "e2e_bf16_bf16y": 2, "e2e_f16_f32y": 4, "e2e_f16_f16y": 2,
               "counters_f32": 0, "counters_bf16": 0, "counters_f16": 0}
    res = {}
    for k, ts in times.items():
        ms = statistics.median(ts) * 1e3
        h2d = graph_h2d + n * d * x_bytes[k]
        d2h = small_d2h + n * d * y_bytes[k]
        form = "column blocks" if y_bytes[k] and column_blocks(d) else "row blocks"
        res[k] = {"ms": ms, "ms_min": min(ts) * 1e3, "ms_max": max(ts) * 1e3, "gedges_s": nnz / (ms * 1e-3) / 1e9,
                  "h2d_bytes": h2d, "d2h_bytes": d2h, "link_gbs": (h2d + d2h) / (ms * 1e-3) / 1e9, "form": form}
    line = {"tool": "tools/e2e_bf16_bench.py", "nodes": n, "headline_graph": n == HEADLINE_NODES,
            "stored_entries": nnz, "dim": d, "classes": C, "norm": "sym D^-1/2 (A+I) D^-1/2 on the fly",
            "reps": args.reps, "warmup": args.warmup, "timer": "host clock around the synchronous call",
            "host_memory": "pinned", "arms": res,
            "speedup_e2e_bf16_f32y": res["e2e_f32"]["ms"] / res["e2e_bf16_f32y"]["ms"],
            "speedup_e2e_bf16_bf16y": res["e2e_f32"]["ms"] / res["e2e_bf16_bf16y"]["ms"],
            "speedup_counters_bf16": res["counters_f32"]["ms"] / res["counters_bf16"]["ms"],
            "speedup_e2e_f16_f32y": res["e2e_f32"]["ms"] / res["e2e_f16_f32y"]["ms"],
            "speedup_e2e_f16_f16y": res["e2e_f32"]["ms"] / res["e2e_f16_f16y"]["ms"],
            "speedup_counters_f16": res["counters_f32"]["ms"] / res["counters_f16"]["ms"],
            "check_counters_identical": bool(counters_equal), "check_sample_rows": int(rows.shape[0]),
            "check_y_f32_max_abs_err": err, "check_y_max_abs": scale,
            "check_y_f32": bool(y_ok), "check_y_bf16_is_rounded_f32": bool(bf16_ok),
            "check_y_f16_f32_max_abs_err": err16, "check_y_f16_f32": bool(y16_ok),
            "check_y_f16_is_rounded_f32": bool(f16_ok), "card": card(device)}
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    if not (counters_equal and y_ok and bf16_ok and y16_ok and f16_ok):
        sys.exit(3)


if __name__ == "__main__":
    main()
