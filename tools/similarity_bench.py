#!/usr/bin/env python
"""Aggregation similarity: the Gram path (gram + class_colsum) against the Gram-free class sums (class_inner_sums), and
the whole-graph similarity on the headline graph (BASELINE.json configs[4], bench.gen_rows: 50M nodes, ~976M stored
entries, 10 classes, d = 128).

    python tools/similarity_bench.py [--reps 10] [--warmup 3] [--out profiles/similarity_r05.json]

Part 1, both paths side by side at m in {10,000, 65,536} x d in {10, 128}: z is the first m rows of A Y (one-hot
labels, d = 10) or of A X (d = 128) of the headline graph, labels its first m labels.  CUDA events, the two paths
alternating within every repetition; median, min and max ms; the largest ulp difference of w between the paths and
the soft-LAS counts (las_count, LP = 1, sum) of both.

Part 2, hm.similarity(oh, A, oh) and hm.similarity(x, A, oh) on the whole graph (m = 50M: the class-sum path): the
end-to-end call with CUDA events, then the time of each stage from a separate torch.profiler run (kernel durations
summed by name).  Algorithmic bytes per stage:
    spmm        nnz (4 + 4 d) + n (8 + 4 d)              column ids and feature rows, rowptr and output rows
    class sums  4 m d + 4 m + 16 P                       z and labels once; P = partial-table doubles, written + read
    class dots  4 m d + 4 m C                            z again, w out
    las_score   4 m + 12 m C                             labels, w, the label rows (read twice: column sums + scores)
and each stage's rate as a fraction of the device-to-device copy_ bandwidth measured in the same run.
Prints one JSON line and writes it to --out.
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "when-do-gnns-help_b200"), os.path.join(ROOT, "tools")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import torch  # noqa: E402

import bench  # noqa: E402
from bf16_bench import card  # noqa: E402

STAGES = {"class_sum_partial_kernel": "class_sums", "class_sum_reduce_kernel": "class_sums",
          "class_dot_kernel": "class_dots", "label_colsum_kernel": "las_score", "las_score_kernel": "las_score"}


def timed(fns, reps, warmup):
    """{name: [ms per rep]}: every fn once per repetition, alternating, CUDA events"""
    for _ in range(warmup):
        for fn in fns.values():
            fn()
    torch.cuda.synchronize()
    ev = {k: [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
          for k in fns}
    for r in range(reps):
        for k, fn in fns.items():
            ev[k][r][0].record()
            fn()
            ev[k][r][1].record()
    torch.cuda.synchronize()
    return {k: [a.elapsed_time(b) for a, b in v] for k, v in ev.items()}


def summary(times):
    return {"ms": statistics.median(times), "ms_min": min(times), "ms_max": max(times)}


def ulp_diff(a, b):
    def key(x):
        i = x.contiguous().view(torch.int32).to(torch.int64)
        return torch.where(i < 0, -(i & 0x7FFFFFFF), i)
    return int((key(a) - key(b)).abs().max().item())


def stage_times(fn, reps):
    """ms per call of every stage, from kernel durations under torch.profiler (a run of its own)"""
    from torch.profiler import ProfilerActivity, profile
    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        us = getattr(e, "device_time_total", None)
        if us is None:
            us = e.cuda_time_total
        name = e.key
        stage = next((s for k, s in STAGES.items() if k in name), "spmm" if "spmm" in name else None)
        if stage is None or us == 0:
            continue
        out.setdefault(stage, {"ms": 0.0, "kernels": {}})
        out[stage]["ms"] += us / 1e3 / reps
        out[stage]["kernels"][name] = us / 1e3 / reps
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--nodes", type=int, default=50_000_000)
    ap.add_argument("--avg-degree", type=float, default=20.0)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--classes", type=int, default=10)
    ap.add_argument("--homophily", type=float, default=0.3)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "similarity_r05.json"))
    args = ap.parse_args()

    import wdgh_b200 as W
    from wdgh_b200 import graph as G
    hm = W.homophily_metrics

    W._lib.require_device()
    device = torch.device("cuda", torch.cuda.current_device())
    n, d, C = args.nodes, args.dim, args.classes
    rowptr, col, x, labels = bench.gen_rows(0, n, n, args.avg_degree, C, args.homophily, d, device)
    nnz = int(col.shape[0])
    g = G.CSRGraph(rowptr, col, None, n)
    _ = g.plan
    oh = torch.zeros((n, C), dtype=torch.float32, device=device)
    oh[torch.arange(n, device=device), labels.long()] = 1.0
    z_oh = G.spmm(g, oh, W.NORM_NONE, False)
    z_x = G.spmm(g, x, W.NORM_NONE, False)
    torch.cuda.synchronize()

    # device-to-device copy bandwidth of this run (read + write)
    src = torch.empty(1 << 30, dtype=torch.float32, device=device)
    dst = torch.empty_like(src)
    cp = timed({"copy": lambda: dst.copy_(src)}, args.reps, args.warmup)["copy"]
    copy_gbs = 2 * src.numel() * 4 / (statistics.median(cp) * 1e-3) / 1e9
    del src, dst
    torch.cuda.empty_cache()

    side = []
    for m in (10_000, 65_536):
        lab = labels[:m].contiguous()
        label_rows = oh[:m].contiguous()
        for dd, zfull in ((C, z_oh), (d, z_x)):
            z = zfull[:m].contiguous()
            out = {}
            fns = {"gram_colsum": lambda: out.__setitem__("gram", G.class_colsum(G.gram(z), lab, C)),
                   "class_inner_sums": lambda: out.__setitem__("inner", G.class_inner_sums(z, lab, C))}
            t = timed(fns, args.reps, args.warmup)
            wg, wi = out["gram"], out["inner"]
            side.append({"m": m, "d": dd, "classes": C,
                         "gram_colsum": summary(t["gram_colsum"]), "class_inner_sums": summary(t["class_inner_sums"]),
                         "speedup": statistics.median(t["gram_colsum"]) / statistics.median(t["class_inner_sums"]),
                         "max_ulp_diff_w": ulp_diff(wg, wi),
                         "las_count_gram": G.las_count(wg, lab, label_rows, False, 1, True),
                         "las_count_inner": G.las_count(wi, lab, label_rows, False, 1, True)})
            del out
            torch.cuda.empty_cache()
    del z_x, z_oh
    torch.cuda.empty_cache()

    # whole graph: hm.similarity with one-hot and with d-wide features (z = A X inside the call)
    whole = {}
    for tag, feats, dd in (("onehot", oh, C), (f"x_d{d}", x, d)):
        res = {}
        t = timed({"similarity": lambda: res.__setitem__("score", hm.similarity(feats, g, oh))}, args.reps,
                  args.warmup)["similarity"]
        ws = int(W._lib.lib.wdgh_class_inner_workspace_doubles(n, dd, C))
        partial = ws - C * (dd + 1)
        alg = {"spmm": nnz * (4 + 4 * dd) + n * (8 + 4 * dd),
               "class_sums": 4 * n * dd + 4 * n + 16 * partial,
               "class_dots": 4 * n * dd + 4 * n * C,
               "las_score": 4 * n + 12 * n * C}
        stages = stage_times(lambda: hm.similarity(feats, g, oh), max(3, args.reps // 2))
        for s, v in stages.items():
            v["algorithmic_bytes"] = alg.get(s)
            if alg.get(s) and v["ms"] > 0:
                v["achieved_gbs"] = alg[s] / (v["ms"] * 1e-3) / 1e9
                v["frac_of_copy"] = v["achieved_gbs"] / copy_gbs
        whole[tag] = {"d": dd, "score": float(res["score"]), "call": summary(t), "stages": stages,
                      "partial_doubles": partial}
        del res
    line = {"tool": "tools/similarity_bench.py", "nodes": n, "stored_entries": nnz, "dim": d, "classes": C,
            "reps": args.reps, "warmup": args.warmup, "copy_gbs": copy_gbs, "side_by_side": side,
            "whole_graph": whole, "threshold_rows": G.GRAM_SIMILARITY_MAX_ROWS, "card": card(device)}
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
