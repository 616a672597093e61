#!/usr/bin/env python
"""The label-statistics pass (`wdgh_structure_counts`) alone on the headline graph (bench.gen_rows: 50M nodes, ~976M
stored entries, avg degree 20, h = 0.3), one or more builds of the library side by side.

    python tools/label_pass_bench.py [--lib PATH ...] [--reps 5] [--calls 10] [--out FILE]

Arms, each on the graph generated for its class count (the class of node v is v % C):
    c10_stream     C = 10:  1-byte label copy, structure_stream_kernel
    c100_rowgroup  C = 100: 1-byte label copy, structure_rowgroup_kernel<uint8_t>
    c300_int32     C = 300: int32 labels, structure_rowgroup_kernel<int32_t>
    c10_rerun      C = 10 with every 97th label -2: the 1-byte pass, then the int32 re-run graph.structure_counts does
                   after it (both calls timed)
Every --lib (default: the in-tree library) is loaded with ctypes; the libraries take turns within every repetition
(A B A B ...), each timed with CUDA events around --calls back-to-back calls.  Per arm and library: median ms per call
and [min, max] over the repetitions.  Checks in the same run: the counters of every library are identical per arm and
node_sum agrees to 1e-12 relative.  Prints one JSON line, writes it to --out and exits non-zero when a check fails.
"""
import argparse
import ctypes
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

ARMS = (("c10_stream", 10, False), ("c100_rowgroup", 100, False), ("c300_int32", 300, False), ("c10_rerun", 10, True))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], help="libwdgh_b200.so to time (repeatable)")
    ap.add_argument("--nodes", type=int, default=50_000_000)
    ap.add_argument("--avg-degree", type=float, default=20.0)
    ap.add_argument("--homophily", type=float, default=0.3)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--calls", type=int, default=10)
    ap.add_argument("--out", default="")
    args = ap.parse_args()

    import wdgh_b200 as W
    from wdgh_b200 import graph as G

    W._lib.require_device()
    device = torch.device("cuda", torch.cuda.current_device())
    paths = [os.path.abspath(p) for p in (args.lib or [W._lib.LIB_PATH])]
    libs = []
    for p in paths:
        fn = ctypes.CDLL(p).wdgh_structure_counts
        fn.argtypes = W._lib.SIGNATURES["wdgh_structure_counts"]
        fn.restype = ctypes.c_int
        libs.append(fn)
    n = args.nodes
    stream = torch.cuda.current_stream().cuda_stream
    res, ok = {}, True
    for arm, C, rerun in ARMS:
        rowptr, col, _, labels = bench.gen_rows(0, n, n, args.avg_degree, C, args.homophily, 128, device,
                                                want_x=False)
        if rerun:
            labels[::97] = -2
        g = G.CSRGraph(rowptr, col, None, n)
        plan, plan_host = g.plan
        nnz = int(col.shape[0])
        counters = torch.empty(W._lib.sc_words(C), dtype=torch.int64, device=device)
        node_sum = torch.empty(2, dtype=torch.float64, device=device)
        deg = torch.empty(n, dtype=torch.int32, device=device)
        match = torch.empty(n, dtype=torch.int32, device=device)
        lab8 = torch.empty(n, dtype=torch.uint8, device=device)
        ptr = W._lib.ptr

        def call(fn, scratch):
            rc = fn(ptr(rowptr), ptr(col), n, nnz, ptr(labels), C, ptr(plan), plan_host, ptr(counters), ptr(node_sum),
                    ptr(deg), ptr(match), ptr(scratch), n, 0, stream)
            if rc:
                raise RuntimeError(f"wdgh_structure_counts failed (rc={rc}) in {arm}")

        def one(fn):
            call(fn, lab8)
            if rerun:
                call(fn, None)

        call(libs[0], lab8)
        torch.cuda.synchronize()
        if rerun and int(counters[W._lib.SC_N_MULTI_NEG].item()) == 0:
            raise RuntimeError("the -2 labels did not trigger the int32 re-run")
        outs = []
        for fn in libs:
            one(fn)
            torch.cuda.synchronize()
            outs.append((counters.cpu().clone(), node_sum.cpu().clone()))
        same = all(torch.equal(c, outs[0][0]) for c, _ in outs) and \
            all(torch.allclose(s, outs[0][1], rtol=1e-12, atol=0) for _, s in outs)
        ok &= same
        times = [[] for _ in libs]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(args.reps):
            for k, fn in enumerate(libs):
                e0.record()
                for _ in range(args.calls):
                    one(fn)
                e1.record()
                torch.cuda.synchronize()
                times[k].append(e0.elapsed_time(e1) / args.calls)
        res[arm] = {"classes": C, "stored_entries": nnz, "outputs_identical": bool(same),
                    "libs": [{"lib": p, "ms": statistics.median(t), "ms_min": min(t), "ms_max": max(t)}
                             for p, t in zip(paths, times)]}
        del rowptr, col, labels, g, plan, counters, node_sum, deg, match, lab8
        torch.cuda.empty_cache()
    line = {"tool": "tools/label_pass_bench.py", "nodes": n, "reps": args.reps, "calls_per_rep": args.calls,
            "timer": "CUDA events around back-to-back calls, libraries alternating within every repetition",
            "arms": res, "check_outputs_identical": bool(ok), "card": card(device)}
    text = json.dumps(line)
    print(text, flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    if not ok:
        sys.exit(3)


if __name__ == "__main__":
    main()
