#!/usr/bin/env python
"""Headline benchmark: GEdges/s for A_hat X aggregation + homophily metrics (BASELINE.json `metric`).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[4]): synthetic CSBM-H graph with power-law row lengths,
50M nodes / ~1B stored entries, d = 128 float32 features, 10 classes; row-sharded over N GPUs
(total work fixed -> "strong" scaling).  One step = one pass of the hot path:
    degree scale D^-1/2  ->  Y = D^-1/2 (A+I) D^-1/2 X  ->  label statistics (edge / node / class /
    adjusted homophily, label informativeness) [-> all-gather / all-reduce when N > 1].
`value` times the pass with inputs resident in HBM; `e2e` times the reference-facing host-buffer
entry (wdgh_pipeline_host) including the H2D copies of every input and the D2H copies of the counters AND of
Y = A_hat X.  `--impl reference` times the reference's own CPU implementation (oracle/_ref, see oracle/build_ref.py)
on a bounded sample.  At N > 1 every element of Y is checked against an independent path and a mismatch exits 3.
Prints ONE JSON line on rank 0.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "when-do-gnns-help_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

METRIC = "aggregation_plus_homophily_throughput"
UNIT = "GEdges/s"
TILE_ROWS = 2_000_000


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nodes", type=int, default=50_000_000)
    ap.add_argument("--avg-degree", type=float, default=20.0)
    ap.add_argument("--dim", type=int, default=128)
    ap.add_argument("--classes", type=int, default=10)
    ap.add_argument("--homophily", type=float, default=0.3)
    ap.add_argument("--cpu-sample-nodes", type=int, default=200_000,
                    help="CPU arm: nodes of the bounded sample the reference's CPU path is timed on")
    ap.add_argument("--no-phased", action="store_true", help="N>1, 1-D: plain all-gather then aggregate (no overlap)")
    ap.add_argument("--partition", default="auto", choices=["auto", "1d", "2d"],
                    help="N>1: 1-D row partition or 2-D (2 row groups x N/2 column groups); auto = 2d for even N")
    ap.add_argument("--overlap", default="auto", choices=["auto", "on", "off"],
                    help="2-D partition: aggregate the own slice next to the NVLink-bound foreign slices on a second "
                         "stream (auto = from 4 column groups on, i.e. N >= 8)")
    ap.add_argument("--no-verify", action="store_true", help="N>1: skip the element-wise check of Y against the "
                                                               "plain all-gather + one-launch aggregation")
    ap.add_argument("--workload", default="csbm", choices=["csbm", "linkx"],
                    help="csbm = BASELINE.json configs[4] (the headline); linkx = configs[2]: a twitch-gamer-sized graph "
                         "through the whole large-dataset flow of homophily_tests.py:88-137 (seconds per flow)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy: the counters, node_sum, and Y = "
                         "A_hat X on a fixed, seeded sample of rows (at most 32 MB of Y)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.workload != "csbm"):
        ap.error("--dump-outputs writes the outputs of --impl ours --workload csbm")
    return args


DUMP_Y_BYTES = 32 << 20


def dump_rows(n, d):
    """Sorted global row ids of the Y sample --dump-outputs writes: the same for every run and every partition."""
    k = min(n, max(1, DUMP_Y_BYTES // (4 * d)))
    return np.sort(np.random.default_rng(0).choice(n, k, replace=False))


def dump_outputs(out_dir, rows, y_local, r0, r1, counters, node_sum, world):
    """Gather the sampled rows of Y from the ranks that own them (all ranks call this); rank 0 writes the .npy files."""
    import torch.distributed as dist
    device = y_local.device
    rows_t = torch.from_numpy(rows).to(device)
    mine = (rows_t >= r0) & (rows_t < r1)
    y_s = torch.zeros((rows.shape[0], y_local.shape[1]), dtype=torch.float32, device=device)
    y_s[mine] = y_local.index_select(0, rows_t[mine] - r0)
    if world > 1:
        dist.all_reduce(y_s)
    if int(os.environ.get("RANK", "0")) != 0:
        return
    os.makedirs(out_dir, exist_ok=True)
    arrays = {"y_sample": y_s.cpu().numpy(), "y_sample_rows": rows.astype(np.float64),
              "counters": counters.cpu().numpy().astype(np.float64), "node_sum": node_sum.cpu().numpy().astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ---------------------------------------------------------------------------
# synthetic CSBM-H / power-law generator (torch on the GPU; outside every timed region)
# ---------------------------------------------------------------------------
def gen_rows(r0, r1, n, avg_deg, C, h, d, device, seed=1234, want_x=True):
    """Rows [r0, r1) of the global graph, generated tile by tile so that the graph does not depend
    on how many ranks share it.  Row lengths ~ Pareto(shape 1.8) with mean avg_deg (cap 1e6); the
    class of node v is v % C; a neighbour has the row's class with probability h, otherwise one of
    the other classes uniformly; within the class it is uniform (no L2-friendly locality)."""
    a = 1.8
    xm = avg_deg * (a - 1) / a
    rowptr_parts, col_parts, x_parts = [torch.zeros(1, dtype=torch.int64, device=device)], [], []
    base = 0
    per_class = n // C
    t0 = (r0 // TILE_ROWS) * TILE_ROWS
    for ts in range(t0, r1, TILE_ROWS):
        te = min(ts + TILE_ROWS, n)
        g = torch.Generator(device=device).manual_seed(seed * 1_000_003 + ts // TILE_ROWS)
        rows = te - ts
        u = torch.rand(rows, device=device, generator=g).clamp_(min=1e-12)
        deg = (xm * u.pow(-1.0 / a)).clamp_(max=1e6).to(torch.int64)
        # drawn even when the caller does not want it: the generator state (hence the column ids drawn below) must
        # not depend on want_x, or a row slice regenerated by a peer (2-D partition) would be a different graph
        xt = torch.randn(rows, d, device=device, generator=g)
        lo, hi = max(ts, r0) - ts, min(te, r1) - ts  # part of this tile that belongs to [r0, r1)
        # generate the whole tile's random stream so the graph is identical for every sharding
        rid = torch.repeat_interleave(torch.arange(rows, device=device), deg)
        e = rid.shape[0]
        own = (rid + ts) % C
        same = torch.rand(e, device=device, generator=g) < h
        other = (own + 1 + torch.randint(0, C - 1, (e,), device=device, generator=g)) % C
        cls = torch.where(same, own, other)
        col = cls + C * torch.randint(0, per_class, (e,), device=device, generator=g)
        key = (rid << 32) | col
        del rid, own, same, other, cls, col
        key = torch.sort(key).values
        ptr = torch.zeros(rows + 1, dtype=torch.int64, device=device)
        ptr[1:] = torch.cumsum(deg, 0)
        e0, e1 = int(ptr[lo]), int(ptr[hi])
        col_parts.append((key[e0:e1] & 0xFFFFFFFF).to(torch.int32))
        rowptr_parts.append(ptr[lo + 1:hi + 1] - ptr[lo] + base)
        base += e1 - e0
        if want_x:
            x_parts.append(xt[lo:hi].clone())
        del key, ptr, deg, u, xt
    rowptr = torch.cat(rowptr_parts)
    col = torch.cat(col_parts) if col_parts else torch.zeros(0, dtype=torch.int32, device=device)
    x = torch.cat(x_parts) if want_x else None
    labels = (torch.arange(r0, r1, device=device) % C).to(torch.int32)
    return rowptr, col, x, labels


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler:
    """`nvidia-smi -lms 50` in the background from process start; `stop(t0, t1)` keeps the samples whose own
    timestamp lies inside the wall-clock window [t0, t1] = warm-up + timed steps (B200_PROFILING.md clocks line).
    Started early because nvidia-smi needs up to a second for its first sample on an 8-GPU box."""
    Q = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, device):
        self.proc = None
        try:
            uuid = str(torch.cuda.get_device_properties(device).uuid)
            sel = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", sel, f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    @staticmethod
    def parse(text, t0, t1):
        """CSV lines -> summary of the samples taken in [t0, t1] (seconds since the epoch, local clock)."""
        import datetime
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in text.strip().splitlines():
            f = [v.strip() for v in line.split(",")]
            if len(f) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                if not (t0 - 0.025 <= ts <= t1 + 0.025):
                    continue
                sm.append(float(f[1])), mx.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm))
        return out

    def stop(self, t0, t1):
        if self.proc is None:
            return self.parse("", t0, t1)
        time.sleep(0.15)
        self.proc.terminate()
        try:
            text, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            return self.parse("", t0, t1)
        return self.parse(text, t0, t1)


def nvlink_bytes(device):
    """(tx, rx) bytes this GPU has moved over NVLink so far, summed over its links (`nvidia-smi nvlink -gt d`); None
    when the counters are not available."""
    import re
    try:
        uuid = str(torch.cuda.get_device_properties(device).uuid)
        sel = uuid if uuid.startswith("GPU-") else "GPU-" + uuid
        out = subprocess.run(["nvidia-smi", "nvlink", "-gt", "d", "-i", sel], capture_output=True, text=True,
                             timeout=20).stdout
        tx = [int(v) for v in re.findall(r"Tx:\s*(\d+)\s*KiB", out)]
        rx = [int(v) for v in re.findall(r"Rx:\s*(\d+)\s*KiB", out)]
        if not tx or not rx:
            if os.environ.get("WDGH_STAGE_TIMES") == "1":
                print("[nvlink] unparsed nvidia-smi output: " + out[:400].replace("\n", " | "), file=sys.stderr)
            return None
        return sum(tx) * 1024, sum(rx) * 1024
    except Exception:
        return None


# ---------------------------------------------------------------------------
# the CPU arm: the reference's own CPU implementation of the path on the host cores
# ---------------------------------------------------------------------------
def load_cpu_arm():
    """-> (kind, once(rowptr, col, x, labels, n)).  kind = "reference": the unmodified reference modules (from
    /root/reference, or from oracle/_ref on the GPU box -- see oracle/build_ref.py) bound to the CPU;
    kind = "port": the oracle restatement, only when no reference tree travelled with the repo."""
    import scipy.sparse as sp
    try:
        from oracle import ref_shim
        hm, uf, _ = ref_shim.load()
    except Exception:
        hm = uf = None
    if hm is not None:
        def once(rowptr, col, x, labels, n):
            # homophily_tests.py:88-110 (large-dataset flow, --symmetric 1) + SGC-1 propagation + every label metric
            adj = sp.csr_matrix((np.ones(col.shape[0], np.float32), col, rowptr), (n, n))
            a_hat = uf.sparse_mx_to_torch_sparse_tensor(uf.sys_normalized_adjacency(adj))   # uf.py:418-426, 400-407
            y = torch.spmm(a_hat, torch.from_numpy(x))                                      # hm.py:192/234
            lab = torch.from_numpy(labels)
            vals = [hm.edge_homophily(a_hat, lab), hm.node_homophily(a_hat, lab),           # hm.py:43-78
                    hm.our_measure(a_hat.coalesce().indices(), lab),                        # hm.py:81-123
                    hm.adjusted_homo(a_hat, lab), hm.label_informativeness(a_hat, lab)]     # hm.py:126-161
            return float(y[0, 0]) + sum(float(v) for v in vals)
        return "reference", once

    def once(rowptr, col, x, labels, n):
        from oracle import ref_port as O
        row = np.repeat(np.arange(n, dtype=np.int64), np.diff(rowptr))
        ones = np.ones(col.shape[0], np.float32)
        r, c, v = O.sys_normalized_adjacency(row, col, ones, n)          # util_funcs.py:418-426
        y = O.spmm(r, c, v, n, x)                                         # hm.py:192/234 torch.spmm
        s = O.structure_counts(r, c, labels, n)                           # hm.py:43-161 (all label metrics)
        return float(y[0, 0]) + s["match_all"]
    return "port", once


def cpu_sample(args, device):
    n_s = min(args.cpu_sample_nodes, args.nodes)
    rowptr, col, x, labels = gen_rows(0, n_s, n_s, args.avg_degree, args.classes, args.homophily, args.dim, device)
    return (rowptr.cpu().numpy(), col.cpu().numpy().astype(np.int64), x.cpu().numpy(),
            labels.cpu().numpy().astype(np.int64), n_s)


def cpu_sample_text(kind, n_s, nnz, args):
    what = ("unmodified reference: sys_normalized_adjacency + sparse_mx_to_torch_sparse_tensor + torch.spmm + edge / "
            "node / class / adjusted homophily + label informativeness" if kind == "reference" else
            "oracle port: sys-normalise + torch.spmm + label counts")
    return (f"SAMPLE, not the full workload: a {n_s}-node graph from the same generator ({nnz} stored entries, "
            f"d={args.dim}, C={args.classes}); {what}")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import warnings
    warnings.filterwarnings("ignore")
    device = torch.device("cuda", 0) if torch.cuda.is_available() else torch.device("cpu")
    rowptr, col, x, labels, n_s = cpu_sample(args, device)
    nnz = int(col.shape[0])
    kind, once = load_cpu_arm()
    for _ in range(max(args.warmup, 1)):
        once(rowptr, col, x, labels, n_s)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        once(rowptr, col, x, labels, n_s)
    dt = (time.perf_counter() - t0) / args.steps
    val = nnz / dt / 1e9
    sample = cpu_sample_text(kind, n_s, nnz, args)
    cfg = workload_config(args, nnz=nnz)
    cfg["workload"] = sample + f"; the GPU arm runs the full {args.nodes}-node graph"
    cfg["nodes"], cfg["partition"], cfg["norm"] = n_s, "host cores, one process", "sym D^-1/2 (A+I) D^-1/2, materialised (scipy)"
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": torch.get_num_threads(), "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def make_slice_graphs(G, grid2, rank, rowptr, col, args, device):
    """2-D partition: the CSR of every row slice of this rank's row group restricted to its column group.  A real
    pipeline would receive these from the loader; here the peers' rows are regenerated (same seeds, same graph)."""
    n, part = args.nodes, grid2.part
    gi, gj = grid2.coords(rank)
    slice_graphs = []
    for srank in grid2.row_group_ranks(gi):
        s0, s1 = part.bounds(srank)
        if srank == rank:
            rp_s, col_s = rowptr, col
        else:
            rp_s, col_s, _, _ = gen_rows(s0, s1, n, args.avg_degree, args.classes, args.homophily, args.dim, device,
                                         want_x=False)
        rp_f, col_f = grid2.filter_slice(rp_s, col_s, gj)
        sg = G.CSRGraph(rp_f, col_f, None, s1 - s0, row_offset=s0, n_global=n)
        _ = sg.plan
        slice_graphs.append(sg)
    torch.cuda.empty_cache()
    return slice_graphs


def workload_config(args, nnz):
    return {"workload": "csbm-h power-law graph (BASELINE.json configs[4]): "
                        f"{args.nodes} nodes, avg row length {args.avg_degree:g}, d={args.dim} f32, "
                        f"{args.classes} classes, h={args.homophily}",
            "nodes": args.nodes, "stored_entries": nnz, "dim": args.dim, "classes": args.classes,
            "norm": "sym D^-1/2 (A+I) D^-1/2 on the fly",
            "partition": (f"rows/{args.gpus}" if not getattr(args, "_use_2d", False) else
                          f"2 row groups x {args.gpus // 2} column groups (peer pull of the partner shard, foreign row "
                          "slices stored into their owners' memory by the aggregation kernel"
                          + (", own slice overlapped on a second stream" if getattr(args, "_overlap", False) else "") + ")"),
            "l2_policy": "inputs (feature matrix >= 25 GB at full size) are far larger than the 126 MB L2"}


# ---------------------------------------------------------------------------
# --workload linkx: BASELINE.json configs[2] -- LINKX-scale homophily metrics + KR on one B200
# ---------------------------------------------------------------------------
LINKX_NODES, LINKX_AVG_DEG, LINKX_DIM, LINKX_CLASSES = 168_114, 40.0, 7, 2   # twitch-gamer: 168,114 nodes, 6.8M edges


def linkx_graph(device):
    """twitch-gamer-shaped synthetic graph: power-law row lengths, symmetrised like `to_undirected` (uf.py:272), binary
    labels, 7 non-negative features.  Returns (row, col) int64 coalesced on the host, labels, features."""
    n = LINKX_NODES
    rowptr, col, x, labels = gen_rows(0, n, n, LINKX_AVG_DEG, LINKX_CLASSES, 0.55, LINKX_DIM, device)
    row = torch.repeat_interleave(torch.arange(n, device=device), rowptr[1:] - rowptr[:-1])
    col = col.to(torch.int64)
    keep = row != col
    key = torch.unique(torch.cat([row[keep] * n + col[keep], col[keep] * n + row[keep]]))
    return ((key // n).cpu(), (key % n).cpu(), labels.to(torch.int64).cpu(), x.abs().cpu())


def linkx_flow(hm, uf, row, col, labels, features, n, to_dev, epochs):
    """homophily_tests.py:88-137 for every metric of METRIC_LIST on one graph; `hm` / `uf` are either the reference's
    modules (CPU arm) or the wdgh_b200 mirrors (CUDA path) -- the same call sequence runs against both."""
    import scipy.sparse as sp
    import torch.nn.functional as f
    out = {}
    adj_raw = sp.coo_matrix((np.ones(row.shape[0]), (row.numpy(), col.numpy())), shape=(n, n))
    feats = f.normalize(features, p=1, dim=1)                                               # :95
    adj = uf.sparse_mx_to_torch_sparse_tensor(uf.sys_normalized_adjacency(adj_raw))         # :98-104 (--symmetric 1)
    adj, feats_d, lab_d = to_dev(adj), to_dev(feats), to_dev(labels)
    out["node_homo"] = float(hm.node_homophily(adj, lab_d))                                 # :108-109
    out["class_homo"] = float(hm.our_measure(adj.coalesce().indices(), lab_d))
    out["label_info"] = float(hm.label_informativeness(adj, lab_d))
    out["adj_homo"] = float(hm.adjusted_homo(adj, lab_d))
    out["edge_homo"] = float(hm.edge_homophily(adj, to_dev(torch.eye(int(labels.max()) + 1)[labels])))   # :110-112
    out["node_hom_generalized"] = float(hm.generalized_edge_homophily(adj, feats_d, lab_d))  # :113-114
    a_raw = to_dev(uf.sparse_mx_to_torch_sparse_tensor(adj_raw))                            # full_load_data_large again, :117
    onehot = to_dev(torch.eye(int(labels.max()) + 1)[labels])
    for key, hard in (("agg_homo_soft", None), ("agg_homo_hard", 1)):                       # :115-128
        las = np.zeros(10)
        for i in range(10):
            idx, _, _ = uf.random_disassortative_splits(labels, labels.max() + 1, 10000 / n)
            las[i] = 2 * float(hm.similarity(onehot, a_raw, onehot, hard=hard, LP=1, idx_train=to_dev(idx))) - 1
        out[key] = float(np.mean(las))
    p, _ = hm.classifier_based_performance_metric(to_dev(features), a_raw, labels, 500,     # :129-133
                                                  base_classifier="kernel_reg1", epochs=epochs)
    out["kernel_reg1_based_homo"] = float(p)
    return out


def linkx_kr_check(hm, row, col, labels, features, n, device, epochs=3):
    """The KR p-value is a t-test over per-epoch accuracies of kernel regressions whose train Gram is rank-deficient
    (d = 7) and fed to pinv(rcond=1e-15): single predictions are decided by float32 rounding noise, so the p-value of two
    float32 implementations may differ while every well-determined prediction agrees.  This is the per-prediction
    contract of tests/test_gpu_parity.py::kr_contract on this workload (checker, untimed): same seeds through the CUDA
    path and the oracle port, predictions compared node by node, flips allowed only on nodes the oracle's perturbation
    analysis (oracle.kr_unstable_nodes) flags as noise-decided."""
    import random
    from oracle import ref_port as O
    a_raw = torch.sparse_coo_tensor(torch.stack([row, col]), torch.ones(row.shape[0]), (n, n)).coalesce()
    random.seed(11), np.random.seed(11), torch.manual_seed(11)
    tr = []
    hm.classifier_based_performance_metric(features.to(device), a_raw.to(device), labels, 500,
                                           base_classifier="kernel_reg1", epochs=epochs, _trace=tr)
    random.seed(11), np.random.seed(11), torch.manual_seed(11)
    rtr = []
    O.kr_metric(features.numpy(), row.numpy(), col.numpy(), np.ones(row.shape[0], np.float32), n, labels.numpy(), 500,
                "kernel_reg1", epochs, trace=rtr)
    out = {"epochs": epochs, "predictions": 0, "flips": 0, "unstable_predictions": 0, "flips_outside_unstable": 0}
    for got, ref in zip(tr, rtr):
        if not torch.equal(got["va"].cpu(), ref["va"]):
            out["flips_outside_unstable"] += 1 << 20     # different validation sets: not comparable, flag loudly
            continue
        for side, kname in (("pred_g", "gram_g"), ("pred_x", "gram_x")):
            changed = got[side].cpu() != ref[side]
            outside, unstable, _ = O.kr_flips_outside_unstable(changed, ref[kname], ref["n_layers"], ref["tr"], ref["va"],
                                                               ref["onehot_tr"])
            out["predictions"] += int(changed.numel())
            out["flips"] += int(changed.sum())
            out["unstable_predictions"] += int(unstable.sum())
            out["flips_outside_unstable"] += outside
    out["ok"] = out["flips_outside_unstable"] == 0
    return out


def run_linkx(args):
    """One JSON line: seconds per complete flow on the CUDA path, the reference's CPU seconds next to it."""
    import random
    import warnings
    warnings.filterwarnings("ignore")
    if int(os.environ.get("RANK", "0")) != 0:
        return
    device = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    row, col, labels, features = linkx_graph(device)
    n, nnz = LINKX_NODES, int(row.shape[0])
    epochs = 100
    cfg = {"workload": f"twitch-gamer-sized synthetic graph (BASELINE.json configs[2]): {n} nodes, {nnz} stored entries "
                       f"(symmetric), d={LINKX_DIM}, {LINKX_CLASSES} classes; homophily_tests.py:88-137 for EVERY metric: "
                       "sys-normalised adjacency, node / class / adjusted / edge homophily, label informativeness, "
                       "generalised edge homophily (10 x 75000 sampled entries), 2 x 10 similarity on 10,000-node samples, "
                       f"KR kernel_reg1 sample_max=500 epochs={epochs}",
           "nodes": n, "stored_entries": nnz, "dim": LINKX_DIM, "classes": LINKX_CLASSES}

    def seed():
        random.seed(7), np.random.seed(7), torch.manual_seed(7)

    if args.impl == "reference":
        from oracle import ref_shim
        hm, uf, _ = ref_shim.load()
        steps = max(1, min(args.steps, 2))
        seed()
        linkx_flow(hm, uf, row, col, labels, features, n, lambda t: t, epochs) if args.warmup else None
        t0 = time.perf_counter()
        for _ in range(steps):
            seed()
            vals = linkx_flow(hm, uf, row, col, labels, features, n, lambda t: t, epochs)
        dt = (time.perf_counter() - t0) / steps
        line = {"impl": "reference", "metric": "linkx_flow_seconds", "value": dt, "unit": "s", "n_gpus": args.gpus,
                "steps": steps, "warmup": min(args.warmup, 1), "ms_per_step": dt * 1e3, "higher_is_better": False,
                "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
                "cpu_baseline": {"value": dt, "unit": "s", "cores": torch.get_num_threads(), "kind": "reference",
                                 "sample": "the full linkx workload (no sampling), unmodified reference on the host cores"},
                "e2e": {"value": dt, "unit": "s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "metrics": vals}
        print(json.dumps(line), flush=True)
        return
    import wdgh_b200 as W
    W._lib.require_device()
    hm, uf = W.homophily_metrics, W.util_funcs
    to_dev = lambda t: t.to(device) if isinstance(t, torch.Tensor) else t   # noqa: E731  (host tensors in: H2D is timed)
    steps = max(1, min(args.steps, 5))
    for _ in range(max(1, min(args.warmup, 2))):
        seed()
        linkx_flow(hm, uf, row, col, labels, features, n, to_dev, epochs)
    torch.cuda.synchronize()
    launches0 = W.launch_count()
    t0 = time.perf_counter()
    for _ in range(steps):
        seed()
        vals = linkx_flow(hm, uf, row, col, labels, features, n, to_dev, epochs)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    cpu = None
    if not args.no_cpu_baseline:
        from oracle import ref_shim
        rhm, ruf, _ = ref_shim.load()
        seed()
        t0 = time.perf_counter()
        ref_vals = linkx_flow(rhm, ruf, row, col, labels, features, n, lambda t: t, epochs)
        cpu_dt = time.perf_counter() - t0
        dev = {k: abs(vals[k] - ref_vals[k]) for k in vals}
        cpu = {"value": cpu_dt, "unit": "s", "cores": torch.get_num_threads(), "kind": "reference",
               "sample": "the full linkx workload, one pass of the unmodified reference on the host cores, same seeds",
               "abs_deviation_of_our_metrics": dev}
    h2d = nnz * 16 + n * (8 + 4 * LINKX_DIM)
    line = {"metric": "linkx_flow_seconds", "value": dt, "unit": "s", "n_gpus": 1, "steps": steps,
            "warmup": max(1, min(args.warmup, 2)), "ms_per_step": dt * 1e3, "higher_is_better": False,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": cfg,
            "cpu_baseline": cpu,
            "e2e": {"value": dt, "unit": "s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 8 * len(vals),
                    "note": "the flow starts from host tensors (as homophily_tests.py does) and ends with host scalars: "
                            "value IS the end-to-end time, host-side pinv / t-test / sampling included"},
            "gpu_launches": int((W.launch_count() - launches0) // steps), "metrics": vals,
            "kr_check": linkx_kr_check(hm, row, col, labels, features, n, device)}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------
def main():
    args = parse()
    if args.workload == "linkx":
        run_linkx(args)
        return
    if args.impl == "reference":
        run_reference(args)
        return

    import torch.distributed as dist
    import wdgh_b200 as W
    from wdgh_b200 import graph as G
    from wdgh_b200.sharded import CudaShardedStats, RowPartition

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    W._lib.require_device()
    sampler = ClockSampler(device)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)
    n, C, d = args.nodes, args.classes, args.dim
    part = RowPartition(n, world)
    r0, r1 = part.bounds(rank)

    rowptr, col, x_local, labels_local = gen_rows(r0, r1, n, args.avg_degree, C, args.homophily, d, device)
    torch.cuda.synchronize()
    nnz_local = int(col.shape[0])
    g = G.CSRGraph(rowptr, col, None, r1 - r0, row_offset=r0, n_global=n)
    _ = g.plan  # degree binning: built once per resident graph
    use_2d = world >= 2 and world % 2 == 0 and d % 4 == 0 and d >= 128 and args.partition in ("2d", "auto")
    if args.partition == "2d" and not use_2d:
        raise SystemExit("--partition 2d needs an even number of GPUs and d >= 128 (multiple of 4)")
    slice_graphs = None
    args._use_2d = use_2d
    if use_2d:
        from wdgh_b200.sharded import Cuda2DShardedStats, Grid2D
        grid2 = Grid2D(n, world, 2)
        slice_graphs = make_slice_graphs(G, grid2, rank, rowptr, col, args, device)
    nnz_t = torch.tensor([nnz_local], dtype=torch.int64, device=device)
    if world > 1:
        dist.all_reduce(nnz_t)
    nnz = int(nnz_t.item())

    pipe = None
    if world == 1:
        y = torch.empty((n, d), dtype=torch.float32, device=device)
        scratch = [None]

        def step():
            g._dinv.clear()
            dinv, _, code = g.degree_scale(W.NORM_SYM, True)
            _, scratch[0] = G.spmm_structure_fused(g, x_local, labels_local, C, W.NORM_SYM, True, out=y, dinv=dinv,
                                                   deg_code=code, scratch=scratch[0])
            return scratch[0][0], scratch[0][1]
    else:
        if use_2d:
            pipe = Cuda2DShardedStats(grid2, rank, slice_graphs, g, x_local, labels_local, C,
                                      overlap={"auto": None, "on": True, "off": False}[args.overlap])
            args._overlap = pipe.overlap
        else:
            pipe = CudaShardedStats(g, part, rank, x_local, labels_local, C,
                                    phased=(False if args.no_phased else None))

        def step():
            _, counters, node_sum = pipe.step(W.NORM_SYM, True)
            return counters, node_sum

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    trace_stages = os.environ.get("WDGH_STAGE_TIMES") == "1" and hasattr(pipe, "_trace")
    if trace_stages:
        pipe._trace = False           # the per-stage events synchronise every step: keep them out of the timed steps
    barrier()
    t_load0 = time.time()             # clock samples are kept from here (warm-up + timed steps, all under load)
    for _ in range(max(args.warmup, 3)):
        counters, node_sum = step()
    nvl0 = nvlink_bytes(device) if world > 1 and rank == 0 else None   # hardware NVLink counters around the timed steps
    barrier()                         # (read BEFORE the barrier: nvidia-smi takes ~0.1-0.5 s on rank 0)
    launches0 = W.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(args.steps):
        counters, node_sum = step()
    ev1.record()
    barrier()
    t_load1 = time.time()
    nvl1 = nvlink_bytes(device) if nvl0 is not None else None
    ms = ev0.elapsed_time(ev1) / args.steps
    launches = W.launch_count() - launches0
    clocks = sampler.stop(t_load0, t_load1)
    ms_t = torch.tensor([ms], dtype=torch.float64, device=device)
    if world > 1:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    ms = float(ms_t.item())
    value = nnz / (ms * 1e-3) / 1e9

    # ---- checksum of Y = A_hat X of the last step: sum and sum |.| over all ranks in float64.  The graph does not
    # depend on the partition, so N = 1, rows/N and the 2-D partition must print the same two numbers (~1e-7).
    y_last = y if world == 1 else pipe._y
    y_chk = torch.zeros(2, dtype=torch.float64, device=device)
    for a0 in range(0, r1 - r0, 1 << 20):
        blk = y_last[a0:min(a0 + (1 << 20), r1 - r0)]
        y_chk[0] += blk.sum(dtype=torch.float64)
        y_chk[1] += blk.abs().sum(dtype=torch.float64)
    if world > 1:
        dist.all_reduce(y_chk)
    y_chk = [float(v) for v in y_chk.tolist()]
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dump_rows(n, d), y_last, r0, r1, counters, node_sum, world)

    # ---- N > 1: EVERY element of Y against an independent path -- plain NCCL all-gather of the features into a
    # fresh buffer, then the N = 1 kernel in one launch on this rank's rows.  A wrong Y fails the run (exit 3).
    verify = None
    if world > 1 and not args.no_verify:
        from wdgh_b200.sharded import _all_gather_rows, _pad_rows
        blk_rows = part.block
        x_all = _all_gather_rows(_pad_rows(x_local, blk_rows), None)
        dv, _, cd = g.degree_scale(W.NORM_SYM, True)
        dv_all = _all_gather_rows(_pad_rows(dv, blk_rows), None)
        cd_all = _all_gather_rows(_pad_rows(cd, blk_rows), None)
        y_ref = G.spmm(g, x_all, W.NORM_SYM, True, dinv=dv_all, deg_code=cd_all)
        stat = torch.zeros(2, dtype=torch.float64, device=device)
        for a0 in range(0, r1 - r0, 1 << 20):
            a1 = min(a0 + (1 << 20), r1 - r0)
            diff = (y_last[a0:a1] - y_ref[a0:a1]).abs()
            diff = torch.where(torch.isnan(diff), torch.full_like(diff, float("inf")), diff)   # NaN must not hide
            stat[0] = torch.maximum(stat[0], diff.max().to(torch.float64))
            stat[1] = torch.maximum(stat[1], y_ref[a0:a1].abs().max().to(torch.float64))
        dist.all_reduce(stat, op=dist.ReduceOp.MAX)
        rel = float(stat[0].item() / max(float(stat[1].item()), 1e-30))
        verify = {"against": "NCCL all-gather + one-launch aggregation (every element of Y, all ranks)",
                  "max_abs_err_over_max_abs": rel, "tolerance": 5e-6, "ok": bool(rel <= 5e-6)}
        del x_all, y_ref, dv_all, cd_all
        torch.cuda.empty_cache()

    # ---- roofline of the dominant kernel (spmm_rowgroup_kernel), timed alone on this rank's shard ----
    if world == 1:
        xs = x_local
        dinv, _, code = g.degree_scale(W.NORM_SYM, True)
        ys = y
    elif not use_2d:
        xs, _, dinv = pipe.gather_inputs(W.NORM_SYM, True)
        code = pipe.code_full
        ys = torch.empty((g.n, d), dtype=torch.float32, device=device)
    if use_2d:
        # the aggregation kernels of this rank's block (pc row slices, raw partial sums), features already gathered
        dinv2, _, code2 = g.degree_scale(W.NORM_SYM, True)
        blk = part.block
        dinv_f = torch.zeros(world * blk, dtype=torch.float32, device=device)
        code_f = torch.zeros(world * blk, dtype=torch.uint8, device=device)
        dist.all_gather_into_tensor(dinv_f, torch.nn.functional.pad(dinv2, (0, blk - dinv2.shape[0])))
        dist.all_gather_into_tensor(code_f, torch.nn.functional.pad(code2, (0, blk - code2.shape[0])))

        x_cols = pipe.x_full.clone()       # the pipeline's own buffer is peer-visible: time on a private copy
        x_cols[torch.isnan(x_cols)] = 0.0  # blocks outside this rank's column group are never read
        out_slice = torch.empty((blk, d), dtype=torch.float32, device=device)

        def spmm_once():
            for si, sg in enumerate(slice_graphs):
                G.spmm_ranged(sg, sg.rowptr[:-1], sg.rowptr[1:], x_cols, out_slice, W.NORM_SYM, True,
                              dinv_f, code_f, pipe._skip[si], False, False, True)
        nnz_local = sum(sg.nnz for sg in slice_graphs)
        rows_local = sum(sg.n for sg in slice_graphs)
    else:
        def spmm_once():
            G.spmm(g, xs, W.NORM_SYM, True, out=ys, dinv=dinv, deg_code=code)
        rows_local = r1 - r0
    if trace_stages:                  # one extra, untimed step with per-stage CUDA events
        pipe._trace = True
        step()
        pipe._trace = False
    if getattr(pipe, "stage_ms", None) and os.environ.get("WDGH_STAGE_TIMES") == "1":
        print(f"[rank {rank}] stages: " + ", ".join(f"{k} {v:.2f}" for k, v in pipe.stage_ms), file=sys.stderr, flush=True)
    for _ in range(2):
        spmm_once()
    torch.cuda.synchronize()
    k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = max(3, min(args.steps, 10))
    k0.record()
    for _ in range(reps):
        spmm_once()
    k1.record()
    torch.cuda.synchronize()
    spmm_ms = k0.elapsed_time(k1) / reps
    # algorithmic bytes of one SpMM launch (DESIGN.md "SpMM roofline"): per stored entry a 4 B column id,
    # a 4 B D^-1/2 gather and a d*4 B feature-row gather; per row 8 B rowptr, 4 B scale, d*4 B self-loop
    # row and d*4 B output row (2-D partition: raw partial rows, no scale / self-loop read).
    if use_2d:
        alg_bytes = nnz_local * (4 + 4 + 4 * d) + rows_local * (8 + 4 * d)
    else:
        alg_bytes = nnz_local * (4 + 4 + 4 * d) + rows_local * (8 + 4 + 4 * d + 4 * d)
    achieved = alg_bytes / (spmm_ms * 1e-3) / 1e9
    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak, peak_src = float(mp["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except Exception:
        pass
    traffic = None
    try:
        traffic = json.load(open(os.path.join(ROOT, "profiles", "spmm_traffic.json"))).get("dram_bytes_per_entry")
        traffic = traffic * nnz_local if traffic is not None else None
    except Exception:
        pass
    roofline = {"kernel": "spmm_rowgroup_kernel<VEC=4,NCH=1,binary,FULL,32 CTAs/SM> (+ spmm_chunks / spmm_heavy_finish for split rows)"
                          + (": the pc row slices of this rank's block as raw partial sums, local stores" if use_2d else ""),
                "bound": "hbm", "achieved": achieved, "peak": peak,
                "unit": "GB/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                "kernel_ms": spmm_ms, "algorithmic_bytes": alg_bytes, "share_of_step": spmm_ms / ms,
                # DRAM bytes actually moved (ncu) / time / peak: stays below 1, whereas `frac` may exceed 1 slightly on a
                # box that is not power-capped -- its numerator counts ~5% of L2-served bytes (degree codes, repeated
                # feature rows) and its denominator is a read+write copy_, not the HBM pin rate (profiles/summary_r02.md)
                "traffic_frac": (traffic / (spmm_ms * 1e-3) / 1e9 / peak) if traffic else None,
                "traffic_source": "profiles/spmm_traffic.json: ncu dram__bytes_read.sum + dram__bytes_write.sum per stored "
                                  "entry of this kernel on a 16M-node instance of the same generator, times this launch's entries"}

    # ---- NVLink: bytes per step from the hardware counters of rank 0's GPU next to what the partition predicts ----
    nvlink = None
    if world > 1:
        shard_bytes = part.block * d * 4
        expect = ((1 + (world // 2 - 1)) if use_2d else (world - 1)) * shard_bytes    # per direction and step
        nvlink = {"expected_bytes_per_direction_per_step": int(expect),
                  "expected_gbs_over_step": expect / (ms * 1e-3) / 1e9,
                  "reference_peer_copy_gbs": 770.0, "note": "B200_PROFILING.md: measured peer copy 770 GB/s per direction"}
        if nvl0 is not None and nvl1 is not None:
            tx, rx = (nvl1[0] - nvl0[0]) / args.steps, (nvl1[1] - nvl0[1]) / args.steps
            nvlink.update(tx_bytes_per_step=tx, rx_bytes_per_step=rx, tx_gbs_over_step=tx / (ms * 1e-3) / 1e9,
                          rx_gbs_over_step=rx / (ms * 1e-3) / 1e9, source="nvidia-smi nvlink -gt d, rank 0's GPU")

    # ---- metrics of the last step (sanity; also proves the counters left the device) ----------------
    h = counters.cpu().numpy()
    metrics = {"edge_homophily_with_self_loops": float((h[0] + n) / (nnz + n)),
               "node_homophily": float(node_sum[0].item() / max(int(h[G._lib.SC_N_NODES_NSL]), 1)),
               "class_pair_hist_total": int(h[G._lib.SC_HEADER + 2 * C:G._lib.SC_HEADER + 2 * C + C * C].sum()),
               "y_sum": y_chk[0], "y_abs_sum": y_chk[1]}

    # ---- e2e: host buffers through the C ABI, copies inside the timed region ------------------------
    e2e = None
    stage_ms = getattr(pipe, "stage_ms", None)
    if not args.no_e2e:
        if world > 1:
            # The e2e arm builds its own (1-D, host-staged) pipeline with a second peer-mapped feature buffer.  Release
            # everything the device-resident part allocated first -- the 2-D pipeline alone holds the full-size
            # x_full (25.6 GB on every rank) and the receive slots -- and agree COLLECTIVELY whether the rest fits: a rank
            # that ran out of memory alone would leave its peers hanging in a collective.
            import gc
            pipe = slice_graphs = y_last = None
            xs = ys = dinv = code = None
            if use_2d:
                x_cols = out_slice = dinv_f = code_f = dinv2 = code2 = None
            gc.collect()
            torch.cuda.empty_cache()
            free_b, _ = torch.cuda.mem_get_info(device)
            rows_l = r1 - r0
            need = (part.padded * d * 4                      # the e2e pipeline's peer-mapped feature buffer
                    + 3 * rows_l * d * 4                      # staged features, Y, and slack for scratch
                    + (world + 2) * rows_l * 8                # column segments per source rank
                    + 3 * (int(g.rowptr.numel()) * 8 + int(g.col.numel()) * 4))
            ok = torch.tensor([1 if free_b >= 1.15 * need else 0], dtype=torch.int32, device=device)
            dist.all_reduce(ok, op=dist.ReduceOp.MIN)
            if int(ok.item()) == 0:
                e2e = {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                       "note": f"skipped: {free_b / 1e9:.0f} GB free on rank {rank} after releasing the device-resident "
                               f"pipeline, the host-staged pipeline needs ~{need / 1e9:.0f} GB"}
        if e2e is None:
            e2e = run_e2e(args, W, G, world, rank, device, g, x_local, labels_local, nnz, part)

    # ---- secondary rooflines (N = 1): the label pass (HBM) and the tcgen05 Gram (tensor pipe) -------
    roofline_labels = roofline_gram = None
    if world == 1:
        roofline_labels = time_label_pass(G, g, labels_local, C, nnz, n, peak, peak_src)
        roofline_gram = time_gram(G, device)

    # ---- CPU baseline (rank 0, N = 1): the reference's own CPU path on a bounded sample --------------
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        import warnings
        warnings.filterwarnings("ignore")
        kind, once = load_cpu_arm()
        rp, cl, xx, lb, n_s = cpu_sample(args, device)
        once(rp, cl, xx, lb, n_s)
        t0 = time.perf_counter()
        reps_cpu = 2
        for _ in range(reps_cpu):
            once(rp, cl, xx, lb, n_s)
        dt = (time.perf_counter() - t0) / reps_cpu
        cpu_baseline = {"value": cl.shape[0] / dt / 1e9, "unit": UNIT, "cores": torch.get_num_threads(),
                        "kind": kind, "sample": cpu_sample_text(kind, n_s, cl.shape[0], args) +
                        f"; {reps_cpu} timed passes, {dt:.2f} s each"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": max(args.warmup, 3), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, nnz),
                "roofline": roofline, "roofline_labels": roofline_labels, "roofline_gram": roofline_gram,
                "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": int(launches),
                "clocks": clocks, "metrics": metrics, "verify": verify, "nvlink": nvlink,
                "stage_ms": stage_ms}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if verify is not None and not verify["ok"]:
        sys.exit(3)   # a fast wrong answer is not a result


def time_label_pass(G, g, labels32, C, nnz, n, peak, peak_src):
    """Label statistics alone (pack + edge pass + split rows), CUDA events.  Algorithmic bytes: 4 B of `col` per stored
    entry; per node 8 B rowptr, 4 B label in, 1 B packed label out + in, 2 x 4 B per-node counts out (DESIGN.md 4)."""
    scratch = None
    for _ in range(3):
        scratch = G.structure_counts_raw(g, labels32, C, scratch)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    e0.record()
    for _ in range(reps):
        scratch = G.structure_counts_raw(g, labels32, C, scratch)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    alg = nnz * 4 + n * (8 + 4 + 1 + 1 + 4 + 4)
    ach = alg / (ms * 1e-3) / 1e9
    return {"kernel": "labels_to_u8 + structure_stream_kernel (+ structure_chunks / heavy_nodes for split rows)",
            "bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": None,
            "peak_source": peak_src, "kernel_ms": ms, "algorithmic_bytes": alg}


def time_gram(G, device, m=8192, d=1024):
    """G = Z Z^T on tcgen05 (3xTF32 split, fp32-faithful chunked accumulation), the shape VERDICT r01 names.
    `achieved` counts the TF32 FLOPs the tensor pipe executes (3 products per fp32 product, upper triangle only:
    3 * m * (m + 128) * d); peak = half the measured dense bf16 rate (kind::tf32 runs at half the bf16 rate)."""
    z = torch.randn(m, d, device=device)
    for _ in range(3):
        G.gram(z, use_tensor_cores=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    e0.record()
    for _ in range(reps):
        G.gram(z, use_tensor_cores=True)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    peak, src = 0.5 * 1590.0, "fallback (B200_PROFILING.md), bf16 / 2"
    try:
        mp = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        peak, src = 0.5 * float(mp["bf16_tflops"]), "MEASURED_PEAKS.json bf16_tflops / 2 (tf32 runs at half the bf16 rate)"
    except Exception:
        pass
    executed = 3.0 * m * (m + 128) * d / (ms * 1e-3) / 1e12
    useful = 2.0 * m * m * d / (ms * 1e-3) / 1e12
    return {"kernel": "gram_split_kernel + gram_tcgen05_kernel", "bound": "tensor", "achieved": executed, "peak": peak,
            "unit": "TFLOP/s", "frac": executed / peak, "traffic": None, "peak_source": src, "kernel_ms": ms,
            "shape": [m, d], "useful_fp32_equivalent_tflops": useful}


def run_e2e(args, W, G, world, rank, device, g, x_local, labels_local, nnz, part):
    """Same metric from HOST buffers, results back in HOST buffers: N = 1 goes through wdgh_pipeline_host (the C-ABI
    entry a reference user binds) with the counters AND Y = A_hat X copied back; N > 1 stages this rank's shard from
    pinned memory, runs the sharded step and copies the rank's Y rows and the counters back."""
    import torch.distributed as dist
    lib = W._lib.lib
    n, d, C = args.nodes, args.dim, args.classes
    rows = g.n
    steps = max(1, min(args.steps, 3))

    def pinned(t):
        return torch.empty(t.shape, dtype=t.dtype, pin_memory=True).copy_(t)

    try:
        rowptr_h, col_h, x_h, lab_h = pinned(g.rowptr), pinned(g.col), pinned(x_local), pinned(labels_local)
        y_h = torch.empty((rows, d), dtype=torch.float32, pin_memory=True)
    except RuntimeError as e:  # not enough pinnable host memory for this size
        return {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "note": f"host staging failed: {str(e)[:80]}"}
    h2d = rowptr_h.numel() * 8 + col_h.numel() * 4 + x_h.numel() * 4 + lab_h.numel() * 4
    n_cnt = G._lib.sc_words(C)
    d2h_small = n_cnt * 8 + 16
    d2h = d2h_small + y_h.numel() * 4
    extra = {}
    if world == 1:
        counters_h = torch.zeros(n_cnt, dtype=torch.int64).pin_memory()
        node_sum_h = torch.zeros(2, dtype=torch.float64).pin_memory()

        def once(y_ptr):
            W._lib.check(lib.wdgh_pipeline_host(rowptr_h.data_ptr(), col_h.data_ptr(), n, g.nnz, x_h.data_ptr(), d,
                                                lab_h.data_ptr(), C, W.NORM_SYM, 1, y_ptr, counters_h.data_ptr(),
                                                node_sum_h.data_ptr()), "wdgh_pipeline_host")

        def timed(y_ptr):
            once(y_ptr)
            t0 = time.perf_counter()
            for _ in range(steps):
                once(y_ptr)
            return (time.perf_counter() - t0) / steps
        dt_small = timed(None)            # counters only: Y stays on the device (what round 1 reported)
        dt = timed(y_h.data_ptr())        # the headline: Y = A_hat X back in host memory as well
        lib.wdgh_pipeline_host_release()
        assert int(counters_h[G._lib.SC_N_LAB]) == nnz
        extra = {"metrics_only": {"value": nnz / dt_small / 1e9, "unit": UNIT, "ms_per_step": dt_small * 1e3,
                                  "d2h_bytes_per_step": int(d2h_small),
                                  "note": "same call with y_host = NULL: Y stays resident for the downstream metrics"},
                 "y_host_checksum": float(y_h[:1 << 20].sum(dtype=torch.float64))}
    else:
        from wdgh_b200.sharded import CudaShardedStats

        # persistent device buffers; every step refills them from pinned host memory, rebuilds the plan /
        # degree scales / column segments and runs the sharded step (peer mappings are set up once)
        gg = G.CSRGraph(torch.empty_like(g.rowptr), torch.empty_like(g.col), None, rows, row_offset=g.row_offset,
                        n_global=n)
        x_dev = torch.empty_like(x_local)
        lab_dev = torch.empty_like(labels_local)
        pipe = CudaShardedStats(gg, part, rank, x_dev, lab_dev, C, phased=(False if args.no_phased else None))

        def once():
            gg.rowptr.copy_(rowptr_h, non_blocking=True)
            gg.col.copy_(col_h, non_blocking=True)
            pipe.x_local[:rows].copy_(x_h, non_blocking=True)
            pipe.labels_local[:rows].copy_(lab_h, non_blocking=True)
            pipe.reset_graph()
            y_dev, counters, node_sum = pipe.step(W.NORM_SYM, True)
            y_h.copy_(y_dev, non_blocking=True)
            return counters.cpu(), node_sum.cpu()
        once()
        dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            once()
        torch.cuda.synchronize()
        dist.barrier()
        dt = (time.perf_counter() - t0) / steps
        t = torch.tensor([dt], dtype=torch.float64, device=device)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    out = {"value": nnz / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
           "steps": steps, "ms_per_step": dt * 1e3,
           "entry": "wdgh_pipeline_host (C ABI, pinned host buffers in, counters + Y out)" if world == 1 else
                    "pinned host shard -> device -> sharded step (1-D, peer pulls) -> Y rows + counters to host"}
    out.update(extra)
    return out


if __name__ == "__main__":
    main()
