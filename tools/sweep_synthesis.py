#!/usr/bin/env python
"""Replay the reference's data_synthesis sweep (synthetic_plot.py:60-110) on the CUDA path, graph by graph, next to
the CPU oracle:

    python tools/sweep_synthesis.py [--limit N] [--kr-epochs E] [--out profiles/sweep_r02.json]
    python tools/sweep_synthesis.py --dump gpurun_out/sweep_gpu.pt          # GPU box: CUDA path only
    python tools/sweep_synthesis.py --compare gpurun_out/sweep_gpu.pt --out profiles/sweep_r02.json   # anywhere: oracle + checks

Input: oracle/_ref/data_synthesis.npz -- the 580 graphs the reference ships under data_synthesis/{800,4000}/<h>/
(2000 nodes, 5 classes, h swept 0.05 .. 0.9, 10 samples each), packed by oracle/build_ref.py (git-ignored, travels with
the repo to the GPU box).  The feature files the reference's script loads (data_synthesis/features/*) are shipped
EMPTY, so features are class-conditional Gaussians drawn from a per-graph seed, then `preprocess_features`-normalised
as synthetic_plot.py:82 does.  Per graph the flow is the script's: adj = normalize(adj + I) (dense), then
edge / node / class homophily, soft LAS aggregation homophily, adjusted homophily, label informativeness, generalised
edge homophily, and the KR metric with the linear and the arccos kernel (`--kr-epochs` epochs instead of the script's
100, identical per-epoch work).

Every scalar metric is compared with the oracle (test infrastructure; this tool is a checker, not product code); KR is
compared prediction by prediction with the contract of tests/test_gpu_parity.py::kr_contract.  Prints ONE JSON line
with the worst deviations and the wall time of the CUDA path and of the CPU oracle over the same graphs, exits 1 on a
violation.
"""
import argparse
import json
import os
import random
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _p in (ROOT, os.path.join(ROOT, "when-do-gnns-help_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

TOL = {"edge_homo": 1e-6, "node_homo": 1e-6, "class_homo": 1e-5, "soft_las": 1.5 / 2000, "adj_homo": 1e-4,
       "label_info": 1e-4, "gen_edge_homo": 1e-4}


def seed_all(s):
    random.seed(s), np.random.seed(s), torch.manual_seed(s)


def graphs(archive, limit):
    keys = sorted({k.rsplit("/", 1)[0] for k in archive.files})
    if limit and limit < len(keys):           # spread the subset over both sizes and the whole h range
        keys = [keys[i] for i in np.linspace(0, len(keys) - 1, limit).astype(int)]
    for k in keys:
        yield k, archive[k + "/edges"].astype(np.int64), archive[k + "/labels"].astype(np.int64)


def features_for(key, labels, d=32):
    # Python's str hash is salted per process: derive the per-graph seed from the key's bytes
    g = torch.Generator().manual_seed(int.from_bytes(key.encode(), "little") % (2 ** 31 - 1))
    c = int(labels.max()) + 1
    centers = torch.randn(c, d, generator=g)
    # non-negative like the bag-of-words features of the reference's base datasets: `preprocess_features` divides by
    # the row SUM, which for signed noise can be ~0 and blows single rows up by 1e3
    return (centers[torch.from_numpy(labels)] + 1.5 * torch.randn(labels.shape[0], d, generator=g)).abs().float()


def gpu_side(W, key, n_graphs, labels, ei, args):
    """The CUDA path on one graph -> ({metric: value}, {clf: [epoch dicts]}, seconds)."""
    hp, uf = W.homophily_plot, W.util_funcs
    n = labels.shape[0]
    c = int(labels.max()) + 1
    feats_raw = features_for(key, labels)
    a0 = torch.zeros(n, n)
    a0[ei[0], ei[1]] = 1.0
    lab_t = torch.from_numpy(labels)
    label = torch.eye(c)[lab_t]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    feats = uf.preprocess_features(feats_raw)
    feats = feats if isinstance(feats, torch.Tensor) else torch.as_tensor(np.asarray(feats))
    adj = uf.normalize((a0 + torch.eye(n)).cuda())
    got = {"edge_homo": float(hp.edge_homophily(adj, label)), "node_homo": float(hp.node_homophily(adj, lab_t)),
           "class_homo": float(hp.our_measure(adj, lab_t)),
           "soft_las": float(hp.similarity(label, adj, label, NTK=None, hard=None, LP=1)),
           "adj_homo": float(hp.adjusted_homo(adj, label)), "label_info": float(hp.label_informativeness(adj, label)),
           "gen_edge_homo": float(hp.generalized_edge_homophily(adj, feats, label))}
    traces = {}
    for clf in ("kernel_reg0", "kernel_reg1"):
        seed_all(1000 + n_graphs)
        traces[clf] = []
        hp.classifier_based_performance_metric(feats, adj, lab_t, args.kr_sample_max, base_classifier=clf,
                                               epochs=args.kr_epochs, _trace=traces[clf])
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    slim = {clf: [{"va": t["va"].cpu(), "pred_g": t["pred_g"].cpu(), "pred_x": t["pred_x"].cpu()} for t in tr]
            for clf, tr in traces.items()}
    return got, slim, dt


def cpu_side(O, key, n_graphs, labels, ei, args, with_kr=True):
    """The CPU oracle on one graph -> ({metric: value}, {clf: [epoch dicts]}, exact-tie node count, seconds).
    with_kr=False: scalar metrics only (the KR oracle and its perturbation analysis dominate the CPU time)."""
    n = labels.shape[0]
    c = int(labels.max()) + 1
    feats_raw = features_for(key, labels)
    a0 = torch.zeros(n, n)
    a0[ei[0], ei[1]] = 1.0
    t0 = time.perf_counter()
    x = O.normalize_tensor(feats_raw.numpy()).numpy()
    a = a0 + torch.eye(n)
    a = (1.0 / a.sum(1))[:, None] * a
    sp_ = a.to_sparse().coalesce()
    row, col, val = sp_.indices()[0].numpy(), sp_.indices()[1].numpy(), sp_.values().numpy()
    oh = np.eye(c, dtype=np.float32)[labels]
    p, p_bar, pc = O.class_distribution(row, col, labels, n)
    s2 = np.float32(np.sum(p_bar.astype(np.float32) ** 2, dtype=np.float32))
    eh = O.plot_edge_homophily(row, col, val, oh)
    ref = {"edge_homo": float(eh), "node_homo": float(O.plot_node_homophily(row, col, labels, n)),
           "class_homo": float(O.plot_class_homophily(row, col, val, labels, n)),
           "soft_las": float(O.plot_similarity(oh, row, col, val, n, oh)),
           "adj_homo": float((eh - s2) / (1 - s2)), "label_info": float(O.label_informativeness(row, col, labels, n)),
           # hp.py:56-65 takes the all-entries branch whenever nnodes < 20000, whatever the entry count
           "gen_edge_homo": float(O.generalized_edge_homophily(row, col, x, n, sample_max=1 << 62))}
    ref_traces = {}
    for clf in ("kernel_reg0", "kernel_reg1") if with_kr else ():
        seed_all(1000 + n_graphs)
        ref_traces[clf] = []
        O.plot_kr_metric(x, a, labels, args.kr_sample_max, clf, args.kr_epochs, trace=ref_traces[clf])
    dt = time.perf_counter() - t0
    # soft LAS is a mean of per-node indicators `ratio >= 1`; on these graphs some nodes sit on an EXACT tie (e.g. one
    # neighbour of every class: ratio = 1 in exact arithmetic), where float32 rounding decides.  Those nodes are counted
    # in float64 (untimed) and may flip, every other node must agree (1.5 / n on top, as in the golden tests).
    near = O.similarity_near_ties(oh, row, col, val, n, oh)
    return ref, ref_traces, near, dt


def compare(O, key, n, got, traces, ref, ref_traces, near, worst, kr, bad):
    for k, tol in TOL.items():
        if k == "soft_las":
            tol = tol + near / n
        # label informativeness is 2 - ratio with the ratio near 2 at low h: absolute, like the golden tests (1e-5)
        dev = abs(got[k] - ref[k]) / (1.0 if k == "soft_las" else 0.1 if k == "label_info" else max(abs(ref[k]), 1e-3))
        worst[k] = max(worst[k], dev)
        if not dev <= tol:
            bad.append((key, k, got[k], ref[k]))
    for clf in ref_traces:
        for e, (g_, r_) in enumerate(zip(traces[clf], ref_traces[clf])):
            if not torch.equal(g_["va"].cpu(), r_["va"]):
                bad.append((key, clf, "validation sets differ", e))
                continue
            kr["epochs_compared"] += 1
            same = True
            for side, kname in (("pred_g", "gram_g"), ("pred_x", "gram_x")):
                changed = g_[side].cpu() != r_[side]
                if bool(changed.any()):
                    same = False
                    outside, _, n_esc = O.kr_flips_outside_unstable(changed, r_[kname], r_["n_layers"], r_["tr"], r_["va"],
                                                                    r_["onehot_tr"])
                    kr["flips"] += int(changed.sum())
                    kr["escalated_analyses"] = kr.get("escalated_analyses", 0) + n_esc
                    kr["flips_outside_unstable"] += outside
                    if outside:
                        bad.append((key, clf, side, e, outside))
            kr["epochs_identical"] += int(same)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--limit", type=int, default=0, help="number of graphs (0 = all of the archive)")
    ap.add_argument("--archive", default=os.path.join("oracle", "_ref", "data_synthesis.npz"),
                    help="graphs to replay, packed as oracle/build_ref.py packs them (relative paths: from the repo root)")
    ap.add_argument("--kr-epochs", type=int, default=2)
    ap.add_argument("--kr-sample-max", type=int, default=500)
    ap.add_argument("--out", default="")
    ap.add_argument("--dump", default="", help="CUDA path only: store every metric and KR prediction in this file "
                    "(torch.save) -- the GPU box's minutes go to the GPU path, the CPU oracle compares elsewhere")
    ap.add_argument("--compare", default="", help="CPU oracle only: check a --dump file (needs no GPU and no libwdgh)")
    ap.add_argument("--kr-every", type=int, default=1, help="run the KR oracle + per-prediction contract on every K-th "
                    "graph only (the scalar metrics are always compared on every graph); the perturbation analysis "
                    "of one graph costs minutes on a small host")
    args = ap.parse_args()
    import warnings
    warnings.filterwarnings("ignore")

    from oracle import ref_port as O
    W = None
    if not args.compare:
        import wdgh_b200 as W
    path = os.path.join(ROOT, args.archive)
    if not os.path.exists(path):
        print(json.dumps({"sweep": "data_synthesis", "unavailable": f"{args.archive} is missing "
                          "(python oracle/build_ref.py packs it from the reference)"}))
        return 0
    archive = np.load(path)
    worst = {k: 0.0 for k in TOL}
    kr = {"epochs_compared": 0, "epochs_identical": 0, "flips": 0, "flips_outside_unstable": 0}
    t_gpu = t_cpu = 0.0
    n_graphs, bad, near_ties_total, kr_graphs = 0, [], 0, 0
    dumped = torch.load(os.path.join(ROOT, args.compare)) if args.compare else None
    if dumped is not None:
        args.limit, args.kr_epochs, args.kr_sample_max = dumped["limit"], dumped["kr_epochs"], dumped["kr_sample_max"]
    store = {"limit": args.limit, "kr_epochs": args.kr_epochs, "kr_sample_max": args.kr_sample_max, "graphs": {}}
    launches0 = W.launch_count() if W is not None else 0
    for key, ei, labels in graphs(archive, args.limit):
        n = labels.shape[0]
        if dumped is None:
            got, traces, dt = gpu_side(W, key, n_graphs, labels, ei, args)
        else:
            got, traces, dt = dumped["graphs"][key]
        t_gpu += dt
        if args.dump:
            store["graphs"][key] = (got, traces, dt)
        else:
            with_kr = n_graphs % max(args.kr_every, 1) == 0
            kr_graphs += int(with_kr)
            ref, ref_traces, near, dt_c = cpu_side(O, key, n_graphs, labels, ei, args, with_kr)
            t_cpu += dt_c
            near_ties_total += near
            compare(O, key, n, got, traces, ref, ref_traces, near, worst, kr, bad)
        n_graphs += 1
    if args.dump:
        store["gpu_launches"] = int(W.launch_count() - launches0)
        torch.save(store, os.path.join(ROOT, args.dump))
        print(json.dumps({"sweep": "data_synthesis (synthetic_plot.py:60-110), CUDA path only", "graphs": n_graphs,
                          "gpu_path_wall_s": round(t_gpu, 3), "gpu_launches": store["gpu_launches"],
                          "dump": args.dump}), flush=True)
        return 0
    line = {"sweep": "data_synthesis (synthetic_plot.py:60-110)", "graphs": n_graphs, "kr_epochs": args.kr_epochs,
            "gpu_path_wall_s": round(t_gpu, 3), "cpu_oracle_wall_s": round(t_cpu, 3),
            "speedup_wall": round(t_cpu / max(t_gpu, 1e-9), 2), "worst_relative_deviation": worst, "tolerance": TOL,
            "soft_las_exact_tie_nodes": near_ties_total, "kr": dict(kr, graphs_checked=kr_graphs),
            "gpu_launches": int(W.launch_count() - launches0) if W is not None else dumped.get("gpu_launches"),
            "violations": [str(b) for b in bad[:10]], "ok": not bad,
            "note": "both walls include the host-side parts the reference keeps on the host (pinv, t-test, RNG); "
                    "2000-node graphs are launch- and host-bound, not bandwidth-bound"
                    + ("; the CUDA path ran on the B200 box (--dump), the oracle comparison on other host cores "
                       "(--compare): the two walls are not from the same machine" if dumped is not None else "")}
    print(json.dumps(line), flush=True)
    if args.out:
        with open(os.path.join(ROOT, args.out), "w") as f:
            json.dump(line, f, indent=1)
    return 0 if not bad else 1


if __name__ == "__main__":
    sys.exit(main())
