"""The datasets the reference ships -- Cora, citeseer (Planetoid files) and the heterophilous texas / cornell / wisconsin /
film graphs (new_data/*) -- loaded by the reference's own loaders and pushed through the homophily_tests.py
small-dataset flow by tests/golden/make_golden.py; here the CUDA path replays the same inputs.

Kept in its own module, collected after test_gpu_parity.py.  The KR metric is compared prediction by prediction on
every dataset (test_gpu_parity.check_kr): there is no tie-sensitive exception list.
"""
import numpy as np
import pytest
import torch

import _golden as G
from test_gpu_parity import W, check_ax, check_gram, check_kr, check_structure, close, sparse  # noqa: F401

pytestmark = pytest.mark.gpu

DATASETS = ["cora", "ds_citeseer", "ds_cornell", "ds_texas", "ds_film", "ds_wisconsin"]


@pytest.mark.parametrize("name", DATASETS)
def test_reference_datasets(W, name):
    """Cora + the other datasets the reference ships (citeseer, texas, cornell, wisconsin, film) through the
    homophily_tests.py small-dataset flow, against the unmodified reference's outputs."""
    uf, hm = W.util_funcs, W.homophily_metrics
    z = G.load(name)
    n = int(z["in_n"])
    labels = z["in_labels"]
    ei = z["in_edge_index"].astype(np.int64)
    x_raw = G.cora_dense_features(z)
    x = uf.normalize_tensor(torch.from_numpy(x_raw))          # homophily_tests.py:80
    close(x.double().sum(1), z["out_features_rownorm_rowsum"], rtol=1e-5)
    ones = np.ones(ei.shape[1], np.float32)
    A_raw = sparse(ei[0], ei[1], ones, n)
    for sym in (0, 1):
        row, col, val = G.dense_normalized_with_self_loops(z, sym)
        A = sparse(row, col, val, n)
        check_structure(W, z, A, row, col, labels, n, f"__sym{sym}")
        close(hm.generalized_edge_homophily(A, x, torch.from_numpy(labels)), z[f"out_gen_edge_homo__sym{sym}"])
        check_ax(z, W.spmm(hm._as_graph(A), x), x.shape[1], f"norm__sym{sym}")
        # the same A_hat X without materialising A_hat: on-the-fly normalisation of the raw graph
        g_raw = W.CSRGraph.from_torch_sparse(A_raw, binary=True)
        y = W.spmm(g_raw, x, W.NORM_SYM if sym else W.NORM_RW, True)
        check_ax(z, y, x.shape[1], f"norm__sym{sym}")
    check_gram(W, z, A_raw, x_raw, labels)
    check_kr(W, z, A_raw, x_raw, labels)
    # LINKX flow normalisers (homophily_tests.py:99-104)
    for key, fn, tag in (("out_sys_norm_values", uf.sys_normalized_adjacency, "sys"),
                          ("out_row_norm_values", uf.row_normalized_adjacency, "rw")):
        gn = fn(A_raw)
        t = uf.sparse_mx_to_torch_sparse_tensor(gn)
        assert np.array_equal(t.indices().cpu().numpy(), z["out_sys_norm_index"])
        close(t.values(), z[key], rtol=1e-6)
        check_ax(z, W.spmm(gn, x), x.shape[1], tag)
        check_ax(z, uf.propagate(A_raw, x, symmetric=(tag == "sys")), x.shape[1], tag)


@pytest.mark.timeout(900)
@pytest.mark.parametrize("name", G.names("linkx_"))
def test_linkx_facebook100(W, name):
    """facebook100 graphs shipped with the reference (Reed98, Amherst41, Johns Hopkins55, Cornell5), loaded by its
    load_fb100_dataset (gender label, -1 = unlabelled) and pushed through the large-dataset flow of
    homophily_tests.py:88-137 by tests/golden/make_golden.py::case_linkx; the CUDA path replays the same inputs."""
    import random
    uf, hm = W.util_funcs, W.homophily_metrics
    z = G.load(name)
    n = int(z["in_n"])
    labels = z["in_labels"]
    lab_t = torch.from_numpy(labels)
    row, col = G.linkx_graph(z)
    A_raw = sparse(row, col, np.ones(row.shape[0], np.float32), n)
    x_raw = torch.from_numpy(z["in_features"].astype(np.float32))
    x = G.l1_normalize(x_raw)                                     # homophily_tests.py:95 (torch, host side upstream too)
    close(x[:: max(1, n // 64)], z["out_features_l1"], rtol=1e-6)
    for sym, fn in ((1, uf.sys_normalized_adjacency), (0, uf.row_normalized_adjacency)):
        sfx = f"__sym{sym}"
        gn = fn(A_raw)                                            # :98-104
        t = uf.sparse_mx_to_torch_sparse_tensor(gn).coalesce()
        close(t.values()[:4096], z["out_adj_values_head" + sfx], rtol=1e-6)
        close(t.values().double().sum(), z["out_adj_values_sum" + sfx], rtol=1e-7)
        ti = t.indices().cpu().numpy()
        check_structure(W, z, t, ti[0], ti[1], labels, n, sfx)    # :108-116 metric dispatch, integers exact
        random.seed(3), np.random.seed(3), torch.manual_seed(3)
        close(hm.generalized_edge_homophily(t, x, lab_t), z["out_gen_edge_homo" + sfx], rtol=1e-4, atol=1e-6)
        check_ax(z, W.spmm(gn, x), x.shape[1], "norm" + sfx)      # SGC-1 propagation, materialised A_hat
        check_ax(z, uf.propagate(A_raw, x, symmetric=sym), x.shape[1], "norm" + sfx)   # ... and on the fly
    num_sample = int(z["in_num_sample"])
    cmax = int(labels.max()) + 1
    oh = torch.eye(cmax)[lab_t]
    for hard, key in ((None, "soft"), (1, "hard")):
        seed = int(z["in_agg_seed"])
        random.seed(seed), np.random.seed(seed), torch.manual_seed(seed)
        las = np.zeros(10)
        m = n
        for i in range(10):
            idx = None
            if n >= num_sample:
                idx, _, _ = uf.random_disassortative_splits(lab_t, lab_t.max() + 1, num_sample / n)
                m = int(idx.sum())
            las[i] = 2 * float(hm.similarity(oh, A_raw, oh, hard=hard, LP=1, idx_train=idx)) - 1
        close(las, z[f"out_agg_homo_{key}_las"], rtol=0, atol=2 * 1.5 / m)
    if "out_kr_p_gnb" in z.files:
        check_kr(W, z, A_raw, x_raw.numpy(), labels)


def test_kr_svm_classifiers(W):
    """hm.py:312-333: the SVM base classifiers (rbf / poly / linear) of the KR metric on texas -- A X and the row
    gathers come from the GPU, sklearn runs on the host as upstream; per-epoch accuracies equal the reference's."""
    import random
    z, s = G.load("ds_texas"), G.load("svm_texas")
    n, labels = int(z["in_n"]), z["in_labels"]
    ei = z["in_edge_index"].astype(np.int64)
    x = G.cora_dense_features(z)
    A = sparse(ei[0], ei[1], np.ones(ei.shape[1], np.float32), n)
    for clf in ("svm_rbf", "svm_poly", "svm_linear"):
        seed = int(s["in_kr_seed"])
        random.seed(seed), np.random.seed(seed), torch.manual_seed(seed)
        trace = []
        p, _ = W.homophily_metrics.classifier_based_performance_metric(
            torch.from_numpy(x), A, torch.from_numpy(labels), int(s["in_kr_sample_max"]), base_classifier=clf,
            epochs=int(s["in_kr_epochs"]), _trace=trace)
        np.testing.assert_allclose([t["acc_g"] for t in trace], s[f"out_kr_acc_g_{clf}"], rtol=0, atol=1e-7)
        np.testing.assert_allclose([t["acc_x"] for t in trace], s[f"out_kr_acc_x_{clf}"], rtol=0, atol=1e-7)
        close(p, s[f"out_kr_p_{clf}"], rtol=1e-6, atol=1e-12)


def golden_synthesis_archive(path):
    """The data_synthesis graphs stored in the golden fixtures (syn_* and plot_syn_*), packed like
    oracle/build_ref.py packs the reference's 580: {"<size>/<h>/<s>/edges": int16 [2, nnz], ".../labels": int8 [n]}."""
    out = {}
    for name in G.names("syn_") + G.names("plot_syn_"):
        z = G.load(name)
        key = "/".join(name.split("_")[-3:])
        out[key + "/edges"] = z["in_edge_index"].astype(np.int16)
        out[key + "/labels"] = z["in_labels"].astype(np.int8)
    np.savez(path, **out)
    return len(out) // 2


@pytest.mark.timeout(3000)
def test_data_synthesis_sweep(W, tmp_path):
    """synthetic_plot.py:60-110 over the data_synthesis graphs the reference ships (tools/sweep_synthesis.py): every
    metric against the oracle on a subset spread over both sizes and the whole h range; WDGH_FULL_SWEEP=1 replays all
    580 graphs (slow: the CPU oracle needs minutes).  Without the packed archive (oracle/build_ref.py, made from the
    reference) the sweep replays the six data_synthesis graphs of the golden fixtures."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    archive = os.path.join(root, "oracle", "_ref", "data_synthesis.npz")
    if os.path.exists(archive):
        limit = "0" if os.environ.get("WDGH_FULL_SWEEP") == "1" else "12"
        expect = 580 if limit == "0" else 12
    else:
        archive = str(tmp_path / "data_synthesis.npz")
        limit, expect = "0", golden_synthesis_archive(archive)
    out = subprocess.run([sys.executable, os.path.join(root, "tools", "sweep_synthesis.py"), "--limit", limit,
                          "--archive", archive], capture_output=True, text=True, timeout=2900, cwd=root)
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith('{"sweep"')]
    assert out.returncode == 0 and lines, out.stdout[-1500:] + out.stderr[-1500:]
    rep = json.loads(lines[-1])
    assert rep["ok"] and rep["graphs"] == expect and rep["kr"]["flips_outside_unstable"] == 0
