"""Drop-in mirror of the reference's `utils/homophily_metrics.py` on the B200 path.

Same function names, argument order, defaults and error behaviour as
/root/reference/utils/homophily_metrics.py (cited per function as hm.py:LINE);
`homophily_tests.py`, `synthetic_plot.py` and friends keep calling

    edge_homophily(A, labels), node_homophily(A, labels), our_measure(edge_index, label),
    adjusted_homo(A, label), label_informativeness(A, label),
    generalized_edge_homophily(adj, features, label), similarity(features, adj, label, ...),
    classifier_based_performance_metric(features, adj, labels, sample_max, ...)

All graph-sized work (edge passes, A_hat X, Gram matrices) runs in the CUDA kernels
of libwdgh_b200.so through the C ABI; what stays on the host is what the reference
itself does on the host (RNG-driven sampling, `np.linalg.pinv`, sklearn, scipy's t-test)
plus O(C^2) scalar arithmetic on the integer counters the kernels return.
`adj` / `A` may be a torch sparse COO tensor (as in the reference) or a resident
`wdgh_b200.CSRGraph`.  Scalars come back as 0-dim float32 CPU tensors.
"""
from __future__ import annotations

import math
import random
import time

import numpy as np
import torch
from scipy.stats import ttest_ind

from . import graph as G
from .graph import CSRGraph
from .util_funcs import accuracy, random_disassortative_splits

pi = math.pi

_GRAPH_CACHE: dict = {}
_GRAPH_CACHE_MAX = 4


def _as_graph(a) -> CSRGraph:
    """torch sparse COO -> resident CSR (cached on the tensor's storage identity)."""
    if isinstance(a, CSRGraph):
        return a
    if not (isinstance(a, torch.Tensor) and a.is_sparse):
        raise TypeError("adjacency must be a torch sparse COO tensor or a wdgh_b200.CSRGraph")
    a = a.coalesce() if not a.is_coalesced() else a
    key = (a.indices().data_ptr(), a.values().data_ptr(), a._nnz(), tuple(a.shape), a.values()._version)
    g = _GRAPH_CACHE.get(key)
    if g is None:
        g = CSRGraph.from_torch_sparse(a)
        g._keepalive = a  # the key holds raw pointers: keep the tensor alive while cached
        if len(_GRAPH_CACHE) >= _GRAPH_CACHE_MAX:
            _GRAPH_CACHE.pop(next(iter(_GRAPH_CACHE)))
        _GRAPH_CACHE[key] = g
    return g


def _counts(g: CSRGraph, labels):
    """Label statistics of (graph, 1-D labels); one kernel pass, cached on the graph."""
    cacheable = isinstance(labels, torch.Tensor)  # numpy inputs can be mutated behind our back
    labels = torch.as_tensor(labels) if not cacheable else labels
    labels = labels.squeeze() if labels.dim() > 1 else labels
    key = (labels.data_ptr(), labels._version, labels.shape[0], str(labels.device))
    hit = g._counts.get(key) if cacheable else None
    if hit is None:
        lab32, mx = G.pack_labels(labels)
        hit = (G.structure_counts(g, lab32, mx + 1), labels)  # holding `labels` pins its address
        if cacheable:
            g._counts = {key: hit}
    return hit[0]


def _f32(v):
    return torch.tensor(np.float32(v))


def remove_self_loops(edge_index, edge_attr=None):
    """hm.py:24-40 (index filtering, torch plumbing)."""
    row, col = edge_index[0], edge_index[1]
    mask = row != col
    edge_attr = edge_attr if edge_attr is None else edge_attr[mask]
    return edge_index[:, mask], edge_attr


def edge_homophily(A, labels, ignore_negative=False):
    """hm.py:43-57.  1-D labels: fraction of stored entries (diagonal included) with equal
    endpoint labels; 2-D labels (homophily_tests.py:115-116): fraction of equal label ENTRIES."""
    g = _as_graph(A)
    lab = torch.as_tensor(labels) if not isinstance(labels, torch.Tensor) else labels
    if lab.dim() == 2:
        if ignore_negative:
            raise TypeError("mean() received an invalid combination of arguments")  # hm.py:54 on tensors
        eq = G.edge_label_rows_equal(g, lab.to(torch.float32))
        tot = g.nnz * lab.shape[1]
        return _f32(eq / tot if tot else float("nan"))
    s = _counts(g, lab)
    if ignore_negative:
        if isinstance(labels, torch.Tensor):
            raise TypeError("mean() received an invalid combination of arguments")  # np.mean(torch bool), hm.py:54
        return float(s.match_lab / s.n_lab) if s.n_lab else float("nan")
    return _f32(s.match_all / s.nnz if s.nnz else float("nan"))


def _node_homo_from_counts(s, num_nodes):
    if s.nbins != num_nodes and s.nbins != 1:  # bincount length vs hs length, hm.py:75-77
        raise RuntimeError(
            f"The size of tensor a ({num_nodes}) must match the size of tensor b ({s.nbins}) at non-singleton dimension 0")
    return _f32(s.node_sum / s.n_nodes_nsl if s.n_nodes_nsl else float("nan"))


def node_homophily(A, labels):
    """hm.py:60-68: mean over nodes (with >= 1 off-diagonal entry) of the same-label neighbour fraction."""
    g = _as_graph(A)
    return _node_homo_from_counts(_counts(g, labels), g.n)


def _counts_coo(edge_idx, labels, num_nodes):
    labels = torch.as_tensor(labels)
    labels = labels.squeeze() if labels.dim() > 1 else labels
    lab32, mx = G.pack_labels(labels)
    n = int(num_nodes) if num_nodes is not None else int(labels.shape[0])
    return G.structure_counts_coo(edge_idx, n, lab32, mx + 1)


def node_homophily_edge_idx(edge_idx, labels, num_nodes):
    """hm.py:71-78; edge_idx is 2 x (number of edges), any order, repeats counted."""
    return _node_homo_from_counts(_counts_coo(edge_idx, labels, num_nodes), int(num_nodes))


def compact_matrix_edge_idx(edge_idx, labels):
    """hm.py:81-102: C x C class compatibility matrix, rows normalised, negative labels ignored."""
    h = _counts_coo(edge_idx, labels, None).hist.astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        h = h / h.sum(1, keepdims=True)
    return torch.from_numpy(h)


def our_measure(edge_index, label):
    """hm.py:105-123: class-insensitive edge homophily \\hat{h}."""
    if isinstance(edge_index, CSRGraph):
        edge_index = edge_index.indices()
    elif isinstance(edge_index, torch.Tensor) and edge_index.is_sparse:
        edge_index = edge_index.coalesce().indices()
    label = torch.as_tensor(label).squeeze()
    s = _counts_coo(edge_index, label, None)
    c = s.num_classes
    h = s.hist.astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        h = h / h.sum(1, keepdims=True)
    neg = int(label.shape[0] - s.class_count.sum())
    counts = s.class_count[s.class_count > 0]  # unique(return_counts) of the non-negative labels, hm.py:113-114
    proportions = counts.astype(np.float32) / np.float32(label.shape[0] - neg)
    val = np.float32(0)
    for k in range(c):
        class_add = h[k, k] - proportions[k]  # IndexError when a class id never occurs, as upstream
        class_add = np.float32(max(class_add, 0)) if not np.isnan(class_add) else class_add
        if not np.isnan(class_add):
            val = np.float32(val + class_add)
    return _f32(val / np.float32(c - 1))


def class_distribution(A, labels):
    """hm.py:126-147 -> (p, p_bar, pc)."""
    g = _as_graph(A)
    s = _counts(g, labels)
    if s.n_empty:
        raise IndexError("index out of bounds: a node without stored entries misaligns `deg` (hm.py:129,141)")
    c = s.num_classes
    n = g.n
    neg = int(n - s.class_count.sum())
    uniq_counts = ([neg] if neg else []) + [int(v) for v in s.class_count if v > 0]
    p = torch.tensor(np.asarray(uniq_counts, dtype=np.int64)) / n                  # hm.py:137
    total = np.float32(s.nnz - n)                                                     # sum(deg - 1), hm.py:132,145
    p_bar = (s.class_deg - s.class_count).astype(np.float32) / total                  # hm.py:141
    pc = s.hist.astype(np.float32) / total                                            # hm.py:144
    p_bar[p_bar == 0] = 1e-8
    pc[pc == 0] = 1e-8
    return p, torch.from_numpy(p_bar.astype(np.float32)), torch.from_numpy(pc.astype(np.float32).reshape(c, c))


def adjusted_homo(A, label):
    """hm.py:150-155."""
    p, p_bar, pc = class_distribution(A, label)
    edge_homo = edge_homophily(A, label)
    return (edge_homo - torch.sum(p_bar ** 2)) / (1 - torch.sum(p_bar ** 2))


def label_informativeness(A, label):
    """hm.py:158-161."""
    p, p_bar, pc = class_distribution(A, label)
    return 2 - torch.sum(pc * torch.log(pc)) / torch.sum(p_bar * torch.log(p_bar))


def generalized_edge_homophily(adj, features, label, sample_max=75000, iteration=10):
    """hm.py:164-187: mean feature cosine over edges (all off-diagonal entries, or sampled entries)."""
    g = _as_graph(adj)
    nedges = g.nnz
    if nedges < sample_max:
        s, cnt = G.edge_cosine(g, features)
        return _f32(s / cnt if cnt else float("nan"))
    g_homo = np.zeros(iteration)
    for i in range(iteration):
        sample = torch.tensor(random.sample(range(nedges), int(sample_max)))     # hm.py:179-180, same draws
        s, cnt = G.edge_cosine(g, features, sample)
        g_homo[i] = np.float32(s / cnt)
    return np.mean(g_homo)


def _propagate(adj, features):
    """torch.spmm(adj, features) / torch.mm(adj, features) (hm.py:192,199,234) on the GPU."""
    if isinstance(adj, torch.Tensor) and not adj.is_sparse:
        g = CSRGraph.from_torch_sparse(adj.to_sparse())  # dense adjacency (synthetic_plot.py flow)
    else:
        g = _as_graph(adj)
    return G.spmm(g, features, G.NORM_NONE, False)


def _ids(mask_or_ids, device):
    t = torch.as_tensor(mask_or_ids)
    if t.dtype == torch.bool:
        t = torch.nonzero(t).view(-1)
    return t.to(device=device, dtype=torch.int64)


def similarity(features, adj, label, hard=None, LP=1, ifsum=1, idx_train=None):
    """hm.py:190-229: aggregation similarity score (soft / hard LAS) from (A X)(A X)^T -- for more than
    graph.GRAM_SIMILARITY_MAX_ROWS rows without forming it (class sums of A X), so whole graphs of any size work.
    bfloat16 / float16 features are aggregated as they are (no fp32 copy) and give the score of features.float()."""
    z = _propagate(adj, features)
    label = G._cuda(label, torch.float32)
    labels = G.argmax_rows(label)                                   # hm.py:193
    if idx_train is not None:
        ids = _ids(idx_train, z.device)
        z = G.gather_rows(z, ids)                                   # hm.py:199
        labels = labels[ids].contiguous()                           # hm.py:196
        label = label[ids].contiguous()                             # hm.py:197
    m = int(z.shape[0])
    c = int(labels.max().item()) + 1
    w = G.las_weights(z, labels, c, is_mean=(ifsum != 1))           # hm.py:192 / 199-206
    if label.shape[1] != c:
        if LP != 1:
            raise RuntimeError(f"The size of tensor a ({c}) must match the size of tensor b ({label.shape[1]})")
        label = label[:, :c].contiguous()
    cnt = G.las_count(w, labels, label, hard is not None, LP, ifsum == 1)
    return _f32(cnt / m if m else float("nan"))


def gntk_homophily_(features, adj, sample, n_layers, _z=None):
    """hm.py:232-257 -> (K_G / 2, K_X / 2) for the sampled nodes, as CUDA tensors."""
    z = _propagate(adj, features) if _z is None else _z
    x = G._cuda(features, torch.float32)
    ids = _ids(sample, z.device)
    tc = G.KR_USE_TENSOR_CORES  # see wdgh_b200/graph.py: pinv amplifies Gram rounding noise -> fp32-faithful mode
    k_g = G.gntk_transform_(G.gram(G.gather_rows(z, ids), use_tensor_cores=tc, faithful=True), 1 if n_layers == 1 else 0)
    k_x = G.gntk_transform_(G.gram(G.gather_rows(x, ids), use_tensor_cores=tc, faithful=True), 1 if n_layers == 1 else 0)
    return k_g, k_x


def classifier_based_performance_metric(features, adj, labels, sample_max, base_classifier='kernel_reg1', epochs=100,
                                        _trace=None):
    """hm.py:260-349: p-value of "graph-aware beats graph-agnostic" (KR / GNB / SVM), plus elapsed seconds.

    A X is computed once and stays resident (the reference recomputes it every epoch);
    sampling, pinv, sklearn and the t-test follow the reference on the host with the same RNG calls.
    `_trace` (not part of the reference signature): a list that receives one dict per epoch -- validation mask,
    arg-max predictions and accuracies of both classifiers -- for the parity tests.
    """
    from sklearn import svm
    from sklearn.naive_bayes import GaussianNB

    labels = torch.as_tensor(labels)
    nnodes = labels.shape[0]
    if labels.dim() > 1:
        labels = labels.flatten()
    labels = labels.cpu()
    G_results, X_results, diff_results = torch.zeros(epochs), torch.zeros(epochs), torch.zeros(epochs)
    t_time = time.time()
    z = _propagate(adj, features)
    x_dev = G._cuda(features, torch.float32)
    for j in range(epochs):
        if nnodes <= sample_max:
            sample = np.arange(nnodes)
            label_onehot = torch.eye(int(labels.max()) + 1)[labels]
            labels_sample = labels
        else:
            sample, _, _ = random_disassortative_splits(labels, labels.max() + 1, sample_max / nnodes)
            sample = sample.cpu()
            label_onehot = torch.eye(int(labels.max()) + 1)[labels][sample, :]
            labels_sample = labels[sample]
        idx_train, idx_val, idx_test = random_disassortative_splits(labels_sample, labels_sample.max() + 1)
        idx_train, idx_val = idx_train.cpu(), (idx_val + idx_test).cpu()
        if base_classifier in {'kernel_reg0', 'kernel_reg1'}:
            nlayers = 0 if base_classifier == 'kernel_reg0' else 1
            K_graph, K = gntk_homophily_(x_dev, adj, sample, nlayers, _z=z)
            K_graph, K = K_graph.cpu(), K.cpu()
            preds = []
            for kk in (K_graph, K):
                k_tt = kk[idx_train, :][:, idx_train]
                k_vt = kk[idx_val, :][:, idx_train]
                preds.append(k_vt @ (torch.tensor(np.linalg.pinv(k_tt.numpy())) @ label_onehot[idx_train]))
            acc_g, acc_x = accuracy(labels_sample[idx_val], preds[0]), accuracy(labels_sample[idx_val], preds[1])
            pred_g, pred_x = preds[0].max(1)[1], preds[1].max(1)[1]
        else:
            ids = _ids(sample, z.device)
            X = G.gather_rows(x_dev, ids).cpu()
            X_agg = G.gather_rows(z, ids).cpu()
            if base_classifier == 'gnb':
                mk = lambda: GaussianNB()  # noqa: E731
            elif base_classifier == 'svm_rbf':
                mk = lambda: svm.SVC(kernel='rbf', gamma=0.5, C=0.1)  # noqa: E731
            elif base_classifier == 'svm_poly':
                mk = lambda: svm.SVC(kernel='poly', degree=3, C=1)  # noqa: E731
            elif base_classifier == 'svm_linear':
                mk = lambda: svm.SVC(kernel='linear')  # noqa: E731
            else:
                raise ValueError(f"unknown base_classifier {base_classifier!r}")
            g_clf = mk().fit(X_agg[idx_train], labels_sample[idx_train])
            x_clf = mk().fit(X[idx_train], labels_sample[idx_train])
            pred_g, pred_x = torch.tensor(g_clf.predict(X_agg[idx_val])), torch.tensor(x_clf.predict(X[idx_val]))
            acc_g = torch.mean(pred_g.eq(labels_sample[idx_val]).float())
            acc_x = torch.mean(pred_x.eq(labels_sample[idx_val]).float())
        diff_results[j] = (acc_g > acc_x)
        G_results[j] = acc_g
        X_results[j] = acc_x
        if _trace is not None:
            _trace.append({"va": idx_val.clone(), "pred_g": pred_g, "pred_x": pred_x, "acc_g": float(acc_g),
                           "acc_x": float(acc_x)})
    _, g_aware_good_p = ttest_ind(X_results.detach().cpu(), G_results.detach().cpu(), axis=0, equal_var=False,
                                  nan_policy='propagate')
    if torch.mean(diff_results) <= 0.5:
        g_aware_good_p = g_aware_good_p / 2
    else:
        g_aware_good_p = 1 - g_aware_good_p / 2
    return g_aware_good_p, time.time() - t_time
