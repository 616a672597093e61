"""Drop-in mirror of the reference's `utils/homophily_plot.py` (the dense-adjacency variants that
`synthetic_plot.py` imports) on the B200 path.

The reference hands these functions a DENSE n x n adjacency (row-normalised, self-loops added,
synthetic_plot.py:94) and a dense one-hot label matrix.  Here the dense matrix is sparsified once
(`adj.to_sparse()`, torch plumbing) into a resident CSRGraph and every metric reuses the same CUDA
kernels as `wdgh_b200.homophily_metrics`.  Differences of the plot variants that are reproduced
(cited as hp.py:LINE):
  * edge_homophily takes the one-hot matrix and sums <l_i, l_j> over off-diagonal positive entries (:43-54);
  * node_homophily does NOT strip self-loops (:81-100);
  * compact_matrix_edge_idx takes an [E, 2] edge list and keeps self-loops (:103-125);
  * our_measure drops the diagonal and gives isolated nodes a self-loop (:128-148);
  * similarity has the NTK branch and applies idx_train (an index list) to the finished Gram (:189-241);
  * classifier_based_performance_metric returns only the p-value (:278-368).
"""
from __future__ import annotations

import math

import numpy as np
import torch
from scipy.stats import ttest_ind

from . import graph as G
from .graph import CSRGraph
from .homophily_metrics import (_as_graph, _counts, _f32, _ids, class_distribution as _class_distribution_sparse,
                                gntk_homophily_ as _gntk_sparse, remove_self_loops)  # noqa: F401
from .util_funcs import random_disassortative_splits

pi = math.pi
_DENSE_CACHE: dict = {}


def _graph_of(adj) -> CSRGraph:
    """Dense torch matrix (or anything homophily_metrics accepts) -> resident CSR, cached per tensor."""
    if isinstance(adj, CSRGraph) or (isinstance(adj, torch.Tensor) and adj.is_sparse):
        return _as_graph(adj)
    adj = torch.as_tensor(adj)
    key = (adj.data_ptr(), adj._version, tuple(adj.shape), str(adj.device))
    g = _DENSE_CACHE.get(key)
    if g is None:
        g = CSRGraph.from_torch_sparse(adj.to(torch.float32).to_sparse())
        g._keepalive = adj
        _DENSE_CACHE.clear()
        _DENSE_CACHE[key] = g
    return g


def edge_homophily(adj, label):
    """hp.py:43-54."""
    g = _graph_of(adj)
    s, cnt = G.edge_cosine(g, G._cuda(label, torch.float32), raw_dot=True)
    return _f32(s / cnt if cnt else float("nan"))


def generalized_edge_homophily(adj, features, label, sample_max=20000, iteration=100):
    """hp.py:56-78.  The reference's >= sample_max branch overwrites `adj` with the sampled sub-matrix in its
    first iteration and dies with IndexError in the second; that is reproduced instead of guessed at."""
    nnodes = label.shape[0]
    if nnodes >= sample_max:
        raise IndexError("homophily_plot.generalized_edge_homophily: index out of range in the 2nd sampling "
                         "iteration (the reference reassigns `adj` inside the loop, hp.py:74)")
    g = _graph_of(adj)
    s, cnt = G.edge_cosine(g, features)
    return _f32(s / cnt if cnt else float("nan"))


def node_homophily(A, labels):
    """hp.py:81-100: self-loops stay in both the numerator and the denominator."""
    g = _graph_of(A)
    s = _counts(g, labels)
    last_row_empty = int((g.rowptr[-1] - g.rowptr[-2]).item()) == 0 if g.n else True
    if last_row_empty:  # bincount(edge_index[0]) would be shorter than num_nodes
        raise RuntimeError("The size of tensor a must match the size of tensor b at non-singleton dimension 0")
    nodes = g.n - s.n_empty
    return _f32(s.node_sum_self / nodes if nodes else float("nan"))


def node_homophily_edge_idx(edge_index, labels, num_nodes):
    """hp.py:92-100 on an explicit 2 x E edge list (self-loops kept)."""
    ei = G._cuda(edge_index, torch.int64)
    vals = torch.ones(ei.shape[1], device=ei.device)
    a = torch.sparse_coo_tensor(ei, vals, (int(num_nodes), int(num_nodes)))
    if not bool((a.coalesce().values() == 1).all()):
        raise NotImplementedError("repeated edges in edge_index are not supported by the plot variant mirror")
    return node_homophily(a, labels)


def _compat_from_counts(s):
    h = s.hist.astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        return h / h.sum(1, keepdims=True)


def compact_matrix_edge_idx(edge_index, labels):
    """hp.py:103-125: `edge_index` is [E, 2] (as `A.nonzero()` returns it); self-loops are counted."""
    ei = torch.as_tensor(edge_index)
    labels = torch.as_tensor(labels).squeeze()
    lab32, mx = G.pack_labels(labels)
    s = G.structure_counts_coo(ei.t().contiguous(), int(labels.shape[0]), lab32, mx + 1, hist_includes_self_loops=True)
    return torch.from_numpy(_compat_from_counts(s))


def our_measure(A, label):
    """hp.py:128-148: diagonal dropped, isolated nodes get a self-loop, then the class-insensitive homophily."""
    g = _graph_of(A)
    label = torch.as_tensor(label).squeeze()
    s = _counts(g, label)
    c = s.num_classes
    hist = s.hist + np.diag(s.class_isolated)      # (i, i) entries of the isolated nodes
    h = hist.astype(np.float32)
    with np.errstate(divide="ignore", invalid="ignore"):
        h = h / h.sum(1, keepdims=True)
    counts = s.class_count[s.class_count > 0]
    proportions = counts.astype(np.float32) / np.float32(s.class_count.sum())
    val = np.float32(0)
    for k in range(c):
        class_add = h[k, k] - proportions[k]
        if not np.isnan(class_add):
            val = np.float32(val + max(class_add, 0))
    return _f32(val / np.float32(c - 1))


def class_distribution(A, labels):
    """hp.py:150-173."""
    return _class_distribution_sparse(_graph_of(A), labels)


def adjusted_homo(A, label):
    """hp.py:175-180."""
    label = torch.as_tensor(label)
    p, p_bar, pc = class_distribution(A, torch.argmax(label, 1))
    edge_homo = edge_homophily(A, label)
    return (edge_homo - torch.sum(p_bar ** 2)) / (1 - torch.sum(p_bar ** 2))


def label_informativeness(A, label):
    """hp.py:183-186."""
    label = torch.as_tensor(label)
    p, p_bar, pc = class_distribution(A, torch.argmax(label, 1))
    return 2 - torch.sum(pc * torch.log(pc)) / torch.sum(p_bar * torch.log(p_bar))


def similarity(features, adj, label, NTK=None, hard=None, LP=1, ifsum=1, idx_train=None):
    """hp.py:189-241."""
    g = _graph_of(adj)
    label = G._cuda(label, torch.float32)
    labels = G.argmax_rows(label)
    ids = None if idx_train is None else _ids(idx_train, label.device)
    if NTK:
        x = G._cuda(features, torch.float32)
        k = G.ntk_clamp_transform_(G.gram(x))                                   # hp.py:191-193
        ak = G.spmm(g, k)                                                       # A K
        gm = G.spmm(g, ak.t().contiguous()).t().contiguous()                    # (A (A K)^T)^T = A K A^T
        if ids is not None:
            gm = G.gather_rows(G.gather_rows(gm, ids).t().contiguous(), ids).t().contiguous()   # [idx][:, idx]
    else:
        z = G.spmm(g, features)
        if ids is not None:
            z = G.gather_rows(z, ids)
    if ids is not None:
        labels = labels[ids].contiguous()
        label = label[ids].contiguous()
    m = int((gm if NTK else z).shape[0])
    c = int(labels.max().item()) + 1
    if NTK:
        w = G.class_colsum(gm, labels, c, is_mean=(ifsum != 1))
    else:
        w = G.las_weights(z, labels, c, is_mean=(ifsum != 1))                  # hp.py:196-206
    if label.shape[1] != c:
        if LP != 1:
            raise RuntimeError(f"The size of tensor a ({c}) must match the size of tensor b ({label.shape[1]})")
        label = label[:, :c].contiguous()
    cnt = G.las_count(w, labels, label, hard is not None, LP, ifsum == 1)
    return _f32(cnt / m if m else float("nan"))


def gntk_homophily_(features, adj, sample, n_layers, _z=None):
    """hp.py:244-275."""
    if not isinstance(sample, torch.Tensor):
        raise AttributeError("'numpy.ndarray' object has no attribute 'device'")   # hp.py:245 on np.arange samples
    return _gntk_sparse(features, _graph_of(adj), sample, n_layers, _z=_z)


def classifier_based_performance_metric(features, adj, labels, sample_max, rcond=1e-15, base_classifier='kernel_reg1',
                                        epochs=100, _trace=None):
    """hp.py:278-368: like the homophily_metrics version but returns only the p-value.
    `_trace` (not part of the reference signature): list receiving one dict per epoch for the parity tests."""
    from sklearn import svm
    from sklearn.naive_bayes import GaussianNB

    labels = torch.as_tensor(labels)
    nnodes = labels.shape[0]
    if labels.dim() > 1:
        labels = labels.flatten()
    labels = labels.cpu()
    G_results, X_results, diff_results = torch.zeros(epochs), torch.zeros(epochs), torch.zeros(epochs)
    g = _graph_of(adj)
    z = G.spmm(g, features)
    x_dev = G._cuda(features, torch.float32)
    for j in range(epochs):
        if nnodes <= sample_max:
            sample = np.arange(nnodes)
            label_onehot = torch.eye(int(labels.max()) + 1)[labels]
            labels_sample = labels
        else:
            sample, _, _ = random_disassortative_splits(labels, labels.max() + 1, sample_max / nnodes)
            label_onehot = torch.eye(int(labels.max()) + 1)[labels][sample, :]
            labels_sample = labels[sample]
        idx_train, idx_val, idx_test = random_disassortative_splits(labels_sample, labels_sample.max() + 1)
        idx_val = idx_val + idx_test
        if base_classifier in {'kernel_reg0', 'kernel_reg1'}:
            nlayers = 0 if base_classifier == 'kernel_reg0' else 1
            K_graph, K = gntk_homophily_(x_dev, g, sample, nlayers, _z=z)
            K_graph, K = K_graph.cpu(), K.cpu()
            preds = []
            for kk in (K_graph, K):
                k_tt, k_vt = kk[idx_train, :][:, idx_train], kk[idx_val, :][:, idx_train]
                preds.append(k_vt @ (torch.tensor(np.linalg.pinv(k_tt.numpy())) @ label_onehot[idx_train]))
            pred_g, pred_x = preds[0].argmax(1), preds[1].argmax(1)
            acc_g = torch.mean(pred_g.eq(labels_sample[idx_val]).float())
            acc_x = torch.mean(pred_x.eq(labels_sample[idx_val]).float())
        else:
            ids = _ids(sample, z.device)
            X, X_agg = G.gather_rows(x_dev, ids).cpu(), G.gather_rows(z, ids).cpu()
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
        G_results[j], X_results[j] = acc_g, acc_x
        if _trace is not None:
            _trace.append({"va": idx_val.clone(), "pred_g": pred_g, "pred_x": pred_x, "acc_g": float(acc_g),
                           "acc_x": float(acc_x)})
    _, g_aware_good_p = ttest_ind(X_results.detach().cpu(), G_results.detach().cpu(), axis=0, equal_var=False,
                                  nan_policy='propagate')
    if torch.mean(diff_results) <= 0.5:
        return g_aware_good_p / 2
    return 1 - g_aware_good_p / 2
