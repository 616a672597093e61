"""Drop-in mirror of the graph-statistics parts of the reference's `utils/util_funcs.py`.

Normalisers (normalize, preprocess_features, normalize_tensor, normalize_adj, sys_/row_normalized_adjacency)
and dataset_edge_balance run on the GPU through libwdgh_b200.so; the split / accuracy helpers are the
reference's host-side RNG logic (they must consume torch's global RNG identically so that
seeded runs reproduce).  Dataset loaders (load_data, full_load_data*, utils/datasets.py) are
out of scope of the hot path -- keep using the reference's.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
import torch

from . import graph as G
from .graph import CSRGraph


def _to_graph(adj, binary=False) -> CSRGraph:
    if isinstance(adj, CSRGraph):
        return adj
    if isinstance(adj, torch.Tensor):
        return CSRGraph.from_torch_sparse(adj if adj.is_sparse else adj.to_sparse(), binary=binary)
    return CSRGraph.from_scipy(sp.coo_matrix(adj), binary=binary)


def normalize_tensor(mx, symmetric=0):
    """Row-normalise (symmetric=0) or D^-1/2 M D^-1/2 (symmetric=1) a dense matrix.  util_funcs.py:365-380."""
    return G.normalize_dense(mx, 1 if symmetric else 0)


def normalize(mx):
    """Row-normalise: diag(1 / rowsum) @ mx, zero-sum rows stay zero.  util_funcs.py:29-36.

    Dense input (torch / numpy; synthetic_plot.py:92 hands it `adj + eye`) -> dense float32 CUDA tensor, which the
    caller's `torch.tensor(...)` wrapper accepts.  scipy sparse input (full_load_data, util_funcs.py:189-190) ->
    resident CSRGraph holding f32(rowsum^-1 * a_ij), products formed in float64 like scipy's."""
    if sp.issparse(mx):
        return _to_graph(mx).normalized(G.NORM_RW_SUM)
    return G.normalize_dense(mx, 0)


def preprocess_features(features):
    """Row-normalise the feature matrix.  util_funcs.py:39-46 (same arithmetic as `normalize`)."""
    if sp.issparse(features):
        return G.CSRGraph.from_scipy(features, rectangular=True).normalized(G.NORM_RW_SUM)
    return G.normalize_dense(features, 0)


def normalize_adj(adj):
    """(A D^-1/2)^T D^-1/2 = D^-1/2 A^T D^-1/2, D = diag(row sums of A), as a resident CSRGraph.  util_funcs.py:429-436.
    Zero row sums give a zero scale (`inf -> 0`), negative ones NaN, exactly like numpy's power(., -0.5)."""
    g = _to_graph(adj)
    scaled = g.normalized(G.NORM_SYM_RAW)            # D^-1/2 A D^-1/2 on A's pattern ...
    t = scaled.to_torch_sparse().t().coalesce()      # ... and its transpose (index plumbing only)
    return CSRGraph.from_coo_indices(t.indices(), t.values(), g.n)


def dataset_edge_balance(adj, labels):
    """Per class: (node count, adjacency mass inside the class, adjacency mass leaving it).  util_funcs.py:439-451.

    A binary adjacency goes through the integer label-statistics kernels (exact counts); a weighted one through the
    aggregation kernel, Z = A [onehot | 1 - onehot], followed by class-wise sums."""
    lab = torch.as_tensor(labels).reshape(-1)
    c = int(lab.max().item()) + 1
    g = _to_graph(adj)
    lab32, _ = G.pack_labels(lab)
    binary = g.val is None or bool((g.val == 1).all().item())
    if binary:
        pairs = G.structure_counts_coo(g.indices(), g.n, lab32, c, hist_includes_self_loops=True)   # diagonal kept
        rows = G.structure_counts(g, lab32, c)                    # class sizes + stored entries per class of the row
        inside = np.diag(pairs.hist).astype(np.float64)
        return rows.class_count.astype(np.float64), np.stack([inside, rows.class_deg.astype(np.float64) - inside], axis=1)
    known = lab32 >= 0
    onehot = torch.zeros((g.n, c), dtype=torch.float32, device=g.device)
    onehot[known, lab32[known].long()] = 1.0
    z = G.spmm(g, torch.cat([onehot, 1.0 - onehot], dim=1))          # [n, 2c]: mass into class k / into the rest
    # class-wise row sums are one more aggregation: P[i, u] = 1 iff label(u) = i (rows >= c empty), sums = (P Z)[:c]
    order = torch.argsort(torch.where(known, lab32, c).long(), stable=True)
    count = torch.bincount(lab32[known].long(), minlength=c)
    rowptr = torch.zeros(g.n + 1, dtype=torch.int64, device=g.device)
    rowptr[1:c + 1] = torch.cumsum(count, 0)
    rowptr[c + 1:] = rowptr[c]
    pool = CSRGraph(rowptr, order[:int(rowptr[c].item())].to(torch.int32).contiguous(), None, g.n)
    sums = G.spmm(pool, z)[:c].cpu().numpy().astype(np.float64)     # [c, 2c]
    idx = np.arange(c)
    return count.cpu().numpy().astype(np.float64), np.stack([sums[idx, idx], sums[idx, c + idx]], axis=1)


def sys_normalized_adjacency(adj):
    """D^-1/2 (A + I) D^-1/2 as a resident CSRGraph.  util_funcs.py:418-426."""
    return _to_graph(adj).with_self_loops().normalized(G.NORM_SYM)


def row_normalized_adjacency(adj):
    """D^-1 (A + I) (l1 row normalisation) as a resident CSRGraph.  util_funcs.py:383-390."""
    return _to_graph(adj).with_self_loops().normalized(G.NORM_RW)


def sparse_mx_to_torch_sparse_tensor(sparse_mx):
    """util_funcs.py:400-407; also accepts the CSRGraph the normalisers above return."""
    if isinstance(sparse_mx, CSRGraph):
        return sparse_mx.to_torch_sparse()
    sparse_mx = sparse_mx.tocoo().astype(np.float32)
    indices = torch.from_numpy(np.vstack((sparse_mx.row, sparse_mx.col)).astype(np.int64))
    values = torch.from_numpy(sparse_mx.data)
    return torch.sparse_coo_tensor(indices, values, torch.Size(sparse_mx.shape))


def propagate(adj, features, symmetric=1, add_self_loop=True, out_dtype=None):
    """SGC-1 / GCN propagation A_hat X without materialising A_hat (on-the-fly D^-1/2 or D^-1).

    bfloat16 and float16 features are read as they are (fp32 accumulation, the bits of the call on features.float());
    out_dtype=torch.bfloat16 / torch.float16, the dtype of the features, returns the result rounded to that type."""
    g = _to_graph(adj, binary=True)
    return G.spmm(g, features, G.NORM_SYM if symmetric else G.NORM_RW, add_self_loop, out_dtype=out_dtype)


def accuracy(labels, output):
    """Fraction of rows whose arg-max equals the label, as a float64 tensor.  util_funcs.py:393-397."""
    predicted = torch.argmax(output, dim=1).to(labels.dtype)
    return (predicted == labels).double().sum() / len(labels)


def index_to_mask(index, size):
    """Boolean mask of length `size` that is True at `index`.  util_funcs.py:478-481."""
    mask = torch.zeros(size, dtype=torch.bool, device=index.device)
    mask[index] = True
    return mask


def random_disassortative_splits(labels, num_classes, training_percentage=0.6):
    """Class-balanced train / val / test masks (60 / 20 / 20 by default).  util_funcs.py:454-475.

    Consumes torch's global RNG in the reference's order -- one `randperm` per class over that class's
    nodes, then one over the left-over nodes -- so seeded runs pick the same nodes as the reference."""
    labels = torch.as_tensor(labels).cpu()
    n = labels.shape[0]
    k = int(num_classes)
    per_class = int(round(training_percentage * (n / k)))
    n_val = int(round(0.2 * n))
    train_parts, rest_parts = [], []
    for cls in range(k):
        members = torch.nonzero(labels == cls).view(-1)
        shuffled = members[torch.randperm(members.size(0))]
        train_parts.append(shuffled[:per_class])
        rest_parts.append(shuffled[per_class:])
    train_index = torch.cat(train_parts, dim=0)
    rest = torch.cat(rest_parts, dim=0)
    rest = rest[torch.randperm(rest.size(0))]
    return index_to_mask(train_index, n), index_to_mask(rest[:n_val], n), index_to_mask(rest[n_val:], n)


def rand_train_test_idx(label, train_prop=.6, valid_prop=.2, ignore_negative=True):
    """Random train / valid / test index split over the labelled nodes (label != -1).  util_funcs.py:484-508.
    Uses numpy's global RNG (`np.random.permutation`) like the reference."""
    pool = torch.where(label != -1)[0] if ignore_negative else label
    count = pool.shape[0]
    n_train, n_valid = int(count * train_prop), int(count * valid_prop)
    order = torch.as_tensor(np.random.permutation(count))
    parts = (order[:n_train], order[n_train:n_train + n_valid], order[n_train + n_valid:])
    if not ignore_negative:
        return parts
    return tuple(pool[p] for p in parts)
