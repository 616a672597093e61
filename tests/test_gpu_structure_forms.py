"""Every form of the label-statistics pass (csrc/structure.cu) against an exact reference, at its dispatch boundaries.

`wdgh_structure_counts` picks its edge kernel from the class count C and the label copy:
  * C <= 63 with the 1-byte label copy: `structure_stream_kernel` ((C+1)^2 <= 4096 pair bins in shared memory);
  * otherwise `structure_rowgroup_kernel<uint8_t>` (C <= 254) or `<int32_t>` (C > 254, no 1-byte scratch, or the
    re-run after labels the 1-byte copy cannot represent: below -1 or >= C), pair table in shared memory while
    C*C <= 4096, class accumulators in shared memory while C <= 2048.
Both reduce the nodes of the rows up to the plan threshold T in their group epilogue; longer rows go through
`structure_chunks_kernel<uint8_t | int32_t>` and then `structure_heavy_nodes_kernel`.  The edge-list form is
`structure_coo_kernel` + `structure_nodes_kernel`.
The reference is `oracle.structure_counts` plus the outputs it does not return, restated here in numpy.  Integers must be
equal; the two float64 node sums may differ by the order of the atomic additions only (rtol 1e-12).  A label >= C is
unlabelled but compared raw (include/wdgh_b200.h): the reference sees it as a distinct negative value, -1000 - v.
"""
import numpy as np
import pytest
import torch

from oracle import ref_port as O

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(300)]


@pytest.fixture(scope="module")
def W():
    import wdgh_b200
    wdgh_b200._lib.require_device()
    return wdgh_b200


# ---------------------------------------------------------------------------
# reference and comparison
# ---------------------------------------------------------------------------
def reference(row, col, labels, n, C, coo=False, hist_self=False):
    """Every output of wdgh_structure_counts (coo=False) or wdgh_structure_counts_coo (coo=True) for the entry list
    (row, col), repeats counted with multiplicity."""
    row, col = np.asarray(row, np.int64), np.asarray(col, np.int64)
    lab = np.asarray(labels, np.int64)
    lab = np.where(lab >= C, -1000 - lab, lab)
    o = O.structure_counts(row, col, lab, n, num_classes=C)
    d_all, d_nsl, m_nsl = o["deg_all"], o["deg_nsl"], o["match_nsl"]
    labelled = lab >= 0
    hist = o["hist"].copy()
    if hist_self:   # compact_matrix_edge_idx keeps (i, i): labelled self loops land on the diagonal
        k = (row == col) & (lab[row] >= 0)
        hist += np.bincount(lab[row[k]] * (C + 1), minlength=C * C).reshape(C, C)
    has = d_nsl > 0
    f32 = np.float32
    r = dict(match_all=o["match_all"], match_lab=o["match_lab"], n_lab=o["n_lab"], n_self=o["n_selfloop"],
             n_nodes_nsl=int(has.sum()), nbins=int(np.flatnonzero(has).max()) + 1 if has.any() else 0,
             class_count=o["class_count"], hist=hist,
             class_isolated=np.bincount(lab[labelled & ~has], minlength=C).astype(np.int64),
             node_sum=float((m_nsl[has].astype(f32) / d_nsl[has].astype(f32)).astype(np.float64).sum()),
             deg_nsl=d_nsl, match_nsl=m_nsl)
    if coo:   # row lengths are unknown to the edge-list form: no degree mass, no empty rows, no diagonal variant
        r.update(class_deg=np.zeros(C, np.int64), n_empty=0, node_sum_self=0.0)
    else:
        cdeg = np.zeros(C, np.int64)
        np.add.at(cdeg, lab[labelled], d_all[labelled])
        a = d_all > 0
        self_sum = (m_nsl[a] + d_all[a] - d_nsl[a]).astype(f32) / d_all[a].astype(f32)
        r.update(class_deg=cdeg, n_empty=int((~a).sum()), node_sum_self=float(self_sum.astype(np.float64).sum()))
    return r


SCALARS = ("match_all", "match_lab", "n_lab", "n_self", "n_empty", "nbins", "n_nodes_nsl")
ARRAYS = ("class_count", "class_deg", "class_isolated", "hist")


def assert_counts(s, ref, tag=""):
    for k in SCALARS:
        assert getattr(s, k) == ref[k], (tag, k, getattr(s, k), ref[k])
    for k in ARRAYS:
        got = getattr(s, k)
        assert np.array_equal(got, ref[k]), (tag, k, np.flatnonzero(got.ravel() != ref[k].ravel())[:8])
    for k in ("deg_nsl", "match_nsl"):
        got = getattr(s, k).cpu().numpy().astype(np.int64)
        assert np.array_equal(got, ref[k]), (tag, k, np.flatnonzero(got != ref[k])[:8])
    for k in ("node_sum", "node_sum_self"):
        assert getattr(s, k) == pytest.approx(ref[k], rel=1e-12, abs=0), (tag, k, getattr(s, k), ref[k])


def assert_same_run(a, b, tag=""):
    """two forms of the pass on the same input: integers equal, node sums up to the atomic summation order"""
    for k in SCALARS:
        assert getattr(a, k) == getattr(b, k), (tag, k)
    for k in ARRAYS:
        assert np.array_equal(getattr(a, k), getattr(b, k)), (tag, k)
    assert torch.equal(a.deg_nsl, b.deg_nsl) and torch.equal(a.match_nsl, b.match_nsl), tag
    for k in ("node_sum", "node_sum_self"):
        assert getattr(a, k) == pytest.approx(getattr(b, k), rel=1e-12, abs=0), (tag, k)


def run(W, g, lab32, C, form):
    """form "auto": graph.structure_counts (1-byte label copy where it applies, int32 re-run after several distinct
    negative labels); "u8": one call with the 1-byte scratch, no re-run; "int32": no scratch, i.e. the int32 rowgroup
    form.  Returns (StructureCounts, the labels-below--1 counter of that call)."""
    if form == "auto":
        s = W.graph.structure_counts(g, lab32, C)
        return s, None
    scratch = None
    if form == "int32":
        dev = g.device
        scratch = (torch.empty(W._lib.sc_words(C), dtype=torch.int64, device=dev),
                   torch.empty(2, dtype=torch.float64, device=dev),
                   torch.empty(g.n, dtype=torch.int32, device=dev),
                   torch.empty(g.n, dtype=torch.int32, device=dev), None)
    counters, node_sum, deg, match, _ = W.graph.structure_counts_raw(g, lab32, C, scratch)
    multi_neg = int(counters[W._lib.SC_N_MULTI_NEG].item())
    return W.graph._unpack_counts(g.n, g.nnz, C, counters, node_sum, deg, match), multi_neg


def labels_with(rng, n, C, neg_frac=0.1):
    lab = rng.integers(0, C, n).astype(np.int64)
    lab[rng.random(n) < neg_frac] = -1
    top = min(n - 1, 5)
    lab[top] = C - 1            # the largest class id is always present
    return lab


def with_out_of_range(rng, labels, C, frac=0.05):
    """labels >= C, which only the C ABI can pass, on about `frac` of the nodes"""
    vals = np.array([C, C + 1, 254, 255, 1000, 2 ** 31 - 1], np.int64)
    vals = np.unique(vals[vals >= C])
    lab = np.asarray(labels, np.int64).copy()
    pick = rng.random(lab.shape[0]) < frac
    lab[pick] = rng.choice(vals, int(pick.sum()))
    return lab


def to_lab32(labels):
    return torch.from_numpy(np.asarray(labels, np.int32)).cuda()


# ---------------------------------------------------------------------------
# graphs
# ---------------------------------------------------------------------------
def powerlaw(n, avg, seed, hub_rows=(0, 1, 2), hub_deg=1500, self_frac=0.3, tail=40):
    """power-law rows, hub rows (split rows, each with its self loop), self loops on a fraction of the rows, ~5% of
    the rows without off-diagonal entries (empty, or a self loop only) and the last `tail` rows without any (so nbins
    stops short of n)"""
    rng = np.random.default_rng(seed)
    deg = np.minimum((rng.pareto(1.8, n) + 1) * avg / 2.2, n // 2).astype(np.int64)
    hubs = np.asarray(hub_rows, np.int64)
    bare = rng.random(n) < 0.05
    bare[hubs] = False
    bare[n - tail:] = True
    src = np.repeat(np.arange(n), deg)
    dst = rng.integers(0, n, src.shape[0])
    hs = np.repeat(hubs, hub_deg)
    hd = rng.integers(0, n, hs.shape[0])
    src, dst = np.concatenate([src, hs, hd]), np.concatenate([dst, hd, hs])
    keep = ~bare[src]
    sl = np.concatenate([np.flatnonzero(rng.random(n) < self_frac), hubs])
    row, col, _ = O.coalesce(np.concatenate([src[keep], sl]), np.concatenate([dst[keep], sl]), None, n)
    return row, col


def csr(W, row, col, n, T):
    rowptr = O.csr_from_coo(row, n)
    return W.CSRGraph.from_csr(torch.from_numpy(rowptr), torch.from_numpy(col.astype(np.int32)), None, n, threshold=T)


# ---------------------------------------------------------------------------
# 1. class counts at every dispatch boundary, through both label widths
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("C", [1, 2, 63, 64, 65, 200, 254, 255, 300, 2048, 2049])
def test_class_count_boundaries(W, C):
    """stream form up to C = 63, uint8 rowgroup with a 4096-bin shared table at 64 and global pair bins from 65, int32
    from 255, global class accumulators from 2049; every C also forced through the int32 rowgroup form"""
    n, T = 20000, 64
    row, col = powerlaw(n, 8, seed=C, hub_rows=(0, 9000, n - 100))
    rng = np.random.default_rng(C)
    labels = labels_with(rng, n, C)
    g = csr(W, row, col, n, T)
    assert g.n_heavy >= 3
    ref = reference(row, col, labels, n, C)
    assert ref["class_count"][C - 1] > 0 and (labels == -1).mean() > 0.05
    lab32 = to_lab32(labels)
    s_auto, _ = run(W, g, lab32, C, "auto")
    assert_counts(s_auto, ref, "auto")
    s_i32, neg = run(W, g, lab32, C, "int32")
    assert neg == 0
    assert_counts(s_i32, ref, "int32")
    assert_same_run(s_auto, s_i32)


# ---------------------------------------------------------------------------
# 2. graph shapes around the 32-row groups and the split threshold
# ---------------------------------------------------------------------------
def shaped_graph(n, T, seed):
    """random short rows, a whole empty 32-row group, rows of exactly T, T + 1 and 2T + 1 entries (the split ones hold
    their self loop), rows whose only entry is a self loop (one labelled, one not), an unlabelled row with a self loop
    among other entries.  Returns (row, col, {role: row id}); the caller fixes the labels of the roles."""
    rng = np.random.default_rng(seed)
    deg = rng.integers(0, 6, n)
    deg[rng.random(n) < 0.3] = 0
    if n >= 64:
        deg[32:64] = 0
    free = [int(r) for r in rng.permutation(n) if not 32 <= r < 64]
    roles = {}
    rows = {}
    for name, length in (("len_T", T), ("len_T1", T + 1), ("len_2T1", 2 * T + 1)):
        if length <= n and free:
            r = free.pop()
            if name == "len_T":
                rows[r] = rng.choice(n, length, replace=False)
            else:   # the split rows carry their self loop
                rows[r] = np.concatenate([rng.choice(np.delete(np.arange(n), r), length - 1, replace=False), [r]])
            roles[name] = r
    for name in ("self_only_lab", "self_only_unlab", "unlab_self_plus"):
        if free:
            r = free.pop()
            rows[r] = np.array([r]) if name != "unlab_self_plus" else \
                np.unique(np.concatenate([[r], rng.integers(0, n, 3)]))
            roles[name] = r
    deg[list(rows)] = 0
    src = np.repeat(np.arange(n), deg)
    dst = rng.integers(0, n, src.shape[0])
    src = np.concatenate([src] + [np.full(len(c), r) for r, c in rows.items()])
    dst = np.concatenate([dst] + list(rows.values()))
    row, col, _ = O.coalesce(src, dst, None, n)
    return row, col, roles


@pytest.mark.parametrize("T", [32, 64])
@pytest.mark.parametrize("n", [1, 31, 32, 33, 95, 20011])
def test_row_group_shapes(W, n, T):
    row, col, roles = shaped_graph(n, T, seed=n * 7 + T)
    deg = np.bincount(row, minlength=n)
    if "len_T1" in roles:
        assert deg[roles["len_T1"]] == T + 1
    g = csr(W, row, col, n, T)
    assert g.n_heavy == int((deg > T).sum())
    for C in (7, 100):   # stream form, uint8 rowgroup form (+ the int32 rowgroup form of both)
        labels = labels_with(np.random.default_rng(n + C), n, C)
        for name, r in roles.items():
            labels[r] = -1 if "unlab" in name else (r % C)
        ref = reference(row, col, labels, n, C)
        lab32 = to_lab32(labels)
        s_auto, _ = run(W, g, lab32, C, "auto")
        assert_counts(s_auto, ref, ("auto", C))
        s_i32, _ = run(W, g, lab32, C, "int32")
        assert_counts(s_i32, ref, ("int32", C))
    if "self_only_lab" in roles:   # self-loop-only rows are isolated, but not empty
        r = roles["self_only_lab"]
        assert ref["deg_nsl"][r] == 0 and deg[r] == 1 and ref["class_isolated"][labels[r]] >= 1


# ---------------------------------------------------------------------------
# 3. several distinct unlabelled values (-1, -2, labels >= C): the 1-byte copy folds them together, the host re-runs
#    on int32 labels
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("C", [3, 64, 200])
def test_distinct_negative_labels(W, C):
    n, T = 20000, 64
    row, col = powerlaw(n, 8, seed=100 + C, hub_rows=(3, 12000))
    rng = np.random.default_rng(C)
    labels = labels_with(rng, n, C, neg_frac=0.15)
    labels[rng.random(n) < 0.1] = -2
    labels = with_out_of_range(rng, labels, C)
    n_below = int(((labels < -1) | (labels >= C)).sum())
    g = csr(W, row, col, n, T)
    lab32 = to_lab32(labels)
    ref = reference(row, col, labels, n, C)
    folded = reference(row, col, np.where((labels >= 0) & (labels < C), labels, -1), n, C)
    assert ref["match_all"] != folded["match_all"]   # raw equality must tell -1, -2 and labels >= C apart
    s_u8, neg = run(W, g, lab32, C, "u8")
    assert neg == n_below
    assert s_u8.match_all == folded["match_all"]     # what the 1-byte copy sees, before the re-run
    s_auto, _ = run(W, g, lab32, C, "auto")
    assert_counts(s_auto, ref, "auto")
    s_i32, neg = run(W, g, lab32, C, "int32")
    assert neg == 0
    assert_counts(s_i32, ref, "int32")


# ---------------------------------------------------------------------------
# 4. row shards: global label ids, local per-row arrays
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("form", ["auto", "int32"])
@pytest.mark.parametrize("C", [7, 300])
@pytest.mark.parametrize("bounds", [(0, 9001, 20000), (0, 5003, 13371, 20000)])
def test_row_shards(W, C, bounds, form):
    """the shards' per-row arrays are slices of the whole-graph run, their counters add up to it, max(nbins) is its
    nbins.  Shard boundaries are not multiples of 32; every shard holds split rows with their self loops."""
    n, T = bounds[-1], 64
    hubs = [b + 17 for b in bounds[:-1]]
    row, col = powerlaw(n, 8, seed=C + len(bounds), hub_rows=hubs)
    labels = labels_with(np.random.default_rng(C), n, C)
    lab32 = to_lab32(labels)
    whole, _ = run(W, csr(W, row, col, n, T), lab32, C, form)
    assert_counts(whole, reference(row, col, labels, n, C), "whole")
    rowptr = O.csr_from_coo(row, n)
    col32 = col.astype(np.int32)
    parts = []
    for r0, r1 in zip(bounds[:-1], bounds[1:]):
        rp = torch.from_numpy(rowptr[r0:r1 + 1] - rowptr[r0]).cuda()
        cs = torch.from_numpy(col32[rowptr[r0]:rowptr[r1]]).cuda()
        sg = W.CSRGraph(rp, cs, None, r1 - r0, threshold=T, row_offset=r0, n_global=n)
        assert sg.n_heavy >= 1
        s, _ = run(W, sg, lab32, C, form)
        assert torch.equal(s.deg_nsl, whole.deg_nsl[r0:r1]) and torch.equal(s.match_nsl, whole.match_nsl[r0:r1])
        parts.append(s)
    for k in ("match_all", "match_lab", "n_lab", "n_self", "n_empty", "n_nodes_nsl"):
        assert sum(getattr(p, k) for p in parts) == getattr(whole, k), k
    assert max(p.nbins for p in parts) == whole.nbins
    for k in ARRAYS:
        assert np.array_equal(sum(getattr(p, k) for p in parts), getattr(whole, k)), k
    for k in ("node_sum", "node_sum_self"):
        assert sum(getattr(p, k) for p in parts) == pytest.approx(getattr(whole, k), rel=1e-12, abs=0), k


# ---------------------------------------------------------------------------
# 5. the edge-list form: unsorted, repeated edges
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("hist_self", [False, True])
@pytest.mark.parametrize("C", [2, 64, 65])
def test_edge_list_form(W, C, hist_self):
    n = 3000
    row, col = powerlaw(n, 6, seed=C, hub_rows=(1, 2000), hub_deg=400)
    rng = np.random.default_rng(C + hist_self)
    rep = rng.random(row.shape[0]) < 0.2                 # repeated edges, self loops among them
    src = np.concatenate([row, row[rep], [7, 7, 7]])
    dst = np.concatenate([col, col[rep], [7, 7, 7]])
    perm = rng.permutation(src.shape[0])
    src, dst = src[perm], dst[perm]
    labels = with_out_of_range(rng, labels_with(rng, n, C), C)
    labels[7] = 0
    ei = torch.from_numpy(np.vstack([src, dst]).astype(np.int64))
    s = W.graph.structure_counts_coo(ei, n, to_lab32(labels), C, hist_includes_self_loops=hist_self)
    assert s.nnz == src.shape[0]
    assert_counts(s, reference(src, dst, labels, n, C, coo=True, hist_self=hist_self))
