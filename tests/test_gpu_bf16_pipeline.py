"""bfloat16 features in the phased aggregation (wdgh_spmm_csr_ranged_bf16, graph.spmm_ranged with a bf16 `x`), in the
host-buffer pipeline (wdgh_pipeline_host_bf16, graph.pipeline_host) and in graph.spmm_structure_fused.

bf16 -> fp32 is exact and a bf16 phase sums every row in the order of the fp32 phase, so a phase is checked exactly
against the fp32 phase on x.float().  The pipeline's fp32 Y is checked exactly against the fp32 pipeline on x.float()
(both feature types take the same copy / compute form), and a bf16 Y exactly against the rounding of the fp32 Y.
"""
import numpy as np
import pytest
import torch

from oracle import ref_port as O

pytestmark = pytest.mark.gpu

BF16 = torch.bfloat16


@pytest.fixture(scope="module")
def W():
    import wdgh_b200
    wdgh_b200._lib.require_device()
    return wdgh_b200


def powerlaw_graph(n, avg_deg, seed, hubs=3, hub_deg=3000):
    rng = np.random.default_rng(seed)
    deg = np.minimum((rng.pareto(1.8, n) + 1) * avg_deg / 2.2, n // 2).astype(np.int64)
    src = np.repeat(np.arange(n), deg)
    dst = rng.integers(0, n, src.shape[0])
    hs = np.repeat(np.arange(hubs), hub_deg)
    hd = rng.integers(0, n, hs.shape[0])
    row, col, _ = O.coalesce(np.concatenate([src, hs, hd]), np.concatenate([dst, hd, hs]), None, n)
    keep = row != col
    return row[keep], col[keep]


def bf16_features(rng, n, d, device="cuda"):
    return torch.from_numpy(rng.standard_normal((n, d)).astype(np.float32)).to(device).to(BF16)


def same(a, b):
    """bit-identical, NaN in the same places (rows a phase has not written yet)"""
    torch.testing.assert_close(a, b, rtol=0, atol=0, equal_nan=True)


# ---------------------------------------------------------------------------
# phased aggregation
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("d", [32, 64, 128, 256])
@pytest.mark.parametrize("weighted,codes", [(False, True), (False, False), (True, False)])
def test_bf16_phases_equal_fp32_phases(W, d, weighted, codes):
    """own-shard phase read in place through x_row0, then the columns before / after it with accumulate, finalize
    and the split rows (threshold 256) -- every phase bit-identical to the fp32 phase on x.float()"""
    n, parts = 20000, 3
    row, col = powerlaw_graph(n, 10, seed=d)
    rng = np.random.default_rng(d)
    val = torch.from_numpy((rng.random(row.shape[0]) + 0.5).astype(np.float32)) if weighted else None
    g = W.CSRGraph.from_coo_indices(torch.from_numpy(np.vstack([row, col])), val, n, threshold=256)
    assert g.n_heavy > 0
    xb = bf16_features(rng, n, d)
    x32 = xb.float()
    dinv, _, code = g.degree_scale(W.NORM_SYM, True)
    code = code if codes else None
    block = (n + parts - 1) // parts
    seg = W.graph.column_segments(g, [b * block for b in range(parts)] + [n])
    skip = W.graph.heavy_flags(g)
    y_ref = W.spmm(g, xb, W.NORM_SYM, True)
    for r in range(parts):
        lo, hi = r * block, min((r + 1) * block, n)
        first, last = r == 0, r == parts - 1
        ys = []
        for x in (xb, x32):
            y = torch.full((n, d), float("nan"), device="cuda")
            calls = [(seg[r], seg[r + 1], x[lo:hi].clone(), False, False, False, lo)]
            if not first:
                calls.append((seg[0], seg[r], x, True, last, last, 0))
            if not last:
                calls.append((seg[r + 1], seg[parts], x, True, True, True, 0))
            states = []
            for b, e, xx, acc, fin, split, row0 in calls:
                W.graph.spmm_ranged(g, b, e, xx, y, W.NORM_SYM, True, dinv, code, skip, acc, fin, split, x_row0=row0)
                states.append(y.clone())
            ys.append(states)
        for sb, sf in zip(*ys):
            same(sb, sf)
        y = ys[0][-1]
        assert not y.isnan().any()
        assert (y - y_ref).abs().max().item() <= 1e-5 * y_ref.abs().max().item()


def test_bf16_phase_errors(W):
    lib = W._lib.lib
    n = 2000
    row, col = powerlaw_graph(n, 6, seed=1, hubs=0)
    g = W.CSRGraph.from_coo_indices(torch.from_numpy(np.vstack([row, col])), None, n, threshold=1 << 20)
    assert g.n_chunks == 0            # no split rows: the calls below need no skip flags
    plan, host = g.plan
    rng = np.random.default_rng(1)
    p = W._lib.ptr
    rb, re = g.rowptr[:-1], g.rowptr[1:]

    def call(x, d, ldx, y):
        return lib.wdgh_spmm_csr_ranged_bf16(p(g.rowptr), p(rb), p(re), p(g.col), None, n, p(x), d, ldx, p(y), d, 0, 1,
                                             None, None, None, 0, 1, 1, p(plan), host, None, 0, None)

    xw = bf16_features(rng, n, 256)
    y = torch.empty(n, 256, device="cuda")
    assert call(xw, 128, 256, y) == 0
    torch.cuda.synchronize()
    for x, d, ldx in ((xw, 96, 256),              # a width the row-group kernel does not take
                      (xw[:, 2:], 128, 256),      # rows on 4-byte boundaries
                      (xw, 128, 130)):            # ldx not a multiple of 4
        assert call(x, d, ldx, y) == -1, (d, ldx)
        err = lib.wdgh_last_error()
        assert err.startswith(b"wdgh_spmm_csr_ranged_bf16: ") and b"8-byte aligned rows" in err, err
    x = xw[:, :128]
    y128 = torch.empty(n, 128, device="cuda")
    with pytest.raises(W.WdghError):
        W.graph.spmm_ranged(g, rb, re, xw[:, :96], y128[:, :96], 0, True, None, None, None, False, True, True)
    with pytest.raises(ValueError):
        W.graph.spmm_ranged(g, rb, re, x, y128, 0, True, None, None, None, False, True, True,
                            extra=torch.zeros(1, n, 128, device="cuda"))
    with pytest.raises(ValueError):
        W.graph.spmm_ranged(g, rb, re, x, y128, 0, True, None, None, None, False, True, True, ctas_per_sm=8)
    with pytest.raises(ValueError):
        W.graph.spmm_ranged(g, rb, re, x, torch.empty(n, 128, dtype=BF16, device="cuda"), 0, True, None, None, None,
                            False, True, True)


# ---------------------------------------------------------------------------
# host-buffer pipeline
# ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host_graph():
    n, c = 50000, 7
    row, col = powerlaw_graph(n, 14, seed=128)
    rng = np.random.default_rng(3)
    labels = rng.integers(0, c, n).astype(np.int32)
    labels[rng.random(n) < 0.1] = -1
    rowptr = torch.from_numpy(O.csr_from_coo(row, n).astype(np.int64))
    return rowptr, torch.from_numpy(col.astype(np.int32)), torch.from_numpy(labels), c, (row, col)


def check_counts(W, counters, node_sum, s):
    """pipeline counters == the resident label pass (integers exactly; node_sum is a float64 atomic sum)"""
    L, H, c = W._lib, W._lib.SC_HEADER, s.num_classes
    head = [s.match_all, s.match_lab, s.n_lab, s.n_self, s.n_empty, s.nbins, s.n_nodes_nsl]
    assert list(counters[:L.SC_N_MULTI_NEG]) == head
    assert np.array_equal(counters[H:H + c], s.class_count)
    assert np.array_equal(counters[H + c:H + 2 * c], s.class_deg)
    assert np.array_equal(counters[H + 2 * c:H + 2 * c + c * c].reshape(c, c), s.hist)
    assert np.array_equal(counters[H + 2 * c + c * c:], s.class_isolated)
    assert abs(node_sum[0] - s.node_sum) <= 1e-12 * max(1.0, s.node_sum)
    assert abs(node_sum[1] - s.node_sum_self) <= 1e-12 * max(1.0, s.node_sum_self)


@pytest.mark.parametrize("d,form", [(128, "two 64-wide column blocks, Y back under the X copies"),
                                    (192, "three column blocks"),
                                    (160, "not a multiple of 64: row blocks, one phase per arriving block"),
                                    (96, "single copy, then one launch"),
                                    (70, "d % 4 != 0: single launch through the bf16 SpMM dispatch")])
def test_bf16_pipeline_forms(W, host_graph, d, form):
    rowptr, col, labels, c, _ = host_graph
    n = int(labels.shape[0])
    P = W.graph.pipeline_host
    xb = bf16_features(np.random.default_rng(d), n, d, device="cpu")
    x32 = xb.float()
    g = W.CSRGraph.from_csr(rowptr, col, None, n)
    assert g.n_heavy > 0
    s = W.graph.structure_counts(g, labels.cuda(), c)
    y_res = W.spmm(g, xb.cuda(), W.NORM_SYM, True).cpu()

    W._lib.lib.wdgh_pipeline_host_release()      # the first call below sizes the feature buffer for bf16
    cnt0, ns0 = P(rowptr, col, xb, labels, c)    # counters only
    check_counts(W, cnt0, ns0, s)
    y1 = torch.empty(n, d)
    cnt1, ns1 = P(rowptr, col, xb, labels, c, y=y1)
    check_counts(W, cnt1, ns1, s)
    y1b = torch.empty(n, d)
    P(rowptr, col, xb, labels, c, y=y1b)         # cached buffers reused
    assert torch.equal(y1, y1b)
    y32 = torch.empty(n, d)
    cnt32, _ = P(rowptr, col, x32, labels, c, y=y32)   # fp32 features: the feature buffer grows
    assert np.array_equal(cnt32, cnt1)
    y2 = torch.empty(n, d, dtype=BF16)
    cnt2, ns2 = P(rowptr, col, xb, labels, c, y=y2)    # bf16 again after the fp32 call
    check_counts(W, cnt2, ns2, s)
    W._lib.lib.wdgh_pipeline_host_release()

    scale = y_res.abs().max().item()
    assert (y1 - y_res).abs().max().item() <= 1e-5 * scale
    assert (y32 - y_res).abs().max().item() <= 1e-5 * scale
    assert torch.equal(y1, y32)          # both feature types take the same schedule (csrc/pipeline_host.cu)
    if d in (96, 70):
        assert torch.equal(y1, y_res)
    assert torch.equal(y2, y1.to(BF16))


def test_bf16_pipeline_distinct_negative_labels(W, host_graph):
    """several negative labels: the 1-byte label copy folds them together, the pipeline re-runs on int32 labels"""
    rowptr, col, labels, c, _ = host_graph
    n, d = int(labels.shape[0]), 128
    lab = labels.clone()
    rng = np.random.default_rng(5)
    neg = torch.from_numpy(rng.random(n) < 0.2)
    lab[neg] = torch.from_numpy(-rng.integers(1, 4, n).astype(np.int32))[neg]
    assert len(set(lab[lab < 0].tolist())) == 3
    g = W.CSRGraph.from_csr(rowptr, col, None, n)
    s = W.graph.structure_counts(g, lab.cuda(), c)
    xb = bf16_features(rng, n, d, device="cpu")
    y = torch.empty(n, d, dtype=BF16)
    cnt, ns = W.graph.pipeline_host(rowptr, col, xb, lab, c, y=y)
    W._lib.lib.wdgh_pipeline_host_release()
    check_counts(W, cnt, ns, s)
    assert cnt[W._lib.SC_N_MULTI_NEG] == 0
    y_res = W.spmm(g, xb.cuda(), W.NORM_SYM, True).cpu()
    assert (y.float() - y_res).abs().max().item() <= 1e-2 * y_res.abs().max().item()


def test_pipeline_host_argument_errors(W, host_graph):
    rowptr, col, labels, c, _ = host_graph
    n, d = int(labels.shape[0]), 64
    P = W.graph.pipeline_host
    xb = torch.zeros(n, d, dtype=BF16)
    x32 = torch.zeros(n, d)
    bad = [
        dict(x=xb.cuda()),                                      # device
        dict(rowptr=rowptr.cuda()),
        dict(x=torch.zeros(n, 2 * d, dtype=BF16)[:, ::2]),      # contiguity
        dict(y=torch.zeros(n, 2 * d)[:, :d]),
        dict(x=xb[: n - 1]),                                    # shape
        dict(y=torch.zeros(n, d + 1, dtype=BF16)),
        dict(labels=labels[:-1]),
        dict(x=x32.double()),                                   # dtypes
        dict(col=col.long()),
        dict(labels=labels.long()),
        dict(y=torch.zeros(n, d, dtype=torch.float64)),
        dict(x=x32, y=torch.zeros(n, d, dtype=BF16)),           # a bf16 y needs bf16 features
    ]
    for kw in bad:
        args = dict(rowptr=rowptr, col=col, x=xb, labels=labels, y=None)
        args.update(kw)
        with pytest.raises(ValueError):
            P(args["rowptr"], args["col"], args["x"], args["labels"], c, y=args["y"])


# ---------------------------------------------------------------------------
# fused step with bf16 features
# ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def big(W):
    """2M nodes, d = 128, a few split rows, 10 classes"""
    n, d = 2_000_000, 128
    gen = torch.Generator(device="cuda").manual_seed(3)
    deg = torch.randint(0, 12, (n,), device="cuda", generator=gen)
    deg[:4] = 5000
    rowptr = torch.zeros(n + 1, dtype=torch.int64, device="cuda")
    rowptr[1:] = torch.cumsum(deg, 0)
    nnz = int(rowptr[-1])
    col = torch.randint(0, n, (nnz,), device="cuda", generator=gen).to(torch.int32)
    g = W.CSRGraph(rowptr, col, None, n)
    xb = torch.randn(n, d, device="cuda", generator=gen).to(BF16)
    labels = torch.randint(0, 10, (n,), device="cuda", generator=gen).to(torch.int32)
    return g, xb, labels


def test_fused_bf16_equals_fp32_route(W, big):
    g, xb, labels = big
    F = W.graph.spmm_structure_fused
    y, (cnt, ns, *_) = F(g, xb, labels, 10)
    y = y.clone()
    cnt, ns = cnt.clone(), ns.clone()
    yb, _ = F(g, xb, labels, 10, out_dtype=BF16)
    assert y.dtype == torch.float32 and yb.dtype == BF16
    y32, (cnt32, ns32, *_) = F(g, xb.float(), labels, 10)
    assert torch.equal(y, y32) and torch.equal(yb, y32.to(BF16))
    assert torch.equal(cnt, cnt32)
    assert torch.allclose(ns, ns32, rtol=1e-12, atol=0)
    with pytest.raises(ValueError):
        F(g, xb.float(), labels, 10, out_dtype=BF16)


def test_fused_bf16_no_fp32_copy(W, big):
    g, xb, labels = big
    F = W.graph.spmm_structure_fused
    F(g, xb, labels, 10)              # plan, degree scale and split-row scratch
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    y, _ = F(g, xb, labels, 10)
    torch.cuda.synchronize()
    grew = torch.cuda.max_memory_allocated() - base
    scratch = g.n_chunks * xb.shape[1] * 4
    assert grew <= y.numel() * 4 + scratch + (64 << 20), grew
