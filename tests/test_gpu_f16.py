"""float16 feature matrices in the A_hat X aggregation (wdgh_spmm_csr_f16), its phased form (wdgh_spmm_csr_ranged_f16),
the host-buffer pipeline (wdgh_pipeline_host_f16) and the fused step.

fp16 -> fp32 is exact for every value (subnormals, +-0, +-inf and NaN included) and the fp16 kernels sum every row in the
order of the fp32 kernels, so the checks here are exact: fp32 output has the bits of the fp32 call on x.float(), fp16
output those of that result .to(torch.float16) (round to nearest even, overflow to +-inf).
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oracle import ref_port as O

pytestmark = pytest.mark.gpu

F16 = torch.float16
BF16 = torch.bfloat16


@pytest.fixture(scope="module")
def W():
    import wdgh_b200
    wdgh_b200._lib.require_device()
    return wdgh_b200


def f16_features(rng, n, d, device="cuda"):
    return torch.from_numpy(rng.standard_normal((n, d)).astype(np.float32)).to(device).to(F16)


_BITS = {torch.float32: torch.int32, torch.float16: torch.int16, torch.bfloat16: torch.int16}


def eq(a, b):
    """bit-identical: same dtype and shape, NaN in the same places, every other element the same bit pattern (so -0.0
    and +0.0 differ, which torch.equal would not see)"""
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    if not a.is_floating_point():
        return torch.equal(a, b)
    nan = a.isnan()
    if not torch.equal(nan, b.isnan()):
        return False
    bits = _BITS[a.dtype]
    return torch.equal(a.contiguous().view(bits)[~nan], b.contiguous().view(bits)[~nan])


def same(a, b):
    assert eq(a, b)


def check_both(W, g, xh, *args, **kw):
    """fp16 call == fp32 call on the upcast matrix (fp32 output), == its rounding (fp16 output)."""
    ref = W.spmm(g, xh.float(), *args, **kw)
    y = W.spmm(g, xh, *args, **kw)
    assert y.dtype == torch.float32
    same(y, ref)
    yh = W.spmm(g, xh, *args, out_dtype=F16, **kw)
    assert yh.dtype == F16
    same(yh, ref.to(F16))
    return ref, y, yh


def powerlaw_graph(n, avg_deg, seed, hubs=3, hub_deg=3000):
    rng = np.random.default_rng(seed)
    deg = np.minimum((rng.pareto(1.8, n) + 1) * avg_deg / 2.2, n // 2).astype(np.int64)
    src = np.repeat(np.arange(n), deg)
    dst = rng.integers(0, n, src.shape[0])
    hs = np.repeat(np.arange(hubs), hub_deg)
    hd = rng.integers(0, n, hs.shape[0])
    return O.coalesce(np.concatenate([src, hs, hd]), np.concatenate([dst, hd, hs]), None, n)


def ei_of(row, col):
    return torch.from_numpy(np.vstack([row, col]).astype(np.int64)).reshape(2, -1)


# ---------------------------------------------------------------------------
# resident aggregation
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("d", [1, 3, 4, 8, 19, 32, 64, 100, 128, 130, 256, 384, 512, 700])
def test_f16_widths(W, d):
    n = 3000
    row, col, _ = powerlaw_graph(n, 6, seed=d)
    rng = np.random.default_rng(d)
    val = torch.from_numpy((rng.random(row.shape[0]) + 0.5).astype(np.float32))
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), val, n, threshold=256)
    assert g.n_heavy >= 3
    check_both(W, g, f16_features(rng, n, d))


@pytest.mark.parametrize("self_loop", [True, False])
@pytest.mark.parametrize("norm", [0, 1, 2])
def test_f16_on_the_fly_norm(W, norm, self_loop):
    """binary graph with rows of >= 255 entries: their degree code is 255 and the SYM scale falls back to dinv"""
    n, d = 5000, 128
    row, col, _ = powerlaw_graph(n, 10, seed=7)
    keep = row != col
    g = W.CSRGraph.from_coo_indices(ei_of(row[keep], col[keep]), None, n)
    assert np.bincount(row[keep], minlength=n).max() >= 255
    check_both(W, g, f16_features(np.random.default_rng(1), n, d), norm, self_loop)


@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 64, 95, 1000])
@pytest.mark.parametrize("d", [32, 64, 128, 200, 256])
def test_f16_row_group_boundaries(W, n, d):
    rng = np.random.default_rng(n * 1000 + d)
    deg = rng.integers(0, 7, n)
    deg[rng.random(n) < 0.4] = 0              # many empty rows
    if n >= 64:
        deg[32:64] = 0                        # one group without any stored entry
    if n > 40:
        deg[n // 2] = min(n, 600)             # a split row (threshold 32 below)
    src = np.repeat(np.arange(n), deg)
    row, col, _ = O.coalesce(src, rng.integers(0, n, src.shape[0]), None, n)
    keep = row != col
    row, col = row[keep], col[keep]
    xh = f16_features(rng, n, d)
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), None, n, threshold=32)
    assert n <= 40 or g.n_heavy >= 1
    for norm in (2, 1):
        check_both(W, g, xh, norm, True)
    val = torch.from_numpy((rng.random(row.shape[0]) + 0.5).astype(np.float32))
    gv = W.CSRGraph.from_coo_indices(ei_of(row, col), val, n, threshold=32)
    _, y, yh = check_both(W, gv, xh)
    empty = torch.from_numpy(np.bincount(row, minlength=n) == 0).cuda()
    assert not y[empty].any() and not yh[empty].any()


def _kernels_launched(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return " ".join(e.key for e in prof.key_averages())


def test_f16_strided_and_misaligned_views(W):
    n, d = 3000, 128
    row, col, _ = powerlaw_graph(n, 6, seed=11)
    rng = np.random.default_rng(11)
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), None, n, threshold=256)
    xw = f16_features(rng, n, 384)
    x = xw[:, 128:256]                                  # ldx = 384 > d, read in place
    assert x.stride(0) == 384
    ref = W.spmm(g, x.float(), 2, True)
    assert eq(W.spmm(g, x, 2, True), ref)
    for dt in (torch.float32, F16):                     # out as a slab of a wider matrix
        yw = torch.full((n, 384), 7.0, dtype=dt, device="cuda")
        out = yw[:, 128:256]
        assert W.spmm(g, x, 2, True, out=out) is out
        assert eq(out, ref.to(dt))
        assert (yw[:, :128] == 7).all() and (yw[:, 256:] == 7).all()
    # a slab starting at column 2: rows are only 4-byte aligned -> the plain row kernel, same bits
    xm = xw[:, 2:2 + d]
    assert xm.data_ptr() % 8 == 4
    refm = W.spmm(g, xm.float(), 2, True)
    names = _kernels_launched(lambda: W.spmm(g, xm, 2, True))
    assert "spmm_rows_kernel" in names and "spmm_rowgroup_kernel" not in names
    assert eq(W.spmm(g, xm, 2, True), refm)
    yw = torch.zeros((n, 384), dtype=F16, device="cuda")
    assert eq(W.spmm(g, xm, 2, True, out=yw[:, 2:2 + d]), refm.to(F16))
    names = _kernels_launched(lambda: W.spmm(g, x, 2, True))
    assert "spmm_rowgroup_kernel" in names


def test_f16_broadcast_and_transposed_views(W):
    """layouts whose row stride is below d (broadcast rows, a transposed column) give the values of x.float()"""
    n, d = 500, 64
    row, col, _ = powerlaw_graph(n, 6, seed=12, hubs=0)
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), None, n)
    rng = np.random.default_rng(12)
    xe = f16_features(rng, 1, d).expand(n, d)           # stride (0, 1)
    assert xe.stride(0) == 0
    check_both(W, g, xe, 2, True)
    g1 = W.CSRGraph.from_coo_indices(torch.zeros(2, 1, dtype=torch.int64), None, 1)
    xt = f16_features(rng, d, 1).t()                    # [1, d] with stride (1, 1)
    assert xt.stride(0) < d
    ref = W.spmm(g1, torch.empty(1, d, device="cuda").copy_(xt), 2, True)
    assert eq(W.spmm(g1, xt, 2, True), ref)
    assert eq(W.spmm(g1, xt, 2, True, out_dtype=F16), ref.to(F16))


def test_f16_row_shard(W):
    """1-D partition: a CSRGraph of rows [r0, r1) with global column ids, global x and the global degree scale"""
    n, d = 4000, 128
    row, col, _ = powerlaw_graph(n, 8, seed=5)
    keep = row != col
    g = W.CSRGraph.from_coo_indices(ei_of(row[keep], col[keep]), None, n, threshold=64)
    dinv, _, code = g.degree_scale(2, True)
    xh = f16_features(np.random.default_rng(5), n, d)
    r0, r1 = 1000, 2500
    rp = g.rowptr[r0:r1 + 1]
    gs = W.CSRGraph(rp - rp[0], g.col[int(rp[0]):int(rp[-1])], None, r1 - r0, threshold=64, row_offset=r0, n_global=n)
    assert gs.n_heavy >= 1
    check_both(W, gs, xh, 2, True, dinv=dinv, deg_code=code)


# ---------------------------------------------------------------------------
# fp16 values: subnormals, signed zeros, the largest finite values, overflow, NaN and inf
# ---------------------------------------------------------------------------
def special_graph(W, n, seed, threshold=64):
    """every row has 2..8 entries, a few rows are split (threshold), weights 1"""
    rng = np.random.default_rng(seed)
    deg = rng.integers(2, 9, n)
    deg[:3] = 300
    src = np.repeat(np.arange(n), deg)
    row, col, _ = O.coalesce(src, rng.integers(0, n, src.shape[0]), None, n)
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), None, n, threshold=threshold)
    assert g.n_heavy >= 1
    return g, rng


@pytest.mark.parametrize("d", [3, 64, 128, 256])
def test_f16_subnormal_zero_and_max_inputs(W, d):
    """inputs drawn from the fp16 subnormals 2^-24 .. 2^-14, +-0 and +-65504 widen exactly"""
    n = 2000
    g, rng = special_graph(W, n, seed=d)
    pool = np.concatenate([2.0 ** np.arange(-24, -13), -(2.0 ** np.arange(-24, -13)), 3 * 2.0 ** np.arange(-24, -15),
                           [0.0, -0.0, 65504.0, -65504.0]]).astype(np.float32)
    x32 = torch.from_numpy(rng.choice(pool, (n, d))).cuda()
    x = x32.to(F16)
    assert eq(x.float(), x32)                 # every value of the pool is an fp16 value
    assert (x.float().abs() < 2.0 ** -14).any() and (x.float().abs() == 65504).any()
    assert (torch.signbit(x) & (x == 0)).any()
    for norm, sl in ((0, False), (0, True), (2, True)):
        check_both(W, g, x, norm, sl)


def test_f16_overflow_and_subnormal_sums(W):
    """sums above 65504 round to the same +-inf as torch's rounding, sums in the fp16 subnormal range to the same
    subnormals"""
    n, d = 2000, 128
    g, rng = special_graph(W, n, seed=3)
    big = torch.from_numpy(rng.choice(np.float32([40000.0, -40000.0, 65504.0]), (n, d))).cuda().to(F16)
    ref, _, yh = check_both(W, g, big)
    assert yh.isinf().sum() > 0 and (yh == float("-inf")).any() and (yh == float("inf")).any()
    assert ref.isfinite().all()
    tiny = torch.from_numpy(rng.choice(np.float32([2.0 ** -24, -(2.0 ** -24), 2.0 ** -20, 3 * 2.0 ** -22]),
                                       (n, d))).cuda().to(F16)
    _, _, yt = check_both(W, g, tiny)
    sub = (yt != 0) & (yt.float().abs() < 2.0 ** -14)
    assert sub.float().mean().item() > 0.5
    # the row-scaled sums: fp16 subnormals, some below the smallest one (rounded to signed zero)
    check_both(W, g, tiny, 1, True)


def test_f16_nan_and_inf_inputs(W):
    """NaN inputs give NaN in the same positions as the fp32 call on x.float(); inf - inf too"""
    n, d = 2000, 128
    g, rng = special_graph(W, n, seed=4)
    x = f16_features(rng, n, d)
    flat = x.view(-1)
    idx = torch.from_numpy(rng.choice(n * d, 300, replace=False)).cuda()
    flat[idx[:100]] = float("nan")
    flat[idx[100:200]] = float("inf")
    flat[idx[200:]] = float("-inf")
    for norm, sl in ((0, False), (2, True), (1, True)):
        ref, y, yh = check_both(W, g, x, norm, sl)
        assert ref.isnan().any() and y.isinf().any()


# ---------------------------------------------------------------------------
# no fp32 copy, determinism (2M nodes, 5000-entry split rows)
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
    xh = torch.randn(n, d, device="cuda", generator=gen).to(F16)
    labels = torch.randint(0, 10, (n,), device="cuda", generator=gen).to(torch.int32)
    return g, xh, labels


def test_f16_big_equals_fp32(W, big):
    g, xh, _ = big
    assert g.n_heavy >= 4
    check_both(W, g, xh, 2, True)


def test_f16_no_fp32_copy(W, big):
    g, xh, _ = big
    W.spmm(g, xh, 2, True)            # plan, degree scale and split-row scratch
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    y = W.spmm(g, xh, 2, True)
    torch.cuda.synchronize()
    grew = torch.cuda.max_memory_allocated() - base
    scratch = g.n_chunks * xh.shape[1] * 4
    assert grew <= y.numel() * 4 + scratch + (64 << 20), grew


def test_f16_deterministic(W, big):
    g, xh, _ = big
    assert eq(W.spmm(g, xh, 2, True), W.spmm(g, xh, 2, True))
    assert eq(W.spmm(g, xh, 2, True, out_dtype=F16), W.spmm(g, xh, 2, True, out_dtype=F16))


def test_fused_f16_equals_fp32_route(W, big):
    g, xh, labels = big
    F = W.graph.spmm_structure_fused
    y, (cnt, ns, *_) = F(g, xh, labels, 10)
    y = y.clone()
    cnt, ns = cnt.clone(), ns.clone()
    yh, _ = F(g, xh, labels, 10, out_dtype=F16)
    assert y.dtype == torch.float32 and yh.dtype == F16
    y32, (cnt32, ns32, *_) = F(g, xh.float(), labels, 10)
    assert eq(y, y32) and eq(yh, y32.to(F16))
    assert eq(cnt, cnt32)
    assert torch.allclose(ns, ns32, rtol=1e-12, atol=0)
    for bad in (BF16, torch.float64):
        with pytest.raises(ValueError):
            F(g, xh, labels, 10, out_dtype=bad)
    with pytest.raises(ValueError):
        F(g, xh.float(), labels, 10, out_dtype=F16)


def test_fused_f16_no_fp32_copy(W, big):
    g, xh, labels = big
    F = W.graph.spmm_structure_fused
    F(g, xh, labels, 10)              # plan, degree scale and split-row scratch
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    y, _ = F(g, xh, labels, 10)
    torch.cuda.synchronize()
    grew = torch.cuda.max_memory_allocated() - base
    scratch = g.n_chunks * xh.shape[1] * 4
    assert grew <= y.numel() * 4 + scratch + (64 << 20), grew


# ---------------------------------------------------------------------------
# phased aggregation
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("d", [32, 64, 128, 256])
@pytest.mark.parametrize("weighted,codes", [(False, True), (False, False), (True, False)])
def test_f16_phases_equal_fp32_phases(W, d, weighted, codes):
    """own-shard phase read in place through x_row0, then the columns before / after it with accumulate, finalize
    and the split rows (threshold 256) -- every phase bit-identical to the fp32 phase on x.float()"""
    n, parts = 20000, 3
    row, col, _ = powerlaw_graph(n, 10, seed=d)
    keep = row != col
    row, col = row[keep], col[keep]
    rng = np.random.default_rng(d)
    val = torch.from_numpy((rng.random(row.shape[0]) + 0.5).astype(np.float32)) if weighted else None
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), val, n, threshold=256)
    assert g.n_heavy > 0
    xh = f16_features(rng, n, d)
    x32 = xh.float()
    dinv, _, code = g.degree_scale(W.NORM_SYM, True)
    code = code if codes else None
    block = (n + parts - 1) // parts
    seg = W.graph.column_segments(g, [b * block for b in range(parts)] + [n])
    skip = W.graph.heavy_flags(g)
    y_ref = W.spmm(g, xh, W.NORM_SYM, True)
    for r in range(parts):
        lo, hi = r * block, min((r + 1) * block, n)
        first, last = r == 0, r == parts - 1
        ys = []
        for x in (xh, x32):
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
        for sh, sf in zip(*ys):
            same(sh, sf)
        y = ys[0][-1]
        assert not y.isnan().any()
        assert (y - y_ref).abs().max().item() <= 1e-5 * y_ref.abs().max().item()


def test_f16_phase_errors(W):
    lib = W._lib.lib
    n = 2000
    row, col, _ = powerlaw_graph(n, 6, seed=1, hubs=0)
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), None, n, threshold=1 << 20)
    assert g.n_chunks == 0
    plan, host = g.plan
    p = W._lib.ptr
    rb, re = g.rowptr[:-1], g.rowptr[1:]
    xw = f16_features(np.random.default_rng(1), n, 256)
    y = torch.empty(n, 256, device="cuda")

    def call(x, d, ldx):
        return lib.wdgh_spmm_csr_ranged_f16(p(g.rowptr), p(rb), p(re), p(g.col), None, n, p(x), d, ldx, p(y), d, 0, 1,
                                            None, None, None, 0, 1, 1, p(plan), host, None, 0, None)

    assert call(xw, 128, 256) == 0
    torch.cuda.synchronize()
    for x, d, ldx in ((xw, 96, 256), (xw[:, 2:], 128, 256), (xw, 128, 130)):
        assert call(x, d, ldx) == -1, (d, ldx)
        err = lib.wdgh_last_error()
        assert err.startswith(b"wdgh_spmm_csr_ranged_f16: ") and b"8-byte aligned rows" in err, err
    x = xw[:, :128]
    y128 = torch.empty(n, 128, device="cuda")
    args = (0, True, None, None, None, False, True, True)
    with pytest.raises(ValueError):
        W.graph.spmm_ranged(g, rb, re, x, y128, *args, extra=torch.zeros(1, n, 128, device="cuda"))
    with pytest.raises(ValueError):
        W.graph.spmm_ranged(g, rb, re, x, y128, *args, ctas_per_sm=8)
    for dt in (F16, BF16):
        with pytest.raises(ValueError):
            W.graph.spmm_ranged(g, rb, re, x, torch.empty(n, 128, dtype=dt, device="cuda"), *args)


# ---------------------------------------------------------------------------
# host-buffer pipeline
# ---------------------------------------------------------------------------
@pytest.fixture(scope="module")
def host_graph():
    n, c = 50000, 7
    row, col, _ = powerlaw_graph(n, 14, seed=128)
    keep = row != col
    row, col = row[keep], col[keep]
    rng = np.random.default_rng(3)
    labels = rng.integers(0, c, n).astype(np.int32)
    labels[rng.random(n) < 0.1] = -1
    rowptr = torch.from_numpy(O.csr_from_coo(row, n).astype(np.int64))
    return rowptr, torch.from_numpy(col.astype(np.int32)), torch.from_numpy(labels), c


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
                                    (160, "not a multiple of 64: 16 row blocks, one phase per arriving block"),
                                    (96, "one copy, then one launch"),
                                    (70, "d % 4 != 0: one launch through the fp16 SpMM dispatch"),
                                    (7, "odd d: the fp16 Y is rounded element by element")])
def test_f16_pipeline_forms(W, host_graph, d, form):
    rowptr, col, labels, c = host_graph
    n = int(labels.shape[0])
    P = W.graph.pipeline_host
    xh = f16_features(np.random.default_rng(d), n, d, device="cpu")
    x32 = xh.float()
    g = W.CSRGraph.from_csr(rowptr, col, None, n)
    assert g.n_heavy > 0
    s = W.graph.structure_counts(g, labels.cuda(), c)
    y_res = W.spmm(g, xh.cuda(), W.NORM_SYM, True).cpu()

    W._lib.lib.wdgh_pipeline_host_release()      # the first call below sizes the feature buffer for fp16
    cnt0, ns0 = P(rowptr, col, xh, labels, c)    # counters only
    check_counts(W, cnt0, ns0, s)
    y1 = torch.empty(n, d)
    cnt1, ns1 = P(rowptr, col, xh, labels, c, y=y1)
    check_counts(W, cnt1, ns1, s)
    y2 = torch.empty(n, d, dtype=F16)
    cnt2, ns2 = P(rowptr, col, xh, labels, c, y=y2)
    check_counts(W, cnt2, ns2, s)
    y32 = torch.empty(n, d)
    cnt32, _ = P(rowptr, col, x32, labels, c, y=y32)   # fp32 features: the feature buffer grows
    assert np.array_equal(cnt32, cnt1)
    yb = torch.empty(n, d, dtype=BF16)
    P(rowptr, col, xh.to(BF16), labels, c, y=yb)       # bf16 between fp16 calls: same cache, same 2-byte staging
    y2b = torch.empty(n, d, dtype=F16)
    P(rowptr, col, xh, labels, c, y=y2b)
    W._lib.lib.wdgh_pipeline_host_release()

    scale = y_res.abs().max().item()
    assert (y1 - y_res).abs().max().item() <= 1e-5 * scale
    assert eq(y1, y32)          # every feature type takes the same schedule (csrc/pipeline_host.cu)
    if d in (96, 70, 7):
        assert eq(y1, y_res)
    assert eq(y2, y1.to(F16)) and eq(y2b, y2)


def test_f16_pipeline_type_errors(W, host_graph):
    rowptr, col, labels, c = host_graph
    n, d = int(labels.shape[0]), 64
    P = W.graph.pipeline_host
    xh = torch.zeros(n, d, dtype=F16)
    for x, y in ((xh, torch.zeros(n, d, dtype=BF16)),           # the half y must have the type of x
                 (xh.to(BF16), torch.zeros(n, d, dtype=F16)),
                 (xh.float(), torch.zeros(n, d, dtype=F16)),
                 (xh, torch.zeros(n, d, dtype=torch.float64))):
        with pytest.raises(ValueError):
            P(rowptr, col, x, labels, c, y=y)
    lib = W._lib.lib
    cnt = np.zeros(W._lib.sc_words(c), np.int64)
    ns = np.zeros(2, np.float64)
    y = torch.zeros(n, d, dtype=F16)
    for fn, x, y_dtype in ((lib.wdgh_pipeline_host_f16, xh, W._lib.DTYPE_BF16),
                           (lib.wdgh_pipeline_host_bf16, xh.to(BF16), W._lib.DTYPE_F16)):
        assert fn(rowptr.data_ptr(), col.data_ptr(), n, int(col.shape[0]), x.data_ptr(), d, labels.data_ptr(), c, 2, 1,
                  y.data_ptr(), y_dtype, cnt.ctypes.data, ns.ctypes.data) == -1
        err = lib.wdgh_last_error()
        assert err.startswith(fn.__name__.encode() + b": ") and b"y_dtype" in err, err


# ---------------------------------------------------------------------------
# C ABI, Python refusals, mirrors
# ---------------------------------------------------------------------------
def test_f16_errors(W):
    lib = W._lib.lib
    n, d = 64, 8
    row, col, _ = powerlaw_graph(n, 4, seed=1, hubs=0)
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), None, n)
    plan, host = g.plan
    xh = f16_features(np.random.default_rng(1), n, d)
    y = torch.empty(n, d, device="cuda")
    p = W._lib.ptr

    def call(fn, x, y_dtype):
        return fn(p(g.rowptr), p(g.col), None, n, p(x), d, d, p(y), d, y_dtype, 0, 1, None, None, p(plan), host,
                  None, 0, None)

    assert call(lib.wdgh_spmm_csr_f16, xh, W._lib.DTYPE_F16) == 0
    torch.cuda.synchronize()
    for fn, x, y_dtype in ((lib.wdgh_spmm_csr_f16, xh, W._lib.DTYPE_BF16),
                           (lib.wdgh_spmm_csr_bf16, xh.to(BF16), W._lib.DTYPE_F16),
                           (lib.wdgh_spmm_csr_f16, xh, 7)):
        assert call(fn, x, y_dtype) == -1
        err = lib.wdgh_last_error()
        assert err.startswith(fn.__name__.encode() + b": ") and b"y_dtype" in err, err
    for bad in (BF16, torch.float64):                  # a half output has the type of the features
        with pytest.raises(ValueError):
            W.spmm(g, xh, out_dtype=bad)
        with pytest.raises(ValueError):
            W.spmm(g, xh, out=torch.empty(n, d, dtype=bad, device="cuda"))
    with pytest.raises(ValueError):
        W.spmm(g, xh.to(BF16), out_dtype=F16)
    with pytest.raises(ValueError):
        W.spmm(g, xh.float(), out_dtype=F16)
    with pytest.raises(ValueError):
        W.spmm(g, xh.float(), out=torch.empty(n, d, dtype=F16, device="cuda"))


def test_f16_vs_oracle(W):
    n, d = 3000, 128
    row, col, _ = powerlaw_graph(n, 6, seed=4)
    rng = np.random.default_rng(4)
    val = (rng.random(row.shape[0]) + 0.5).astype(np.float32)
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), torch.from_numpy(val), n, threshold=256)
    xh = f16_features(rng, n, d)
    y = W.spmm(g, xh).cpu().numpy()
    ref = O.spmm(row, col, val, n, xh.float().cpu().numpy())
    np.testing.assert_allclose(y, ref, rtol=1e-4, atol=1e-5 * np.abs(ref).max())


def test_propagate_f16(W):
    n, d = 2000, 64
    rng = np.random.default_rng(9)
    a = sp.random(n, n, density=0.004, format="csr", random_state=9)
    adj = ((a + a.T) > 0).astype(np.float32)
    xh = f16_features(rng, n, d)
    ref = W.util_funcs.propagate(adj, xh.float())
    y = W.util_funcs.propagate(adj, xh)
    assert y.dtype == torch.float32 and eq(y, ref)
    yh = W.util_funcs.propagate(adj, xh, out_dtype=F16)
    assert yh.dtype == F16 and eq(yh, ref.to(F16))


def test_similarity_f16_one_hot(W):
    """fp16 one-hot features are aggregated without the fp32 copy and give the fp32 score"""
    n, c = 3000, 5
    row, col, _ = powerlaw_graph(n, 6, seed=21, hubs=0)
    idx = ei_of(row, col)
    A = torch.sparse_coo_tensor(idx, torch.ones(idx.shape[1]), (n, n)).coalesce().cuda()
    labels = torch.from_numpy(np.random.default_rng(21).integers(0, c, n))
    oh = torch.eye(c)[labels]
    hm = W.homophily_metrics
    for kw in (dict(hard=None, LP=1), dict(hard=1, LP=1), dict(hard=None, LP=1, ifsum=0)):
        want = hm.similarity(oh, A, oh, **kw)
        got = hm.similarity(oh.half(), A, oh, **kw)
        assert eq(got, want), kw
