"""bfloat16 feature matrices in the A_hat X aggregation (wdgh_spmm_csr_bf16, graph.spmm with a bf16 `x`).

bf16 -> fp32 is exact and the bf16 kernels sum every row in the order of the fp32 kernels, so the checks here are
exact: fp32 output is torch.equal to the fp32 call on x.float(), bf16 output to that result .to(torch.bfloat16).
"""
import numpy as np
import pytest
import scipy.sparse as sp
import torch

from oracle import ref_port as O

pytestmark = pytest.mark.gpu

RTOL = 1e-4
BF16 = torch.bfloat16


@pytest.fixture(scope="module")
def W():
    import wdgh_b200
    wdgh_b200._lib.require_device()
    return wdgh_b200


def bf16_features(rng, n, d):
    return torch.from_numpy(rng.standard_normal((n, d)).astype(np.float32)).cuda().to(BF16)


def check_both(W, g, xb, *args, **kw):
    """bf16 call == fp32 call on the upcast matrix (fp32 output), == its rounding (bf16 output)."""
    ref = W.spmm(g, xb.float(), *args, **kw)
    y = W.spmm(g, xb, *args, **kw)
    assert y.dtype == torch.float32 and torch.equal(y, ref)
    yb = W.spmm(g, xb, *args, out_dtype=BF16, **kw)
    assert yb.dtype == BF16 and torch.equal(yb, ref.to(BF16))
    return ref, y, yb


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


@pytest.mark.parametrize("d", [1, 3, 4, 8, 19, 32, 64, 100, 128, 130, 256, 384, 512, 700])
def test_bf16_widths(W, d):
    n = 3000
    row, col, _ = powerlaw_graph(n, 6, seed=d)
    rng = np.random.default_rng(d)
    val = torch.from_numpy((rng.random(row.shape[0]) + 0.5).astype(np.float32))
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), val, n, threshold=256)
    assert g.n_heavy >= 3
    check_both(W, g, bf16_features(rng, n, d))


@pytest.mark.parametrize("norm,self_loop", [(1, True), (2, True), (1, False), (2, False)])
def test_bf16_on_the_fly_norm(W, norm, self_loop):
    """binary graph with rows of >= 255 entries: their degree code is 255 and the SYM scale falls back to dinv"""
    n, d = 5000, 128
    row, col, _ = powerlaw_graph(n, 10, seed=7)
    keep = row != col
    g = W.CSRGraph.from_coo_indices(ei_of(row[keep], col[keep]), None, n)
    assert np.bincount(row[keep], minlength=n).max() >= 255
    check_both(W, g, bf16_features(np.random.default_rng(1), n, d), norm, self_loop)


@pytest.mark.parametrize("n", [1, 2, 31, 32, 33, 64, 95, 1000])
@pytest.mark.parametrize("d", [32, 64, 128, 200, 256])
def test_bf16_row_group_boundaries(W, n, d):
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
    xb = bf16_features(rng, n, d)
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), None, n, threshold=32)
    assert n <= 40 or g.n_heavy >= 1
    for norm in (2, 1):
        check_both(W, g, xb, norm, True)
    val = torch.from_numpy((rng.random(row.shape[0]) + 0.5).astype(np.float32))
    gv = W.CSRGraph.from_coo_indices(ei_of(row, col), val, n, threshold=32)
    _, y, yb = check_both(W, gv, xb)
    empty = torch.from_numpy(np.bincount(row, minlength=n) == 0).cuda()
    assert not y[empty].any() and not yb[empty].any()


def _kernels_launched(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return " ".join(e.key for e in prof.key_averages())


def test_bf16_strided_and_misaligned_views(W):
    n, d = 3000, 128
    row, col, _ = powerlaw_graph(n, 6, seed=11)
    rng = np.random.default_rng(11)
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), None, n, threshold=256)
    xw = bf16_features(rng, n, 384)
    x = xw[:, 128:256]                                  # ldx = 384 > d, read in place
    assert x.stride(0) == 384
    ref = W.spmm(g, x.float(), 2, True)
    assert torch.equal(W.spmm(g, x, 2, True), ref)
    for dt in (torch.float32, BF16):                    # out as a slab of a wider matrix
        yw = torch.full((n, 384), 7.0, dtype=dt, device="cuda")
        out = yw[:, 128:256]
        assert W.spmm(g, x, 2, True, out=out) is out
        assert torch.equal(out, ref.to(dt))
        assert (yw[:, :128] == 7).all() and (yw[:, 256:] == 7).all()
    # a slab starting at column 2: rows are only 4-byte aligned -> the plain row kernel, same bits
    xm = xw[:, 2:2 + d]
    assert xm.data_ptr() % 8 == 4
    refm = W.spmm(g, xm.float(), 2, True)
    names = _kernels_launched(lambda: W.spmm(g, xm, 2, True))
    assert "spmm_rows_kernel" in names and "spmm_rowgroup_kernel" not in names
    assert torch.equal(W.spmm(g, xm, 2, True), refm)
    yw = torch.zeros((n, 384), dtype=BF16, device="cuda")
    assert torch.equal(W.spmm(g, xm, 2, True, out=yw[:, 2:2 + d]), refm.to(BF16))
    names = _kernels_launched(lambda: W.spmm(g, x, 2, True))
    assert "spmm_rowgroup_kernel" in names


def test_bf16_broadcast_and_transposed_views(W):
    """layouts whose row stride is below d (broadcast rows, a transposed column) give the values of x.float()"""
    n, d = 500, 64
    row, col, _ = powerlaw_graph(n, 6, seed=12, hubs=0)
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), None, n)
    rng = np.random.default_rng(12)
    xe = bf16_features(rng, 1, d).expand(n, d)          # stride (0, 1)
    assert xe.stride(0) == 0
    check_both(W, g, xe, 2, True)
    g1 = W.CSRGraph.from_coo_indices(torch.zeros(2, 1, dtype=torch.int64), None, 1)
    xt = bf16_features(rng, d, 1).t()                   # [1, d] with stride (1, 1)
    assert xt.stride(0) < d
    ref = W.spmm(g1, torch.empty(1, d, device="cuda").copy_(xt), 2, True)
    assert torch.equal(W.spmm(g1, xt, 2, True), ref)
    assert torch.equal(W.spmm(g1, xt, 2, True, out_dtype=BF16), ref.to(BF16))


def test_bf16_row_shard(W):
    """1-D partition: a CSRGraph of rows [r0, r1) with global column ids, global x and the global degree scale"""
    n, d = 4000, 128
    row, col, _ = powerlaw_graph(n, 8, seed=5)
    keep = row != col
    g = W.CSRGraph.from_coo_indices(ei_of(row[keep], col[keep]), None, n, threshold=64)
    dinv, _, code = g.degree_scale(2, True)
    xb = bf16_features(np.random.default_rng(5), n, d)
    r0, r1 = 1000, 2500
    rp = g.rowptr[r0:r1 + 1]
    gs = W.CSRGraph(rp - rp[0], g.col[int(rp[0]):int(rp[-1])], None, r1 - r0, threshold=64, row_offset=r0, n_global=n)
    assert gs.n_heavy >= 1
    check_both(W, gs, xb, 2, True, dinv=dinv, deg_code=code)


@pytest.fixture(scope="module")
def big(W):
    """2M nodes, d = 128, a few split rows"""
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
    return g, xb


def test_bf16_no_fp32_copy(W, big):
    g, xb = big
    W.spmm(g, xb, 2, True)            # plan, degree scale and split-row scratch
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    y = W.spmm(g, xb, 2, True)
    torch.cuda.synchronize()
    grew = torch.cuda.max_memory_allocated() - base
    scratch = g.n_chunks * xb.shape[1] * 4
    assert grew <= y.numel() * 4 + scratch + (64 << 20), grew


def test_bf16_deterministic(W, big):
    g, xb = big
    a = W.spmm(g, xb, 2, True)
    b = W.spmm(g, xb, 2, True)
    assert torch.equal(a, b)
    assert torch.equal(W.spmm(g, xb, 2, True, out_dtype=BF16), W.spmm(g, xb, 2, True, out_dtype=BF16))


def test_propagate_bf16(W):
    n, d = 2000, 64
    rng = np.random.default_rng(9)
    a = sp.random(n, n, density=0.004, format="csr", random_state=9)
    adj = ((a + a.T) > 0).astype(np.float32)
    xb = bf16_features(rng, n, d)
    ref = W.util_funcs.propagate(adj, xb.float())
    y = W.util_funcs.propagate(adj, xb)
    assert y.dtype == torch.float32 and torch.equal(y, ref)
    yb = W.util_funcs.propagate(adj, xb, out_dtype=BF16)
    assert yb.dtype == BF16 and torch.equal(yb, ref.to(BF16))


def test_bf16_errors(W):
    lib = W._lib.lib
    n, d = 64, 8
    row, col, _ = powerlaw_graph(n, 4, seed=1, hubs=0)
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), None, n)
    plan, host = g.plan
    xb = bf16_features(np.random.default_rng(1), n, d)
    y = torch.empty(n, d, device="cuda")
    dinv = g.degree_scale(2, True)[0]
    p = W._lib.ptr

    def call(x=xb, ldx=d, yp=None, y_dtype=0, norm=0, dv=None):
        return lib.wdgh_spmm_csr_bf16(p(g.rowptr), p(g.col), None, n, p(x), d, ldx, p(y) if yp is None else yp, d,
                                      y_dtype, norm, 1, p(dv), None, p(plan), host, None, 0, None)

    assert call(dv=dinv, norm=2) == 0
    torch.cuda.synchronize()
    for kw, msg in ((dict(y_dtype=7), b"y_dtype"), (dict(yp=p(xb)), b"in-place"), (dict(ldx=d - 1), b"bad shape"),
                    (dict(norm=2), b"norm requires dinv")):
        assert call(**kw) == -1, kw
        err = lib.wdgh_last_error()
        assert err.startswith(b"wdgh_spmm_csr_bf16: ") and msg in err, err
    with pytest.raises(ValueError):
        W.spmm(g, xb, out=torch.empty(n, d, dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        W.spmm(g, xb.float(), out=torch.empty(n, d, dtype=torch.float64, device="cuda"))
    with pytest.raises(ValueError):
        W.spmm(g, xb.float(), out_dtype=BF16)
    with pytest.raises(ValueError):
        W.spmm(g, xb.float(), out=torch.empty(n, d, dtype=BF16, device="cuda"))


def test_bf16_vs_oracle(W):
    n, d = 3000, 128
    row, col, _ = powerlaw_graph(n, 6, seed=4)
    rng = np.random.default_rng(4)
    val = (rng.random(row.shape[0]) + 0.5).astype(np.float32)
    g = W.CSRGraph.from_coo_indices(ei_of(row, col), torch.from_numpy(val), n, threshold=256)
    xb = bf16_features(rng, n, d)
    y = W.spmm(g, xb).cpu().numpy()
    ref = O.spmm(row, col, val, n, xb.float().cpu().numpy())
    np.testing.assert_allclose(y, ref, rtol=RTOL, atol=1e-5 * np.abs(ref).max())
