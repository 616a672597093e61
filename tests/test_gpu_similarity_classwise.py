"""The Gram-free aggregation similarity (csrc/class_sums.cu, graph.class_inner_sums / graph.las_weights): w[i][c] =
<z_i, s_c> with fp64 class sums s_c, against exact references and against the Gram path it replaces above
graph.GRAM_SIMILARITY_MAX_ROWS rows.

* Integer z with every partial sum of both paths below 2^24: w equals the float64 restatement and class_colsum(gram(z))
  in all three Gram modes bit for bit, at the segment / tile / class-tile boundaries.
* Random floats: one final rounding plus fp64-accumulation slack, tighter than the Gram path's own bound.
* The mirrors (homophily_metrics / homophily_plot similarity) on the new path reproduce the golden fixtures.
* A whole 131,073-node graph with the shipped threshold: no Gram, exact integer w.
"""
import numpy as np
import pytest
import torch

import _golden as GD
from oracle import ref_port as O

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]

MODES = {"simt": 0, "tc": 1, "tc_faithful": 2}   # GRAM_SIMT, GRAM_TC, GRAM_TC_FAITHFUL (include/wdgh_b200.h)


@pytest.fixture(scope="module")
def W():
    import wdgh_b200
    wdgh_b200._lib.require_device()
    return wdgh_b200


def gram_mode(W, z, mode):
    lib = W._lib.lib
    m, d = z.shape
    g = torch.empty((m, m), dtype=torch.float32, device="cuda")
    ws = torch.empty(max(1, int(lib.wdgh_gram_workspace_floats(m, d))), dtype=torch.float32, device="cuda")
    rc = lib.wdgh_gram(z.data_ptr(), m, d, z.stride(0), g.data_ptr(), m, mode, ws.data_ptr(), W._lib.stream_ptr())
    assert rc == 0, W._lib.last_error()
    return g


def restate(z64, labels, n_cls, is_mean):
    """float64 restatement: exact whenever every partial sum is an integer below 2^53."""
    y = np.zeros((z64.shape[0], n_cls))
    ok = (labels >= 0) & (labels < n_cls)
    y[np.nonzero(ok)[0], labels[ok]] = 1
    s = y.T @ z64                                   # [C, d]
    w = z64 @ s.T                                   # [m, C]
    if is_mean:
        with np.errstate(invalid="ignore", divide="ignore"):
            w = w / y.sum(0)
    return w


# ---------------------------------------------------------------------------
# 1. exact on integer inputs
# ---------------------------------------------------------------------------
M_EDGES = [1, 31, 32, 33, 255, 256, 257, 4099]


@pytest.mark.parametrize("n_cls", [1, 2, 10, 64, 65, 300])
@pytest.mark.parametrize("d", [1, 2, 7, 16, 32, 33, 128, 129, 300])
def test_integer_inputs_exact(W, d, n_cls):
    """z in [-3, 3]: |partial sums| <= 4099 * 300 * 9 < 2^24 in either path, so every order gives the exact value"""
    for m in M_EDGES:
        gen = torch.Generator(device="cuda").manual_seed(m * 7919 + d * 31 + n_cls)
        z = torch.randint(-3, 4, (m, d), generator=gen, device="cuda").to(torch.float32)
        labels = torch.randint(0, n_cls, (m,), generator=gen, device="cuda").to(torch.int32)
        lab = labels.cpu().numpy()
        z64 = z.cpu().numpy().astype(np.float64)
        grams = {k: gram_mode(W, z, v) for k, v in MODES.items()}
        for is_mean in (False, True):
            got = W.graph.class_inner_sums(z, labels, n_cls, is_mean=is_mean).cpu().numpy()
            want = restate(z64, lab, n_cls, is_mean).astype(np.float32)
            assert np.array_equal(got, want, equal_nan=True), (m, d, n_cls, is_mean)
            for mode, g in grams.items():
                ref = W.graph.class_colsum(g, labels, n_cls, is_mean=is_mean).cpu().numpy()
                assert np.array_equal(got, ref, equal_nan=True), (m, d, n_cls, is_mean, mode)


# ---------------------------------------------------------------------------
# 2. edge cases
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("m,d,ldz", [(300, 7, 9), (1000, 128, 131), (4099, 33, 64)])
def test_strided_view_same_bits(W, m, d, ldz):
    """ldz > d: NaN in the unused columns (never read), same bits as the contiguous copy"""
    gen = torch.Generator(device="cuda").manual_seed(ldz)
    buf = torch.full((m, ldz), float("nan"), device="cuda")
    buf[:, :d] = torch.randn((m, d), generator=gen, device="cuda")
    labels = torch.randint(0, 5, (m,), generator=gen, device="cuda").to(torch.int32)
    view = buf[:, :d]
    assert view.stride(0) == ldz
    for is_mean in (False, True):
        a = W.graph.class_inner_sums(view, labels, 5, is_mean=is_mean)
        b = W.graph.class_inner_sums(view.contiguous(), labels, 5, is_mean=is_mean)
        assert torch.equal(a, b)
        assert not torch.isnan(a).any()


def test_out_of_range_labels_join_no_class(W):
    n_cls, m, d = 4, 1000, 12
    rng = np.random.default_rng(1)
    z = rng.integers(-5, 6, (m, d)).astype(np.float32)
    labels = rng.integers(0, n_cls, m).astype(np.int64)
    odd = rng.permutation(m)[:200]
    labels[odd] = rng.choice([-1, n_cls, 254, 2 ** 31 - 1], 200)
    lab32 = torch.from_numpy(labels.astype(np.int32)).cuda()
    zt = torch.from_numpy(z).cuda()
    for is_mean in (False, True):
        got = W.graph.class_inner_sums(zt, lab32, n_cls, is_mean=is_mean).cpu().numpy()
        want = restate(z.astype(np.float64), labels, n_cls, is_mean).astype(np.float32)
        assert np.array_equal(got, want)
        ref = W.graph.class_colsum(W.graph.gram(zt), lab32, n_cls, is_mean=is_mean).cpu().numpy()
        assert np.array_equal(got, ref)


def test_empty_class_and_empty_input(W):
    m, d, n_cls = 500, 9, 6
    rng = np.random.default_rng(2)
    z = torch.from_numpy(rng.integers(-4, 5, (m, d)).astype(np.float32)).cuda()
    labels = rng.integers(0, n_cls, m)
    labels[labels == 3] = 5                           # class 3 empty
    lab32 = torch.from_numpy(labels.astype(np.int32)).cuda()
    s = W.graph.class_inner_sums(z, lab32, n_cls).cpu().numpy()
    mean = W.graph.class_inner_sums(z, lab32, n_cls, is_mean=True).cpu().numpy()
    assert (s[:, 3] == 0).all() and np.signbit(s[:, 3]).sum() == 0
    assert np.isnan(mean[:, 3]).all() and not np.isnan(np.delete(mean, 3, 1)).any()
    w0 = W.graph.class_inner_sums(torch.empty((0, d), device="cuda"), lab32[:0], n_cls)
    assert w0.shape == (0, n_cls)
    lib = W._lib.lib
    assert lib.wdgh_class_inner_sums(None, 0, d, d, None, n_cls, 0, None, None, None) == 0   # m = 0: no-op
    assert lib.wdgh_class_inner_sums(None, 4, d, d - 1, None, n_cls, 0, None, None, None) < 0
    assert lib.wdgh_class_inner_workspace_doubles(10, 0, 3) == -1


# ---------------------------------------------------------------------------
# 3. accuracy on random floats
# ---------------------------------------------------------------------------
def gram_bound(mode, d):
    """Relative bound of the Gram kernels (tests/test_gpu_gram_modes.py::bound)."""
    u = 2.0 ** -24
    if mode == "simt":
        return d * u / (1 - d * u)
    chunk = 1 if mode == "tc_faithful" else 4
    n_chunks = -(-(-(-d // 32)) // chunk)
    return 3 * (1 + 2.0 ** -10) * 2.0 ** -22 + 10 * (12 * chunk) * 2.0 ** -23 * (1 + 2.0 ** -10) + n_chunks * u


@pytest.mark.parametrize("d", [10, 128])
def test_accuracy_random_floats(W, d):
    m, n_cls = 20_011, 7
    rng = np.random.default_rng(d)
    z = rng.standard_normal((m, d)).astype(np.float32)
    labels = rng.integers(0, n_cls, m)
    z64 = z.astype(np.float64)
    w64 = restate(z64, labels, n_cls, False)
    y = np.eye(n_cls)[labels]
    mass = np.abs(z64) @ (y.T @ np.abs(z64)).T        # (|z| a^T)[i][c], a_c = sum_{j in c} |z_j|
    zt = torch.from_numpy(z).cuda()
    lab32 = torch.from_numpy(labels.astype(np.int32)).cuda()
    got = W.graph.class_inner_sums(zt, lab32, n_cls).cpu().numpy().astype(np.float64)
    err = np.abs(got - w64)
    assert (err <= 2.0 ** -24 * np.abs(w64) + 2.0 ** -30 * mass).all(), float((err / mass).max())
    # the Gram path (the tensor-core mode las_weights uses at d > 32, the SIMT kernel below) within its own bound:
    # Gram entries per tests/test_gpu_gram_modes.py, then class_colsum's fp32 sum of ceil(m / 32) terms per lane and
    # a 5-level warp tree
    mode = "tc" if d > 32 else "simt"
    gw = W.graph.class_colsum(W.graph.gram(zt), lab32, n_cls).cpu().numpy().astype(np.float64)
    err_g = np.abs(gw - w64)
    tol_g = (gram_bound(mode, d) + (-(-m // 32) + 6) * 2.0 ** -24) * mass
    assert (err_g <= tol_g).all(), float((err_g / mass).max())
    print(f"d={d}: max err / mass: class sums {float((err / mass).max()):.3e}, Gram {float((err_g / mass).max()):.3e}")
    assert (err / mass).max() <= (err_g / mass).max()


# ---------------------------------------------------------------------------
# 4. determinism
# ---------------------------------------------------------------------------
def test_deterministic(W):
    gen = torch.Generator(device="cuda").manual_seed(4)
    z = torch.randn((300_001, 128), generator=gen, device="cuda")
    labels = torch.randint(0, 10, (300_001,), generator=gen, device="cuda").to(torch.int32)
    a = W.graph.class_inner_sums(z, labels, 10)
    b = W.graph.class_inner_sums(z, labels, 10)
    assert torch.equal(a, b)
    z1 = z[:, :10].contiguous()
    assert torch.equal(W.graph.class_inner_sums(z1, labels, 10, True), W.graph.class_inner_sums(z1, labels, 10, True))


# ---------------------------------------------------------------------------
# 5. the mirrors on the new path reproduce the golden fixtures
# ---------------------------------------------------------------------------
def sparse(row, col, val, n):
    idx = torch.from_numpy(np.vstack([row, col]).astype(np.int64))
    return torch.sparse_coo_tensor(idx, torch.from_numpy(np.asarray(val, dtype=np.float32)), (n, n)).coalesce().cuda()


def close_flips(got, want, m, ties):
    """within 1.5 / m (one indicator on a float tie, as the Gram-path tests allow), or the number of exact-arithmetic
    ties of the fixture (oracle.similarity_near_ties) where it has more than one"""
    allowed = (max(1, ties) + 0.5) / m
    assert abs(float(got) - float(want)) <= allowed, (float(got), float(want), m, ties)


def mirror_keys(W, z, A, row, col, val, labels, tag=""):
    hm = W.homophily_metrics
    n = labels.shape[0]
    c = int(labels.max()) + 1
    oh = torch.eye(c)[torch.from_numpy(labels)]
    ties = O.similarity_near_ties(oh.numpy(), row, col, val, n, oh.numpy())
    for kw, key in (({"hard": None, "LP": 1}, "out_soft_las"), ({"hard": 1, "LP": 1}, "out_hard_las"),
                    ({"hard": None, "LP": 0}, "out_soft_las_lp0"), ({"hard": 1, "LP": 0}, "out_hard_las_lp0"),
                    ({"hard": None, "LP": 1, "ifsum": 0}, "out_soft_las_mean")):
        close_flips(hm.similarity(oh, A, oh, **kw), z[key + tag], n, ties)
    mask = torch.from_numpy(z[f"in_idx_train{tag}"])
    for kw, key in (({"hard": None, "LP": 1}, "out_soft_las_idx"), ({"hard": 1, "LP": 1}, "out_hard_las_idx")):
        close_flips(hm.similarity(oh, A, oh, idx_train=mask, **kw), z[key + tag], int(mask.sum()), ties)


@pytest.fixture
def new_path(W, monkeypatch):
    monkeypatch.setattr(W.graph, "GRAM_SIMILARITY_MAX_ROWS", 0)
    calls = []
    inner = W.graph.class_inner_sums
    monkeypatch.setattr(W.graph, "class_inner_sums", lambda *a, **k: calls.append(1) or inner(*a, **k))
    return calls


@pytest.mark.parametrize("name", GD.names("syn_") + GD.names("ec_") + ["cora", "ds_citeseer", "ds_cornell", "ds_texas",
                                                                       "ds_film", "ds_wisconsin"])
def test_mirror_golden_on_class_sums(W, new_path, name):
    z = GD.load(name)
    if "out_soft_las" not in z.files:
        pytest.skip("fixture without similarity outputs")
    n = int(z["in_n"])
    labels = z["in_labels"]
    ei = z["in_edge_index"].astype(np.int64)
    val = z["in_edge_values"] if name.startswith("ec_") else np.ones(ei.shape[1], np.float32)
    A = sparse(ei[0], ei[1], val, n)
    mirror_keys(W, z, A, ei[0], ei[1], val, labels)
    if name.startswith("syn_"):
        uf = W.util_funcs
        ones = np.ones(ei.shape[1], np.float32)
        for sym, fn, ofn in ((1, uf.sys_normalized_adjacency, O.sys_normalized_adjacency),
                             (0, uf.row_normalized_adjacency, O.row_normalized_adjacency)):
            sfx = f"__sym{sym}"
            An = uf.sparse_mx_to_torch_sparse_tensor(fn(A))
            r, c, v = ofn(ei[0], ei[1], ones, n)
            zz = {k.replace("_norm" + sfx, "") + "@": z[k] for k in z.files if k.endswith("_norm" + sfx)}
            mirror_keys(W, zz, An, r, c, v, labels, tag="@")
    assert new_path


@pytest.mark.parametrize("name", GD.names("plot_"))
def test_plot_mirror_golden_on_class_sums(W, new_path, name):
    hp = W.homophily_plot
    z = GD.load(name)
    n = int(z["in_n"])
    labels = torch.from_numpy(z["in_labels"])
    adj = GD.plot_flow_adjacency(z)
    c = int(labels.max()) + 1
    label = torch.eye(c)[labels]
    r, cc = np.nonzero(adj.numpy())
    ties = O.similarity_near_ties(label.numpy(), r, cc, adj.numpy()[r, cc], n, label.numpy())
    adj = adj.cuda()
    close_flips(hp.similarity(label, adj, label, NTK=None, hard=None, LP=1), z["out_soft_las"], n, ties)
    close_flips(hp.similarity(label, adj, label, NTK=None, hard=1, LP=1), z["out_hard_las"], n, ties)
    idx = torch.from_numpy(z["in_idx_train"])
    close_flips(hp.similarity(label, adj, label, NTK=None, hard=None, LP=1, idx_train=idx), z["out_soft_las_idx"],
                idx.shape[0], ties)
    assert len(new_path) == 3


# ---------------------------------------------------------------------------
# 6. a whole graph beyond the threshold, with the shipped threshold
# ---------------------------------------------------------------------------
def las_restated(w, labels, cnt, hard, is_sum):
    """las_score_kernel's decisions (LP = 1) on float32 w, op by op in float32 (classes summed in order)"""
    f = np.float32
    m, n_cls = w.shape
    if hard:
        return torch.from_numpy(w).argmax(1).numpy() == labels
    if is_sum:
        nnodes, degs = f(m), cnt[labels].astype(f)
    else:
        nnodes, degs = f(n_cls), f(1)
    tot = np.zeros(m, f)
    for c in range(n_cls):
        tot = tot + w[:, c]
    own = w[np.arange(m), labels]
    with np.errstate(all="ignore"):
        ratio = (own / degs) / ((tot - own) / (nnodes - degs))
    ratio[np.isnan(ratio)] = 0
    return ratio >= 1


def test_whole_graph_beyond_threshold(W):
    hm = W.homophily_metrics
    n, n_cls = 131_073, 5
    assert n > W.graph.GRAM_SIMILARITY_MAX_ROWS
    rng = np.random.default_rng(6)
    src = np.repeat(np.arange(n), 10)
    dst = rng.integers(0, n, src.shape[0])
    row, col, _ = O.coalesce(np.concatenate([src, dst]), np.concatenate([dst, src]), None, n)
    A = sparse(row, col, np.ones(row.shape[0], np.float32), n)
    labels = rng.integers(0, n_cls, n)
    oh = torch.eye(n_cls)[torch.from_numpy(labels)]
    # exact integer references: z = A Y (neighbour counts), s = Y^T z, W = z s^T
    y = np.eye(n_cls, dtype=np.int64)[labels]
    z = np.zeros((n, n_cls), np.int64)
    np.add.at(z, row, y[col])
    s = y.T @ z
    w_exact = z @ s.T
    cnt = y.sum(0)
    assert w_exact.max() < 2 ** 53
    zt = W.spmm(hm._as_graph(A), oh)
    assert np.array_equal(zt.cpu().numpy(), z.astype(np.float32))
    lab32 = torch.from_numpy(labels.astype(np.int32)).cuda()
    w_sum = W.graph.las_weights(zt, lab32, n_cls, is_mean=False).cpu().numpy()
    w_mean = W.graph.las_weights(zt, lab32, n_cls, is_mean=True).cpu().numpy()
    assert np.array_equal(w_sum, w_exact.astype(np.float32))
    assert np.array_equal(w_mean, (w_exact.astype(np.float64) / cnt).astype(np.float32))
    own = w_exact[np.arange(n), labels].astype(np.float64)
    tot = w_exact.sum(1).astype(np.float64)
    deg = cnt[labels].astype(np.float64)
    with np.errstate(all="ignore"):
        near = {1: np.abs((own / deg) / ((tot - own) / (n - deg)) - 1) <= 1e-6,
                0: np.abs((own / deg) / (((w_exact / cnt).sum(1) - own / deg) / (n_cls - 1)) - 1) <= 1e-6}
    torch.cuda.synchronize()
    for hard in (None, 1):
        for ifsum in (1, 0):
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            score = float(hm.similarity(oh, A, oh, hard=hard, LP=1, ifsum=ifsum))
            rise = torch.cuda.max_memory_allocated() - base
            assert rise < 2 ** 30, rise                       # the Gram would be 4 n^2 bytes = 64 GiB
            ok = las_restated(w_sum if ifsum == 1 else w_mean, labels, cnt, hard is not None, ifsum == 1)
            want = int(ok.sum())
            got = round(score * n)
            slack = 0 if hard is not None else int(near[ifsum].sum())
            assert abs(got - want) <= slack, (hard, ifsum, got, want, slack)
            assert score == float(np.float32(got / n))
            score_bf16 = float(hm.similarity(oh.bfloat16(), A, oh, hard=hard, LP=1, ifsum=ifsum))
            assert score_bf16 == score, (hard, ifsum)


# ---------------------------------------------------------------------------
# 7. the threshold
# ---------------------------------------------------------------------------
def test_threshold(W):
    G = W.graph
    lim = G.GRAM_SIMILARITY_MAX_ROWS
    assert lim == 65536
    gen = torch.Generator(device="cuda").manual_seed(7)
    z = torch.randn((lim + 1, 8), generator=gen, device="cuda")
    labels = torch.randint(0, 4, (lim + 1,), generator=gen, device="cuda").to(torch.int32)
    at = z[:lim]
    w = G.las_weights(at, labels, 4, is_mean=False)
    assert torch.equal(w, G.class_colsum(G.gram(at), labels, 4))
    del w
    torch.cuda.empty_cache()
    torch.cuda.synchronize()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    w = G.las_weights(z, labels, 4, is_mean=True)
    assert torch.cuda.max_memory_allocated() - base < 2 ** 30   # the Gram of 65,537 rows would be 17 GB
    assert torch.equal(w, G.class_inner_sums(z, labels, 4, is_mean=True))
