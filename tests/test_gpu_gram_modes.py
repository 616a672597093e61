"""The three Gram modes (csrc/dense.cu, csrc/gram_tc.cu) and the similarity helpers after them, against references that
are exact where the arithmetic allows it and discriminating where it does not.

* Integer inputs in [-8, 8] are exact in TF32 (lo = 0), every product is exact and every partial sum stays below 2^24:
  all three modes must equal the float64 product bit for bit, at the tile-schedule boundaries and across the SIMT
  routing boundary d = 32 -> 33.
* Accuracy: inputs on which every TF32 rounding errs the same way, bounded per mode from the kernel's arithmetic; a
  kernel without one of the two cross products of 3xTF32 is ~4x past the fast-mode bound.
* class_colsum / las_count on integer values (every sum exact, IEEE division), gntk_transform_ bit-equal to a float32
  op-by-op restatement with a correctly rounded acos.
"""
import math

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


MODES = {"simt": 0, "tc": 1, "tc_faithful": 2}   # GRAM_SIMT, GRAM_TC, GRAM_TC_FAITHFUL (include/wdgh_b200.h)


def gram_abi(W, z, m, d, ldz, g, ldg, mode):
    """wdgh_gram on raw buffers: z [m, ldz] and g [m, ldg] are device tensors, only z[:, :d] / g[:, :m] are used"""
    lib = W._lib.lib
    ws = torch.empty(max(1, int(lib.wdgh_gram_workspace_floats(m, d))), dtype=torch.float32, device="cuda")
    rc = lib.wdgh_gram(z.data_ptr(), m, d, ldz, g.data_ptr(), ldg, mode, ws.data_ptr(), W._lib.stream_ptr())
    assert rc == 0, W._lib.last_error()
    torch.cuda.synchronize()


def gram(W, z, mode):
    m, d = z.shape
    g = torch.empty((m, m), dtype=torch.float32, device="cuda")
    gram_abi(W, z, m, d, d, g, m, mode)
    return g


def int_matrix(m, d, seed):
    gen = torch.Generator(device="cuda").manual_seed(seed)
    return torch.randint(-8, 9, (m, d), generator=gen, device="cuda").to(torch.float32)


# ---------------------------------------------------------------------------
# 1. bit-exact on integer inputs
# ---------------------------------------------------------------------------
M_EDGES = [1, 127, 128, 129, 255, 256, 257, 383, 384, 385, 511, 512, 513]


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("d", [32, 33, 64, 65, 96, 97, 160, 300])
def test_integer_inputs_exact(W, mode, d):
    """|partial sums| <= 64 d < 2^24: the float64 product is representable and every order of summation gives it"""
    for m in M_EDGES:
        z = int_matrix(m, d, seed=m * 1000 + d)
        g = gram(W, z, MODES[mode])
        ref = (z.double() @ z.double().T).float()
        assert torch.equal(g, ref), (mode, m, d, (g - ref).abs().max().item())
        assert torch.equal(g, g.T), (mode, m, d)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("d", [96, 300])
def test_integer_inputs_exact_more_tiles_than_ctas(W, mode, d):
    """m = 2900: 155 live 128 x 256 tiles on 148 SMs, so some CTAs take a second tile.  d = 96 has 3 k-blocks (3 chunks
    in the faithful mode), d = 300 has 10 (3 chunks of 4 in the fast mode): an odd chunk count per tile carries the
    ping-pong accumulator parity from one tile into the next."""
    m = 2900
    z = int_matrix(m, d, seed=d)
    g = gram(W, z, MODES[mode])
    ref = (z.double() @ z.double().T).float()
    assert torch.equal(g, ref), (mode, d, int((g != ref).sum()))
    assert torch.equal(g, g.T)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("m,d,ldz", [(100, 20, 23), (129, 33, 40), (257, 97, 100), (513, 300, 301)])
def test_strided_operands(W, mode, m, d, ldz):
    """ldz > d with NaN in the unused columns of z (never read), ldg = m + 1 (rows not 16-byte aligned: the scalar
    store path) with NaN in the padding column of g (never written)"""
    zbuf = torch.full((m, ldz), float("nan"), device="cuda")
    z = int_matrix(m, d, seed=ldz)
    zbuf[:, :d] = z
    ldg = m + 1
    gbuf = torch.full((m, ldg), float("nan"), device="cuda")
    gram_abi(W, zbuf, m, d, ldz, gbuf, ldg, MODES[mode])
    ref = (z.double() @ z.double().T).float()
    assert torch.equal(gbuf[:, :m], ref), (mode, m, d)
    assert torch.isnan(gbuf[:, m]).all()


# ---------------------------------------------------------------------------
# 2. accuracy that tells 3xTF32 from a kernel missing one of its cross products
# ---------------------------------------------------------------------------
U = 2.0 ** -24           # fp32 unit roundoff
FRAC = 4014 / 8192       # 0.48999...: a multiple of 2^-13, so z below has at most 24 significant bits


def tf32_skewed(m, d, seed):
    """z = (1 + (k + FRAC) 2^-10) 2^e, k in [0, 1024), e in [-2, 2]: every element sits 0.49 TF32 ulp above a TF32
    value, so hi = (1 + k 2^-10) 2^e (rounded down), lo = FRAC 2^-10 2^e exactly, and all errors have one sign."""
    rng = np.random.default_rng(seed)
    k = rng.integers(0, 1024, (m, d))
    e = rng.integers(-2, 3, (m, d)).astype(np.float64)
    hi = (1 + k * 2.0 ** -10) * 2.0 ** e
    lo = FRAC * 2.0 ** -10 * 2.0 ** e
    z = (hi + lo).astype(np.float32)
    assert np.array_equal(z.astype(np.float64), hi + lo)
    return z, hi, lo


def bound(mode, d):
    """Largest e_ij / s_ij the mode may show, s_ij = sum_k |z_ik z_jk|.

    SIMT: one fp32 FMA chain per element, |e| <= gamma_d s with gamma_d = d u / (1 - d u), u = 2^-24.

    Tensor cores (3xTF32).  z = hi + lo + r with hi = RN_tf32(z), lo = RN_tf32(z - hi): a TF32 significand has 11
    bits, so |z - hi| <= 2^-11 |z|, |lo| <= 2^-11 |z| (1 + 2^-11) and the split residual |r| <= 2^-22 |z|.  The kernel
    sums hi hi + hi lo + lo hi; what it leaves out of z_i z_j is lo_i lo_j + (hi_i + lo_i) r_j + r_i z_j,
    in all <= 3 (1 + 2^-10) 2^-22 |z_i z_j|.

    Each tcgen05.mma (K = 8) adds 8 exact TF32 products into the fp32 TMEM accumulator.  The model bounded here: the
    9 addends are aligned to the largest one (magnitude M) and truncated at fp32 precision, then the sum is truncated
    to fp32 -- at most 9 * 2^-23 M + 2^-23 |sum| <= 10 * 2^-23 s_chunk per instruction, where s_chunk is the sum of
    |products| the chunk adds (M and |sum| cannot exceed it).  A chunk is `chunk` k-blocks of 12 instructions (4 k-steps
    x 3 products): 12 in the fp32-faithful mode (chunk = 1), 48 in the fast mode (chunk = 4), so a chunk errs by at most
    10 * I * 2^-23 s_chunk with I = 12 or 48, and the chunks together by 10 * I * 2^-23 (1 + 2^-10) s (the lo terms add
    2^-10 to s).  The drained chunks are added in fp32 registers with round to nearest: n_chunks * u s more.

    A kernel without lo_a hi_b (or hi_a lo_b) misses sum_k lo_ik hi_jk >= 0.245 * 2^-10 (1 - 2^-10) s ~ 2.39e-4 s on
    the inputs of `tf32_skewed` (lo / z >= FRAC 2^-10 / 2), ~4x the fast-mode bound at d = 1433 (5.9e-5) and ~13x the
    faithful one (1.8e-5)."""
    if mode == "simt":
        return d * U / (1 - d * U)
    chunk = 1 if mode == "tc_faithful" else 4
    k_blocks = -(-d // 32)
    n_chunks = -(-k_blocks // chunk)
    split = 3 * (1 + 2.0 ** -10) * 2.0 ** -22
    tmem = 10 * (12 * chunk) * 2.0 ** -23 * (1 + 2.0 ** -10)
    return split + tmem + n_chunks * U


@pytest.mark.parametrize("m,d", [(1000, 1433), (300, 96)])
def test_accuracy_bound_per_mode(W, m, d):
    z, hi, lo = tf32_skewed(m, d, seed=d)
    z64 = z.astype(np.float64)
    s = z64 @ z64.T                                     # all entries positive: s_ij = sum_k |z_ik z_jk| = G_ij
    # the inputs discriminate: dropping either cross product errs by far more than the fast-mode bound
    missing = (lo @ hi.T) / s
    assert missing.min() > 3 * bound("tc", d), (missing.min(), bound("tc", d))
    zt = torch.from_numpy(z).cuda()
    worst = {}
    for mode in MODES:
        g = gram(W, zt, MODES[mode]).cpu().numpy().astype(np.float64)
        worst[mode] = float((np.abs(g - s) / s).max())
        print(f"gram accuracy m={m} d={d} {mode}: max e/s = {worst[mode]:.3e}, bound {bound(mode, d):.3e}")
    assert all(worst[mode] <= bound(mode, d) for mode in MODES), worst


# ---------------------------------------------------------------------------
# 3. class_colsum: integer G, every sum exact
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("m", [1, 33, 300])
@pytest.mark.parametrize("n_cls", [1, 9, 40])
def test_class_colsum_exact(W, m, n_cls):
    """9 and 40 classes: more classes than the 8 warps of a CTA.  One class id below the largest is absent: its sum is
    0, its mean 0/0 = NaN as torch.mean of an empty selection gives.  G is a column slab of a wider buffer (ldg > m)."""
    rng = np.random.default_rng(m * 100 + n_cls)
    g = rng.integers(-50, 51, (m, m)).astype(np.float32)
    labels = rng.integers(0, n_cls, m).astype(np.int32)
    if n_cls > 1:
        labels[labels == n_cls // 2] = n_cls - 1        # absent class
    buf = torch.full((m, m + 5), float("nan"), device="cuda")
    buf[:, :m] = torch.from_numpy(g).cuda()
    lab32 = torch.from_numpy(labels).cuda()
    sums = np.zeros((m, n_cls), np.float64)
    for c in range(n_cls):
        sums[:, c] = g[:, labels == c].astype(np.float64).sum(1)
    cnt = np.bincount(labels, minlength=n_cls).astype(np.float32)
    with np.errstate(invalid="ignore", divide="ignore"):
        means = sums.astype(np.float32) / cnt            # IEEE float32 division, 0/0 = NaN
    got_sum = W.graph.class_colsum(buf[:, :m], lab32, n_cls, is_mean=False).cpu().numpy()
    got_mean = W.graph.class_colsum(buf[:, :m], lab32, n_cls, is_mean=True).cpu().numpy()
    assert np.array_equal(got_sum, sums.astype(np.float32))
    assert np.array_equal(got_mean, means, equal_nan=True)
    if n_cls > 1:
        assert np.isnan(got_mean[:, n_cls // 2]).all()
        ref = torch.from_numpy(g)[:, torch.from_numpy(labels) == n_cls // 2].mean(1)   # hm.py:205
        assert torch.isnan(ref).all()


# ---------------------------------------------------------------------------
# 4. las_count: every branch, exact ties
# ---------------------------------------------------------------------------
def las_reference(w, labels, lab, hard, lp, is_sum):
    """hm.py:207-229 in numpy float32.  w is integer-valued (or NaN), so every sum is exact in any order."""
    m, n_cls = w.shape
    f = np.float32
    with np.errstate(all="ignore"):
        if not hard:
            if lp == 1:
                if is_sum:
                    nnodes, degs = f(m), (lab @ lab.T).sum(1).astype(f)               # :210
                else:
                    nnodes, degs = f(n_cls), f(1)
                own = w[np.arange(m), labels]
                ratio = (own / degs) / ((w.sum(1) - own) / (nnodes - degs))          # :216-218
                ratio[np.isnan(ratio)] = 0
                ok = ratio >= 1
            else:
                ok = ((w - w * lab).sum(1) <= 0) & ((w * lab).sum(1) >= 0)
        elif lp == 1:
            ok = torch.from_numpy(w).argmax(1).numpy() == labels                      # :226, NaN counts as maximum
        else:
            ok = ((w - w * lab).max(1) <= 0) & ((w * lab).sum(1) >= 0)
    return int(ok.sum())


def las_inputs(n_cls, seed):
    rng = np.random.default_rng(seed)
    m = 96
    w = rng.integers(-20, 21, (m, n_cls)).astype(np.float32)
    labels = rng.integers(0, n_cls, m).astype(np.int64)
    rows = iter(range(m))
    special = {}
    if n_cls >= 3:
        for y in (0, 2):                       # all columns equal: mean ratio exactly 1; argmax = column 0
            i = next(rows)
            w[i], labels[i] = 5, y
            special.setdefault("flat", []).append(i)
        for c2, y in ((1, 2), (2, 1)):         # two equal maxima: the first one wins
            i = next(rows)
            w[i], labels[i] = rng.integers(-5, 5, n_cls), y
            w[i, [c2, y]] = 50
            special.setdefault("tie", []).append(i)
        for y in (n_cls - 1, 1):               # a NaN column wins the argmax, poisons every sum
            i = next(rows)
            w[i, n_cls - 1], labels[i] = np.nan, y
        i = next(rows)                         # off == 0 and on == 0 with nonzero entries
        w[i], labels[i] = 0, 2
        w[i, 0], w[i, 1] = 3, -3
        special["zero_sums"] = [i]
        i = next(rows)                         # an all-zero row
        w[i], labels[i] = 0, 0
        special["zero_sums"].append(i)
    sizes = np.bincount(labels, minlength=n_cls)
    i = next(rows)                             # w proportional to the class sizes: sum ratio exactly 1
    w[i] = 2 * sizes
    special["proportional"] = [i]
    lab = np.eye(n_cls, dtype=np.float32)[labels]
    return w, labels, lab, special


@pytest.mark.parametrize("n_cls", [1, 9])
@pytest.mark.parametrize("hard", [False, True])
@pytest.mark.parametrize("lp", [1, 2])
@pytest.mark.parametrize("is_sum", [True, False])
def test_las_count_branches(W, n_cls, hard, lp, is_sum):
    w, labels, lab, special = las_inputs(n_cls, seed=n_cls)
    if n_cls >= 3:   # the ties are ties in float32, as constructed
        f = np.float32
        i = special["proportional"][0]
        y = labels[i]
        deg = f((labels == y).sum())
        assert (w[i, y] / deg) / ((w[i].sum() - w[i, y]) / (f(len(labels)) - deg)) == 1
        i = special["flat"][0]
        assert (w[i, labels[i]] / f(1)) / ((w[i].sum() - w[i, labels[i]]) / f(n_cls - 1)) == 1
    want = las_reference(w, labels, lab, hard, lp, is_sum)
    got = W.graph.las_count(torch.from_numpy(w).cuda(), torch.from_numpy(labels.astype(np.int32)).cuda(),
                            torch.from_numpy(lab).cuda(), hard, lp, is_sum)
    assert got == want, (got, want)


# ---------------------------------------------------------------------------
# 5. gntk_transform_: torch's float32 rounding sequence, sqrt and acos correctly rounded
# ---------------------------------------------------------------------------
def cr_sqrt(x):
    with np.errstate(invalid="ignore"):    # float64, then float32: correctly rounded for sqrt
        return np.sqrt(x.astype(np.float64)).astype(np.float32)


def cr_acos(x):
    with np.errstate(invalid="ignore"):
        return np.arccos(x.astype(np.float64)).astype(np.float32)


def torch_op(fn):
    return lambda x: fn(torch.from_numpy(x)).numpy()


def gntk_reference(g, n_layers, sqrt=cr_sqrt, acos=cr_acos, calls=None):
    """homophily_metrics.py:236-244 (oracle._arccos_kernel, then / 2) op by op in numpy float32.  Every +, -, *, / is
    an IEEE float32 operation as in torch; `sqrt` / `acos` are the two library functions (correctly rounded by
    default).  `calls` collects (name, argument) of each library call, with the shapes torch sees."""
    f = np.float32
    g = g.astype(f)
    if n_layers != 1:
        return g / f(2)
    calls = [] if calls is None else calls
    diag = np.ascontiguousarray(np.diag(g))
    calls.append(("sqrt", diag))
    dsq = sqrt(diag)
    raw = dsq[:, None] * dsq[None, :]
    eps = f(1e-8)
    norm = (raw > eps).astype(f) * raw + eps * (raw <= eps).astype(f)
    with np.errstate(invalid="ignore"):
        x = g / norm
        diff = norm * norm - g * g
        calls += [("acos", x), ("sqrt", diff)]
        ac = acos(x)
        root = sqrt(diff)
    ac[np.isnan(ac)] = 0
    root[np.isnan(root)] = 0
    k = f(1 / math.pi) * (g * (f(math.pi) - ac) + root)
    return k / f(2)


def ulps(a, b):
    def key(x):
        i = x.astype(np.float32).view(np.int32).astype(np.int64)
        return np.where(i < 0, -(i & 0x7FFFFFFF), i)
    return np.abs(key(a) - key(b))


def gntk_inputs(kind):
    rng = np.random.default_rng(7)
    if kind == "integer":
        z = rng.integers(-3, 4, (60, 6)).astype(np.float64)
        z[2], z[3] = [3, 4, 0, 0, 0, 0], [6, 8, 0, 0, 0, 0]     # |z| = 5, 10: g / norm = 1 exactly
        z[5] = -z[0]                                         # anti-parallel: acos near pi
    else:
        z = rng.standard_normal((200, 64))
    z[1] = 2 * z[0]                                          # parallel rows: root = sqrt(~0)
    z[4] = 0                                                 # zero row: norm = eps
    return (z @ z.T).astype(np.float32)


@pytest.mark.parametrize("n_layers", [0, 1])
@pytest.mark.parametrize("kind", ["integer", "float"])
def test_gntk_transform_rounding(W, kind, n_layers):
    """The kernel equals the float32 restatement with correctly rounded sqrt / acos bit for bit.  Against torch the
    comparison is per library call: the same restatement fed torch's own sqrt / acos reproduces torch's result bit for
    bit (the sequence of roundings is torch's), and torch's sqrt / acos are within 1 ulp of the correctly rounded
    values on every argument they get here.  The result itself has no ulp bound against torch: near (anti-)parallel
    rows x (pi - acos) + root cancels, so a 1-ulp acos difference moves K by many ulps."""
    g = gntk_inputs(kind)
    m = g.shape[0]
    buf = torch.full((m, m + 3), float("nan"), device="cuda")
    buf[:, :m] = torch.from_numpy(g).cuda()
    W.graph.gntk_transform_(buf[:, :m], n_layers)
    out = buf.cpu().numpy()
    assert np.isnan(out[:, m:]).all()
    got = out[:, :m]
    calls = []
    want = gntk_reference(g, n_layers, calls=calls)
    assert np.array_equal(got, want), (kind, n_layers, np.argwhere(got != want)[:5])
    ref = (O._arccos_kernel(torch.from_numpy(g), n_layers) / 2).numpy()
    assert np.array_equal(gntk_reference(g, n_layers, torch_op(torch.sqrt), torch_op(torch.acos)), ref)
    for name, x in calls:
        fn_torch, fn_cr = {"sqrt": (torch.sqrt, cr_sqrt), "acos": (torch.acos, cr_acos)}[name]
        a, b = torch_op(fn_torch)(x), fn_cr(x)
        assert np.array_equal(np.isnan(a), np.isnan(b)), name
        ok = ~np.isnan(b)
        assert ulps(a[ok], b[ok]).max(initial=0) <= 1, (name, ulps(a[ok], b[ok]).max())
