"""HBM-resident CSR graph + thin typed wrappers over the C ABI (include/wdgh_b200.h).

torch is used for device memory, streams and dtype plumbing only; every
arithmetic step on the path is a kernel of libwdgh_b200.so.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import NamedTuple

import numpy as np
import torch

from . import _lib
from ._lib import NORM_NONE, NORM_RW, NORM_RW_SUM, NORM_SYM, NORM_SYM_RAW, check, lib, ptr, stream_ptr

HEAVY_THRESHOLD = 512  # entries; longer rows are split into chunks of this many (degree binning)


class _HalfEntries(NamedTuple):
    code: int        # WDGH_DTYPE of an output of this type
    spmm: str        # the C-ABI entries that read features of this type as they are (fp32 accumulation)
    ranged: str
    pipeline: str


# The 16-bit feature types the aggregation reads without an fp32 copy.  Each writes float32, or its own type.
_HALF = {
    torch.bfloat16: _HalfEntries(_lib.DTYPE_BF16, "wdgh_spmm_csr_bf16", "wdgh_spmm_csr_ranged_bf16",
                                 "wdgh_pipeline_host_bf16"),
    torch.float16: _HalfEntries(_lib.DTYPE_F16, "wdgh_spmm_csr_f16", "wdgh_spmm_csr_ranged_f16",
                                "wdgh_pipeline_host_f16"),
}


def _dev():
    _lib.require_device()
    return torch.device("cuda", torch.cuda.current_device())


def _cuda(t, dtype=None):
    """Move to the current CUDA device (plumbing), contiguous, optional dtype."""
    if not isinstance(t, torch.Tensor):
        t = torch.as_tensor(np.asarray(t))
    if t.device.type != "cuda":
        t = t.to(_dev(), non_blocking=True)
    if dtype is not None and t.dtype != dtype:
        t = t.to(dtype)
    return t.contiguous()


class CSRGraph:
    """Adjacency in CSR (rowptr int64, col int32, optional float32 values), resident in HBM.

    Row-major order with sorted columns -- the order `A.coalesce().indices()` produces,
    which every reference metric starts from (utils/homophily_metrics.py:50,63,127,165).
    """

    def __init__(self, rowptr, col, val, n, threshold=HEAVY_THRESHOLD, row_offset=0, n_global=None):
        self.rowptr, self.col, self.val = rowptr, col, val
        self.n, self.nnz = int(n), int(col.shape[0])
        # a 1-D row shard holds rows [row_offset, row_offset + n) of an n_global x n_global matrix
        self.row_offset = int(row_offset)
        self.n_global = int(n_global) if n_global is not None else int(n)
        self.threshold = int(threshold)
        self.device = rowptr.device
        self.n_cols = self.n_global       # a rectangular row-scaled matrix (preprocess_features) overrides this
        self._plan = None
        self._rows = None
        self._dinv = {}
        self._counts = {}
        self._partial = {}

    # ---- constructors ----------------------------------------------------
    @classmethod
    def from_coo_indices(cls, indices, values, n, threshold=HEAVY_THRESHOLD):
        """indices: int64 [2, nnz], coalesced (row-major sorted, unique)."""
        dev = _dev()
        indices = _cuda(indices, torch.int64)
        nnz = int(indices.shape[1])
        rowptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
        col = torch.empty(nnz, dtype=torch.int32, device=dev)
        check(lib.wdgh_coo_to_csr(ptr(indices), nnz, n, ptr(rowptr), ptr(col), stream_ptr()), "wdgh_coo_to_csr")
        val = None if values is None else _cuda(values, torch.float32)
        g = cls(rowptr, col, val, n, threshold)
        g._indices = indices
        return g

    @classmethod
    def from_torch_sparse(cls, a, threshold=HEAVY_THRESHOLD, binary=False):
        """a: torch sparse COO tensor (any device).  Coalesced first if it is not (torch plumbing)."""
        if not a.is_sparse:
            raise TypeError("expected a torch sparse COO tensor")
        if a.device.type != "cuda":
            a = a.to(_dev())
        a = a.coalesce()
        vals = None if binary else a.values()
        return cls.from_coo_indices(a.indices(), vals, a.shape[0], threshold)

    @classmethod
    def from_scipy(cls, m, threshold=HEAVY_THRESHOLD, binary=False, rectangular=False):
        """scipy sparse matrix -> resident CSR.  `rectangular=True` admits an n x d matrix (a sparse feature matrix):
        such a container only supports the row scalings (`normalized(NORM_RW / NORM_RW_SUM)`) and the exports."""
        m = m.tocsr()
        if m.shape[0] != m.shape[1] and not rectangular:
            raise ValueError(f"adjacency must be square, got {m.shape}")
        m.sum_duplicates()
        m.sort_indices()
        dev = _dev()
        rowptr = torch.from_numpy(m.indptr.astype(np.int64)).to(dev)
        col = torch.from_numpy(m.indices.astype(np.int32)).to(dev)
        val = None if binary else torch.from_numpy(m.data.astype(np.float32)).to(dev)
        g = cls(rowptr, col, val, m.shape[0], threshold)
        g.n_cols = int(m.shape[1])
        return g

    @classmethod
    def from_csr(cls, rowptr, col, val, n, threshold=HEAVY_THRESHOLD):
        return cls(_cuda(rowptr, torch.int64), _cuda(col, torch.int32),
                   None if val is None else _cuda(val, torch.float32), n, threshold)

    # ---- derived data ----------------------------------------------------
    @property
    def plan(self):
        """(device plan tensor, host int64[4] ctypes array) -- built once per graph."""
        if self._plan is None:
            cap = 2 * self.nnz // self.threshold + 2
            words = _lib.PLAN_HEADER + 3 * cap
            plan = torch.empty(words, dtype=torch.int64, device=self.device)
            host = (C.c_int64 * 8)()
            check(lib.wdgh_plan_build(ptr(self.rowptr), self.n, self.nnz, self.threshold, ptr(plan), cap, host,
                                      stream_ptr()), "wdgh_plan_build")
            self._plan = (plan, host)
        return self._plan

    @property
    def n_chunks(self):
        return int(self.plan[1][1])

    @property
    def n_heavy(self):
        return int(self.plan[1][0])

    def rows(self):
        """int64 row id of every stored entry (COO view)."""
        if self._rows is None:
            r = torch.empty(self.nnz, dtype=torch.int64, device=self.device)
            check(lib.wdgh_csr_to_coo_rows(ptr(self.rowptr), self.n, self.nnz, ptr(r), stream_ptr()),
                  "wdgh_csr_to_coo_rows")
            self._rows = r
        return self._rows

    def indices(self):
        """torch-style int64 [2, nnz] index tensor."""
        return torch.stack([self.rows(), self.col.to(torch.int64)])

    def degree_scale(self, norm, self_loop, want64=False):
        """(dinv float32[n], dinv64 or None, deg_code uint8[n] or None) -- cached per (norm, self_loop)."""
        key = (norm, bool(self_loop), want64)
        if key not in self._dinv:
            dinv = torch.empty(self.n, dtype=torch.float32, device=self.device)
            d64 = torch.empty(self.n, dtype=torch.float64, device=self.device) if want64 else None
            code = torch.empty(self.n, dtype=torch.uint8, device=self.device) if self.val is None else None
            check(lib.wdgh_degree_scale(ptr(self.rowptr), ptr(self.val), self.n, norm, int(bool(self_loop)),
                                        ptr(dinv), ptr(d64), ptr(code), stream_ptr()), "wdgh_degree_scale")
            self._dinv[key] = (dinv, d64, code)
        return self._dinv[key]

    def with_self_loops(self):
        """CSR of A + I (diagonal merged or inserted), util_funcs.py:385,420."""
        dev = self.device
        n, nnz = self.n, self.nnz
        out_rowptr = torch.empty(n + 1, dtype=torch.int64, device=dev)
        out_col = torch.empty(nnz + n, dtype=torch.int32, device=dev)
        out_val = torch.empty(nnz + n, dtype=torch.float32, device=dev)
        scratch = torch.empty(n + 2 * ((n + 1023) // 1024) + 8, dtype=torch.int64, device=dev)
        check(lib.wdgh_add_self_loops(ptr(self.rowptr), ptr(self.col), ptr(self.val), n, ptr(out_rowptr),
                                      ptr(out_col), ptr(out_val), ptr(scratch), stream_ptr()), "wdgh_add_self_loops")
        new_nnz = int(out_rowptr[-1].item())
        return CSRGraph(out_rowptr, out_col[:new_nnz], out_val[:new_nnz], n, self.threshold)

    def normalized(self, norm):
        """Materialised D^-1/2 A D^-1/2 (SYM) or D^-1 A (RW) of THIS matrix (no self-loop added)."""
        if norm in (NORM_SYM, NORM_SYM_RAW) and self.n_cols != self.n:
            raise ValueError("a symmetric scaling needs a square matrix")
        d64 = self.degree_scale(norm, False, want64=True)[1]
        out = torch.empty(self.nnz, dtype=torch.float32, device=self.device)
        check(lib.wdgh_scale_values(ptr(self.rowptr), ptr(self.col), ptr(self.val), self.n, norm, ptr(d64), ptr(out),
                                    stream_ptr()), "wdgh_scale_values")
        g = CSRGraph(self.rowptr, self.col, out, self.n, self.threshold)
        g._plan, g._rows, g.n_cols = self._plan, self._rows, self.n_cols
        return g

    def to_torch_sparse(self):
        v = self.val if self.val is not None else torch.ones(self.nnz, dtype=torch.float32, device=self.device)
        return torch.sparse_coo_tensor(self.indices(), v, (self.n, self.n_cols), is_coalesced=True)

    def to_scipy(self):
        """Host copy as scipy CSR (float32 values) -- what the scipy-returning reference normalisers hand back."""
        import scipy.sparse as sp
        v = self.val if self.val is not None else torch.ones(self.nnz, dtype=torch.float32, device=self.device)
        return sp.csr_matrix((v.cpu().numpy(), self.col.cpu().numpy(), self.rowptr.cpu().numpy()),
                             shape=(self.n, self.n_cols))

    def todense(self):
        """numpy matrix like scipy's `.todense()` (full_load_data densifies the row-normalised features this way)."""
        return self.to_scipy().todense()


# ---------------------------------------------------------------------------
# A_hat X aggregation
# ---------------------------------------------------------------------------
def spmm(g: CSRGraph, x, norm=NORM_NONE, add_self_loop=False, out=None, dinv=None, deg_code=None, out_dtype=None):
    """y = norm(A [+I]) x on the GPU with fp32 accumulation (hm.py:192,199,234; util_funcs.py:383-390,418-426).

    A bfloat16 or float16 `x` is read as it is (no fp32 copy); its result is bit-identical to the one of `x.float()`.
    The result has the dtype of `out` if given, else `out_dtype`, else float32; a half output (round to nearest even;
    float16 overflows to +-inf) must have the dtype of the features.  Any other `x` dtype is converted to float32 first.
    For a row shard `x` (and `dinv`, the all-gathered degree scale) are global, the result is local."""
    half = _HALF.get(x.dtype) if isinstance(x, torch.Tensor) else None
    if out is not None:
        if out_dtype is not None and out_dtype != out.dtype:
            raise ValueError(f"out has dtype {out.dtype}, out_dtype asks for {out_dtype}")
        out_dtype = out.dtype
    out_dtype = torch.float32 if out_dtype is None else out_dtype
    if out_dtype not in ((torch.float32, x.dtype) if half else (torch.float32,)):
        raise ValueError(f"cannot write a {out_dtype} result from {x.dtype if half else 'float32'} features "
                         "(float32 output, or the half type of the features)")
    if half:
        # views with a unit column stride and whole rows apart (a column slab of a wider matrix) are read in place;
        # any other layout (transposed, broadcast rows) is copied like the float32 path does
        x = x.to(_dev(), non_blocking=True) if x.device.type != "cuda" else x
        if x.dim() == 2 and (x.stride(1) != 1 or x.stride(0) < x.shape[1]):
            x = x.new_empty(x.shape).copy_(x)   # (not .contiguous(): a [1, d] view with row stride 1 counts as such)
    else:
        x = _cuda(x, torch.float32)
    if x.dim() != 2 or x.shape[0] < g.n_global or (x.shape[0] != g.n_global and g.n_global == g.n):
        raise ValueError(f"features must be [n={g.n_global}, d], got {tuple(x.shape)}")
    d = int(x.shape[1])
    y = out if out is not None else torch.empty((g.n, d), dtype=out_dtype, device=g.device)
    if y.shape != (g.n, d) or y.stride(1) != 1:
        raise ValueError("out must be [n, d] with unit column stride (a column slab of a wider matrix is fine)")
    plan, plan_host = g.plan
    partial = _partial_scratch(g, d)
    if norm != NORM_NONE and dinv is None:
        if g.n_global != g.n:
            raise ValueError("a row shard needs the all-gathered degree scale (dinv=...)")
        dinv, _, deg_code = g.degree_scale(norm, add_self_loop)
    if half:
        y_dtype = half.code if out_dtype == x.dtype else _lib.DTYPE_F32
        check(getattr(lib, half.spmm)(ptr(g.rowptr), ptr(g.col), ptr(g.val), g.n, ptr(x), d, x.stride(0), ptr(y),
                                      y.stride(0), y_dtype, norm, int(bool(add_self_loop)), ptr(dinv), ptr(deg_code),
                                      ptr(plan), plan_host, ptr(partial), g.row_offset, stream_ptr()), half.spmm)
        return y
    check(lib.wdgh_spmm_csr(ptr(g.rowptr), ptr(g.col), ptr(g.val), g.n, ptr(x), d, x.stride(0), ptr(y), y.stride(0),
                            norm, int(bool(add_self_loop)), ptr(dinv), ptr(deg_code), ptr(plan), plan_host,
                            ptr(partial), g.row_offset, stream_ptr()), "wdgh_spmm_csr")
    return y


def _partial_scratch(g: CSRGraph, d: int):
    """Scratch for the rows whose sum is assembled from pieces: one partial row per chunk of a split row."""
    ldp = (d + 3) & ~3
    n_part = g.n_chunks * ldp
    partial = g._partial.get(n_part)
    if partial is None and n_part:
        partial = torch.empty(n_part, dtype=torch.float32, device=g.device)
        g._partial = {n_part: partial}
    return partial


def column_segments(g: CSRGraph, bounds):
    """int64 [len(bounds), n]: per row, the first stored entry whose column id is >= each bound."""
    b = _cuda(torch.as_tensor(bounds, dtype=torch.int64), torch.int64)
    seg = torch.empty((int(b.shape[0]), g.n), dtype=torch.int64, device=g.device)
    check(lib.wdgh_column_segments(ptr(g.rowptr), ptr(g.col), g.n, ptr(b), int(b.shape[0]), ptr(seg), stream_ptr()),
          "wdgh_column_segments")
    return seg


def heavy_flags(g: CSRGraph):
    """uint8 [n]: 1 for the rows the plan splits into chunks."""
    plan, plan_host = g.plan
    flags = torch.empty(g.n, dtype=torch.uint8, device=g.device)
    check(lib.wdgh_plan_heavy_flags(ptr(plan), plan_host, g.n, ptr(flags), stream_ptr()), "wdgh_plan_heavy_flags")
    return flags


def spmm_ranged(g: CSRGraph, range_begin, range_end, x, y, norm, add_self_loop, dinv, deg_code, skip_rows,
                accumulate, finalize, run_split_rows, x_row0=0, extra=None, extra_split=0, ctas_per_sm=0):
    """One phase of the aggregation: entries [range_begin[r], range_end[r]) of every row (see wdgh_spmm_csr_ranged).

    x_row0: global node id of x[0] -- lets a phase that only touches columns [x_row0, x_row0 + len(x)) read a
    feature shard in place (the kernel is handed the address x[0] would have at global id 0).
    extra: [parts, rows >= n, d] tensor of raw partial sums of the same rows (possibly peer-mapped), added to every row
    as it is aggregated; the split-row pass adds only the last `extra_split` parts.  y may be peer memory.
    ctas_per_sm: 0 = default grid, smaller = leave room for a kernel running concurrently on another stream.
    A bfloat16 or float16 `x` (float32 `y`, no `extra`, no `ctas_per_sm`) is read as it is; every phase sums in fp32
    and is bit-identical to the same call on `x.float()`."""
    d = int(x.shape[1])
    x_ptr = x.data_ptr() - int(x_row0) * x.stride(0) * x.element_size()
    plan, plan_host = g.plan
    partial = _partial_scratch(g, d)
    half = _HALF.get(x.dtype)
    if half:
        if extra is not None or ctas_per_sm:
            raise ValueError("extra partial sums and ctas_per_sm need float32 features")
        if y.dtype != torch.float32:
            raise ValueError(f"a phase writes float32 partial sums, got a {y.dtype} y")
        check(getattr(lib, half.ranged)(ptr(g.rowptr), ptr(range_begin), ptr(range_end), ptr(g.col), ptr(g.val),
                                        g.n, x_ptr, d, x.stride(0), ptr(y), y.stride(0), norm,
                                        int(bool(add_self_loop)), ptr(dinv), ptr(deg_code), ptr(skip_rows),
                                        int(bool(accumulate)), int(bool(finalize)), int(bool(run_split_rows)),
                                        ptr(plan), plan_host, ptr(partial), g.row_offset, stream_ptr()), half.ranged)
        return y
    n_extra = part_rows = ld_extra = 0
    if extra is not None:
        if extra.dim() != 3 or extra.shape[1] < g.n or extra.shape[2] != d or extra.stride(2) != 1:
            raise ValueError("extra partial sums must be a [parts, rows >= n, d] tensor")
        n_extra, ld_extra = int(extra.shape[0]), int(extra.stride(1))
        if n_extra > 1 and extra.stride(0) % ld_extra:
            raise ValueError("the parts of `extra` must be a whole number of rows apart")
        part_rows = int(extra.stride(0)) // ld_extra if n_extra > 1 else int(extra.shape[1])
    check(lib.wdgh_spmm_csr_ranged(ptr(g.rowptr), ptr(range_begin), ptr(range_end), ptr(g.col), ptr(g.val), g.n,
                                   x_ptr, d, x.stride(0), ptr(y), y.stride(0), norm, int(bool(add_self_loop)),
                                   ptr(dinv), ptr(deg_code), ptr(skip_rows), int(bool(accumulate)), int(bool(finalize)),
                                   int(bool(run_split_rows)), ptr(extra), n_extra, int(extra_split), part_rows,
                                   ld_extra, int(ctas_per_sm), ptr(plan), plan_host, ptr(partial), g.row_offset,
                                   stream_ptr()), "wdgh_spmm_csr_ranged")
    return y


# ---------------------------------------------------------------------------
# label statistics
# ---------------------------------------------------------------------------
@dataclass
class StructureCounts:
    """Exact integer statistics of one (graph, labels) pair (see include/wdgh_b200.h)."""
    n: int
    nnz: int
    num_classes: int
    match_all: int
    match_lab: int
    n_lab: int
    n_self: int
    n_empty: int
    nbins: int
    n_nodes_nsl: int
    class_count: np.ndarray   # [C] int64
    class_deg: np.ndarray     # [C] int64, sum of stored entries per row over the class
    hist: np.ndarray          # [C, C] int64
    node_sum: float           # sum_i f32(match_i)/f32(deg_i), diagonal excluded
    node_sum_self: float      # same with stored diagonal entries kept and counted as matches
    class_isolated: np.ndarray  # [C] int64, class-c nodes without an off-diagonal entry
    deg_nsl: torch.Tensor     # [n] int32 (device)
    match_nsl: torch.Tensor   # [n] int32 (device)


def pack_labels(labels):
    """int64 label tensor -> (int32 device tensor, max label)."""
    labels = _cuda(labels).reshape(-1)
    if labels.dtype != torch.int64:
        labels = labels.to(torch.int64)
    n = labels.shape[0]
    out = torch.empty(n, dtype=torch.int32, device=labels.device)
    mx = torch.empty(1, dtype=torch.int32, device=labels.device)
    check(lib.wdgh_pack_labels(ptr(labels), n, ptr(out), ptr(mx), stream_ptr()), "wdgh_pack_labels")
    return out, int(mx.item())


def _unpack_counts(n, nnz, c, counters, node_sum, deg, match):
    h = counters.cpu().numpy()
    H = _lib.SC_HEADER
    return StructureCounts(
        n=n, nnz=nnz, num_classes=c,
        match_all=int(h[_lib.SC_MATCH_ALL]), match_lab=int(h[_lib.SC_MATCH_LAB]), n_lab=int(h[_lib.SC_N_LAB]),
        n_self=int(h[_lib.SC_N_SELF]), n_empty=int(h[_lib.SC_N_EMPTY]), nbins=int(h[_lib.SC_NBINS]),
        n_nodes_nsl=int(h[_lib.SC_N_NODES_NSL]),
        class_count=h[H:H + c].copy(), class_deg=h[H + c:H + 2 * c].copy(),
        hist=h[H + 2 * c:H + 2 * c + c * c].reshape(c, c).copy(),
        node_sum=float(node_sum[0].item()), node_sum_self=float(node_sum[1].item()),
        class_isolated=h[H + 2 * c + c * c:H + 3 * c + c * c].copy(), deg_nsl=deg, match_nsl=match)


def structure_counts_raw(g: CSRGraph, labels32, num_classes, scratch=None):
    """Launch the label-statistics kernels; returns DEVICE tensors (counters, node_sum, deg, match), no sync.

    `labels32` is indexed by global node id (length n_global for a row shard)."""
    c = int(num_classes)
    dev = g.device
    n_labels = int(labels32.shape[0])
    if n_labels < g.row_offset + g.n:
        raise ValueError("labels must cover every (global) node id of the shard")
    if scratch is None:
        scratch = (torch.empty(_lib.sc_words(c), dtype=torch.int64, device=dev),
                   torch.empty(2, dtype=torch.float64, device=dev),
                   torch.empty(g.n, dtype=torch.int32, device=dev),
                   torch.empty(g.n, dtype=torch.int32, device=dev),
                   torch.empty(n_labels, dtype=torch.uint8, device=dev))
    counters, node_sum, deg, match, lab8 = scratch
    plan, plan_host = g.plan
    check(lib.wdgh_structure_counts(ptr(g.rowptr), ptr(g.col), g.n, g.nnz, ptr(labels32), c, ptr(plan), plan_host,
                                    ptr(counters), ptr(node_sum), ptr(deg), ptr(match), ptr(lab8), n_labels,
                                    g.row_offset, stream_ptr()), "wdgh_structure_counts")
    return counters, node_sum, deg, match, lab8


def structure_counts(g: CSRGraph, labels32, num_classes) -> StructureCounts:
    counters, node_sum, deg, match, _ = structure_counts_raw(g, labels32, num_classes)
    if int(counters[_lib.SC_N_MULTI_NEG].item()):
        # labels below -1 or >= num_classes: the 1-byte label copy folds them together with -1, redo on int32 labels
        c = int(num_classes)
        scratch = (counters, node_sum, deg, match, None)
        counters, node_sum, deg, match, _ = structure_counts_raw(g, labels32, c, scratch)
    return _unpack_counts(g.n, g.nnz, int(num_classes), counters, node_sum, deg, match)


def spmm_structure_fused(g: CSRGraph, x, labels32, num_classes, norm=NORM_SYM, add_self_loop=True, out=None,
                         dinv=None, deg_code=None, scratch=None, out_dtype=None):
    """One call: y = norm(A [+I]) x and the label statistics (device tensors, no sync).

    Returns (y, (counters, node_sum, deg, match, labels_u8)); binary adjacency only.  A bfloat16 or float16 `x` is read
    as it is (the half aggregation, then the label pass on the same stream); `out_dtype` / `out` as in `spmm`."""
    if g.val is not None:
        raise ValueError("the fused pass needs a binary adjacency (values = None)")
    if isinstance(x, torch.Tensor) and x.dtype in _HALF:
        y = spmm(g, x, norm, add_self_loop, out=out, dinv=dinv, deg_code=deg_code, out_dtype=out_dtype)
        return y, structure_counts_raw(g, labels32, num_classes, scratch)
    if out_dtype not in (None, torch.float32):
        raise ValueError(f"cannot write a {out_dtype} result from float32 features (a half output needs features of "
                         "that type)")
    x = _cuda(x, torch.float32)
    d = int(x.shape[1])
    c = int(num_classes)
    dev = g.device
    y = out if out is not None else torch.empty((g.n, d), dtype=torch.float32, device=dev)
    n_labels = int(labels32.shape[0])
    if scratch is None:
        scratch = (torch.empty(_lib.sc_words(c), dtype=torch.int64, device=dev),
                   torch.empty(2, dtype=torch.float64, device=dev),
                   torch.empty(g.n, dtype=torch.int32, device=dev),
                   torch.empty(g.n, dtype=torch.int32, device=dev),
                   torch.empty(n_labels, dtype=torch.uint8, device=dev))
    counters, node_sum, deg, match, lab8 = scratch
    plan, plan_host = g.plan
    partial = _partial_scratch(g, d)
    if norm != NORM_NONE and dinv is None:
        dinv, _, deg_code = g.degree_scale(norm, add_self_loop)
    check(lib.wdgh_spmm_structure_fused(ptr(g.rowptr), ptr(g.col), g.n, g.nnz, ptr(x), d, x.stride(0), ptr(y),
                                        y.stride(0), norm, int(bool(add_self_loop)), ptr(dinv), ptr(deg_code),
                                        ptr(labels32), c, ptr(plan), plan_host, ptr(partial), ptr(counters),
                                        ptr(node_sum), ptr(deg), ptr(match), ptr(lab8), n_labels, g.row_offset,
                                        stream_ptr()), "wdgh_spmm_structure_fused")
    return y, scratch


def pipeline_host(rowptr, col, x, labels, num_classes, norm=NORM_SYM, add_self_loop=True, y=None):
    """The whole pass from HOST memory (wdgh_pipeline_host / _bf16 / _f16): copies in, plan, degree scale,
    y = norm(A [+I]) x, label statistics, copies back.  Synchronous; device buffers are cached between calls.

    rowptr int64 [n+1], col int32 [nnz], labels int32 [n] and x [n, d] float32, bfloat16 or float16 (a half type
    halves the feature bytes on the link) are contiguous CPU tensors -- pinned memory lets the copies run at the full
    link rate.  y: None (counters only) or a contiguous [n, d] CPU tensor, filled in place: float32, or the half type of
    the features (the float32 result rounded to nearest even).  Returns (counters int64[sc_words(C)], node_sum
    float64[2]) as numpy arrays."""
    feature_dtypes = (torch.float32,) + tuple(_HALF)
    named = [("rowptr", rowptr, (torch.int64,)), ("col", col, (torch.int32,)), ("labels", labels, (torch.int32,)),
             ("x", x, feature_dtypes)]
    if y is not None:
        named.append(("y", y, feature_dtypes))
    for name, t, dtypes in named:
        if not isinstance(t, torch.Tensor) or t.device.type != "cpu":
            raise ValueError(f"{name} must be a CPU tensor")
        if not t.is_contiguous():
            raise ValueError(f"{name} must be contiguous")
        if t.dtype not in dtypes:
            raise ValueError(f"{name} must be {' or '.join(str(d) for d in dtypes)}, got {t.dtype}")
    if x.dim() != 2:
        raise ValueError(f"x must be [n, d], got {tuple(x.shape)}")
    n, d = int(x.shape[0]), int(x.shape[1])
    if rowptr.shape != (n + 1,) or col.dim() != 1 or labels.shape != (n,):
        raise ValueError(f"rowptr must be [{n + 1}], col 1-D and labels [{n}]; got {tuple(rowptr.shape)}, "
                         f"{tuple(col.shape)}, {tuple(labels.shape)}")
    half = _HALF.get(x.dtype)
    if y is not None:
        if y.shape != (n, d):
            raise ValueError(f"y must be [{n}, {d}], got {tuple(y.shape)}")
        if y.dtype not in (torch.float32, x.dtype):
            raise ValueError(f"a {y.dtype} y needs {y.dtype} features, got {x.dtype}")
    c = int(num_classes)
    counters = np.zeros(_lib.sc_words(c), np.int64)
    node_sum = np.zeros(2, np.float64)
    _lib.require_device()
    args = (ptr(rowptr), ptr(col), n, int(col.shape[0]), ptr(x), d, ptr(labels), c, norm, int(bool(add_self_loop)))
    if half:
        y_dtype = half.code if y is not None and y.dtype == x.dtype else _lib.DTYPE_F32
        check(getattr(lib, half.pipeline)(*args, ptr(y), y_dtype, counters.ctypes.data, node_sum.ctypes.data),
              half.pipeline)
    else:
        check(lib.wdgh_pipeline_host(*args, ptr(y), counters.ctypes.data, node_sum.ctypes.data), "wdgh_pipeline_host")
    return counters, node_sum


def structure_counts_coo(edge_index, n, labels32, num_classes, hist_includes_self_loops=False) -> StructureCounts:
    ei = _cuda(edge_index, torch.int64)
    c = int(num_classes)
    e = int(ei.shape[1])
    dev = ei.device
    counters = torch.empty(_lib.sc_words(c), dtype=torch.int64, device=dev)
    node_sum = torch.empty(2, dtype=torch.float64, device=dev)
    deg = torch.empty(n, dtype=torch.int32, device=dev)
    match = torch.empty(n, dtype=torch.int32, device=dev)
    check(lib.wdgh_structure_counts_coo(ptr(ei), e, n, ptr(labels32), c, ptr(counters), ptr(node_sum), ptr(deg),
                                        ptr(match), int(bool(hist_includes_self_loops)), stream_ptr()),
          "wdgh_structure_counts_coo")
    return _unpack_counts(n, e, c, counters, node_sum, deg, match)


def edge_label_rows_equal(g: CSRGraph, label_rows) -> int:
    lab = _cuda(label_rows, torch.float32)
    out = torch.empty(1, dtype=torch.int64, device=g.device)
    check(lib.wdgh_edge_label_rows_equal(ptr(g.rowptr), ptr(g.col), g.n, ptr(lab), lab.shape[1], lab.stride(0),
                                         ptr(out), stream_ptr()), "wdgh_edge_label_rows_equal")
    return int(out.item())


def edge_cosine(g: CSRGraph, x, entry_ids=None, raw_dot=False):
    """(sum of cosines -- or plain dot products --, entries counted): all off-diagonal positive entries,
    or the listed entry ids."""
    x = _cuda(x, torch.float32)
    s = torch.empty(1, dtype=torch.float64, device=g.device)
    cnt = torch.empty(1, dtype=torch.int64, device=g.device)
    if entry_ids is None:
        mode, ids, n_ids = 0, None, g.nnz
    else:
        ids = _cuda(entry_ids, torch.int64)
        mode, n_ids = 1, int(ids.shape[0])
    mode |= 2 if raw_dot else 0
    check(lib.wdgh_edge_cosine(ptr(g.rowptr), ptr(g.col), ptr(g.val), g.n, ptr(x), x.shape[1], x.stride(0), mode,
                               ptr(ids), n_ids, ptr(s), ptr(cnt), stream_ptr()), "wdgh_edge_cosine")
    return float(s.item()), int(cnt.item())


# ---------------------------------------------------------------------------
# dense contractions
# ---------------------------------------------------------------------------
GRAM_SIMT, GRAM_TC, GRAM_TC_FAITHFUL = 0, 1, 2   # include/wdgh_b200.h
USE_TENSOR_CORES = True  # tcgen05 / TMEM Gram (csrc/gram_tc.cu); False selects the SIMT fp32 cross-check kernel
# The KR metric feeds its Gram to np.linalg.pinv(rcond=1e-15): the matrix is rank-deficient (rank <= d), so rounding
# noise of the Gram is amplified into the predictions.  KR therefore uses the fp32-faithful tensor-core mode (every
# k-block drained from TMEM and added in fp32 registers); False falls back to the SIMT fp32-FMA kernel.
KR_USE_TENSOR_CORES = True


def gather_rows(x, ids):
    x = _cuda(x, torch.float32)
    ids = _cuda(ids, torch.int64)
    m, d = int(ids.shape[0]), int(x.shape[1])
    out = torch.empty((m, d), dtype=torch.float32, device=x.device)
    check(lib.wdgh_gather_rows(ptr(x), d, x.stride(0), ptr(ids), m, ptr(out), d, stream_ptr()), "wdgh_gather_rows")
    return out


def gram(z, use_tensor_cores=None, faithful=False):
    """g = z z^T (float32).  faithful=True: fp32-level accumulation on the tensor cores (KR path)."""
    z = _cuda(z, torch.float32)
    m, d = int(z.shape[0]), int(z.shape[1])
    g = torch.empty((m, m), dtype=torch.float32, device=z.device)
    tc = USE_TENSOR_CORES if use_tensor_cores is None else use_tensor_cores
    mode = (GRAM_TC_FAITHFUL if faithful else GRAM_TC) if tc else GRAM_SIMT
    ws = None
    if tc:
        ws = torch.empty(int(lib.wdgh_gram_workspace_floats(m, d)), dtype=torch.float32, device=z.device)
    check(lib.wdgh_gram(ptr(z), m, d, z.stride(0), ptr(g), m, mode, ptr(ws), stream_ptr()), "wdgh_gram")
    return g


def class_colsum(gm, labels32, num_classes, is_mean=False):
    m = int(gm.shape[0])
    w = torch.empty((m, num_classes), dtype=torch.float32, device=gm.device)
    check(lib.wdgh_class_colsum(ptr(gm), m, gm.stride(0), ptr(labels32), num_classes, int(bool(is_mean)), ptr(w),
                                stream_ptr()), "wdgh_class_colsum")
    return w


def class_inner_sums(z, labels32, num_classes, is_mean=False):
    """w[m, C]: sum (or mean) over the rows j of class c of <z_i, z_j>, computed as <z_i, s_c> with fp64 class sums
    s_c (two passes over z, no m x m Gram; include/wdgh_b200.h wdgh_class_inner_sums).  A float32 view with unit
    column stride (a row gather or a column slab of a wider matrix) is read in place."""
    if not (isinstance(z, torch.Tensor) and z.device.type == "cuda" and z.dtype == torch.float32 and z.dim() == 2
            and z.stride(1) == 1 and z.stride(0) >= z.shape[1]):
        z = _cuda(z, torch.float32)
    m, d, c = int(z.shape[0]), int(z.shape[1]), int(num_classes)
    if labels32.shape[0] < m:
        raise ValueError(f"labels must cover the {m} rows of z, got {labels32.shape[0]}")
    w = torch.empty((m, c), dtype=torch.float32, device=z.device)
    words = int(lib.wdgh_class_inner_workspace_doubles(m, d, c))
    if words < 0:
        raise ValueError(f"bad class-sum shape m={m} d={d} C={c}")
    ws = torch.empty(max(1, words), dtype=torch.float64, device=z.device)
    check(lib.wdgh_class_inner_sums(ptr(z), m, d, max(1, z.stride(0)), ptr(labels32), c, int(bool(is_mean)), ptr(ws),
                                    ptr(w), stream_ptr()), "wdgh_class_inner_sums")
    return w


# Above this many rows las_weights takes the Gram-free class sums: the Gram is 4 m^2 bytes (17 GB at 65,536 rows).
# Up to it the Gram path is kept, so every result of earlier releases at those sizes stays bit-identical.
GRAM_SIMILARITY_MAX_ROWS = 65536


def las_weights(z, labels32, num_classes, is_mean):
    """The class table w[m, C] of the aggregation similarity (hm.py:199-206): class sums (or means) of the rows of
    z z^T.  Up to GRAM_SIMILARITY_MAX_ROWS rows from the Gram (class_colsum(gram(z))), above from class_inner_sums."""
    if int(z.shape[0]) <= GRAM_SIMILARITY_MAX_ROWS:
        return class_colsum(gram(z), labels32, num_classes, is_mean=is_mean)
    return class_inner_sums(z, labels32, num_classes, is_mean=is_mean)


def las_count(w, labels32, label_rows, hard, lp, is_sum) -> int:
    m, c = int(w.shape[0]), int(w.shape[1])
    label_rows = _cuda(label_rows, torch.float32)
    scratch = torch.empty(c, dtype=torch.float32, device=w.device)
    cnt = torch.empty(1, dtype=torch.int64, device=w.device)
    check(lib.wdgh_las_score(ptr(w), ptr(labels32), ptr(label_rows), m, c, int(bool(hard)), int(lp), int(bool(is_sum)),
                             ptr(scratch), ptr(cnt), stream_ptr()), "wdgh_las_score")
    return int(cnt.item())


def gntk_transform_(gm, n_layers):
    m = int(gm.shape[0])
    scratch = torch.empty(m, dtype=torch.float32, device=gm.device)
    check(lib.wdgh_gntk_transform(ptr(gm), m, gm.stride(0), int(n_layers), ptr(scratch), stream_ptr()),
          "wdgh_gntk_transform")
    return gm


def ntk_clamp_transform_(gm):
    check(lib.wdgh_ntk_clamp_transform(ptr(gm), int(gm.shape[0]), gm.stride(0), stream_ptr()), "wdgh_ntk_clamp_transform")
    return gm


def argmax_rows(m):
    m = _cuda(m, torch.float32)
    out = torch.empty(m.shape[0], dtype=torch.int32, device=m.device)
    check(lib.wdgh_argmax_rows(ptr(m), m.shape[0], m.shape[1], m.stride(0), ptr(out), stream_ptr()),
          "wdgh_argmax_rows")
    return out


def normalize_dense(x, symmetric=0):
    x = _cuda(x, torch.float32)
    n, d = int(x.shape[0]), int(x.shape[1])
    out = torch.empty((n, d), dtype=torch.float32, device=x.device)
    scratch = torch.empty(n, dtype=torch.float32, device=x.device)
    check(lib.wdgh_normalize_dense(ptr(x), n, d, x.stride(0), int(symmetric), ptr(scratch), ptr(out), d,
                                   stream_ptr()), "wdgh_normalize_dense")
    return out
