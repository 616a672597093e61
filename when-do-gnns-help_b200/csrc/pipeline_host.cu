// End-to-end entry with HOST buffers: what a reference user calls when the graph lives in host
// memory (homophily_tests.py moves everything with `.to(device)` first).  H2D copies, plan,
// normaliser, A_hat X, label statistics and the D2H result copies are all inside the caller's
// timed region (bench.py "e2e").
//
// The pass is PCIe-bound (the feature matrix is 85% of the bytes), so the entry is a pipeline on three streams.  The CSR
// and the labels go first on a copy stream, and the feature matrix follows on the same stream as KC = d / W column
// blocks of width W, each in R row chunks.  Meanwhile the compute stream builds the plan and runs the label pass, then
// aggregates every chunk as it arrives: with R > 1 one phase per chunk (wdgh_spmm_csr_ranged: the entries whose source
// node lies in the chunk, y +=, self loop + scale with the last chunk), with R = 1 one full launch.  When Y comes back,
// each Y block leaves on the third stream as soon as its last phase is done.  So only the last chunk's phase is exposed
// after the H2D copies end.  schedule() picks (W, KC, R):
//
//   case                                                  W    KC       R
//   Y wanted, d % 64 == 0 and 2 <= d / 64 <= 64           64   d / 64   4, halved while KC * R > 64
//   otherwise, d % 4 == 0 and d in {32, 64} or d >= 128   d    1        16   (row blocks)
//   otherwise (widths the ranged entries do not take)     d    1        1    (one copy, one launch)
//
// Why column blocks when Y comes back: with row blocks the D2H copy of Y would follow the whole H2D stream -- Y depends
// on every feature ROW block -- and the step would cost H2D + D2H back to back (1070 ms for 30.1 + 25.6 GB).  PCIe is
// full duplex, and a COLUMN block of Y needs only the same column block of X, so the feature matrix is split by columns
// instead: pitched copies (cudaMemcpy2DAsync), aggregation of a column block on strided views (ldx = ldy = d;
// bit-identical to the one-launch result, tools/colblock_probe.py) phased by arriving row chunk, so that only the last
// chunk's phase separates the end of a block's H2D copy from the start of its D2H copy, and the D2H copy of block k runs
// under the H2D copy of block k + 1.
//
// bfloat16 and float16 features (wdgh_pipeline_host_bf16 / _f16) take the same body with their aggregation entries
// (Elem below): half the bytes of X on the link, fp32 phases (a phase is bit-identical to the fp32 phase on the upcast
// matrix).  Y is always aggregated in fp32 into the device Y buffer; for a half Y (the type of X) the last phase of a
// block is followed by a rounding pass into a 2-byte staging buffer, which the D2H copy reads -- so a half Y is exactly
// the rounding of the fp32 Y of the same schedule, and the schedule depends neither on the type of X nor on that of Y.
#include <algorithm>
#include <mutex>

#include "internal.cuh"

namespace wdgh {

// Block chunks (KC * R) of one call: each has its own H2D event, and each column block its own Y event.
constexpr int kMaxChunks = 64;

// Row chunks when the feature matrix travels whole-width (1 = copy everything, then compute).  Measured (30.1 GB per
// pass): 1 -> 635 ms, 4 -> 587, 8 -> 579, 16 -> 574 ms; the copies alone take ~548 ms.
constexpr int kRowChunks = 16;

// Width (elements) of the column blocks when Y comes back.  64 floats = 256-byte rows: the narrowest pitched copy that
// still runs at the full PCIe rate in both directions (55.6 / 53.5 GB/s alone, 48 + 50 GB/s both directions at once;
// 128-byte rows: 34 + 40 GB/s, tools/pcie_probe.cu), and a width the row-group aggregation kernel runs natively.
// bf16 and fp16 features take the same 64 columns, i.e. 128-byte rows (the slower pitched copy): measured on the 50M-node /
// 976M-entry graph at d = 128 (tools/e2e_bf16_bench.py, NVIDIA B200, 1000 W power limit, each form in its own process),
// column blocks 735.7 ms with fp32 Y back and 536.8 ms with bf16 Y back, against 795.1 / 578.3 ms for row blocks (full-rate
// contiguous H2D, Y copied after the last phase).
constexpr int64_t kColWidth = 64;

// Row chunks per column block: the block's aggregation is phased by arriving row chunk, so that only the last chunk's
// phase -- not a whole-graph launch -- stands between the end of a block's H2D copy and the start of its D2H copy.  A
// phase over 50M rows costs 20-23 ms at 64 columns whatever the range length (tools/phase_probe.py; 52.8 ms for the
// whole block in one launch), so the phases of a block must fit under its 230 ms H2D copy.  Measured per step: 858.9 ms
// (1 chunk), 831.7 ms (4), 828.9 ms (8); 4 keeps the larger margin.
constexpr int kColRows = 4;

// The feature matrix travels as KC = d / W column blocks of width W, each in R row chunks.
struct Schedule {
  int64_t W;
  int KC, R;
};

static Schedule schedule(int64_t d, bool y_wanted) {
  if (y_wanted && d % kColWidth == 0 && d / kColWidth >= 2 && d / kColWidth <= kMaxChunks) {
    const int KC = (int)(d / kColWidth);
    int R = kColRows;
    while (R > 1 && KC * R > kMaxChunks) R /= 2;
    return {kColWidth, KC, R};
  }
  // the widths the ranged aggregation entries take (16-byte fp32 / 8-byte bf16 and fp16 rows, row-group kernel widths)
  if (d % 4 == 0 && (d == 32 || d == 64 || d >= 128)) return {d, 1, kRowChunks};
  return {d, 1, 1};
}

struct HostPipelineCache {
  int64_t n = -1, nnz = -1, d = -1, cap = -1;
  int C = -1, device = -1;
  // The feature buffer is sized in bytes and grows when a call needs more (an fp32 call after a half one); a half call
  // after an fp32 one reuses it, so a caller alternating feature types does not reallocate the largest buffer.
  size_t x_bytes = 0, ystage_bytes = 0, partial_bytes = 0;
  int64_t *rowptr = nullptr;
  int32_t *col = nullptr;
  void *x = nullptr;
  float *y = nullptr, *dinv = nullptr, *partial = nullptr;
  void *ystage = nullptr;  // half Y (bf16 or fp16) rounded for the D2H copy (allocated by the first half-Y call)
  int32_t *labels = nullptr, *deg = nullptr, *match = nullptr;
  uint8_t *labels8 = nullptr, *deg_code = nullptr;
  int64_t *plan = nullptr, *counters = nullptr;
  double *node_sum = nullptr;
  int64_t *seg = nullptr, *bounds = nullptr;  // column segments of the feature row chunks
  uint8_t *skip = nullptr;
  cudaStream_t st = nullptr, st_copy = nullptr, st_back = nullptr;
  cudaEvent_t ev_csr = nullptr, ev_x[kMaxChunks] = {nullptr}, ev_y[kMaxChunks] = {nullptr};
  void release() {
    cudaFree(seg); cudaFree(bounds); cudaFree(skip);
    if (st_copy) cudaStreamDestroy(st_copy);
    if (st_back) cudaStreamDestroy(st_back);
    if (ev_csr) cudaEventDestroy(ev_csr);
    for (auto &e : ev_x) if (e) cudaEventDestroy(e);
    for (auto &e : ev_y) if (e) cudaEventDestroy(e);
    cudaFree(rowptr); cudaFree(col); cudaFree(x); cudaFree(y); cudaFree(ystage); cudaFree(dinv); cudaFree(partial);
    cudaFree(labels); cudaFree(labels8); cudaFree(deg_code); cudaFree(deg); cudaFree(match); cudaFree(plan); cudaFree(counters); cudaFree(node_sum);
    if (st) cudaStreamDestroy(st);
    *this = HostPipelineCache();
  }
};
static HostPipelineCache g_cache;  // one cached pipeline per process, guarded by g_cache_mu
static std::mutex g_cache_mu;
constexpr int64_t kHostPipelineThreshold = 512;

// The buffers of the cache that only grow (features, half Y staging, split-row partial sums): reallocates p when it
// holds fewer than `bytes`.
template <typename T>
static cudaError_t grow(T *&p, size_t &cap, size_t bytes) {
  if (cap >= bytes) return cudaSuccess;
  cudaFree(p);
  p = nullptr;
  cap = 0;
  const cudaError_t e = cudaMalloc(&p, bytes);
  if (e == cudaSuccess) cap = bytes;
  return e;
}

#define WDGH_REQUIRE_AT(cond, what)                                      \
  do {                                                                   \
    if (!(cond)) {                                                       \
      snprintf(g_err, sizeof(g_err), "%s: %s", fn, what);                \
      return WDGH_EINVAL;                                                \
    }                                                                    \
  } while (0)

// What the body needs of a feature type T: the element type of its C-ABI pointers (Bits), and its full aggregation
// launch and phase entry, both with fp32 Y, in the argument order of the half-type entries.  The half Y it may return
// is kHalfY<T>, rounded by round_to_half<T>.
template <typename T>
struct Elem;
template <>
struct Elem<float> {
  using Bits = float;
  static int full(const int64_t *rowptr, const int32_t *col, const float *val, int64_t n, const float *x, int64_t d,
                  int64_t ldx, void *y, int64_t ldy, int /* y_dtype: always WDGH_DTYPE_F32 */, int norm,
                  int add_self_loop, const float *dinv, const uint8_t *deg_code, int64_t *plan_i64,
                  const int64_t *plan_host, float *partial, int64_t row_offset, void *stream) {
    return wdgh_spmm_csr(rowptr, col, val, n, x, d, ldx, static_cast<float *>(y), ldy, norm, add_self_loop, dinv,
                         deg_code, plan_i64, plan_host, partial, row_offset, stream);
  }
  static int phase(const int64_t *rowptr, const int64_t *range_begin, const int64_t *range_end, const int32_t *col,
                   const float *val, int64_t n, const float *x, int64_t d, int64_t ldx, float *y, int64_t ldy, int norm,
                   int add_self_loop, const float *dinv, const uint8_t *deg_code, const uint8_t *skip_rows,
                   int accumulate, int finalize, int run_split_rows, int64_t *plan_i64, const int64_t *plan_host,
                   float *partial, int64_t row_offset, void *stream) {
    return wdgh_spmm_csr_ranged(rowptr, range_begin, range_end, col, val, n, x, d, ldx, y, ldy, norm, add_self_loop,
                                dinv, deg_code, skip_rows, accumulate, finalize, run_split_rows, nullptr, 0, 0, 0, 0, 0,
                                plan_i64, plan_host, partial, row_offset, stream);
  }
};
template <>
struct Elem<bf16> {
  using Bits = uint16_t;
  static constexpr auto full = wdgh_spmm_csr_bf16;
  static constexpr auto phase = wdgh_spmm_csr_ranged_bf16;
};
template <>
struct Elem<f16> {
  using Bits = uint16_t;
  static constexpr auto full = wdgh_spmm_csr_f16;
  static constexpr auto phase = wdgh_spmm_csr_ranged_f16;
};

// The body of wdgh_pipeline_host (T = float), wdgh_pipeline_host_bf16 and wdgh_pipeline_host_f16.
template <typename T>
static int pipeline_host(const char *fn, const int64_t *rowptr_host, const int32_t *col_host, int64_t n, int64_t nnz,
                         const typename Elem<T>::Bits *x_host, int64_t d, const int32_t *labels_host,
                         int32_t num_classes, int norm, int add_self_loop, void *y_host, int y_dtype,
                         int64_t *counters_host, double *node_sum_host) {
  using E = Elem<T>;
  using Tin = typename E::Bits;
  WDGH_REQUIRE_AT(rowptr_host && x_host && labels_host && counters_host && node_sum_host, "null pointer");
  WDGH_REQUIRE_AT(n > 0 && nnz >= 0 && d > 0 && num_classes >= 1 && (col_host || nnz == 0), "bad shape");
  WDGH_REQUIRE_AT(y_dtype == WDGH_DTYPE_F32 || y_dtype == kHalfY<T>, "bad y_dtype (float32, or the type of x)");
  std::lock_guard<std::mutex> lock(g_cache_mu);  // the cached buffers and streams serve one call at a time
  HostPipelineCache &c = g_cache;
  const int C = num_classes;
  int device = -1;
  WDGH_CUDA(cudaGetDevice(&device));
  const size_t n_counters = WDGH_SC_WORDS((size_t)C);
  const int64_t cap = 2 * nnz / kHostPipelineThreshold + 2;
  if (c.n != n || c.nnz != nnz || c.d != d || c.C != C || c.device != device) {
    c.release();
    WDGH_CUDA(cudaStreamCreateWithFlags(&c.st, cudaStreamNonBlocking));
    WDGH_CUDA(cudaMalloc(&c.rowptr, (n + 1) * sizeof(int64_t)));
    WDGH_CUDA(cudaMalloc(&c.col, (nnz > 0 ? nnz : 1) * sizeof(int32_t)));
    WDGH_CUDA(cudaMalloc(&c.y, n * d * sizeof(float)));
    WDGH_CUDA(cudaMalloc(&c.dinv, n * sizeof(float)));
    WDGH_CUDA(cudaMalloc(&c.labels, n * sizeof(int32_t)));
    WDGH_CUDA(cudaMalloc(&c.labels8, n));
    WDGH_CUDA(cudaMalloc(&c.deg_code, n));
    WDGH_CUDA(cudaMalloc(&c.deg, n * sizeof(int32_t)));
    WDGH_CUDA(cudaMalloc(&c.match, n * sizeof(int32_t)));
    WDGH_CUDA(cudaMalloc(&c.plan, WDGH_PLAN_WORDS(cap) * sizeof(int64_t)));
    WDGH_CUDA(cudaMalloc(&c.counters, n_counters * sizeof(int64_t)));
    WDGH_CUDA(cudaMalloc(&c.node_sum, 2 * sizeof(double)));
    WDGH_CUDA(cudaStreamCreateWithFlags(&c.st_copy, cudaStreamNonBlocking));
    WDGH_CUDA(cudaStreamCreateWithFlags(&c.st_back, cudaStreamNonBlocking));
    WDGH_CUDA(cudaEventCreateWithFlags(&c.ev_csr, cudaEventDisableTiming));
    for (auto &e : c.ev_x) WDGH_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    for (auto &e : c.ev_y) WDGH_CUDA(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    WDGH_CUDA(cudaMalloc(&c.seg, (size_t)(kRowChunks + 1) * (size_t)n * sizeof(int64_t)));
    WDGH_CUDA(cudaMalloc(&c.bounds, (kRowChunks + 1) * sizeof(int64_t)));
    WDGH_CUDA(cudaMalloc(&c.skip, (size_t)n));
    c.n = n; c.nnz = nnz; c.d = d; c.C = C; c.cap = cap; c.device = device;
  }
  WDGH_CUDA(grow(c.x, c.x_bytes, (size_t)(n * d) * sizeof(Tin)));
  const bool y16 = y_host && y_dtype != WDGH_DTYPE_F32;
  if (y16) WDGH_CUDA(grow(c.ystage, c.ystage_bytes, (size_t)(n * d) * 2));
  const size_t ysz = y16 ? 2 : sizeof(float);  // bytes of one element of Y on the host
  Tin *x = static_cast<Tin *>(c.x);
  cudaStream_t st = c.st, sc = c.st_copy, sb = c.st_back;
  const Schedule sched = schedule(d, y_host != nullptr);
  const int64_t W = sched.W;
  const int KC = sched.KC, R = sched.R;
  // rows [r0, r0 + rows) of column block kc between two row-major n x d matrices: contiguous when the block is the
  // whole width, pitched otherwise
  auto copy_block = [&](void *dst, const void *src, size_t esz, int kc, int64_t r0, int64_t rows, cudaMemcpyKind kind,
                        cudaStream_t stream) -> cudaError_t {
    const size_t off = (size_t)(r0 * d + kc * W) * esz;
    char *to = static_cast<char *>(dst) + off;
    const char *from = static_cast<const char *>(src) + off;
    if (W == d) return cudaMemcpyAsync(to, from, (size_t)(rows * d) * esz, kind, stream);
    return cudaMemcpy2DAsync(to, d * esz, from, d * esz, W * esz, rows, kind, stream);
  };
  // 1. graph + labels first (the compute stream needs them at once) ...
  WDGH_CUDA(cudaMemcpyAsync(c.rowptr, rowptr_host, (n + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, sc));
  if (nnz) WDGH_CUDA(cudaMemcpyAsync(c.col, col_host, nnz * sizeof(int32_t), cudaMemcpyHostToDevice, sc));
  WDGH_CUDA(cudaMemcpyAsync(c.labels, labels_host, n * sizeof(int32_t), cudaMemcpyHostToDevice, sc));
  WDGH_CUDA(cudaEventRecord(c.ev_csr, sc));
  // 2. ... then the feature matrix on the copy stream, block by block and chunk by chunk (rows [bounds_h[r],
  //    bounds_h[r + 1]) form row chunk r)
  const int64_t blk = (n + R - 1) / R;
  int64_t bounds_h[kRowChunks + 1];
  for (int r = 0; r <= R; ++r) bounds_h[r] = std::min((int64_t)r * blk, n);
  for (int kc = 0; kc < KC; ++kc) {
    for (int r = 0; r < R; ++r) {
      if (bounds_h[r + 1] > bounds_h[r])
        WDGH_CUDA(copy_block(x, x_host, sizeof(Tin), kc, bounds_h[r], bounds_h[r + 1] - bounds_h[r],
                             cudaMemcpyHostToDevice, sc));
      WDGH_CUDA(cudaEventRecord(c.ev_x[kc * R + r], sc));
    }
  }
  WDGH_CUDA(cudaStreamWaitEvent(st, c.ev_csr, 0));
  int64_t plan_host[8];
  int rc = wdgh_plan_build(c.rowptr, n, nnz, kHostPipelineThreshold, c.plan, cap, plan_host, st);
  if (rc) return rc;
  const int64_t ldp = (d + 3) & ~int64_t(3);
  WDGH_CUDA(grow(c.partial, c.partial_bytes, (size_t)(plan_host[1] * ldp) * sizeof(float)));
  if (norm != WDGH_NORM_NONE) {
    rc = wdgh_degree_scale(c.rowptr, nullptr, n, norm, add_self_loop, c.dinv, nullptr, c.deg_code, st);
    if (rc) return rc;
  }
  const float *dinv = norm != WDGH_NORM_NONE ? c.dinv : nullptr;
  const uint8_t *code = norm != WDGH_NORM_NONE ? c.deg_code : nullptr;
  // one launch over every row of a column slab of width w (fp32 Y)
  auto full = [&](const Tin *xb, int64_t w, float *yb) -> int {
    return E::full(c.rowptr, c.col, nullptr, n, xb, w, d, yb, d, WDGH_DTYPE_F32, norm, add_self_loop, dinv, code, c.plan,
                   plan_host, c.partial, 0, st);
  };
  // the phase of row chunk k: y (+)= the entries whose column lies in chunk k; the last phase finalizes
  auto phase = [&](int k, const Tin *xb, int64_t w, float *yb, int accumulate, int last) -> int {
    const int64_t *b = c.seg + (size_t)k * n, *e = c.seg + (size_t)(k + 1) * n;
    return E::phase(c.rowptr, b, e, c.col, nullptr, n, xb, w, d, yb, d, norm, add_self_loop, dinv, code, c.skip,
                    accumulate, last, last, c.plan, plan_host, c.partial, 0, st);
  };
  // 3. label pass: needs only the graph and the labels, runs under the feature copy
  rc = wdgh_structure_counts(c.rowptr, c.col, n, nnz, c.labels, C, c.plan, plan_host, c.counters, c.node_sum, c.deg,
                             c.match, c.labels8, n, 0, st);
  if (rc) return rc;
  // 4. per column block: one aggregation phase per arriving row chunk (R = 1: one full launch); the Y block leaves on
  //    the third stream as soon as its last phase (and, for a half Y, its rounding) is done
  if (R > 1) {
    WDGH_CUDA(cudaMemcpyAsync(c.bounds, bounds_h, (R + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    rc = wdgh_column_segments(c.rowptr, c.col, n, c.bounds, R + 1, c.seg, st);
    if (rc) return rc;
    rc = wdgh_plan_heavy_flags(c.plan, plan_host, n, c.skip, st);
    if (rc) return rc;
  }
  for (int kc = 0; kc < KC; ++kc) {
    const Tin *xb = x + kc * W;
    float *yb = c.y + kc * W;
    for (int r = 0; r < R; ++r) {
      WDGH_CUDA(cudaStreamWaitEvent(st, c.ev_x[kc * R + r], 0));
      rc = (R == 1) ? full(xb, W, yb) : phase(r, xb, W, yb, r > 0, r == R - 1);
      if (rc) return rc;
    }
    if (!y_host) continue;
    if constexpr (kHalfY<T> != WDGH_DTYPE_F32) {
      if (y16) {
        rc = round_to_half<T>(yb, n, W, d, static_cast<uint16_t *>(c.ystage) + kc * W, d, st);
        if (rc) return rc;
      }
    }
    WDGH_CUDA(cudaEventRecord(c.ev_y[kc], st));
    WDGH_CUDA(cudaStreamWaitEvent(sb, c.ev_y[kc], 0));
    WDGH_CUDA(copy_block(y_host, y16 ? c.ystage : static_cast<void *>(c.y), ysz, kc, 0, n, cudaMemcpyDeviceToHost, sb));
  }
  WDGH_CUDA(cudaMemcpyAsync(counters_host, c.counters, n_counters * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
  WDGH_CUDA(cudaMemcpyAsync(node_sum_host, c.node_sum, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
  WDGH_CUDA(cudaStreamSynchronize(st));
  if (counters_host[WDGH_SC_N_MULTI_NEG] != 0) {
    // labels below -1 or >= C: the 1-byte label copy folds them together with -1, but the reference compares raw
    // labels (hm.py:51) -- redo the label pass on the int32 labels
    rc = wdgh_structure_counts(c.rowptr, c.col, n, nnz, c.labels, C, c.plan, plan_host, c.counters, c.node_sum, c.deg,
                               c.match, nullptr, n, 0, st);
    if (rc) return rc;
    WDGH_CUDA(cudaMemcpyAsync(counters_host, c.counters, n_counters * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
    WDGH_CUDA(cudaMemcpyAsync(node_sum_host, c.node_sum, 2 * sizeof(double), cudaMemcpyDeviceToHost, st));
    WDGH_CUDA(cudaStreamSynchronize(st));
  }
  if (y_host) WDGH_CUDA(cudaStreamSynchronize(sb));
  return 0;
}
#undef WDGH_REQUIRE_AT

}  // namespace wdgh

using namespace wdgh;

extern "C" int wdgh_pipeline_host_release(void) {
  std::lock_guard<std::mutex> lock(g_cache_mu);
  g_cache.release();
  return 0;
}

extern "C" int wdgh_pipeline_host(const int64_t *rowptr_host, const int32_t *col_host, int64_t n, int64_t nnz,
                                  const float *x_host, int64_t d, const int32_t *labels_host, int32_t num_classes,
                                  int norm, int add_self_loop, float *y_host, int64_t *counters_host,
                                  double *node_sum_host) {
  return pipeline_host<float>("wdgh_pipeline_host", rowptr_host, col_host, n, nnz, x_host, d, labels_host, num_classes, norm,
                       add_self_loop, y_host, WDGH_DTYPE_F32, counters_host, node_sum_host);
}

extern "C" int wdgh_pipeline_host_bf16(const int64_t *rowptr_host, const int32_t *col_host, int64_t n, int64_t nnz,
                                       const uint16_t *x_host, int64_t d, const int32_t *labels_host,
                                       int32_t num_classes, int norm, int add_self_loop, void *y_host, int y_dtype,
                                       int64_t *counters_host, double *node_sum_host) {
  return pipeline_host<bf16>("wdgh_pipeline_host_bf16", rowptr_host, col_host, n, nnz, x_host, d, labels_host,
                             num_classes, norm, add_self_loop, y_host, y_dtype, counters_host, node_sum_host);
}

extern "C" int wdgh_pipeline_host_f16(const int64_t *rowptr_host, const int32_t *col_host, int64_t n, int64_t nnz,
                                      const uint16_t *x_host, int64_t d, const int32_t *labels_host,
                                      int32_t num_classes, int norm, int add_self_loop, void *y_host, int y_dtype,
                                      int64_t *counters_host, double *node_sum_host) {
  return pipeline_host<f16>("wdgh_pipeline_host_f16", rowptr_host, col_host, n, nnz, x_host, d, labels_host,
                            num_classes, norm, add_self_loop, y_host, y_dtype, counters_host, node_sum_host);
}
