// Aggregation similarity without the m x m Gram (utils/homophily_metrics.py:199-206, homophily_plot.py non-NTK
// branch).  The class sum of the Gram is linear in z:
//     w[i][c] = sum_{j: l_j = c} <z_i, z_j> = <z_i, s_c>,   s_c = sum_{j: l_j = c} z_j   (s = Y^T z, [C][d])
// so two streaming passes over z replace the O(m^2 d) Gram and its O(m^2) memory.
//
//   class_sum_partial_kernel  rows cut into `nseg` contiguous segments; segment q -> partial fp64 table
//                             part[q][c][0..d) (column sums) and part[q][c][d] (row count).  Inside a CTA, `groups`
//                             thread groups of `gw` threads each own one private shared-memory table; thread kk of
//                             group g adds column k0 + kk of rows r0 + g, r0 + g + groups, ... in row order, and the
//                             group tables are added in group order at the end.  No atomics.
//   class_sum_reduce_kernel   s[c][k] = sum of the nseg partials: 8 contiguous runs of segments, each summed in
//                             segment order, then the 8 run sums in run order.
//   class_dot_kernel          w[i][c] = f32(sum_k z[i][k] * s[c][k]), products and sum in fp64 (one FMA chain in k
//                             order), rounded once; is_mean divides by the class count in fp64 first.
// Every tiling parameter is a function of (m, d, C) only: the result does not depend on the SM count or on
// scheduling.
#include "common.cuh"

namespace wdgh {

constexpr int kCsThreads = 256;
constexpr int kCsSmemBytes = 48 * 1024;          // group tables of one CTA (default dynamic shared-memory limit)
constexpr int64_t kCsSegRowsMin = 256;           // rows per segment at least ...
constexpr int64_t kCsMaxSegs = 1024;             // ... and at most this many segments ...
constexpr int64_t kCsPartialDoubles = 1 << 22;   // ... whose partial tables fit 32 MiB (unless one table is larger)
constexpr int kCsUnroll = 8;                     // rows in flight per thread

struct ClassSumShape {
  int gw;         // columns per column tile = threads per group
  int n_kt;       // column tiles
  int ct;         // classes per class tile
  int n_ct;       // class tiles
  int groups;     // row-interleaved thread groups of a CTA
  int threads;
  size_t smem;
  int64_t nseg, seg_rows;
};

// d = C <= 16 (one-hot features): ~256 / d groups of d threads, each warp reads several whole rows at once.
// d = 128: two groups of 128 threads, one column per thread.  d > 128: column tiles of <= 128.  C * gw too large
// for one table: class tiles (a row whose label is outside the tile is not read).
static ClassSumShape class_sum_shape(int64_t m, int64_t d, int64_t C) {
  ClassSumShape s;
  s.n_kt = (int)ceil_div(d, 128);
  s.gw = (int)ceil_div(d, s.n_kt);
  const int64_t per_class = (int64_t)(s.gw + 1) * 8;  // one table row: gw column sums + the count
  const int64_t fit = kCsSmemBytes / per_class;        // >= 46 since gw <= 128
  s.n_ct = (int)ceil_div(C, fit < C ? fit : C);
  s.ct = (int)ceil_div(C, s.n_ct);
  const int64_t gmax = kCsThreads / s.gw;
  int64_t groups = kCsSmemBytes / (s.ct * per_class);
  groups = groups < gmax ? groups : gmax;
  s.groups = (int)(groups < 1 ? 1 : groups);
  s.threads = (int)ceil_div((int64_t)s.groups * s.gw, kWarp) * kWarp;
  s.smem = (size_t)s.groups * s.ct * per_class;
  const int64_t table = C * (d + 1);
  int64_t cap = kCsPartialDoubles / table;
  cap = cap < kCsMaxSegs ? cap : kCsMaxSegs;
  cap = cap < 1 ? 1 : cap;
  const int64_t want = ceil_div(m < 1 ? 1 : m, kCsSegRowsMin);
  s.nseg = want < cap ? want : cap;
  s.seg_rows = ceil_div(m < 1 ? 1 : m, s.nseg);
  s.nseg = ceil_div(m < 1 ? 1 : m, s.seg_rows);
  return s;
}

// grid: nseg * n_kt * n_ct CTAs, x = ((seg * n_kt) + kt) * n_ct + ct_tile
__global__ void __launch_bounds__(kCsThreads)
class_sum_partial_kernel(const float *__restrict__ z, int64_t m, int64_t d, int64_t ldz,
                         const int32_t *__restrict__ labels, int C, int64_t seg_rows, int gw, int n_kt, int groups,
                         int ct, int n_ct, double *__restrict__ part) {
  extern __shared__ double tab[];  // [groups][ct][gw + 1]
  const int64_t b = blockIdx.x;
  const int ctile = (int)(b % n_ct);
  const int kt = (int)((b / n_ct) % n_kt);
  const int64_t seg = b / ((int64_t)n_ct * n_kt);
  const int64_t k0 = (int64_t)kt * gw;
  const int c0 = ctile * ct;
  const int cend = (C - c0 < ct) ? C : c0 + ct;
  const int row_len = gw + 1;
  for (int t = threadIdx.x; t < groups * ct * row_len; t += blockDim.x) tab[t] = 0.0;
  __syncthreads();

  const int g = threadIdx.x / gw, kk = threadIdx.x - g * gw;
  const int64_t k = k0 + kk;
  const bool col_ok = k < d;
  const bool counter = kt == 0 && kk == 0;  // one thread per group counts the rows (column tile 0 only)
  if (g < groups) {
    double *my = tab + (int64_t)g * ct * row_len;
    const int64_t r0 = seg * seg_rows;
    const int64_t r1 = (m - r0 < seg_rows) ? m : r0 + seg_rows;
    const int64_t step = (int64_t)groups * kCsUnroll;
    for (int64_t j = r0 + g; j < r1; j += step) {
      int slot[kCsUnroll];
      float v[kCsUnroll];
#pragma unroll
      for (int u = 0; u < kCsUnroll; ++u) {
        const int64_t r = j + (int64_t)u * groups;
        slot[u] = -1;
        v[u] = 0.f;
        if (r < r1) {
          const int lab = __ldg(labels + r);
          if (lab >= c0 && lab < cend) {  // any other label (negative, >= C, another tile) joins no class here
            slot[u] = lab - c0;
            if (col_ok) v[u] = __ldg(z + r * ldz + k);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < kCsUnroll; ++u) {
        if (slot[u] < 0) continue;
        double *row = my + slot[u] * row_len;
        if (col_ok) row[kk] += (double)v[u];
        if (counter) row[gw] += 1.0;
      }
    }
  }
  __syncthreads();

  for (int t = threadIdx.x; t < ct * row_len; t += blockDim.x) {
    const int c = t / row_len, q = t - c * row_len;
    if (c0 + c >= C) continue;
    int64_t col;
    if (q < gw) {
      col = k0 + q;
      if (col >= d) continue;
    } else {
      if (kt != 0) continue;
      col = d;
    }
    double acc = 0.0;
    for (int gg = 0; gg < groups; ++gg) acc += tab[((int64_t)gg * ct + c) * row_len + q];
    part[(seg * C + c0 + c) * (d + 1) + col] = acc;
  }
}

// s[e] = sum over segments of part[seg][e], e < width = C * (d + 1).  32 entries per CTA (one per lane), 8 warps.
__global__ void __launch_bounds__(256)
class_sum_reduce_kernel(const double *__restrict__ part, int64_t nseg, int64_t width, double *__restrict__ s) {
  __shared__ double run[8][32];
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t e = (int64_t)blockIdx.x * 32 + lane;
  const int64_t q0 = nseg * wid / 8, q1 = nseg * (wid + 1) / 8;
  double acc = 0.0;
  if (e < width) {
#pragma unroll 8
    for (int64_t q = q0; q < q1; ++q) acc += __ldg(part + q * width + e);
  }
  run[wid][lane] = acc;
  __syncthreads();
  if (wid == 0 && e < width) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += run[w][lane];
    s[e] = t;
  }
}

// w[i][c0 .. c0 + CT) for 512 rows per CTA, two rows per thread.  z is staged through shared memory in 16-column
// steps (coalesced whatever ldz is), the class tile of s likewise; columns past d are zero in both.
constexpr int kDotThreads = 256;
constexpr int kDotRows = 2 * kDotThreads;
constexpr int kDotKT = 16;
constexpr int kDotMaxCT = 16;

template <int CT>
__global__ void __launch_bounds__(kDotThreads)
class_dot_kernel(const float *__restrict__ z, int64_t m, int64_t d, int64_t ldz, const double *__restrict__ s,
                 int C, int n_ct, int is_mean, float *__restrict__ w) {
  __shared__ float zs[kDotRows][kDotKT + 1];
  __shared__ double ss[CT][kDotKT];
  const int64_t row0 = (int64_t)(blockIdx.x / n_ct) * kDotRows;
  const int c0 = (int)(blockIdx.x % n_ct) * CT;
  double acc[2][CT];
#pragma unroll
  for (int c = 0; c < CT; ++c) acc[0][c] = acc[1][c] = 0.0;
  for (int64_t k0 = 0; k0 < d; k0 += kDotKT) {
    for (int i = threadIdx.x; i < kDotRows * kDotKT; i += kDotThreads) {
      const int r = i / kDotKT, kk = i % kDotKT;
      const int64_t row = row0 + r, k = k0 + kk;
      zs[r][kk] = (row < m && k < d) ? __ldg(z + row * ldz + k) : 0.f;
    }
    for (int i = threadIdx.x; i < CT * kDotKT; i += kDotThreads) {
      const int c = i / kDotKT, kk = i % kDotKT;
      const int64_t k = k0 + kk;
      ss[c][kk] = (c0 + c < C && k < d) ? __ldg(s + (int64_t)(c0 + c) * (d + 1) + k) : 0.0;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kDotKT; ++kk) {
      const double a0 = (double)zs[threadIdx.x][kk];
      const double a1 = (double)zs[threadIdx.x + kDotThreads][kk];
#pragma unroll
      for (int c = 0; c < CT; ++c) {
        const double bv = ss[c][kk];
        acc[0][c] = fma(a0, bv, acc[0][c]);
        acc[1][c] = fma(a1, bv, acc[1][c]);
      }
    }
    __syncthreads();
  }
  const int64_t ra = row0 + threadIdx.x, rb = ra + kDotThreads;
#pragma unroll
  for (int c = 0; c < CT; ++c) {
    if (c0 + c < C) {
      double va = acc[0][c], vb = acc[1][c];
      if (is_mean) {  // empty class: 0 / 0 = NaN
        const double cnt = __ldg(s + (int64_t)(c0 + c) * (d + 1) + d);
        va = va / cnt;
        vb = vb / cnt;
      }
      if (ra < m) w[ra * C + c0 + c] = (float)va;
      if (rb < m) w[rb * C + c0 + c] = (float)vb;
    }
  }
}

template <int CT>
static void launch_class_dot(unsigned grid, const float *z, int64_t m, int64_t d, int64_t ldz, const double *s, int C,
                             int n_ct, int is_mean, float *w, cudaStream_t st) {
  class_dot_kernel<CT><<<grid, kDotThreads, 0, st>>>(z, m, d, ldz, s, C, n_ct, is_mean, w);
}

}  // namespace wdgh

using namespace wdgh;

extern "C" int64_t wdgh_class_inner_workspace_doubles(int64_t m, int64_t d, int32_t num_classes) {
  if (m < 0 || d < 1 || num_classes < 1 || d > (INT64_C(1) << 40) / num_classes) return -1;
  const ClassSumShape s = class_sum_shape(m, d, num_classes);
  return (s.nseg + 1) * (int64_t)num_classes * (d + 1);
}

extern "C" int wdgh_class_inner_sums(const float *z, int64_t m, int64_t d, int64_t ldz, const int32_t *labels,
                                     int32_t num_classes, int is_mean, double *workspace, float *w, void *stream) {
  WDGH_REQUIRE(m >= 0 && d >= 1 && ldz >= d && num_classes >= 1 && (is_mean == 0 || is_mean == 1),
               "wdgh_class_inner_sums: bad arguments");
  WDGH_REQUIRE(d <= (INT64_C(1) << 40) / num_classes, "wdgh_class_inner_sums: C * d too large");
  if (m == 0) return 0;
  WDGH_REQUIRE(z && labels && workspace && w, "wdgh_class_inner_sums: null pointer");
  cudaStream_t st = as_stream(stream);
  const int C = num_classes;
  const ClassSumShape sh = class_sum_shape(m, d, C);
  const int64_t width = (int64_t)C * (d + 1);
  double *s = workspace;           // [C][d + 1]: column sums, then the count
  double *part = workspace + width;  // [nseg][C][d + 1]
  const int64_t n_cta = sh.nseg * sh.n_kt * sh.n_ct;
  WDGH_REQUIRE(n_cta <= INT32_MAX, "wdgh_class_inner_sums: too many column / class tiles");
  class_sum_partial_kernel<<<(unsigned)n_cta, sh.threads, sh.smem, st>>>(z, m, d, ldz, labels, C, sh.seg_rows, sh.gw,
                                                                         sh.n_kt, sh.groups, sh.ct, sh.n_ct, part);
  WDGH_LAUNCHED("class_sum_partial_kernel");
  class_sum_reduce_kernel<<<(unsigned)ceil_div(width, 32), 256, 0, st>>>(part, sh.nseg, width, s);
  WDGH_LAUNCHED("class_sum_reduce_kernel");

  const int ct = (int)ceil_div(C, ceil_div(C, kDotMaxCT));  // balanced class tiles of <= 16
  const int n_ct = (int)ceil_div(C, ct);
  const int64_t n_dot = ceil_div(m, kDotRows) * n_ct;
  WDGH_REQUIRE(n_dot <= INT32_MAX, "wdgh_class_inner_sums: too many rows x class tiles");
  const unsigned grid = (unsigned)n_dot;
  switch (ct) {
#define WDGH_DOT_CASE(N) \
  case N: launch_class_dot<N>(grid, z, m, d, ldz, s, C, n_ct, is_mean, w, st); break;
    WDGH_DOT_CASE(1) WDGH_DOT_CASE(2) WDGH_DOT_CASE(3) WDGH_DOT_CASE(4) WDGH_DOT_CASE(5) WDGH_DOT_CASE(6)
    WDGH_DOT_CASE(7) WDGH_DOT_CASE(8) WDGH_DOT_CASE(9) WDGH_DOT_CASE(10) WDGH_DOT_CASE(11) WDGH_DOT_CASE(12)
    WDGH_DOT_CASE(13) WDGH_DOT_CASE(14) WDGH_DOT_CASE(15) WDGH_DOT_CASE(16)
#undef WDGH_DOT_CASE
    default: return fail(WDGH_EINVAL, "wdgh_class_inner_sums: class tile");
  }
  WDGH_LAUNCHED("class_dot_kernel");
  return 0;
}
