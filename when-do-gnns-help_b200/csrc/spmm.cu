// A_hat X aggregation: CSR SpMM in float32 with on-the-fly D^-1/2 / D^-1 scaling.
//
// Replaces torch.spmm(adj, features) / torch.mm(adj, features) of the reference
// (utils/homophily_metrics.py:192,199,234,299,315) together with the materialised
// normalisers of utils/util_funcs.py:383-390 (row) and :418-426 (symmetric):
//     y_i = s_i * ( sum_{j in row i} w_ij * t_j * x_j  +  [self loop] t_i * x_i )
// with s = t = D^-1/2 (SYM), s = D^-1, t = 1 (RW), s = t = 1 (NONE).  A_hat itself is
// never written to memory.
//
// HBM-bound gather kernel (no tensor cores: there is no dense operand reuse):
//   * a group of G lanes owns one row; lane g holds VEC contiguous floats of NCH
//     column chunks, so one neighbour row is fetched with coalesced 16-byte loads
//     (d=128: one warp, one float4 per lane, 512 B per neighbour);
//   * the group loads G column indices (+ weights) with one coalesced load, keeps
//     them in registers ("row segment staged on chip") and broadcasts them with
//     shuffles; the inner loop issues U independent row gathers before the FMAs so
//     every warp keeps U*512 B in flight;
//   * degree-binned load balance: rows longer than the plan's threshold are skipped
//     here and split into fixed-size chunks, one warp per chunk, summed in a fixed
//     order by a second small kernel (deterministic, no float atomics).
//
// bfloat16 features (wdgh_spmm_csr_bf16): the same kernels with the element type of x (Tin) and of y (Tout) as
// template parameters.  Loads widen bf16 -> fp32 exactly (a 16-bit shift), the accumulators are fp32 and every row is
// summed in the order of the fp32 instances -- stored entries in CSR order as fmaf(w, x_j, acc) per column, then the
// self loop, then the row scale; split rows through the same chunks and the same fixed-order finish -- so a bf16 launch
// with fp32 output is bit-identical to the fp32 launch on x.float(), and with bf16 output (round to nearest even) to
// that result .to(bfloat16).  The fp32 instances are unchanged.  The phased form (wdgh_spmm_csr_ranged_bf16) takes bf16
// features with fp32 output only: its partial sums stay fp32, so a phase is bit-identical to the fp32 phase on x.float().
//
// float16 features (wdgh_spmm_csr_f16, wdgh_spmm_csr_ranged_f16): the same instances with Tin = __half.  fp16 -> fp32 is
// exact for every value (subnormals, +-0, +-inf and NaN included; one HADD2.F32 per element), the order is the one
// above, so fp32 output is bit-identical to the fp32 launch on x.float() and fp16 output (round to nearest even,
// overflow to +-inf) to that result .to(float16).  A half Y has the type of X: no fp16 -> bf16 or bf16 -> fp16 launch.
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <limits.h>
#include <stdlib.h>

#include <type_traits>

#include "internal.cuh"

namespace wdgh {

// bf16 -> fp32 is exact: the bf16 bits are the upper half of the float
__device__ __forceinline__ float bf16_lo(unsigned u) { return __uint_as_float(u << 16); }
__device__ __forceinline__ float bf16_hi(unsigned u) { return __uint_as_float(u & 0xffff0000u); }
__device__ __forceinline__ unsigned bf16x2_rn(float a, float b) {  // round to nearest even, a in the low half
  const __nv_bfloat162 h = __float22bfloat162_rn(make_float2(a, b));
  return *reinterpret_cast<const unsigned *>(&h);
}

// The 16-bit feature types: a packed pair (low half first) or one value widened to fp32 exactly, a pair or one value
// rounded to nearest even
template <typename H>
struct Half;
template <>
struct Half<bf16> {
  static __device__ __forceinline__ float2 widen2(unsigned u) { return make_float2(bf16_lo(u), bf16_hi(u)); }
  static __device__ __forceinline__ float widen1(unsigned short u) { return bf16_lo(u); }
  static __device__ __forceinline__ unsigned round2(float a, float b) { return bf16x2_rn(a, b); }
  static __device__ __forceinline__ bf16 round1(float v) { return __float2bfloat16_rn(v); }
};
template <>
struct Half<f16> {  // overflow rounds to +-inf, as Tensor.to(torch.float16) does
  static __device__ __forceinline__ float2 widen2(unsigned u) { return __half22float2(*reinterpret_cast<const __half2 *>(&u)); }
  static __device__ __forceinline__ float widen1(unsigned short u) { return __half2float(__ushort_as_half(u)); }
  static __device__ __forceinline__ unsigned round2(float a, float b) {
    const __half2 h = __float22half2_rn(make_float2(a, b));
    return *reinterpret_cast<const unsigned *>(&h);
  }
  static __device__ __forceinline__ f16 round1(float v) { return __float2half_rn(v); }
};

// scalar element access of the split-row finish
__device__ __forceinline__ float load1(const float *p) { return __ldg(p); }
__device__ __forceinline__ float load1(const bf16 *p) { return __bfloat162float(__ldg(p)); }
__device__ __forceinline__ float load1(const f16 *p) { return __half2float(__ldg(p)); }
__device__ __forceinline__ void store1(float *p, float v) { *p = v; }
template <typename H>
__device__ __forceinline__ void store1(H *p, float v) { *p = Half<H>::round1(v); }

template <int VEC>
struct Vec;
template <>
struct Vec<4> {
  float4 v;
  __device__ __forceinline__ void zero() { v = make_float4(0.f, 0.f, 0.f, 0.f); }
  __device__ __forceinline__ void load(const float *p) { v = ldg_na(reinterpret_cast<const float4 *>(p)); }
  __device__ __forceinline__ void load_plain(const float *p) { v = *reinterpret_cast<const float4 *>(p); }
  __device__ __forceinline__ void fma(float w, const Vec &o) {
    v.x = fmaf(w, o.v.x, v.x);
    v.y = fmaf(w, o.v.y, v.y);
    v.z = fmaf(w, o.v.z, v.z);
    v.w = fmaf(w, o.v.w, v.w);
  }
  __device__ __forceinline__ void add(const Vec &o) {
    v.x += o.v.x; v.y += o.v.y; v.z += o.v.z; v.w += o.v.w;
  }
  __device__ __forceinline__ void scale(float s) { v.x *= s; v.y *= s; v.z *= s; v.w *= s; }
  __device__ __forceinline__ void store_stream(float *p) const { st_cs(reinterpret_cast<float4 *>(p), v); }
  __device__ __forceinline__ void store(float *p) const { *reinterpret_cast<float4 *>(p) = v; }
  template <typename H>
  __device__ __forceinline__ void load(const H *p) {  // 8 bytes
    unsigned a, b;
    asm("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(a), "=r"(b) : "l"(p));
    const float2 lo = Half<H>::widen2(a), hi = Half<H>::widen2(b);
    v = make_float4(lo.x, lo.y, hi.x, hi.y);
  }
  template <typename H>
  __device__ __forceinline__ void store_stream(H *p) const {
    asm volatile("st.global.cs.v2.u32 [%0], {%1, %2};" ::"l"(p), "r"(Half<H>::round2(v.x, v.y)),
                 "r"(Half<H>::round2(v.z, v.w))
                 : "memory");
  }
};
template <>
struct Vec<2> {
  float2 v;
  __device__ __forceinline__ void zero() { v = make_float2(0.f, 0.f); }
  __device__ __forceinline__ void load(const float *p) {
    asm("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(v.x), "=f"(v.y) : "l"(p));
  }
  __device__ __forceinline__ void load_plain(const float *p) { v = *reinterpret_cast<const float2 *>(p); }
  __device__ __forceinline__ void fma(float w, const Vec &o) {
    v.x = fmaf(w, o.v.x, v.x);
    v.y = fmaf(w, o.v.y, v.y);
  }
  __device__ __forceinline__ void add(const Vec &o) { v.x += o.v.x; v.y += o.v.y; }
  __device__ __forceinline__ void scale(float s) { v.x *= s; v.y *= s; }
  __device__ __forceinline__ void store_stream(float *p) const {
    asm volatile("st.global.cs.v2.f32 [%0], {%1, %2};" ::"l"(p), "f"(v.x), "f"(v.y) : "memory");
  }
  __device__ __forceinline__ void store(float *p) const { *reinterpret_cast<float2 *>(p) = v; }
  template <typename H>
  __device__ __forceinline__ void load(const H *p) {  // 4 bytes
    unsigned a;
    asm("ld.global.nc.L1::no_allocate.u32 %0, [%1];" : "=r"(a) : "l"(p));
    v = Half<H>::widen2(a);
  }
  template <typename H>
  __device__ __forceinline__ void store_stream(H *p) const {
    asm volatile("st.global.cs.u32 [%0], %1;" ::"l"(p), "r"(Half<H>::round2(v.x, v.y)) : "memory");
  }
};
template <>
struct Vec<1> {
  float v;
  __device__ __forceinline__ void zero() { v = 0.f; }
  __device__ __forceinline__ void load(const float *p) { v = __ldg(p); }
  __device__ __forceinline__ void load_plain(const float *p) { v = *p; }
  __device__ __forceinline__ void fma(float w, const Vec &o) { v = fmaf(w, o.v, v); }
  __device__ __forceinline__ void add(const Vec &o) { v += o.v; }
  __device__ __forceinline__ void scale(float s) { v *= s; }
  __device__ __forceinline__ void store_stream(float *p) const { __stcs(p, v); }
  __device__ __forceinline__ void store(float *p) const { *p = v; }
  template <typename H>
  __device__ __forceinline__ void load(const H *p) {  // 2 bytes
    unsigned short a;
    asm("ld.global.nc.L1::no_allocate.u16 %0, [%1];" : "=h"(a) : "l"(p));
    v = Half<H>::widen1(a);
  }
  template <typename H>
  __device__ __forceinline__ void store_stream(H *p) const { __stcs(p, Half<H>::round1(v)); }
};

// Accumulate entries [s, e) of one row into acc[NCH].  All G lanes of the group call this together.
template <int G, int VEC, int NCH, bool HAS_VAL, typename Tin>
__device__ __forceinline__ void accumulate_range(Vec<VEC> (&acc)[NCH], int64_t s, int64_t e,
                                                 const int32_t *__restrict__ col, const float *__restrict__ val,
                                                 const float *__restrict__ tscale,  // t_j or nullptr
                                                 const Tin *__restrict__ x, int64_t ldx, int cbase, int d,
                                                 int gl, unsigned gmask) {
  constexpr int U0 = (NCH >= 4) ? 2 : (NCH == 2 ? 4 : 8);  // independent gathers in flight per lane
  constexpr int U = U0 < G ? U0 : G;
  bool live[NCH];
#pragma unroll
  for (int t = 0; t < NCH; ++t) live[t] = cbase + (t * G + gl) * VEC < d;

  for (int64_t base = s; base < e; base += G) {
    const int64_t idx = base + gl;
    int j = 0;
    float w = 0.f;
    if (idx < e) {
      j = __ldg(col + idx);
      w = HAS_VAL ? __ldg(val + idx) : 1.f;
      if (tscale != nullptr) w *= __ldg(tscale + j);
    }
    const int cnt = (int)min((int64_t)G, e - base);
    for (int k = 0; k < cnt; k += U) {
      Vec<VEC> v[U][NCH];
      float ww[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
        // slots past the end of the segment are predicated off (group-uniform condition)
        const bool on = k + u < cnt;
        const int src = on ? k + u : 0;
        const int jj = __shfl_sync(gmask, j, src, G);
        ww[u] = __shfl_sync(gmask, w, src, G);
        const Tin *xr = x + (int64_t)jj * ldx + cbase;
#pragma unroll
        for (int t = 0; t < NCH; ++t) {
          if (on && live[t]) v[u][t].load(xr + (t * G + gl) * VEC);
          else v[u][t].zero();
        }
      }
#pragma unroll
      for (int u = 0; u < U; ++u) {
#pragma unroll
        for (int t = 0; t < NCH; ++t) acc[t].fma(ww[u], v[u][t]);
      }
    }
  }
}

// One group of G lanes per row; rows longer than `threshold` are left to the chunk kernels.
template <int G, int VEC, int NCH, bool HAS_VAL, typename Tin = float, typename Tout = float>
__global__ void __launch_bounds__(256)
spmm_rows_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                 const float *__restrict__ val, int64_t n, const Tin *__restrict__ x, int d, int64_t ldx,
                 Tout *__restrict__ y, int64_t ldy, int norm, int self_loop, const float *__restrict__ dinv,
                 int64_t threshold, int64_t row_offset) {
  constexpr int RPW = 32 / G;
  const int lane = threadIdx.x & 31;
  const int gl = lane % G;
  const int grp = lane / G;
  const unsigned gmask = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (grp * G));
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t row = warp * RPW + grp;
  const int cbase = blockIdx.y * (G * VEC * NCH);
  if (row >= n) return;
  const int64_t s = __ldg(rowptr + row), e = __ldg(rowptr + row + 1);
  if (e - s > threshold) return;

  Vec<VEC> acc[NCH];
#pragma unroll
  for (int t = 0; t < NCH; ++t) acc[t].zero();
  accumulate_range<G, VEC, NCH, HAS_VAL>(acc, s, e, col, val, norm == WDGH_NORM_SYM ? dinv : nullptr, x, ldx,
                                         cbase, d, gl, gmask);
  const int64_t grow = row + row_offset;  // id of this row in the global (column) index space
  const float si = (norm != WDGH_NORM_NONE) ? __ldg(dinv + grow) : 1.f;
  const float self_w = (norm == WDGH_NORM_SYM) ? si : 1.f;
#pragma unroll
  for (int t = 0; t < NCH; ++t) {
    const int c = cbase + (t * G + gl) * VEC;
    if (c < d) {
      if (self_loop) {
        Vec<VEC> xi;
        xi.load(x + grow * ldx + c);
        acc[t].fma(self_w, xi);
      }
      acc[t].scale(si);
      acc[t].store_stream(y + row * ldy + c);
    }
  }
}

// One warp per chunk of a split row: partial[chunk][:] = sum over the chunk's entries (unscaled by s_i).
template <int VEC, int NCH, bool HAS_VAL, typename Tin = float>
__global__ void __launch_bounds__(256)
spmm_chunks_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                   const float *__restrict__ val, const Tin *__restrict__ x, int d, int64_t ldx, int norm,
                   const float *__restrict__ dinv, const int64_t *__restrict__ plan, int64_t n_chunks,
                   float *__restrict__ partial, int64_t ldp) {
  const int lane = threadIdx.x & 31;
  const int64_t chunk = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int cbase = blockIdx.y * (32 * VEC * NCH);
  if (chunk >= n_chunks) return;
  const int64_t cap = plan[kPlanCapacity], T = plan[kPlanThreshold];
  const int64_t k = plan_chunk_owner(plan, cap)[chunk];
  const int64_t row = plan_heavy_row(plan)[k];
  const int64_t part = chunk - plan_heavy_chunk0(plan, cap)[k];
  const int64_t s = __ldg(rowptr + row) + part * T;
  const int64_t e = min(s + T, __ldg(rowptr + row + 1));

  Vec<VEC> acc[NCH];
#pragma unroll
  for (int t = 0; t < NCH; ++t) acc[t].zero();
  accumulate_range<32, VEC, NCH, HAS_VAL>(acc, s, e, col, val, norm == WDGH_NORM_SYM ? dinv : nullptr, x, ldx,
                                          cbase, d, lane, 0xffffffffu);
#pragma unroll
  for (int t = 0; t < NCH; ++t) {
    const int c = cbase + (t * 32 + lane) * VEC;
    if (c < d) acc[t].store(partial + chunk * ldp + c);
  }
}

// Ranged / phased aggregation: the kernel normally walks CSR rows [rowptr[r], rowptr[r+1]); with row_end set it
// walks [rowptr[r], row_end[r]) instead (a column range of every row, e.g. the entries whose source node lives on
// one rank), optionally adding to what Y already holds and deferring the self-loop + D^-1/2 scaling to the last phase.
// ExtraParts lists further raw partial sums of the same rows (local-row indexed like y): `n` parts of one buffer,
// part q starting `part_rows` rows after part q - 1 (the receive slots of the 2-D partition are one [pc][rows][d]
// array).  They enter the row's stream as VIRTUAL trailing entries with weight 1 -- like the self loop -- so they are
// fetched in the same unpredicated gather batches as the feature rows, fully pipelined: the 2-D partition finishes a
// row slice in the launch that aggregates its last column range (or, with an empty range, in a pure streaming
// reduction) -- the partial of the earlier range and the slices the peers stored into this rank's memory ride along,
// no separate reduce pass.  (Adding them when a row is flushed was measured at 4.5 TB/s: every flush stalled on a
// dependent load; as stream entries the phase runs like any other gather pass.)
constexpr int kMaxExtra = 8;
struct ExtraParts {
  int n;                // number of parts
  int64_t ld;           // row stride in floats
  int64_t part_rows;    // rows between consecutive parts
  const float *base;    // part 0, row 0
};
struct RangeArgs {
  const int64_t *row_end;  // nullptr: plain CSR
  const uint8_t *skip;     // nullptr, or 1 for rows that are handled elsewhere (split rows)
  int accumulate;          // y += partial instead of y = partial
  int finalize;            // apply self loop and row scale (0: store the raw partial sum)
  ExtraParts ex;
};

// One CTA per split row: fixed-order sum of its chunk partials, self loop, s_i scaling.
template <typename Tin = float, typename Tout = float>
__global__ void __launch_bounds__(128)
spmm_heavy_finish_kernel(const int64_t *__restrict__ rowptr, const Tin *__restrict__ x, int d, int64_t ldx,
                         Tout *__restrict__ y, int64_t ldy, int norm, int self_loop,
                         const float *__restrict__ dinv, const int64_t *__restrict__ plan,
                         const float *__restrict__ partial, int64_t ldp, int64_t row_offset, int finalize,
                         ExtraParts ex) {
  const int64_t k = blockIdx.x;
  const int64_t cap = plan[kPlanCapacity], T = plan[kPlanThreshold];
  const int64_t row = plan_heavy_row(plan)[k];
  const int64_t c0 = plan_heavy_chunk0(plan, cap)[k];
  const int64_t deg = __ldg(rowptr + row + 1) - __ldg(rowptr + row);
  const int64_t nch = (deg + T - 1) / T;
  const int64_t grow = row + row_offset;
  const float si = (norm != WDGH_NORM_NONE && finalize) ? __ldg(dinv + grow) : 1.f;
  const float self_w = (norm == WDGH_NORM_SYM) ? si : 1.f;
  for (int c = threadIdx.x; c < d; c += blockDim.x) {
    float acc = 0.f;
    for (int64_t p = 0; p < nch; ++p) acc += partial[(c0 + p) * ldp + c];
    for (int q = 0; q < ex.n; ++q) acc += ex.base[(q * ex.part_rows + row) * ex.ld + c];
    if (self_loop && finalize) acc = fmaf(self_w, load1(x + grow * ldx + c), acc);
    store1(y + row * ldy + c, acc * si);  // finalize == 0: the raw partial sum (2-D partition: reduced across ranks later)
  }
}

// ---------------------------------------------------------------------------
// Row-group kernel: the persistent one-warp CTA walks GROUPS of 32 consecutive rows and treats the stored
// entries of a group as one stream.  The gather batches (U feature rows in flight per lane) are cut from the
// stream, not from a row, so short rows no longer mean short batches: a row of 3 entries shares its batch
// with its neighbours, every batch but the last of a group is full and unpredicated.  Row boundaries are
// found on the consuming side (each entry carries its row slot; a change flushes the accumulator).
//   * lane l owns row 32 g + l of the group: bounds, D^-1/2 scale and skip flag are one coalesced load each;
//   * an inclusive warp scan of the row lengths gives the stream offsets (shared memory, double buffered so
//     that the next group's first segment is requested while the current group's last batch is in flight);
//   * each lane finds the row of its stream position with a 5-step search in the offsets;
//   * the self loop is a virtual LAST entry of its row (column = the row itself, weight = s_i): its feature
//     row rides in the gather batches instead of being fetched after them, and the summation order -- stored
//     entries in CSR order, then the self loop -- is the one of the row kernels, so results are bit-identical.
// Split ("heavy") rows contribute no entries and are not stored; the chunk kernels own them.
// ---------------------------------------------------------------------------
template <int VEC, int NCH, bool HAS_VAL, bool FULL, int MINB, bool EXTRA, typename Tin = float,
          typename Tout = float, bool PHASED = true>
__global__ void __launch_bounds__(32, MINB)
spmm_rowgroup_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                     const float *__restrict__ val, int64_t n, const Tin *__restrict__ x, int d, int64_t ldx,
                     Tout *__restrict__ y, int64_t ldy, int norm, int self_loop,
                     const float *__restrict__ dinv, const uint8_t *__restrict__ deg_code, int64_t threshold,
                     int64_t row_offset, RangeArgs ra, unsigned long long *__restrict__ sched) {
  constexpr int TILE = 32 * VEC * NCH;
  constexpr int U0 = 32 / (VEC * NCH);
  // gather batch: feature rows in flight per lane.  Capped at 8: with 16 (the natural value for 64 / 32 columns) the
  // 64-column kernel ran the full graph in 76.3 ms and a short-range phase in 55-65 ms; with 8 it takes 52.8 ms and
  // 20-21 ms (tools/phase_probe.py, profiles/phase_probe_r02.txt)
  constexpr int U = U0 > 8 ? 8 : (U0 < 2 ? 2 : U0);
  constexpr unsigned kFull = 0xffffffffu;
  // PHASED: the phased forms (y +=, raw partial sums) are compiled in; they need fp32 output, a phase never rounds its
  // partial sum.  bf16 features get them only in the instances of wdgh_spmm_csr_ranged_bf16: compiled into the
  // instances of wdgh_spmm_csr_bf16 as well, they made its d = 128 launch slower (64.87 against 64.52 ms on the full
  // graph, same call, non-overlapping spreads).  The extra partial sums ride in the gather batches as rows of x, so they
  // exist for fp32 features only.
  static_assert(!PHASED || std::is_same<Tout, float>::value, "phases store fp32 partial sums");
  static_assert(std::is_same<Tin, float>::value || !EXTRA, "extra partial sums are fp32");
  __shared__ float table[256];
  __shared__ int s_off[2][33];      // stream offset of every row slot of the group (exclusive scan), [32] = total
  __shared__ int64_t s_beg[2][32];  // first stored entry of every row slot
  const int lane = threadIdx.x;
  const bool sym = (norm == WDGH_NORM_SYM);
  const bool coded = sym && deg_code != nullptr;
  const bool virt = self_loop && ra.finalize;  // self loop = virtual trailing entry of its row
  const int n_virt = (virt ? 1 : 0) + (EXTRA ? ra.ex.n : 0);   // ... followed by the extra partial sums of the row
  if (coded) {
    for (int c = lane; c < 256; c += 32) {
      double rs = (double)c + (self_loop ? 1.0 : 0.0);
      if (rs == 0.0) rs = 1.0;
      table[c] = (float)(1.0 / sqrt(rs));  // same expression as degree_scale_kernel -> same bits
    }
    __syncwarp();
  }
  const int cbase = FULL ? 0 : blockIdx.y * TILE;
  bool live[NCH];
#pragma unroll
  for (int t = 0; t < NCH; ++t) live[t] = FULL || (cbase + (t * 32 + lane) * VEC < d);
  const int64_t W = gridDim.x;
  const int64_t n_groups = (n + 31) >> 5;
  const int ld32 = (int)ldx;
  const Tin *xl = x + cbase + lane * VEC;

  auto load_bounds = [&](int64_t g, int64_t &b, int64_t &e, int &flag) {
    b = 0;
    e = 0;
    flag = 0;
    const int64_t r = (g << 5) + lane;
    if (r < n) {
      b = __ldg(rowptr + r);
      e = ra.row_end ? __ldg(ra.row_end + r) : __ldg(rowptr + r + 1);
      if (ra.skip) flag = __ldg(ra.skip + r);
    }
  };
  // scan the row lengths of group g into s_off[buf] / s_beg[buf]
  auto publish = [&](int buf, int64_t g, int64_t b, int64_t e, int flag, unsigned &nostore, int &total, float &si) {
    const int64_t r = (g << 5) + lane;
    const bool inr = r < n;
    const bool hv = inr && (flag != 0 || e - b > threshold);
    int inc = (!inr || hv) ? 0 : (int)(e - b) + n_virt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(kFull, inc, o);
      if (lane >= o) inc += v;
    }
    s_off[buf][lane + 1] = inc;
    if (lane == 0) s_off[buf][0] = 0;
    s_beg[buf][lane] = b;
    nostore = __ballot_sync(kFull, !inr || hv);
    total = __shfl_sync(kFull, inc, 31);
    si = (norm != WDGH_NORM_NONE && ra.finalize && inr) ? __ldg(dinv + r + row_offset) : 1.f;
    if (PHASED && FULL && ra.accumulate && inr && !hv && (e > b || ra.finalize)) {
      // `y +=` phase: flush_row reads the row's earlier partial sum right before it stores -- a dependent HBM round
      // trip per row, 32 in a row per group.  Ask for the lines one group ahead so that the read is an L2 hit
      // (measured on the 16-phase e2e schedule at 64 columns: 59 -> 56 ms per phase).
      const Tout *yp = y + r * ldy;
#pragma unroll
      for (int c0 = 0; c0 < TILE; c0 += 32) asm volatile("prefetch.global.L2 [%0];" ::"l"(yp + c0));
    }
    __syncwarp();
  };
  // column id, weight and row slot of stream position t0 + lane of group g
  auto load_seg = [&](int buf, int64_t g, int t0, int total, int &j, float &w, int &rho) {
    j = 0;
    w = 0.f;
    rho = 0;
    const int t = t0 + lane;
    if (t < total) {
      int lo = 0;
#pragma unroll
      for (int step = 16; step >= 1; step >>= 1)
        if (s_off[buf][lo + step] <= t) lo += step;
      rho = lo;
      const int k = t - s_off[buf][lo];
      const int real = s_off[buf][lo + 1] - s_off[buf][lo] - n_virt;   // stored entries of this row in the stream
      if (k >= real) {
        const int q = k - real;
        if (virt && q == 0) {   // the self loop
          const int64_t grow = (g << 5) + lo + row_offset;
          j = (int)grow;
          w = sym ? __ldg(dinv + grow) : 1.f;
        } else {                // part q' of the extra partial sums: row index inside the parts buffer, top bit set
          const int64_t part = q - (virt ? 1 : 0);
          j = (int)(0x80000000u | (unsigned)(part * ra.ex.part_rows + (g << 5) + lo));
          w = 1.f;
        }
      } else {
        const int64_t idx = s_beg[buf][lo] + k;
        j = __ldg(col + idx);
        w = HAS_VAL ? __ldg(val + idx) : 1.f;
        if (coded) {
          const int c = __ldg(deg_code + j);
          w *= (c < 255) ? table[c] : __ldg(dinv + j);
        } else if (sym) {
          w *= __ldg(dinv + j);
        }
      }
    }
  };
  // address of the feature (or extra partial) row a stream entry gathers
  const float *el = EXTRA ? ra.ex.base + cbase + lane * VEC : nullptr;
  const int lde32 = EXTRA ? (int)ra.ex.ld : 0;
  auto row_ptr = [&](int ju) -> const Tin * {
    if constexpr (EXTRA) {
      if (ju < 0) return el + (int64_t)(ju & 0x7fffffff) * lde32;
    }
    return xl + (int64_t)ju * ld32;
  };

  // group order: a ticket counter (FULL: one column tile) -- row lengths are heavy-tailed, with tickets a warp
  // that drew long rows simply takes fewer groups -- or a static stride W when several column tiles share the rows
  auto take = [&](int64_t prev) -> int64_t {
    if (!FULL) return prev + W;
    unsigned long long t = 0;
    if (lane == 0) t = atomicAdd(&sched[0], 1ull);
    return (int64_t)__shfl_sync(kFull, t, 0) + W;  // tickets start after the W groups handed out by blockIdx
  };
  int64_t g = blockIdx.x;  // the grid never exceeds the number of groups
  int64_t b, e;
  int flag;
  load_bounds(g, b, e, flag);
  int buf = 0;
  unsigned nostore, n_nostore = kFull;
  int total, n_total = 0;
  float si_l, n_si = 1.f;
  publish(0, g, b, e, flag, nostore, total, si_l);
  int64_t gn = take(g);
  int64_t gnn = 0;
  load_bounds(gn, b, e, flag);  // the next group's bounds travel while this group is aggregated
  int j, rho, nj = 0, nrho = 0;
  float w, nw = 0.f;
  load_seg(0, g, 0, total, j, w, rho);
  Vec<VEC> acc[NCH];
#pragma unroll
  for (int t = 0; t < NCH; ++t) acc[t].zero();

  // store row slot `cur` of the current group (accumulator -> y) and clear the accumulator
  auto flush_row = [&](int cur) {
    if (!((nostore >> cur) & 1u)) {
      const int64_t row = (g << 5) + cur;
      const float si = __shfl_sync(kFull, si_l, cur);
      const bool had = s_off[buf][cur + 1] != s_off[buf][cur];
      if (had || ra.finalize || !ra.accumulate) {  // an empty range adds nothing to an earlier phase's sum
#pragma unroll
        for (int t = 0; t < NCH; ++t) {
          if (live[t]) {
            const int c = cbase + (t * 32 + lane) * VEC;
            if constexpr (PHASED) {
              if (ra.accumulate) {
                Vec<VEC> prev;
                prev.load_plain(y + row * ldy + c);
                acc[t].add(prev);
              }
              if (ra.finalize) {
                acc[t].scale(si);
                acc[t].store_stream(y + row * ldy + c);
              } else {
                acc[t].store(y + row * ldy + c);
              }
            } else {
              acc[t].scale(si);
              acc[t].store_stream(y + row * ldy + c);
            }
          }
        }
      }
    }
#pragma unroll
    for (int t = 0; t < NCH; ++t) acc[t].zero();
  };

  while (true) {
    int cur = 0;
    auto prefetch = [&](int t0, bool last_seg) {
      if (!last_seg) {
        load_seg(buf, g, t0 + 32, total, nj, nw, nrho);
      } else {  // next group: offsets, first segment, and the bounds of the group after it
        publish(buf ^ 1, gn, b, e, flag, n_nostore, n_total, n_si);
        load_seg(buf ^ 1, gn, 0, n_total, nj, nw, nrho);
        gnn = take(gn);
        load_bounds(gnn, b, e, flag);
      }
    };
    // (a group without entries still makes one pass with cnt = 0: every gather predicated off, nothing consumed -- it
    // is what fetches the next group, so that the prefetch code exists once)
    for (int t0 = 0; t0 < total || t0 == 0; t0 += 32) {
      const int cnt = min(32, total - t0);
      const bool last_seg = t0 + 32 >= total;
      bool next_issued = false;
      // One batch loop: the gathers come in two flavours -- every batch but the last of a segment is full and issues
      // U unpredicated loads -- but the prefetch of the next segment / group and the consuming side (row flush + fma)
      // exist ONCE.  (They used to be duplicated for the predicated last batch: the kernel was 4096 SASS instructions,
      // and a launch over short row ranges, which runs the whole body once per group, was instruction-fetch bound:
      // 78% of its stall samples, profiles/summary_r02.md.)
#pragma unroll 1
      for (int k = 0; k < cnt || k == 0; k += U) {
        Vec<VEC> v[U][NCH];
        if (k + U <= cnt) {
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const Tin *xr = row_ptr(__shfl_sync(kFull, j, k + u));
#pragma unroll
            for (int t = 0; t < NCH; ++t) {
              if (live[t]) v[u][t].load(xr + t * (32 * VEC));
              else v[u][t].zero();
            }
          }
        } else {
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const bool on = k + u < cnt;
            const Tin *xr = row_ptr(__shfl_sync(kFull, j, on ? k + u : 0));
#pragma unroll
            for (int t = 0; t < NCH; ++t) {
              if (on && live[t]) v[u][t].load(xr + t * (32 * VEC));
              else v[u][t].zero();
            }
          }
        }
        if (!next_issued) {
          prefetch(t0, last_seg);
          next_issued = true;
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          if (k + u < cnt) {  // warp-uniform
            const int ru = __shfl_sync(kFull, rho, k + u);
            while (cur < ru) flush_row(cur++);
            const float wu = __shfl_sync(kFull, w, k + u);
#pragma unroll
            for (int t = 0; t < NCH; ++t) acc[t].fma(wu, v[u][t]);
          }
        }
      }
      j = nj; w = nw; rho = nrho;
    }
    while (cur < 32) flush_row(cur++);
    g = gn;
    gn = gnn;
    buf ^= 1;
    nostore = n_nostore; total = n_total; si_l = n_si;
    if (g >= n_groups) break;
  }
  if (FULL) sched_retire(sched, gridDim.x);  // the last CTA re-arms the ticket counter for the next launch
}

struct SpmmArgs {
  const int64_t *rowptr;
  const int32_t *col;
  const float *val;
  int64_t n;
  const void *x;  // float, bf16 or f16 (the Tin of the launch)
  int d;
  int64_t ldx;
  void *y;        // float, or Tin when it is a half type (Tout)
  int64_t ldy;
  int norm, self_loop;
  const float *dinv;
  const uint8_t *deg_code;
  int64_t *plan;
  int64_t threshold, n_heavy, n_chunks, row_offset;
  RangeArgs ra = {nullptr, nullptr, 0, 1, {0, 0, 0, nullptr}};
  int cta_limit = 0;       // row-group kernel: CTAs per SM (0 = the default for the tile shape)
  bool heavy_pass = true;  // run the split-row chunk kernels
  float *partial;
  int64_t ldp;
  cudaStream_t st;
};

// Plain row kernel (any width / alignment): one-warp CTAs keep warp slots busy when row lengths are skewed (a CTA's
// slots are only recycled when its longest row finishes; measured on the 1B-entry graph: 256 threads 123.8 ms,
// 128 -> 114.7, 64 -> 112.4, 32 -> 111.3).
template <int G, int VEC, int NCH, bool HAS_VAL, typename Tin, typename Tout>
static int launch_rows(const SpmmArgs &a) {
  constexpr int RPW = 32 / G;
  const int tile = G * VEC * NCH;
  dim3 grid((unsigned)ceil_div(a.n, RPW), (unsigned)ceil_div(a.d, tile));
  spmm_rows_kernel<G, VEC, NCH, HAS_VAL, Tin, Tout><<<grid, 32, 0, a.st>>>(
      a.rowptr, a.col, a.val, a.n, static_cast<const Tin *>(a.x), a.d, a.ldx, static_cast<Tout *>(a.y), a.ldy, a.norm,
      a.self_loop, a.dinv, a.threshold, a.row_offset);
  WDGH_LAUNCHED("spmm_rows_kernel");
  return 0;
}

// split rows: one warp per chunk, then one CTA per row (fixed-order sum, extras, self loop, scale)
template <int VEC, int NCH, bool HAS_VAL, typename Tin = float, typename Tout = float>
static int launch_heavy(const SpmmArgs &a, const ExtraParts &ex) {
  if (a.n_chunks == 0) return 0;
  const int tile = 32 * VEC * NCH;
  const Tin *x = static_cast<const Tin *>(a.x);
  dim3 grid((unsigned)ceil_div(a.n_chunks, 8), (unsigned)ceil_div(a.d, tile));
  spmm_chunks_kernel<VEC, NCH, HAS_VAL, Tin><<<grid, 256, 0, a.st>>>(a.rowptr, a.col, a.val, x, a.d, a.ldx, a.norm,
                                                                    a.dinv, a.plan, a.n_chunks, a.partial, a.ldp);
  WDGH_LAUNCHED("spmm_chunks_kernel");
  spmm_heavy_finish_kernel<Tin, Tout><<<(unsigned)a.n_heavy, 128, 0, a.st>>>(
      a.rowptr, x, a.d, a.ldx, static_cast<Tout *>(a.y), a.ldy, a.norm, a.self_loop, a.dinv, a.plan, a.partial, a.ldp,
      a.row_offset, a.ra.finalize, ex);
  WDGH_LAUNCHED("spmm_heavy_finish_kernel");
  return 0;
}

// Row-group kernel: persistent grid of one-warp CTAs, 32 per SM for a single 128-column tile (measured on the
// 1B-entry graph, d = 128: 16 CTAs/SM 118.1 ms, 24 -> 100.4, 32 -> 95.6), 16 per SM for the wider tiles.
template <int VEC, int NCH, bool HAS_VAL, typename Tin, typename Tout, bool PHASED>
static int launch_rowgroup(const SpmmArgs &a) {
  constexpr int TILE = 32 * VEC * NCH;
  constexpr int MINB = (NCH == 1) ? 32 : 16;
  const int64_t n_groups = (a.n + 31) / 32;
  const int per_sm = (a.cta_limit > 0 && a.cta_limit < MINB) ? a.cta_limit : MINB;
  int64_t ctas = (int64_t)sm_count() * per_sm;
  if (ctas > n_groups) ctas = n_groups;
  dim3 grid((unsigned)ctas, (unsigned)ceil_div(a.d, TILE));
  const bool full = (a.d == TILE);
  unsigned long long *sched = plan_sched(a.plan, kPlanSpmmTicket);
#define WDGH_RG_LAUNCH(FULLV, MINBV, EXTRAV)                                                                        \
  spmm_rowgroup_kernel<VEC, NCH, HAS_VAL, FULLV, MINBV, EXTRAV, Tin, Tout, PHASED><<<grid, 32, 0, a.st>>>(            \
      a.rowptr, a.col, a.val, a.n, static_cast<const Tin *>(a.x), a.d, a.ldx, static_cast<Tout *>(a.y), a.ldy, a.norm, \
      a.self_loop, a.dinv, a.deg_code, a.threshold, a.row_offset, a.ra, sched)
  constexpr bool F32 = std::is_same<Tin, float>::value && std::is_same<Tout, float>::value;
  if (F32 && a.ra.ex.n > 0) {  // (the bf16 entry has no extra partial sums)
    if (VEC != 4) return fail(WDGH_EINVAL, "wdgh_spmm_csr_ranged: extra partial sums need d >= 128");
    if (full) WDGH_RG_LAUNCH(true, MINB, (F32 && VEC == 4));
    else WDGH_RG_LAUNCH(false, 16, (F32 && VEC == 4));
  } else if (full) {
    WDGH_RG_LAUNCH(true, MINB, false);
  } else {
    WDGH_RG_LAUNCH(false, 16, false);
  }
#undef WDGH_RG_LAUNCH
  WDGH_LAUNCHED("spmm_rowgroup_kernel");
  return 0;
}

static bool rowgroup_width(int64_t d) { return d >= 128 || d == 64 || d == 32; }

// PHASED: the row-group instances carry the phased forms (the ranged entries, and every fp32 launch)
template <bool HAS_VAL, typename Tin, typename Tout, bool PHASED>
static int dispatch(const SpmmArgs &a, bool vec4) {
  int rc;
  const int d = a.d;
  const ExtraParts none = {0, 0, 0, nullptr};
  if (vec4 && rowgroup_width(d)) {
    if (d == 32) rc = launch_rowgroup<1, 1, HAS_VAL, Tin, Tout, PHASED>(a);
    else if (d == 64) rc = launch_rowgroup<2, 1, HAS_VAL, Tin, Tout, PHASED>(a);
    else if (d <= 128) rc = launch_rowgroup<4, 1, HAS_VAL, Tin, Tout, PHASED>(a);
    else if (d <= 256) rc = launch_rowgroup<4, 2, HAS_VAL, Tin, Tout, PHASED>(a);
    else rc = launch_rowgroup<4, 4, HAS_VAL, Tin, Tout, PHASED>(a);
    if (rc || !a.heavy_pass) return rc;
    if (d <= 128) return launch_heavy<4, 1, HAS_VAL, Tin, Tout>(a, none);
    if (d <= 256) return launch_heavy<4, 2, HAS_VAL, Tin, Tout>(a, none);
    return launch_heavy<4, 4, HAS_VAL, Tin, Tout>(a, none);
  }
  if (vec4) {
    if (d <= 4) rc = launch_rows<1, 4, 1, HAS_VAL, Tin, Tout>(a);
    else if (d <= 8) rc = launch_rows<2, 4, 1, HAS_VAL, Tin, Tout>(a);
    else if (d <= 16) rc = launch_rows<4, 4, 1, HAS_VAL, Tin, Tout>(a);
    else if (d <= 32) rc = launch_rows<8, 4, 1, HAS_VAL, Tin, Tout>(a);
    else if (d <= 64) rc = launch_rows<16, 4, 1, HAS_VAL, Tin, Tout>(a);
    else rc = launch_rows<32, 4, 1, HAS_VAL, Tin, Tout>(a);
    if (rc) return rc;
    return launch_heavy<4, 1, HAS_VAL, Tin, Tout>(a, none);
  }
  if (d <= 1) rc = launch_rows<1, 1, 1, HAS_VAL, Tin, Tout>(a);
  else if (d <= 2) rc = launch_rows<2, 1, 1, HAS_VAL, Tin, Tout>(a);
  else if (d <= 4) rc = launch_rows<4, 1, 1, HAS_VAL, Tin, Tout>(a);
  else if (d <= 8) rc = launch_rows<8, 1, 1, HAS_VAL, Tin, Tout>(a);
  else if (d <= 16) rc = launch_rows<16, 1, 1, HAS_VAL, Tin, Tout>(a);
  else if (d <= 32) rc = launch_rows<32, 1, 1, HAS_VAL, Tin, Tout>(a);
  else if (d <= 64) rc = launch_rows<32, 1, 2, HAS_VAL, Tin, Tout>(a);
  else rc = launch_rows<32, 1, 4, HAS_VAL, Tin, Tout>(a);
  if (rc) return rc;
  if (d <= 32) return launch_heavy<1, 1, HAS_VAL, Tin, Tout>(a, none);
  if (d <= 64) return launch_heavy<1, 2, HAS_VAL, Tin, Tout>(a, none);
  return launch_heavy<1, 4, HAS_VAL, Tin, Tout>(a, none);
}

// every row of x / y starts on a 4-element boundary (16 bytes for fp32, 8 for bf16 / f16)
template <typename Tin, typename Tout>
static bool rows_vec4(const Tin *x, int64_t d, int64_t ldx, const Tout *y, int64_t ldy, const float *partial) {
  return (d % 4 == 0) && (ldx % 4 == 0) && (ldy % 4 == 0) && (reinterpret_cast<uintptr_t>(x) % (4 * sizeof(Tin)) == 0) &&
         (reinterpret_cast<uintptr_t>(y) % (4 * sizeof(Tout)) == 0) &&
         (partial == nullptr || reinterpret_cast<uintptr_t>(partial) % 16 == 0);
}

}  // namespace wdgh

using namespace wdgh;

namespace wdgh {
// argument checks and dispatch shared by wdgh_spmm_csr (Tin = float), wdgh_spmm_csr_bf16 and wdgh_spmm_csr_f16; `fn`
// names the entry in the error messages
#define WDGH_REQUIRE_AT(cond, what)                                      \
  do {                                                                   \
    if (!(cond)) {                                                       \
      snprintf(g_err, sizeof(g_err), "%s: %s", fn, what);                \
      return WDGH_EINVAL;                                                \
    }                                                                    \
  } while (0)
template <typename Tin>
static int spmm_csr(const char *fn, const int64_t *rowptr, const int32_t *col, const float *val, int64_t n,
                    const Tin *x, int64_t d, int64_t ldx, void *y, int64_t ldy, int y_dtype, int norm,
                    int add_self_loop, const float *dinv, const uint8_t *deg_code, int64_t *plan_i64,
                    const int64_t *plan_host, float *partial, int64_t row_offset, void *stream) {
  WDGH_REQUIRE_AT(rowptr && x && y && plan_i64 && plan_host, "null pointer");  // col may be NULL iff nnz == 0
  WDGH_REQUIRE_AT(n >= 0 && d > 0 && d <= (1 << 24) && ldx >= d && ldy >= d, "bad shape");
  WDGH_REQUIRE_AT(norm == WDGH_NORM_NONE || norm == WDGH_NORM_RW || norm == WDGH_NORM_SYM, "bad norm");
  WDGH_REQUIRE_AT(norm == WDGH_NORM_NONE || dinv != nullptr, "norm requires dinv");
  WDGH_REQUIRE_AT(static_cast<const void *>(x) != y, "in-place aggregation is not supported");
  WDGH_REQUIRE_AT(row_offset >= 0, "negative row_offset");
  WDGH_REQUIRE_AT(y_dtype == WDGH_DTYPE_F32 || y_dtype == kHalfY<Tin>, "bad y_dtype (float32, or the type of x)");
  if (n == 0) return 0;
  SpmmArgs a;
  a.rowptr = rowptr; a.col = col; a.val = val; a.n = n; a.x = x; a.d = (int)d; a.ldx = ldx; a.y = y; a.ldy = ldy;
  a.norm = norm; a.self_loop = add_self_loop ? 1 : 0; a.dinv = dinv; a.deg_code = (val == nullptr) ? deg_code : nullptr; a.plan = plan_i64;
  a.n_heavy = plan_host[0]; a.n_chunks = plan_host[1]; a.threshold = plan_host[2];
  a.partial = partial; a.ldp = (d + 3) & ~int64_t(3);
  a.row_offset = row_offset;
  a.st = as_stream(stream);
  WDGH_REQUIRE_AT(a.n_chunks == 0 || partial != nullptr, "split rows need the partial buffer");
  if constexpr (!std::is_same<Tin, float>::value) {  // (fp32 features have fp32 output only)
    if (y_dtype == kHalfY<Tin>) {
      const bool vec4 = rows_vec4(x, d, ldx, static_cast<const Tin *>(y), ldy, partial);
      return val ? dispatch<true, Tin, Tin, false>(a, vec4) : dispatch<false, Tin, Tin, false>(a, vec4);
    }
  }
  const bool vec4 = rows_vec4(x, d, ldx, static_cast<const float *>(y), ldy, partial);
  constexpr bool F32 = std::is_same<Tin, float>::value;
  return val ? dispatch<true, Tin, float, F32>(a, vec4) : dispatch<false, Tin, float, F32>(a, vec4);
}
}  // namespace wdgh

extern "C" int wdgh_spmm_csr(const int64_t *rowptr, const int32_t *col, const float *val, int64_t n,
                             const float *x, int64_t d, int64_t ldx, float *y, int64_t ldy, int norm,
                             int add_self_loop, const float *dinv, const uint8_t *deg_code, int64_t *plan_i64,
                             const int64_t *plan_host, float *partial, int64_t row_offset, void *stream) {
  return spmm_csr("wdgh_spmm_csr", rowptr, col, val, n, x, d, ldx, y, ldy, WDGH_DTYPE_F32, norm, add_self_loop, dinv,
                  deg_code, plan_i64, plan_host, partial, row_offset, stream);
}

extern "C" int wdgh_spmm_csr_bf16(const int64_t *rowptr, const int32_t *col, const float *val, int64_t n,
                                  const uint16_t *x, int64_t d, int64_t ldx, void *y, int64_t ldy, int y_dtype,
                                  int norm, int add_self_loop, const float *dinv, const uint8_t *deg_code,
                                  int64_t *plan_i64, const int64_t *plan_host, float *partial, int64_t row_offset,
                                  void *stream) {
  return spmm_csr("wdgh_spmm_csr_bf16", rowptr, col, val, n, reinterpret_cast<const bf16 *>(x), d, ldx, y, ldy, y_dtype,
                  norm, add_self_loop, dinv, deg_code, plan_i64, plan_host, partial, row_offset, stream);
}

extern "C" int wdgh_spmm_csr_f16(const int64_t *rowptr, const int32_t *col, const float *val, int64_t n,
                                 const uint16_t *x, int64_t d, int64_t ldx, void *y, int64_t ldy, int y_dtype, int norm,
                                 int add_self_loop, const float *dinv, const uint8_t *deg_code, int64_t *plan_i64,
                                 const int64_t *plan_host, float *partial, int64_t row_offset, void *stream) {
  return spmm_csr("wdgh_spmm_csr_f16", rowptr, col, val, n, reinterpret_cast<const f16 *>(x), d, ldx, y, ldy, y_dtype,
                  norm, add_self_loop, dinv, deg_code, plan_i64, plan_host, partial, row_offset, stream);
}

extern "C" int wdgh_structure_counts(const int64_t *, const int32_t *, int64_t, int64_t, const int32_t *, int32_t,
                                     int64_t *, const int64_t *, int64_t *, double *, int32_t *, int32_t *,
                                     uint8_t *, int64_t, int64_t, void *);

// The aggregation and the label pass back to back on one stream.  Folding the per-entry label work into the
// aggregation kernel was measured twice (round 1: 111.3 vs 105.9 ms per step on the 1B-entry graph) and costs more
// than the separate pass: the gather kernel sits at the HBM roofline and is issue- and register-bound at 64
// registers / thread, so the single-kernel form was removed.
extern "C" int wdgh_spmm_structure_fused(const int64_t *rowptr, const int32_t *col, int64_t n, int64_t nnz,
                                         const float *x, int64_t d, int64_t ldx, float *y, int64_t ldy, int norm,
                                         int add_self_loop, const float *dinv, const uint8_t *deg_code,
                                         const int32_t *labels, int32_t num_classes, int64_t *plan_i64,
                                         const int64_t *plan_host, float *partial, int64_t *counters, double *node_sum,
                                         int32_t *deg_nsl, int32_t *match_nsl, uint8_t *labels_u8_scratch,
                                         int64_t n_labels, int64_t row_offset, void *stream) {
  WDGH_REQUIRE(rowptr && x && y && labels && plan_i64 && plan_host && counters && node_sum && deg_nsl && match_nsl,
               "wdgh_spmm_structure_fused: null pointer");
  int rc = wdgh_spmm_csr(rowptr, col, nullptr, n, x, d, ldx, y, ldy, norm, add_self_loop, dinv, deg_code, plan_i64,
                         plan_host, partial, row_offset, stream);
  if (rc) return rc;
  return wdgh_structure_counts(rowptr, col, n, nnz, labels, num_classes, plan_i64, plan_host, counters, node_sum,
                               deg_nsl, match_nsl, labels_u8_scratch, n_labels, row_offset, stream);
}

// ---------------------------------------------------------------------------
// Ranged / phased aggregation (multi-GPU overlap, host-buffer pipeline): see RangeArgs.
// ---------------------------------------------------------------------------
namespace wdgh {
__global__ void column_segments_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col, int64_t n,
                                       const int64_t *__restrict__ bounds, int nb, int64_t *__restrict__ seg) {
  // seg[b][r] = first entry of row r whose column is >= bounds[b]   (thread per row, binary search per boundary)
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; r < n; r += stride) {
    const int64_t s = rowptr[r], e = rowptr[r + 1];
    for (int b = 0; b < nb; ++b) {
      const int64_t key = bounds[b];
      int64_t lo = s, hi = e;
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if ((int64_t)col[mid] < key) lo = mid + 1;
        else hi = mid;
      }
      seg[(int64_t)b * n + r] = lo;
    }
  }
}
__global__ void heavy_flags_kernel(const int64_t *__restrict__ plan, uint8_t *__restrict__ flags) {
  const int64_t n_heavy = plan[kPlanNHeavy];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_heavy; k += stride)
    flags[plan_heavy_row(plan)[k]] = 1;
}
}  // namespace wdgh

extern "C" int wdgh_column_segments(const int64_t *rowptr, const int32_t *col, int64_t n, const int64_t *bounds_dev,
                                    int32_t num_bounds, int64_t *seg, void *stream) {
  WDGH_REQUIRE(rowptr && bounds_dev && seg && n >= 0 && num_bounds >= 1, "wdgh_column_segments: bad arguments");
  if (n == 0) return 0;
  column_segments_kernel<<<persistent_grid(ceil_div(n, 256), 8), 256, 0, as_stream(stream)>>>(rowptr, col, n, bounds_dev,
                                                                                            num_bounds, seg);
  WDGH_LAUNCHED("column_segments_kernel");
  return 0;
}

extern "C" int wdgh_plan_heavy_flags(const int64_t *plan_i64, const int64_t *plan_host, int64_t n, uint8_t *flags,
                                     void *stream) {
  WDGH_REQUIRE(plan_i64 && plan_host && flags && n >= 0, "wdgh_plan_heavy_flags: bad arguments");
  cudaStream_t st = as_stream(stream);
  WDGH_CUDA(cudaMemsetAsync(flags, 0, (size_t)n, st));
  if (plan_host[0] > 0) {
    heavy_flags_kernel<<<persistent_grid(ceil_div(plan_host[0], 256), 4), 256, 0, st>>>(plan_i64, flags);
    WDGH_LAUNCHED("heavy_flags_kernel");
  }
  return 0;
}

namespace wdgh {
// fp32 -> H (bf16 or f16) of a strided block, round to nearest even (the rounding of the streaming stores): one warp
// per row
template <typename H>
__global__ void round_half_kernel(const float *__restrict__ x, int64_t rows, int64_t cols, int64_t ldx,
                                  H *__restrict__ y, int64_t ldy, int pairs) {
  const int lane = threadIdx.x & 31;
  const int64_t warps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  for (int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < rows; r += warps) {
    const float *xr = x + r * ldx;
    H *yr = y + r * ldy;
    if (pairs) {
      for (int64_t c = 2 * lane; c < cols; c += 64) {
        const float2 v = *reinterpret_cast<const float2 *>(xr + c);
        *reinterpret_cast<unsigned *>(yr + c) = Half<H>::round2(v.x, v.y);
      }
    } else {
      for (int64_t c = lane; c < cols; c += 32) yr[c] = Half<H>::round1(xr[c]);
    }
  }
}

template <typename H>
int round_to_half(const float *x, int64_t rows, int64_t cols, int64_t ldx, void *y, int64_t ldy, cudaStream_t st) {
  if (rows == 0) return 0;
  const int pairs = (cols % 2 == 0) && (ldx % 2 == 0) && (ldy % 2 == 0) && (reinterpret_cast<uintptr_t>(x) % 8 == 0) &&
                    (reinterpret_cast<uintptr_t>(y) % 4 == 0);
  round_half_kernel<H><<<persistent_grid(ceil_div(rows, 8), 8), 256, 0, st>>>(x, rows, cols, ldx, static_cast<H *>(y),
                                                                             ldy, pairs);
  WDGH_LAUNCHED("round_half_kernel");
  return 0;
}
template int round_to_half<bf16>(const float *, int64_t, int64_t, int64_t, void *, int64_t, cudaStream_t);
template int round_to_half<f16>(const float *, int64_t, int64_t, int64_t, void *, int64_t, cudaStream_t);

// argument checks and dispatch shared by wdgh_spmm_csr_ranged (Tin = float), wdgh_spmm_csr_ranged_bf16 and
// wdgh_spmm_csr_ranged_f16 (no extra partial sums, n_extra = 0)
template <typename Tin>
static int spmm_ranged(const char *fn, const int64_t *rowptr, const int64_t *range_begin, const int64_t *range_end,
                       const int32_t *col, const float *val, int64_t n, const Tin *x, int64_t d, int64_t ldx, float *y,
                       int64_t ldy, int norm, int add_self_loop, const float *dinv, const uint8_t *deg_code,
                       const uint8_t *skip_rows, int accumulate, int finalize, int run_split_rows,
                       const float *extra_parts, int32_t n_extra, int32_t n_extra_split, int64_t extra_part_rows,
                       int64_t ld_extra, int32_t ctas_per_sm, int64_t *plan_i64, const int64_t *plan_host,
                       float *partial, int64_t row_offset, void *stream) {
  WDGH_REQUIRE_AT(rowptr && range_begin && range_end && x && y && plan_i64 && plan_host, "null pointer");
  WDGH_REQUIRE_AT(n >= 0 && d > 0 && ldx >= d && ldy >= d, "bad shape");
  WDGH_REQUIRE_AT(norm == WDGH_NORM_NONE || dinv != nullptr, "norm requires dinv");
  WDGH_REQUIRE_AT(rows_vec4(x, d, ldx, y, ldy, partial) && rowgroup_width(d),
                  sizeof(Tin) == 4 ? "needs 16-byte aligned rows and d in {32, 64} or d >= 128"
                                   : "needs 8-byte aligned rows (d, ldx multiples of 4) and d in {32, 64} or d >= 128");
  WDGH_REQUIRE_AT(plan_host[1] == 0 || skip_rows != nullptr, "split rows need skip_rows (wdgh_plan_heavy_flags)");
  WDGH_REQUIRE_AT(n_extra >= 0 && n_extra <= kMaxExtra && n_extra_split >= 0 && n_extra_split <= n_extra &&
                      (n_extra == 0 || (extra_parts != nullptr && ld_extra >= d && ld_extra % 4 == 0 && d >= 128 &&
                                        extra_part_rows >= n && reinterpret_cast<uintptr_t>(extra_parts) % 16 == 0 &&
                                        (int64_t)n_extra * extra_part_rows < ((int64_t)1 << 31))),
                  "bad extra partial sums");
  WDGH_REQUIRE_AT(ctas_per_sm >= 0, "bad ctas_per_sm");
  if (n == 0) return 0;
  SpmmArgs a;
  a.rowptr = range_begin; a.col = col; a.val = val; a.n = n; a.x = x; a.d = (int)d; a.ldx = ldx; a.y = y; a.ldy = ldy;
  a.norm = norm; a.self_loop = add_self_loop ? 1 : 0; a.dinv = dinv; a.deg_code = (val == nullptr) ? deg_code : nullptr;
  a.plan = plan_i64;
  a.n_heavy = plan_host[0]; a.n_chunks = plan_host[1]; a.threshold = INT64_MAX / 4;  // ranges are never "heavy" by length
  a.partial = partial; a.ldp = (d + 3) & ~int64_t(3);
  a.row_offset = row_offset;
  a.st = as_stream(stream);
  a.ra.row_end = range_end; a.ra.skip = skip_rows; a.ra.accumulate = accumulate ? 1 : 0; a.ra.finalize = finalize ? 1 : 0;
  a.ra.ex = ExtraParts{n_extra, ld_extra, extra_part_rows, extra_parts};
  a.cta_limit = ctas_per_sm;
  a.heavy_pass = false;
  int rc = val ? dispatch<true, Tin, float, true>(a, true) : dispatch<false, Tin, float, true>(a, true);
  if (rc || !run_split_rows || a.n_chunks == 0) return rc;
  // split rows: always over their full column range, after the last phase (they overwrite their Y rows); of the
  // extra partial sums only the LAST n_extra_split apply (an earlier phase of this rank never stored split rows)
  WDGH_REQUIRE_AT(partial != nullptr, "split rows need the partial buffer");
  ExtraParts ex = {n_extra_split, ld_extra, extra_part_rows,
                   n_extra ? extra_parts + (int64_t)(n_extra - n_extra_split) * extra_part_rows * ld_extra : nullptr};
  a.rowptr = rowptr; a.threshold = plan_host[2];
  a.ra = RangeArgs{nullptr, nullptr, 0, finalize ? 1 : 0, {0, 0, 0, nullptr}};
  if (val) {
    if (d <= 128) return launch_heavy<4, 1, true, Tin>(a, ex);
    if (d <= 256) return launch_heavy<4, 2, true, Tin>(a, ex);
    return launch_heavy<4, 4, true, Tin>(a, ex);
  }
  if (d <= 128) return launch_heavy<4, 1, false, Tin>(a, ex);
  if (d <= 256) return launch_heavy<4, 2, false, Tin>(a, ex);
  return launch_heavy<4, 4, false, Tin>(a, ex);
}
#undef WDGH_REQUIRE_AT
}  // namespace wdgh

extern "C" int wdgh_spmm_csr_ranged(const int64_t *rowptr, const int64_t *range_begin, const int64_t *range_end,
                                    const int32_t *col, const float *val, int64_t n, const float *x, int64_t d,
                                    int64_t ldx, float *y, int64_t ldy, int norm, int add_self_loop,
                                    const float *dinv, const uint8_t *deg_code, const uint8_t *skip_rows,
                                    int accumulate, int finalize, int run_split_rows,
                                    const float *extra_parts, int32_t n_extra, int32_t n_extra_split,
                                    int64_t extra_part_rows, int64_t ld_extra, int32_t ctas_per_sm, int64_t *plan_i64,
                                    const int64_t *plan_host, float *partial, int64_t row_offset, void *stream) {
  return spmm_ranged("wdgh_spmm_csr_ranged", rowptr, range_begin, range_end, col, val, n, x, d, ldx, y, ldy, norm,
                     add_self_loop, dinv, deg_code, skip_rows, accumulate, finalize, run_split_rows, extra_parts,
                     n_extra, n_extra_split, extra_part_rows, ld_extra, ctas_per_sm, plan_i64, plan_host, partial,
                     row_offset, stream);
}

extern "C" int wdgh_spmm_csr_ranged_bf16(const int64_t *rowptr, const int64_t *range_begin, const int64_t *range_end,
                                         const int32_t *col, const float *val, int64_t n, const uint16_t *x, int64_t d,
                                         int64_t ldx, float *y, int64_t ldy, int norm, int add_self_loop,
                                         const float *dinv, const uint8_t *deg_code, const uint8_t *skip_rows,
                                         int accumulate, int finalize, int run_split_rows, int64_t *plan_i64,
                                         const int64_t *plan_host, float *partial, int64_t row_offset, void *stream) {
  return spmm_ranged("wdgh_spmm_csr_ranged_bf16", rowptr, range_begin, range_end, col, val, n,
                     reinterpret_cast<const bf16 *>(x), d, ldx, y, ldy, norm, add_self_loop, dinv, deg_code, skip_rows,
                     accumulate, finalize, run_split_rows, nullptr, 0, 0, 0, 0, 0, plan_i64, plan_host, partial,
                     row_offset, stream);
}

extern "C" int wdgh_spmm_csr_ranged_f16(const int64_t *rowptr, const int64_t *range_begin, const int64_t *range_end,
                                        const int32_t *col, const float *val, int64_t n, const uint16_t *x, int64_t d,
                                        int64_t ldx, float *y, int64_t ldy, int norm, int add_self_loop,
                                        const float *dinv, const uint8_t *deg_code, const uint8_t *skip_rows,
                                        int accumulate, int finalize, int run_split_rows, int64_t *plan_i64,
                                        const int64_t *plan_host, float *partial, int64_t row_offset, void *stream) {
  return spmm_ranged("wdgh_spmm_csr_ranged_f16", rowptr, range_begin, range_end, col, val, n,
                     reinterpret_cast<const f16 *>(x), d, ldx, y, ldy, norm, add_self_loop, dinv, deg_code, skip_rows,
                     accumulate, finalize, run_split_rows, nullptr, 0, 0, 0, 0, 0, plan_i64, plan_host, partial,
                     row_offset, stream);
}
