// Label metrics: every integer statistic behind edge / node / class / adjusted homophily and
// label informativeness (utils/homophily_metrics.py:43-161) in ONE pass over the stored entries.
//
//   edge pass  : per entry (i,j): label gather, match flags, class-pair key a*C+b.
//                Key multiplicities inside a warp are folded with __match_any_sync + popc and a
//                single shared-memory atomic per distinct key (C*C <= 4096 bins in shared memory,
//                global 64-bit atomics beyond that); the scalar counters travel as per-lane
//                registers and are combined by warp shuffles -- all counts are exact integers.
//   node part  : per node: f32(match)/f32(deg) for node homophily (hm.py:77-78), class sizes,
//                class degree mass (hm.py:141), empty rows, bincount length -- in the group epilogue of
//                the edge kernel; split rows after their chunks (structure_heavy_nodes_kernel).
// HBM traffic per entry: 4 B of `col` plus one label gather that is served by L2 whenever the
// label array (4 B/node) fits its 126 MB.
#include <limits.h>
#include <stdlib.h>

#include "internal.cuh"

namespace wdgh {

constexpr int kClassSmemClasses = 2048;  // 2*C 64-bit class accumulators kept in shared memory per CTA

// A label indexes the class tables only when 0 <= l < C.  Any other value -- negative, or >= C through the C ABI --
// is unlabelled; match counts compare raw labels all the same (hm.py:51).
__device__ __forceinline__ bool labelled(int l, int C) { return (unsigned)l < (unsigned)C; }

struct EdgeAcc {
  unsigned match_all = 0, match_lab = 0, n_lab = 0, n_self = 0;

  // one stored entry with endpoint labels li, lj; returns its class-pair key (both endpoints labelled, off the
  // diagonal unless hist_self), -1 for none
  __device__ __forceinline__ int add(int li, int lj, bool self, int C, bool hist_self = false) {
    const bool same = (li == lj);
    const bool both = labelled(li, C) && labelled(lj, C);
    match_all += same;
    match_lab += (same && both);
    n_lab += both;
    n_self += self;
    return (both && (!self || hist_self)) ? li * C + lj : -1;
  }
  __device__ __forceinline__ void flush(unsigned long long *counters) {
    long long v0 = warp_sum((long long)match_all), v1 = warp_sum((long long)match_lab);
    long long v2 = warp_sum((long long)n_lab), v3 = warp_sum((long long)n_self);
    if ((threadIdx.x & 31) == 0) {
      if (v0) atomicAdd(&counters[WDGH_SC_MATCH_ALL], (unsigned long long)v0);
      if (v1) atomicAdd(&counters[WDGH_SC_MATCH_LAB], (unsigned long long)v1);
      if (v2) atomicAdd(&counters[WDGH_SC_N_LAB], (unsigned long long)v2);
      if (v3) atomicAdd(&counters[WDGH_SC_N_SELF], (unsigned long long)v3);
    }
  }
};

// Per-node reductions of the rows a thread owns: node-homophily sums, rows with an off-diagonal entry, empty rows and
// the bincount length.  flush() combines them per warp (every lane of the warp calls it).
struct NodeAcc {
  double sum = 0.0, sum_self = 0.0;
  unsigned n_nsl = 0, n_empty = 0;
  long long nbins = 0;

  // a row with d_nsl off-diagonal entries, m_nsl of them label matches (edge-list input: row lengths unknown)
  __device__ __forceinline__ void add_nsl(int d_nsl, int m_nsl, int64_t global_row) {
    if (d_nsl > 0) {
      sum += (double)((float)m_nsl / (float)d_nsl);  // float32 division as torch does (hm.py:77)
      n_nsl += 1;
      nbins = max(nbins, (long long)(global_row + 1));  // rows do not come in order
    }
  }
  // the same with the stored row length deg_all known: empty rows, and the variant that counts the stored diagonal
  // entries as matches (homophily_plot.py:92-100, which does not strip self loops)
  __device__ __forceinline__ void add(int d_nsl, int m_nsl, int deg_all, int64_t global_row) {
    add_nsl(d_nsl, m_nsl, global_row);
    if (deg_all == 0) n_empty += 1;
    else sum_self += (double)((float)(m_nsl + (deg_all - d_nsl)) / (float)deg_all);
  }
  // class size, class degree mass and (rare: no off-diagonal entry) isolated count of a node with label l
  template <typename T>
  static __device__ __forceinline__ void add_class(int l, int C, int d_nsl, T deg_all, T *cls_count, T *cls_deg,
                                                   unsigned long long *counters) {
    if (!labelled(l, C)) return;
    atomicAdd(&cls_count[l], (T)1);
    atomicAdd(&cls_deg[l], deg_all);
    if (d_nsl == 0) atomicAdd(&counters[WDGH_SC_HEADER + 2 * C + (size_t)C * C + l], 1ull);
  }
  __device__ __forceinline__ void flush(unsigned long long *counters, double *node_sum) {
    const double s0 = warp_sum(sum), s1 = warp_sum(sum_self);
    const long long a0 = warp_sum((long long)n_nsl), a1 = warp_sum((long long)n_empty);
    long long nbm = nbins;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) nbm = max(nbm, __shfl_xor_sync(0xffffffffu, nbm, o));
    if ((threadIdx.x & 31) == 0) {
      if (s0 != 0.0) atomicAdd(node_sum, s0);
      if (s1 != 0.0) atomicAdd(node_sum + 1, s1);
      if (a0) atomicAdd(&counters[WDGH_SC_N_NODES_NSL], (unsigned long long)a0);
      if (a1) atomicAdd(&counters[WDGH_SC_N_EMPTY], (unsigned long long)a1);
      if (nbm) atomicMax(&counters[WDGH_SC_NBINS], (unsigned long long)nbm);
    }
  }
};

// Counts of one CTA bound for global 64-bit counters: shared-memory words T while the table fits, otherwise the global
// counters themselves.  Every thread of the CTA constructs it; the constructor ends with __syncthreads().
template <typename T>
struct CtaTable {
  T *s;
  unsigned long long *g;
  int words;
  bool smem;
  __device__ __forceinline__ CtaTable(T *s_words, unsigned long long *g_words, int n_words, bool fits)
      : s(s_words), g(g_words), words(n_words), smem(fits) {
    if (smem)
      for (int b = threadIdx.x; b < words; b += blockDim.x) s[b] = 0;
    __syncthreads();
  }
  __device__ __forceinline__ T *ptr() const { return smem ? s : g; }         // T = unsigned long long
  __device__ __forceinline__ void fold(int key) { fold_keys(key, s, g, smem); }  // T = unsigned
  __device__ __forceinline__ void flush() {
    if (!smem) return;
    __syncthreads();
    for (int b = threadIdx.x; b < words; b += blockDim.x)
      if (s[b]) atomicAdd(&g[b], (unsigned long long)s[b]);
  }
};
// the C x C class-pair histogram: 32-bit shared bins while C*C <= kHistSmemBins
__device__ __forceinline__ CtaTable<unsigned> pair_table(unsigned *s, unsigned long long *counters, int C) {
  return CtaTable<unsigned>(s, counters + WDGH_SC_HEADER + 2 * C, C * C, C * C <= kHistSmemBins);
}
// [C] class sizes, [C] class degree mass: 64-bit shared words while C <= kClassSmemClasses
__device__ __forceinline__ CtaTable<unsigned long long> class_table(unsigned long long *s, unsigned long long *counters,
                                                                    int C) {
  return CtaTable<unsigned long long>(s, counters + WDGH_SC_HEADER, 2 * C, C <= kClassSmemClasses);
}
static size_t pair_smem(int C) { return ((size_t)C * C <= (size_t)kHistSmemBins) ? (size_t)C * C * sizeof(unsigned) : 0; }
static size_t class_smem(int C) { return (C <= kClassSmemClasses) ? 2 * (size_t)C * sizeof(unsigned long long) : 0; }

// label fetch: int32 labels as given, or the uint8 copy (0xFF = unlabelled) that keeps the gathered
// array L2-resident for graphs up to ~100M nodes
template <typename L>
__device__ __forceinline__ int load_label(const L *p, int64_t i);
template <>
__device__ __forceinline__ int load_label<int32_t>(const int32_t *p, int64_t i) { return __ldg(p + i); }
template <>
__device__ __forceinline__ int load_label<uint8_t>(const uint8_t *p, int64_t i) {
  const int v = __ldg(p + i);
  return v == 255 ? -1 : v;
}

// Row-group form of the edge pass: a warp takes GROUPS of 32 consecutive rows (ticket counter: row lengths are
// heavy-tailed) and walks the stored entries of a group as one stream, 4 x 32 entries per iteration, so every
// lane carries an entry whatever the row lengths are (the G-lanes-per-row kernel above idles ~1/3 of its
// lanes on a power-law graph).  The row slot of a stream position comes from a 5-step search in the scanned
// row lengths; per-row counts are popcounts over the runs of equal row slots inside a 32-entry slice,
// accumulated in shared memory and written coalesced at the end of the group.  Column ids are requested one
// iteration ahead (and across the group boundary), label gathers right before they are consumed.  The per-node
// reductions of the group's non-split rows ride in the group epilogue, as in the stream form below.
// 4 CTAs / SM: the grid never holds more (launch in wdgh_structure_counts).
template <typename L>
__global__ void __launch_bounds__(256, 4)
structure_rowgroup_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col, int64_t n,
                          const L *__restrict__ labels, int C, int64_t threshold,
                          unsigned long long *__restrict__ counters, double *__restrict__ node_sum,
                          int32_t *__restrict__ deg_nsl, int32_t *__restrict__ match_nsl, int64_t row_offset,
                          unsigned long long *__restrict__ sched) {
  extern __shared__ unsigned long long s_dyn64[];  // class_smem(C) bytes of class table, then the pair table
  __shared__ int s_off[8][2][33];
  __shared__ int64_t s_beg[8][2][32];
  __shared__ int s_match[8][2][32], s_self[8][2][32];
  constexpr unsigned kFull = 0xffffffffu;
  constexpr int EPL = 4;
  CtaTable<unsigned long long> cls = class_table(s_dyn64, counters, C);
  CtaTable<unsigned> pairs = pair_table(reinterpret_cast<unsigned *>(s_dyn64 + (cls.smem ? 2 * C : 0)), counters, C);
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const int64_t W = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t n_groups = (n + 31) >> 5;
  EdgeAcc acc;
  NodeAcc nodes;

  auto take = [&]() -> int64_t {
    unsigned long long t = 0;
    if (lane == 0) t = atomicAdd(&sched[0], 1ull);
    return (int64_t)__shfl_sync(kFull, t, 0) + W;  // the first W groups are handed out by position
  };
  auto load_bounds = [&](int64_t g, int64_t &b, int64_t &e, int &li) {
    b = 0;
    e = 0;
    li = -1;
    const int64_t r = (g << 5) + lane;
    if (r < n) {
      b = __ldg(rowptr + r);
      e = __ldg(rowptr + r + 1);
      li = load_label<L>(labels, r + row_offset);
    }
  };
  // scan the row lengths of group g; split rows count as empty here (structure_chunks_kernel owns them)
  auto publish = [&](int buf, int64_t b, int64_t e, int &total, int &len) {
    len = (e - b > threshold) ? 0 : (int)(e - b);
    int inc = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(kFull, inc, o);
      if (lane >= o) inc += v;
    }
    s_off[wid][buf][lane + 1] = inc;
    if (lane == 0) s_off[wid][buf][0] = 0;
    s_beg[wid][buf][lane] = b;
    s_match[wid][buf][lane] = 0;
    s_self[wid][buf][lane] = 0;
    total = __shfl_sync(kFull, inc, 31);
    __syncwarp();
  };
  // column ids and row slots of stream positions t0 + 32 k + lane, k = 0 .. 3 (j = -1: past the end)
  auto load_cols = [&](int buf, int t0, int total, int (&j)[EPL], int (&rho)[EPL]) {
#pragma unroll
    for (int k = 0; k < EPL; ++k) {
      const int t = t0 + 32 * k + lane;
      j[k] = -1;
      rho[k] = 0;
      if (t < total) {
        int lo = 0;
#pragma unroll
        for (int step = 16; step >= 1; step >>= 1)
          if (s_off[wid][buf][lo + step] <= t) lo += step;
        rho[k] = lo;
        j[k] = __ldg(col + s_beg[wid][buf][lo] + (t - s_off[wid][buf][lo]));
      }
    }
  };

  int64_t g = (int64_t)blockIdx.x * 8 + wid;
  if (g < n_groups) {
    int64_t b, e;
    int li_cur, li_next = -1, li_load, dall, n_dall = 0;  // dall: full row length (split rows included)
    load_bounds(g, b, e, li_cur);
    int buf = 0, total, len, n_total = 0, n_len = 0;
    publish(0, b, e, total, len);
    dall = (int)(e - b);
    int64_t gn = take(), gnn = 0;
    load_bounds(gn, b, e, li_load);
    int j[EPL], rho[EPL], nj[EPL], nrho[EPL];
    load_cols(0, 0, total, j, rho);
    while (true) {
      bool next_ready = false;
      auto prefetch = [&](int t0) {
        if (t0 + 32 * EPL < total) {
          load_cols(buf, t0 + 32 * EPL, total, nj, nrho);
        } else {
          publish(buf ^ 1, b, e, n_total, n_len);
          n_dall = (int)(e - b);
          li_next = li_load;
          load_cols(buf ^ 1, 0, n_total, nj, nrho);
          gnn = take();
          load_bounds(gnn, b, e, li_load);
          next_ready = true;
        }
      };
      for (int t0 = 0; t0 < total; t0 += 32 * EPL) {
        int lj[EPL];
#pragma unroll
        for (int k = 0; k < EPL; ++k) lj[k] = (j[k] >= 0) ? load_label<L>(labels, j[k]) : -1;
        prefetch(t0);
#pragma unroll
        for (int k = 0; k < EPL; ++k) {
          const bool valid = j[k] >= 0;
          if (__ballot_sync(kFull, valid) == 0u) continue;  // warp-uniform
          const int lie = __shfl_sync(kFull, li_cur, rho[k]);
          const int64_t grow = (g << 5) + rho[k] + row_offset;
          const bool self = valid && ((int64_t)j[k] == grow);
          pairs.fold(valid ? acc.add(lie, lj[k], self, C) : -1);
          // per-row counts: one popcount per run of equal row slots
          const unsigned m = __ballot_sync(kFull, valid && !self && lie == lj[k]), sf = __ballot_sync(kFull, self);
          const int prev = __shfl_up_sync(kFull, rho[k], 1);
          const bool head = valid && (lane == 0 || prev != rho[k]);
          const unsigned heads = __ballot_sync(kFull, head);
          if (head) {
            const unsigned above = (lane == 31) ? 0u : (heads & (kFull << (lane + 1)));
            const int end = above ? (__ffs(above) - 1) : 32;
            const unsigned mask = ((end == 32) ? kFull : ((1u << end) - 1u)) & (kFull << lane);
            const int cm = __popc(m & mask), cs = __popc(sf & mask);
            if (cm) s_match[wid][buf][rho[k]] += cm;
            if (cs) s_self[wid][buf][rho[k]] += cs;
          }
          __syncwarp();
        }
#pragma unroll
        for (int k = 0; k < EPL; ++k) {
          j[k] = nj[k];
          rho[k] = nrho[k];
        }
      }
      if (!next_ready) {  // a group without entries
        prefetch(0);
#pragma unroll
        for (int k = 0; k < EPL; ++k) {
          j[k] = nj[k];
          rho[k] = nrho[k];
        }
      }
      __syncwarp();
      // group epilogue: per-row outputs (split rows: zero here, the chunk kernel adds atomically) and the per-node
      // reductions of the non-split rows this warp owns (split rows: structure_heavy_nodes_kernel)
      const int64_t r = (g << 5) + lane;
      if (r < n) {
        const int dn = len - s_self[wid][buf][lane], mn = s_match[wid][buf][lane];
        deg_nsl[r] = dn;
        match_nsl[r] = mn;
        if (dall <= threshold) {
          nodes.add(dn, mn, len, r + row_offset);
          NodeAcc::add_class(li_cur, C, dn, (unsigned long long)len, cls.ptr(), cls.ptr() + C, counters);
        }
      }
      g = gn;
      gn = gnn;
      buf ^= 1;
      total = n_total;
      len = n_len;
      dall = n_dall;
      li_cur = li_next;
      if (g >= n_groups) break;
    }
  }
  acc.flush(counters);
  nodes.flush(counters, node_sum);
  cls.flush();
  pairs.flush();
  sched_retire(sched, gridDim.x);
}

// ---------------------------------------------------------------------------
// Stream form of the edge pass -- the default (1-byte labels, (C+1)^2 <= 4096 pair bins).  A warp takes GROUPS of 32
// consecutive rows from a ticket counter and walks the group's stored entries as one stream, EPL x 32 entries per
// iteration.  What makes it ~4x cheaper per entry than the row-group kernel above:
//   * the row of a stream position comes from two warp-wide bit operations instead of a 5-step search per lane:
//     REDUX.OR builds the mask of rows that START inside a 32-entry slice, a ballot counts the rows that started
//     before it; rank = count + popc(mask & lanes_le) - 1 indexes a compacted table of the non-empty rows
//     ({row slot, label, address correction}: one 8-byte shared-memory load);
//   * ONE pair table over (C+1) x (C+1) label values, unlabelled = C, self loops excluded: the four scalar counters
//     (matches, labelled matches, labelled entries) are sums over its bins taken once per CTA, so the per-entry
//     work is a single key fold (__match_any_sync + one shared atomic per distinct key);
//   * per-row match counts are taken on the OWNER side: lane r intersects the slice's match ballot with the bit
//     range of its own row -- no run detection, no shared-memory counters;
//   * the per-node reductions (node homophily sum, class sizes / degree mass, empty rows, bincount length) ride in
//     the group epilogue, where the row owner has everything in registers -- no second pass over the node arrays.
// Split rows contribute no entries here (structure_chunks_kernel + structure_heavy_nodes_kernel own them).
// ---------------------------------------------------------------------------
constexpr int kStreamEPL = 4;
__global__ void __launch_bounds__(256, 4)
structure_stream_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col, int64_t n,
                        const uint8_t *__restrict__ labels8, int C, int64_t threshold,
                        unsigned long long *__restrict__ counters, double *__restrict__ node_sum,
                        int32_t *__restrict__ deg_nsl, int32_t *__restrict__ match_nsl, int64_t row_offset,
                        unsigned long long *__restrict__ sched) {
  extern __shared__ unsigned s_dyn[];  // [(C+1)^2] pair table, [C+1] class sizes, [C+1] class degree mass
  __shared__ int2 s_pack[8][2][32];    // per warp, double buffered: {(row slot << 8) | label, address correction}
  constexpr unsigned kFull = 0xffffffffu;
  constexpr int EPL = kStreamEPL;
  const int C1 = C + 1;
  unsigned *s_hist = s_dyn, *s_cnt = s_dyn + C1 * C1, *s_deg = s_cnt + C1;
  for (int b = threadIdx.x; b < C1 * C1 + 2 * C1; b += blockDim.x) s_dyn[b] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
  const unsigned lanes_lt = (1u << lane) - 1u, lanes_le = lanes_lt | (1u << lane);
  const int64_t W = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t n_groups = (n + 31) >> 5;
  unsigned n_self = 0, n_self_lab = 0;                  // warp-uniform
  NodeAcc nodes;                                        // per lane (row owner)

  auto take = [&]() -> int64_t {
    unsigned long long t = 0;
    if (lane == 0) t = atomicAdd(&sched[0], 1ull);
    return (int64_t)__shfl_sync(kFull, t, 0) + W;  // the first W groups are handed out by position
  };
  auto load_bounds = [&](int64_t g, int64_t &b, int64_t &e, int &li) {
    b = 0;
    e = 0;
    li = C;
    const int64_t r = (g << 5) + lane;
    if (r < n) {
      b = __ldg(rowptr + r);
      e = __ldg(rowptr + r + 1);
      const int v = __ldg(labels8 + r + row_offset);
      li = (v == 255) ? C : v;
    }
  };
  // scan the row lengths of a group and publish the compacted row table
  auto publish = [&](int buf, int64_t b, int64_t e, int li, int &off, int &len, int &total, const int32_t *&cp) {
    len = (e - b > threshold) ? 0 : (int)(e - b);
    int inc = len;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int v = __shfl_up_sync(kFull, inc, o);
      if (lane >= o) inc += v;
    }
    off = inc - len;
    total = __shfl_sync(kFull, inc, 31);
    const int64_t gbeg = __shfl_sync(kFull, b, 0);
    cp = col + gbeg;
    const unsigned ne = __ballot_sync(kFull, len > 0);
    if (len > 0) s_pack[wid][buf][__popc(ne & lanes_lt)] = make_int2((lane << 8) | li, (int)(b - gbeg) - off);
    __syncwarp();
  };
  // column ids and row records of stream positions t0 + 32 k + lane (j = -1: past the end)
  auto load_cols = [&](int buf, int t0, int total, int off, int len, const int32_t *cp, int (&j)[EPL], int (&pk)[EPL]) {
#pragma unroll
    for (int k = 0; k < EPL; ++k) {
      const int tk = t0 + 32 * k;
      j[k] = -1;
      pk[k] = 0;
      if (tk < total) {  // warp-uniform
        const int rel = off - tk;
        const unsigned heads = __reduce_or_sync(kFull, (len > 0 && rel >= 0 && rel < 32) ? (1u << rel) : 0u);
        const int before = __popc(__ballot_sync(kFull, len > 0 && rel < 0));
        if (tk + lane < total) {
          const int2 rec = s_pack[wid][buf][before + __popc(heads & lanes_le) - 1];
          pk[k] = rec.x;
          j[k] = __ldg(cp + (tk + lane + rec.y));
        }
      }
    }
  };

  int64_t g = (int64_t)blockIdx.x * 8 + wid;
  if (g < n_groups) {
    int64_t b, e;
    int li_load, li_cur, li_next = C, dall, n_dall = 0;  // dall: full row length (split rows included)
    load_bounds(g, b, e, li_load);
    int buf = 0, off, len, total, n_off = 0, n_len = 0, n_total = 0;
    const int32_t *cp, *n_cp = col;
    publish(0, b, e, li_load, off, len, total, cp);
    dall = (int)(e - b); li_cur = li_load;
    int64_t gn = take(), gnn = 0;
    load_bounds(gn, b, e, li_load);
    int j[EPL], pk[EPL], nj[EPL], npk[EPL];
    load_cols(0, 0, total, off, len, cp, j, pk);
    while (true) {
      bool next_ready = false;
      int my_match = 0, my_self = 0;
      auto prefetch = [&](int t0) {
        if (t0 + 32 * EPL < total) {
          load_cols(buf, t0 + 32 * EPL, total, off, len, cp, nj, npk);
        } else {
          publish(buf ^ 1, b, e, li_load, n_off, n_len, n_total, n_cp);
          n_dall = (int)(e - b); li_next = li_load;
          load_cols(buf ^ 1, 0, n_total, n_off, n_len, n_cp, nj, npk);
          gnn = take();
          load_bounds(gnn, b, e, li_load);
          next_ready = true;
        }
      };
      const int grow0 = (int)((g << 5) + row_offset);
      for (int t0 = 0; t0 < total; t0 += 32 * EPL) {
        int lj[EPL];
#pragma unroll
        for (int k = 0; k < EPL; ++k) lj[k] = (j[k] >= 0) ? (int)__ldg(labels8 + j[k]) : 255;
        prefetch(t0);
#pragma unroll
        for (int k = 0; k < EPL; ++k) {
          const int tk = t0 + 32 * k;
          if (tk >= total) continue;  // warp-uniform
          const bool valid = j[k] >= 0;
          const int lie = pk[k] & 0xff, slot = pk[k] >> 8;
          const int ljx = (lj[k] == 255) ? C : lj[k];
          const bool self = valid && (j[k] == grow0 + slot);
          const bool same = valid && !self && (lie == ljx);
          fold_keys((valid && !self) ? lie * C1 + ljx : -1, s_hist, nullptr, true);
          const unsigned m = __ballot_sync(kFull, same), sf = __ballot_sync(kFull, self);
          // owner side: bits of this slice that belong to my row
          const int lo = min(max(off - tk, 0), 32), hi = min(max(off + len - tk, 0), 32);
          const unsigned upto_hi = (hi >= 32) ? kFull : ((1u << hi) - 1u);
          const unsigned mask = (hi > lo) ? (upto_hi & ~((1u << lo) - 1u)) : 0u;
          my_match += __popc(m & mask);
          if (sf) {  // warp-uniform and rare: stored diagonal entries
            my_self += __popc(sf & mask);
            n_self += __popc(sf);
            n_self_lab += __popc(__ballot_sync(kFull, self && lie < C));
          }
        }
#pragma unroll
        for (int k = 0; k < EPL; ++k) {
          j[k] = nj[k];
          pk[k] = npk[k];
        }
      }
      if (!next_ready) {  // a group without entries
        prefetch(0);
#pragma unroll
        for (int k = 0; k < EPL; ++k) {
          j[k] = nj[k];
          pk[k] = npk[k];
        }
      }
      // group epilogue: per-row outputs and the per-node reductions of the rows this warp owns
      const int64_t r = (g << 5) + lane;
      if (r < n) {
        const bool heavy = dall > threshold;
        const int dn = len - my_self;
        deg_nsl[r] = heavy ? 0 : dn;       // split rows: zero here, the chunk kernel adds atomically
        match_nsl[r] = heavy ? 0 : my_match;
        if (!heavy) {                      // len == dall
          nodes.add(dn, my_match, dall, r + row_offset);
          NodeAcc::add_class(li_cur, C, dn, (unsigned)len, s_cnt, s_deg, counters);
        }
      }
      g = gn;
      gn = gnn;
      buf ^= 1;
      off = n_off; len = n_len; total = n_total; cp = n_cp;
      dall = n_dall; li_cur = li_next;
      if (g >= n_groups) break;
    }
  }
  // ---- per-warp scalars ----
  nodes.flush(counters, node_sum);
  if (lane == 0) {
    if (n_self) {
      atomicAdd(&counters[WDGH_SC_N_SELF], (unsigned long long)n_self);
      atomicAdd(&counters[WDGH_SC_MATCH_ALL], (unsigned long long)n_self);
    }
    if (n_self_lab) {
      atomicAdd(&counters[WDGH_SC_MATCH_LAB], (unsigned long long)n_self_lab);
      atomicAdd(&counters[WDGH_SC_N_LAB], (unsigned long long)n_self_lab);
    }
  }
  // ---- per-CTA tables: the pair table also yields the scalar counters ----
  __syncthreads();
  unsigned long long *g_cls = counters + WDGH_SC_HEADER;
  unsigned long long *g_hist = counters + WDGH_SC_HEADER + 2 * C;
  long long m_all = 0, m_lab = 0, n_lab = 0;
  for (int bin = threadIdx.x; bin < C1 * C1; bin += blockDim.x) {
    const unsigned v = s_hist[bin];
    if (v == 0) continue;
    const int a = bin / C1, b2 = bin - a * C1;
    if (a == b2) m_all += v;
    if (a < C && b2 < C) {
      n_lab += v;
      if (a == b2) m_lab += v;
      atomicAdd(&g_hist[a * C + b2], (unsigned long long)v);
    }
  }
  m_all = warp_sum(m_all);
  m_lab = warp_sum(m_lab);
  n_lab = warp_sum(n_lab);
  if (lane == 0) {
    if (m_all) atomicAdd(&counters[WDGH_SC_MATCH_ALL], (unsigned long long)m_all);
    if (m_lab) atomicAdd(&counters[WDGH_SC_MATCH_LAB], (unsigned long long)m_lab);
    if (n_lab) atomicAdd(&counters[WDGH_SC_N_LAB], (unsigned long long)n_lab);
  }
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    if (s_cnt[c]) atomicAdd(&g_cls[c], (unsigned long long)s_cnt[c]);
    if (s_deg[c]) atomicAdd(&g_cls[C + c], (unsigned long long)s_deg[c]);
  }
  sched_retire(sched, gridDim.x);
}

// per-node reductions of the split rows, after structure_chunks_kernel completed their counts
__global__ void structure_heavy_nodes_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ labels,
                                             int C, const int64_t *__restrict__ plan,
                                             const int32_t *__restrict__ deg_nsl, const int32_t *__restrict__ match_nsl,
                                             unsigned long long *__restrict__ counters, double *__restrict__ node_sum,
                                             int64_t row_offset) {
  const int64_t n_heavy = plan[kPlanNHeavy];
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  unsigned long long *g_cls = counters + WDGH_SC_HEADER;
  NodeAcc nodes;
  for (int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; k < n_heavy; k += stride) {
    const int64_t i = plan_heavy_row(plan)[k];
    const int d = deg_nsl[i], m = match_nsl[i];
    const int deg_all = (int)(rowptr[i + 1] - rowptr[i]);
    nodes.add(d, m, deg_all, i + row_offset);
    NodeAcc::add_class(labels[i + row_offset], C, d, (unsigned long long)deg_all, g_cls, g_cls + C, counters);
  }
  nodes.flush(counters, node_sum);
}

// int32 labels -> uint8 (0xFF = unlabelled); requires C <= 254.
// counters[WDGH_SC_N_MULTI_NEG] counts the labels the 1-byte copy cannot represent exactly, those below -1 or >= C:
// they all map to 0xFF like -1, so their mutual (in)equality (hm.py:51 compares raw labels) is only exact on the
// int32 path -- the host re-runs it.
__global__ void labels_to_u8_kernel(const int32_t *__restrict__ in, int64_t n, int C, uint8_t *__restrict__ out,
                                    unsigned long long *__restrict__ counters) {
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  long long odd = 0;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int v = in[i];
    const bool lab = labelled(v, C);
    out[i] = lab ? (uint8_t)v : (uint8_t)255;
    odd += (!lab && v != -1);
  }
  odd = warp_sum(odd);
  if ((threadIdx.x & 31) == 0 && odd) atomicAdd(&counters[WDGH_SC_N_MULTI_NEG], (unsigned long long)odd);
}

// One warp per chunk of a split row.
template <typename L>
__global__ void __launch_bounds__(256)
structure_chunks_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col,
                        const L *__restrict__ labels, int C, const int64_t *__restrict__ plan,
                        int64_t n_chunks, unsigned long long *__restrict__ counters,
                        int32_t *__restrict__ deg_nsl, int32_t *__restrict__ match_nsl, int64_t row_offset) {
  extern __shared__ unsigned s_hist[];
  CtaTable<unsigned> pairs = pair_table(s_hist, counters, C);
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  const int64_t cap = plan[kPlanCapacity], T = plan[kPlanThreshold];
  EdgeAcc acc;
  for (int64_t chunk = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; chunk < n_chunks; chunk += nwarps) {
    const int64_t k = plan_chunk_owner(plan, cap)[chunk];
    const int64_t row = plan_heavy_row(plan)[k];
    const int64_t part = chunk - plan_heavy_chunk0(plan, cap)[k];
    const int64_t s = __ldg(rowptr + row) + part * T;
    const int64_t e = min(s + T, __ldg(rowptr + row + 1));
    const int li = load_label<L>(labels, row + row_offset);
    int m_nsl = 0, d_nsl = 0;
    for (int64_t base = s; base < e; base += 32) {  // warp-uniform trip count
      const int64_t idx = base + lane;
      int key = -1;
      if (idx < e) {
        const int j = __ldg(col + idx);
        const int lj = load_label<L>(labels, j);
        const bool self = (j == row + row_offset);
        key = acc.add(li, lj, self, C);
        d_nsl += !self;
        m_nsl += (!self && li == lj);
      }
      pairs.fold(key);
    }
    m_nsl = (int)warp_sum((long long)m_nsl);
    d_nsl = (int)warp_sum((long long)d_nsl);
    if (lane == 0) {
      atomicAdd(&deg_nsl[row], d_nsl);
      atomicAdd(&match_nsl[row], m_nsl);
    }
  }
  acc.flush(counters);
  pairs.flush();
}

// Edge-list input (an arbitrary, possibly unsorted / repeated `edge_index` as handed to
// node_homophily_edge_idx / compact_matrix_edge_idx, hm.py:71,81): one lane per listed edge,
// per-node counts through 32-bit global atomics.  deg / match must be zeroed by the caller.
__global__ void __launch_bounds__(256)
structure_coo_kernel(const int64_t *__restrict__ edge_index, int64_t E, const int32_t *__restrict__ labels, int C,
                     unsigned long long *__restrict__ counters, int32_t *__restrict__ deg_nsl,
                     int32_t *__restrict__ match_nsl, bool hist_self) {
  extern __shared__ unsigned s_hist[];
  CtaTable<unsigned> pairs = pair_table(s_hist, counters, C);
  EdgeAcc acc;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  const int64_t rounds = (E + stride - 1) / stride;  // uniform trip count for the warp-wide fold
  for (int64_t r = 0; r < rounds; ++r) {
    const int64_t t = r * stride + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int key = -1;
    if (t < E) {
      const int64_t src = edge_index[t], dst = edge_index[E + t];
      const int li = __ldg(labels + src), lj = __ldg(labels + dst);
      const bool self = (dst == src);
      key = acc.add(li, lj, self, C, hist_self);
      if (!self) {
        atomicAdd(&deg_nsl[src], 1);
        if (li == lj) atomicAdd(&match_nsl[src], 1);
      }
    }
    pairs.fold(key);
  }
  acc.flush(counters);
  pairs.flush();
}

// Per-node reductions of the edge-list form.  Row lengths are unknown there: no empty rows, no diagonal variant of
// the node sum, no class degree mass.
__global__ void __launch_bounds__(256)
structure_nodes_kernel(int64_t n, const int32_t *__restrict__ labels, int C, const int32_t *__restrict__ deg_nsl,
                       const int32_t *__restrict__ match_nsl, unsigned long long *__restrict__ counters,
                       double *__restrict__ node_sum) {
  extern __shared__ unsigned long long s_cls[];
  CtaTable<unsigned long long> cls = class_table(s_cls, counters, C);
  NodeAcc nodes;
  const int64_t stride = (int64_t)gridDim.x * blockDim.x;
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
    const int d = deg_nsl[i], m = match_nsl[i];
    nodes.add_nsl(d, m, i);
    NodeAcc::add_class(labels[i], C, d, 0ull, cls.ptr(), cls.ptr() + C, counters);
  }
  nodes.flush(counters, node_sum);
  cls.flush();
}

// edge_homophily with a 2-D label matrix: elementwise equality of the two label rows (hm.py:51)
__global__ void __launch_bounds__(256)
label_rows_equal_kernel(const int64_t *__restrict__ rowptr, const int32_t *__restrict__ col, int64_t n,
                        const float *__restrict__ lab, int64_t c, int64_t ld, unsigned long long *__restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
  long long cnt = 0;
  for (int64_t row = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; row < n; row += nwarps) {
    const int64_t s = rowptr[row], e = rowptr[row + 1];
    const float *li = lab + row * ld;
    for (int64_t q = s + lane; q < e; q += 32) {
      const float *lj = lab + (int64_t)col[q] * ld;
      for (int64_t k = 0; k < c; ++k) cnt += (li[k] == lj[k]);
    }
  }
  cnt = warp_sum(cnt);
  if (lane == 0 && cnt) atomicAdd(out, (unsigned long long)cnt);
}

}  // namespace wdgh

using namespace wdgh;

// zero the counters, optionally build the 1-byte label copy (returns it, or nullptr when the int32 labels must be
// used: C > 254 or no scratch)
static int structure_prepare(const int32_t *labels, int64_t n_labels, int C, uint8_t *labels_u8_scratch,
                             int64_t *counters, double *node_sum, const uint8_t **labels8_out, cudaStream_t st) {
  const size_t n_counters = WDGH_SC_WORDS((size_t)C);
  WDGH_CUDA(cudaMemsetAsync(counters, 0, n_counters * sizeof(int64_t), st));
  WDGH_CUDA(cudaMemsetAsync(node_sum, 0, 2 * sizeof(double), st));
  *labels8_out = nullptr;
  if (labels_u8_scratch != nullptr && C <= 254 && n_labels > 0) {
    labels_to_u8_kernel<<<persistent_grid(ceil_div(n_labels, 256), 8), 256, 0, st>>>(
        labels, n_labels, C, labels_u8_scratch, reinterpret_cast<unsigned long long *>(counters));
    WDGH_LAUNCHED("labels_to_u8_kernel");
    *labels8_out = labels_u8_scratch;
  }
  return 0;
}

extern "C" int wdgh_structure_counts(const int64_t *rowptr, const int32_t *col, int64_t n, int64_t nnz,
                                     const int32_t *labels, int32_t num_classes, int64_t *plan_i64,
                                     const int64_t *plan_host, int64_t *counters, double *node_sum,
                                     int32_t *deg_nsl, int32_t *match_nsl, uint8_t *labels_u8_scratch,
                                     int64_t n_labels, int64_t row_offset, void *stream) {
  WDGH_REQUIRE(rowptr && labels && plan_i64 && plan_host && counters && node_sum && deg_nsl && match_nsl,
               "wdgh_structure_counts: null pointer");
  WDGH_REQUIRE(n >= 0 && nnz >= 0 && (col || nnz == 0), "wdgh_structure_counts: bad shape");
  WDGH_REQUIRE(num_classes >= 1 && num_classes <= 46340, "wdgh_structure_counts: num_classes out of range");
  WDGH_REQUIRE(labels_u8_scratch == nullptr || n_labels >= n + row_offset, "wdgh_structure_counts: n_labels too small");
  cudaStream_t st = as_stream(stream);
  const int C = num_classes;
  const uint8_t *labels8 = nullptr;
  int rc = structure_prepare(labels, n == 0 ? 0 : n_labels, C, labels_u8_scratch, counters, node_sum, &labels8, st);
  if (rc || n == 0) return rc;
  unsigned long long *cnt = reinterpret_cast<unsigned long long *>(counters);
  unsigned long long *sched = plan_sched(plan_i64, kPlanLabelTicket);
  const size_t hist_smem = pair_smem(C);
  const int64_t threshold = plan_host[2], n_heavy = plan_host[0], n_chunks = plan_host[1];
  const unsigned edge_grid = persistent_grid(ceil_div(ceil_div(n, 32), 8), 4);
  // every form: edge pass with the per-node reductions of the non-split rows -> split-row chunks -> split-row nodes
  const bool stream_form = labels8 != nullptr && (size_t)(C + 1) * (C + 1) <= (size_t)kHistSmemBins &&
                           n + row_offset < (int64_t)INT32_MAX;
  if (stream_form) {
    const size_t smem = ((size_t)(C + 1) * (C + 1) + 2 * (size_t)(C + 1)) * sizeof(unsigned);
    // 4 CTAs / SM (64 registers, 76 B of spills): 5.89 ms on the 976M-entry graph against 6.16 ms at 3 CTAs / SM
    // (76 registers, no spills) and 6.71 ms at 5 (48 registers)
    structure_stream_kernel<<<edge_grid, 256, smem, st>>>(rowptr, col, n, labels8, C, threshold, cnt, node_sum,
                                                          deg_nsl, match_nsl, row_offset, sched);
    WDGH_LAUNCHED("structure_stream_kernel");
  } else {
    const size_t smem = class_smem(C) + hist_smem;
    if (labels8)
      structure_rowgroup_kernel<uint8_t><<<edge_grid, 256, smem, st>>>(rowptr, col, n, labels8, C, threshold, cnt,
                                                                       node_sum, deg_nsl, match_nsl, row_offset, sched);
    else
      structure_rowgroup_kernel<int32_t><<<edge_grid, 256, smem, st>>>(rowptr, col, n, labels, C, threshold, cnt,
                                                                       node_sum, deg_nsl, match_nsl, row_offset, sched);
    WDGH_LAUNCHED("structure_rowgroup_kernel");
  }
  if (n_chunks > 0) {  // split rows: one warp per chunk
    const unsigned grid = persistent_grid(ceil_div(n_chunks, 8), 8);
    if (labels8)
      structure_chunks_kernel<uint8_t><<<grid, 256, hist_smem, st>>>(rowptr, col, labels8, C, plan_i64, n_chunks, cnt,
                                                                    deg_nsl, match_nsl, row_offset);
    else
      structure_chunks_kernel<int32_t><<<grid, 256, hist_smem, st>>>(rowptr, col, labels, C, plan_i64, n_chunks, cnt,
                                                                    deg_nsl, match_nsl, row_offset);
    WDGH_LAUNCHED("structure_chunks_kernel");
  }
  if (n_heavy > 0) {
    structure_heavy_nodes_kernel<<<persistent_grid(ceil_div(n_heavy, 256), 4), 256, 0, st>>>(
        rowptr, labels, C, plan_i64, deg_nsl, match_nsl, cnt, node_sum, row_offset);
    WDGH_LAUNCHED("structure_heavy_nodes_kernel");
  }
  return 0;
}

extern "C" int wdgh_structure_counts_coo(const int64_t *edge_index, int64_t num_edges, int64_t n,
                                         const int32_t *labels, int32_t num_classes, int64_t *counters,
                                         double *node_sum, int32_t *deg_nsl, int32_t *match_nsl,
                                         int hist_includes_self_loops, void *stream) {
  WDGH_REQUIRE(labels && counters && node_sum && deg_nsl && match_nsl && (edge_index || num_edges == 0),
               "wdgh_structure_counts_coo: null pointer");
  WDGH_REQUIRE(n >= 0 && num_edges >= 0 && num_classes >= 1 && num_classes <= 46340,
               "wdgh_structure_counts_coo: bad shape");
  cudaStream_t st = as_stream(stream);
  const int C = num_classes;
  const uint8_t *labels8 = nullptr;
  int rc = structure_prepare(labels, 0, C, nullptr, counters, node_sum, &labels8, st);
  if (rc || n == 0) return rc;
  WDGH_CUDA(cudaMemsetAsync(deg_nsl, 0, n * sizeof(int32_t), st));
  WDGH_CUDA(cudaMemsetAsync(match_nsl, 0, n * sizeof(int32_t), st));
  unsigned long long *cnt = reinterpret_cast<unsigned long long *>(counters);
  if (num_edges > 0) {
    structure_coo_kernel<<<persistent_grid(ceil_div(num_edges, 256), 8), 256, pair_smem(C), st>>>(
        edge_index, num_edges, labels, C, cnt, deg_nsl, match_nsl, hist_includes_self_loops != 0);
    WDGH_LAUNCHED("structure_coo_kernel");
  }
  structure_nodes_kernel<<<persistent_grid(ceil_div(n, 256), 8), 256, class_smem(C), st>>>(n, labels, C, deg_nsl,
                                                                                          match_nsl, cnt, node_sum);
  WDGH_LAUNCHED("structure_nodes_kernel");
  return 0;
}

extern "C" int wdgh_edge_label_rows_equal(const int64_t *rowptr, const int32_t *col, int64_t n,
                                          const float *label_rows, int64_t c, int64_t ld,
                                          unsigned long long *equal_count, void *stream) {
  WDGH_REQUIRE(rowptr && label_rows && equal_count && n >= 0 && c >= 1 && ld >= c,
               "wdgh_edge_label_rows_equal: bad arguments");
  cudaStream_t st = as_stream(stream);
  WDGH_CUDA(cudaMemsetAsync(equal_count, 0, sizeof(unsigned long long), st));
  if (n == 0) return 0;
  label_rows_equal_kernel<<<persistent_grid(ceil_div(n, 8), 8), 256, 0, st>>>(rowptr, col, n, label_rows, c, ld,
                                                                             equal_count);
  WDGH_LAUNCHED("label_rows_equal_kernel");
  return 0;
}
