// Internal (non-ABI) entry points shared between translation units.
#pragma once
#include "common.cuh"

namespace wdgh {

constexpr int kHistSmemBins = 4096;  // C*C bins kept in shared memory per CTA

// y[r][c] = bf16(x[r][c]) rounded to nearest even, r < rows, c < cols (spmm.cu); y holds raw bf16 bits
int round_to_bf16(const float *x, int64_t rows, int64_t cols, int64_t ldx, void *y, int64_t ldy, cudaStream_t st);

// Folds one warp-wide batch of class-pair keys (key < 0: nothing to count) into the histogram:
// one atomic per distinct key, multiplicity from __match_any_sync + popc.
__device__ __forceinline__ void fold_keys(int key, unsigned *s_hist, unsigned long long *g_hist, bool use_smem) {
  const unsigned peers = __match_any_sync(0xffffffffu, key);
  if (key >= 0 && (threadIdx.x & 31) == (__ffs(peers) - 1)) {
    const unsigned c = __popc(peers);
    if (use_smem) atomicAdd(&s_hist[key], c);
    else atomicAdd(&g_hist[key], (unsigned long long)c);
  }
}

}  // namespace wdgh
