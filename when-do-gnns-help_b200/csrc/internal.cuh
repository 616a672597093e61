// Internal (non-ABI) entry points shared between translation units.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace wdgh {

constexpr int kHistSmemBins = 4096;  // C*C bins kept in shared memory per CTA

using bf16 = __nv_bfloat16;
using f16 = __half;

// The WDGH_DTYPE of the half Y an aggregation with features of type T may write besides fp32: the type of the features
// itself (fp32 features: fp32 Y only)
template <typename T>
constexpr int kHalfY = WDGH_DTYPE_F32;
template <>
constexpr int kHalfY<bf16> = WDGH_DTYPE_BF16;
template <>
constexpr int kHalfY<f16> = WDGH_DTYPE_F16;

// y[r][c] = x[r][c] rounded to nearest even to H (bf16 or f16; fp16 overflow -> +-inf), r < rows, c < cols (spmm.cu);
// y holds raw H bits
template <typename H>
int round_to_half(const float *x, int64_t rows, int64_t cols, int64_t ldx, void *y, int64_t ldy, cudaStream_t st);

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
