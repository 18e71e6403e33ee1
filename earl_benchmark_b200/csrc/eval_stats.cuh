// eval_stats.cuh -- the device reduction behind earl_eval_stats, earl_tt3_eval_stats and earl_mjk_eval_stats: four fp64
// per-thread partial sums (episode return, #success at the last step, #success at any step, #envs) reduced over the block
// and added to out4.
#pragma once

#include <cuda_runtime.h>

namespace earl {

// Every thread of the block must call it (it synchronises the block); blockDim.x is a multiple of 32, at most 1024.
// out4 must be zeroed before the launch; blocks add their sums with fp64 atomics, so the order of the additions across
// blocks is not fixed (exact for the integer counts and for sums of integer rewards).
__device__ __forceinline__ void block_add_eval_stats(double ret, double last, double any, double cnt, double* __restrict__ out4) {
#pragma unroll
  for (int o = 16; o; o >>= 1) {
    ret += __shfl_xor_sync(0xffffffffu, ret, o);
    last += __shfl_xor_sync(0xffffffffu, last, o);
    any += __shfl_xor_sync(0xffffffffu, any, o);
    cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
  }
  __shared__ double sm[4][32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { sm[0][warp] = ret; sm[1][warp] = last; sm[2][warp] = any; sm[3][warp] = cnt; }
  __syncthreads();
  if (warp == 0) {
    const int nw = blockDim.x >> 5;
    double v[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      v[k] = lane < nw ? sm[k][lane] : 0.0;
#pragma unroll
      for (int o = 16; o; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
    }
    if (lane == 0) {
#pragma unroll
      for (int k = 0; k < 4; ++k) atomicAdd(out4 + k, v[k]);
    }
  }
}

}  // namespace earl
