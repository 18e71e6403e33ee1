// final_obs.cuh -- EARL_FLAG_FINAL_OBS capture of the tasks whose auto-reset is a separate pass after the step (sawyer_door,
// sawyer_peg: earl_mj_impl.inc; kitchen: earl_mj_kitchen.cu).  Launched in the step's stream after the step, redo and
// ordering kernels and before the reset pass, it copies the observation row of every env whose horizon fired (done != 0)
// to final_obs: the row the step returns without auto-reset.  Rows of the other envs are not touched.
#pragma once
#include <cstdint>
#include <cuda_runtime.h>

namespace earl {

// obs, final_obs [n, dim] row-major; one thread per element, grid-stride.  Reads the n done bytes (once per element, from
// L1 / L2) and the obs rows it copies: the traffic follows the number of resets.
template <typename T>
__global__ void final_obs_capture_kernel(const T* __restrict__ obs, const uint8_t* __restrict__ done, T* __restrict__ final_obs,
                                         long long n, int dim) {
  const long long total = n * dim;
  for (long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x; k < total; k += (long long)gridDim.x * blockDim.x)
    if (done[k / dim]) final_obs[k] = obs[k];
}

// one launch of the capture in `stream`, at most 4 blocks of 256 threads per SM
template <typename T>
cudaError_t launch_final_obs_capture(const T* obs, const uint8_t* done, T* final_obs, int n, int dim, int sm_count,
                                     cudaStream_t stream) {
  long long blocks = ((long long)n * dim + 255) / 256;
  if (blocks > 4LL * sm_count) blocks = 4LL * sm_count;
  final_obs_capture_kernel<T><<<(unsigned)(blocks > 0 ? blocks : 1), 256, 0, stream>>>(obs, done, final_obs, n, dim);
  return cudaGetLastError();
}

}  // namespace earl
