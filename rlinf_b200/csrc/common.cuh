// Shared helpers for the rlinf_b200 kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/rlinf_b200.h"

#define RB_CHECK_CUDA(expr)                                   \
  do {                                                        \
    cudaError_t _e = (expr);                                  \
    if (_e != cudaSuccess) return (int)_e;                    \
  } while (0)

#define RB_RETURN_LAUNCH()                                    \
  do {                                                        \
    cudaError_t _e = cudaPeekAtLastError();                   \
    return _e == cudaSuccess ? RB200_OK : (int)_e;            \
  } while (0)

namespace rb {

constexpr int kWarp = 32;

__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Block-wide sum of K doubles per thread; result valid in thread 0. blockDim.x multiple of 32, <=1024.
template <int K>
__device__ __forceinline__ void block_sum(double (&v)[K], double* smem /* K*32 doubles */) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = (blockDim.x + 31) >> 5;
#pragma unroll
  for (int k = 0; k < K; ++k) v[k] = warp_sum(v[k]);
  if (lane == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) smem[k * 32 + warp] = v[k];
  }
  __syncthreads();
  if (warp == 0) {
#pragma unroll
    for (int k = 0; k < K; ++k) {
      double x = lane < nwarp ? smem[k * 32 + lane] : 0.0;
      v[k] = warp_sum(x);
    }
  }
}

// number of kernels this library has launched (host-side counter; bench.py's gpu_launches)
void count_launch(int n = 1);

inline cudaStream_t as_stream(rb200_stream_t s) { return reinterpret_cast<cudaStream_t>(s); }

// Per-device scratch (reduction slots); allocated on first use, never freed.
double* device_scratch(int n_doubles_min);  // defined in abi.cu; returns nullptr on failure

// Cross-block sums without floating-point atomics, so that a result does not depend on the order in which blocks
// finish: each block stores its partial sums in a row of `part` (stride floats apart), then sum_partials adds the rows
// in a fixed order.  One segment per output array: out[k] += sum_b part[b * stride + off + k], k < K.
struct PartialSeg {
  float* out;
  int64_t off, K;
};
int sum_partials(const float* part, int nparts, int64_t stride, const PartialSeg* segs, int nseg, cudaStream_t st);

inline int sm_count() {
  static int cached[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
}

}  // namespace rb
