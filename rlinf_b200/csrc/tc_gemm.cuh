// Host-side interface of the fp16-split tcgen05 GEMMs of the MLP towers (tc_gemm_h.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rb {
namespace tc {

constexpr int BM = 128, BN = 256, BK = 32;  // BK fp32 = 128 bytes = one swizzle span

enum Epi { EPI_STORE = 0, EPI_BIAS_TANH = 1, EPI_TANHGRAD = 2 };

}  // namespace tc

// ---- fp16-split tensor-core GEMMs, grouped over up to two towers per launch ---------------------------------------------
namespace tch {

struct GemmLaunch {        // one group (tower) of a forward / dgrad launch
  const float* a;          // [M,K] fp32 streamed operand (activations or activation gradients)
  const float* b_hi;       // PACKED fp16 weight tiles of w * 2^10 for this launch's mode (pack_weights): per k-block of 32
                           // one contiguous 32 KB block = hi tile | lo tile, pre-swizzled as the MMA reads them; b_mn = 0
                           // takes the forward pack, b_mn = 1 the dgrad pack
  const float* b_lo;       // unused (kept for the aggregate initialisers)
  float* c;                // [M,256] fp32 result
  const float* bias;       // EPI_BIAS_TANH
  const float* h;          // EPI_TANHGRAD: previous activation [M,256]
  float* colsum;           // EPI_TANHGRAD: [256] += column sums of the output, or NULL
  const float* amax_in;    // device max|a| (gradient operands: scaled into fp16 range), or NULL
  float* amax_out;         // EPI_TANHGRAD: atomicMax of |output| (feeds the next gradient GEMM), or NULL
};
struct WgradLaunch {
  const float* z;          // [n,256] activation gradients
  const float* h;          // [n,IN]  layer inputs
  float* dW;               // [256,IN] +=
  const float* amax_z;     // device max|z| or NULL
};
struct SplitSpec {
  const float* src;        // weight matrix [256 out, K in] fp32
  float* hi;               // forward pack: 256*K floats of storage (typed float*: the cache lives in the fp32 wsplit buffer)
  float* lo;               // dgrad pack (K == 256 only) or NULL
  int64_t n;               // 256 * K
};

// epi: rb::tc::Epi.  b_mn = 0: C = epi(A . W^T) (forward, W [256,K]);  b_mn = 1: C = epi(A . W) (dgrad, W [256,256]).
// The gradient sums of the two launches (dW of wgrad, the column sums of an EPI_TANHGRAD launch with colsum) are stored
// per sample chunk / CTA in `part` and added by rb::sum_partials in a fixed order: the result does not depend on the order
// in which CTAs finish.  `part` needs wgrad_part_floats / launch_part_floats floats (launch: may be NULL without colsum);
// calls sharing it must be stream-ordered.
int64_t launch_part_floats(int ngroups, int64_t M);
int64_t wgrad_part_floats(int ngroups, int64_t n, int IN);
int launch(const GemmLaunch* groups, int ngroups, int64_t M, int K, int epi, int b_mn, float* part, cudaStream_t st);
int wgrad(const WgradLaunch* groups, int ngroups, int64_t n, int IN, float* part, cudaStream_t st);
// Weight packs (one launch for all matrices).  Forward pack: k-block kb (32 input features) = the [256 out x 32 k] tile
// in the K-major SWIZZLE_64B layout, hi (16 KB) then lo (16 KB).  Dgrad pack: k-block kb (32 OUTPUT features = the
// reduction index of dZ . W) = four [32 out x 64 in] SWIZZLE_128B groups, hi (16 KB) then lo (16 KB).  Both are what
// TMA tensor loads of the plain [256, K] fp16 copies produced in the first version - as 512 / 256 row requests of 64 /
// 128 bytes per k-block, which is what bounded the kernel (tools/gemm_role_probe.py: 884 clk per k-block waiting for the
// weight tile); packed, a k-block is one 32 KB bulk copy.
int split_weights(const SplitSpec* specs, int count, cudaStream_t st);

}  // namespace tch
}  // namespace rb
