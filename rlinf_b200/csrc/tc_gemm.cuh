// Host-side interface of the tcgen05 3xTF32 GEMMs (tc_gemm.cu).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace rb {
namespace tc {

constexpr int BM = 128, BN = 256, BK = 32;  // BK fp32 = 128 bytes = one swizzle span

enum Epi { EPI_STORE = 0, EPI_BIAS_TANH = 1, EPI_TANHGRAD = 2 };

struct Params {
  int64_t M;
  int K;              // multiple of 32
  const float* bias;  // [256]                         (EPI_BIAS_TANH)
  const float* h;     // [M,256] previous activation   (EPI_TANHGRAD: out = acc * (1 - h^2))
  float* c;           // [M,256] fp32 result
  float* colsum;      // [256] += column sums of the output (bias gradient of the producing layer), or NULL
  int epi;
};

// debug/experiment switches (rb200_debug_set_flags): bit 0 = also mask the streamed operand's hi part in shared memory
// (default off: the tensor core ignores the low 13 mantissa bits of a kind::tf32 operand - verified bit-identical), bit 1 (2) = round-1
// fused-rollout layers (one-k-step weight prefetch), bit 3 (8) = round-1 3xTF32 GEMMs instead of the fp16-split kernels, bit 5 (32) = one
// fp16-split GEMM launch per tower, bit 6 (64) = 8 transform warps in the fp16-split forward kernel, bits 8-15 = TF32 kernels' L2
// prefetch distance in k-blocks (0 = default)
extern int g_debug_flags;

// C[M,256] = epi( A[M,K] . (B_hi+B_lo)[256,K]^T ).  A is plain fp32 (split into exact-TF32 hi/lo inside the kernel);
// B is a pre-split weight matrix (rb::tc::split).  All pointers 16-byte aligned.
int launch(const float* a, const float* b_hi, const float* b_lo, const Params& p, cudaStream_t st);
// dW[256, IN] += Z[n,256]^T . H[n,IN]   (IN % 32 == 0, <= 256), plain fp32 operands, fp32 atomics into dW
int wgrad(const float* z, const float* h, float* dW, int64_t n, int IN, cudaStream_t st);
// x -> (hi, lo) exact-TF32 pair, hi + lo ~= x to 2^-21 relative; hi may alias x.
int split(const float* x, float* hi, float* lo, int64_t n, cudaStream_t st);
// out[c][r] = split(x[r][c]) for a small [R,C] matrix
int split_transpose(const float* x, float* hi, float* lo, int R, int C, cudaStream_t st);

}  // namespace tc

// ---- round 2: fp16-split tensor-core GEMMs (tc_gemm_h.cu), grouped over up to two towers per launch -------------------
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
