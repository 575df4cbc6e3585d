#include "tma.cuh"
#include <cudaTypedefs.h>

namespace rb {

static PFN_cuTensorMapEncodeTiled_v12000 get_encode() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled_v12000>(p);
  }
  return fn;
}

int encode_tmap_2d(CUtensorMap* out, const void* base, int elem_bytes, uint64_t rows, uint64_t cols,
                   uint32_t box_rows, uint32_t box_cols) {
  auto enc = get_encode();
  if (!enc) return -1;
  CUtensorMapDataType dt;
  switch (elem_bytes) {
    case 1: dt = CU_TENSOR_MAP_DATA_TYPE_UINT8; break;
    case 4: dt = CU_TENSOR_MAP_DATA_TYPE_FLOAT32; break;
    default: return -2;
  }
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * (uint64_t)elem_bytes};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, dt, 2, const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)r;
}


namespace tch {
// fp32 [rows, cols] row-major, box [box_rows x 32 floats], SWIZZLE_128B (landing tiles of the fp16-split kernels)
int encode_f32_sw128(CUtensorMap* out, const float* base, uint64_t rows, uint64_t cols, uint32_t box_rows) {
  auto enc = get_encode();
  if (!enc) return -1;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * 4ull};
  cuuint32_t box[2] = {32u, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)r;
}
// fp16 [rows, cols] row-major, box [box_rows x box_cols], SWIZZLE_64B / SWIZZLE_128B (pre-split weight copies)
int encode_f16(CUtensorMap* out, const void* base, uint64_t rows, uint64_t cols, uint32_t box_cols, uint32_t box_rows,
               int swizzle_bytes) {
  auto enc = get_encode();
  if (!enc) return -1;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * 2ull};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  const CUtensorMapSwizzle swz = swizzle_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : (int)r;
}
}  // namespace tch

}  // namespace rb
