// The one TMA tensor-map builder of the library (declared in internal.cuh).
#include <cuda.h>

#include "internal.cuh"

namespace sg {

namespace {
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// the driver's tiled encoder, looked up through the runtime (no link dependency on libcuda); null when unavailable
EncodeTiledFn lookup_encode_tiled() {
  void* p = nullptr;
  cudaDriverEntryPointQueryResult q;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
      q == cudaDriverEntryPointSuccess)
    return reinterpret_cast<EncodeTiledFn>(p);
  (void)cudaGetLastError();
  return nullptr;
}
}  // namespace

bool make_tensor_map_2d(CUtensorMap* map, CUtensorMapDataType dtype, const void* base, uint64_t rows, uint64_t cols,
                        uint64_t pitch_bytes, uint32_t box_rows, uint32_t box_cols, CUtensorMapSwizzle swizzle) {
  static const EncodeTiledFn enc = lookup_encode_tiled();
  if (enc == nullptr) return false;
  const cuuint64_t dims[2] = {cols, rows};
  const cuuint64_t strides[1] = {pitch_bytes};
  const cuuint32_t box[2] = {box_cols, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  return enc(map, dtype, 2, const_cast<void*>(base), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
             CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace sg
