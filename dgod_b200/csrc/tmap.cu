// Host side of tmap.cuh: tensor maps are encoded by the driver (cuTensorMapEncodeTiled); the entry point is
// fetched through the runtime so that libdgod_b200.so needs no link-time dependency on libcuda.
#include "tmap.cuh"

namespace dgod {

PFN_cuTensorMapEncodeTiled tensor_map_encoder() {
  static PFN_cuTensorMapEncodeTiled fn = nullptr;
  static bool looked = false;
  if (!looked) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_cuTensorMapEncodeTiled>(p);
    else
      (void)cudaGetLastError();
    looked = true;
  }
  return fn;
}

int encode_words_2d(CUtensorMap* map, const void* base, unsigned long long rows, unsigned row_words, unsigned box_rows) {
  PFN_cuTensorMapEncodeTiled enc = tensor_map_encoder();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from this driver");
    return DGOD_ERR_CUDA;
  }
  const cuuint64_t dims[2] = {row_words, rows ? rows : 1};
  const cuuint64_t strides[1] = {(cuuint64_t)row_words * 4};
  const cuuint32_t box[2] = {row_words, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with code %d (rows %llu, row_words %u, box_rows %u)", (int)r, rows, row_words, box_rows);
    return DGOD_ERR_CUDA;
  }
  return DGOD_OK;
}

int encode_f32_2d_sw128(CUtensorMap* map, const void* base, unsigned long long rows, unsigned long long cols, unsigned box_rows) {
  PFN_cuTensorMapEncodeTiled enc = tensor_map_encoder();
  if (!enc) {
    set_error("cuTensorMapEncodeTiled is not available from this driver");
    return DGOD_ERR_CUDA;
  }
  const cuuint64_t dims[2] = {cols, rows};
  const cuuint64_t strides[1] = {(cuuint64_t)cols * 4};
  const cuuint32_t box[2] = {32, box_rows};
  const cuuint32_t estr[2] = {1, 1};
  const CUresult r = enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<void*>(base), dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed with code %d (rows %llu, cols %llu, box_rows %u)", (int)r, rows, cols, box_rows);
    return DGOD_ERR_CUDA;
  }
  return DGOD_OK;
}

}  // namespace dgod
