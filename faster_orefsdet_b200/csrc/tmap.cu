// Host side of TMA: tensor-map encoding through the driver entry point (no libcuda link).
#include "common.cuh"
#include "tc05.cuh"

namespace fod {

PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !p) {
    set_error("cuTensorMapEncodeTiled entry point not available: %s", cudaGetErrorString(e));
    return nullptr;
  }
  fn = reinterpret_cast<PFN_encodeTiled>(p);
  return fn;
}

int make_nhwc_map(CUtensorMap* out, const float* base, int N, int H, int W, int C, long pixel_stride, int bc, int bw, int bh,
                  int estride, CUtensorMapSwizzle swizzle) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return FOD_ERR_CUDA;
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)pixel_stride * 4, (cuuint64_t)W * pixel_stride * 4, (cuuint64_t)H * W * pixel_stride * 4};
  cuuint32_t box[4] = {(cuuint32_t)bc, (cuuint32_t)bw, (cuuint32_t)bh, 1};
  cuuint32_t estr[4] = {1, (cuuint32_t)estride, (cuuint32_t)estride, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<float*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for map [%d,%d,%d,%d] pixel stride %ld box [%d,%d,%d] element stride %d", (int)r,
              N, H, W, C, pixel_stride, bc, bw, bh, estride);
    return FOD_ERR_CUDA;
  }
  return FOD_OK;
}

int make_matrix_map(CUtensorMap* out, const float* base, long rows, long cols, int box_cols, int box_rows) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return FOD_ERR_CUDA;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 4};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for matrix [%ld,%ld] box [%d,%d]", (int)r, rows, cols, box_cols, box_rows);
    return FOD_ERR_CUDA;
  }
  return FOD_OK;
}

int make_matrix_map_f16(CUtensorMap* out, const void* base, long rows, long cols, int box_cols, int box_rows) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return FOD_ERR_CUDA;
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)cols * 2};
  cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d) for fp16 matrix [%ld,%ld] box [%d,%d]", (int)r, rows, cols, box_cols, box_rows);
    return FOD_ERR_CUDA;
  }
  return FOD_OK;
}

}  // namespace fod
