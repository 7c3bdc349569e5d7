// csrc/tma_host.cu -- TMA tensor-map encoding for the tcgen05 kernels (see tma_host.cuh).
#include "tma_host.cuh"

namespace slq {

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *,
                                  CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                  CUtensorMapFloatOOBfill);
typedef CUresult (*EncodeIm2colFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                   const cuuint64_t *, const int *, const int *, cuuint32_t, cuuint32_t,
                                   const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                   CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// the driver's encoders, looked up on first use (the library links the runtime only, not libcuda)
static int get_encoders(EncodeTiledFn *tiled, EncodeIm2colFn *im2col) {
  static EncodeTiledFn f_tiled = nullptr;
  static EncodeIm2colFn f_im2col = nullptr;
  if (!f_tiled || !f_im2col) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult qr;
    SLQ_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qr));
    if (qr != cudaDriverEntryPointSuccess || !p) {
      set_error("cuTensorMapEncodeTiled not available from the driver");
      return SLQ_ERR_CUDA;
    }
    f_tiled = (EncodeTiledFn)p;
    p = nullptr;
    SLQ_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &p, cudaEnableDefault, &qr));
    if (qr != cudaDriverEntryPointSuccess || !p) {
      set_error("cuTensorMapEncodeIm2col not available from the driver");
      return SLQ_ERR_CUDA;
    }
    f_im2col = (EncodeIm2colFn)p;
  }
  *tiled = f_tiled;
  *im2col = f_im2col;
  return SLQ_OK;
}

int encode_tiled(CUtensorMap *tm, CUtensorMapDataType dtype, int rank, const void *ptr, const cuuint64_t *dims,
                 const cuuint64_t *strides_bytes, const cuuint32_t *box, CUtensorMapSwizzle swizzle, const char *what) {
  EncodeTiledFn enc_tiled;
  EncodeIm2colFn enc_im2col;
  int rc = get_encoders(&enc_tiled, &enc_im2col);
  if (rc != SLQ_OK) return rc;
  const cuuint32_t es[3] = {1, 1, 1};
  const CUresult r = enc_tiled(tm, dtype, (cuuint32_t)rank, const_cast<void *>(ptr), dims, strides_bytes, box, es,
                               CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled(%s) failed: CUresult %d", what, (int)r);
    return SLQ_ERR_CUDA;
  }
  return SLQ_OK;
}

int encode_tiled_u8(CUtensorMap *tm, const void *ptr, long long rows, int cols, int box_cols, int box_rows,
                    CUtensorMapSwizzle swizzle, const char *what) {
  const cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)cols};
  const cuuint32_t box[2] = {(cuuint32_t)box_cols, (cuuint32_t)box_rows};
  return encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, ptr, dims, strides, box, swizzle, what);
}

int encode_im2col_u8(CUtensorMap *tm, const void *ptr, int N, int H, int W, int C, const int lower[2],
                     const int upper[2], int stride, int channels, int pixels, CUtensorMapSwizzle swizzle,
                     const char *what) {
  EncodeTiledFn enc_tiled;
  EncodeIm2colFn enc_im2col;
  int rc = get_encoders(&enc_tiled, &enc_im2col);
  if (rc != SLQ_OK) return rc;
  const cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  const cuuint64_t strides[3] = {(cuuint64_t)C, (cuuint64_t)W * C, (cuuint64_t)H * W * C};
  const cuuint32_t es[4] = {1, (cuuint32_t)stride, (cuuint32_t)stride, 1};
  const CUresult r = enc_im2col(tm, CU_TENSOR_MAP_DATA_TYPE_UINT8, 4, const_cast<void *>(ptr), dims, strides, lower,
                                upper, (cuuint32_t)channels, (cuuint32_t)pixels, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                swizzle, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeIm2col(%s) failed: CUresult %d", what, (int)r);
    return SLQ_ERR_CUDA;
  }
  // Known driver issue (<= 13.1): im2col maps of tensors below 128 KiB come back with bit 21 of
  // the second descriptor word set and then fault; CUTLASS clears it the same way.
  int drv = 0;
  if (cudaDriverGetVersion(&drv) == cudaSuccess && drv <= 13010 && (long long)N * H * W * C < 131072)
    reinterpret_cast<uint64_t *>(tm)[1] &= ~(1ull << 21);
  return SLQ_OK;
}

}  // namespace slq
