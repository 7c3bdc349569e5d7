// csrc/tma_host.cuh -- host side of the tcgen05 kernels: TMA tensor-map encoding, the once-per-device shared-memory
// limit and the programmatic-dependent launch.  The encoders live in tma_host.cu.
#pragma once
#include <cuda.h>

#include <utility>

#include "common.cuh"

namespace slq {

// Tiled map over a tensor of rank <= 3 (dims innermost first, rank - 1 byte strides of the outer dims), element
// strides 1.  `what` names the operand in the error message.  SLQ_OK or SLQ_ERR_CUDA (message set).
int encode_tiled(CUtensorMap *tm, CUtensorMapDataType dtype, int rank, const void *ptr, const cuuint64_t *dims,
                 const cuuint64_t *strides_bytes, const cuuint32_t *box, CUtensorMapSwizzle swizzle, const char *what);

// [rows, cols] u8 matrix, box = box_cols x box_rows
int encode_tiled_u8(CUtensorMap *tm, const void *ptr, long long rows, int cols, int box_cols, int box_rows,
                    CUtensorMapSwizzle swizzle, const char *what);

// NHWC u8 tensor [N, H, W, C] in im2col mode: each load is `pixels` base pixels, `stride` apart in W and H, times
// `channels` channels; the filter window runs from lower to upper ({W, H}) around the base pixel.
int encode_im2col_u8(CUtensorMap *tm, const void *ptr, int N, int H, int W, int C, const int lower[2],
                     const int upper[2], int stride, int channels, int pixels, CUtensorMapSwizzle swizzle,
                     const char *what);

// Raises the dynamic shared-memory limit of Kernel to `bytes`, once per device (function attributes are per device).
template <auto Kernel>
cudaError_t set_smem_limit_once(int bytes) {
  static bool done[kMaxDevices] = {false};
  const int dev = current_device();
  if (dev < kMaxDevices && done[dev]) return cudaSuccess;
  const cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess && dev < kMaxDevices) done[dev] = true;
  return e;
}

// Programmatic dependent launch: the grid's CTAs may start (barrier / TMEM set-up, resident weights) on an SM as soon
// as the previous kernel's CTA there has exited; griddepcontrol.wait in the kernel holds everything that touches the
// previous kernel's outputs until that grid has completed.
template <typename... Params, typename... Args>
cudaError_t launch_pdl(void (*kernel)(Params...), int grid, int block, int smem_bytes, cudaStream_t st,
                       Args &&...args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3((unsigned)block);
  cfg.dynamicSmemBytes = (size_t)smem_bytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

}  // namespace slq
