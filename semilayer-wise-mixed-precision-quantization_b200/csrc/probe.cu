// csrc/probe.cu -- measures the roofline denominator of the conv kernels ON THE BOX bench.py runs on:
// the dense kind::i8 rate of the 5th-generation tensor cores (SURVEY.md 8d: "expect INT8 ~ 2x bf16; measure it").
//
// Every SM runs one CTA whose two issuing warps stream tcgen05.mma.kind::i8 (M = 128, N = 256, K = 32,
// u8 x u8 -> s32, operands in 128-byte-swizzled shared memory, two TMEM accumulators) back to back with no
// loads in between: the tensor pipe's own speed (r1 measurement: 7518 MAC/clk/SM = 97 % of the nominal
// 8192).  bench.py times the launch with CUDA events -- once short (burst clocks) and once for >= 2 s
// (sustained, under the power cap) -- and divides the conv kernels' achieved ops by it.
#include "conv_common.cuh"
#include "tma_host.cuh"
#include "umma_ptx.cuh"

namespace slq {

constexpr int kProbeN = 256;
constexpr int kProbeSmem = 2 * (16384 + kProbeN * 128) + 1024;  // two {A, B} operand sets

__global__ void __launch_bounds__(128, 1) probe_i8_kernel(int iters) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem = smem_raw + (base - smem_u32(smem_raw));
  __shared__ uint32_t tmem_slot;
  __shared__ __align__(8) uint64_t bars[2][4];
  const int w = threadIdx.x >> 5;
  for (int i = threadIdx.x; i < (kProbeSmem - 1024) / 4; i += blockDim.x) reinterpret_cast<uint32_t *>(smem)[i] = 0x01010101u;
  if (threadIdx.x == 0) {
    for (int i = 0; i < 8; ++i) mbar_init(smem_u32(&bars[i >> 2][i & 3]), 1);
    fence_barrier_init();
  }
  if (w == 3) tmem_alloc(&tmem_slot, 512);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem = tmem_slot;
  if (w < 2) {
    const uint32_t bar0 = smem_u32(&bars[w][0]);
    const uint32_t idesc = (2u << 4) | ((uint32_t)(kProbeN >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    const uint64_t dflags = make_smem_desc<128>(0);
    const uint32_t acc = tmem + (uint32_t)w * 256u;
    const uint32_t lo = (((base + (uint32_t)w * (16384 + kProbeN * 128)) & 0x3FFFFu) >> 4);
    const uint64_t da = dflags | lo, db = dflags | (lo + (16384 >> 4));
    // One commit per 4 K blocks (16 MMAs), commit k on barrier k % 4; commit k - 3 is waited for before
    // commit k + 1 is issued.  A parity wait is only meaningful while the barrier is at most ONE phase ahead
    // of its waiter, hence a ring of four barriers: barrier j completes its phase n with commit 4n + j and
    // cannot complete phase n + 1 before the waiter has seen phase n (it has not issued that commit yet).
    uint32_t commits = 0, waited = 0;
    for (int i = 0; i < iters; ++i) {
      if (elect_one()) {
#pragma unroll
        for (int k = 0; k < 4; ++k) umma_i8(acc, da + 2 * k, db + 2 * k, idesc, 1);
        if ((i & 3) == 3) umma_commit(bar0 + 8u * (commits & 3));
      }
      __syncwarp();
      if ((i & 3) == 3) {
        ++commits;
        if (commits - waited > 3) { mbar_wait(bar0 + 8u * (waited & 3), (waited >> 2) & 1); ++waited; }
      }
    }
    for (; waited < commits; ++waited) mbar_wait(bar0 + 8u * (waited & 3), (waited >> 2) & 1);
  }
  tc_fence_before();
  __syncthreads();
  if (w == 3) {
    tc_fence_after();
    tmem_dealloc(tmem, 512);
  }
}

}  // namespace slq

using namespace slq;

extern "C" int slq_probe_i8_peak(int32_t iters, int64_t *ops_out, void *stream) {
  SLQ_CHECK_ARG(iters > 0 && (iters & 3) == 0, "slq_probe_i8_peak: iters must be a positive multiple of 4");
  SLQ_CUDA(set_smem_limit_once<probe_i8_kernel>(kProbeSmem));
  const int ctas = sm_count();
  probe_i8_kernel<<<ctas, 128, kProbeSmem, (cudaStream_t)stream>>>(iters);
  SLQ_LAUNCH_CHECK();
  // 2 warps x iters x 4 MMAs x (128 x 256 x 32) MACs, 2 ops per MAC
  if (ops_out) *ops_out = (int64_t)ctas * 2 * iters * 4 * (2LL * 128 * kProbeN * 32);
  return SLQ_OK;
}
