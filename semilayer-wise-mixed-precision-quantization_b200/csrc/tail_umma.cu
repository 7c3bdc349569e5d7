// csrc/tail_umma.cu -- the un-quantised tail of the network on the tensor cores.
//
// Replaces resnet.py:216-218: adaptive_avg_pool2d((1,1)) + flatten + fc (fp32 weights and bias; the reference
// keeps them in fp32, SURVEY.md F3).  Three launches:
//   avgpool_v2_kernel   u8 NHWC [N, HW, C] -> pooled fp32 [N, C]   (exact integer sums, one fp32 multiply)
//   fc_umma_kernel      split-K GEMM  partial[s][n][o] = sum_{k in split s} pooled[n][k] * W[o][k]
//                       TMA (fp32 tiles, 128-byte swizzle) -> tcgen05.mma.kind::tf32 (fp32 accumulate in TMEM)
//                       M = 128 images, N = 128 outputs, K = C / splits per CTA: 2 x 8 x 8 = 128 CTAs for the
//                       256 x 1000 x 2048 problem (a single pass over K on 16 CTAs would be bound by one SM's
//                       L2 path)
//   fc_reduce_kernel    logits[n][o] = (sum over splits, FIXED order) + bias[o]
// Round 1 ran this GEMM on the CUDA cores (55 us of a 2.3 ms step).  A TF32 operand carries a 10-bit significand,
// so BOTH operands are split into two TF32 terms, x = x_hi + x_lo with x_hi = x truncated to TF32 and x_lo the
// exact remainder, and the product is taken as  a_lo*w_hi + a_hi*w_lo + a_hi*w_hi  (three passes over K into the
// same fp32 accumulator; the dropped a_lo*w_lo term is ~2^-20 relative): fp32-class accuracy for weights the
// reference keeps in fp32, at three times a cost that is small to begin with.  Bias and the reduction over the
// splits are fp32.
#include <algorithm>

#include "conv_common.cuh"
#include "tma_host.cuh"
#include "umma_ptx.cuh"

namespace slq {

// x truncated to TF32 (sign, 8-bit exponent, 10-bit significand): exactly representable, so the tensor core adds no
// rounding of its own; x - tf32_hi(x) is exact in fp32
__device__ __forceinline__ float tf32_hi(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }

// fc weights -> {hi, lo} planes: w2[0][i] = tf32_hi(w[i]), w2[1][i] = w[i] - w2[0][i]
__global__ void __launch_bounds__(256) fc_split_kernel(const float *__restrict__ w, long long n, float *__restrict__ w2) {
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = w[i], h = tf32_hi(v);
    w2[i] = h;
    w2[n + i] = __fsub_rn(v, h);
  }
}

// ------------------------------------------------------------------------------------------
// global average pool: one CTA per image; a thread owns 16 channels (16-byte loads) of ONE PART of the image's
// pixels -- 512 threads = C/16 channel groups x P pixel parts, every load of a thread in flight at once -- and the
// parts meet in shared memory (integer atomics: exact, order-free).  One CTA of 128 threads walking all 49 pixels
// (round 2's first version) kept 7 loads per thread in flight: 20.7 us for 25.7 MB.
// ------------------------------------------------------------------------------------------
constexpr int kPoolThreads = 512;
constexpr int kPoolMaxPix = 16;  // pixels per thread and pass (unrolled: that many 16-byte loads in flight)

__global__ void __launch_bounds__(kPoolThreads) avgpool_v2_kernel(const uint8_t *__restrict__ x, int HW, int C,
                                                                  const float *__restrict__ act_scales, int in_id,
                                                                  float *__restrict__ pooled_hi, float *__restrict__ pooled_lo) {
  extern __shared__ uint32_t pool_sum[];  // [16][C / 16]: channel 16 g + j at j * groups + g
  const int n = blockIdx.x;
  const int groups = C / 16;
  for (int i = threadIdx.x; i < C; i += blockDim.x) pool_sum[i] = 0;
  __syncthreads();
  const int gpp = groups < (int)blockDim.x ? groups : (int)blockDim.x;  // channel groups per pass
  const int P = (int)blockDim.x / gpp;                                  // pixel parts
  const int part = threadIdx.x / gpp, gl = threadIdx.x - part * gpp;
  const int per = (HW + P - 1) / P;
  const int i0 = part * per, i1 = min(HW, i0 + per);
  if (part < P) {
    for (int g = gl; g < groups; g += gpp) {
      const uint4 *p = reinterpret_cast<const uint4 *>(x + (long long)n * HW * C) + g;
      unsigned s[16];
#pragma unroll
      for (int j = 0; j < 16; ++j) s[j] = 0;
      for (int ib = i0; ib < i1; ib += kPoolMaxPix) {
        uint4 v[kPoolMaxPix];
#pragma unroll
        for (int k = 0; k < kPoolMaxPix; ++k)
          v[k] = ib + k < i1 ? __ldg(p + (long long)(ib + k) * groups) : make_uint4(0, 0, 0, 0);
#pragma unroll
        for (int k = 0; k < kPoolMaxPix; ++k) {
          const uint32_t w[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            s[4 * q] += w[q] & 255; s[4 * q + 1] += (w[q] >> 8) & 255;
            s[4 * q + 2] += (w[q] >> 16) & 255; s[4 * q + 3] += w[q] >> 24;
          }
        }
      }
#pragma unroll
      for (int j = 0; j < 16; ++j) atomicAdd(&pool_sum[j * groups + g], s[j]);  // channel 16 g + j; conflict-free
    }
  }
  __syncthreads();
  const float k = __fdiv_rn(act_scales[in_id], (float)HW);
  for (int c4 = threadIdx.x; c4 * 4 < C; c4 += blockDim.x) {
    float v[4], h[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      v[e] = __fmul_rn((float)pool_sum[((4 * c4 + e) & 15) * groups + (c4 >> 2)], k);
      h[e] = tf32_hi(v[e]);
    }
    reinterpret_cast<float4 *>(pooled_hi + (long long)n * C)[c4] = make_float4(h[0], h[1], h[2], h[3]);
    reinterpret_cast<float4 *>(pooled_lo + (long long)n * C)[c4] =
        make_float4(__fsub_rn(v[0], h[0]), __fsub_rn(v[1], h[1]), __fsub_rn(v[2], h[2]), __fsub_rn(v[3], h[3]));
  }
}

// ------------------------------------------------------------------------------------------
// split-K TF32 GEMM
// ------------------------------------------------------------------------------------------
constexpr int kFcStages = 4;
constexpr int kFcTileBytes = 128 * 128;                     // 128 rows x 32 floats
constexpr int kFcSmemBytes = 1024 + kFcStages * 2 * kFcTileBytes + 256;
constexpr int kFcThreads = 192;                             // warp 0 TMA, warp 1 MMA, warps 2-5 epilogue

__global__ void __launch_bounds__(kFcThreads, 1) fc_umma_kernel(const __grid_constant__ CUtensorMap tmAhi,
                                                                const __grid_constant__ CUtensorMap tmAlo,
                                                                const __grid_constant__ CUtensorMap tmBhi,
                                                                const __grid_constant__ CUtensorMap tmBlo, int N, int O,
                                                                int kb_per_split, float *__restrict__ partial) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + kFcStages * 2 * kFcTileBytes;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kFcStages + s); };
  const uint32_t tfull_bar = bar_base + 8u * (2 * kFcStages);
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem + kFcStages * 2 * kFcTileBytes + 8 * (2 * kFcStages + 1));
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const int n_tile = blockIdx.x, m_tile = blockIdx.y, split = blockIdx.z;
  if (threadIdx.x == 0) {
    prefetch_tmap(&tmAhi);
    prefetch_tmap(&tmAlo);
    prefetch_tmap(&tmBhi);
    prefetch_tmap(&tmBlo);
    for (int s = 0; s < kFcStages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tfull_bar, 1);
    fence_barrier_init();
  }
  if (warp == 1) tmem_alloc(tmem_slot, 128);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int kb0 = split * kb_per_split;
  const int steps = 3 * kb_per_split;  // three passes over this CTA's K range: lo*hi, hi*lo, hi*hi
  if (warp == 0) {
    for (int i = 0; i < steps; ++i) {
      const int s = i % kFcStages;
      const int seg = i / kb_per_split, kb = kb0 + (i - seg * kb_per_split);
      mbar_wait(empty_bar(s), (uint32_t)(((i / kFcStages) & 1) ^ 1));
      if (elect_one()) {
        const uint32_t sa = smem_base + s * 2 * kFcTileBytes;
        mbar_expect_tx(full_bar(s), 2 * kFcTileBytes);  // rows past N / O are zero-filled by the TMA and still counted
        tma_load_2d(sa, seg == 0 ? &tmAlo : &tmAhi, full_bar(s), kb * 32, m_tile * 128);
        tma_load_2d(sa + kFcTileBytes, seg == 1 ? &tmBlo : &tmBhi, full_bar(s), kb * 32, n_tile * 128);
      }
      __syncwarp();
    }
  } else if (warp == 1) {
    // instruction descriptor: D = f32, A = B = tf32 (K-major), M = 128, N = 128
    const uint32_t idesc = (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    for (int i = 0; i < steps; ++i) {
      const int s = i % kFcStages;
      mbar_wait(full_bar(s), (uint32_t)((i / kFcStages) & 1));
      tc_fence_after();
      if (elect_one()) {
        const uint64_t da = make_smem_desc<128>(smem_base + s * 2 * kFcTileBytes);
        const uint64_t db = make_smem_desc<128>(smem_base + s * 2 * kFcTileBytes + kFcTileBytes);
#pragma unroll
        for (int k = 0; k < 4; ++k)  // UMMA_K = 8 tf32 = 32 bytes
          umma_tf32(tmem_base, da + 2 * k, db + 2 * k, idesc, (uint32_t)((i | k) != 0));
        umma_commit(empty_bar(s));
        if (i == steps - 1) umma_commit(tfull_bar);
      }
      __syncwarp();
    }
  } else {
    const int wq = warp & 3;  // TMEM lane quarter of this warp (warps 2..5 -> 2, 3, 0, 1)
    const int row = wq * 32 + lane;
    const int n = m_tile * 128 + row;
    mbar_wait(tfull_bar, 0);
    tc_fence_after();
    float *dst = partial + ((long long)split * N + n) * O + n_tile * 128;
#pragma unroll 1
    for (int c0 = 0; c0 < 128; c0 += 32) {
      uint32_t v[32];
      tmem_ld32(tmem_base + ((uint32_t)(wq * 32) << 16) + c0, v);
      tmem_ld_wait();
      if (n < N) {
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const int o = n_tile * 128 + c0 + j;
          if (o + 3 < O && (O & 3) == 0) {
            *reinterpret_cast<float4 *>(dst + c0 + j) = make_float4(__uint_as_float(v[j]), __uint_as_float(v[j + 1]),
                                                                    __uint_as_float(v[j + 2]), __uint_as_float(v[j + 3]));
          } else {
            for (int e = 0; e < 4; ++e)
              if (o + e < O) dst[c0 + j + e] = __uint_as_float(v[j + e]);
          }
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 128);
  }
}

__global__ void __launch_bounds__(256) fc_reduce_kernel(const float *__restrict__ partial, int splits, int N, int O,
                                                        const float *__restrict__ bias, float *__restrict__ logits) {
  const long long total = (long long)N * O;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    float acc = partial[i];
    for (int s = 1; s < splits; ++s) acc = __fadd_rn(acc, partial[(long long)s * total + i]);
    logits[i] = __fadd_rn(acc, bias[(int)(i % O)]);
  }
}

// [rows, K] fp32 matrix, box = 32 floats (128 bytes) x 128 rows
static int encode_f32_rows(CUtensorMap *tm, const float *ptr, int rows, int K) {
  const cuuint64_t dims[2] = {(cuuint64_t)K, (cuuint64_t)rows};
  const cuuint64_t strides[1] = {(cuuint64_t)K * 4};
  const cuuint32_t box[2] = {32, 128};
  return encode_tiled(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, ptr, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B,
                      "fc operand");
}

static int fc_splits(int C) {
  int splits = 8;
  while (splits > 1 && (C / 32) % splits != 0) splits >>= 1;
  return splits;
}

}  // namespace slq

using namespace slq;

extern "C" int64_t slq_tail_workspace_bytes(int32_t N, int32_t C, int32_t O) {
  if (N <= 0 || C <= 0 || O <= 0) return -1;
  return (2 * (int64_t)N * C + (int64_t)fc_splits(C) * N * O) * 4;
}

extern "C" int slq_tail_split_weights(const float *fc_w, int32_t O, int32_t C, float *fc_w_split, void *stream) {
  SLQ_CHECK_ARG(fc_w && fc_w_split && O > 0 && C > 0, "slq_tail_split_weights: bad argument");
  const long long n = (long long)O * C;
  fc_split_kernel<<<(unsigned)std::min<long long>(ceil_div(n, 256), (long long)sm_count() * 8), 256, 0, (cudaStream_t)stream>>>(
      fc_w, n, fc_w_split);
  SLQ_LAUNCH_CHECK();
  return SLQ_OK;
}

extern "C" int slq_tail_forward(const uint8_t *x, int32_t N, int32_t HW, int32_t C, const float *act_scales,
                                int32_t in_id, const float *fc_w_split, const float *fc_b, int32_t O, float *workspace,
                                float *logits, void *stream) {
  const float *fc_w = fc_w_split;
  SLQ_CHECK_ARG(x && act_scales && fc_w && fc_b && workspace && logits, "slq_tail_forward: null pointer argument");
  SLQ_CHECK_ARG(N > 0 && HW > 0 && C > 0 && C % 32 == 0 && C <= 12288 && O > 0,
                "slq_tail_forward: bad shape (C must be a multiple of 32, at most 12288: the pool keeps C sums in shared memory)");
  SLQ_CHECK_ARG(reinterpret_cast<uintptr_t>(x) % 16 == 0 && reinterpret_cast<uintptr_t>(fc_w) % 16 == 0 &&
                    reinterpret_cast<uintptr_t>(workspace) % 16 == 0,
                "slq_tail_forward: x, fc_w and workspace must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  float *pooled_hi = workspace, *pooled_lo = workspace + (int64_t)N * C, *partial = workspace + 2 * (int64_t)N * C;
  avgpool_v2_kernel<<<N, kPoolThreads, (size_t)C * 4, st>>>(x, HW, C, act_scales, in_id, pooled_hi, pooled_lo);
  SLQ_LAUNCH_CHECK();
  CUtensorMap tmAhi, tmAlo, tmBhi, tmBlo;
  int rc = encode_f32_rows(&tmAhi, pooled_hi, N, C);
  if (rc == SLQ_OK) rc = encode_f32_rows(&tmAlo, pooled_lo, N, C);
  if (rc == SLQ_OK) rc = encode_f32_rows(&tmBhi, fc_w, O, C);
  if (rc == SLQ_OK) rc = encode_f32_rows(&tmBlo, fc_w + (int64_t)O * C, O, C);
  if (rc != SLQ_OK) return rc;
  SLQ_CUDA(set_smem_limit_once<fc_umma_kernel>(kFcSmemBytes));
  const int splits = fc_splits(C);
  dim3 grid((unsigned)ceil_div(O, 128), (unsigned)ceil_div(N, 128), (unsigned)splits);
  fc_umma_kernel<<<grid, kFcThreads, kFcSmemBytes, st>>>(tmAhi, tmAlo, tmBhi, tmBlo, N, O, C / 32 / splits, partial);
  SLQ_LAUNCH_CHECK();
  const long long total = (long long)N * O;
  fc_reduce_kernel<<<(unsigned)std::min<long long>(ceil_div(total, 256), (long long)sm_count() * 8), 256, 0, st>>>(
      partial, splits, N, O, fc_b, logits);
  SLQ_LAUNCH_CHECK();
  return SLQ_OK;
}
