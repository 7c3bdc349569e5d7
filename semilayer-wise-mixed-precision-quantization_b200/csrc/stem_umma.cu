// csrc/stem_umma.cu -- the un-quantised stem on Blackwell tensor cores, ONE fused kernel.
//
// Replaces resnet.py:206-209 (conv1 7x7 s2 p3, 3->64, fp32 weights; bn1; relu; maxpool 3x3 s2 p1).
// The reference keeps these weights in fp32 (SURVEY.md F3), so this layer is NOT quantised to 8 bit:
// operands go through the tensor core as fp16 (11-bit significand, fp32 accumulation in TMEM),
// a relative error ~3e-4, an order of magnitude below the u8 activation quantisation that follows.
//
// Data path: the fp32 NCHW image is read from HBM exactly once and the pooled u8 NHWC tensor is
// written exactly once; im2col, the conv output and the pre-pool rows never leave the SM.
//   work unit  = (image, 14 pooled rows) -> 29 conv rows (one recomputed at the seam), units are
//                dealt round-robin to one persistent CTA per SM
//   builders   (warps 0-15) fp32 input rows -> fp16 row ring in smem (next row's loads are in flight
//                while this row is built) -> implicit-GEMM A tile of one conv row in the UMMA
//                K-major SWIZZLE_128B layout: row = output column q, K = (c, r, s padded to 8):
//                every 16-byte chunk is the 8 consecutive input pixels x[c][2p-3+r][2q-3 .. 2q+4]
//   MMA        (warps 24,25) D[128 x 64] = A[128 x 192] * W[64 x 192]^T, tcgen05.mma kind::f16, weights
//                resident in smem, A and the TMEM accumulator double-buffered.  One thread gets a
//                tcgen05.mma out only every ~100 cycles whatever its size (32 tensor cycles here), so
//                even and odd conv rows are issued by two different warps
//   epilogue   (warps 16-23) tcgen05.ld -> folded BN + ReLU -> u8 (scale of the POOLED tensor: max
//                commutes with a monotone map) -> 4-row ring in smem -> 3x3/s2 max-pool -> coalesced
//                stores of the pooled row
// Calibration (SLQ_OUT_F32) writes the fp32 conv rows to a scratch tensor and pools them with the
// fp32 pool kernel of layers.cu.
#include <algorithm>
#include <cstdlib>
#include <cuda_fp16.h>
#include <new>

#include "conv_common.cuh"
#include "tma_host.cuh"
#include "umma_ptx.cuh"

struct slq_stem {
  int N, H, W, Hc, Wc, Hp, Wp;
  __half *wh;  // [64, 192] fp16, zero padded; K order of the kernel in use (see the two weight kernels)
  float *wf;   // the same matrix in fp32 (stem_ts_kernel folds the BN scale into it before rounding to fp16)
  int num_ctas;
  int use_ts;  // 1: stem_ts_kernel (A operand in TMEM; needs 16-byte input rows: W % 16 == 0), 0: stem_fused_kernel
};

namespace slq {

constexpr int kSfK = 192;                       // padded K: 24 chunks of 8 halfs (21 real)
constexpr int kSfChunks = 24;
constexpr int kSfABytes = 3 * 16384;            // one A tile: 3 K blocks x (128 rows x 128 B)
constexpr int kSfBBytes = 3 * 8192;             // weights: 3 K blocks x (64 rows x 128 B)
constexpr int kSfRowP = 264;                    // halfs per ring row: column cc = w + 3, w in [-3, 2*127+4]
constexpr int kSfRing = 16;                     // input rows kept (7 live + 2 arriving fit twice)
constexpr int kSfRingBytes = kSfRing * 3 * kSfRowP * 2;
constexpr int kSfConvRing = 4;                  // u8 conv rows kept for pooling
constexpr int kSfConvRowBytes = 128 * 64;
constexpr int kSfAOff = 0;
constexpr int kSfBOff = kSfAOff + 2 * kSfABytes;
constexpr int kSfRingOff = kSfBOff + kSfBBytes;
constexpr int kSfConvOff = kSfRingOff + ((kSfRingBytes + 1023) / 1024) * 1024;
constexpr int kSfPrmOff = kSfConvOff + kSfConvRing * kSfConvRowBytes;
constexpr int kSfBarOff = kSfPrmOff + 64 * 8;
constexpr int kSfSmemBytes = 1024 + kSfBarOff + 128;
constexpr int kSfThreads = 26 * 32;  // 16 builder + 8 epilogue + 2 MMA warps
constexpr int kSfBuilders = 512, kSfEpi = 256;
constexpr int kSfBW = kSfBuilders / 32;          // builder warps; epilogue = warps kSfBW..kSfBW+7, MMA = the last two
constexpr int kSfUnitRows = 14;                 // pooled rows per work unit
constexpr int kSfTmemCols = 128;                // 2 accumulators x 64 columns
static_assert(kSfSmemBytes <= 232448, "stem kernel exceeds 227 KB of shared memory");

// w fp32 [64, 3, 7, 7] -> wh fp16 [64, 192]: wh[oc][(c*7 + r)*8 + s], zero for s == 7 and the pad chunks
__global__ void stem_weights_kernel(const float *__restrict__ w, __half *__restrict__ wh) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * kSfK) return;
  const int k = idx % kSfK, oc = idx / kSfK;
  const int chunk = k >> 3, s = k & 7;
  float v = 0.f;
  if (chunk < 21 && s < 7) {
    const int c = chunk / 7, r = chunk % 7;
    v = w[((oc * 3 + c) * 7 + r) * 7 + s];
  }
  wh[idx] = __float2half_rn(v);
}

struct StemArgs {
  const void *x;       // [N,3,H,W]: fp32 | fp16 | u8 (slq_stem_launch_in)
  float nmean[3], nstd[3];  // u8 input: value = (u/255 - mean[c]) / std[c]  (imagenet.py:14-15 ToTensor + Normalize)
  int N, H, W, Hc, Wc, Hp, Wp;
  const __half *wh;
  const float *wf;
  const float *bn_a, *bn_b, *act_scales;
  int out_id, out_mode;
  void *out;  // u8 pooled [N,Hp,Wp,64]  |  fp32 conv rows [N,Hc,Wc,64] (SLQ_OUT_F32)
  uint32_t *out_rowsum;  // [N*Hp*Wp] channel sum of every pooled u8 pixel (or NULL): slq_epilogue.in_rowsum of layer 1
  int units_per_img, total_units;
  long long *trace;  // debug timeline of CTA 0 (slq_debug_set_trace): 24 issuers x cap/24 events
  int trace_cap;
  int dbg;  // $SLQ_STEM_DBG bit mask (timing experiments only): 1 skip A build, 2 skip pooling, 4 skip epilogue math
};

#define SF_DBG(a) (kDebugTrace ? (a).dbg : 0)
__device__ __forceinline__ void stem_trace(const StemArgs &a, int issuer, int &n, int ev, int idx) {
  if (!kDebugTrace || a.trace == nullptr || blockIdx.x != 0) return;
  const int per = a.trace_cap / 24;
  if (n < per) {
    long long *p = a.trace + 3LL * (issuer * per + n);
    p[0] = ev + 1;
    p[1] = idx;
    p[2] = clock64();
    ++n;
  }
}

// A load whose ISSUE POINT the compiler must keep: __ldg() is an invariant load that gets sunk to its
// first use (after the A-tile build), which exposes the whole DRAM latency once per conv row.
// IN selects the element type of the image in HBM (SLQ_IN_*); the value is returned RAW (fp32 bits, fp16
// bits or the byte) and turned into the fp32 pixel by stem_pixel() after the build, so that only the
// load itself is pinned.
template <int IN>
__device__ __forceinline__ uint32_t ldg_pinned(const void *base, long long idx) {
  uint32_t v;
  if (IN == SLQ_IN_F32) asm volatile("ld.global.nc.b32 %0, [%1];" : "=r"(v) : "l"(reinterpret_cast<const float *>(base) + idx) : "memory");
  else if (IN == SLQ_IN_F16) {
    uint16_t h;
    asm volatile("ld.global.nc.b16 %0, [%1];" : "=h"(h) : "l"(reinterpret_cast<const uint16_t *>(base) + idx) : "memory");
    v = h;
  } else asm volatile("ld.global.nc.u8 %0, [%1];" : "=r"(v) : "l"(reinterpret_cast<const uint8_t *>(base) + idx) : "memory");
  return v;
}
// raw element -> the fp32 pixel value the reference's model would see (then rounded to fp16 by the caller)
template <int IN>
__device__ __forceinline__ float stem_pixel(uint32_t raw, float mean, float stdv) {
  if (IN == SLQ_IN_F32) return __uint_as_float(raw);
  if (IN == SLQ_IN_F16) return __half2float(__ushort_as_half((unsigned short)raw));
  // torchvision ToTensor: u8 -> fp32 / 255 ; Normalize: (t - mean) / std -- three separately rounded fp32 ops
  return __fdiv_rn(__fsub_rn(__fdiv_rn((float)raw, 255.0f), mean), stdv);
}

// conv rows [p0, p1) of unit u and the pooled rows [j0, j1) it owns
__device__ __forceinline__ void unit_rows(const StemArgs &a, int u, int &n, int &j0, int &j1, int &p0, int &p1) {
  n = u / a.units_per_img;
  const int q = u - n * a.units_per_img;
  j0 = q * kSfUnitRows;
  j1 = min(j0 + kSfUnitRows, a.Hp);
  p0 = max(2 * j0 - 1, 0);
  p1 = min(2 * j1, a.Hc);  // last conv row needed is 2*(j1-1)+1
}

// Chunks [J0, J1) of output column q of one conv row: every index that depends on the chunk is a
// compile-time constant after unrolling (c, r, K block, chunk-in-block), so a chunk costs 4 LDS.32 +
// 1 STS.128 + a handful of integer ops.  ring_q = ring + 2q halfs; atile_q = tile + q*128; qx = q & 7.
template <int J0, int J1>
__device__ __forceinline__ void stem_build_chunks(const __half *ring_q, uint8_t *atile_q, int qx, int p) {
#pragma unroll
  for (int j = J0; j < J1; ++j) {
    constexpr int dummy = 0;
    (void)dummy;
    const int c = j / 7, r = j % 7;
    const int slot = (2 * p + 13 + r) & (kSfRing - 1);  // (2p - 3 + r + 16) mod 16
    const uint32_t *src = reinterpret_cast<const uint32_t *>(ring_q + (slot * 3 + c) * kSfRowP);
    const uint4 v = make_uint4(src[0], src[1], src[2], src[3]);
    const int kb = j >> 3, cj = j & 7;
    *reinterpret_cast<uint4 *>(atile_q + kb * 16384 + ((cj ^ qx) << 4)) = v;
  }
}

template <int IN>
__global__ void __launch_bounds__(kSfThreads, 1) stem_fused_kernel(const StemArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + kSfBarOff;
  auto afull_bar = [&](int b) { return bar_base + 8u * b; };         // A tile built      (256 arrivals)
  auto aempty_bar = [&](int b) { return bar_base + 8u * (2 + b); };  // A tile consumed   (commit)
  auto tfull_bar = [&](int b) { return bar_base + 8u * (4 + b); };   // accumulator ready (commit)
  auto tempty_bar = [&](int b) { return bar_base + 8u * (6 + b); };  // accumulator drained (256)
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem + kSfBarOff + 64);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // ---- one-time setup -------------------------------------------------------------------------
  if (threadIdx.x == 0) {
    for (int b = 0; b < 2; ++b) {
      mbar_init(afull_bar(b), kSfBuilders);
      mbar_init(aempty_bar(b), 1);
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), kSfEpi);
    }
    fence_barrier_init();
  }
  if (warp == kSfBW + 8) tmem_alloc(tmem_slot, kSfTmemCols);
  // zero the input ring (its pad columns are never written again) and stage weights + BN constants
  for (int i = threadIdx.x; i < kSfRingBytes / 16; i += blockDim.x)
    reinterpret_cast<uint4 *>(smem + kSfRingOff)[i] = make_uint4(0, 0, 0, 0);
  for (int i = threadIdx.x; i < 64 * kSfChunks; i += blockDim.x) {
    const int oc = i / kSfChunks, j = i % kSfChunks;
    const uint4 v = __ldg(reinterpret_cast<const uint4 *>(a.wh + oc * kSfK + j * 8));
    const int kb = j >> 3, cj = j & 7;
    *reinterpret_cast<uint4 *>(smem + kSfBOff + kb * 8192 + oc * 128 + ((cj ^ (oc & 7)) << 4)) = v;
  }
  for (int i = threadIdx.x; i < 2 * 128 * 3; i += blockDim.x) {  // K-pad chunks 21..23 of both A tiles stay zero
    const int ab = i / 384, rem = i % 384, q = rem / 3, j = 21 + rem % 3;
    *reinterpret_cast<uint4 *>(smem + kSfAOff + ab * kSfABytes + (j >> 3) * 16384 + q * 128 + (((j & 7) ^ (q & 7)) << 4)) =
        make_uint4(0, 0, 0, 0);
  }
  if (threadIdx.x < 64) {  // u8 output: the re-quantisation multiply is folded into the BN constants
    const float inv = a.out_mode == SLQ_OUT_F32 ? 1.f : __fdiv_rn(1.0f, a.act_scales[a.out_id]);
    reinterpret_cast<float2 *>(smem + kSfPrmOff)[threadIdx.x] =
        make_float2(__fmul_rn(a.bn_a[threadIdx.x], inv), __fmul_rn(a.bn_b[threadIdx.x], inv));
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp < kSfBW) {
    // ================================ builders ================================================
    const int t = threadIdx.x;                       // 0..511
    const int q = t & 127, part = t >> 7;            // output column, which quarter of the 21 chunks
    const int lt = t & 255, lrow = t >> 8;           // loader role: input column, which of the two new rows
    __half *ring = reinterpret_cast<__half *>(smem + kSfRingOff);
    constexpr int kMaxPer = 3;                       // ring elements per thread per step: 3 channels of one row
    int tn = 0;
    int rc = 0;                                      // conv rows built so far (A buffer parity / phase)
    for (int u = blockIdx.x; u < a.total_units; u += gridDim.x) {
      int n, j0, j1, p0, p1;
      unit_rows(a, u, n, j0, j1, p0, p1);
      const long long xn = (long long)n * 3 * a.H * a.W;  // element index of image n
      // rows [lo, hi) of the image (may be outside: zeros) -> ring, through registers
      auto load_rows = [&](int lo, int hi, uint32_t (&v)[kMaxPer], bool first) {
        const int per_row = 3 * a.W;
        const int total = (hi - lo) * per_row;
        if (first) {  // unit start: 7 rows at once, written straight away
          for (int e = t; e < total; e += kSfBuilders) {
            const int ri = e / per_row, rem = e - ri * per_row;
            const int c = rem / a.W, w = rem - c * a.W;
            const int h = lo + ri;
            const float f = (h >= 0 && h < a.H)
                                ? stem_pixel<IN>(ldg_pinned<IN>(a.x, xn + ((long long)c * a.H + h) * a.W + w), a.nmean[c], a.nstd[c])
                                : 0.f;
            ring[(((h + 16) & (kSfRing - 1)) * 3 + c) * kSfRowP + w + 3] = __float2half_rn(f);
          }
          return;
        }
        // steady state: thread = (one of the two new rows, one column), three channels: no divisions
        const int h = lo + lrow;
        const bool ok = lt < a.W && lrow < hi - lo && h >= 0 && h < a.H;
        const long long src = xn + (long long)h * a.W + lt;
#pragma unroll
        for (int c = 0; c < 3; ++c) v[c] = ok ? ldg_pinned<IN>(a.x, src + (long long)c * a.H * a.W) : 0u;
      };
      auto store_rows = [&](int lo, int hi, const uint32_t (&v)[kMaxPer]) {
        const int h = lo + lrow;
        const bool inside = h >= 0 && h < a.H;  // rows outside the image are the conv's zero padding
        if (lt < a.W && lrow < hi - lo) {
          __half *dst = ring + ((h + 16) & (kSfRing - 1)) * 3 * kSfRowP + lt + 3;
#pragma unroll
          for (int c = 0; c < 3; ++c)
            dst[c * kSfRowP] = __float2half_rn(inside ? stem_pixel<IN>(v[c], a.nmean[c], a.nstd[c]) : 0.f);
        }
      };
      uint32_t nxt[kMaxPer];
      named_bar_sync(1, kSfBuilders);  // nobody still builds from the previous unit's rows
      load_rows(2 * p0 - 3, 2 * p0 + 4, nxt, true);
      named_bar_sync(1, kSfBuilders);
      for (int p = p0; p < p1; ++p, ++rc) {
        const int ab = rc & 1;
        if (t == 0) stem_trace(a, 0, tn, 0, rc);
        if (p + 1 < p1 && !(SF_DBG(a) & 16)) load_rows(2 * p + 4, 2 * p + 6, nxt, false);  // in flight during the build
        mbar_wait(aempty_bar(ab), (uint32_t)(((rc >> 1) & 1) ^ 1));
        if (t == 0) stem_trace(a, 0, tn, 1, rc);
        uint8_t *atile = smem + kSfAOff + ab * kSfABytes;
        if (!(SF_DBG(a) & 1)) {
          if (part == 0) stem_build_chunks<0, 6>(ring + 2 * q, atile + q * 128, q & 7, p);
          else if (part == 1) stem_build_chunks<6, 11>(ring + 2 * q, atile + q * 128, q & 7, p);
          else if (part == 2) stem_build_chunks<11, 16>(ring + 2 * q, atile + q * 128, q & 7, p);
          else stem_build_chunks<16, 21>(ring + 2 * q, atile + q * 128, q & 7, p);
        }
        if (t == 0) stem_trace(a, 0, tn, 2, rc);
        if (!(SF_DBG(a) & 8)) fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core (async proxy)
        mbar_arrive(afull_bar(ab));
        if (t == 0) stem_trace(a, 0, tn, 3, rc);
        if (p + 1 < p1) {
          if (!(SF_DBG(a) & 16)) store_rows(2 * p + 4, 2 * p + 6, nxt);
          named_bar_sync(1, kSfBuilders);  // the next row's inputs are complete
        }
        if (t == 0) stem_trace(a, 0, tn, 8, rc);
      }
    }
  } else if (warp >= kSfBW + 8) {
    // ================================ MMA issuers (convergent warps, elected lane) =============
    const int my_par = warp - (kSfBW + 8);  // this warp issues the rows with rc % 2 == my_par
    int tn = 0;
    const uint32_t idesc = (1u << 4) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);  // f16 x f16 -> f32
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    int rc = 0;
    for (int u = blockIdx.x; u < a.total_units; u += gridDim.x) {
      int n, j0, j1, p0, p1;
      unit_rows(a, u, n, j0, j1, p0, p1);
      for (int p = p0; p < p1; ++p, ++rc) {
        const int ab = rc & 1;
        if (ab != my_par) continue;
        const uint32_t ph = (uint32_t)((rc >> 1) & 1);
        mbar_wait(tempty_bar(ab), ph ^ 1);
        mbar_wait(afull_bar(ab), ph);
        tc_fence_after();
        if (lane == 0) stem_trace(a, 16 + my_par, tn, 4, rc);
        const uint32_t tmem_d = tmem_u + ab * 64;
        const uint64_t da = make_smem_desc<128>(smem_base + kSfAOff + ab * kSfABytes);
        const uint64_t db = make_smem_desc<128>(smem_base + kSfBOff);
        if (elect_one()) {
#pragma unroll
          for (int kb = 0; kb < 3; ++kb)
#pragma unroll
            for (int k = 0; k < 4; ++k)  // UMMA_K = 16 halfs = 32 bytes
              umma_f16(tmem_d, da + (uint64_t)(kb * (16384 >> 4) + 2 * k), db + (uint64_t)(kb * (8192 >> 4) + 2 * k),
                       idesc, (kb | k) != 0);
          umma_commit(aempty_bar(ab));
          umma_commit(tfull_bar(ab));
        }
        __syncwarp();
        if (lane == 0) stem_trace(a, 16 + my_par, tn, 9, rc);
      }
    }
  } else {
    // ================================ epilogue + pooling (warps 8-15) ==========================
    const int et = threadIdx.x - kSfBuilders;        // 0..255
    const int wq = warp & 3, half = (warp - kSfBW) >> 2; // TMEM lane quarter, channel half
    const int q = wq * 32 + lane;
    const float2 *prm = reinterpret_cast<const float2 *>(smem + kSfPrmOff);
    uint8_t *cring = smem + kSfConvOff;
    const bool f32_out = a.out_mode == SLQ_OUT_F32;
    int tn = 0;
    int rc = 0;
    for (int u = blockIdx.x; u < a.total_units; u += gridDim.x) {
      int n, j0, j1, p0, p1;
      unit_rows(a, u, n, j0, j1, p0, p1);
      for (int p = p0; p < p1; ++p, ++rc) {
        const int ab = rc & 1;
        mbar_wait(tfull_bar(ab), (uint32_t)((rc >> 1) & 1));
        tc_fence_after();
        if (et == 0) stem_trace(a, 18, tn, 5, rc);
        uint32_t acc[32];
        tmem_ld32(tmem_base + ((uint32_t)(wq * 32) << 16) + ab * 64 + half * 32, acc);
        tmem_ld_wait();
        tc_fence_before();
        mbar_arrive(tempty_bar(ab));  // accumulator is in registers: the next row may start
        if (SF_DBG(a) & 4) continue;
        float y[32];
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          const float2 p2 = prm[half * 32 + j];
          y[j] = __fmaf_rn(__uint_as_float(acc[j]), p2.x, p2.y);  // u8: in units of the output scale
        }
        if (f32_out) {
          if (q < a.Wc) {
            float4 *o = reinterpret_cast<float4 *>(reinterpret_cast<float *>(a.out) +
                                                   (((long long)n * a.Hc + p) * a.Wc + q) * 64 + half * 32);
#pragma unroll
            for (int j = 0; j < 8; ++j)
              o[j] = make_float4(fmaxf(y[4 * j], 0.f), fmaxf(y[4 * j + 1], 0.f), fmaxf(y[4 * j + 2], 0.f),
                                 fmaxf(y[4 * j + 3], 0.f));
          }
          continue;
        }
        uint32_t pk[8];
#pragma unroll
        for (int j = 0; j < 8; ++j)  // saturation at 0 is the ReLU
          pk[j] = epi_pack4<false>(y[4 * j], y[4 * j + 1], y[4 * j + 2], y[4 * j + 3]);
        uint4 *dst = reinterpret_cast<uint4 *>(cring + (p & (kSfConvRing - 1)) * kSfConvRowBytes + q * 64 + half * 32);
        dst[0] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
        dst[1] = make_uint4(pk[4], pk[5], pk[6], pk[7]);
        if (et == 0) stem_trace(a, 18, tn, 10, rc);
        named_bar_sync(2, kSfEpi);  // conv row p is complete in the ring
        if (et == 0) stem_trace(a, 18, tn, 11, rc);
        // pooled row j = max over conv rows 2j-1..2j+1: complete after an odd row or the last row
        if (!((p & 1) || p == a.Hc - 1) || (SF_DBG(a) & 2)) continue;
        const int j = p >> 1;
        if (j < j0) continue;  // the seam row only feeds this unit's first pooled row
        // one thread per (pooled column, 16 channels): 9 clamped 16-byte loads (a duplicated row or
        // column does not change a max), byte-wise max, one 16-byte coalesced store
        const int r0 = max(2 * j - 1, 0), r1 = 2 * j, r2 = min(2 * j + 1, a.Hc - 1);
        const uint8_t *row0 = cring + (r0 & (kSfConvRing - 1)) * kSfConvRowBytes;
        const uint8_t *row1 = cring + (r1 & (kSfConvRing - 1)) * kSfConvRowBytes;
        const uint8_t *row2 = cring + (r2 & (kSfConvRing - 1)) * kSfConvRowBytes;
        uint4 *orow = reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(a.out) +
                                                (((long long)n * a.Hp + j) * a.Wp) * 64);
        uint32_t *rsrow = a.out_rowsum ? a.out_rowsum + ((long long)n * a.Hp + j) * a.Wp : nullptr;
        for (int base = et & ~31; base < a.Wp * 4; base += kSfEpi) {  // whole warps walk the loop (shuffles below)
          const int idx = base + lane;
          const bool live = idx < a.Wp * 4;
          const int i = idx >> 2, g = (idx & 3) * 16;
          uint4 m = make_uint4(0, 0, 0, 0);
          if (live) {
            const int c0 = max(2 * i - 1, 0) * 64 + g, c1 = 2 * i * 64 + g, c2 = min(2 * i + 1, a.Wc - 1) * 64 + g;
            m = *reinterpret_cast<const uint4 *>(row0 + c0);
            auto mx = [&](const uint8_t *ptr) {
              const uint4 v = *reinterpret_cast<const uint4 *>(ptr);
              m.x = __vmaxu4(m.x, v.x); m.y = __vmaxu4(m.y, v.y); m.z = __vmaxu4(m.z, v.z); m.w = __vmaxu4(m.w, v.w);
            };
            mx(row0 + c1); mx(row0 + c2);
            mx(row1 + c0); mx(row1 + c1); mx(row1 + c2);
            mx(row2 + c0); mx(row2 + c1); mx(row2 + c2);
            orow[idx] = m;
          }
          // channel sum of the pooled pixel: 16 channels per thread, four neighbouring lanes per pixel
          uint32_t ps = __dp4a(m.x, 0x01010101u, __dp4a(m.y, 0x01010101u, __dp4a(m.z, 0x01010101u, __dp4a(m.w, 0x01010101u, 0u))));
          ps += __shfl_xor_sync(0xffffffffu, ps, 1);
          ps += __shfl_xor_sync(0xffffffffu, ps, 2);
          if (live && rsrow && (idx & 3) == 0) rsrow[i] = ps;
        }
        if (et == 0) stem_trace(a, 18, tn, 6, rc);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kSfBW + 8) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kSfTmemCols);
  }
}

// ================================================================================================
// Stem v2: A operand in TENSOR MEMORY (tcgen05.mma TS form)
// ================================================================================================
// The 7x7 stride-2 conv as an implicit GEMM whose K dimension is cut into "pair slabs": slab (c, t) is the
// [128 output columns q] x [16 halfs] matrix  { x[c][2t][2q-3 .. 2q+4], x[c][2t+1][2q-3 .. 2q+4] }
// (input-row pair t of channel c).  Conv row p needs the four pairs t = p-2 .. p+1: pair i = t - p + 2
// multiplies the filter rows r = 2i-1 (first row of the pair; r = -1 -> zero weights) and r = 2i, i.e. a
// FIXED 64 x 16 weight slice per (c, i).  Going from conv row p to p+1 therefore adds ONE new pair (3
// slabs) and retires one -- round 1 rebuilt all 21 (c, r) chunks of every conv row in shared memory
// (2688 16-byte chunks per row through LDS.32 / STS.128; the stem was bound by exactly that).
//   producer (warp 0)    TMA bulk copies of the raw input rows of pair t into an 8-deep staging ring
//   builders (8 warps)   staging -> fp16 rows (each element converted once) -> the thread that owns output
//                        column q writes its 16-byte window of each of the six rows straight into the
//                        slab's TMEM columns (tcgen05.st): the A operand never exists in shared memory
//   MMA (4 warps)        conv row rc -> warp rc & 3, accumulator rc & 3: 12 tcgen05.mma.kind::f16
//                        (A from TMEM, 64 x 16 weight slices resident in shared memory, M128 N64 K16)
//   epilogue (8 warps)   tcgen05.ld -> folded BN + ReLU -> u8 -> 4-row ring -> 3x3/s2 max-pool -> store
// TMEM: columns [0, 256) four accumulators; [256, 448) eight pair slots x 3 channels x 8 columns.

constexpr int kTsSlots = 8;                       // staged input-row pairs == TMEM pair slots
constexpr int kTsRowP = 264;                      // halfs per converted row: column cc = w + 3, w in [-3, 2*127+4]
constexpr int kTsMaxRowBytes = 1024;              // W <= 256 fp32 elements
constexpr int kTsStageBytes = 6 * kTsMaxRowBytes; // one pair: 3 channels x 2 rows, raw
constexpr int kTsStageOff = 0;
constexpr int kTsRowBufOff = kTsStageOff + kTsSlots * kTsStageBytes;
constexpr int kTsRowBufBytes = 4 * 6 * kTsRowP * 2;   // fp16 rows of one pair: two buffers per builder group
constexpr int kTsBOff = ((kTsRowBufOff + kTsRowBufBytes + 1023) / 1024) * 1024;
constexpr int kTsConvOff = kTsBOff + kSfBBytes;
constexpr int kTsPrmOff = kTsConvOff + kSfConvRing * kSfConvRowBytes;
constexpr int kTsBarOff = kTsPrmOff + 64 * 8;
constexpr int kTsSmemBytes = 1024 + kTsBarOff + 512;
constexpr int kTsBuildW = 8, kTsMmaW = 2, kTsEpiW = 16, kTsPoolW = 4;
constexpr int kTsWarps = 1 + kTsBuildW + kTsMmaW + kTsEpiW + kTsPoolW;  // producer + builders + MMA + epilogue + pool = 31
constexpr int kTsThreads = kTsWarps * 32;
constexpr int kTsGroupW = kTsBuildW / 2, kTsGroup = kTsGroupW * 32, kTsEpi = kTsEpiW * 32;  // two builder groups of 4 warps
constexpr int kTsAccCols = 64, kTsSlabBase = 256, kTsSlotCols = 24;
constexpr int kTsTmemCols = 512;
static_assert(kTsSmemBytes <= 232448, "stem v2 exceeds 227 KB of shared memory");

// w fp32 [64, 3, 7, 7] -> wh fp16 [64, 192]: wh[oc][c*64 + ch*8 + s] = w[oc][c][ch-1][s]  (ch = 2i + j is
// the row of pair i: filter row r = ch - 1; ch = 0 and s = 7 are zero)
__global__ void stem_weights_ts_kernel(const float *__restrict__ w, float *__restrict__ wh) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 64 * kSfK) return;
  const int k = idx % kSfK, oc = idx / kSfK;
  const int c = k >> 6, ch = (k >> 3) & 7, s = k & 7;
  float v = 0.f;
  if (ch >= 1 && s < 7) v = w[((oc * 3 + c) * 7 + (ch - 1)) * 7 + s];
  wh[idx] = v;
}

template <int IN>
__global__ void __launch_bounds__(kTsThreads, 1) stem_ts_kernel(const __grid_constant__ CUtensorMap tmX, const StemArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + kTsBarOff;
  auto sfull_bar = [&](int s) { return bar_base + 8u * s; };          // raw rows of a pair landed (TMA tx)
  auto sempty_bar = [&](int s) { return bar_base + 8u * (8 + s); };   // builders have converted them (8 warps)
  auto pfull_bar = [&](int s) { return bar_base + 8u * (16 + s); };   // pair slabs written to TMEM (8 warps)
  auto pfree_bar = [&](int s) { return bar_base + 8u * (24 + s); };   // the 4 conv rows using the pair are done (4 commits)
  auto tfull_bar = [&](int b) { return bar_base + 8u * (32 + b); };   // accumulator ready (commit)
  auto tempty_bar = [&](int b) { return bar_base + 8u * (36 + b); };  // accumulator drained (8 epilogue warps)
  auto vfull_bar = [&](int b) { return bar_base + 8u * (40 + b); };   // vertically pooled row written (8 epilogue warps)
  auto vfree_bar = [&](int b) { return bar_base + 8u * (44 + b); };   // ... and consumed by the pool warps (4 warps)
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem + kTsBarOff + 8 * 48);
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  constexpr int ESZ = IN == SLQ_IN_F32 ? 4 : (IN == SLQ_IN_F16 ? 2 : 1);
  const int row_bytes = a.W * ESZ;

  // ---- one-time setup -------------------------------------------------------------------------
  if (threadIdx.x == 0) {
    for (int s = 0; s < kTsSlots; ++s) {
      mbar_init(sfull_bar(s), 1);
      mbar_init(sempty_bar(s), kTsGroupW);
      mbar_init(pfull_bar(s), kTsGroupW);
      mbar_init(pfree_bar(s), 4);
    }
    for (int b = 0; b < 4; ++b) {
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), kTsEpiW);
      mbar_init(vfull_bar(b), kTsEpiW);
      mbar_init(vfree_bar(b), kTsPoolW);
    }
    fence_barrier_init();
  }
  if (warp == 0) {
    if (lane == 0) prefetch_tmap(&tmX);
    tmem_alloc(tmem_slot, kTsTmemCols);
  }
  // converted-row buffers: the pad columns are never written again; weights + BN constants
  for (int i = threadIdx.x; i < kTsRowBufBytes / 16; i += blockDim.x)
    reinterpret_cast<uint4 *>(smem + kTsRowBufOff)[i] = make_uint4(0, 0, 0, 0);
  for (int i = threadIdx.x; i < 64 * kSfChunks; i += blockDim.x) {
    const int oc = i / kSfChunks, j = i % kSfChunks;
    // the BN scale of the output channel goes into the weights BEFORE they are rounded to fp16 (one rounding, like
    // the plain fp16 weights had): the epilogue is then y = acc * inv + b' with a scalar inv and 16 per-channel b'
    // that stay in registers -- no constant loads in its loop
    const float4 w0 = __ldg(reinterpret_cast<const float4 *>(a.wf + oc * kSfK + j * 8));
    const float4 w1 = __ldg(reinterpret_cast<const float4 *>(a.wf + oc * kSfK + j * 8 + 4));
    const float sa = a.bn_a[oc];
    const __half2 h0 = __floats2half2_rn(__fmul_rn(w0.x, sa), __fmul_rn(w0.y, sa)), h1 = __floats2half2_rn(__fmul_rn(w0.z, sa), __fmul_rn(w0.w, sa));
    const __half2 h2 = __floats2half2_rn(__fmul_rn(w1.x, sa), __fmul_rn(w1.y, sa)), h3 = __floats2half2_rn(__fmul_rn(w1.z, sa), __fmul_rn(w1.w, sa));
    const uint4 v = make_uint4(*reinterpret_cast<const uint32_t *>(&h0), *reinterpret_cast<const uint32_t *>(&h1),
                               *reinterpret_cast<const uint32_t *>(&h2), *reinterpret_cast<const uint32_t *>(&h3));
    const int kb = j >> 3, cj = j & 7;  // kb = channel c, cj = 2i + j: 32 bytes per pair i inside the 128-byte row
    *reinterpret_cast<uint4 *>(smem + kTsBOff + kb * 8192 + oc * 128 + ((cj ^ (oc & 7)) << 4)) = v;
  }
  const float inv_out = a.out_mode == SLQ_OUT_F32 ? 1.f : __fdiv_rn(1.0f, a.act_scales[a.out_id]);
  if (threadIdx.x < 64)  // u8 output: in units of the output scale
    reinterpret_cast<float *>(smem + kTsPrmOff)[threadIdx.x] = __fmul_rn(a.bn_b[threadIdx.x], inv_out);
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // Every role walks the same units; running counters: rc = conv rows so far, g = pairs so far.  A unit
  // of R conv rows consumes R + 3 pairs (the first row needs four), so row rc of the u-th unit uses the
  // pairs g_lo .. g_lo + 3 with g_lo = rc + 3 u.
  if (warp == 0) {
    // ================================ producer: raw rows -> staging ring ======================
    // ONE tensor load per pair: box {W, 2 rows, 3 channels} of the image viewed as [3N planes][H][W]; rows
    // above / below the image are zero-filled by the TMA unit (the conv's padding).  (Six 1-D bulk copies
    // per pair cost the issuing thread ~1800 cycles -- more than everything else in the kernel.)
    int g = 0, tn = 0;
    const uint32_t pair_bytes = (uint32_t)(6 * row_bytes);
    for (int u = blockIdx.x; u < a.total_units; u += gridDim.x) {
      int n, j0, j1, p0, p1;
      unit_rows(a, u, n, j0, j1, p0, p1);
      for (int t = p0 - 2; t <= p1; ++t, ++g) {
        const int s = g & (kTsSlots - 1);
        if (lane == 0) stem_trace(a, 0, tn, 0, g);
        mbar_wait(sempty_bar(s), (uint32_t)(((g >> 3) & 1) ^ 1));
        if (lane == 0) stem_trace(a, 0, tn, 1, g);
        if (elect_one()) {
          mbar_expect_tx(sfull_bar(s), pair_bytes);
          tma_load_3d(smem_base + kTsStageOff + s * kTsStageBytes, &tmX, sfull_bar(s), 0, 2 * t, 3 * n);
        }
        __syncwarp();
      }
    }
  } else if (warp <= kTsBuildW) {
    // ================================ builders ================================================
    // Two groups of four warps (one warp per TMEM lane quarter), pair g -> group g & 1: while one group writes its
    // pair's slabs to tensor memory the other converts the next pair -- a pair's chain (wait, convert, barrier,
    // wait for the slot, six tcgen05.st, wait::st, arrive) is ~1500 cycles of mostly latency, and with all eight
    // warps walking it together it was the pace of the whole kernel.
    const int group = (warp - 1) >> 2;
    const int bt = threadIdx.x - 32 - group * kTsGroup;  // 0..127 inside the group
    const int quarter = warp & 3;                    // the TMEM lanes this warp may touch
    const int q = quarter * 32 + lane;               // output column == TMEM lane
    __half *rowbuf = reinterpret_cast<__half *>(smem + kTsRowBufOff);
    const int w4 = a.W >> 2;                         // 4-element groups per row (<= 64)
    int g = 0, tn = 0;
    for (int u = blockIdx.x; u < a.total_units; u += gridDim.x) {
      int n, j0, j1, p0, p1;
      unit_rows(a, u, n, j0, j1, p0, p1);
      for (int t = p0 - 2; t <= p1; ++t, ++g) {
        if ((g & 1) != group) continue;
        const int s = g & (kTsSlots - 1);
        const uint32_t ph = (uint32_t)((g >> 3) & 1);
        __half *rb = rowbuf + (group * 2 + ((g >> 1) & 1)) * 6 * kTsRowP;
        const int tr = group ? 8 : 1;  // trace issuer
        if (bt == 0) stem_trace(a, tr, tn, 2, g);
        mbar_wait(sfull_bar(s), ph);
        if (bt == 0) stem_trace(a, tr, tn, 3, g);
        // 1. raw -> fp16, every element once: thread = (row r6 of the six, 4-element group c4); three passes
        const uint8_t *stg = smem + kTsStageOff + s * kTsStageBytes;
#pragma unroll
        for (int pass = 0; pass < 3; ++pass) {
          const int r6 = pass * 2 + (bt >> 6), c4 = bt & 63;
          if (c4 >= w4 || (SF_DBG(a) & 1)) continue;
          const int c = r6 >> 1;
          float f[4];
          const uint8_t *src = stg + r6 * row_bytes + c4 * 4 * ESZ;  // rows outside the image arrive as zeros
          if (IN == SLQ_IN_F32) {
            const float4 v = *reinterpret_cast<const float4 *>(src);
            f[0] = v.x; f[1] = v.y; f[2] = v.z; f[3] = v.w;
          } else if (IN == SLQ_IN_F16) {
            const uint2 v = *reinterpret_cast<const uint2 *>(src);
            f[0] = stem_pixel<IN>(v.x & 0xffffu, 0.f, 1.f); f[1] = stem_pixel<IN>(v.x >> 16, 0.f, 1.f);
            f[2] = stem_pixel<IN>(v.y & 0xffffu, 0.f, 1.f); f[3] = stem_pixel<IN>(v.y >> 16, 0.f, 1.f);
          } else {
            const uint32_t v = *reinterpret_cast<const uint32_t *>(src);
            const int h = 2 * t + (r6 & 1);
            const bool inside = h >= 0 && h < a.H;  // a zero BYTE is a pixel value: padding rows must become 0.0
#pragma unroll
            for (int e = 0; e < 4; ++e) f[e] = inside ? stem_pixel<IN>((v >> (8 * e)) & 255u, a.nmean[c], a.nstd[c]) : 0.f;
          }
          __half *dst = rb + r6 * kTsRowP + 3 + 4 * c4;  // 2-byte aligned (cc = w + 3)
          dst[0] = __float2half_rn(f[0]);
          *reinterpret_cast<__half2 *>(dst + 1) = __floats2half2_rn(f[1], f[2]);
          dst[3] = __float2half_rn(f[3]);
        }
        named_bar_sync(1 + group, kTsGroup);  // rows complete; also: nobody in the group still reads the buffer of pair g - 4
        if (lane == 0) mbar_arrive(sempty_bar(s));  // the staging slot may be refilled
        // 2. the pair's TMEM slot must be free: the four conv rows that used pair g - 8 have completed
        if (bt == 0) stem_trace(a, tr, tn, 4, g);
        if (g >= kTsSlots) mbar_wait(pfree_bar(s), ph ^ 1);
        if (bt == 0) stem_trace(a, tr, tn, 5, g);
        tc_fence_after();
        // 3. this thread's 16-byte windows x[c][h][2q-3 .. 2q+4] -> the slab's TMEM columns
        const uint32_t tslab = tmem_base + ((uint32_t)(quarter * 32) << 16) + kTsSlabBase + s * kTsSlotCols;
#pragma unroll
        for (int k = 0; k < 6 && !(SF_DBG(a) & 2); ++k) {
          const int r6 = k;  // = c * 2 + j
          const uint32_t *src = reinterpret_cast<const uint32_t *>(rb + r6 * kTsRowP + 2 * q);
          tmem_st4(tslab + (r6 >> 1) * 8 + (r6 & 1) * 4, src[0], src[1], src[2], src[3]);
        }
        tmem_st_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(pfull_bar(s));
        if (bt == 0) stem_trace(a, tr, tn, 6, g);
      }
    }
  } else if (warp <= kTsBuildW + kTsMmaW) {
    // ================================ MMA issuers (convergent warps, elected lane) =============
    const int mw = warp - (kTsBuildW + 1);  // conv rows with rc % kTsMmaW == mw
    const uint32_t idesc = (1u << 4) | ((uint32_t)(64 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);  // f16 x f16 -> f32
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint64_t db0 = make_smem_desc<128>(smem_base + kTsBOff);
    int rc = 0, u_ord = 0, tn = 0;
    for (int u = blockIdx.x; u < a.total_units; u += gridDim.x, ++u_ord) {
      int n, j0, j1, p0, p1;
      unit_rows(a, u, n, j0, j1, p0, p1);
      for (int p = p0; p < p1; ++p, ++rc) {
        if ((rc & (kTsMmaW - 1)) != mw) continue;
        const int acc = rc & 3;
        const int g_lo = rc + 3 * u_ord;
        if (lane == 0) stem_trace(a, 2 + mw, tn, 7, rc);
        if (rc >= 4) mbar_wait(tempty_bar(acc), (uint32_t)(((rc >> 2) & 1) ^ 1));
        if (lane == 0) stem_trace(a, 2 + mw, tn, 8, rc);
        // each builder group completes its pairs in order: the newest pair of either group implies the older ones
        mbar_wait(pfull_bar((g_lo + 2) & (kTsSlots - 1)), (uint32_t)(((g_lo + 2) >> 3) & 1));
        mbar_wait(pfull_bar((g_lo + 3) & (kTsSlots - 1)), (uint32_t)(((g_lo + 3) >> 3) & 1));
        tc_fence_after();
        if (lane == 0) stem_trace(a, 2 + mw, tn, 9, rc);
        if (elect_one()) {
#pragma unroll
          for (int i = 0; i < 4 && !(SF_DBG(a) & 8); ++i) {
            const uint32_t ta = tmem_u + kTsSlabBase + ((g_lo + i) & (kTsSlots - 1)) * kTsSlotCols;
#pragma unroll
            for (int c = 0; c < 3; ++c)
              umma_f16_ts(tmem_u + acc * kTsAccCols, ta + c * 8, db0 + (uint64_t)(c * (8192 >> 4) + 2 * i), idesc,
                          (uint32_t)((i | c) != 0));
          }
          // a pair slab is read by the MMAs of FOUR conv rows, issued by four different threads, and a commit
          // only tracks its own thread's MMAs: every row arrives once on each of its four pairs ...
#pragma unroll
          for (int i = 0; i < 4; ++i) umma_commit(pfree_bar((g_lo + i) & (kTsSlots - 1)));
          // ... and the rows at the ends of a unit stand in for the users their pairs do not have
          // (the first pair of a unit is used by 1 row, the second by 2, the third by 3; same at the end)
          // pair k of a unit has min(k, 3) + 1 users at its start and as few at its end: the first row adds the
          // 3 - i arrivals its pair i lacks, the last row the i arrivals its pair i lacks
          for (int i = 0; i < 4; ++i) {
            const int extra = (p == p0 ? 3 - i : 0) + (p == p1 - 1 ? i : 0);
            for (int k = 0; k < extra; ++k) umma_commit(pfree_bar((g_lo + i) & (kTsSlots - 1)));
          }
          umma_commit(tfull_bar(acc));
        }
        __syncwarp();
        if (lane == 0) stem_trace(a, 2 + mw, tn, 10, rc);
      }
    }
  } else if (warp <= kTsBuildW + kTsMmaW + kTsEpiW) {
    // ================================ epilogue: accumulator -> u8, vertical half of the pooling ====
    const int et = threadIdx.x - (1 + kTsBuildW + kTsMmaW) * 32;  // 0..511
    // TMEM lane quarter, and which 16 of the 64 channels: sixteen warps drain a conv row together, so the row's
    // accumulator is free again (and the row is pooled) in half the time eight warps with 32 channels each needed --
    // the per-row chain wait -> tcgen05.ld -> convert -> pack of these warps is what paced the whole kernel
    const int wq = warp & 3, sl = (warp - (1 + kTsBuildW + kTsMmaW)) >> 2;
    const int q = wq * 32 + lane;
    float2 kb2[8];  // b' of this thread's 16 channels, for the CTA's whole life
#pragma unroll
    for (int j = 0; j < 8; ++j) kb2[j] = reinterpret_cast<const float2 *>(smem + kTsPrmOff)[sl * 8 + j];
    const float2 inv2 = make_float2(inv_out, inv_out);
    uint8_t *cring = smem + kTsConvOff;
    const bool f32_out = a.out_mode == SLQ_OUT_F32;
    uint32_t vm[4] = {0, 0, 0, 0};  // running vertical maximum of the pooling window (packed u8)
    int rc = 0, ve = 0, tn = 0;                  // conv rows / pooled rows handled so far by this CTA
    for (int u = blockIdx.x; u < a.total_units; u += gridDim.x) {
      int n, j0, j1, p0, p1;
      unit_rows(a, u, n, j0, j1, p0, p1);
      for (int p = p0; p < p1; ++p, ++rc) {
        const int acc = rc & 3;
        if (et == 0) stem_trace(a, 6, tn, 11, rc);
        mbar_wait(tfull_bar(acc), (uint32_t)((rc >> 2) & 1));
        if (et == 0) stem_trace(a, 6, tn, 12, rc);
        tc_fence_after();
        uint32_t av[16];
        tmem_ld16(tmem_base + ((uint32_t)(wq * 32) << 16) + acc * kTsAccCols + sl * 16, av);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(tempty_bar(acc));  // accumulator is in registers: row rc + 4 may start
        if (et == 0) stem_trace(a, 6, tn, 13, rc);
        if (SF_DBG(a) & 4) continue;
        float y[16];
#pragma unroll
        for (int j = 0; j < 16; j += 2) {
          const float2 r = ffma2(make_float2(__uint_as_float(av[j]), __uint_as_float(av[j + 1])), inv2, kb2[j >> 1]);
          y[j] = r.x; y[j + 1] = r.y;
        }
        if (f32_out) {
          if (q < a.Wc) {
            float4 *o = reinterpret_cast<float4 *>(reinterpret_cast<float *>(a.out) +
                                                   (((long long)n * a.Hc + p) * a.Wc + q) * 64 + sl * 16);
#pragma unroll
            for (int j = 0; j < 4; ++j)
              o[j] = make_float4(fmaxf(y[4 * j], 0.f), fmaxf(y[4 * j + 1], 0.f), fmaxf(y[4 * j + 2], 0.f),
                                 fmaxf(y[4 * j + 3], 0.f));
          }
          continue;
        }
        uint32_t pk[4];
#pragma unroll
        for (int j = 0; j < 4; ++j)  // saturation at 0 is the ReLU
          pk[j] = epi_pack4<false>(y[4 * j], y[4 * j + 1], y[4 * j + 2], y[4 * j + 3]);
        // 3x3 / stride-2 max-pool, separable: the VERTICAL maximum over conv rows 2j-1, 2j, 2j+1 is kept in
        // registers (this thread always owns the same column and channels), so only every second row goes to
        // shared memory and costs a barrier; the horizontal maximum then reads 3 pixels instead of 9
        if (p == p0) {  // the first conv row of a unit opens a window (and closes none)
#pragma unroll
          for (int j = 0; j < 4; ++j) vm[j] = pk[j];
        } else {        // rows 2j and 2j+1 extend the window that row 2j-1 opened
#pragma unroll
          for (int j = 0; j < 4; ++j) vm[j] = __vmaxu4(vm[j], pk[j]);
        }
        const int jrow = p >> 1;
        // pooled row jrow is complete with an odd conv row (or the last one); the seam row 2 j0 - 1 at the start
        // of a unit belongs to the previous unit's pooled row and only opens this unit's first window
        const bool emit = ((p & 1) || p == a.Hc - 1) && jrow >= j0 && p != p0;
        if (emit) {
          // hand the vertically pooled row to the pool warps through a 4-slot ring
          const int vs = ve & 3;
          if (et == 0) stem_trace(a, 6, tn, 14, rc);
          if (ve >= 4) mbar_wait(vfree_bar(vs), (uint32_t)(((ve >> 2) & 1) ^ 1));
          if (et == 0) stem_trace(a, 6, tn, 15, rc);
          *reinterpret_cast<uint4 *>(cring + vs * kSfConvRowBytes + q * 64 + sl * 16) = make_uint4(vm[0], vm[1], vm[2], vm[3]);
          __syncwarp();
          if (lane == 0) mbar_arrive(vfull_bar(vs));
          ++ve;
        }
        if (p & 1) {  // an odd row also opens the next window
#pragma unroll
          for (int j = 0; j < 4; ++j) vm[j] = pk[j];
        }
      }
    }
  } else {
    // ================================ pool warps: horizontal half of the pooling, stores ============
    // (their own role, so that the epilogue warps' chain per conv row -- wait, tcgen05.ld, convert -- never waits
    // for a pooled row to be written out)
    const int pt = threadIdx.x - (1 + kTsBuildW + kTsMmaW + kTsEpiW) * 32;  // 0..127
    const uint8_t *cring = smem + kTsConvOff;
    int ve = 0, tn = 0;
    if (a.out_mode != SLQ_OUT_F32 && !(SF_DBG(a) & 4)) {  // (debug bit 4: the epilogue emits nothing)
      for (int u = blockIdx.x; u < a.total_units; u += gridDim.x) {
        int n, j0, j1, p0, p1;
        unit_rows(a, u, n, j0, j1, p0, p1);
        for (int jrow = j0; jrow < j1; ++jrow, ++ve) {
          const int vs = ve & 3;
          if (pt == 0) stem_trace(a, 7, tn, 16, ve);
          mbar_wait(vfull_bar(vs), (uint32_t)((ve >> 2) & 1));
          if (pt == 0) stem_trace(a, 7, tn, 17, ve);
          const uint8_t *vrow = cring + vs * kSfConvRowBytes;
          uint4 *orow = reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(a.out) +
                                                  (((long long)n * a.Hp + jrow) * a.Wp) * 64);
          uint32_t *rsrow = a.out_rowsum ? a.out_rowsum + ((long long)n * a.Hp + jrow) * a.Wp : nullptr;
          for (int base = pt & ~31; base < a.Wp * 4 && !(SF_DBG(a) & 16); base += kTsPoolW * 32) {  // whole warps (shuffles below)
            const int idx = base + lane;
            const bool live = idx < a.Wp * 4;
            const int i = idx >> 2, gch = (idx & 3) * 16;
            uint4 m = make_uint4(0, 0, 0, 0);
            if (live) {
              // clamped columns: a duplicated column does not change a maximum
              const int c0 = max(2 * i - 1, 0) * 64 + gch, c1 = 2 * i * 64 + gch, c2 = min(2 * i + 1, a.Wc - 1) * 64 + gch;
              m = *reinterpret_cast<const uint4 *>(vrow + c0);
              const uint4 v1 = *reinterpret_cast<const uint4 *>(vrow + c1), v2 = *reinterpret_cast<const uint4 *>(vrow + c2);
              m.x = __vmaxu4(__vmaxu4(m.x, v1.x), v2.x); m.y = __vmaxu4(__vmaxu4(m.y, v1.y), v2.y);
              m.z = __vmaxu4(__vmaxu4(m.z, v1.z), v2.z); m.w = __vmaxu4(__vmaxu4(m.w, v1.w), v2.w);
              orow[idx] = m;
            }
            uint32_t ps = __dp4a(m.x, 0x01010101u, __dp4a(m.y, 0x01010101u, __dp4a(m.z, 0x01010101u, __dp4a(m.w, 0x01010101u, 0u))));
            ps += __shfl_xor_sync(0xffffffffu, ps, 1);
            ps += __shfl_xor_sync(0xffffffffu, ps, 2);
            if (live && rsrow && (idx & 3) == 0) rsrow[i] = ps;
          }
          __syncwarp();
          if (lane == 0) mbar_arrive(vfree_bar(vs));
          if (pt == 0) stem_trace(a, 7, tn, 18, ve);
        }
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTsTmemCols);
  }
}

}  // namespace slq

using namespace slq;

static void stem_dims(int H, int W, int *Hc, int *Wc, int *Hp, int *Wp) {
  *Hc = (H + 6 - 7) / 2 + 1;
  *Wc = (W + 6 - 7) / 2 + 1;
  *Hp = (*Hc + 2 - 3) / 2 + 1;
  *Wp = (*Wc + 2 - 3) / 2 + 1;
}

extern "C" int64_t slq_stem_workspace_bytes(int32_t N, int32_t H, int32_t W) {
  if (N <= 0 || H < 7 || W < 7) return -1;
  return 64 * kSfK * (2 + 4);  // the weight matrix in fp16 and in fp32; activations never leave the SM
}

extern "C" int slq_stem_create(int32_t N, int32_t H, int32_t W, void *workspace, slq_stem **out) {
  SLQ_CHECK_ARG(workspace && out, "slq_stem_create: null pointer argument");
  SLQ_CHECK_ARG(N > 0 && H >= 7 && W >= 7, "slq_stem_create: bad shape");
  SLQ_CHECK_ARG(reinterpret_cast<uintptr_t>(workspace) % 256 == 0, "slq_stem_create: workspace must be 256-byte aligned");
  slq_stem *s = new (std::nothrow) slq_stem();
  SLQ_CHECK_ARG(s != nullptr, "slq_stem_create: out of host memory");
  s->N = N; s->H = H; s->W = W;
  stem_dims(H, W, &s->Hc, &s->Wc, &s->Hp, &s->Wp);
  if (s->Wc > 128 || 3 * W > 3 * 256) {
    delete s;
    set_error("slq_stem_create: the tcgen05 stem maps one output row to one 128-pixel tile (W <= 256); use slq_stem_forward");
    return SLQ_ERR_UNSUPPORTED;
  }
  s->wh = reinterpret_cast<__half *>(workspace);
  s->wf = reinterpret_cast<float *>(reinterpret_cast<uint8_t *>(workspace) + 64 * kSfK * 2);
  s->use_ts = (W % 16 == 0) ? 1 : 0;
#if SLQ_DEBUG_TRACE
  if (getenv("SLQ_STEM_OLD")) s->use_ts = 0;  // A/B timing of the round-1 kernel (debug build only)
#endif
  const int units_per_img = (s->Hp + kSfUnitRows - 1) / kSfUnitRows;
  s->num_ctas = (int)std::min<long long>((long long)N * units_per_img, sm_count());
  cudaError_t e = set_smem_limit_once<stem_fused_kernel<SLQ_IN_F32>>(kSfSmemBytes);
  if (e == cudaSuccess) e = set_smem_limit_once<stem_fused_kernel<SLQ_IN_F16>>(kSfSmemBytes);
  if (e == cudaSuccess) e = set_smem_limit_once<stem_fused_kernel<SLQ_IN_U8>>(kSfSmemBytes);
  if (e == cudaSuccess) e = set_smem_limit_once<stem_ts_kernel<SLQ_IN_F32>>(kTsSmemBytes);
  if (e == cudaSuccess) e = set_smem_limit_once<stem_ts_kernel<SLQ_IN_F16>>(kTsSmemBytes);
  if (e == cudaSuccess) e = set_smem_limit_once<stem_ts_kernel<SLQ_IN_U8>>(kTsSmemBytes);
  if (e != cudaSuccess) {
    delete s;
    set_error("slq_stem_create: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    return SLQ_ERR_CUDA;
  }
  *out = s;
  return SLQ_OK;
}

extern "C" void slq_stem_destroy(slq_stem *s) { delete s; }

extern "C" int slq_stem_set_weights(slq_stem *s, const float *w, void *stream) {
  SLQ_CHECK_ARG(s && w, "slq_stem_set_weights: null pointer argument");
  if (s->use_ts) stem_weights_ts_kernel<<<(64 * kSfK + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, s->wf);
  else stem_weights_kernel<<<(64 * kSfK + 255) / 256, 256, 0, (cudaStream_t)stream>>>(w, s->wh);
  SLQ_LAUNCH_CHECK();
  return SLQ_OK;
}

extern "C" int slq_stem_launch(slq_stem *s, const float *x, const float *bn_a, const float *bn_b,
                               const float *act_scales, int32_t out_id, void *out, int32_t out_mode,
                               float *f32_scratch, uint32_t *out_rowsum, void *stream) {
  return slq_stem_launch_in(s, x, SLQ_IN_F32, nullptr, bn_a, bn_b, act_scales, out_id, out, out_mode, f32_scratch,
                            out_rowsum, stream);
}

extern "C" int slq_stem_launch_in(slq_stem *s, const void *x, int32_t in_kind, const float *norm, const float *bn_a,
                                  const float *bn_b, const float *act_scales, int32_t out_id, void *out,
                                  int32_t out_mode, float *f32_scratch, uint32_t *out_rowsum, void *stream) {
  SLQ_CHECK_ARG(s && x && bn_a && bn_b && out, "slq_stem_launch: null pointer argument");
  SLQ_CHECK_ARG(in_kind == SLQ_IN_F32 || in_kind == SLQ_IN_F16 || in_kind == SLQ_IN_U8, "slq_stem_launch: in_kind %d", in_kind);
  SLQ_CHECK_ARG(in_kind != SLQ_IN_U8 || norm != nullptr, "slq_stem_launch: u8 input needs norm = {mean[3], std[3]}");
  SLQ_CHECK_ARG(out_mode == SLQ_OUT_U8 || out_mode == SLQ_OUT_F32, "slq_stem_launch: out_mode %d", out_mode);
  SLQ_CHECK_ARG(out_mode == SLQ_OUT_U8 ? act_scales != nullptr : f32_scratch != nullptr,
                "slq_stem_launch: act_scales (u8) / f32_scratch (fp32) required");
  cudaStream_t st = (cudaStream_t)stream;
  StemArgs a;
  a.x = x;
  for (int c = 0; c < 3; ++c) {
    a.nmean[c] = in_kind == SLQ_IN_U8 ? norm[c] : 0.f;
    a.nstd[c] = in_kind == SLQ_IN_U8 ? norm[3 + c] : 1.f;
  }
  a.N = s->N; a.H = s->H; a.W = s->W; a.Hc = s->Hc; a.Wc = s->Wc; a.Hp = s->Hp; a.Wp = s->Wp;
  a.wh = s->wh;
  a.wf = s->wf;
  a.bn_a = bn_a; a.bn_b = bn_b; a.act_scales = act_scales; a.out_id = out_id; a.out_mode = out_mode;
  a.out = out_mode == SLQ_OUT_U8 ? out : (void *)f32_scratch;
  a.out_rowsum = out_mode == SLQ_OUT_U8 ? out_rowsum : nullptr;
  a.units_per_img = (s->Hp + kSfUnitRows - 1) / kSfUnitRows;
  a.total_units = s->N * a.units_per_img;
  {
    int cap = 0;
    debug_trace_buffer(&a.trace, &cap);
    a.trace_cap = cap;
#if SLQ_DEBUG_TRACE
    const char *d = getenv("SLQ_STEM_DBG");
    a.dbg = d ? atoi(d) : 0;
#else
    a.dbg = 0;
#endif
  }
  if (s->use_ts) {
    SLQ_CHECK_ARG(reinterpret_cast<uintptr_t>(x) % 16 == 0, "slq_stem_launch: the image must be 16-byte aligned");
    // the image as a 3-D tensor [3N planes][H][W]; one box = {W, 2 rows, 3 channels} = one input-row pair
    const int esz = in_kind == SLQ_IN_F32 ? 4 : (in_kind == SLQ_IN_F16 ? 2 : 1);
    CUtensorMap tmX;
    const cuuint64_t dims[3] = {(cuuint64_t)s->W, (cuuint64_t)s->H, (cuuint64_t)3 * s->N};
    const cuuint64_t strides[2] = {(cuuint64_t)s->W * esz, (cuuint64_t)s->H * s->W * esz};
    const cuuint32_t box[3] = {(cuuint32_t)s->W, 2, 3};
    const CUtensorMapDataType dt = in_kind == SLQ_IN_F32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                   : (in_kind == SLQ_IN_F16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16 : CU_TENSOR_MAP_DATA_TYPE_UINT8);
    const int rc = encode_tiled(&tmX, dt, 3, x, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_NONE, "stem image");
    if (rc != SLQ_OK) return rc;
    if (in_kind == SLQ_IN_F32) stem_ts_kernel<SLQ_IN_F32><<<s->num_ctas, kTsThreads, kTsSmemBytes, st>>>(tmX, a);
    else if (in_kind == SLQ_IN_F16) stem_ts_kernel<SLQ_IN_F16><<<s->num_ctas, kTsThreads, kTsSmemBytes, st>>>(tmX, a);
    else stem_ts_kernel<SLQ_IN_U8><<<s->num_ctas, kTsThreads, kTsSmemBytes, st>>>(tmX, a);
  } else if (in_kind == SLQ_IN_F32) stem_fused_kernel<SLQ_IN_F32><<<s->num_ctas, kSfThreads, kSfSmemBytes, st>>>(a);
  else if (in_kind == SLQ_IN_F16) stem_fused_kernel<SLQ_IN_F16><<<s->num_ctas, kSfThreads, kSfSmemBytes, st>>>(a);
  else stem_fused_kernel<SLQ_IN_U8><<<s->num_ctas, kSfThreads, kSfSmemBytes, st>>>(a);
  SLQ_LAUNCH_CHECK();
  if (out_mode == SLQ_OUT_F32)
    return launch_stem_pool(f32_scratch, s->N, s->Hc, s->Wc, s->Hp, s->Wp, act_scales, out_id, out, SLQ_OUT_F32, nullptr, st);
  return SLQ_OK;
}
