// csrc/block_tail.cu -- the tail of a residual block WITH a downsample branch as ONE kernel.
//
// Replaces, for the first block of a stage (resnet.py:107-114 Bottleneck.forward; :60-66 BasicBlock has 3x3
// convs and is not covered),
//     out = conv3(y2) ; out = bn3(out)                         1x1, quantised weights (<= 8-bit codes)
//     identity = downsample(x) = bn_d(conv1x1_stride_s(x))     weights the reference keeps in fp32: 16-bit codes
//     out += identity ; out = relu(out)
// Round 1 ran the downsample conv as its own two-limb launch that WROTE the identity as an s8 tensor (205 MB at
// 56x56) for conv3's epilogue to READ back as its residual: four launches that cost 290 us of a 2.3 ms step, all
// of them epilogue-bound.  Here both 1x1 GEMMs of a 128-pixel x 64-channel tile accumulate side by side in
// tensor memory,
//     columns [0, 64)   acc3 = y2 . W3^T     (u8 x u8, K = Cmid)   + ones column 64  -> S3 = sum_k y2
//     columns [80, 144) low limbs  \  x . Wd^T  (u8 x two u8 limbs, K = Cin, stride s through the im2col TMA)
//     columns [144, 208) high limbs /                               + ones column 208 -> Sd = sum_k x
// and ONE epilogue folds them:  y = A3 (acc3 + z3 S3) + Ad ((lo + 256 hi) + zd Sd) + B ; ReLU ; u8.  The identity
// never exists in HBM (and is never rounded to 8 bits).
//
// Roles (640 threads, 1 CTA/SM): two operand pipelines (tile i -> pipeline i & 1: a TMA producer warp, an MMA warp, an
// operand ring and a TMEM accumulator each) feed ONE epilogue crew of 16 warps that drains every tile together
// (warp = TMEM lane quarter x 16-channel slice): the accumulator of tile i is free again after ~1/2 of the time an
// 8-warp team needs, and while the crew works on tile i the other pipeline's MMAs for tile i + 1 run -- with one
// accumulator per pipeline (2 x 224 of the 512 TMEM columns) the epilogue and the MMAs of the SAME pipeline can never
// overlap, so a team per pipeline (the first version) paid MMA + epilogue per tile.  The CTA keeps the weights of ONE
// 64-channel n-tile (both convs) resident in shared memory for its whole life.  sm_100a only.
//
// Measured and NOT kept: reading the accumulators in the 16x256b (mma fragment) shape, so that a thread always owns
// the same four channels and their 20 constants stay in registers instead of 1.25 broadcast LDS.128 per output --
// bit-identical results, but 166 / 97 / 82 us per launch against 140 / 93 / 76 us for this version (the byte-pair
// shared-memory stores and the quad shuffles of the window sums cost more than the constant loads they replace).
#include <algorithm>
#include <new>

#include "conv_common.cuh"
#include "tma_host.cuh"
#include "umma_ptx.cuh"

struct slq_blocktail {
  slq_blocktail_desc d;
  int Ho, Wo, swz, k3_blocks, kd_blocks, stages, smem_bytes, grid, n_tiles;
  long long M;
  const uint8_t *y2, *x, *wg3, *wgd;
  CUtensorMap tmA3, tmAd, tmB3, tmBd, tmO;
  const void *out_ptr;
};

namespace slq {

constexpr int kBtThreads = 640;
constexpr int kBtCrew = 512;      // epilogue threads
constexpr int kBtStage = 3;       // output staging tiles (TMA store of tile i in flight while i + 1, i + 2 are staged)
constexpr int kBtN3 = 80;    // UMMA N of the conv3 part: 64 channels + the ones group
constexpr int kBtNd = 144;   // UMMA N of the downsample part: 64 low + 64 high limbs + the ones group
constexpr int kBtAccCols = 256;  // TMEM columns per pipeline (224 used)
constexpr int kBtMaxStages = 4;

struct BtArgs {
  long long M;
  int N, H, W, Ho, Wo, stride, Cin, Cmid, Cout;
  int k3_blocks, kd_blocks, stages, m_tiles, n_tiles, d_im2col;
  int b3_off, bd_off, ring_off, out_off, prm_off, bar_off;  // byte offsets from the 1024-aligned smem base
  const float *wscale3, *zf3, *bias3, *wscaled, *zfd, *biasd, *act_scales;
  int in3_id, ind_id, out_id, out_mode;
  void *out;
  uint32_t *out_rowsum;
  long long *stats;  // debug build: wait statistics of CTA 0, or NULL
  int dbg;  // $SLQ_BT_DBG (debug build only, timing experiments): 1 no constant loads, 2 no limb TMEM loads, 4 no staging /
            // store, 8 no downsample MMAs, 32 results overwritten (the arithmetic itself still runs: a runtime flag)
};
#define BT_DBG(a) (kDebugTrace ? (a).dbg : 0)

// per-channel constants of the fused epilogue, structure of arrays in shared memory (64 channels):
//   A3 = wscale3 * s_y2 [* inv] ; Z3 = zf3 * A3 ; Ad = wscaled * s_x [* inv] ; Zd = zfd * Ad ; B = (bias3 + biasd) [* inv]
// y = fma(accd, Ad, fma(acc3, A3, fma(Sd, Zd, fma(S3, Z3, B)))) with accd = fma(f32(hi), 256, f32(lo))
struct BtChan { float a3, z3, ad, zd, b; };
__host__ __device__ inline BtChan bt_chan(float wscale3, float zf3, float bias3, float wscaled, float zfd, float biasd,
                                          float s_y2, float s_x, float inv, bool quantised) {
  BtChan c;
#ifdef __CUDA_ARCH__
  c.a3 = __fmul_rn(wscale3, s_y2);
  c.ad = __fmul_rn(wscaled, s_x);
  c.b = __fadd_rn(bias3, biasd);
  if (quantised) { c.a3 = __fmul_rn(c.a3, inv); c.ad = __fmul_rn(c.ad, inv); c.b = __fmul_rn(c.b, inv); }
  c.z3 = __fmul_rn(zf3, c.a3);
  c.zd = __fmul_rn(zfd, c.ad);
#else
  c.a3 = wscale3 * s_y2; c.ad = wscaled * s_x; c.b = bias3 + biasd;
  if (quantised) { c.a3 *= inv; c.ad *= inv; c.b *= inv; }
  c.z3 = zf3 * c.a3; c.zd = zfd * c.ad;
#endif
  return c;
}

template <int SWZ, int OUT>  // OUT: SLQ_OUT_U8 | SLQ_OUT_F32
__global__ void __launch_bounds__(kBtThreads, 1)
block_tail_kernel(const __grid_constant__ CUtensorMap tmA3, const __grid_constant__ CUtensorMap tmAd,
                  const __grid_constant__ CUtensorMap tmB3, const __grid_constant__ CUtensorMap tmBd,
                  const __grid_constant__ CUtensorMap tmO, const BtArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem = smem_raw + (smem_base - smem_u32(smem_raw));
  constexpr int kABytes = kTileM * SWZ;
  const uint32_t bar_base = smem_base + a.bar_off;
  // barriers: per pipeline p (0/1): full[p][s], empty[p][s] (s < stages), tfull[p], tempty[p]; bfull once
  auto full_bar = [&](int p, int s) { return bar_base + 8u * (p * 2 * kBtMaxStages + s); };
  auto empty_bar = [&](int p, int s) { return bar_base + 8u * (p * 2 * kBtMaxStages + kBtMaxStages + s); };
  auto tfull_bar = [&](int p) { return bar_base + 8u * (4 * kBtMaxStages + p); };
  auto tempty_bar = [&](int p) { return bar_base + 8u * (4 * kBtMaxStages + 2 + p); };
  const uint32_t bfull_bar = bar_base + 8u * (4 * kBtMaxStages + 4);
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(smem + a.bar_off + 8 * (4 * kBtMaxStages + 5));
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;

  // this CTA's n-tile (fixed) and m-tiles (strided), like the resident-weight walk of conv_umma.cu
  const int per_n = (int)gridDim.x / a.n_tiles;
  const int my_n = (int)blockIdx.x % a.n_tiles;
  const int first_m = (int)blockIdx.x / a.n_tiles;
  const int count = first_m < a.m_tiles ? (a.m_tiles - first_m + per_n - 1) / per_n : 0;
  const int kb_tile = a.k3_blocks + a.kd_blocks;

  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA3); prefetch_tmap(&tmAd); prefetch_tmap(&tmB3); prefetch_tmap(&tmBd);
    if (OUT == SLQ_OUT_U8) prefetch_tmap(&tmO);
  }
  if (warp == 1 && lane == 0) {
    for (int p = 0; p < 2; ++p) {
      for (int s = 0; s < a.stages; ++s) { mbar_init(full_bar(p, s), 1); mbar_init(empty_bar(p, s), 1); }
      mbar_init(tfull_bar(p), 1);
      mbar_init(tempty_bar(p), kBtCrew / 32);  // one arrival per crew warp
    }
    mbar_init(bfull_bar, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, 512);
  // the ones groups behind the weight rows of every resident B tile (row 0 of the group = 0x01.., rows 1..15 = 0)
  for (int i = threadIdx.x; i < kb_tile * 16 * (SWZ / 16); i += blockDim.x) {
    const int t = i / (16 * (SWZ / 16)), rem = i % (16 * (SWZ / 16));
    const int row = rem / (SWZ / 16), chunk = rem % (SWZ / 16);
    const uint4 v = row == 0 ? make_uint4(0x01010101u, 0x01010101u, 0x01010101u, 0x01010101u) : make_uint4(0, 0, 0, 0);
    const int base = t < a.k3_blocks ? a.b3_off + t * (kBtN3 * SWZ) + 64 * SWZ
                                     : a.bd_off + (t - a.k3_blocks) * (kBtNd * SWZ) + 128 * SWZ;
    *reinterpret_cast<uint4 *>(smem + base + row * SWZ + chunk * 16) = v;
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0 || warp == 2) {
    // ================================ producers (pipeline p = tiles i with i & 1 == p) ===========
    const int p = warp >> 1;
    if (p == 0 && count > 0) {  // the resident weights of this CTA's n-tile, once
      if (elect_one()) {
        mbar_expect_tx(bfull_bar, (uint32_t)(a.k3_blocks * 64 * SWZ + a.kd_blocks * 128 * SWZ));
        for (int kb = 0; kb < a.k3_blocks; ++kb)
          tma_load_2d(smem_base + a.b3_off + kb * (kBtN3 * SWZ), &tmB3, bfull_bar, kb * SWZ, my_n * 64);
        for (int kb = 0; kb < a.kd_blocks; ++kb)
          tma_load_2d(smem_base + a.bd_off + kb * (kBtNd * SWZ), &tmBd, bfull_bar, kb * SWZ, my_n * 128);
      }
      __syncwarp();
    }
    grid_dependency_wait();  // activations of the previous layers
    int c = 0;  // pipeline steps issued by this producer
    long long w_empty = 0;
    const bool st_on = kDebugTrace && a.stats != nullptr && blockIdx.x == 0;
    const long long t_begin = clock64();
    for (int i = p; i < count; i += 2) {
      const int m0 = (first_m + i * per_n) * kTileM;
      int dn = 0, dh = 0, dw = 0;
      if (a.d_im2col) {  // base pixel of the tile in the block input (stride s, no padding)
        const int hw = a.Ho * a.Wo;
        dn = m0 / hw;
        const int rem = m0 - dn * hw, ph = rem / a.Wo;
        dh = ph * a.stride;
        dw = (rem - ph * a.Wo) * a.stride;
      }
      for (int kb = 0; kb < kb_tile; ++kb, ++c) {
        const int s = c % a.stages;
        mbar_wait_stat(empty_bar(p, s), (uint32_t)(((c / a.stages) & 1) ^ 1), w_empty, st_on);
        if (elect_one()) {
          const uint32_t dst = smem_base + a.ring_off + (p * a.stages + s) * kABytes;
          mbar_expect_tx(full_bar(p, s), kABytes);
          if (kb < a.k3_blocks) tma_load_2d(dst, &tmA3, full_bar(p, s), kb * SWZ, m0);
          else if (a.d_im2col) tma_load_im2col_4d(dst, &tmAd, full_bar(p, s), (kb - a.k3_blocks) * SWZ, dw, dh, dn, 0, 0);
          else tma_load_2d(dst, &tmAd, full_bar(p, s), (kb - a.k3_blocks) * SWZ, m0);
        }
        __syncwarp();
      }
    }
    if (st_on && lane == 0) { a.stats[p] = w_empty; a.stats[2 + p] = clock64() - t_begin; }
  } else if (warp == 1 || warp == 3) {
    // ================================ MMA issuers ==============================================
    const int p = warp >> 1;
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0) + p * kBtAccCols;
    const uint32_t idesc3 = (2u << 4) | ((uint32_t)(kBtN3 >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
    const uint32_t idescd = (2u << 4) | ((uint32_t)(kBtNd >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
    if (count > p) {
      mbar_wait(bfull_bar, 0);
      tc_fence_after();
    }
    int c = 0, t = 0;
    long long w_full = 0, w_tempty = 0;
    const bool st_on = kDebugTrace && a.stats != nullptr && blockIdx.x == 0;
    const long long t_begin = clock64();
    for (int i = p; i < count; i += 2, ++t) {
      if (t >= 1) mbar_wait_stat(tempty_bar(p), (uint32_t)((t - 1) & 1), w_tempty, st_on);  // the crew drained this pipeline's previous tile
      tc_fence_after();
      for (int kb = 0; kb < kb_tile; ++kb, ++c) {
        const int s = c % a.stages;
        mbar_wait_stat(full_bar(p, s), (uint32_t)((c / a.stages) & 1), w_full, st_on);
        tc_fence_after();
        if (elect_one()) {
          const uint64_t da = make_smem_desc<SWZ>(smem_base + a.ring_off + (p * a.stages + s) * kABytes);
          const bool is3 = kb < a.k3_blocks;
          const uint64_t db = make_smem_desc<SWZ>(smem_base + (is3 ? a.b3_off + kb * (kBtN3 * SWZ)
                                                                   : a.bd_off + (kb - a.k3_blocks) * (kBtNd * SWZ)));
          const bool first = is3 ? kb == 0 : kb == a.k3_blocks;  // first K block of its accumulator
#pragma unroll
          for (int k = 0; k < SWZ / 32 && !(!is3 && (BT_DBG(a) & 8)); ++k)
            umma_i8(tmem_u + (is3 ? 0 : kBtN3), da + 2 * k, db + 2 * k, is3 ? idesc3 : idescd, (uint32_t)(!first || k != 0));
          umma_commit(empty_bar(p, s));
          if (kb == kb_tile - 1) umma_commit(tfull_bar(p));
        }
        __syncwarp();
      }
    }
    if (st_on && lane == 0) { a.stats[4 + p] = w_full; a.stats[6 + p] = w_tempty; a.stats[8 + p] = clock64() - t_begin; }
  } else if (warp >= 4) {
    // ================================ epilogue crew ============================================
    grid_dependency_wait();
    const int slice = (warp - 4) >> 2;        // channels [16 slice, 16 slice + 16) of the tile
    const int wq = warp & 3;                  // TMEM lane quarter this warp may read
    const int et = threadIdx.x - 128;
    const int row = wq * 32 + lane;
    constexpr bool kQuant = OUT == SLQ_OUT_U8;
    float *prm = reinterpret_cast<float *>(smem + a.prm_off);  // A3 | Z3 | Ad | Zd | B, 64 floats each
    const uint32_t prm_s = smem_base + a.prm_off + (uint32_t)slice * 64;
    volatile uint32_t *rs_base = reinterpret_cast<volatile uint32_t *>(smem + a.prm_off + 5 * 64 * 4);  // [2][3][128]
    const uint32_t row_byte = (uint32_t)(row * 64), row_sw = (uint32_t)((row >> 1) & 3);
    if (et < 64) {  // the n-tile never changes: constants once
      const int oc = my_n * 64 + et;
      const float inv = kQuant ? __fdiv_rn(1.0f, a.act_scales[a.out_id]) : 1.0f;
      const BtChan c = bt_chan(a.wscale3[oc], a.zf3[oc], a.bias3[oc], a.wscaled[oc], a.zfd[oc], a.biasd[oc],
                               a.act_scales[a.in3_id], a.act_scales[a.ind_id], inv, kQuant);
      prm[et] = c.a3; prm[64 + et] = c.z3; prm[128 + et] = c.ad; prm[192 + et] = c.zd; prm[256 + et] = c.b;
    }
    named_bar_sync(1, kBtCrew);
    const uint32_t tlane = tmem_base + ((uint32_t)(wq * 32) << 16);
    const int c0 = slice * 16;
    const bool want_rs = kQuant && a.out_rowsum != nullptr;
    long long w_tfull = 0, w_bar = 0, seg[6] = {0, 0, 0, 0, 0, 0}, tseg = 0;
#define BT_SEG(k) do { if (st_on) { const long long now__ = clock64(); seg[k] += now__ - tseg; tseg = now__; } } while (0)
    const bool st_on = kDebugTrace && a.stats != nullptr && blockIdx.x == 0 && et == 0;
    const long long t_begin = clock64();
    for (int i = 0; i < count; ++i) {
      const int p = i & 1, t = i >> 1;          // pipeline / accumulator, and its tile ordinal
      const int m_tile = first_m + i * per_n;
      const long long m = (long long)m_tile * kTileM + row;
      const bool valid = m < a.M;
      const uint32_t tcol = tlane + p * kBtAccCols;
      mbar_wait_stat(tfull_bar(p), (uint32_t)(t & 1), w_tfull, st_on);
      if (st_on) tseg = clock64();
      tc_fence_after();
      uint32_t a3[16], lo[16], hi[16];
      tmem_ld16(tcol + c0, a3);
      if (!(BT_DBG(a) & 2)) {
        tmem_ld16(tcol + kBtN3 + c0, lo);
        tmem_ld16(tcol + kBtN3 + 64 + c0, hi);
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) { lo[j] = a3[(j + 1) & 15]; hi[j] = a3[(j + 2) & 15]; }
      }
      const float S3 = (float)(int)tmem_ld1(tcol + 64);
      const float Sd = (float)(int)tmem_ld1(tcol + kBtN3 + 128);
      tmem_ld_wait();
      BT_SEG(0);   // TMEM loads
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar(p));  // everything of this tile is in registers: the pipeline's next MMAs may start
      BT_SEG(1);   // fence + arrive
      uint32_t pk[4];
      float *of = reinterpret_cast<float *>(a.out) + m * a.Cout + my_n * 64 + c0;
#pragma unroll
      for (int q4 = 0; q4 < 4; ++q4) {
        const uint32_t pofs = prm_s + (uint32_t)q4 * 16;
        uint4 pa3, pz3, pad, pzd, pb;
        if (!(BT_DBG(a) & 1)) {
          pa3 = lds128(pofs); pz3 = lds128(pofs + 256); pad = lds128(pofs + 512); pzd = lds128(pofs + 768); pb = lds128(pofs + 1024);
        } else {
          pa3 = pz3 = pad = pzd = pb = make_uint4(0x3a000000u + q4, 0x3a100000u, 0x3a200000u, 0x3a300000u);
        }
        const uint32_t va3[4] = {pa3.x, pa3.y, pa3.z, pa3.w}, vz3[4] = {pz3.x, pz3.y, pz3.z, pz3.w};
        const uint32_t vad[4] = {pad.x, pad.y, pad.z, pad.w}, vzd[4] = {pzd.x, pzd.y, pzd.z, pzd.w};
        const uint32_t vb[4] = {pb.x, pb.y, pb.z, pb.w};
        float v[4];
#pragma unroll
        for (int b = 0; b < 4; b += 2) {
          const int j = 4 * q4 + b;
          const float2 f3 = make_float2((float)(int)a3[j], (float)(int)a3[j + 1]);
          const float2 fd = ffma2(make_float2((float)(int)hi[j], (float)(int)hi[j + 1]), make_float2(256.0f, 256.0f),
                                  make_float2((float)(int)lo[j], (float)(int)lo[j + 1]));
          float2 y = ffma2(make_float2(S3, S3), make_float2(__uint_as_float(vz3[b]), __uint_as_float(vz3[b + 1])),
                           make_float2(__uint_as_float(vb[b]), __uint_as_float(vb[b + 1])));
          y = ffma2(make_float2(Sd, Sd), make_float2(__uint_as_float(vzd[b]), __uint_as_float(vzd[b + 1])), y);
          y = ffma2(f3, make_float2(__uint_as_float(va3[b]), __uint_as_float(va3[b + 1])), y);
          y = ffma2(fd, make_float2(__uint_as_float(vad[b]), __uint_as_float(vad[b + 1])), y);
          v[b] = y.x; v[b + 1] = y.y;
        }
        if (BT_DBG(a) & 32) { v[0] = __uint_as_float(a3[4 * q4] ^ lo[4 * q4]); v[1] = v[2] = v[3] = __uint_as_float(hi[4 * q4]); }
        if (!kQuant) {
          if (valid) reinterpret_cast<float4 *>(of)[q4] = make_float4(fmaxf(v[0], 0.f), fmaxf(v[1], 0.f), fmaxf(v[2], 0.f), fmaxf(v[3], 0.f));
        } else {
          pk[q4] = epi_pack4<false>(v[0], v[1], v[2], v[3]);  // saturation at 0 is the ReLU
        }
      }
      if (kQuant) {
        const uint32_t stg = smem_base + a.out_off + (uint32_t)(i % kBtStage) * (kTileM * 64);
        if (!(BT_DBG(a) & 4)) sts128(stg + row_byte + (((uint32_t)slice ^ row_sw) << 4), make_uint4(pk[0], pk[1], pk[2], pk[3]));
        else if ((pk[0] ^ pk[1] ^ pk[2] ^ pk[3]) == 0x12345679u) sts128(stg, make_uint4(pk[0], pk[1], pk[2], pk[3]));
        uint32_t rsum = 0;
        volatile uint32_t *rs_scratch = rs_base + (i & 1) * 384;  // tile i + 1 must not overwrite what tile i still reads
        if (want_rs) {
          rsum = __dp4a(pk[0], 0x01010101u, __dp4a(pk[1], 0x01010101u, __dp4a(pk[2], 0x01010101u, __dp4a(pk[3], 0x01010101u, 0u))));
          if (slice != 0) rs_scratch[(slice - 1) * 128 + row] = rsum;
        }
        BT_SEG(2);   // arithmetic, pack, staging store
        fence_proxy_async_smem();
        BT_SEG(3);   // proxy fence
        const long long tb0 = st_on ? clock64() : 0;
        named_bar_sync(1, kBtCrew);
        if (st_on) w_bar += clock64() - tb0;
        BT_SEG(4);   // crew barrier
        if (et == 0 && !(BT_DBG(a) & 4)) {
          tma_store_2d(&tmO, stg, my_n * 64, m_tile * kTileM);
          tma_store_commit();
          // at most the two newest stores still read their staging tiles: the tile that tile i + 1 overwrites
          // (i + 1 - kBtStage = i - 2) is free before this thread reaches the next barrier
          asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
        }
        if (want_rs && slice == 0) {
          if (valid) a.out_rowsum[(long long)my_n * a.M + m] = rsum + rs_scratch[row] + rs_scratch[128 + row] + rs_scratch[256 + row];
        }
        BT_SEG(5);   // store issue, wait for the staging tile two tiles back
      }
    }
    if (st_on) {
      a.stats[10] = w_tfull; a.stats[11] = w_bar; a.stats[12] = clock64() - t_begin; a.stats[13] = count;
      for (int k = 0; k < 6; ++k) a.stats[16 + k] = seg[k];
    }
    if (kQuant && et == 0) tma_store_wait_all();
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------
// SIMT checker of the same fused operation: thread = (output pixel, output channel)
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) block_tail_simt_kernel(BtArgs a, const uint8_t *__restrict__ y2,
                                                              const uint8_t *__restrict__ x,
                                                              const uint8_t *__restrict__ wg3,
                                                              const uint8_t *__restrict__ wgd) {
  const int oc = blockIdx.y * 32 + (threadIdx.x & 31);
  const long long m = (long long)blockIdx.x * 4 + (threadIdx.x >> 5);
  if (m >= a.M || oc >= a.Cout) return;
  const int wo = (int)(m % a.Wo), ho = (int)((m / a.Wo) % a.Ho), n = (int)(m / ((long long)a.Wo * a.Ho));
  unsigned acc3 = 0, S3 = 0, lo = 0, hi = 0, Sd = 0;
  const uint32_t *yp = reinterpret_cast<const uint32_t *>(y2 + m * a.Cmid);
  const uint32_t *w3 = reinterpret_cast<const uint32_t *>(wg3 + (long long)oc * a.Cmid);
  for (int c4 = 0; c4 < a.Cmid / 4; ++c4) {
    const uint32_t v = __ldg(yp + c4);
    acc3 = __dp4a(v, __ldg(w3 + c4), acc3);
    S3 = __dp4a(v, 0x01010101u, S3);
  }
  const uint32_t *xp = reinterpret_cast<const uint32_t *>(x + (((long long)n * a.H + ho * a.stride) * a.W + wo * a.stride) * a.Cin);
  const uint32_t *wl = reinterpret_cast<const uint32_t *>(wgd + (long long)gemm_row_of(oc, 0, 1) * a.Cin);
  const uint32_t *wh = reinterpret_cast<const uint32_t *>(wgd + (long long)gemm_row_of(oc, 1, 1) * a.Cin);
  for (int c4 = 0; c4 < a.Cin / 4; ++c4) {
    const uint32_t v = __ldg(xp + c4);
    lo = __dp4a(v, __ldg(wl + c4), lo);
    hi = __dp4a(v, __ldg(wh + c4), hi);
    Sd = __dp4a(v, 0x01010101u, Sd);
  }
  const bool quantised = a.out_mode == SLQ_OUT_U8;
  const float inv = quantised ? __fdiv_rn(1.0f, a.act_scales[a.out_id]) : 1.0f;
  const BtChan c = bt_chan(a.wscale3[oc], a.zf3[oc], a.bias3[oc], a.wscaled[oc], a.zfd[oc], a.biasd[oc],
                           a.act_scales[a.in3_id], a.act_scales[a.ind_id], inv, quantised);
  const float fd = __fmaf_rn((float)(int)hi, 256.0f, (float)(int)lo);
  float y = __fmaf_rn((float)(int)S3, c.z3, c.b);
  y = __fmaf_rn((float)(int)Sd, c.zd, y);
  y = __fmaf_rn((float)(int)acc3, c.a3, y);
  y = __fmaf_rn(fd, c.ad, y);
  if (quantised) reinterpret_cast<uint8_t *>(a.out)[m * a.Cout + oc] = (uint8_t)epi_quant_u8(y);
  else reinterpret_cast<float *>(a.out)[m * a.Cout + oc] = fmaxf(y, 0.f);
}

template <int SWZ, int OUT>
static int bt_launch(slq_blocktail *h, const BtArgs &a, cudaStream_t st) {
  constexpr auto kernel = block_tail_kernel<SWZ, OUT>;
  SLQ_CUDA(set_smem_limit_once<kernel>(232448));
  SLQ_CUDA(launch_pdl(kernel, h->grid, kBtThreads, h->smem_bytes, st, h->tmA3, h->tmAd, h->tmB3, h->tmBd, h->tmO, a));
  return SLQ_OK;
}

}  // namespace slq

using namespace slq;

// shared-memory plan: resident weights of one n-tile (both convs) + two operand rings + three staging tiles +
// constants + barriers.  Returns the bytes to request, or -1 if it does not fit (the caller then keeps the two
// separate launches).
static int bt_plan(const slq_blocktail_desc *d, int swz, int *stages, int off[6]) {
  const int k3 = d->Cmid / swz, kd = d->Cin / swz;
  const int b3 = k3 * kBtN3 * swz, bd = kd * kBtNd * swz;
  const int fixed = b3 + bd + kBtStage * kTileM * 64 + (5 * 64 * 4 + 2 * 3 * 128 * 4) + 512 + 1024;
  const int a_bytes = kTileM * swz;
  int st = std::min(kBtMaxStages, (232448 - fixed) / (2 * a_bytes));
  if (st < 2) return -1;
  *stages = st;
  off[0] = 0;                        // b3
  off[1] = b3;                       // bd
  off[2] = b3 + bd;                  // ring (both pipelines)
  off[3] = off[2] + 2 * st * a_bytes;  // output staging
  off[4] = off[3] + kBtStage * kTileM * 64;   // constants + row-sum scratch
  off[5] = off[4] + 5 * 64 * 4 + 2 * 3 * 128 * 4;  // barriers
  return 1024 + off[5] + 512;
}

extern "C" int slq_blocktail_create(const slq_blocktail_desc *d, const uint8_t *y2, const uint8_t *x, const uint8_t *wg3,
                                    const uint8_t *wgd, slq_blocktail **out) {
  SLQ_CHECK_ARG(d && y2 && x && wg3 && wgd && out, "slq_blocktail_create: null pointer argument");
  SLQ_CHECK_ARG(d->N > 0 && d->H > 0 && d->W > 0 && (d->stride == 1 || d->stride == 2), "slq_blocktail_create: bad shape");
  SLQ_CHECK_ARG(d->Cin % 64 == 0 && d->Cmid % 64 == 0 && d->Cout % 64 == 0 && d->Cin > 0 && d->Cmid > 0 && d->Cout > 0,
                "slq_blocktail_create: channel counts must be multiples of 64");
  SLQ_CHECK_ARG(d->impl == SLQ_IMPL_UMMA || d->impl == SLQ_IMPL_SIMT, "slq_blocktail_create: impl %d", d->impl);
  const int swz = (d->Cmid % 128 == 0 && d->Cin % 128 == 0) ? 128 : 64;
  int stages = 0, off[6];
  const int smem = bt_plan(d, swz, &stages, off);
  if (smem < 0) {  // also for the checker: both engines must take the same schedule
    set_error("slq_blocktail_create: the weights of one n-tile (Cmid %d, Cin %d) do not fit in shared memory", d->Cmid, d->Cin);
    return SLQ_ERR_UNSUPPORTED;
  }
  slq_blocktail *h = new (std::nothrow) slq_blocktail();
  SLQ_CHECK_ARG(h != nullptr, "slq_blocktail_create: out of host memory");
  h->d = *d;
  h->Ho = (d->H - 1) / d->stride + 1;
  h->Wo = (d->W - 1) / d->stride + 1;
  h->M = (long long)d->N * h->Ho * h->Wo;
  h->swz = swz;
  h->k3_blocks = d->Cmid / swz;
  h->kd_blocks = d->Cin / swz;
  h->stages = stages;
  h->smem_bytes = smem;
  h->n_tiles = d->Cout / 64;
  h->y2 = y2; h->x = x; h->wg3 = wg3; h->wgd = wgd;
  h->out_ptr = nullptr;
  const long long m_tiles = ceil_div(h->M, kTileM);
  h->grid = (int)(std::min<long long>(std::max(sm_count() / h->n_tiles, 1), m_tiles)) * h->n_tiles;
  if (d->impl == SLQ_IMPL_UMMA) {
    const CUtensorMapSwizzle sw = swz == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    int rc = encode_tiled_u8(&h->tmA3, y2, h->M, d->Cmid, swz, kTileM, sw, "y2");
    if (rc == SLQ_OK) rc = encode_tiled_u8(&h->tmB3, wg3, d->Cout, d->Cmid, swz, 64, sw, "W3");
    if (rc == SLQ_OK) rc = encode_tiled_u8(&h->tmBd, wgd, (long long)h->n_tiles * 128, d->Cin, swz, 128, sw, "Wd");
    if (rc == SLQ_OK) {
      if (d->stride == 1) {
        rc = encode_tiled_u8(&h->tmAd, x, h->M, d->Cin, swz, kTileM, sw, "x");
      } else {  // strided 1x1: the im2col-mode map walks every stride-th pixel
        const int lower[2] = {0, 0}, upper[2] = {0, 0};
        rc = encode_im2col_u8(&h->tmAd, x, d->N, d->H, d->W, d->Cin, lower, upper, d->stride, swz, kTileM, sw, "x");
      }
    }
    if (rc != SLQ_OK) {
      delete h;
      return rc;
    }
    h->tmO = h->tmB3;
  }
  *out = h;
  return SLQ_OK;
}

extern "C" void slq_blocktail_destroy(slq_blocktail *h) { delete h; }

extern "C" int32_t slq_blocktail_rowsum_planes(const slq_blocktail *h) {
  return (h && h->d.impl == SLQ_IMPL_UMMA) ? h->n_tiles : 0;
}

extern "C" int slq_blocktail_launch(slq_blocktail *h, const slq_blocktail_epilogue *e, void *stream) {
  SLQ_CHECK_ARG(h && e, "slq_blocktail_launch: null handle/epilogue");
  SLQ_CHECK_ARG(e->wscale3 && e->zf3 && e->bias3 && e->wscaled && e->zfd && e->biasd && e->act_scales && e->out,
                "slq_blocktail_launch: epilogue vectors missing");
  SLQ_CHECK_ARG(e->out_mode == SLQ_OUT_U8 || e->out_mode == SLQ_OUT_F32, "slq_blocktail_launch: out_mode %d", e->out_mode);
  SLQ_CHECK_ARG(reinterpret_cast<uintptr_t>(e->out) % 16 == 0, "slq_blocktail_launch: out must be 16-byte aligned");
  const slq_blocktail_desc &d = h->d;
  BtArgs a{};
  a.M = h->M; a.N = d.N; a.H = d.H; a.W = d.W; a.Ho = h->Ho; a.Wo = h->Wo; a.stride = d.stride;
  a.Cin = d.Cin; a.Cmid = d.Cmid; a.Cout = d.Cout;
  a.k3_blocks = h->k3_blocks; a.kd_blocks = h->kd_blocks; a.stages = h->stages;
  a.m_tiles = (int)ceil_div(h->M, kTileM); a.n_tiles = h->n_tiles; a.d_im2col = d.stride != 1;
  a.wscale3 = e->wscale3; a.zf3 = e->zf3; a.bias3 = e->bias3; a.wscaled = e->wscaled; a.zfd = e->zfd; a.biasd = e->biasd;
  a.act_scales = e->act_scales; a.in3_id = e->in3_id; a.ind_id = e->ind_id; a.out_id = e->out_id; a.out_mode = e->out_mode;
  a.out = e->out; a.out_rowsum = e->out_mode == SLQ_OUT_U8 ? e->out_rowsum : nullptr;
  a.dbg = 0;
  a.stats = nullptr;
#if SLQ_DEBUG_TRACE
  {
    int cap = 0;
    debug_trace_buffer(&a.stats, &cap);
    if (cap > -16) a.stats = nullptr;  // statistics mode: slq_debug_set_trace(buf, -16 or below)
  }
  if (const char *d = getenv("SLQ_BT_DBG")) a.dbg = atoi(d);
#endif
  cudaStream_t st = (cudaStream_t)stream;
  if (d.impl == SLQ_IMPL_SIMT) {
    dim3 grid((unsigned)ceil_div(h->M, 4), (unsigned)ceil_div(d.Cout, 32));
    block_tail_simt_kernel<<<grid, 128, 0, st>>>(a, h->y2, h->x, h->wg3, h->wgd);
    SLQ_LAUNCH_CHECK();
    return SLQ_OK;
  }
  int stages = 0, off[6];
  bt_plan(&d, h->swz, &stages, off);
  a.b3_off = off[0]; a.bd_off = off[1]; a.ring_off = off[2]; a.out_off = off[3]; a.prm_off = off[4]; a.bar_off = off[5];
  if (e->out_mode == SLQ_OUT_U8 && h->out_ptr != e->out) {
    int rc = encode_tiled_u8(&h->tmO, e->out, h->M, d.Cout, 64, kTileM, CU_TENSOR_MAP_SWIZZLE_64B, "out");
    if (rc != SLQ_OK) return rc;
    h->out_ptr = e->out;
  }
  if (h->swz == 128)
    return e->out_mode == SLQ_OUT_U8 ? bt_launch<128, SLQ_OUT_U8>(h, a, st) : bt_launch<128, SLQ_OUT_F32>(h, a, st);
  return e->out_mode == SLQ_OUT_U8 ? bt_launch<64, SLQ_OUT_U8>(h, a, st) : bt_launch<64, SLQ_OUT_F32>(h, a, st);
}
