/*
 * include/slq.h -- C ABI of libslq_b200.so: the B200 (sm_100a) hot path of
 * kenm-28/Semilayer-Wise-Mixed-Precision-Quantization.
 *
 * The reference has no FFI of its own (it is pure Python on torch).  Each entry point below cites
 * the reference call site whose ATen kernels it replaces; INTEGRATION.md shows the ctypes binding a
 * maintainer adds to functions.py / resnet.py.
 *
 * Conventions
 *   - plain C types only: pointers + sizes, no torch types, no C++ exceptions across the boundary;
 *   - the caller owns every buffer (the Python host allocates them with torch) -- the library
 *     allocates device memory only inside the *_host convenience calls;
 *   - `stream` is a cudaStream_t passed as void* (NULL = legacy default stream);
 *   - every function returns SLQ_OK or an SLQ_ERR_* code; slq_last_error() gives the message;
 *   - device entry points only enqueue work: they never synchronise;
 *   - safe to call from one host thread per device.
 */
#ifndef SLQ_H_
#define SLQ_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SLQ_ABI_VERSION 1

#if defined(__GNUC__)
#define SLQ_API __attribute__((visibility("default")))
#else
#define SLQ_API
#endif

/* ---- status codes ------------------------------------------------------------------------- */
#define SLQ_OK 0
#define SLQ_ERR_INVALID 1     /* bad argument (message says which) */
#define SLQ_ERR_CUDA 2        /* a CUDA runtime / driver call failed */
#define SLQ_ERR_ZERO_RANGE 3  /* constant row: the reference raises ZeroDivisionError (functions.py:40) */
#define SLQ_ERR_UNSUPPORTED 4 /* shape outside what the kernels implement */

/* per-row status written by the quantizer kernels (bit flags) */
#define SLQ_ROW_OK 0
#define SLQ_ROW_ZERO_RANGE 1 /* max == min: scale == 0 (row left untouched) */
#define SLQ_ROW_CODE_RANGE 2 /* a code fell outside [0, 2^bit-1] and was clamped */

/* fp32 divide flavour of functions.py:41 `tensor/scale` (SURVEY.md F5) */
#define SLQ_DIV_TRUE 0  /* IEEE fp32 divide: what ATen does for CPU tensors */
#define SLQ_DIV_RECIP 1 /* multiply by float32(1.0 / scale64): ATen CUDA div by a CPU scalar */

SLQ_API const char *slq_last_error(void);
SLQ_API int slq_abi_version(void);
/* sm_count / cc_major / cc_minor of the current device (any pointer may be NULL) */
SLQ_API int slq_device_info(int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor);

/* =============================================================================================
 * 1. Per-channel affine quantizer
 *    replaces  functions.py:25-43  quantize_wgt(tensor, bit)
 *              functions.py:9-23   channel_wise_quantizationperchan(tensor, bit, i)
 *    (min/max -> fp64 scale, z -> five separately rounded fp32 ops; SURVEY.md Appendix A)
 * ============================================================================================= */

/* Bytes of one packed row: bit 8/6 -> K, 4 -> ceil(K/2), 2 -> ceil(K/4), 16 -> 2K (lo plane, hi plane).
 * Codes are little-endian inside a byte: element i of a 4-bit row sits in byte i/2, bits 4*(i%2).. */
SLQ_API int64_t slq_packed_row_bytes(int64_t K, int32_t bit);

/* One launch for a work-list of (row, bit) jobs over ONE contiguous fp32 weight tensor [n_rows, K]
 * (an OIHW conv weight viewed as rows).  A semilayer is such a list with one bit-width; the whole
 * model's layers can be issued back to back on the same stream.
 *   w          in/out  device [n_rows*K] fp32; row rows[j] is overwritten with its de-quantised
 *                      value when write_back != 0 (the in-place contract of functions.py:22)
 *   rows, bits in      device [n_jobs] int32   (bit in 1..8)
 *   codes      out     device blob or NULL; job j's packed codes start at codes + code_offsets[j]
 *   code_offsets in    device [n_jobs] int64, each a multiple of 4 (ignored when codes == NULL)
 *   z, s32     out     device [n_jobs] or NULL: zero point (functions.py:40) and float32(scale)
 *   status     out     device [n_jobs] SLQ_ROW_* flags (required)
 * Real weight of element i of job j: (code + z[j]) * s32[j].                                     */
SLQ_API int slq_quantize_rows(float *w, int64_t n_rows, int64_t K, const int32_t *rows, const int32_t *bits,
                      int32_t n_jobs, int32_t div_mode, int32_t write_back, uint8_t *codes,
                      const int64_t *code_offsets, int32_t *z, float *s32, int32_t *status,
                      void *stream);

/* Same operation on HOST buffers (what an FFI caller without device memory binds; also the `e2e`
 * leg of bench.py): copies w to the device, runs slq_quantize_rows, copies the results back and
 * synchronises.  Returns SLQ_ERR_ZERO_RANGE if any job hit a constant row (results of the other
 * jobs are still valid), like the reference's ZeroDivisionError.                                  */
SLQ_API int slq_quantize_rows_host(float *w, int64_t n_rows, int64_t K, const int32_t *rows,
                           const int32_t *bits, int32_t n_jobs, int32_t div_mode, int32_t write_back,
                           uint8_t *codes, const int64_t *code_offsets, int32_t *z, float *s32,
                           int32_t *status);

/* The same quantizer over a MULTI-TENSOR job table: one launch for every (row, bit) job of a whole model
 * (resnet50_main.py:189-197 walks all 22,656 rows of the 48 quantised convs once per bit-width phase).
 * jobs is a DEVICE array sorted by the caller into three classes, in this order:
 *   n_small jobs with K <= 288, n_mid jobs with K <= 1152, n_large jobs with K <= 4608;
 * every row pointer must be 16-byte aligned and K a multiple of 4 (rows that are not go through
 * slq_quantize_rows).  z / s32 (may be NULL) / status are indexed like jobs.                         */
typedef struct slq_qjob {
  float *row;     /* device: K contiguous fp32, overwritten in place when write_back != 0          */
  uint8_t *codes; /* device: where this row's packed codes go (slq_packed_row_bytes), or NULL     */
  int32_t K;
  int32_t bit;    /* 1..8 */
} slq_qjob;
SLQ_API int slq_quantize_jobs(const slq_qjob *jobs, int32_t n_small, int32_t n_mid, int32_t n_large,
                              int32_t div_mode, int32_t write_back, int32_t *z, float *s32, int32_t *status,
                              void *stream);

/* Packed rows -> fp32: w[row, e] = fp32((code + z[row]) * s[row]).  For rows of <= 8 bits this is exactly the
 * value the quantizer wrote back (functions.py:41: (round(w/scale + z) - z) * scale), so a packed snapshot
 * restores a fake-quantised model bit for bit -- the device-resident replacement of the mains' undo buffer
 * torch.save(net.state_dict()) / torch.load (resnet50_main.py:212, :233-234) and the loader of the packed
 * on-disk format.  codes / code_offsets / bit / z / s as written by slq_quantize_rows or slq_encode_rows. */
SLQ_API int slq_decode_rows(const uint8_t *codes, const int64_t *code_offsets, const int32_t *bit,
                            const int32_t *z, const float *s, int64_t n_rows, int64_t K, float *w, void *stream);

/* Content-derived classification used when the forward has to consume weights that were quantised
 * elsewhere (the mains mutate conv.weight.data and reload fp32 state_dicts; SURVEY.md H4):
 * for every row of w [n_rows, K] find the smallest bit in {2,4,6,8} whose affine grid (spanned by
 * the row's own min/max) already contains every element; rows that are on no such grid (never
 * quantised) get bit 16.  Writes bit/z/s per row.  No codes are produced here.
 * For rows of <= 8 bits the scale is then refined to the neighbouring float (within 2 ulp) for which
 * fp32(rint(w / s) * s) == w holds for EVERY element, i.e. the scale the row was quantised with:
 * exact[row] (may be NULL) = 1 when such a scale exists -- the packed row then decodes bit for bit
 * (slq_decode_rows) -- else 0 (the row is still within 0.02 grid steps of the grid found).          */
SLQ_API int slq_classify_rows(const float *w, int64_t n_rows, int64_t K, int32_t *bit, int32_t *z, float *s,
                      int32_t *exact, void *stream);

/* Packs rows whose (bit, z, s) are already known (from slq_classify_rows): code = clamp(rint(w/s) - z).
 * Job j reads row j (all rows, in order).                                                        */
SLQ_API int slq_encode_rows(const float *w, int64_t n_rows, int64_t K, const int32_t *bit, const int32_t *z,
                    const float *s, uint8_t *codes, const int64_t *code_offsets, void *stream);

/* =============================================================================================
 * 2. Quantised convolution = implicit GEMM on tcgen05 (u8 x u8 -> s32 in TMEM) + fused epilogue
 *    replaces  resnet.py:22-30 nn.Conv2d (called resnet.py:57,60,99,103,107 and the downsample
 *              convs :63,:111) + native_batch_norm (:58,61,100,104,108) + add_ (:65,:113)
 *              + relu_ (:59,66,101,105,114)
 * ============================================================================================= */

#define SLQ_IMPL_UMMA 0 /* TMA + tcgen05.mma kind::i8 + TMEM (the product path) */
#define SLQ_IMPL_SIMT 1 /* CUDA-core dp4a kernel: on-device cross-check used by tests */

#define SLQ_A_AUTO 0      /* 1x1 stride-1: tiled TMA over [M, Cin]; otherwise im2col TMA */
#define SLQ_A_IM2COL 1    /* force im2col-mode TMA */
#define SLQ_A_TILED 2     /* force tiled TMA (1x1 stride-1 pad-0 only) */

#define SLQ_OUT_U8 0  /* u8 NHWC, re-quantised with act_scales[out_id] (the inference path) */
#define SLQ_OUT_F32 1 /* fp32 NHWC after BN/residual/ReLU (calibration pass) */
#define SLQ_OUT_ACC 2 /* raw s32 accumulators (parity tests): out[M, Cout] (w16: [M, 2*Cout], low
                         limb block then high limb block) and window sums out_S[M] */
#define SLQ_OUT_S8 3  /* s8 NHWC with scale absmax/127: tensors that are not post-ReLU, i.e. the
                         downsample branch bn(conv1x1(x)) of resnet.py:63/:111 */

typedef struct slq_conv_desc {
  int32_t N, H, W, Cin;              /* input activations: u8 NHWC */
  int32_t Cout, kh, kw, stride, pad; /* cross-correlation, no bias, groups=1, dilation=1 */
  int32_t w16;                       /* 0: 8-bit codes (one limb); 1: 16-bit codes (two u8 limbs) */
  int32_t impl;                      /* SLQ_IMPL_* */
  int32_t a_mode;                    /* SLQ_A_* */
} slq_conv_desc;

typedef struct slq_conv slq_conv; /* opaque: tensor maps + launch geometry of one layer */

/* Rows of the GEMM-ready weight matrix for a layer and its K extent (= kh*kw*Cin). */
SLQ_API int64_t slq_gemm_weight_rows(const slq_conv_desc *d);

/* Builds the GEMM-ready B operand from the packed per-row store:
 *   wg [slq_gemm_weight_rows(d), kh*kw*Cin] u8, K ordered (r, s, c) to match NHWC activations.
 *   w8 : row oc = codes of channel oc (bit <= 8 rows, 2/4-bit rows unpacked), zero rows up to a
 *        multiple of the N tile.
 *   w16: per 64-channel tile t, rows [128t, 128t+64) = low limbs, [128t+64, 128t+128) = high limbs.
 * packed rows are in OIHW order (c, r, s) as slq_quantize_rows / slq_encode_rows wrote them.      */
SLQ_API int slq_build_gemm_weights(const slq_conv_desc *d, const uint8_t *codes, const int64_t *code_offsets,
                           const int32_t *bit, uint8_t *wg, void *stream);

SLQ_API int slq_conv_create(const slq_conv_desc *d, const uint8_t *in, const uint8_t *wg, slq_conv **out);

/* PACKED weights, unpacked to int8 in shared memory (BASELINE north_star; SURVEY.md H5).
 * Layers whose whole n-tile of weights stays resident in shared memory (the 1x1 convs up to K = 512 and the
 * 3x3 64->64 convs of ResNet-50) can take their B operand as the packed store itself: per n-tile and K block,
 * the rows' codes back to back -- rows of <= 4 bits two codes per byte (low nibble = even k), wider rows one code
 * per byte -- fetched with one bulk copy per K block and expanded in place by the epilogue warps before the first MMA.
 *   slq_conv_tiling          the tiling the kernel uses for this layer: columns (rows of B) per n-tile, n-tiles,
 *                            codes of K per K block, K blocks, and whether the weights are resident (packable)
 *   layout (computed by the caller from the per-channel bit-widths):
 *     row_offsets[t][r]  (uint16, r = 0..bn_cols)  byte offset of row r inside one (n-tile t, K block) segment;
 *                        a row takes k_block/2 bytes (bit <= 4) or k_block bytes; rows past Cout count as 4-bit
 *     seg_bytes[t] = row_offsets[t][bn_cols];  tile_base[t] = sum over earlier tiles of num_kb * seg_bytes
 *   slq_build_packed_gemm_weights   fills wgp from the per-row packed store (slq_quantize_rows / slq_encode_rows)
 *   slq_conv_set_packed_weights     attaches it to the handle (all four pointers are DEVICE pointers; NULL wgp
 *                                   detaches); launches of non-resident / two-limb layers ignore it            */
SLQ_API int slq_conv_tiling(const slq_conv_desc *d, int32_t *bn_cols, int32_t *n_tiles, int32_t *k_block,
                            int32_t *num_kb, int32_t *resident);
SLQ_API int slq_build_packed_gemm_weights(const slq_conv_desc *d, const uint8_t *codes, const int64_t *code_offsets,
                                          const int32_t *bit, const int64_t *tile_base, const int32_t *seg_bytes,
                                          const uint16_t *row_offsets, uint8_t *wgp, void *stream);
SLQ_API int slq_conv_set_packed_weights(slq_conv *c, const uint8_t *wgp, const int64_t *tile_base,
                                        const int32_t *seg_bytes, const uint16_t *row_offsets);
SLQ_API void slq_conv_destroy(slq_conv *c);

typedef struct slq_epilogue {
  const float *wscale;     /* [Cout] s32[oc] * bn_a[oc]   (bn_a = gamma / sqrt(var + eps))        */
  const float *zf;         /* [Cout] (float) z[oc]                                                 */
  const float *bias;       /* [Cout] bn_b[oc] = beta - mean * bn_a                                 */
  const float *act_scales; /* device array of per-tensor activation scales                        */
  int32_t in_id, out_id, res_id; /* indices into act_scales; res_id < 0: no residual              */
  const uint8_t *res;      /* [M, Cout] NHWC residual (block identity) or NULL                    */
  int32_t res_signed;      /* 0: res is u8 (a post-ReLU tensor); 1: s8 (a SLQ_OUT_S8 tensor)       */
  void *out;               /* see SLQ_OUT_*                                                        */
  int32_t *out_S;          /* SLQ_OUT_ACC only: [M] window sums, may be NULL                       */
  int32_t out_mode;
  int32_t relu;
  /* Window sums S[m] of the INPUT for the zero-point term z[oc] * S[m].  Layers that run 64- / 128-channel tiles
   * let the tensor core produce S (a row of ones behind the weight rows) and ignore these fields.  Layers that run
   * 256-channel tiles (slq_conv_needs_rowsum) gather S from a ROWSUM side tensor of their input: a stack of PLANES of
   * one uint32 per pixel whose sum is the channel sum of the pixel.  A producer whose output feeds such a layer is
   * given out_rowsum and writes one plane per n-tile of its launch (plain stores: no atomics, nothing to zero).   */
  const uint32_t *in_rowsum; /* [in_planes][in_plane_stride], in_plane_stride >= N*H*W pixels of the input; may be
                                NULL unless slq_conv_needs_rowsum()                                            */
  uint32_t *out_rowsum;      /* SLQ_OUT_U8 only, may be NULL: [slq_conv_rowsum_planes()][M] planes of the output */
  int32_t in_planes;
  int64_t in_plane_stride;
} slq_epilogue;

/* Debug timeline: when buf != NULL, CTA 0 of every later slq_conv_launch logs (event+1, index, SM clock)
 * triples into buf (3*capacity_events int64, zeroed by the caller; 24 issuers own capacity/24 slots
 * each).  Events: 0/1 A load issue begin/end, 2/3 B load issue begin/end, 4 MMA saw K block, 5/6
 * epilogue tile begin/end.  NULL switches tracing off.  Not for production use.                    */
SLQ_API int slq_debug_set_trace(int64_t *buf, int32_t capacity_events);

/* Planes a launch of this layer writes into slq_epilogue.out_rowsum (= n-tiles of the tiling it will use, which
 * depends on whether the launch has a residual); 0 for the SIMT checker.                                  */
SLQ_API int32_t slq_conv_rowsum_planes(const slq_conv *c, int32_t has_residual);
/* 1 when a launch of this layer (with / without residual) gathers its window sums from slq_epilogue.in_rowsum. */
SLQ_API int32_t slq_conv_needs_rowsum(const slq_conv *c, int32_t has_residual);

/* y[m, oc] = (acc[m,oc] + z[oc] * S[m]) * wscale[oc] * act_scales[in_id] + bias[oc]
 *            (+ res[m,oc] * act_scales[res_id]) ; ReLU ; u8 = clamp(rint(y / act_scales[out_id])) */
SLQ_API int slq_conv_launch(slq_conv *c, const slq_epilogue *e, void *stream);

/* ---------------------------------------------------------------------------------------------
 * 2b. Tail of a residual block WITH a downsample branch as one launch
 *     replaces  resnet.py:107-114 (Bottleneck.forward): out = bn3(conv3(y2)); identity = downsample(x) =
 *               bn_d(conv1x1_stride_s(x)); out += identity; out = relu(out)
 * Both 1x1 GEMMs of a 128-pixel x 64-channel tile accumulate side by side in tensor memory (conv3: u8 x u8 codes;
 * downsample: u8 x two u8 limbs of its 16-bit codes, the reference keeps these weights in fp32) and ONE epilogue
 * folds them, so the identity tensor never exists in HBM and is never rounded to 8 bits:
 *   per channel : A3 = wscale3*s[in3_id] ; Ad = wscaled*s[ind_id] ; B = bias3 + biasd     (u8 out: each * 1/s[out_id])
 *                 Z3 = zf3*A3 ; Zd = zfd*Ad
 *   per element : accd = fma(f32(hi), 256, f32(lo))
 *                 y = fma(accd, Ad, fma(f32(acc3), A3, fma(f32(Sd), Zd, fma(f32(S3), Z3, B))))
 *   fp32 out    : max(y, 0)          u8 out : sat_u8(rint(y))
 * (oracle/slq_oracle.py `block_tail` / `block_tail_q` restate it).  The kernel keeps the weights of one 64-channel
 * n-tile of BOTH convs resident in shared memory: slq_blocktail_create returns SLQ_ERR_UNSUPPORTED when they do
 * not fit (Cmid = 512 / Cin = 1024, the last stage of ResNet-50) -- the caller then launches the two convs
 * separately (slq_conv_launch with the downsample output as s8 residual).
 * ------------------------------------------------------------------------------------------- */
typedef struct slq_blocktail_desc {
  int32_t N, H, W, Cin; /* block input x: u8 NHWC [N, H, W, Cin]                                        */
  int32_t stride;       /* of the downsample conv (1 or 2); outputs are Ho = (H-1)/stride + 1 pixels     */
  int32_t Cmid;         /* channels of y2 = conv3's input: u8 NHWC [N, Ho, Wo, Cmid]                     */
  int32_t Cout;         /* output channels of both convs                                                 */
  int32_t impl;         /* SLQ_IMPL_UMMA, or SLQ_IMPL_SIMT: the dp4a checker of the same arithmetic      */
} slq_blocktail_desc;

typedef struct slq_blocktail slq_blocktail; /* opaque */

typedef struct slq_blocktail_epilogue {
  const float *wscale3, *zf3, *bias3; /* conv3 + bn3, as in slq_epilogue                                 */
  const float *wscaled, *zfd, *biasd; /* downsample conv + its BN                                        */
  const float *act_scales;
  int32_t in3_id, ind_id, out_id;     /* scales of y2, of x and of the output                            */
  void *out;                          /* [M, Cout] u8 (SLQ_OUT_U8) or fp32 (SLQ_OUT_F32)                 */
  int32_t out_mode;
  uint32_t *out_rowsum;               /* SLQ_OUT_U8, may be NULL: [slq_blocktail_rowsum_planes()][M]      */
} slq_blocktail_epilogue;

/* y2, x: the two input activations; wg3: GEMM-ready weights of conv3 built with w16 = 0, wgd: of the downsample conv
 * built with w16 = 1 (slq_build_gemm_weights).  All four are device pointers the handle keeps.            */
SLQ_API int slq_blocktail_create(const slq_blocktail_desc *d, const uint8_t *y2, const uint8_t *x, const uint8_t *wg3,
                                 const uint8_t *wgd, slq_blocktail **out);
SLQ_API void slq_blocktail_destroy(slq_blocktail *h);
SLQ_API int32_t slq_blocktail_rowsum_planes(const slq_blocktail *h);
SLQ_API int slq_blocktail_launch(slq_blocktail *h, const slq_blocktail_epilogue *e, void *stream);

/* =============================================================================================
 * 3. Un-quantised ends of the network and calibration helpers
 * ============================================================================================= */

/* Stem: resnet.py:206-209  conv1 7x7 s2 p3 (3->64, fp32 weights) + bn1 + relu + maxpool 3x3 s2 p1.
 * x fp32 NCHW [N,3,H,W] -> out NHWC [N,Hp,Wp,64], Hp = ((H+1)/2+1)/2 (u8 via act_scales[out_id], or
 * fp32 when out_mode == SLQ_OUT_F32).  `scratch` holds the pre-pool activations:
 * N*Hc*Wc*64 floats with Hc = (H+1)/2.  out_rowsum (SLQ_OUT_U8, may be NULL): [N*Hp*Wp] channel sum of
 * every output pixel: the single rowsum plane of the stem's output (see slq_epilogue.in_rowsum).        */
SLQ_API int slq_stem_forward(const float *x, int32_t N, int32_t H, int32_t W, const float *w,
                     const float *bn_a, const float *bn_b, const float *act_scales, int32_t out_id,
                     float *scratch, void *out, int32_t out_mode, uint32_t *out_rowsum, void *stream);

/* The same stem on the tensor cores (the product path; slq_stem_forward above is the exact-fp32
 * CUDA-core version kept as on-device checker and for W > 256).  Operands pass through tcgen05 as
 * fp16 with fp32 accumulation -- these weights are NOT quantised (the reference keeps them fp32).
 * `workspace` (slq_stem_workspace_bytes, 256-byte aligned, caller-owned) holds the weight matrix in the
 * kernel's K order (fp16 and fp32: the BN scale is folded in before the rounding to fp16); activations
 * never leave the SM.
 * out: u8 NHWC [N,Hp,Wp,64] (SLQ_OUT_U8, scale act_scales[out_id]) or fp32 (SLQ_OUT_F32; then
 * f32_scratch must hold N*Hc*Wc*64 floats).                                                      */
typedef struct slq_stem slq_stem;
SLQ_API int64_t slq_stem_workspace_bytes(int32_t N, int32_t H, int32_t W);
SLQ_API int slq_stem_create(int32_t N, int32_t H, int32_t W, void *workspace, slq_stem **out);
SLQ_API void slq_stem_destroy(slq_stem *s);
/* w: fp32 [64,3,7,7] device pointer (resnet.py:143 conv1.weight) */
SLQ_API int slq_stem_set_weights(slq_stem *s, const float *w, void *stream);
SLQ_API int slq_stem_launch(slq_stem *s, const float *x, const float *bn_a, const float *bn_b,
                            const float *act_scales, int32_t out_id, void *out, int32_t out_mode,
                            float *f32_scratch, uint32_t *out_rowsum, void *stream);
/* The same launch for the other element types a loader may hand over (the data format on the host side
 * of the path, imagenet.py:14-40): SLQ_IN_F16 = the fp32 image already rounded to fp16 (the stem rounds
 * its operands to fp16 anyway, so the logits are bit-identical to the fp32 call); SLQ_IN_U8 = raw pixels,
 * normalised on the fly exactly as torchvision's ToTensor + Normalize (imagenet.py:14-15):
 * (u8 / 255 - mean[c]) / std[c] in fp32; `norm` = HOST floats {mean[3], std[3]} (SLQ_IN_U8 only).     */
#define SLQ_IN_F32 0
#define SLQ_IN_F16 1
#define SLQ_IN_U8 2
SLQ_API int slq_stem_launch_in(slq_stem *s, const void *x, int32_t in_kind, const float *norm,
                               const float *bn_a, const float *bn_b, const float *act_scales, int32_t out_id,
                               void *out, int32_t out_mode, float *f32_scratch, uint32_t *out_rowsum, void *stream);

/* Tail: resnet.py:216-218  adaptive_avg_pool2d((1,1)) + flatten + fc (fp32 weights + bias).
 * x u8 NHWC [N, HW, C] -> logits fp32 [N, O].  The fc runs as a split-K GEMM on the tensor cores
 * (tcgen05.mma kind::tf32, fp32 accumulation).  A TF32 operand carries 10 significand bits, so both operands
 * are split into two TF32 terms (x = x_hi + x_lo, exact) and three products are accumulated
 * (lo*hi + hi*lo + hi*hi): fp32-class accuracy for weights the reference keeps in fp32.
 *   slq_tail_split_weights: fc_w fp32 [O, C] -> fc_w_split fp32 [2][O][C] ({hi, lo} planes), once per weight change
 *   workspace: slq_tail_workspace_bytes(N, C, O) bytes, 16-byte aligned, caller-owned (pooled {hi, lo} +
 *   the per-split partial sums, which are added in a fixed order: the result is deterministic).
 *   C: a multiple of 32, at most 12288 (the pool keeps C integer sums in shared memory).               */
SLQ_API int64_t slq_tail_workspace_bytes(int32_t N, int32_t C, int32_t O);
SLQ_API int slq_tail_split_weights(const float *fc_w, int32_t O, int32_t C, float *fc_w_split, void *stream);
SLQ_API int slq_tail_forward(const uint8_t *x, int32_t N, int32_t HW, int32_t C, const float *act_scales,
                     int32_t in_id, const float *fc_w_split, const float *fc_b, int32_t O, float *workspace,
                     float *logits, void *stream);

/* Calibration of the static per-tensor activation scales (the reference never quantises
 * activations, SURVEY.md F2; this path must): act_scales[id] = max|y| / qmax (1.0 if max == 0),
 * qmax = 255 for post-ReLU (u8) tensors, 127 for signed (s8) ones.
 * `tmp` is one device uint32 of scratch, zeroed by the call.                                     */
SLQ_API int slq_absmax_scale(const float *y, int64_t n, float *act_scales, int32_t id, int32_t qmax,
                     uint32_t *tmp, void *stream);

/* Histogram calibration (opt-in; abs-max above is the default).  A scale set by the single largest element
 * only grows with more data; a threshold read from the distribution of |y| does not.
 * slq_act_histogram ADDS the counts of |y[0..n)| (y 4-byte aligned, any offset) to histogram `id` of
 * hist [.][bins + 1] (device uint64, zeroed by the caller before the first call):
 *   hist[id][0]      exact zeros (either sign)
 *   hist[id][1 + j]  0 < |y| with j = min(trunc(fp32(|y| * fp32(bins / range[id]))), bins - 1): values at or
 *                    above range[id] land in the last bin
 * slq_hist_scales turns histograms [n_tensors][bins + 1] into act_scales[0..n_tensors), one CTA per tensor, in
 * fp64.  Candidate thresholds T_k = fp32(fp32(range * k) / bins), k = 1..bins (T_bins == range).
 *   SLQ_CALIB_PERCENTILE  smallest k with zeros + n_0 + .. + n_{k-1} >= ceil(percentile / 100 * total),
 *                         total including the zeros; 0 < percentile <= 100
 *   SLQ_CALIB_MSE         k minimising sum_j n_j * (c_j - Q(c_j))^2 over the bin centres c_j = (j + 0.5) * range / bins,
 *                         Q(v) = D * min(rint(v / D), qmax), D = T_k / qmax; exact ties go to the larger k
 *   SLQ_CALIB_ENTROPY     k minimising the KL divergence D_k (TensorRT's and pytorch-quantization's entropy
 *                         calibrator; bins >= 128).  n_j = hist[1 + j], N = sum_j n_j (zeros left out: they
 *                         quantise to 0 at every threshold), nq = qmax + 1 levels; candidates k = 128..bins:
 *                           o_k = sum_{j >= k} n_j (outliers), clipped onto the last bin:
 *                             P_j = n_j (j < k - 1), P_{k-1} = n_{k-1} + o_k
 *                           group(j) = floor(j * nq / k) (integers); m_g = sum of n_j over group g, c_g = its
 *                             bins with n_j > 0; Q_j = m_g / c_g where n_j > 0, else 0 (sum Q = N - o_k)
 *                           D_k = sum_{P_j > 0} (P_j / N) ln((P_j / N) / (Q_j / (N - o_k))); +inf when some
 *                             P_j > 0 has Q_j = 0 (n_{k-1} = 0 < o_k, or N == o_k); D_bins is finite
 *                         exact ties go to the larger k.  The device sums, per candidate, in fp64 and in
 *                         increasing j over the bins with n_j > 0:
 *                           D_k = (sum_j P_j * ln((P_j * (c_g * (N - o_k))) / (m_g * N))) / N,  g = group(j)
 *                         so a bin with P_j == Q_j adds exactly 0 when o_k == 0.
 *   act_scales[t] = fp32(fp32(T_k / qmax[t]) * headroom), or 1.0 when the tensor has no non-zero element.
 * bins: a power of two, at most 2048.  Counts are integers (below 2^53) and every fp64 sum runs in a fixed
 * order: the results are deterministic.                                                                 */
#define SLQ_CALIB_PERCENTILE 1
#define SLQ_CALIB_MSE 2
#define SLQ_CALIB_ENTROPY 3
SLQ_API int slq_act_histogram(const float *y, int64_t n, const float *range, int32_t id, int32_t bins,
                              uint64_t *hist, void *stream);
SLQ_API int slq_hist_scales(const uint64_t *hist, int32_t n_tensors, int32_t bins, const float *range,
                            const int32_t *qmax, int32_t method, double percentile, float headroom,
                            float *act_scales, void *stream);
/* out[i] = clamp(rint(y[i] / act_scales[id]), 0, 255)  (is_signed: clamp to [-128, 127], s8: the range of
 * every s8 producer, cvt.rni.sat.s8, and of slq_oracle.requant_s8) */
SLQ_API int slq_quantize_act(const float *y, int64_t n, const float *act_scales, int32_t id,
                     int32_t is_signed, uint8_t *out, void *stream);

/* =============================================================================================
 * 4. Evaluation tail (callers of the forward)
 *    replaces  functions.py:109-122  output.max(1) + CrossEntropyLoss + Softmax, per batch
 *              functions.py:142-146  KLdiv: a Python loop with one reduction per SAMPLE
 * ============================================================================================= */

/* logits [B, C] fp32 (device).  labels [B] int64 or NULL.  probs_out [B, C] or NULL: softmax(logits).
 * ref_probs [B, C] or NULL: p of KL(p || softmax(logits)), i.e. the stored outputs of the un-quantised model.
 * rows: scratch, 3*B floats.  accum: 4 doubles on the device, zeroed by the caller before the first batch:
 *   accum[0] += number of argmax == label      accum[1] += batch-mean cross-entropy (one value per batch)
 *   accum[2] += sum over the batch of KL_b      accum[3] += B
 * Deterministic (fixed summation order); nothing is synchronised.                                      */
SLQ_API int slq_eval_tail(const float *logits, const int64_t *labels, int32_t B, int32_t C, float *probs_out,
                          const float *ref_probs, float *rows, double *accum, void *stream);
/* KL(p || q) of two probability tensors [B, C]: accum[2] += sum_b sum_c p*log(p/q), accum[3] += B. */
SLQ_API int slq_kl_rows(const float *p, const float *q, int32_t B, int32_t C, float *rows, double *accum,
                        void *stream);

/* =============================================================================================
 * 5. Roofline probe
 * ============================================================================================= */

/* Enqueues, on every SM, `iters` (a multiple of 4) K blocks of back-to-back tcgen05.mma.kind::i8
 * (M = 128, N = 256, K = 4 x 32, u8 x u8 -> s32) from two warps: the dense INT8 rate of this GPU, the
 * denominator of the conv kernels' roofline fraction.  *ops_out (host, may be NULL) = 2 * MACs enqueued.
 * The caller times the launch with CUDA events.                                                        */
SLQ_API int slq_probe_i8_peak(int32_t iters, int64_t *ops_out, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* SLQ_H_ */
