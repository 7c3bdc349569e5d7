// csrc/conv_umma.cu -- quantised convolution as an implicit GEMM on Blackwell tensor cores.
//
// Replaces aten::convolution + native_batch_norm + add_ + relu_ of the reference's residual blocks
// (resnet.py:55-68 BasicBlock.forward, :97-116 Bottleneck.forward; conv modules resnet.py:22-30).
//
//   D[m, oc] = sum_k A[m, k] * B[oc, k]         u8 x u8 -> s32, tcgen05.mma kind::i8, D in TMEM
//   A = NHWC u8 activations, gathered by TMA: im2col-mode tensor map for 3x3 / strided layers
//       (zero padding and the (r,s) filter offsets are resolved by the TMA unit), tiled map for
//       1x1 stride-1 layers;  B = GEMM-ready weight codes [rows, K], K ordered (r, s, c).
//   The zero-point correction z[oc]*S[m] (SURVEY.md H3) needs the window sum S[m] = sum_k A[m, k].
//   64- and 128-channel tiles let the tensor core produce it: a constant row of ones behind the B rows of every
//   tile (UMMA N = bn + 16) puts S[m] into one more accumulator column.  The 256-channel tiles of the K-heavy
//   layers have no column to spare (N = 256 is the largest UMMA): there the epilogue gathers S from a ROWSUM side
//   tensor -- one plane of 4 bytes per pixel per n-tile of the producing launch (one DP4A per four outputs in the
//   producer's epilogue, the two half-tile warps combine through shared memory, one coalesced store per pixel) --
//   adding the planes over the <= 9 taps of its window one tile ahead.  Only the small late-stage tensors that
//   feed such layers carry a rowsum; the gather's latency hides behind the long tiles of those layers (in the
//   epilogue-bound early layers both the gather and atomics were measured to cost 10-30 %).
//   K-heavy layers (weights streamed, Cout % 256 == 0) run 256-channel tiles: UMMA N = 256 is the shape at
//   which one tcgen05.mma occupies the tensor pipe for as long as a warp needs to issue the next one
//   (128 cycles, tools/issue_bench.cu), and a K block then moves 48 KB per 512 tensor cycles instead of
//   32 KB per 288 -- the L2 -> SM path (~75 B/clk/SM through TMA) was what capped the 128-channel tiles.
//
// Persistent, warp-specialised CTA (640 threads, 1 CTA/SM):
//   warps 0, 2  TMA producers: pipeline step c (one smem stage = 1-4 K blocks of A, plus the K block's B tile
//               when the weights are streamed) belongs to producer c & 1; warp 0 also loads the resident
//               weights once and one residual tile per output tile; warp 2 allocates TMEM first
//   warps 1, 3  tcgen05.mma issuers: steps (or, on short tiles, whole tiles) alternate between the two;
//               accumulator ring of 3 in TMEM
//   warps 4-11  epilogue team 0  \  tile i -> team i&1, accumulator buffer i%3.  A team is 8 warps:
//   warps 12-19 epilogue team 1  /  two per TMEM lane quarter, each taking half of the tile's channels:
//               tcgen05.ld -> dequant + folded BN + residual + ReLU -> u8 into a swizzled smem tile
//               -> ONE TMA store per tile, so the epilogue's global traffic is coalesced 128-byte
//               lines in both directions.  The epilogue is the issue-bound part of the small-K layers
//               (16 warps = 4 per scheduler keep it near one instruction per cycle per scheduler) and is
//               compiled per (output kind, residual kind) so that no mode branch survives in the loop.
#include <algorithm>
#include <cstdlib>
#include <new>

#include "conv_common.cuh"
#include "tma_host.cuh"
#include "umma_ptx.cuh"

namespace slq {

constexpr int kThreads = 640;   // 20 warps: 96 registers per thread (the epilogue needs them)
constexpr int kTeam = 256;  // threads of one epilogue team
// u8 output / residual staging tile: 128 rows x bn_ch bytes -- 16 KB for 128-channel tiles, 8 KB for 64-channel tiles
// (the 8 KB that a fixed 16 KB stride wasted per tile are what the 3x3 Cin = 64 layers' ring needs to stay 6 deep)
inline int out_tile_bytes(const ConvGeom &g) {
#ifdef SLQ_OUT_TILE_16K  // A/B build: the fixed stride of before
  return kTileM * 128;
#endif
  return kTileM * (g.bn_ch < 128 ? g.bn_ch : 128);
}

constexpr int kMaxStages = 8;
constexpr int kSmemLimit = 232448;  // 227 KB: the most dynamic shared memory one CTA may own

// Shared-memory carve-up of one layer (byte offsets from the 1024-aligned base), decided on the host.
//   streamed B : every pipeline stage holds {A tile, B tile}; B is re-fetched for every tile.
//   resident B : the n-tile's whole weight matrix (num_kb B tiles) stays in smem for all the M tiles a
//                CTA works on, stages hold A only -- `group` consecutive K blocks (A tiles) per stage, so
//                that one barrier round trip, one expect_tx and one loop trip of the issuing warps cover
//                several TMA boxes / MMAs (a warp's control code runs at ~5-10 cycles per dependent
//                instruction, which is what bounds the small-K layers; tools/issue_bench.cu).
struct SmemPlan {
  int stages;        // pipeline depth (even, see make_plan)
  int stage_bytes;   // stride between stages
  int group;         // K blocks per stage (1 when B is streamed)
  int a_bytes;       // kTileM * SWZ
  int b_tile_bytes;  // (bn_cols + 16 rows of the ones group when bn_cols < 256) * SWZ
  int b_resident;    // 1: B tiles at b_off + kb * b_tile_bytes ; 0: inside each stage after A
  int mma_warps;     // 2: warps 1 and 3 issue MMAs (1: warp 1 only; experiments)
  int b_off;
  int res_bufs;      // depth of the residual (block identity) prefetch ring, 0 without residual
  int out_bufs;      // output staging tiles: TWO per epilogue team (resident weights, when they fit: the TMA store of a
                     // tile is still reading one while the team fills the other -- one team barrier per tile), one
                     // per team, ONE shared by both (streamed weights), or NONE (256-channel tiles store from registers)
  int out_tile;      // bytes of one output / residual staging tile (out_tile_bytes)
  int out_off, res_off, prm_off, bar_off;
  int total;         // dynamic smem bytes to request (including 1024 B of alignment slack)
};

constexpr int kMaxResBufs = 4;
constexpr int kPrmBytes = 2 * 3 * 256 * 4 + 4 * 128 * 4;  // per team: A[256] | Z[256] | B[256] floats; then 2 x 128 u32 of row-sum scratch per team
constexpr int kMaxGroup = 4;

inline SmemPlan make_plan(const ConvGeom &g, int swz, bool has_res) {
  SmemPlan p{};
  p.a_bytes = kTileM * swz;
  const int kOutTileBytes = p.out_tile = out_tile_bytes(g);
  p.b_tile_bytes = (g.bn_cols + (g.bn_cols < 256 ? 16 : 0)) * swz;
  const int num_kb = g.Ktot / swz;
  const long long b_all = (long long)num_kb * p.b_tile_bytes;
#if SLQ_DEBUG_TRACE  // experiment knobs exist only in the debug build of the library
  static const int force_group = getenv("SLQ_GROUP") ? atoi(getenv("SLQ_GROUP")) : 0;
  static const int force_mma = getenv("SLQ_MMA_WARPS") ? atoi(getenv("SLQ_MMA_WARPS")) : 0;
#else
  constexpr int force_group = 0, force_mma = 0;
#endif
  // EVEN depth: stage-sized step c goes to producer / MMA warp c & 1 and to stage c % stages, so with an
  // even depth every stage barrier is always waited on by the same warp (an mbarrier wait only names a
  // phase parity; a warp that saw every other phase of a barrier could not tell them apart)
  p.stages = 0;
  for (int rb = has_res ? kMaxResBufs : 0; g.bn_ch != 256 && p.stages == 0 && rb >= (has_res ? 2 : 0); rb -= 2) {
    // out staging (2), residual ring, prm, barriers, alignment slack
    const int fixed = (2 + rb) * kOutTileBytes + kPrmBytes + 512 + 1024;
    const long long room = (long long)kSmemLimit - fixed - b_all;  // for A stages when B is resident
    for (int grp = std::min(kMaxGroup, num_kb); grp >= 1; --grp) {
      if (num_kb % grp != 0 || (force_group && grp > force_group)) continue;
      const int st = (int)std::min<long long>(kMaxStages, room / ((long long)grp * p.a_bytes)) & ~1;
      if (st >= (grp == 1 ? 4 : 4)) {
        p.b_resident = 1; p.group = grp; p.stages = st; p.stage_bytes = grp * p.a_bytes; p.res_bufs = rb; p.out_bufs = 2;
        const int st4 = (int)std::min<long long>(kMaxStages, (room - 2 * kOutTileBytes) / ((long long)grp * p.a_bytes)) & ~1;
        // measured: the residual (expansion) layers gain 6-9 % from it even with a 4-deep ring; the K = 512
        // reductions lose more from a ring cut from 6 to 4 stages than they gain
        if (st4 >= st || (has_res && st4 >= 4)) { p.out_bufs = 4; p.stages = st4; }
        break;
      }
    }
    if (!has_res) break;
  }
  if (p.stages == 0) {
    // streamed weights: these are the K-heavy layers -- few tiles per CTA, epilogue teams idle 80 % of the
    // time, and the {A, B} ring is what runs short (2 -> 4 stages: 54 -> 37 us on the 3x3 256 layer), so
    // the two teams share ONE staging tile and the 16 KB go to the ring (6 stages without residual)
    p.res_bufs = has_res ? kMaxResBufs : 0;
    p.out_bufs = g.bn_ch == 256 ? 0 : 1;
    const int fixed = (p.out_bufs + p.res_bufs) * kOutTileBytes + kPrmBytes + 512 + 1024;
    p.b_resident = 0;
    p.group = 1;
    p.stage_bytes = p.a_bytes + p.b_tile_bytes;
    p.stages = std::min(kMaxStages, (kSmemLimit - fixed) / p.stage_bytes) & ~1;
  }
  p.mma_warps = force_mma ? force_mma : 2;
  p.b_off = p.stages * p.stage_bytes;
  p.out_off = p.b_off + (p.b_resident ? (int)b_all : 0);
  p.res_off = p.out_off + p.out_bufs * kOutTileBytes;
  p.prm_off = p.res_off + p.res_bufs * kOutTileBytes;
  p.bar_off = p.prm_off + kPrmBytes;
  p.total = 1024 + p.bar_off + 512;
  return p;
}

// CTAs to launch: one per SM; with resident weights every CTA keeps ONE n-tile for its whole life, so
// the grid is the largest multiple of n_tiles that fits (148 -> 144 for 8 or 16 n-tiles).
inline int plan_grid(const ConvGeom &g, const SmemPlan &p, int sms) {
  const long long m_tiles = (g.M + kTileM - 1) / kTileM;
  if (p.b_resident) {
    const int per_n = (int)std::min<long long>(std::max(sms / g.n_tiles, 1), m_tiles);
    return per_n * g.n_tiles;
  }
  return (int)std::min<long long>(m_tiles * g.n_tiles, sms);
}

struct KernelArgs {
  ConvGeom g;
  EpiDev e;
  SmemPlan sp;
  int a_im2col;
  int num_kb;          // K blocks per tile = kh*kw*Cin / SWZ
  int num_grp;         // pipeline steps per tile = num_kb / sp.group
  int chunks_per_tap;  // Cin / SWZ
  int tma_out;         // 1: u8/s8 output through the smem tile + TMA store
  int mma_warps_per_tile;  // MMA warps that touch one tile: 2, or 1 when a tile is a single K block / tile_alt
  int tile_alt;            // the two MMA warps alternate whole tiles instead of pipeline steps
  int acc_bufs, acc_stride;  // TMEM accumulator ring: 3 x 160 columns (N <= 128), 2 x 256 (N = 256)
  // packed weights (resident-B layers): the n-tile's codes arrive as the PACKED store (4-bit rows two codes per
  // byte) and are expanded to the u8 operand tiles in shared memory (SURVEY.md H5 / north_star "unpacked in SMEM")
  const uint8_t *wgp;          // NULL: weights come as u8 through tmB
  const long long *wgp_tile;   // [n_tiles] byte offset of the n-tile's first (kb = 0) segment
  const int *wgp_seg;          // [n_tiles] bytes of one (n-tile, kb) segment
  const uint16_t *wgp_rowoff;  // [n_tiles][bn_cols + 1] byte offset of every row inside a segment
  long long m_tiles;
  int half_b;          // debug build: $SLQ_HALF_B experiment (see the producer loop)
  long long *trace;    // debug: CTA 0 logs (event, index, clock) triples here (slq_debug_set_trace)
  int trace_cap;
};

// debug timeline (CTA 0 only): every issuer owns a private region of the buffer, so logging is one
// fire-and-forget store (no atomics: their latency would distort the very thing being measured)
constexpr int kTraceIssuers = 24;
// trace_cap < 0 selects "wait statistics only": every role adds up the cycles it spends blocked in its
// mbarrier waits (mbar_wait_stat) and CTA 0 writes one total per role at the end (slot = role) -- no per-step overhead
__device__ __forceinline__ void trace_ev(const KernelArgs &a, int issuer, int &n, int ev, int idx) {
  if (!kDebugTrace || a.trace == nullptr || a.trace_cap < 0 || blockIdx.x != 0) return;
  const int per = a.trace_cap / kTraceIssuers;
  if (n < per) {
    long long *p = a.trace + 3LL * (issuer * per + n);
    p[0] = ev + 1;  // 0 = empty slot
    p[1] = idx;
    p[2] = clock64();
    ++n;
  }
}

// The tiles one CTA works on, in the order every role walks them.  Both orders are m-major in time
// (CTAs that run together touch neighbouring pixels: A tiles are shared through L2 and the channel
// slices of an output row are written close together).
//   streamed B : tile = blockIdx + i*grid over (m_tile, n_tile) pairs
//   resident B : n_tile = blockIdx % n_tiles for the CTA's whole life, m_tile strided
struct TileWalk {  // everything fits 32 bits (M <= 2^31): no 64-bit divisions on the issue paths
  int count, first_m, step_m;
  int first, step;
  int n_tiles, fixed_n, my_n;
  __device__ TileWalk(const KernelArgs &a) {
    n_tiles = a.g.n_tiles;
    fixed_n = a.sp.b_resident;
    const int m_tiles = (int)a.m_tiles;
    if (fixed_n) {
      const int per_n = (int)gridDim.x / n_tiles;
      my_n = (int)blockIdx.x % n_tiles;
      first_m = (int)blockIdx.x / n_tiles;
      step_m = per_n;
      count = first_m < m_tiles ? (m_tiles - first_m + per_n - 1) / per_n : 0;
      first = step = 0;
    } else {
      const int total = m_tiles * n_tiles;
      first = (int)blockIdx.x;
      step = (int)gridDim.x;
      count = first < total ? (total - first + step - 1) / step : 0;
      my_n = 0; first_m = step_m = 0;
    }
  }
  __device__ void at(int i, int &m_tile, int &n_tile) const {
    if (fixed_n) { n_tile = my_n; m_tile = first_m + i * step_m; }
    else { const int t = first + i * step; m_tile = t / n_tiles; n_tile = t - m_tile * n_tiles; }
  }
};

// accumulator ring in TMEM: tile i -> buffer i % acc_bufs (KernelArgs: 3 buffers 160 columns apart, or 2 x 256
// for the 256-channel tiles)
constexpr int kTileBars = 6;     // per-tile barrier sets: tile i -> set i % 6 (a multiple of acc_bufs and of the 2 teams)
constexpr int kTmemCols = 512;

// byte offset of 16-byte chunk c of row r inside a staging tile whose rows are bn_ch (64|128) bytes,
// stored with the TMA swizzle of that width (so that thread-per-row accesses are conflict-free)
__device__ __forceinline__ uint32_t stage_off(int r, int c, int bn_ch) {
  return bn_ch == 128 ? (uint32_t)(r * 128 + ((c ^ (r & 7)) << 4))
                      : (uint32_t)(r * 64 + ((c ^ ((r >> 1) & 3)) << 4));
}

// Two residual bytes (b, b + 1 of word w; b = 0 or 2) as exact floats.  `I2F.U8` runs on the quarter-rate XU pipe
// through the MIO queue -- with one per output it was the busiest pipe of the expansion layers' epilogue (48 % under
// ncu, profiles/r2_conv_expand_stall_sites.txt) -- so the LOW pair of every word goes another way: a byte permute
// plants each byte in the mantissa of 2^23 (0x4B0000xx = 8388608 + x) and one packed fma(m, 1, -2^23) takes the
// offset off again (exact: the difference is an integer < 2^24).  Measured on 64->256 @56^2: all four bytes through
// I2F.U8 119.2 us, all four through PRMT 115.2, two and two (this) another 2 % better (tools/gpu_r2_call32.sh).
__device__ __forceinline__ float2 res_pair(uint32_t w, int b, bool is_signed) {
  const uint32_t b0 = (w >> (8 * b)) & 255u, b1 = (w >> (8 * b + 8)) & 255u;
  // signed residuals (BasicBlock downsample branches) keep the conversion unit: measured 1.4 % faster there
  if (is_signed) return make_float2((float)(int)(int8_t)b0, (float)(int)(int8_t)b1);
  if (b == 2) return make_float2((float)b0, (float)b1);
  const uint32_t m0 = __byte_perm(w, 0x4B000000u, 0x7440), m1 = __byte_perm(w, 0x4B000000u, 0x7441);
  return ffma2(make_float2(__uint_as_float(m0), __uint_as_float(m1)), make_float2(1.0f, 1.0f),
               make_float2(-8388608.0f, -8388608.0f));
}

// OUT: SLQ_OUT_*;  RES: residual kind
constexpr int kResNone = 0, kResU8 = 1, kResS8 = 2, kResDyn = 3;  // Dyn: decided at run time (fp32/raw outputs)
constexpr int kResWide = 4;  // no residual, 256-channel tile: quantised outputs are stored straight from registers

template <int SWZ, bool W16, int OUT, int RES>
__global__ void __launch_bounds__(kThreads, 1)
conv_umma_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                 const __grid_constant__ CUtensorMap tmO, const __grid_constant__ CUtensorMap tmR,
                 const KernelArgs a) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t *smem = smem_raw + (smem_base - smem_u32(smem_raw));
  const SmemPlan &sp = a.sp;
  const uint32_t bar_base = smem_base + sp.bar_off;
  // barrier slots (8 bytes each)
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (kMaxStages + s); };
  // Per-tile barriers are indexed by tile % kTileBars (6 = lcm of the 3 accumulators and the 2 teams /
  // MMA warps): an mbarrier wait only names a phase PARITY, so every barrier must always be waited on by
  // the same party, which then sees each of its phases in turn.  Tile i uses accumulator i % 3.
  auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * kMaxStages + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * kMaxStages + kTileBars + b); };
  auto tstart_bar = [&](int b) { return bar_base + 8u * (2 * kMaxStages + 2 * kTileBars + b); };
  auto rfull_bar = [&](int b) { return bar_base + 8u * (2 * kMaxStages + 3 * kTileBars + b); };
  auto rempty_bar = [&](int b) { return bar_base + 8u * (2 * kMaxStages + 3 * kTileBars + kMaxResBufs + b); };
  const uint32_t bfull_bar = bar_base + 8u * (2 * kMaxStages + 3 * kTileBars + 2 * kMaxResBufs);  // resident B landed
  auto stfree_bar = [&](int t) { return bar_base + 8u * (2 * kMaxStages + 3 * kTileBars + 2 * kMaxResBufs + 2 + t); };
  const uint32_t bready_bar = bar_base + 8u * (2 * kMaxStages + 3 * kTileBars + 2 * kMaxResBufs + 4);  // packed B expanded
  volatile uint32_t *tmem_slot = reinterpret_cast<volatile uint32_t *>(
      smem + sp.bar_off + 8 * (2 * kMaxStages + 3 * kTileBars + 2 * kMaxResBufs + 1));

  // warp index through a shuffle: the compiler then knows it is warp-uniform and keeps the control loops
  // (stage / barrier / descriptor arithmetic, branches) on the uniform datapath instead of R2UR-ing every
  // TMA / MMA operand out of vector registers
  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0), lane = threadIdx.x & 31;
  const ConvGeom &g = a.g;
  const EpiDev &e = a.e;
  const int bn_cols = g.bn_cols;
  const bool ones_row = bn_cols < 256;  // S[m] from the tensor core (else from the rowsum side tensor)
  const int umma_n = bn_cols + (ones_row ? 16 : 0);
  constexpr bool kWide = RES == kResWide;
  const bool has_res = RES == kResDyn ? (e.res != nullptr) : (RES != kResNone && RES != kResWide);
  const TileWalk walk(a);

  // ---- one-time setup -----------------------------------------------------------------------
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the next kernel may queue behind this one
  const long long t_entry = clock64();
  if (warp == 0 && lane == 0) {
    prefetch_tmap(&tmA);
    prefetch_tmap(&tmB);
    if (!kWide && a.tma_out) prefetch_tmap(&tmO);
    if (has_res) prefetch_tmap(&tmR);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < sp.stages; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int b = 0; b < kTileBars; ++b) {
      mbar_init(tfull_bar(b), (uint32_t)a.mma_warps_per_tile);
      mbar_init(tempty_bar(b), kTeam / 32);  // one arrival per epilogue warp of the team
      mbar_init(tstart_bar(b), 1);
    }
    for (int b = 0; b < sp.res_bufs; ++b) {
      mbar_init(rfull_bar(b), 1);
      mbar_init(rempty_bar(b), kTeam / 32);
    }
    mbar_init(bfull_bar, 1);
    mbar_init(bready_bar, 2 * kTeam);
    mbar_init(stfree_bar(0), 1);
    mbar_init(stfree_bar(1), 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(tmem_slot, kTmemCols);
  // constant "ones" row group behind the B rows of every B tile:
  // row bn_cols = 0x01.., rows bn_cols+1 .. +15 = 0  (identical bytes are swizzle-invariant)
  if (ones_row) {
    const int b_tiles = sp.b_resident ? a.num_kb : sp.stages;
    const int b_stride = sp.b_resident ? sp.b_tile_bytes : sp.stage_bytes;
    const int b_first = sp.b_resident ? sp.b_off : sp.a_bytes;
    for (int i = threadIdx.x; i < b_tiles * 16 * (SWZ / 16); i += blockDim.x) {
      const int t = i / (16 * (SWZ / 16));
      const int rem = i % (16 * (SWZ / 16));
      const int row = rem / (SWZ / 16), chunk = rem % (SWZ / 16);
      uint4 v = row == 0 ? make_uint4(0x01010101u, 0x01010101u, 0x01010101u, 0x01010101u) : make_uint4(0, 0, 0, 0);
      *reinterpret_cast<uint4 *>(smem + b_first + t * b_stride + (bn_cols + row) * SWZ + chunk * 16) = v;
    }
  }
  fence_proxy_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // ================================ TMA producers ===============================================
  // What ONE warp can issue is the unit of throughput here (tools/issue_bench.cu, B200): a warp that
  // walks a division-free loop in convergent code and lets one elected lane issue sustains one TMA box
  // per ~300 cycles (tiled or im2col alike) and one tcgen05.mma per ~140 cycles (128-byte swizzle;
  // ~260 with the 64-byte swizzle) WHATEVER the box size or the MMA's N; issuing from a divergent
  // `if (lane == 0)` region instead makes the compiler wrap every such instruction in an
  // ELECT / R2UR.BROADCAST loop that costs 2-4x more.  Different warps issue concurrently, so the four
  // control warps are dealt as (SmemPlan::mma_warps == 1 frees warp 3 for a third producer):
  //   warps 0 + 2 (+ 3) : producers; pipeline step c (a stage = sp.group K blocks of A, plus the B tile
  //                       of the K block when weights are streamed) belongs to producer c % n_prod
  //   warps 1 + 3       : MMA issuers; step c belongs to MMA warp c & 1
  //   residual tiles    : warp 0, one box per tile, up to a tile ahead of the A tiles it is loading
  //   resident weights  : land once, issued by warp 0
  const int w_mma1 = sp.mma_warps == 2 ? 3 : -1;  // second MMA warp
  const int a_idx = warp == 0 ? 0 : (warp == 2 ? 1 : -1);
  if (a_idx >= 0) {
    const uint32_t b_bytes = (uint32_t)(bn_cols * SWZ);
    const int grp = sp.group;
    const uint32_t tx_bytes = (uint32_t)(grp * sp.a_bytes) + (sp.b_resident ? 0u : b_bytes);
    if (warp == 0 && sp.b_resident && walk.count > 0) {  // this CTA's n-tile never changes
      if (elect_one()) {
        if (a.wgp != nullptr) {
          // packed store: one bulk copy per K block, landing at the END of the block's operand tile; the
          // epilogue warps expand it in place (below) before the first MMA
          const uint32_t seg = (uint32_t)a.wgp_seg[walk.my_n];
          const uint8_t *src = a.wgp + a.wgp_tile[walk.my_n];
          mbar_expect_tx(bfull_bar, seg * (uint32_t)a.num_kb);
          for (int kb = 0; kb < a.num_kb; ++kb)
            bulk_g2s(smem_base + sp.b_off + kb * sp.b_tile_bytes + bn_cols * SWZ - seg, src + (long long)kb * seg, seg, bfull_bar);
        } else {
          mbar_expect_tx(bfull_bar, b_bytes * (uint32_t)a.num_kb);
          for (int kb = 0; kb < a.num_kb; ++kb)
            tma_load_2d(smem_base + sp.b_off + kb * sp.b_tile_bytes, &tmB, bfull_bar, kb * SWZ, walk.my_n * bn_cols);
        }
      }
      __syncwarp();
    }
    grid_dependency_wait();  // activations of the previous layer (weights above are static)
    const int ngrp = a.num_grp, cpt = a.chunks_per_tap;
    const int items = walk.count * ngrp;
    int tn = 0;
    const int tid_ = a_idx * 4;
    const int first = a_idx;
    constexpr int step = 2;  // two producer warps; the pipeline depth is even
    // Everything a step needs is carried incrementally (a warp's control code runs at 5-10 cycles per
    // dependent instruction: ~100 instructions per step were the bottleneck of the K-heavy layers):
    //   (tile i, step gi inside the tile), first K block kb0 = gi * grp, its filter tap (tap_r, tap_s) and
    //   channel chunk, the stage's shared-memory address / barrier / phase; tile coordinates and the tap
    //   state are recomputed (with divisions) only when the tile changes.
    int i = first / ngrp, gi = first - i * ngrp;
    int stage = first % sp.stages;
    uint32_t phase = (uint32_t)((first / sp.stages) & 1);
    uint32_t sa = smem_base + (uint32_t)(stage * sp.stage_bytes);
    const uint32_t sa_step = (uint32_t)(step * sp.stage_bytes), sa_end = smem_base + (uint32_t)(sp.stages * sp.stage_bytes);
    int cur_i = -1, n_tile = 0, m0 = 0, cw = 0, chh = 0, cn = 0;
    int kb0 = 0, tap_r = 0, tap_s = 0, cchunk = 0;
    const int kb_step = step * grp;
    const bool tracing = kDebugTrace && a.trace != nullptr && a.trace_cap >= 0;
    const bool stats = kDebugTrace && a.trace != nullptr && a.trace_cap < 0 && blockIdx.x == 0;
    long long wsum = 0;
    const long long tstart_clk = clock64();
    const bool im2col = a.a_im2col != 0, streamed = !sp.b_resident;
    const int kw = g.kw;
    // residual (block identity) tiles: a ring of res_bufs boxes, filled by warp 0
    const bool res_warp = has_res && warp == 0;
    const uint32_t res_bytes = (uint32_t)(kTileM * g.bn_ch);
    int res_next = 0, res_buf = 0;
    uint32_t res_ph = 0;
    auto issue_residuals = [&](int upto) {  // residual boxes of tiles [res_next, upto]
      for (; res_next <= upto && res_next < walk.count; ++res_next) {
        int mt, nt;
        walk.at(res_next, mt, nt);
        mbar_wait(rempty_bar(res_buf), res_ph ^ 1);
        if (elect_one()) {
          mbar_expect_tx(rfull_bar(res_buf), res_bytes);
          tma_load_2d(smem_base + sp.res_off + res_buf * sp.out_tile, &tmR, rfull_bar(res_buf), nt * g.bn_ch,
                      mt * kTileM);
        }
        __syncwarp();
        if (++res_buf == sp.res_bufs) { res_buf = 0; res_ph ^= 1; }
      }
    };
    for (int c = first; c < items; c += step) {
      if (i != cur_i) {  // new tile: coordinates and tap state from scratch
        if (res_warp) issue_residuals(i + sp.res_bufs - 3);  // never waits on a tile whose A tiles are not loaded yet
        int m_tile;
        walk.at(i, m_tile, n_tile);
        m0 = m_tile * kTileM;
        kb0 = gi * grp;
        if (im2col) {
          const int hw = g.Wo * g.Ho;
          cn = m0 / hw;
          const int rem = m0 - cn * hw;
          const int p = rem / g.Wo;
          cw = (rem - p * g.Wo) * g.stride - g.pad;
          chh = p * g.stride - g.pad;
          const int tap = kb0 / cpt;
          cchunk = kb0 - tap * cpt;
          tap_r = tap / kw;
          tap_s = tap - tap_r * kw;
        }
        cur_i = i;
      }
      const uint32_t fb = full_bar(stage);
      mbar_wait_stat(empty_bar(stage), phase ^ 1, wsum, stats);
      if (tracing && lane == 0) trace_ev(a, tid_, tn, 0, c);
      // debug build, $SLQ_HALF_B: fetch the weight tile only on every other pipeline step (wrong results; shows how
      // much of a streamed-weight layer's time is the B traffic through L2)
      const bool skip_b = kDebugTrace && a.half_b && (c & 2);
      if (elect_one()) {
        mbar_expect_tx(fb, skip_b ? tx_bytes - b_bytes : tx_bytes);
        if (im2col) {
          int cc = cchunk, ts = tap_s, tr = tap_r;
          for (int j = 0; j < grp; ++j) {
            tma_load_im2col_4d(sa + j * sp.a_bytes, &tmA, fb, cc * SWZ, cw, chh, cn, (uint16_t)ts, (uint16_t)tr);
            if (++cc == cpt) { cc = 0; if (++ts == kw) { ts = 0; ++tr; } }
          }
        } else {
          for (int j = 0; j < grp; ++j) tma_load_2d(sa + j * sp.a_bytes, &tmA, fb, (kb0 + j) * SWZ, m0);
        }
        if (streamed && !skip_b) tma_load_2d(sa + sp.a_bytes, &tmB, fb, kb0 * SWZ, n_tile * bn_cols);
      }
      __syncwarp();
      if (tracing && lane == 0) trace_ev(a, tid_, tn, 1, c);
      // advance by `step` pipeline steps
      gi += step;
      kb0 += kb_step;
      if (gi >= ngrp) {
        do { gi -= ngrp; ++i; } while (gi >= ngrp);  // tile change: state is rebuilt at the top of the loop
      } else if (im2col) {
        cchunk += kb_step;
        while (cchunk >= cpt) { cchunk -= cpt; if (++tap_s == kw) { tap_s = 0; ++tap_r; } }
      }
      stage += step; sa += sa_step;
      if (stage >= sp.stages) { stage -= sp.stages; sa -= sa_end - smem_base; phase ^= 1; }
    }
    if (res_warp) issue_residuals(walk.count - 1);
    if (stats && lane == 0) { a.trace[a_idx] = wsum; a.trace[8 + a_idx] = clock64() - tstart_clk; if (a_idx == 0) a.trace[14] = tstart_clk - t_entry; }
  } else if (warp == 1 || warp == w_mma1) {
    // ================================ MMA issuers =============================================
    // With two issuing warps, pipeline step c (counted over all the tiles of this CTA) belongs to warp
    // c & 1 and both accumulate into the tile's TMEM buffer (integer accumulation commutes).  A single
    // warp retires one tcgen05.mma per ~140 cycles whatever its N, i.e. half the tensor pipe at N = 144.
    // Ordering inside a tile: the MMAs of its first step overwrite the accumulator, so the warp that
    // does not own that step waits (tstart) until they have completed before its own first MMA; the
    // accumulator goes to the epilogue (tfull) when BOTH warps' MMAs of the tile have completed.
    // Each WHOLE warp walks the loop (convergent, every operand warp-uniform, so the descriptors live
    // in uniform registers) and one elected lane issues.
    // instruction descriptor: D=s32, A=B=u8, both K-major, M=128, N=umma_n
    const int w = warp == 1 ? 0 : 1;
    const int nmw = sp.mma_warps;
    const uint32_t idesc = (2u << 4) | ((uint32_t)(umma_n >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
    const uint32_t tmem_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint64_t desc_hi = make_smem_desc<SWZ>(0) & 0xffffffff00000000ull;
    const uint32_t desc_lo0 = (uint32_t)(make_smem_desc<SWZ>(0) & 0xffffffffull);  // flags of the low word
    const int n_stages = sp.stages, ngrp = a.num_grp, grp = sp.group;
    const int nw = a.mma_warps_per_tile;  // MMA warps that touch one tile
    const uint32_t stage16 = (uint32_t)sp.stage_bytes >> 4, a16 = (uint32_t)sp.a_bytes >> 4;
    const uint32_t btile16 = (uint32_t)sp.b_tile_bytes >> 4;
    const uint32_t a_lo_first = desc_lo0 | ((smem_base & 0x3FFFFu) >> 4);
    const uint32_t b_lo_first = desc_lo0 | (((smem_base + (uint32_t)sp.b_off) & 0x3FFFFu) >> 4);
    const bool resident = sp.b_resident != 0;
    const bool tracing = kDebugTrace && a.trace != nullptr && a.trace_cap >= 0;
    const bool stats = kDebugTrace && a.trace != nullptr && a.trace_cap < 0 && blockIdx.x == 0;
    long long wfull = 0, wacc = 0;
    const long long tstart_clk = clock64();
    const int items = walk.count * ngrp;
    int tn = 0;
    if (resident && walk.count > 0) {
      mbar_wait(a.wgp != nullptr ? bready_bar : bfull_bar, 0);  // the CTA's weights are in shared memory (as u8)
      tc_fence_after();
    }
    // Which steps this warp issues.  Default: alternate steps (c = w, w + 2, ...), both warps feed the same
    // tile.  tile_alt: alternate whole TILES (tile i -> warp i & 1), so short tiles (2-3 steps) do not make
    // the second warp idle through the first step waiting for tstart; the host enables it when the pipeline
    // depth is a multiple of 2 * steps-per-tile (each stage barrier then always has the same waiter).
    const bool tile_alt = a.tile_alt != 0;
    int i = tile_alt ? w : w / ngrp, gi = tile_alt ? 0 : w - i * ngrp;  // w < 2
    int c0 = tile_alt ? w * ngrp : w;
    int stage = c0 % n_stages;
    uint32_t phase = (uint32_t)((c0 / n_stages) & 1);
    int cur_i = -1, acc = 0, tb = 0;
    for (int c = c0; c < items;) {
      if (i != cur_i) {  // this warp's first step of tile i
        cur_i = i;
        acc = i % a.acc_bufs;
        tb = i % kTileBars;
        if (gi == 0) {  // the epilogue of tile i - 3 has drained this accumulator
          if (i >= a.acc_bufs) mbar_wait_stat(tempty_bar((i - a.acc_bufs) % kTileBars), (uint32_t)(((i - a.acc_bufs) / kTileBars) & 1), wacc, stats);
        } else {        // the overwriting MMAs of this tile have completed
          mbar_wait_stat(tstart_bar(tb), (uint32_t)((i / kTileBars) & 1), wacc, stats);
        }
        tc_fence_after();
      }
      const uint32_t tmem_d = tmem_u + acc * a.acc_stride;
      const uint32_t a_lo = a_lo_first + (uint32_t)stage * stage16;
      const uint32_t b_lo = resident ? b_lo_first + (uint32_t)(gi * grp) * btile16 : a_lo + a16;
      const bool last_mine = tile_alt ? gi + 1 == ngrp : gi + nmw >= ngrp;  // this warp's last step of the tile
      if (tracing && lane == 0) trace_ev(a, 16 + 3 * w, tn, 7, c);
      mbar_wait_stat(full_bar(stage), phase, wfull, stats);
      tc_fence_after();
      if (tracing && lane == 0) trace_ev(a, 16 + 3 * w, tn, 4, c);
      if (elect_one()) {
        for (int j = 0; j < grp; ++j) {
          const uint64_t da = desc_hi | (a_lo + (uint32_t)j * a16), db = desc_hi | (b_lo + (uint32_t)j * btile16);
#pragma unroll
          for (int k = 0; k < SWZ / 32; ++k)  // UMMA_K = 32 bytes of K per instruction
            umma_i8(tmem_d, da + 2 * k, db + 2 * k, idesc, (uint32_t)(gi | j | k) != 0u);
        }
        umma_commit(empty_bar(stage));  // frees the smem slot when these MMAs retire
        if (gi == 0 && nw > 1) umma_commit(tstart_bar(tb));
        if (last_mine) umma_commit(tfull_bar(tb));  // this warp's share of the accumulator is complete
      }
      __syncwarp();
      if (tile_alt) {
        int adv = 1;
        if (++gi == ngrp) { gi = 0; i += 2; adv += ngrp; }  // skip the other warp's tile
        c += adv; stage += adv;
        while (stage >= n_stages) { stage -= n_stages; phase ^= 1; }
      } else {
        c += nmw;
        gi += nmw;
        while (gi >= ngrp) { gi -= ngrp; ++i; }
        stage += nmw;
        if (stage >= n_stages) { stage -= n_stages; phase ^= 1; }
      }
    }
    if (stats && lane == 0) { a.trace[2 + w] = wfull; a.trace[4 + w] = wacc; a.trace[10 + w] = clock64() - tstart_clk; }
  } else if (warp >= 4) {
    // ================================ epilogue (2 teams of 8 warps) ============================
    grid_dependency_wait();  // before the first global write / residual read
    constexpr bool kQuant = OUT == SLQ_OUT_U8 || OUT == SLQ_OUT_S8;
    constexpr int CW = W16 ? 16 : 32;              // accumulator columns per TMEM load
    const int team = (warp - 4) >> 3;              // tile i -> team i & 1
    const int half = ((warp - 4) >> 2) & 1;        // which half of the tile's channel units
    const int wq = warp & 3;                       // TMEM lane quarter this warp may touch
    const int et = threadIdx.x - 128 - team * kTeam;  // 0..255 inside the team (warps 4..19)
    const int row = wq * 32 + lane;                // tile row == TMEM lane
    // per-channel constants of the team's current n-tile, structure-of-arrays: A[128] | Z[128] | B[128] floats.
    // A warp-wide broadcast LDS.128 costs the LSU four wavefronts whatever it delivers (measured: the LSU
    // data pipe was the busiest unit of the epilogue with one {A,Z,B,pad} load per output), so one load
    // fetches the same constant of FOUR channels: 3 wavefronts per channel instead of 4, 0.75 loads per output.
    float *prm = reinterpret_cast<float *>(smem + sp.prm_off) + team * 768;
    volatile uint32_t *rs_base = reinterpret_cast<volatile uint32_t *>(smem + sp.prm_off + 2 * 3072) + team * 256;
    const uint32_t prm_s = smem_base + sp.prm_off + team * 3072;
    const bool shared_stg = sp.out_bufs == 1;  // both teams stage through one tile (stfree hand-off below)
    const bool dbl_stg = sp.out_bufs == 4;     // two tiles per team, alternating: no wait for the store at the loop top
    const uint32_t stg_base = smem_base + sp.out_off + (shared_stg ? 0 : team * (dbl_stg ? 2 : 1)) * sp.out_tile;
    float s_in = 1.f, s_res = 0.f, inv_out = 1.f;
    if (OUT != SLQ_OUT_ACC) {
      s_in = e.act_scales[e.in_id];
      if (kQuant) inv_out = __fdiv_rn(1.0f, e.act_scales[e.out_id]);
      if (has_res) s_res = kQuant ? __fmul_rn(e.act_scales[e.res_id], inv_out) : e.act_scales[e.res_id];
    }
    const bool res_signed = RES == kResDyn ? (e.res_signed != 0) : (RES == kResS8);
    // this thread's row inside a staging / residual tile (rows of bn_ch bytes, TMA swizzle of that width)
    const uint32_t row_byte = (uint32_t)(row * g.bn_ch);
    const uint32_t row_sw = g.bn_ch == 128 ? (uint32_t)(row & 7) : (uint32_t)((row >> 1) & 3);
    const int units = g.bn_ch / CW;
    const int u0 = half * (units >> 1), u1 = u0 + (units >> 1);
    int last_n_tile = -1;
    int tn = 0;
    long long wepi = 0;
    const long long tstart_clk = clock64();
    // S[m] = sum over the conv window of the per-pixel channel sums the producing kernel accumulated
    // (slq_epilogue.in_rowsum).  1x1 stride-1 layers -- all the epilogue-bound ones -- read one value at index m;
    // the others split m into (image, row, column) with a float reciprocal (M < 2^24: exact after one fix-up).
    const bool same_grid = g.kh == 1 && g.stride == 1;
    const float inv_hw = __frcp_rn((float)(g.Ho * g.Wo)), inv_wo = __frcp_rn((float)g.Wo);
    auto window_sum = [&](int mm) -> uint32_t {
      if (mm >= g.M) return 0u;
      if (same_grid) {
        uint32_t sum = 0;
        for (int pl = 0; pl < e.in_planes; ++pl) sum += __ldg(e.in_rowsum + (long long)pl * e.in_plane_stride + mm);
        return sum;
      }
      const int hw = g.Ho * g.Wo;
      int n_img, rem, ho, wo;
      if (g.M < (1 << 24)) {  // every index is an exact float: the reciprocal quotient is off by at most one
        n_img = (int)((float)mm * inv_hw);
        rem = mm - n_img * hw;
        if (rem < 0) { --n_img; rem += hw; } else if (rem >= hw) { ++n_img; rem -= hw; }
        ho = (int)((float)rem * inv_wo);
        wo = rem - ho * g.Wo;
        if (wo < 0) { --ho; wo += g.Wo; } else if (wo >= g.Wo) { ++ho; wo -= g.Wo; }
      } else {
        n_img = mm / hw; rem = mm - n_img * hw;
        ho = rem / g.Wo; wo = rem - ho * g.Wo;
      }
      uint32_t sum = 0;
      for (int pl = 0; pl < e.in_planes; ++pl) {
        const uint32_t *rs = e.in_rowsum + (long long)pl * e.in_plane_stride + (long long)n_img * g.H * g.W;
        if (g.kh == 1) { sum += __ldg(rs + (ho * g.stride) * g.W + wo * g.stride); continue; }
        const int h0 = ho * g.stride - g.pad, w0 = wo * g.stride - g.pad;
#pragma unroll
        for (int r = 0; r < 3; ++r) {
          const int hi = h0 + r;
          if (hi < 0 || hi >= g.H) continue;
#pragma unroll
          for (int q = 0; q < 3; ++q) {
            const int wi = w0 + q;
            if (wi >= 0 && wi < g.W) sum += __ldg(rs + hi * g.W + wi);
          }
        }
      }
      return sum;
    };
    if (a.wgp != nullptr && sp.b_resident && walk.count > 0) {
      // ---- packed weights -> u8 operand tiles, in shared memory (all 16 epilogue warps, once per CTA) ----
      // Row r of a K block arrives as SWZ/2 bytes (<= 4 bit: two codes per byte, low nibble first) or SWZ bytes
      // (8 / 6 bit) at offset rowoff[r] of the block's segment, which sits at the END of the block's tile.  A
      // thread owns (row, 16-byte output chunk) pairs: every source of a tile is read into registers, the
      // warps meet at a barrier, then every chunk is written to its swizzled place -- reads and writes of the
      // same tile never overlap in time, so the expansion is in place.
      const int tid = threadIdx.x - 128;  // 0 .. 511
      constexpr int kChunks = SWZ / 16;
      const int n_chunks = bn_cols * kChunks;  // per K block: <= 2048
      const uint32_t seg = (uint32_t)a.wgp_seg[walk.my_n];
      const uint16_t *rowoff = a.wgp_rowoff + (long long)walk.my_n * (bn_cols + 1);
      // this thread's (row, chunk) items: idx = tid + 512 * j
      uint32_t src_off[4], src_len[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int idx = tid + 512 * j;
        src_off[j] = 0; src_len[j] = 0;
        if (idx < n_chunks) {
          const int r = idx / kChunks, c = idx % kChunks;
          const uint32_t o0 = rowoff[r], o1 = rowoff[r + 1];
          const bool half = (o1 - o0) == (uint32_t)(SWZ / 2);  // a 4-bit row
          src_len[j] = half ? 8u : 16u;
          src_off[j] = o0 + (uint32_t)c * src_len[j];
        }
      }
      mbar_wait(bfull_bar, 0);
      for (int kb = 0; kb < a.num_kb; ++kb) {
        const uint32_t tile_s = smem_base + sp.b_off + kb * sp.b_tile_bytes;
        const uint32_t raw_s = tile_s + (uint32_t)(bn_cols * SWZ) - seg;  // behind it: the ones group
        uint4 v[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (src_len[j] == 16u) v[j] = lds128(raw_s + src_off[j]);
          else if (src_len[j] == 8u) {
            uint2 w;
            asm volatile("ld.shared.v2.u32 {%0, %1}, [%2];" : "=r"(w.x), "=r"(w.y) : "r"(raw_s + src_off[j]));
            // 16 nibbles -> 16 bytes: byte 2i = low nibble of byte i, byte 2i+1 = its high nibble
            const uint32_t l0 = w.x & 0x0f0f0f0fu, h0 = (w.x >> 4) & 0x0f0f0f0fu;
            const uint32_t l1 = w.y & 0x0f0f0f0fu, h1 = (w.y >> 4) & 0x0f0f0f0fu;
            v[j] = make_uint4(__byte_perm(l0, h0, 0x5140), __byte_perm(l0, h0, 0x7362), __byte_perm(l1, h1, 0x5140),
                              __byte_perm(l1, h1, 0x7362));
          }
        }
        named_bar_sync(3, 2 * kTeam);  // every source of this tile is in registers
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int idx = tid + 512 * j;
          if (src_len[j] != 0u) {
            const int r = idx / kChunks, c = idx % kChunks;
            const uint32_t sw = SWZ == 128 ? (uint32_t)(c ^ (r & 7)) : (uint32_t)(c ^ ((r >> 1) & 3));
            sts128(tile_s + (uint32_t)r * SWZ + (sw << 4), v[j]);
          }
        }
      }
      fence_proxy_async_smem();  // generic-proxy writes -> visible to the tensor core (async proxy)
      mbar_arrive(bready_bar);
    }
    // debug build, statistics mode: where one epilogue warp (warp 4 of CTA 0) spends a tile -- cycle sums per segment
    const bool seg_on = kDebugTrace && a.trace != nullptr && a.trace_cap < 0 && blockIdx.x == 0 && warp == 4;
    long long seg_t = 0, seg_sum[6] = {0, 0, 0, 0, 0, 0};
    auto seg = [&](int k) {
      if (seg_on) { const long long t = clock64(); seg_sum[k] += t - seg_t; seg_t = t; }
    };
    if (seg_on) seg_t = clock64();
    uint32_t S_next = 0;
    if (!ones_row && team < walk.count) {
      int mt0, nt0;
      walk.at(team, mt0, nt0);
      S_next = window_sum(mt0 * kTileM + row);
    }
    for (int it = team; it < walk.count; it += 2) {
      int m_tile, n_tile;
      walk.at(it, m_tile, n_tile);
      const int acc = it % a.acc_bufs, tb = it % kTileBars;
      const uint32_t ph = (uint32_t)((it / kTileBars) & 1);
      const uint32_t stg = stg_base + (dbl_stg ? (uint32_t)((it >> 1) & 1) * sp.out_tile : 0u);
      volatile uint32_t *rs_scratch = rs_base + ((it >> 1) & 1) * 128;
      if ((!dbl_stg && (kWide || a.tma_out)) || (n_tile != last_n_tile && OUT != SLQ_OUT_ACC)) {
        // staging tile free again? (the previous TMA store of this team has read it)  With two staging tiles per
        // team nothing is waited for here; the barrier is then only needed before the constants are rewritten
        if (!kWide && a.tma_out && et == 0 && !dbl_stg) tma_store_wait_read();
        named_bar_sync(1 + team, kTeam);
      }
      if (n_tile != last_n_tile && OUT != SLQ_OUT_ACC) {
        if (et < g.bn_ch) {
          const int oc = n_tile * g.bn_ch + et;
          ChanParam p = {0.f, 0.f, 0.f, 0.f};
          if (oc < g.Cout) p = make_chan_param(e.wscale[oc], e.zf[oc], e.bias[oc], s_in, inv_out, kQuant);
          prm[et] = p.wsc; prm[256 + et] = p.zw; prm[512 + et] = p.bias;
        }
        last_n_tile = n_tile;
        named_bar_sync(1 + team, kTeam);
      }
      // window sum of the INPUT activation for this thread's output pixel: gathered one tile AHEAD (the loads
      // of tile it + 2 are in flight while tile it is converted), so their latency is never exposed
      const long long m = (long long)m_tile * kTileM + row;
      const bool valid = m < g.M;
      uint32_t S_raw = S_next;
      if (!ones_row && it + 2 < walk.count) {
        int mt2, nt2;
        walk.at(it + 2, mt2, nt2);
        S_next = window_sum(mt2 * kTileM + row);
      }
      seg(0);  // loop top: staging / constants barriers, window-sum gather
      mbar_wait_stat(tfull_bar(tb), ph, wepi, kDebugTrace && a.trace != nullptr && a.trace_cap < 0 && blockIdx.x == 0);
      tc_fence_after();
      seg(1);  // accumulator ready
      if (kDebugTrace && a.trace != nullptr && et == 0) trace_ev(a, 17 + team, tn, 5, (int)it);
      const int rbuf = has_res ? (int)(it % sp.res_bufs) : 0;
      const uint32_t rsb = smem_base + sp.res_off + rbuf * sp.out_tile;
      if (has_res) mbar_wait(rfull_bar(rbuf), (uint32_t)((it / sp.res_bufs) & 1));
      const uint32_t trow = tmem_base + ((uint32_t)(wq * 32) << 16) + acc * a.acc_stride;
      if (ones_row) {
        S_raw = tmem_ld1(trow + bn_cols);
        tmem_ld_wait();
      }
      seg(2);  // residual tile landed, window sum read from TMEM
      const float Sf = (float)S_raw;  // <= 9 * 2048 * 255 < 2^24: exact
      uint32_t rsum = 0;              // channel sum of this thread's u8 outputs of the tile
      const bool want_rs_any = e.out_rowsum != nullptr;
      if (OUT == SLQ_OUT_ACC && e.out_S && valid && n_tile == 0 && half == 0) e.out_S[m] = (int)S_raw;
      for (int u = u0; u < u1; ++u) {
        uint32_t lo[CW], hi[CW];
        tmem_ld<CW>(trow + u * CW, lo);
        if constexpr (W16) tmem_ld<CW>(trow + 64 + u * CW, hi);
        uint32_t rw[CW / 4];
        if (has_res) {
#pragma unroll
          for (int i = 0; i < CW / 16; ++i) {
            const uint4 r = lds128(rsb + row_byte + ((((uint32_t)(u * (CW / 16) + i)) ^ row_sw) << 4));
            rw[4 * i] = r.x; rw[4 * i + 1] = r.y; rw[4 * i + 2] = r.z; rw[4 * i + 3] = r.w;
          }
        }
        tmem_ld_wait();
        const int cb = n_tile * g.bn_ch + u * CW;  // first output channel of this unit
        if (OUT == SLQ_OUT_ACC) {
          if (!valid || cb >= g.Cout) continue;
          const long long ld = (long long)(W16 ? 2 : 1) * g.Cout;
          int4 *o = reinterpret_cast<int4 *>(reinterpret_cast<int32_t *>(e.out) + m * ld + cb);
#pragma unroll
          for (int j = 0; j < CW / 4; ++j) o[j] = make_int4(lo[4 * j], lo[4 * j + 1], lo[4 * j + 2], lo[4 * j + 3]);
          if (W16) {
            int4 *oh = reinterpret_cast<int4 *>(reinterpret_cast<int32_t *>(e.out) + m * ld + g.Cout + cb);
#pragma unroll
            for (int j = 0; j < CW / 4; ++j) oh[j] = make_int4(hi[4 * j], hi[4 * j + 1], hi[4 * j + 2], hi[4 * j + 3]);
          }
          continue;
        }
        const bool store_ok = valid && cb < g.Cout;
        float4 *of = reinterpret_cast<float4 *>(reinterpret_cast<float *>(e.out) + m * g.Cout + cb);
        uint32_t pk[CW / 4];
        const float2 S2 = make_float2(Sf, Sf), R2 = make_float2(s_res, s_res);
#pragma unroll
        for (int q4 = 0; q4 < CW / 4; ++q4) {
          float v[4];
          const uint32_t pofs = prm_s + (uint32_t)(u * CW + 4 * q4) * 4;  // warp-wide broadcast loads
          const uint4 pa = lds128(pofs), pz = lds128(pofs + 1024), pb = lds128(pofs + 2048);
          const uint32_t pav[4] = {pa.x, pa.y, pa.z, pa.w}, pzv[4] = {pz.x, pz.y, pz.z, pz.w}, pbv[4] = {pb.x, pb.y, pb.z, pb.w};
          // two channels per FFMA2 (packed fp32 pairs): the arithmetic of epi_value / epi_add_res, component-wise
#pragma unroll
          for (int b = 0; b < 4; b += 2) {
            const int j = 4 * q4 + b;
            float2 accf = make_float2((float)(int)lo[j], (float)(int)lo[j + 1]);
            if (W16) accf = ffma2(make_float2((float)(int)hi[j], (float)(int)hi[j + 1]), make_float2(256.0f, 256.0f), accf);
            const float2 c2 = ffma2(S2, make_float2(__uint_as_float(pzv[b]), __uint_as_float(pzv[b + 1])),
                                    make_float2(__uint_as_float(pbv[b]), __uint_as_float(pbv[b + 1])));
            float2 y = ffma2(accf, make_float2(__uint_as_float(pav[b]), __uint_as_float(pav[b + 1])), c2);
            if (has_res) {
              y = ffma2(res_pair(rw[q4], b, res_signed), R2, y);
            }
            v[b] = y.x; v[b + 1] = y.y;
          }
          if (!kQuant) {
            if (e.relu) {
#pragma unroll
              for (int b = 0; b < 4; ++b) v[b] = fmaxf(v[b], 0.f);
            }
            if (store_ok) of[q4] = make_float4(v[0], v[1], v[2], v[3]);
          } else {
            pk[q4] = epi_pack4<OUT == SLQ_OUT_S8>(v[0], v[1], v[2], v[3]);
            // (the channel sums of the outputs, below, only where a consumer gathers them)
          }
        }
        if (OUT == SLQ_OUT_U8 && want_rs_any) {  // one uniform branch around the unit's dot products: layers whose
#pragma unroll                                  // outputs nobody gathers (every expansion of stages 1-2) skip them
          for (int q4 = 0; q4 < CW / 4; ++q4) rsum = __dp4a(pk[q4], 0x01010101u, rsum);
        }
        if (kQuant) {
          if (!kWide && a.tma_out) {
            // shared staging tile: the other team's store of the previous tile must have read it
            if (shared_stg && u == u0 && it >= 1) mbar_wait(stfree_bar(team ^ 1), (uint32_t)(((it - 1) >> 1) & 1));
#pragma unroll
            for (int i = 0; i < CW / 16; ++i)
              sts128(stg + row_byte + ((((uint32_t)(u * (CW / 16) + i)) ^ row_sw) << 4),
                     make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]));
          } else if (store_ok) {
            // 256-channel tiles: no staging tile (the smem goes to the {A, B} ring); a thread owns 128 contiguous
            // bytes of its pixel, written as 16-byte stores that complete whole lines over the unit loop
            uint4 *o = reinterpret_cast<uint4 *>(reinterpret_cast<uint8_t *>(e.out) + m * g.Cout + cb);
#pragma unroll
            for (int i = 0; i < CW / 16; ++i) o[i] = make_uint4(pk[4 * i], pk[4 * i + 1], pk[4 * i + 2], pk[4 * i + 3]);
          }
        }
      }
      seg(3);  // the unit loop: TMEM loads, arithmetic, staging stores
      const bool want_rs = OUT == SLQ_OUT_U8 && e.out_rowsum != nullptr;
      if (want_rs && half == 1) rs_scratch[row] = rsum;  // the other half of the tile's channels adds it below
      tc_fence_before();
      if (kDebugTrace && a.trace != nullptr && et == 0) trace_ev(a, 17 + team, tn, 6, (int)it);
      // ONE arrival per warp instead of one per thread (256 shared-memory atomics on the barrier's word per tile
      // and barrier; measured: no difference in time, kept for the lower LSU traffic)
      __syncwarp();
      if (lane == 0) {
        mbar_arrive(tempty_bar(tb));  // kTeam / 32 arrivals release the accumulator buffer
        if (has_res) mbar_arrive(rempty_bar(rbuf));
      }
      if (kWide || !a.tma_out) {
        if (want_rs) named_bar_sync(1 + team, kTeam);  // the scratch row sums are visible
      } else {
        fence_proxy_async_smem();  // generic-proxy smem writes -> visible to the TMA (async proxy)
        // two staging tiles: the store issued one tile ago (it read the OTHER tile, which the team fills next) has
        // long finished reading; making sure of it before the barrier costs nothing and keeps the hand-off exact
        if (dbl_stg && et == 0) tma_store_wait_read();
        named_bar_sync(1 + team, kTeam);
        if (et == 0) {
          tma_store_2d(&tmO, stg, n_tile * g.bn_ch, (int)(m_tile * kTileM));  // rows >= M are clipped
          tma_store_commit();
          if (shared_stg) {  // hand the tile to the other team as soon as the TMA engine has read it
            tma_store_wait_read();
            mbar_arrive(stfree_bar(team));
          }
        }
      }
      seg(4);  // hand-offs: accumulator / residual release, proxy fence, team barrier, TMA store issue
      // per-pixel channel sum of this tile's u8 outputs -> side tensor of the output activation.  LAST in the
      // iteration: a fire-and-forget reduction issued before the proxy fence / barrier above would have its
      // round trip to L2 waited for there, once per tile
      if (OUT == SLQ_OUT_U8 && e.out_rowsum != nullptr && half == 0 && valid)
        e.out_rowsum[(long long)n_tile * g.M + m] = rsum + rs_scratch[row];  // plane n_tile: the whole tile's channels
      seg(5);
    }
    if (seg_on && lane == 0) {
      for (int k = 0; k < 6; ++k) a.trace[56 + k] = seg_sum[k];
      a.trace[62] = (walk.count + 1 - team) / 2;
    }
    if (!kWide && a.tma_out && et == 0) tma_store_wait_all();
    if (kDebugTrace && a.trace != nullptr && a.trace_cap < 0 && blockIdx.x == 0 && et == 0) { a.trace[6 + team] = wepi; a.trace[12 + team] = clock64() - tstart_clk; }
  }

  // ---- teardown -----------------------------------------------------------------------------
  tc_fence_before();
  __syncthreads();
  if (kDebugTrace && a.trace != nullptr && a.trace_cap < 0 && threadIdx.x == 0) {
    if (blockIdx.x == 0) a.trace[15] = clock64() - t_entry;
    if (blockIdx.x < 32) a.trace[16 + blockIdx.x] = clock64() - t_entry;  // lifetime of the first CTAs
    if (blockIdx.x >= gridDim.x - 8) a.trace[48 + blockIdx.x - (gridDim.x - 8)] = clock64() - t_entry;
  }
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------------------------------
// host side: tensor maps + launch
// ------------------------------------------------------------------------------------------
// [M, Cout] u8 tensor (output or residual) as a tiled map with box = bn_ch channels x 128 pixels
static int encode_out_map(CUtensorMap *tm, const void *ptr, const ConvGeom &g, const char *what) {
  return encode_tiled_u8(tm, ptr, g.M, g.Cout, g.bn_ch, kTileM,
                         g.bn_ch == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, what);
}

static int build_tensor_maps(slq_conv *c) {
  const ConvGeom &g = c->g;
  const int swz = c->swizzle;
  const CUtensorMapSwizzle sw = swz == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
  for (int wide = 0; wide <= (c->wide_ok ? 1 : 0); ++wide) {
    // B: GEMM-ready weights [gemm_rows, Ktot] u8, box = SWZ bytes of K x bn_cols rows (one map per tiling)
    const ConvGeom &gb = wide ? c->g_wide : c->g;
    const int rc = encode_tiled_u8(wide ? &c->tmB_wide : &c->tmB, c->wg, gb.gemm_rows, gb.Ktot, swz, gb.bn_cols, sw, "B");
    if (rc != SLQ_OK) return rc;
  }
  if (!c->a_im2col)  // A: [M, Cin] u8 (1x1 stride-1), box = SWZ channels x 128 pixels
    return encode_tiled_u8(&c->tmA, c->in, g.M, g.Cin, swz, kTileM, sw, "A");
  // A: NHWC u8 through im2col mode; base pixel = top-left tap of each output pixel
  const int lower[2] = {-g.pad, -g.pad};                          // {W, H}
  const int upper[2] = {g.pad - (g.kw - 1), g.pad - (g.kh - 1)};  // {W, H}
  return encode_im2col_u8(&c->tmA, c->in, g.N, g.H, g.W, g.Cin, lower, upper, g.stride, swz, kTileM, sw, "A");
}

static long long *g_trace = nullptr;  // slq_debug_set_trace
static int g_trace_cap = 0;
void debug_trace_buffer(long long **buf, int *cap) { *buf = g_trace; *cap = g_trace_cap; }

template <int SWZ, bool W16, int OUT, int RES>
static int launch_one(slq_conv *c, const EpiDev &e, int tma_out, cudaStream_t st) {
  constexpr auto kernel = conv_umma_kernel<SWZ, W16, OUT, RES>;
  SLQ_CUDA(set_smem_limit_once<kernel>(kSmemLimit));
  // K-heavy layers (weights streamed) without residual run 256-channel tiles
  const bool wide = c->wide_ok && e.res == nullptr && !W16;
  const ConvGeom &geom = wide ? c->g_wide : c->g;
  KernelArgs a;
  a.g = geom;
  a.e = e;
  a.sp = make_plan(geom, SWZ, e.res != nullptr);
  a.acc_bufs = wide ? 2 : 3;
  a.acc_stride = wide ? 256 : 160;
  const bool packed = c->wgp != nullptr && a.sp.b_resident && !W16 && !wide;
  a.wgp = packed ? c->wgp : nullptr;
  a.wgp_tile = c->wgp_tile; a.wgp_seg = c->wgp_seg; a.wgp_rowoff = c->wgp_rowoff;
  if (wide) tma_out = 0;  // straight from registers (no staging tile: the smem goes to the operand ring)
  // (measured, tools/gpu_r2_call24.sh: storing the resident-weight layers' outputs from registers as well -- no staging
  // tile, no team barrier, no TMA store -- costs 159 us against 128 on 64->256 @56^2 and 82 against 70 on 128->512
  // @28^2: half-filled 32-byte sectors from 32 lanes at a Cout-byte pitch; equal within 5 % on the small layers)
  const int grid = plan_grid(geom, a.sp, sm_count());
  a.trace = g_trace;
  a.trace_cap = g_trace_cap;
  a.half_b = 0;
#if SLQ_DEBUG_TRACE
  a.half_b = getenv("SLQ_HALF_B") != nullptr;
#endif
  a.a_im2col = c->a_im2col;
  a.chunks_per_tap = geom.Cin / SWZ;
  a.num_kb = geom.kh * geom.kw * a.chunks_per_tap;
  a.num_grp = a.num_kb / a.sp.group;
  a.tile_alt = (a.sp.mma_warps == 2 && a.num_grp >= 2 && a.sp.stages % (2 * a.num_grp) == 0) ? 1 : 0;
  a.mma_warps_per_tile = (a.sp.mma_warps == 2 && a.num_grp >= 2 && !a.tile_alt) ? 2 : 1;
  a.m_tiles = ceil_div(geom.M, kTileM);
  a.tma_out = tma_out;
  SLQ_CUDA(launch_pdl(kernel, grid, kThreads, a.sp.total, st, c->tmA, wide ? c->tmB_wide : c->tmB, c->tmO, c->tmR, a));
  return SLQ_OK;
}

// picks the compiled (output kind, residual kind) variant
template <int SWZ, bool W16>
static int launch_umma(slq_conv *c, const EpiDev &e, int tma_out, cudaStream_t st) {
  const int res = e.res == nullptr ? kResNone : (e.res_signed ? kResS8 : kResU8);
  if constexpr (SWZ == 128 && !W16) {
    if (c->wide_ok && res == kResNone) {  // K-heavy layer: 256-channel tiles, quantised outputs straight from registers
      if (e.out_mode == SLQ_OUT_U8) return launch_one<SWZ, W16, SLQ_OUT_U8, kResWide>(c, e, 0, st);
      if (e.out_mode == SLQ_OUT_S8) return launch_one<SWZ, W16, SLQ_OUT_S8, kResWide>(c, e, 0, st);
    }
  }
  switch (e.out_mode) {
    case SLQ_OUT_U8:
      if (res == kResNone) return launch_one<SWZ, W16, SLQ_OUT_U8, kResNone>(c, e, tma_out, st);
      if (res == kResU8) return launch_one<SWZ, W16, SLQ_OUT_U8, kResU8>(c, e, tma_out, st);
      return launch_one<SWZ, W16, SLQ_OUT_U8, kResS8>(c, e, tma_out, st);
    case SLQ_OUT_S8:
      if (res == kResNone) return launch_one<SWZ, W16, SLQ_OUT_S8, kResNone>(c, e, tma_out, st);
      if (res == kResU8) return launch_one<SWZ, W16, SLQ_OUT_S8, kResU8>(c, e, tma_out, st);
      return launch_one<SWZ, W16, SLQ_OUT_S8, kResS8>(c, e, tma_out, st);
    case SLQ_OUT_F32:
      return launch_one<SWZ, W16, SLQ_OUT_F32, kResDyn>(c, e, tma_out, st);
    default:
      return launch_one<SWZ, W16, SLQ_OUT_ACC, kResNone>(c, e, tma_out, st);
  }
}

}  // namespace slq

using namespace slq;

extern "C" int slq_conv_create(const slq_conv_desc *d, const uint8_t *in, const uint8_t *wg, slq_conv **out) {
  int rc = validate_desc(d);
  if (rc != SLQ_OK) return rc;
  SLQ_CHECK_ARG(in && wg && out, "slq_conv_create: null pointer argument");
  SLQ_CHECK_ARG(d->impl == SLQ_IMPL_UMMA || d->impl == SLQ_IMPL_SIMT, "slq_conv_create: impl %d", d->impl);
  SLQ_CHECK_ARG(reinterpret_cast<uintptr_t>(in) % 16 == 0 && reinterpret_cast<uintptr_t>(wg) % 16 == 0,
                "slq_conv_create: buffers must be 16-byte aligned");
  slq_conv *c = new (std::nothrow) slq_conv();
  SLQ_CHECK_ARG(c != nullptr, "slq_conv_create: out of host memory");
  c->desc = *d;
  c->g = make_geom(*d);
  if (c->g.M > 0x7fff0000LL) {
    delete c;
    set_error("slq_conv_create: more than 2^31 output pixels");
    return SLQ_ERR_UNSUPPORTED;
  }
  c->in = in;
  c->wg = wg;
  c->swizzle = (d->Cin % 128 == 0) ? 128 : 64;
  c->g_wide = make_geom(*d, 1);
  // wide tiles only where the 128-channel tiling has to stream its weights anyway (K-heavy layers)
  c->wide_ok = (d->impl == SLQ_IMPL_UMMA && c->g_wide.bn_ch == 256 && c->swizzle == 128 &&
                !make_plan(c->g, c->swizzle, false).b_resident) ? 1 : 0;
#if SLQ_DEBUG_TRACE
  if (getenv("SLQ_NO_WIDE")) c->wide_ok = 0;  // A/B timing against the 128-channel tiling (debug build only)
#endif
  c->out_ptr = nullptr;
  c->res_ptr = nullptr;
  c->wgp = nullptr; c->wgp_tile = nullptr; c->wgp_seg = nullptr; c->wgp_rowoff = nullptr;
  const bool can_tile = d->kh == 1 && d->kw == 1 && d->stride == 1 && d->pad == 0;
  if (d->a_mode == SLQ_A_TILED && !can_tile) {
    delete c;
    set_error("slq_conv_create: SLQ_A_TILED needs a 1x1 stride-1 layer");
    return SLQ_ERR_INVALID;
  }
  c->a_im2col = (d->a_mode == SLQ_A_IM2COL) ? 1 : (d->a_mode == SLQ_A_TILED ? 0 : (can_tile ? 0 : 1));
  if (d->impl == SLQ_IMPL_UMMA) {
    if (d->Cout % 64 != 0) {
      delete c;
      set_error("slq_conv_create: the tcgen05 path needs Cout %% 64 == 0 (got %d)", d->Cout);
      return SLQ_ERR_UNSUPPORTED;
    }
    rc = build_tensor_maps(c);
    if (rc != SLQ_OK) {
      delete c;
      return rc;
    }
    c->tmO = c->tmB;  // placeholders until the first launch names the output / residual buffers
    c->tmR = c->tmB;
    const long long tiles = ceil_div(c->g.M, kTileM) * c->g.n_tiles;
    c->num_ctas = (int)std::min<long long>(tiles, sm_count());
    c->smem_bytes = make_plan(c->g, c->swizzle, true).total;
  }
  *out = c;
  return SLQ_OK;
}

extern "C" void slq_conv_destroy(slq_conv *c) { delete c; }

extern "C" int slq_debug_set_trace(int64_t *buf, int32_t capacity_events) {
  if (!kDebugTrace && buf != nullptr) {
    set_error("slq_debug_set_trace: this library was built without SLQ_DEBUG_TRACE (python slq_build.py --debug)");
    return SLQ_ERR_UNSUPPORTED;
  }
  g_trace = reinterpret_cast<long long *>(buf);
  g_trace_cap = buf ? capacity_events : 0;
  return SLQ_OK;
}

extern "C" int slq_conv_launch(slq_conv *c, const slq_epilogue *ep, void *stream) {
  SLQ_CHECK_ARG(c && ep, "slq_conv_launch: null handle/epilogue");
  SLQ_CHECK_ARG(ep->out != nullptr, "slq_conv_launch: out is NULL");
  SLQ_CHECK_ARG(ep->out_mode >= SLQ_OUT_U8 && ep->out_mode <= SLQ_OUT_S8, "slq_conv_launch: out_mode %d", ep->out_mode);
  if (ep->out_mode != SLQ_OUT_ACC) {
    SLQ_CHECK_ARG(ep->wscale && ep->zf && ep->bias && ep->act_scales, "slq_conv_launch: epilogue vectors missing");
    SLQ_CHECK_ARG(!ep->res || ep->res_id >= 0, "slq_conv_launch: residual without res_id");
  }
  SLQ_CHECK_ARG(reinterpret_cast<uintptr_t>(ep->out) % 16 == 0 &&
                    (!ep->res || reinterpret_cast<uintptr_t>(ep->res) % 16 == 0),
                "slq_conv_launch: out/res must be 16-byte aligned");
  EpiDev e;
  e.wscale = ep->wscale; e.zf = ep->zf; e.bias = ep->bias; e.act_scales = ep->act_scales;
  e.in_rowsum = ep->in_rowsum; e.out_rowsum = ep->out_rowsum;
  e.in_planes = ep->in_planes; e.in_plane_stride = ep->in_plane_stride;
  e.res = ep->out_mode == SLQ_OUT_ACC ? nullptr : ep->res;
  e.out = ep->out; e.out_S = ep->out_S;
  e.in_id = ep->in_id; e.out_id = ep->out_id; e.res_id = ep->res_id;
  e.out_mode = ep->out_mode; e.relu = ep->relu; e.res_signed = ep->res_signed;
  e.Cout = c->g.Cout; e.w16 = c->g.w16; e.M = c->g.M;
  cudaStream_t st = (cudaStream_t)stream;
  if (c->desc.impl == SLQ_IMPL_SIMT) return launch_conv_simt(c->g, c->in, c->wg, e, st);
  const bool wide_launch = c->wide_ok && ep->res == nullptr && !c->g.w16;
  SLQ_CHECK_ARG(!wide_launch || (ep->in_rowsum != nullptr && ep->in_planes >= 1 &&
                                 ep->in_plane_stride >= (int64_t)c->g.N * c->g.H * c->g.W),
                "slq_conv_launch: this layer runs 256-channel tiles and needs in_rowsum (per-pixel channel sums of its "
                "input: planes, plane stride; slq_conv_needs_rowsum)");
  const int tma_out = (ep->out_mode == SLQ_OUT_U8 || ep->out_mode == SLQ_OUT_S8) ? 1 : 0;
  if (tma_out && c->out_ptr != ep->out) {  // (re)encode the store map for this output buffer
    int rc = encode_out_map(&c->tmO, ep->out, c->g, "out");
    if (rc != SLQ_OK) return rc;
    c->out_ptr = ep->out;
  }
  if (e.res && c->res_ptr != e.res) {
    int rc = encode_out_map(&c->tmR, e.res, c->g, "residual");
    if (rc != SLQ_OK) return rc;
    c->res_ptr = e.res;
  }
  if (c->swizzle == 128)
    return c->g.w16 ? launch_umma<128, true>(c, e, tma_out, st) : launch_umma<128, false>(c, e, tma_out, st);
  return c->g.w16 ? launch_umma<64, true>(c, e, tma_out, st) : launch_umma<64, false>(c, e, tma_out, st);
}

extern "C" int slq_conv_tiling(const slq_conv_desc *d, int32_t *bn_cols, int32_t *n_tiles, int32_t *k_block,
                               int32_t *num_kb, int32_t *resident) {
  int rc = validate_desc(d);
  if (rc != SLQ_OK) return rc;
  const ConvGeom g = make_geom(*d);
  const int swz = (d->Cin % 128 == 0) ? 128 : 64;
  if (bn_cols) *bn_cols = g.bn_cols;
  if (n_tiles) *n_tiles = g.n_tiles;
  if (k_block) *k_block = swz;
  if (num_kb) *num_kb = g.Ktot / swz;
  // resident with AND without a residual tile ring (the caller does not know the epilogue yet)
  if (resident) *resident = (make_plan(g, swz, true).b_resident && make_plan(g, swz, false).b_resident && !g.w16) ? 1 : 0;
  return SLQ_OK;
}

extern "C" int slq_conv_set_packed_weights(slq_conv *c, const uint8_t *wgp, const int64_t *tile_base,
                                           const int32_t *seg_bytes, const uint16_t *row_offsets) {
  SLQ_CHECK_ARG(c != nullptr, "slq_conv_set_packed_weights: null handle");
  SLQ_CHECK_ARG(wgp == nullptr || (tile_base && seg_bytes && row_offsets), "slq_conv_set_packed_weights: layout tables missing");
  SLQ_CHECK_ARG(reinterpret_cast<uintptr_t>(wgp) % 16 == 0, "slq_conv_set_packed_weights: wgp must be 16-byte aligned");
  c->wgp = wgp;
  c->wgp_tile = reinterpret_cast<const long long *>(tile_base);
  c->wgp_seg = seg_bytes;
  c->wgp_rowoff = row_offsets;
  return SLQ_OK;
}

extern "C" int32_t slq_conv_needs_rowsum(const slq_conv *c, int32_t has_residual) {
  if (!c || c->desc.impl != SLQ_IMPL_UMMA) return 0;
  return (c->wide_ok && !has_residual && !c->g.w16) ? 1 : 0;
}

extern "C" int32_t slq_conv_rowsum_planes(const slq_conv *c, int32_t has_residual) {
  if (!c) return -1;
  if (c->desc.impl != SLQ_IMPL_UMMA) return 0;  // the SIMT checker computes its own window sums and writes none
  return (c->wide_ok && !has_residual && !c->g.w16) ? c->g_wide.n_tiles : c->g.n_tiles;
}
