// csrc/calib.cu -- histogram calibration of the static activation scales (include/slq.h section 3):
//   * act_histogram_kernel: |y| of one fp32 layer output into a uint64 histogram (HBM-bound)
//   * hist_scales_kernel:   one CTA per tensor, histogram -> percentile or MSE threshold -> scale (fp64)
//   * hist_entropy_kernel:  one CTA per tensor, histogram -> entropy (KL-divergence) threshold -> scale (fp64)
// The binning rule is exact fp32 and the counts are integers, so the result is deterministic and
// tests/calib_oracle.py (act_histogram, hist_scale) restates it bit for bit; tests/calib_entropy_oracle.py restates
// the entropy rule.
#include <math_constants.h>

#include <algorithm>

#include "common.cuh"

namespace slq {

constexpr int kHistThreads = 256;
constexpr int kHistCopies = 4;        // privatised sub-histograms per CTA (two warps share one)
constexpr int kHistMaxBins = 2048;    // (bins + 1) * 4 B * kHistCopies = 32 KB of shared memory at most

// counter of one element: 0 for an exact zero (either sign), else 1 + min(trunc(|v| * inv), bins - 1)
__device__ __forceinline__ int hist_counter(float v, float inv, int bins) {
  const float a = fabsf(v);
  if (a == 0.f) return 0;
  return 1 + min(__float2int_rz(__fmul_rn(a, inv)), bins - 1);
}

// Lanes with the same counter add once, through their lowest lane: post-ReLU tensors are about half zeros and
// the rest crowds into the low bins, so one shared atomic per element would serialise on a few addresses.
// Every lane of the warp must call this; a lane without an element passes -1.
__device__ __forceinline__ void hist_add_warp(uint32_t *sh, int c) {
  const unsigned same = __match_any_sync(0xffffffffu, c);
  if (c >= 0 && (threadIdx.x & 31) == __ffs(same) - 1) atomicAdd(sh + c, (uint32_t)__popc(same));
}

__global__ void __launch_bounds__(kHistThreads) act_histogram_kernel(const float *__restrict__ y, long long n,
                                                                     const float *__restrict__ range, int id,
                                                                     int bins, unsigned long long *__restrict__ hist) {
  extern __shared__ uint32_t sh_hist[];  // [kHistCopies][bins + 1]
  const int stride_c = bins + 1;
  for (int i = threadIdx.x; i < kHistCopies * stride_c; i += blockDim.x) sh_hist[i] = 0;
  __syncthreads();
  const float inv = __fdiv_rn((float)bins, range[id]);
  uint32_t *sh = sh_hist + ((threadIdx.x >> 5) % kHistCopies) * stride_c;
  // aligned body: float4 loads from the first 16-byte boundary on; the (at most 3 + 3) elements before it and
  // after the last whole float4 are added by CTA 0 one by one
  const long long head = min((long long)(((16 - (reinterpret_cast<uintptr_t>(y) & 15)) & 15) >> 2), n);
  const long long n4 = (n - head) >> 2;
  const float4 *y4 = reinterpret_cast<const float4 *>(y + head);
  const int lane = threadIdx.x & 31;
  const long long step = (long long)gridDim.x * blockDim.x;
  for (long long base = blockIdx.x * (long long)blockDim.x + (threadIdx.x - lane); base < n4; base += step) {
    const long long i = base + lane;  // the loop bound is per warp: every lane reaches the match below
    int c0 = -1, c1 = -1, c2 = -1, c3 = -1;
    if (i < n4) {
      const float4 v = __ldg(y4 + i);
      c0 = hist_counter(v.x, inv, bins);
      c1 = hist_counter(v.y, inv, bins);
      c2 = hist_counter(v.z, inv, bins);
      c3 = hist_counter(v.w, inv, bins);
    }
    hist_add_warp(sh, c0);
    hist_add_warp(sh, c1);
    hist_add_warp(sh, c2);
    hist_add_warp(sh, c3);
  }
  if (blockIdx.x == 0) {
    const long long tail0 = head + (n4 << 2);
    const long long rest = head + (n - tail0);
    for (long long t = threadIdx.x; t < rest; t += blockDim.x) {
      const long long i = t < head ? t : tail0 + (t - head);
      atomicAdd(sh + hist_counter(y[i], inv, bins), 1u);
    }
  }
  __syncthreads();
  unsigned long long *out = hist + (long long)id * stride_c;
  for (int b = threadIdx.x; b < stride_c; b += blockDim.x) {
    uint32_t s = 0;
#pragma unroll
    for (int c = 0; c < kHistCopies; ++c) s += sh_hist[c * stride_c + b];
    if (s) atomicAdd(out + b, (unsigned long long)s);
  }
}

// T_k = range * k / bins in fp32 (bins a power of two: the divide is exact, T_bins == range)
__device__ __forceinline__ float hist_threshold(float range, int k, int bins) {
  return __fdiv_rn(__fmul_rn(range, (float)k), (float)bins);
}

constexpr int kScaleThreads = 256;

// Arg-min of (err, k) over the CTA, exact ties to the larger k; k == 0 marks a thread without a candidate.  Every
// thread of the CTA calls this once and gets the winning k.
__device__ int cta_argmin_larger_k(double best, int kb) {
  __shared__ double sh_best_err[kScaleThreads / 32];
  __shared__ int sh_best_k[kScaleThreads / 32];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    const double oe = __shfl_xor_sync(0xffffffffu, best, off);
    const int ok = __shfl_xor_sync(0xffffffffu, kb, off);
    if (ok != 0 && (kb == 0 || oe < best || (oe == best && ok > kb))) best = oe, kb = ok;
  }
  if ((threadIdx.x & 31) == 0) sh_best_err[threadIdx.x >> 5] = best, sh_best_k[threadIdx.x >> 5] = kb;
  __syncthreads();
  best = sh_best_err[0], kb = sh_best_k[0];
  for (int w = 1; w < kScaleThreads / 32; ++w) {
    const double oe = sh_best_err[w];
    const int ok = sh_best_k[w];
    if (ok != 0 && (kb == 0 || oe < best || (oe == best && ok > kb))) best = oe, kb = ok;
  }
  return kb;
}

__global__ void __launch_bounds__(kScaleThreads) hist_scales_kernel(const unsigned long long *__restrict__ hist,
                                                                   int bins, const float *__restrict__ range,
                                                                   const int32_t *__restrict__ qmax_arr, int method,
                                                                   double percentile, float headroom,
                                                                   float *__restrict__ act_scales) {
  // the non-empty bins of this tensor, compacted: bin centre and count (zeros contribute no error)
  __shared__ double sh_c[kHistMaxBins], sh_n[kHistMaxBins];
  __shared__ int sh_nnz;
  const int t = blockIdx.x;
  const unsigned long long *h = hist + (long long)t * (bins + 1);
  const float rng = range[t];
  const int qmax = qmax_arr[t];
  for (int j = threadIdx.x; j < bins; j += blockDim.x) {
    sh_c[j] = __ddiv_rn(__dmul_rn((double)j + 0.5, (double)rng), (double)bins);
    sh_n[j] = (double)h[1 + j];
  }
  __syncthreads();
  if (threadIdx.x == 0) {  // compacted in bin order (in place), so every run sums in the same order
    int m = 0;
    for (int j = 0; j < bins; ++j)
      if (sh_n[j] != 0.0) sh_c[m] = sh_c[j], sh_n[m] = sh_n[j], ++m;
    sh_nnz = m;
  }
  __syncthreads();
  const int nnz = sh_nnz;
  int k_best = bins;
  if (nnz == 0) {
    if (threadIdx.x == 0) act_scales[t] = 1.0f;
    return;
  }
  if (method == SLQ_CALIB_PERCENTILE) {
    if (threadIdx.x != 0) return;
    unsigned long long total = 0;
    for (int j = 0; j <= bins; ++j) total += h[j];
    const double target = ceil(percentile / 100.0 * (double)total);
    unsigned long long cum = h[0];
    for (k_best = 1; k_best < bins; ++k_best) {
      cum += h[k_best];  // zeros + n_0 .. n_{k-1}
      if ((double)cum >= target) break;
    }
  } else {
    // every candidate k on its own thread, summed over the non-empty bins (shared-memory broadcast reads);
    // separately rounded fp64 ops, as the oracle writes them
    double best = 0.0;
    int kb = 0;
    const double dq = (double)qmax;
    for (int k = 1 + threadIdx.x; k <= bins; k += blockDim.x) {
      const double D = __ddiv_rn((double)hist_threshold(rng, k, bins), dq);
      double err = 0.0;
      for (int s = 0; s < nnz; ++s) {
        const double c = sh_c[s];
        const double q = fmin(rint(__ddiv_rn(c, D)), dq);
        const double e = __dsub_rn(c, __dmul_rn(D, q));
        err = __dadd_rn(err, __dmul_rn(sh_n[s], __dmul_rn(e, e)));
      }
      if (kb == 0 || err <= best) best = err, kb = k;  // k rises along the loop: ties go to the larger k
    }
    k_best = cta_argmin_larger_k(best, kb);
    if (threadIdx.x != 0) return;
  }
  act_scales[t] = __fmul_rn(__fdiv_rn(hist_threshold(rng, k_best, bins), (float)qmax), headroom);
}

constexpr int kEntropyStartBin = 128;  // first candidate k of the entropy rule (pytorch-quantization's start_bin)

// The entropy (KL-divergence) rule of include/slq.h section 3, one CTA per tensor: every candidate k on its own
// thread, O(k) fp64 work from the prefix sums of the counts, then the CTA arg-min.
__global__ void __launch_bounds__(kScaleThreads) hist_entropy_kernel(const unsigned long long *__restrict__ hist,
                                                                    int bins, const float *__restrict__ range,
                                                                    const int32_t *__restrict__ qmax_arr,
                                                                    float headroom, float *__restrict__ act_scales) {
  // n_j, and M[j] = n_0 + .. + n_{j-1}, C[j] = bins with n > 0 among 0 .. j-1: a group's m_g and c_g in O(1)
  // (counts below 2^53: exact in fp64)
  __shared__ double sh_n[kHistMaxBins], sh_m[kHistMaxBins + 1];
  __shared__ int sh_c[kHistMaxBins + 1];
  const int t = blockIdx.x;
  const unsigned long long *h = hist + (long long)t * (bins + 1);
  for (int j = threadIdx.x; j < bins; j += blockDim.x) sh_n[j] = (double)h[1 + j];
  __syncthreads();
  if (threadIdx.x == 0) {
    double m = 0.0;
    int c = 0;
    for (int j = 0; j < bins; ++j) {
      sh_m[j] = m, sh_c[j] = c;
      m += sh_n[j], c += sh_n[j] != 0.0;
    }
    sh_m[bins] = m, sh_c[bins] = c;
  }
  __syncthreads();
  const double N = sh_m[bins];
  if (N == 0.0) {
    if (threadIdx.x == 0) act_scales[t] = 1.0f;
    return;
  }
  const int qmax = qmax_arr[t];
  // nq >= k splits every candidate into single bins, so capping nq at bins changes no group and keeps g * k
  // within int
  const int nq = min(qmax, bins - 1) + 1;
  double best = 0.0;
  int kb = 0;
  for (int k = kEntropyStartBin + threadIdx.x; k <= bins; k += blockDim.x) {
    const double kept = sh_m[k], o = N - kept;  // o_k: the outliers clipped onto bin k - 1
    double d = CUDART_INF;
    if (o == 0.0 || sh_n[k - 1] != 0.0) {
      double acc = 0.0;
      for (int g = 0, lo = 0; g < nq; ++g) {
        const int hi = ((g + 1) * k + nq - 1) / nq;  // group g: bins ceil(g k / nq) .. ceil((g + 1) k / nq) - 1
        const double m = sh_m[hi] - sh_m[lo];
        if (m != 0.0) {
          const double num = __dmul_rn((double)(sh_c[hi] - sh_c[lo]), kept), den = __dmul_rn(m, N);
          for (int j = lo; j < hi; ++j) {
            const double n = sh_n[j];
            if (n == 0.0) continue;
            const double p = j == k - 1 ? n + o : n;
            acc = __dadd_rn(acc, __dmul_rn(p, log(__ddiv_rn(__dmul_rn(p, num), den))));
          }
        }
        lo = hi;
      }
      d = __ddiv_rn(acc, N);
    }
    if (kb == 0 || d <= best) best = d, kb = k;  // k rises along the loop: ties go to the larger k
  }
  const int k_best = cta_argmin_larger_k(best, kb);
  if (threadIdx.x == 0)
    act_scales[t] = __fmul_rn(__fdiv_rn(hist_threshold(range[t], k_best, bins), (float)qmax), headroom);
}

}  // namespace slq

using namespace slq;

static bool hist_bins_ok(int32_t bins) { return bins >= 1 && bins <= kHistMaxBins && (bins & (bins - 1)) == 0; }

extern "C" int slq_act_histogram(const float *y, int64_t n, const float *range, int32_t id, int32_t bins,
                                 uint64_t *hist, void *stream) {
  SLQ_CHECK_ARG(y && range && hist && n > 0 && id >= 0, "slq_act_histogram: bad argument");
  SLQ_CHECK_ARG(hist_bins_ok(bins), "slq_act_histogram: bins=%d must be a power of two in [1, %d]", bins,
                kHistMaxBins);
  SLQ_CHECK_ARG(reinterpret_cast<uintptr_t>(y) % 4 == 0, "slq_act_histogram: y must be 4-byte aligned");
  const int blocks = (int)std::min<int64_t>(ceil_div(n / 4 + 1, kHistThreads), (int64_t)sm_count() * 8);
  const size_t smem = (size_t)kHistCopies * (bins + 1) * sizeof(uint32_t);
  act_histogram_kernel<<<blocks, kHistThreads, smem, (cudaStream_t)stream>>>(
      y, n, range, id, bins, reinterpret_cast<unsigned long long *>(hist));
  SLQ_LAUNCH_CHECK();
  return SLQ_OK;
}

extern "C" int slq_hist_scales(const uint64_t *hist, int32_t n_tensors, int32_t bins, const float *range,
                               const int32_t *qmax, int32_t method, double percentile, float headroom,
                               float *act_scales, void *stream) {
  SLQ_CHECK_ARG(hist && range && qmax && act_scales && n_tensors > 0, "slq_hist_scales: bad argument");
  SLQ_CHECK_ARG(hist_bins_ok(bins), "slq_hist_scales: bins=%d must be a power of two in [1, %d]", bins, kHistMaxBins);
  SLQ_CHECK_ARG(method == SLQ_CALIB_PERCENTILE || method == SLQ_CALIB_MSE || method == SLQ_CALIB_ENTROPY,
                "slq_hist_scales: method %d", method);
  SLQ_CHECK_ARG(method != SLQ_CALIB_ENTROPY || bins >= kEntropyStartBin,
                "slq_hist_scales: entropy needs at least %d bins, got bins=%d", kEntropyStartBin, bins);
  SLQ_CHECK_ARG(method != SLQ_CALIB_PERCENTILE || (percentile > 0.0 && percentile <= 100.0),
                "slq_hist_scales: percentile %g outside (0, 100]", percentile);
  SLQ_CHECK_ARG(headroom > 0.f, "slq_hist_scales: headroom must be positive");
  const auto *h = reinterpret_cast<const unsigned long long *>(hist);
  if (method == SLQ_CALIB_ENTROPY)
    hist_entropy_kernel<<<n_tensors, kScaleThreads, 0, (cudaStream_t)stream>>>(h, bins, range, qmax, headroom,
                                                                              act_scales);
  else
    hist_scales_kernel<<<n_tensors, kScaleThreads, 0, (cudaStream_t)stream>>>(h, bins, range, qmax, method,
                                                                             percentile, headroom, act_scales);
  SLQ_LAUNCH_CHECK();
  return SLQ_OK;
}
