// PSIS leave-one-out (sm_100a): per row of a [nrows][ld] fp64 matrix of per-draw log-likelihoods, the Pareto-smoothed
// importance-sampling estimate of the leave-one-out log predictive density, the log pointwise predictive density
// and the Pareto k-hat diagnostic (include/spmf_b200.h states the algorithm; the scalar pieces are in spmf_loo.cuh).
//
// Mapping: one CTA of 256 threads per row.  The row's S values go to shared memory (P = next power of two >= S
// doubles, padded with +inf, at most 64 KB) and are sorted ascending by a bitonic network; ascending
// log-likelihood is descending log-ratio, so the tail is the first n sorted entries.  The generalised Pareto fit
// takes one warp per grid point (lanes over the tail) for k_j, one thread per grid point for the weights, and
// thread 0 for the weighted grid mean.  Every reduction has a fixed order: a strided per-thread partial, a warp
// butterfly, then the warps' results in warp order.  Nothing is accumulated with atomics, so the outputs are
// bit-identical from run to run and a row's result does not depend on the other rows or on nrows.
// With `lw` given, each thread then writes the normalised log weights of its draws in draw order: a draw of the
// tail finds its sorted position by a binary search of the sorted row (tied draws of the tail are ranked by
// draw index, as a stable sort of the log-ratios ranks them).
#include <cuda_runtime.h>
#include <float.h>
#include <math.h>

#include "../../include/spmf_b200.h"
#include "spmf_loo.cuh"

namespace spmf {

constexpr int kLooThreads = 256;
constexpr int kLooWarps = kLooThreads / 32;

__device__ __forceinline__ double loo_warp_sum(double v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

// the block's sum (max) of one value per thread, returned to every thread
__device__ __forceinline__ double loo_block_sum(double v, double* red) {
  v = loo_warp_sum(v);
  __syncthreads();                                   // red[] may still be read by a previous reduction
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = 0.0;
#pragma unroll
  for (int w = 0; w < kLooWarps; ++w) t += red[w];
  return t;
}

__device__ __forceinline__ double loo_block_max(double v, double* red) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, off));
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
  __syncthreads();
  double t = red[0];
#pragma unroll
  for (int w = 1; w < kLooWarps; ++w) t = fmax(t, red[w]);
  return t;
}

// LW: also write the log weights (spmf_psis_loo_lw).  A template argument rather than a run-time test of lw, so
// that the instance without them compiles to the kernel spmf_psis_loo always ran (60 registers, no spills).
template <bool LW>
__global__ void __launch_bounds__(kLooThreads)
psis_loo_kernel(const double* __restrict__ ll, long long ld, int S, int P, double* __restrict__ elpd,
                double* __restrict__ lppd, float* __restrict__ khat, double* __restrict__ lw, long long ldw) {
  extern __shared__ double sv[];                     // [P] the row, sorted ascending (padding +inf)
  __shared__ double red[kLooWarps];
  __shared__ double tl[kLooMaxTail];                 // tail: y ascending, then its smoothed log weights
  __shared__ double gb[kLooMaxGrid], gL[kLooMaxGrid], gw[kLooMaxGrid];
  __shared__ double bhat_s;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long row = blockIdx.x;
  const double* x = ll + row * ld;
  const double INF = __longlong_as_double(0x7ff0000000000000ll);
  const double NaN = __longlong_as_double(0x7ff8000000000000ll);

  bool bad = false, neg = false;
  double mx = -INF;
  for (int i = tid; i < P; i += kLooThreads) {
    double v = INF;
    if (i < S) {
      v = __ldg(x + i);
      bad |= isnan(v) || v == INF;
      neg |= v == -INF;
      mx = fmax(mx, v);
    }
    sv[i] = v;
  }
  if (__syncthreads_or(bad)) {                       // NaN or +inf: nothing is defined
    if (tid == 0) {
      elpd[row] = lppd[row] = NaN;
      khat[row] = __int_as_float(0x7fc00000);
    }
    if (LW)
      for (int s = tid; s < S; s += kLooThreads) lw[row * ldw + s] = NaN;
    return;
  }
  neg = __syncthreads_or(neg);
  // lppd = log mean_s exp(ll_s), max-shifted
  mx = loo_block_max(mx, red);
  double acc = 0.0;
  for (int i = tid; i < S; i += kLooThreads) acc += exp(sv[i] - mx);
  acc = loo_block_sum(acc, red);
  const double lp = mx == -INF ? -INF : mx + log(acc) - log((double)S);
  if (neg) {                                         // some p = 0: the importance-sampling estimate 1/mean(1/p) is 0
    if (tid == 0) {
      elpd[row] = -INF;
      lppd[row] = lp;
      khat[row] = __int_as_float(0x7f800000);
    }
    if (LW)
      for (int s = tid; s < S; s += kLooThreads) lw[row * ldw + s] = NaN;
    return;
  }

  // bitonic sort, ascending
  for (int k = 2; k <= P; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      __syncthreads();
      for (int t = tid; t < (P >> 1); t += kLooThreads) {
        const int i = 2 * j * (t / j) + (t % j), p = i + j;
        const double a = sv[i], b = sv[p];
        if (((i & k) == 0) == (a > b)) {
          sv[i] = b;
          sv[p] = a;
        }
      }
    }
  }
  __syncthreads();

  // log-ratios r = -ll - max(-ll), descending along the sorted row: r_t = -sv[t] - rmax
  const double rmax = -sv[0];
  const int M = loo_tail_len(S);
  const double cut = fmax(-sv[M] - rmax, kLooLogDblMin);
  const double ecut = exp(cut);
  int n = 0;
  for (int i0 = 0; i0 < M; i0 += kLooThreads) {
    const int i = i0 + tid;
    n += __syncthreads_count(i < M && -sv[i] - rmax > cut);
  }
  double kh = INF;
  bool smooth = false;
  if (n > 4) {
    for (int i = tid; i < n; i += kLooThreads) tl[i] = exp(-sv[n - 1 - i] - rmax) - ecut;
    __syncthreads();
    const int m = loo_grid_size(n);
    const double y_last = tl[n - 1], y_quart = tl[loo_quartile_index(n)];
    for (int j = tid; j < m; j += kLooThreads) gb[j] = loo_grid_b(j + 1, m, y_last, y_quart);
    __syncthreads();
    for (int j = warp; j < m; j += kLooWarps) {      // k_j and the profile L_j: a warp per grid point
      const double b = gb[j];
      double s = 0.0;
      for (int i = lane; i < n; i += 32) s += log1p(-b * tl[i]);
      s = loo_warp_sum(s);
      if (lane == 0) gL[j] = loo_profile(n, b, s / n);
    }
    __syncthreads();
    // w_j = 1 / sum_i exp(L_i - L_j); an exp that overflows gives w_j = 0
    for (int j = tid; j < m; j += kLooThreads) {
      double t = 0.0;
      for (int i = 0; i < m; ++i) t += exp(gL[i] - gL[j]);
      gw[j] = 1.0 / t;
    }
    __syncthreads();
    if (tid == 0) {                                  // drop w_j < 10 eps (NaN included), renormalise, b-hat
      double wsum = 0.0;
      for (int j = 0; j < m; ++j)
        if (gw[j] >= 10.0 * DBL_EPSILON) wsum += gw[j];
      double b = 0.0;
      for (int j = 0; j < m; ++j)
        if (gw[j] >= 10.0 * DBL_EPSILON) b += gb[j] * (gw[j] / wsum);
      bhat_s = b;
    }
    __syncthreads();
    const double bhat = bhat_s;
    double s = 0.0;
    for (int i = tid; i < n; i += kLooThreads) s += log1p(-bhat * tl[i]);
    s = loo_block_sum(s, red);                       // (its barriers also end every read of y)
    const double k = s / n;
    const double sigma = -k / bhat;
    kh = (n * k + 5.0) / (n + 10.0);
    if (isfinite(kh) && isfinite(sigma) && sigma > 0.0) {
      for (int i = tid; i < n; i += kLooThreads) {
        const double w = log(loo_gpd_quantile((i + 0.5) / n, kh, sigma) + ecut);
        tl[i] = w > 0.0 ? 0.0 : w;                   // clamped at the largest raw log weight, 0
      }
      smooth = true;
    } else {
      kh = INF;
    }
    __syncthreads();
  }

  // normalised log weights lw_t = r_t - logsumexp(r); elpd = logsumexp(lw + ll)
  auto rw = [&](int t) { return (smooth && t < n) ? tl[n - 1 - t] : -sv[t] - rmax; };
  double m1 = -INF;
  for (int t = tid; t < S; t += kLooThreads) m1 = fmax(m1, rw(t));
  m1 = loo_block_max(m1, red);
  double s1 = 0.0;
  for (int t = tid; t < S; t += kLooThreads) s1 += exp(rw(t) - m1);
  const double lse_r = m1 + log(loo_block_sum(s1, red));
  double m2 = -INF;
  for (int t = tid; t < S; t += kLooThreads) m2 = fmax(m2, (rw(t) - lse_r) + sv[t]);
  m2 = loo_block_max(m2, red);
  double s2 = 0.0;
  for (int t = tid; t < S; t += kLooThreads) s2 += exp(((rw(t) - lse_r) + sv[t]) - m2);
  s2 = loo_block_sum(s2, red);
  if (tid == 0) {
    elpd[row] = m2 + log(s2);
    lppd[row] = lp;
    khat[row] = (float)kh;
  }
  if (!LW) return;
  // lw in draw order: the tail draws take their smoothed weight from their position in the sorted row
  for (int s = tid; s < S; s += kLooThreads) {
    const double v = __ldg(x + s);
    double r = -v - rmax;
    if (smooth) {
      int lo = 0, hi = n;                            // first sorted position holding v, if v is in the tail sv[0, n)
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (sv[mid] < v) lo = mid + 1; else hi = mid;
      }
      if (lo < n) {
        int t = lo;
        if (lo + 1 < n && sv[lo + 1] == v)           // tied tail draws: a later draw takes an earlier position
          for (int j = s + 1; j < S; ++j) t += __ldg(x + j) == v;
        r = tl[n - 1 - t];
      }
    }
    lw[row * ldw + s] = r - lse_r;
  }
}

}  // namespace spmf

using namespace spmf;

static int psis_loo_launch(const double* ll, long long ld, int nrows, int S, double* elpd, double* lppd, float* khat,
                           double* lw, long long ldw, void* stream) {
  if (!ll || !elpd || !lppd || !khat) return SPMF_ERR_BAD_ARG;
  if (nrows <= 0 || S < 1 || S > SPMF_LOO_MAX_S || ld < S) return SPMF_ERR_BAD_ARG;
  int P = 1;
  while (P < S) P <<= 1;
  const size_t smem = sizeof(double) * (size_t)P;
  auto kern = lw ? psis_loo_kernel<true> : psis_loo_kernel<false>;
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  kern<<<(unsigned)nrows, kLooThreads, smem, (cudaStream_t)stream>>>(ll, ld, S, P, elpd, lppd, khat, lw, ldw);
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? SPMF_OK : (int)e;
}

extern "C" {

int spmf_psis_loo(const double* ll, long long ld, int nrows, int S, double* elpd, double* lppd, float* khat,
                  void* stream) {
  return psis_loo_launch(ll, ld, nrows, S, elpd, lppd, khat, nullptr, 0, stream);
}

int spmf_psis_loo_lw(const double* ll, long long ld, int nrows, int S, double* elpd, double* lppd, float* khat,
                     double* lw, long long ldw, void* stream) {
  if (!lw || ldw < S) return SPMF_ERR_BAD_ARG;
  return psis_loo_launch(ll, ld, nrows, S, elpd, lppd, khat, lw, ldw, stream);
}

}  // extern "C"
