// LOO-PIT (sm_100a): the leave-one-row-out predictive CDF of every (row, feature) entry of a batch, weighted by
// the row's PSIS weights and summed over the draws, and the per-feature PIT histograms of the result
// (include/spmf_b200.h states the contracts; the CDFs and the binning are in spmf_pit.cuh).
//
// spmf_loo_pit_accum -- mapping: the row pass of spmf_dense.cu, as the posterior predictive check uses it.  A thread
// owns one (row, draw) and up to 32 latent dims of it (2 or 4 adjacent lanes per owner for K > 32); the CTA stages
// the EV records, phi and the observed count tile of 32 features in shared memory.  Unlike the check, one CTA walks
// every draw group q of the chunk for its rows (grid.y splits the feature tiles instead), so that the sum over the
// draws of an entry stays in the CTA: per tile of 32 features and per q, the owner lane forms the rate (link_rate), the two CDFs in fp64 and
// the weighted pair exp(lw) (F(x-1), F(x)); the pairs of 8 features go to shared memory, and one thread per entry
// adds them into the tile's accumulator in draw order (q outer, sv inner: ascending s).  After the last q the tile's
// sums are added to acc in global memory, which only this CTA touches.  Every sum has a fixed order that depends
// neither on nrows nor on the launch geometry, and there are no atomics, so acc is bit-identical from run to run.
//
// spmf_loo_pit_hist -- one thread per (feature, slot) and row block of kPitRowBlock rows: slots 0..J-1 are the
// bins, slot J counts the valid entries, slot J+1 sums their mean PIT.  A thread walks its rows in order and
// writes a partial; a second kernel adds the partials of the row blocks in order into the caller's outputs.
#include <cuda_runtime.h>
#include <float.h>

#include "../../include/spmf_b200.h"
#include "spmf_dense.cuh"
#include "spmf_pit.cuh"

namespace spmf {

constexpr int kPitSub = 8;             // features per shared-memory round of the weighted CDF pairs
constexpr int kPitRowBlock = 1024;     // rows per partial of the histogram pass
constexpr int kPitTargetCtas = 4096;   // accumulation grid: row tiles x feature groups of about this many CTAs

template <int KC, int LINK>
__global__ void __launch_bounds__(128)
loo_pit_accum_kernel(const float* __restrict__ xd, int nrows, int D, DenseGeom g, const float* __restrict__ EV,
                     const float* __restrict__ PH, const float* __restrict__ z, const double* __restrict__ lw,
                     long long ldw, double* __restrict__ acc, int* __restrict__ inv, float* __restrict__ rate_out) {
  extern __shared__ __align__(16) double pit_sm[];
  const RecMap rm = rec_map(g.KP);
  const int tile = blockIdx.x;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sv = warp % g.SV, grp = warp / g.SV;
  const int kq = lane % g.NKQ, ol = lane / g.NKQ;
  const int rloc = grp * g.OW + ol;
  const int row = tile * g.OB + rloc;
  const bool live = row < nrows;
  const bool owner = live && kq == 0;
  const int XS = g.OB + 1;
  const int nr = min(g.OB, nrows - tile * g.OB);    // live rows of this CTA
  double2* as = reinterpret_cast<double2*>(pit_sm);   // [kTile][OB]            the tile's sums over the draws
  double2* cs = as + kTile * g.OB;                    // [SV][kPitSub][OB]      weighted pairs of one round
  int* ai = reinterpret_cast<int*>(cs + g.SV * kPitSub * g.OB);   // [kTile][OB]  invalid draws
  int* ci = ai + kTile * g.OB;                                   // [SV][kPitSub][OB]
  float* es = reinterpret_cast<float*>(ci + g.SV * kPitSub * g.OB);   // [kTile][SV][KP]
  float* ps = es + kTile * g.REC;                                     // [kTile][SV]
  float* xs = ps + kTile * g.SV;                                      // [kTile][OB + 1]  observed counts
  const int ntile = kTile * g.OB;
  for (int d0 = blockIdx.y * kTile; d0 < D; d0 += gridDim.y * kTile) {
    const int nc = min(kTile, D - d0);
    __syncthreads();                                  // the previous tile's sums are written out
    for (int idx = threadIdx.x; idx < ntile; idx += blockDim.x) {
      as[idx] = make_double2(0.0, 0.0);
      ai[idx] = 0;
    }
    for (int idx = threadIdx.x; idx < g.OB * kTile; idx += blockDim.x) {
      const int r = idx / kTile, c = idx - r * kTile;
      const int rr = tile * g.OB + r, d = d0 + c;
      xs[c * XS + r] = (rr < nrows && d < D) ? __ldg(xd + (size_t)rr * D + d) : 0.f;
    }
    for (int q = 0; q < g.NQ; ++q) {
      __syncthreads();
      stage_records(es, EV + (size_t)q * D * g.REC, d0, kTile, D, g, rm);
      for (int idx = threadIdx.x; idx < kTile * g.SV; idx += blockDim.x) {
        const int c = idx / g.SV;
        ps[idx] = d0 + c < D ? __ldg(PH + ((size_t)q * D + d0 + c) * g.SV + (idx - c * g.SV)) : 1.f;
      }
      float zr[KC];
      const float* zq = z + ((size_t)q * nrows + (live ? row : 0)) * g.REC;
#pragma unroll
      for (int j = 0; j < KC; ++j) zr[j] = live ? __ldg(zq + rec_pos(g.KP, g.SV, sv, kq * KC + j)) : 0.f;
      const int s = q * g.SV + sv;
      const double w = owner ? exp(__ldg(lw + (size_t)row * ldw + s)) : 0.0;
      __syncthreads();
      for (int c0 = 0; c0 < nc; c0 += kPitSub) {
        const int ns = min(kPitSub, nc - c0);
        for (int cc = 0; cc < ns; ++cc) {
          const int c = c0 + cc;
          float e[KC];
          ld_slice<KC>(e, es + (c * g.SV + sv) * g.KP + kq * KC);
          float p = 0.f;
#pragma unroll
          for (int j = 0; j < KC; ++j) p = fmaf(zr[j], e[j], p);
          p = lanes_sum(p, g.NKQ);
          if (!owner) continue;
          const float rate = link_rate<LINK>(p, ps[c * g.SV + sv]);
          const float x = xs[c * XS + rloc];
          double fm = 0.0, fp = 0.0;
          bool ok;
          if (LINK < 2) {                              // Poisson(rate)
            ok = poisson_rate_ok(rate) && pit_count_ok(x, false);
            if (ok) poisson_cdf_pair((double)x, (double)rate, &fm, &fp);
          } else {                                     // Bernoulli(sigmoid(rate))
            ok = fabsf(rate) <= FLT_MAX && pit_count_ok(x, true);
            if (ok) {
              const double f0 = bernoulli_cdf(0.0, (double)rate);
              fm = x == 0.f ? 0.0 : f0;
              fp = x == 0.f ? f0 : 1.0;
            }
          }
          const int i = (sv * kPitSub + cc) * g.OB + rloc;
          cs[i] = ok ? make_double2(w * fm, w * fp) : make_double2(0.0, 0.0);
          ci[i] = !ok;
          if (rate_out) rate_out[((size_t)s * nrows + row) * D + d0 + c] = rate;
        }
        __syncthreads();
        // one thread per entry: the round's pairs in draw order
        for (int idx = threadIdx.x; idx < ns * g.OB; idx += blockDim.x) {
          const int cc = idx / g.OB, r = idx - cc * g.OB;
          if (r >= nr) continue;
          double2 a = as[(c0 + cc) * g.OB + r];
          int n = ai[(c0 + cc) * g.OB + r];
          for (int v = 0; v < g.SV; ++v) {
            const int i = (v * kPitSub + cc) * g.OB + r;
            a.x += cs[i].x;
            a.y += cs[i].y;
            n += ci[i];
          }
          as[(c0 + cc) * g.OB + r] = a;
          ai[(c0 + cc) * g.OB + r] = n;
        }
        __syncthreads();
      }
    }
    // the chunk's sums into acc (coalesced along the features)
    for (int idx = threadIdx.x; idx < nr * kTile; idx += blockDim.x) {
      const int r = idx / kTile, c = idx - r * kTile;
      if (c >= nc) continue;
      const size_t e = (size_t)(tile * g.OB + r) * D + d0 + c;
      const double2 a = as[c * g.OB + r];
      double2* o = reinterpret_cast<double2*>(acc) + e;
      double2 t = *o;
      t.x += a.x;
      t.y += a.y;
      *o = t;
      inv[e] += ai[c * g.OB + r];
    }
  }
}

static size_t pit_smem(const DenseGeom& g) {
  return sizeof(double2) * ((size_t)kTile * g.OB + (size_t)g.SV * kPitSub * g.OB) +
         sizeof(int) * ((size_t)kTile * g.OB + (size_t)g.SV * kPitSub * g.OB) +
         sizeof(float) * ((size_t)kTile * g.REC + (size_t)kTile * g.SV + (size_t)kTile * (g.OB + 1));
}

// partial[blockIdx.y][d][slot] over the rows of one row block, in row order
__global__ void __launch_bounds__(128)
loo_pit_hist_kernel(const double* __restrict__ acc, const int* __restrict__ inv, int nrows, int D, int J,
                    double* __restrict__ partial) {
  const int NS = J + 2;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)D * NS) return;
  const int d = (int)(t / NS), j = (int)(t - (long long)d * NS);
  const int r0 = blockIdx.y * kPitRowBlock, r1 = min(nrows, r0 + kPitRowBlock);
  const double2* a2 = reinterpret_cast<const double2*>(acc);
  double s = 0.0;
  for (int r = r0; r < r1; ++r) {
    const size_t e = (size_t)r * D + d;
    const double2 a = __ldg(a2 + e);
    if (__ldg(inv + e) != 0 || !isfinite(a.x) || !isfinite(a.y)) continue;   // invalid entry / excluded row
    if (j < J)
      s += czado_bin_mass(a.x, a.y, j, J);
    else if (j == J)
      s += 1.0;
    else
      s += 0.5 * (fmin(fmax(a.x, 0.0), 1.0) + fmin(fmax(a.y, 0.0), 1.0));
  }
  partial[(size_t)blockIdx.y * D * NS + t] = s;
}

__global__ void loo_pit_hist_reduce_kernel(const double* __restrict__ partial, int nblk, int D, int J,
                                           double* __restrict__ col_hist, long long* __restrict__ col_n,
                                           double* __restrict__ col_pit_sum) {
  const int NS = J + 2;
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (long long)D * NS) return;
  const int d = (int)(t / NS), j = (int)(t - (long long)d * NS);
  double s = 0.0;
  for (int b = 0; b < nblk; ++b) s += partial[(size_t)b * D * NS + t];
  if (j < J)
    col_hist[(size_t)d * J + j] += s;
  else if (j == J)
    col_n[d] += (long long)s;                      // an exact integer below 2^53
  else
    col_pit_sum[d] += s;
}

}  // namespace spmf

using namespace spmf;

extern "C" {

int spmf_loo_pit_accum(const float* xd, int nrows, int D, int K, int S, int link, const float* EV, const float* PH,
                       const float* z, const double* lw, long long ldw, double* acc, int* inv, float* rate_out,
                       void* stream) {
  if (!xd || !EV || !PH || !z || !lw || !acc || !inv) return SPMF_ERR_BAD_ARG;
  if (nrows <= 0 || D <= 0 || K <= 0 || K > SPMF_MAX_K || S <= 0 || S > SPMF_LOO_PIT_MAX_DRAWS || ldw < S)
    return SPMF_ERR_BAD_ARG;
  if (link < SPMF_LINK_POISSON || link > SPMF_LINK_BERNOULLI_LOG) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  cudaStream_t st = (cudaStream_t)stream;
#define CALL_L(KC, L)                                                                                          \
  {                                                                                                            \
    const DenseGeom g = dense_geom<KC>(KP, SV, NQ);                                                            \
    const size_t sm = pit_smem(g);                                                                             \
    int rc = set_smem(loo_pit_accum_kernel<KC, L>, sm);                                                        \
    if (rc) return rc;                                                                                         \
    const int gx = (nrows + g.OB - 1) / g.OB;                                                                 \
    const int gy = min((D + kTile - 1) / kTile, max(1, (kPitTargetCtas + gx - 1) / gx));                       \
    loo_pit_accum_kernel<KC, L><<<dim3(gx, gy), 128, sm, st>>>(xd, nrows, D, g, EV, PH, z, lw, ldw, acc, inv,     \
                                                             rate_out);                                        \
  }
#define CALL_K(KC) DENSE_LINK(KC, link, CALL_L)
  DENSE_KC(KP, CALL_K);
#undef CALL_K
#undef CALL_L
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? SPMF_OK : (int)e;
}

long long spmf_loo_pit_hist_scratch_doubles(int nrows, int D, int J) {
  if (nrows <= 0 || D <= 0 || J < 1 || J > SPMF_LOO_PIT_MAX_BINS) return -1;
  return (long long)((nrows + kPitRowBlock - 1) / kPitRowBlock) * D * (J + 2);
}

int spmf_loo_pit_hist(const double* acc, const int* inv, int nrows, int D, int J, double* col_hist,
                      long long* col_n, double* col_pit_sum, double* scratch, void* stream) {
  if (!acc || !inv || !col_hist || !col_n || !col_pit_sum || !scratch) return SPMF_ERR_BAD_ARG;
  if (nrows <= 0 || D <= 0 || J < 1 || J > SPMF_LOO_PIT_MAX_BINS) return SPMF_ERR_BAD_ARG;
  const int nblk = (nrows + kPitRowBlock - 1) / kPitRowBlock;
  const long long slots = (long long)D * (J + 2);
  const unsigned gx = (unsigned)((slots + 127) / 128);
  cudaStream_t st = (cudaStream_t)stream;
  loo_pit_hist_kernel<<<dim3(gx, nblk), 128, 0, st>>>(acc, inv, nrows, D, J, scratch);
  loo_pit_hist_reduce_kernel<<<gx, 128, 0, st>>>(scratch, nblk, D, J, col_hist, col_n, col_pit_sum);
  const cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? SPMF_OK : (int)e;
}

}  // extern "C"
