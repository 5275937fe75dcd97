// Posterior predictive check (sm_100a): replicated counts x_rep ~ p(x | theta_s) for every (draw, row, feature)
// entry of a batch and the check statistics of the replicates, in one pass that never writes the (S,B,D) rate
// tensor -- nor the replicates, unless asked to.
//
// Mapping: the row pass of spmf_dense.cu.  A thread owns one (row, draw) and up to 32 latent dims of it (2 or 4
// adjacent lanes per owner for K > 32); the CTA stages the EV records, phi and the observed count tile of 32
// features in shared memory.  Per entry the owner lane forms the rate exactly as the data term does
// (link_rate), draws the replicate (poisson_draw / bernoulli_draw, spmf_math.cuh) from the Philox stream keyed
// by (seed, draw, global row, feature), and accumulates in registers: the row's replicated total and nonzero
// count, and the realised discrepancies D(x_rep, theta) and D(x, theta) in fp64, summed in feature order.
// The replicates of a tile go to shared memory; one thread per (feature, draw) then sums them over the CTA's
// rows and adds the column total, sum of squares and nonzero count to global memory with integer atomics.
// Integer sums do not depend on the order of the additions, and every fp64 sum has a fixed order, so every
// output is bit-identical from run to run and does not depend on the launch geometry.
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include "../../include/spmf_b200.h"
#include "spmf_dense.cuh"

namespace spmf {

#define SPMF_CHECK_LAUNCH()                      \
  do {                                           \
    cudaError_t e__ = cudaGetLastError();        \
    if (e__ != cudaSuccess) return (int)e__;     \
  } while (0)

struct PpcOut {
  long long* row_total;               // [S][nrows]
  int* row_nnz;                       // [S][nrows]
  double* row_disc;                   // [S][nrows][2]: D(x_rep, theta), D(x, theta)
  unsigned long long* col_total;      // [S][D]   (accumulated)
  unsigned long long* col_sumsq;      // [S][D]
  unsigned int* col_nnz;              // [S][D]
  unsigned int* draw_max;             // [S]
  unsigned long long* draw_invalid;   // [S]
  int* out;                           // [S][nrows][D] or NULL
};

// (y - m)^2 / v of one entry; v == 0 (rate 0, or a logit saturated in fp32): 0 where y == m, +inf elsewhere
__device__ __forceinline__ float disc_term(float dy, float v) {
  return v > 0.f ? dy * dy / v : (dy == 0.f ? 0.f : __int_as_float(0x7f800000));
}

template <int KC, int LINK>
__global__ void __launch_bounds__(128)
ppc_rows_kernel(const float* __restrict__ xd, int nrows, int D, DenseGeom g, const float* __restrict__ EV,
                const float* __restrict__ PH, const float* __restrict__ z, Key2 key, long long row_offset, PpcOut o) {
  extern __shared__ __align__(16) float dsm[];
  const RecMap rm = rec_map(g.KP);
  const int tile = blockIdx.x, q = blockIdx.y;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sv = warp % g.SV, grp = warp / g.SV;
  const int kq = lane % g.NKQ, ol = lane / g.NKQ;
  const int rloc = grp * g.OW + ol;
  const int row = tile * g.OB + rloc;
  const bool live = row < nrows;
  const bool owner = live && kq == 0;
  const int XS = g.OB + 1;
  const int nr = min(g.OB, nrows - tile * g.OB);    // live rows of this CTA
  float* es = dsm;                                  // [kTile][SV][KP]
  float* ps = es + kTile * g.REC;                   // [kTile][SV]
  float* xs = ps + kTile * g.SV;                    // [kTile][OB + 1]       observed counts
  int* ys = reinterpret_cast<int*>(xs + kTile * XS);   // [SV][kTile][OB + 1]  replicates
  float zr[KC];
  const float* zq = z + ((size_t)q * nrows + (live ? row : 0)) * g.REC;
#pragma unroll
  for (int j = 0; j < KC; ++j) zr[j] = live ? zq[rec_pos(g.KP, g.SV, sv, kq * KC + j)] : 0.f;
  const int s = q * g.SV + sv;
  const long long grow = row_offset + row;
  long long tot = 0;
  int nnz = 0;
  unsigned ymax = 0u, ninv = 0u;
  double drep = 0.0, dobs = 0.0;
  for (int d0 = 0; d0 < D; d0 += kTile) {
    __syncthreads();
    stage_records(es, EV + (size_t)q * D * g.REC, d0, kTile, D, g, rm);
    for (int idx = threadIdx.x; idx < kTile * g.SV; idx += blockDim.x) {
      const int c = idx / g.SV;
      ps[idx] = d0 + c < D ? __ldg(PH + ((size_t)q * D + d0 + c) * g.SV + (idx - c * g.SV)) : 1.f;
    }
    for (int idx = threadIdx.x; idx < g.OB * kTile; idx += blockDim.x) {
      const int r = idx / kTile, c = idx - r * kTile;
      const int rr = tile * g.OB + r, d = d0 + c;
      xs[c * XS + r] = (rr < nrows && d < D) ? __ldg(xd + (size_t)rr * D + d) : 0.f;
    }
    __syncthreads();
    const int nc = min(kTile, D - d0);
    for (int c = 0; c < nc; ++c) {
      float e[KC];
      ld_slice<KC>(e, es + (c * g.SV + sv) * g.KP + kq * KC);
      float p = 0.f;
#pragma unroll
      for (int j = 0; j < KC; ++j) p = fmaf(zr[j], e[j], p);
      p = lanes_sum(p, g.NKQ);
      if (!owner) continue;
      const float rate = link_rate<LINK>(p, ps[c * g.SV + sv]);
      const float x = xs[c * XS + rloc];
      const U4 ctr = ppc_counter(s, grow, d0 + c);
      int y = 0;
      if (LINK < 2) {                                  // Poisson(rate)
        if (poisson_rate_ok(rate)) {
          y = poisson_draw(rate, key, ctr);
          drep += (double)disc_term((float)y - rate, rate);
          dobs += (double)disc_term(x - rate, rate);
        } else {
          ++ninv;
        }
      } else {                                         // Bernoulli(sigmoid(rate)); p and 1 - p without cancellation
        if (fabsf(rate) <= FLT_MAX) {
          const float ex = __expf(-fabsf(rate));
          const float r = __fdividef(1.f, 1.f + ex);
          const float sg = rate >= 0.f ? r : ex * r, oms = rate >= 0.f ? ex * r : r;
          y = bernoulli_draw(sg, key, ctr);
          const float v = sg * oms;
          drep += (double)disc_term(y ? oms : -sg, v);
          dobs += (double)disc_term(x == 1.f ? oms : x - sg, v);
        } else {
          ++ninv;
        }
      }
      tot += y;
      nnz += y != 0;
      ymax = max(ymax, (unsigned)y);
      ys[(sv * kTile + c) * XS + rloc] = y;
    }
    __syncthreads();
    // per (feature, draw): sums over the CTA's rows, then one integer atomic each into global memory
    {
      const int c = threadIdx.x % kTile, cs = threadIdx.x / kTile;
      if (cs < g.SV && c < nc) {
        const int* col = ys + (cs * kTile + c) * XS;
        unsigned long long t = 0ull, t2 = 0ull;
        unsigned n = 0u;
        for (int r = 0; r < nr; ++r) {
          const unsigned long long y = (unsigned)col[r];
          t += y;
          t2 += y * y;
          n += y != 0ull;
        }
        if (t) {
          const size_t i = (size_t)(q * g.SV + cs) * D + d0 + c;
          atomicAdd(o.col_total + i, t);
          atomicAdd(o.col_sumsq + i, t2);
          atomicAdd(o.col_nnz + i, n);
        }
      }
    }
    if (o.out) {                                       // materialisation: coalesced along the features
      for (int idx = threadIdx.x; idx < g.SV * nr * kTile; idx += blockDim.x) {
        const int c = idx % kTile, t = idx / kTile, r = t % nr, v = t / nr;
        if (c < nc)
          o.out[((size_t)(q * g.SV + v) * nrows + tile * g.OB + r) * D + d0 + c] = ys[(v * kTile + c) * XS + r];
      }
    }
  }
  // per draw: maximum replicate and invalid entries, one atomic per warp (its lanes share the draw)
  const unsigned wmax = __reduce_max_sync(0xffffffffu, ymax);
  const unsigned winv = __reduce_add_sync(0xffffffffu, ninv);
  if (lane == 0) {
    if (wmax) atomicMax(o.draw_max + s, wmax);
    if (winv) atomicAdd(o.draw_invalid + s, (unsigned long long)winv);
  }
  if (!owner) return;
  const size_t i = (size_t)s * nrows + row;
  o.row_total[i] = tot;
  o.row_nnz[i] = nnz;
  o.row_disc[2 * i] = drep;
  o.row_disc[2 * i + 1] = dobs;
}

// observed statistics of a CSR batch: warp per row (fixed-order shuffle sums), fp64 / integer atomics per column
__global__ void ppc_observed_kernel(const long long* __restrict__ rowptr, const int* __restrict__ cols,
                                    const float* __restrict__ vals, int nrows, double* __restrict__ row_total,
                                    int* __restrict__ row_nnz, double* __restrict__ col_total,
                                    double* __restrict__ col_sumsq, unsigned int* __restrict__ col_nnz) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= nrows) return;
  double t = 0.0;
  int n = 0;
  for (long long j = rowptr[row] + lane; j < rowptr[row + 1]; j += 32) {
    const double x = fabsf(__ldg(vals + j));     // |x|: the value the dense scatter gives the check pass
    if (x == 0.0) continue;
    const int d = __ldg(cols + j);
    t += x;
    ++n;
    atomicAdd(col_total + d, x);
    atomicAdd(col_sumsq + d, x * x);
    atomicAdd(col_nnz + d, 1u);
  }
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    t += __shfl_xor_sync(0xffffffffu, t, off);
    n += __shfl_xor_sync(0xffffffffu, n, off);
  }
  if (lane == 0) {
    row_total[row] = t;
    row_nnz[row] = n;
  }
}

static size_t ppc_smem(const DenseGeom& g) {
  return sizeof(float) * ((size_t)kTile * g.REC + (size_t)kTile * g.SV + (size_t)kTile * (g.OB + 1)) +
         sizeof(int) * (size_t)g.SV * kTile * (g.OB + 1);
}

}  // namespace spmf

using namespace spmf;

extern "C" {

int spmf_ppc_rows(const float* xd, int nrows, int D, int K, int S, int link, const float* EV, const float* PH,
                  const float* z, unsigned long long seed, long long row_offset, long long* row_total, int* row_nnz,
                  double* row_disc, unsigned long long* col_total, unsigned long long* col_sumsq,
                  unsigned int* col_nnz, unsigned int* draw_max, unsigned long long* draw_invalid, int* out,
                  double* disc_sum, double* scratch, void* stream) {
  if (!xd || !EV || !PH || !z || !row_total || !row_nnz || !row_disc || !col_total || !col_sumsq || !col_nnz ||
      !draw_max || !draw_invalid || !disc_sum || !scratch)
    return SPMF_ERR_BAD_ARG;
  if (nrows <= 0 || D <= 0 || K <= 0 || K > SPMF_MAX_K || S <= 0 || S > SPMF_PPC_MAX_S) return SPMF_ERR_BAD_ARG;
  if (link < SPMF_LINK_POISSON || link > SPMF_LINK_BERNOULLI_LOG) return SPMF_ERR_BAD_ARG;
  if (row_offset < 0 || row_offset + nrows > SPMF_PPC_MAX_ROW) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  const Key2 key = ppc_key(seed);
  const PpcOut o{row_total, row_nnz, row_disc, col_total, col_sumsq, col_nnz, draw_max, draw_invalid, out};
  cudaStream_t st = (cudaStream_t)stream;
#define CALL_L(KC, L)                                                                                     \
  {                                                                                                       \
    const DenseGeom g = dense_geom<KC>(KP, SV, NQ);                                                       \
    const size_t sm = ppc_smem(g);                                                                        \
    int rc = set_smem(ppc_rows_kernel<KC, L>, sm);                                                        \
    if (rc) return rc;                                                                                    \
    ppc_rows_kernel<KC, L><<<dim3((nrows + g.OB - 1) / g.OB, NQ), 128, sm, st>>>(xd, nrows, D, g, EV, PH, z, \
                                                                                 key, row_offset, o);      \
  }
#define CALL_K(KC) DENSE_LINK(KC, link, CALL_L)
  DENSE_KC(KP, CALL_K);
#undef CALL_K
#undef CALL_L
  SPMF_CHECK_LAUNCH();
  return spmf_colsum_f64(row_disc, nrows, 2, S, disc_sum, scratch, stream);
}

int spmf_ppc_observed(const long long* rowptr, const int* cols, const float* vals, int nrows, int D,
                      double* row_total, int* row_nnz, double* col_total, double* col_sumsq, unsigned int* col_nnz,
                      void* stream) {
  if (!rowptr || !cols || !vals || !row_total || !row_nnz || !col_total || !col_sumsq || !col_nnz || nrows <= 0 ||
      D <= 0)
    return SPMF_ERR_BAD_ARG;
  ppc_observed_kernel<<<(unsigned)((nrows + 7) / 8), 256, 0, (cudaStream_t)stream>>>(
      rowptr, cols, vals, nrows, row_total, row_nnz, col_total, col_sumsq, col_nnz);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

}  // extern "C"
