// Dense evaluation of the data term on the CUDA cores (sm_100a): every (draw, row, feature) entry of
// the rate matrix is visited -- tile by tile, in registers, never written to memory.
//
// Three users:
//   * the link functions that have no closed form for sum(rate): `log_transform=True`
//     (poisson.py:41-42, 52-53: encoder log(x/eta + 1), decoder exp(y*eta) - 1) and the
//     Bernoulli-logit likelihood of BernoulliFactorization (bernoulli.py:148);
//   * the EXACT non-finite guard of poisson.py:606-616 for the default (linear) link: when the fast
//     sparse / tensor-core path has seen an entry whose log-likelihood is not finite, the whole data
//     term of that step is re-evaluated here with the reference's semantics -- non-finite entries
//     are replaced by  min(finite entries over the whole (S,B,D) tensor) - 10  in the value, carry no
//     gradient of their own, and the gradient of that minimum flows to the entry attaining it;
//   * WAIC / row_log_likelihood for those links.
//
// Mapping: a thread owns one (row, draw) of the row pass [or one (feature, draw) of the column pass]
// and up to 32 latent dims of it (wider latent spaces split a row over 2 or 4 adjacent lanes); it
// keeps its z (EV) slice and the gradient accumulators in registers and walks the features (rows) of
// the batch; the operand records and the count tile it meets on the way are staged in shared memory
// by the whole CTA (coalesced global reads, broadcast / conflict-free shared reads).  This is the
// "x tile in shared memory, rate recomputed in registers, dL/drate feeding dz and dv in the same
// pass" formulation; it is FMA-bound (2*K FMAs per entry and pass against K/4 + 1 shared loads).
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include "../../include/spmf_b200.h"
#include "spmf_dense.cuh"
#include "spmf_guard.cuh"

namespace spmf {

#define SPMF_CHECK_LAUNCH()                      \
  do {                                           \
    cudaError_t e__ = cudaGetLastError();        \
    if (e__ != cudaSuccess) return (int)e__;     \
  } while (0)

constexpr int LINK_POIS_LIN = SPMF_LINK_POISSON;
constexpr int MODE_OPT = SPMF_DENSE_OPTIMISTIC, MODE_STATS = SPMF_DENSE_STATS, MODE_GUARD = SPMF_DENSE_GUARDED;

__device__ __forceinline__ float lgamma1p(float x) { return (x == 0.f || x == 1.f) ? 0.f : lgammaf(x + 1.f); }

// ---------------------------------------------------------------------------------------------------
// densify: xd[B][D] (fp32, TABLE order: column = table row of the feature) from a CSR batch whose
// column ids are already table rows; hybrid batches flag covered entries with a negative sign.
// ---------------------------------------------------------------------------------------------------
__device__ void phase_zero(float* __restrict__ p, long long n, long long tid, long long nth) {
  float4* p4 = reinterpret_cast<float4*>(p);
  const long long n4 = n >> 2;
  for (long long i = tid; i < n4; i += nth) p4[i] = make_float4(0.f, 0.f, 0.f, 0.f);
  for (long long i = (n4 << 2) + tid; i < n; i += nth) p[i] = 0.f;
}
__device__ void phase_scatter(const long long* __restrict__ rowptr, const int* __restrict__ cols,
                              const float* __restrict__ vals, int nrows, int D, float* __restrict__ xd,
                              long long wid, long long nw, int lane) {
  for (long long row = wid; row < nrows; row += nw) {           // warp per row
    const long long j0 = rowptr[row], j1 = rowptr[row + 1];
    for (long long j = j0 + lane; j < j1; j += 32) xd[row * D + cols[j]] = fabsf(vals[j]);
  }
}

// densify from the raw dense upload (feature order) of a dense-ingested batch
template <typename T>
__device__ void phase_scatter_raw(const T* __restrict__ raw, const int* __restrict__ rank, int nrows, int D,
                                  float* __restrict__ xd, long long tid, long long nth) {
  const long long n = (long long)nrows * D;
  for (long long i = tid; i < n; i += nth) {
    const long long row = i / D;
    const int d = (int)(i - row * D);
    xd[row * D + (rank ? rank[d] : d)] = (float)raw[i];
  }
}

__global__ void dense_zero_kernel(float* __restrict__ p, long long n, const GuardState* __restrict__ gs, int cond) {
  if (cond && !(gs && (gs->flag & 1))) return;
  phase_zero(p, n, (long long)blockIdx.x * blockDim.x + threadIdx.x, (long long)gridDim.x * blockDim.x);
}
__global__ void dense_scatter_kernel(const long long* __restrict__ rowptr, const int* __restrict__ cols,
                                     const float* __restrict__ vals, int nrows, int D, float* __restrict__ xd) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  phase_scatter(rowptr, cols, vals, nrows, D, xd, t >> 5, ((long long)gridDim.x * blockDim.x) >> 5, threadIdx.x & 31);
}

// ---------------------------------------------------------------------------------------------------
// encode (log link): z_b = r_b sum_d log(x_bd/eta_d + 1) A'_d        poisson.py:41-42, 640-649
// ---------------------------------------------------------------------------------------------------
struct DenseBatch {
  const float* xd;            // [nrows][D]
  const float* rowsum;        // [nrows]
  const float* lgam;          // [nrows] sum_d lgamma(x+1)
  const float* eta_enc;       // [D] table order: encoder divisor (log link) -- may be NULL for the linear encoder
  float inv_xi;
  int scale_rows, nrows, D;
};

template <int KC, int LINK>
__device__ void phase_encode(const DenseBatch& b, const DenseGeom& g, const float* __restrict__ Ap,
                             float* __restrict__ z, float* sm, int tile, int q) {
  const RecMap rm = rec_map(g.KP);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sv = warp % g.SV, grp = warp / g.SV;
  const int kq = lane % g.NKQ, ol = lane / g.NKQ;
  const int rloc = grp * g.OW + ol;
  const int row = tile * g.OB + rloc;
  float* as = sm;                                   // [kTile][SV][KP]
  float* xs = as + kTile * g.REC;                   // [kTile][OB + 1]
  const int XS = g.OB + 1;
  float acc[KC];
#pragma unroll
  for (int j = 0; j < KC; ++j) acc[j] = 0.f;
  for (int d0 = 0; d0 < b.D; d0 += kTile) {
    __syncthreads();
    stage_records(as, Ap + (size_t)q * b.D * g.REC, d0, kTile, b.D, g, rm);
    for (int idx = threadIdx.x; idx < g.OB * kTile; idx += blockDim.x) {
      const int r = idx / kTile, c = idx - r * kTile;
      const int rr = tile * g.OB + r, d = d0 + c;
      float e = 0.f;
      if (rr < b.nrows && d < b.D) {
        const float x = __ldg(b.xd + (size_t)rr * b.D + d);
        if (LINK & 1) e = x > 0.f ? log1pf(x / __ldg(b.eta_enc + d)) : 0.f;   // poisson.py:41-42
        else e = x;                                                          // 1/eta is folded into A'
      }
      xs[c * XS + r] = e;
    }
    __syncthreads();
    const int nc = min(kTile, b.D - d0);
    for (int c = 0; c < nc; ++c) {
      const float e = xs[c * XS + rloc];
      float a[KC];
      ld_slice<KC>(a, as + (c * g.SV + sv) * g.KP + kq * KC);
#pragma unroll
      for (int j = 0; j < KC; ++j) acc[j] = fmaf(e, a[j], acc[j]);
    }
  }
  if (row < b.nrows) {
    const float r = b.scale_rows ? b.rowsum[row] * b.inv_xi : 1.f;      // poisson.py:644-649 (raw row sums)
    float* zq = z + ((size_t)q * b.nrows + row) * g.REC;
#pragma unroll
    for (int j = 0; j < KC; ++j) zq[rec_pos(g.KP, g.SV, sv, kq * KC + j)] = r * acc[j];
  }
}

// ---------------------------------------------------------------------------------------------------
// row pass: per (row, draw): sum_d ll, dz = sum_d dL/dlin EV_d, finished in place:
//   dzr = r (dz - z)  (z prior HalfNormal(1), poisson.py:599-604),  rowacc = (sum ll, 0, |z|^2, #bad)
// mode OPT: no guard input (bad entries dropped and counted); STATS: counts / minimum only;
// GUARD: reads gs (nbad over all draws, arg-min entry) and adds the gradient of the minimum.
// ---------------------------------------------------------------------------------------------------
template <int KC, int LINK>
__device__ void phase_rows(const DenseBatch& b, const DenseGeom& g, const float* __restrict__ EV,
                           const float* __restrict__ PH, const float* __restrict__ z, float* __restrict__ dzr,
                           float* __restrict__ rowacc, GuardState* gs, int mode, float* sm, int tile, int q) {
  const RecMap rm = rec_map(g.KP);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sv = warp % g.SV, grp = warp / g.SV;
  const int kq = lane % g.NKQ, ol = lane / g.NKQ;
  const int rloc = grp * g.OW + ol;
  const int row = tile * g.OB + rloc;
  const bool live = row < b.nrows;
  float* es = sm;                                   // [kTile][SV][KP]
  float* ps = es + kTile * g.REC;                   // [kTile][SV]
  float* xs = ps + kTile * g.SV;                    // [kTile][OB + 1]
  const int XS = g.OB + 1;
  float zr[KC], dz[KC];
  const float* zq = z + ((size_t)q * b.nrows + (live ? row : 0)) * g.REC;
#pragma unroll
  for (int j = 0; j < KC; ++j) {
    zr[j] = live ? zq[rec_pos(g.KP, g.SV, sv, kq * KC + j)] : 0.f;
    dz[j] = 0.f;
  }
  const int s = q * g.SV + sv;
  const bool want_ll = mode != MODE_OPT;            // per-entry lgamma only when the minimum is tracked
  int nbad_all = 0;
  unsigned argmin_lo = 0;
  bool has_min = false;
  if (mode == MODE_GUARD) {
    nbad_all = gs->nbad;
    argmin_lo = (unsigned)(gs->minkey & 0xffffffffull);
    has_min = nbad_all > 0 && gs->minkey != ~0ull;
  }
  float llsum = 0.f, badlg = 0.f;
  int nbad = 0;
  unsigned long long mykey = ~0ull;
  for (int d0 = 0; d0 < b.D; d0 += kTile) {
    __syncthreads();
    stage_records(es, EV + (size_t)q * b.D * g.REC, d0, kTile, b.D, g, rm);
    for (int idx = threadIdx.x; idx < kTile * g.SV; idx += blockDim.x) {
      const int c = idx / g.SV;
      ps[idx] = d0 + c < b.D ? __ldg(PH + ((size_t)q * b.D + d0 + c) * g.SV + (idx - c * g.SV)) : 1.f;
    }
    for (int idx = threadIdx.x; idx < g.OB * kTile; idx += blockDim.x) {
      const int r = idx / kTile, c = idx - r * kTile;
      const int rr = tile * g.OB + r, d = d0 + c;
      xs[c * XS + r] = (rr < b.nrows && d < b.D) ? __ldg(b.xd + (size_t)rr * b.D + d) : 0.f;
    }
    __syncthreads();
    const int nc = min(kTile, b.D - d0);
    for (int c = 0; c < nc; ++c) {
      const float x = xs[c * XS + rloc];
      float e[KC];
      ld_slice<KC>(e, es + (c * g.SV + sv) * g.KP + kq * KC);
      float p = 0.f;
#pragma unroll
      for (int j = 0; j < KC; ++j) p = fmaf(zr[j], e[j], p);
      p = lanes_sum(p, g.NKQ);
      const Elem el = link_elem<LINK>(x, p, ps[c * g.SV + sv]);
      float wgt = 1.f;
      if (!el.ok) {
        ++nbad;
        if (LINK < 2) badlg += lgamma1p(x);
      } else if (want_ll) {
        const float ll = el.ll - (LINK < 2 ? lgamma1p(x) : 0.f);
        const unsigned lo = (unsigned)((((unsigned long long)s * b.nrows + row) * b.D + d0 + c) & 0xffffffffull);
        if (mode == MODE_STATS) {
          const unsigned long long key = ((unsigned long long)ordered_bits(ll) << 32) | lo;
          mykey = key < mykey ? key : mykey;
        } else if (has_min && lo == argmin_lo) {
          wgt = 1.f + (float)nbad_all;              // d/dtheta of nbad * (min - 10): poisson.py:609-616
        }
      }
      llsum += el.ll;
      const float gl = el.glin * wgt;
#pragma unroll
      for (int j = 0; j < KC; ++j) dz[j] = fmaf(gl, e[j], dz[j]);
    }
  }
  if (mode == MODE_STATS) {
    if (live && kq == 0) {
      if (nbad) atomicAdd(&gs->nbad, nbad);
      if (mykey != ~0ull) atomicMin(&gs->minkey, mykey);
    }
    return;
  }
  float z2 = 0.f;
#pragma unroll
  for (int j = 0; j < KC; ++j) z2 = fmaf(zr[j], zr[j], z2);
  z2 = lanes_sum(z2, g.NKQ);          // (full-warp shuffle: before any lane leaves)
  if (!live) return;
  const float r = b.scale_rows ? b.rowsum[row] * b.inv_xi : 1.f;
  float* dq = dzr + ((size_t)q * b.nrows + row) * g.REC;
#pragma unroll
  for (int j = 0; j < KC; ++j) dq[rec_pos(g.KP, g.SV, sv, kq * KC + j)] = r * (dz[j] - zr[j]);
  if (kq == 0) {
    float* ra = rowacc + ((size_t)q * b.nrows + row) * 4 * g.SV;
    // Poisson: sum over the finite entries of -lgamma(x+1) = -(row total) + (the bad entries' share)
    ra[0 * g.SV + sv] = llsum - (LINK < 2 ? b.lgam[row] - badlg : 0.f);
    ra[1 * g.SV + sv] = 0.f;
    ra[2 * g.SV + sv] = z2;
    ra[3 * g.SV + sv] = (float)nbad;
    if (mode == MODE_OPT && nbad) atomicOr(&gs->flag, 1);      // the statistics pass will count them
  }
}

// ---------------------------------------------------------------------------------------------------
// column pass: per (feature, draw): GEV_d = sum_b dL/dlin z_b, Gphi_d = sum_b dL/dphi and (with_ga)
// GA'_d = sum_b enc(x_bd) dzr_b; accumulated with atomics over row splits (tables zeroed before).
// Guard-aware through gs (nbad > 0: bad entries carry no gradient, the arg-min entry nbad more).
// ---------------------------------------------------------------------------------------------------
template <int KC, int LINK>
__device__ void phase_cols(const DenseBatch& b, const DenseGeom& g, const float* __restrict__ EV,
                           const float* __restrict__ PH, const float* __restrict__ z, const float* __restrict__ dzr,
                           float* __restrict__ GAp, float* __restrict__ GEV, float* __restrict__ Gph,
                           const GuardState* gs, int with_ga, float* sm, int ctile, int q, int r_begin, int r_end) {
  const RecMap rm = rec_map(g.KP);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int sv = warp % g.SV, grp = warp / g.SV;
  const int kq = lane % g.NKQ, ol = lane / g.NKQ;
  const int cloc = grp * g.OW + ol;
  const int d = ctile * g.OB + cloc;
  const bool live = d < b.D;
  float* zs = sm;                                   // [kTile][SV][KP]
  float* ds = zs + kTile * g.REC;                   // [kTile][SV][KP]   (with_ga)
  float* xs = ds + (with_ga ? kTile * g.REC : 0);   // [kTile][OB]
  float ev[KC], gev[KC], ga[KC];
  const float* eq = EV + ((size_t)q * b.D + (live ? d : 0)) * g.REC;
#pragma unroll
  for (int j = 0; j < KC; ++j) {
    ev[j] = live ? eq[rec_pos(g.KP, g.SV, sv, kq * KC + j)] : 0.f;
    gev[j] = 0.f;
    ga[j] = 0.f;
  }
  const float phi = live ? PH[((size_t)q * b.D + d) * g.SV + sv] : 1.f;
  const float eta_e = (live && (LINK & 1)) ? b.eta_enc[d] : 1.f;
  const int s = q * g.SV + sv;
  const int nbad_all = gs ? gs->nbad : 0;
  const bool has_min = nbad_all > 0 && gs->minkey != ~0ull;
  const unsigned argmin_lo = has_min ? (unsigned)(gs->minkey & 0xffffffffull) : 0u;
  float gphi = 0.f;
  for (int r0 = r_begin; r0 < r_end; r0 += kTile) {
    __syncthreads();
    const int nr = min(kTile, r_end - r0);
    stage_records(zs, z + (size_t)q * b.nrows * g.REC, r0, nr, b.nrows, g, rm);
    if (with_ga) stage_records(ds, dzr + (size_t)q * b.nrows * g.REC, r0, nr, b.nrows, g, rm);
    for (int idx = threadIdx.x; idx < nr * g.OB; idx += blockDim.x) {
      const int r = idx / g.OB, c = idx - r * g.OB;
      const int dd = ctile * g.OB + c;
      xs[idx] = dd < b.D ? __ldg(b.xd + (size_t)(r0 + r) * b.D + dd) : 0.f;
    }
    __syncthreads();
    for (int r = 0; r < nr; ++r) {
      const float x = xs[r * g.OB + cloc];
      float zz[KC];
      ld_slice<KC>(zz, zs + (r * g.SV + sv) * g.KP + kq * KC);
      float p = 0.f;
#pragma unroll
      for (int j = 0; j < KC; ++j) p = fmaf(zz[j], ev[j], p);
      p = lanes_sum(p, g.NKQ);
      const Elem el = link_elem<LINK>(x, p, phi);
      float wgt = 1.f;
      if (has_min && el.ok) {
        const unsigned lo = (unsigned)((((unsigned long long)s * b.nrows + r0 + r) * b.D + d) & 0xffffffffull);
        if (lo == argmin_lo) wgt = 1.f + (float)nbad_all;
      }
      const float gl = el.glin * wgt;
      gphi = fmaf(el.gphi, wgt, gphi);
#pragma unroll
      for (int j = 0; j < KC; ++j) gev[j] = fmaf(gl, zz[j], gev[j]);
      if (with_ga) {
        const float e = (LINK & 1) ? (x > 0.f ? log1pf(x / eta_e) : 0.f) : x;
        float dd[KC];
        ld_slice<KC>(dd, ds + (r * g.SV + sv) * g.KP + kq * KC);
#pragma unroll
        for (int j = 0; j < KC; ++j) ga[j] = fmaf(e, dd[j], ga[j]);
      }
    }
  }
  if (!live) return;
  const size_t o = ((size_t)q * b.D + d) * g.REC;
#pragma unroll
  for (int j = 0; j < KC; ++j) {
    const int p = rec_pos(g.KP, g.SV, sv, kq * KC + j);
    atomicAdd(GEV + o + p, gev[j]);
    if (with_ga) atomicAdd(GAp + o + p, ga[j]);
  }
  if (kq == 0) atomicAdd(Gph + ((size_t)q * b.D + d) * g.SV + sv, gphi);
}

// ---------------------------------------------------------------------------------------------------
// kernels: one phase per launch (dense-link path) ...
// ---------------------------------------------------------------------------------------------------
template <int KC, int LINK>
__global__ void __launch_bounds__(128)
dense_encode_kernel(DenseBatch b, DenseGeom g, const float* __restrict__ Ap, float* __restrict__ z) {
  extern __shared__ __align__(16) float dsm[];
  phase_encode<KC, LINK>(b, g, Ap, z, dsm, blockIdx.x, blockIdx.y);
}

// cond != 0: run only when the step has met non-finite entries (gs->flag bit 0)
template <int KC, int LINK>
__global__ void __launch_bounds__(128)
dense_rows_kernel(DenseBatch b, DenseGeom g, const float* __restrict__ EV, const float* __restrict__ PH,
                  const float* __restrict__ z, float* __restrict__ dzr, float* __restrict__ rowacc, GuardState* gs,
                  int mode, int cond) {
  extern __shared__ __align__(16) float dsm[];
  if (cond && !(gs->flag & 1)) return;
  phase_rows<KC, LINK>(b, g, EV, PH, z, dzr, rowacc, gs, mode, dsm, blockIdx.x, blockIdx.y);
}

template <int KC, int LINK>
__global__ void __launch_bounds__(128)
dense_cols_kernel(DenseBatch b, DenseGeom g, const float* __restrict__ EV, const float* __restrict__ PH,
                  const float* __restrict__ z, const float* __restrict__ dzr, float* __restrict__ GAp,
                  float* __restrict__ GEV, float* __restrict__ Gph, const GuardState* gs, int with_ga, int rows_per_split) {
  extern __shared__ __align__(16) float dsm[];
  const int r0 = blockIdx.z * rows_per_split;
  phase_cols<KC, LINK>(b, g, EV, PH, z, dzr, GAp, GEV, Gph, gs, with_ga, dsm, blockIdx.x, blockIdx.y, r0,
                       min(b.nrows, r0 + rows_per_split));
}

// ... and the exact-guard slow path of the linear link as TWO conditional launches (they return at once
// unless gs->flag is set, so a step that meets no non-finite entry pays two empty launches of one CTA
// per SM): rows fix = densify -> statistics -> guarded row pass; columns fix = zero GEV / Gphi ->
// guarded column pass.  GA' needs no fix of its own: it is computed from the (fixed) dzr afterwards.
// The phases of one launch are separated by a grid barrier.  These are ordinary launches of at most
// one CTA per SM (a cooperative launch would make every step wait for the whole grid to be
// co-resident, i.e. drain the kernels of the other streams, even when the guard does not fire -- measured
// +70 us per step); the barrier is a monotonic arrival counter in the guard state: all CTAs become
// resident as soon as the kernels running beside them finish (nothing those kernels wait for is
// produced here), and a bounded spin turns a barrier that could not complete into a flagged error
// instead of a hang.
__device__ __forceinline__ bool grid_barrier(GuardState* gs, unsigned nblocks, unsigned phase) {
  __shared__ int ok_s;
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    atomicAdd(&gs->bar, 1u);
    const unsigned target = (phase + 1u) * nblocks;
    int ok = 0;
    for (long long spin = 0; spin < (1ll << 24); ++spin) {          // ~10 s at 0.5 us per poll
      if (*(volatile unsigned*)&gs->bar >= target) { ok = 1; break; }
      __nanosleep(500);
    }
    __threadfence();
    ok_s = ok;
  }
  __syncthreads();
  return ok_s != 0;
}
// last CTA out re-arms the barrier for the next launch
__device__ __forceinline__ void grid_leave(GuardState* gs, unsigned nblocks) {
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    if (atomicAdd(&gs->done, 1u) == nblocks - 1u) {
      gs->bar = 0u;
      gs->done = 0u;
      __threadfence();
    }
  }
}
#define GRID_BARRIER_OR_FAIL(gs, phase)                       \
  do {                                                        \
    if (!grid_barrier(gs, gridDim.x, phase)) {                \
      if (threadIdx.x == 0) atomicOr(&(gs)->flag, 4);         \
      grid_leave(gs, gridDim.x);                              \
      return;                                                 \
    }                                                         \
  } while (0)
struct GuardFixArgs {
  DenseBatch b;
  DenseGeom g;
  const long long* rowptr; const int* cols; const float* vals;      // CSR in table order (|vals|)
  const void* raw; int raw_dtype; const int* rank;                   // or: the raw dense upload (feature order)
  float* xd;
  const float *EV, *PH, *z;
  float *dzr, *rowacc, *GEV, *Gph;
  GuardState* gs;
  int rows_per_split, nsplit;
};

template <int KC>
__global__ void __launch_bounds__(128)
guard_rows_fix_kernel(GuardFixArgs a) {
  extern __shared__ __align__(16) float dsm[];
  if (!(a.gs->flag & 1)) return;                             // uniform over the grid (nobody writes it here)
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, nth = (long long)gridDim.x * blockDim.x;
  if (tid == 0) { a.gs->nbad = 0; a.gs->minkey = ~0ull; }
  if (a.raw) {                       // every element is written: no zero fill needed
    if (a.raw_dtype == SPMF_DENSE_U8) phase_scatter_raw((const unsigned char*)a.raw, a.rank, a.b.nrows, a.b.D, a.xd, tid, nth);
    else if (a.raw_dtype == SPMF_DENSE_U16) phase_scatter_raw((const unsigned short*)a.raw, a.rank, a.b.nrows, a.b.D, a.xd, tid, nth);
    else phase_scatter_raw((const float*)a.raw, a.rank, a.b.nrows, a.b.D, a.xd, tid, nth);
  } else {
    phase_zero(a.xd, (long long)a.b.nrows * a.b.D, tid, nth);
  }
  GRID_BARRIER_OR_FAIL(a.gs, 0u);
  if (!a.raw) phase_scatter(a.rowptr, a.cols, a.vals, a.b.nrows, a.b.D, a.xd, tid >> 5, nth >> 5, threadIdx.x & 31);
  GRID_BARRIER_OR_FAIL(a.gs, 1u);
  DenseBatch b = a.b;
  b.xd = a.xd;
  const int ntile = (b.nrows + a.g.OB - 1) / a.g.OB;
  for (int w = blockIdx.x; w < ntile * a.g.NQ; w += gridDim.x)
    phase_rows<KC, LINK_POIS_LIN>(b, a.g, a.EV, a.PH, a.z, a.dzr, a.rowacc, a.gs, MODE_STATS, dsm, w % ntile, w / ntile);
  GRID_BARRIER_OR_FAIL(a.gs, 2u);
  for (int w = blockIdx.x; w < ntile * a.g.NQ; w += gridDim.x)
    phase_rows<KC, LINK_POIS_LIN>(b, a.g, a.EV, a.PH, a.z, a.dzr, a.rowacc, a.gs, MODE_GUARD, dsm, w % ntile, w / ntile);
  grid_leave(a.gs, gridDim.x);
}

template <int KC>
__global__ void __launch_bounds__(128)
guard_cols_fix_kernel(GuardFixArgs a) {
  extern __shared__ __align__(16) float dsm[];
  if (!(a.gs->flag & 1)) return;
  const long long tid = (long long)blockIdx.x * blockDim.x + threadIdx.x, nth = (long long)gridDim.x * blockDim.x;
  phase_zero(a.GEV, (long long)a.g.NQ * a.b.D * a.g.REC, tid, nth);
  phase_zero(a.Gph, (long long)a.g.NQ * a.b.D * a.g.SV, tid, nth);
  GRID_BARRIER_OR_FAIL(a.gs, 0u);
  DenseBatch b = a.b;
  b.xd = a.xd;
  const int nct = (b.D + a.g.OB - 1) / a.g.OB;
  const int total = nct * a.g.NQ * a.nsplit;
  for (int w = blockIdx.x; w < total; w += gridDim.x) {
    const int ct = w % nct, rest = w / nct;
    const int q = rest % a.g.NQ, sp = rest / a.g.NQ;
    const int r0 = sp * a.rows_per_split;
    phase_cols<KC, LINK_POIS_LIN>(b, a.g, a.EV, a.PH, a.z, nullptr, nullptr, a.GEV, a.Gph, a.gs, 0, dsm, ct, q, r0,
                                  min(b.nrows, r0 + a.rows_per_split));
  }
  grid_leave(a.gs, gridDim.x);
}

__global__ void guard_reset_kernel(GuardState* gs, int flag) {
  gs->flag = flag;
  gs->nbad = 0;
  gs->minkey = ~0ull;
  gs->bar = 0u;
  gs->done = 0u;
}

static size_t rows_smem(const DenseGeom& g) {
  return sizeof(float) * ((size_t)kTile * g.REC + (size_t)kTile * g.SV + (size_t)kTile * (g.OB + 1));
}
static size_t cols_smem(const DenseGeom& g, int with_ga) {
  return sizeof(float) * ((size_t)kTile * g.REC * (with_ga ? 2 : 1) + (size_t)kTile * g.OB);
}

}  // namespace spmf

using namespace spmf;

static bool dense_shape_ok(int nrows, int D, int K, int S) {
  return nrows > 0 && D > 0 && K > 0 && K <= SPMF_MAX_K && S > 0;
}

extern "C" {

int spmf_guard_state_bytes(void) { return (int)sizeof(GuardState); }

int spmf_guard_reset(void* gs, int flag, void* stream) {
  if (!gs) return SPMF_ERR_BAD_ARG;
  guard_reset_kernel<<<1, 1, 0, (cudaStream_t)stream>>>((GuardState*)gs, flag);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_guard_decode(const void* gs_host, int* flag, int* nbad, float* min_ll) {
  if (!gs_host) return SPMF_ERR_BAD_ARG;
  const GuardState* g = (const GuardState*)gs_host;
  if (flag) *flag = g->flag;
  if (nbad) *nbad = g->nbad;
  if (min_ll) *min_ll = guard_min_val(g->minkey);      /* the replacement value: min(finite) - 10 */
  return SPMF_OK;
}

int spmf_dense_scatter(const long long* rowptr, const int* cols, const float* vals, int nrows, int D, float* xd,
                       void* stream) {
  if (!rowptr || !cols || !vals || !xd || nrows <= 0 || D <= 0) return SPMF_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const long long n = (long long)nrows * D;
  dense_zero_kernel<<<(unsigned)((n / 4 + 255) / 256 > 4096 ? 4096 : (n / 4 + 255) / 256 + 1), 256, 0, st>>>(xd, n, nullptr, 0);
  dense_scatter_kernel<<<(unsigned)((nrows + 7) / 8), 256, 0, st>>>(rowptr, cols, vals, nrows, D, xd);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_dense_encode(const float* xd, const float* eta_enc, const float* rowsum, float inv_xi, int scale_rows,
                      int nrows, int D, int K, int S, int link, const float* Ap, float* z, void* stream) {
  if (!xd || !rowsum || !Ap || !z || !dense_shape_ok(nrows, D, K, S)) return SPMF_ERR_BAD_ARG;
  if ((link & 1) && !eta_enc) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  DenseBatch b{xd, rowsum, nullptr, eta_enc, inv_xi, scale_rows, nrows, D};
  cudaStream_t st = (cudaStream_t)stream;
#define CALL_L(KC, L)                                                                             \
  {                                                                                               \
    const DenseGeom g = dense_geom<KC>(KP, SV, NQ);                                               \
    const size_t sm = sizeof(float) * ((size_t)kTile * g.REC + (size_t)kTile * (g.OB + 1));       \
    int rc = set_smem(dense_encode_kernel<KC, L>, sm);                                            \
    if (rc) return rc;                                                                            \
    dense_encode_kernel<KC, L><<<dim3((nrows + g.OB - 1) / g.OB, NQ), 128, sm, st>>>(b, g, Ap, z); \
  }
#define CALL_K(KC) DENSE_LINK(KC, link, CALL_L)
  DENSE_KC(KP, CALL_K);
#undef CALL_K
#undef CALL_L
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_dense_rows(const float* xd, const float* rowsum, const float* lgam, float inv_xi, int scale_rows, int nrows,
                    int D, int K, int S, int link, int mode, int conditional, const float* EV, const float* PH,
                    const float* z, float* dzr, float* rowacc, void* gs, void* stream) {
  if (!xd || !rowsum || !lgam || !EV || !PH || !z || !dzr || !rowacc || !gs || !dense_shape_ok(nrows, D, K, S))
    return SPMF_ERR_BAD_ARG;
  if (mode < SPMF_DENSE_OPTIMISTIC || mode > SPMF_DENSE_GUARDED) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  DenseBatch b{xd, rowsum, lgam, nullptr, inv_xi, scale_rows, nrows, D};
  cudaStream_t st = (cudaStream_t)stream;
#define CALL_L(KC, L)                                                                                     \
  {                                                                                                       \
    const DenseGeom g = dense_geom<KC>(KP, SV, NQ);                                                       \
    const size_t sm = rows_smem(g);                                                                       \
    int rc = set_smem(dense_rows_kernel<KC, L>, sm);                                                      \
    if (rc) return rc;                                                                                    \
    dense_rows_kernel<KC, L><<<dim3((nrows + g.OB - 1) / g.OB, NQ), 128, sm, st>>>(b, g, EV, PH, z, dzr,   \
                                                                                   rowacc, (GuardState*)gs, \
                                                                                   mode, conditional);     \
  }
#define CALL_K(KC) DENSE_LINK(KC, link, CALL_L)
  DENSE_KC(KP, CALL_K);
#undef CALL_K
#undef CALL_L
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_dense_cols(const float* xd, const float* eta_enc, int nrows, int D, int K, int S, int link, int with_ga,
                    const float* z, const float* dzr, const float* EV, const float* PH, float* GAp, float* GEV,
                    float* Gph, const void* gs, void* stream) {
  if (!xd || !z || !EV || !PH || !GEV || !Gph || !dense_shape_ok(nrows, D, K, S)) return SPMF_ERR_BAD_ARG;
  if (with_ga && (!dzr || !GAp)) return SPMF_ERR_BAD_ARG;
  if ((link & 1) && !eta_enc) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  DenseBatch b{xd, nullptr, nullptr, eta_enc, 1.f, 0, nrows, D};
  cudaStream_t st = (cudaStream_t)stream;
#define CALL_L(KC, L)                                                                                       \
  {                                                                                                         \
    const DenseGeom g = dense_geom<KC>(KP, SV, NQ);                                                         \
    const size_t sm = cols_smem(g, with_ga);                                                                \
    int rc = set_smem(dense_cols_kernel<KC, L>, sm);                                                        \
    if (rc) return rc;                                                                                      \
    const int nct = (D + g.OB - 1) / g.OB;                                                                  \
    int nsplit = (4 * 148 + nct * NQ - 1) / (nct * NQ);                                                     \
    const int maxsplit = (nrows + 4 * kTile - 1) / (4 * kTile);                                             \
    if (nsplit > maxsplit) nsplit = maxsplit;                                                               \
    if (nsplit < 1) nsplit = 1;                                                                             \
    const int per = ((nrows + nsplit - 1) / nsplit + kTile - 1) / kTile * kTile;                            \
    nsplit = (nrows + per - 1) / per;                                                                       \
    dense_cols_kernel<KC, L><<<dim3(nct, NQ, nsplit), 128, sm, st>>>(b, g, EV, PH, z, dzr, GAp, GEV, Gph,    \
                                                                     (const GuardState*)gs, with_ga, per);   \
  }
#define CALL_K(KC) DENSE_LINK(KC, link, CALL_L)
  DENSE_KC(KP, CALL_K);
#undef CALL_K
#undef CALL_L
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

}  // extern "C"

// Conditional exact-guard launches of the linear link (see guard_rows_fix_kernel).  `xd` is scratch of
// nrows*D floats, touched only when the guard fires.
template <int KC, typename Kern>
static int launch_fix(Kern kern, GuardFixArgs& a, size_t sm, cudaStream_t st) {
  static size_t cached_sm = ~(size_t)0;          // per instantiation: set the shared-memory attribute once per size
  static int cached_grid = 0;
  if (cached_sm != sm) {
    int rc = set_smem(kern, sm);
    if (rc) return rc;
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (sms < 1) return SPMF_ERR_UNSUPPORTED;
    cached_grid = sms;                           // one CTA per SM: always able to become co-resident
    cached_sm = sm;
  }
  kern<<<cached_grid, 128, sm, st>>>(a);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? SPMF_OK : (int)e;
}

extern "C" {

static int guard_rows_fix_impl(const long long* rowptr, const int* cols, const float* vals, const void* raw,
                               int raw_dtype, const int* rank, const float* rowsum, const float* lgam, float inv_xi,
                               int scale_rows, int nrows, int D, int K, int S, const float* EV, const float* PH,
                               const float* z, float* dzr, float* rowacc, float* xd, void* gs, void* stream);

int spmf_guard_rows_fix(const long long* rowptr, const int* cols, const float* vals, const float* rowsum,
                        const float* lgam, float inv_xi, int scale_rows, int nrows, int D, int K, int S,
                        const float* EV, const float* PH, const float* z, float* dzr, float* rowacc, float* xd,
                        void* gs, void* stream) {
  if (!rowptr || !cols || !vals) return SPMF_ERR_BAD_ARG;
  return guard_rows_fix_impl(rowptr, cols, vals, nullptr, 0, nullptr, rowsum, lgam, inv_xi, scale_rows, nrows, D, K, S,
                             EV, PH, z, dzr, rowacc, xd, gs, stream);
}

int spmf_guard_rows_fix_dense(const void* raw, int raw_dtype, const int* rank, const float* rowsum, const float* lgam,
                              float inv_xi, int scale_rows, int nrows, int D, int K, int S, const float* EV,
                              const float* PH, const float* z, float* dzr, float* rowacc, float* xd, void* gs,
                              void* stream) {
  if (!raw || (raw_dtype != SPMF_DENSE_U8 && raw_dtype != SPMF_DENSE_U16 && raw_dtype != SPMF_DENSE_F32))
    return SPMF_ERR_BAD_ARG;
  return guard_rows_fix_impl(nullptr, nullptr, nullptr, raw, raw_dtype, rank, rowsum, lgam, inv_xi, scale_rows, nrows,
                             D, K, S, EV, PH, z, dzr, rowacc, xd, gs, stream);
}

static int guard_rows_fix_impl(const long long* rowptr, const int* cols, const float* vals, const void* raw,
                               int raw_dtype, const int* rank, const float* rowsum, const float* lgam, float inv_xi,
                               int scale_rows, int nrows, int D, int K, int S, const float* EV, const float* PH,
                               const float* z, float* dzr, float* rowacc, float* xd, void* gs, void* stream) {
  if (false || !rowsum || !lgam || !EV || !PH || !z || !dzr || !rowacc || !xd || !gs ||
      !dense_shape_ok(nrows, D, K, S))
    return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  GuardFixArgs a{};
  a.b = DenseBatch{xd, rowsum, lgam, nullptr, inv_xi, scale_rows, nrows, D};
  a.rowptr = rowptr; a.cols = cols; a.vals = vals; a.xd = xd;
  a.raw = raw; a.raw_dtype = raw_dtype; a.rank = rank;
  a.EV = EV; a.PH = PH; a.z = z; a.dzr = dzr; a.rowacc = rowacc; a.gs = (GuardState*)gs;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = SPMF_OK;
#define CALL_K(KC)                                                    \
  {                                                                   \
    a.g = dense_geom<KC>(KP, SV, NQ);                                 \
    rc = launch_fix<KC>(guard_rows_fix_kernel<KC>, a, rows_smem(a.g), st); \
  }
  DENSE_KC(KP, CALL_K);
#undef CALL_K
  return rc;
}

int spmf_guard_cols_fix(int nrows, int D, int K, int S, const float* EV, const float* PH, const float* z,
                        float* GEV, float* Gph, const float* xd, void* gs, void* stream) {
  if (!EV || !PH || !z || !GEV || !Gph || !xd || !gs || !dense_shape_ok(nrows, D, K, S)) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  GuardFixArgs a{};
  a.b = DenseBatch{xd, nullptr, nullptr, nullptr, 1.f, 0, nrows, D};
  a.xd = const_cast<float*>(xd);
  a.EV = EV; a.PH = PH; a.z = z; a.GEV = GEV; a.Gph = Gph; a.gs = (GuardState*)gs;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = SPMF_OK;
#define CALL_K(KC)                                                                   \
  {                                                                                  \
    a.g = dense_geom<KC>(KP, SV, NQ);                                                \
    const int nct = (D + a.g.OB - 1) / a.g.OB;                                       \
    int nsplit = (4 * 148 + nct * NQ - 1) / (nct * NQ);                              \
    const int maxsplit = (nrows + 4 * kTile - 1) / (4 * kTile);                      \
    if (nsplit > maxsplit) nsplit = maxsplit;                                        \
    if (nsplit < 1) nsplit = 1;                                                      \
    a.rows_per_split = ((nrows + nsplit - 1) / nsplit + kTile - 1) / kTile * kTile;  \
    a.nsplit = (nrows + a.rows_per_split - 1) / a.rows_per_split;                    \
    rc = launch_fix<KC>(guard_cols_fix_kernel<KC>, a, cols_smem(a.g, 0), st);        \
  }
  DENSE_KC(KP, CALL_K);
#undef CALL_K
  return rc;
}

}  // extern "C"
