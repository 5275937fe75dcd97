// Data term of the ADVI step on sparse (CSR + CSC) count batches, sm_100a.
//
// Never materialises the (S,B,D) rate matrix of the reference (poisson.py:174-184).  Per nonzero:
//   row pass    (CSR, row-owned outputs):  z_b = r_b sum_d x A'_d ;  lambda = z_b.EV_d + phi_d ;
//               x log lambda ;  dz_b = sum_d (x/lambda) EV_d - vsum - z_b
//   column pass (CSC, column-owned outputs, recomputes lambda):  GEV_d = sum_b (x/lambda) z_b ;
//               Gphi_d = sum_b x/lambda ;  GA'_d = sum_b x r_b dz_b
// The -sum(rate) part of the Poisson log-likelihood is closed form (SURVEY.md 3.4) and handled
// by vsum / zcolsum / phisum, O(BK + KD).
//
// Thread mapping: see `Map` below and spmf_record.cuh -- a slot of LPN = SV*RG lanes owns one
// nonzero at a time and gathers its record with VPL coalesced vector loads; every lane holds up to
// 16 latent dims of one draw, so the k-contraction is in-lane FMAs plus log2(RG) shuffle steps.
#include <cuda_runtime.h>
#include <stdlib.h>
#include <stdint.h>

#include "../../include/spmf_b200.h"
#include "spmf_record.cuh"
#include "spmf_umma_layout.cuh"

namespace spmf {

#define SPMF_CHECK_LAUNCH()                      \
  do {                                           \
    cudaError_t e__ = cudaGetLastError();        \
    if (e__ != cudaSuccess) return (int)e__;     \
  } while (0)

// ---- thread mapping shared by the row and column passes -------------------------------------
// Operand records are [SV][KP] floats (k innermost).  A "slot" of LPN lanes owns one nonzero at a
// time: lane_in = s*RG + kg holds, for draw s, the k-vectors nv = i*RG + kg (i < VPL), each VW wide.
// The k-contraction is VW*VPL FMAs in-lane followed by a butterfly over the RG lanes of draw s.
template <int KP, int SV>
struct Map {
  static constexpr int VW = KP < 4 ? KP : 4;            // floats per vector load (over k)
  static constexpr int NV = KP / VW;                     // k-vectors per draw
  static constexpr int VPL = NV < 4 ? NV : 4;            // vectors per lane (<= 16 latent dims)
  static constexpr int RG = NV / VPL;                    // lanes sharing one draw
  static constexpr int LPN = SV * RG;                    // lanes per nonzero slot (<= 32)
  static_assert(LPN <= 32, "a nonzero slot must fit in one warp (REC = SV*KP <= 512)");
  static constexpr int REC = SV * KP;                    // floats per record
  static constexpr int THREADS = 128;
  static constexpr int NSLOT = THREADS / LPN;            // slots per CTA
  static constexpr int SPW = 32 / LPN;                   // slots per warp
  // float offset of vector i of lane (s,kg) inside a record -- see spmf_record.cuh
  __device__ static __forceinline__ int off(int i, int s, int kg) { return ((i * SV + s) * RG + kg) * VW; }
};

template <int VW>
__device__ __forceinline__ void ldv(float (&r)[VW], const float* __restrict__ p) {
  if constexpr (VW == 4) {
    float4 t = __ldg(reinterpret_cast<const float4*>(p));
    r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w;
  } else if constexpr (VW == 2) {
    float2 t = __ldg(reinterpret_cast<const float2*>(p));
    r[0] = t.x; r[1] = t.y;
  } else {
    r[0] = __ldg(p);
  }
}
template <int VW>
__device__ __forceinline__ void ldv_s(float (&r)[VW], const float* p) {   // shared / generic
  if constexpr (VW == 4) {
    float4 t = *reinterpret_cast<const float4*>(p);
    r[0] = t.x; r[1] = t.y; r[2] = t.z; r[3] = t.w;
  } else if constexpr (VW == 2) {
    float2 t = *reinterpret_cast<const float2*>(p);
    r[0] = t.x; r[1] = t.y;
  } else {
    r[0] = *p;
  }
}
template <int VW>
__device__ __forceinline__ void stv(float* p, const float (&r)[VW]) {
  if constexpr (VW == 4) {
    *reinterpret_cast<float4*>(p) = make_float4(r[0], r[1], r[2], r[3]);
  } else if constexpr (VW == 2) {
    *reinterpret_cast<float2*>(p) = make_float2(r[0], r[1]);
  } else {
    p[0] = r[0];
  }
}

template <int RG>
__device__ __forceinline__ float group_sum(float v, unsigned mask) {
#pragma unroll
  for (int o = RG / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o);
  return v;
}

// sum over the slots of a warp (lanes with equal position inside their slot); every lane of the
// warp must call it.  The xor butterfly is symmetric, so all lanes end with identical bits.
template <int LPN>
__device__ __forceinline__ float warp_slot_sum(float v) {
#pragma unroll
  for (int o = LPN; o < 32; o <<= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <int LPN>
__device__ __forceinline__ unsigned slot_mask(int lane) {
  if constexpr (LPN == 32) return 0xffffffffu;
  else return ((1u << LPN) - 1u) << ((lane / LPN) * LPN);
}

// ------------------------------------------------------------------ row pass
// One CTA per row, NSLOT slots striding over the row's nonzeros; slot partials meet in shared
// memory.  z stays in registers between the two sweeps; the rate matrix is never written.
// Hot loops use 32-bit row-local indices, U nonzeros per slot in flight, and fetch the next
// batch's (col,val) pairs while the current records are gathered.

// rate guard (poisson.py:606-616): an entry whose rate is not a positive finite number has a
// non-finite log-likelihood; it is dropped from value and gradient and counted.
__device__ __forceinline__ bool rate_ok(float lam) { return lam > 0.f && lam <= 3.402823466e38f; }
// single-MUFU log2 / reciprocal (flush-to-zero forms: no subnormal fix-up code in the hot loop;
// a rate is a sum of positive terms >= phi and never subnormal)
__device__ __forceinline__ float fast_lg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float fast_rcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// U consecutive (col,val) pairs as one vector load each (U = 4: 16 B, U = 2: 8 B; p aligned)
template <int U>
__device__ __forceinline__ void ld_idx(const int* __restrict__ pc, const float* __restrict__ pv,
                                       int (&d)[U], float (&x)[U]) {
  if constexpr (U == 4) {
    const int4 c = __ldg(reinterpret_cast<const int4*>(pc));
    const float4 v = __ldg(reinterpret_cast<const float4*>(pv));
    d[0] = c.x; d[1] = c.y; d[2] = c.z; d[3] = c.w;
    x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
  } else {
    const int2 c = __ldg(reinterpret_cast<const int2*>(pc));
    const float2 v = __ldg(reinterpret_cast<const float2*>(pv));
    d[0] = c.x; d[1] = c.y;
    x[0] = v.x; x[1] = v.y;
  }
}

// MODE 0: training row pass.  MODE 1: encode only (z).
// MODE 3: cold part of the tile-hybrid step -- the hot-column block of the encode product already sits
// in z (tcgen05 GEMM, spmf_umma.cu); both sweeps visit only the entries the tensor cores do not cover
// (stored after rowmid[row], positive values; the tcgen05 tile kernel, spmf_hot_tile.cu, owns the
// others) and dzr / rowacc receive RAW partial sums (un-scaled sum w.EV, sum x log lambda,
// #non-finite) that spmf_rows_finish completes.
constexpr int kRowsTrain = 0, kRowsEncode = 1, kRowsCold = 3;

template <int KP, int SV, int MODE>
__device__ __forceinline__ void
csr_rows_body(const long long* __restrict__ rowptr, const int* __restrict__ cols,
              const float* __restrict__ vals, const float* __restrict__ rowsum,
              const float* __restrict__ lgam, float inv_xi, int scale_rows, int nrows, int D,
              const float* __restrict__ Ap, const float* __restrict__ EV,
              const float* __restrict__ PH, const double* __restrict__ vsum,
              float* __restrict__ z, float* __restrict__ dzr, float* __restrict__ rowacc,
              const int* __restrict__ rowmid, int* __restrict__ gflag) {
  constexpr bool ENCODE_ONLY = (MODE == kRowsEncode);
  constexpr bool COLD = (MODE == kRowsCold);
  using M = Map<KP, SV>;
  constexpr int VW = M::VW, LPN = M::LPN, RG = M::RG, VPL = M::VPL, REC = M::REC, NSLOT = M::NSLOT;
  constexpr int U = VPL >= 4 ? 2 : 4;
  constexpr int NWARP = 4;
  __shared__ __align__(16) float part[NWARP * REC];
  __shared__ float sc[NWARP][SV][2];
  const int lane = threadIdx.x & 31;
  const int slot = threadIdx.x / LPN;
  const int li = threadIdx.x % LPN;
  const int s = li / RG, kg = li % RG;
  const int row = blockIdx.x, q = blockIdx.y;
  const unsigned gmask = slot_mask<LPN>(lane);
  int off[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) off[i] = M::off(i, s, kg);

  // Row-local index space.  The nonzero stream is consumed in aligned groups of U (one 16-byte
  // load for U columns, one for U values, shared by the whole slot): `head` elements up to the
  // first aligned position, `ng` full groups dealt round-robin to the slots, then a tail; head and
  // tail (< 2U elements) go through a scalar path on the last slot.
  struct Range {
    int head, ng, my_groups, n_extra;
    const int* gc; const float* gv; const int* rc; const float* rv;
    __device__ __forceinline__ int extra_index(int e) const { return e < head ? e : e + ng * U; }
  };
  auto make_range = [&](long long jstart, int cnt) {
    Range R;
    R.head = min(cnt, (int)((U - (jstart & (U - 1))) & (U - 1)));
    R.ng = (cnt - R.head) / U;
    R.gc = cols + jstart + R.head;   // aligned group base
    R.gv = vals + jstart + R.head;
    R.rc = cols + jstart;
    R.rv = vals + jstart;
    R.my_groups = slot < R.ng ? (R.ng - slot + NSLOT - 1) / NSLOT : 0;
    R.n_extra = (slot == NSLOT - 1) ? cnt - R.ng * U : 0;   // [0,head) U [head + ng*U, cnt)
    return R;
  };
  const long long j0 = rowptr[row];
  const int n = (int)(rowptr[row + 1] - j0);
  const int mid = COLD ? rowmid[row] : 0;            // both sweeps start here in the cold mode
  const Range R = make_range(j0 + mid, n - mid);
  const float r = scale_rows ? rowsum[row] * inv_xi : 1.f;   // poisson.py:644-649

  // ---- z = r * sum_d x A'_d          (poisson.py:640-643 with 1/eta folded into A')
  const float* Apl = Ap + (size_t)q * D * REC;
  float zz[VPL][VW];
#pragma unroll
  for (int i = 0; i < VPL; ++i)
#pragma unroll
    for (int w = 0; w < VW; ++w) zz[i][w] = 0.f;
  {
    int dcur[U];
    float xcur[U];
    if (R.my_groups > 0) ld_idx<U>(R.gc + slot * U, R.gv + slot * U, dcur, xcur);
    for (int b = 0; b < R.my_groups; ++b) {
      float a[U][VPL][VW];
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int i = 0; i < VPL; ++i) ldv<VW>(a[u][i], Apl + (unsigned)dcur[u] * REC + off[i]);
      const int gn = slot + min(b + 1, R.my_groups - 1) * NSLOT;   // last iteration re-reads its own group
      int dn[U];
      float xn[U];
      ld_idx<U>(R.gc + gn * U, R.gv + gn * U, dn, xn);
#pragma unroll
      for (int u = 0; u < U; ++u) {
#pragma unroll
        for (int i = 0; i < VPL; ++i)
#pragma unroll
          for (int w = 0; w < VW; ++w) zz[i][w] = fmaf(xcur[u], a[u][i][w], zz[i][w]);
        dcur[u] = dn[u];
        xcur[u] = xn[u];
      }
    }
    for (int e = 0; e < R.n_extra; ++e) {
      const int t = R.extra_index(e);
      const int d = __ldg(R.rc + t);
      const float x = __ldg(R.rv + t);
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        float a[VW];
        ldv<VW>(a, Apl + (unsigned)d * REC + off[i]);
#pragma unroll
        for (int w = 0; w < VW; ++w) zz[i][w] = fmaf(x, a[w], zz[i][w]);
      }
    }
  }
  // slot partials -> row total: shuffle across the slots of a warp, then the 4 warps through smem
  const int warp = threadIdx.x >> 5;
  const bool warp_lead = (lane < LPN);            // slot 0 of this warp
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
#pragma unroll
    for (int w = 0; w < VW; ++w) zz[i][w] = warp_slot_sum<LPN>(zz[i][w]);
    if (warp_lead) stv<VW>(part + warp * REC + off[i], zz[i]);
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
#pragma unroll
    for (int w = 0; w < VW; ++w) zz[i][w] = 0.f;
#pragma unroll
    for (int t = 0; t < NWARP; ++t) {       // fixed order: every slot ends with the same bits
      float a[VW];
      ldv_s<VW>(a, part + t * REC + off[i]);
#pragma unroll
      for (int w = 0; w < VW; ++w) zz[i][w] += a[w];
    }
  }
  float* zq = z + ((size_t)q * nrows + row) * REC;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    if constexpr (COLD) {                   // hot-column block of x.A' from the tensor-core GEMM
      float a[VW];
      ldv_s<VW>(a, zq + off[i]);
#pragma unroll
      for (int w = 0; w < VW; ++w) zz[i][w] += a[w];
    }
#pragma unroll
    for (int w = 0; w < VW; ++w) zz[i][w] *= r;
  }
  if constexpr (COLD) __syncthreads();      // every slot has read the GEMM block before slot 0 overwrites it
#pragma unroll
  for (int i = 0; i < VPL; ++i)
    if (slot == 0) stv<VW>(zq + off[i], zz[i]);
  if constexpr (ENCODE_ONLY) return;

  // ---- lambda at the nonzeros, x log lambda, dz      (poisson.py:174-184)
  const float* EVl = EV + (size_t)q * D * REC;
  const float* PHl = PH + (size_t)q * D * SV + s;
  float dz[VPL][VW];
  float xlog2 = 0.f;     // sum x log2(lambda); scaled by ln 2 at the end
  int bad = 0;
#pragma unroll
  for (int i = 0; i < VPL; ++i)
#pragma unroll
    for (int w = 0; w < VW; ++w) dz[i][w] = 0.f;
  {
    int dcur[U];
    float xcur[U];
    if (R.my_groups > 0) ld_idx<U>(R.gc + slot * U, R.gv + slot * U, dcur, xcur);
    for (int b = 0; b < R.my_groups; ++b) {
      float e[U][VPL][VW], ph[U], p[U];
#pragma unroll
      for (int u = 0; u < U; ++u) {
#pragma unroll
        for (int i = 0; i < VPL; ++i) ldv<VW>(e[u][i], EVl + (unsigned)dcur[u] * REC + off[i]);
        ph[u] = __ldg(PHl + (unsigned)dcur[u] * SV);
      }
      const int gn = slot + min(b + 1, R.my_groups - 1) * NSLOT;
      int dn[U];
      float xn[U];
      ld_idx<U>(R.gc + gn * U, R.gv + gn * U, dn, xn);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        p[u] = 0.f;
#pragma unroll
        for (int i = 0; i < VPL; ++i)
#pragma unroll
          for (int w = 0; w < VW; ++w) p[u] = fmaf(zz[i][w], e[u][i][w], p[u]);
      }
#pragma unroll
      for (int u = 0; u < U; ++u) p[u] = group_sum<RG>(p[u], gmask);
#pragma unroll
      for (int u = 0; u < U; ++u) {
        const float lam = p[u] + ph[u];                        // poisson.py:177
        const bool ok = rate_ok(lam);
        const float lg = ok ? fast_lg2(lam) : 0.f;
        const float gq = ok ? xcur[u] * fast_rcp(lam) : 0.f;
        bad += ok ? 0 : 1;
        xlog2 = fmaf(xcur[u], lg, xlog2);
#pragma unroll
        for (int i = 0; i < VPL; ++i)
#pragma unroll
          for (int w = 0; w < VW; ++w) dz[i][w] = fmaf(gq, e[u][i][w], dz[i][w]);
        dcur[u] = dn[u];
        xcur[u] = xn[u];
      }
    }
    for (int ex = 0; ex < R.n_extra; ++ex) {
      const int t = R.extra_index(ex);
      const int d = __ldg(R.rc + t);
      const float x = __ldg(R.rv + t);
      float e[VPL][VW];
      float p = 0.f;
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        ldv<VW>(e[i], EVl + (unsigned)d * REC + off[i]);
#pragma unroll
        for (int w = 0; w < VW; ++w) p = fmaf(zz[i][w], e[i][w], p);
      }
      const float lam = group_sum<RG>(p, gmask) + __ldg(PHl + (unsigned)d * SV);
      const bool ok = rate_ok(lam);
      const float lg = ok ? fast_lg2(lam) : 0.f;
      const float gq = ok ? x * fast_rcp(lam) : 0.f;
      bad += ok ? 0 : 1;
      xlog2 = fmaf(x, lg, xlog2);
#pragma unroll
      for (int i = 0; i < VPL; ++i)
#pragma unroll
        for (int w = 0; w < VW; ++w) dz[i][w] = fmaf(gq, e[i][w], dz[i][w]);
    }
  }
  float xlog = xlog2 * 0.6931471805599453f;
  float fbad = (float)bad;
  __syncthreads();   // everyone is done reading `part` (z partials)
  xlog = warp_slot_sum<LPN>(xlog);
  fbad = warp_slot_sum<LPN>(fbad);
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
#pragma unroll
    for (int w = 0; w < VW; ++w) dz[i][w] = warp_slot_sum<LPN>(dz[i][w]);
    if (warp_lead) stv<VW>(part + warp * REC + off[i], dz[i]);
  }
  if (warp_lead && kg == 0) { sc[warp][s][0] = xlog; sc[warp][s][1] = fbad; }
  __syncthreads();
  if (slot != 0) return;
  xlog = 0.f; fbad = 0.f;
#pragma unroll
  for (int t = 0; t < NWARP; ++t) { xlog += sc[t][s][0]; fbad += sc[t][s][1]; }
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
#pragma unroll
    for (int w = 0; w < VW; ++w) dz[i][w] = 0.f;
#pragma unroll
    for (int t = 0; t < NWARP; ++t) {
      float a[VW];
      ldv_s<VW>(a, part + t * REC + off[i]);
#pragma unroll
      for (int w = 0; w < VW; ++w) dz[i][w] += a[w];
    }
  }
  float* dq = dzr + ((size_t)q * nrows + row) * REC;
  if constexpr (COLD) {       // raw partial sums; spmf_hot_tile adds its share, spmf_rows_finish completes
#pragma unroll
    for (int i = 0; i < VPL; ++i) stv<VW>(dq + off[i], dz[i]);
    if (kg == 0) {
      float* ra = rowacc + ((size_t)q * nrows + row) * 4 * SV;
      ra[0 * SV + s] = xlog;
      ra[1 * SV + s] = 0.f;
      ra[2 * SV + s] = 0.f;
      ra[3 * SV + s] = fbad;
      if (gflag && fbad > 0.f) atomicOr(gflag, 1);     // exact guard (poisson.py:606-616) takes over this step
    }
    return;
  }
  // ---- closed-form parts and per-row scalars (slot 0 only from here)
  const double* vsq = vsum + (size_t)q * REC;
  float zv = 0.f, z2 = 0.f;
#pragma unroll
  for (int i = 0; i < VPL; ++i) {
    float o[VW];
#pragma unroll
    for (int w = 0; w < VW; ++w) {
      const float vs = (float)vsq[off[i] + w];
      zv = fmaf(zz[i][w], vs, zv);
      z2 = fmaf(zz[i][w], zz[i][w], z2);
      o[w] = r * (dz[i][w] - vs - zz[i][w]);   // dL/dz includes the HalfNormal(1) z prior (:599-604)
    }
    stv<VW>(dq + off[i], o);
  }
  zv = group_sum<RG>(zv, gmask);
  z2 = group_sum<RG>(z2, gmask);
  if (kg == 0) {
    float* ra = rowacc + ((size_t)q * nrows + row) * 4 * SV;
    ra[0 * SV + s] = xlog - lgam[row];
    ra[1 * SV + s] = zv;
    ra[2 * SV + s] = z2;
    ra[3 * SV + s] = fbad;
    // a non-finite entry among the nonzeros, or a non-finite closed-form sum(rate) of this row (some
    // zero entry's rate is not finite): the exact guard of poisson.py:606-616 takes over this step
    if (gflag && (fbad > 0.f || !(fabsf(zv) <= 3.402823466e38f))) atomicOr(gflag, 1);
  }
}

#define SPMF_ROWS_PARAMS                                                                                        \
  const long long *__restrict__ rowptr, const int *__restrict__ cols, const float *__restrict__ vals,          \
      const float *__restrict__ rowsum, const float *__restrict__ lgam, float inv_xi, int scale_rows, int nrows, \
      int D, const float *__restrict__ Ap, const float *__restrict__ EV, const float *__restrict__ PH,          \
      const double *__restrict__ vsum, float *__restrict__ z, float *__restrict__ dzr,                          \
      float *__restrict__ rowacc, const int *__restrict__ rowmid, int *__restrict__ gflag
#define SPMF_ROWS_ARGS \
  rowptr, cols, vals, rowsum, lgam, inv_xi, scale_rows, nrows, D, Ap, EV, PH, vsum, z, dzr, rowacc, rowmid, gflag

template <int KP, int SV, int MODE>
__global__ void __launch_bounds__(128) csr_rows_kernel(SPMF_ROWS_PARAMS) {
  csr_rows_body<KP, SV, MODE>(SPMF_ROWS_ARGS);
}
// the cold pass of the tile-hybrid step at 128-float records: capped at 96 registers for 5 CTAs per SM
// (the kernel is bound by the L1 data pipe and latency; 4 -> 5 resident CTAs measured -6 %, 6 with
// spills +10 %)
template <int KP, int SV>
__global__ void __launch_bounds__(128, 5) csr_rows_cold5_kernel(SPMF_ROWS_PARAMS) {
  csr_rows_body<KP, SV, kRowsCold>(SPMF_ROWS_ARGS);
}

// ------------------------------------------------------------------ column pass
// Each slot walks a fixed-length slice of the CSC nonzero stream (perfect balance, coalesced
// streaming), keeps the current column's EV record and accumulators in registers and flushes with
// atomics when the column changes (only columns that straddle slices are contended).
constexpr int kSliceLen = 256;

// `nnz_bound` sizes the grid; the actual count is colptr[D] (known on the device only).
template <int KP, int SV>
__global__ void __launch_bounds__(128, KP > 128 ? 3 : 4)
csc_cols_kernel(const int* __restrict__ colptr, const int* __restrict__ rows,
                const float* __restrict__ vals, int nnz_bound, int nrows, int D,
                const float* __restrict__ z, const float* __restrict__ dzr,
                const float* __restrict__ EV, const float* __restrict__ PH,
                float* __restrict__ GAp, float* __restrict__ GEV, float* __restrict__ Gphi, int slice_len) {
  using M = Map<KP, SV>;
  constexpr int VW = M::VW, LPN = M::LPN, RG = M::RG, VPL = M::VPL, REC = M::REC, NSLOT = M::NSLOT;
  constexpr int U = VPL >= 4 ? 2 : 4;
  const int lane = threadIdx.x & 31;
  const int slot = threadIdx.x / LPN;
  const int li = threadIdx.x % LPN;
  const int s = li / RG, kg = li % RG;
  const int q = blockIdx.y;
  const unsigned gmask = slot_mask<LPN>(lane);
  const int slice = blockIdx.x * NSLOT + slot;
  const int j0 = slice * slice_len;          // slice_len is a multiple of 4: 16-byte index loads stay aligned
  const int nnz = min(nnz_bound, __ldg(colptr + D));
  if (j0 >= nnz) return;
  const int j1 = min(j0 + slice_len, nnz);
  int off[VPL];
#pragma unroll
  for (int i = 0; i < VPL; ++i) off[i] = M::off(i, s, kg);

  const float* zl = z + (size_t)q * nrows * REC;
  const float* dl = dzr + (size_t)q * nrows * REC;
  const float* EVl = EV + (size_t)q * D * REC;
  const float* PHl = PH + (size_t)q * D * SV + s;
  float* GApq = GAp + (size_t)q * D * REC;
  float* GEVq = GEV + (size_t)q * D * REC;
  float* Gphq = Gphi + (size_t)q * D * SV + s;

  // column containing position j0: largest d with colptr[d] <= j0  (colptr[D] = nnz > j0)
  int lo = 0, hi = D;
  while (hi - lo > 1) {
    int mid = (lo + hi) >> 1;
    if (__ldg(colptr + mid) <= j0) lo = mid; else hi = mid;
  }
  int d = lo;
  int next = __ldg(colptr + d + 1);

  float ev[VPL][VW], aEV[VPL][VW], aAp[VPL][VW], ph, aPh;
  auto load_col = [&](int dd) {
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      ldv<VW>(ev[i], EVl + (unsigned)dd * REC + off[i]);
#pragma unroll
      for (int w = 0; w < VW; ++w) {
        aEV[i][w] = 0.f;
        aAp[i][w] = 0.f;
      }
    }
    ph = __ldg(PHl + (unsigned)dd * SV);
    aPh = 0.f;
  };
  auto flush_col = [&](int dd) {
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      const unsigned o = (unsigned)dd * REC + off[i];
#pragma unroll
      for (int w = 0; w < VW; ++w) {
        atomicAdd(GEVq + o + w, aEV[i][w]);
        atomicAdd(GApq + o + w, aAp[i][w]);
      }
    }
    if (kg == 0) atomicAdd(Gphq + (unsigned)dd * SV, aPh);
  };
  auto one = [&](int j, float x, const float (&zz)[VPL][VW], const float (&dd)[VPL][VW]) {
    if (j >= next) {
      flush_col(d);
      do {
        ++d;
        next = __ldg(colptr + d + 1);
      } while (j >= next);
      load_col(d);
    }
    float p = 0.f;
#pragma unroll
    for (int i = 0; i < VPL; ++i)
#pragma unroll
      for (int w = 0; w < VW; ++w) p = fmaf(zz[i][w], ev[i][w], p);
    const float lam = group_sum<RG>(p, gmask) + ph;
    const float gq = rate_ok(lam) ? x * fast_rcp(lam) : 0.f;    // same entries the row pass dropped
    aPh += gq;
#pragma unroll
    for (int i = 0; i < VPL; ++i)
#pragma unroll
      for (int w = 0; w < VW; ++w) {
        aEV[i][w] = fmaf(gq, zz[i][w], aEV[i][w]);
        aAp[i][w] = fmaf(x, dd[i][w], aAp[i][w]);
      }
  };
  load_col(d);
  const int nfull = (j1 - j0) / U;
  for (int b = 0; b < nfull; ++b) {
    const int jb = j0 + b * U;
    int bb[U];
    float xx[U];
    if constexpr (U == 4) {                       // slices start 256-aligned: 16-byte vector loads
      const int4 b4 = __ldg(reinterpret_cast<const int4*>(rows + jb));
      const float4 x4 = __ldg(reinterpret_cast<const float4*>(vals + jb));
      bb[0] = b4.x; bb[1] = b4.y; bb[2] = b4.z; bb[3] = b4.w;
      xx[0] = x4.x; xx[1] = x4.y; xx[2] = x4.z; xx[3] = x4.w;
    } else {
      const int2 b2 = __ldg(reinterpret_cast<const int2*>(rows + jb));
      const float2 x2 = __ldg(reinterpret_cast<const float2*>(vals + jb));
      bb[0] = b2.x; bb[1] = b2.y;
      xx[0] = x2.x; xx[1] = x2.y;
    }
    float zz[U][VPL][VW], dd[U][VPL][VW];
#pragma unroll
    for (int u = 0; u < U; ++u)
#pragma unroll
      for (int i = 0; i < VPL; ++i) {
        ldv<VW>(zz[u][i], zl + (unsigned)bb[u] * REC + off[i]);
        ldv<VW>(dd[u][i], dl + (unsigned)bb[u] * REC + off[i]);
      }
#pragma unroll
    for (int u = 0; u < U; ++u) one(jb + u, xx[u], zz[u], dd[u]);
  }
  for (int j = j0 + nfull * U; j < j1; ++j) {     // tail of the last slice
    const int b = __ldg(rows + j);
    const float x = __ldg(vals + j);
    float zz[VPL][VW], dd[VPL][VW];
#pragma unroll
    for (int i = 0; i < VPL; ++i) {
      ldv<VW>(zz[i], zl + (unsigned)b * REC + off[i]);
      ldv<VW>(dd[i], dl + (unsigned)b * REC + off[i]);
    }
    one(j, x, zz, dd);
  }
  flush_col(d);
}

// ------------------------------------------------------------------ data-format kernels
// lgamma(x+1) for integer counts x < 64 (almost every entry of a count matrix)
__constant__ float kLgamTab[64] = {0.000000000e+00f, 0.000000000e+00f, 6.931471806e-01f, 1.791759469e+00f, 3.178053830e+00f, 4.787491743e+00f, 6.579251212e+00f, 8.525161361e+00f, 1.060460290e+01f, 1.280182748e+01f, 1.510441257e+01f, 1.750230785e+01f, 1.998721450e+01f, 2.255216385e+01f, 2.519122118e+01f, 2.789927138e+01f, 3.067186011e+01f, 3.350507345e+01f, 3.639544521e+01f, 3.933988419e+01f, 4.233561646e+01f, 4.538013890e+01f, 4.847118135e+01f, 5.160667557e+01f, 5.478472940e+01f, 5.800360522e+01f, 6.126170176e+01f, 6.455753863e+01f, 6.788974314e+01f, 7.125703897e+01f, 7.465823635e+01f, 7.809222355e+01f, 8.155795946e+01f, 8.505446702e+01f, 8.858082754e+01f, 9.213617560e+01f, 9.571969454e+01f, 9.933061245e+01f, 1.029681986e+02f, 1.066317603e+02f, 1.103206397e+02f, 1.140342118e+02f, 1.177718814e+02f, 1.215330815e+02f, 1.253172711e+02f, 1.291239336e+02f, 1.329525750e+02f, 1.368027226e+02f, 1.406739236e+02f, 1.445657439e+02f, 1.484777670e+02f, 1.524095926e+02f, 1.563608363e+02f, 1.603311282e+02f, 1.643201123e+02f, 1.683274454e+02f, 1.723527971e+02f, 1.763958484e+02f, 1.804562914e+02f, 1.845338289e+02f, 1.886281734e+02f, 1.927390473e+02f, 1.968661817e+02f, 2.010093164e+02f};

__device__ __forceinline__ float lgamma1p_count(float x) {
  const int i = (int)x;
  return (x >= 0.f && x < 64.f && (float)i == x) ? kLgamTab[i] : lgammaf(x + 1.f);
}

__global__ void csr_row_consts_kernel(const long long* __restrict__ rowptr,
                                      const float* __restrict__ vals, long long nrows,
                                      float* __restrict__ rowsum, float* __restrict__ lgam) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= nrows) return;
  const long long j0 = rowptr[row], j1 = rowptr[row + 1];
  float s = 0.f, l = 0.f;
  for (long long j = j0 + lane; j < j1; j += 32) {
    const float x = __ldg(vals + j);
    s += x;
    l += lgamma1p_count(x);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    l += __shfl_xor_sync(0xffffffffu, l, o);
  }
  if (lane == 0) { rowsum[row] = s; lgam[row] = l; }
}

__global__ void csr_colstats_kernel(const int* __restrict__ cols, const float* __restrict__ vals,
                                    long long nnz, double* __restrict__ colsum,
                                    float* __restrict__ colnnz) {
  long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; j < nnz; j += stride) {
    const float x = __ldg(vals + j);
    const int d = __ldg(cols + j);
    atomicAdd(colsum + d, (double)x);
    if (x > 0.f) atomicAdd(colnnz + d, 1.0f);   // fp32 counter as poisson.py:126-130
  }
}

// Row r's entries of one part of a partitioned CSR (spmf_hot_split): part 0 = the first rowmid[r]
// entries, part 1 = the rest; rowmid == nullptr = the whole row.
__device__ __forceinline__ void part_range(const long long* __restrict__ rowptr, const int* __restrict__ rowmid,
                                           int part, int row, long long& j0, long long& j1) {
  j0 = rowptr[row];
  j1 = rowptr[row + 1];
  if (rowmid) {
    const long long m = j0 + rowmid[row];
    if (part == 0) j1 = m; else j0 = m;
  }
}

__global__ void count_cols_kernel(const long long* __restrict__ rowptr, const int* __restrict__ rowmid, int part,
                                  const int* __restrict__ cols, int nrows, int* __restrict__ cnt) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= nrows) return;
  long long j0, j1;
  part_range(rowptr, rowmid, part, row, j0, j1);
  for (long long j = j0 + lane; j < j1; j += 32) atomicAdd(cnt + __ldg(cols + j), 1);
}

// ---- block-partitioned transpose (D*4 bytes fit in shared memory) -------------------------------
// The batch's rows are cut into kTrBlocks contiguous ranges of equal nonzero count.  Pass 1: each
// CTA histograms its range's columns in shared memory.  Pass 2: per column, exclusive scan over the
// CTAs.  Pass 3: each CTA scatters its range with shared-memory cursors.  No global atomics, and
// column segments come out ordered by row block.
constexpr int kTrBlocks = 148;
constexpr int kTrThreads = 1024;

__device__ __forceinline__ int tr_row_bound(const long long* __restrict__ rowptr, int nrows, long long target) {
  int lo = 0, hi = nrows;        // first row r with rowptr[r] >= target
  while (lo < hi) {
    int mid = (lo + hi) >> 1;
    if (rowptr[mid] < target) lo = mid + 1; else hi = mid;
  }
  return lo;
}

__global__ void __launch_bounds__(kTrThreads)
csc_block_hist_kernel(const long long* __restrict__ rowptr, const int* __restrict__ rowmid, int part,
                      const int* __restrict__ cols, int nrows, int D, int* __restrict__ blockhist) {
  extern __shared__ int h[];
  for (int d = threadIdx.x; d < D; d += blockDim.x) h[d] = 0;
  __syncthreads();
  const long long base = rowptr[0], nnz = rowptr[nrows] - base;
  const int r0 = tr_row_bound(rowptr, nrows, base + nnz * blockIdx.x / gridDim.x);
  const int r1 = (blockIdx.x + 1 == gridDim.x) ? nrows
                                               : tr_row_bound(rowptr, nrows, base + nnz * (blockIdx.x + 1) / gridDim.x);
  if (!rowmid) {
    const long long j0 = rowptr[r0], j1 = rowptr[r1];
    for (long long j = j0 + threadIdx.x; j < j1; j += blockDim.x) atomicAdd(&h[__ldg(cols + j)], 1);
  } else {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    for (int row = r0 + warp; row < r1; row += nwarp) {
      long long j0, j1;
      part_range(rowptr, rowmid, part, row, j0, j1);
#pragma unroll 4
      for (long long j = j0 + lane; j < j1; j += 32) atomicAdd(&h[__ldcs(cols + j)], 1);   // (loads batched 4 deep)
    }
  }
  __syncthreads();
  int* out = blockhist + (long long)blockIdx.x * D;
  for (int d = threadIdx.x; d < D; d += blockDim.x) out[d] = h[d];
}

__global__ void csc_block_scan_kernel(int* __restrict__ blockhist, int nblocks, int D, int* __restrict__ colcnt) {
  const int d = blockIdx.x * blockDim.x + threadIdx.x;
  if (d >= D) return;
  int run = 0;
  for (int b0 = 0; b0 < nblocks; b0 += 16) {          // 16 independent loads in flight per thread
    int t[16];
#pragma unroll
    for (int i = 0; i < 16; ++i) t[i] = (b0 + i < nblocks) ? blockhist[(long long)(b0 + i) * D + d] : 0;
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (b0 + i < nblocks) blockhist[(long long)(b0 + i) * D + d] = run;
      run += t[i];
    }
  }
  colcnt[d] = run;
}

__global__ void __launch_bounds__(kTrThreads)
csc_block_scatter_kernel(const long long* __restrict__ rowptr, const int* __restrict__ rowmid, int part,
                         const int* __restrict__ cols, const float* __restrict__ vals, int nrows, int D,
                         const int* __restrict__ colptr, const int* __restrict__ blockhist,
                         int* __restrict__ rows_out, float* __restrict__ vals_out) {
  extern __shared__ int cur[];
  const int* bh = blockhist + (long long)blockIdx.x * D;
  for (int d = threadIdx.x; d < D; d += blockDim.x) cur[d] = colptr[d] + bh[d];
  __syncthreads();
  const long long base = rowptr[0], nnz = rowptr[nrows] - base;
  const int r0 = tr_row_bound(rowptr, nrows, base + nnz * blockIdx.x / gridDim.x);
  const int r1 = (blockIdx.x + 1 == gridDim.x) ? nrows
                                               : tr_row_bound(rowptr, nrows, base + nnz * (blockIdx.x + 1) / gridDim.x);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  for (int row = r0 + warp; row < r1; row += nwarp) {
    long long j0, j1;
    part_range(rowptr, rowmid, part, row, j0, j1);
#pragma unroll 4
    for (long long j = j0 + lane; j < j1; j += 32) {
      // (streaming hints: this build runs on the copy stream under the previous step, whose gather kernels
      // live off the L2-resident operand tables)
      const int pos = atomicAdd(&cur[__ldcs(cols + j)], 1);
      __stcs(rows_out + pos, row);
      __stcs(vals_out + pos, fabsf(__ldcs(vals + j)));     // the sign is the hot-split coverage flag
    }
  }
}

// single-block exclusive scan: out[0..n] (n+1 entries), also copies to cursor
__global__ void exscan_int_kernel(const int* __restrict__ in, int n, int* __restrict__ out,
                                  int* __restrict__ cursor) {
  __shared__ int warp_tot[32];
  __shared__ int carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int base = 0; base < n; base += blockDim.x) {
    const int i = base + threadIdx.x;
    const int v = i < n ? in[i] : 0;
    int x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      int y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[w] = x;
    __syncthreads();
    if (w == 0) {
      int t = lane < (blockDim.x >> 5) ? warp_tot[lane] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        int y = __shfl_up_sync(0xffffffffu, t, o);
        if (lane >= o) t += y;
      }
      warp_tot[lane] = t;   // inclusive over warps
    }
    __syncthreads();
    const int excl = carry + (w ? warp_tot[w - 1] : 0) + x - v;
    if (i < n) { out[i] = excl; if (cursor) cursor[i] = excl; }
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry = excl + v;
    __syncthreads();
  }
  if (threadIdx.x == 0) { out[n] = carry; if (cursor) cursor[n] = carry; }
}

__global__ void scatter_csc_kernel(const long long* __restrict__ rowptr, const int* __restrict__ rowmid, int part,
                                   const int* __restrict__ cols, const float* __restrict__ vals, int nrows,
                                   int* __restrict__ cursor, int* __restrict__ rows_out,
                                   float* __restrict__ vals_out) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= nrows) return;
  long long j0, j1;
  part_range(rowptr, rowmid, part, row, j0, j1);
  for (long long j = j0 + lane; j < j1; j += 32) {
    const int d = __ldg(cols + j);
    const int pos = atomicAdd(cursor + d, 1);
    rows_out[pos] = row;
    vals_out[pos] = fabsf(__ldg(vals + j));
  }
}

// compact host format -> device CSR arrays: uint16 column ids (D <= 65536) and/or uint16 counts
__global__ void csr_unpack16_kernel(const unsigned short* __restrict__ c16,
                                    const unsigned short* __restrict__ v16, long long nnz,
                                    int* __restrict__ cols, float* __restrict__ vals) {
  long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long stride = (long long)gridDim.x * blockDim.x;
  for (; j < nnz; j += stride) {
    if (c16) cols[j] = (int)c16[j];
    if (v16) vals[j] = (float)v16[j];
  }
}

// 2-byte transfer format of a CSR batch (1 byte per column id + 1 byte per count): per row the stored
// byte of entry j is  col_j - col_{j-1} - 1  (col_{-1} = -1), so a row's column ids are an inclusive prefix
// sum; gaps wider than 256 are bridged on the host by explicit zero-valued entries, counts above 254 are
// sent as the byte 255 and patched from a short (entry index, value) list.  One warp per row.
__global__ void __launch_bounds__(256)
csr_unpack8_kernel(const long long* __restrict__ rowptr, const unsigned char* __restrict__ gaps8,
                   const unsigned char* __restrict__ vals8, int nrows, int* __restrict__ cols,
                   float* __restrict__ vals) {
  const int lane = threadIdx.x & 31;
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= nrows) return;
  const long long j0 = rowptr[row], j1 = rowptr[row + 1];
  int base = -1;                                              // column of the previous entry
  for (long long j = j0; j < j1; j += 32) {
    const long long jj = j + lane;
    int g = jj < j1 ? (int)gaps8[jj] + 1 : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {                        // inclusive warp scan
      const int t = __shfl_up_sync(0xffffffffu, g, o);
      if (lane >= o) g += t;
    }
    if (jj < j1) {
      cols[jj] = base + g;
      vals[jj] = (float)vals8[jj];
    }
    base += __shfl_sync(0xffffffffu, g, 31);
  }
}
__global__ void csr_patch_vals_kernel(const int* __restrict__ idx, const float* __restrict__ val, int n,
                                      float* __restrict__ vals) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) vals[idx[i]] = val[i];
}

__global__ void dense_count_kernel(const float* __restrict__ x, int nrows, int D,
                                   long long* __restrict__ cnt) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= nrows) return;
  int c = 0;
  for (int d = lane; d < D; d += 32) c += (x[(long long)row * D + d] != 0.f);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) c += __shfl_xor_sync(0xffffffffu, c, o);
  if (lane == 0) cnt[row + 1] = c;
  if (row == 0 && lane == 0) cnt[0] = 0;
}

// single-block inclusive scan in place over rowptr[1..n] (int64)
__global__ void incscan_ll_kernel(long long* __restrict__ a, int n) {
  __shared__ long long warp_tot[32];
  __shared__ long long carry;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int base = 0; base < n; base += blockDim.x) {
    const int i = base + threadIdx.x;
    long long x = i < n ? a[1 + i] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      long long y = __shfl_up_sync(0xffffffffu, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) warp_tot[w] = x;
    __syncthreads();
    if (w == 0) {
      long long t = lane < (blockDim.x >> 5) ? warp_tot[lane] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        long long y = __shfl_up_sync(0xffffffffu, t, o);
        if (lane >= o) t += y;
      }
      warp_tot[lane] = t;
    }
    __syncthreads();
    const long long incl = carry + (w ? warp_tot[w - 1] : 0) + x;
    if (i < n) a[1 + i] = incl;
    __syncthreads();
    if (threadIdx.x == blockDim.x - 1) carry = incl;
    __syncthreads();
  }
}

__global__ void dense_fill_kernel(const float* __restrict__ x, int nrows, int D,
                                  const long long* __restrict__ rowptr, int* __restrict__ cols,
                                  float* __restrict__ vals) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= nrows) return;
  long long pos = rowptr[row];
  for (int d0 = 0; d0 < D; d0 += 32) {
    const int d = d0 + lane;
    const float v = d < D ? x[(long long)row * D + d] : 0.f;
    const unsigned m = __ballot_sync(0xffffffffu, v != 0.f);
    if (v != 0.f) {
      const long long o = pos + __popc(m & ((1u << lane) - 1u));
      cols[o] = d;
      vals[o] = v;
    }
    pos += __popc(m);
  }
}

__device__ __forceinline__ bool hot_covered(int r, float x, int H) {   // rank in the block, x > 0 exact in bf16
  return r < H && x > 0.f && __uint_as_float(__float_as_uint(x) & 0xffff0000u) == x;
}

// One CTA per row of the 128-row-padded batch.  STAGED: the row's dense hot vector (Hp bf16) is assembled
// in shared memory and written out as whole 16-byte chunks -- zeros included, so xhot needs no memset and
// the DRAM side sees full chunks instead of 2-byte read-modify-writes; rows >= nrows (tile padding) are
// written as zeros.  !STAGED (very wide hot blocks): direct 2-byte scatter into a pre-zeroed xhot.
constexpr int kSplitThreads = 256, kSplitWarps = kSplitThreads / 32;
constexpr int kSplitStash = 2048;     // (rank, value) pairs per row kept between the two passes

// count of entry e of the 2-byte format: the byte, or (byte 255) its value in the sorted overflow list
__device__ __forceinline__ float u8_count(const unsigned char* __restrict__ vals8, long long e,
                                          const int* __restrict__ ovf_idx, const float* __restrict__ ovf_val, int novf) {
  const unsigned b = __ldcs(vals8 + e);
  if (b != 255u) return (float)b;
  int lo = 0, hi = novf - 1;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(ovf_idx + mid) < (int)e) lo = mid + 1; else hi = mid;
  }
  return (novf > 0 && __ldg(ovf_idx + lo) == (int)e) ? __ldg(ovf_val + lo) : 255.f;
}

// CT / VT: int / float, or unsigned short for the compact upload format (spmf_csr_unpack16 fused in).
// GAPS (CT = VT = unsigned char): the 2-byte format of spmf_csr_unpack8 fused in -- `cols` holds the column
// gaps (a row's column ids are their inclusive prefix sum: warp scans, chained across the warps' pieces),
// `vals` the count bytes with the overflow list beside them; entry indices are relative to rowptr[0].
template <bool STAGED, typename CT, typename VT, bool GAPS = false>
__global__ void __launch_bounds__(kSplitThreads, 2048 / kSplitThreads)
hot_split_kernel(const long long* __restrict__ rowptr, const CT* __restrict__ cols,
                 const VT* __restrict__ vals, int nrows, const int* __restrict__ rank, int H,
                 long long* __restrict__ rowptr_out, int* __restrict__ cols_out,
                 float* __restrict__ vals_out, int* __restrict__ rowmid,
                 unsigned short* __restrict__ xhot, long long hchunks, float* __restrict__ rowsum,
                 float* __restrict__ lgam, const int* __restrict__ ovf_idx = nullptr,
                 const float* __restrict__ ovf_val = nullptr, int novf = 0) {
  extern __shared__ __align__(16) unsigned short xrow[];        // [Hp] when STAGED, then the stash
  __shared__ int s_cov[kSplitWarps];
  __shared__ int s_gap[kSplitWarps];
  __shared__ float s_sum[kSplitWarps], s_lg[kSplitWarps];
  const int row = blockIdx.x;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int hp = (int)hchunks * 64;
  if constexpr (STAGED) {
    for (int i = threadIdx.x; i < hp / 8; i += blockDim.x) reinterpret_cast<uint4*>(xrow)[i] = make_uint4(0u, 0u, 0u, 0u);
  }
  if (row >= nrows) {                                            // padding row of the last 128-row tile
    if constexpr (STAGED) {
      for (int c = threadIdx.x; c < hp / 8; c += blockDim.x)
        *reinterpret_cast<uint4*>(xhot + tiledA_index(row, 8LL * c, hchunks)) = make_uint4(0u, 0u, 0u, 0u);
    }
    return;
  }
  // the warps take contiguous, equal pieces of the row (the kernel is a chain of dependent gathers
  // per 32 entries: more warps per row = more of them in flight)
  const long long base = rowptr[0];
  const long long j0 = rowptr[row], j1 = rowptr[row + 1];
  const long long o0 = j0 - base;
  if (threadIdx.x == 0) {
    rowptr_out[row] = o0;
    if (row == nrows - 1) rowptr_out[nrows] = j1 - base;
  }
  const long long n = j1 - j0;
  const long long seg = (n + kSplitThreads - 1) / kSplitThreads * 32;     // entries per warp, a multiple of 32
  const long long a0 = min(j1, j0 + w * seg), a1 = min(j1, a0 + seg);
  // pass 1: covered entries of my piece (and, if asked, the row constants of spmf_csr_row_consts);
  // the (rank, value) pairs of the first kSplitStash entries of the row are kept in shared memory so
  // that pass 2 does not repeat the two dependent gathers
  int2* stash = reinterpret_cast<int2*>(xrow + (STAGED ? hp : 0));
  int ncov = 0;
  float rs = 0.f, rl = 0.f;
  int cstart = -1;                                              // GAPS: column before my piece's first entry
  if constexpr (GAPS) {
    int gs = 0;
    for (long long j = a0 + lane; j < a1; j += 32) gs += (int)__ldcs(cols + j) + 1;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) gs += __shfl_xor_sync(0xffffffffu, gs, o);
    if (lane == 0) s_gap[w] = gs;
    __syncthreads();
    for (int t = 0; t < w; ++t) cstart += s_gap[t];
    int cbase = cstart;
    for (long long jb = a0; jb < a1; jb += 32) {
      const long long j = jb + lane;
      const bool in = j < a1;
      int g = in ? (int)__ldcs(cols + j) + 1 : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {                         // inclusive warp scan of the gaps
        const int t = __shfl_up_sync(0xffffffffu, g, o);
        if (lane >= o) g += t;
      }
      const int c = cbase + g;
      cbase += __shfl_sync(0xffffffffu, g, 31);
      if (in) {
        const int r = rank ? __ldg(rank + c) : c;
        const float x = u8_count(reinterpret_cast<const unsigned char*>(vals), j - base, ovf_idx, ovf_val, novf);
        if (j - j0 < kSplitStash) stash[j - j0] = make_int2(r, __float_as_int(x));
        ncov += hot_covered(r, x, H) ? 1 : 0;
        if (rowsum) { rs += x; rl += lgamma1p_count(x); }
      }
    }
  } else {
#pragma unroll 4
    for (long long j = a0 + lane; j < a1; j += 32) {
      const int c = (int)__ldcs(cols + j);
      const int r = rank ? __ldg(rank + c) : c;
      const float x = (float)__ldcs(vals + j);
      if (j - j0 < kSplitStash) stash[j - j0] = make_int2(r, __float_as_int(x));
      ncov += hot_covered(r, x, H) ? 1 : 0;
      if (rowsum) { rs += x; rl += lgamma1p_count(x); }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ncov += __shfl_xor_sync(0xffffffffu, ncov, o);
    rs += __shfl_xor_sync(0xffffffffu, rs, o);
    rl += __shfl_xor_sync(0xffffffffu, rl, o);
  }
  if (lane == 0) { s_cov[w] = ncov; s_sum[w] = rs; s_lg[w] = rl; }
  __syncthreads();                                           // (also: xrow is zeroed)
  int cov_before = 0, cov_total = 0;
  float tsum = 0.f, tlg = 0.f;
#pragma unroll
  for (int t = 0; t < kSplitWarps; ++t) {
    if (t < w) cov_before += s_cov[t];
    cov_total += s_cov[t];
    tsum += s_sum[t];
    tlg += s_lg[t];
  }
  if (threadIdx.x == 0) {
    rowmid[row] = cov_total;
    if (rowsum) {
      rowsum[row] = tsum;
      lgam[row] = tlg;
    }
  }
  // pass 2: stable partition -- covered entries first (negated), the others after cov_total
  long long pc = o0 + cov_before, pu = o0 + cov_total + ((a0 - j0) - cov_before);
  const bool rescan = GAPS && n > kSplitStash;                  // (CTA-uniform) rows longer than the stash
  int cbase2 = cstart;
  for (long long jb = a0; jb < a1; jb += 32) {
    const long long j = jb + lane;
    const bool in = j < a1;
    int r = 0;
    float x = 0.f;
    int cscan = 0;
    if constexpr (GAPS) {
      if (rescan) {
        int g = in ? (int)__ldcs(cols + j) + 1 : 0;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
          const int t = __shfl_up_sync(0xffffffffu, g, o);
          if (lane >= o) g += t;
        }
        cscan = cbase2 + g;
        cbase2 += __shfl_sync(0xffffffffu, g, 31);
      }
    }
    if (in) {
      if (j - j0 < kSplitStash) {                               // (written by this same lane in pass 1)
        const int2 e = stash[j - j0];
        r = e.x;
        x = __int_as_float(e.y);
      } else if constexpr (GAPS) {
        r = rank ? __ldg(rank + cscan) : cscan;
        x = u8_count(reinterpret_cast<const unsigned char*>(vals), j - base, ovf_idx, ovf_val, novf);
      } else {
        const int c = (int)__ldcs(cols + j);
        r = rank ? __ldg(rank + c) : c;
        x = (float)__ldcs(vals + j);
      }
    }
    const bool cov = in && hot_covered(r, x, H);
    const unsigned mc = __ballot_sync(0xffffffffu, cov);
    const unsigned mu = __ballot_sync(0xffffffffu, in && !cov);
    const unsigned below = (1u << lane) - 1u;
    if (cov) {
      const long long o = pc + __popc(mc & below);
      __stcs(cols_out + o, r);
      __stcs(vals_out + o, -x);
      const unsigned short hx = (unsigned short)(__float_as_uint(x) >> 16);
      if constexpr (STAGED) xrow[r] = hx;
      else xhot[tiledA_index(row, r, hchunks)] = hx;           // UMMA-tiled X[nrows][Hp]
    } else if (in) {
      const long long o = pu + __popc(mu & below);
      __stcs(cols_out + o, r);
      __stcs(vals_out + o, x);
    }
    pc += __popc(mc);
    pu += __popc(mu);
  }
  if constexpr (STAGED) {
    __syncthreads();
    for (int c = threadIdx.x; c < hp / 8; c += blockDim.x)
      __stcs(reinterpret_cast<uint4*>(xhot + tiledA_index(row, 8LL * c, hchunks)), reinterpret_cast<const uint4*>(xrow)[c]);
  }
}

// ---- the 2-byte transfer format straight to the hybrid form, one pass ------------------------------------------
// The streamed end-to-end step pays for this kernel in full (the device is busy under it), and the generic
// kernel above is issue-bound (~340 warp instructions per 32 nonzeros, profiles/r2_final_ncu_upload_kernels_summary.txt):
// two sweeps with a (rank, value) stash between them, 64-bit indices, a constant-memory table read with
// divergent indices.  Here: row-local 32-bit indices; after the warps' gap sums are known ONE sweep does the
// column scan, the rank lookup, the row constants and the placement -- covered entries are appended from the
// front of the row's output range, the others from its back, through two shared-memory cursors bumped once per
// warp and 32 entries (the order inside either part is irrelevant to every consumer: the cold row pass, the CSC
// build and the guard's scatter are order-free, the dense block is position-indexed).
__global__ void __launch_bounds__(kSplitThreads, 2048 / kSplitThreads)
hot_split8_kernel(const long long* __restrict__ rowptr, const unsigned char* __restrict__ gaps8,
                  const unsigned char* __restrict__ vals8, int nrows, const int* __restrict__ rank, int H,
                  long long* __restrict__ rowptr_out, int* __restrict__ cols_out, float* __restrict__ vals_out,
                  int* __restrict__ rowmid, unsigned short* __restrict__ xhot, long long hchunks,
                  float* __restrict__ rowsum, float* __restrict__ lgam, const int* __restrict__ ovf_idx,
                  const float* __restrict__ ovf_val, int novf) {
  extern __shared__ __align__(16) unsigned short xrow[];        // [Hp]
  __shared__ int s_gap[kSplitWarps], s_cur[2];
  __shared__ float s_sum[kSplitWarps], s_lg[kSplitWarps], s_tab[64];
  const int row = blockIdx.x;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int hp = (int)hchunks * 64;
  for (int i = threadIdx.x; i < hp / 8; i += blockDim.x) reinterpret_cast<uint4*>(xrow)[i] = make_uint4(0u, 0u, 0u, 0u);
  if (row >= nrows) {                                            // padding row of the last 128-row tile
    for (int c = threadIdx.x; c < hp / 8; c += blockDim.x)
      __stcs(reinterpret_cast<uint4*>(xhot + tiledA_index(row, 8LL * c, hchunks)), make_uint4(0u, 0u, 0u, 0u));
    return;
  }
  if (threadIdx.x < 64) s_tab[threadIdx.x] = kLgamTab[threadIdx.x];
  if (threadIdx.x < 2) s_cur[threadIdx.x] = 0;
  const long long base = rowptr[0], j0 = rowptr[row], j1 = rowptr[row + 1];
  const int n = (int)(j1 - j0);
  const long long o0 = j0 - base;
  if (threadIdx.x == 0) {
    rowptr_out[row] = o0;
    if (row == nrows - 1) rowptr_out[nrows] = j1 - base;
  }
  const unsigned char* __restrict__ g8 = gaps8 + j0;            // row-local from here on
  const unsigned char* __restrict__ v8 = vals8 + j0;
  int* __restrict__ co = cols_out + o0;
  float* __restrict__ vo = vals_out + o0;
  const int e0 = (int)o0;                                        // entry index of the row's first entry (overflow list key)
  const int seg = (n + kSplitThreads - 1) / kSplitThreads * 32;  // entries per warp, a multiple of 32
  const int a0 = min(n, w * seg), a1 = min(n, a0 + seg);
  int gs = 0;
  for (int t = a0 + lane; t < a1; t += 32) gs += (int)__ldcs(g8 + t) + 1;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) gs += __shfl_xor_sync(0xffffffffu, gs, o);
  if (lane == 0) s_gap[w] = gs;
  __syncthreads();                                               // (also: xrow zeroed, table and cursors set)
  int cbase = -1;                                                // column before my piece's first entry
  for (int t = 0; t < w; ++t) cbase += s_gap[t];
  float rs = 0.f, rl = 0.f;
  const unsigned below = (1u << lane) - 1u;
  for (int tb = a0; tb < a1; tb += 32) {
    const int t = tb + lane;
    const bool in = t < a1;
    int g = in ? (int)__ldcs(g8 + t) + 1 : 0;
    const unsigned b = in ? (unsigned)__ldcs(v8 + t) : 0u;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {                           // inclusive warp scan of the gaps
      const int u = __shfl_up_sync(0xffffffffu, g, o);
      if (lane >= o) g += u;
    }
    const int c = cbase + g;
    cbase += __shfl_sync(0xffffffffu, g, 31);
    int r = 0;
    float x = 0.f;
    if (in) {
      r = rank ? __ldg(rank + c) : c;
      x = (float)b;
      if (b == 255u) {                                           // count above 254: sorted overflow list
        const int e = e0 + t;
        int lo = 0, hi = novf - 1;
        while (lo < hi) {
          const int mid = (lo + hi) >> 1;
          if (__ldg(ovf_idx + mid) < e) lo = mid + 1; else hi = mid;
        }
        if (novf > 0 && __ldg(ovf_idx + lo) == e) x = __ldg(ovf_val + lo);
      }
      rs += x;
      rl += (b < 64u) ? s_tab[b] : lgammaf(x + 1.f);
    }
    const bool cov = in && hot_covered(r, x, H);
    const unsigned mc = __ballot_sync(0xffffffffu, cov);
    const unsigned mu = __ballot_sync(0xffffffffu, in && !cov);
    int bc = 0, bu = 0;
    if (lane == 0) {
      if (mc) bc = atomicAdd(&s_cur[0], __popc(mc));
      if (mu) bu = atomicAdd(&s_cur[1], __popc(mu));
    }
    bc = __shfl_sync(0xffffffffu, bc, 0);
    bu = __shfl_sync(0xffffffffu, bu, 0);
    if (cov) {
      const int o = bc + __popc(mc & below);
      __stcs(co + o, r);
      __stcs(vo + o, -x);
      xrow[r] = (unsigned short)(__float_as_uint(x) >> 16);
    } else if (in) {
      const int o = n - 1 - (bu + __popc(mu & below));
      __stcs(co + o, r);
      __stcs(vo + o, x);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    rs += __shfl_xor_sync(0xffffffffu, rs, o);
    rl += __shfl_xor_sync(0xffffffffu, rl, o);
  }
  if (lane == 0) { s_sum[w] = rs; s_lg[w] = rl; }
  __syncthreads();
  if (threadIdx.x == 0) {
    rowmid[row] = s_cur[0];
    if (rowsum) {
      float ts = 0.f, tl = 0.f;
#pragma unroll
      for (int t = 0; t < kSplitWarps; ++t) { ts += s_sum[t]; tl += s_lg[t]; }
      rowsum[row] = ts;
      lgam[row] = tl;
    }
  }
  for (int c = threadIdx.x; c < hp / 8; c += blockDim.x)
    __stcs(reinterpret_cast<uint4*>(xhot + tiledA_index(row, 8LL * c, hchunks)), reinterpret_cast<const uint4*>(xrow)[c]);
}

// ---- direct dense ingest: dense (B,D) counts in feature order -> hybrid form, no CSR round trip ------------
// For dense-origin workloads (BASELINE C2 / C3: every column is hot) the batch arrives as a dense matrix
// of small integers; going through CSR would write and re-read 8 B per nonzero only to scatter it back
// into the dense block.  Kernel 1: one CTA per row assembles the row's hot vector (bf16, rank order) in
// shared memory from the dense row, writes it as whole 16-byte chunks of the UMMA-tiled block, and emits
// the row constants and the number of UNCOVERED nonzeros (cold column, or a count that is not exact in
// bf16).  Kernel 2 (after a scan of those counts): the uncovered entries as a ranked CSR -- all the gather
// kernels of the tile-hybrid step read (rowmid = 0: the covered part of the CSR is never visited there).
template <typename T>
__global__ void __launch_bounds__(kSplitThreads, 2048 / kSplitThreads)
dense_hot_rows_kernel(const T* __restrict__ x, int nrows, int D, const int* __restrict__ rank, int H,
                      unsigned short* __restrict__ xhot, long long hchunks, float* __restrict__ rowsum,
                      float* __restrict__ lgam, long long* __restrict__ uncount, int* __restrict__ rowmid) {
  extern __shared__ __align__(16) unsigned short xrow[];        // [Hp]
  __shared__ int s_unc[kSplitWarps];
  __shared__ float s_sum[kSplitWarps], s_lg[kSplitWarps];
  const int row = blockIdx.x;
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const int hp = (int)hchunks * 64;
  for (int i = threadIdx.x; i < hp / 8; i += blockDim.x) reinterpret_cast<uint4*>(xrow)[i] = make_uint4(0u, 0u, 0u, 0u);
  if (row >= nrows) {                                            // padding row of the last 128-row tile
    for (int c = threadIdx.x; c < hp / 8; c += blockDim.x)
      *reinterpret_cast<uint4*>(xhot + tiledA_index(row, 8LL * c, hchunks)) = make_uint4(0u, 0u, 0u, 0u);
    return;
  }
  __syncthreads();
  const T* xr = x + (size_t)row * D;
  int nunc = 0;
  float rs = 0.f, rl = 0.f;
  for (int d = threadIdx.x; d < D; d += blockDim.x) {
    const float v = (float)xr[d];
    if (v != 0.f) {
      const int r = rank ? __ldg(rank + d) : d;
      rs += v;
      rl += lgamma1p_count(v);
      if (hot_covered(r, v, H)) xrow[r] = (unsigned short)(__float_as_uint(v) >> 16);
      else ++nunc;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    nunc += __shfl_xor_sync(0xffffffffu, nunc, o);
    rs += __shfl_xor_sync(0xffffffffu, rs, o);
    rl += __shfl_xor_sync(0xffffffffu, rl, o);
  }
  if (lane == 0) { s_unc[w] = nunc; s_sum[w] = rs; s_lg[w] = rl; }
  __syncthreads();
  if (threadIdx.x == 0) {
    int tu = 0;
    float ts = 0.f, tl = 0.f;
#pragma unroll
    for (int t = 0; t < kSplitWarps; ++t) { tu += s_unc[t]; ts += s_sum[t]; tl += s_lg[t]; }
    uncount[row + 1] = tu;
    if (row == 0) uncount[0] = 0;
    rowsum[row] = ts;
    lgam[row] = tl;
    rowmid[row] = 0;
  }
  for (int c = threadIdx.x; c < hp / 8; c += blockDim.x)
    *reinterpret_cast<uint4*>(xhot + tiledA_index(row, 8LL * c, hchunks)) = reinterpret_cast<const uint4*>(xrow)[c];
}

template <typename T>
__global__ void dense_uncovered_fill_kernel(const T* __restrict__ x, int nrows, int D, const int* __restrict__ rank,
                                            int H, const long long* __restrict__ rowptr, int* __restrict__ cols,
                                            float* __restrict__ vals) {
  const int row = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= nrows) return;
  if (rowptr[row + 1] == rowptr[row]) return;                    // (the common case for dense-origin counts)
  long long pos = rowptr[row];
  const T* xr = x + (size_t)row * D;
  for (int d0 = 0; d0 < D; d0 += 32) {
    const int d = d0 + lane;
    const float v = d < D ? (float)xr[d] : 0.f;
    const int r = (d < D && v != 0.f) ? (rank ? __ldg(rank + d) : d) : 0;
    const bool unc = v != 0.f && !hot_covered(r, v, H);
    const unsigned m = __ballot_sync(0xffffffffu, unc);
    if (unc) {
      const long long o = pos + __popc(m & ((1u << lane) - 1u));
      cols[o] = r;
      vals[o] = v;
    }
    pos += __popc(m);
  }
}

template <typename T>
static int launch_dense_hot_split(const T* x, int nrows, int D, const int* rank, int H, long long* rowptr_out,
                                  int* cols_out, float* vals_out, int* rowmid, void* xhot, float* rowsum, float* lgam,
                                  cudaStream_t st) {
  const long long hp = (H + 63) / 64 * 64;
  const size_t smem = (size_t)hp * 2;
  if (smem > 200 * 1024) return SPMF_ERR_UNSUPPORTED;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(dense_hot_rows_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    if (e != cudaSuccess) return (int)e;
    attr = true;
  }
  dense_hot_rows_kernel<T><<<(nrows + 127) / 128 * 128, kSplitThreads, smem, st>>>(
      x, nrows, D, rank, H, (unsigned short*)xhot, hp / 64, rowsum, lgam, rowptr_out, rowmid);
  incscan_ll_kernel<<<1, 1024, 0, st>>>(rowptr_out, nrows);
  dense_uncovered_fill_kernel<T><<<(nrows + 7) / 8, 256, 0, st>>>(x, nrows, D, rank, H, rowptr_out, cols_out, vals_out);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

// ------------------------------------------------------------------ dispatch
template <int KP, int SV, int MODE>
static int launch_rows(const long long* rowptr, const int* cols, const float* vals,
                       const float* rowsum, const float* lgam, float inv_xi, int scale_rows, int nrows,
                       int D, int NQ, const float* Ap, const float* EV, const float* PH,
                       const double* vsum, float* z, float* dzr, float* rowacc, const int* rowmid,
                       int* gflag, cudaStream_t st) {
  dim3 grid(nrows, NQ);
  if constexpr (MODE == kRowsCold && KP * SV == 128)
    csr_rows_cold5_kernel<KP, SV><<<grid, 128, 0, st>>>(
        rowptr, cols, vals, rowsum, lgam, inv_xi, scale_rows, nrows, D, Ap, EV, PH, vsum, z, dzr, rowacc, rowmid, gflag);
  else
    csr_rows_kernel<KP, SV, MODE><<<grid, 128, 0, st>>>(
        rowptr, cols, vals, rowsum, lgam, inv_xi, scale_rows, nrows, D, Ap, EV, PH, vsum, z, dzr, rowacc, rowmid, gflag);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

template <int KP, int SV>
static int launch_cols(const int* colptr, const int* rows, const float* vals, int nnz, int nrows,
                       int D, int NQ, const float* z, const float* dzr, const float* EV,
                       const float* PH, float* GAp, float* GEV, float* Gphi, cudaStream_t st,
                       int slice_len = kSliceLen) {
  constexpr int NSLOT = Map<KP, SV>::NSLOT;
  const int nslices = (nnz + slice_len - 1) / slice_len;
  if (nslices == 0) return SPMF_OK;
  dim3 grid((nslices + NSLOT - 1) / NSLOT, NQ);
  csc_cols_kernel<KP, SV><<<grid, 128, 0, st>>>(colptr, rows, vals, nnz, nrows, D, z, dzr, EV, PH,
                                               GAp, GEV, Gphi, slice_len);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

#define SPMF_DISPATCH_KP_SV(KP, SV, CALL)                                    \
  do {                                                                       \
    switch (KP) {                                                            \
      case 1: SPMF_DISPATCH_SV(1, SV, CALL); break;                          \
      case 2: SPMF_DISPATCH_SV(2, SV, CALL); break;                          \
      case 4: SPMF_DISPATCH_SV(4, SV, CALL); break;                          \
      case 8: SPMF_DISPATCH_SV(8, SV, CALL); break;                          \
      case 16: SPMF_DISPATCH_SV(16, SV, CALL); break;                        \
      case 32: SPMF_DISPATCH_SV(32, SV, CALL); break;                        \
      case 64: SPMF_DISPATCH_SV(64, SV, CALL); break;                        \
      case 128: SPMF_DISPATCH_SV(128, SV, CALL); break;                      \
      /* wide records: SV = spmf_draw_vec_k(K, S) keeps SV*KP <= 512 */       \
      case 256:                                                              \
        if (SV == 2) { CALL(256, 2); } else if (SV == 1) { CALL(256, 1); }   \
        else return SPMF_ERR_UNSUPPORTED;                                    \
        break;                                                               \
      case 512:                                                              \
        if (SV == 1) { CALL(512, 1); } else return SPMF_ERR_UNSUPPORTED;     \
        break;                                                               \
      default: return SPMF_ERR_UNSUPPORTED;                                  \
    }                                                                        \
  } while (0)
#define SPMF_DISPATCH_SV(KPC, SV, CALL)                                      \
  do {                                                                       \
    if (SV == 4) { CALL(KPC, 4); } else if (SV == 2) { CALL(KPC, 2); } else { CALL(KPC, 1); } \
  } while (0)

}  // namespace spmf

using namespace spmf;

extern "C" {

int spmf_csr_row_consts(const long long* rowptr, const float* vals, long long nrows, float* rowsum,
                        float* lgam, void* stream) {
  if (!rowptr || !vals || !rowsum || !lgam || nrows <= 0) return SPMF_ERR_BAD_ARG;
  csr_row_consts_kernel<<<(unsigned)((nrows + 3) / 4), 128, 0, (cudaStream_t)stream>>>(rowptr, vals, nrows, rowsum, lgam);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_csr_rows(const long long* rowptr, const int* cols, const float* vals, const float* rowsum,
                  const float* lgam, float inv_xi, int scale_rows, int nrows, int D, int K, int S,
                  const float* Ap, const float* EV, const float* PH, const double* vsum, float* z,
                  float* dzr, float* rowacc, int variant, void* gs, void* stream) {
  if (!rowptr || !cols || !vals || !rowsum || !lgam || !Ap || !EV || !PH || !vsum || !z || !dzr || !rowacc)
    return SPMF_ERR_BAD_ARG;
  if (nrows <= 0 || D <= 0 || K <= 0 || K > SPMF_MAX_K || S <= 0) return SPMF_ERR_BAD_ARG;
  if (variant != 0) return SPMF_ERR_UNSUPPORTED;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = SPMF_OK;
#define CALL_ROWS(KPC, SVC) rc = launch_rows<KPC, SVC, kRowsTrain>(rowptr, cols, vals, rowsum, lgam, inv_xi, scale_rows, nrows, D, NQ, Ap, EV, PH, vsum, z, dzr, rowacc, nullptr, (int*)gs, st)
  SPMF_DISPATCH_KP_SV(KP, SV, CALL_ROWS);
#undef CALL_ROWS
  return rc;
}

int spmf_csr_encode(const long long* rowptr, const int* cols, const float* vals, const float* rowsum,
                    float inv_xi, int scale_rows, int nrows, int D, int K, int S, const float* Ap,
                    float* z, void* stream) {
  if (!rowptr || !cols || !vals || !rowsum || !Ap || !z) return SPMF_ERR_BAD_ARG;
  if (nrows <= 0 || D <= 0 || K <= 0 || K > SPMF_MAX_K || S <= 0) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = SPMF_OK;
#define CALL_ENC(KPC, SVC) rc = launch_rows<KPC, SVC, kRowsEncode>(rowptr, cols, vals, rowsum, nullptr, inv_xi, scale_rows, nrows, D, NQ, Ap, nullptr, nullptr, nullptr, z, nullptr, nullptr, nullptr, nullptr, st)
  SPMF_DISPATCH_KP_SV(KP, SV, CALL_ENC);
#undef CALL_ENC
  return rc;
}

int spmf_csc_cols(const int* colptr, const int* rows, const float* vals, int nnz, int nrows, int D,
                  int K, int S, const float* z, const float* dzr, const float* EV, const float* PH,
                  float* GAp, float* GEVnz, float* Gphinz, int variant, void* stream) {
  if (!colptr || !rows || !vals || !z || !dzr || !EV || !PH || !GAp || !GEVnz || !Gphinz) return SPMF_ERR_BAD_ARG;
  if (nnz < 0 || nrows <= 0 || D <= 0 || K <= 0 || K > SPMF_MAX_K || S <= 0) return SPMF_ERR_BAD_ARG;
  if (variant != 0) return SPMF_ERR_UNSUPPORTED;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t nb = (size_t)NQ * D * KP * SV * sizeof(float);
  cudaError_t e = cudaMemsetAsync(GAp, 0, nb, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(GEVnz, 0, nb, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(Gphinz, 0, (size_t)NQ * D * SV * sizeof(float), st);
  if (e != cudaSuccess) return (int)e;
  int rc = SPMF_OK;
#define CALL_COLS(KPC, SVC) rc = launch_cols<KPC, SVC>(colptr, rows, vals, nnz, nrows, D, NQ, z, dzr, EV, PH, GAp, GEVnz, Gphinz, st)
  SPMF_DISPATCH_KP_SV(KP, SV, CALL_COLS);
#undef CALL_COLS
  return rc;
}

// ---- hybrid (tensor-core hot block + gather) variants --------------------------------------------
// Supported record shapes: REC = KP*SV in {32, 64, 128} (the N of the tcgen05 GEMM).
#define SPMF_DISPATCH_HYBRID(KP, SV, CALL)                                   \
  do {                                                                       \
    if (KP == 32 && SV == 4) { CALL(32, 4); }                                \
    else if (KP == 32 && SV == 2) { CALL(32, 2); }                           \
    else if (KP == 32 && SV == 1) { CALL(32, 1); }                           \
    else if (KP == 16 && SV == 4) { CALL(16, 4); }                           \
    else if (KP == 16 && SV == 2) { CALL(16, 2); }                           \
    else if (KP == 8 && SV == 4) { CALL(8, 4); }                             \
    else if (KP == 64 && SV == 4) { CALL(64, 4); }                           \
    else if (KP == 64 && SV == 2) { CALL(64, 2); }                           \
    else if (KP == 64 && SV == 1) { CALL(64, 1); }                           \
    else if (KP == 128 && SV == 4) { CALL(128, 4); }                         \
    else if (KP == 128 && SV == 2) { CALL(128, 2); }                         \
    else if (KP == 128 && SV == 1) { CALL(128, 1); }                         \
    else return SPMF_ERR_UNSUPPORTED;                                        \
  } while (0)

/* 0: gather kernels only; 2: tile-hybrid (GEMMs + fused tile kernel, spmf_hot_tile.cu) */
int spmf_hybrid_supported(int K, int S) {
  if (K <= 0 || K > SPMF_MAX_TILE_K || S <= 0) return 0;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S);
  if ((KP == 32 && (SV == 4 || SV == 2 || SV == 1)) || (KP == 16 && (SV == 4 || SV == 2)) || (KP == 8 && SV == 4))
    return 2;
  if (KP == 64 || KP == 128) return 2;     // fused tile kernel with 64 / 128 latent dims (spmf_hot_tile.cu)
  return 0;
}

int spmf_csr_rows_cold(const long long* rowptr, const int* cols, const float* vals, const int* rowmid,
                       const float* rowsum, float inv_xi, int scale_rows, int nrows, int D, int K, int S,
                       const float* Ap, const float* EV, const float* PH, float* z, float* dzacc, float* rowacc,
                       void* gs, void* stream) {
  if (!rowptr || !cols || !vals || !rowmid || !rowsum || !Ap || !EV || !PH || !z || !dzacc || !rowacc)
    return SPMF_ERR_BAD_ARG;
  if (nrows <= 0 || D <= 0 || K <= 0 || K > SPMF_MAX_TILE_K || S <= 0) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = SPMF_OK;
#define CALL_ROWS_C(KPC, SVC) rc = launch_rows<KPC, SVC, kRowsCold>(rowptr, cols, vals, rowsum, nullptr, inv_xi, scale_rows, nrows, D, NQ, Ap, EV, PH, nullptr, z, dzacc, rowacc, rowmid, (int*)gs, st)
  SPMF_DISPATCH_HYBRID(KP, SV, CALL_ROWS_C);
#undef CALL_ROWS_C
  return rc;
}

int spmf_zero_col_grads(float* GAp, float* GEVnz, float* Gphinz, int D, int K, int S, void* stream) {
  if (!GAp || !GEVnz || !Gphinz || D <= 0 || K <= 0 || K > SPMF_MAX_K || S <= 0) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t nb = (size_t)NQ * D * KP * SV * sizeof(float);
  cudaError_t e = cudaMemsetAsync(GAp, 0, nb, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(GEVnz, 0, nb, st);
  if (e == cudaSuccess) e = cudaMemsetAsync(Gphinz, 0, (size_t)NQ * D * SV * sizeof(float), st);
  return e == cudaSuccess ? SPMF_OK : (int)e;
}

int spmf_csc_cols_accum(const int* colptr, const int* rows, const float* vals, int nnz_bound, int nrows, int D,
                        int K, int S, const float* z, const float* dzr, const float* EV, const float* PH,
                        float* GAp, float* GEVnz, float* Gphinz, void* stream) {
  if (!colptr || !rows || !vals || !z || !dzr || !EV || !PH || !GAp || !GEVnz || !Gphinz) return SPMF_ERR_BAD_ARG;
  if (nnz_bound < 0 || nrows <= 0 || D <= 0 || K <= 0 || K > SPMF_MAX_TILE_K || S <= 0) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  cudaStream_t st = (cudaStream_t)stream;
  int rc = SPMF_OK;
  // sparse remainder: short slices keep every SM busy on a small stream
#define CALL_COLS_COLD(KPC, SVC) rc = launch_cols<KPC, SVC>(colptr, rows, vals, nnz_bound, nrows, D, NQ, z, dzr, EV, PH, GAp, GEVnz, Gphinz, st, 64)
  SPMF_DISPATCH_HYBRID(KP, SV, CALL_COLS_COLD);
#undef CALL_COLS_COLD
  return rc;
}

// ---- hot split: CSR batch (original column ids) -> ranked, partitioned CSR + dense bf16 hot block ----
// A nonzero is "covered" by the tensor-core products when its column's rank is < H and its value
// is exactly representable in bf16 (integer counts <= 256).  Per row, covered entries come first
// (stored with a negative sign as their flag), the rest after rowmid[row]; column ids become ranks.
// xhot[b][rank] receives the covered values.
}  // extern "C"

// test hook: exercise the wide-block fallback (unstaged split kernels) on small inputs
static bool split_unstaged() {
  static const bool on = [] {
    const char* e = getenv("SPMF_SPLIT_UNSTAGED");
    return e && e[0] == '1';
  }();
  return on;
}

template <typename CT, typename VT>
static int launch_hot_split(const long long* rowptr, const CT* cols, const VT* vals, int nrows, const int* rank, int H,
                            long long* rowptr_out, int* cols_out, float* vals_out, int* rowmid, void* xhot,
                            float* rowsum, float* lgam, cudaStream_t st) {
  const long long hp = (H + 63) / 64 * 64;
  const size_t stash = (size_t)kSplitStash * sizeof(int2);
  const size_t smem = (size_t)hp * 2 + stash;
  if (smem <= 112 * 1024 && !split_unstaged()) {
    // staged: every 16-byte chunk of the 128-row-padded block is written by the kernel (no memset)
    static bool attr = false;
    if (!attr) {
      cudaError_t e = cudaFuncSetAttribute(hot_split_kernel<true, CT, VT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           112 * 1024);
      if (e != cudaSuccess) return (int)e;
      attr = true;
    }
    hot_split_kernel<true, CT, VT><<<(nrows + 127) / 128 * 128, kSplitThreads, smem, st>>>(
        rowptr, cols, vals, nrows, rank, H, rowptr_out, cols_out, vals_out, rowmid, (unsigned short*)xhot, hp / 64,
        rowsum, lgam);
  } else {
    cudaError_t e = cudaMemsetAsync(xhot, 0, (size_t)spmf_umma_tiled_a_elems(nrows, hp) * 2, st);
    if (e != cudaSuccess) return (int)e;
    hot_split_kernel<false, CT, VT><<<nrows, kSplitThreads, stash, st>>>(rowptr, cols, vals, nrows, rank, H, rowptr_out, cols_out,
                                                          vals_out, rowmid, (unsigned short*)xhot, hp / 64, rowsum,
                                                          lgam);
  }
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

static int launch_hot_split8(const long long* rowptr, const unsigned char* gaps8, const unsigned char* vals8,
                             const int* ovf_idx, const float* ovf_val, int novf, int nrows, const int* rank, int H,
                             long long* rowptr_out, int* cols_out, float* vals_out, int* rowmid, void* xhot,
                             float* rowsum, float* lgam, cudaStream_t st) {
  const long long hp = (H + 63) / 64 * 64;
  const size_t stash = (size_t)kSplitStash * sizeof(int2);
  const size_t smem = (size_t)hp * 2 + stash;
  if (smem <= 112 * 1024 && !split_unstaged()) {
    static bool attr = false;
    if (!attr) {
      cudaError_t e = cudaFuncSetAttribute(hot_split8_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 112 * 1024);
      if (e != cudaSuccess) return (int)e;
      attr = true;
    }
    hot_split8_kernel<<<(nrows + 127) / 128 * 128, kSplitThreads, (size_t)hp * 2, st>>>(
        rowptr, gaps8, vals8, nrows, rank, H, rowptr_out, cols_out, vals_out, rowmid, (unsigned short*)xhot, hp / 64,
        rowsum, lgam, ovf_idx, ovf_val, novf);
  } else {
    cudaError_t e = cudaMemsetAsync(xhot, 0, (size_t)spmf_umma_tiled_a_elems(nrows, hp) * 2, st);
    if (e != cudaSuccess) return (int)e;
    hot_split_kernel<false, unsigned char, unsigned char, true><<<nrows, kSplitThreads, stash, st>>>(
        rowptr, gaps8, vals8, nrows, rank, H, rowptr_out, cols_out, vals_out, rowmid, (unsigned short*)xhot, hp / 64,
        rowsum, lgam, ovf_idx, ovf_val, novf);
  }
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

extern "C" {

int spmf_hot_split_u8(const long long* rowptr, const unsigned char* gaps8, const unsigned char* vals8,
                      const int* ovf_idx, const float* ovf_val, int novf, int nrows, const int* rank, int H,
                      long long* rowptr_out, int* cols_out, float* vals_out, int* rowmid, void* xhot, float* rowsum,
                      float* lgam, void* stream) {
  if (!rowptr || !gaps8 || !vals8 || !rowptr_out || !cols_out || !vals_out || !rowmid || !xhot) return SPMF_ERR_BAD_ARG;
  if ((rowsum == nullptr) != (lgam == nullptr) || novf < 0 || (novf > 0 && (!ovf_idx || !ovf_val))) return SPMF_ERR_BAD_ARG;
  if (nrows <= 0 || H <= 0) return SPMF_ERR_BAD_ARG;
  return launch_hot_split8(rowptr, gaps8, vals8, ovf_idx, ovf_val, novf, nrows, rank, H, rowptr_out, cols_out, vals_out,
                           rowmid, xhot, rowsum, lgam, (cudaStream_t)stream);
}

int spmf_hot_split_packed(const long long* rowptr, const int* cols, const unsigned short* cols16, const float* vals,
                          const unsigned short* vals16, int nrows, long long nnz, const int* rank, int H,
                          long long* rowptr_out, int* cols_out, float* vals_out, int* rowmid, void* xhot,
                          float* rowsum, float* lgam, void* stream) {
  if (!rowptr || (!cols == !cols16) || (!vals == !vals16) || !rowptr_out || !cols_out || !vals_out || !rowmid || !xhot)
    return SPMF_ERR_BAD_ARG;
  if ((rowsum == nullptr) != (lgam == nullptr)) return SPMF_ERR_BAD_ARG;
  if (nrows <= 0 || nnz < 0 || H <= 0) return SPMF_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  int rc;
#define SPMF_SPLIT_ARGS nrows, rank, H, rowptr_out, cols_out, vals_out, rowmid, xhot, rowsum, lgam, st
  if (cols && vals) rc = launch_hot_split(rowptr, cols, vals, SPMF_SPLIT_ARGS);
  else if (cols) rc = launch_hot_split(rowptr, cols, vals16, SPMF_SPLIT_ARGS);
  else if (vals) rc = launch_hot_split(rowptr, cols16, vals, SPMF_SPLIT_ARGS);
  else rc = launch_hot_split(rowptr, cols16, vals16, SPMF_SPLIT_ARGS);
#undef SPMF_SPLIT_ARGS
  return rc;
}

int spmf_hot_split(const long long* rowptr, const int* cols, const float* vals, int nrows, long long nnz,
                   const int* rank, int H, long long* rowptr_out, int* cols_out, float* vals_out, int* rowmid,
                   void* xhot, float* rowsum, float* lgam, void* stream) {
  if (!cols || !vals) return SPMF_ERR_BAD_ARG;
  return spmf_hot_split_packed(rowptr, cols, nullptr, vals, nullptr, nrows, nnz, rank, H, rowptr_out, cols_out,
                               vals_out, rowmid, xhot, rowsum, lgam, stream);
}

int spmf_csr_colstats(const int* cols, const float* vals, long long nnz, int D, double* colsum,
                      float* colnnz, void* stream) {
  if (!cols || !vals || !colsum || !colnnz || nnz < 0 || D <= 0) return SPMF_ERR_BAD_ARG;
  if (nnz == 0) return SPMF_OK;
  long long blocks = (nnz + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  csr_colstats_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(cols, vals, nnz, colsum, colnnz);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

long long spmf_csc_scratch_ints(int D) { return (long long)(kTrBlocks + 1) * ((long long)D + 1); }

int spmf_csr_to_csc(const long long* rowptr, const int* cols, const float* vals, int nrows, int D,
                    int* colptr, int* rows_out, float* vals_out, int* scratch, void* stream) {
  return spmf_csr_to_csc_part(rowptr, nullptr, 0, cols, vals, nrows, D, colptr, rows_out, vals_out, scratch, stream);
}

int spmf_csr_to_csc_part(const long long* rowptr, const int* rowmid, int part, const int* cols, const float* vals,
                         int nrows, int D, int* colptr, int* rows_out, float* vals_out, int* scratch,
                         void* stream) {
  if (!rowptr || !cols || !vals || !colptr || !rows_out || !vals_out || !scratch) return SPMF_ERR_BAD_ARG;
  if (nrows <= 0 || D <= 0 || (part != 0 && part != 1)) return SPMF_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  int* colcnt = scratch;                       // [D+1]
  int* blockhist = scratch + (D + 1);          // [kTrBlocks][D]
  const size_t smem = (size_t)D * sizeof(int);
  if (smem <= 200 * 1024) {
    static bool attr_set = false;
    if (!attr_set) {
      cudaFuncSetAttribute(csc_block_hist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      cudaFuncSetAttribute(csc_block_scatter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
      attr_set = true;
    }
    const int nb = nrows < kTrBlocks ? nrows : kTrBlocks;
    csc_block_hist_kernel<<<nb, kTrThreads, smem, st>>>(rowptr, rowmid, part, cols, nrows, D, blockhist);
    csc_block_scan_kernel<<<(D + 63) / 64, 64, 0, st>>>(blockhist, nb, D, colcnt);
    exscan_int_kernel<<<1, 1024, 0, st>>>(colcnt, D, colptr, nullptr);
    csc_block_scatter_kernel<<<nb, kTrThreads, smem, st>>>(rowptr, rowmid, part, cols, vals, nrows, D, colptr,
                                                          blockhist, rows_out, vals_out);
  } else {                                     // very wide matrices: global atomic cursors
    cudaError_t e = cudaMemsetAsync(colcnt, 0, (size_t)(D + 1) * sizeof(int), st);
    if (e != cudaSuccess) return (int)e;
    count_cols_kernel<<<(nrows + 7) / 8, 256, 0, st>>>(rowptr, rowmid, part, cols, nrows, colcnt);
    exscan_int_kernel<<<1, 1024, 0, st>>>(colcnt, D, colptr, colcnt);
    scatter_csc_kernel<<<(nrows + 3) / 4, 128, 0, st>>>(rowptr, rowmid, part, cols, vals, nrows, colcnt, rows_out,
                                                       vals_out);
  }
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_csr_unpack16(const unsigned short* cols16, const unsigned short* vals16, long long nnz,
                      int* cols, float* vals, void* stream) {
  if ((!cols16 && !vals16) || (cols16 && !cols) || (vals16 && !vals) || nnz < 0) return SPMF_ERR_BAD_ARG;
  if (nnz == 0) return SPMF_OK;
  long long blocks = (nnz + 255) / 256;
  if (blocks > 148 * 16) blocks = 148 * 16;
  csr_unpack16_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(cols16, vals16, nnz, cols, vals);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_csr_unpack8(const long long* rowptr, const unsigned char* gaps8, const unsigned char* vals8, int nrows,
                     const int* ovf_idx, const float* ovf_val, int n_ovf, int* cols, float* vals, void* stream) {
  if (!rowptr || !gaps8 || !vals8 || !cols || !vals || nrows <= 0 || n_ovf < 0 || (n_ovf && (!ovf_idx || !ovf_val)))
    return SPMF_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  csr_unpack8_kernel<<<(unsigned)((nrows + 7) / 8), 256, 0, st>>>(rowptr, gaps8, vals8, nrows, cols, vals);
  if (n_ovf) csr_patch_vals_kernel<<<(unsigned)((n_ovf + 255) / 256), 256, 0, st>>>(ovf_idx, ovf_val, n_ovf, vals);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_dense_count(const float* x, int nrows, int D, long long* rowptr, void* stream) {
  if (!x || !rowptr || nrows <= 0 || D <= 0) return SPMF_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  dense_count_kernel<<<(nrows + 3) / 4, 128, 0, st>>>(x, nrows, D, rowptr);
  incscan_ll_kernel<<<1, 1024, 0, st>>>(rowptr, nrows);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_dense_fill(const float* x, int nrows, int D, const long long* rowptr, int* cols, float* vals,
                    void* stream) {
  if (!x || !rowptr || !cols || !vals || nrows <= 0 || D <= 0) return SPMF_ERR_BAD_ARG;
  dense_fill_kernel<<<(nrows + 3) / 4, 128, 0, (cudaStream_t)stream>>>(x, nrows, D, rowptr, cols, vals);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_dense_hot_split(const void* x, int dtype, int nrows, int D, const int* rank, int H, long long* rowptr_out,
                         int* cols_out, float* vals_out, int* rowmid, void* xhot, float* rowsum, float* lgam,
                         void* stream) {
  if (!x || !rowptr_out || !cols_out || !vals_out || !rowmid || !xhot || !rowsum || !lgam) return SPMF_ERR_BAD_ARG;
  if (nrows <= 0 || D <= 0 || H <= 0 || H > D) return SPMF_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  switch (dtype) {
    case SPMF_DENSE_U8: return launch_dense_hot_split<unsigned char>((const unsigned char*)x, nrows, D, rank, H, rowptr_out, cols_out, vals_out, rowmid, xhot, rowsum, lgam, st);
    case SPMF_DENSE_U16: return launch_dense_hot_split<unsigned short>((const unsigned short*)x, nrows, D, rank, H, rowptr_out, cols_out, vals_out, rowmid, xhot, rowsum, lgam, st);
    case SPMF_DENSE_F32: return launch_dense_hot_split<float>((const float*)x, nrows, D, rank, H, rowptr_out, cols_out, vals_out, rowmid, xhot, rowsum, lgam, st);
    default: return SPMF_ERR_BAD_ARG;
  }
}

const char* spmf_version(void) { return "spmf_b200 0.2 (sm_100a)"; }

}  // extern "C"
