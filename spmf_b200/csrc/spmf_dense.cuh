// Pieces of the dense CUDA-core evaluation shared by the data-term kernels (spmf_dense.cu) and the
// posterior predictive check (spmf_ppc.cu): the per-entry link, the (row|feature, draw) thread geometry and
// the shared-memory staging of the operand records.
#pragma once
#include <cuda_runtime.h>
#include <float.h>
#include <stdint.h>

#include "../../include/spmf_b200.h"
#include "spmf_record.cuh"

namespace spmf {

// One entry: lin = z.EV  ->  rate = f(lin) + phi  ->  log-likelihood core (without -lgamma(x+1)),
// dL/dlin, dL/dphi.  `ok` = the log-likelihood is finite (poisson.py:606-608 is_finite).
struct Elem { float ll, glin, gphi; bool ok; };

// rate = f(lin) + phi: the Poisson rate (links 0, 1) or the Bernoulli logit (links 2, 3)
template <int LINK>
__device__ __forceinline__ float link_rate(float lin, float phi) {
  const float t = (LINK & 1) ? __expf(lin) - 1.f : lin;   // poisson.py:52-53 decoder exp(y*eta) - 1 (eta folded into EV)
  return t + phi;                                          // poisson.py:177
}

template <int LINK>
__device__ __forceinline__ Elem link_elem(float x, float lin, float phi) {
  const float dt = (LINK & 1) ? __expf(lin) : 1.f;
  const float rate = link_rate<LINK>(lin, phi);
  Elem o;
  if (LINK < 2) {                         // tfd.Poisson(rate).log_prob(x) = multiply_no_nan(log rate, x) - lgamma(1+x) - rate
    const bool fin = fabsf(rate) <= FLT_MAX;
    o.ok = x > 0.f ? (rate > 0.f && fin) : fin;
    const float rs = o.ok ? rate : 1.f;
    const float lg = x > 0.f ? __logf(rs) : 0.f;
    o.ll = fmaf(x, lg, -rs);
    const float dr = x > 0.f ? fmaf(x, __fdividef(1.f, rs), -1.f) : -1.f;
    o.gphi = o.ok ? dr : 0.f;
  } else {                                // tfd.Bernoulli(logits=rate).log_prob(x) = x*rate - softplus(rate)
    o.ok = fabsf(rate) <= FLT_MAX;
    const float rs = o.ok ? rate : 0.f;
    const float e = __expf(-fabsf(rs));
    const float sp = fmaxf(rs, 0.f) + log1pf(e);
    const float r = __fdividef(1.f, 1.f + e);
    const float sg = rs >= 0.f ? r : e * r;
    o.ll = fmaf(x, rs, -sp);
    o.gphi = o.ok ? x - sg : 0.f;
  }
  o.glin = o.gphi * dt;
  if (!o.ok) o.ll = 0.f;
  return o;
}

// (sv, k) of position p inside a record -- inverse of rec_pos (spmf_record.cuh)
__device__ __forceinline__ void rec_unpos(const RecMap& m, int SV, int p, int* sv, int* k) {
  const int w = p % m.VW;
  int t = p / m.VW;
  const int kg = t % m.RG;
  t /= m.RG;
  *sv = t % SV;
  const int i = t / SV;
  *k = (i * m.RG + kg) * m.VW + w;
}

struct DenseGeom {
  int KP, SV, NQ, REC;
  int NKQ;          // lanes sharing one (row|feature, draw): KP / KC
  int OW;           // owners (rows or features) per warp: 32 / NKQ
  int WG;           // owner groups per CTA: 4 / SV   (warp w: sv = w % SV, group = w / SV)
  int OB;           // owners per CTA: OW * WG
};
template <int KC>
__host__ __device__ __forceinline__ DenseGeom dense_geom(int KP, int SV, int NQ) {
  DenseGeom g;
  g.KP = KP; g.SV = SV; g.NQ = NQ; g.REC = KP * SV;
  g.NKQ = KP / KC;
  g.OW = 32 / g.NKQ;
  g.WG = 4 / SV;
  g.OB = g.OW * g.WG;
  return g;
}
constexpr int kTile = 32;           // features (row pass) / rows (column pass) staged per step

// stage `n` records of a gather table (rows first .. first+n) into shared memory in plain [i][sv][k]
// order; records beyond `limit` are zero
__device__ __forceinline__ void stage_records(float* dst, const float* __restrict__ tab, long long first, int n,
                                              long long limit, const DenseGeom& g, const RecMap& rm) {
  const int total = n * g.REC;
  for (int idx = threadIdx.x; idx < total; idx += blockDim.x) {
    const int i = idx / g.REC, p = idx - i * g.REC;
    int sv, k;
    rec_unpos(rm, g.SV, p, &sv, &k);
    dst[(i * g.SV + sv) * g.KP + k] = (first + i < limit) ? __ldg(tab + (first + i) * g.REC + p) : 0.f;
  }
}

template <int KC>
__device__ __forceinline__ void ld_slice(float (&r)[KC], const float* p) {
  if constexpr (KC >= 4) {
#pragma unroll
    for (int j = 0; j < KC; j += 4) {
      const float4 t = *reinterpret_cast<const float4*>(p + j);
      r[j] = t.x; r[j + 1] = t.y; r[j + 2] = t.z; r[j + 3] = t.w;
    }
  } else {
#pragma unroll
    for (int j = 0; j < KC; ++j) r[j] = p[j];
  }
}

__device__ __forceinline__ float lanes_sum(float v, int nkq) {      // lanes kq = lane % nkq are adjacent
  for (int o = nkq >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

template <typename Kern>
static int set_smem(Kern k, size_t bytes) {
  if (bytes <= 48 * 1024) return SPMF_OK;
  cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  return e == cudaSuccess ? SPMF_OK : (int)e;
}

}  // namespace spmf

// dispatch on the per-lane latent slice KC = min(KP, 32) and the link
#define DENSE_KC(KP, CALL)                     \
  do {                                         \
    switch ((KP) > 32 ? 32 : (KP)) {           \
      case 32: CALL(32); break;                \
      case 16: CALL(16); break;                \
      case 8: CALL(8); break;                  \
      case 4: CALL(4); break;                  \
      case 2: CALL(2); break;                  \
      case 1: CALL(1); break;                  \
      default: return SPMF_ERR_UNSUPPORTED;    \
    }                                          \
  } while (0)
#define DENSE_LINK(KC, LINK, CALL)                                 \
  do {                                                             \
    switch (LINK) {                                                \
      case SPMF_LINK_POISSON: CALL(KC, 0); break;                  \
      case SPMF_LINK_POISSON_LOG: CALL(KC, 1); break;              \
      case SPMF_LINK_BERNOULLI: CALL(KC, 2); break;                \
      case SPMF_LINK_BERNOULLI_LOG: CALL(KC, 3); break;            \
      default: return SPMF_ERR_UNSUPPORTED;                        \
    }                                                              \
  } while (0)
