// O(D*K*S) kernels around the data term: noise generation, reparameterised draws ->
// gather operands, prior/entropy forward+backward chained with the data-term gradients,
// deterministic reductions, Adam.  One warp per feature d, lanes over latent k; the
// per-element math lives in spmf_model.cuh (shared with the CPU host check).
//
// Replaces, for the ADVI step of mederrata_spmf/poisson.py (paths relative to /root/reference):
//   surrogate_distribution.sample / log_prob   [EXT L3], poisson.py:403-573
//   prior_distribution.log_prob_parts           poisson.py:590
//   encoding_matrix / intercept_matrix          poisson.py:652-701
//   tf.GradientTape backward + Adam             [EXT L4]
#include <cuda_runtime.h>
#include <stdint.h>
#include <string.h>

#include "../../include/spmf_b200.h"
#include "spmf_guard.cuh"
#include "spmf_model.cuh"
#include "spmf_record.cuh"

namespace spmf {

#define SPMF_CHECK_LAUNCH()                      \
  do {                                           \
    cudaError_t e__ = cudaGetLastError();        \
    if (e__ != cudaSuccess) return (int)e__;     \
  } while (0)

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------ noise
// Normal variables (blockIdx.y = v,w,u,s): 4 normals per Philox call; element e -> (call e/4, slot e%4).
__global__ void fill_normal_kernel(Layout L, float* __restrict__ noise, uint32_t step, uint32_t k0,
                                   uint32_t k1, const StepState* __restrict__ sst) {
  if (sst) step = sst->rng_step;
  const int v = blockIdx.y;
  const long long n = L.vsize[v] * L.S;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long base = i * 4;
  if (base >= n) return;
  float* out = noise + L.noff[v];
  U4 ctr = {(uint32_t)(i & 0xffffffffu), (uint32_t)(i >> 32), (uint32_t)v, step};
  U4 r = philox4x32_10(ctr, k0, k1);
  float x[4];
  box_muller(r.x, r.y, &x[0], &x[1]);
  box_muller(r.z, r.w, &x[2], &x[3]);
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (base + j < n) out[base + j] = x[j];
}

// Gamma variables (blockIdx.y = the 8 InverseGamma-based ones), one thread per element, all S
// draws: g[s][e] ~ Gamma(softplus(conc_raw[e]), 1) (Philox stream keyed by s*nelem+e) when `draw`,
// and dg/dalpha of every draw (implicit reparameterisation) -- it depends on (alpha, g) only, so
// it is evaluated here, fully parallel, off the critical path of the data term.
// The continued-fraction regime of the gradient (draws well above alpha, ~20 % of them) is not evaluated
// in place -- that would run its long loop once per draw slot with a fifth of the lanes active -- but
// queued in shared memory and worked off by the whole CTA with (nearly) full warps.
// The grid is the concatenation of each variable's ceil(vsize / 128) CTAs (gamma_grid_blocks): the
// variables range from K to D*K elements, and a grid of 8 x the largest left ~70 % of the CTAs with
// nothing to do.
static unsigned gamma_grid_blocks(const Layout& L) {
  long long nb = 0;
  for (int v = VAR_UETA; v < NUM_VARS; ++v) nb += (L.vsize[v] + 127) / 128;
  return (unsigned)nb;
}

__global__ void __launch_bounds__(128)
gamma_kernel(Layout L, const float* __restrict__ P, float* __restrict__ N, float* __restrict__ G,
             int draw, int grad, uint32_t step, uint32_t k0, uint32_t k1, const StepState* __restrict__ sst) {
  if (sst) step = sst->rng_step;
  __shared__ float4 cfq[128 * 4];              // (alpha, digamma(alpha), draw, slot = draw index * 128 + thread)
  __shared__ int cfn;
  int v = VAR_UETA;
  long long blk = blockIdx.x;
  for (; v < NUM_VARS - 1; ++v) {
    const long long nb = (L.vsize[v] + 127) / 128;
    if (blk < nb) break;
    blk -= nb;
  }
  const long long nelem = L.vsize[v];
  const long long e0 = blk * blockDim.x;
  const long long e = e0 + threadIdx.x;
  const bool live = e < nelem;
  if (threadIdx.x == 0) cfn = 0;
  __syncthreads();
  const float alpha = live ? softplusf(P[L.toff[2 * v] + e]) : 1.f;
  const float psi = (grad && live) ? digammaf_pos(alpha) : 0.f;
  float* Nv = N + L.noff[v];
  float* Gv = G + L.noff[v];
  for (int s0 = 0; s0 < L.S; s0 += 4) {
    const int ns = L.S - s0 < 4 ? L.S - s0 : 4;
    bool queued = false;
    if (live) {
      float g[4] = {1.f, 1.f, 1.f, 1.f}, o[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (j < ns) {
          const long long i = (long long)(s0 + j) * nelem + e;
          if (draw) {
            // stream id folds the step so that (element, iteration) keep the whole counter space
            g[j] = gamma_draw(alpha, (uint32_t)(i & 0xffffffffu), (uint32_t)(i >> 32),
                              (uint32_t)v ^ (step * 0x9E3779B9u), k0, k1 ^ step);
            Nv[i] = g[j];
          } else {
            g[j] = Nv[i];
          }
        }
      }
      if (grad) {
        const unsigned cf = gamma_der_series4(alpha, psi, g, ns, o);
        queued = cf != 0u;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (j < ns) {
            if (cf & (1u << j)) {
              cfq[atomicAdd(&cfn, 1)] = make_float4(alpha, psi, g[j], __int_as_float(j * 128 + (int)threadIdx.x));
            } else {
              Gv[(long long)(s0 + j) * nelem + e] = o[j];
            }
          }
        }
      }
    }
    // the queue is worked off (and emptied for the next group of draws) only when some lane filled it
    if (grad && __syncthreads_or(queued)) {
      const int nq = cfn;
      for (int t = threadIdx.x; t < nq; t += blockDim.x) {
        const float4 q = cfq[t];
        const int slot = __float_as_int(q.w);
        Gv[(long long)(s0 + (slot >> 7)) * nelem + e0 + (slot & 127)] = gamma_der_cf(q.x, q.y, q.z);
      }
      if (s0 + 4 < L.S) {
        __syncthreads();
        if (threadIdx.x == 0) cfn = 0;
        __syncthreads();
      }
    }
  }
}

// ------------------------------------------------------------------ draw -> operands
// Only the four Normal-based variables enter the operands (u, v per (d,k); w, s per feature), so this
// kernel initialises just those -- no lgamma / digamma of the InverseGamma factors (that was 80 % of
// its instructions) -- and needs softplus(t) alone, not its derivatives.  (Launch bounds: 0 = no
// occupancy target; the wide instantiations, KK >= 8, ask for 3 CTAs per SM, which keeps them free of spills.)
template <int KK>
__global__ void __launch_bounds__(128, KK >= 8 ? 3 : 0)
draw_operands_kernel(Layout L, const float* __restrict__ P, const float* __restrict__ N,
                     const float* __restrict__ eta, const int* __restrict__ rank, int SV, int KP,
                     float* __restrict__ Ap, float* __restrict__ EV, float* __restrict__ PH, int vw_identity) {
  const int lane = threadIdx.x & 31;
  const int d = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (d >= L.D) return;
  const int dr = rank ? rank[d] : d;      // table row of feature d (hot-column ordering)
  const long long D = L.D, DK = (long long)L.D * L.K;
  float ul[KK], us[KK], vl[KK], vs[KK];
#pragma unroll
  for (int i = 0; i < KK; ++i) {
    const int k = lane + 32 * i;
    ul[i] = us[i] = vl[i] = vs[i] = 0.f;
    if (k < L.K) {
      const long long e = (long long)d * L.K + k;
      ul[i] = P[L.toff[U_LOC] + e]; us[i] = softplusf(P[L.toff[U_RHO] + e]);
      vl[i] = P[L.toff[V_LOC] + e]; vs[i] = softplusf(P[L.toff[V_RHO] + e]);
    }
  }
  const float wl = P[L.toff[W_LOC] + d], wsg = softplusf(P[L.toff[W_RHO] + d]);
  const float s0l = P[L.toff[S_LOC] + d], s0s = softplusf(P[L.toff[S_RHO] + d]);
  const float s1l = P[L.toff[S_LOC] + D + d], s1s = softplusf(P[L.toff[S_RHO] + D + d]);
  const float eta_dec = eta[d], ieta_enc = 1.f / eta[D + d];
  // position of (sv, k) inside a record = position of (0, k) + sv * RG * VW  (spmf_record.cuh): the
  // integer divisions of rec_pos leave the draw loop
  const RecMap rm = rec_map(KP);
  const int sv_stride = rm.RG * rm.VW;
  int pos0[KK];
#pragma unroll
  for (int i = 0; i < KK; ++i) pos0[i] = (lane + 32 * i) < KP ? rec_pos(KP, SV, 0, lane + 32 * i) : 0;
  // per-feature quantities of draw s (a_d, b_d, phi) are computed by lane s % 32 and broadcast, not by all
  // 32 lanes redundantly (two softplus and a division per draw were a third of this kernel's instructions)
  for (int s0 = 0; s0 < L.S; s0 += 32) {
    const int sm = s0 + lane;
    float a_mine = 0.f;
    if (sm < L.S) {
      const float y0 = softplus4(fmaf(s0s, N[L.noff[VAR_S] + (long long)sm * 2 * D + d], s0l)).y;
      const float y1 = softplus4(fmaf(s1s, N[L.noff[VAR_S] + (long long)sm * 2 * D + D + d], s1l)).y;
      const float inv = 1.f / (y0 + y1);
      a_mine = y0 * inv;                                         // poisson.py:661-663
      const float tw = fmaf(wsg, N[L.noff[VAR_W] + (long long)sm * D + d], wl);
      const int qm = sm / SV, svm = sm - qm * SV;
      PH[((long long)qm * D + dr) * SV + svm] = eta_dec * (y1 * inv) * (vw_identity ? tw : softplus4(tw).y);   // poisson.py:694-701
    }
    const int ns = min(32, L.S - s0);
    for (int j = 0; j < ns; ++j) {
      const int s = s0 + j;
      const int q = s / SV, sv = s - q * SV;
      const float a_d = __shfl_sync(0xffffffffu, a_mine, j);
#pragma unroll
      for (int i = 0; i < KK; ++i) {
        const int k = lane + 32 * i;
        if (k < KP) {
          float ap = 0.f, ev = 0.f;
          if (k < L.K) {
            const long long e = (long long)s * DK + (long long)d * L.K + k;
            ap = a_d * softplus4(fmaf(us[i], N[L.noff[VAR_U] + e], ul[i])).y * ieta_enc;   // A' (poisson.py:665, 43)
            const float tv = fmaf(vs[i], N[L.noff[VAR_V] + e], vl[i]);
            ev = eta_dec * (vw_identity ? tv : softplus4(tv).y);                         // eta v (poisson.py:54)
          }
          const long long idx = ((long long)q * D + dr) * SV * KP + pos0[i] + sv * sv_stride;
          Ap[idx] = ap;
          EV[idx] = ev;
        }
      }
    }
  }
}

// Optional: materialise the draws themselves (API surface: surrogate_distribution.sample()).
// out[var][s][elem] in the same layout as the noise buffer.
__global__ void sample_kernel(Layout L, const float* __restrict__ P, const float* __restrict__ N,
                              float* __restrict__ out, int vw_identity) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  for (int v = 0; v < NUM_VARS; ++v) {
    long long n = L.vsize[v] * L.S;
    if (i < n) {
      long long e = i % L.vsize[v];
      float a = P[L.toff[2 * v] + e], b = P[L.toff[2 * v + 1] + e];
      float nz = N[L.noff[v] + i];
      float y;
      if (v <= VAR_S) {
        NParam p = nparam_init(a, b);
        y = ndraw_sel(p, nz, vw_identity && (v == VAR_V || v == VAR_W)).y;
      } else {
        y = softplusf(softplusf(b) / nz);
      }
      out[L.noff[v] + i] = y;
    }
  }
}

// ------------------------------------------------------------------ u_tau draws, per (s,k)
// utab[s][k] = utau_y (spmf_model.cuh): the one value of u_tau the (d,k) programs read, evaluated once
// per step here rather than D times per (s,k) inside them.
__global__ void utau_table_kernel(Layout L, const float* __restrict__ P, const float* __restrict__ N,
                                  float* __restrict__ utab) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= L.S * L.K) return;
  utab[i] = utau_y(softplusf(P[L.toff[UTAU_B] + i % L.K]), N[L.noff[VAR_UTAU] + i]);
}

static void launch_utau_table(const Layout& L, const float* P, const float* N, float* utab, cudaStream_t st) {
  utau_table_kernel<<<(L.S * L.K + 127) / 128, 128, 0, st>>>(L, P, N, utab);
}

// ------------------------------------------------------------------ backward, (d,k)-shaped tensors
// One warp per feature d, lanes over k: u, v, u_eta, u_eta_a.  Emits da[s][d] = sum_k GA' u / eta
// (needed by the per-feature kernel), the per-(s,d,k) contribution to d prior_u / d u_tau, and
// this feature's share of the prior / log q sums.
// PRE = true: the data-independent half of the backward (prior + entropy terms of every tensor, all
// loss parts) with the upstream data gradients taken as zero; it also stores, per (s,d,k), the three
// factors the data half needs -- cu = a_d sigmoid'(u)/eta_d, cv = eta_d sigmoid'(v), uy = u/eta_d -- so
// that backward_dk_post_kernel is a pure streaming pass.  The gradient is linear in the upstream
// terms, so pre + post == the one-pass kernel.  PRE runs on the side stream under the data term.
// Latent dims k0 + [0, 32*KK) of feature d: a warp covers a wide latent space in 128-wide chunks
// (backward_dk_wide_kernel) with the register budget of KK = 4.  The first chunk stores the per-(s,d)
// sums (da, prior / log q parts), later chunks add to them.  `lane` below is the latent index of lane 0
// of the chunk plus the lane, as the spmf_model.cuh bodies expect (k = lane + 32 * i).
#define SPMF_DK_PARAMS                                                                                  \
  Layout L, Hyper h, const float *__restrict__ P, const float *__restrict__ N, const float *__restrict__ G, \
      const float *__restrict__ eta, const int *__restrict__ rank, int SV, int KP,                       \
      const float *__restrict__ GAp, const float *__restrict__ GEVnz, const double *__restrict__ zcolsum, \
      float *__restrict__ grads, float *__restrict__ scr_utau, float *__restrict__ scr_parts,            \
      float *__restrict__ scr_da, float *__restrict__ fac, const float *__restrict__ utab,               \
      const int *__restrict__ gflag
#define SPMF_DK_ARGS L, h, P, N, G, eta, rank, SV, KP, GAp, GEVnz, zcolsum, grads, scr_utau, scr_parts, scr_da, fac, utab, gflag

template <int KK, bool PRE>
__device__ __forceinline__ void backward_dk_body(SPMF_DK_PARAMS, int k0, bool first) {
  const int wlane = threadIdx.x & 31, lane = k0 + wlane;
  const int d = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (d >= L.D) return;
  const int dr = (!PRE && rank) ? rank[d] : d;
  const bool dense = !PRE && gflag && *gflag;      // dense data term: no closed-form -sum_b z_b in GEV
  LaneState<KK> st;
  lane_init<KK>(st, L, P, d, lane, h.decay);
  const NParam s0 = nparam_init(P[L.toff[S_LOC] + d], P[L.toff[S_RHO] + d]);
  const NParam s1 = nparam_init(P[L.toff[S_LOC] + L.D + d], P[L.toff[S_RHO] + L.D + d]);
  const float eta_dec = eta[d], ieta = 1.f / eta[L.D + d];   // decoder scale, 1 / encoder divisor
  const RecMap rmap = rec_map(KP);                 // rec_pos(sv, k) = rec_pos(0, k) + sv * RG * VW
  const int sv_stride = rmap.RG * rmap.VW;
  int pos0[KK];
#pragma unroll
  for (int i = 0; i < KK; ++i) pos0[i] = (lane + 32 * i) < KP ? rec_pos(KP, SV, 0, lane + 32 * i) : 0;
  float a_mine[2] = {0.f, 0.f};                    // a_d of draws lane, lane + 32 (S <= 64 on this path)
#pragma unroll
  for (int h2 = 0; h2 < 2; ++h2) {
    const int sm = wlane + 32 * h2;
    if (sm < L.S) {
      const float y0 = ndraw(s0, N[L.noff[VAR_S] + (long long)sm * 2 * L.D + d]).y;
      const float y1 = ndraw(s1, N[L.noff[VAR_S] + (long long)sm * 2 * L.D + L.D + d]).y;
      a_mine[h2] = y0 / (y0 + y1);                          // poisson.py:661-663
    }
  }
  for (int s = 0; s < L.S; ++s) {
    const int q = s / SV, sv = s - q * SV;
    float a_d;
    if (L.S <= 64) {
      a_d = __shfl_sync(0xffffffffu, s < 32 ? a_mine[0] : a_mine[1], s & 31);
    } else {
      const float y0 = ndraw(s0, N[L.noff[VAR_S] + (long long)s * 2 * L.D + d]).y;
      const float y1 = ndraw(s1, N[L.noff[VAR_S] + (long long)s * 2 * L.D + L.D + d]).y;
      a_d = y0 / (y0 + y1);
    }
    float da = 0.f, pp[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int i = 0; i < KK; ++i) {
      int k = lane + 32 * i;
      if (k < L.K) {
        const int rp = pos0[i] + sv * sv_stride;
        long long idx = ((long long)q * L.D + dr) * SV * KP + rp;
        DkUp up;
        if constexpr (PRE) {
          up.GAp = 0.f;
          up.GEV = 0.f;
        } else {
          up.GAp = GAp[idx];
          up.GEV = GEVnz[idx] - (dense ? 0.f : (float)zcolsum[(long long)q * SV * KP + rp]);
        }
        DkOut o = lane_step<KK>(st, L, h, N, G, eta_dec, ieta, d, lane, i, s, a_d, __ldg(&utab[s * L.K + k]), up);
        if constexpr (PRE) {
          const long long e = ((long long)s * L.D + d) * L.K + k;
          const long long nsdk = (long long)L.S * L.D * L.K;
          fac[e] = a_d * ieta * o.usg;
          fac[nsdk + e] = eta_dec * o.vsg;
          fac[2 * nsdk + e] = o.uy * ieta;
        }
        da += o.da;
        scr_utau[((long long)s * L.D + d) * L.K + k] = o.dutau;
#pragma unroll
        for (int j = 0; j < 5; ++j) pp[j] += o.parts[j];
      }
    }
    da = warp_sum(da);
#pragma unroll
    for (int j = 0; j < 5; ++j) pp[j] = warp_sum(pp[j]);
    if (wlane == 0 && first) {
      if constexpr (!PRE) scr_da[(long long)s * L.D + d] = da;
      float* o = scr_parts + ((long long)d * L.S + s) * NUM_PARTS;
#pragma unroll
      for (int j = 0; j < NUM_PARTS; ++j) o[j] = 0.f;
      o[P_U] = pp[0]; o[P_V] = pp[1]; o[P_UETA] = pp[2]; o[P_UETAA] = pp[3]; o[P_LOGQ] = pp[4];
    } else if (wlane == 0) {
      if constexpr (!PRE) scr_da[(long long)s * L.D + d] += da;
      float* o = scr_parts + ((long long)d * L.S + s) * NUM_PARTS;
      o[P_U] += pp[0]; o[P_V] += pp[1]; o[P_UETA] += pp[2]; o[P_UETAA] += pp[3]; o[P_LOGQ] += pp[4];
    }
  }
  const float invS = 1.f / (float)L.S;
  const float wer = h.w_entropy * h.rep_scale;
#pragma unroll
  for (int i = 0; i < KK; ++i) {
    int k = lane + 32 * i;
    if (k < L.K) {
      long long e = (long long)d * L.K + k;
      nparam_finish(st.u[i], P[L.toff[U_RHO] + e], invS, wer, &grads[L.toff[U_LOC] + e], &grads[L.toff[U_RHO] + e]);
      nparam_finish(st.v[i], P[L.toff[V_RHO] + e], invS, wer, &grads[L.toff[V_LOC] + e], &grads[L.toff[V_RHO] + e]);
      gparam_finish(st.ue[i], P[L.toff[UETA_C] + e], P[L.toff[UETA_B] + e], invS, &grads[L.toff[UETA_C] + e], &grads[L.toff[UETA_B] + e]);
      gparam_finish(st.ua[i], P[L.toff[UETAA_C] + e], P[L.toff[UETAA_B] + e], invS, &grads[L.toff[UETAA_C] + e], &grads[L.toff[UETAA_B] + e]);
    }
  }
}

template <int KK, bool PRE>
__global__ void __launch_bounds__(128, KK == 1 ? 6 : 3) backward_dk_kernel(SPMF_DK_PARAMS) {
  backward_dk_body<KK, PRE>(SPMF_DK_ARGS, 0, true);
}

// KP in {256, 512}: the warp of feature d walks the latent space in chunks of 128
template <bool PRE>
__global__ void __launch_bounds__(128, 3) backward_dk_wide_kernel(SPMF_DK_PARAMS) {
  if (blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5) >= L.D) return;
  for (int k0 = 0; k0 < L.K; k0 += 128) backward_dk_body<4, PRE>(SPMF_DK_ARGS, k0, k0 == 0);
}

// Data half of the backward: u and v per (d,k) -- grads += (1/S) sum_s of the upstream terms times the
// stored factors (see PRE above) -- then, with da[s] = sum_k GA' u / eta still in registers, w and s of
// the same feature.
template <int KK>
__global__ void __launch_bounds__(128)
backward_dk_post_kernel(Layout L, Hyper h, const float* __restrict__ P, const float* __restrict__ N,
                        const float* __restrict__ eta, const int* __restrict__ rank, int SV, int KP,
                        const float* __restrict__ GAp, const float* __restrict__ GEVnz,
                        const float* __restrict__ Gphinz, const double* __restrict__ zcolsum,
                        const float* __restrict__ fac, float* __restrict__ grads, const int* __restrict__ gflag) {
  const int lane = threadIdx.x & 31;
  const int d = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (d >= L.D) return;
  const int dr = rank ? rank[d] : d;
  const bool dense = gflag && *gflag;              // dense data term: no closed-form terms (-sum z, -B)
  const float cf_rows = dense ? 0.f : h.batch_rows;
  const long long nsdk = (long long)L.S * L.D * L.K;
  float au[KK], aue[KK], av[KK], ave[KK];
#pragma unroll
  for (int i = 0; i < KK; ++i) { au[i] = 0.f; aue[i] = 0.f; av[i] = 0.f; ave[i] = 0.f; }
  float da_mine[2] = {0.f, 0.f};               // S <= 64 draws (checked by the launcher)
  const RecMap rmap = rec_map(KP);                 // rec_pos(sv, k) = rec_pos(0, k) + sv * RG * VW
  const int sv_stride = rmap.RG * rmap.VW;
  int pos0[KK];
#pragma unroll
  for (int i = 0; i < KK; ++i) pos0[i] = (lane + 32 * i) < KP ? rec_pos(KP, SV, 0, lane + 32 * i) : 0;
  for (int s = 0; s < L.S; ++s) {
    const int q = s / SV, sv = s - q * SV;
    float da = 0.f;
#pragma unroll
    for (int i = 0; i < KK; ++i) {
      const int k = lane + 32 * i;
      if (k < L.K) {
        const int rp = pos0[i] + sv * sv_stride;
        const long long idx = ((long long)q * L.D + dr) * SV * KP + rp;
        const long long e = ((long long)s * L.D + d) * L.K + k;
        const float ga = GAp[idx];
        const float gv = GEVnz[idx] - (dense ? 0.f : (float)zcolsum[(long long)q * SV * KP + rp]);
        const float dtu = -ga * fac[e], dtv = -gv * fac[nsdk + e];
        au[i] += dtu;
        aue[i] = fmaf(dtu, N[L.noff[VAR_U] + e], aue[i]);
        av[i] += dtv;
        ave[i] = fmaf(dtv, N[L.noff[VAR_V] + e], ave[i]);
        da = fmaf(ga, fac[2 * nsdk + e], da);
      }
    }
    da = warp_sum(da);
    if ((s & 31) == lane) da_mine[s >> 5] = da;       // lane s % 32 keeps draw s for the per-feature half below
  }
  const float invS = 1.f / (float)L.S;
  // per-feature tensors w, s (poisson.py:661-663, 694-701 chain rule): lane s takes draw s, the six
  // accumulators meet in a butterfly.  (Was a kernel of its own reading da[s][d] back.)
  {
    const long long D = L.D;
    FeatState f;
    f.w = nparam_init(P[L.toff[W_LOC] + d], P[L.toff[W_RHO] + d]);
    f.s0 = nparam_init(P[L.toff[S_LOC] + d], P[L.toff[S_RHO] + d]);
    f.s1 = nparam_init(P[L.toff[S_LOC] + D + d], P[L.toff[S_RHO] + D + d]);
    float aw = 0.f, awe = 0.f, a0 = 0.f, a0e = 0.f, a1 = 0.f, a1e = 0.f;
    for (int s = lane; s < L.S; s += 32) {
      const int q = s / SV, sv = s - q * SV;
      const FeatDraw fd = feat_draw(f, L, N, d, s, h.vw_identity);
      const float da = da_mine[s >> 5];
      const float Gphi = Gphinz[((long long)q * D + dr) * SV + sv] - cf_rows;          // d L / d phi_d
      const float dw_data = eta[d] * fd.b * Gphi;                                     // phi = eta b w
      const float db = eta[d] * fd.w.y * Gphi;
      const float inv = 1.f / (fd.s0.y + fd.s1.y), inv2 = inv * inv;
      const float ds0_data = (da - db) * fd.s1.y * inv2;
      const float ds1_data = (db - da) * fd.s0.y * inv2;
      const float tw = -dw_data * fd.w.sg, t0 = -ds0_data * fd.s0.sg, t1 = -ds1_data * fd.s1.sg;
      aw += tw;  awe = fmaf(tw, N[L.noff[VAR_W] + s * D + d], awe);
      a0 += t0;  a0e = fmaf(t0, N[L.noff[VAR_S] + s * 2 * D + d], a0e);
      a1 += t1;  a1e = fmaf(t1, N[L.noff[VAR_S] + s * 2 * D + D + d], a1e);
    }
    aw = warp_sum(aw);  awe = warp_sum(awe);
    a0 = warp_sum(a0);  a0e = warp_sum(a0e);
    a1 = warp_sum(a1);  a1e = warp_sum(a1e);
    if (lane == 0) {
      grads[L.toff[W_LOC] + d] += aw * invS;
      grads[L.toff[W_RHO] + d] += awe * invS * sigmoidf(P[L.toff[W_RHO] + d]);
      grads[L.toff[S_LOC] + d] += a0 * invS;
      grads[L.toff[S_RHO] + d] += a0e * invS * sigmoidf(P[L.toff[S_RHO] + d]);
      grads[L.toff[S_LOC] + D + d] += a1 * invS;
      grads[L.toff[S_RHO] + D + d] += a1e * invS * sigmoidf(P[L.toff[S_RHO] + D + d]);
    }
  }
#pragma unroll
  for (int i = 0; i < KK; ++i) {
    const int k = lane + 32 * i;
    if (k < L.K) {
      const long long e = (long long)d * L.K + k;
      grads[L.toff[U_LOC] + e] += au[i] * invS;
      grads[L.toff[U_RHO] + e] += aue[i] * invS * sigmoidf(P[L.toff[U_RHO] + e]);
      grads[L.toff[V_LOC] + e] += av[i] * invS;
      grads[L.toff[V_RHO] + e] += ave[i] * invS * sigmoidf(P[L.toff[V_RHO] + e]);
    }
  }
}

// ------------------------------------------------------------------ backward, per-feature tensors
// G = SV lanes per feature d, each taking every G-th draw: w, s, s_eta, s_tau, s_eta_a, s_tau_a
// (runs after backward_dk_kernel).  Accumulators meet through a fixed xor butterfly.
__device__ __forceinline__ void group_add(float& v, int G) {
  for (int o = G >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
}

__global__ void __launch_bounds__(128, 4)
backward_feat_kernel(Layout L, Hyper h, const float* __restrict__ P, const float* __restrict__ N,
                     const float* __restrict__ G, const float* __restrict__ eta,
                     const int* __restrict__ rank, int SV,
                     const float* __restrict__ Gphinz, const float* __restrict__ scr_da,
                     float* __restrict__ grads, float* __restrict__ scr_parts, int pre,
                     const int* __restrict__ gflag) {
  if (!pre && gflag && *gflag) h.batch_rows = 0.f;  // dense data term: Gphi carries no closed-form -B
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  const int dreal = t / SV, sg = t - dreal * SV;
  const bool valid = dreal < L.D;
  const int d = valid ? dreal : L.D - 1;           // out-of-range lanes shadow the last feature (no writes)
  const int dr = (!pre && rank) ? rank[d] : d;
  FeatState f;
  feat_init(f, L, P, d);
  for (int s = sg; s < L.S; s += SV) {
    const int q = s / SV, sv = s - q * SV;
    FeatDraw fd = feat_draw(f, L, N, d, s, h.vw_identity);
    float fp[7];
    // pre: data-independent half (upstream da = 0, dL/dphi = 0); the data half of backward_dk_post_kernel adds the rest
    feat_step(f, fd, L, h, N, G, eta, d, s, pre ? 0.f : scr_da[(long long)s * L.D + d],
              pre ? h.batch_rows : Gphinz[((long long)q * L.D + dr) * SV + sv], fp);
    if (valid) {
      float* o = scr_parts + ((long long)d * L.S + s) * NUM_PARTS;
      o[P_W] = fp[0]; o[P_S] = fp[1]; o[P_SETA] = fp[2]; o[P_STAU] = fp[3];
      o[P_SETAA] = fp[4]; o[P_STAUA] = fp[5]; o[P_LOGQ] += fp[6];
    }
  }
  NParam* np[3] = {&f.w, &f.s0, &f.s1};
  GParam* gp[6] = {&f.se0, &f.se1, &f.st, &f.sea0, &f.sea1, &f.sta};
#pragma unroll
  for (int i = 0; i < 3; ++i) { group_add(np[i]->acc_dt, SV); group_add(np[i]->acc_dte, SV); }
#pragma unroll
  for (int i = 0; i < 6; ++i) { group_add(gp[i]->acc_da, SV); group_add(gp[i]->acc_db, SV); }
  if (!valid || sg != 0) return;
  const float invS = 1.f / (float)L.S;
  const float wer = h.w_entropy * h.rep_scale;
  const int D = L.D;
  nparam_finish(f.w, P[L.toff[W_RHO] + d], invS, wer, &grads[L.toff[W_LOC] + d], &grads[L.toff[W_RHO] + d]);
  nparam_finish(f.s0, P[L.toff[S_RHO] + d], invS, wer, &grads[L.toff[S_LOC] + d], &grads[L.toff[S_RHO] + d]);
  nparam_finish(f.s1, P[L.toff[S_RHO] + D + d], invS, wer, &grads[L.toff[S_LOC] + D + d], &grads[L.toff[S_RHO] + D + d]);
  gparam_finish(f.se0, P[L.toff[SETA_C] + d], P[L.toff[SETA_B] + d], invS, &grads[L.toff[SETA_C] + d], &grads[L.toff[SETA_B] + d]);
  gparam_finish(f.se1, P[L.toff[SETA_C] + D + d], P[L.toff[SETA_B] + D + d], invS, &grads[L.toff[SETA_C] + D + d], &grads[L.toff[SETA_B] + D + d]);
  gparam_finish(f.st, P[L.toff[STAU_C] + d], P[L.toff[STAU_B] + d], invS, &grads[L.toff[STAU_C] + d], &grads[L.toff[STAU_B] + d]);
  gparam_finish(f.sea0, P[L.toff[SETAA_C] + d], P[L.toff[SETAA_B] + d], invS, &grads[L.toff[SETAA_C] + d], &grads[L.toff[SETAA_B] + d]);
  gparam_finish(f.sea1, P[L.toff[SETAA_C] + D + d], P[L.toff[SETAA_B] + D + d], invS, &grads[L.toff[SETAA_C] + D + d], &grads[L.toff[SETAA_B] + D + d]);
  gparam_finish(f.sta, P[L.toff[STAUA_C] + d], P[L.toff[STAUA_B] + d], invS, &grads[L.toff[STAUA_C] + d], &grads[L.toff[STAUA_B] + d]);
}

// ------------------------------------------------------------------ backward (per latent k)
__global__ void backward_lat_kernel(Layout L, Hyper h, const float* __restrict__ P,
                                    const float* __restrict__ N, const float* __restrict__ G,
                                    const double* __restrict__ dutau,
                                    float* __restrict__ grads, float* __restrict__ scr_lat) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= L.K) return;
  LatState t;
  lat_init(t, L, P, k);
  for (int s = 0; s < L.S; ++s) {
    float pp[3];
    lat_step(t, L, h, N, G, k, s, (float)dutau[(long long)s * L.K + k], pp);
    float* o = scr_lat + ((long long)k * L.S + s) * NUM_PARTS;
    for (int j = 0; j < NUM_PARTS; ++j) o[j] = 0.f;
    o[P_UTAU] = pp[0]; o[P_UTAUA] = pp[1]; o[P_LOGQ] = pp[2];
  }
  const float invS = 1.f / (float)L.S;
  gparam_finish(t.ut, P[L.toff[UTAU_C] + k], P[L.toff[UTAU_B] + k], invS, &grads[L.toff[UTAU_C] + k], &grads[L.toff[UTAU_B] + k]);
  gparam_finish(t.uta, P[L.toff[UTAUA_C] + k], P[L.toff[UTAUA_B] + k], invS, &grads[L.toff[UTAUA_C] + k], &grads[L.toff[UTAUA_B] + k]);
}

// ------------------------------------------------------------------ deterministic reductions
// out[q][split][c] = sum over rows of in[q][row][c] for rows of this split (fixed order).
template <typename TIn>
__global__ void reduce_rows_kernel(const TIn* __restrict__ in, double* __restrict__ out,
                                   long long n, int c, int nsplit) {
  __shared__ double sm[8][33];
  const int cx = blockIdx.x * 32 + threadIdx.x;
  const int split = blockIdx.y, q = blockIdx.z;
  const long long chunk = (n + nsplit - 1) / nsplit;
  const long long r0 = split * chunk;
  long long r1 = r0 + chunk;
  if (r1 > n) r1 = n;
  double acc = 0.0;
  if (cx < c) {
    const TIn* base = in + (long long)q * n * c + cx;
    for (long long r = r0 + threadIdx.y; r < r1; r += 8) acc += (double)base[r * c];
  }
  sm[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && cx < c) {
    double t = 0.0;
#pragma unroll
    for (int j = 0; j < 8; ++j) t += sm[j][threadIdx.x];
    out[((long long)q * nsplit + split) * c + cx] = t;
  }
}

// parts[s][p] (double) and loss from the reduced pieces.
//   featparts[S*16], latparts[S*16]: prior/logq sums;
//   data[NQ][4][SV]: (sum_nz x log lam - sum lgamma(x+1), sum z.vsum, sum z^2, #non-finite)
//   Lx = sum_nz [x log lam - lgamma(x+1)] - sum z.vsum - B * phisum   (SURVEY 3.4 closed form)
//   Lz = B*K*0.5*log(2/pi) - 0.5 * sum z^2                            (poisson.py:599-604)
__global__ void finalize_parts_kernel(int S, int SV, int K, const double* __restrict__ featparts,
                                      const double* __restrict__ latparts,
                                      const double* __restrict__ data, const double* __restrict__ phisum,
                                      double batch_rows, double w_entropy,
                                      double w_prior, double* __restrict__ parts_out,
                                      float* __restrict__ comm, GuardState* __restrict__ gs) {
  int s = threadIdx.x;
  const int gflag = gs ? gs->flag : 0;
  const double min_val = gs ? (double)guard_min_val(gs->minkey) : 0.0;
  __syncthreads();
  if (gs && threadIdx.x == 0) {        // last reader of the step: re-arm the guard for the next one
    gs->flag = gflag & 2;              // (the dense-link bit is configuration, not state; bit 2 = barrier
                                       //  failure of the slow path, sticky in the reports only)
    gs->nbad = 0;
    gs->minkey = ~0ull;
  }
  if (s >= S) return;
  double* o = parts_out + (long long)s * NUM_PARTS;
  for (int p = 0; p <= P_LOGQ; ++p) o[p] = featparts[s * NUM_PARTS + p] + latparts[s * NUM_PARTS + p];
  const int q = s / SV, sv = s - q * SV;
  const double* dd = data + ((long long)q * 4) * SV;   // data[q][4][SV]
  double xlog = dd[0 * SV + sv], zv = dd[1 * SV + sv], z2 = dd[2 * SV + sv];
  if (gflag) {
    // dense data term: dd[0] already sums the finite entries; the others take min(finite) - 10
    // (poisson.py:606-616)
    const double nb = dd[3 * SV + sv];
    o[P_X] = xlog + (nb > 0.0 ? nb * min_val : 0.0);
  } else {
    o[P_X] = xlog - zv - batch_rows * phisum[q * SV + sv];
  }
  o[P_Z] = batch_rows * (double)K * (double)kHalfLog2OverPi - 0.5 * z2;
  double prior = 0.0;
  for (int p = 0; p < P_LOGQ; ++p) prior += o[p];
  o[15] = w_entropy * o[P_LOGQ] - w_prior * prior - o[P_Z] - o[P_X];   // per-draw loss
  // data parts as (hi, lo) float pairs inside the all-reduced gradient block: summed across ranks
  // by the same collective as the gradients and recombined in double on the host side.
  if (4 * s + 3 < kCommSlack) {
    float zh = (float)o[P_Z], xh = (float)o[P_X];
    comm[4 * s + 0] = zh; comm[4 * s + 1] = (float)(o[P_Z] - (double)zh);
    comm[4 * s + 2] = xh; comm[4 * s + 3] = (float)(o[P_X] - (double)xh);
  }
}

// After the all-reduce of the gradient block: recombine the summed ('z','x') (hi,lo) pairs into
// parts[s][13..14], recompute the per-draw loss, emit the mean loss, clear the scalar slack.
__global__ void unpack_parts_kernel(int S, double w_entropy, double w_prior, float* __restrict__ comm, int slack,
                                    double* __restrict__ parts, double* __restrict__ loss_out) {
  __shared__ double sl[64];
  const int s = threadIdx.x;
  double l = 0.0;
  if (s < S) {
    double* o = parts + (long long)s * NUM_PARTS;
    o[P_Z] = (double)comm[4 * s + 0] + (double)comm[4 * s + 1];
    o[P_X] = (double)comm[4 * s + 2] + (double)comm[4 * s + 3];
    double prior = 0.0;
    for (int p = 0; p < P_LOGQ; ++p) prior += o[p];
    l = w_entropy * o[P_LOGQ] - w_prior * prior - o[P_Z] - o[P_X];
    o[15] = l;
  }
  if (s < 64) sl[s] = l;
  __syncthreads();
  for (int i = threadIdx.x; i < slack; i += blockDim.x) comm[i] = 0.f;
  if (s == 0) {
    double t = 0.0;
    for (int i = 0; i < S && i < 64; ++i) t += sl[i];
    *loss_out = t / (double)S;
  }
}

// blocks [0, n/256): Adam over the all-reduced gradient block; the extra last block: unpack_parts_kernel's job
__global__ void unpack_adam_kernel(int S, double w_entropy, double w_prior, float* __restrict__ comm, int slack,
                                   double* __restrict__ parts, double* __restrict__ loss_out,
                                   const float* __restrict__ g, long long n, AdamCfg adam) {
  if (blockIdx.x + 1 < gridDim.x) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long c0 = comm - g;                       // the scalar slack is bookkeeping, not a gradient
    if (i < n && adam.lr > 0.f && !(i >= c0 && i < c0 + slack)) adam_apply(adam, i, g[i]);
    return;
  }
  __shared__ double sl[64];
  const int s = threadIdx.x;
  double l = 0.0;
  if (s < S) {
    double* o = parts + (long long)s * NUM_PARTS;
    o[P_Z] = (double)comm[4 * s + 0] + (double)comm[4 * s + 1];
    o[P_X] = (double)comm[4 * s + 2] + (double)comm[4 * s + 3];
    double prior = 0.0;
    for (int p = 0; p < P_LOGQ; ++p) prior += o[p];
    l = w_entropy * o[P_LOGQ] - w_prior * prior - o[P_Z] - o[P_X];
    o[15] = l;
  }
  if (s < 64) sl[s] = l;
  __syncthreads();
  for (int i = threadIdx.x; i < slack; i += blockDim.x) comm[i] = 0.f;
  if (s == 0) {
    double t = 0.0;
    for (int i = 0; i < S && i < 64; ++i) t += sl[i];
    *loss_out = t / (double)S;
  }
}

// ------------------------------------------------------------------ Adam  [EXT L4]
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, long long n, float lr, float b1, float b2, float eps,
                            float bc1, float bc2, float clip_value, float grad_scale,
                            const StepState* __restrict__ sst) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  if (sst) { lr = sst->lr; b1 = sst->b1; b2 = sst->b2; eps = sst->eps; bc1 = sst->bc1; bc2 = sst->bc2; clip_value = sst->clip; }
  float gi = g[i] * grad_scale;
  if (!isfinite(gi)) gi = 0.f;                 // non-finite gradients are dropped, not propagated
  if (clip_value > 0.f) gi = fminf(fmaxf(gi, -clip_value), clip_value);
  float mi = b1 * m[i] + (1.f - b1) * gi;
  float vi = b2 * v[i] + (1.f - b2) * gi * gi;
  m[i] = mi;
  v[i] = vi;
  p[i] -= lr * (mi / bc1) / (sqrtf(vi / bc2) + eps);
}

__global__ void step_state_kernel(StepState* dst, StepState v) { *dst = v; }

// sum of squares (double) of a float vector, deterministic two-stage via reduce_rows
__global__ void square_kernel(const float* __restrict__ g, float* __restrict__ out, long long n) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) {
    float x = g[i];
    out[i] = isfinite(x) ? x * x : 0.f;
  }
}

static Hyper make_hyper(float u_tau_scale, float s_tau_scale, float decay, float w_entropy,
                        float w_prior, int world, float batch_rows, int model = 0) {
  Hyper h;
  h.vw_identity = model == SPMF_MODEL_BERNOULLI;
  h.u_tau_b = 1.f / (u_tau_scale * u_tau_scale);
  h.s_tau_b = 1.f / (s_tau_scale * s_tau_scale);
  h.decay = decay;
  h.w_entropy = w_entropy;
  h.w_prior = w_prior;
  h.rep_scale = 1.f / (float)world;
  h.batch_rows = batch_rows;
  return h;
}

static AdamCfg make_adam(const spmf_adam_args* a) {
  AdamCfg c{};
  if (!a || !(a->lr > 0.f) || !a->params || !a->m || !a->v || a->step <= 0) return c;     // lr = 0: off
  c.lr = a->lr; c.b1 = a->beta1; c.b2 = a->beta2; c.eps = a->eps;
  c.bc1 = 1.f - powf(a->beta1, (float)a->step);
  c.bc2 = 1.f - powf(a->beta2, (float)a->step);
  c.clip = a->clip_value;
  c.grad_scale = a->grad_scale > 0.f ? a->grad_scale : 1.f;
  c.p = a->params; c.m = a->m; c.v = a->v;
  return c;
}

static int nsplit_for(long long n) {
  long long s = (n + 255) / 256;
  if (s < 1) s = 1;
  if (s > 64) s = 64;
  return (int)s;
}

// Two independent column-sum jobs per launch (they always come in pairs around the data term).
struct RJob { const void* in; double* out; long long n; int c, q, ns; };

template <typename TIn>
__global__ void reduce_rows2_kernel(RJob A, RJob B) {
  __shared__ double sm[8][33];
  const bool isB = (int)blockIdx.z >= A.q;
  const RJob J = isB ? B : A;
  const int q = isB ? blockIdx.z - A.q : blockIdx.z;
  const int split = blockIdx.y;
  if (split >= J.ns || (int)blockIdx.x * 32 >= J.c) return;
  const int cx = blockIdx.x * 32 + threadIdx.x;
  const long long chunk = (J.n + J.ns - 1) / J.ns;
  const long long r0 = split * chunk;
  long long r1 = r0 + chunk;
  if (r1 > J.n) r1 = J.n;
  double acc = 0.0;
  if (cx < J.c) {
    const TIn* base = (const TIn*)J.in + (long long)q * J.n * J.c + cx;
    for (long long r = r0 + threadIdx.y; r < r1; r += 8) acc += (double)base[r * J.c];
  }
  sm[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && cx < J.c) {
    double t = 0.0;
#pragma unroll
    for (int j = 0; j < 8; ++j) t += sm[j][threadIdx.x];
    J.out[((long long)q * J.ns + split) * J.c + cx] = t;
  }
}

// outA/outB = column sums of two float arrays; 2 launches in total (fixed summation order).
static int reduce_rows_pair(const float* inA, double* outA, long long nA, int cA, int qA,
                            const float* inB, double* outB, long long nB, int cB, int qB,
                            double* scratch, cudaStream_t st) {
  if (nA <= 0 || cA <= 0 || qA <= 0 || nB <= 0 || cB <= 0 || qB <= 0) return SPMF_ERR_BAD_ARG;
  const int nsA = nsplit_for(nA), nsB = nsplit_for(nB);
  double* pA = scratch;
  double* pB = scratch + (long long)qA * nsA * cA;
  const int cmax = cA > cB ? cA : cB, nsmax = nsA > nsB ? nsA : nsB;
  dim3 blk(32, 8);
  RJob a1{inA, nsA == 1 ? outA : pA, nA, cA, qA, nsA}, b1{inB, nsB == 1 ? outB : pB, nB, cB, qB, nsB};
  reduce_rows2_kernel<float><<<dim3((cmax + 31) / 32, nsmax, qA + qB), blk, 0, st>>>(a1, b1);
  if (nsA > 1 || nsB > 1) {
    // second stage over the split partials; a job that needed no split gets an empty descriptor
    RJob a2{pA, outA, nsA, cA, nsA > 1 ? qA : 0, 1}, b2{pB, outB, nsB, cB, nsB > 1 ? qB : 0, 1};
    if (a2.q + b2.q > 0)
      reduce_rows2_kernel<double><<<dim3((cmax + 31) / 32, 1, a2.q + b2.q), blk, 0, st>>>(a2, b2);
  }
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

// out (double[q][c]) = column sums of in[q][n][c]; scratch needs q*nsplit*c doubles.
template <typename TIn>
static int reduce_rows(const TIn* in, double* out, double* scratch, long long n, int c, int q,
                       cudaStream_t st) {
  if (n <= 0 || c <= 0 || q <= 0) return SPMF_ERR_BAD_ARG;
  int ns = nsplit_for(n);
  dim3 blk(32, 8);
  if (ns == 1) {
    reduce_rows_kernel<TIn><<<dim3((c + 31) / 32, 1, q), blk, 0, st>>>(in, out, n, c, 1);
  } else {
    reduce_rows_kernel<TIn><<<dim3((c + 31) / 32, ns, q), blk, 0, st>>>(in, scratch, n, c, ns);
    reduce_rows_kernel<double><<<dim3((c + 31) / 32, 1, q), blk, 0, st>>>(scratch, out, ns, c, 1);
  }
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

}  // namespace spmf

using namespace spmf;

extern "C" {

int spmf_kpad(int K) {
  int kp = 1;
  while (kp < K) kp <<= 1;
  return kp;
}

int spmf_draw_vec(int S) { return (S % 4 == 0) ? 4 : (S % 2 == 0) ? 2 : 1; }

// A gather record holds at most 512 floats (one warp-wide slot of 16 floats per lane, spmf_sparse.cu):
// wide latent spaces take fewer draws per record.  KP <= 128 always fits 4 draws, so there this is
// spmf_draw_vec(S).
int spmf_draw_vec_k(int K, int S) {
  const int KP = spmf_kpad(K);
  for (int sv = 4; sv > 1; sv >>= 1)
    if (S % sv == 0 && (long long)KP * sv <= 512) return sv;
  return 1;
}

int spmf_rec_pos(int KP, int SV, int sv, int k) {
  if (KP <= 0 || (KP & (KP - 1)) || SV <= 0 || sv < 0 || sv >= SV || k < 0 || k >= KP) return SPMF_ERR_BAD_ARG;
  return rec_pos(KP, SV, sv, k);
}

int spmf_layout(int D, int K, int S, long long* tensor_offsets, long long* noise_offsets) {
  if (D <= 0 || K <= 0 || S <= 0 || K > SPMF_MAX_K) return SPMF_ERR_BAD_ARG;
  Layout L = make_layout(D, K, S);
  for (int i = 0; i <= NUM_TENSORS; ++i) tensor_offsets[i] = L.toff[i];
  for (int i = 0; i <= NUM_VARS; ++i) noise_offsets[i] = L.noff[i];
  return SPMF_OK;
}

int spmf_fill_noise(float* noise, const float* params, int D, int K, int S, unsigned long long seed,
                    unsigned int step, int which, void* stream) {
  return spmf_fill_noise_dev(noise, params, D, K, S, seed, step, which, nullptr, stream);
}

int spmf_fill_noise_dev(float* noise, const float* params, int D, int K, int S, unsigned long long seed,
                        unsigned int step, int which, const void* step_state, void* stream) {
  const StepState* sst = (const StepState*)step_state;
  if (!noise || !params || D <= 0 || K <= 0 || S <= 0 || K > SPMF_MAX_K || !(which & 3)) return SPMF_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  Layout L = make_layout(D, K, S);
  uint32_t k0 = (uint32_t)(seed & 0xffffffffu), k1 = (uint32_t)(seed >> 32);
  long long nmax = (long long)D * K * S;
  if (nmax < 2LL * D * S) nmax = 2LL * D * S;
  if (which & SPMF_NOISE_NORMAL) {
    dim3 grid((unsigned)(((nmax + 3) / 4 + 255) / 256), VAR_S + 1);
    fill_normal_kernel<<<grid, 256, 0, st>>>(L, noise, step, k0, k1, sst);
  }
  if (which & SPMF_NOISE_GAMMA) {
    gamma_kernel<<<gamma_grid_blocks(L), 128, 0, st>>>(L, params, noise, noise, 1, 0, step, k0, k1, sst);
  }
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_sample(const float* params, const float* noise, int D, int K, int S, float* samples,
                void* stream) {
  return spmf_sample_m(params, noise, D, K, S, samples, SPMF_MODEL_POISSON, stream);
}

int spmf_sample_m(const float* params, const float* noise, int D, int K, int S, float* samples, int model,
                  void* stream) {
  if (!params || !noise || !samples || K > SPMF_MAX_K) return SPMF_ERR_BAD_ARG;
  Layout L = make_layout(D, K, S);
  long long nmax = (long long)D * K * S;
  if (nmax < 2LL * D * S) nmax = 2LL * D * S;
  sample_kernel<<<(unsigned)((nmax + 255) / 256), 256, 0, (cudaStream_t)stream>>>(L, params, noise, samples, model == SPMF_MODEL_BERNOULLI);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_draw_operands(const float* params, const float* noise, const float* eta, int D, int K, int S,
                       float* Ap, float* EV, float* PH, double* vsum, double* phisum,
                       double* scratch, void* stream) {
  return spmf_draw_operands_ranked(params, noise, eta, nullptr, D, K, S, Ap, EV, PH, vsum, phisum, scratch, stream);
}

int spmf_draw_operands_ranked(const float* params, const float* noise, const float* eta, const int* rank,
                              int D, int K, int S, float* Ap, float* EV, float* PH, double* vsum,
                              double* phisum, double* scratch, void* stream) {
  return spmf_draw_operands_ranked_m(params, noise, eta, rank, D, K, S, Ap, EV, PH, vsum, phisum, scratch,
                                     SPMF_MODEL_POISSON, stream);
}

int spmf_draw_operands_ranked_m(const float* params, const float* noise, const float* eta, const int* rank,
                                int D, int K, int S, float* Ap, float* EV, float* PH, double* vsum,
                                double* phisum, double* scratch, int model, void* stream) {
  const int vwid = model == SPMF_MODEL_BERNOULLI;
  if (!params || !noise || !eta || !Ap || !EV || !PH) return SPMF_ERR_BAD_ARG;
  if ((vsum == nullptr) != (phisum == nullptr) || (vsum && !scratch)) return SPMF_ERR_BAD_ARG;
  if (D <= 0 || K <= 0 || S <= 0 || K > SPMF_MAX_K) return SPMF_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  Layout L = make_layout(D, K, S);
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S);
  dim3 grid((D + 3) / 4);
  if (KP <= 32) draw_operands_kernel<1><<<grid, 128, 0, st>>>(L, params, noise, eta, rank, SV, KP, Ap, EV, PH, vwid);
  else if (KP <= 64) draw_operands_kernel<2><<<grid, 128, 0, st>>>(L, params, noise, eta, rank, SV, KP, Ap, EV, PH, vwid);
  else if (KP <= 128) draw_operands_kernel<4><<<grid, 128, 0, st>>>(L, params, noise, eta, rank, SV, KP, Ap, EV, PH, vwid);
  else if (KP == 256) draw_operands_kernel<8><<<grid, 128, 0, st>>>(L, params, noise, eta, rank, SV, KP, Ap, EV, PH, vwid);
  else if (KP == 512) draw_operands_kernel<16><<<grid, 128, 0, st>>>(L, params, noise, eta, rank, SV, KP, Ap, EV, PH, vwid);
  else return SPMF_ERR_UNSUPPORTED;
  SPMF_CHECK_LAUNCH();
  if (!vsum) return SPMF_OK;        // the caller runs spmf_operand_sums itself (on another stream)
  return spmf_operand_sums(EV, PH, D, K, S, vsum, phisum, scratch, stream);
}

/* vsum[q][rec] = sum_d EV, phisum[q][sv] = sum_d PH (fp64): the closed-form -sum lambda terms. */
int spmf_operand_sums(const float* EV, const float* PH, int D, int K, int S, double* vsum, double* phisum,
                      double* scratch, void* stream) {
  if (!EV || !PH || !vsum || !phisum || !scratch) return SPMF_ERR_BAD_ARG;
  if (D <= 0 || K <= 0 || S <= 0 || K > SPMF_MAX_K) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  return reduce_rows_pair(EV, vsum, D, KP * SV, NQ, PH, phisum, D, SV, NQ, scratch, (cudaStream_t)stream);
}

int spmf_gamma_grad(const float* params, const float* noise, int D, int K, int S, float* dgda,
                    void* stream) {
  if (!params || !noise || !dgda || D <= 0 || K <= 0 || S <= 0 || K > SPMF_MAX_K) return SPMF_ERR_BAD_ARG;
  Layout L = make_layout(D, K, S);
  gamma_kernel<<<gamma_grid_blocks(L), 128, 0, (cudaStream_t)stream>>>(L, params, const_cast<float*>(noise), dgda, 0, 1, 0, 0, 0, nullptr);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

/* Gamma draws and their implicit gradients in one pass (what a training step uses). */
int spmf_gamma_draw_grad(const float* params, float* noise, float* dgda, int D, int K, int S,
                         unsigned long long seed, unsigned int step, void* stream) {
  return spmf_gamma_draw_grad_dev(params, noise, dgda, D, K, S, seed, step, nullptr, stream);
}

int spmf_gamma_draw_grad_dev(const float* params, float* noise, float* dgda, int D, int K, int S,
                             unsigned long long seed, unsigned int step, const void* step_state, void* stream) {
  if (!params || !noise || !dgda || D <= 0 || K <= 0 || S <= 0 || K > SPMF_MAX_K) return SPMF_ERR_BAD_ARG;
  Layout L = make_layout(D, K, S);
  gamma_kernel<<<gamma_grid_blocks(L), 128, 0, (cudaStream_t)stream>>>(L, params, noise, dgda, 1, 1, step,
                                                      (uint32_t)(seed & 0xffffffffu), (uint32_t)(seed >> 32),
                                                      (const StepState*)step_state);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_backward_params(const float* params, const float* noise, const float* dgda, const float* eta,
                         int D, int K, int S, const float* GAp, const float* GEVnz, const float* Gphinz,
                         const double* zcolsum, const double* datasums, const double* phisum,
                         float batch_rows, float u_tau_scale, float s_tau_scale,
                         float decay, float w_entropy, float w_prior, int world_size, float* grads,
                         double* parts, float* scr_f, double* scr_d, void* gs, void* stream) {
  return spmf_backward_params_ranked(params, noise, dgda, eta, nullptr, D, K, S, GAp, GEVnz, Gphinz, zcolsum,
                                     datasums, phisum, batch_rows, u_tau_scale, s_tau_scale, decay, w_entropy,
                                     w_prior, world_size, grads, parts, scr_f, scr_d, gs, stream);
}

int spmf_backward_params_ranked(const float* params, const float* noise, const float* dgda, const float* eta,
                                const int* rank, int D, int K, int S, const float* GAp, const float* GEVnz,
                                const float* Gphinz, const double* zcolsum, const double* datasums,
                                const double* phisum, float batch_rows, float u_tau_scale, float s_tau_scale,
                                float decay, float w_entropy, float w_prior, int world_size, float* grads,
                                double* parts, float* scr_f, double* scr_d, void* gs, void* stream) {
  return spmf_backward_params_ranked_m(params, noise, dgda, eta, rank, D, K, S, GAp, GEVnz, Gphinz, zcolsum, datasums,
                                       phisum, batch_rows, u_tau_scale, s_tau_scale, decay, w_entropy, w_prior,
                                       world_size, grads, parts, scr_f, scr_d, gs, SPMF_MODEL_POISSON, stream);
}

int spmf_backward_params_ranked_m(const float* params, const float* noise, const float* dgda, const float* eta,
                                  const int* rank, int D, int K, int S, const float* GAp, const float* GEVnz,
                                  const float* Gphinz, const double* zcolsum, const double* datasums,
                                  const double* phisum, float batch_rows, float u_tau_scale, float s_tau_scale,
                                  float decay, float w_entropy, float w_prior, int world_size, float* grads,
                                  double* parts, float* scr_f, double* scr_d, void* gs, int model, void* stream) {
  if (!params || !noise || !dgda || !eta || !GAp || !GEVnz || !Gphinz || !zcolsum || !datasums ||
      !phisum || !grads || !parts || !scr_f || !scr_d)
    return SPMF_ERR_BAD_ARG;
  if (D <= 0 || K <= 0 || S <= 0 || K > SPMF_MAX_K || world_size <= 0) return SPMF_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  Layout L = make_layout(D, K, S);
  Hyper h = make_hyper(u_tau_scale, s_tau_scale, decay, w_entropy, w_prior, world_size, batch_rows, model);
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S);
  // float scratch: scr_utau [S][D][K] | scr_parts [D][S*16] | scr_lat [K][S*16] | scr_da [S][D] |
  // (fac [3][S][D][K], split backward only) | utab [S][K]
  float* scr_utau = scr_f;
  float* scr_parts = scr_utau + (long long)S * D * K;
  float* scr_lat = scr_parts + (long long)D * S * NUM_PARTS;
  // double scratch: dutau [S][K] | featparts [S*16] | latparts [S*16] | reduce scratch
  double* dutau = scr_d;
  double* featparts = dutau + (long long)S * K;
  double* latparts = featparts + (long long)S * NUM_PARTS;
  double* rscr = latparts + (long long)S * NUM_PARTS;
  float* scr_da = scr_lat + (long long)K * S * NUM_PARTS;
  float* utab = scr_da + (long long)S * D + 3LL * S * D * K;
  dim3 grid((D + 3) / 4);
  launch_utau_table(L, params, noise, utab, st);
  if (KP <= 32) backward_dk_kernel<1, false><<<grid, 128, 0, st>>>(L, h, params, noise, dgda, eta, rank, SV, KP, GAp, GEVnz, zcolsum, grads, scr_utau, scr_parts, scr_da, nullptr, utab, (const int*)gs);
  else if (KP <= 64) backward_dk_kernel<2, false><<<grid, 128, 0, st>>>(L, h, params, noise, dgda, eta, rank, SV, KP, GAp, GEVnz, zcolsum, grads, scr_utau, scr_parts, scr_da, nullptr, utab, (const int*)gs);
  else if (KP <= 128) backward_dk_kernel<4, false><<<grid, 128, 0, st>>>(L, h, params, noise, dgda, eta, rank, SV, KP, GAp, GEVnz, zcolsum, grads, scr_utau, scr_parts, scr_da, nullptr, utab, (const int*)gs);
  else if (KP <= 512) backward_dk_wide_kernel<false><<<grid, 128, 0, st>>>(L, h, params, noise, dgda, eta, rank, SV, KP, GAp, GEVnz, zcolsum, grads, scr_utau, scr_parts, scr_da, nullptr, utab, (const int*)gs);
  else return SPMF_ERR_UNSUPPORTED;
  backward_feat_kernel<<<(int)(((long long)D * SV + 127) / 128), 128, 0, st>>>(L, h, params, noise, dgda, eta, rank, SV, Gphinz, scr_da, grads, scr_parts, 0, (const int*)gs);
  SPMF_CHECK_LAUNCH();
  int rc = reduce_rows_pair(scr_utau, dutau, D, K, S, scr_parts, featparts, D, S * NUM_PARTS, 1, rscr, st);
  if (rc) return rc;
  backward_lat_kernel<<<(K + 63) / 64, 64, 0, st>>>(L, h, params, noise, dgda, dutau, grads, scr_lat);
  SPMF_CHECK_LAUNCH();
  rc = reduce_rows<float>(scr_lat, latparts, rscr, K, S * NUM_PARTS, 1, st);
  if (rc) return rc;
  finalize_parts_kernel<<<1, ((S + 31) / 32) * 32, 0, st>>>(S, SV, K, featparts, latparts, datasums, phisum,
                                                           (double)batch_rows,
                                                           (double)w_entropy, (double)w_prior, parts,
                                                           grads + L.comm_off, (GuardState*)gs);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

long long spmf_backward_scratch_floats(int D, int K, int S) {
  // scr_utau | scr_parts | scr_lat | scr_da | fac (3 factors per (s,d,k), split backward only) | utab
  return 4LL * S * D * K + (long long)D * S * NUM_PARTS + (long long)K * S * NUM_PARTS + (long long)S * D +
         (long long)S * K;
}

/* Split backward: spmf_backward_pre = everything that does not depend on the data term (runs under it on
 * a side stream), spmf_backward_post = the data half + the loss parts.  pre + post == spmf_backward_params. */
int spmf_backward_pre(const float* params, const float* noise, const float* dgda, const float* eta, int D, int K,
                      int S, float batch_rows, float u_tau_scale, float s_tau_scale, float decay, float w_entropy,
                      float w_prior, int world_size, float* grads, float* scr_f, double* scr_d, void* stream) {
  return spmf_backward_pre_m(params, noise, dgda, eta, D, K, S, batch_rows, u_tau_scale, s_tau_scale, decay, w_entropy,
                             w_prior, world_size, grads, scr_f, scr_d, SPMF_MODEL_POISSON, stream);
}

int spmf_backward_pre_m(const float* params, const float* noise, const float* dgda, const float* eta, int D, int K,
                        int S, float batch_rows, float u_tau_scale, float s_tau_scale, float decay, float w_entropy,
                        float w_prior, int world_size, float* grads, float* scr_f, double* scr_d, int model,
                        void* stream) {
  if (!params || !noise || !dgda || !eta || !grads || !scr_f || !scr_d) return SPMF_ERR_BAD_ARG;
  if (D <= 0 || K <= 0 || S <= 0 || K > SPMF_MAX_K || world_size <= 0) return SPMF_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  Layout L = make_layout(D, K, S);
  Hyper h = make_hyper(u_tau_scale, s_tau_scale, decay, w_entropy, w_prior, world_size, batch_rows, model);
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S);
  float* scr_utau = scr_f;
  float* scr_parts = scr_utau + (long long)S * D * K;
  float* scr_lat = scr_parts + (long long)D * S * NUM_PARTS;
  float* scr_da = scr_lat + (long long)K * S * NUM_PARTS;
  float* fac = scr_da + (long long)S * D;
  float* utab = fac + 3LL * S * D * K;
  double* dutau = scr_d;
  double* featparts = dutau + (long long)S * K;
  double* latparts = featparts + (long long)S * NUM_PARTS;
  double* rscr = latparts + (long long)S * NUM_PARTS;
  dim3 grid((D + 3) / 4);
  launch_utau_table(L, params, noise, utab, st);
  if (KP <= 32) backward_dk_kernel<1, true><<<grid, 128, 0, st>>>(L, h, params, noise, dgda, eta, nullptr, SV, KP, nullptr, nullptr, nullptr, grads, scr_utau, scr_parts, scr_da, fac, utab, nullptr);
  else if (KP <= 64) backward_dk_kernel<2, true><<<grid, 128, 0, st>>>(L, h, params, noise, dgda, eta, nullptr, SV, KP, nullptr, nullptr, nullptr, grads, scr_utau, scr_parts, scr_da, fac, utab, nullptr);
  else if (KP <= 128) backward_dk_kernel<4, true><<<grid, 128, 0, st>>>(L, h, params, noise, dgda, eta, nullptr, SV, KP, nullptr, nullptr, nullptr, grads, scr_utau, scr_parts, scr_da, fac, utab, nullptr);
  else if (KP <= 512) backward_dk_wide_kernel<true><<<grid, 128, 0, st>>>(L, h, params, noise, dgda, eta, nullptr, SV, KP, nullptr, nullptr, nullptr, grads, scr_utau, scr_parts, scr_da, fac, utab, nullptr);
  else return SPMF_ERR_UNSUPPORTED;
  backward_feat_kernel<<<(int)(((long long)D * SV + 127) / 128), 128, 0, st>>>(L, h, params, noise, dgda, eta, nullptr, SV, nullptr, nullptr, grads, scr_parts, 1, nullptr);
  SPMF_CHECK_LAUNCH();
  int rc = reduce_rows_pair(scr_utau, dutau, D, K, S, scr_parts, featparts, D, S * NUM_PARTS, 1, rscr, st);
  if (rc) return rc;
  backward_lat_kernel<<<(K + 63) / 64, 64, 0, st>>>(L, h, params, noise, dgda, dutau, grads, scr_lat);
  SPMF_CHECK_LAUNCH();
  return reduce_rows<float>(scr_lat, latparts, rscr, K, S * NUM_PARTS, 1, st);
}

int spmf_backward_post(const float* params, const float* noise, const float* eta, const int* rank, int D, int K,
                       int S, const float* GAp, const float* GEVnz, const float* Gphinz, const double* zcolsum,
                       const double* datasums, const double* phisum, float batch_rows, float u_tau_scale,
                       float s_tau_scale, float decay, float w_entropy, float w_prior, int world_size,
                       float* grads, double* parts, float* scr_f, const double* scr_d, void* gs, void* stream) {
  return spmf_backward_post_m(params, noise, eta, rank, D, K, S, GAp, GEVnz, Gphinz, zcolsum, datasums, phisum,
                              batch_rows, u_tau_scale, s_tau_scale, decay, w_entropy, w_prior, world_size, grads,
                              parts, scr_f, scr_d, gs, SPMF_MODEL_POISSON, stream);
}

int spmf_backward_post_m(const float* params, const float* noise, const float* eta, const int* rank, int D, int K,
                         int S, const float* GAp, const float* GEVnz, const float* Gphinz, const double* zcolsum,
                         const double* datasums, const double* phisum, float batch_rows, float u_tau_scale,
                         float s_tau_scale, float decay, float w_entropy, float w_prior, int world_size,
                         float* grads, double* parts, float* scr_f, const double* scr_d, void* gs, int model,
                         void* stream) {
  if (!params || !noise || !eta || !GAp || !GEVnz || !Gphinz || !zcolsum || !datasums || !phisum || !grads ||
      !parts || !scr_f || !scr_d)
    return SPMF_ERR_BAD_ARG;
  if (D <= 0 || K <= 0 || S <= 0 || K > SPMF_MAX_K || world_size <= 0) return SPMF_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  Layout L = make_layout(D, K, S);
  Hyper h = make_hyper(u_tau_scale, s_tau_scale, decay, w_entropy, w_prior, world_size, batch_rows, model);
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S);
  float* scr_da = scr_f + (long long)S * D * K + (long long)D * S * NUM_PARTS + (long long)K * S * NUM_PARTS;
  const float* fac = scr_da + (long long)S * D;
  const double* featparts = scr_d + (long long)S * K;
  const double* latparts = featparts + (long long)S * NUM_PARTS;
  dim3 grid((D + 3) / 4);
  if (S > 64) return SPMF_ERR_BAD_ARG;
  if (KP <= 32) backward_dk_post_kernel<1><<<grid, 128, 0, st>>>(L, h, params, noise, eta, rank, SV, KP, GAp, GEVnz, Gphinz, zcolsum, fac, grads, (const int*)gs);
  else if (KP <= 64) backward_dk_post_kernel<2><<<grid, 128, 0, st>>>(L, h, params, noise, eta, rank, SV, KP, GAp, GEVnz, Gphinz, zcolsum, fac, grads, (const int*)gs);
  else if (KP <= 128) backward_dk_post_kernel<4><<<grid, 128, 0, st>>>(L, h, params, noise, eta, rank, SV, KP, GAp, GEVnz, Gphinz, zcolsum, fac, grads, (const int*)gs);
  else if (KP == 256) backward_dk_post_kernel<8><<<grid, 128, 0, st>>>(L, h, params, noise, eta, rank, SV, KP, GAp, GEVnz, Gphinz, zcolsum, fac, grads, (const int*)gs);
  else if (KP == 512) backward_dk_post_kernel<16><<<grid, 128, 0, st>>>(L, h, params, noise, eta, rank, SV, KP, GAp, GEVnz, Gphinz, zcolsum, fac, grads, (const int*)gs);
  else return SPMF_ERR_UNSUPPORTED;
  finalize_parts_kernel<<<1, ((S + 31) / 32) * 32, 0, st>>>(S, SV, K, featparts, latparts, datasums, phisum,
                                                           (double)batch_rows, (double)w_entropy, (double)w_prior,
                                                           parts, grads + L.comm_off, (GuardState*)gs);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}
long long spmf_backward_scratch_doubles(int D, int K, int S) {
  long long c = (long long)S * NUM_PARTS;
  if (c < K) c = K;
  return (long long)S * K + 2LL * S * NUM_PARTS + 64LL * S * (K + NUM_PARTS) + 64LL * S * c +
         64LL * (spmf_kpad(K) + 8) * S + 1024;
}

int spmf_adam_step(float* params, const float* grads, float* m, float* v, long long n, float lr,
                   float beta1, float beta2, float eps, int step, float clip_value, float grad_scale,
                   void* stream) {
  return spmf_adam_step_dev(params, grads, m, v, n, lr, beta1, beta2, eps, step, clip_value, grad_scale, nullptr, stream);
}

int spmf_step_state_bytes(void) { return (int)sizeof(StepState); }

/* host-side value of the per-step device scalars (what the first node of a step graph writes) */
static StepState make_step_state(unsigned rng_step, int adam_t, float lr, float b1, float b2, float eps, float clip) {
  StepState v;
  v.rng_step = rng_step; v.adam_t = adam_t; v.lr = lr; v.b1 = b1; v.b2 = b2; v.eps = eps; v.clip = clip;
  const int t = adam_t > 0 ? adam_t : 1;
  v.bc1 = 1.f - powf(b1, (float)t);
  v.bc2 = 1.f - powf(b2, (float)t);
  return v;
}

int spmf_step_state_set(void* step_state, unsigned int rng_step, int adam_t, float lr, float beta1, float beta2,
                        float eps, float clip_value, void* stream) {
  if (!step_state) return SPMF_ERR_BAD_ARG;
  step_state_kernel<<<1, 1, 0, (cudaStream_t)stream>>>((StepState*)step_state,
                                                       make_step_state(rng_step, adam_t, lr, beta1, beta2, eps, clip_value));
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

/* the kernel and the argument image of spmf_step_state_set, for graph node updates (spmf_step.cu) */
const void* spmf_step_state_kernel_ptr(void) { return (const void*)step_state_kernel; }
int spmf_step_state_value(unsigned int rng_step, int adam_t, float lr, float beta1, float beta2, float eps,
                          float clip_value, void* out36) {
  if (!out36) return SPMF_ERR_BAD_ARG;
  const StepState v = make_step_state(rng_step, adam_t, lr, beta1, beta2, eps, clip_value);
  memcpy(out36, &v, sizeof(v));
  return SPMF_OK;
}

int spmf_adam_step_dev(float* params, const float* grads, float* m, float* v, long long n, float lr,
                       float beta1, float beta2, float eps, int step, float clip_value, float grad_scale,
                       const void* step_state, void* stream) {
  if (!params || !grads || !m || !v || n <= 0 || (step <= 0 && !step_state)) return SPMF_ERR_BAD_ARG;
  const int t = step > 0 ? step : 1;
  float bc1 = 1.f - powf(beta1, (float)t), bc2 = 1.f - powf(beta2, (float)t);
  adam_kernel<<<(unsigned)((n + 255) / 256), 256, 0, (cudaStream_t)stream>>>(params, grads, m, v, n, lr, beta1, beta2, eps, bc1, bc2, clip_value, grad_scale, (const StepState*)step_state);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

/* Multi-GPU tail of a step in one launch: fold the all-reduced ('z','x') pairs back into parts / the mean
 * loss (spmf_unpack_parts) and apply Adam to grads[0, n) (the whole flat parameter buffer). */
int spmf_unpack_adam(float* comm_slack, int slack_floats, int S, float w_entropy, float w_prior, double* parts,
                     double* loss_out, const float* grads, long long n_data, const spmf_adam_args* adam,
                     void* stream) {
  if (!comm_slack || !parts || !loss_out || !grads || S <= 0 || S > 64 || slack_floats < 4 * S || n_data <= 0)
    return SPMF_ERR_BAD_ARG;
  const AdamCfg ad = make_adam(adam);
  const unsigned nblk = (unsigned)((n_data + 255) / 256);
  unpack_adam_kernel<<<nblk + 1, 256, 0, (cudaStream_t)stream>>>(S, (double)w_entropy, (double)w_prior, comm_slack,
                                                                slack_floats, parts, loss_out, grads, n_data, ad);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_unpack_parts(float* comm_slack, int slack_floats, int S, float w_entropy, float w_prior, double* parts,
                      double* loss_out, void* stream) {
  if (!comm_slack || !parts || !loss_out || S <= 0 || S > 64 || slack_floats < 4 * S) return SPMF_ERR_BAD_ARG;
  unpack_parts_kernel<<<1, 64, 0, (cudaStream_t)stream>>>(S, (double)w_entropy, (double)w_prior, comm_slack,
                                                          slack_floats, parts, loss_out);
  SPMF_CHECK_LAUNCH();
  return SPMF_OK;
}

int spmf_sumsq(const float* g, long long n, float* tmp, double* out, double* scratch, void* stream) {
  if (!g || !tmp || !out || !scratch || n <= 0) return SPMF_ERR_BAD_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  square_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(g, tmp, n);
  SPMF_CHECK_LAUNCH();
  // view tmp as [rows][32] (tail handled by treating n as rows of 1 channel when not divisible)
  long long rows = n / 32;
  int rc;
  if (rows * 32 == n) {
    rc = reduce_rows<float>(tmp, scratch + 64 * 32, scratch, rows, 32, 1, st);
    if (rc) return rc;
    return reduce_rows<double>(scratch + 64 * 32, out, scratch, 32, 1, 1, st);
  }
  return reduce_rows<float>(tmp, out, scratch, n, 1, 1, st);
}

int spmf_batch_sums(const float* z, const float* rowacc, int nrows, int K, int S, double* zcolsum,
                    double* datasums, double* scratch, void* stream) {
  if (!z || !rowacc || !zcolsum || !datasums || !scratch || nrows <= 0 || K <= 0 || K > SPMF_MAX_K || S <= 0)
    return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  return reduce_rows_pair(z, zcolsum, nrows, KP * SV, NQ, rowacc, datasums, nrows, 4 * SV, NQ, scratch,
                          (cudaStream_t)stream);
}

int spmf_colsum(const float* in, long long n, int c, int q, double* out, double* scratch, void* stream) {
  if (!in || !out || !scratch) return SPMF_ERR_BAD_ARG;
  return reduce_rows<float>(in, out, scratch, n, c, q, (cudaStream_t)stream);
}

int spmf_colsum_f64(const double* in, long long n, int c, int q, double* out, double* scratch, void* stream) {
  if (!in || !out || !scratch) return SPMF_ERR_BAD_ARG;
  return reduce_rows<double>(in, out, scratch, n, c, q, (cudaStream_t)stream);
}

}  // extern "C"
