// Per-element bodies of the surrogate draw / prior / entropy forward+backward.
//
// Everything here is __host__ __device__: the CUDA kernels in spmf_params.cu call these
// bodies one warp per feature d (lanes over latent k), and csrc/hostcheck.cpp runs the very
// same bodies in serial loops on the CPU so the math can be parity-checked without a GPU.
//
// Model restated (file:line relative to /root/reference):
//   surrogate q:  mederrata_spmf/poisson.py:403-539  (Softplus o Normal / Softplus o InverseGamma)
//   priors:       mederrata_spmf/poisson.py:225-377  (horseshoe+ hierarchy, horshoe_plus=True)
//   operands:     poisson.py:652-701 (encoding_matrix / intercept_matrix / decoding_matrix)
#pragma once
#include "spmf_math.cuh"

namespace spmf {

// ---- flat parameter buffer: data-touched tensors first (they are the all-reduced block) ----
enum TensorId {
  V_LOC = 0, V_RHO, W_LOC, W_RHO, U_LOC, U_RHO, S_LOC, S_RHO,
  UETA_C, UETA_B, UTAU_C, UTAU_B, SETA_C, SETA_B, STAU_C, STAU_B,
  UETAA_C, UETAA_B, UTAUA_C, UTAUA_B, SETAA_C, SETAA_B, STAUA_C, STAUA_B,
  NUM_TENSORS
};
enum VarId { VAR_V = 0, VAR_W, VAR_U, VAR_S, VAR_UETA, VAR_UTAU, VAR_SETA, VAR_STAU,
             VAR_UETAA, VAR_UTAUA, VAR_SETAA, VAR_STAUA, NUM_VARS };
// loss parts, reference var_list order (poisson.py:572) then log q, z, x
enum PartId { P_V = 0, P_W, P_U, P_UETA, P_UTAU, P_SETA, P_STAU, P_S, P_UETAA, P_UTAUA,
              P_SETAA, P_STAUA, P_LOGQ, P_Z, P_X, NUM_PARTS = 16 };

struct Layout {
  int D, K, S;
  long long toff[NUM_TENSORS + 1];  // float offsets into params / grads / adam moments
  long long noff[NUM_VARS + 1];     // float offsets into the noise buffer ([var][s][elem])
  long long vsize[NUM_VARS];
  long long comm_off;               // kCommSlack floats after the data-touched block (all-reduced scalars)
};
constexpr int kCommSlack = 1024;

inline long long pad32(long long n) { return (n + 31) / 32 * 32; }

inline Layout make_layout(int D, int K, int S) {
  Layout L;
  L.D = D; L.K = K; L.S = S;
  const long long DK = (long long)D * K;
  const long long vs[NUM_VARS] = {DK, D, DK, 2LL * D, DK, K, 2LL * D, D, DK, K, 2LL * D, D};
  long long o = 0, n = 0;
  for (int v = 0; v < NUM_VARS; ++v) {
    L.vsize[v] = vs[v];
    L.toff[2 * v] = o; o += pad32(vs[v]);
    L.toff[2 * v + 1] = o; o += pad32(vs[v]);
    if (v == VAR_S) { L.comm_off = o; o += kCommSlack; }
    L.noff[v] = n; n += pad32((long long)S * vs[v]);
  }
  L.toff[NUM_TENSORS] = o;
  L.noff[NUM_VARS] = n;
  return L;
}

struct Hyper {
  int vw_identity;   // BernoulliFactorization: v, w use an Identity bijector and Normal priors (bernoulli.py:186-215)
  float u_tau_b;     // 1/u_tau_scale^2   (poisson.py:339)
  float s_tau_b;     // 1/s_tau_scale^2   (poisson.py:375)
  float decay;       // symmetry_breaking_decay (poisson.py:225)
  float w_entropy;   // weight of log q        (1 = reference)
  float w_prior;     // weight of prior terms  (1 = reference, poisson.py:577)
  float rep_scale;   // 1/world_size: prior+entropy share carried by each rank for the all-reduced tensors
  float batch_rows;  // rows in this rank's minibatch (closed-form -B term of dphi)
};

// ---------------- per-step scalars on the device ----------------
// What changes from one step to the next (Philox step, optimiser step and rates) lives in device memory
// when the step is replayed as a CUDA graph: kernel arguments of a graph are frozen at capture, so the
// kernels read these from `StepState` instead (written by the first node of the graph, whose argument is
// the only thing updated per launch).  NULL state pointer = use the launch arguments.
struct StepState {
  unsigned rng_step;
  int adam_t;
  float lr, b1, b2, eps, bc1, bc2, clip;
};

// ---------------- Adam [EXT L4: tf.optimizers.Adam in bayesianquilts' loop] ----------------
// m, v = first / second moments; bc1, bc2 = 1 - beta^t; a non-finite gradient is dropped, `clip` > 0 clips
// the gradient by value.  lr <= 0: off.  (Fusing this into the backward kernels was tried in round 2
// and measured slower: they are latency-bound, and the extra dependent loads of m, v, p cost more than
// the separate streaming pass -- 80 us against 33 us at C4.)
struct AdamCfg {
  float lr, b1, b2, eps, bc1, bc2, clip, grad_scale;
  float* p;     // parameters (same flat layout as the gradients)
  float* m;
  float* v;
};
SPMF_HD void adam_apply(const AdamCfg& a, long long i, float g) {
  g *= a.grad_scale;
  if (!(fabsf(g) <= 3.402823466e38f)) g = 0.f;
  if (a.clip > 0.f) g = fminf(fmaxf(g, -a.clip), a.clip);
  const float mi = a.b1 * a.m[i] + (1.f - a.b1) * g;
  const float vi = a.b2 * a.v[i] + (1.f - a.b2) * g * g;
  a.m[i] = mi;
  a.v[i] = vi;
  a.p[i] -= a.lr * (mi / a.bc1) / (sqrtf(vi / a.bc2) + a.eps);
}

#ifdef SPMF_B200_H
// host: C-ABI optimiser arguments -> kernel configuration (lr = 0: off)
inline AdamCfg make_adam_cfg(const spmf_adam_args* a) {
  AdamCfg c{};
  if (!a || !(a->lr > 0.f) || !a->params || !a->m || !a->v || a->step <= 0) return c;
  c.lr = a->lr; c.b1 = a->beta1; c.b2 = a->beta2; c.eps = a->eps;
  c.bc1 = 1.f - powf(a->beta1, (float)a->step);
  c.bc2 = 1.f - powf(a->beta2, (float)a->step);
  c.clip = a->clip_value;
  c.grad_scale = a->grad_scale > 0.f ? a->grad_scale : 1.f;
  c.p = a->params; c.m = a->m; c.v = a->v;
  return c;
}
#endif

// ---------------- Normal-based factor:  y = softplus(loc + softplus(rho) * eps) ----------------
struct NParam { float loc, sig, logsig, acc_dt, acc_dte; };
struct NDraw { float t, y, sg, oms, lsg; };   // pre-softplus t, softplus, sigmoid, 1-sigmoid, log sigmoid

SPMF_HD NParam nparam_init(float loc, float rho) {
  float sig = softplusf(rho);
  return NParam{loc, sig, logf(sig), 0.f, 0.f};
}
SPMF_HD NDraw ndraw(const NParam& p, float eps) {
  NDraw d;
  d.t = fmaf(p.sig, eps, p.loc);
  const Sp4 f = softplus4(d.t);
  d.y = f.y; d.sg = f.sg; d.oms = f.oms; d.lsg = f.lsg;
  return d;
}
// Identity bijector (v, w of BernoulliFactorization, bernoulli.py:186-195): y = t, no Jacobian term
SPMF_HD NDraw ndraw_id(const NParam& p, float eps) {
  NDraw d;
  d.t = fmaf(p.sig, eps, p.loc);
  d.y = d.t; d.sg = 1.f; d.oms = 0.f; d.lsg = 0.f;
  return d;
}
SPMF_HD NDraw ndraw_sel(const NParam& p, float eps, int identity) { return identity ? ndraw_id(p, eps) : ndraw(p, eps); }
// log q(y) = log N(t; loc, sig) - log sigmoid(t)     [EXT tfb.Softplus fldj]
SPMF_HD float nlogq(const NParam& p, const NDraw& d, float eps) {
  return -0.5f * eps * eps - p.logsig - kHalfLog2Pi - d.lsg;
}
// Gy = d loss_s / d y (data+prior part, already weighted); we = entropy weight
SPMF_HD void nparam_bwd(NParam& p, const NDraw& d, float eps, float Gy, float we) {
  float dt = Gy * d.sg - we * d.oms;
  p.acc_dt += dt;
  p.acc_dte += dt * eps;
}
SPMF_HD void nparam_finish(const NParam& p, float rho, float invS, float we, float* g_loc, float* g_rho) {
  float sr = sigmoidf(rho);
  *g_loc = p.acc_dt * invS;
  *g_rho = p.acc_dte * invS * sr - we * sr / p.sig;
}

// ------------- InverseGamma-based factor:  y = softplus(beta / g),  g ~ Gamma(alpha,1) -------------
struct GParam { float alpha, beta, psi, c0, acc_da, acc_db; };   // c0 = -log(beta) - lgamma(alpha)
struct GDraw { float t, y, sg, oms, lsg, g; };

SPMF_HD GParam gparam_init(float conc_raw, float scale_raw) {
  GParam p;
  p.alpha = softplusf(conc_raw);
  p.beta = softplusf(scale_raw);
  p.psi = digammaf_pos(p.alpha);
  p.c0 = -logf(p.beta) - lgammaf(p.alpha);
  p.acc_da = 0.f;
  p.acc_db = 0.f;
  return p;
}
SPMF_HD GDraw gdraw(const GParam& p, float g) {
  GDraw d;
  d.g = g;
  d.t = p.beta * SPMF_RCPF(g);
  const Sp4 f = softplus4(d.t);
  d.y = f.y; d.sg = f.sg; d.oms = f.oms; d.lsg = f.lsg;
  return d;
}
// log q(y) = log InvGamma(t; alpha, beta) - log sigmoid(t), with beta/t = g, log t = log beta - log g
SPMF_HD float glogq(const GParam& p, const GDraw& d) {
  return p.c0 + (p.alpha + 1.f) * SPMF_LOGF(d.g) - d.g - d.lsg;
}
// dgda = d g / d alpha of the Gamma draw (implicit reparameterisation), precomputed per draw by
// gamma_grad_kernel since it depends on (alpha, g) only.
SPMF_HD void gparam_bwd(GParam& p, const GDraw& d, float dgda, float Gy, float we) {
  float g = d.g;
  const float ig = SPMF_RCPF(g), ib = SPMF_RCPF(p.beta);
  float dlogq_dt = (g * ib) * (g - (p.alpha + 1.f)) - d.oms;
  float dt = Gy * d.sg + we * dlogq_dt;
  p.acc_da += we * (SPMF_LOGF(g) - p.psi) - dt * (p.beta * ig * ig) * dgda;
  p.acc_db += we * (p.alpha - g) * ib + dt * ig;
}
SPMF_HD void gparam_finish(const GParam& p, float conc_raw, float scale_raw, float invS,
                           float* g_conc, float* g_scale) {
  *g_conc = p.acc_da * invS * sigmoidf(conc_raw);
  *g_scale = p.acc_db * invS * sigmoidf(scale_raw);
}

// ---------------- prior log-densities with derivatives [EXT TFP definitions] ----------------
// HalfNormal(y; sigma): value, d/dy, d/dsigma
SPMF_HD float halfnormal(float y, float sigma, float* dy, float* dsigma) {
  float is = SPMF_RCPF(sigma), r = y * is;
  *dy = -r * is;
  *dsigma = (r * r - 1.f) * is;
  return kHalfLog2OverPi - SPMF_LOGF(sigma) - 0.5f * r * r;
}
// Normal(y; 0, sigma): value, d/dy   (priors of v, w in bernoulli.py:200-215)
SPMF_HD float normal0(float y, float sigma, float* dy) {
  float is = SPMF_RCPF(sigma), r = y * is;
  *dy = -r * is;
  return -kHalfLog2Pi - SPMF_LOGF(sigma) - 0.5f * r * r;
}
// SqrtInverseGamma(y; 0.5, scale = 1/a): value, d/dy, d/da
SPMF_HD float sqrt_ig_half(float y, float a, float* dy, float* da) {
  float iy = SPMF_RCPF(y), ia = SPMF_RCPF(a), iy2 = iy * iy;
  *dy = -2.f * iy + 2.f * ia * iy2 * iy;
  *da = -0.5f * ia + ia * ia * iy2;
  return -0.5f * SPMF_LOGF(a) - kLgammaHalf - 2.f * SPMF_LOGF(y) - ia * iy2 + kLog2;
}
// InverseGamma(a; 0.5, b): value, d/da
SPMF_HD float ig_half(float a, float b, float* da) {
  float ia = SPMF_RCPF(a);
  *da = -1.5f * ia + b * ia * ia;
  return 0.5f * SPMF_LOGF(b) - kLgammaHalf - 1.5f * SPMF_LOGF(a) - b * ia;
}

// ---------------------------------------------------------------------------------------
// Row program for one feature d.  `LaneState` holds what one lane (k = lane, lane+32, ...)
// keeps across the draw loop; `FeatState` what lane 0 keeps for the per-feature variables.
// ---------------------------------------------------------------------------------------
template <int KK>
struct LaneState {
  NParam u[KK], v[KK];
  GParam ue[KK], ua[KK];
  float utb[KK];   // softplus(scale_raw) of u_tau[k]: read by the host form of lane_step only
  float ck[KK];    // symmetry_breaking_decay^k (poisson.py:225-226)
};
struct FeatState {
  NParam w, s0, s1;
  GParam se0, se1, st, sea0, sea1, sta;
};

// `eta` everywhere below is [2][D]: row 0 = the decoder scale eta_i (EV = eta v, phi = eta b w), row 1 =
// the encoder divisor (A' = a u / eta_enc): eta_i for the linear encoder x/eta, 1 under log_transform
// (the encoder log(x/eta + 1) is then applied to the counts themselves; poisson.py:34-54).
struct ModelPtrs {
  const float* params;   // flat
  const float* noise;    // flat
  const float* eta;      // [2][D]
};


template <int KK>
SPMF_HD void lane_init(LaneState<KK>& st, const Layout& L, const float* P, int d, int lane,
                       float decay = 1.f) {
  for (int i = 0; i < KK; ++i) {
    int k = lane + 32 * i;
    st.ck[i] = powf(decay, (float)k);
    if (k < L.K) {
      long long e = (long long)d * L.K + k;
      st.u[i] = nparam_init(P[L.toff[U_LOC] + e], P[L.toff[U_RHO] + e]);
      st.v[i] = nparam_init(P[L.toff[V_LOC] + e], P[L.toff[V_RHO] + e]);
      st.ue[i] = gparam_init(P[L.toff[UETA_C] + e], P[L.toff[UETA_B] + e]);
      st.ua[i] = gparam_init(P[L.toff[UETAA_C] + e], P[L.toff[UETAA_B] + e]);
      st.utb[i] = softplusf(P[L.toff[UTAU_B] + k]);
    }
  }
}

SPMF_HD void feat_init(FeatState& f, const Layout& L, const float* P, int d) {
  const int D = L.D;
  f.w = nparam_init(P[L.toff[W_LOC] + d], P[L.toff[W_RHO] + d]);
  f.s0 = nparam_init(P[L.toff[S_LOC] + d], P[L.toff[S_RHO] + d]);
  f.s1 = nparam_init(P[L.toff[S_LOC] + D + d], P[L.toff[S_RHO] + D + d]);
  f.se0 = gparam_init(P[L.toff[SETA_C] + d], P[L.toff[SETA_B] + d]);
  f.se1 = gparam_init(P[L.toff[SETA_C] + D + d], P[L.toff[SETA_B] + D + d]);
  f.st = gparam_init(P[L.toff[STAU_C] + d], P[L.toff[STAU_B] + d]);
  f.sea0 = gparam_init(P[L.toff[SETAA_C] + d], P[L.toff[SETAA_B] + d]);
  f.sea1 = gparam_init(P[L.toff[SETAA_C] + D + d], P[L.toff[SETAA_B] + D + d]);
  f.sta = gparam_init(P[L.toff[STAUA_C] + d], P[L.toff[STAUA_B] + d]);
}

// Draws of the per-feature variables needed by every lane (a_d, b_d and the draws themselves).
struct FeatDraw { NDraw w, s0, s1; float a, b; };
SPMF_HD FeatDraw feat_draw(const FeatState& f, const Layout& L, const float* N, int d, int s, int vw_identity = 0) {
  FeatDraw r;
  const long long D = L.D;
  r.w = ndraw_sel(f.w, N[L.noff[VAR_W] + s * D + d], vw_identity);
  r.s0 = ndraw(f.s0, N[L.noff[VAR_S] + s * 2 * D + d]);
  r.s1 = ndraw(f.s1, N[L.noff[VAR_S] + s * 2 * D + D + d]);
  float inv = 1.f / (r.s0.y + r.s1.y);
  r.a = r.s0.y * inv;   // poisson.py:661-663
  r.b = r.s1.y * inv;   // poisson.py:694-697
  return r;
}

// ---- forward operands for one (d,k,s):  A' = a_d u / eta_d,  EV = eta_d v  (poisson.py:665,174-175,43) ----
template <int KK>
SPMF_HD void lane_operands(const LaneState<KK>& st, const Layout& L, const float* N, const float* eta,
                           int d, int lane, int i, int s, float a_d, float* Ap, float* EV,
                           float* u_out, float* v_out, int vw_identity = 0) {
  int k = lane + 32 * i;
  long long e = (long long)s * L.D * L.K + (long long)d * L.K + k;
  NDraw u = ndraw(st.u[i], N[L.noff[VAR_U] + e]);
  NDraw v = ndraw_sel(st.v[i], N[L.noff[VAR_V] + e], vw_identity);
  *Ap = a_d * u.y / eta[L.D + d];      // encoder divisor: eta_d, or 1 under log_transform (poisson.py:41-43)
  *EV = eta[d] * v.y;
  if (u_out) *u_out = u.y;
  if (v_out) *v_out = v.y;
}

// u_tau[k] enters the (d,k) programs through its draw y = softplus(beta_k / g_sk) only, a function of
// (s,k): the kernels evaluate it once per step into an [S][K] table (utau_table_kernel) instead of once
// per (d,k,s).  beta = softplus(scale_raw[k]).
SPMF_HD float utau_y(float beta, float g) { return softplus4(beta * SPMF_RCPF(g)).y; }

// Upstream gradients of the data term for one (d,k,s)
struct DkUp { float GAp, GEV; };   // dL/dA'_dk (sum over rows), dL/dEV_dk (closed form already applied)
// parts: U, V, UETA, UETAA, LOGQ; uy, usg, vsg: the u draw, sigmoid'(u) and sigmoid'(v) of this (d,k,s),
// which the split backward stores for its data half
struct DkOut { float da; float dutau; float parts[5]; float uy, usg, vsg; };

// One (d,k,s) of the (d,k) program.  eta_dec = eta[d], ieta = 1 / eta[D + d] (the encoder divisor) and
// ut_y = utau_y of (s,k) are per-feature / per-draw values the caller holds.
template <int KK>
SPMF_HD DkOut lane_step(LaneState<KK>& st, const Layout& L, const Hyper& h, const float* N,
                        const float* G, float eta_dec, float ieta, int d, int lane, int i, int s, float a_d,
                        float ut_y, DkUp up) {
  DkOut o;
  int k = lane + 32 * i;
  const long long DK = (long long)L.D * L.K;
  long long e = (long long)s * DK + (long long)d * L.K + k;
  float eps_u = N[L.noff[VAR_U] + e], eps_v = N[L.noff[VAR_V] + e];
  NDraw u = ndraw(st.u[i], eps_u);
  NDraw v = ndraw_sel(st.v[i], eps_v, h.vw_identity);
  GDraw ue = gdraw(st.ue[i], N[L.noff[VAR_UETA] + e]);
  GDraw ua = gdraw(st.ua[i], N[L.noff[VAR_UETAA] + e]);
  const float ck = st.ck[i];
  float sigma = ue.y * ut_y * ck;
  float du, dsig, dv, dtmp, due, dua, dua2;
  float pu = halfnormal(u.y, sigma, &du, &dsig);                 // poisson.py:247-251
  float pv = h.vw_identity ? normal0(v.y, 0.1f, &dv)             // bernoulli.py:200-208
                           : halfnormal(v.y, 0.1f, &dv, &dtmp);  // poisson.py:229-235
  float pue = sqrt_ig_half(ue.y, ua.y, &due, &dua);              // poisson.py:303-311
  float pua = ig_half(ua.y, 1.0f, &dua2);                        // poisson.py:312-322
  const float wpr = h.w_prior * h.rep_scale, wer = h.w_entropy * h.rep_scale;
  float Gy_u = -(wpr * du + up.GAp * a_d * ieta);
  float Gy_v = -(wpr * dv + eta_dec * up.GEV);
  float Gy_ue = -h.w_prior * (dsig * ut_y * ck + due);
  float Gy_ua = -h.w_prior * (dua + dua2);
  nparam_bwd(st.u[i], u, eps_u, Gy_u, wer);
  nparam_bwd(st.v[i], v, eps_v, Gy_v, wer);
  gparam_bwd(st.ue[i], ue, G[L.noff[VAR_UETA] + e], Gy_ue, h.w_entropy);
  gparam_bwd(st.ua[i], ua, G[L.noff[VAR_UETAA] + e], Gy_ua, h.w_entropy);
  o.da = up.GAp * u.y * ieta;                    // d L / d a_d contribution
  o.dutau = dsig * ue.y * ck;                    // d prior_u / d u_tau[k] contribution
  o.parts[0] = pu; o.parts[1] = pv; o.parts[2] = pue; o.parts[3] = pua;
  o.parts[4] = nlogq(st.u[i], u, eps_u) + nlogq(st.v[i], v, eps_v) + glogq(st.ue[i], ue) +
               glogq(st.ua[i], ua);
  o.uy = u.y; o.usg = u.sg; o.vsg = v.sg;
  return o;
}

// Host form (tests/hostcheck): draws u_tau from the lane state and reads eta itself.
template <int KK>
SPMF_HD DkOut lane_step(LaneState<KK>& st, const Layout& L, const Hyper& h, const float* N,
                        const float* G, const float* eta, int d, int lane, int i, int s, float a_d,
                        DkUp up) {
  const int k = lane + 32 * i;
  const float ut_y = utau_y(st.utb[i], N[L.noff[VAR_UTAU] + (long long)s * L.K + k]);
  return lane_step<KK>(st, L, h, N, G, eta[d], 1.f / eta[L.D + d], d, lane, i, s, a_d, ut_y, up);
}

// per-feature step (lane 0): w, s, s_eta, s_tau, s_eta_a, s_tau_a.  da = sum_k GAp u / eta (reduced),
// Gphi = sum over nonzeros of x/lambda (closed-form -B applied here).
// parts out: W, S, SETA, STAU, SETAA, STAUA, LOGQ
SPMF_HD void feat_step(FeatState& f, const FeatDraw& fd, const Layout& L, const Hyper& h,
                       const float* N, const float* G, const float* eta, int d, int s, float da,
                       float Gphi_nz, float parts[7]) {
  const long long D = L.D;
  float eps_w = N[L.noff[VAR_W] + s * D + d];
  float eps_s0 = N[L.noff[VAR_S] + s * 2 * D + d];
  float eps_s1 = N[L.noff[VAR_S] + s * 2 * D + D + d];
  GDraw se0 = gdraw(f.se0, N[L.noff[VAR_SETA] + s * 2 * D + d]);
  GDraw se1 = gdraw(f.se1, N[L.noff[VAR_SETA] + s * 2 * D + D + d]);
  GDraw st = gdraw(f.st, N[L.noff[VAR_STAU] + s * D + d]);
  GDraw sea0 = gdraw(f.sea0, N[L.noff[VAR_SETAA] + s * 2 * D + d]);
  GDraw sea1 = gdraw(f.sea1, N[L.noff[VAR_SETAA] + s * 2 * D + D + d]);
  GDraw sta = gdraw(f.sta, N[L.noff[VAR_STAUA] + s * D + d]);
  const float wpr = h.w_prior * h.rep_scale, wer = h.w_entropy * h.rep_scale;

  float Gphi = Gphi_nz - h.batch_rows;                        // d L / d phi_d
  float dw_data = eta[d] * fd.b * Gphi;                       // phi = eta b w   (poisson.py:701)
  float db = eta[d] * fd.w.y * Gphi;
  float inv = 1.f / (fd.s0.y + fd.s1.y), inv2 = inv * inv;
  float ds0_data = (da - db) * fd.s1.y * inv2;
  float ds1_data = (db - da) * fd.s0.y * inv2;

  float dw, dtmp, d_s0, dsig0, d_s1, dsig1;
  float pw = h.vw_identity ? normal0(fd.w.y, 1.0f, &dw)        // bernoulli.py:209-215
                           : halfnormal(fd.w.y, 1.0f, &dw, &dtmp);   // poisson.py:236-242
  float ps0 = halfnormal(fd.s0.y, se0.y * st.y, &d_s0, &dsig0);  // poisson.py:273-277
  float ps1 = halfnormal(fd.s1.y, se1.y * st.y, &d_s1, &dsig1);
  float dse0, dsea0, dse1, dsea1, dst, dsta, dsea0b, dsea1b, dstab;
  float pse0 = sqrt_ig_half(se0.y, sea0.y, &dse0, &dsea0);     // poisson.py:343-351
  float pse1 = sqrt_ig_half(se1.y, sea1.y, &dse1, &dsea1);
  float pst = sqrt_ig_half(st.y, sta.y, &dst, &dsta);          // poisson.py:360-367
  float psea0 = ig_half(sea0.y, 1.0f, &dsea0b);                // poisson.py:352-359
  float psea1 = ig_half(sea1.y, 1.0f, &dsea1b);
  float psta = ig_half(sta.y, h.s_tau_b, &dstab);              // poisson.py:368-377

  nparam_bwd(f.w, fd.w, eps_w, -(wpr * dw + dw_data), wer);
  nparam_bwd(f.s0, fd.s0, eps_s0, -(wpr * d_s0 + ds0_data), wer);
  nparam_bwd(f.s1, fd.s1, eps_s1, -(wpr * d_s1 + ds1_data), wer);
  gparam_bwd(f.se0, se0, G[L.noff[VAR_SETA] + s * 2 * D + d], -h.w_prior * (dsig0 * st.y + dse0), h.w_entropy);
  gparam_bwd(f.se1, se1, G[L.noff[VAR_SETA] + s * 2 * D + D + d], -h.w_prior * (dsig1 * st.y + dse1), h.w_entropy);
  gparam_bwd(f.st, st, G[L.noff[VAR_STAU] + s * D + d], -h.w_prior * (dsig0 * se0.y + dsig1 * se1.y + dst), h.w_entropy);
  gparam_bwd(f.sea0, sea0, G[L.noff[VAR_SETAA] + s * 2 * D + d], -h.w_prior * (dsea0 + dsea0b), h.w_entropy);
  gparam_bwd(f.sea1, sea1, G[L.noff[VAR_SETAA] + s * 2 * D + D + d], -h.w_prior * (dsea1 + dsea1b), h.w_entropy);
  gparam_bwd(f.sta, sta, G[L.noff[VAR_STAUA] + s * D + d], -h.w_prior * (dsta + dstab), h.w_entropy);

  parts[0] = pw;
  parts[1] = ps0 + ps1;
  parts[2] = pse0 + pse1;
  parts[3] = pst;
  parts[4] = psea0 + psea1;
  parts[5] = psta;
  parts[6] = nlogq(f.w, fd.w, eps_w) + nlogq(f.s0, fd.s0, eps_s0) + nlogq(f.s1, fd.s1, eps_s1) +
             glogq(f.se0, se0) + glogq(f.se1, se1) + glogq(f.st, st) + glogq(f.sea0, sea0) +
             glogq(f.sea1, sea1) + glogq(f.sta, sta);
}

// per-latent step (one thread per k): u_tau, u_tau_a.  dutau = sum_d d prior_u / d u_tau[k].
// parts out: UTAU, UTAUA, LOGQ
struct LatState { GParam ut, uta; };
SPMF_HD void lat_init(LatState& t, const Layout& L, const float* P, int k) {
  t.ut = gparam_init(P[L.toff[UTAU_C] + k], P[L.toff[UTAU_B] + k]);
  t.uta = gparam_init(P[L.toff[UTAUA_C] + k], P[L.toff[UTAUA_B] + k]);
}
SPMF_HD void lat_step(LatState& t, const Layout& L, const Hyper& h, const float* N, const float* G,
                      int k, int s, float dutau, float parts[3]) {
  GDraw ut = gdraw(t.ut, N[L.noff[VAR_UTAU] + (long long)s * L.K + k]);
  GDraw uta = gdraw(t.uta, N[L.noff[VAR_UTAUA] + (long long)s * L.K + k]);
  float dut, duta, duta2;
  float put = sqrt_ig_half(ut.y, uta.y, &dut, &duta);           // poisson.py:323-331
  float puta = ig_half(uta.y, h.u_tau_b, &duta2);               // poisson.py:332-341
  gparam_bwd(t.ut, ut, G[L.noff[VAR_UTAU] + (long long)s * L.K + k], -h.w_prior * (dutau + dut), h.w_entropy);
  gparam_bwd(t.uta, uta, G[L.noff[VAR_UTAUA] + (long long)s * L.K + k], -h.w_prior * (duta + duta2), h.w_entropy);
  parts[0] = put;
  parts[1] = puta;
  parts[2] = glogq(t.ut, ut) + glogq(t.uta, uta);
}

}  // namespace spmf
