// Scalar fp32 math shared by the sampling / prior kernels.  Every function is
// __host__ __device__ so tests can run the exact same code on the CPU
// (csrc/hostcheck.cpp) without a GPU.
//
// Restates TFP / bayesianquilts semantics needed by the ADVI step of
// mederrata_spmf/poisson.py (surrogate at :403-539, priors at :225-377); see
// SURVEY.md section 3.4.
#pragma once
#include <math.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define SPMF_HD __host__ __device__ __forceinline__
#else
#define SPMF_HD inline
#endif
// Per-draw elementwise math: single-MUFU forms on the device (relative error ~1e-6, two orders
// below the 1e-4 parity tolerance), libm on the host so the CPU host check stays the accurate
// reference for the same formulas.  log1p is kept accurate everywhere (softplus of very negative
// arguments is the scale of every u, v, w).
#if defined(__CUDA_ARCH__)
#define SPMF_RCP(x) __frcp_rn(x)
#define SPMF_LOGF(x) __logf(x)
#define SPMF_EXPF(x) __expf(x)
#define SPMF_RCPF(x) __fdividef(1.f, (x))
#define SPMF_COSF(x) __cosf(x)
#else
#define SPMF_RCP(x) (1.f / (x))
#define SPMF_LOGF(x) logf(x)
#define SPMF_EXPF(x) expf(x)
#define SPMF_RCPF(x) (1.f / (x))
#define SPMF_COSF(x) cosf(x)
#endif

namespace spmf {

constexpr float kHalfLog2OverPi = -0.22579135264472743f;  // 0.5*log(2/pi)
constexpr float kHalfLog2Pi = 0.9189385332046727f;        // 0.5*log(2*pi)
constexpr float kLgammaHalf = 0.5723649429247001f;        // lgamma(0.5)
constexpr float kLog2 = 0.6931471805599453f;

SPMF_HD float softplusf(float x) { return fmaxf(x, 0.f) + log1pf(expf(-fabsf(x))); }
SPMF_HD float sigmoidf(float x) {
  float e = expf(-fabsf(x));
  float s = 1.f / (1.f + e);
  return x >= 0.f ? s : e * s;
}
// 1 - sigmoid(x) without cancellation
SPMF_HD float one_minus_sigmoidf(float x) { return sigmoidf(-x); }
SPMF_HD float log_sigmoidf(float x) { return -softplusf(-x); }

// log1p(e) for e in [0, 1] (e = exp(-|t|) of a softplus): relative error < 1e-6.  Small e: 8-term series
// (truncation (e^9/9)/log1p(e) < 1e-8 at e = 1/8); otherwise the single-MUFU log of 1 + e, whose absolute
// error (~1e-7) is small against log1p(e) >= 0.117.  ~14 instructions against ~30 of libdevice's log1pf.
SPMF_HD float log1p_unit(float e) {
#if defined(__CUDA_ARCH__)
  const float p = e * (1.f + e * (-0.5f + e * (0.33333334f + e * (-0.25f + e * (0.2f + e * (-0.16666667f +
                  e * (0.14285715f + e * -0.125f)))))));
  return e < 0.125f ? p : __logf(1.f + e);
#else
  return log1pf(e);
#endif
}

// softplus(t), sigmoid(t), 1 - sigmoid(t) and log sigmoid(t) from ONE exp, one log1p, one reciprocal
struct Sp4 { float y, sg, oms, lsg; };
SPMF_HD Sp4 softplus4(float t) {
  const float e = SPMF_EXPF(-fabsf(t));
  const float l = log1p_unit(e);
  const float r = SPMF_RCPF(1.f + e);
  Sp4 o;
  o.y = fmaxf(t, 0.f) + l;
  o.sg = t >= 0.f ? r : e * r;
  o.oms = t >= 0.f ? e * r : r;
  o.lsg = fminf(t, 0.f) - l;
  return o;
}

SPMF_HD float digammaf_pos(float x) {
  // x > 0.  Shift to x >= 6 with psi(x) = psi(x+1) - 1/x, then the asymptotic series.
  float acc = 0.f;
  while (x < 6.f) {
    acc -= 1.f / x;
    x += 1.f;
  }
  float r = 1.f / x, r2 = r * r;
  return acc + logf(x) - 0.5f * r -
         r2 * (1.f / 12.f - r2 * (1.f / 120.f - r2 * (1.f / 252.f)));
}

// dg/dalpha of a standard Gamma(alpha) draw g at fixed quantile (implicit
// reparameterisation, Figurnov et al. 2018 -- what tf.random.gamma's gradient returns).
//   g <= max(1, alpha+1): power series  (g/a) [sum T_n H_n - (log g - psi(a+1)) sum T_n]
//   otherwise: Cephes igamc continued fraction differentiated in alpha.
SPMF_HD float gamma_sample_der_alpha(float a, float x) {
  if (!(x > 0.f)) return 0.f;
  if (x <= 1.f || x <= a + 1.f) {
    float T = 1.f, H = 0.f, sT = 1.f, sTH = 0.f;
    for (int n = 1; n < 400; ++n) {
      float inv = SPMF_RCP(a + (float)n);
      T *= x * inv;
      H += inv;
      sT += T;
      sTH += T * H;
      if (T * (1.f + H) < 1e-7f * sT) break;
    }
    return (x / a) * (sTH - (logf(x) - digammaf_pos(a + 1.f)) * sT);
  }
  float y = 1.f - a, z = x + y + 1.f;
  float pkm2 = 1.f, qkm2 = x, pkm1 = x + 1.f, qkm1 = z * x;
  float dpkm2 = 0.f, dqkm2 = 0.f, dpkm1 = 0.f, dqkm1 = -x;
  float ans = pkm1 / qkm1;
  float dans = (dpkm1 - ans * dqkm1) / qkm1;
  for (int c = 1; c < 400; ++c) {
    y += 1.f;
    z += 2.f;
    float fc = (float)c;
    float yc = y * fc, dyc = -fc;
    float pk = pkm1 * z - pkm2 * yc;
    float qk = qkm1 * z - qkm2 * yc;
    float dpk = dpkm1 * z - pkm1 - dpkm2 * yc - pkm2 * dyc;
    float dqk = dqkm1 * z - qkm1 - dqkm2 * yc - qkm2 * dyc;
    float nans = pk / qk;
    float ndans = (dpk - nans * dqk) / qk;
    float delta = fabsf(ndans - dans);
    float scale = fabsf(ndans) + 1e-30f;
    ans = nans;
    dans = ndans;
    pkm2 = pkm1; pkm1 = pk; qkm2 = qkm1; qkm1 = qk;
    dpkm2 = dpkm1; dpkm1 = dpk; dqkm2 = dqkm1; dqkm1 = dqk;
    if (fabsf(pk) > 1e18f || fabsf(qk) > 1e18f) {
      const float sc = 1e-18f;
      pkm2 *= sc; pkm1 *= sc; qkm2 *= sc; qkm1 *= sc;
      dpkm2 *= sc; dpkm1 *= sc; dqkm2 *= sc; dqkm1 *= sc;
    }
    if (delta < 1e-6f * scale && c > 3) break;
  }
  return x * (dans + ans * (logf(x) - digammaf_pos(a)));
}

// Same gradient for up to 4 draws of ONE variable (shared alpha): the series terms 1/(a+n) and
// H_n, digamma and the loop control are shared, which is how the per-step kernel evaluates it.
// psi = digamma(a).  Results match gamma_sample_der_alpha() to rounding.
SPMF_HD float gamma_der_cf(float a, float psi, float x) {
  float y = 1.f - a, z = x + y + 1.f;
  float pkm2 = 1.f, qkm2 = x, pkm1 = x + 1.f, qkm1 = z * x;
  float dpkm2 = 0.f, dqkm2 = 0.f, dpkm1 = 0.f, dqkm1 = -x;
  float ans = pkm1 / qkm1;
  float dans = (dpkm1 - ans * dqkm1) / qkm1;
  for (int c = 1; c < 400; ++c) {
    y += 1.f;
    z += 2.f;
    const float fc = (float)c;
    const float yc = y * fc;
    const float pk = pkm1 * z - pkm2 * yc;
    const float qk = qkm1 * z - qkm2 * yc;
    const float dpk = dpkm1 * z - pkm1 - dpkm2 * yc + pkm2 * fc;
    const float dqk = dqkm1 * z - qkm1 - dqkm2 * yc + qkm2 * fc;
    const float iq = SPMF_RCPF(qk);
    const float nans = pk * iq;
    const float ndans = (dpk - nans * dqk) * iq;
    const float delta = fabsf(ndans - dans);
    const float scale = fabsf(ndans) + 1e-30f;
    ans = nans;
    dans = ndans;
    pkm2 = pkm1; pkm1 = pk; qkm2 = qkm1; qkm1 = qk;
    dpkm2 = dpkm1; dpkm1 = dpk; dqkm2 = dqkm1; dqkm1 = dqk;
    if (fabsf(pk) > 1e18f || fabsf(qk) > 1e18f) {
      const float sc = 1e-18f;
      pkm2 *= sc; pkm1 *= sc; qkm2 *= sc; qkm1 *= sc;
      dpkm2 *= sc; dpkm1 *= sc; dqkm2 *= sc; dqkm1 *= sc;
    }
    if (delta < 1e-6f * scale && c > 3) break;
  }
  return x * (dans + ans * (SPMF_LOGF(x) - psi));
}

// Series half: fills out[j] for the draws in the power-series regime and returns the mask of the draws
// that need the continued fraction instead (gamma_der_cf).
SPMF_HD unsigned gamma_der_series4(float a, float psi, const float (&x)[4], int n, float (&out)[4]) {
  bool ser[4];
  bool any_ser = false;
  unsigned cf = 0u;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    ser[j] = j < n && x[j] > 0.f && (x[j] <= 1.f || x[j] <= a + 1.f);
    any_ser = any_ser || ser[j];
    out[j] = 0.f;
    if (j < n && !ser[j] && x[j] > 0.f) cf |= 1u << j;
  }
  if (any_ser) {
    float T[4], sT[4], sTH[4], xs[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) { T[j] = 1.f; sT[j] = 1.f; sTH[j] = 0.f; xs[j] = ser[j] ? x[j] : 0.f; }
    float H = 0.f;
    for (int k = 1; k < 400; ++k) {
      const float inv = SPMF_RCPF(a + (float)k);
      H += inv;
      bool done = true;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        T[j] *= xs[j] * inv;
        sT[j] += T[j];
        sTH[j] = fmaf(T[j], H, sTH[j]);
        done = done && (T[j] * (1.f + H) < 1e-7f * sT[j]);
      }
      if (done) break;
    }
    const float psi1 = psi + 1.f / a;          // digamma(a+1)
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (ser[j]) out[j] = (x[j] / a) * (sTH[j] - (SPMF_LOGF(x[j]) - psi1) * sT[j]);
  }
  return cf;
}

SPMF_HD void gamma_sample_der_alpha4(float a, float psi, const float (&x)[4], int n, float (&out)[4]) {
  const unsigned cf = gamma_der_series4(a, psi, x, n, out);
#pragma unroll
  for (int j = 0; j < 4; ++j)
    if (cf & (1u << j)) out[j] = gamma_der_cf(a, psi, x[j]);
}

// ---------------------------------------------------------------------------
// Philox4x32-10 counter RNG (Salmon et al. 2011).  Own implementation so that the
// stream is a pure function of (seed, var, step, element) and identical on every rank.
// ---------------------------------------------------------------------------
struct U4 { uint32_t x, y, z, w; };

SPMF_HD uint32_t mulhi32(uint32_t a, uint32_t b) { return (uint32_t)(((uint64_t)a * b) >> 32); }

SPMF_HD U4 philox4x32_10(U4 ctr, uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = mulhi32(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = mulhi32(M1, ctr.z), lo1 = M1 * ctr.z;
    U4 n;
    n.x = hi1 ^ ctr.y ^ k0;
    n.y = lo1;
    n.z = hi0 ^ ctr.w ^ k1;
    n.w = lo0;
    ctr = n;
    k0 += W0;
    k1 += W1;
  }
  return ctr;
}

// (0,1] uniform from 32 random bits
SPMF_HD float u01(uint32_t r) { return ((float)(r >> 8) + 1.0f) * (1.0f / 16777216.0f); }

SPMF_HD void box_muller(uint32_t r0, uint32_t r1, float* n0, float* n1) {
  float u = u01(r0), v = u01(r1);
  float rad = sqrtf(-2.f * logf(u));
  float ang = 6.283185307179586f * v;
  *n0 = rad * cosf(ang);
  *n1 = rad * sinf(ang);
}

// Marsaglia-Tsang standard Gamma(alpha) draw; one private Philox stream per element.
SPMF_HD float gamma_draw(float alpha, uint32_t elem_lo, uint32_t elem_hi, uint32_t stream,
                         uint32_t k0, uint32_t k1) {
  float a = alpha < 1.f ? alpha + 1.f : alpha;
  float d = a - 1.f / 3.f;
  float c = 1.f / sqrtf(9.f * d);
  float boost = 1.f;
  float g = d;
  for (uint32_t it = 0; it < 64; ++it) {
    U4 ctr = {elem_lo, elem_hi, stream, it};
    U4 r = philox4x32_10(ctr, k0, k1);
    const float n0 = sqrtf(-2.f * SPMF_LOGF(u01(r.x))) * SPMF_COSF(6.283185307179586f * u01(r.y));
    if (it == 0 && alpha < 1.f) boost = powf(u01(r.w), 1.f / alpha);
    float v = 1.f + c * n0;
    if (v <= 0.f) continue;
    v = v * v * v;
    float u = u01(r.z);
    float x2 = n0 * n0;
    if (u < 1.f - 0.0331f * x2 * x2 || SPMF_LOGF(u) < 0.5f * x2 + d * (1.f - v + SPMF_LOGF(v))) {
      g = d * v;
      break;
    }
  }
  g *= boost;
  return fmaxf(g, 1.17549435e-38f);
}

// ---------------------------------------------------------------------------
// Poisson and Bernoulli draws of the posterior predictive replicates (csrc/spmf_ppc.cu).  Pure functions
// of the parameter, a Philox key and a counter: the i-th Philox call of a draw uses `ctr` with ctr.w + i.
// ---------------------------------------------------------------------------
struct Key2 { uint32_t k0, k1; };

constexpr float kPoissonInvMax = 10.f;        // inversion below this rate, PTRS from it on
constexpr int kPoissonInvCap = 64;            // inversion search stops at this count
constexpr int kPoissonPtrsCalls = 8;          // Philox calls of one PTRS draw: 2 candidates each
// Largest valid Poisson rate: keeps every replicate an exact int32 and the per-column sums of squares
// of a batch well inside 64 bits.
constexpr float kPoissonMaxRate = 16777216.f;  // 2^24

SPMF_HD bool poisson_rate_ok(float lam) { return lam >= 0.f && lam <= kPoissonMaxRate; }   // false for NaN

// Sequential-search inversion of the CDF at u in (0,1].  The search stops where the next pmf term no
// longer changes F in fp32 (or at kPoissonInvCap): the tail mass beyond that point -- a few times 2^-24,
// the resolution of u01 -- lands on the count reached there.
SPMF_HD int poisson_inversion(float lam, float u) {
  float p = expf(-lam), F = p;
  int k = 0;
  while (u > F && k < kPoissonInvCap) {
    ++k;
    p *= lam / (float)k;
    const float Fn = F + p;
    if (Fn == F) break;
    F = Fn;
  }
  return k;
}

// log k! in double for integer k >= 0 (numpy's random_loggam: Stirling series from 7 on, the recurrence below)
SPMF_HD double log_factorial(double k) {
  double x = k + 1.0, shift = 0.0;
  if (x <= 2.0) return 0.0;
  while (x < 7.0) {
    shift += log(x);
    x += 1.0;
  }
  const double x2 = 1.0 / (x * x);
  const double g = 8.333333333333333e-02 + x2 * (-2.777777777777778e-03 + x2 * (7.936507936507937e-04 +
                   x2 * (-5.952380952380952e-04 + x2 * (8.417508417508418e-04 + x2 * (-1.917526917526918e-03 +
                   x2 * (6.410256410256410e-03 + x2 * (-2.955065359477124e-02 + x2 * (1.796443723688307e-01 +
                   x2 * -1.39243221690590e+00))))))));
  return g / x + 0.9189385332046727 + (x - 0.5) * log(x) - x - shift;
}

// Transformed rejection with squeeze (PTRS, Hoermann 1993; the method of numpy's random_poisson_ptrs)
// for lam >= kPoissonInvMax.  The acceptance test -lam + k log lam - log k! is evaluated in double: in fp32
// the two large terms (~1e6 at lam = 1e5) cancel to O(1) and lgammaf alone is off by about one unit.  A
// candidate is accepted with probability above 0.9, so all 2*kPoissonPtrsCalls candidates are rejected with
// probability below 1e-15; the draw then returns floor(lam), the mode.
SPMF_HD int poisson_ptrs(float lam, Key2 key, U4 ctr) {
  const float slam = sqrtf(lam);
  const double dlam = (double)lam, dloglam = log(dlam);
  const float b = 0.931f + 2.53f * slam;
  const float a = -0.059f + 0.02483f * b;
  const float log_invalpha = logf(1.1239f + 1.1328f / (b - 3.4f));
  const float vr = 0.9277f - 3.6224f / (b - 2.f);
  for (int call = 0; call < kPoissonPtrsCalls; ++call) {
    U4 c = ctr;
    c.w += (uint32_t)call;
    const U4 r = philox4x32_10(c, key.k0, key.k1);
    for (int h = 0; h < 2; ++h) {
      const float U = u01(h ? r.z : r.x) - 0.5f, V = u01(h ? r.w : r.y);
      const float us = 0.5f - fabsf(U);
      if (us < 0.013f && V > us) continue;          // (also every us == 0, before 2a/us is formed)
      const double k = floor((double)(2.f * a / us + b) * (double)U + dlam + 0.43);
      if (us >= 0.07f && V <= vr) return (int)k;
      if (k < 0.0) continue;
      const double rhs = -dlam + k * dloglam - log_factorial(k);
      if ((double)(logf(V) + log_invalpha - logf(a / (us * us) + b)) <= rhs) return (int)k;
    }
  }
  return (int)floorf(lam);
}

// Poisson(lam) for a valid rate (poisson_rate_ok); 0 for lam == 0 and for anything invalid.
SPMF_HD int poisson_draw(float lam, Key2 key, U4 ctr) {
  if (!(lam > 0.f) || !(lam <= kPoissonMaxRate)) return 0;
  if (lam < kPoissonInvMax) return poisson_inversion(lam, u01(philox4x32_10(ctr, key.k0, key.k1).x));
  return poisson_ptrs(lam, key, ctr);
}

// Bernoulli(p): 1 iff u01 <= p, so P(1) = floor(p * 2^24) / 2^24 -- p is resolved to 2^-24 (p = 0 never
// gives 1, p = 1 always does).
SPMF_HD int bernoulli_draw(float p, Key2 key, U4 ctr) {
  return u01(philox4x32_10(ctr, key.k0, key.k1).x) <= p ? 1 : 0;
}

// Replicate stream of entry (draw s, global row, feature d) under a check seed.  The seed is mixed with a
// constant, so the key differs from the training noise key (the model seed) even for equal seeds; the
// counter holds (d, row bits 0-31, row bits 32-47 | s << 16, call).  Needs s < 2^16 and row < 2^48.
SPMF_HD Key2 ppc_key(uint64_t seed) { return Key2{(uint32_t)seed, (uint32_t)(seed >> 32) ^ 0x50504331u}; }
SPMF_HD U4 ppc_counter(int s, long long row, int d) {
  const uint64_t r = (uint64_t)row;
  return U4{(uint32_t)d, (uint32_t)r, (uint32_t)((r >> 32) & 0xffffu) | ((uint32_t)s << 16), 0u};
}

}  // namespace spmf
