// Predictive CDFs and the Czado PIT binning of the LOO-PIT pass (csrc/spmf_pit.cu), in fp64 and
// __host__ __device__ so that tests/pit_math.cpp runs the kernel's own code on the CPU.
//
// poisson_cdf(x, lam) = P(X <= x) for X ~ Poisson(lam) is the regularised upper incomplete gamma Q(x + 1, lam):
// the series of P(a, lam) below lam < a = x + 1 (Q = 1 - P) and the modified Lentz continued fraction of Q from
// lam >= a on (Numerical Recipes 6.2).  Both are scaled by a Poisson pmf taken in Loader's saddle-point form
// (stirlerr + bd0, as R's dpois_raw), which keeps its relative error near 1e-15 where the direct
// exp(x log lam - lam - lgamma(x + 1)) would lose ~x log lam * eps (3e-8 at x = 2^24).
#pragma once
#include <math.h>

#include "spmf_math.cuh"

namespace spmf {

constexpr double kPitMaxValue = 16777216.0;   // 2^24: the largest count and Poisson rate the CDF takes
// Iteration bound of both the series and the continued fraction.  The worst case is lam just either side of
// a = x + 1 at the top of the range, where both need ~sqrt(74 a) terms (terms fall like exp(-n^2 / 2a) down to
// eps): 35,200 at a = 2^24 + 1.  tests/test_pit_host.py measures the largest count used over the grid.
constexpr int kPitMaxIter = 40000;

// Stirling's error log(n!) - ((n + 1/2) log n - n + log sqrt(2 pi)), n >= 32 (five terms: error < 1e-20)
SPMF_HD double pit_stirlerr(double n) {
  const double nn = 1.0 / (n * n);
  return (1.0 / 12 - (1.0 / 360 - (1.0 / 1260 - (1.0 / 1680 - nn / 1188) * nn) * nn) * nn) / n;
}

// Loader's deviance term x log(x / m) + m - x, without cancellation for x close to m
SPMF_HD double pit_bd0(double x, double m) {
  if (fabs(x - m) < 0.1 * (x + m)) {
    double v = (x - m) / (x + m);
    double s = (x - m) * v, ej = 2.0 * x * v;
    v *= v;
    for (int j = 1; j < 100; ++j) {                  // v^2 < 0.0083: at most ~9 terms
      ej *= v;
      const double s1 = s + ej / (2 * j + 1);
      if (s1 == s) return s1;
      s = s1;
    }
    return s;
  }
  return x * log(x / m) + m - x;
}

// Poisson pmf lam^k e^-lam / k!, k a non-negative integer, lam >= 0
SPMF_HD double pit_poisson_pmf(double k, double lam) {
  if (lam == 0.0) return k == 0.0 ? 1.0 : 0.0;
  if (k == 0.0) return exp(-lam);
  if (k < 32.0) return exp(k * log(lam) - lam - lgamma(k + 1.0));
  return exp(-pit_stirlerr(k) - pit_bd0(k, lam)) / sqrt(6.283185307179586476925 * k);
}

// (F(x - 1), F(x)) of Poisson(lam) for an integer 0 <= x <= 2^24 and 0 <= lam <= 2^24, sharing one evaluation:
// F(x - 1) = F(x) - pmf(x), clamped at 0.  *iters (may be NULL) = terms used.
SPMF_HD void poisson_cdf_pair(double x, double lam, double* fm, double* fp, int* iters = nullptr) {
  if (x == 0.0) {                                    // the zeros: F(-1) = 0, F(0) = e^-lam
    *fm = 0.0;
    *fp = exp(-lam);
    if (iters) *iters = 0;
    return;
  }
  const double a = x + 1.0;
  double q, pmf;
  int it = 0;
  if (lam < a) {                                     // P(a, lam) = pmf(a) sum_n lam^n / ((a+1)...(a+n))
    const double pa = pit_poisson_pmf(a, lam);
    double del = 1.0, sum = 1.0, ap = a;
    for (it = 1; it <= kPitMaxIter; ++it) {
      ap += 1.0;
      del *= lam / ap;
      sum += del;
      if (del < sum * 1e-17) break;
    }
    q = 1.0 - pa * sum;
    pmf = lam > 0.0 ? pa * a / lam : (x == 0.0 ? 1.0 : 0.0);   // pmf(x) = pmf(x + 1) (x + 1) / lam
  } else {                                           // Q(a, lam) = lam pmf(x) / (lam + 1 - a - 1(1-a)/(lam + 3 - a - ...))
    pmf = pit_poisson_pmf(x, lam);
    const double tiny = 1e-300;
    double b = lam + 1.0 - a, c = 1.0 / tiny, d = 1.0 / b, h = d;
    for (it = 1; it <= kPitMaxIter; ++it) {
      const double an = -it * (it - a);
      b += 2.0;
      d = an * d + b;
      if (fabs(d) < tiny) d = tiny;
      c = b + an / c;
      if (fabs(c) < tiny) c = tiny;
      d = 1.0 / d;
      const double del = d * c;
      h *= del;
      if (fabs(del - 1.0) < 1e-16) break;
    }
    q = lam * pmf * h;
  }
  q = fmin(fmax(q, 0.0), 1.0);
  *fp = q;
  *fm = fmax(q - pmf, 0.0);
  if (iters) *iters = it;
}

// P(X <= x), X ~ Poisson(lam): integer x >= -1 (F(-1) = 0), 0 <= x, lam <= 2^24
SPMF_HD double poisson_cdf(double x, double lam) {
  if (x < 0.0) return 0.0;
  double fm, fp;
  poisson_cdf_pair(x, lam, &fm, &fp);
  return fp;
}

// P(X <= x), X ~ Bernoulli(sigmoid(logit)): F(-1) = 0, F(0) = 1 - sigmoid(logit) = sigmoid(-logit), F(1) = 1
SPMF_HD double bernoulli_cdf(double x, double logit) {
  if (x < 0.0) return 0.0;
  if (x >= 1.0) return 1.0;
  if (logit >= 0.0) {
    const double e = exp(-logit);
    return e / (1.0 + e);
  }
  return 1.0 / (1.0 + exp(logit));
}

// an observed value the CDF takes: an integer in the support (0 <= x <= 2^24 for Poisson, x in {0, 1} for
// Bernoulli); false for NaN
SPMF_HD bool pit_count_ok(float x, bool bernoulli) {
  return x >= 0.f && x <= (bernoulli ? 1.f : (float)kPitMaxValue) && x == floorf(x);
}

// Czado, Gneiting & Held (2009): the non-randomised PIT of one entry has the distribution function
// F(u) = 0 (u <= lo), (u - lo) / (hi - lo) (lo < u < hi), 1 (u >= hi), with lo, hi = P-, P+ clamped to [0, 1].
SPMF_HD double czado_cdf(double u, double lo, double hi) {
  if (u <= lo) return 0.0;
  if (u >= hi) return 1.0;
  return (u - lo) / (hi - lo);
}

// the mass of bin j = 0..J-1 (the interval (j/J, (j+1)/J]) of one entry: F((j+1)/J) - F(j/J); if hi <= lo the
// entry puts unit mass in bin min(J - 1, floor(hi J))
SPMF_HD double czado_bin_mass(double pm, double pp, int j, int J) {
  const double lo = fmin(fmax(pm, 0.0), 1.0), hi = fmin(fmax(pp, 0.0), 1.0);
  if (hi <= lo) {
    const int b = (int)fmin((double)(J - 1), floor(hi * J));
    return b == j ? 1.0 : 0.0;
  }
  return czado_cdf((double)(j + 1) / J, lo, hi) - czado_cdf((double)j / J, lo, hi);
}

}  // namespace spmf
