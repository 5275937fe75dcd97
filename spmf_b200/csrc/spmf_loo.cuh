// Scalar fp64 pieces of Pareto-smoothed importance-sampling leave-one-out (PSIS-LOO, Vehtari, Gelman & Gabry
// 2017; the generalised Pareto fit of Zhang & Stephens 2009 with Vehtari's weakly informative prior), as ArviZ's
// _psislw / _gpdfit compute them with r_eff = 1.  Every function is __host__ __device__ so that
// tests/test_loo_host.py runs the kernel's own math on the CPU (through tests/loo_math.cpp) against
// oracle/psis.py.  The kernel that uses them is csrc/spmf_loo.cu.
#pragma once
#include <math.h>

#include "spmf_math.cuh"

namespace spmf {

constexpr double kLooLogDblMin = -708.3964185322641;   // log(DBL_MIN): the lowest cutoff of the tail
constexpr int kLooMaxTail = 272;                       // loo_tail_len(SPMF_LOO_MAX_S = 8192)
constexpr int kLooMaxGrid = 46;                        // loo_grid_size(kLooMaxTail)

// M = ceil(min(0.2 S, 3 sqrt(S))) draws of largest log-ratio may form the tail; the cutoff is the (M+1)-th largest
// value.  At S = 1 the formula gives M = S, which leaves no cutoff value: M is capped at S - 1 (no tail).
SPMF_HD int loo_tail_len(int S) {
  const int M = (int)ceil(fmin(0.2 * S, 3.0 * sqrt((double)S)));
  return M < S - 1 ? M : S - 1;
}

// grid of the profile fit: m = 30 + floor(sqrt(n)) points for a tail of n values
SPMF_HD int loo_grid_size(int n) { return 30 + (int)floor(sqrt((double)n)); }

// index (0-based, ascending tail) of the first-quartile value the grid is scaled by: floor(n/4 + 1/2) - 1
SPMF_HD int loo_quartile_index(int n) { return (int)(n / 4.0 + 0.5) - 1; }

// grid point b_j, j = 1..m:  1/y_n + (1 - sqrt(m/(j - 1/2))) / (3 y_q)
SPMF_HD double loo_grid_b(int j, int m, double y_last, double y_quart) {
  return (1.0 - sqrt(m / (j - 0.5))) / (3.0 * y_quart) + 1.0 / y_last;
}

// profile log-likelihood of grid point b with k = mean_i log1p(-b y_i):  n (log(-b/k) - k - 1)
SPMF_HD double loo_profile(int n, double b, double k) { return n * (log(-(b / k)) - k - 1.0); }

// generalised Pareto quantile at p of shape k and scale sigma (location 0); k -> 0 is the exponential quantile
SPMF_HD double loo_gpd_quantile(double p, double k, double sigma) {
  if (fabs(k) < 2.220446049250313e-16) return sigma * -log1p(-p);
  return expm1(-k * log1p(-p)) / k * sigma;
}

}  // namespace spmf
