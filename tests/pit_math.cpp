// Test-side C wrappers of the predictive CDFs and the Czado binning of spmf_b200/csrc/spmf_pit.cuh (all
// __host__ __device__), so tests/test_pit_host.py can run the kernel's own code on the CPU.  Compiled by that
// test with g++ into a temporary directory; never shipped.
#include "../spmf_b200/csrc/spmf_pit.cuh"

using namespace spmf;

extern "C" {

void hc_poisson_cdf(const double* x, const double* lam, double* out, long long n) {
  for (long long i = 0; i < n; ++i) out[i] = poisson_cdf(x[i], lam[i]);
}
// (F(x - 1), F(x)) and the terms used
void hc_poisson_cdf_pair(const double* x, const double* lam, double* fm, double* fp, int* iters, long long n) {
  for (long long i = 0; i < n; ++i) poisson_cdf_pair(x[i], lam[i], fm + i, fp + i, iters + i);
}
void hc_bernoulli_cdf(const double* x, const double* logit, double* out, long long n) {
  for (long long i = 0; i < n; ++i) out[i] = bernoulli_cdf(x[i], logit[i]);
}
// out[i][j] = czado_bin_mass(pm[i], pp[i], j, J)
void hc_czado_bins(const double* pm, const double* pp, long long n, int J, double* out) {
  for (long long i = 0; i < n; ++i)
    for (int j = 0; j < J; ++j) out[i * J + j] = czado_bin_mass(pm[i], pp[i], j, J);
}
int hc_count_ok(float x, int bernoulli) { return pit_count_ok(x, bernoulli != 0); }

}  // extern "C"
