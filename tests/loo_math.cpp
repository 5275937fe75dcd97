// Test-side C wrappers of the PSIS-LOO pieces of spmf_b200/csrc/spmf_loo.cuh (__host__ __device__), so
// tests/test_loo_host.py can run the kernel's own scalar math on the CPU.  Compiled by that test with g++ into a
// temporary directory; never shipped.
#include "../spmf_b200/csrc/spmf_loo.cuh"

using namespace spmf;

extern "C" {

int hc_tail_len(int S) { return loo_tail_len(S); }
int hc_grid_size(int n) { return loo_grid_size(n); }
int hc_quartile_index(int n) { return loo_quartile_index(n); }
double hc_grid_b(int j, int m, double y_last, double y_quart) { return loo_grid_b(j, m, y_last, y_quart); }
double hc_profile(int n, double b, double k) { return loo_profile(n, b, k); }
double hc_gpd_quantile(double p, double k, double sigma) { return loo_gpd_quantile(p, k, sigma); }
double hc_log_dbl_min() { return kLooLogDblMin; }
int hc_max_tail() { return kLooMaxTail; }
int hc_max_grid() { return kLooMaxGrid; }

}  // extern "C"
