// Test-side C wrappers of the replicate samplers of spmf_b200/csrc/spmf_math.cuh (poisson_draw /
// bernoulli_draw are __host__ __device__), so tests/test_ppc_host.py can run the kernel's own sampling code
// on the CPU.  Compiled by that test with g++ into a temporary directory; never shipped.
#include "../spmf_b200/csrc/spmf_math.cuh"

using namespace spmf;

extern "C" {

// draw i: parameter p[i], key (k0, k1), counter (i_lo, i_hi, c2, 0)
void hc_poisson(const float* lam, int* out, long long n, unsigned k0, unsigned k1, unsigned c2) {
  for (long long i = 0; i < n; ++i)
    out[i] = poisson_draw(lam[i], Key2{k0, k1}, U4{(uint32_t)i, (uint32_t)(i >> 32), c2, 0u});
}
void hc_bernoulli(const float* p, int* out, long long n, unsigned k0, unsigned k1, unsigned c2) {
  for (long long i = 0; i < n; ++i)
    out[i] = bernoulli_draw(p[i], Key2{k0, k1}, U4{(uint32_t)i, (uint32_t)(i >> 32), c2, 0u});
}

}  // extern "C"
