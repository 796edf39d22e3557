// Device driver of loo_psis_kernel (hmc.jl_b200/csrc/loo.cuh) for tests/test_loo.py: the PSIS step of hmcgpu_loo on caller-given
// pointwise terms, so that ratio sets the sampler does not produce on demand (ties with the cutoff, heavy tails) reach the
// device code.  Reads "R n_dates" and then, per date, R values of ell followed by R values of F (stdin); prints per date
// "elpd lppd pareto_k pit".  Built with nvcc for sm_100a by the test.
#include <cstdio>
#include <vector>

#include "loo.cuh"

#define CHECK(x)                                                                   \
    do {                                                                           \
        const cudaError_t e_ = (x);                                                \
        if (e_ != cudaSuccess) {                                                   \
            fprintf(stderr, "%s: %s\n", #x, cudaGetErrorString(e_));               \
            return 1;                                                              \
        }                                                                          \
    } while (0)

int main() {
    using namespace hmc;
    long long R = 0, n = 0;
    if (scanf("%lld %lld", &R, &n) != 2 || R < 2 || R > kLooMaxDraws || n < 1) return 2;
    std::vector<double> ell((size_t)R * n), F((size_t)R * n);
    for (long long j = 0; j < n; ++j) {
        for (long long d = 0; d < R; ++d)
            if (scanf("%lf", &ell[(size_t)j * R + d]) != 1) return 2;
        for (long long d = 0; d < R; ++d)
            if (scanf("%lf", &F[(size_t)j * R + d]) != 1) return 2;
    }
    double *d_ell, *d_F, *d_out;
    CHECK(cudaMalloc(&d_ell, ell.size() * sizeof(double)));
    CHECK(cudaMalloc(&d_F, F.size() * sizeof(double)));
    CHECK(cudaMalloc(&d_out, 4 * (size_t)n * sizeof(double)));
    CHECK(cudaMemcpy(d_ell, ell.data(), ell.size() * sizeof(double), cudaMemcpyHostToDevice));
    CHECK(cudaMemcpy(d_F, F.data(), F.size() * sizeof(double), cudaMemcpyHostToDevice));
    const size_t smem = loo_psis_smem(R);
    if (smem > 48 * 1024) CHECK(cudaFuncSetAttribute(loo_psis_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    loo_psis_kernel<<<(unsigned)n, kLooThreads, smem>>>(R, 0, d_ell, d_F, d_out, d_out + n, d_out + 2 * n, d_out + 3 * n);
    CHECK(cudaGetLastError());
    std::vector<double> out(4 * (size_t)n);
    CHECK(cudaMemcpy(out.data(), d_out, out.size() * sizeof(double), cudaMemcpyDeviceToHost));
    for (long long j = 0; j < n; ++j) printf("%.17g %.17g %.17g %.17g\n", out[j], out[n + j], out[2 * n + j], out[3 * n + j]);
    cudaFree(d_ell);
    cudaFree(d_F);
    cudaFree(d_out);
    return 0;
}
