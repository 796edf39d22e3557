// psis.cuh — the numerics of Pareto-smoothed importance sampling (HMCGPU_FLAG_LOO), shared by the device (loo.cuh) and by
// the CPU test driver tests/psis_driver.cpp: plain C++17 that nvcc compiles as __host__ __device__ and g++ compiles as is.
//
// This is the algorithm of the R package `loo` 2.x with r_eff = 1 (Vehtari, Gelman & Gabry 2017; Zhang & Stephens 2009):
// n_pareto_draws (the tail length), gpdfit (wip = TRUE, min_grid_pts = 30, prior 3), qgpd, and the k̂ threshold of
// pareto_k_table.  The sort, the selection of the tail and the reductions over all draws live with their callers.
#pragma once
#include <cmath>

#ifdef __CUDACC__
#define HMC_PSIS_FN __host__ __device__ inline
#else
#define HMC_PSIS_FN inline
#endif

namespace hmc {

constexpr long long kLooMaxDraws = 1ll << 24;   // R = n_chains * nrun per window; the tail then holds at most 3 * 2^12 values
constexpr int kLooMaxTail = 12288;

// M = ceil(min(0.2 R, 3 sqrt(R))): the draws in the smoothed tail (the largest M log ratios)
HMC_PSIS_FN int psis_tail_len(long long R) {
    const double a = 0.2 * (double)R, b = 3.0 * sqrt((double)R);
    return (int)ceil(a < b ? a : b);
}

// min(1 - 1/log10(R), 0.7): above it the importance-sampling estimate of a date is unreliable
HMC_PSIS_FN double psis_k_threshold(long long R) {
    const double t = 1.0 - 1.0 / log10((double)R);
    return t < 0.7 ? t : 0.7;
}

// points of gpdfit's grid over theta for a tail of M values
HMC_PSIS_FN int gpd_grid_len(int M) { return 30 + (int)floor(sqrt((double)M)); }

// grid point j = 1..m: theta_j = 1/x_(M) + (1 - sqrt(m / (j - 1/2))) / (prior x*), x* = x_(floor(M/4 + 1/2)) (1-based, x sorted)
HMC_PSIS_FN double gpd_theta(int j, int m, double x_last, double xstar) {
    return 1.0 / x_last + (1.0 - sqrt((double)m / ((double)j - 0.5))) / 3.0 / xstar;
}

// M times the profile log-likelihood at theta, from mean_log1p = (1/M) sum_i log1p(-theta x_i)  (`loo`'s lx)
HMC_PSIS_FN double gpd_profile(double theta, double mean_log1p, int M) {
    return (double)M * (log(-theta / mean_log1p) - mean_log1p - 1.0);
}

// From the posterior mean theta_hat of the grid and mean_log1p = (1/M) sum_i log1p(-theta_hat x_i): sigma = -k / theta_hat with
// the raw k, then the weakly informative prior k <- (M k + 5) / (M + 10); a NaN k becomes +inf.
HMC_PSIS_FN void gpd_finish(double theta_hat, double mean_log1p, int M, double* k, double* sigma) {
    const double kr = mean_log1p;
    *sigma = -kr / theta_hat;
    double kk = kr * M / (M + 10.0) + 10.0 * 0.5 / (M + 10.0);
    if (kk != kk) kk = INFINITY;
    *k = kk;
}

// the generalised Pareto quantile sigma expm1(-k log1p(-p)) / k (NaN when sigma is not positive, as `loo`'s qgpd)
HMC_PSIS_FN double gpd_quantile(double p, double k, double sigma) {
    if (!(sigma > 0.0)) return NAN;
    return sigma * expm1(-k * log1p(-p)) / k;
}

// Serial gpdfit of x[0..M) sorted ascending (every sum in index order); the device runs the same steps in parallel (loo.cuh).
HMC_PSIS_FN void gpdfit(const double* x, int M, double* k, double* sigma) {
    const int m = gpd_grid_len(M);
    const double xstar = x[(int)floor(M / 4.0 + 0.5) - 1], xl = x[M - 1];
    double lmax = -INFINITY;
    for (int j = 1; j <= m; ++j) {
        const double th = gpd_theta(j, m, xl, xstar);
        double s = 0.0;
        for (int i = 0; i < M; ++i) s += log1p(-th * x[i]);
        const double l = gpd_profile(th, s / M, M);
        if (l > lmax) lmax = l;
    }
    double sw = 0.0, swt = 0.0;
    for (int j = 1; j <= m; ++j) {
        const double th = gpd_theta(j, m, xl, xstar);
        double s = 0.0;
        for (int i = 0; i < M; ++i) s += log1p(-th * x[i]);
        const double e = exp(gpd_profile(th, s / M, M) - lmax);
        sw += e;
        swt += th * e;
    }
    const double theta_hat = swt / sw;
    double s = 0.0;
    for (int i = 0; i < M; ++i) s += log1p(-theta_hat * x[i]);
    gpd_finish(theta_hat, s / M, M, k, sigma);
}

}  // namespace hmc
