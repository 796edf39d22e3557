// CPU driver of hmc.jl_b200/csrc/psis.cuh for tests/test_loo.py: the PSIS steps of include/hmcgpu.h (hmcgpu_loo) around the
// header's tail length, gpdfit, GPD quantile and k̂ threshold, compiled with g++.
//   psis_driver params R         -> "M m threshold"
//   psis_driver psis < R r_1..r_R -> k̂, then the truncated log weights lw_d (before normalisation), one per line
#include <algorithm>
#include <cfloat>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <numeric>
#include <vector>

#include "psis.cuh"

int main(int argc, char** argv) {
    using namespace hmc;
    if (argc >= 3 && !strcmp(argv[1], "params")) {
        const long long R = atoll(argv[2]);
        const int M = psis_tail_len(R);
        printf("%d %d %.17g\n", M, gpd_grid_len(M), psis_k_threshold(R));
        return 0;
    }
    if (argc < 2 || strcmp(argv[1], "psis")) { fprintf(stderr, "usage: psis_driver params R | psis < ratios\n"); return 2; }
    long long R = 0;
    if (scanf("%lld", &R) != 1 || R < 2) return 2;
    std::vector<double> lw(R);
    for (auto& v : lw)
        if (scanf("%lf", &v) != 1) return 2;
    const double mx = *std::max_element(lw.begin(), lw.end());
    for (auto& v : lw) v -= mx;
    const int M = psis_tail_len(R);
    double k = INFINITY;
    if (M >= 5) {
        std::vector<int> ord(R);
        std::iota(ord.begin(), ord.end(), 0);
        std::sort(ord.begin(), ord.end(), [&](int a, int b) { return lw[a] < lw[b] || (lw[a] == lw[b] && a < b); });
        const int* tail = ord.data() + (R - M);
        if (std::fabs(lw[tail[M - 1]] - lw[tail[0]]) >= DBL_EPSILON / 100) {
            const double cutoff = lw[ord[R - M - 1]], ec = std::exp(cutoff);
            std::vector<double> x(M);
            for (int j = 0; j < M; ++j) x[j] = std::exp(lw[tail[j]]) - ec;
            double sigma;
            gpdfit(x.data(), M, &k, &sigma);
            if (std::isfinite(k))
                for (int j = 0; j < M; ++j) lw[tail[j]] = std::log(gpd_quantile((j + 0.5) / M, k, sigma) + ec);
        }
    }
    printf("%.17g\n", k);
    for (auto v : lw) printf("%.17g\n", std::min(v, 0.0));
    return 0;
}
