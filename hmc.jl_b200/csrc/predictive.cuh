// predictive.cuh — posterior predictive distribution of every forecast (HMCGPU_FLAG_PREDICTIVE), streamed over the saved draws
// as they pass through the per-chunk buffer out[(f*chunk + i)*n_slots + slot].
//
// Draw d of a window defines, for horizon h, the Gaussian mixture with weights v = pi_end' A^h and components N(mu_s, sigma2_s).
// Per (slot, horizon) a running fp64 state keeps, in draw order:
//   cdf[g]  = sum_d F_d(grid[g])                     F_d(x) = sum_s v_s Phi((x - mu_s) / sigma_s)
//   pit     = sum_d F_d(y+)                          y+ = y[end + h] (NaN past the series)
//   dens    = sum_d p_d(y+)                          p_d(x) = sum_s v_s phi((x - mu_s) / sigma_s) / sigma_s
//   m1..m3  = sum_d sum_s v_s E[(Y_s - c)^k]         raw moments of the draw's mixture about the window's last observation c
// pred_finish_kernel then adds the window's chains in chain order and divides by R.  No atomics: a window's outputs do not
// depend on the chunk size, the batch or the sharding (the per-chain draws being equal).  All arithmetic is fp64 on the draws
// converted to double.  tests/test_predictive.py holds the numpy definition it matches.
#pragma once
#include <cuda_runtime.h>
#include "gibbs_kernel.cuh"     // kMaxH

namespace hmc {

constexpr int kPredThreads = 256;
constexpr int kPredScores = 5;      // pit, dens, m1, m2, m3

// horizons ascending and their position in the caller's list (as GibbsArgs::h_sorted / h_slot)
struct PredHorizons {
    int h_sorted[kMaxH];
    int h_slot[kMaxH];
};

// Dynamic shared memory of pred_accum_kernel for `pairs` (slot, draw) pairs per tile.
inline size_t pred_smem_bytes(int K, int n_h, int pairs) {
    return ((size_t)pairs * K * (5 + n_h) + (size_t)kMaxH * 8 * kPredScores) * sizeof(double) + (size_t)pairs * sizeof(int);
}

// Adds draws [0, n_i) of a chunk buffer to the running state of `sb` = kPredThreads / tg consecutive slots (one block).  Draws
// are taken in tiles of td; per tile the block
//   1. stages mu, sigma2, sigma and pi_end of every (slot, draw) pair in shared memory and flags pairs with a non-finite
//      mu / sigma2 / A / pi_end value;
//   2. walks the horizons in ascending order, one transition step v <- v A per __syncthreads, thread per (pair, state), and
//      keeps v for every horizon (the weights, computed once per pair);
//   3. thread (slot b, grid point g [+ tg]) evaluates Phi((g - mu_s) / sigma_s) once per state and adds v_s Phi to the CDF sums
//      of every horizon, draw after draw; thread (slot b, horizon j) adds the draw's F(y+), p(y+) and raw moments.
// The CDF sums live in registers for the whole chunk (one block per SM: with fewer registers ptxas spills).  first != 0 starts
// from zero (first chunk of a run).
template <typename R, int GPT>
__global__ void __launch_bounds__(kPredThreads, 1) pred_accum_kernel(int K, int n_h, int n_grid, int n_slots, int chunk, int n_i,
                                                                  int first, int tg, int td, PredHorizons hz,
                                                                  const int* __restrict__ slot_win, const double* __restrict__ cshift_w,
                                                                  const double* __restrict__ yfut_w, const double* __restrict__ grid,
                                                                  const R* __restrict__ out, double* __restrict__ cdf_state,
                                                                  double* __restrict__ score_state) {
    extern __shared__ double psm[];
    const int sb = kPredThreads / tg, P = sb * td, PK = P * K;
    double* s_mu = psm;                 // [P][K]
    double* s_s2 = s_mu + PK;           // [P][K]
    double* s_sd = s_s2 + PK;           // [P][K]
    double* s_cur = s_sd + PK;          // [2][P][K] the vector of the recursion
    double* s_w = s_cur + 2 * PK;       // [P][n_h][K] weights, in the caller's horizon order
    double* s_sc = s_w + (size_t)PK * n_h;  // [sb][n_h][5] the score sums of the block's slots (in shared memory: registers go to the CDF)
    int* s_bad = reinterpret_cast<int*>(s_sc + (size_t)kMaxH * 8 * kPredScores);   // [P]
    const int tid = threadIdx.x;
    const int slot0 = blockIdx.x * sb;
    const size_t cs = (size_t)chunk * n_slots;
    const int fA = 2 * K, fpi = 2 * K + K * K, nf = 3 * K + K * K;

    // CDF role: slot b, grid points g0 + k * tg
    const int b = tid / tg, g0 = tid % tg;
    const int slot = slot0 + b;
    const int w = slot_win[slot];
    double x[GPT], acc[GPT][kMaxH];
#pragma unroll
    for (int k = 0; k < GPT; ++k) {
        const int g = g0 + k * tg;
        x[k] = g < n_grid ? grid[g] : 0.0;
#pragma unroll
        for (int j = 0; j < kMaxH; ++j)
            acc[k][j] = (!first && w >= 0 && g < n_grid && j < n_h) ? cdf_state[((size_t)slot * n_h + j) * n_grid + g] : 0.0;
    }
    // score role: slot bs, horizon js
    const bool scorer = tid < sb * n_h;
    const int bs = scorer ? tid / n_h : 0, js = scorer ? tid % n_h : 0;
    const int sslot = slot0 + bs;
    const int ws = slot_win[sslot];
    const bool sown = scorer && ws >= 0;
    double* sc = s_sc + (size_t)tid * kPredScores;
    if (scorer)
        for (int q = 0; q < kPredScores; ++q) sc[q] = (sown && !first) ? score_state[((size_t)sslot * n_h + js) * kPredScores + q] : 0.0;

    for (int i0 = 0; i0 < n_i; i0 += td) {
        const int m = min(td, n_i - i0);
        const int pm = sb * m;                      // pairs in this tile: (bb, t) -> p = bb * td + t
        __syncthreads();                            // the previous tile's readers are done
        for (int e = tid; e < pm; e += kPredThreads) s_bad[(e / m) * td + e % m] = 0;
        __syncthreads();
        // 1. stage the pairs' parameters; flag non-finite draws
        for (int e = tid; e < pm * nf; e += kPredThreads) {
            const int pl = e / nf, f = e % nf;
            const int bb = pl / m, t = pl % m, p = bb * td + t;
            const int sl = slot0 + bb;
            if (slot_win[sl] < 0) {                 // padding slot: harmless values, results never stored
                if (f < K) { s_mu[p * K + f] = 0.0; s_s2[p * K + f] = 1.0; s_sd[p * K + f] = 1.0; }
                else if (f >= fpi) s_cur[p * K + f - fpi] = 0.0;
                continue;
            }
            const double v = (double)out[(size_t)f * cs + (size_t)(i0 + t) * n_slots + sl];
            if (!isfinite(v)) s_bad[p] = 1;
            if (f < K) s_mu[p * K + f] = v;
            else if (f < fA) { s_s2[p * K + f - K] = v; s_sd[p * K + f - K] = sqrt(v); }
            else if (f >= fpi) s_cur[p * K + f - fpi] = v;
        }
        __syncthreads();
        // 2. weights v = pi' A^h for the horizons in ascending order (A[r][s] is field 2K + s*K + r)
        int h = 0, cb = 0;
        for (int j = 0; j < n_h; ++j) {
            for (; h < hz.h_sorted[j]; ++h) {
                const double* cur = s_cur + cb * PK;
                double* nxt = s_cur + (cb ^ 1) * PK;
                for (int e = tid; e < pm * K; e += kPredThreads) {
                    const int pl = e / K, s = e % K;
                    const int bb = pl / m, t = pl % m, p = bb * td + t;
                    const int sl = slot0 + bb;
                    double a = 0.0;
                    if (slot_win[sl] >= 0) {
                        const R* col = out + (size_t)(fA + s * K) * cs + (size_t)(i0 + t) * n_slots + sl;
                        a = cur[p * K] * (double)col[0];
                        for (int r = 1; r < K; ++r) a = fma(cur[p * K + r], (double)col[(size_t)r * cs], a);
                    }
                    nxt[p * K + s] = a;
                }
                __syncthreads();
                cb ^= 1;
            }
            const double* cur = s_cur + cb * PK;
            for (int e = tid; e < pm * K; e += kPredThreads) {
                const int pl = e / K, s = e % K;
                const int p = (pl / m) * td + pl % m;
                s_w[((size_t)p * n_h + hz.h_slot[j]) * K + s] = cur[p * K + s];
            }
        }
        __syncthreads();
        // 3. accumulate, draw after draw
        for (int t = 0; t < m; ++t) {
            const int p = b * td + t;
            const double* wp = s_w + (size_t)p * n_h * K;
            if (s_bad[p]) {
#pragma unroll
                for (int k = 0; k < GPT; ++k)
#pragma unroll
                    for (int j = 0; j < kMaxH; ++j) acc[k][j] += NAN;
                continue;
            }
            for (int s = 0; s < K; ++s) {
                const double mu = s_mu[p * K + s], sd = s_sd[p * K + s];
                double phi[GPT];
#pragma unroll
                for (int k = 0; k < GPT; ++k) phi[k] = normcdf((x[k] - mu) / sd);
#pragma unroll
                for (int j = 0; j < kMaxH; ++j) {
                    if (j < n_h) {
                        const double v = wp[j * K + s];
#pragma unroll
                        for (int k = 0; k < GPT; ++k) acc[k][j] = fma(v, phi[k], acc[k][j]);
                    }
                }
            }
        }
        if (scorer) {
            const double yp = sown ? yfut_w[(size_t)ws * n_h + js] : 0.0;
            const double cw = sown ? cshift_w[ws] : 0.0;
            for (int t = 0; t < m; ++t) {
                const int p = bs * td + t;
                if (s_bad[p]) {
                    for (int q = 0; q < kPredScores; ++q) sc[q] += NAN;
                    continue;
                }
                const double* wp = s_w + ((size_t)p * n_h + js) * K;
                double F = 0.0, dens = 0.0, r1 = 0.0, r2 = 0.0, r3 = 0.0;
                for (int s = 0; s < K; ++s) {
                    const double v = wp[s], mu = s_mu[p * K + s], s2 = s_s2[p * K + s], sd = s_sd[p * K + s];
                    const double z = (yp - mu) / sd;
                    F = fma(v, normcdf(z), F);
                    dens = fma(v, exp(-0.5 * z * z) * 0.3989422804014327 / sd, dens);   // 1 / sqrt(2 pi)
                    const double d = mu - cw, d2 = d * d;
                    r1 = fma(v, d, r1);
                    r2 = fma(v, d2 + s2, r2);
                    r3 = fma(v, d2 * d + 3.0 * d * s2, r3);
                }
                sc[0] += F; sc[1] += dens; sc[2] += r1; sc[3] += r2; sc[4] += r3;
            }
        }
    }
    if (w >= 0) {
#pragma unroll
        for (int k = 0; k < GPT; ++k) {
            const int g = g0 + k * tg;
            if (g < n_grid) {
#pragma unroll
                for (int j = 0; j < kMaxH; ++j)
                    if (j < n_h) cdf_state[((size_t)slot * n_h + j) * n_grid + g] = acc[k][j];
            }
        }
    }
    if (sown) {
        for (int q = 0; q < kPredScores; ++q) score_state[((size_t)sslot * n_h + js) * kPredScores + q] = sc[q];
    }
}

// Per (window, horizon, e) in caller order, e < n_grid: the CDF at grid[e]; e == n_grid: pit, log score and the moments.  Sums
// the window's chains in chain order, then divides by R = n_chains * nrun.
__global__ void pred_finish_kernel(int n_windows, int n_h, int n_grid, int n_chains, double R, const int* __restrict__ win_slot0,
                                   const double* __restrict__ cshift_w, const double* __restrict__ cdf_state,
                                   const double* __restrict__ score_state, double* __restrict__ cdf, double* __restrict__ pit,
                                   double* __restrict__ log_score, double* __restrict__ moments) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const int ne = n_grid + 1;
    if (i >= (long long)n_windows * n_h * ne) return;
    const int e = (int)(i % ne), j = (int)(i / ne % n_h), w = (int)(i / ne / n_h);
    const size_t wj = (size_t)w * n_h + j;
    const int s0 = win_slot0[w];
    if (e < n_grid) {
        double a = 0.0;
        for (int c = 0; c < n_chains; ++c) a += cdf_state[((size_t)(s0 + c) * n_h + j) * n_grid + e];
        cdf[wj * n_grid + e] = a / R;
        return;
    }
    double S[kPredScores] = {0.0, 0.0, 0.0, 0.0, 0.0};
    for (int c = 0; c < n_chains; ++c)
        for (int q = 0; q < kPredScores; ++q) S[q] += score_state[((size_t)(s0 + c) * n_h + j) * kPredScores + q];
    const double m1 = S[2] / R, m2 = S[3] / R, m3 = S[4] / R;
    const double var = m2 - m1 * m1;
    pit[wj] = S[0] / R;
    log_score[wj] = log(S[1] / R);
    moments[wj * 3 + 0] = cshift_w[w] + m1;
    moments[wj * 3 + 1] = var;
    moments[wj * 3 + 2] = (m3 - 3.0 * m1 * m2 + 2.0 * m1 * m1 * m1) / (var * sqrt(var));
}

}  // namespace hmc
