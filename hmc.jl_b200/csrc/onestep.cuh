// onestep.cuh — one-step-ahead posterior predictive scores of every in-sample date (HMCGPU_FLAG_ONESTEP), streamed over the
// saved draws as they pass through the per-chunk buffer out[(f*chunk + i)*n_slots + slot].
//
// Each saved draw d of a window (mu_s, sigma2_s, A[r][s]) is run through the forward filter from the uniform initial
// distribution over the window's own observations (the rows the chain saw, read from the plan's time-major series yr), in the
// log domain and in the plan's precision:
//   l_t,s = log w_t,s + log phi(y_t; mu_s, sigma2_s),   ell_t,d = log sum_s exp(l_t,s),   F_t,d = sum_s w_t,s Phi(z_t,s),
//   w_t+1,s = sum_r exp(l_t,r - ell_t,d) A[r][s],        w_1,s = 1/K.
// Per (slot, date) a running fp64 state keeps, in draw order:
//   [0] sum_d F_t,d                  (PIT)
//   [1] max_d ell_t,d, [2] sum_d exp(ell_t,d - max)      (log-sum-exp)
//   [3] mean_d ell_t,d, [4] sum_d (ell_t,d - mean)^2     (Welford)
// stored component-major: state[q * n_state + base + t] with base = (date offset of the window) * n_chains + chain * N_w.
//
// onestep_accum_kernel: one warp per slot, lane = draw, tiles of 32 draws taken in draw order.  Every lane filters its draw over
// 32 dates, the 32 x 32 (ell, F) tile is transposed through shared memory, and lane j then folds the tile's draws, in draw
// order, into the state of date t0 + j.  The fold of a (slot, date) is therefore one sequential chain of fp64 operations over
// the chain's draws, whatever the chunking.  onestep_finish_kernel combines a window's chains in chain order (log-sum-exp
// pairs, Chan's pairwise update of (n, mean, M2), the PIT sums) and forms the window's WAIC row with t ascending.  No atomics:
// a window's outputs are bit-identical however the windows are batched, chunked or sharded.  tests/test_onestep.py holds the
// numpy definition it matches.
#pragma once
#include <cuda_runtime.h>
#include "hmm_device.cuh"     // Emission, Real

namespace hmc {

constexpr int kOsState = 5;          // running values per (slot, date), see above
constexpr int kOsMaxK = 8;

// fp64 at K = 8 holds A in shared memory (in registers ptxas spills there), one warp per block to keep the static shared memory
// under 48 KB; every other case holds A in registers, two warps (slots) per block.
template <typename R, int K> __host__ __device__ constexpr bool os_a_smem() { return sizeof(R) == 8 && K == kOsMaxK; }
template <typename R, int K> __host__ __device__ constexpr int os_warps() { return os_a_smem<R, K>() ? 1 : 2; }

// the lane's transition matrix A[r][s]
template <typename R, int K, bool SMEM> struct OsTrans {
    R a[K][K];
    __device__ __forceinline__ R& at(int r, int s) { return a[r][s]; }
};
template <typename R, int K> struct OsTrans<R, K, true> {
    R* p;                                // [K*K][32], lane-minor
    int lane;
    __device__ __forceinline__ R& at(int r, int s) { return p[(r * K + s) * 32 + lane]; }
};

// log w in the log base of the plan's precision (log2 in fp32, as the fp32 emission; natural in fp64)
template <typename R> __device__ __forceinline__ R os_log(R x) {
    if constexpr (sizeof(R) == 4) return Real<float>::lg2(x);
    else return log(x);
}

// log phi(y; mu_s, sigma2_s) in that base
template <typename R, int K>
__device__ __forceinline__ R os_log_emission(const Emission<R, K>& em, const R (&lnrm)[K], int s, R y) {
    if constexpr (sizeof(R) == 4) { const float d = y - em.mu[s]; return fmaf(d * d, em.q[s], em.c[s]); }
    else { const double z = (y - em.mu[s]) * em.isd[s]; return lnrm[s] - 0.5 * (z * z); }
}

// One step of the forward filter at y_t from the predictive weights wt = w_t (the step of onestep_accum_kernel, shared with
// loo_terms_kernel): l[s] = log w_t,s + log phi_s(y_t) in the precision's log base, cdf[s] = Phi(z_t,s),
// ell = log p(y_t | y_1..t-1) (natural log, fp64), F = sum_s w_t,s cdf[s]; then wt <- w_t+1 = alpha_t A.
template <typename R, int K, typename Trans>
__device__ __forceinline__ void os_forward_step(const Emission<R, K>& em, const R (&isd)[K], const R (&lnrm)[K], R yt, R (&wt)[K],
                                                Trans& A, R (&l)[K], R (&cdf)[K], double& ell, R& F) {
    R a[K], mx;
    F = R(0);
    if constexpr (sizeof(R) == 4) {                  // log2 domain, as the fp32 emission
#pragma unroll
        for (int s = 0; s < K; ++s) {
            const float d = yt - em.mu[s];
            l[s] = Real<float>::lg2(wt[s]) + fmaf(d * d, em.q[s], em.c[s]);
            cdf[s] = normcdff(d * isd[s]);
            F = fmaf(wt[s], cdf[s], F);
        }
        mx = l[0];
#pragma unroll
        for (int s = 1; s < K; ++s) mx = fmaxf(mx, l[s]);
        float sum = 0.f;
#pragma unroll
        for (int s = 0; s < K; ++s) { a[s] = Real<float>::ex2(l[s] - mx); sum += a[s]; }
        ell = ((double)mx + (double)Real<float>::lg2(sum)) * 0.6931471805599453;
        const float inv = Real<float>::rcp(sum);
#pragma unroll
        for (int s = 0; s < K; ++s) a[s] *= inv;
    } else {
#pragma unroll
        for (int s = 0; s < K; ++s) {
            const double z = (yt - em.mu[s]) * isd[s];
            l[s] = log(wt[s]) + lnrm[s] - 0.5 * (z * z);
            cdf[s] = normcdf(z);
            F = fma(wt[s], cdf[s], F);
        }
        mx = l[0];
#pragma unroll
        for (int s = 1; s < K; ++s) mx = fmax(mx, l[s]);
        double sum = 0.0;
#pragma unroll
        for (int s = 0; s < K; ++s) { a[s] = exp(l[s] - mx); sum += a[s]; }
        ell = mx + log(sum);
#pragma unroll
        for (int s = 0; s < K; ++s) a[s] /= sum;
    }
    // a holds the filtered probabilities alpha_t; predict the next date's weights
#pragma unroll
    for (int s = 0; s < K; ++s) {
        R v = a[0] * A.at(0, s);
#pragma unroll
        for (int r = 1; r < K; ++r) v = fma(a[r], A.at(r, s), v);
        wt[s] = v;
    }
}

// Adds draws [0, n_i) of a chunk (draws d0 .. d0 + n_i - 1 of every chain) to the running state.  d0 == 0 starts from the empty
// state (first chunk of a run).
template <typename R, int K>
__global__ void __launch_bounds__(32 * os_warps<R, K>()) onestep_accum_kernel(int n_slots, int chunk, int n_i, long long d0, int n_chains,
                                                                    const int* __restrict__ slot_win, const int* __restrict__ slot_chain,
                                                                    const int* __restrict__ wT, const long long* __restrict__ win_pib_off,
                                                                    const long long* __restrict__ ybase, int yld, const R* __restrict__ y,
                                                                    const R* __restrict__ out, double* __restrict__ state, long long n_state) {
    constexpr int W = os_warps<R, K>();
    constexpr bool SM = os_a_smem<R, K>();
    __shared__ double s_ell[W][32][33];
    __shared__ double s_F[W][32][33];
    __shared__ R s_A[SM ? W * K * K * 32 : 1];
    const int wp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int slot = blockIdx.x * W + wp;
    if (slot >= n_slots) return;
    const int w = slot_win[slot];
    if (w < 0) return;                                       // padding slot
    const int N = wT[w];
    const long long base = win_pib_off[w] / K * n_chains + (long long)slot_chain[slot] * N;
    const R* ys = y + ybase[slot];
    double* st = state + base;
    const size_t cs = (size_t)chunk * n_slots;
    double (*tl)[33] = s_ell[wp];
    double (*tF)[33] = s_F[wp];

    for (int i0 = 0; i0 < n_i; i0 += 32) {
        const int m = min(32, n_i - i0);
        // this lane's draw (lanes past the tile run a harmless uniform model whose results are never folded)
        R mu[K], s2[K];
        OsTrans<R, K, SM> A;
        if constexpr (SM) { A.p = s_A + wp * K * K * 32; A.lane = lane; }
        bool bad = false;
        const R* o = out + (size_t)(i0 + min(lane, m - 1)) * n_slots + slot;
#pragma unroll
        for (int s = 0; s < K; ++s) {
            mu[s] = o[(size_t)s * cs];
            s2[s] = o[(size_t)(K + s) * cs];
            bad |= !isfinite(mu[s]) || !isfinite(s2[s]);
#pragma unroll
            for (int r = 0; r < K; ++r) {
                A.at(r, s) = o[(size_t)(2 * K + s * K + r) * cs];
                bad |= !isfinite(A.at(r, s));
            }
        }
        if (bad) {
#pragma unroll
            for (int s = 0; s < K; ++s) {
                mu[s] = R(0); s2[s] = R(1);
#pragma unroll
                for (int r = 0; r < K; ++r) A.at(r, s) = R(1) / R(K);
            }
        }
        Emission<R, K> em;
        em.prepare(mu, s2);
        R isd[K], lnrm[K];                                   // 1 / sd; log normaliser (fp64 only: fp32 reads em.c)
#pragma unroll
        for (int s = 0; s < K; ++s) {
            if constexpr (sizeof(R) == 4) { isd[s] = rsqrtf(s2[s]); lnrm[s] = 0.f; }
            else { isd[s] = em.isd[s]; lnrm[s] = log(em.nrm[s]); }
        }
        R wt[K];
#pragma unroll
        for (int s = 0; s < K; ++s) wt[s] = R(1) / R(K);

        for (int t0 = 0; t0 < N; t0 += 32) {
            const int nt = min(32, N - t0);
            const R yl = (t0 + lane < N) ? ys[(long long)(t0 + lane) * yld] : R(0);
            for (int tt = 0; tt < nt; ++tt) {
                const R yt = __shfl_sync(0xffffffffu, yl, tt);
                R l[K], cdf[K], F;
                double ell;
                os_forward_step<R, K>(em, isd, lnrm, yt, wt, A, l, cdf, ell, F);
                tl[lane][tt] = bad ? (double)NAN : ell;
                tF[lane][tt] = bad ? (double)NAN : (double)F;
            }
            __syncwarp();
            if (lane < nt) {
                const long long t = t0 + lane;
                double pit, mx, sc, mean, m2;
                if (d0 == 0 && i0 == 0) { pit = 0.0; mx = -INFINITY; sc = 0.0; mean = 0.0; m2 = 0.0; }
                else { pit = st[t]; mx = st[n_state + t]; sc = st[2 * n_state + t]; mean = st[3 * n_state + t]; m2 = st[4 * n_state + t]; }
                for (int i = 0; i < m; ++i) {
                    const double x = tl[i][lane], f = tF[i][lane];
                    if (isnan(x) || isnan(f)) { pit = mx = sc = mean = m2 = NAN; continue; }
                    pit += f;
                    if (x > mx) { sc = sc * exp(mx - x) + 1.0; mx = x; }
                    else sc += exp(x - mx);
                    const double n = (double)(d0 + i0 + i + 1);
                    const double dl = x - mean;
                    mean += dl / n;
                    m2 += dl * (x - mean);
                }
                st[t] = pit; st[n_state + t] = mx; st[2 * n_state + t] = sc; st[3 * n_state + t] = mean; st[4 * n_state + t] = m2;
            }
            __syncwarp();
        }
    }
}

template <typename R>
inline cudaError_t launch_onestep_accum(int K, int n_slots, int chunk, int n_i, long long d0, int n_chains, const int* slot_win,
                                        const int* slot_chain, const int* wT, const long long* win_pib_off, const long long* ybase,
                                        int yld, const R* y, const R* out, double* state, long long n_state, cudaStream_t st) {
#define HMC_OS_CASE(KK)                                                                                                       \
    case KK: {                                                                                                                \
        constexpr int W = os_warps<R, KK>();                                                                                  \
        onestep_accum_kernel<R, KK><<<(unsigned)((n_slots + W - 1) / W), 32 * W, 0, st>>>(                                    \
            n_slots, chunk, n_i, d0, n_chains, slot_win, slot_chain, wT, win_pib_off, ybase, yld, y, out, state, n_state);    \
    } break;
    switch (K) {
        HMC_OS_CASE(2) HMC_OS_CASE(3) HMC_OS_CASE(4) HMC_OS_CASE(5) HMC_OS_CASE(6) HMC_OS_CASE(7) HMC_OS_CASE(8)
        default: return cudaErrorInvalidValue;
    }
#undef HMC_OS_CASE
    return cudaGetLastError();
}

// One block per window (caller order).  Per date t: the window's chains summed in chain order; then thread 0 forms
// waic[w] = {lppd, p_waic, elpd_waic, se} with t ascending.  pit / lpd / lpd_var are per date, windows concatenated at
// win_pib_off[w] / K.
__global__ void onestep_finish_kernel(int K, int n_chains, long long nrun, const int* __restrict__ wT,
                                      const long long* __restrict__ win_pib_off, const double* __restrict__ state, long long n_state,
                                      double* __restrict__ pit, double* __restrict__ lpd, double* __restrict__ lpd_var,
                                      double* __restrict__ waic) {
    const int w = blockIdx.x;
    const int N = wT[w];
    const long long off = win_pib_off[w] / K;
    const double R = (double)n_chains * (double)nrun, nb = (double)nrun;
    for (int t = threadIdx.x; t < N; t += blockDim.x) {
        double sf = 0.0, mx = -INFINITY;
        bool nan = false;
        for (int c = 0; c < n_chains; ++c) {
            const long long i = off * n_chains + (long long)c * N + t;
            sf += state[i];
            const double m = state[n_state + i];
            nan |= isnan(m);
            mx = fmax(mx, m);
        }
        double sc = 0.0, na = 0.0, mean = 0.0, m2 = 0.0;
        for (int c = 0; c < n_chains; ++c) {
            const long long i = off * n_chains + (long long)c * N + t;
            sc += state[2 * n_state + i] * exp(state[n_state + i] - mx);
            const double n = na + nb, d = state[3 * n_state + i] - mean;
            mean += d * (nb / n);
            m2 += state[4 * n_state + i] + d * d * (na * nb / n);
            na = n;
        }
        pit[off + t] = nan ? (double)NAN : sf / R;
        lpd[off + t] = nan ? (double)NAN : mx + log(sc / R);
        lpd_var[off + t] = nan ? (double)NAN : m2 / (R - 1.0);
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        double lppd = 0.0, pw = 0.0;
        for (int t = 0; t < N; ++t) { lppd += lpd[off + t]; pw += lpd_var[off + t]; }
        const double me = (lppd - pw) / N;
        double v = 0.0;
        for (int t = 0; t < N; ++t) { const double e = lpd[off + t] - lpd_var[off + t] - me; v += e * e; }
        waic[(size_t)w * 4 + 0] = lppd;
        waic[(size_t)w * 4 + 1] = pw;
        waic[(size_t)w * 4 + 2] = lppd - pw;
        waic[(size_t)w * 4 + 3] = sqrt(N * (v / (N - 1)));
    }
}

}  // namespace hmc
