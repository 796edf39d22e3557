// loo.cuh — PSIS-LOO of every in-sample date (HMCGPU_FLAG_LOO): leave-one-out predictive density, Pareto k̂ and LOO-PIT,
// recomputed at fetch from the parameter draws kept on the device.
//
// plan_run keeps the fields mu, sigma2 and A (the first F' = 2K + K^2 summary fields) of every saved draw with ranked_keep_kernel
// (ranked.cuh), keep[((w*Fs + f)*n_chains + c)*nrun + i], Fs = F' (or the full F of HMCGPU_FLAG_RANKED's buffer when that flag
// is set too, which then holds them already).  hmcgpu_plan_fetch_loo works through batches of dates (pieces of windows) whose
// scratch stays under Tuning::loo_scratch (4 GiB; HMCGPU_LOO_SCRATCH_MB):
//   loo_terms_kernel<R, K>  one lane per draw d (a window's R = n_chains*nrun draws are contiguous in every kept field): the
//                           backward pass from t = N writes the max-free log b_t of the piece's dates to lb; the forward pass from
//                           the uniform start (os_forward_step, the step of onestep_accum_kernel) then writes ell_t,d and F_t,d in
//                           fp64, date-major ell[t][d], so that each date's R values are contiguous;
//   loo_psis_kernel         one block per date: the max log ratio, the (M + 1) largest by radix select on ranked_key (8-bit
//                           digits, then the draw index for ties), the tail sorted by (value, d) in shared memory (bitonic), the
//                           generalised Pareto fit (psis.cuh), truncation, and the per-date reductions in a fixed tree order;
//   loo_finish_kernel       the per-window row.
// Every value of a date is computed by one lane or one block in a fixed order with no atomics on values (the radix histograms
// count with shared-memory atomics, whose totals do not depend on order): a window's outputs are bit-identical however the
// windows are batched, chunked or sharded.  tests/test_loo.py holds the numpy definition it matches.
#pragma once
#include <cuda_runtime.h>
#include <cfloat>
#include "onestep.cuh"     // os_forward_step, OsTrans, os_a_smem / os_warps, kOsMaxK
#include "ranked.cuh"      // ranked_key, key_value, ranked_keep_kernel
#include "psis.cuh"

namespace hmc {

constexpr int kLooThreads = 256;                  // loo_psis_kernel
constexpr int kLooSummary = 6;

// bytes of fetch scratch per date: ell and F in fp64, and K log b values in the plan's precision, per draw
inline size_t loo_date_bytes(long long R_draws, int K, int prec_bytes) { return (size_t)R_draws * (16 + (size_t)K * prec_bytes); }

// A date range [t0, t1) of window w whose terms land at date row `row` of the batch's scratch.
struct LooPiece { int w, t0, t1, row; };

template <typename R, int K>
__global__ void __launch_bounds__(32 * os_warps<R, K>()) loo_terms_kernel(long long Rd, int Fs, const LooPiece* __restrict__ pieces,
                                                                 const R* __restrict__ keep, const int* __restrict__ wT,
                                                                 const int* __restrict__ win_slot0, const long long* __restrict__ ybase,
                                                                 int yld, const R* __restrict__ y, R* __restrict__ lb,
                                                                 double* __restrict__ ell_out, double* __restrict__ F_out) {
    constexpr int W = os_warps<R, K>();
    constexpr bool SM = os_a_smem<R, K>();
    __shared__ R s_A[SM ? W * K * K * 32 : 1];
    const int wp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const LooPiece pc = pieces[blockIdx.y];
    const long long d = ((long long)blockIdx.x * W + wp) * 32 + lane;
    if (d >= Rd) return;
    const int w = pc.w, N = wT[w];
    const R* ys = y + ybase[win_slot0[w]];
    const R* o = keep + (size_t)w * Fs * Rd + d;
    R mu[K], s2[K];
    OsTrans<R, K, SM> A;
    if constexpr (SM) { A.p = s_A + wp * K * K * 32; A.lane = lane; }
    bool bad = false;
#pragma unroll
    for (int s = 0; s < K; ++s) {
        mu[s] = o[(size_t)s * Rd];
        s2[s] = o[(size_t)(K + s) * Rd];
        bad |= !isfinite(mu[s]) || !isfinite(s2[s]);
#pragma unroll
        for (int r = 0; r < K; ++r) {
            A.at(r, s) = o[(size_t)(2 * K + s * K + r) * Rd];
            bad |= !isfinite(A.at(r, s));
        }
    }
    if (bad) {                                   // a harmless model; the outputs are NaN
#pragma unroll
        for (int s = 0; s < K; ++s) {
            mu[s] = R(0); s2[s] = R(1);
#pragma unroll
            for (int r = 0; r < K; ++r) A.at(r, s) = R(1) / R(K);
        }
    }
    Emission<R, K> em;
    em.prepare(mu, s2);
    R isd[K], lnrm[K];
#pragma unroll
    for (int s = 0; s < K; ++s) {
        if constexpr (sizeof(R) == 4) { isd[s] = rsqrtf(s2[s]); lnrm[s] = 0.f; }
        else { isd[s] = em.isd[s]; lnrm[s] = log(em.nrm[s]); }
    }
    // backward: b_N = 1; log b_t,r = log sum_s A[r][s] exp(log phi_s(y_t+1) + log b_t+1,s - m), m dropped (a rescaling per t)
    R* lbp = lb + (size_t)pc.row * K * Rd + d;
    R b[K];
#pragma unroll
    for (int s = 0; s < K; ++s) b[s] = R(0);
    for (int t = N - 1; t >= pc.t0; --t) {
        if (t < N - 1) {
            const R yn = ys[(long long)(t + 1) * yld];
            R u[K], m;
#pragma unroll
            for (int s = 0; s < K; ++s) u[s] = os_log_emission<R, K>(em, lnrm, s, yn) + b[s];
            m = u[0];
#pragma unroll
            for (int s = 1; s < K; ++s) m = fmax(m, u[s]);
#pragma unroll
            for (int s = 0; s < K; ++s) {
                if constexpr (sizeof(R) == 4) u[s] = Real<float>::ex2(u[s] - m);
                else u[s] = exp(u[s] - m);
            }
#pragma unroll
            for (int r = 0; r < K; ++r) {
                R v = A.at(r, 0) * u[0];
#pragma unroll
                for (int s = 1; s < K; ++s) v = fma(A.at(r, s), u[s], v);
                b[r] = os_log<R>(v);
            }
        }
        if (t < pc.t1) {
#pragma unroll
            for (int s = 0; s < K; ++s) lbp[((size_t)(t - pc.t0) * K + s) * Rd] = b[s];
        }
    }
    // forward from the uniform start: the one-step step, then the leave-one-out term with b_t
    R wt[K];
#pragma unroll
    for (int s = 0; s < K; ++s) wt[s] = R(1) / R(K);
    for (int t = 0; t < pc.t1; ++t) {
        R w0[K];
#pragma unroll
        for (int s = 0; s < K; ++s) w0[s] = wt[s];
        R l[K], cdf[K], F1;
        double ell1;
        os_forward_step<R, K>(em, isd, lnrm, ys[(long long)t * yld], wt, A, l, cdf, ell1, F1);
        if (t < pc.t0) continue;
        R num[K], den[K], mn, md;
#pragma unroll
        for (int s = 0; s < K; ++s) {
            const R bs = lbp[((size_t)(t - pc.t0) * K + s) * Rd];
            num[s] = l[s] + bs;                  // log w_t,s phi_s(y_t) b_t,s
            den[s] = os_log<R>(w0[s]) + bs;      // log w_t,s b_t,s
        }
        mn = num[0]; md = den[0];
#pragma unroll
        for (int s = 1; s < K; ++s) { mn = fmax(mn, num[s]); md = fmax(md, den[s]); }
        R sn = R(0), sd = R(0), sf = R(0);
#pragma unroll
        for (int s = 0; s < K; ++s) {
            R en, ed;
            if constexpr (sizeof(R) == 4) { en = Real<float>::ex2(num[s] - mn); ed = Real<float>::ex2(den[s] - md); }
            else { en = exp(num[s] - mn); ed = exp(den[s] - md); }
            sn += en;
            sd += ed;
            sf = fma(ed, cdf[s], sf);
        }
        double ell, F;
        if constexpr (sizeof(R) == 4)
            ell = (((double)mn + (double)Real<float>::lg2(sn)) - ((double)md + (double)Real<float>::lg2(sd))) * 0.6931471805599453;
        else
            ell = (mn + log(sn)) - (md + log(sd));
        F = (double)sf / (double)sd;
        const size_t q = (size_t)(pc.row + t - pc.t0) * Rd + d;
        ell_out[q] = bad ? (double)NAN : ell;
        F_out[q] = bad ? (double)NAN : F;
    }
}

template <typename R>
inline cudaError_t launch_loo_terms(int K, long long Rd, int Fs, int n_pieces, const LooPiece* pieces, const R* keep, const int* wT,
                                    const int* win_slot0, const long long* ybase, int yld, const R* y, R* lb, double* ell,
                                    double* F, cudaStream_t st) {
    // one piece per grid row, in launches of at most 65 535 rows (the limit of gridDim.y)
    for (int p0 = 0; p0 < n_pieces; p0 += 65535) {
        const unsigned np = (unsigned)(n_pieces - p0 < 65535 ? n_pieces - p0 : 65535);
#define HMC_LOO_CASE(KK)                                                                                                       \
        case KK: {                                                                                                             \
            constexpr int W = os_warps<R, KK>();                                                                               \
            const dim3 grid((unsigned)((Rd + 32 * W - 1) / (32 * W)), np);                                                     \
            loo_terms_kernel<R, KK><<<grid, 32 * W, 0, st>>>(Rd, Fs, pieces + p0, keep, wT, win_slot0, ybase, yld, y, lb, ell, F); \
        } break;
        switch (K) {
            HMC_LOO_CASE(2) HMC_LOO_CASE(3) HMC_LOO_CASE(4) HMC_LOO_CASE(5) HMC_LOO_CASE(6) HMC_LOO_CASE(7) HMC_LOO_CASE(8)
            default: return cudaErrorInvalidValue;
        }
#undef HMC_LOO_CASE
        const cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return e;
    }
    return cudaSuccess;
}

// ---------------------------------------------------------------------------------------------------------------- PSIS

// block-wide reduction of one value per thread in a fixed tree (every thread gets the result)
template <typename Op>
__device__ __forceinline__ double loo_block_reduce(double v, double* sh, Op op) {
    const int tid = threadIdx.x;
    __syncthreads();
    sh[tid] = v;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (tid < s) sh[tid] = op(sh[tid], sh[tid + s]);
        __syncthreads();
    }
    return sh[0];
}

// the smallest power of two >= n
__host__ __device__ inline int loo_pow2(int n) { int p = 1; while (p < n) p <<= 1; return p; }

// dynamic shared memory of loo_psis_kernel: the tail's keys (later its values) and draw indices, padded to a power of two
inline size_t loo_psis_smem(long long Rd) {
    const int M = psis_tail_len(Rd);
    return M >= 5 ? (size_t)loo_pow2(M) * (sizeof(unsigned long long) + sizeof(int)) : 0;
}

struct LooTerm { const double* ell; double maxr; };
// the shifted log ratio lw_d = -ell_d - max_d(-ell_d) and its key
__device__ __forceinline__ double loo_lw(const LooTerm& a, int d) { return -a.ell[d] - a.maxr; }

// One block per date of the batch (row j = blockIdx.x of ell / F, date g0 + j of the outputs).
__global__ void __launch_bounds__(kLooThreads) loo_psis_kernel(long long Rd, long long g0, const double* __restrict__ ell_b,
                                                               const double* __restrict__ F_b, double* __restrict__ elpd,
                                                               double* __restrict__ lppd, double* __restrict__ pareto_k,
                                                               double* __restrict__ pit) {
    extern __shared__ unsigned long long s_key[];            // [P] keys, then the tail's x / smoothed values as doubles
    __shared__ double red[kLooThreads];
    __shared__ unsigned hist[256];
    __shared__ unsigned long long s_sel[4];                  // selected key prefix, d prefix, flags
    __shared__ double s_prof[160];                           // gpdfit's profile log-likelihood per grid point (m <= 140)
    __shared__ unsigned s_cnt;
    const int tid = threadIdx.x, nt = blockDim.x;
    const int R = (int)Rd;
    const long long j = blockIdx.x;
    const double* ell = ell_b + (size_t)j * Rd;
    const double* Fd = F_b + (size_t)j * Rd;
    const long long g = g0 + j;
    // max of r = -ell, and NaN
    double mx = -INFINITY, nan = 0.0, mxl = -INFINITY;
    for (int d = tid; d < R; d += nt) {
        const double e = ell[d], f = Fd[d];
        if (isnan(e) || isnan(f)) nan = 1.0;
        mx = fmax(mx, -e);
        mxl = fmax(mxl, e);
    }
    nan = loo_block_reduce(nan, red, [](double a, double b) { return fmax(a, b); });
    if (nan != 0.0) {
        if (tid == 0) { elpd[g] = NAN; lppd[g] = NAN; pareto_k[g] = NAN; pit[g] = NAN; }
        return;
    }
    mx = loo_block_reduce(mx, red, [](double a, double b) { return fmax(a, b); });
    mxl = loo_block_reduce(mxl, red, [](double a, double b) { return fmax(a, b); });
    const LooTerm lt{ell, mx};
    const int M = psis_tail_len(Rd);
    int* s_idx = nullptr;
    double* s_val = reinterpret_cast<double*>(s_key);
    bool smooth = false;
    double k = INFINITY;
    unsigned long long kc = 0;                               // the cutoff draw's (key, d)
    int dc = 0;
    if (M >= 5) {
        const int P = loo_pow2(M);
        s_idx = reinterpret_cast<int*>(s_key + P);
        // radix select of ascending position R - M - 1 in the (key, d) order: 8 digits of the key, then 4 of d
        unsigned long long kp = 0, km = 0;
        unsigned dp = 0, dm = 0;
        unsigned rank = (unsigned)(R - M - 1);
        bool done = false;
        for (int pass = 0; pass < 12 && !done; ++pass) {
            const bool on_key = pass < 8;
            const int shift = on_key ? 56 - 8 * pass : 24 - 8 * (pass - 8);
            for (int b = tid; b < 256; b += nt) hist[b] = 0u;
            __syncthreads();
            for (int d = tid; d < R; d += nt) {
                const unsigned long long key = ranked_key(loo_lw(lt, d));
                if ((key & km) != kp || ((unsigned)d & dm) != dp) continue;
                const unsigned dig = on_key ? (unsigned)(key >> shift) & 255u : ((unsigned)d >> shift) & 255u;
                atomicAdd(&hist[dig], 1u);
            }
            __syncthreads();
            if (tid == 0) {
                unsigned dig = 255, r = rank;
                for (unsigned b = 0; b < 256; ++b) {
                    if (r < hist[b]) { dig = b; break; }
                    r -= hist[b];
                }
                s_sel[0] = dig; s_sel[1] = r; s_sel[2] = hist[dig];
            }
            __syncthreads();
            const unsigned dig = (unsigned)s_sel[0];
            rank = (unsigned)s_sel[1];
            if (on_key) { kp |= (unsigned long long)dig << shift; km |= 255ull << shift; }
            else { dp |= dig << shift; dm |= 255u << shift; }
            if (s_sel[2] == 1u) {                            // one candidate left: read it
                __syncthreads();
                for (int d = tid; d < R; d += nt) {
                    const unsigned long long key = ranked_key(loo_lw(lt, d));
                    if ((key & km) == kp && ((unsigned)d & dm) == dp) { s_sel[0] = key; s_sel[1] = (unsigned)d; }
                }
                __syncthreads();
                kp = s_sel[0]; dp = (unsigned)s_sel[1];
                done = true;
            }
            __syncthreads();
        }
        kc = kp; dc = (int)dp;
        // gather the M draws above the cutoff in the (key, d) order; pad to P with keys that sort last
        if (tid == 0) s_cnt = 0u;
        for (int i = M + tid; i < P; i += nt) { s_key[i] = ~0ull; s_idx[i] = 0x7fffffff; }
        __syncthreads();
        for (int d = tid; d < R; d += nt) {
            const unsigned long long key = ranked_key(loo_lw(lt, d));
            if (key > kc || (key == kc && d > dc)) {
                const unsigned q = atomicAdd(&s_cnt, 1u);
                if (q < (unsigned)M) { s_key[q] = key; s_idx[q] = d; }
            }
        }
        __syncthreads();
        // bitonic sort by (key, d) ascending
        for (int size = 2; size <= P; size <<= 1) {
            for (int stride = size >> 1; stride > 0; stride >>= 1) {
                for (int i = tid; i < P; i += nt) {
                    const int p = i ^ stride;
                    if (p > i) {
                        const bool up = (i & size) == 0;
                        const unsigned long long ka = s_key[i], kb = s_key[p];
                        const int da = s_idx[i], db = s_idx[p];
                        const bool gt = ka > kb || (ka == kb && da > db);
                        if (gt == up) { s_key[i] = kb; s_key[p] = ka; s_idx[i] = db; s_idx[p] = da; }
                    }
                }
                __syncthreads();
            }
        }
        const double lo = key_value(s_key[0]), hi = key_value(s_key[M - 1]), cutoff = key_value(kc);
        __syncthreads();
        if (fabs(hi - lo) >= DBL_EPSILON / 100) {
            smooth = true;
            const double ec = exp(cutoff);
            for (int i = tid; i < M; i += nt) s_val[i] = exp(key_value(s_key[i])) - ec;   // x_i, ascending
            __syncthreads();
            // gpdfit: one warp per grid point, lanes over the tail, a fixed shuffle tree
            const int m = gpd_grid_len(M);
            const double xl = s_val[M - 1], xstar = s_val[(int)floor(M / 4.0 + 0.5) - 1];
            const int lane = tid & 31, wp = tid >> 5, nw = nt >> 5;
            for (int q = wp; q < m; q += nw) {
                const double th = gpd_theta(q + 1, m, xl, xstar);
                double s = 0.0;
                for (int i = lane; i < M; i += 32) s += log1p(-th * s_val[i]);
                for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
                if (lane == 0) s_prof[q] = gpd_profile(th, s / M, M);
            }
            __syncthreads();
            if (tid == 0) {
                double lm = -INFINITY;
                for (int q = 0; q < m; ++q) lm = fmax(lm, s_prof[q]);
                double sw = 0.0, swt = 0.0;
                for (int q = 0; q < m; ++q) {
                    const double e = exp(s_prof[q] - lm);
                    sw += e;
                    swt += gpd_theta(q + 1, m, xl, xstar) * e;
                }
                red[0] = swt / sw;
            }
            __syncthreads();
            const double theta_hat = red[0];
            double s = 0.0;
            for (int i = tid; i < M; i += nt) s += log1p(-theta_hat * s_val[i]);
            s = loo_block_reduce(s, red, [](double a, double b) { return a + b; });
            double sigma;
            gpd_finish(theta_hat, s / M, M, &k, &sigma);
            __syncthreads();
            if (isfinite(k)) {
                for (int i = tid; i < M; i += nt) s_val[i] = log(gpd_quantile((i + 0.5) / M, k, sigma) + ec);
            } else {
                for (int i = tid; i < M; i += nt) s_val[i] = loo_lw(lt, s_idx[i]);   // (s_key now holds x: the draw's own lw)
            }
            __syncthreads();
        }
    }
    // the truncated log weights: the tail's (smoothed) values from shared memory, every other draw its own lw_d
    auto in_tail = [&](int d) -> bool {
        if (!smooth) return false;
        const unsigned long long key = ranked_key(loo_lw(lt, d));
        return key > kc || (key == kc && d > dc);
    };
    // pass 1: the max of lw_d + ell_d; pass 2: sum exp(lw), sum exp(lw + ell - max), sum exp(lw) F, sum exp(ell - max ell)
    double m2 = -INFINITY;
    for (int d = tid; d < R; d += nt)
        if (!in_tail(d)) m2 = fmax(m2, fmin(loo_lw(lt, d), 0.0) + ell[d]);
    if (smooth)
        for (int i = tid; i < M; i += nt) m2 = fmax(m2, fmin(s_val[i], 0.0) + ell[s_idx[i]]);
    m2 = loo_block_reduce(m2, red, [](double a, double b) { return fmax(a, b); });
    double s0 = 0.0, s1 = 0.0, sf = 0.0, sl = 0.0;
    for (int d = tid; d < R; d += nt) {
        sl += exp(ell[d] - mxl);
        if (in_tail(d)) continue;
        const double lw = fmin(loo_lw(lt, d), 0.0), e = exp(lw);
        s0 += e;
        s1 += exp(lw + ell[d] - m2);
        sf += e * Fd[d];
    }
    if (smooth) {
        for (int i = tid; i < M; i += nt) {
            const int d = s_idx[i];
            const double lw = fmin(s_val[i], 0.0), e = exp(lw);
            s0 += e;
            s1 += exp(lw + ell[d] - m2);
            sf += e * Fd[d];
        }
    }
    auto add = [](double a, double b) { return a + b; };
    s0 = loo_block_reduce(s0, red, add);
    s1 = loo_block_reduce(s1, red, add);
    sf = loo_block_reduce(sf, red, add);
    sl = loo_block_reduce(sl, red, add);
    if (tid == 0) {
        elpd[g] = m2 + log(s1) - log(s0);
        lppd[g] = mxl + log(sl / (double)Rd);
        pareto_k[g] = k;
        pit[g] = sf / s0;
    }
}

// One thread per window: summary[w*6 + 0..5] = elpd_loo, se, p_loo, lppd, max k̂, #(k̂ > threshold), t ascending; NaN everywhere
// when a date is NaN.
__global__ void loo_finish_kernel(int n_windows, int K, long long Rd, const int* __restrict__ wT, const long long* __restrict__ win_pib_off,
                                  const double* __restrict__ elpd, const double* __restrict__ lppd, const double* __restrict__ pareto_k,
                                  double* __restrict__ summary) {
    const int w = blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= n_windows) return;
    const int N = wT[w];
    const long long off = win_pib_off[w] / K;
    const double thr = psis_k_threshold(Rd);
    double se = 0.0, sl = 0.0, kmax = -INFINITY, nbad = 0.0;
    bool nan = false;
    for (int t = 0; t < N; ++t) {
        const double e = elpd[off + t], l = lppd[off + t], kk = pareto_k[off + t];
        nan |= isnan(e) || isnan(l) || isnan(kk);
        se += e;
        sl += l;
        kmax = fmax(kmax, kk);
        nbad += kk > thr ? 1.0 : 0.0;
    }
    const double me = se / N;
    double v = 0.0, pl = 0.0;
    for (int t = 0; t < N; ++t) {
        const double e = elpd[off + t] - me;
        v += e * e;
        pl += lppd[off + t] - elpd[off + t];
    }
    double* out = summary + (size_t)w * kLooSummary;
    out[0] = nan ? (double)NAN : se;
    out[1] = nan ? (double)NAN : sqrt(N * (v / (N - 1)));
    out[2] = nan ? (double)NAN : pl;
    out[3] = nan ? (double)NAN : sl;
    out[4] = nan ? (double)NAN : kmax;
    out[5] = nan ? (double)NAN : nbad;
}

}  // namespace hmc
