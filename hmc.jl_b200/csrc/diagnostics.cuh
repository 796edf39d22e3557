// diagnostics.cuh — split-R̂ and effective sample size per (window, field) (HMCGPU_FLAG_DIAGNOSTICS), streamed over the saved
// draws as they pass through the per-chunk buffer out[(f*chunk + i)*n_slots + slot].
//
// Every chain's nrun saved draws form two sequences of n = nrun/2 draws (the middle draw of an odd nrun is dropped).  One
// sequence at a time is accumulated per (slot, field), shifted by its first value x_0 (y_t = x_t - x_0, so that the centred
// sums below do not cancel; DESIGN.md section 5 records the same problem for sigma^2):
//   S1 = sum_t y_t,  P_l = sum_{t<n-l} y_t y_{t+l} (l = 0..63),  the first 64 raw values (head) and the last 64 (ring).
// When a sequence ends, diag_half_kernel turns these into the sequence's mean, variance and centred lag sums
//   G_l = sum_{t<n-l} (y_t - ybar)(y_{t+l} - ybar) = P_l - ybar (sum_{t<n-l} y_t + sum_{t>=l} y_t) + (n-l) ybar^2,
// the two partial sums coming from S1 minus the tail (ring) or the head, and adds G_l over the window's chains in chain order.
// diag_finish_kernel then computes R̂ and the ESS (Geyer's initial monotone sequence, lags capped at 63) per (window, field).
//
// Every sum runs in draw order or chain order, with no atomics: a window's result does not depend on the chunk size, the
// batch or the sharding (the per-chain draws being equal).  tests/test_diagnostics.py holds the numpy definition it matches.
#pragma once
#include <cuda_runtime.h>

namespace hmc {

constexpr int kDiagLags = 64;   // autocovariance lags 0..63: 32 Geyer pairs

// Streaming state of the current sequence of every (slot, field); sf = f * n_slots + slot, n_sf = F * n_slots.
template <typename R>
struct DiagState {
    double* P;      // [sf][64] lag-product sums P_l
    double* S1;     // [sf]
    R* head;        // [64][sf] raw value t < 64 at head[t * n_sf + sf]; head[sf] is the shift x_0
    R* ring;        // [64][sf] raw value t of the last 64 at ring[(t & 63) * n_sf + sf]
    long long n_sf;
};

// Adds draws [i_lo, i_lo + n_i) of a chunk buffer — sequence positions t0 .. t0 + n_i - 1 — to the state of 32 consecutive
// slots x one field (block (32, 32), grid (n_slots / 32, fields)).  The block stages the draws, shifted, in a circular buffer
// of 128 positions per slot; then warp w walks slot w's draws in order with lane l accumulating lags l and l + 32.
// t0 == 0 starts a new sequence (the state left by the previous one is ignored).
template <typename R>
__global__ void __launch_bounds__(1024) diag_accum_kernel(int n_slots, int chunk, int i_lo, int n_i, long long t0,
                                                          const R* __restrict__ out, DiagState<R> st) {
    __shared__ double sy[32][129];            // (odd row length: the loader's column writes spread over the banks)
    __shared__ double cs[32];
    const int x = threadIdx.x, w = threadIdx.y, f = blockIdx.y;
    const int slot0 = blockIdx.x * 32;
    const size_t sfx = (size_t)f * n_slots + slot0 + x;     // loader role: slot x
    const size_t sfw = (size_t)f * n_slots + slot0 + w;     // walker role: slot w
    const R* src = out + ((size_t)f * chunk + i_lo) * n_slots + slot0 + x;
    if (w == 0) cs[x] = t0 == 0 ? (double)src[0] : (double)st.head[sfx];
    __syncthreads();
    const double cx = cs[x];
    // the 64 positions before t0: the previous call's ring, or zeros (= no contribution) before the start of the sequence
    for (int k = w; k < 64; k += 32) {
        const long long t = t0 - 64 + k;
        sy[x][t & 127] = t >= 0 ? (double)st.ring[(size_t)(t & 63) * st.n_sf + sfx] - cx : 0.0;
    }
    double p0 = 0.0, p1 = 0.0, s1 = 0.0;
    if (t0 > 0) {
        p0 = st.P[sfw * kDiagLags + x];
        p1 = st.P[sfw * kDiagLags + 32 + x];
        if (w == 0) s1 = st.S1[sfx];
    }
    const double* col = sy[w];
    const long long t_end = t0 + n_i;
    for (int r0 = 0; r0 < n_i; r0 += 64) {
        const int m = min(64, n_i - r0);
        __syncthreads();                        // the previous tile's walks are done with the positions this tile overwrites
        for (int r = w; r < m; r += 32) {
            const long long t = t0 + r0 + r;
            const R v = src[(size_t)(r0 + r) * n_slots];
            sy[x][t & 127] = (double)v - cx;
            if (t < 64) st.head[(size_t)t * st.n_sf + sfx] = v;
            if (t >= t_end - 64) st.ring[(size_t)(t & 63) * st.n_sf + sfx] = v;
        }
        __syncthreads();
        const unsigned tb = (unsigned)(t0 + r0);
        if (w == 0)
            for (int r = 0; r < m; ++r) s1 += sy[x][(tb + r) & 127];
        for (int r = 0; r < m; ++r) {
            const unsigned t = tb + r;
            const double y = col[t & 127];
            p0 = __fma_rn(y, col[(t - x) & 127], p0);
            p1 = __fma_rn(y, col[(t - x - 32) & 127], p1);
        }
    }
    st.P[sfw * kDiagLags + x] = p0;
    st.P[sfw * kDiagLags + 32 + x] = p1;
    if (w == 0) st.S1[sfx] = s1;
}

// End of a sequence of n draws (half 0 or 1): per (window, field) (grid (n_windows, fields), 64 threads = lags), the
// sequence mean and variance of every chain into seq_mean / seq_var [(w*F + f)*M + half*n_chains + chain] (M = 2 n_chains),
// and sum over the chains, in chain order, of the centred lag sums G_l into gsum [(w*F + f)*64 + l] (set by half 0,
// added to by half 1).
template <typename R>
__global__ void __launch_bounds__(kDiagLags) diag_half_kernel(int F, int n_slots, int n_chains, long long n, int half,
                                                              const int* __restrict__ win_slot0, DiagState<R> st,
                                                              double* __restrict__ seq_mean, double* __restrict__ seq_var,
                                                              double* __restrict__ gsum) {
    __shared__ double hy[kDiagLags], ty[kDiagLags];
    const int wnd = blockIdx.x, f = blockIdx.y, l = threadIdx.x;
    const int M = 2 * n_chains;
    const size_t wf = (size_t)wnd * F + f;
    const double dn = (double)n;
    double acc = 0.0;
    for (int c = 0; c < n_chains; ++c) {
        const size_t sf = (size_t)f * n_slots + win_slot0[wnd] + c;
        const double c0 = (double)st.head[sf];
        const double S1 = st.S1[sf];
        __syncthreads();                        // the previous chain's hy / ty have been read
        {
            const long long t = n - kDiagLags + l;   // tail value t (if it exists)
            hy[l] = l < n ? (double)st.head[(size_t)l * st.n_sf + sf] - c0 : 0.0;
            ty[l] = t >= 0 ? (double)st.ring[(size_t)(t & 63) * st.n_sf + sf] - c0 : 0.0;
        }
        __syncthreads();
        const double ybar = S1 / dn;
        const double P = st.P[sf * kDiagLags + l];
        if (l == 0) {
            seq_mean[wf * M + half * n_chains + c] = c0 + ybar;
            seq_var[wf * M + half * n_chains + c] = (P - S1 * ybar) / (dn - 1.0);
        }
        if (l < n) {
            double hs = 0.0, ts = 0.0;          // sum_{t<l} y_t and sum_{t>=n-l} y_t
            for (int k = 0; k < l; ++k) hs += hy[k];
            for (int k = kDiagLags - l; k < kDiagLags; ++k) ts += ty[k];
            acc += P - ybar * ((S1 - ts) + (S1 - hs)) + (dn - (double)l) * ybar * ybar;
        }
    }
    gsum[wf * kDiagLags + l] = half == 0 ? acc : gsum[wf * kDiagLags + l] + acc;
}

// Per (window, field) in caller order: split-R̂, ESS and the last lag of the autocorrelation sum (ess_lag).  NaN (ess_lag -1)
// for a field with a non-finite draw, no within-sequence variance (W = 0), or the log-likelihood field without its flag.
__global__ void diag_finish_kernel(long long n_elems, int F, int n_chains, long long n, int has_loglik,
                                   const double* __restrict__ seq_mean, const double* __restrict__ seq_var,
                                   const double* __restrict__ gsum, double* __restrict__ rhat, double* __restrict__ ess,
                                   int* __restrict__ ess_lag) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n_elems) return;
    const int M = 2 * n_chains;
    const double* mu = seq_mean + (size_t)i * M;
    const double* s2 = seq_var + (size_t)i * M;
    const double* g = gsum + (size_t)i * kDiagLags;
    bool ok = has_loglik || (int)(i % F) != F - 1;
    double W = 0.0, mbar = 0.0;
    for (int m = 0; m < M; ++m) {
        ok = ok && isfinite(mu[m]) && isfinite(s2[m]);
        W += s2[m];
        mbar += mu[m];
    }
    for (int l = 0; l < kDiagLags; ++l) ok = ok && isfinite(g[l]);
    W /= M;
    mbar /= M;
    if (!ok || !(W > 0.0)) { rhat[i] = NAN; ess[i] = NAN; ess_lag[i] = -1; return; }
    double Bn = 0.0;                            // B / n: variance of the sequence means
    for (int m = 0; m < M; ++m) { const double d = mu[m] - mbar; Bn += d * d; }
    Bn /= (M - 1);
    const double dn = (double)n, Mn = (double)M * dn;
    const double varp = (dn - 1.0) / dn * W + Bn;
    rhat[i] = sqrt(varp / W);
    auto rho = [&](int l) { return l == 0 ? 1.0 : 1.0 - (W - g[l] / Mn) / varp; };
    const long long cap = n - 1 < kDiagLags - 1 ? n - 1 : kDiagLags - 1;   // last lag that may be summed, made odd below
    double sum = 0.0, prev = INFINITY;
    int last = -1;
    for (int k = 0; 2 * k + 1 <= cap; ++k) {
        double Pk = rho(2 * k) + rho(2 * k + 1);
        if (!(Pk > 0.0)) break;
        Pk = fmin(Pk, prev);
        prev = Pk;
        sum += Pk;
        last = 2 * k + 1;
    }
    const double tau = fmax(-1.0 + 2.0 * sum, 1.0 / log10(Mn));
    ess[i] = Mn / tau;
    ess_lag[i] = last;
}

}  // namespace hmc
