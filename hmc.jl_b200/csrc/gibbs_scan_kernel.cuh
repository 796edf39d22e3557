// gibbs_scan_kernel.cuh — the Gibbs sweep for NARROW batches (a few thousand chains or fewer): ONE WARP PER CHAIN,
// parallel in time.  This is the regime of the reference itself (one chain per end date, code/run_hmm.jl:119): with a
// thread per chain the GPU holds a few hundred serial chains and every sweep costs T dependent steps; here the 32 lanes
// of a warp split the window into contiguous chunks of C = ceil(T/32) steps and both recursions become scans:
//
//   forward filter (forwardupdate_P!, src/Hmc.jl:371-440): pif_t ∝ pif_{t-1} · (A diag(e_t)).  Phase 1: every lane
//   multiplies the K x K matrices of its chunk (renormalised each step).  Phase 2: Kogge-Stone scan of the 32 chunk
//   products with warp shuffles gives each lane the filtered vector entering its chunk.  Phase 3: the lane runs the
//   ordinary recursion over its chunk (same forward_step as the other kernels, so normalisers / log-likelihood are
//   the usual ones) and stores the rows in shared memory.
//
//   backward sampling (update_X!, :459-484): X_t = f_t(X_{t+1}) where f_t is the K -> K map "categorical draw from
//   pif[t,:]·A[:,x] with this step's uniform".  Phase 1: every lane walks its chunk for all K possible entering states
//   at once (one walk after they have coalesced), recording the paths, which gives the chunk's composite map.  Phase 2:
//   suffix scan of the maps (4-bit packed, function composition).  Phase 3: each lane now knows the state entering its
//   chunk from above, decodes the recorded path of that state (chunks longer than 32 steps are walked again) and
//   accumulates the next sweep's sufficient statistics (:254-258, :291-294, :362-365); warp reductions pool them.
//
// Same Philox streams, same draw order and the same buffers as the thread-per-chain kernel (gibbs_kernel.cuh): the two
// are interchangeable behind the plan and the fp64 chain follows the oracle's chain (the scans only change the
// association of the products that bring the filtered vector to a chunk boundary).  K <= 4; plain sweep and the signals
// tier (SIG: signal mask, kappa-weighted statistics, pi_row_back — estimatesignals! runs 100 copies x ONE chain); no
// smoothed-mean accumulators.
#pragma once
#include "lane_draws.cuh"
#include "plan_policy.cuh"    // kScanThreads, scan_max_T

namespace hmc {

// per-warp shared memory: pif rows [T][K], uniforms [T], A by columns [K][4]
template <typename R, int K> __host__ __device__ constexpr size_t scan_warp_bytes(int max_T) {
    return (sizeof(R) * ((size_t)max_T * K + (size_t)max_T + 4 * K) + 15) / 16 * 16;
}

template <typename R, int K, bool LOGLIK, bool SIG = false>
struct ScanWarp {
    static constexpr unsigned kFull = 0xffffffffu;

    // any positive common factor will do (only the direction of the products is used): row sums in parallel, approx rcp
    static __device__ __forceinline__ void normalise(R (&P)[K][K]) {
        R rs[K];
#pragma unroll
        for (int i = 0; i < K; ++i) {
            rs[i] = P[i][0];
#pragma unroll
            for (int j = 1; j < K; ++j) rs[i] += P[i][j];
        }
        R s = rs[0];
#pragma unroll
        for (int i = 1; i < K; ++i) s += rs[i];
        const R inv = Real<R>::rcp(s);
#pragma unroll
        for (int i = 0; i < K; ++i)
#pragma unroll
            for (int j = 0; j < K; ++j) P[i][j] *= inv;
    }
    // C = L · Rm
    static __device__ __forceinline__ void matmul(const R (&L)[K][K], const R (&Rm)[K][K], R (&C)[K][K]) {
#pragma unroll
        for (int i = 0; i < K; ++i)
#pragma unroll
            for (int j = 0; j < K; ++j) {
                R acc = L[i][0] * Rm[0][j];
#pragma unroll
                for (int r = 1; r < K; ++r) acc = fma(L[i][r], Rm[r][j], acc);
                C[i][j] = acc;
            }
    }
    static __device__ __forceinline__ R wsum(R v) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
        return v;
    }
    static __device__ __forceinline__ unsigned long long wsum64(unsigned long long v) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
        return v;
    }
    // (F ∘ Q)[h] = F[Q[h]] on 4-bit packed maps
    static __device__ __forceinline__ unsigned compose(unsigned F, unsigned Q) {
        unsigned r = 0;
#pragma unroll
        for (int h = 0; h < K; ++h) r |= ((F >> (4 * ((Q >> (4 * h)) & 15u))) & 15u) << (4 * h);
        return r;
    }

    // Conjugate draws with the K*K + 2K gamma variates spread over the lanes (each has its own Philox purpose stream, so
    // they are independent): lane i < K draws the gamma of sigma2_i, lane K+i that of rho_i, lane 2K + i*K + j that of
    // A[i][j].  The posterior of each state is state_posterior, the streams those of draw_params (hmm_device.cuh): same
    // results.  (The segment kernel's draw_params_lanes with L = 32 draws the same bits, but here its variate selection
    // costs ~20 more instructions per sweep on the critical path of a one-chain run: C1 0.2 % slower, B200 at 1000 W.)
    static __device__ __forceinline__ int draw_params_warp(const int lane, const int (&cnt)[K], const R (&Sd)[K], const R (&Qd)[K],
                                                          const int (&trans)[K][K], R c, const Hyper<R, K>& hp, const RngKey& key,
                                                          uint32_t sweep, R (&sig2)[K], R (&mu)[K], R (&rho)[K], R (&A)[K][K],
                                                          const SigStats<R, K>& sg) {
        int events = 0;
        StatePosterior<R> post[K];
        R shape = R(1);
        uint32_t purpose = (KIND_RHO << 16);
        bool mine = false;
#pragma unroll
        for (int i = 0; i < K; ++i) {
            if constexpr (SIG)
                post[i] = state_posterior<R, true>(cnt[i], Sd[i], Qd[i], c, hp.alpha[i], hp.beta[i], hp.nu[i], hp.xi[i],
                                                   sg.m[i], sg.Sm[i], sg.Qm[i], sg.k1);
            else
                post[i] = state_posterior<R>(cnt[i], Sd[i], Qd[i], c, hp.alpha[i], hp.beta[i], hp.nu[i], hp.xi[i]);
            if (lane == i) { shape = post[i].a; purpose = (KIND_SIGMA << 16) | (uint32_t)i; mine = post[i].a > R(0) && post[i].b > R(0); }
            if (lane == K + i) { shape = R(1); purpose = (KIND_RHO << 16) | (uint32_t)i; mine = true; }
#pragma unroll
            for (int j = 0; j < K; ++j)
                if (lane == 2 * K + i * K + j) { shape = (R)(trans[i][j] + 1); purpose = (KIND_A << 16) | (uint32_t)(i * K + j); mine = true; }
        }
        R g = R(1);
        if (mine) g = gamma_mt<R>(shape, key, sweep, purpose);
        R z = R(0);
        if (lane < K) {
            const uint4 w = rng_block(key, sweep, (KIND_MU << 16), (uint32_t)(lane >> 1));
            z = (lane & 1) ? normal_from<R>(w.z, w.w) : normal_from<R>(w.x, w.y);
        }
#pragma unroll
        for (int i = 0; i < K; ++i) {
            const R gi = __shfl_sync(kFull, g, i);
            if (post[i].a > R(0) && post[i].b > R(0)) sig2[i] = post[i].b / gi; else ++events;
        }
#pragma unroll
        for (int i = 0; i < K; ++i) mu[i] = post[i].mean(c, hp.nu[i], hp.xi[i]) + post[i].sd(sig2[i], hp.nu[i]) * __shfl_sync(kFull, z, i);
        {
            R tot = R(0);
#pragma unroll
            for (int i = 0; i < K; ++i) { rho[i] = __shfl_sync(kFull, g, K + i); tot += rho[i]; }
#pragma unroll
            for (int i = 0; i < K; ++i) rho[i] /= tot;
        }
#pragma unroll
        for (int i = 0; i < K; ++i) {
            R tot = R(0);
#pragma unroll
            for (int j = 0; j < K; ++j) { A[i][j] = __shfl_sync(kFull, g, 2 * K + i * K + j); tot += A[i][j]; }
#pragma unroll
            for (int j = 0; j < K; ++j) A[i][j] /= tot;
        }
        return events;
    }

    // emission of row t; signal rows (sw < 0) use sd x (1+kappa) (:382): z scaled by |sw| = 1/(1+kappa).  Returns the log2
    // of the factor divided out (fp32), including the 1/(1+kappa) of the signal pdf.
    static __device__ __forceinline__ R emission(const Emission<R, K>& em, R y, R sw, R (&e)[K]) {
        if constexpr (!SIG) {
            return em.eval(y, e);
        } else if constexpr (sizeof(R) == 8) {
            em.eval_scaled(y, sw, e);
            return R(0);
        } else {
            const float a = fabsf((float)sw);
            float l[K];
#pragma unroll
            for (int s = 0; s < K; ++s) { const float d = ((float)y - em.mu[s]) * a; l[s] = fmaf(d * d, em.q[s], em.c[s]); }
            float m = l[0];
#pragma unroll
            for (int s = 1; s < K; ++s) m = fmaxf(m, l[s]);
#pragma unroll
            for (int s = 0; s < K; ++s) e[s] = Real<float>::ex2(l[s] - m);
            return (R)(m + Real<float>::lg2(a));
        }
    }

    // one backward draw: X_t | X_{t+1} = xn  (src/Hmc.jl:466-481 in the pif form, quirk Q5 included)
    static __device__ __forceinline__ int draw_step(const R* __restrict__ pis, const R* __restrict__ As, int t, int xn, R u) {
        R p[K];
        const R gate = pis[(t + 1) * K + xn];
#pragma unroll
        for (int r = 0; r < K; ++r) p[r] = pis[t * K + r] * As[xn * 4 + r];
        if (!(gate > Real<R>::eps())) {
#pragma unroll
            for (int r = 0; r < K; ++r) p[r] = R(1);
        }
        return categorical_unnorm<R, K>(p, u);
    }

    static __device__ void run(const GibbsArgs& a, const int slot, const int lane, unsigned char* smem_warp, const int max_T) {
        const int ns = a.n_slots;
        const int T = a.T[slot];
        if (T <= 0) return;                                         // padding slot: the whole warp leaves
        R* const pis = reinterpret_cast<R*>(smem_warp);             // [T][K]
        R* const us = pis + (size_t)max_T * K;                      // [T] uniform of step t
        R* const As = us + max_T;                                   // As[x*4 + r] = A[r][x]
        const long long yld = a.yld;
        const R* __restrict__ const y0 = reinterpret_cast<const R*>(a.y) + a.ybase[slot];
        const R c = reinterpret_cast<const R*>(a.cshift)[slot];
        const RngKey key{a.k0, a.k1, a.chain_id[slot]};
        R* __restrict__ const out = reinterpret_cast<R*>(a.out);
        const int C = (T + 31) / 32;                                // chunk length
        const int t0 = min(lane * C, T), t1 = min(t0 + C, T);       // this lane's steps [t0, t1)
        const int lastlane = (T - 1) / C;                           // owner of step T-1

        // chain state: every lane holds the same copy
        int cnt[K], trans[K][K];
        R Sd[K], Qd[K], sig2[K], mu[K], rho[K], A[K][K];
        Hyper<R, K> hp;
        SigStats<R, K> sg;                                          // statistics of the signals (SIG; cnt/Sd/Qd: observations)
        load_chain_stats<R, K, SIG>(a, ns, slot, cnt, Sd, Qd, trans, hp, &sg);
#pragma unroll
        for (int i = 0; i < K; ++i) sig2[i] = R(1);
        int events = 0;
        const R* s0 = nullptr;                                      // emission z-scale of row t: s0[t*sld], sign = signal flag
        long long sld = 0;
        if constexpr (SIG) {
            sld = a.sld;
            s0 = reinterpret_cast<const R*>(a.sigw) + a.sbase[slot];
        }
        auto sw_at = [&](int t) -> R {
            if constexpr (SIG) return ld_ro(s0 + (long long)t * sld);
            else return R(1);
        };

        for (int sw = 0; sw < a.n_sweeps; ++sw) {
            const long long gs = a.sweep0 + sw;
            const uint32_t sweep = (uint32_t)gs;
            // ---- 1. conjugate draws (identical in every lane: same statistics, same counters)
#pragma unroll
            for (int i = 0; i < K; ++i) hp.beta[i] = (R)(gs == 0 ? a.beta0[i] : a.beta[i]);
            events += draw_params_warp(lane, cnt, Sd, Qd, trans, c, hp, key, sweep, sig2, mu, rho, A, sg);
            if (lane < K) {
#pragma unroll
                for (int r = 0; r < K; ++r) As[lane * 4 + r] = A[r][lane];
            }
            // uniforms of the backward pass: the i-th consumed (i = T-1-t) is word i&3 of Philox block i>>2
            for (int b = lane; 4 * b < T; b += 32) {
                const uint4 w = rng_block_states(key, sweep, (uint32_t)b);
                const int i = 4 * b;
                us[T - 1 - i] = u01<R>(w.x);
                if (i + 1 < T) us[T - 2 - i] = u01<R>(w.y);
                if (i + 2 < T) us[T - 3 - i] = u01<R>(w.z);
                if (i + 3 < T) us[T - 4 - i] = u01<R>(w.w);
            }

            // ---- 2. forward filter by scan
            Emission<R, K> em;
            em.prepare(mu, sig2);
            R P[K][K];
#pragma unroll
            for (int i = 0; i < K; ++i)
#pragma unroll
                for (int j = 0; j < K; ++j) P[i][j] = (i == j) ? R(1) : R(0);
            for (int t = t0; t < t1; ++t) {                         // phase 1: product of the chunk's A diag(e_t)
                R e[K], N[K][K];
                emission(em, ld_ro(y0 + (long long)t * yld), sw_at(t), e);
                matmul(P, A, N);
#pragma unroll
                for (int i = 0; i < K; ++i)
#pragma unroll
                    for (int s = 0; s < K; ++s) P[i][s] = N[i][s] * e[s];
                normalise(P);
            }
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {                      // phase 2: inclusive scan of the chunk products
                R Q[K][K], N[K][K];
#pragma unroll
                for (int i = 0; i < K; ++i)
#pragma unroll
                    for (int j = 0; j < K; ++j) Q[i][j] = __shfl_up_sync(kFull, P[i][j], d);
                if (lane >= d) {
                    matmul(Q, P, N);
#pragma unroll
                    for (int i = 0; i < K; ++i)
#pragma unroll
                        for (int j = 0; j < K; ++j) P[i][j] = N[i][j];
                    normalise(P);
                }
            }
            R pf[K];                                                // filtered vector entering this lane's chunk
            {
                R Q[K][K];
#pragma unroll
                for (int i = 0; i < K; ++i)
#pragma unroll
                    for (int j = 0; j < K; ++j) Q[i][j] = __shfl_up_sync(kFull, P[i][j], 1);
                R tot = R(0);
#pragma unroll
                for (int s = 0; s < K; ++s) {
                    R acc = rho[0] * Q[0][s];
#pragma unroll
                    for (int r = 1; r < K; ++r) acc = fma(rho[r], Q[r][s], acc);
                    pf[s] = acc;
                    tot += acc;
                }
                const R inv = R(1) / tot;
#pragma unroll
                for (int s = 0; s < K; ++s) pf[s] = (lane == 0) ? rho[s] : pf[s] * inv;   // t = 1 uses ρ (:390)
            }
            R ll = R(0);
            bool bad = false;
            for (int t = t0; t < t1; ++t) {                         // phase 3: the ordinary recursion over the chunk
                R e[K];
                const R m2 = emission(em, ld_ro(y0 + (long long)t * yld), sw_at(t), e);
                bool ok;
                const R tot = forward_step<R, K>(A, e, pf, ok);
                bad = bad || !ok;
                if (LOGLIK) {
                    if (sizeof(R) == 4) ll += (R)((Real<float>::lg2((float)tot) + (float)m2) * 0.6931471805599453f);
                    else ll += (R)log((double)tot);
                }
#pragma unroll
                for (int s = 0; s < K; ++s) pis[t * K + s] = pf[s];
            }
            {   // a chunk entered with a non-finite vector is bad as well (its own normalisers may still look fine)
                R chk = pf[0];
#pragma unroll
                for (int s = 1; s < K; ++s) chk += pf[s];
                bad = bad || (t1 > t0 && !(chk > R(0.5) && chk < R(2)));
            }
            if (__builtin_expect(__any_sync(kFull, bad), 0)) {
                // zero / non-finite normaliser somewhere (the reference only warns, :435): redo the filter serially with
                // the per-step reset to the uniform vector, every lane computing the same thing
                ll = R(0);
#pragma unroll
                for (int s = 0; s < K; ++s) pf[s] = rho[s];
                int ev = 0;
                for (int t = 0; t < T; ++t) {
                    R e[K];
                    const R m2 = emission(em, ld_ro(y0 + (long long)t * yld), sw_at(t), e);
                    bool ok;
                    const R tot = forward_step<R, K>(A, e, pf, ok);
                    if (!ok) {
                        ++ev;
#pragma unroll
                        for (int s = 0; s < K; ++s) pf[s] = R(1) / R(K);
                    }
                    if (LOGLIK && lane == 0) {
                        if (sizeof(R) == 4) ll += (R)((Real<float>::lg2((float)tot) + (float)m2) * 0.6931471805599453f);
                        else ll += (R)log((double)tot);
                    }
                    if (lane == 0) {
#pragma unroll
                        for (int s = 0; s < K; ++s) pis[t * K + s] = pf[s];
                    }
                }
                events += ev;
            } else {
#pragma unroll
                for (int s = 0; s < K; ++s) pf[s] = __shfl_sync(kFull, pf[s], lastlane);   // pif[T,:] in chain labels
            }
            if (LOGLIK) ll = wsum(ll);
            __syncwarp();
            R pend[K];                                              // what the draw reports as pi_end
#pragma unroll
            for (int s = 0; s < K; ++s) pend[s] = pf[s];
            if constexpr (SIG) {
                // samples.πb[:, endIndex, :] (:893): the smoothed marginal pi_back rows before the end of the window
                const int nback = a.pi_back < T - 1 ? a.pi_back : T - 1;
                for (int i = 1; i <= nback; ++i) {
                    R row[K];
#pragma unroll
                    for (int s = 0; s < K; ++s) row[s] = pis[(T - 1 - i) * K + s];
                    smooth_step<R, K>(A, row, pend);
                }
            }

            // ---- 3. relabel (:501-513) and emit the draw in increasing-μ order (lane 0 writes)
            int rank[K];
            ranks_of<R, K>(mu, rank);
            const long long draw_idx = gs - a.burnin;
            const bool save = draw_idx >= 0;
            if (save) {
                const size_t i = (size_t)(draw_idx - a.draw0);
                const size_t cs = (size_t)a.chunk * ns;
                R* o = out + i * ns + slot;
                const int f0 = 3 * K + K * K;
                R v[K];
#pragma unroll
                for (int s = 0; s < K; ++s) v[s] = pf[s];
                if (lane == 0) {
#pragma unroll
                    for (int s = 0; s < K; ++s) {
                        o[(size_t)(rank[s]) * cs] = mu[s];
                        o[(size_t)(K + rank[s]) * cs] = sig2[s];
                        o[(size_t)(2 * K + K * K + rank[s]) * cs] = pend[s];
#pragma unroll
                        for (int r = 0; r < K; ++r) o[(size_t)(2 * K + rank[s] * K + rank[r]) * cs] = A[r][s];
                    }
                    if (LOGLIK) o[(size_t)(f0 + 2 * a.n_h) * cs] = ll;
                }
                // lane j owns horizon j: it fetches the realised value up front and stores the pair at the end, so the
                // serial v <- v·A chain never waits for a global load
                const R yr = (lane < a.n_h) ? reinterpret_cast<const R*>(a.yfut)[(size_t)a.h_slot[lane] * ns + slot] : R(0);
                R myf = R(0);
                int h = 0;
                for (int j = 0; j < a.n_h; ++j) {                   // forecasts pib_T' A^h μ (:658-667, :858-862)
                    for (; h < a.h_sorted[j]; ++h) {
                        R nv[K];
#pragma unroll
                        for (int s = 0; s < K; ++s) {
                            R acc = v[0] * A[0][s];
#pragma unroll
                            for (int r = 1; r < K; ++r) acc = fma(v[r], A[r][s], acc);
                            nv[s] = acc;
                        }
#pragma unroll
                        for (int s = 0; s < K; ++s) v[s] = nv[s];
                    }
                    R f = v[0] * mu[0];
#pragma unroll
                    for (int s = 1; s < K; ++s) f = fma(v[s], mu[s], f);
                    if (lane == j) myf = f;
                }
                if (lane < a.n_h) {
                    o[(size_t)(f0 + 2 * a.h_slot[lane]) * cs] = myf;
                    o[(size_t)(f0 + 2 * a.h_slot[lane] + 1) * cs] = myf - yr;
                }
            }

            // ---- 4. backward sampling by composition of maps
            int xN;
            {   // X[N] ~ Categorical(pif[N,:]); with quirk Q1 the relabelled row is used with chain labels (:512-514)
                R pN[K];
                if (a.flags & 1u) {
#pragma unroll
                    for (int k = 0; k < K; ++k) {
                        R vsel = R(0);
#pragma unroll
                        for (int s = 0; s < K; ++s) vsel = (rank[s] == k) ? pf[s] : vsel;
                        pN[k] = vsel;
                    }
                } else {
#pragma unroll
                    for (int s = 0; s < K; ++s) pN[s] = pf[s];
                }
                xN = categorical_unnorm<R, K>(pN, us[T - 1]);
            }
            // this lane draws X_t for t in [t0, tw): the owner of step T-1 leaves that step out (it is X[N])
            const int tw = (lane == lastlane) ? T - 1 : t1;
            unsigned long long rec[K], recc = 0ull;                 // recorded paths: per entering state until coalescence, common after
#pragma unroll
            for (int h = 0; h < K; ++h) rec[h] = 0ull;
            unsigned F = 0x3210u;                                   // phase 1: composite map of the chunk (identity if it has no steps)
            if (lane <= lastlane) {
                // the K walks (one per entering state) advance together; once they have coalesced one walk is enough
                // the walked paths are recorded (2 bits per step; chunks of up to 32 steps) so that phase 3 only decodes
                int x[K];
#pragma unroll
                for (int h = 0; h < K; ++h) { x[h] = (lane == lastlane) ? xN : h; rec[h] = 0ull; }
                int t = tw - 1;
                for (; t >= t0; --t) {
                    bool same = true;
#pragma unroll
                    for (int h = 1; h < K; ++h) same = same && (x[h] == x[0]);
                    if (same) break;
                    const R u = us[t];
                    const int sh = 2 * ((tw - 1 - t) & 31);
#pragma unroll
                    for (int h = 0; h < K; ++h) { x[h] = draw_step(pis, As, t, x[h], u); rec[h] |= (unsigned long long)x[h] << sh; }
                }
                if (t >= t0) {
                    int x0 = x[0];
                    for (; t >= t0; --t) { x0 = draw_step(pis, As, t, x0, us[t]); recc |= (unsigned long long)x0 << (2 * ((tw - 1 - t) & 31)); }
#pragma unroll
                    for (int h = 0; h < K; ++h) x[h] = x0;
                }
                F = 0;
#pragma unroll
                for (int h = 0; h < K; ++h) F |= (unsigned)x[h] << (4 * h);
                if (K < 4) F |= 0x3000u;
            }
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {                      // phase 2: suffix scan, S_l = F_l ∘ F_{l+1} ∘ ...
                const unsigned Q = __shfl_down_sync(kFull, F, d);
                if (lane + d < 32) F = compose(F, Q);
            }
            int g = (int)(__shfl_down_sync(kFull, F, 1) & 15u);     // state entering this lane's chunk from above
            if (lane >= lastlane) g = xN;
            // phase 3: the actual path of this chunk and its statistics
            unsigned long long tr[K];
            R sdl[K], qdl[K], sml[K], qml[K];                       // observations / signals (SIG)
            int mil[K];
#pragma unroll
            for (int i = 0; i < K; ++i) { tr[i] = 0ull; sdl[i] = R(0); qdl[i] = R(0); sml[i] = R(0); qml[i] = R(0); mil[i] = 0; }
            {
                int xn = g;
                unsigned long long path = recc;
#pragma unroll
                for (int h = 0; h < K; ++h) path |= (g == h) ? rec[h] : 0ull;
                const bool recorded = C <= 32;                      // longer chunks are walked again
                for (int t = tw - 1; t >= t0; --t) {
                    const int x = recorded ? (int)((path >> (2 * (tw - 1 - t))) & 3ull) : draw_step(pis, As, t, xn, us[t]);
                    const R d = ld_ro(y0 + (long long)t * yld) - c, dd = d * d;
                    const unsigned long long inc = 1ull << (16 * xn);
                    const bool obs = !SIG || !(sw_at(t) < R(0));
#pragma unroll
                    for (int i = 0; i < K; ++i)
                        if (x == i) {
                            tr[i] += inc;
                            if (obs) { sdl[i] += d; qdl[i] += dd; }
                            else { sml[i] += d; qml[i] += dd; mil[i] += 1; }
                        }
                    xn = x;
                }
            }
            if (lane == lastlane) {                                 // X[N] itself: occupancy and sums, no outgoing transition
                const R d = ld_ro(y0 + (long long)(T - 1) * yld) - c, dd = d * d;
                const bool obs = !SIG || !(sw_at(T - 1) < R(0));
#pragma unroll
                for (int i = 0; i < K; ++i)
                    if (xN == i) {
                        if (obs) { sdl[i] += d; qdl[i] += dd; }
                        else { sml[i] += d; qml[i] += dd; mil[i] += 1; }
                    }
            }
#pragma unroll
            for (int i = 0; i < K; ++i) {
                const unsigned long long row = wsum64(tr[i]);
                Sd[i] = wsum(sdl[i]);
                Qd[i] = wsum(qdl[i]);
                int n = (xN == i) ? 1 : 0;
#pragma unroll
                for (int j = 0; j < K; ++j) { trans[i][j] = (int)((row >> (16 * j)) & 0xffffull); n += trans[i][j]; }
                if constexpr (SIG) {                              // split the occupancy into observations and signals
                    sg.m[i] = (int)wsum((R)mil[i]);
                    sg.Sm[i] = wsum(sml[i]);
                    sg.Qm[i] = wsum(qml[i]);
                    if (sg.m[i] == 0) { sg.Sm[i] = R(0); sg.Qm[i] = R(0); }
                    n -= sg.m[i];
                }
                cnt[i] = n;
                if (n == 0) { Sd[i] = R(0); Qd[i] = R(0); }
            }
            __syncwarp();
        }

        if (lane == 0) store_chain_stats<R, K, SIG>(a, ns, slot, cnt, Sd, Qd, trans, events, &sg);
    }
};

template <typename R, int K, bool LOGLIK, bool SIG = false>
__global__ void __launch_bounds__(kScanThreads) gibbs_scan_kernel(const GibbsArgs a, const int max_T) {
    extern __shared__ __align__(16) unsigned char scan_smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.x * (kScanThreads / 32) + warp;
    if (slot >= a.n_slots) return;
    ScanWarp<R, K, LOGLIK, SIG>::run(a, slot, lane, scan_smem + (size_t)warp * scan_warp_bytes<R, K>(max_T), max_T);
}

template <typename R, int K> cudaError_t launch_gibbs_scan(const GibbsLaunch& cfg, const GibbsArgs& a, cudaStream_t st);

}  // namespace hmc
