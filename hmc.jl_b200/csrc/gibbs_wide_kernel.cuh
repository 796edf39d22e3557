// gibbs_wide_kernel.cuh — the Gibbs sweep for K = 5..32 states: lane-per-state mapping.
//
// One chain is owned by a group of W lanes (W = 8, 16 or 32, the smallest that holds K); lane s of the group holds
// state s: its mean/variance, its filtered probability, its sufficient statistics, and it draws row s of A.  32/W
// chains share a warp.  The K x K transition matrix and the transition counters of a chain live in shared memory (rows
// padded to an odd stride so that both row and column accesses are conflict-free); for the forward recursion lane s
// keeps COLUMN s of A in registers and the filtered vector is broadcast through a double-buffered shared-memory line
// (one STS + W/4 LDS.128 per lane instead of K shuffles), the emission maximum is one CREDUX (W = 32) or a shuffle
// tree, the normaliser a shuffle tree, and the backward categorical draw a group prefix sum + ballot/popc.  Same
// arithmetic, same Philox streams and the same buffers as the thread-per-chain kernels (gibbs_kernel.cuh), so the two
// are interchangeable behind the plan.
// Reference lines as in gibbs_kernel.cuh (src/Hmc.jl:231-369 draws, :371-440 forward, :459-484 backward, :501-513 relabel).
#pragma once
#include "gibbs_kernel.cuh"

namespace hmc {

constexpr int kWideThreads = 128;

template <typename R, int W>
struct WideChain {
    static constexpr unsigned kFull = 0xffffffffu;
    static __device__ __forceinline__ unsigned group_mask(int lane) {
        return W == 32 ? kFull : (((1u << W) - 1u) << ((lane / W) * W));
    }
    static __device__ __forceinline__ R gsum(R v, unsigned m) {
#pragma unroll
        for (int o = W / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o, W);
        return v;
    }
    static __device__ __forceinline__ R gmax(R v, unsigned m) {
        if constexpr (W == 32 && sizeof(R) == 4) {                 // sm_100a: one warp-wide float max (CREDUX.MAX.F32)
            float r;
            asm volatile("redux.sync.max.f32 %0, %1, 0xffffffff;" : "=f"(r) : "f"((float)v));
            return (R)r;
        } else {
#pragma unroll
            for (int o = W / 2; o > 0; o >>= 1) { const R w = __shfl_xor_sync(m, v, o, W); v = v > w ? v : w; }
            return v;
        }
    }
    static __device__ __forceinline__ R gscan(R v, unsigned m, int s) {   // inclusive prefix sum over the group
#pragma unroll
        for (int o = 1; o < W; o <<= 1) { const R w = __shfl_up_sync(m, v, o, W); if (s >= o) v += w; }
        return v;
    }
};

// dynamic shared memory per chain group: broadcast lines [2][W] R (first: 16-byte aligned), A [K][K|1] R, transition
// counters [K*K] int; padded to 16 bytes
__host__ __device__ constexpr int wide_row_stride(int K) { return K | 1; }
template <typename R> __host__ __device__ constexpr size_t wide_group_bytes(int K, int W) {
    return (sizeof(R) * ((size_t)K * wide_row_stride(K) + 2 * (size_t)W) + sizeof(int) * (size_t)K * K + 15) / 16 * 16;
}

#ifndef HMC_WIDE_MINBLOCKS32
#define HMC_WIDE_MINBLOCKS32 5
#endif
template <typename R, int W, bool LOGLIK>
__global__ void __launch_bounds__(kWideThreads, sizeof(R) == 8 ? 3 : (W == 32 ? HMC_WIDE_MINBLOCKS32 : 4)) gibbs_wide_kernel(const GibbsArgs a, const int K, const long long* __restrict__ slot_pi_off) {
    using WC = WideChain<R, W>;
    extern __shared__ __align__(16) unsigned char wide_smem[];
    const int lane = threadIdx.x & 31;
    const int s = lane % W;                                   // state of this lane
    const int grp = threadIdx.x / W;                          // chain group within the block
    const int slot = blockIdx.x * (kWideThreads / W) + grp;
    const unsigned gm = WC::group_mask(lane);
    const int ns = a.n_slots;
    const bool live = slot < ns;
    const int T = live ? a.T[slot] : 0;
    if (T <= 0) return;                                       // whole group leaves together (T is group-uniform)
    const bool act = s < K;
    unsigned char* base = wide_smem + (size_t)grp * wide_group_bytes<R>(K, W);
    const int KP = wide_row_stride(K);
    R* const scratch = reinterpret_cast<R*>(base);                              // [2][W] broadcast lines
    R* const Asm = scratch + 2 * W;                                             // A[r*KP + c]
    int* const tr = reinterpret_cast<int*>(Asm + (size_t)K * KP);               // n_rc of the path being sampled

    const long long yld = a.yld;
    const R* __restrict__ const y0 = reinterpret_cast<const R*>(a.y) + a.ybase[slot];
    R* __restrict__ const pi0 = reinterpret_cast<R*>(a.pi) + slot_pi_off[slot];   // row t: pi0[t*K + s]
    const R c = reinterpret_cast<const R*>(a.cshift)[slot];
    const RngKey key{a.k0, a.k1, a.chain_id[slot]};
    R* __restrict__ const out = reinterpret_cast<R*>(a.out);

    // chain state of this lane's state
    int cnt = act ? a.cnt[s * ns + slot] : 0;
    R Sd = act ? reinterpret_cast<const R*>(a.Sd)[s * ns + slot] : R(0);
    R Qd = act ? reinterpret_cast<const R*>(a.Qd)[s * ns + slot] : R(0);
    const R xi = act ? reinterpret_cast<const R*>(a.xi)[s * ns + slot] : R(0);
    const R alpha = act ? (R)a.alpha[s] : R(1), nu = act ? (R)a.nu[s] : R(1);
    if (act) for (int j = 0; j < K; ++j) tr[s * K + j] = a.trans[(s * K + j) * ns + slot];
    __syncwarp(gm);
    R sig2 = R(1), mu = R(0);
    int events = 0;

    for (int sw = 0; sw < a.n_sweeps; ++sw) {
        const long long gs = a.sweep0 + sw;
        const uint32_t sweep = (uint32_t)gs;
        // ---- 1. conjugate draws: lane s draws sigma2_s, mu_s, its share of rho and row s of A
        R rho = R(0);
        if (act) {
            const R beta = (R)(gs == 0 ? a.beta0[s] : a.beta[s]);
            const R n = (R)cnt;
            const R dbar = cnt > 0 ? Sd / n : R(0);
            R s2 = Qd - n * dbar * dbar;
            s2 = s2 > R(0) ? s2 : R(0);
            const R totalbar = cnt > 0 ? dbar + c : R(0);
            const R dev = totalbar - xi;
            const R ga = alpha + R(0.5) * n;
            const R gb = beta + R(0.5) * s2 + R(0.5) * n * nu / (n + nu) * (dev * dev);
            if (ga > R(0) && gb > R(0)) sig2 = gb / gamma_mt<R>(ga, key, sweep, (KIND_SIGMA << 16) | (uint32_t)s);
            else ++events;
            const R m = (Sd + n * c + nu * xi) / (n + nu);
            const R sd = M<R>::sqrt(sig2 / (n + nu));
            const uint4 w = rng_block(key, sweep, (KIND_MU << 16), (uint32_t)(s >> 1));
            mu = m + sd * ((s & 1) ? normal_from<R>(w.z, w.w) : normal_from<R>(w.x, w.y));
            rho = gamma_mt<R>(R(1), key, sweep, (KIND_RHO << 16) | (uint32_t)s);
            R rowsum = R(0);
            for (int j = 0; j < K; ++j) {
                const R g = gamma_mt<R>((R)(tr[s * K + j] + 1), key, sweep, (KIND_A << 16) | (uint32_t)(s * K + j));
                Asm[s * KP + j] = g;
                rowsum += g;
            }
            const R inv = R(1) / rowsum;
            for (int j = 0; j < K; ++j) { Asm[s * KP + j] *= inv; tr[s * K + j] = 0; }
        }
        rho = rho / WC::gsum(rho, gm);
        __syncwarp(gm);
        // column s of A in registers (zero outside K x K): pred_s = sum_r pf_r A[r][s]
        R Ac[W];
#pragma unroll
        for (int r = 0; r < W; r += 2) {
            const R a0 = (act && r < K) ? Asm[r * KP + s] : R(0), a1 = (act && r + 1 < K) ? Asm[(r + 1) * KP + s] : R(0);
            Ac[r] = a0; Ac[r + 1] = a1;
        }

        // ---- 2. forward filter
        R q = R(0), cc = R(0), isd = R(1), nrm = R(0);
        if (sizeof(R) == 4) {
            q = (R)(-0.72134752044448170368) / sig2;
            cc = act ? (R)(-0.5f * Real<float>::lg2(6.283185307179586f * (float)sig2)) : (R)(-3.0e38);
        } else {
            const R sd = M<R>::sqrt(sig2);
            isd = R(1) / sd;
            nrm = act ? (R)0.3989422804014327 / sd : R(0);
        }
        R pf = rho;
        R ll = R(0);
        constexpr bool kMaxScale = (W == 32) && (sizeof(R) == 4);
        R pfn = rho;                                       // normalised filtered probability of the current row (kMaxScale)
        float lc = 0.f;
        // observations: batches of 8 steps, fetched into registers one batch ahead, their lines pulled into L1 two more
        // batches ahead (every chain of a wide batch streams its own series from HBM)
        // (W = 32 already keeps a 32-register column of A: there only the L1 prefetch is used, registers buy occupancy)
        constexpr bool kPipe = W < 32;
        R ybn[8];
        if constexpr (kPipe) {
#pragma unroll
            for (int j = 0; j < 8; ++j) ybn[j] = (j < T) ? y0[(long long)j * yld] : R(0);
        }
        for (int t0 = 0; t0 < T; t0 += 8) {
          R yb8[8];
          if (s < 8 && t0 + 24 + s < T) prefetch_l1(y0 + (long long)(t0 + 24 + s) * yld);
          if constexpr (kPipe) {
#pragma unroll
            for (int j = 0; j < 8; ++j) yb8[j] = ybn[j];
#pragma unroll
            for (int j = 0; j < 8; ++j) ybn[j] = (t0 + 8 + j < T) ? y0[(long long)(t0 + 8 + j) * yld] : R(0);
          } else {
#pragma unroll
            for (int j = 0; j < 8; ++j) yb8[j] = (t0 + j < T) ? y0[(long long)(t0 + j) * yld] : R(0);
          }
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int t = t0 + j;
            if (t >= T) break;
            const R yt = yb8[j];
            R e, m2 = R(0);
            if (sizeof(R) == 4) {
                const R d = yt - mu;
                const R l = act ? fma(d * d, q, cc) : (R)(-3.0e38);
                m2 = WC::gmax(l, gm);
                e = (R)Real<float>::ex2((float)(l - m2));
            } else {
                const R z = (yt - mu) * isd;
                e = (R)exp_nonpos<false>(-0.5 * (double)(z * z)) * nrm;
            }
            // broadcast pf through shared memory (double-buffered: one __syncwarp per step is enough)
            R* const line = scratch + (t & 1) * W;
            line[s] = pf;
            __syncwarp(gm);
            R acc[4] = {R(0), R(0), R(0), R(0)};
            constexpr int kVec = 16 / (int)sizeof(R);                  // elements per 16-byte shared-memory load
            using V = typename std::conditional<sizeof(R) == 4, float4, double2>::type;
#pragma unroll
            for (int r0 = 0; r0 < W; r0 += kVec) {
                const V v = *reinterpret_cast<const V*>(line + r0);
                if constexpr (sizeof(R) == 4) {
                    acc[0] = fma((R)v.x, Ac[r0], acc[0]); acc[1] = fma((R)v.y, Ac[r0 + 1], acc[1]);
                    acc[2] = fma((R)v.z, Ac[r0 + 2], acc[2]); acc[3] = fma((R)v.w, Ac[r0 + 3], acc[3]);
                } else {
                    acc[(r0 / 2) & 3] = fma((R)v.x, Ac[r0], acc[(r0 / 2) & 3]);
                    acc[(r0 / 2 + 1) & 3] = fma((R)v.y, Ac[r0 + 1], acc[(r0 / 2 + 1) & 3]);
                }
            }
            const R pred = (acc[0] + acc[1]) + (acc[2] + acc[3]);
            const R qq = pred * e;
            if constexpr (kMaxScale) {
                // W = 32, fp32: the recursion continues with qq rescaled by the exact power of two of its maximum (one
                // CREDUX), so the 5-step shuffle sum is needed only for the STORED row and the log-likelihood and
                // overlaps the next step instead of sitting in the dependent chain (measured: the largest stall).
                const float mx = (float)WC::gmax(qq, gm);
                const bool ok = (mx > 0.f) && (mx < 3.0e38f);
                const float scale = __int_as_float(0x7f000000 - (__float_as_int(mx) & 0x7f800000));   // 2^-floor(log2 mx)
                const R tot = WC::gsum(qq, gm);
                pfn = ok ? qq * Real<R>::rcp(tot) : (act ? R(1) / R(K) : R(0));
                pf = ok ? (R)((float)qq * scale) : pfn;
                if (!ok && s == 0) ++events;
                if (LOGLIK) {   // tot is relative to the scale lc = log2(sum of the previous recursion vector)
                    ll += (R)((Real<float>::lg2((float)tot) - lc + (float)m2) * 0.6931471805599453f);
                    lc = ok ? Real<float>::lg2((float)tot * scale) : 0.f;
                }
                if (act) pi0[(long long)t * K + s] = pfn;
            } else {
            const R tot = WC::gsum(qq, gm);
            const bool ok = (tot > R(0)) && (tot < R(3.0e38));
            pf = ok ? qq * Real<R>::rcp(tot) : (act ? R(1) / R(K) : R(0));
            if (!ok && s == 0) ++events;
            if (LOGLIK) {
                if (sizeof(R) == 4) ll += (R)((Real<float>::lg2((float)tot) + (float)m2) * 0.6931471805599453f);
                else ll += (R)log((double)tot);
            }
            if (act) pi0[(long long)t * K + s] = pf;
            }
          }
        }
        if constexpr (kMaxScale) pf = pfn;                 // pif[N,:], normalised
        __syncwarp(gm);

        // ---- 3. relabel and emit
        int rank = 0;
        for (int j = 0; j < K; ++j) {
            const R mj = __shfl_sync(gm, mu, j, W);
            rank += (mj < mu || (mj == mu && j < s)) ? 1 : 0;
        }
        const long long draw = gs - a.burnin;
        const bool save = draw >= 0;
        if (save) {
            const size_t i = (size_t)(draw - a.draw0);
            const size_t cs = (size_t)a.chunk * ns;
            R* o = out + i * ns + slot;
            if (act) {
                o[(size_t)rank * cs] = mu;
                o[(size_t)(K + rank) * cs] = sig2;
                o[(size_t)(2 * K + K * K + rank) * cs] = pf;
            }
            for (int r = 0; r < K; ++r) {
                const int rr = __shfl_sync(gm, rank, r, W);
                if (act) o[(size_t)(2 * K + rank * K + rr) * cs] = Asm[r * KP + s];     // emitted A[rr][rank] = A[r][s]
            }
            const int f0 = 3 * K + K * K;
            R v = pf;
            int h = 0;
            for (int j = 0; j < a.n_h; ++j) {
                for (; h < a.h_sorted[j]; ++h) {
                    R nv = R(0);
                    for (int r = 0; r < K; ++r) nv = fma(__shfl_sync(gm, v, r, W), act ? Asm[r * KP + s] : R(0), nv);
                    v = nv;
                }
                const R f = WC::gsum(act ? v * mu : R(0), gm);
                if (s == 0) {
                    const R yr = reinterpret_cast<const R*>(a.yfut)[(size_t)a.h_slot[j] * ns + slot];
                    o[(size_t)(f0 + 2 * a.h_slot[j]) * cs] = f;
                    o[(size_t)(f0 + 2 * a.h_slot[j] + 1) * cs] = f - yr;
                }
            }
            if (LOGLIK && s == 0) o[(size_t)(f0 + 2 * a.n_h) * cs] = ll;
        }

        // ---- 4. backward sampling fused with the next sweep's statistics
        cnt = 0; Sd = R(0); Qd = R(0);
        int xn = 0;
        R gate = R(1), Acol = R(0);
        uint4 w = make_uint4(0, 0, 0, 0);
        // rows and observations are fetched 8 steps at a time (they do not depend on the sampled states), so one
        // HBM/L2 latency is paid per 8 steps instead of per step
        constexpr int kBatch = 8;
        R ptn[kBatch], ytn[kBatch];                       // the batch after the one being processed
        auto fetch = [&](int i0) {
#pragma unroll
            for (int j = 0; j < kBatch; ++j) {
                const int t = T - 1 - (i0 + j);
                ptn[j] = (t >= 0 && act && (i0 + j) > 0) ? pi0[(long long)t * K + s] : R(0);
                ytn[j] = (t >= 0) ? y0[(long long)t * yld] : R(0);
            }
        };
        if constexpr (kPipe) fetch(0);
        for (int i0 = 0; i0 < T; i0 += kBatch) {
            R ptb[kBatch], ytb[kBatch];
            if constexpr (!kPipe) fetch(i0);
#pragma unroll
            for (int j = 0; j < kBatch; ++j) { ptb[j] = ptn[j]; ytb[j] = ytn[j]; }
            {   // lines of the batch after next: lanes 0..7 of the group take one row each (y and the first line of the pif row)
                const int t = T - 1 - (i0 + 2 * kBatch + s);
                if (s < kBatch && t >= 0) { prefetch_l1(y0 + (long long)t * yld); prefetch_l1(pi0 + (long long)t * K); }
            }
            if constexpr (kPipe) fetch(i0 + kBatch);
            if ((i0 & (4 * W - 1)) == 0) w = rng_block_states(key, sweep, (uint32_t)((i0 >> 2) + s));   // block of steps i0 + 4s .. + 3
#pragma unroll
            for (int j = 0; j < kBatch; ++j) {
                const int i = i0 + j;
                if (i >= T) break;
                // uniforms: every lane of the group generated ONE Philox block of the next 4W steps (see above), so a step costs
                // one shuffle instead of a quarter of a Philox evaluation in every lane
                const uint32_t wsel = (j & 3) == 0 ? w.x : (j & 3) == 1 ? w.y : (j & 3) == 2 ? w.z : w.w;
                const uint32_t wi = __shfl_sync(gm, wsel, (i >> 2) & (W - 1), W);
                const R u = u01<R>(wi);
                R pt, p;
                if (i == 0) {
                    pt = pf;
                    if (a.flags & 1u) {                      // quirk Q1: the relabelled row, used with chain labels
                        if (act) scratch[rank] = pf;
                        __syncwarp(gm);
                        p = act ? scratch[s] : R(0);
                        __syncwarp(gm);
                    } else {
                        p = act ? pf : R(0);
                    }
                } else {
                    pt = ptb[j];
                    p = (gate > Real<R>::eps()) ? pt * Acol : (act ? R(1) : R(0));
                }
                const R cum = WC::gscan(p, gm, s);
                const R tot = __shfl_sync(gm, cum, K - 1, W);
                const R thr = u * tot;
                const unsigned below = __ballot_sync(gm, (cum < thr) && (s < K - 1)) & gm;
                const int x = __popc(below);
                const R d = ytb[j] - c;
                if (s == x) {
                    cnt += 1; Sd += d; Qd += d * d;
                    if (i > 0) tr[x * K + xn] += 1;
                }
                xn = x;
                gate = __shfl_sync(gm, pt, x, W);
                Acol = act ? Asm[s * KP + x] : R(0);
            }
        }
        __syncwarp(gm);
    }

    if (act) {
        a.cnt[s * ns + slot] = cnt;
        reinterpret_cast<R*>(a.Sd)[s * ns + slot] = Sd;
        reinterpret_cast<R*>(a.Qd)[s * ns + slot] = Qd;
        for (int j = 0; j < K; ++j) a.trans[(s * K + j) * ns + slot] = tr[s * K + j];
    }
    const int ev = (int)WC::gsum((R)events, gm);
    if (s == 0) a.events[slot] += ev;
}

template <typename R> cudaError_t launch_gibbs_wide(const GibbsLaunch& cfg, const GibbsArgs& a, int K, const long long* slot_pi_off, cudaStream_t st);

}  // namespace hmc
