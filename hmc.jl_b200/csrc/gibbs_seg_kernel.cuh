// gibbs_seg_kernel.cuh — the Gibbs sweep for MID-WIDTH batches (a few thousand to a few ten thousand chains): L lanes per
// chain, each lane owning one contiguous time SEGMENT of the window; 32/L chains per warp.
//
// Why.  With a thread per chain (gibbs_kernel.cuh) a batch of 16 000 chains is 500 warps on 592 warp schedulers: every warp
// runs alone, in order, at ~3.3 cycles per instruction, and the job lasts as long as its longest window (T steps, one after
// the other).  With a warp per chain (gibbs_scan_kernel.cuh) the per-sweep work (draws, scans) is paid per chain instead of
// per 32 chains and the kernel is instruction-bound from ~4000 chains.  Here the window is cut into L = 4 or 8 segments: L times
// more warps with L times shorter dependent chains, and the per-sweep work is still shared by 32/L chains.  This is one GPU's
// share of the fixed 500 x 256 rolling job when it is sharded over 8 GPUs (strong scaling; the reference's parallel unit is one
// process per end date, slurmscripts/base_estimation.sh:5,17).
//
// Segments are cut in BACKWARD index space (i = 0 is X[N]) in multiples of 4 steps, so Philox blocks never straddle lanes:
// segment q holds i in [qC, (q+1)C), C = 4 ceil(T_warp / 4L); segment 0 is the END of the window, the last one is ragged.
// Inside its segment a lane is exactly a (ragged) lane of the thread-per-chain kernel: same right-aligned tile frame of C
// rows, same spill layout, same cp.async ring.
//
//   forward filter (forwardupdate_P!, src/Hmc.jl:371-440).  Phase 1: every lane multiplies the K x K matrices A diag(e_t) of
//   its segment.  Phase 2: the chain's lanes pass the filtered vector along: v_q = normalise(v_{q+1} M_{q+1}) (L-1 rounds of
//   shuffles).  Phase 3: the lane runs the ordinary recursion from its entering vector — GibbsWarp::forward_pass itself, so
//   rows, normalisers and log-likelihood are the usual ones — and spills its rows.
//
//   backward sampling (update_X!, :459-484).  A lane does not know the state entering its segment from above.  Pass A: it
//   walks all K candidates at once, 4 steps at a time, until (warp-wide) every lane's candidates have coalesced — sticky
//   chains do within a few steps.  Pass B: one walk from the coalesced state to the end of the segment, accumulating the next
//   sweep's statistics (:254-258, :291-294, :362-365).  The composite maps (entering state -> leaving state, 2 bits each) are
//   chained through the L lanes, after which every lane knows its true entering state and (pass C) replays the few
//   speculative steps with statistics.  Exactly the serial algorithm's path for the same uniforms.
//
// Same Philox streams, draw order, buffers and outputs as the other sweep kernels (interchangeable behind the plan); the fp64
// chain follows the oracle's chain (phase 2 only re-associates the products that carry the filtered vector to a segment
// boundary).  K <= 4, plain sweep (no smoothed means, no signals), segment length <= 2^(32/K) - 1.
#pragma once
#include "lane_draws.cuh"
#include "plan_policy.cuh"    // kSegThreads (threads per block), seg_max_T

namespace hmc {

static_assert(kSegThreads % kGibbsThreads == 0, "whole selection tables");

// (the selection table of GibbsWarp is laid out for kGibbsThreads threads: one table per kGibbsThreads threads of the block)
template <typename R, int K> __host__ __device__ constexpr size_t seg_smem_bytes(int n_h, int threads) {
    return sizeof(GibbsEntry<R, K, false>) * K * (size_t)threads                                 // selection tables (pass B)
           + sizeof(R) * (size_t)(threads / 32) * gibbs_ring_stages<R, K>() * 4 * K * 32         // cp.async rings
           + sizeof(R) * (size_t)(n_h > 0 ? n_h : 1) * threads;                                  // realised y at end+h, per thread
}

template <typename R, int K, int L, bool LOGLIK>
struct SegWarp {
    static_assert(L == 2 || L == 4 || L == 8 || L == 16, "lanes per chain");
    static constexpr unsigned kFull = 0xffffffffu;
    static constexpr int kCPW = 32 / L;                               // chains per warp
    using GW = GibbsWarp<R, K, false, LOGLIK, false, false>;
    using Chain = typename GW::Chain;
    using Vec = typename GW::Vec;
    using FwdOut = typename GW::FwdOut;
    static constexpr int kRing = GW::kRing;
    static constexpr int kBits = 32 / K;                              // packed transition counters: row[origin], one field per destination
    static constexpr unsigned kFieldMask = (kBits >= 32) ? 0xffffffffu : ((1u << kBits) - 1u);

    struct Mat { R m[K][K]; bool bad; };

    static __device__ __forceinline__ bool normalise(R (&P)[K][K]) {
        R s = R(0);
#pragma unroll
        for (int i = 0; i < K; ++i)
#pragma unroll
            for (int j = 0; j < K; ++j) s += P[i][j];
        const R inv = Real<R>::rcp(s);
#pragma unroll
        for (int i = 0; i < K; ++i)
#pragma unroll
            for (int j = 0; j < K; ++j) P[i][j] *= inv;
        return (s > R(0)) && (s < R(3.0e38));
    }

    // phase 1: M = prod_t A diag(e_t) over the lane's rows (any positive scale; identity for an empty segment)
    template <bool STREAM>
    static __device__ __noinline__ Mat seg_product(const Chain ch, const Emission<R, K> em) {
        Mat o;
        R (&P)[K][K] = o.m;
#pragma unroll
        for (int i = 0; i < K; ++i)
#pragma unroll
            for (int j = 0; j < K; ++j) P[i][j] = (i == j) ? R(1) : R(0);
        const long long yld = STREAM ? ch.yld : 1ll;                 // (one shared series: stride 1, as in forward_pass)
        const R* yp = ch.y0 + (long long)ch.off * yld;
        bool ok = true;
        auto step = [&](const R yt) {
            R e[K], N[K][K];
            em.eval(yt, e);
#pragma unroll
            for (int i = 0; i < K; ++i)
#pragma unroll
                for (int s = 0; s < K; ++s) {
                    R acc = P[i][0] * ch.A[0][s];
#pragma unroll
                    for (int r = 1; r < K; ++r) acc = fma(P[i][r], ch.A[r][s], acc);
                    N[i][s] = acc * e[s];
                }
#pragma unroll
            for (int i = 0; i < K; ++i)
#pragma unroll
                for (int s = 0; s < K; ++s) P[i][s] = N[i][s];
        };
        int j = ch.off;
        if constexpr (sizeof(R) == 4) {
            // the fp32 emissions are scaled to a maximum of one: the product shrinks by at most min(A) per step and is
            // renormalised every 4 steps
            for (; j + 3 < ch.Tw; j += 4, yp += 4 * yld) {
                const R y0 = ld_ro(yp), y1 = ld_ro(yp + yld), y2 = ld_ro(yp + 2 * yld), y3 = ld_ro(yp + 3 * yld);
                step(y0); step(y1); step(y2); step(y3);
                ok = normalise(P) && ok;
            }
        }
        for (; j < ch.Tw; ++j, yp += yld) {
            step(ld_ro(yp));
            ok = normalise(P) && ok;
        }
        o.bad = !ok;
        return o;
    }


    // The filtered vector entering a segment, WITHOUT the products of phase 1: the filter forgets its initial condition, so the
    // recursion is started from the flat vector W time steps before the segment (from ρ itself when that reaches t = 1, which is
    // then exact).  The result is only USED when it agrees with the final row of the segment before (known after phase 3) within
    // kWarmTol — otherwise the chain's segments are filtered again from the exact vectors of phases 1-2.  Rows computed from a
    // verified vector differ from the exact ones by less than the rounding noise of the recursion itself.
    static __device__ __forceinline__ R warm_tol() { return sizeof(R) == 4 ? R(2.0e-7) : R(1.0e-13); }
    template <bool STREAM>
    static __device__ __noinline__ Vec seg_warmup(const Chain ch, const Emission<R, K> em, const Vec start, const int W) {
        Vec o;
        R (&pi)[K] = o.v;
#pragma unroll
        for (int s = 0; s < K; ++s) pi[s] = start.v[s];
        const long long yld = STREAM ? ch.yld : 1ll;
        const R* yp = ch.y0 + (long long)(ch.off - W) * yld;         // rows off-W .. off-1: the W time steps before the segment
        for (int j = 0; j < W; ++j, yp += yld) {
            R e[K];
            em.eval(ld_ro(yp), e);
            bool ok;
            forward_step<R, K>(ch.A, e, pi, ok);
        }
        return o;
    }

    // one backward draw X_t | X_{t+1} = xl (src/Hmc.jl:466-481 in the pif form): pt = pif[t,:], pl = pif[t+1,:] (quirk Q5 gate).
    // Same operations as GibbsWarp::back_step (gated form).
    static __device__ __forceinline__ int draw_from(const R (&A)[K][K], int xl, const R (&pt)[K], const R (&pl)[K], R u) {
        R p[K];
#pragma unroll
        for (int r = 0; r < K; ++r) p[r] = pt[r] * select_k<R, K>(A[r], xl);
        const R gate = select_k<R, K>(pl, xl);
        if (!(gate > Real<R>::eps())) {
#pragma unroll
            for (int r = 0; r < K; ++r) p[r] = R(1);
        }
        return categorical_unnorm<R, K>(p, u);
    }

    struct SpecState { int s[K]; R pl[K]; bool coal; };              // state of each candidate (entering state h), the later step's row
    struct GroupRows { R c[4][K]; R y[4]; uint4 w; };                // 4 steps: filtered rows, observations, Philox block

    // 4 steps of the speculative walk (pass A): all K candidates advance; X[N] itself is step 0 of segment 0.  Rolled and out
    // of line on purpose (runs about once per sweep).
    static __device__ __noinline__ SpecState spec_group(const Chain ch, SpecState st, const GroupRows gr, const int i0, const int n, const int q, const int xN) {
#pragma unroll 1
        for (int u = 0; u < 4; ++u) {
            if (i0 + u < n) {
                const uint32_t word = u == 0 ? gr.w.x : u == 1 ? gr.w.y : u == 2 ? gr.w.z : gr.w.w;
                const R u_ = u01<R>(word);
                R pt[K];
#pragma unroll
                for (int k = 0; k < K; ++k) pt[k] = gr.c[u][k];
                if (q == 0 && i0 + u == 0) {
#pragma unroll
                    for (int h = 0; h < K; ++h) st.s[h] = xN;
                } else {
#pragma unroll 1
                    for (int h = 0; h < K; ++h) st.s[h] = draw_from(ch.A, st.s[h], pt, st.pl, u_);
                }
#pragma unroll
                for (int k = 0; k < K; ++k) st.pl[k] = pt[k];
            }
        }
        bool same = true;
#pragma unroll
        for (int h = 1; h < K; ++h) same = same && (st.s[h] == st.s[0]);
        st.coal = same;
        return st;
    }
    // 4 steps of pass B with the per-lane end-of-segment test (the groups around the end of the warp's shortest segments)
    static __device__ __noinline__ typename GW::Back passB_group_guarded(const Chain ch, typename GW::Back b, const GroupRows gr, const int i0, const int n) {
        bool badq = false;
#pragma unroll 1
        for (int u = 0; u < 4; ++u) {
            if (i0 + u < n) {
                const uint32_t word = u == 0 ? gr.w.x : u == 1 ? gr.w.y : u == 2 ? gr.w.z : gr.w.w;
                R pt[K];
#pragma unroll
                for (int k = 0; k < K; ++k) pt[k] = gr.c[u][k];
                GW::template back_step<true>(b, ch, pt, nullptr, nullptr, gr.y[u], R(1), word, false, badq);
            }
        }
        return b;
    }

    struct BackOut { R Sd[K - 1], Qd[K - 1]; unsigned row[K]; int xN; };

    template <bool STREAM>
    static __device__ __noinline__ BackOut seg_backward(const Chain ch, const Vec pf_end, const RngKey key, const uint32_t sweep,
                                                        const unsigned flags, const int q, const int Cc, unsigned long long* diag) {
        BackOut o;
        const int C = ch.Tw, n = ch.T;                               // rows of the frame, steps of this lane (right-aligned)
        const int n_min = (int)__reduce_min_sync(kFull, (unsigned)n); // steps every lane of the warp has
        const int lane = threadIdx.x & 31;
        const int base_lane = lane - q;                              // lane of the chain's segment 0
        const long long ys = STREAM ? ch.yld : 1ll;
        const uint32_t blk0 = (uint32_t)(q * (Cc >> 2));             // Philox block of this segment's first step (Cc: rows per segment of this chain)
        R Sd[K - 1], Qd[K - 1];
        unsigned row[K];
#pragma unroll
        for (int i = 0; i < K - 1; ++i) { Sd[i] = R(0); Qd[i] = R(0); }
#pragma unroll
        for (int i = 0; i < K; ++i) row[i] = 0u;
        // row j of the frame, state s: tile layout of gibbs_kernel.cuh with pad = 0 (C is a multiple of 4)
        auto row_ptr = [&](int jrow) -> const R* { return ch.pi0 + (size_t)(jrow >> 2) * (4 * K * 32) + (jrow & 3); };
        const R* const ytop = ch.y0 + (long long)(C - 1) * ys;       // observation of step i' = 0
        // the filtered row of the step above this segment (quirk Q5 gate of step i' = 0): the neighbour lane's row 0
        R pabove[K];
#pragma unroll
        for (int s = 0; s < K; ++s) pabove[s] = R(1);
        if (q > 0 && n > 0) {                                        // (that segment is full: Cc rows, right-aligned in the frame of C)
            const R* rp = ch.pi0 - 4 + (size_t)((C - Cc) >> 2) * (4 * K * 32);
#pragma unroll
            for (int s = 0; s < K; ++s) pabove[s] = ld_stream(rp + s * 128);
        }
        // X[N] ~ Categorical(pif[N,:]) by the lane of segment 0; with quirk Q1 the relabelled row is used with chain labels (:512-514)
        int xN = 0;
        if (q == 0 && n > 0) {
            R pN[K];
            if (flags & 1u) {
#pragma unroll
                for (int k = 0; k < K; ++k) {
                    R vsel = R(0);
#pragma unroll
                    for (int s = 0; s < K; ++s) vsel = (ch.rank[s] == k) ? pf_end.v[s] : vsel;
                    pN[k] = vsel;
                }
            } else {
#pragma unroll
                for (int s = 0; s < K; ++s) pN[s] = pf_end.v[s];
            }
            const uint4 w0 = rng_block_states(key, sweep, 0u);
            xN = categorical_unnorm<R, K>(pN, u01<R>(w0.x));
        }
        auto book = [&](int x, int xl, bool has_later, R yt) {      // state x at this step, xl at the later one
            const unsigned inc = 1u << (kBits * xl);
            const R d = yt - ch.c;
#pragma unroll
            for (int i = 0; i < K; ++i) if (x == i && has_later) row[i] += inc;
#pragma unroll
            for (int i = 0; i < K - 1; ++i) if (x == i) { Sd[i] += d; Qd[i] = fma(d, d, Qd[i]); }
        };

        // ---- passes A and B over the ring
        constexpr int kGroupElems = 4 * K * 32;
        constexpr int kChunksPerLane = (int)(kGroupElems * sizeof(R) / 16 / 32);
        constexpr unsigned kGroupBytes = (unsigned)(kGroupElems * sizeof(R));
        R* const ring = reinterpret_cast<R*>(smem_base() + ch.ring_off);
        const int n_groups = C >> 2;
        const char* nsrc = reinterpret_cast<const char*>(ch.pi0 - lane * 4 + (long long)(C - 4) * K * 32) + lane * 16;   // tile of group 0
        const unsigned ring_s = (unsigned)__cvta_generic_to_shared(ring) + (unsigned)lane * 16u;
        const unsigned ring_rd = (unsigned)__cvta_generic_to_shared(ring) + (unsigned)(lane * 4 * sizeof(R));   // this lane's rows of state 0, stage 0
        unsigned nstage = 0, rstage = 0;
        int nleft = n_groups;
        auto issue = [&]() {
            if (nleft > 0) {
#pragma unroll
                for (int m = 0; m < kChunksPerLane; ++m) cp_async16_s(ring_s + nstage + 512u * m, nsrc + 512 * m);
            }
            cp_async_commit();
            --nleft;
            nsrc -= kGroupBytes;
            nstage = (nstage + kGroupBytes == kRing * kGroupBytes) ? 0u : nstage + kGroupBytes;
        };
#pragma unroll
        for (int g = 0; g < kRing - 1; ++g) issue();
        SpecState sp;                                                // candidates of the speculative walk
#pragma unroll
        for (int h = 0; h < K; ++h) sp.s[h] = h;
#pragma unroll
        for (int k = 0; k < K; ++k) sp.pl[k] = pabove[k];
        sp.coal = false;
        bool spec = true;                                            // uniform over the chain's lanes: still walking candidates
        int spec_groups = 0;
        typename GW::Back b;                                         // pass B state: GibbsWarp's backward step (statistics, packed counters, selections)
#pragma unroll
        for (int i = 0; i < K - 1; ++i) { b.Sd[i] = R(0); b.Qd[i] = R(0); }
        b.tr.clear();
        b.inc = 0; b.gate = R(1);
#pragma unroll
        for (int k = 0; k < K; ++k) { b.Acol[k] = R(0); b.pb[k] = R(0); }
        const R* yp = ytop;
        // the next group of 4 rows out of the ring (position 3 of a tile = its highest row = the group's first step), its
        // observations and its Philox block
        auto next_group = [&](GroupRows& gr, const int g, const bool guard_y) {
            issue();
            cp_async_wait<kRing - 1>();
            __syncwarp();
            // (read through a 32-bit shared address computed once per pass, like the thread-per-chain kernel's ring loop)
            const unsigned rd = ring_rd + rstage;
            rstage = (rstage + kGroupBytes == kRing * kGroupBytes) ? 0u : rstage + kGroupBytes;
#pragma unroll
            for (int k = 0; k < K; ++k) lds_quad(rd + (unsigned)(k * 128 * sizeof(R)), gr.c[3][k], gr.c[2][k], gr.c[1][k], gr.c[0][k]);
#pragma unroll
            for (int u = 0; u < 4; ++u) gr.y[u] = (!guard_y || 4 * g + u < n) ? ld_ro(yp - u * ys) : R(0);
            yp -= 4 * ys;
            gr.w = rng_block_states(key, sweep, blk0 + (uint32_t)g);
        };
        int g = 0;
        // ---- loop A: while some chain of the warp still walks candidates (about one group per sweep).  Chains that have
        // coalesced already run pass B on these groups.  Both bodies are out of line: they must not sit in the hot loop's cache lines.
        for (; g < n_groups; ++g) {
            const unsigned open_lanes = __ballot_sync(kFull, spec && (4 * g < n) && !sp.coal);
            if (spec) {
                // decided per CHAIN (its L lanes), not per warp: which steps are replayed then depends on the chain alone, so the
                // summation order of its statistics — and with it every result bit — is independent of the rest of the batch
                spec = ((open_lanes >> base_lane) & ((1u << L) - 1u)) != 0u;
                if (!spec) {                                         // pass B starts: the later step's state is s[0], its row pl
                    bool ltx[K - 1];
#pragma unroll
                    for (int i = 0; i < K - 1; ++i) ltx[i] = sp.s[0] > i;
                    GW::select_later(b, ch, ltx, sp.pl);
                }
            }
            if (open_lanes == 0u) break;
            GroupRows gr;
            next_group(gr, g, true);
            if (spec) { sp = spec_group(ch, sp, gr, 4 * g, n, q, xN); ++spec_groups; }
            else b = passB_group_guarded(ch, b, gr, 4 * g, n);
            __syncwarp();
        }
        // ---- loop B: groups every lane of the warp has in full — the hot loop: no per-lane tests, 4 inlined steps
        {
            bool badq = false;
            for (; g < n_groups && 4 * g + 3 < n_min; ++g) {
                GroupRows gr;
                next_group(gr, g, false);
                GW::template back_step<true>(b, ch, gr.c[0], nullptr, nullptr, gr.y[0], R(1), gr.w.x, false, badq);
                GW::template back_step<true>(b, ch, gr.c[1], nullptr, nullptr, gr.y[1], R(1), gr.w.y, false, badq);
                GW::template back_step<true>(b, ch, gr.c[2], nullptr, nullptr, gr.y[2], R(1), gr.w.z, false, badq);
                GW::template back_step<true>(b, ch, gr.c[3], nullptr, nullptr, gr.y[3], R(1), gr.w.w, false, badq);
                __syncwarp();
            }
        }
        // ---- loop C: the last groups, where the shortest segments of the warp have ended
        for (; g < n_groups; ++g) {
            GroupRows gr;
            next_group(gr, g, true);
            b = passB_group_guarded(ch, b, gr, 4 * g, n);
            __syncwarp();
        }
        cp_async_wait<0>();
        int s[K];
#pragma unroll
        for (int h = 0; h < K; ++h) s[h] = sp.s[h];
        if (!spec) {                                                 // pass B ran: every candidate leaves through its last state
            const bool ranB = 4 * spec_groups < n;
            const int xlast = (__ffs((int)b.inc) - 1) / kBits;       // b.inc = 1 << (kBits * state of the last step)
#pragma unroll
            for (int h = 0; h < K; ++h) s[h] = ranB ? xlast : s[h];
        }
        // ---- the chain's lanes compose their maps (entering state -> leaving state): the true entering state of every segment
        unsigned Fp = 0u;
#pragma unroll
        for (int h = 0; h < K; ++h) Fp |= (unsigned)s[h] << (2 * h);
        int xin = 0, cur = 0;
#pragma unroll
        for (int qq = 0; qq < L; ++qq) {
            const unsigned Fq = __shfl_sync(kFull, Fp, base_lane + qq);
            if (qq == q) xin = cur;
            cur = (int)((Fq >> (2 * cur)) & 3u);
        }
        xN = __shfl_sync(kFull, xN, base_lane);
        if (diag && q == 0) atomicAdd(diag + 1, (unsigned long long)spec_groups);
        // ---- pass C: the speculative steps again, from the true entering state, with statistics
        {
            const int nrep = min(4 * spec_groups, n);
            int xc = xin;
            R plc[K];
#pragma unroll
            for (int k = 0; k < K; ++k) plc[k] = pabove[k];
            const R* ypc = ytop;
            uint4 wc = make_uint4(0u, 0u, 0u, 0u);
            for (int i = 0; i < nrep; ++i, ypc -= ys) {
                R pt[K];
                const R* rp = row_ptr(C - 1 - i);
#pragma unroll
                for (int k = 0; k < K; ++k) pt[k] = ld_stream(rp + k * 128);
                const R yt = ld_ro(ypc);
                if ((i & 3) == 0) wc = rng_block_states(key, sweep, blk0 + (uint32_t)(i >> 2));
                const uint32_t word = (i & 3) == 0 ? wc.x : (i & 3) == 1 ? wc.y : (i & 3) == 2 ? wc.z : wc.w;
                if (q == 0 && i == 0) {
                    book(xN, 0, false, yt);
                    xc = xN;
                } else {
                    const int xn_ = draw_from(ch.A, xc, pt, plc, u01<R>(word));
                    book(xn_, xc, true, yt);
                    xc = xn_;
                }
#pragma unroll
                for (int k = 0; k < K; ++k) plc[k] = pt[k];
            }
        }
#pragma unroll
        for (int i = 0; i < K - 1; ++i) { o.Sd[i] = b.Sd[i] + Sd[i]; o.Qd[i] = b.Qd[i] + Qd[i]; }    // pass B + replayed steps
#pragma unroll
        for (int i = 0; i < K; ++i) o.row[i] = b.tr.row[i] + row[i];
        o.xN = xN;
        return o;
    }

    // Conjugate draws with the K*K + 2K gamma variates spread over the L lanes of a chain (each variate has its own Philox
    // purpose stream, so they are independent): variate g is drawn by lane g % L in its round g / L and handed round by shuffles.
    // The posterior of each state is state_posterior, the streams those of draw_params (hmm_device.cuh): same results, bit for bit.
    static constexpr int kNG = K * K + 2 * K;
    static constexpr int kRounds = (kNG + L - 1) / L;
    static __device__ __forceinline__ int draw_params_lanes(const int q, const int base_lane, const int (&cnt)[K], const R (&Sd)[K],
                                                            const R (&Qd)[K], const int (&trans)[K][K], R c, const Hyper<R, K>& hp,
                                                            const RngKey& key, uint32_t sweep, R (&sig2)[K], R (&mu)[K], R (&rho)[K],
                                                            R (&A)[K][K]) {
        int events = 0;
        StatePosterior<R> post[K];
        R shape[kNG];
        uint32_t purpose[kNG];
        bool valid[kNG];
#pragma unroll
        for (int i = 0; i < K; ++i) {
            post[i] = state_posterior<R>(cnt[i], Sd[i], Qd[i], c, hp.alpha[i], hp.beta[i], hp.nu[i], hp.xi[i]);
            shape[i] = post[i].a; purpose[i] = (KIND_SIGMA << 16) | (uint32_t)i; valid[i] = post[i].a > R(0) && post[i].b > R(0);
            shape[K + i] = R(1); purpose[K + i] = (KIND_RHO << 16) | (uint32_t)i; valid[K + i] = true;
#pragma unroll
            for (int j = 0; j < K; ++j) {
                shape[2 * K + i * K + j] = (R)(trans[i][j] + 1);
                purpose[2 * K + i * K + j] = (KIND_A << 16) | (uint32_t)(i * K + j);
                valid[2 * K + i * K + j] = true;
            }
        }
        R gl[kRounds];
#pragma unroll
        for (int m = 0; m < kRounds; ++m) {
            R sh = R(1);
            uint32_t pu = 0u;
            bool mine = false;
#pragma unroll
            for (int l = 0; l < L; ++l) {
                const int g = m * L + l;
                if (g < kNG && q == l) { sh = shape[g]; pu = purpose[g]; mine = valid[g]; }
            }
            gl[m] = R(1);
            if (mine) gl[m] = gamma_mt<R>(sh, key, sweep, pu);
        }
        R z = R(0);                                                  // normals of mu: lane i draws state i's (every lane when L < K)
        R zs[K];
        if constexpr (L >= K) {
            if (q < K) {
                const uint4 w = rng_block(key, sweep, (KIND_MU << 16), (uint32_t)(q >> 1));
                z = (q & 1) ? normal_from<R>(w.z, w.w) : normal_from<R>(w.x, w.y);
            }
#pragma unroll
            for (int i = 0; i < K; ++i) zs[i] = __shfl_sync(kFull, z, base_lane + i);
        } else {
#pragma unroll
            for (int i = 0; i < K; ++i) {
                const uint4 w = rng_block(key, sweep, (KIND_MU << 16), (uint32_t)(i >> 1));
                zs[i] = (i & 1) ? normal_from<R>(w.z, w.w) : normal_from<R>(w.x, w.y);
            }
        }
        auto G = [&](int g) -> R { return __shfl_sync(kFull, gl[g / L], base_lane + g % L); };
#pragma unroll
        for (int i = 0; i < K; ++i) {
            const R gi = G(i);
            if (valid[i]) sig2[i] = post[i].b / gi; else ++events;     // :320 InverseGamma(a,b); reference: catch + keep old value (:321-329)
        }
#pragma unroll
        for (int i = 0; i < K; ++i) mu[i] = post[i].mean(c, hp.nu[i], hp.xi[i]) + post[i].sd(sig2[i], hp.nu[i]) * zs[i];   // :331-334
        {
            R tot = R(0);
#pragma unroll
            for (int i = 0; i < K; ++i) { rho[i] = G(K + i); tot += rho[i]; }
#pragma unroll
            for (int i = 0; i < K; ++i) rho[i] /= tot;
        }
#pragma unroll
        for (int i = 0; i < K; ++i) {
            R tot = R(0);
#pragma unroll
            for (int j = 0; j < K; ++j) { A[i][j] = G(2 * K + i * K + j); tot += A[i][j]; }
#pragma unroll
            for (int j = 0; j < K; ++j) A[i][j] /= tot;
        }
        return events;
    }

    template <typename V> static __device__ __forceinline__ V gsum(V v) {   // sum over the L lanes of a chain
#pragma unroll
        for (int o = 1; o < L; o <<= 1) v += __shfl_xor_sync(kFull, v, o);
        return v;
    }

    // the active warps of the block meet before the filter and before the sampler (see kSegThreads)
    static __device__ __forceinline__ void phase_barrier(const int nact) {
        if (nact > 32) asm volatile("bar.sync 1, %0;" ::"r"(nact) : "memory");
    }

    static __device__ __forceinline__ void run(const GibbsArgs& a, const int task, const int lane, const int nact) {
        const int q = lane % L;                                      // segment of this lane (0 = the end of the window)
        const int base_lane = lane - q;
        const int slot = task * kCPW + lane / L;
        const int ns = a.n_slots;
        const int T = a.T[slot];
        const int C = a.warp_T[task];
        // The segments of a chain depend on ITS window length alone (Cc rows each), whatever else shares the warp, so its
        // results are bit-identical in any batch; the warp's frame holds C >= Cc rows and shorter segments are right-aligned in it.
        const int Cc = T > 0 ? (T + 4 * L - 1) / (4 * L) * 4 : 4;
        Chain ch;
        {
            int n = T - q * Cc;
            n = n < 0 ? 0 : (n > Cc ? Cc : n);
            const int t_lo = T - q * Cc - n;
            ch.T = n; ch.Tw = C; ch.off = C - n;
            ch.yld = a.yld;
            ch.y0 = reinterpret_cast<const R*>(a.y) + a.ybase[slot] + (long long)(t_lo - ch.off) * ch.yld;
        }
        ch.rag_rows = (int)__reduce_max_sync(kFull, (unsigned)ch.off);   // (ragged only in the tiles before the start of the shortest segment)
        ch.pi0 = reinterpret_cast<R*>(a.pi) + a.warp_pi_off[task] + lane * 4;
        ch.pacc0 = nullptr; ch.facc0 = nullptr; ch.n_hi = 0; ch.mh_off = 0;
        const unsigned tab_byte = (unsigned)((threadIdx.x / kGibbsThreads) * (K * kGibbsThreads * sizeof(typename GW::Entry))
                                             + (threadIdx.x % kGibbsThreads) * sizeof(typename GW::Entry));
        ch.tab_s = (unsigned)__cvta_generic_to_shared(smem_base()) + tab_byte;
        // shared memory of a block of nt threads: selection tables | cp.async rings | realised future observations
        const unsigned nt = blockDim.x;
        const unsigned tab_total = (unsigned)(sizeof(typename GW::Entry) * K) * nt, ring_total = (unsigned)(sizeof(R) * kRing * 4 * K * 32) * (nt >> 5);
        ch.ring_off = tab_total + (unsigned)(sizeof(R) * (threadIdx.x >> 5) * (kRing * 4 * K * 32));
        ch.c = reinterpret_cast<const R*>(a.cshift)[slot];
        const unsigned yf_off = tab_total + ring_total + (unsigned)(threadIdx.x * sizeof(R));
        if (q == 0) {
            R* yf = reinterpret_cast<R*>(smem_base() + yf_off);
            for (int j = 0; j < a.n_h; ++j) yf[j * blockDim.x] = reinterpret_cast<const R*>(a.yfut)[(size_t)a.h_slot[j] * ns + slot];
        }
        const bool stream_y = a.yld != 1;
        const R totS = reinterpret_cast<const R*>(a.totS)[slot], totQ = reinterpret_cast<const R*>(a.totQ)[slot];
        const RngKey key{a.k0, a.k1, a.chain_id[slot]};
        R* __restrict__ const out = reinterpret_cast<R*>(a.out);

        // chain state: the L lanes of a chain hold the same copy
        int cnt[K], trans[K][K];
        R Sd[K], Qd[K], sig2[K], mu[K], rho[K];
        Hyper<R, K> hp;
        load_chain_stats<R, K>(a, ns, slot, cnt, Sd, Qd, trans, hp);
#pragma unroll
        for (int i = 0; i < K; ++i) sig2[i] = R(1);
        int events = 0;                                              // this lane's share (summed over the chain's lanes at the end)
        const int warm_steps = a.seg_warm;                           // time steps of warm-up in front of a segment (seg_warmup)

        for (int sw = 0; sw < a.n_sweeps; ++sw) {
            const long long gs = a.sweep0 + sw;
            const uint32_t sweep = (uint32_t)gs;
            // ---- 1. conjugate draws (identical in the L lanes of a chain: same statistics, same counters)
#pragma unroll
            for (int i = 0; i < K; ++i) hp.beta[i] = (R)(gs == 0 ? a.beta0[i] : a.beta[i]);
            {
                const int ev = draw_params_lanes(q, base_lane, cnt, Sd, Qd, trans, ch.c, hp, key, sweep, sig2, mu, rho, ch.A);
                if (q == 0) events += ev;
            }
            // ---- 2. forward filter
            if (a.seg_barriers > 0) phase_barrier(nact);
            Emission<R, K> em;
            em.prepare(mu, sig2);
            R pf[K], ll;
            {
                // entering vector by warm-up (see seg_warmup); t_lo = first time step of this segment
                const int t_lo = T - q * Cc - ch.T;
                const bool first_seg = (t_lo <= 0) || ch.T == 0;     // the window's earliest segment (or an empty one): starts from ρ
                const int W = first_seg ? 0 : (t_lo < warm_steps ? t_lo : warm_steps);
                const bool exact_start = first_seg || W == t_lo;     // the warm-up itself starts at t = 1 from ρ: exact
                Vec rv;
#pragma unroll
                for (int s = 0; s < K; ++s) rv.v[s] = exact_start ? rho[s] : R(1) / R(K);
                if (W > 0) rv = stream_y ? seg_warmup<true>(ch, em, rv, W) : seg_warmup<false>(ch, em, rv, W);
                FwdOut fo = stream_y ? GW::template forward_pass<true, false, true>(ch, em, rv) : GW::template forward_pass<true, false>(ch, em, rv);
                // verification: the vector this lane started from against the final row of the segment before it (lane q + 1)
                bool redo;
                {
                    R err = R(0);
#pragma unroll
                    for (int s = 0; s < K; ++s) {
                        const R prev = __shfl_sync(kFull, fo.pf.v[s], (lane + 1) & 31);
                        const R d = rv.v[s] - prev;
                        err = fmax(err, d < R(0) ? -d : d);
                    }
                    const bool mine_bad = !exact_start && !(err <= warm_tol());     // (a NaN fails the test)
                    redo = ((__ballot_sync(kFull, mine_bad) >> base_lane) & ((1u << L) - 1u)) != 0u;
                }
                R chk = fo.pf.v[0];
#pragma unroll
                for (int s = 1; s < K; ++s) chk += fo.pf.v[s];
                bool bad = ch.T > 0 && !(chk > R(0.5) && chk < R(2));
                if (__any_sync(kFull, redo)) {
                    // some chain of the warp failed the verification: exact entering vectors for it.  Phase 1: every lane of that
                    // chain multiplies the K x K matrices of its segment; phase 2: v_q = normalise(v_{q+1} M_{q+1}) along the chain
                    Mat M;
#pragma unroll
                    for (int i = 0; i < K; ++i)
#pragma unroll
                        for (int j = 0; j < K; ++j) M.m[i][j] = (i == j) ? R(1) : R(0);
                    M.bad = false;
                    if (redo) M = stream_y ? seg_product<true>(ch, em) : seg_product<false>(ch, em);
                    __syncwarp();
                    R vin[K], cur[K];
#pragma unroll
                    for (int s = 0; s < K; ++s) { vin[s] = rho[s]; cur[s] = rho[s]; }          // t = 1 uses ρ (:390)
#pragma unroll
                    for (int sq = L - 1; sq >= 1; --sq) {            // cur = vector leaving segment sq (sq = L-1 is the earliest)
                        R nx[K], tot = R(0);
#pragma unroll
                        for (int s = 0; s < K; ++s) nx[s] = R(0);
#pragma unroll
                        for (int r = 0; r < K; ++r)
#pragma unroll
                            for (int s = 0; s < K; ++s) nx[s] = fma(cur[r], __shfl_sync(kFull, M.m[r][s], base_lane + sq), nx[s]);
#pragma unroll
                        for (int s = 0; s < K; ++s) tot += nx[s];
                        const R inv = R(1) / tot;
#pragma unroll
                        for (int s = 0; s < K; ++s) cur[s] = nx[s] * inv;
                        if (q == sq - 1) {
#pragma unroll
                            for (int s = 0; s < K; ++s) vin[s] = cur[s];
                        }
                    }
                    if (redo) {
#pragma unroll
                        for (int s = 0; s < K; ++s) rv.v[s] = vin[s];
                        fo = stream_y ? GW::template forward_pass<true, false, true>(ch, em, rv) : GW::template forward_pass<true, false>(ch, em, rv);
                        chk = fo.pf.v[0];
#pragma unroll
                        for (int s = 1; s < K; ++s) chk += fo.pf.v[s];
                        bad = M.bad || (ch.T > 0 && !(chk > R(0.5) && chk < R(2)));
                        if (q == 0 && a.diag) atomicAdd(a.diag, 1ull);
                    }
                    __syncwarp();
                }
                if (__builtin_expect(__any_sync(kFull, bad), 0)) {
                    // a zero / non-finite normaliser somewhere in the warp (the reference only warns, :435): the segments are
                    // filtered again one after the other with per-step handling, each from the final row of the one before
                    R carry[K];
#pragma unroll
                    for (int s = 0; s < K; ++s) carry[s] = rho[s];
                    for (int sq = L - 1; sq >= 0; --sq) {
                        if (q == sq) {
#pragma unroll
                            for (int s = 0; s < K; ++s) rv.v[s] = carry[s];
                            fo = GW::template forward_pass<true, true>(ch, em, rv);
                            if (ch.T > 0) {
#pragma unroll
                                for (int s = 0; s < K; ++s) carry[s] = fo.pf.v[s];
                            }
                        }
                        __syncwarp();
#pragma unroll
                        for (int s = 0; s < K; ++s) carry[s] = __shfl_sync(kFull, carry[s], base_lane + sq);
                    }
                }
#pragma unroll
                for (int s = 0; s < K; ++s) pf[s] = fo.pf.v[s];
                ll = fo.ll;
                events += fo.events;
            }
            if (LOGLIK) ll = gsum(ch.T > 0 ? ll : R(0));
            // pf of the lane of segment 0 is pif[T,:] in chain labels

            // ---- 3. relabel (:501-513) and emit the draw in increasing-μ order (the lane of segment 0 writes)
            ranks_of<R, K>(mu, ch.rank);
            const long long draw_idx = gs - a.burnin;
            const bool save = (draw_idx >= 0) && (T > 0) && (q == 0);
            if (save) {
                const size_t i = (size_t)(draw_idx - a.draw0);
                const size_t cs = (size_t)a.chunk * ns;
                R* o = out + i * ns + slot;
#pragma unroll
                for (int s = 0; s < K; ++s) {
                    o[(size_t)(ch.rank[s]) * cs] = mu[s];
                    o[(size_t)(K + ch.rank[s]) * cs] = sig2[s];
                    o[(size_t)(2 * K + K * K + ch.rank[s]) * cs] = pf[s];
#pragma unroll
                    for (int r = 0; r < K; ++r) o[(size_t)(2 * K + ch.rank[s] * K + ch.rank[r]) * cs] = ch.A[r][s];
                }
                const int f0 = 3 * K + K * K;
                R v[K];
#pragma unroll
                for (int s = 0; s < K; ++s) v[s] = pf[s];
                int h = 0;
                for (int j = 0; j < a.n_h; ++j) {                    // forecasts pib_T' A^h μ (:658-667, :858-862)
                    for (; h < a.h_sorted[j]; ++h) {
                        R nv[K];
#pragma unroll
                        for (int s = 0; s < K; ++s) {
                            R acc = v[0] * ch.A[0][s];
#pragma unroll
                            for (int r = 1; r < K; ++r) acc = fma(v[r], ch.A[r][s], acc);
                            nv[s] = acc;
                        }
#pragma unroll
                        for (int s = 0; s < K; ++s) v[s] = nv[s];
                    }
                    R f = v[0] * mu[0];
#pragma unroll
                    for (int s = 1; s < K; ++s) f = fma(v[s], mu[s], f);
                    const R yr = reinterpret_cast<const R*>(smem_base() + yf_off)[j * blockDim.x];
                    o[(size_t)(f0 + 2 * a.h_slot[j]) * cs] = f;
                    o[(size_t)(f0 + 2 * a.h_slot[j] + 1) * cs] = f - yr;
                }
                if (LOGLIK) o[(size_t)(f0 + 2 * a.n_h) * cs] = ll;
            }
            __syncwarp();

            // ---- 4. backward sampling + the next sweep's statistics
            if (a.seg_barriers > 1) phase_barrier(nact);
            {
                typename GW::Entry* tab = reinterpret_cast<typename GW::Entry*>(smem_base() + tab_byte);
#pragma unroll
                for (int xx = 0; xx < K; ++xx) {                     // this thread's private selection table (GibbsWarp::select_later)
                    typename GW::Entry en;
#pragma unroll
                    for (int r = 0; r < K; ++r) en.a[r] = ch.A[r][xx];
                    en.inc = 1u << (kBits * xx);
                    tab[xx * kGibbsThreads] = en;
                }
            }
            Vec pv;
#pragma unroll
            for (int s = 0; s < K; ++s) pv.v[s] = pf[s];
            const BackOut bo = stream_y ? seg_backward<true>(ch, pv, key, sweep, a.flags, q, Cc, a.diag) : seg_backward<false>(ch, pv, key, sweep, a.flags, q, Cc, a.diag);
            {
                R sS = R(0), sQ = R(0);
#pragma unroll
                for (int i = 0; i < K; ++i) {
                    int nocc = (T > 0 && bo.xN == i) ? 1 : 0;
#pragma unroll
                    for (int j = 0; j < K; ++j) {
                        trans[i][j] = gsum((int)((bo.row[i] >> (kBits * j)) & kFieldMask));
                        nocc += trans[i][j];
                    }
                    cnt[i] = nocc;
                }
#pragma unroll
                for (int i = 0; i < K - 1; ++i) { Sd[i] = gsum(bo.Sd[i]); Qd[i] = gsum(bo.Qd[i]); sS += Sd[i]; sQ += Qd[i]; }
                Sd[K - 1] = totS - sS; Qd[K - 1] = totQ - sQ;
                if (cnt[K - 1] == 0) { Sd[K - 1] = R(0); Qd[K - 1] = R(0); }
            }
        }

        events = gsum(events);
        if (q == 0) store_chain_stats<R, K>(a, ns, slot, cnt, Sd, Qd, trans, events);
    }
};

template <typename R, int K, int L, bool LOGLIK>
__global__ void __launch_bounds__(kSegThreads, (sizeof(R) == 8 ? 384 : 512) / kSegThreads) gibbs_seg_kernel(const GibbsArgs a) {
    const int lane = threadIdx.x & 31;
    const int wpb = (int)(blockDim.x >> 5);                          // the host picks 128 or 256 threads (launch_gibbs_seg)
    const int g0 = blockIdx.x * wpb;
    const int g = g0 + (threadIdx.x >> 5);
    if (g >= a.n_tasks) return;
    const int nact = 32 * min(wpb, a.n_tasks - g0);                  // threads of this block that have a task (they meet at the phase barriers)
    SegWarp<R, K, L, LOGLIK>::run(a, a.task0 + g * a.task_stride, lane, nact);
}

// lanes per chain; a warp task holds 32 / lanes chains (plan.seg_lanes); threads per block (<= kSegThreads)
template <typename R, int K> cudaError_t launch_gibbs_seg(const GibbsLaunch& cfg, const GibbsArgs& a, int lanes, int threads, cudaStream_t st);

}  // namespace hmc
