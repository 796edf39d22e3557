// plan_policy.cuh — what a plan runs, decided on the host: the sweep kernel (choose_sweep), the chain slots and warp tasks
// (layout_slots), the draw chunks (draw_chunks) and the order of the sweep launches and per-chunk post-processing
// (launch_schedule).  Plain C++17 without CUDA, so that g++ compiles it too and tests/test_plan_policy.py checks the policy
// and the schedule on the CPU; hmcgpu.cu issues what it decides.
#pragma once
#include "../../include/hmcgpu.h"

#include <algorithm>
#include <cstddef>
#include <cstdint>
#include <cstdlib>
#include <numeric>
#include <optional>
#include <vector>

namespace hmc {

// threads per block of the warp-per-chain kernel (gibbs_scan_kernel.cuh): 4 chains per block
constexpr int kScanThreads = 128;

// Threads per block of the segment kernel (gibbs_seg_kernel.cuh).  The warps of a block step through the phases of a sweep
// together (two named barriers per sweep): a scheduler then holds warps that run the SAME loop, which keeps that loop in the
// ~6 KB L0 instruction cache.  Without the alignment the four warps of a scheduler sit in different loops (filter, sampler,
// draws, ...), every 128-byte line of every loop misses L0 and the kernel spends 2.5 cycles per issued instruction waiting
// for instructions (ncu stall_no_instruction).
#ifndef HMC_SEG_THREADS
#define HMC_SEG_THREADS 256
#endif
constexpr int kSegThreads = HMC_SEG_THREADS;

// largest window the scan kernel can hold in shared memory (4 chains per block); precision 32 or 64
constexpr int scan_max_T(int precision, int K) { return (200 * 1024 / (kScanThreads / 32) - 64) / (precision / 8 * (K + 1)); }
// longest window the segment kernel takes with this many lanes per chain (packed 32-bit transition counters per segment)
constexpr long long seg_max_T(int K, int lanes) { return (long long)lanes * (((1ll << (32 / K)) - 1) / 4 * 4); }

// The HMCGPU_* tuning variables (INTEGRATION.md), read once per plan at hmcgpu_plan_create.  An unset optional leaves the
// choice to the plan; the bools are "value != 0".
struct Tuning {
    bool lane_kernel = false, seg_mixed = true, y_smem = true, launch_timing = true, verbose = false;
    int seg_warm = 32, seg_barriers = 2;
    std::optional<long long> scan_max_chains, seg_long;
    std::optional<int> seg_lanes, groups, seg_threads, sweeps_per_launch;
    // HMCGPU_FLAG_LOO: the fetch scratch of one batch of dates (ell, F and the backward vectors), HMCGPU_LOO_SCRATCH_MB; a smaller
    // bound only cuts the dates into more batches, whose outputs are the same bit for bit
    size_t loo_scratch = 4ull << 30;
};
inline Tuning read_tuning() {
    Tuning t;
    const char* e;
    if ((e = getenv("HMCGPU_LANE_KERNEL"))) t.lane_kernel = atoi(e) != 0;
    if ((e = getenv("HMCGPU_SCAN_MAX_CHAINS"))) t.scan_max_chains = atoll(e);
    if ((e = getenv("HMCGPU_SEG_LANES"))) t.seg_lanes = atoi(e);
    if ((e = getenv("HMCGPU_SEG_MIXED"))) t.seg_mixed = atoi(e) != 0;
    if ((e = getenv("HMCGPU_SEG_LONG"))) t.seg_long = atoll(e);
    if ((e = getenv("HMCGPU_GROUPS"))) t.groups = std::max(1, std::min(8, atoi(e)));
    if ((e = getenv("HMCGPU_Y_SMEM"))) t.y_smem = atoi(e) != 0;
    if ((e = getenv("HMCGPU_SEG_WARMUP"))) t.seg_warm = std::max(0, atoi(e));
    if ((e = getenv("HMCGPU_SEG_BARRIERS"))) t.seg_barriers = atoi(e);
    if ((e = getenv("HMCGPU_SEG_THREADS"))) t.seg_threads = atoi(e);
    if ((e = getenv("HMCGPU_SWEEPS_PER_LAUNCH"))) t.sweeps_per_launch = std::max(1, atoi(e));
    if ((e = getenv("HMCGPU_LAUNCH_TIMING"))) t.launch_timing = atoi(e) != 0;
    if ((e = getenv("HMCGPU_VERBOSE"))) t.verbose = atoi(e) != 0;
    if ((e = getenv("HMCGPU_LOO_SCRATCH_MB"))) t.loo_scratch = (size_t)std::max(1LL, atoll(e)) << 20;
    return t;
}

// sweeps: thread-per-chain kernels for K = 2..8, lane-per-state kernel for K = 9..32 (HMCGPU_LANE_KERNEL=1: also for 5..8)
inline bool k_thread_sweep(int K, const Tuning& t) { return (K >= 2 && K <= 4) || (K >= 5 && K <= 8 && !t.lane_kernel); }

enum class SweepKernel : int32_t { thread = HMCGPU_KERNEL_THREAD, scan = HMCGPU_KERNEL_SCAN, lane = HMCGPU_KERNEL_LANE, seg = HMCGPU_KERNEL_SEG };

// Which sweep kernel a plan runs, and how (choose_sweep)
struct SweepChoice {
    SweepKernel kernel = SweepKernel::thread;
    int seg_lanes = 0;           // segment kernel: L lanes per chain (a warp task holds 32 / L chains)
    // Mixed segment counts (mid-width batches with spare thread slots): the n_long longest windows run with 8 lanes per chain,
    // in their own slot range with their own warp-task tables (task id = slot / 4)
    int n_long = 0;
    int sweeps_per_launch = 16;
    int seg_threads = 128;       // threads per block of the segment kernel
};

// The sweep-kernel policy (SweepChoice) on a device of sm_count SMs.  wT / order: the window lengths and the windows by
// decreasing length.  Returns HMCGPU_OK, or an error code with *err set to its message.
inline int choose_sweep(int sm_count, const hmcgpu_problem* p, const std::vector<int>& wT, const std::vector<int>& order,
                        const Tuning& t, SweepChoice& c, const char** err) {
    const int K = p->K, nw = p->n_windows, nc = p->n_chains, max_T = wT[order[0]];
    const bool sig = p->is_signal != nullptr || p->pi_row_back != 0;
    const bool acc_mean = p->flags & (HMCGPU_FLAG_SMOOTHED_MEAN | HMCGPU_FLAG_FILTERED_MEAN);   // per-date means: thread-per-chain kernels only
    const long long n_real = (long long)nw * nc;
    const long long full = (long long)sm_count * 16 * 32;          // one wave of thread slots (16 warps per SM)
    c = SweepChoice{};
    if (!k_thread_sweep(K, t)) c.kernel = SweepKernel::lane;
    if (K <= 4 && !acc_mean) {
        // Narrow batches (the reference's own regime: one chain per end date) cannot fill the GPU with a thread per chain:
        // below kScanMaxChains chains the time-parallel warp-per-chain kernel is used (K <= 4, plain sweep, window in smem).
        // (the signals tier has no segment kernel: there the warp-per-chain kernel serves up to 12 288 chains; for the plain
        //  sweep the segment kernel takes over from ~4000 chains — measured crossover on C2, DESIGN.md section 7)
        const bool seg_ok = !sig && !(t.seg_lanes && *t.seg_lanes == 0);
        long long lim = t.scan_max_chains.value_or(seg_ok ? 4096 : 12288);
        // long windows leave room for fewer resident warps (the window lives in shared memory): scale the bound with them
        const size_t wb = (size_t)(p->precision / 8) * ((size_t)max_T * (K + 1) + 4 * K);
        const long long blocks = std::max<long long>(1, std::min<long long>(5, (long long)((227 * 1024) / (4 * wb + 1024))));
        lim = lim * blocks / 5;
        if (n_real <= lim && max_T <= scan_max_T(p->precision, K)) c.kernel = SweepKernel::scan;
    }
    // Mid-width batches (too many chains for a warp each, too few to fill the schedulers with a thread each): L lanes per
    // chain, one time segment per lane (gibbs_seg_kernel.cuh).  L is chosen so that the batch yields about one full wave of
    // warps; HMCGPU_SEG_LANES forces it (0 = never).  K <= 4, plain sweep.
    if (K <= 4 && !acc_mean && !sig && c.kernel != SweepKernel::scan) {
        int lanes = 0;
        // measured on C2 (500 windows x c chains, B200): 4 lanes per chain are best up to ~38 000 chains, 2 lanes up to ~90 000,
        // the thread-per-chain kernel beyond (DESIGN.md section 7); in units of one wave of thread slots:
        if (n_real * 2 <= full) lanes = 4;
        // (2 lanes only when the chains share one series: a batch of distinct series streams every observation from HBM in each
        //  of the segment kernel's passes — C4, 65 536 series: 143 ms with 2 lanes, 139 ms with 4, 109 ms with a thread per chain)
        else if (n_real * 4 <= 5 * full && p->n_series == 1) lanes = 2;
        if (t.seg_lanes) lanes = *t.seg_lanes;
        if (lanes != 0 && lanes != 2 && lanes != 4 && lanes != 8) {
            *err = "HMCGPU_SEG_LANES must be 0, 2, 4 or 8";
            return HMCGPU_ERR_ARG;
        }
        if (lanes && max_T > seg_max_T(K, lanes)) lanes = 0;
        if (lanes) c.kernel = SweepKernel::seg;
        c.seg_lanes = lanes;
        // With 4 lanes per chain and thread slots to spare, the sweep time is the serial time of the LONGEST windows (every warp is
        // resident from the start; a 16 000-chain batch leaves a fifth of the slots empty).  The longest tenth of the windows (in
        // `order`) then gets 8 lanes per chain — half the dependent steps per sweep — as far as the slots last.  Measured on C2
        // (HMCGPU_SEG_LONG sweep, scripts/r2_call_j.sh): 50 of 500 windows +7 % at 16 chains per window, +2 % at 24, +4 % at 32;
        // 100 windows +7 % at 32 but -5 % at 24; 300 or all of them lose everywhere (8 lanes pay more per-sweep work per chain).
        // HMCGPU_SEG_MIXED=0 disables it; a forced HMCGPU_SEG_LANES is uniform.
        if (lanes == 4 && !t.seg_lanes && t.seg_mixed) {
            const long long spare = full * 115 / 100 - n_real * 4;
            long long n8 = spare > 0 ? std::min<long long>(nw / 10, spare / ((long long)nc * 4)) : 0;
            while (n8 > 0 && wT[order[n8 - 1]] < 128) --n8;          // (segments of fewer than 16 steps are all warm-up)
            if (t.seg_long) n8 = std::max(0ll, std::min<long long>(nw, *t.seg_long));
            if (n8 * nc >= 32 && max_T <= seg_max_T(K, 8)) c.n_long = (int)n8;
        }
    }
    if (c.kernel == SweepKernel::seg) {
        // 256-thread blocks (8 warps stepping through the phases of a sweep together) when that still gives every SM a block
        // and a half; otherwise 128.  Warp tasks: 4 chains each in the long class, 32 / L in the rest, each class padded to 32.
        const long long n8c = (long long)c.n_long * nc, tasks = (n8c + 31) / 32 * 8 + (n_real - n8c + 31) / 32 * c.seg_lanes;
        c.seg_threads = t.seg_threads.value_or(tasks / (kSegThreads / 32) >= sm_count * 3 / 2 ? kSegThreads : 128);
    }
    // Sweeps per launch.  Short launches bound the damage of the priority-based warp arbiter (a starved warp can only fall
    // behind by one launch) and give the block scheduler a steady supply of pending blocks from the other groups.  A scan
    // sweep is a few µs.
    c.sweeps_per_launch = t.sweeps_per_launch.value_or(c.kernel == SweepKernel::scan ? 64 : 16);
    return HMCGPU_OK;
}

// An interleaved subset of the (longest-first) warp tasks of a class, driven through its own stream: tasks task0,
// task0 + stride, ... (n_tasks of them), with `lanes` lanes per chain
struct TaskGroup { int task0, stride, n_tasks, lanes; bool long_class; };

// Host tables of the chain slots and warp tasks (uploaded by plan_build), and the task groups
struct SlotLayout {
    std::vector<int> slot_win, slot_chain, Ts, win_slot0, warp_T, warp_T_long;
    std::vector<long long> ybase, warp_off, warp_off_long, slot_off;   // slot_off: the lane kernel's pi row of each slot
    std::vector<unsigned> chain_id;
    long long pi_elems = 0;
    int n_slots = 0, n_warps = 0, n_tasks = 0;                         // (n_tasks: warp tasks of both classes)
    std::vector<TaskGroup> groups;
};

// Lays out the chain slots, warp tasks, pi offsets and task groups of a plan for its SweepChoice c.  wT / order as for
// choose_sweep.
inline SlotLayout layout_slots(const hmcgpu_problem* p, const std::vector<int>& wT, const std::vector<int>& order,
                               const SweepChoice& c, const Tuning& t) {
    const int K = p->K, nw = p->n_windows, nc = p->n_chains, nser = p->n_series;
    const bool seg = c.kernel == SweepKernel::seg;
    const int ts = 32;
    // slots: windows by decreasing T, chains consecutive; [long class (8 lanes), padded to 32][the rest, padded to 32]
    const int long_slots = (int)(((long long)c.n_long * nc + ts - 1) / ts * ts);
    const int n_slots = long_slots + (int)(((long long)nw * nc - (long long)c.n_long * nc + ts - 1) / ts * ts);
    const int cpt = seg ? 32 / c.seg_lanes : ts;            // chains per warp task
    const int n_warps = n_slots / cpt;                      // number of warp tasks (task id = slot / cpt; ids below long_slots / cpt are unused when there is a long class)
    SlotLayout s;
    s.n_slots = n_slots; s.n_warps = n_warps;
    s.slot_win.assign(n_slots, -1); s.slot_chain.assign(n_slots, 0); s.Ts.assign(n_slots, 0); s.ybase.assign(n_slots, 0);
    s.chain_id.assign(n_slots, 0); s.slot_off.assign(n_slots, 0); s.win_slot0.assign(nw, 0);
    s.warp_T.assign(n_warps, 0); s.warp_off.assign(n_warps, 0);
    for (int j = 0; j < nw; ++j) {
        const int w = order[j];
        const int s0w = j < c.n_long ? j * nc : long_slots + (j - c.n_long) * nc;
        s.win_slot0[w] = s0w;
        const unsigned long long wid = p->win_id ? (unsigned long long)p->win_id[w] : (unsigned long long)w;
        for (int cidx = 0; cidx < nc; ++cidx) {
            const int slot = s0w + cidx;
            s.slot_win[slot] = w; s.slot_chain[slot] = cidx; s.Ts[slot] = wT[w];
            s.ybase[slot] = (long long)(p->win_start[w] - 1) * nser + (p->win_series ? p->win_series[w] : 0);   // time-major [y_len][n_series] (the sweeps)
            s.chain_id[slot] = (unsigned)(wid * (unsigned long long)nc + (unsigned long long)cidx);
        }
    }
    // the long class first (8 lanes per chain: 4 chains per task, task id = slot / 4)
    s.warp_T_long.assign(long_slots / 4, 0);
    s.warp_off_long.assign(long_slots / 4, 0);
    for (int wp = 0; wp < long_slots / 4; ++wp) {
        int m = 0;
        for (int l = 0; l < 4; ++l) m = std::max(m, s.Ts[wp * 4 + l]);
        const int Cs = std::max(4, (m + 31) / 32 * 4);
        s.warp_T_long[wp] = Cs;
        s.warp_off_long[wp] = s.pi_elems;
        s.pi_elems += (long long)Cs * K * 32;
    }
    for (int wp = long_slots / cpt; wp < n_warps; ++wp) {
        int m = 0;
        for (int l = 0; l < cpt; ++l) m = std::max(m, s.Ts[wp * cpt + l]);
        s.warp_T[wp] = m;
        s.warp_off[wp] = s.pi_elems;
        if (seg) {
            // segment kernel: every lane owns a frame of C = 4 ceil(T / 4L) rows (warp_T holds C), tiled like the thread kernel's
            const int Cs = std::max(4, (m + 4 * c.seg_lanes - 1) / (4 * c.seg_lanes) * 4);
            s.warp_T[wp] = Cs;
            s.pi_elems += (long long)Cs * K * 32;
        }
        // thread-per-chain kernels: rows right-aligned to tiles of 4 time steps (gibbs_kernel.cuh, st_quad)
        else if (c.kernel != SweepKernel::lane) s.pi_elems += (long long)((m + 3) / 4 * 4) * K * ts;
        else for (int l = 0; l < ts; ++l) { s.slot_off[wp * ts + l] = s.pi_elems; s.pi_elems += (long long)s.Ts[wp * ts + l] * K; }
    }
    // task groups: interleaved subsets of the (longest-first) warp tasks of a class, each driven through its own stream
    auto add_groups = [&](int task0, int tasks, int lanes, bool long_class) {
        if (tasks <= 0) return;
        int g = t.groups.value_or((c.kernel == SweepKernel::lane || c.kernel == SweepKernel::scan) ? 1 : (tasks >= 1024 ? 4 : (tasks >= 256 ? 2 : 1)));
        g = std::max(1, std::min(g, tasks));
        for (int q = 0; q < g; ++q) s.groups.push_back({task0 + q, g, (tasks - q + g - 1) / g, lanes, long_class});
    };
    const int t_long = long_slots / 4, t_first = long_slots / cpt, t_rest = n_warps - t_first;
    add_groups(0, t_long, 8, true);
    add_groups(t_first, t_rest, c.seg_lanes, false);
    s.n_tasks = t_long + t_rest;
    return s;
}

// Draws per chunk buffer and the number of buffers
struct DrawChunks { int chunk, n_bufs; };

// F fields per draw of n_slots slots of elem_bytes each.  Double-buffered draw chunks let the groups drift apart (not with the
// smoothing accumulators, which are shared); the chunk buffers are bounded to ~2 GiB in total.
inline DrawChunks draw_chunks(int n_groups, unsigned flags, int F, int n_slots, size_t elem_bytes, long long nrun) {
    const unsigned kAccMean = HMCGPU_FLAG_SMOOTHED_MEAN | HMCGPU_FLAG_FILTERED_MEAN;
    const int n_bufs = (n_groups > 1 && !(flags & kAccMean)) ? 2 : 1;
    const size_t per_draw = (size_t)F * n_slots * elem_bytes;
    long long chunk = std::max<long long>(1, (long long)((2ull << 30) / n_bufs / per_draw));
    chunk = std::min<long long>(chunk, std::min<long long>(nrun, 1024));
    return {(int)chunk, n_bufs};
}

// One operation of a plan run, in enqueue order: a sweep launch of a task group, or the post-processing of a draw chunk
struct RunOp {
    bool post;                // false: a sweep launch; true: the post-processing of draw chunk `chunk`
    int group;                // (launch) its task group
    long long sweep0, n_sweeps;
    long long chunk;          // the draw chunk the launch writes (-1 during burn-in), or the chunk posted
    long long wait;           // (launch) the chunk whose post-processing must have released its buffer first, or -1
    bool closes_chunk;        // (launch) the group's last launch into `chunk`
    bool last;                // (launch) the group's last launch
};

// The launches of a run of burnin + nrun sweeps over n_groups task groups (sweeps_per_launch sweeps each) and the
// post-processing of its draw chunks (chunk draws each, in n_bufs buffers used in turn).  Launches go round-robin over the
// groups, laggards first; the first launch of group g is (g+1)/G of a normal one, so that the groups' launch boundaries
// interleave.  A launch never crosses the end of burn-in or of a draw chunk.  A group whose next chunk's buffer has not been
// released by the post-processing of chunk k - n_bufs sits the round out.  A chunk is post-processed as soon as every group
// has closed it.
inline std::vector<RunOp> launch_schedule(long long burnin, long long nrun, long long chunk, int n_bufs, int n_groups,
                                          int sweeps_per_launch) {
    const int G = n_groups, L = sweeps_per_launch;
    const long long S = burnin + nrun, n_chunks = (nrun + chunk - 1) / chunk;
    std::vector<RunOp> ops;
    std::vector<long long> next(G, 0);                       // next sweep of each group
    std::vector<std::vector<char>> closed(n_chunks, std::vector<char>(G, 0));
    long long posted = 0;                                    // chunks whose post-processing has been scheduled
    bool more = true;
    for (long long round = 0; more; ++round) {
        more = false;
        std::vector<int> gorder(G);
        std::iota(gorder.begin(), gorder.end(), 0);
        std::stable_sort(gorder.begin(), gorder.end(), [&](int x, int y) { return next[x] < next[y]; });   // laggards first
        for (int g : gorder) {
            const long long s0 = next[g];
            if (s0 >= S) continue;
            more = true;
            RunOp op{false, g, s0, 0, -1, -1, false, false};
            if (s0 >= burnin) {
                op.chunk = (s0 - burnin) / chunk;
                if ((s0 - burnin) % chunk == 0 && op.chunk >= n_bufs) {
                    op.wait = op.chunk - n_bufs;
                    if (op.wait >= posted) continue;         // buffer not released yet: next round
                }
            }
            long long n = (round == 0 && G > 1) ? std::max<long long>(1, (long long)L * (g + 1) / G) : L;
            const long long limit = s0 < burnin ? burnin : burnin + std::min<long long>(nrun, (op.chunk + 1) * chunk);
            op.n_sweeps = std::min(n, limit - s0);
            next[g] = s0 + op.n_sweeps;
            op.last = next[g] >= S;
            op.closes_chunk = op.chunk >= 0 && next[g] == limit;
            ops.push_back(op);
            if (op.closes_chunk) closed[op.chunk][g] = 1;
            // post-process every chunk all groups have closed
            while (posted < n_chunks && std::all_of(closed[posted].begin(), closed[posted].end(), [](char x) { return x != 0; }))
                ops.push_back(RunOp{true, -1, 0, 0, posted++, -1, false, false});
        }
    }
    return ops;
}

}  // namespace hmc
