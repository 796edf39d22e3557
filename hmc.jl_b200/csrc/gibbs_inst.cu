// gibbs_inst.cu — one explicit instantiation of the Gibbs sweep kernel family per translation unit:
// compiled with -DHMC_R=<float|double> -DHMC_K=<2|3|4> (hmc.jl_b200/build.py builds the six units in parallel).
#include <algorithm>
#include "gibbs_kernel.cuh"
#if HMC_K <= 4
#include "gibbs_scan_kernel.cuh"
#include "gibbs_seg_kernel.cuh"
#endif

namespace hmc {

// calls f(kernel) with the variant the flags / window length select
template <typename R, int K, bool WIDE, typename F> static auto with_variant(const GibbsLaunch& cfg, F f) {
    const bool smooth = cfg.flags & 8u /*HMCGPU_FLAG_SMOOTHED_MEAN*/, ll = cfg.flags & 16u /*HMCGPU_FLAG_LOGLIK*/;
    if constexpr (K > 4) {   // K = 5..8: the plain sweep and the smoothed means (the host rejects signals for K > 4)
        if (smooth && ll) return f(gibbs_sweeps_kernel<R, K, true, true, WIDE>);
        if (smooth) return f(gibbs_sweeps_kernel<R, K, true, false, WIDE>);
        if (ll) return f(gibbs_sweeps_kernel<R, K, false, true, WIDE>);
        return f(gibbs_sweeps_kernel<R, K, false, false, WIDE>);
    } else {
    if (cfg.sig) {   // signals tier (mask, kappa-weighted statistics, pi_row_back); never combined with the smoothed means
        if (ll) return f(gibbs_sweeps_kernel<R, K, false, true, WIDE, true>);
        return f(gibbs_sweeps_kernel<R, K, false, false, WIDE, true>);
    }
    if (smooth && ll) return f(gibbs_sweeps_kernel<R, K, true, true, WIDE>);
    if (smooth) return f(gibbs_sweeps_kernel<R, K, true, false, WIDE>);
    if (ll) return f(gibbs_sweeps_kernel<R, K, false, true, WIDE>);
    return f(gibbs_sweeps_kernel<R, K, false, false, WIDE>);
    }
}
// packed transition counters: 32-bit rows hold fields of 32/K bits; longer windows use 64-bit rows
template <int K> static bool wide_rows(const GibbsLaunch& cfg) { return (long long)cfg.max_T - 1 > TransPack<K, false>::kMaxT; }
template <typename R, int K, typename F> static auto with_rows(const GibbsLaunch& cfg, F f) {
    if constexpr (K > 4) return with_variant<R, K, true>(cfg, f);        // always 64-bit rows, flushed
    else {
        if (wide_rows<K>(cfg)) return with_variant<R, K, true>(cfg, f);
        return with_variant<R, K, false>(cfg, f);
    }
}

template <typename R, int K> cudaError_t launch_gibbs(const GibbsLaunch& cfg, const GibbsArgs& a, cudaStream_t st) {
    const unsigned grid = (unsigned)((a.n_tasks + kGibbsThreads / 32 - 1) / (kGibbsThreads / 32));
    auto go = [&](auto kern, size_t smem) -> cudaError_t {
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        kern<<<grid, kGibbsThreads, smem, st>>>(a);
        return cudaGetLastError();
    };
    const bool smooth = cfg.flags & (8u | 64u);   // smoothed or filtered means: the A^h mu vectors of the in-sample forecasts live in shared memory
    const bool wr = K > 4 || wide_rows<K>(cfg);
    const size_t ysm = a.y_sm_elems > 0 ? ((size_t)a.y_sm_elems * sizeof(R) + 15) / 16 * 16 : 0;   // the block's copy of the one series
    const size_t smem = (wr ? gibbs_smem_bytes<R, K, true>(smooth, cfg.n_h) : gibbs_smem_bytes<R, K, false>(smooth, cfg.n_h)) + ysm;
    return with_rows<R, K>(cfg, [&](auto kern) { return go(kern, smem); });
}

template cudaError_t launch_gibbs<HMC_R, HMC_K>(const GibbsLaunch&, const GibbsArgs&, cudaStream_t);

#if HMC_K <= 4
// narrow batches: one warp per chain, time-parallel (gibbs_scan_kernel.cuh); covers every slot in one launch
template <typename R, int K> cudaError_t launch_gibbs_scan(const GibbsLaunch& cfg, const GibbsArgs& a, cudaStream_t st) {
    const unsigned grid = (unsigned)((a.n_slots + kScanThreads / 32 - 1) / (kScanThreads / 32));
    const size_t smem = (kScanThreads / 32) * scan_warp_bytes<R, K>(cfg.max_T);
    auto go = [&](auto kern) -> cudaError_t {
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        kern<<<grid, kScanThreads, smem, st>>>(a, cfg.max_T);
        return cudaGetLastError();
    };
    if (cfg.sig) {
        if (cfg.flags & 16u) return go(gibbs_scan_kernel<R, K, true, true>);
        return go(gibbs_scan_kernel<R, K, false, true>);
    }
    if (cfg.flags & 16u) return go(gibbs_scan_kernel<R, K, true>);
    return go(gibbs_scan_kernel<R, K, false>);
}
template cudaError_t launch_gibbs_scan<HMC_R, HMC_K>(const GibbsLaunch&, const GibbsArgs&, cudaStream_t);

// mid-width batches: `lanes` lanes per chain, one time segment per lane (gibbs_seg_kernel.cuh); a task is 32 / lanes chains
template <typename R, int K> cudaError_t launch_gibbs_seg(const GibbsLaunch& cfg, const GibbsArgs& a, int lanes, int threads, cudaStream_t st) {
    if (threads != 128 && threads != kSegThreads) return cudaErrorInvalidValue;
    const unsigned grid = (unsigned)((a.n_tasks + threads / 32 - 1) / (threads / 32));
    const size_t smem = seg_smem_bytes<R, K>(cfg.n_h, threads);
    const bool ll = cfg.flags & 16u;
    auto go = [&](auto kern) -> cudaError_t {
        if (smem > 48 * 1024) {
            cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
        }
        kern<<<grid, threads, smem, st>>>(a);
        return cudaGetLastError();
    };
    switch (lanes) {
        case 2: return ll ? go(gibbs_seg_kernel<R, K, 2, true>) : go(gibbs_seg_kernel<R, K, 2, false>);
        case 4: return ll ? go(gibbs_seg_kernel<R, K, 4, true>) : go(gibbs_seg_kernel<R, K, 4, false>);
        case 8: return ll ? go(gibbs_seg_kernel<R, K, 8, true>) : go(gibbs_seg_kernel<R, K, 8, false>);
        default: return cudaErrorInvalidValue;
    }
}
template cudaError_t launch_gibbs_seg<HMC_R, HMC_K>(const GibbsLaunch&, const GibbsArgs&, int, int, cudaStream_t);
#endif

}  // namespace hmc
