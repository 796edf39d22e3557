// ranked.cuh — exact posterior quantiles, rank-normalised split-R̂ and bulk / tail ESS per (window, field)
// (HMCGPU_FLAG_RANKED), from every saved draw kept on the device.
//
// plan_run copies each draw chunk out of the per-chunk buffer out[(f*chunk + i)*n_slots + slot] into the retained buffer
//   keep[((w*F + f)*n_chains + c)*nrun + i]
// so that the R = n_chains*nrun draws of a (window, field) form one contiguous segment.  hmcgpu_plan_fetch_ranked then works
// through batches of segments (bounded scratch):
//   1. order-preserving 64-bit keys of the draws as doubles (-0 made +0), sorted per segment with their positions (CUB's stable
//      segmented radix sort);
//   2. from the sorted segment: the requested quantiles and q(0.05), q(0.5), q(0.95) (type 7), and the average rank r of every
//      draw (the run of equal keys around its sorted position), written back at the draw's position as the normal score
//      z = Phi^-1((r - 3/8) / (R + 1/4));
//   3. the split statistics of a transformed sequence (z, the indicators 1[x <= q(0.05)] and 1[x <= q(0.95)]): per chain and
//      half the mean, the variance and the centred lag sums G_l (l = 0..63), computed in two passes on the resident data, and
//      G_l summed over the chains in chain order, in the layout diag_finish_kernel (diagnostics.cuh) reads;
//   4. the same keys, sort and ranks for |x - q(0.5)| (fp64) give the folded normal scores and their statistics.
// diag_finish_kernel turns each of the four into R̂ / ESS, and ranked_combine_kernel forms rhat_rank = max(bulk, folded),
// ess_bulk and ess_tail = min(tail 5 %, tail 95 %).
//
// Every computation belongs to one segment, and every sum runs in a fixed order (within a sequence, then over the chains in
// chain order) with no atomics: a window's outputs are bit-identical however the windows are batched, chunked or sharded.
// tests/test_ranked.py holds the numpy definition it matches.
#pragma once
#include <cuda_runtime.h>
#include <cub/device/device_segmented_radix_sort.cuh>
#include "diagnostics.cuh"

namespace hmc {

constexpr int kRankedMaxProbs = 64;
constexpr int kRankedQuants = 3;            // q(0.05), q(0.5), q(0.95): the tail indicators and the fold
constexpr int kRankedSeqWarps = 8;          // warps (sequences) per block of ranked_stats_kernel

// Retention: draws [d0, d0 + n_i) of a chunk, per (window, field) block, through a 32 x 32 shared tile (reads along the
// slots, writes along the draws).  Block (32, 8), grid (n_windows, F).
template <typename R>
__global__ void __launch_bounds__(256) ranked_keep_kernel(int F, int n_slots, int chunk, int n_i, long long d0, long long nrun,
                                                          int n_chains, const int* __restrict__ win_slot0,
                                                          const R* __restrict__ out, R* __restrict__ keep) {
    __shared__ R tile[32][33];
    const int w = blockIdx.x, f = blockIdx.y, tx = threadIdx.x, ty = threadIdx.y;
    const int s0 = win_slot0[w];
    R* seg = keep + ((size_t)w * F + f) * (size_t)n_chains * nrun;
    const int ct = (n_chains + 31) / 32, it = (n_i + 31) / 32;
    for (int t = 0; t < ct * it; ++t) {
        const int c0 = (t % ct) * 32, i0 = (t / ct) * 32;
        __syncthreads();                        // the previous tile has been written out
        for (int r = ty; r < 32; r += 8) {
            const int c = c0 + tx, i = i0 + r;
            if (c < n_chains && i < n_i) tile[r][tx] = out[((size_t)f * chunk + i) * n_slots + s0 + c];
        }
        __syncthreads();
        for (int r = ty; r < 32; r += 8) {
            const int c = c0 + r, i = i0 + tx;
            if (c < n_chains && i < n_i) seg[(size_t)c * nrun + d0 + i] = tile[tx][r];
        }
    }
}

// Order-preserving unsigned key of a double: -0 and +0 share the key of +0, every NaN gets the largest key (so a non-finite
// draw always sorts to an end of its segment, where ranked_quantiles_kernel looks for it), the rest map by a sign-dependent
// XOR.  NaN is classified before any bit is flipped: from `(u >> 63) ? ~u : (u | sign)` nvcc forms u | sign as the bits of
// the fp64 -|x|, which leaves a NaN's sign bit clear and so sorted NaN among the negative numbers.  (The magnitude test stays
// right however it is formed: any NaN bit pattern, signed or not, compares above the bits of infinity.)  key_value inverts the
// map (NaN for the NaN key).
__device__ __forceinline__ unsigned long long ranked_key(double x) {
    constexpr unsigned long long kSign = 0x8000000000000000ull;
    const unsigned long long u = (unsigned long long)__double_as_longlong(x), mag = u & ~kSign;
    if (mag == 0) return kSign;
    if (mag > 0x7ff0000000000000ull) return ~0ull;
    return u ^ ((unsigned long long)((long long)u >> 63) | kSign);
}
__device__ __forceinline__ double key_value(unsigned long long k) {
    return __longlong_as_double((long long)(k ^ (((k >> 63) - 1ull) | 0x8000000000000000ull)));
}

// Keys of the n elements of a batch (segments of length Rs from x) and their positions.  qs != NULL: the key of |x - q(0.5)|
// (ranked_quantiles_kernel's qs), the fold.
template <typename R>
__global__ void ranked_keys_kernel(long long n, long long Rs, const R* __restrict__ x, const double* __restrict__ qs,
                                   unsigned long long* __restrict__ keys, int* __restrict__ pos) {
    const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (j >= n) return;
    double v = (double)x[j];
    if (qs) v = fabs(v - qs[j / Rs * kRankedQuants + 1]);
    keys[j] = ranked_key(v);
    pos[j] = (int)j;
}

// Sorted element j of a batch: its average rank within its segment (the run of equal keys around j, found by binary search)
// as the normal score, written at the element's position.
__global__ void ranked_scores_kernel(long long n, long long Rs, const unsigned long long* __restrict__ keys,
                                     const int* __restrict__ pos, double* __restrict__ z) {
    const long long j = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (j >= n) return;
    const long long b = j / Rs * Rs, e = b + Rs;
    const unsigned long long k = keys[j];
    long long lo = j, hi = j + 1;               // [lo, hi): the run of keys equal to k
    if (lo > b && keys[lo - 1] == k) {
        long long a = b, c = j;                 // first index in [b, j] with key == k
        while (a < c) { const long long m = (a + c) / 2; if (keys[m] < k) a = m + 1; else c = m; }
        lo = a;
    }
    if (hi < e && keys[hi] == k) {
        long long a = j + 1, c = e;             // first index in [j + 1, e] with key > k
        while (a < c) { const long long m = (a + c) / 2; if (keys[m] <= k) a = m + 1; else c = m; }
        hi = a;
    }
    const double r = 0.5 * (double)((lo - b + 1) + (hi - b));      // ranks lo-b+1 .. hi-b, averaged
    z[pos[j]] = normcdfinv((r - 0.375) / ((double)Rs + 0.25));
}

// type-7 quantile of a sorted segment of Rs keys
__device__ __forceinline__ double ranked_quantile(const unsigned long long* __restrict__ k, long long Rs, double p) {
    const double h = (double)(Rs - 1) * p;
    const double fl = floor(h);
    const long long i = (long long)fl;
    const double lo = key_value(k[i]);
    if (i + 1 >= Rs) return lo;
    return lo + (h - fl) * (key_value(k[i + 1]) - lo);
}

// Per segment of the batch (segment index s0 + s overall, field (s0 + s) % F): whether it is unusable (a non-finite draw, which
// sorts to one end, or the log-likelihood field without its flag), the requested quantiles into quant[(s0 + s)*n_probs + k]
// (NaN when unusable), and q(0.05), q(0.5), q(0.95) into qs[s*3 + ...].
struct RankedProbs { double p[kRankedMaxProbs]; int n; };
__global__ void ranked_quantiles_kernel(int n_seg, long long s0, long long Rs, int F, int has_loglik,
                                        const unsigned long long* __restrict__ keys, RankedProbs pr, double* __restrict__ quant,
                                        double* __restrict__ qs, unsigned char* __restrict__ bad) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    const unsigned long long* k = keys + (size_t)s * Rs;
    const bool b = !isfinite(key_value(k[0])) || !isfinite(key_value(k[Rs - 1])) || (!has_loglik && (int)((s0 + s) % F) == F - 1);
    bad[s] = b;
    for (int q = 0; q < pr.n; ++q) quant[(size_t)(s0 + s) * pr.n + q] = b ? NAN : ranked_quantile(k, Rs, pr.p[q]);
    qs[(size_t)s * kRankedQuants + 0] = ranked_quantile(k, Rs, 0.05);
    qs[(size_t)s * kRankedQuants + 1] = ranked_quantile(k, Rs, 0.5);
    qs[(size_t)s * kRankedQuants + 2] = ranked_quantile(k, Rs, 0.95);
}

// Split statistics of one sequence per warp: sequence (segment s, half h, chain c) holds elements
// [s*Rs + c*nrun + h*(nrun - n), + n) of the batch, transformed: z[...] when z != NULL, else 1[x[...] <= qs[s*3 + qi]].
// Writes seq_mean / seq_var [s*M + h*n_chains + c] (M = 2 n_chains) and the centred lag sums G_l, l = 0..63, to
// g[(s*M + h*n_chains + c)*64 + l].  The values are shifted by the sequence's first one (a constant sequence then has exactly
// zero variance, W = 0).  Pass 1: the mean (a fixed-order tree per tile of 32, tiles in draw order); pass 2: lane l accumulates
// lags l and l + 32 over a ring of the last 128 centred values.
template <typename R>
__global__ void __launch_bounds__(32 * kRankedSeqWarps) ranked_stats_kernel(long long n_seqs, int n_chains, long long nrun, long long n,
                                                                            long long Rs, const double* __restrict__ z,
                                                                            const R* __restrict__ x, const double* __restrict__ qs, int qi,
                                                                            double* __restrict__ seq_mean, double* __restrict__ seq_var,
                                                                            double* __restrict__ g) {
    __shared__ double ring[kRankedSeqWarps][128];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    const long long q = blockIdx.x * (long long)kRankedSeqWarps + wp;
    if (q >= n_seqs) return;
    const int M = 2 * n_chains;
    const long long s = q / M;
    const int hc = (int)(q % M), h = hc / n_chains, c = hc % n_chains;
    const size_t base = (size_t)s * Rs + (size_t)c * nrun + (size_t)h * (nrun - n);
    const double thr = z ? 0.0 : qs[s * kRankedQuants + qi];
    auto raw = [&](long long t) -> double { return z ? z[base + t] : ((double)x[base + t] <= thr ? 1.0 : 0.0); };
    const double x0 = raw(0);
    auto value = [&](long long t) -> double { return raw(t) - x0; };
    double sum = 0.0;
    for (long long t0 = 0; t0 < n; t0 += 32) {
        double v = t0 + lane < n ? value(t0 + lane) : 0.0;
        for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
        sum += __shfl_sync(0xffffffffu, v, 0);
    }
    const double mean = sum / (double)n;
    double* rg = ring[wp];
    rg[64 + lane] = 0.0;                        // positions -64 .. -1: no contribution
    rg[96 + lane] = 0.0;
    double p0 = 0.0, p1 = 0.0;
    for (long long t0 = 0; t0 < n; t0 += 32) {
        __syncwarp();                           // the previous tile's reads are done with the positions written here
        if (t0 + lane < n) rg[(t0 + lane) & 127] = value(t0 + lane) - mean;
        __syncwarp();
        const int m = n - t0 < 32 ? (int)(n - t0) : 32;
        for (int r = 0; r < m; ++r) {
            const unsigned t = (unsigned)(t0 + r);
            const double y = rg[t & 127];
            p0 = __fma_rn(y, rg[(t - lane) & 127], p0);
            p1 = __fma_rn(y, rg[(t - lane - 32) & 127], p1);
        }
    }
    double* gq = g + (size_t)q * kDiagLags;
    gq[lane] = p0;
    gq[32 + lane] = p1;
    if (lane == 0) {
        seq_mean[q] = x0 + mean;
        seq_var[q] = p0 / (double)(n - 1);
    }
}

// gsum[s*64 + l] = (sum over chains, in chain order, of half 0's G_l) + (the same for half 1), as diag_half_kernel forms it
__global__ void ranked_chain_sum_kernel(long long n_elems, int n_chains, const double* __restrict__ g, double* __restrict__ gsum) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n_elems) return;
    const long long s = i / kDiagLags;
    const int l = (int)(i % kDiagLags);
    double acc[2];
    for (int h = 0; h < 2; ++h) {
        double a = 0.0;
        for (int c = 0; c < n_chains; ++c) a += g[((size_t)(s * 2 + h) * n_chains + c) * kDiagLags + l];
        acc[h] = a;
    }
    gsum[i] = acc[0] + acc[1];
}

// The four diag_finish_kernel results of a batch (rh / es [4][n_seg]: bulk, folded, tail 5 %, tail 95 %) into the outputs of
// segments s0 .. s0 + n_seg - 1.  NaN where the segment is unusable or either part is NaN.
__global__ void ranked_combine_kernel(int n_seg, long long s0, const unsigned char* __restrict__ bad, const double* __restrict__ rh,
                                      const double* __restrict__ es, double* __restrict__ rhat_rank, double* __restrict__ ess_bulk,
                                      double* __restrict__ ess_tail) {
    const int s = blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= n_seg) return;
    const bool b = bad[s];
    const double rb = rh[s], rf = rh[n_seg + s], t5 = es[2 * n_seg + s], t95 = es[3 * n_seg + s];
    if (rhat_rank) rhat_rank[s0 + s] = (b || isnan(rb) || isnan(rf)) ? NAN : fmax(rb, rf);
    if (ess_bulk) ess_bulk[s0 + s] = b ? NAN : es[s];
    if (ess_tail) ess_tail[s0 + s] = (b || isnan(t5) || isnan(t95)) ? NAN : fmin(t5, t95);
}

// Stable sort of every segment of a batch by key, carrying the positions (d_temp == NULL: the scratch size into temp_bytes).
inline cudaError_t ranked_sort(void* d_temp, size_t& temp_bytes, cub::DoubleBuffer<unsigned long long>& keys, cub::DoubleBuffer<int>& pos,
                               int n, int n_seg, const int* offsets, cudaStream_t st) {
    return cub::DeviceSegmentedRadixSort::SortPairs(d_temp, temp_bytes, keys, pos, n, n_seg, offsets, offsets + 1, 0, 64, st);
}

}  // namespace hmc
