// hmcgpu.cu — C ABI (include/hmcgpu.h) and kernels of the B200 Gibbs/FFBS path.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 --shared (see hmc.jl_b200/build.py).
#include "../../include/hmcgpu.h"
#include "gibbs_wide_kernel.cuh"
#include "gibbs_scan_kernel.cuh"
#include "gibbs_seg_kernel.cuh"
#include "diagnostics.cuh"
#include "predictive.cuh"
#include "ranked.cuh"
#include "onestep.cuh"
#include "loo.cuh"
#include "plan_policy.cuh"

#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <exception>
#include <map>
#include <memory>
#include <mutex>
#include <new>
#include <numeric>
#include <optional>
#include <string>
#include <thread>
#include <vector>

using namespace hmc;

// ============================================================================================ context
struct DevPool;
struct hmcgpu_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    std::string err;
    int sm_count = 0;
    std::shared_ptr<DevPool> pool;      // recycled device buffers (see DevPool)
    // pinned staging buffers of large host -> device uploads (staged_upload); allocated on first use, freed with the context
    void* stage[2] = {nullptr, nullptr};
    cudaEvent_t stage_free[2] = {nullptr, nullptr};
    size_t stage_bytes = 0;
};

static thread_local std::string g_create_err;

static int fail(hmcgpu_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf; else g_create_err = buf;
    return code;
}

#define CU(ctx, call)                                                                                   \
    do {                                                                                                \
        cudaError_t e__ = (call);                                                                       \
        if (e__ != cudaSuccess)                                                                         \
            return fail(ctx, e__ == cudaErrorMemoryAllocation ? HMCGPU_ERR_ALLOC : HMCGPU_ERR_CUDA,     \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__);   \
    } while (0)

// No C++ exception may cross the C ABI (include/hmcgpu.h): host-side allocation failures become HMCGPU_ERR_ALLOC.
#define GUARD(ctx, expr)                                                                                \
    try {                                                                                               \
        return (expr);                                                                                  \
    } catch (const std::bad_alloc&) {                                                                   \
        return fail(ctx, HMCGPU_ERR_ALLOC, "%s: host allocation failed", __func__);                     \
    } catch (const std::exception& e__) {                                                               \
        return fail(ctx, HMCGPU_ERR_ALLOC, "%s: %s", __func__, e__.what());                             \
    }

// Device memory is recycled per context: repeated estimations of the same shape (the rolling-window driver calls
// hmcgpu_estimate once per batch) reuse their multi-GB buffers instead of paying cudaMalloc/cudaFree every call.
struct DevPool {
    std::mutex mu;
    std::multimap<size_t, void*> free_blocks;
    size_t pooled = 0;
    // Upper bound of idle memory kept for reuse (HMCGPU_POOL_MAX_GB overrides; 0 disables pooling).  Idle blocks are also
    // released by hmcgpu_ctx_trim, when another allocation on this context fails, and when the context is destroyed, so
    // other allocators on the same GPU (torch, NCCL, a second context) are never starved by memory nobody is using.
    size_t max_pooled = 16ull << 30;
    static constexpr size_t kMaxBlocks = 64;
    DevPool() {
        if (const char* e = getenv("HMCGPU_POOL_MAX_GB")) max_pooled = (size_t)(atof(e) * (double)(1ull << 30));
    }
    cudaError_t get(size_t n, void** out) {
        {
            std::lock_guard<std::mutex> g(mu);
            auto it = free_blocks.find(n);
            if (it != free_blocks.end()) { *out = it->second; pooled -= n; free_blocks.erase(it); return cudaSuccess; }
        }
        cudaError_t e = cudaMalloc(out, n);
        if (e == cudaErrorMemoryAllocation) {                     // make room and retry once
            cudaGetLastError();
            release_all();
            e = cudaMalloc(out, n);
        }
        return e;
    }
    void put(size_t n, void* p) {
        std::lock_guard<std::mutex> g(mu);
        if (n > max_pooled) { cudaFree(p); return; }
        // make room by dropping the smallest idle blocks first (big buffers are the expensive ones to re-allocate)
        while (!free_blocks.empty() && (pooled + n > max_pooled || free_blocks.size() >= kMaxBlocks)) {
            auto it = free_blocks.begin();
            cudaFree(it->second);
            pooled -= it->first;
            free_blocks.erase(it);
        }
        free_blocks.emplace(n, p);
        pooled += n;
    }
    void release_all() {
        std::lock_guard<std::mutex> g(mu);
        for (auto& kv : free_blocks) cudaFree(kv.second);
        free_blocks.clear();
        pooled = 0;
    }
    ~DevPool() { release_all(); }
};
static thread_local std::shared_ptr<DevPool> tl_pool;     // set by the API entry points for the context they run on

// RAII device buffer
struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    std::shared_ptr<DevPool> pool;
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void release() {
        if (!p) return;
        if (pool) pool->put(bytes, p); else cudaFree(p);
        p = nullptr;
    }
    cudaError_t alloc(size_t n) {
        release();
        bytes = n;
        if (n == 0) return cudaSuccess;
        pool = tl_pool;
        return pool ? pool->get(n, &p) : cudaMalloc(&p, n);
    }
    template <typename T> T* as() const { return reinterpret_cast<T*>(p); }
};

extern "C" int hmcgpu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

extern "C" int hmcgpu_ctx_create(int device, hmcgpu_ctx** out) {
    if (!out) return fail(nullptr, HMCGPU_ERR_ARG, "out is NULL");
    *out = nullptr;
    int n = hmcgpu_device_count();
    if (n <= 0) return fail(nullptr, HMCGPU_ERR_NODEVICE, "no CUDA device visible (this library has no CPU fallback)");
    if (device < 0 || device >= n) return fail(nullptr, HMCGPU_ERR_ARG, "device %d out of range (0..%d)", device, n - 1);
    std::unique_ptr<hmcgpu_ctx> ctx(new hmcgpu_ctx());     // released into *out only when everything below succeeded
    ctx->device = device;
    CU(nullptr, cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(nullptr, cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        return fail(nullptr, HMCGPU_ERR_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a (B200) only",
                    device, prop.major, prop.minor);
    }
    ctx->sm_count = prop.multiProcessorCount;
    CU(nullptr, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    ctx->pool = std::make_shared<DevPool>();
    *out = ctx.release();
    return HMCGPU_OK;
}

// releases the idle device buffers this context keeps for reuse (they are also released on allocation failure and at destroy)
extern "C" int hmcgpu_ctx_trim(hmcgpu_ctx* ctx) {
    if (!ctx) return HMCGPU_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    if (ctx->pool) ctx->pool->release_all();
    return HMCGPU_OK;
}

extern "C" void hmcgpu_ctx_destroy(hmcgpu_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaDeviceSynchronize();
    if (tl_pool == ctx->pool) tl_pool.reset();
    if (ctx->pool) ctx->pool->release_all();
    for (int i = 0; i < 2; ++i) {
        if (ctx->stage[i]) cudaFreeHost(ctx->stage[i]);
        if (ctx->stage_free[i]) cudaEventDestroy(ctx->stage_free[i]);
    }
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

extern "C" const char* hmcgpu_last_error(const hmcgpu_ctx* ctx) { return ctx ? ctx->err.c_str() : g_create_err.c_str(); }

extern "C" int hmcgpu_ctx_sync(hmcgpu_ctx* ctx) {
    if (!ctx) return HMCGPU_ERR_ARG;
    CU(ctx, cudaSetDevice(ctx->device));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return HMCGPU_OK;
}

static bool k_supported(int K) { return K >= 2 && K <= 32; }
static bool k_thread(int K) { return K >= 2 && K <= 4; }       // every feature (smoothed means, signals, K-templated entry points)

#define DISPATCH_K(K, ...)                          \
    switch (K) {                                    \
        case 2: { constexpr int KK = 2; __VA_ARGS__; } break; \
        case 3: { constexpr int KK = 3; __VA_ARGS__; } break; \
        case 4: { constexpr int KK = 4; __VA_ARGS__; } break; \
        default: break;                             \
    }
#ifdef HMC_DEV_F3   /* experiment builds: only the fp32 K=3 sweep kernels are linked */
#define DISPATCH_RUN(pl, rc) do { if ((pl)->precision == 32) { if ((pl)->sw.kernel == SweepKernel::lane) rc = plan_run_t<float, 0>(pl); else if ((pl)->K == 3) rc = plan_run_t<float, 3>(pl); } } while (0)
#elif defined(HMC_DEV_D3)   /* ... or only the fp64 K=3 ones */
#define DISPATCH_RUN(pl, rc) do { if ((pl)->precision == 64) { if ((pl)->sw.kernel == SweepKernel::lane) rc = plan_run_t<double, 0>(pl); else if ((pl)->K == 3) rc = plan_run_t<double, 3>(pl); } } while (0)
#else
#define DISPATCH_K8(K, ...)                         \
    switch (K) {                                    \
        case 2: { constexpr int KK = 2; __VA_ARGS__; } break; \
        case 3: { constexpr int KK = 3; __VA_ARGS__; } break; \
        case 4: { constexpr int KK = 4; __VA_ARGS__; } break; \
        case 5: { constexpr int KK = 5; __VA_ARGS__; } break; \
        case 6: { constexpr int KK = 6; __VA_ARGS__; } break; \
        case 7: { constexpr int KK = 7; __VA_ARGS__; } break; \
        case 8: { constexpr int KK = 8; __VA_ARGS__; } break; \
        default: break;                             \
    }
#define DISPATCH_RUN(pl, rc)                                                                                          \
    do {                                                                                                            \
        if ((pl)->sw.kernel == SweepKernel::lane) rc = ((pl)->precision == 32) ? plan_run_t<float, 0>(pl) : plan_run_t<double, 0>(pl);       \
        else DISPATCH_K8((pl)->K, { rc = ((pl)->precision == 32) ? plan_run_t<float, KK>(pl) : plan_run_t<double, KK>(pl); }) \
    } while (0)
#endif

// ============================================================================================ deterministic entry points
// One thread per batch element; host arrays are fp64 row-major and are converted on the fly.

// sig (may be NULL): signal flag per time step, shared by the batch; signal rows use sd*(1+kappa) (src/Hmc.jl:382)
template <typename R, int K>
__global__ void filter_kernel(long long B, long long T, const double* __restrict__ y, long long ystride,
                              const double* __restrict__ A, const double* __restrict__ mu, const double* __restrict__ sig2,
                              const double* __restrict__ rho, double* __restrict__ pif, double* __restrict__ totals,
                              double* __restrict__ loglik, const unsigned char* __restrict__ sig, double kappa) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= B) return;
    R a[K][K], m[K], s2[K], pf[K];
#pragma unroll
    for (int r = 0; r < K; ++r) {
        m[r] = (R)mu[b * K + r]; s2[r] = (R)sig2[b * K + r]; pf[r] = (R)rho[b * K + r];
#pragma unroll
        for (int s = 0; s < K; ++s) a[r][s] = (R)A[(b * K + r) * K + s];
    }
    Emission<R, K> em;
    em.prepare(m, s2);
    const double* yb = y + b * ystride;
    double ll = 0.0;
    const R k1 = (R)(1.0 / (1.0 + kappa));
    for (long long t = 0; t < T; ++t) {
        R e[K];
        R m2;
        if (sig && sig[t]) {                                  // z scaled by 1/(1+kappa), pdf by the same factor
            if constexpr (sizeof(R) == 8) {
                em.template eval_scaled<true>((R)yb[t], k1, e);          // entry points keep libm's exp
                m2 = R(0);
            } else {
                // fp32: the scaled series point (y - mu)*k1 = (y*k1 - mu*k1) is not an affine image of y for all states at
                // once, so evaluate the quadratic directly
                float l[K];
#pragma unroll
                for (int s = 0; s < K; ++s) { const float d = ((float)yb[t] - (float)em.mu[s]) * (float)k1; l[s] = fmaf(d * d, (float)em.q[s], (float)em.c[s]); }
                float mx = l[0];
#pragma unroll
                for (int s = 1; s < K; ++s) mx = fmaxf(mx, l[s]);
#pragma unroll
                for (int s = 0; s < K; ++s) e[s] = (R)Real<float>::ex2(l[s] - mx);
                m2 = (R)(mx + Real<float>::lg2((float)k1));
            }
        } else {
            m2 = em.template eval<true>((R)yb[t], e);
        }
        bool ok;
        const R tot = forward_step<R, K>(a, e, pf, ok);
        if (!ok) {
#pragma unroll
            for (int s = 0; s < K; ++s) pf[s] = R(1) / R(K);
        }
        // natural-log normaliser of the unscaled recursion (what the reference's `total` is, :417/:430)
        const double lt = (sizeof(R) == 4) ? ((double)Real<float>::lg2((float)tot) + (double)m2) * 0.6931471805599453
                                           : log((double)tot);
        ll += lt;
        if (totals) totals[b * T + t] = (sizeof(R) == 4) ? exp(lt) : (double)tot;
#pragma unroll
        for (int s = 0; s < K; ++s) pif[(b * T + t) * K + s] = (double)pf[s];
    }
    if (loglik) loglik[b] = ll;
}

template <typename R, int K>
__global__ void smooth_kernel(long long B, long long T, const double* __restrict__ A, const double* __restrict__ pif,
                              double* __restrict__ pib) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= B) return;
    R a[K][K], pb[K], pf[K];
#pragma unroll
    for (int r = 0; r < K; ++r)
#pragma unroll
        for (int s = 0; s < K; ++s) a[r][s] = (R)A[(b * K + r) * K + s];
#pragma unroll
    for (int s = 0; s < K; ++s) { pb[s] = (R)pif[(b * T + T - 1) * K + s]; pib[(b * T + T - 1) * K + s] = (double)pb[s]; }
    for (long long t = T - 2; t >= 0; --t) {
#pragma unroll
        for (int s = 0; s < K; ++s) pf[s] = (R)pif[(b * T + t) * K + s];
        smooth_step<R, K>(a, pf, pb);
#pragma unroll
        for (int s = 0; s < K; ++s) pib[(b * T + t) * K + s] = (double)pb[s];
    }
}

// fp64, operation-for-operation the oracle's pif form (bit-exact state paths under injected uniforms)
template <int K>
__global__ void sample_states_kernel(long long B, long long T, const double* __restrict__ A, const double* __restrict__ pif,
                                     const double* __restrict__ piN, const double* __restrict__ u, long long* __restrict__ X) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= B) return;
    double a[K][K], p[K];
#pragma unroll
    for (int r = 0; r < K; ++r)
#pragma unroll
        for (int s = 0; s < K; ++s) a[r][s] = A[(b * K + r) * K + s];
#pragma unroll
    for (int s = 0; s < K; ++s) p[s] = piN ? piN[b * K + s] : pif[(b * T + T - 1) * K + s];
    int x = categorical_exact<K>(p, u[b * T + T - 1]);
    X[b * T + T - 1] = x + 1;
    for (long long k = T - 2; k >= 0; --k) {
        double total = 0.0;
#pragma unroll
        for (int r = 0; r < K; ++r) {
            p[r] = __dmul_rn(pif[(b * T + k) * K + r], select_k<double, K>(a[r], x));
            total = __dadd_rn(total, p[r]);
        }
        const double gate = pif[(b * T + k + 1) * K + x];
        if (gate > 2.220446049250313e-16 && total > 0.0) {
#pragma unroll
            for (int r = 0; r < K; ++r) p[r] = __ddiv_rn(p[r], total);
        } else {
#pragma unroll
            for (int r = 0; r < K; ++r) p[r] = 1.0 / K;
        }
        x = categorical_exact<K>(p, u[b * T + k]);
        X[b * T + k] = x + 1;
    }
}

// Mi / Sm / Sm2 (may be NULL): counts, sums and centred sums of squares of the noisy signals per state (src/Hmc.jl:267-300)
template <typename R, int K>
__global__ void draw_params_kernel(long long B, const long long* __restrict__ Ni, const double* __restrict__ S,
                                   const double* __restrict__ S2, const long long* __restrict__ Mi, const double* __restrict__ Sm,
                                   const double* __restrict__ Sm2, double kappa, const long long* __restrict__ trans,
                                   const double* __restrict__ xi, const double* __restrict__ alpha, const double* __restrict__ nu,
                                   const double* __restrict__ beta, unsigned k0, unsigned k1, unsigned chain0, unsigned sweep,
                                   double* __restrict__ sig2o, double* __restrict__ muo, double* __restrict__ rhoo,
                                   double* __restrict__ Ao) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= B) return;
    int cnt[K], tr[K][K];
    R Sd[K], Qd[K], sig2[K], mu[K], rho[K], A[K][K];
    Hyper<R, K> hp;
#pragma unroll
    for (int i = 0; i < K; ++i) {
        cnt[i] = (int)Ni[b * K + i];
        const double s = S[b * K + i], n = (double)cnt[i];
        const double ybar = cnt[i] > 0 ? s / n : 0.0;
        Sd[i] = (R)s;                                // shift c = 0
        Qd[i] = (R)(S2[b * K + i] + n * ybar * ybar); // raw second moment
        hp.xi[i] = (R)xi[i]; hp.alpha[i] = (R)alpha[i]; hp.nu[i] = (R)nu[i]; hp.beta[i] = (R)beta[i];
        sig2[i] = R(1);
#pragma unroll
        for (int j = 0; j < K; ++j) tr[i][j] = (int)trans[(b * K + i) * K + j] - 1;  // API counts include the +1 prior
    }
    const RngKey key{k0, k1, chain0 + (unsigned)b};
    if (Mi) {
        SigStats<R, K> sg;
#pragma unroll
        for (int i = 0; i < K; ++i) {
            sg.m[i] = (int)Mi[b * K + i];
            const double m = (double)sg.m[i], sbar = sg.m[i] > 0 ? Sm[b * K + i] / m : 0.0;
            sg.Sm[i] = (R)Sm[b * K + i];
            sg.Qm[i] = (R)(Sm2[b * K + i] + m * sbar * sbar);
        }
        sg.k1 = (R)(1.0 / (1.0 + kappa));
        draw_params<R, K, true>(cnt, Sd, Qd, tr, R(0), hp, key, sweep, sig2, mu, rho, A, &sg);
    } else {
        draw_params<R, K>(cnt, Sd, Qd, tr, R(0), hp, key, sweep, sig2, mu, rho, A);
    }
#pragma unroll
    for (int i = 0; i < K; ++i) {
        sig2o[b * K + i] = (double)sig2[i]; muo[b * K + i] = (double)mu[i]; rhoo[b * K + i] = (double)rho[i];
#pragma unroll
        for (int j = 0; j < K; ++j) Ao[(b * K + i) * K + j] = (double)A[i][j];
    }
}

template <int K>
__global__ void forecast_kernel(long long B, const double* __restrict__ mu, const double* __restrict__ A,
                                const double* __restrict__ pi, const int* __restrict__ horizons, int n_h,
                                const double* __restrict__ yreal, double* __restrict__ out) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= B) return;
    double a[K][K], m[K];
#pragma unroll
    for (int r = 0; r < K; ++r) {
        m[r] = mu[b * K + r];
#pragma unroll
        for (int s = 0; s < K; ++s) a[r][s] = A[(b * K + r) * K + s];
    }
    for (int j = 0; j < n_h; ++j) {
        double v[K];
#pragma unroll
        for (int s = 0; s < K; ++s) v[s] = pi[b * K + s];
        for (int h = 0; h < horizons[j]; ++h) {
            double nv[K];
#pragma unroll
            for (int s = 0; s < K; ++s) {
                double acc = v[0] * a[0][s];
#pragma unroll
                for (int r = 1; r < K; ++r) acc = fma(v[r], a[r][s], acc);
                nv[s] = acc;
            }
#pragma unroll
            for (int s = 0; s < K; ++s) v[s] = nv[s];
        }
        double f = 0.0;
#pragma unroll
        for (int s = 0; s < K; ++s) f = fma(v[s], m[s], f);
        out[(b * n_h + j) * 2] = f;
        out[(b * n_h + j) * 2 + 1] = f - yreal[j];
    }
}


// ---- runtime-K (5..32) versions of the deterministic entry points: same arithmetic, small local arrays, A read from
//      global memory.  These are checking utilities, not hot paths.
constexpr int kMaxK = 32;
constexpr int kMaxHorizon = 100000;   // forecast horizons run an in-kernel loop of that length per saved draw

template <typename R>
__global__ void filter_kernel_generic(int K, long long B, long long T, const double* __restrict__ y, long long ystride,
                                      const double* __restrict__ A, const double* __restrict__ mu, const double* __restrict__ sig2,
                                      const double* __restrict__ rho, double* __restrict__ pif, double* __restrict__ totals,
                                      double* __restrict__ loglik) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= B) return;
    R pf[kMaxK], q[kMaxK], m[kMaxK], c0[kMaxK], c1[kMaxK];
    for (int s = 0; s < K; ++s) {
        pf[s] = (R)rho[b * K + s]; m[s] = (R)mu[b * K + s];
        const R v = (R)sig2[b * K + s];
        if (sizeof(R) == 4) { c0[s] = (R)(-0.72134752044448170368) / v; c1[s] = (R)(-0.5f * Real<float>::lg2(6.283185307179586f * (float)v)); }
        else { const R sd = (R)sqrt((double)v); c0[s] = R(1) / sd; c1[s] = (R)0.3989422804014327 / sd; }
    }
    const double* Ab = A + b * K * K;
    const double* yb = y + b * ystride;
    double ll = 0.0;
    for (long long t = 0; t < T; ++t) {
        const R yt = (R)yb[t];
        R mx = (R)(-3.0e38);
        if (sizeof(R) == 4) for (int s = 0; s < K; ++s) { const R d = yt - m[s]; q[s] = fma(d * d, c0[s], c1[s]); mx = q[s] > mx ? q[s] : mx; }
        R tot = R(0);
        for (int s = 0; s < K; ++s) {
            R e;
            if (sizeof(R) == 4) e = (R)Real<float>::ex2((float)(q[s] - mx));
            else { const R z = (yt - m[s]) * c0[s]; e = (R)exp(-0.5 * (double)(z * z)) * c1[s]; }
            R pred = R(0);
            for (int r = 0; r < K; ++r) pred = fma(pf[r], (R)Ab[r * K + s], pred);
            q[s] = pred * e;
            tot += q[s];
        }
        const bool ok = (tot > R(0)) && (tot < R(3.0e38));
        for (int s = 0; s < K; ++s) pf[s] = ok ? q[s] / tot : R(1) / R(K);
        const double lt = (sizeof(R) == 4) ? ((double)Real<float>::lg2((float)tot) + (double)mx) * 0.6931471805599453 : log((double)tot);
        ll += lt;
        if (totals) totals[b * T + t] = (sizeof(R) == 4) ? exp(lt) : (double)tot;
        for (int s = 0; s < K; ++s) pif[(b * T + t) * K + s] = (double)pf[s];
    }
    if (loglik) loglik[b] = ll;
}

template <typename R>
__global__ void smooth_kernel_generic(int K, long long B, long long T, const double* __restrict__ A, const double* __restrict__ pif,
                                      double* __restrict__ pib) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= B) return;
    R pb[kMaxK], w[kMaxK];
    const double* Ab = A + b * K * K;
    for (int s = 0; s < K; ++s) { pb[s] = (R)pif[(b * T + T - 1) * K + s]; pib[(b * T + T - 1) * K + s] = (double)pb[s]; }
    for (long long t = T - 2; t >= 0; --t) {
        const double* f = pif + (b * T + t) * K;
        for (int s = 0; s < K; ++s) {
            R pred = R(0);
            for (int r = 0; r < K; ++r) pred = fma((R)f[r], (R)Ab[r * K + s], pred);
            w[s] = pred > R(0) ? pb[s] / pred : R(0);
        }
        for (int r = 0; r < K; ++r) {
            R acc = R(0);
            for (int s2 = 0; s2 < K; ++s2) acc = fma((R)Ab[r * K + s2], w[s2], acc);
            pb[r] = (R)f[r] * acc;
        }
        for (int s = 0; s < K; ++s) pib[(b * T + t) * K + s] = (double)pb[s];
    }
}

__global__ void sample_states_kernel_generic(int K, long long B, long long T, const double* __restrict__ A, const double* __restrict__ pif,
                                             const double* __restrict__ piN, const double* __restrict__ u, long long* __restrict__ X) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= B) return;
    double p[kMaxK];
    const double* Ab = A + b * K * K;
    auto cat = [&](double uu) { int i = 0; double c = p[0]; while (c < uu && i < K - 1) { ++i; c = __dadd_rn(c, p[i]); } return i; };
    for (int s = 0; s < K; ++s) p[s] = piN ? piN[b * K + s] : pif[(b * T + T - 1) * K + s];
    int x = cat(u[b * T + T - 1]);
    X[b * T + T - 1] = x + 1;
    for (long long k = T - 2; k >= 0; --k) {
        double total = 0.0;
        for (int r = 0; r < K; ++r) { p[r] = __dmul_rn(pif[(b * T + k) * K + r], Ab[r * K + x]); total = __dadd_rn(total, p[r]); }
        const double gate = pif[(b * T + k + 1) * K + x];
        if (gate > 2.220446049250313e-16 && total > 0.0) { for (int r = 0; r < K; ++r) p[r] = __ddiv_rn(p[r], total); }
        else { for (int r = 0; r < K; ++r) p[r] = 1.0 / K; }
        x = cat(u[b * T + k]);
        X[b * T + k] = x + 1;
    }
}

__global__ void forecast_kernel_generic(int K, long long B, const double* __restrict__ mu, const double* __restrict__ A,
                                        const double* __restrict__ pi, const int* __restrict__ horizons, int n_h,
                                        const double* __restrict__ yreal, double* __restrict__ out) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= B) return;
    double v[kMaxK], nv[kMaxK];
    const double* Ab = A + b * K * K;
    for (int j = 0; j < n_h; ++j) {
        for (int s = 0; s < K; ++s) v[s] = pi[b * K + s];
        for (int h = 0; h < horizons[j]; ++h) {
            for (int s = 0; s < K; ++s) { double acc = 0.0; for (int r = 0; r < K; ++r) acc = fma(v[r], Ab[r * K + s], acc); nv[s] = acc; }
            for (int s = 0; s < K; ++s) v[s] = nv[s];
        }
        double f = 0.0;
        for (int s = 0; s < K; ++s) f = fma(v[s], mu[b * K + s], f);
        out[(b * n_h + j) * 2] = f;
        out[(b * n_h + j) * 2 + 1] = f - yreal[j];
    }
}

template <typename R>
__global__ void draw_params_kernel_generic(int K, long long B, const long long* __restrict__ Ni, const double* __restrict__ S,
                                           const double* __restrict__ S2, const long long* __restrict__ trans,
                                           const double* __restrict__ xi, const double* __restrict__ alpha, const double* __restrict__ nu,
                                           const double* __restrict__ beta, unsigned k0, unsigned k1, unsigned chain0, unsigned sweep,
                                           double* __restrict__ sig2o, double* __restrict__ muo, double* __restrict__ rhoo,
                                           double* __restrict__ Ao) {
    const long long b = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (b >= B) return;
    const RngKey key{k0, k1, chain0 + (unsigned)b};
    R rsum = R(0);
    for (int i = 0; i < K; ++i) {
        const R n = (R)Ni[b * K + i];
        const R ybar = n > R(0) ? (R)S[b * K + i] / n : R(0);
        const R dev = ybar - (R)xi[i];
        const R a = (R)alpha[i] + R(0.5) * n;
        const R bb = (R)beta[i] + R(0.5) * (R)S2[b * K + i] + R(0.5) * n * (R)nu[i] / (n + (R)nu[i]) * (dev * dev);
        R v = R(1);
        if (a > R(0) && bb > R(0)) v = bb / gamma_mt<R>(a, key, sweep, (KIND_SIGMA << 16) | (uint32_t)i);
        sig2o[b * K + i] = (double)v;
        const R m = ((R)S[b * K + i] + (R)nu[i] * (R)xi[i]) / (n + (R)nu[i]);
        const R sd = M<R>::sqrt(v / (n + (R)nu[i]));
        const uint4 w = rng_block(key, sweep, (KIND_MU << 16), (uint32_t)(i >> 1));
        muo[b * K + i] = (double)(m + sd * ((i & 1) ? normal_from<R>(w.z, w.w) : normal_from<R>(w.x, w.y)));
        const R g = gamma_mt<R>(R(1), key, sweep, (KIND_RHO << 16) | (uint32_t)i);
        rhoo[b * K + i] = (double)g;
        rsum += g;
        R tot = R(0);
        for (int j = 0; j < K; ++j) {
            const R ga = gamma_mt<R>((R)trans[(b * K + i) * K + j], key, sweep, (KIND_A << 16) | (uint32_t)(i * K + j));
            Ao[(b * K + i) * K + j] = (double)ga;
            tot += ga;
        }
        for (int j = 0; j < K; ++j) Ao[(b * K + i) * K + j] = (double)((R)Ao[(b * K + i) * K + j] / tot);
    }
    for (int i = 0; i < K; ++i) rhoo[b * K + i] = (double)((R)rhoo[b * K + i] / rsum);
}

__global__ void philox_kernel(long long n, int rounds, const unsigned* __restrict__ ctr, const unsigned* __restrict__ key, unsigned* __restrict__ out) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint4 r = rounds == kStateRounds ? philox4x32<kStateRounds>(ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3], key[2 * i], key[2 * i + 1])
                                           : philox4x32<10>(ctr[4 * i], ctr[4 * i + 1], ctr[4 * i + 2], ctr[4 * i + 3], key[2 * i], key[2 * i + 1]);
    out[4 * i] = r.x; out[4 * i + 1] = r.y; out[4 * i + 2] = r.z; out[4 * i + 3] = r.w;
}

// ---- host helpers for the deterministic calls
struct Xfer {
    hmcgpu_ctx* ctx;
    std::vector<DevBuf*> owned;
    // error paths return with copies / kernels still queued on the stream: nothing may go back to the pool before they finish
    ~Xfer() { cudaStreamSynchronize(ctx->stream); for (auto* b : owned) delete b; }
    template <typename T> int up(const T* host, size_t n, T** dev) {
        DevBuf* b = new DevBuf();
        owned.push_back(b);
        CU(ctx, b->alloc(n * sizeof(T)));
        if (host) CU(ctx, cudaMemcpyAsync(b->p, host, n * sizeof(T), cudaMemcpyHostToDevice, ctx->stream));
        *dev = b->as<T>();
        return 0;
    }
    template <typename T> int down(T* host, const T* dev, size_t n) {
        if (host) CU(ctx, cudaMemcpyAsync(host, dev, n * sizeof(T), cudaMemcpyDeviceToHost, ctx->stream));
        return 0;
    }
};

#define TRY(x) do { int rc__ = (x); if (rc__ != 0) return rc__; } while (0)

// Large uploads from the caller's (pageable) memory.  A plain cudaMemcpyAsync from pageable memory is staged by the driver on
// ONE thread at a few GB/s (measured: the 1 GB series upload of the wide batch C4 was twice its device time).  Here the copy is
// cut into chunks that several host threads copy into one of two pinned buffers while the DMA engine drains the other: one
// cudaMemcpyAsync per chunk, limited by host memory bandwidth / PCIe instead of a single core.  HMCGPU_STAGE_MB sets the
// chunk size (0: plain copy), HMCGPU_STAGE_THREADS the copying threads.
static cudaError_t staged_upload(hmcgpu_ctx* ctx, void* dev, const void* host, size_t bytes, cudaStream_t st) {
    const size_t chunk = [] { const char* e = getenv("HMCGPU_STAGE_MB"); return (size_t)std::max(0ll, std::min(1024ll, e ? atoll(e) : 32ll)) << 20; }();
    const int n_thr = [] {
        const char* e = getenv("HMCGPU_STAGE_THREADS");
        const int hw = (int)std::thread::hardware_concurrency();
        return std::max(1, std::min(64, e ? atoi(e) : std::min(8, hw > 1 ? hw / 2 : 1)));
    }();
    if (chunk == 0 || bytes < 2 * chunk) return cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, st);
    {   // a caller that already hands over page-locked memory needs no staging: the DMA engine reads it directly
        cudaPointerAttributes at;
        if (cudaPointerGetAttributes(&at, host) == cudaSuccess && at.type == cudaMemoryTypeHost)
            return cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, st);
        cudaGetLastError();
    }
    if (ctx->stage_bytes != chunk) {
        for (int i = 0; i < 2; ++i) {
            if (ctx->stage[i]) { cudaFreeHost(ctx->stage[i]); ctx->stage[i] = nullptr; }
            cudaError_t e = cudaHostAlloc(&ctx->stage[i], chunk, cudaHostAllocDefault);
            if (e != cudaSuccess) { ctx->stage[i] = nullptr; ctx->stage_bytes = 0; cudaGetLastError(); return cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, st); }
            if (!ctx->stage_free[i] && (e = cudaEventCreateWithFlags(&ctx->stage_free[i], cudaEventDisableTiming)) != cudaSuccess) return e;
        }
        ctx->stage_bytes = chunk;
    }
    const char* src = static_cast<const char*>(host);
    char* dst = static_cast<char*>(dev);
    // persistent copy threads for this upload: thread t copies its slice of every chunk; the caller's thread drives the DMA
    struct Shared { std::mutex mu; std::condition_variable cv; long long filling = -1; int done = 0; bool quit = false; } sh;
    const size_t n_chunks = (bytes + chunk - 1) / chunk;
    auto chunk_len = [&](size_t c) { return std::min(chunk, bytes - c * chunk); };
    auto worker = [&](int t) {
        long long seen = -1;
        for (;;) {
            long long c;
            {
                std::unique_lock<std::mutex> lk(sh.mu);
                sh.cv.wait(lk, [&] { return sh.quit || sh.filling > seen; });
                if (sh.quit) return;
                c = seen = sh.filling;
            }
            const size_t len = chunk_len((size_t)c), per = (len / n_thr + 63) & ~(size_t)63;
            const size_t lo = std::min(len, per * t), hi = (t == n_thr - 1) ? len : std::min(len, per * (t + 1));
            if (hi > lo) memcpy(static_cast<char*>(ctx->stage[c & 1]) + lo, src + (size_t)c * chunk + lo, hi - lo);
            {
                std::lock_guard<std::mutex> lk(sh.mu);
                ++sh.done;
            }
            sh.cv.notify_all();
        }
    };
    std::vector<std::thread> pool;
    try {
        for (int t = 1; t < n_thr; ++t) pool.emplace_back(worker, t);
    } catch (...) {                                                              // no threads to be had: stop the ones that started, plain copy
        {
            std::lock_guard<std::mutex> lk(sh.mu);
            sh.quit = true;
        }
        sh.cv.notify_all();
        for (auto& t : pool) t.join();
        return cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, st);
    }
    cudaError_t rc = cudaSuccess;
    for (size_t c = 0; c < n_chunks && rc == cudaSuccess; ++c) {
        if (c >= 2) rc = cudaEventSynchronize(ctx->stage_free[c & 1]);          // the DMA out of this buffer (chunk c-2) has finished
        if (rc != cudaSuccess) break;
        {
            std::lock_guard<std::mutex> lk(sh.mu);
            sh.filling = (long long)c; sh.done = 0;
        }
        sh.cv.notify_all();
        {                                                                        // the caller's thread copies slice 0
            const size_t len = chunk_len(c), per = (len / n_thr + 63) & ~(size_t)63;
            const size_t hi = n_thr == 1 ? len : std::min(len, per);
            memcpy(ctx->stage[c & 1], src + c * chunk, hi);
        }
        {
            std::unique_lock<std::mutex> lk(sh.mu);
            sh.cv.wait(lk, [&] { return sh.done == n_thr - 1; });
        }
        rc = cudaMemcpyAsync(dst + c * chunk, ctx->stage[c & 1], chunk_len(c), cudaMemcpyHostToDevice, st);
        if (rc == cudaSuccess) rc = cudaEventRecord(ctx->stage_free[c & 1], st);
    }
    {
        std::lock_guard<std::mutex> lk(sh.mu);
        sh.quit = true;
    }
    sh.cv.notify_all();
    for (auto& t : pool) t.join();
    // the staging buffers are reused by the next upload on this context: it starts by overwriting them, so drain the DMA first
    if (rc == cudaSuccess) rc = cudaEventSynchronize(ctx->stage_free[(n_chunks - 1) & 1]);
    return rc;
}

// HMCGPU_VERBOSE=1: wall-clock phases of an estimation on stderr
struct PhaseTrace {
    const bool on = getenv("HMCGPU_VERBOSE") != nullptr && atoi(getenv("HMCGPU_VERBOSE")) != 0;
    std::chrono::steady_clock::time_point t0 = std::chrono::steady_clock::now();
    void sync_mark(cudaStream_t st, const char* what) {      // (tracing only) drains the stream first: device time of what was queued
        if (!on) return;
        cudaStreamSynchronize(st);
        mark(what);
    }
    void mark(const char* what) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[hmcgpu] %-28s %9.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

static int check_common(hmcgpu_ctx* ctx, int K, long long B, long long T) {
    if (!ctx) return HMCGPU_ERR_ARG;
    if (!k_supported(K)) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "K=%d not supported (2..32)", K);
    if (B <= 0 || T <= 0) return fail(ctx, HMCGPU_ERR_ARG, "empty batch (B=%lld, T=%lld)", B, T);
    if (cudaSetDevice(ctx->device) != cudaSuccess) return fail(ctx, HMCGPU_ERR_CUDA, "cudaSetDevice failed");
    tl_pool = ctx->pool;
    return 0;
}

static inline unsigned grid_for(long long n, int block) { return (unsigned)((n + block - 1) / block); }

static int filter_impl(hmcgpu_ctx* ctx, int32_t precision, int32_t K, int64_t B, int64_t T, const double* y,
                       int64_t ystride, const uint8_t* is_signal, double kappa, const double* A, const double* mu,
                       const double* sigma2, const double* rho, double* pif, double* totals, double* loglik) {
    TRY(check_common(ctx, K, B, T));
    if (is_signal && !k_thread(K)) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "the signal mask is only implemented for K <= 4");
    if (is_signal && !(kappa >= 0.0)) return fail(ctx, HMCGPU_ERR_ARG, "kappa must be >= 0");
    if (!y || !A || !mu || !sigma2 || !rho || !pif) return fail(ctx, HMCGPU_ERR_ARG, "NULL input");
    if (precision != 32 && precision != 64) return fail(ctx, HMCGPU_ERR_ARG, "precision must be 32 or 64");
    if (ystride != 0 && ystride < T) return fail(ctx, HMCGPU_ERR_ARG, "y_batch_stride < T");
    Xfer x{ctx};
    double *dy, *dA, *dmu, *ds, *dr, *dp, *dt = nullptr, *dl = nullptr;
    TRY(x.up(y, (size_t)(ystride ? B * ystride : T), &dy));
    TRY(x.up(A, (size_t)B * K * K, &dA)); TRY(x.up(mu, (size_t)B * K, &dmu));
    TRY(x.up(sigma2, (size_t)B * K, &ds)); TRY(x.up(rho, (size_t)B * K, &dr));
    TRY(x.up((double*)nullptr, (size_t)B * T * K, &dp));
    if (totals) TRY(x.up((double*)nullptr, (size_t)B * T, &dt));
    if (loglik) TRY(x.up((double*)nullptr, (size_t)B, &dl));
    unsigned char* dsig = nullptr;
    if (is_signal) TRY(x.up(reinterpret_cast<const unsigned char*>(is_signal), (size_t)T, &dsig));
    if (!k_thread(K)) {
        if (precision == 32) filter_kernel_generic<float><<<grid_for(B, 64), 64, 0, ctx->stream>>>(K, B, T, dy, ystride, dA, dmu, ds, dr, dp, dt, dl);
        else filter_kernel_generic<double><<<grid_for(B, 64), 64, 0, ctx->stream>>>(K, B, T, dy, ystride, dA, dmu, ds, dr, dp, dt, dl);
    }
    DISPATCH_K(K, {
        if (precision == 32) filter_kernel<float, KK><<<grid_for(B, 64), 64, 0, ctx->stream>>>(B, T, dy, ystride, dA, dmu, ds, dr, dp, dt, dl, dsig, kappa);
        else filter_kernel<double, KK><<<grid_for(B, 64), 64, 0, ctx->stream>>>(B, T, dy, ystride, dA, dmu, ds, dr, dp, dt, dl, dsig, kappa);
    });
    CU(ctx, cudaGetLastError());
    TRY(x.down(pif, dp, (size_t)B * T * K)); TRY(x.down(totals, dt, (size_t)B * T)); TRY(x.down(loglik, dl, (size_t)B));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return HMCGPU_OK;
}

extern "C" int hmcgpu_filter(hmcgpu_ctx* ctx, int32_t precision, int32_t K, int64_t B, int64_t T, const double* y,
                             int64_t ystride, const double* A, const double* mu, const double* sigma2, const double* rho,
                             double* pif, double* totals, double* loglik) {
    return filter_impl(ctx, precision, K, B, T, y, ystride, nullptr, 1.0, A, mu, sigma2, rho, pif, totals, loglik);
}

extern "C" int hmcgpu_filter_masked(hmcgpu_ctx* ctx, int32_t precision, int32_t K, int64_t B, int64_t T, const double* y,
                                    int64_t ystride, const uint8_t* is_signal, double kappa, const double* A, const double* mu,
                                    const double* sigma2, const double* rho, double* pif, double* totals, double* loglik) {
    return filter_impl(ctx, precision, K, B, T, y, ystride, is_signal, kappa, A, mu, sigma2, rho, pif, totals, loglik);
}

extern "C" int hmcgpu_smooth(hmcgpu_ctx* ctx, int32_t precision, int32_t K, int64_t B, int64_t T, const double* A,
                             const double* pif, double* pib) {
    TRY(check_common(ctx, K, B, T));
    if (!A || !pif || !pib) return fail(ctx, HMCGPU_ERR_ARG, "NULL input");
    if (precision != 32 && precision != 64) return fail(ctx, HMCGPU_ERR_ARG, "precision must be 32 or 64");
    Xfer x{ctx};
    double *dA, *dp, *db;
    TRY(x.up(A, (size_t)B * K * K, &dA)); TRY(x.up(pif, (size_t)B * T * K, &dp)); TRY(x.up((double*)nullptr, (size_t)B * T * K, &db));
    if (!k_thread(K)) {
        if (precision == 32) smooth_kernel_generic<float><<<grid_for(B, 64), 64, 0, ctx->stream>>>(K, B, T, dA, dp, db);
        else smooth_kernel_generic<double><<<grid_for(B, 64), 64, 0, ctx->stream>>>(K, B, T, dA, dp, db);
    }
    DISPATCH_K(K, {
        if (precision == 32) smooth_kernel<float, KK><<<grid_for(B, 64), 64, 0, ctx->stream>>>(B, T, dA, dp, db);
        else smooth_kernel<double, KK><<<grid_for(B, 64), 64, 0, ctx->stream>>>(B, T, dA, dp, db);
    });
    CU(ctx, cudaGetLastError());
    TRY(x.down(pib, db, (size_t)B * T * K));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return HMCGPU_OK;
}

extern "C" int hmcgpu_sample_states(hmcgpu_ctx* ctx, int32_t K, int64_t B, int64_t T, const double* A, const double* pif,
                                    const double* piN, const double* u, int64_t* X) {
    TRY(check_common(ctx, K, B, T));
    if (!A || !pif || !u || !X) return fail(ctx, HMCGPU_ERR_ARG, "NULL input");
    Xfer x{ctx};
    double *dA, *dp, *dn = nullptr, *du;
    long long* dX;
    TRY(x.up(A, (size_t)B * K * K, &dA)); TRY(x.up(pif, (size_t)B * T * K, &dp)); TRY(x.up(u, (size_t)B * T, &du));
    if (piN) TRY(x.up(piN, (size_t)B * K, &dn));
    TRY(x.up((long long*)nullptr, (size_t)B * T, &dX));
    if (!k_thread(K)) sample_states_kernel_generic<<<grid_for(B, 64), 64, 0, ctx->stream>>>(K, B, T, dA, dp, dn, du, dX);
    DISPATCH_K(K, { sample_states_kernel<KK><<<grid_for(B, 64), 64, 0, ctx->stream>>>(B, T, dA, dp, dn, du, dX); });
    CU(ctx, cudaGetLastError());
    TRY(x.down(reinterpret_cast<long long*>(X), dX, (size_t)B * T));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return HMCGPU_OK;
}

static int draw_params_impl(hmcgpu_ctx* ctx, int32_t precision, int32_t K, int64_t B, const int64_t* Ni,
                            const double* S, const double* S2, const int64_t* Mi, const double* Sm, const double* Sm2, double kappa,
                            const int64_t* trans, const double* xi,
                            const double* alpha, const double* nu, const double* beta, uint64_t seed,
                            uint32_t chain0, uint32_t sweep, double* sigma2, double* mu, double* rho, double* A) {
    TRY(check_common(ctx, K, B, 1));
    if (Mi && (!Sm || !Sm2)) return fail(ctx, HMCGPU_ERR_ARG, "Mi given without Sm / Sm2");
    if (Mi && !k_thread(K)) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "signal statistics are only implemented for K <= 4");
    if (Mi && !(kappa >= 0.0)) return fail(ctx, HMCGPU_ERR_ARG, "kappa must be >= 0");
    if (!Ni || !S || !S2 || !trans || !xi || !alpha || !nu || !beta || !sigma2 || !mu || !rho || !A)
        return fail(ctx, HMCGPU_ERR_ARG, "NULL input");
    if (precision != 32 && precision != 64) return fail(ctx, HMCGPU_ERR_ARG, "precision must be 32 or 64");
    Xfer x{ctx};
    long long *dN, *dT;
    double *dS, *dS2, *dxi, *dal, *dnu, *dbe, *o1, *o2, *o3, *o4;
    TRY(x.up(reinterpret_cast<const long long*>(Ni), (size_t)B * K, &dN));
    TRY(x.up(reinterpret_cast<const long long*>(trans), (size_t)B * K * K, &dT));
    TRY(x.up(S, (size_t)B * K, &dS)); TRY(x.up(S2, (size_t)B * K, &dS2));
    TRY(x.up(xi, (size_t)K, &dxi)); TRY(x.up(alpha, (size_t)K, &dal)); TRY(x.up(nu, (size_t)K, &dnu)); TRY(x.up(beta, (size_t)K, &dbe));
    TRY(x.up((double*)nullptr, (size_t)B * K, &o1)); TRY(x.up((double*)nullptr, (size_t)B * K, &o2));
    TRY(x.up((double*)nullptr, (size_t)B * K, &o3)); TRY(x.up((double*)nullptr, (size_t)B * K * K, &o4));
    long long* dM = nullptr;
    double *dSm = nullptr, *dSm2 = nullptr;
    if (Mi) {
        TRY(x.up(reinterpret_cast<const long long*>(Mi), (size_t)B * K, &dM));
        TRY(x.up(Sm, (size_t)B * K, &dSm)); TRY(x.up(Sm2, (size_t)B * K, &dSm2));
    }
    const unsigned k0 = (unsigned)seed, k1 = (unsigned)(seed >> 32);
    if (!k_thread(K)) {
        if (precision == 32) draw_params_kernel_generic<float><<<grid_for(B, 64), 64, 0, ctx->stream>>>(K, B, dN, dS, dS2, dT, dxi, dal, dnu, dbe, k0, k1, chain0, sweep, o1, o2, o3, o4);
        else draw_params_kernel_generic<double><<<grid_for(B, 64), 64, 0, ctx->stream>>>(K, B, dN, dS, dS2, dT, dxi, dal, dnu, dbe, k0, k1, chain0, sweep, o1, o2, o3, o4);
    }
    DISPATCH_K(K, {
        if (precision == 32) draw_params_kernel<float, KK><<<grid_for(B, 64), 64, 0, ctx->stream>>>(B, dN, dS, dS2, dM, dSm, dSm2, kappa, dT, dxi, dal, dnu, dbe, k0, k1, chain0, sweep, o1, o2, o3, o4);
        else draw_params_kernel<double, KK><<<grid_for(B, 64), 64, 0, ctx->stream>>>(B, dN, dS, dS2, dM, dSm, dSm2, kappa, dT, dxi, dal, dnu, dbe, k0, k1, chain0, sweep, o1, o2, o3, o4);
    });
    CU(ctx, cudaGetLastError());
    TRY(x.down(sigma2, o1, (size_t)B * K)); TRY(x.down(mu, o2, (size_t)B * K)); TRY(x.down(rho, o3, (size_t)B * K));
    TRY(x.down(A, o4, (size_t)B * K * K));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return HMCGPU_OK;
}

extern "C" int hmcgpu_draw_params(hmcgpu_ctx* ctx, int32_t precision, int32_t K, int64_t B, const int64_t* Ni,
                                  const double* S, const double* S2, const int64_t* trans, const double* xi,
                                  const double* alpha, const double* nu, const double* beta, uint64_t seed,
                                  uint32_t chain0, uint32_t sweep, double* sigma2, double* mu, double* rho, double* A) {
    return draw_params_impl(ctx, precision, K, B, Ni, S, S2, nullptr, nullptr, nullptr, 1.0, trans, xi, alpha, nu, beta, seed, chain0,
                            sweep, sigma2, mu, rho, A);
}

extern "C" int hmcgpu_draw_params_signals(hmcgpu_ctx* ctx, int32_t precision, int32_t K, int64_t B, const int64_t* Ni,
                                          const double* S, const double* S2, const int64_t* Mi, const double* Sm, const double* Sm2,
                                          double kappa, const int64_t* trans, const double* xi, const double* alpha,
                                          const double* nu, const double* beta, uint64_t seed, uint32_t chain0, uint32_t sweep,
                                          double* sigma2, double* mu, double* rho, double* A) {
    if (!Mi) return fail(ctx, HMCGPU_ERR_ARG, "Mi is NULL");
    return draw_params_impl(ctx, precision, K, B, Ni, S, S2, Mi, Sm, Sm2, kappa, trans, xi, alpha, nu, beta, seed, chain0, sweep,
                            sigma2, mu, rho, A);
}

extern "C" int hmcgpu_forecast(hmcgpu_ctx* ctx, int32_t K, int64_t B, const double* mu, const double* A, const double* pi,
                               const int32_t* horizons, int32_t n_h, const double* yreal, double* out) {
    TRY(check_common(ctx, K, B, 1));
    if (!mu || !A || !pi || !horizons || !yreal || !out || n_h <= 0) return fail(ctx, HMCGPU_ERR_ARG, "NULL/empty input");
    for (int j = 0; j < n_h; ++j) if (horizons[j] < 0) return fail(ctx, HMCGPU_ERR_ARG, "negative horizon");
    Xfer x{ctx};
    double *dm, *dA, *dp, *dy, *dout;
    int* dh;
    TRY(x.up(mu, (size_t)B * K, &dm)); TRY(x.up(A, (size_t)B * K * K, &dA)); TRY(x.up(pi, (size_t)B * K, &dp));
    TRY(x.up(yreal, (size_t)n_h, &dy)); TRY(x.up(horizons, (size_t)n_h, &dh)); TRY(x.up((double*)nullptr, (size_t)B * 2 * n_h, &dout));
    if (!k_thread(K)) forecast_kernel_generic<<<grid_for(B, 64), 64, 0, ctx->stream>>>(K, B, dm, dA, dp, dh, n_h, dy, dout);
    DISPATCH_K(K, { forecast_kernel<KK><<<grid_for(B, 64), 64, 0, ctx->stream>>>(B, dm, dA, dp, dh, n_h, dy, dout); });
    CU(ctx, cudaGetLastError());
    TRY(x.down(out, dout, (size_t)B * 2 * n_h));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return HMCGPU_OK;
}

extern "C" int hmcgpu_philox_rounds(hmcgpu_ctx* ctx, int32_t rounds, int64_t n, const uint32_t* ctr, const uint32_t* key, uint32_t* out);
extern "C" int hmcgpu_philox(hmcgpu_ctx* ctx, int64_t n, const uint32_t* ctr, const uint32_t* key, uint32_t* out) {
    return hmcgpu_philox_rounds(ctx, 10, n, ctr, key, out);
}

extern "C" int hmcgpu_philox_rounds(hmcgpu_ctx* ctx, int32_t rounds, int64_t n, const uint32_t* ctr, const uint32_t* key, uint32_t* out) {
    if (!ctx || n <= 0 || !ctr || !key || !out) return fail(ctx, HMCGPU_ERR_ARG, "bad arguments");
    if (rounds != 10 && rounds != kStateRounds) return fail(ctx, HMCGPU_ERR_ARG, "rounds must be 10 (parameter draws) or %d (state uniforms)", kStateRounds);
    CU(ctx, cudaSetDevice(ctx->device));
    tl_pool = ctx->pool;
    Xfer x{ctx};
    unsigned *dc, *dk, *dout;
    TRY(x.up(ctr, (size_t)n * 4, &dc)); TRY(x.up(key, (size_t)n * 2, &dk)); TRY(x.up((unsigned*)nullptr, (size_t)n * 4, &dout));
    philox_kernel<<<grid_for(n, 128), 128, 0, ctx->stream>>>(n, rounds, dc, dk, dout);
    CU(ctx, cudaGetLastError());
    TRY(x.down(out, dout, (size_t)n * 4));
    CU(ctx, cudaStreamSynchronize(ctx->stream));
    return HMCGPU_OK;
}

// ============================================================================================ estimation plan
// ---- window initialisation: HyperParams (:132-142) + makeParams (:161-195) + the statistics of X0, one block per window
struct WinInit {          // per window, fp64
    double mean;          // ξ default and the shift c
    double cnt[32], Sd[32], Qd[32], trans[1024];
    double totS, totQ;    // sum over the window's observations of (y-mean), (y-mean)^2
    // noisy signals (src/Hmc.jl:267-300): cnt/Sd/Qd/totS/totQ above then cover the plain observations only
    double cntM[32], Sm[32], Qm[32], totSm, totQm, totM;
};

__device__ __forceinline__ unsigned long long orderable(double v) {
    unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return (b & 0x8000000000000000ull) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double from_orderable(unsigned long long k) {
    unsigned long long b = (k & 0x8000000000000000ull) ? (k & 0x7fffffffffffffffull) : ~k;
    return __longlong_as_double((long long)b);
}

template <typename T, typename Op>
__device__ T block_reduce(T v, T* sh, Op op) {   // deterministic tree, result broadcast
    const int tid = threadIdx.x;
    sh[tid] = v;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (tid < s) sh[tid] = op(sh[tid], sh[tid + s]);
        __syncthreads();
    }
    T r = sh[0];
    __syncthreads();
    return r;
}

// k-th smallest (0-based) by radix select on the order-preserving 64-bit image of the doubles: passes of 4 bits from the top,
// per-warp histograms in shared memory (sh: at least 8 x 16 + 16 + 2 words), bins summed by 16 threads and walked by one; as soon
// as the selected bin holds a single candidate (typically after the exponent and ~3 mantissa digits) that element is the answer
__device__ double block_select(const double* y, size_t yld, int N, int k, unsigned long long* sh) {
    unsigned* const hist = reinterpret_cast<unsigned*>(sh);       // [warp][16]
    const int nwarp = (int)(blockDim.x >> 5), warp = (int)(threadIdx.x >> 5);
    unsigned* const bins = hist + nwarp * 16;                     // [16] block totals
    unsigned* const pick = bins + 16;                             // [0] digit, [1] k inside the bin, [2] candidates in the bin
    unsigned long long* const found = sh + 128;                   // the single remaining candidate (behind the histograms in the 256 x 8-byte scratch)
    unsigned long long prefix = 0, mask = 0;
    for (int shift = 60; shift >= 0; shift -= 4) {
        for (int q = threadIdx.x; q < nwarp * 16; q += blockDim.x) hist[q] = 0u;
        __syncthreads();
        for (int i = threadIdx.x; i < N; i += blockDim.x) {
            const unsigned long long key = orderable(y[(size_t)i * yld]);
            if ((key & mask) == prefix) atomicAdd(&hist[warp * 16 + (int)((key >> shift) & 15ull)], 1u);
        }
        __syncthreads();
        if (threadIdx.x < 16) {
            unsigned c = 0;
            for (int w = 0; w < nwarp; ++w) c += hist[w * 16 + threadIdx.x];
            bins[threadIdx.x] = c;
        }
        __syncthreads();
        if (threadIdx.x == 0) {
            int digit = 15, kk = k;
            for (int b = 0; b < 16; ++b) {
                if ((unsigned)kk < bins[b]) { digit = b; break; }
                kk -= (int)bins[b];
            }
            pick[0] = (unsigned)digit; pick[1] = (unsigned)kk; pick[2] = bins[digit];
        }
        __syncthreads();
        prefix |= (unsigned long long)pick[0] << shift;
        mask |= 15ull << shift;
        k = (int)pick[1];
        if (pick[2] == 1u && shift > 0) {                         // one candidate left: fetch it
            for (int i = threadIdx.x; i < N; i += blockDim.x) {
                const unsigned long long key = orderable(y[(size_t)i * yld]);
                if ((key & mask) == prefix) *found = key;
            }
            __syncthreads();
            prefix = *found;
            __syncthreads();
            break;
        }
    }
    __syncthreads();
    return from_orderable(prefix);
}

// y: the series the chain runs on; yi: the series the makeParams / HyperParams rules read (estimatesignals! initialises
// from the real data and estimates on a perturbed copy, :888-892); sig: signal flag per absolute time index (or NULL);
// X0u: user-supplied initial paths (1-based states) at offset x0_off[w] (or NULL = makeParams rule).
__global__ void __launch_bounds__(256) window_init_kernel(int K, const double* __restrict__ y64, int yld,
                                                          const long long* __restrict__ wbase, const long long* __restrict__ wbase_init,
                                                          const int* __restrict__ wT, const unsigned char* __restrict__ sig,
                                                          const long long* __restrict__ wsbase, int sld,
                                                          const long long* __restrict__ X0u, const long long* __restrict__ x0_off,
                                                          WinInit* __restrict__ out) {
    extern __shared__ unsigned char x0[];                 // X0, one byte per time step
    __shared__ double shd[256];
    __shared__ unsigned long long shu[256];
    __shared__ double mu0[32];
    const int w = blockIdx.x;
    const int N = wT[w];
    const double* y = y64 + wbase[w];
    const double* yi = wbase_init ? y64 + wbase_init[w] : y;
    const unsigned char* sg = sig ? sig + wsbase[w] : nullptr;          // time-major mask, stride sld between time steps
    const size_t ld = (size_t)yld;
    auto add = [](double a, double b) { return a + b; };
    double s = 0.0, mn = 1e300, mx = -1e300;
    for (int i = threadIdx.x; i < N; i += blockDim.x) { const double v = yi[i * ld]; s += v; mn = fmin(mn, v); mx = fmax(mx, v); }
    const double mean = block_reduce<double>(s, shd, add) / N;
    mn = block_reduce<double>(mn, shd, [](double a, double b) { return fmin(a, b); });
    mx = block_reduce<double>(mx, shd, [](double a, double b) { return fmax(a, b); });
    double ss = 0.0;
    for (int i = threadIdx.x; i < N; i += blockDim.x) { const double d = yi[i * ld] - mean; ss += d * d; }
    const double sd = sqrt(block_reduce<double>(ss, shd, add) / (N - 1));             // Statistics.std (:177)
    double med = block_select(yi, ld, N, N / 2, shu);
    if (!(N & 1)) med = 0.5 * (block_select(yi, ld, N, N / 2 - 1, shu) + med);
    // :175-176.  Rounded operation by operation (no FMA contraction), like the oracle: with an odd window length and an
    // even K the median observation sits exactly on the boundary between two initial states, and which side it falls on
    // is decided by the last bit of these grid points.
    const double R = mx - mn, lo = __dsub_rn(med, __dmul_rn(0.25, R)), hi = __dadd_rn(med, __dmul_rn(0.25, R));
    if ((int)threadIdx.x < K)
        mu0[threadIdx.x] = (K > 1) ? __dadd_rn(lo, __dmul_rn(__dsub_rn(hi, lo), (double)threadIdx.x / (double)(K - 1))) : med;
    __syncthreads();
    for (int i = threadIdx.x; i < N; i += blockDim.x) {                               // :185-187 findmax of the pdfs
        if (X0u) { x0[i] = (unsigned char)(X0u[x0_off[w] + i] - 1); continue; }
        const double v = yi[i * ld];
        // first maximum of pdf(Normal(mu0_k, sd), v) = first minimum of |v - mu0_k| (all states share sd): exact, independent of
        // the exp implementation and of the last bits of sd, so near-ties (the median observation between two grid points)
        // resolve exactly as in the oracle; exact ties go to the lower state like findmax
        int best = 0;
        double bv = fabs(__dsub_rn(v, mu0[0]));
        for (int k = 1; k < K; ++k) {
            const double pv = fabs(__dsub_rn(v, mu0[k]));
            if (pv < bv) { bv = pv; best = k; }
        }
        x0[i] = (unsigned char)best;
    }
    __syncthreads();
    // statistics of X0, deterministic (fixed reduction trees; the integer counts are exact in any order).  Transition pairs: integer
    // atomics on a shared K x K table.  Per-state sums: one warp per state, lanes striding through time, shuffle tree.  (A single
    // thread per quantity walking the window in time order made this kernel 15 ms for 65 536 windows of 2000 observations.)
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarp = (int)(blockDim.x >> 5);
    __shared__ int trc[32 * 32];
    __shared__ double stat[6][32];
    for (int q = tid; q < K * K; q += blockDim.x) trc[q] = 0;
    __syncthreads();
    for (int i = tid; i + 1 < N; i += blockDim.x) atomicAdd(&trc[(int)x0[i] * K + (int)x0[i + 1]], 1);
    for (int q = warp; q < K; q += nwarp) {
        double c = 0.0, sdv = 0.0, qd = 0.0, cm = 0.0, sm = 0.0, qm = 0.0;
        for (int i = lane; i < N; i += 32)
            if (x0[i] == q) {
                const double d = y[i * ld] - mean;
                if (sg && sg[(size_t)i * sld]) { cm += 1.0; sm += d; qm += d * d; }
                else { c += 1.0; sdv += d; qd += d * d; }
            }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            c += __shfl_xor_sync(0xffffffffu, c, o); sdv += __shfl_xor_sync(0xffffffffu, sdv, o); qd += __shfl_xor_sync(0xffffffffu, qd, o);
            cm += __shfl_xor_sync(0xffffffffu, cm, o); sm += __shfl_xor_sync(0xffffffffu, sm, o); qm += __shfl_xor_sync(0xffffffffu, qm, o);
        }
        if (lane == 0) { stat[0][q] = c; stat[1][q] = sdv; stat[2][q] = qd; stat[3][q] = cm; stat[4][q] = sm; stat[5][q] = qm; }
    }
    __syncthreads();
    for (int q = tid; q < K; q += blockDim.x) {
        out[w].cnt[q] = stat[0][q]; out[w].Sd[q] = stat[1][q]; out[w].Qd[q] = stat[2][q];
        out[w].cntM[q] = stat[3][q]; out[w].Sm[q] = stat[4][q]; out[w].Qm[q] = stat[5][q];
    }
    for (int j = tid; j < K * K; j += blockDim.x) out[w].trans[j] = (double)trc[j];
    if (tid == 0) {
        out[w].mean = mean;
        // window totals of both classes = the per-state sums added in state order (the kernels derive the last state's statistics
        // as total minus the others: the two are consistent to the last bit by construction)
        double a = 0.0, b = 0.0, am = 0.0, bm = 0.0, m = 0.0;
        for (int q = 0; q < K; ++q) { a += stat[1][q]; b += stat[2][q]; am += stat[4][q]; bm += stat[5][q]; m += stat[3][q]; }
        out[w].totS = a; out[w].totQ = b; out[w].totSm = am; out[w].totQm = bm; out[w].totM = m;
    }
}

template <typename R>
__global__ void chain_init_kernel(int K, int n_slots, const int* __restrict__ slot_win, const WinInit* __restrict__ wi,
                                  const double* __restrict__ xi_user, int* cnt, int* trans, R* Sd, R* Qd, R* cshift, R* xi,
                                  R* totS, R* totQ, int* events, int* cntM, R* Sm, R* Qm, R* totSm, R* totQm, int* totM) {
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n_slots) return;
    const int w = slot_win[slot];
    events[slot] = 0;
    for (int i = 0; i < K; ++i) {
        cnt[i * n_slots + slot] = w < 0 ? 0 : (int)wi[w].cnt[i];
        Sd[i * n_slots + slot] = w < 0 ? R(0) : (R)wi[w].Sd[i];
        Qd[i * n_slots + slot] = w < 0 ? R(0) : (R)wi[w].Qd[i];
        xi[i * n_slots + slot] = w < 0 ? R(0) : (R)(xi_user ? xi_user[i] : wi[w].mean);
        if (cntM) {
            cntM[i * n_slots + slot] = w < 0 ? 0 : (int)wi[w].cntM[i];
            Sm[i * n_slots + slot] = w < 0 ? R(0) : (R)wi[w].Sm[i];
            Qm[i * n_slots + slot] = w < 0 ? R(0) : (R)wi[w].Qm[i];
        }
        for (int j = 0; j < K; ++j) trans[(i * K + j) * n_slots + slot] = w < 0 ? 0 : (int)wi[w].trans[i * K + j];
    }
    cshift[slot] = w < 0 ? R(0) : (R)wi[w].mean;
    totS[slot] = w < 0 ? R(0) : (R)wi[w].totS;
    totQ[slot] = w < 0 ? R(0) : (R)wi[w].totQ;
    if (cntM) {
        totSm[slot] = w < 0 ? R(0) : (R)wi[w].totSm;
        totQm[slot] = w < 0 ? R(0) : (R)wi[w].totQm;
        totM[slot] = w < 0 ? 0 : (int)wi[w].totM;
    }
}

// signal mask (series-major [S][y_len] as the host gives it, S = 1 or n_series) -> time-major [y_len][S] flags and the
// emission z-scale: +1 = observation, -1/(1+kappa) = signal (the sign is the signal flag)
template <typename R>
__global__ void sigw_kernel(long long y_len, int S, const unsigned char* __restrict__ sig, double kappa,
                            unsigned char* __restrict__ mask_tm, R* __restrict__ out) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= y_len * S) return;
    const long long t = i / S;
    const int s = (int)(i % S);
    const bool f = sig && sig[(long long)s * y_len + t];
    if (mask_tm) mask_tm[i] = f ? 1 : 0;
    out[i] = f ? (R)(-1.0 / (1.0 + kappa)) : R(1);
}

// y (fp64, series-major as the host gives it) -> time-major copy in the sweep precision (yr[t * n_series + s]); 32 x 32 tiles
// through shared memory so that both the reads (along time) and the writes (along the series) are coalesced
template <typename R>
__global__ void __launch_bounds__(256) y_layout_kernel(long long y_len, int n_series, const double* __restrict__ in, R* __restrict__ yr) {
    __shared__ double tile[32][33];
    const long long s0 = (long long)blockIdx.x * 32, t0 = (long long)blockIdx.y * 32;
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;          // 32 x 8 threads
#pragma unroll
    for (int j = ty; j < 32; j += 8) {
        const long long sidx = s0 + j, t = t0 + tx;
        if (sidx < n_series && t < y_len) tile[j][tx] = in[sidx * y_len + t];
    }
    __syncthreads();
#pragma unroll
    for (int j = ty; j < 32; j += 8) {
        const long long t = t0 + j, sidx = s0 + tx;
        if (sidx < n_series && t < y_len) yr[t * n_series + sidx] = (R)tile[tx][j];
    }
}

// per-window posterior summaries from the accumulated sums: mean and (population) variance over the n saved draws of a window;
// the log-likelihood field (last of the F) is zero unless it was produced
__global__ void summary_finish_kernel(long long n_elems, int F, double n, int has_loglik, const double* __restrict__ sum,
                                      const double* __restrict__ sumsq, double* __restrict__ mean, double* __restrict__ var) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i >= n_elems) return;
    const bool zero = !has_loglik && (int)(i % F) == F - 1;
    const double m = sum[i] / n;
    mean[i] = zero ? 0.0 : m;
    var[i] = zero ? 0.0 : fmax(0.0, __dsub_rn(sumsq[i] / n, __dmul_rn(m, m)));      // rounded operation by operation, as the host did
}

// per-date posterior means (pib_mean, insample_forecast_mean) from the sums over the n saved draws of a window
__global__ void mean_finish_kernel(long long n_elems, double n, const double* __restrict__ sum, double* __restrict__ mean) {
    const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (i < n_elems) mean[i] = sum[i] / n;
}

template <typename R>
__global__ void yfut_kernel(int n_slots, int n_h, const int* __restrict__ slot_win, const double* __restrict__ yfut_w, R* __restrict__ out) {
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n_slots) return;
    const int w = slot_win[slot];
    for (int j = 0; j < n_h; ++j) out[(size_t)j * n_slots + slot] = w < 0 ? R(0) : (R)yfut_w[(size_t)w * n_h + j];
}

// ---- per-chunk post-processing
// chunk buffer out[(f*chunk + i)*n_slots + slot]  ->  Julia column-major per-window draw arrays (fp64)
template <typename R>
__global__ void gather_draws_kernel(int K, int n_h, int n_slots, int chunk, int n_i, long long draw0, long long nrun, int n_chains,
                                    const int* __restrict__ slot_win, const int* __restrict__ slot_chain,
                                    const R* __restrict__ out, double* mu, double* sig2, double* A, double* pie, double* fc, double* ll) {
    const int i = blockIdx.y * blockDim.y + threadIdx.y;
    const int slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= n_slots || i >= n_i) return;
    const int w = slot_win[slot];
    if (w < 0) return;
    const long long Rr = (long long)n_chains * nrun;
    const long long d = (long long)slot_chain[slot] * nrun + draw0 + i;
    const size_t cs = (size_t)chunk * n_slots;
    const R* o = out + (size_t)i * n_slots + slot;
    int f = 0;
    for (int k = 0; k < K; ++k, ++f) if (mu) mu[(size_t)w * Rr * K + (size_t)k * Rr + d] = (double)o[f * cs];
    for (int k = 0; k < K; ++k, ++f) if (sig2) sig2[(size_t)w * Rr * K + (size_t)k * Rr + d] = (double)o[f * cs];
    for (int k = 0; k < K * K; ++k, ++f) if (A) A[(size_t)w * Rr * K * K + (size_t)k * Rr + d] = (double)o[f * cs];
    for (int k = 0; k < K; ++k, ++f) if (pie) pie[(size_t)w * Rr * K + (size_t)k * Rr + d] = (double)o[f * cs];
    for (int k = 0; k < 2 * n_h; ++k, ++f) if (fc) fc[(size_t)w * Rr * 2 * n_h + (size_t)k * Rr + d] = (double)o[f * cs];
    if (ll) ll[(size_t)w * Rr + d] = (double)o[f * cs];
}

// per (window, field): sum and sum of squares over the window's chains and the chunk's draws, accumulated in fp64
template <typename R>
__global__ void __launch_bounds__(128) summary_accum_kernel(int F, int n_slots, int chunk, int n_i, int n_chains,
                                                            const int* __restrict__ win_slot0, const R* __restrict__ out,
                                                            double* __restrict__ sum, double* __restrict__ sumsq) {
    __shared__ double sh[128];
    const int w = blockIdx.x, f = blockIdx.y;
    const int s0 = win_slot0[w];
    double a = 0.0, b = 0.0;
    const long long n = (long long)n_chains * n_i;
    for (long long j = threadIdx.x; j < n; j += blockDim.x) {
        const int cidx = (int)(j % n_chains), i = (int)(j / n_chains);
        const double v = (double)out[((size_t)f * chunk + i) * n_slots + s0 + cidx];
        a += v; b += v * v;
    }
    auto add = [](double x, double y2) { return x + y2; };
    a = block_reduce<double>(a, sh, add);
    b = block_reduce<double>(b, sh, add);
    if (threadIdx.x == 0) { sum[(size_t)w * F + f] += a; sumsq[(size_t)w * F + f] += b; }
}

// smoothed-probability sums of this chunk, pooled over the window's chains, added to the fp64 per-window accumulator
// Tile of per-(row, column) sums: tile[(row*ncols + col)*32 + lane] per warp task at offset warp_pi_off/K*ncols (ncols = K for the
// smoothed probabilities, n_h for the in-sample forecasts).  Pools the window's chains and adds to the fp64 per-window sums.
template <typename R>
__global__ void tile_reduce_kernel(int K, int ncols, int n_chains, const int* __restrict__ win_slot0, const int* __restrict__ wT,
                                   const long long* __restrict__ warp_pi_off, const int* __restrict__ warp_T,
                                   const long long* __restrict__ win_off, R* __restrict__ acc_tile, double* __restrict__ win_sum) {
    const int w = blockIdx.x;
    const int N = wT[w];
    const int s0 = win_slot0[w];
    double* dst = win_sum + win_off[w] / K * ncols;
    for (int e = threadIdx.x; e < N * ncols; e += blockDim.x) {
        const int t = e / ncols, k = e % ncols;
        double acc = 0.0;
        for (int cidx = 0; cidx < n_chains; ++cidx) {
            const int slot = s0 + cidx;
            const int row = t + (warp_T[slot >> 5] - N);     // windows are right-aligned inside their warp task
            R* p = acc_tile + warp_pi_off[slot >> 5] / K * ncols + (size_t)(row * ncols + k) * 32 + (slot & 31);
            acc += (double)*p;
            *p = R(0);
        }
        dst[(size_t)k * N + t] += acc;                       // column-major N_w x ncols
    }
}

struct hmcgpu_plan {
    hmcgpu_ctx* ctx = nullptr;
    // problem (host copies)
    int K = 0, n_chains = 0, n_windows = 0, n_h = 0, precision = 32;
    long long burnin = 0, nrun = 0;
    unsigned flags = 0;
    unsigned long long seed = 0;
    int F = 0;
    std::vector<int> wT;                 // per window (caller order)
    std::vector<int> order;              // windows sorted by T descending: order[j] = caller index
    std::vector<long long> pib_off;      // per window (caller order) offset in pib_mean
    std::vector<int> slot0;              // per window (caller order) its first chain slot (SlotLayout::win_slot0)
    long long state_steps = 0;
    int n_slots = 0, n_warps = 0, n_tasks = 0, chunk = 0, max_T = 0;   // (n_tasks: warp tasks of both classes)
    GibbsArgs args{};
    // device buffers
    DevBuf yr, wbase, wTd, wi, slot_win, slot_chain, T, ybase, warp_T, warp_pi_off, pi, pacc, facc, cnt, trans, Sd, Qd,
        events, cshift, xi, xi_user, chain_id, out, yfut_w, yfut, win_slot0, win_pib_off, totS, totQ, slot_pi_off;
    DevBuf sigmask, sigmask_tm, sigw, sbase, wsbase, wbase_init, X0, x0_off, cntM, Sm, Qm, totSm, totQm, totM;    // signals tier / user initial states
    bool sig = false;    // SIG kernels: signal mask and / or pi_row_back
    Tuning tuning;
    SweepChoice sw;
    // fp64 series-major upload, read by the window statistics.  A plan member so that it outlives a failed plan_build until
    // plan_create_impl has drained the stream; released once the stream has drained at the end of plan_build.
    DevBuf yin;
    DevBuf warp_T_long, warp_pi_off_long;     // warp-task tables of the long class (SweepChoice::n_long)
    std::vector<TaskGroup> groups;            // one stream each (plan_run)
    int n_bufs = 1;
    std::vector<cudaStream_t> gstreams;
    std::vector<cudaEvent_t> pool_events;
    std::vector<cudaEvent_t> timing_events;   // pairs around every sweep launch + one end-of-sweeps event per group (timing enabled)
    double launch_ms_sum = 0.0;
    DevBuf d_sum, d_sumsq, d_pibsum, d_fcsum;
    // the per-window outputs (window_outputs), laid out like the caller's arrays: the draws gathered per chunk, the rest
    // finished at fetch
    DevBuf d_mu, d_sig2, d_A, d_pie, d_fc, d_ll, d_mean, d_var, d_pib, d_ifc, d_rhat, d_ess, d_lag, d_cdf, d_pit, d_ls, d_mom, d_quant,
        d_rrank, d_essb, d_esst;
    // HMCGPU_FLAG_DIAGNOSTICS (diagnostics.cuh): streaming state per (slot, field), per-sequence means / variances and lag sums
    // per (window, field)
    DevBuf dg_P, dg_S1, dg_head, dg_ring, dg_mean, dg_var, dg_gsum;
    // HMCGPU_FLAG_PREDICTIVE (predictive.cuh): the grid, the shift c_w per window, running sums per (slot, horizon)
    DevBuf pr_grid, pr_cshift, pr_cdf, pr_score;
    int n_grid = 0, pr_tg = 32, pr_td = 1;    // threads per slot and draws per tile of pred_accum_kernel
    PredHorizons pr_h{};
    // HMCGPU_FLAG_RANKED (ranked.cuh): every saved draw, keep[((w*F + f)*n_chains + c)*nrun + i]
    DevBuf rk_keep;
    // HMCGPU_FLAG_ONESTEP (onestep.cuh): kOsState running values per (slot, date), os_n = n_chains * sum_w T_w of each
    DevBuf os_state, d_ospit, d_oslpd, d_osvar, d_waic;
    long long os_n = 0;
    // HMCGPU_FLAG_LOO (loo.cuh): mu, sigma2, A of every saved draw, keep[((w*F' + f)*n_chains + c)*nrun + i], F' = 2K + K^2
    // (not allocated with HMCGPU_FLAG_RANKED, whose rk_keep holds them); the per-date and per-window outputs
    DevBuf lo_keep, d_lelpd, d_llppd, d_lpk, d_lpit, d_lsum;
    DevBuf d_diag;       // segment kernel: chain-sweeps that fell back to the exact entering vectors
    unsigned long long seg_fallbacks[2] = {0, 0};   // [0] chain-sweeps on the exact path, [1] speculative groups (sum over chain-sweeps)
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, evk0 = nullptr, evk1 = nullptr;
    double gpu_ms = 0.0, sweep_ms = 0.0;
    long long n_launches = 0, n_sweep_launches = 0, h2d = 0, d2h = 0;
    bool ran = false;
    ~hmcgpu_plan() {
        for (auto s2 : gstreams) cudaStreamDestroy(s2);
        for (auto e : pool_events) cudaEventDestroy(e);
        for (auto e : timing_events) cudaEventDestroy(e);
        if (ev0) cudaEventDestroy(ev0);
        if (ev1) cudaEventDestroy(ev1);
        if (evk0) cudaEventDestroy(evk0);
        if (evk1) cudaEventDestroy(evk1);
    }
};

// F: fields per window of the summaries and diagnostics (mu[K], sigma2[K], A[K*K], pi_end[K], forecasts[2*n_h], loglik)
static int summary_fields(int K, int n_h) { return 3 * K + K * K + 2 * n_h + 1; }

// One per-window output of hmcgpu_result / hmcgpu_predictive / hmcgpu_ranked / hmcgpu_onestep / hmcgpu_loo.  Window w holds
// per_window + per_step * T_w elements; the windows are concatenated in caller order, in the caller's array and in the plan's
// device buffer `dev` alike.
enum class OutStruct { result, predictive, ranked, onestep, loo };
struct WinOut {
    const char* name;
    OutStruct in;              // the struct that holds the caller's pointer
    size_t field;              // offset of the caller's pointer in that struct
    size_t elem;               // bytes per element
    long long per_window, per_step;
    bool on;                   // the flags produce it
    bool gated;                // the caller's pointer is read only when `on` (fields appended to the ABI: older structs end before them)
    const char* need;          // the flag that is missing when it is not on
    DevBuf hmcgpu_plan::*dev;  // NULL for status, which is read from the chain slots
    // elements of n windows of sum_T steps in all; elems(w, T_0 + ... + T_{w-1}) is the offset of window w
    long long elems(long long n, long long sum_T) const { return per_window * n + per_step * sum_T; }
    void* base(const hmcgpu_result* r, const hmcgpu_predictive* pr, const hmcgpu_ranked* rk, const hmcgpu_onestep* os,
               const hmcgpu_loo* lo) const {
        switch (in) {
            case OutStruct::result: return (void*)r;
            case OutStruct::predictive: return (void*)pr;
            case OutStruct::ranked: return (void*)rk;
            case OutStruct::onestep: return (void*)os;
            default: return (void*)lo;
        }
    }
    // NULL: not requested, or not readable
    void* get(const hmcgpu_result* r, const hmcgpu_predictive* pr, const hmcgpu_ranked* rk = nullptr,
              const hmcgpu_onestep* os = nullptr, const hmcgpu_loo* lo = nullptr) const {
        const void* s = base(r, pr, rk, os, lo);
        void* p = nullptr;
        if (s && (on || !gated)) memcpy(&p, (const char*)s + field, sizeof p);
        return p;
    }
    void set(hmcgpu_result* r, hmcgpu_predictive* pr, hmcgpu_ranked* rk, hmcgpu_onestep* os, hmcgpu_loo* lo, void* p) const {
        memcpy((char*)base(r, pr, rk, os, lo) + field, &p, sizeof p);
    }
};

// n_probs: quantiles per field of the ranked outputs (known at hmcgpu_plan_fetch_ranked)
static std::vector<WinOut> window_outputs(int K, int n_h, int n_chains, long long nrun, int n_grid, int n_probs, unsigned flags) {
    const long long R = (long long)n_chains * nrun, F = summary_fields(K, n_h);
    const bool draws = flags & HMCGPU_FLAG_DRAWS, summary = flags & HMCGPU_FLAG_SUMMARY, diag = flags & HMCGPU_FLAG_DIAGNOSTICS,
               pred = flags & HMCGPU_FLAG_PREDICTIVE, mean = flags & (HMCGPU_FLAG_SMOOTHED_MEAN | HMCGPU_FLAG_FILTERED_MEAN),
               ranked = flags & HMCGPU_FLAG_RANKED, onestep = flags & HMCGPU_FLAG_ONESTEP, loo = flags & HMCGPU_FLAG_LOO;
    const bool ll = draws && (flags & HMCGPU_FLAG_LOGLIK);
    const char* D = "HMCGPU_FLAG_DRAWS";
    const char* M = "HMCGPU_FLAG_SMOOTHED_MEAN or HMCGPU_FLAG_FILTERED_MEAN";
    const size_t f8 = sizeof(double), i4 = sizeof(int32_t);
    using P = hmcgpu_plan;
#define RES(f) #f, OutStruct::result, offsetof(hmcgpu_result, f)
#define PRED(f) #f, OutStruct::predictive, offsetof(hmcgpu_predictive, f)
#define RANK(f) #f, OutStruct::ranked, offsetof(hmcgpu_ranked, f)
#define ONE(f) #f, OutStruct::onestep, offsetof(hmcgpu_onestep, f)
#define LOO(f) #f, OutStruct::loo, offsetof(hmcgpu_loo, f)
    std::vector<WinOut> o = {
        {RES(mu), f8, R * K, 0, draws, false, D, &P::d_mu},
        {RES(sigma2), f8, R * K, 0, draws, false, D, &P::d_sig2},
        {RES(A), f8, R * K * K, 0, draws, false, D, &P::d_A},
        {RES(pi_end), f8, R * K, 0, draws, false, D, &P::d_pie},
        {RES(forecasts), f8, R * 2 * n_h, 0, draws, false, D, &P::d_fc},
        {RES(loglik), f8, R, 0, ll, false, draws ? "HMCGPU_FLAG_LOGLIK" : D, &P::d_ll},
        {RES(summary_mean), f8, F, 0, summary, false, "HMCGPU_FLAG_SUMMARY", &P::d_mean},
        {RES(summary_var), f8, F, 0, summary, false, "HMCGPU_FLAG_SUMMARY", &P::d_var},
        {RES(pib_mean), f8, 0, K, mean, false, M, &P::d_pib},
        {RES(insample_forecast_mean), f8, 0, n_h, mean, false, M, &P::d_ifc},
        {RES(status), i4, n_chains, 0, true, false, "", nullptr},
        {RES(rhat), f8, F, 0, diag, true, "", &P::d_rhat},
        {RES(ess), f8, F, 0, diag, true, "", &P::d_ess},
        {RES(ess_lag), i4, F, 0, diag, true, "", &P::d_lag},
        {PRED(cdf), f8, (long long)n_h * n_grid, 0, pred, true, "", &P::d_cdf},
        {PRED(pit), f8, n_h, 0, pred, true, "", &P::d_pit},
        {PRED(log_score), f8, n_h, 0, pred, true, "", &P::d_ls},
        {PRED(moments), f8, 3ll * n_h, 0, pred, true, "", &P::d_mom},
        {RANK(quantiles), f8, F * n_probs, 0, ranked, true, "", &P::d_quant},
        {RANK(rhat_rank), f8, F, 0, ranked, true, "", &P::d_rrank},
        {RANK(ess_bulk), f8, F, 0, ranked, true, "", &P::d_essb},
        {RANK(ess_tail), f8, F, 0, ranked, true, "", &P::d_esst},
        {ONE(pit), f8, 0, 1, onestep, true, "", &P::d_ospit},
        {ONE(lpd), f8, 0, 1, onestep, true, "", &P::d_oslpd},
        {ONE(lpd_var), f8, 0, 1, onestep, true, "", &P::d_osvar},
        {ONE(waic), f8, 4, 0, onestep, true, "", &P::d_waic},
        {LOO(elpd), f8, 0, 1, loo, true, "", &P::d_lelpd},
        {LOO(lppd), f8, 0, 1, loo, true, "", &P::d_llppd},
        {LOO(pareto_k), f8, 0, 1, loo, true, "", &P::d_lpk},
        {LOO(pit), f8, 0, 1, loo, true, "", &P::d_lpit},
        {LOO(summary), f8, kLooSummary, 0, loo, true, "", &P::d_lsum},
    };
#undef RES
#undef PRED
#undef RANK
#undef ONE
#undef LOO
    return o;
}

static int validate_problem(hmcgpu_ctx* ctx, const hmcgpu_problem* p, const Tuning& t) {
    if (!ctx) return HMCGPU_ERR_ARG;
    if (!p) return fail(ctx, HMCGPU_ERR_ARG, "problem is NULL");
    if (!p->y || p->y_len < 2 || p->n_series < 1) return fail(ctx, HMCGPU_ERR_ARG, "empty series");
    if (p->n_windows < 1 || !p->win_start || !p->win_end) return fail(ctx, HMCGPU_ERR_ARG, "no windows");
    if (!k_supported(p->K)) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "K=%d not supported (2..32)", p->K);
    if (!k_thread_sweep(p->K, t) && (p->flags & HMCGPU_FLAG_SMOOTHED_MEAN))
        return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "smoothed means are only implemented for K <= 8 (thread-per-chain kernels)");
    if (p->K > 4 && (p->flags & (HMCGPU_FLAG_SMOOTHED_MEAN | HMCGPU_FLAG_FILTERED_MEAN)) && p->n_h > 0) {
        // the A^h mu vectors of the in-sample forecasts live in shared memory next to the selection tables and the rings
        const size_t b = p->precision / 8;
        const size_t need = (size_t)(p->K * b + 8 + 15) / 16 * 16 * p->K * 128 + b * 4 * 3 * 4 * p->K * 32 + b * (size_t)p->n_h * (p->K + 1) * 128;
        if (need > 200 * 1024)
            return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "K=%d with %d in-sample forecast horizons needs %zu KB of shared memory per block: use fewer horizons", p->K, p->n_h, need / 1024);
    }
    if (p->flags & HMCGPU_FLAG_FILTERED_MEAN) {
        if (!k_thread_sweep(p->K, t)) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "filtered means are only implemented for K <= 8");
        if (p->flags & HMCGPU_FLAG_SMOOTHED_MEAN) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "HMCGPU_FLAG_FILTERED_MEAN and HMCGPU_FLAG_SMOOTHED_MEAN share their output arrays: one per call");
        if (p->is_signal || p->pi_row_back != 0) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "is_signal / pi_row_back cannot be combined with HMCGPU_FLAG_FILTERED_MEAN");
    }
    if (p->n_chains < 1) return fail(ctx, HMCGPU_ERR_ARG, "n_chains < 1");
    // chain slots are indexed with 32-bit ints (padded to a multiple of 64); the Philox chain id is 32 bits as well
    if ((long long)p->n_windows * p->n_chains > 0x7fffffffLL - 64)
        return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "n_windows * n_chains = %lld exceeds 2^31 - 65 chains per call", (long long)p->n_windows * p->n_chains);
    if (p->burnin < 0 || p->nrun < 1) return fail(ctx, HMCGPU_ERR_ARG, "burnin < 0 or nrun < 1");
    if (p->burnin + p->nrun > 0xffffffffLL) return fail(ctx, HMCGPU_ERR_ARG, "more than 2^32 sweeps");
    if ((p->flags & HMCGPU_FLAG_DIAGNOSTICS) && p->nrun < 4) return fail(ctx, HMCGPU_ERR_ARG, "HMCGPU_FLAG_DIAGNOSTICS needs nrun >= 4 (two sequences of >= 2 draws per chain)");
    if (p->flags & HMCGPU_FLAG_RANKED) {
        if (p->nrun < 4) return fail(ctx, HMCGPU_ERR_ARG, "HMCGPU_FLAG_RANKED needs nrun >= 4 (two sequences of >= 2 draws per chain)");
        // (positions within a field's draws are 32-bit in the sort)
        if ((long long)p->n_chains * p->nrun >= 0x80000000LL)
            return fail(ctx, HMCGPU_ERR_ARG, "HMCGPU_FLAG_RANKED needs n_chains * nrun < 2^31 (got %lld)", (long long)p->n_chains * p->nrun);
    }
    if (p->flags & HMCGPU_FLAG_ONESTEP) {
        if ((long long)p->n_chains * p->nrun < 2)
            return fail(ctx, HMCGPU_ERR_ARG, "HMCGPU_FLAG_ONESTEP needs n_chains * nrun >= 2 draws per window (lpd_var divides by R - 1)");
        if (p->is_signal)
            return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "HMCGPU_FLAG_ONESTEP with is_signal (signal rows have another emission; their scores are not one-step-ahead predictions)");
        if (p->K > kOsMaxK) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "HMCGPU_FLAG_ONESTEP is only implemented for K <= %d (got K=%d)", kOsMaxK, p->K);
    }
    if (p->flags & HMCGPU_FLAG_LOO) {
        const long long R = (long long)p->n_chains * p->nrun;
        if (R < 2) return fail(ctx, HMCGPU_ERR_ARG, "HMCGPU_FLAG_LOO needs n_chains * nrun >= 2 draws per window");
        // (the Pareto tail of up to 3 sqrt(R) values and their draw indices sits in shared memory)
        if (R > kLooMaxDraws)
            return fail(ctx, HMCGPU_ERR_ARG, "HMCGPU_FLAG_LOO needs n_chains * nrun <= 2^24 draws per window (got %lld)", R);
        if (p->is_signal)
            return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "HMCGPU_FLAG_LOO with is_signal (signal rows have another emission; their scores are not predictions of the data)");
        if (p->K > kOsMaxK) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "HMCGPU_FLAG_LOO is only implemented for K <= %d (got K=%d)", kOsMaxK, p->K);
    }
    if (p->precision != 32 && p->precision != 64) return fail(ctx, HMCGPU_ERR_ARG, "precision must be 32 or 64");
    if (p->n_h < 0 || p->n_h > kMaxH || (p->n_h > 0 && !p->horizons)) return fail(ctx, HMCGPU_ERR_ARG, "0 <= n_h <= %d", kMaxH);
    if (p->flags & HMCGPU_FLAG_PREDICTIVE) {
        if (p->n_h == 0) return fail(ctx, HMCGPU_ERR_ARG, "HMCGPU_FLAG_PREDICTIVE needs at least one forecast horizon");
        if (p->n_grid < 1 || p->n_grid > 512 || !p->pred_grid) return fail(ctx, HMCGPU_ERR_ARG, "HMCGPU_FLAG_PREDICTIVE needs 1 <= n_grid <= 512 grid points");
        for (int g = 0; g < p->n_grid; ++g) {
            if (!std::isfinite(p->pred_grid[g])) return fail(ctx, HMCGPU_ERR_ARG, "pred_grid[%d] is not finite", g);
            if (g > 0 && !(p->pred_grid[g] > p->pred_grid[g - 1])) return fail(ctx, HMCGPU_ERR_ARG, "pred_grid is not strictly increasing at %d", g);
        }
        if (p->pi_row_back != 0)
            return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "HMCGPU_FLAG_PREDICTIVE with pi_row_back != 0 (pi_end is then a smoothed row, not the forecasts' vector)");
    }
    if (p->is_signal || p->pi_row_back != 0) {
        if (!k_thread(p->K)) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "is_signal / pi_row_back are only implemented for K <= 4");
        if (p->flags & HMCGPU_FLAG_SMOOTHED_MEAN) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "is_signal / pi_row_back cannot be combined with HMCGPU_FLAG_SMOOTHED_MEAN");
        if (p->is_signal && !(p->kappa >= 0.0)) return fail(ctx, HMCGPU_ERR_ARG, "kappa must be >= 0 with is_signal");
        if (p->pi_row_back < 0) return fail(ctx, HMCGPU_ERR_ARG, "pi_row_back < 0");
    }
    for (int j = 0; j < p->n_h; ++j)
        if (p->horizons[j] < 0 || p->horizons[j] > kMaxHorizon) return fail(ctx, HMCGPU_ERR_ARG, "horizons must be in 0..%d", kMaxHorizon);
    // The InverseGamma draw needs a > 0 and b > 0 (the reference catches the exception and keeps the old value, :319-329);
    // with positive priors both always hold for finite statistics, so a skipped draw can only follow a NaN.
    for (int i = 0; i < p->K; ++i) {
        if ((p->alpha && !(p->alpha[i] > 0.0)) || (p->nu && !(p->nu[i] > 0.0)) || (p->beta0 && !(p->beta0[i] > 0.0)) || (p->beta && !(p->beta[i] > 0.0)))
            return fail(ctx, HMCGPU_ERR_ARG, "alpha, nu, beta0 and beta must be > 0 (state %d)", i + 1);
        if (p->xi && !std::isfinite(p->xi[i])) return fail(ctx, HMCGPU_ERR_ARG, "xi[%d] is not finite", i);
    }
    for (int w = 0; w < p->n_windows; ++w) {
        // the Philox chain id win_id * n_chains + chain is a 32-bit counter word: ids must not wrap (distinct windows would share streams)
        const long long wid = p->win_id ? (long long)p->win_id[w] : (long long)w;
        if (wid < 0 || (wid + 1) * (long long)p->n_chains > 0x100000000LL)
            return fail(ctx, HMCGPU_ERR_ARG, "window %d: win_id %lld with %d chains per window leaves the 32-bit chain-id range", w, wid, p->n_chains);
        const long long s = p->win_start[w], e = p->win_end[w];
        if (s < 1 || e > p->y_len || e - s + 1 < 2) return fail(ctx, HMCGPU_ERR_ARG, "window %d: [%lld,%lld] outside 1..%lld or shorter than 2", w, s, e, (long long)p->y_len);
        if (p->win_series && (p->win_series[w] < 0 || p->win_series[w] >= p->n_series)) return fail(ctx, HMCGPU_ERR_ARG, "window %d: bad series index", w);
        if (p->win_init_series && (p->win_init_series[w] < 0 || p->win_init_series[w] >= p->n_series)) return fail(ctx, HMCGPU_ERR_ARG, "window %d: bad init series index", w);
        if (p->pi_row_back >= e - s + 1) return fail(ctx, HMCGPU_ERR_ARG, "window %d: pi_row_back %d >= window length", w, p->pi_row_back);
    }
    if (p->X0) {
        size_t off = 0;
        for (int w = 0; w < p->n_windows; ++w) {
            const long long n = (long long)p->win_end[w] - p->win_start[w] + 1;
            for (long long i = 0; i < n; ++i)
                if (p->X0[off + i] < 1 || p->X0[off + i] > p->K) return fail(ctx, HMCGPU_ERR_ARG, "X0: state %lld of window %d is outside 1..%d", (long long)p->X0[off + i], w, p->K);
            off += (size_t)n;
        }
    }
    return 0;
}

template <typename R>
static int plan_build(hmcgpu_plan* pl, const hmcgpu_problem* p) {
    hmcgpu_ctx* ctx = pl->ctx;
    cudaStream_t st = ctx->stream;
    const int K = p->K, nw = p->n_windows, nc = p->n_chains, nser = p->n_series;
    pl->K = K; pl->n_chains = nc; pl->n_windows = nw; pl->n_h = p->n_h; pl->precision = p->precision;
    pl->burnin = p->burnin; pl->nrun = p->nrun; pl->flags = p->flags; pl->seed = p->seed;
    pl->F = summary_fields(K, p->n_h);
    pl->wT.resize(nw);
    pl->order.resize(nw);
    pl->pib_off.resize(nw);
    // per-window tables; forecasts: realised y at end+h per window (NaN outside the series)
    std::vector<long long> wbase(nw), wbase_init(nw), x0_off(nw);
    std::vector<double> yfut_w((size_t)nw * std::max(1, p->n_h), NAN);
    long long sumT = 0, pib_total = 0;
    for (int w = 0; w < nw; ++w) {
        pl->wT[w] = p->win_end[w] - p->win_start[w] + 1;
        pl->pib_off[w] = pib_total;
        pib_total += (long long)pl->wT[w] * K;
        x0_off[w] = sumT;
        sumT += pl->wT[w];
        pl->max_T = std::max(pl->max_T, pl->wT[w]);
        const int ser = p->win_series ? p->win_series[w] : 0;
        // the window statistics read the fp64 series as uploaded (series-major: a window is contiguous)
        wbase[w] = (long long)ser * p->y_len + (p->win_start[w] - 1);
        wbase_init[w] = (long long)(p->win_init_series ? p->win_init_series[w] : ser) * p->y_len + (p->win_start[w] - 1);
        for (int j = 0; j < p->n_h; ++j) {
            const long long idx = (long long)p->win_end[w] + p->horizons[j];   // 1-based
            if (idx <= p->y_len) yfut_w[(size_t)w * p->n_h + j] = p->y[(size_t)ser * p->y_len + idx - 1];
        }
    }
    if (k_thread(K) && (long long)pl->max_T - 1 > ((1ll << (64 / K)) - 1)) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "window too long for K=%d", K);
    pl->state_steps = sumT * nc * (p->burnin + p->nrun);
    std::iota(pl->order.begin(), pl->order.end(), 0);
    std::stable_sort(pl->order.begin(), pl->order.end(), [&](int a, int b) { return pl->wT[a] > pl->wT[b]; });

    pl->sig = p->is_signal != nullptr || p->pi_row_back != 0;
    const char* msg = nullptr;
    if (const int rc = choose_sweep(ctx->sm_count, p, pl->wT, pl->order, pl->tuning, pl->sw, &msg)) return fail(ctx, rc, "%s", msg);
    const SlotLayout lay = layout_slots(p, pl->wT, pl->order, pl->sw, pl->tuning);
    const int n_slots = lay.n_slots, n_warps = lay.n_warps;
    pl->n_slots = n_slots; pl->n_warps = n_warps; pl->n_tasks = lay.n_tasks; pl->groups = lay.groups;
    std::vector<int> hs(p->n_h);                            // horizons sorted ascending
    std::iota(hs.begin(), hs.end(), 0);
    std::stable_sort(hs.begin(), hs.end(), [&](int a, int b) { return p->horizons[a] < p->horizons[b]; });
    const DrawChunks dc = draw_chunks((int)pl->groups.size(), p->flags, pl->F, n_slots, sizeof(R), p->nrun);
    pl->chunk = dc.chunk; pl->n_bufs = dc.n_bufs;
    const unsigned kAccMean = HMCGPU_FLAG_SMOOTHED_MEAN | HMCGPU_FLAG_FILTERED_MEAN;
    const size_t per_draw = (size_t)pl->F * n_slots * sizeof(R);

    // ---- device allocation + upload
    auto up = [&](DevBuf& b, const void* host, size_t bytes) -> cudaError_t {
        cudaError_t e = b.alloc(bytes);
        if (e != cudaSuccess) return e;
        pl->h2d += (long long)bytes;
        return staged_upload(ctx, b.p, host, bytes, st);
    };
    DevBuf& yin = pl->yin;
    const size_t ny = (size_t)p->y_len * nser;
    PhaseTrace tr;
    if ((p->y_len + 31) / 32 > 65535) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "series longer than %d observations", 65535 * 32);
    CU(ctx, pl->yr.alloc(ny * sizeof(R)));
    CU(ctx, up(yin, p->y, ny * sizeof(double)));
    tr.mark("  series upload enqueued");
    y_layout_kernel<R><<<dim3((unsigned)((nser + 31) / 32), (unsigned)((p->y_len + 31) / 32)), 256, 0, st>>>(p->y_len, nser, yin.as<double>(), pl->yr.as<R>());
    CU(ctx, cudaGetLastError());
    tr.sync_mark(st, "  series layout kernel");
    CU(ctx, up(pl->wbase, wbase.data(), nw * sizeof(long long)));
    CU(ctx, up(pl->wTd, pl->wT.data(), nw * sizeof(int)));
    CU(ctx, up(pl->slot_win, lay.slot_win.data(), n_slots * sizeof(int)));
    CU(ctx, up(pl->slot_chain, lay.slot_chain.data(), n_slots * sizeof(int)));
    CU(ctx, up(pl->T, lay.Ts.data(), n_slots * sizeof(int)));
    CU(ctx, up(pl->ybase, lay.ybase.data(), n_slots * sizeof(long long)));
    CU(ctx, up(pl->warp_T, lay.warp_T.data(), n_warps * sizeof(int)));
    CU(ctx, up(pl->warp_pi_off, lay.warp_off.data(), n_warps * sizeof(long long)));
    if (!lay.warp_T_long.empty()) {
        CU(ctx, up(pl->warp_T_long, lay.warp_T_long.data(), lay.warp_T_long.size() * sizeof(int)));
        CU(ctx, up(pl->warp_pi_off_long, lay.warp_off_long.data(), lay.warp_off_long.size() * sizeof(long long)));
    }
    if (pl->sw.kernel == SweepKernel::lane) CU(ctx, up(pl->slot_pi_off, lay.slot_off.data(), n_slots * sizeof(long long)));
    CU(ctx, up(pl->chain_id, lay.chain_id.data(), n_slots * sizeof(unsigned)));
    CU(ctx, up(pl->win_slot0, lay.win_slot0.data(), nw * sizeof(int)));
    pl->slot0 = lay.win_slot0;
    CU(ctx, up(pl->win_pib_off, pl->pib_off.data(), nw * sizeof(long long)));
    CU(ctx, up(pl->yfut_w, yfut_w.data(), yfut_w.size() * sizeof(double)));
    if (p->xi) CU(ctx, up(pl->xi_user, p->xi, K * sizeof(double)));
    if (p->win_init_series) CU(ctx, up(pl->wbase_init, wbase_init.data(), nw * sizeof(long long)));
    if (p->X0) {
        CU(ctx, up(pl->X0, p->X0, (size_t)sumT * sizeof(long long)));
        CU(ctx, up(pl->x0_off, x0_off.data(), nw * sizeof(long long)));
    }
    const int sld = (p->is_signal && p->is_signal_per_series) ? nser : 1;
    if (p->is_signal) CU(ctx, up(pl->sigmask, p->is_signal, (size_t)p->y_len * sld));
    if (pl->sig) {
        std::vector<long long> sbase(n_slots, 0), wsbase(nw, 0);
        for (int w = 0; w < nw; ++w) wsbase[w] = (long long)(p->win_start[w] - 1) * sld + (sld > 1 ? (p->win_series ? p->win_series[w] : 0) : 0);
        for (int slot = 0; slot < n_slots; ++slot) if (lay.slot_win[slot] >= 0) sbase[slot] = wsbase[lay.slot_win[slot]];
        CU(ctx, up(pl->sbase, sbase.data(), n_slots * sizeof(long long)));
        CU(ctx, up(pl->wsbase, wsbase.data(), nw * sizeof(long long)));
        CU(ctx, pl->sigw.alloc((size_t)p->y_len * sld * sizeof(R)));
        CU(ctx, pl->sigmask_tm.alloc((size_t)p->y_len * sld));
        sigw_kernel<R><<<grid_for(p->y_len * sld, 256), 256, 0, st>>>(p->y_len, sld, pl->sigmask.as<unsigned char>(), p->kappa,
                                                                       pl->sigmask_tm.as<unsigned char>(), pl->sigw.as<R>());
        CU(ctx, cudaGetLastError());
        CU(ctx, pl->cntM.alloc((size_t)K * n_slots * sizeof(int)));
        CU(ctx, pl->Sm.alloc((size_t)K * n_slots * sizeof(R)));
        CU(ctx, pl->Qm.alloc((size_t)K * n_slots * sizeof(R)));
        CU(ctx, pl->totSm.alloc((size_t)n_slots * sizeof(R)));
        CU(ctx, pl->totQm.alloc((size_t)n_slots * sizeof(R)));
        CU(ctx, pl->totM.alloc((size_t)n_slots * sizeof(int)));
    }
    CU(ctx, pl->wi.alloc(nw * sizeof(WinInit)));
    CU(ctx, pl->pi.alloc((size_t)lay.pi_elems * sizeof(R)));
    CU(ctx, pl->cnt.alloc((size_t)K * n_slots * sizeof(int)));
    CU(ctx, pl->trans.alloc((size_t)K * K * n_slots * sizeof(int)));
    CU(ctx, pl->Sd.alloc((size_t)K * n_slots * sizeof(R)));
    CU(ctx, pl->Qd.alloc((size_t)K * n_slots * sizeof(R)));
    CU(ctx, pl->events.alloc((size_t)n_slots * sizeof(int)));
    CU(ctx, pl->cshift.alloc((size_t)n_slots * sizeof(R)));
    CU(ctx, pl->xi.alloc((size_t)K * n_slots * sizeof(R)));
    CU(ctx, pl->totS.alloc((size_t)n_slots * sizeof(R)));
    CU(ctx, pl->totQ.alloc((size_t)n_slots * sizeof(R)));
    CU(ctx, pl->out.alloc(per_draw * (size_t)pl->chunk * pl->n_bufs));
    CU(ctx, pl->yfut.alloc((size_t)std::max(1, p->n_h) * n_slots * sizeof(R)));
    if (p->flags & HMCGPU_FLAG_SUMMARY) {
        CU(ctx, pl->d_sum.alloc((size_t)nw * pl->F * sizeof(double)));
        CU(ctx, pl->d_sumsq.alloc((size_t)nw * pl->F * sizeof(double)));
    }
    if (p->flags & HMCGPU_FLAG_DIAGNOSTICS) {
        const size_t n_sf = (size_t)pl->F * n_slots, nwf = (size_t)nw * pl->F;
        CU(ctx, pl->dg_P.alloc(n_sf * kDiagLags * sizeof(double)));
        CU(ctx, pl->dg_S1.alloc(n_sf * sizeof(double)));
        CU(ctx, pl->dg_head.alloc(n_sf * kDiagLags * sizeof(R)));
        CU(ctx, pl->dg_ring.alloc(n_sf * kDiagLags * sizeof(R)));
        CU(ctx, pl->dg_mean.alloc(nwf * 2 * nc * sizeof(double)));
        CU(ctx, pl->dg_var.alloc(nwf * 2 * nc * sizeof(double)));
        CU(ctx, pl->dg_gsum.alloc(nwf * kDiagLags * sizeof(double)));
    }
    if (p->flags & HMCGPU_FLAG_PREDICTIVE) {
        std::vector<double> cw(nw);
        for (int w = 0; w < nw; ++w) cw[w] = p->y[(size_t)(p->win_series ? p->win_series[w] : 0) * p->y_len + p->win_end[w] - 1];
        pl->n_grid = p->n_grid;
        CU(ctx, up(pl->pr_grid, p->pred_grid, (size_t)p->n_grid * sizeof(double)));
        CU(ctx, up(pl->pr_cshift, cw.data(), nw * sizeof(double)));
        CU(ctx, pl->pr_cdf.alloc((size_t)n_slots * p->n_h * p->n_grid * sizeof(double)));
        CU(ctx, pl->pr_score.alloc((size_t)n_slots * p->n_h * kPredScores * sizeof(double)));
        // threads per slot: the grid rounded up to a power of two >= 32 (two points per thread above 256); then as many draws per
        // tile as ~45 KB of shared memory hold
        int tg = 32;
        while (tg < std::min(p->n_grid, kPredThreads)) tg *= 2;
        const int sb = kPredThreads / tg;
        pl->pr_tg = tg;
        pl->pr_td = (int)std::max<size_t>(1, std::min<size_t>(32, (45u << 10) / pred_smem_bytes(K, p->n_h, sb)));
        for (int j = 0; j < p->n_h; ++j) { pl->pr_h.h_sorted[j] = p->horizons[hs[j]]; pl->pr_h.h_slot[j] = hs[j]; }
    }
    if (p->flags & kAccMean) {
        CU(ctx, pl->pacc.alloc((size_t)lay.pi_elems * sizeof(R)));
        if (p->n_h > 0) {
            CU(ctx, pl->facc.alloc((size_t)lay.pi_elems / K * p->n_h * sizeof(R)));
            CU(ctx, pl->d_fcsum.alloc((size_t)pib_total / K * p->n_h * sizeof(double)));
        }
        CU(ctx, pl->d_pibsum.alloc((size_t)pib_total * sizeof(double)));
    }
    // (the ranked outputs are allocated at hmcgpu_plan_fetch_ranked, which knows n_probs)
    for (const WinOut& o : window_outputs(K, p->n_h, nc, p->nrun, pl->n_grid, 0, p->flags))
        if (o.on && o.dev && o.in != OutStruct::ranked) CU(ctx, (pl->*o.dev).alloc((size_t)o.elems(nw, sumT) * o.elem));
    if (p->flags & HMCGPU_FLAG_RANKED) CU(ctx, pl->rk_keep.alloc((size_t)nw * pl->F * nc * (size_t)p->nrun * sizeof(R)));
    if ((p->flags & HMCGPU_FLAG_LOO) && !(p->flags & HMCGPU_FLAG_RANKED))
        CU(ctx, pl->lo_keep.alloc((size_t)nw * (2 * K + K * K) * nc * (size_t)p->nrun * sizeof(R)));
    if (p->flags & HMCGPU_FLAG_ONESTEP) {
        pl->os_n = (long long)nc * sumT;
        CU(ctx, pl->os_state.alloc((size_t)kOsState * pl->os_n * sizeof(double)));
    }
    // window statistics (once per plan)
    const size_t smem = (size_t)pl->max_T;
    if (smem > 200 * 1024) return fail(ctx, HMCGPU_ERR_UNSUPPORTED, "window longer than %d observations", 200 * 1024);
    if (smem > 48 * 1024) CU(ctx, cudaFuncSetAttribute(window_init_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    window_init_kernel<<<nw, 256, smem, st>>>(K, yin.as<double>(), 1, pl->wbase.as<long long>(), pl->wbase_init.as<long long>(),
                                              pl->wTd.as<int>(), p->is_signal ? pl->sigmask_tm.as<unsigned char>() : nullptr,
                                              pl->wsbase.as<long long>(), sld, pl->X0.as<long long>(),
                                              pl->x0_off.as<long long>(), pl->wi.as<WinInit>());
    CU(ctx, cudaGetLastError());
    tr.sync_mark(st, "  tables, allocations, window statistics");
    yfut_kernel<R><<<grid_for(n_slots, 128), 128, 0, st>>>(n_slots, p->n_h, pl->slot_win.as<int>(), pl->yfut_w.as<double>(), pl->yfut.as<R>());
    CU(ctx, cudaGetLastError());

    GibbsArgs& a = pl->args;
    a.n_slots = n_slots; a.T = pl->T.as<int>(); a.ybase = pl->ybase.as<long long>(); a.yld = nser; a.y = pl->yr.p;
    a.warp_T = pl->warp_T.as<int>(); a.warp_pi_off = pl->warp_pi_off.as<long long>(); a.pi = pl->pi.p; a.pib_acc = pl->pacc.p; a.fc_acc = pl->facc.p;
    a.cnt = pl->cnt.as<int>(); a.trans = pl->trans.as<int>(); a.Sd = pl->Sd.p; a.Qd = pl->Qd.p; a.events = pl->events.as<int>();
    a.cshift = pl->cshift.p; a.xi = pl->xi.p; a.totS = pl->totS.p; a.totQ = pl->totQ.p; a.n_warps = n_warps;
    for (int i = 0; i < 32; ++i) {
        a.alpha[i] = (p->alpha && i < K) ? p->alpha[i] : 1.0;      // :137
        a.nu[i] = (p->nu && i < K) ? p->nu[i] : 1.0;               // :140
        a.beta0[i] = (p->beta0 && i < K) ? p->beta0[i] : 1.0;      // :179
        a.beta[i] = (p->beta && i < K) ? p->beta[i] : 2.0;         // :347
    }
    a.k0 = (unsigned)p->seed; a.k1 = (unsigned)(p->seed >> 32); a.chain_id = pl->chain_id.as<unsigned>();
    a.burnin = p->burnin; a.out = pl->out.p; a.chunk = pl->chunk; a.n_h = p->n_h;
    for (int j = 0; j < p->n_h; ++j) { a.h_sorted[j] = p->horizons[hs[j]]; a.h_slot[j] = hs[j]; }
    a.yfut = pl->yfut.p; a.flags = p->flags;
    a.sigw = pl->sigw.p; a.sbase = pl->sbase.as<long long>(); a.sld = sld; a.cntM = pl->cntM.as<int>(); a.Sm = pl->Sm.p; a.Qm = pl->Qm.p; a.totSm = pl->totSm.p; a.totQm = pl->totQm.p;
    a.totM = pl->totM.as<int>(); a.kappa = p->kappa; a.pi_back = p->pi_row_back;
    // one short series shared by every window (the rolling job), fp64: the thread-per-chain kernel keeps a copy in shared memory
    a.y_sm_elems = (y_in_smem<R>() && nser == 1 && K <= 4 && pl->sw.kernel == SweepKernel::thread && (size_t)p->y_len * sizeof(R) <= (size_t)kYSmemMaxBytes &&
                    pl->tuning.y_smem) ? (int)p->y_len : 0;
    a.all_signal = 0;
    if (p->is_signal) {
        const size_t nm = (size_t)p->y_len * sld;
        size_t ones = 0;
        for (size_t q = 0; q < nm; ++q) ones += p->is_signal[q] != 0;
        a.all_signal = ones == nm;
    }
    a.seg_warm = pl->tuning.seg_warm; a.seg_barriers = pl->tuning.seg_barriers;
    if (pl->sw.kernel == SweepKernel::seg) CU(ctx, pl->d_diag.alloc(2 * sizeof(unsigned long long)));
    a.diag = pl->d_diag.as<unsigned long long>();
    for (size_t g = 0; g < pl->groups.size(); ++g) {
        cudaStream_t s2;
        CU(ctx, cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking));
        pl->gstreams.push_back(s2);
    }
    CU(ctx, cudaEventCreate(&pl->ev0)); CU(ctx, cudaEventCreate(&pl->ev1));
    CU(ctx, cudaEventCreate(&pl->evk0)); CU(ctx, cudaEventCreate(&pl->evk1));
    tr.mark("  tables, allocations, init");
    CU(ctx, cudaStreamSynchronize(st));
    tr.mark("  stream drained");
    pl->yin.release();                                       // only the window statistics read the fp64 upload
    return HMCGPU_OK;
}

template <typename R, int K>
static int plan_run_t(hmcgpu_plan* pl) {
    hmcgpu_ctx* ctx = pl->ctx;
    cudaStream_t st = ctx->stream;
    const int ns = pl->n_slots, G = (int)pl->groups.size();
    const int Kr = pl->K;                                    // runtime K (the template K is 0 for the lane-per-state kernel)
    pl->n_launches = 0; pl->n_sweep_launches = 0; pl->sweep_ms = 0.0;
    size_t ev_used = 0;
    auto new_event = [&](cudaEvent_t* e) -> cudaError_t {
        if (ev_used == pl->pool_events.size()) {
            cudaEvent_t x;
            cudaError_t rc = cudaEventCreateWithFlags(&x, cudaEventDisableTiming);
            if (rc != cudaSuccess) return rc;
            pl->pool_events.push_back(x);
        }
        *e = pl->pool_events[ev_used++];
        return cudaSuccess;
    };
    CU(ctx, cudaEventRecord(pl->ev0, st));
    chain_init_kernel<R><<<grid_for(ns, 128), 128, 0, st>>>(Kr, ns, pl->slot_win.as<int>(), pl->wi.as<WinInit>(),
                                                             pl->xi_user.as<double>(), pl->cnt.as<int>(), pl->trans.as<int>(),
                                                             pl->Sd.as<R>(), pl->Qd.as<R>(), pl->cshift.as<R>(), pl->xi.as<R>(),
                                                             pl->totS.as<R>(), pl->totQ.as<R>(), pl->events.as<int>(),
                                                             pl->cntM.as<int>(), pl->Sm.as<R>(), pl->Qm.as<R>(), pl->totSm.as<R>(),
                                                             pl->totQm.as<R>(), pl->totM.as<int>());
    CU(ctx, cudaGetLastError());
    ++pl->n_launches;
    if (pl->d_diag.p) CU(ctx, cudaMemsetAsync(pl->d_diag.p, 0, 2 * sizeof(unsigned long long), st));
    if (pl->d_sum.p) { CU(ctx, cudaMemsetAsync(pl->d_sum.p, 0, pl->d_sum.bytes, st)); CU(ctx, cudaMemsetAsync(pl->d_sumsq.p, 0, pl->d_sumsq.bytes, st)); }
    if (pl->pacc.p) { CU(ctx, cudaMemsetAsync(pl->pacc.p, 0, pl->pacc.bytes, st)); CU(ctx, cudaMemsetAsync(pl->d_pibsum.p, 0, pl->d_pibsum.bytes, st)); }
    if (pl->facc.p) { CU(ctx, cudaMemsetAsync(pl->facc.p, 0, pl->facc.bytes, st)); CU(ctx, cudaMemsetAsync(pl->d_fcsum.p, 0, pl->d_fcsum.bytes, st)); }
    cudaEvent_t ev_init;
    CU(ctx, new_event(&ev_init));
    CU(ctx, cudaEventRecord(ev_init, st));
    CU(ctx, cudaEventRecord(pl->evk0, st));                  // start of the sweeps (sweep_kernel_ms)
    for (int g = 0; g < G; ++g) CU(ctx, cudaStreamWaitEvent(pl->gstreams[g], ev_init, 0));
    // an event pair around every sweep launch (its own duration, on its own stream) and one event per group after its last launch
    size_t tev_used = 0;
    auto timing_event = [&](cudaEvent_t* e) -> cudaError_t {
        if (tev_used == pl->timing_events.size()) {
            cudaEvent_t x;
            cudaError_t rc = cudaEventCreate(&x);
            if (rc != cudaSuccess) return rc;
            pl->timing_events.push_back(x);
        }
        *e = pl->timing_events[tev_used++];
        return cudaSuccess;
    };
    std::vector<cudaEvent_t> gend(G, nullptr);
    for (int g = 0; g < G; ++g) CU(ctx, timing_event(&gend[g]));
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> launch_pairs;

    const GibbsLaunch cfg{pl->flags, pl->max_T, ctx->sm_count, pl->n_h, pl->sig};
    const long long S = pl->burnin + pl->nrun;
    const long long n_chunks = (pl->nrun + pl->chunk - 1) / pl->chunk;
    const size_t buf_elems = (size_t)pl->F * pl->chunk * ns;
    std::vector<cudaEvent_t> post_done(n_chunks, nullptr);   // post-processing of chunk k finished
    std::vector<std::vector<cudaEvent_t>> chunk_done(n_chunks, std::vector<cudaEvent_t>(G, nullptr));
    auto enqueue_post = [&](long long k) -> int {
        for (int g = 0; g < G; ++g) CU(ctx, cudaStreamWaitEvent(st, chunk_done[k][g], 0));
        const long long d0 = k * pl->chunk;
        const int n = (int)std::min<long long>(pl->chunk, pl->nrun - d0);
        const R* buf = pl->out.as<R>() + (size_t)(k % pl->n_bufs) * buf_elems;
        if (pl->flags & HMCGPU_FLAG_DRAWS) {
            dim3 blk(32, 8), grd(grid_for(ns, 32), grid_for(n, 8));
            gather_draws_kernel<R><<<grd, blk, 0, st>>>(Kr, pl->n_h, ns, pl->chunk, n, d0, pl->nrun, pl->n_chains, pl->slot_win.as<int>(),
                                                         pl->slot_chain.as<int>(), buf, pl->d_mu.as<double>(), pl->d_sig2.as<double>(),
                                                         pl->d_A.as<double>(), pl->d_pie.as<double>(), pl->d_fc.as<double>(), pl->d_ll.as<double>());
            CU(ctx, cudaGetLastError());
            ++pl->n_launches;
        }
        if (pl->flags & HMCGPU_FLAG_SUMMARY) {
            dim3 grd(pl->n_windows, pl->F);
            summary_accum_kernel<R><<<grd, 128, 0, st>>>(pl->F, ns, pl->chunk, n, pl->n_chains, pl->win_slot0.as<int>(), buf,
                                                         pl->d_sum.as<double>(), pl->d_sumsq.as<double>());
            CU(ctx, cudaGetLastError());
            ++pl->n_launches;
        }
        if (pl->flags & HMCGPU_FLAG_DIAGNOSTICS) {
            // split-R̂ / ESS: draws [0, nh) form a chain's first sequence, [nrun - nh, nrun) its second; each sequence is reduced
            // per window right after the chunk holding its last draw, and the state is then reused by the next sequence
            const long long nh = pl->nrun / 2, h2 = pl->nrun - nh;
            const int Fd = (pl->flags & HMCGPU_FLAG_LOGLIK) ? pl->F : pl->F - 1;     // (no log-likelihood draws to look at)
            const DiagState<R> ds{pl->dg_P.as<double>(), pl->dg_S1.as<double>(), pl->dg_head.as<R>(), pl->dg_ring.as<R>(), (long long)pl->F * ns};
            auto sequence = [&](long long lo, long long hi, long long seq0, long long seq_end, int half) -> int {
                if (lo >= hi) return 0;
                diag_accum_kernel<R><<<dim3(ns / 32, Fd), dim3(32, 32), 0, st>>>(ns, pl->chunk, (int)(lo - d0), (int)(hi - lo), lo - seq0, buf, ds);
                CU(ctx, cudaGetLastError());
                ++pl->n_launches;
                if (hi == seq_end) {
                    diag_half_kernel<R><<<dim3(pl->n_windows, Fd), kDiagLags, 0, st>>>(pl->F, ns, pl->n_chains, nh, half, pl->win_slot0.as<int>(), ds,
                                                                                       pl->dg_mean.as<double>(), pl->dg_var.as<double>(), pl->dg_gsum.as<double>());
                    CU(ctx, cudaGetLastError());
                    ++pl->n_launches;
                }
                return 0;
            };
            TRY(sequence(d0, std::min<long long>(d0 + n, nh), 0, nh, 0));
            TRY(sequence(std::max(d0, h2), d0 + n, h2, pl->nrun, 1));
        }
        if (pl->flags & HMCGPU_FLAG_RANKED) {
            ranked_keep_kernel<R><<<dim3(pl->n_windows, pl->F), dim3(32, 8), 0, st>>>(pl->F, ns, pl->chunk, n, d0, pl->nrun, pl->n_chains,
                                                                                     pl->win_slot0.as<int>(), buf, pl->rk_keep.as<R>());
            CU(ctx, cudaGetLastError());
            ++pl->n_launches;
        }
        if ((pl->flags & HMCGPU_FLAG_LOO) && !(pl->flags & HMCGPU_FLAG_RANKED)) {
            const int Fl = 2 * Kr + Kr * Kr;                 // mu, sigma2, A: the leading summary fields
            ranked_keep_kernel<R><<<dim3(pl->n_windows, Fl), dim3(32, 8), 0, st>>>(Fl, ns, pl->chunk, n, d0, pl->nrun, pl->n_chains,
                                                                                 pl->win_slot0.as<int>(), buf, pl->lo_keep.as<R>());
            CU(ctx, cudaGetLastError());
            ++pl->n_launches;
        }
        if (pl->flags & HMCGPU_FLAG_PREDICTIVE) {
            const int sb = kPredThreads / pl->pr_tg;
            const size_t smem = pred_smem_bytes(Kr, pl->n_h, sb * pl->pr_td);
            auto accum = pl->n_grid > kPredThreads ? pred_accum_kernel<R, 2> : pred_accum_kernel<R, 1>;
            accum<<<ns / sb, kPredThreads, smem, st>>>(Kr, pl->n_h, pl->n_grid, ns, pl->chunk, n, k == 0, pl->pr_tg, pl->pr_td, pl->pr_h,
                                                       pl->slot_win.as<int>(), pl->pr_cshift.as<double>(), pl->yfut_w.as<double>(),
                                                       pl->pr_grid.as<double>(), buf, pl->pr_cdf.as<double>(), pl->pr_score.as<double>());
            CU(ctx, cudaGetLastError());
            ++pl->n_launches;
        }
        if (pl->flags & HMCGPU_FLAG_ONESTEP) {
            CU(ctx, launch_onestep_accum<R>(Kr, ns, pl->chunk, n, d0, pl->n_chains, pl->slot_win.as<int>(), pl->slot_chain.as<int>(),
                                            pl->wTd.as<int>(), pl->win_pib_off.as<long long>(), pl->ybase.as<long long>(),
                                            pl->args.yld, pl->yr.as<R>(), buf, pl->os_state.as<double>(), pl->os_n, st));
            ++pl->n_launches;
        }
        if (pl->flags & (HMCGPU_FLAG_SMOOTHED_MEAN | HMCGPU_FLAG_FILTERED_MEAN)) {
            tile_reduce_kernel<R><<<pl->n_windows, 256, 0, st>>>(Kr, Kr, pl->n_chains, pl->win_slot0.as<int>(), pl->wTd.as<int>(),
                                                                 pl->warp_pi_off.as<long long>(), pl->warp_T.as<int>(), pl->win_pib_off.as<long long>(),
                                                                 pl->pacc.as<R>(), pl->d_pibsum.as<double>());
            CU(ctx, cudaGetLastError());
            ++pl->n_launches;
            if (pl->facc.p) {
                tile_reduce_kernel<R><<<pl->n_windows, 256, 0, st>>>(Kr, pl->n_h, pl->n_chains, pl->win_slot0.as<int>(), pl->wTd.as<int>(),
                                                                     pl->warp_pi_off.as<long long>(), pl->warp_T.as<int>(), pl->win_pib_off.as<long long>(),
                                                                     pl->facc.as<R>(), pl->d_fcsum.as<double>());
                CU(ctx, cudaGetLastError());
                ++pl->n_launches;
            }
        }
        CU(ctx, new_event(&post_done[k]));
        CU(ctx, cudaEventRecord(post_done[k], st));
        return 0;
    };
    PhaseTrace trr;
    GibbsArgs a = pl->args;
    // the sweep launches and the per-chunk post-processing, in the order launch_schedule gives
    for (const RunOp& op : launch_schedule(pl->burnin, pl->nrun, pl->chunk, pl->n_bufs, G, pl->sw.sweeps_per_launch)) {
        if (op.post) {
            TRY(enqueue_post(op.chunk));
            continue;
        }
        const int g = op.group;
        cudaStream_t gs = pl->gstreams[g];
        if (op.wait >= 0) CU(ctx, cudaStreamWaitEvent(gs, post_done[op.wait], 0));   // the chunk's buffer has been consumed
        a.draw0 = op.chunk >= 0 ? op.chunk * pl->chunk : 0;
        a.out = op.chunk >= 0 ? pl->out.as<R>() + (size_t)(op.chunk % pl->n_bufs) * buf_elems : pl->out.as<R>();
        a.sweep0 = op.sweep0; a.n_sweeps = (int)op.n_sweeps;
        const TaskGroup& grp = pl->groups[g];
        a.task0 = grp.task0; a.task_stride = grp.stride; a.n_tasks = grp.n_tasks;
        a.warp_T = grp.long_class ? pl->warp_T_long.as<int>() : pl->warp_T.as<int>();
        a.warp_pi_off = grp.long_class ? pl->warp_pi_off_long.as<long long>() : pl->warp_pi_off.as<long long>();
        cudaEvent_t lt0 = nullptr, lt1 = nullptr;
        if (pl->tuning.launch_timing) { CU(ctx, timing_event(&lt0)); CU(ctx, timing_event(&lt1)); CU(ctx, cudaEventRecord(lt0, gs)); }
        if constexpr (K == 0) {
            CU(ctx, (launch_gibbs_wide<R>(cfg, a, pl->K, pl->slot_pi_off.as<long long>(), gs)));
        } else if constexpr (K <= 4) {
            switch (pl->sw.kernel) {
                case SweepKernel::scan: CU(ctx, (launch_gibbs_scan<R, K>(cfg, a, gs))); break;
                case SweepKernel::seg: CU(ctx, (launch_gibbs_seg<R, K>(cfg, a, grp.lanes, pl->sw.seg_threads, gs))); break;
                default: CU(ctx, (launch_gibbs<R, K>(cfg, a, gs)));
            }
        } else {
            CU(ctx, (launch_gibbs<R, K>(cfg, a, gs)));
        }
        if (pl->tuning.launch_timing) { CU(ctx, cudaEventRecord(lt1, gs)); launch_pairs.emplace_back(lt0, lt1); }
        ++pl->n_launches; ++pl->n_sweep_launches;
        if (op.last) CU(ctx, cudaEventRecord(gend[g], gs));
        if (op.closes_chunk) {
            CU(ctx, new_event(&chunk_done[op.chunk][g]));
            CU(ctx, cudaEventRecord(chunk_done[op.chunk][g], gs));
        }
    }
    CU(ctx, cudaEventRecord(pl->ev1, st));                   // st has waited for every group through the last chunk's post
    trr.mark("    launches enqueued");
    CU(ctx, cudaEventSynchronize(pl->ev1));
    trr.mark("    device drained");
    for (int g = 0; g < G; ++g) CU(ctx, cudaStreamSynchronize(pl->gstreams[g]));
    float ms = 0.f;
    CU(ctx, cudaEventElapsedTime(&ms, pl->ev0, pl->ev1));
    pl->gpu_ms = ms;
    // the launches of different groups overlap: sweep_ms is the interval from the start of the first sweep launch to the end of
    // the last one (it leaves out the init kernel and the post-processing tail); launch_ms_sum adds up each launch's own duration
    pl->sweep_ms = 0.0;
    for (int g = 0; g < G; ++g) {
        float t = 0.f;
        CU(ctx, cudaEventElapsedTime(&t, pl->evk0, gend[g]));
        pl->sweep_ms = std::max(pl->sweep_ms, (double)t);
    }
    pl->launch_ms_sum = 0.0;
    for (auto& pr : launch_pairs) {
        float t = 0.f;
        CU(ctx, cudaEventElapsedTime(&t, pr.first, pr.second));
        pl->launch_ms_sum += t;
    }
    if (pl->d_diag.p) {
        CU(ctx, cudaMemcpy(pl->seg_fallbacks, pl->d_diag.p, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
        if (pl->tuning.verbose) {
            const double cs = (double)pl->n_windows * pl->n_chains * (double)S;
            if (pl->sw.n_long) fprintf(stderr, "[hmcgpu] segment kernel: the %d longest of %d windows with 8 lanes per chain\n", pl->sw.n_long, pl->n_windows);
            fprintf(stderr, "[hmcgpu] segment kernel (%d lanes per chain, warm-up %d): %llu of %.0f chain-sweeps used the exact entering vectors; "
                            "%.2f speculative groups of 4 steps per chain-sweep\n",
                    pl->sw.seg_lanes, pl->args.seg_warm, pl->seg_fallbacks[0], cs, (double)pl->seg_fallbacks[1] / cs);
        }
    }
    pl->ran = true;
    return HMCGPU_OK;
}

static int plan_create_impl(hmcgpu_ctx* ctx, const hmcgpu_problem* p, hmcgpu_plan** out) {
    const Tuning t = read_tuning();
    TRY(validate_problem(ctx, p, t));
    CU(ctx, cudaSetDevice(ctx->device));
    if (p->flags & HMCGPU_FLAG_RANKED) {
        // the retained draws are the one allocation that grows with nrun: refuse a shape whose draws cannot fit before allocating
        size_t free_b = 0, total_b = 0;
        CU(ctx, cudaMemGetInfo(&free_b, &total_b));
        const double keep = (double)p->n_windows * summary_fields(p->K, p->n_h) * p->n_chains * (double)p->nrun * (p->precision / 8);
        if (keep > (double)total_b)
            return fail(ctx, HMCGPU_ERR_ALLOC, "HMCGPU_FLAG_RANKED retains %.0f bytes of draws, more than the device's %zu bytes", keep, total_b);
    }
    if (p->flags & HMCGPU_FLAG_ONESTEP) {
        // kOsState fp64 values per (chain, date): checked before anything is allocated, like the retained draws
        size_t free_b = 0, total_b = 0;
        CU(ctx, cudaMemGetInfo(&free_b, &total_b));
        double dates = 0.0;
        for (int w = 0; w < p->n_windows; ++w) dates += (double)p->win_end[w] - p->win_start[w] + 1;
        const double need = dates * p->n_chains * kOsState * sizeof(double);
        if (need > (double)total_b)
            return fail(ctx, HMCGPU_ERR_ALLOC, "HMCGPU_FLAG_ONESTEP keeps %.0f bytes of running state, more than the device's %zu bytes", need, total_b);
    }
    if (p->flags & HMCGPU_FLAG_LOO) {
        // the kept mu / sigma2 / A draws (none beyond HMCGPU_FLAG_RANKED's) and one batch of fetch scratch
        size_t free_b = 0, total_b = 0;
        CU(ctx, cudaMemGetInfo(&free_b, &total_b));
        double dates = 0.0;
        for (int w = 0; w < p->n_windows; ++w) dates += (double)p->win_end[w] - p->win_start[w] + 1;
        const double R = (double)p->n_chains * (double)p->nrun, per_date = (double)loo_date_bytes((long long)R, p->K, p->precision / 8);
        const double keep = (p->flags & HMCGPU_FLAG_RANKED) ? 0.0 : (double)p->n_windows * (2 * p->K + p->K * p->K) * R * (p->precision / 8);
        const double need = keep + std::min(dates, std::max(1.0, std::floor((double)t.loo_scratch / per_date))) * per_date;
        if (need > (double)total_b)
            return fail(ctx, HMCGPU_ERR_ALLOC, "HMCGPU_FLAG_LOO needs %.0f bytes of kept draws and fetch scratch, more than the device's %zu bytes", need, total_b);
    }
    tl_pool = ctx->pool;
    std::unique_ptr<hmcgpu_plan> pl(new hmcgpu_plan());
    pl->ctx = ctx;
    pl->tuning = t;
    int rc = (p->precision == 32) ? plan_build<float>(pl.get(), p) : plan_build<double>(pl.get(), p);
    if (rc != 0) {
        cudaStreamSynchronize(ctx->stream);    // uploads / init kernels may still be queued on buffers the plan is about to release
        cudaGetLastError();
        return rc;
    }
    *out = pl.release();
    return HMCGPU_OK;
}

extern "C" int hmcgpu_plan_create(hmcgpu_ctx* ctx, const hmcgpu_problem* p, hmcgpu_plan** out) {
    if (!out) return fail(ctx, HMCGPU_ERR_ARG, "out is NULL");
    *out = nullptr;
    GUARD(ctx, plan_create_impl(ctx, p, out));
}

static int plan_run_impl(hmcgpu_plan* pl) {
    hmcgpu_ctx* ctx = pl->ctx;
    CU(ctx, cudaSetDevice(ctx->device));
    int rc = HMCGPU_ERR_UNSUPPORTED;
    DISPATCH_RUN(pl, rc);
    return rc;
}

extern "C" int hmcgpu_plan_run(hmcgpu_plan* pl) {
    if (!pl) return HMCGPU_ERR_ARG;
    GUARD(pl->ctx, plan_run_impl(pl));
}

static int plan_fetch_impl(hmcgpu_plan* pl, hmcgpu_result* r);
extern "C" int hmcgpu_plan_fetch(hmcgpu_plan* pl, hmcgpu_result* r) {
    if (!pl || !r) return HMCGPU_ERR_ARG;
    GUARD(pl->ctx, plan_fetch_impl(pl, r));
}

// Enqueues the copy of every requested output the plan holds (of r, pr, rk, os or lo) into the caller's arrays; adds the bytes
// to *bytes (NULL: the predictive, ranked, one-step and LOO outputs, which hmcgpu_result's d2h_bytes does not count)
static int download(hmcgpu_plan* pl, const std::vector<WinOut>& outs, const hmcgpu_result* r, const hmcgpu_predictive* pr,
                    const hmcgpu_ranked* rk, const hmcgpu_onestep* os, const hmcgpu_loo* lo, long long* bytes) {
    for (const WinOut& o : outs) {
        void* host = o.get(r, pr, rk, os, lo);
        if (!host || !o.dev || !(pl->*o.dev).p) continue;         // (an output of no elements has no buffer)
        const DevBuf& b = pl->*o.dev;
        CU(pl->ctx, cudaMemcpyAsync(host, b.p, b.bytes, cudaMemcpyDeviceToHost, pl->ctx->stream));
        if (bytes) *bytes += (long long)b.bytes;
    }
    return HMCGPU_OK;
}

static int plan_fetch_impl(hmcgpu_plan* pl, hmcgpu_result* r) {
    hmcgpu_ctx* ctx = pl->ctx;
    if (!pl->ran) return fail(ctx, HMCGPU_ERR_ARG, "plan_fetch before plan_run");
    const std::vector<WinOut> outs = window_outputs(pl->K, pl->n_h, pl->n_chains, pl->nrun, pl->n_grid, 0, pl->flags);
    for (const WinOut& o : outs)
        if (!o.on && o.get(r, nullptr)) return fail(ctx, HMCGPU_ERR_ARG, "%s requested without %s", o.name, o.need);
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const int nc = pl->n_chains, has_ll = (pl->flags & HMCGPU_FLAG_LOGLIK) ? 1 : 0;
    const double n = (double)nc * (double)pl->nrun;
    // finished on the device from the run's sums (these launches are not plan_run's: n_launches leaves them out)
    const long long ne = (long long)pl->n_windows * pl->F, npib = (long long)(pl->d_pib.bytes / sizeof(double)),
                    nifc = (long long)(pl->d_ifc.bytes / sizeof(double));
    if (pl->d_mean.p)
        summary_finish_kernel<<<grid_for(ne, 256), 256, 0, st>>>(ne, pl->F, n, has_ll, pl->d_sum.as<double>(), pl->d_sumsq.as<double>(),
                                                                 pl->d_mean.as<double>(), pl->d_var.as<double>());
    if (pl->d_rhat.p)
        diag_finish_kernel<<<grid_for(ne, 128), 128, 0, st>>>(ne, pl->F, nc, pl->nrun / 2, has_ll, pl->dg_mean.as<double>(),
                                                              pl->dg_var.as<double>(), pl->dg_gsum.as<double>(), pl->d_rhat.as<double>(),
                                                              pl->d_ess.as<double>(), pl->d_lag.as<int>());
    if (pl->d_pib.p) mean_finish_kernel<<<grid_for(npib, 256), 256, 0, st>>>(npib, n, pl->d_pibsum.as<double>(), pl->d_pib.as<double>());
    if (pl->d_ifc.p) mean_finish_kernel<<<grid_for(nifc, 256), 256, 0, st>>>(nifc, n, pl->d_fcsum.as<double>(), pl->d_ifc.as<double>());
    CU(ctx, cudaGetLastError());
    long long d2h = 0;
    TRY(download(pl, outs, r, nullptr, nullptr, nullptr, nullptr, &d2h));
    std::vector<int> ev(pl->n_slots);
    CU(ctx, cudaMemcpyAsync(ev.data(), pl->events.p, ev.size() * sizeof(int), cudaMemcpyDeviceToHost, st));
    d2h += (long long)(ev.size() * sizeof(int));
    CU(ctx, cudaStreamSynchronize(st));
    int bad = 0;
    for (int w = 0; w < pl->n_windows; ++w) {
        for (int c = 0; c < nc; ++c) {
            const int e = ev[(size_t)pl->slot0[w] + c];
            if (r->status) r->status[(size_t)w * nc + c] = e;
            bad += e != 0;
        }
    }
    r->gpu_ms = pl->gpu_ms; r->sweep_kernel_ms = pl->sweep_ms; r->n_launches = pl->n_launches;
    r->n_sweep_launches = pl->n_sweep_launches; r->h2d_bytes = pl->h2d; r->d2h_bytes = d2h; r->state_steps = pl->state_steps;
    r->sweep_launch_ms_sum = pl->launch_ms_sum;
    r->sweep_kernel = (int32_t)pl->sw.kernel;
    r->n_tasks = pl->n_tasks;
    return bad;
}

static int plan_fetch_predictive_impl(hmcgpu_plan* pl, hmcgpu_predictive* pr) {
    hmcgpu_ctx* ctx = pl->ctx;
    if (!(pl->flags & HMCGPU_FLAG_PREDICTIVE)) return fail(ctx, HMCGPU_ERR_ARG, "plan_fetch_predictive on a plan without HMCGPU_FLAG_PREDICTIVE");
    if (!pl->ran) return fail(ctx, HMCGPU_ERR_ARG, "plan_fetch_predictive before plan_run");
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    const long long nwh = (long long)pl->n_windows * pl->n_h;
    pred_finish_kernel<<<grid_for(nwh * (pl->n_grid + 1), 128), 128, 0, st>>>(pl->n_windows, pl->n_h, pl->n_grid, pl->n_chains,
                                                                              (double)pl->n_chains * (double)pl->nrun, pl->win_slot0.as<int>(),
                                                                              pl->pr_cshift.as<double>(), pl->pr_cdf.as<double>(),
                                                                              pl->pr_score.as<double>(), pl->d_cdf.as<double>(), pl->d_pit.as<double>(),
                                                                              pl->d_ls.as<double>(), pl->d_mom.as<double>());
    CU(ctx, cudaGetLastError());
    TRY(download(pl, window_outputs(pl->K, pl->n_h, pl->n_chains, pl->nrun, pl->n_grid, 0, pl->flags), nullptr, pr, nullptr, nullptr, nullptr, nullptr));
    CU(ctx, cudaStreamSynchronize(st));
    return HMCGPU_OK;
}

extern "C" int hmcgpu_plan_fetch_predictive(hmcgpu_plan* pl, hmcgpu_predictive* pr) {
    if (!pl || !pr) return HMCGPU_ERR_ARG;
    GUARD(pl->ctx, plan_fetch_predictive_impl(pl, pr));
}

static int check_ranked(hmcgpu_ctx* ctx, const hmcgpu_ranked* rk) {
    if (rk->n_probs < 0 || rk->n_probs > kRankedMaxProbs)
        return fail(ctx, HMCGPU_ERR_ARG, "hmcgpu_ranked.n_probs = %d is outside 0..%d", rk->n_probs, kRankedMaxProbs);
    if (rk->n_probs > 0 && !rk->probs) return fail(ctx, HMCGPU_ERR_ARG, "hmcgpu_ranked.probs is NULL with n_probs = %d", rk->n_probs);
    for (int k = 0; k < rk->n_probs; ++k)
        if (!std::isfinite(rk->probs[k]) || rk->probs[k] < 0.0 || rk->probs[k] > 1.0)
            return fail(ctx, HMCGPU_ERR_ARG, "hmcgpu_ranked.probs[%d] = %g is not a finite probability in [0, 1]", k, rk->probs[k]);
    return HMCGPU_OK;
}

// The ranked outputs of every (window, field) segment of the retained draws (ranked.cuh), in batches of segments whose scratch
// stays near 2 GiB (at least one segment).  These launches are not plan_run's: n_launches leaves them out.
template <typename R>
static int fetch_ranked_t(hmcgpu_plan* pl, const hmcgpu_ranked* rk) {
    hmcgpu_ctx* ctx = pl->ctx;
    cudaStream_t st = ctx->stream;
    const int nc = pl->n_chains, M = 2 * nc;
    const long long Rs = (long long)nc * pl->nrun, n_seg = (long long)pl->n_windows * pl->F, nh = pl->nrun / 2;
    RankedProbs probs{};
    probs.n = rk->n_probs;
    for (int k = 0; k < rk->n_probs; ++k) probs.p[k] = rk->probs[k];
    CU(ctx, pl->d_quant.alloc((size_t)n_seg * rk->n_probs * sizeof(double)));
    CU(ctx, pl->d_rrank.alloc((size_t)n_seg * sizeof(double)));
    CU(ctx, pl->d_essb.alloc((size_t)n_seg * sizeof(double)));
    CU(ctx, pl->d_esst.alloc((size_t)n_seg * sizeof(double)));
    // per segment: two key and two position buffers for the sort, the normal scores, the per-sequence statistics
    const size_t seg_bytes = (size_t)Rs * (2 * sizeof(unsigned long long) + 2 * sizeof(int) + sizeof(double)) +
                             (size_t)M * (kDiagLags + 2) * sizeof(double) + 256;
    const long long B = std::max<long long>(1, std::min<long long>({n_seg, (long long)((2ull << 30) / seg_bytes), 0x7fffffffLL / Rs}));
    const size_t nB = (size_t)B * Rs;
    DevBuf keys0, keys1, pos0, pos1, z, g, smean, svar, gsum, qs, bad, rh, es, lag, offs, temp;
    CU(ctx, keys0.alloc(nB * sizeof(unsigned long long)));
    CU(ctx, keys1.alloc(nB * sizeof(unsigned long long)));
    CU(ctx, pos0.alloc(nB * sizeof(int)));
    CU(ctx, pos1.alloc(nB * sizeof(int)));
    CU(ctx, z.alloc(nB * sizeof(double)));
    CU(ctx, g.alloc((size_t)B * M * kDiagLags * sizeof(double)));
    CU(ctx, smean.alloc((size_t)B * M * sizeof(double)));
    CU(ctx, svar.alloc((size_t)B * M * sizeof(double)));
    CU(ctx, gsum.alloc((size_t)B * kDiagLags * sizeof(double)));
    CU(ctx, qs.alloc((size_t)B * kRankedQuants * sizeof(double)));
    CU(ctx, bad.alloc((size_t)B));
    CU(ctx, rh.alloc((size_t)4 * B * sizeof(double)));
    CU(ctx, es.alloc((size_t)4 * B * sizeof(double)));
    CU(ctx, lag.alloc((size_t)4 * B * sizeof(int)));
    std::vector<int> off(B + 1);
    for (long long s = 0; s <= B; ++s) off[s] = (int)(s * Rs);
    CU(ctx, offs.alloc(off.size() * sizeof(int)));
    CU(ctx, cudaMemcpyAsync(offs.p, off.data(), off.size() * sizeof(int), cudaMemcpyHostToDevice, st));
    for (long long s0 = 0; s0 < n_seg; s0 += B) {
        const int nb = (int)std::min<long long>(B, n_seg - s0);
        const long long N = (long long)nb * Rs;
        const R* x = pl->rk_keep.as<R>() + (size_t)s0 * Rs;
        // keys of x (fold: of |x - q(0.5)|) sorted per segment, then the normal scores of their ranks into z; returns the sorted keys
        auto scores = [&](const double* fold, const unsigned long long** sorted) -> int {
            ranked_keys_kernel<R><<<grid_for(N, 256), 256, 0, st>>>(N, Rs, x, fold, keys0.as<unsigned long long>(), pos0.as<int>());
            CU(ctx, cudaGetLastError());
            cub::DoubleBuffer<unsigned long long> kb(keys0.as<unsigned long long>(), keys1.as<unsigned long long>());
            cub::DoubleBuffer<int> pb(pos0.as<int>(), pos1.as<int>());
            size_t tb = 0;
            CU(ctx, ranked_sort(nullptr, tb, kb, pb, (int)N, nb, offs.as<int>(), st));
            if (tb > temp.bytes) CU(ctx, temp.alloc(tb));
            CU(ctx, ranked_sort(temp.p, tb, kb, pb, (int)N, nb, offs.as<int>(), st));
            ranked_scores_kernel<<<grid_for(N, 256), 256, 0, st>>>(N, Rs, kb.Current(), pb.Current(), z.as<double>());
            CU(ctx, cudaGetLastError());
            *sorted = kb.Current();
            return HMCGPU_OK;
        };
        // split R̂ / ESS of one transformed sequence (normal scores z, or the indicator 1[x <= qs[qi]]) into rh / es row t
        auto split = [&](bool use_z, int qi, int t) -> int {
            const long long n_seqs = (long long)nb * M;
            ranked_stats_kernel<R><<<grid_for(n_seqs, kRankedSeqWarps), 32 * kRankedSeqWarps, 0, st>>>(
                n_seqs, nc, pl->nrun, nh, Rs, use_z ? z.as<double>() : nullptr, x, qs.as<double>(), qi, smean.as<double>(),
                svar.as<double>(), g.as<double>());
            ranked_chain_sum_kernel<<<grid_for((long long)nb * kDiagLags, 256), 256, 0, st>>>((long long)nb * kDiagLags, nc, g.as<double>(),
                                                                                           gsum.as<double>());
            // (has_loglik = 1: ranked_quantiles_kernel's `bad` covers the log-likelihood field)
            diag_finish_kernel<<<grid_for(nb, 128), 128, 0, st>>>(nb, pl->F, nc, nh, 1, smean.as<double>(), svar.as<double>(), gsum.as<double>(),
                                                                  rh.as<double>() + (size_t)t * nb, es.as<double>() + (size_t)t * nb,
                                                                  lag.as<int>() + (size_t)t * nb);
            CU(ctx, cudaGetLastError());
            return HMCGPU_OK;
        };
        const unsigned long long* sorted = nullptr;
        TRY(scores(nullptr, &sorted));
        ranked_quantiles_kernel<<<grid_for(nb, 128), 128, 0, st>>>(nb, s0, Rs, pl->F, (pl->flags & HMCGPU_FLAG_LOGLIK) ? 1 : 0, sorted, probs,
                                                                   pl->d_quant.as<double>(), qs.as<double>(), bad.as<unsigned char>());
        CU(ctx, cudaGetLastError());
        TRY(split(true, 0, 0));                 // bulk
        TRY(split(false, 0, 2));                // tail: 1[x <= q(0.05)]
        TRY(split(false, 2, 3));                // tail: 1[x <= q(0.95)]
        TRY(scores(qs.as<double>(), &sorted));  // folded about q(0.5)
        TRY(split(true, 0, 1));
        ranked_combine_kernel<<<grid_for(nb, 128), 128, 0, st>>>(nb, s0, bad.as<unsigned char>(), rh.as<double>(), es.as<double>(),
                                                                 pl->d_rrank.as<double>(), pl->d_essb.as<double>(), pl->d_esst.as<double>());
        CU(ctx, cudaGetLastError());
    }
    TRY(download(pl, window_outputs(pl->K, pl->n_h, nc, pl->nrun, pl->n_grid, rk->n_probs, pl->flags), nullptr, nullptr, rk, nullptr, nullptr, nullptr));
    CU(ctx, cudaStreamSynchronize(st));         // (the scratch goes back to the pool when this returns)
    return HMCGPU_OK;
}

static int plan_fetch_ranked_impl(hmcgpu_plan* pl, hmcgpu_ranked* rk) {
    hmcgpu_ctx* ctx = pl->ctx;
    if (!(pl->flags & HMCGPU_FLAG_RANKED)) return fail(ctx, HMCGPU_ERR_ARG, "plan_fetch_ranked on a plan without HMCGPU_FLAG_RANKED");
    if (!pl->ran) return fail(ctx, HMCGPU_ERR_ARG, "plan_fetch_ranked before plan_run");
    TRY(check_ranked(ctx, rk));
    CU(ctx, cudaSetDevice(ctx->device));
    tl_pool = ctx->pool;
    return pl->precision == 32 ? fetch_ranked_t<float>(pl, rk) : fetch_ranked_t<double>(pl, rk);
}

extern "C" int hmcgpu_plan_fetch_ranked(hmcgpu_plan* pl, hmcgpu_ranked* rk) {
    if (!pl) return HMCGPU_ERR_ARG;
    if (!rk) return fail(pl->ctx, HMCGPU_ERR_ARG, "hmcgpu_ranked is NULL");
    GUARD(pl->ctx, plan_fetch_ranked_impl(pl, rk));
}

static int plan_fetch_onestep_impl(hmcgpu_plan* pl, hmcgpu_onestep* os) {
    hmcgpu_ctx* ctx = pl->ctx;
    if (!(pl->flags & HMCGPU_FLAG_ONESTEP)) return fail(ctx, HMCGPU_ERR_ARG, "plan_fetch_onestep on a plan without HMCGPU_FLAG_ONESTEP");
    if (!pl->ran) return fail(ctx, HMCGPU_ERR_ARG, "plan_fetch_onestep before plan_run");
    CU(ctx, cudaSetDevice(ctx->device));
    cudaStream_t st = ctx->stream;
    // (not plan_run's launch: n_launches leaves it out)
    onestep_finish_kernel<<<pl->n_windows, 128, 0, st>>>(pl->K, pl->n_chains, pl->nrun, pl->wTd.as<int>(), pl->win_pib_off.as<long long>(),
                                                         pl->os_state.as<double>(), pl->os_n, pl->d_ospit.as<double>(),
                                                         pl->d_oslpd.as<double>(), pl->d_osvar.as<double>(), pl->d_waic.as<double>());
    CU(ctx, cudaGetLastError());
    TRY(download(pl, window_outputs(pl->K, pl->n_h, pl->n_chains, pl->nrun, pl->n_grid, 0, pl->flags), nullptr, nullptr, nullptr, os, nullptr, nullptr));
    CU(ctx, cudaStreamSynchronize(st));
    return HMCGPU_OK;
}

extern "C" int hmcgpu_plan_fetch_onestep(hmcgpu_plan* pl, hmcgpu_onestep* os) {
    if (!pl) return HMCGPU_ERR_ARG;
    if (!os) return fail(pl->ctx, HMCGPU_ERR_ARG, "hmcgpu_onestep is NULL");
    GUARD(pl->ctx, plan_fetch_onestep_impl(pl, os));
}

// PSIS-LOO of every date (loo.cuh), in batches of dates whose scratch stays under Tuning::loo_scratch (at least one date).  These
// launches are not plan_run's: n_launches leaves them out.
template <typename R>
static int fetch_loo_t(hmcgpu_plan* pl, const hmcgpu_loo* lo) {
    hmcgpu_ctx* ctx = pl->ctx;
    cudaStream_t st = ctx->stream;
    const int K = pl->K, nw = pl->n_windows;
    const long long Rd = (long long)pl->n_chains * pl->nrun;
    const bool rk = pl->flags & HMCGPU_FLAG_RANKED;
    const R* keep = rk ? pl->rk_keep.as<R>() : pl->lo_keep.as<R>();
    const int Fs = rk ? pl->F : 2 * K + K * K;
    long long sumT = 0;
    for (int w = 0; w < nw; ++w) sumT += pl->wT[w];
    const size_t per_date = loo_date_bytes(Rd, K, sizeof(R));
    const long long B = std::max<long long>(1, std::min<long long>(sumT, (long long)(pl->tuning.loo_scratch / per_date)));
    // the pieces of every batch: batch b covers the dates [b*B, (b+1)*B) of the windows concatenated in caller order
    std::vector<LooPiece> pieces;
    std::vector<long long> first{0};
    for (long long g0 = 0; g0 < sumT; g0 += B) {
        const long long g1 = std::min(sumT, g0 + B);
        for (int w = 0; w < nw; ++w) {
            const long long o = pl->pib_off[w] / K, e = o + pl->wT[w];
            if (e <= g0 || o >= g1) continue;
            pieces.push_back({w, (int)(std::max(g0, o) - o), (int)(std::min(g1, e) - o), (int)(std::max(g0, o) - g0)});
        }
        first.push_back((long long)pieces.size());
    }
    DevBuf dp, ell, F, lb;
    CU(ctx, dp.alloc(pieces.size() * sizeof(LooPiece)));
    CU(ctx, cudaMemcpyAsync(dp.p, pieces.data(), pieces.size() * sizeof(LooPiece), cudaMemcpyHostToDevice, st));
    CU(ctx, ell.alloc((size_t)B * Rd * sizeof(double)));
    CU(ctx, F.alloc((size_t)B * Rd * sizeof(double)));
    CU(ctx, lb.alloc((size_t)B * K * Rd * sizeof(R)));
    const size_t smem = loo_psis_smem(Rd);
    if (smem > 48 * 1024) CU(ctx, cudaFuncSetAttribute(loo_psis_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    for (size_t b = 0; b + 1 < first.size(); ++b) {
        const long long g0 = (long long)b * B, nb = std::min(sumT, g0 + B) - g0;
        CU(ctx, launch_loo_terms<R>(K, Rd, Fs, (int)(first[b + 1] - first[b]), dp.as<LooPiece>() + first[b], keep, pl->wTd.as<int>(),
                                    pl->win_slot0.as<int>(), pl->ybase.as<long long>(), pl->args.yld, pl->yr.as<R>(), lb.as<R>(),
                                    ell.as<double>(), F.as<double>(), st));
        loo_psis_kernel<<<(unsigned)nb, kLooThreads, smem, st>>>(Rd, g0, ell.as<double>(), F.as<double>(), pl->d_lelpd.as<double>(),
                                                               pl->d_llppd.as<double>(), pl->d_lpk.as<double>(), pl->d_lpit.as<double>());
        CU(ctx, cudaGetLastError());
    }
    loo_finish_kernel<<<grid_for(nw, 128), 128, 0, st>>>(nw, K, Rd, pl->wTd.as<int>(), pl->win_pib_off.as<long long>(), pl->d_lelpd.as<double>(),
                                                        pl->d_llppd.as<double>(), pl->d_lpk.as<double>(), pl->d_lsum.as<double>());
    CU(ctx, cudaGetLastError());
    TRY(download(pl, window_outputs(K, pl->n_h, pl->n_chains, pl->nrun, pl->n_grid, 0, pl->flags), nullptr, nullptr, nullptr, nullptr, lo, nullptr));
    CU(ctx, cudaStreamSynchronize(st));         // (the scratch goes back to the pool when this returns)
    return HMCGPU_OK;
}

static int plan_fetch_loo_impl(hmcgpu_plan* pl, hmcgpu_loo* lo) {
    hmcgpu_ctx* ctx = pl->ctx;
    if (!(pl->flags & HMCGPU_FLAG_LOO)) return fail(ctx, HMCGPU_ERR_ARG, "plan_fetch_loo on a plan without HMCGPU_FLAG_LOO");
    if (!pl->ran) return fail(ctx, HMCGPU_ERR_ARG, "plan_fetch_loo before plan_run");
    CU(ctx, cudaSetDevice(ctx->device));
    tl_pool = ctx->pool;
    return pl->precision == 32 ? fetch_loo_t<float>(pl, lo) : fetch_loo_t<double>(pl, lo);
}

extern "C" int hmcgpu_plan_fetch_loo(hmcgpu_plan* pl, hmcgpu_loo* lo) {
    if (!pl) return HMCGPU_ERR_ARG;
    if (!lo) return fail(pl->ctx, HMCGPU_ERR_ARG, "hmcgpu_loo is NULL");
    GUARD(pl->ctx, plan_fetch_loo_impl(pl, lo));
}

extern "C" void hmcgpu_plan_destroy(hmcgpu_plan* pl) {
    if (!pl) return;
    cudaSetDevice(pl->ctx->device);
    cudaStreamSynchronize(pl->ctx->stream);            // nothing may still be using the buffers that go back to the pool
    for (auto s2 : pl->gstreams) cudaStreamSynchronize(s2);
    delete pl;
}

extern "C" int hmcgpu_estimate(hmcgpu_ctx* ctx, const hmcgpu_problem* p, hmcgpu_result* r) {
    return hmcgpu_estimate_predictive(ctx, p, r, nullptr);
}

extern "C" int hmcgpu_estimate_predictive(hmcgpu_ctx* ctx, const hmcgpu_problem* p, hmcgpu_result* r, hmcgpu_predictive* pr) {
    return hmcgpu_estimate_ranked(ctx, p, r, pr, nullptr);
}

extern "C" int hmcgpu_estimate_ranked(hmcgpu_ctx* ctx, const hmcgpu_problem* p, hmcgpu_result* r, hmcgpu_predictive* pr, hmcgpu_ranked* rk) {
    return hmcgpu_estimate_onestep(ctx, p, r, pr, rk, nullptr);
}

extern "C" int hmcgpu_estimate_onestep(hmcgpu_ctx* ctx, const hmcgpu_problem* p, hmcgpu_result* r, hmcgpu_predictive* pr, hmcgpu_ranked* rk,
                                       hmcgpu_onestep* os) {
    return hmcgpu_estimate_loo(ctx, p, r, pr, rk, os, nullptr);
}

extern "C" int hmcgpu_estimate_loo(hmcgpu_ctx* ctx, const hmcgpu_problem* p, hmcgpu_result* r, hmcgpu_predictive* pr, hmcgpu_ranked* rk,
                                   hmcgpu_onestep* os, hmcgpu_loo* lo) {
    if (!r) return fail(ctx, HMCGPU_ERR_ARG, "result is NULL");
    if (p && (p->flags & HMCGPU_FLAG_LOO) && !lo)
        return fail(ctx, HMCGPU_ERR_ARG, "HMCGPU_FLAG_LOO without hmcgpu_loo outputs (use hmcgpu_estimate_loo)");
    if (p && (p->flags & HMCGPU_FLAG_ONESTEP) && !os)
        return fail(ctx, HMCGPU_ERR_ARG, "HMCGPU_FLAG_ONESTEP without hmcgpu_onestep outputs (use hmcgpu_estimate_onestep)");
    if (p && (p->flags & HMCGPU_FLAG_PREDICTIVE) && !pr)
        return fail(ctx, HMCGPU_ERR_ARG, "HMCGPU_FLAG_PREDICTIVE without hmcgpu_predictive outputs (use hmcgpu_estimate_predictive)");
    if (p && (p->flags & HMCGPU_FLAG_RANKED)) {
        if (!rk) return fail(ctx, HMCGPU_ERR_ARG, "HMCGPU_FLAG_RANKED without hmcgpu_ranked outputs (use hmcgpu_estimate_ranked)");
        TRY(check_ranked(ctx, rk));             // (before the chains run)
    }
    hmcgpu_plan* pl = nullptr;
    PhaseTrace tr;
    TRY(hmcgpu_plan_create(ctx, p, &pl));
    tr.mark("plan_create (upload, init)");
    int rc = hmcgpu_plan_run(pl);
    tr.mark("plan_run (all sweeps)");
    if (rc == 0) rc = hmcgpu_plan_fetch(pl, r);
    if (rc >= 0 && (p->flags & HMCGPU_FLAG_PREDICTIVE)) {
        const int rp = hmcgpu_plan_fetch_predictive(pl, pr);
        if (rp < 0) rc = rp;
    }
    if (rc >= 0 && (p->flags & HMCGPU_FLAG_RANKED)) {
        const int rp = hmcgpu_plan_fetch_ranked(pl, rk);
        if (rp < 0) rc = rp;
    }
    if (rc >= 0 && (p->flags & HMCGPU_FLAG_ONESTEP)) {
        const int rp = hmcgpu_plan_fetch_onestep(pl, os);
        if (rp < 0) rc = rp;
    }
    if (rc >= 0 && (p->flags & HMCGPU_FLAG_LOO)) {
        const int rp = hmcgpu_plan_fetch_loo(pl, lo);
        if (rp < 0) rc = rp;
    }
    tr.mark("plan_fetch (download)");
    hmcgpu_plan_destroy(pl);
    tr.mark("plan_destroy");
    return rc;
}

// Windows sharded over devices by longest-processing-time-first on T_w; one host thread per device, no collectives.
static int estimate_multi_impl(const int* devices, int n_dev, const hmcgpu_problem* p, hmcgpu_result* r, hmcgpu_predictive* pr,
                               hmcgpu_ranked* rk, hmcgpu_onestep* os, hmcgpu_loo* lo);
extern "C" int hmcgpu_estimate_multi(const int* devices, int n_dev, const hmcgpu_problem* p, hmcgpu_result* r) {
    return hmcgpu_estimate_multi_ranked(devices, n_dev, p, r, nullptr, nullptr);
}

extern "C" int hmcgpu_estimate_multi_predictive(const int* devices, int n_dev, const hmcgpu_problem* p, hmcgpu_result* r,
                                                hmcgpu_predictive* pr) {
    return hmcgpu_estimate_multi_ranked(devices, n_dev, p, r, pr, nullptr);
}

extern "C" int hmcgpu_estimate_multi_ranked(const int* devices, int n_dev, const hmcgpu_problem* p, hmcgpu_result* r,
                                            hmcgpu_predictive* pr, hmcgpu_ranked* rk) {
    return hmcgpu_estimate_multi_onestep(devices, n_dev, p, r, pr, rk, nullptr);
}

extern "C" int hmcgpu_estimate_multi_onestep(const int* devices, int n_dev, const hmcgpu_problem* p, hmcgpu_result* r,
                                             hmcgpu_predictive* pr, hmcgpu_ranked* rk, hmcgpu_onestep* os) {
    return hmcgpu_estimate_multi_loo(devices, n_dev, p, r, pr, rk, os, nullptr);
}

extern "C" int hmcgpu_estimate_multi_loo(const int* devices, int n_dev, const hmcgpu_problem* p, hmcgpu_result* r,
                                         hmcgpu_predictive* pr, hmcgpu_ranked* rk, hmcgpu_onestep* os, hmcgpu_loo* lo) {
    if (!devices || n_dev < 1 || !p || !r) return fail(nullptr, HMCGPU_ERR_ARG, "bad arguments");
    if ((p->flags & HMCGPU_FLAG_LOO) && !lo)
        return fail(nullptr, HMCGPU_ERR_ARG, "HMCGPU_FLAG_LOO without hmcgpu_loo outputs (use hmcgpu_estimate_multi_loo)");
    if ((p->flags & HMCGPU_FLAG_ONESTEP) && !os)
        return fail(nullptr, HMCGPU_ERR_ARG, "HMCGPU_FLAG_ONESTEP without hmcgpu_onestep outputs (use hmcgpu_estimate_multi_onestep)");
    if ((p->flags & HMCGPU_FLAG_PREDICTIVE) && !pr)
        return fail(nullptr, HMCGPU_ERR_ARG, "HMCGPU_FLAG_PREDICTIVE without hmcgpu_predictive outputs (use hmcgpu_estimate_multi_predictive)");
    if (p->flags & HMCGPU_FLAG_RANKED) {
        if (!rk) return fail(nullptr, HMCGPU_ERR_ARG, "HMCGPU_FLAG_RANKED without hmcgpu_ranked outputs (use hmcgpu_estimate_multi_ranked)");
        TRY(check_ranked(nullptr, rk));
    }
    GUARD(nullptr, estimate_multi_impl(devices, n_dev, p, r, (p->flags & HMCGPU_FLAG_PREDICTIVE) ? pr : nullptr,
                                       (p->flags & HMCGPU_FLAG_RANKED) ? rk : nullptr, (p->flags & HMCGPU_FLAG_ONESTEP) ? os : nullptr,
                                       (p->flags & HMCGPU_FLAG_LOO) ? lo : nullptr));
}

static int estimate_multi_impl(const int* devices, int n_dev, const hmcgpu_problem* p, hmcgpu_result* r, hmcgpu_predictive* pr,
                               hmcgpu_ranked* rk, hmcgpu_onestep* os, hmcgpu_loo* lo) {
    if (p->n_windows < 1 || !p->win_start || !p->win_end) return fail(nullptr, HMCGPU_ERR_ARG, "no windows");
    const int nw = p->n_windows;
    std::vector<int> ord(nw);
    std::iota(ord.begin(), ord.end(), 0);
    auto Tw = [&](int w) { return p->win_end[w] - p->win_start[w] + 1; };
    std::stable_sort(ord.begin(), ord.end(), [&](int a, int b) { return Tw(a) > Tw(b); });
    std::vector<std::vector<int>> shard(n_dev);
    std::vector<long long> load(n_dev, 0);
    for (int w : ord) {
        const int d = (int)(std::min_element(load.begin(), load.end()) - load.begin());
        shard[d].push_back(w);
        load[d] += Tw(w);
    }
    std::vector<long long> T0(nw + 1, 0);                   // T_0 + ... + T_{w-1}: window w's offset in X0 and the ragged outputs
    for (int w = 0; w < nw; ++w) T0[w + 1] = T0[w] + Tw(w);
    // (pr is given only with HMCGPU_FLAG_PREDICTIVE, the only case in which n_grid may be read; rk only with HMCGPU_FLAG_RANKED)
    const std::vector<WinOut> outs = window_outputs(p->K, p->n_h, p->n_chains, p->nrun, pr ? p->n_grid : 0, rk ? rk->n_probs : 0, p->flags);
    std::vector<int> rcs(n_dev, 0);
    std::vector<std::string> errs(n_dev);
    std::vector<hmcgpu_result> parts(n_dev);
    std::vector<std::thread> th;
    for (int d = 0; d < n_dev; ++d) {
        th.emplace_back([&, d]() {
          hmcgpu_ctx* ctx = nullptr;
          try {
            const std::vector<int>& ws = shard[d];
            const int n = (int)ws.size();
            memset(&parts[d], 0, sizeof(hmcgpu_result));
            if (n == 0) return;
            int rc = hmcgpu_ctx_create(devices[d], &ctx);
            if (rc != 0) { rcs[d] = rc; errs[d] = hmcgpu_last_error(nullptr); return; }
            std::vector<int32_t> ser(n), iser(n), st(n), en(n);
            std::vector<int64_t> id(n), x0;
            long long sum_T = 0;
            for (int j = 0; j < n; ++j) {
                const int w = ws[j];
                ser[j] = p->win_series ? p->win_series[w] : 0; st[j] = p->win_start[w]; en[j] = p->win_end[w];
                iser[j] = p->win_init_series ? p->win_init_series[w] : ser[j];
                id[j] = p->win_id ? p->win_id[w] : w;
                sum_T += Tw(w);
                if (p->X0) x0.insert(x0.end(), p->X0 + T0[w], p->X0 + T0[w + 1]);
            }
            hmcgpu_problem q = *p;
            q.n_windows = n; q.win_series = ser.data(); q.win_start = st.data(); q.win_end = en.data(); q.win_id = id.data();
            if (p->win_init_series) q.win_init_series = iser.data();
            if (p->X0) q.X0 = x0.data();
            // the shard's outputs in host staging arrays (of at least one byte: a requested output stays a non-NULL pointer)
            hmcgpu_result& o = parts[d];
            hmcgpu_predictive pq{};
            hmcgpu_ranked rq{};
            hmcgpu_onestep oq{};
            hmcgpu_loo lq{};
            if (rk) { rq.probs = rk->probs; rq.n_probs = rk->n_probs; }
            std::vector<std::vector<char>> stage(outs.size());
            for (size_t i = 0; i < outs.size(); ++i) {
                if (!outs[i].get(r, pr, rk, os, lo)) continue;
                stage[i].resize(std::max<size_t>(1, (size_t)outs[i].elems(n, sum_T) * outs[i].elem));
                outs[i].set(&o, &pq, &rq, &oq, &lq, stage[i].data());
            }
            rc = hmcgpu_estimate_loo(ctx, &q, &o, pr ? &pq : nullptr, rk ? &rq : nullptr, os ? &oq : nullptr, lo ? &lq : nullptr);
            rcs[d] = rc;
            if (rc < 0) errs[d] = hmcgpu_last_error(ctx);
            for (size_t i = 0; rc >= 0 && i < outs.size(); ++i) {   // scatter this shard's windows into the caller's arrays
                const WinOut& x = outs[i];
                char* dst = (char*)x.get(r, pr, rk, os, lo);
                if (!dst) continue;
                long long t = 0;                                 // steps of the shard's windows before window j
                for (int j = 0; j < n; ++j) {
                    const int w = ws[j];
                    memcpy(dst + x.elems(w, T0[w]) * x.elem, stage[i].data() + x.elems(j, t) * x.elem, x.elems(1, Tw(w)) * x.elem);
                    t += Tw(w);
                }
            }
            hmcgpu_ctx_destroy(ctx);
          } catch (const std::exception& e) {     // an exception escaping a std::thread would terminate the host process
            rcs[d] = HMCGPU_ERR_ALLOC; errs[d] = std::string("host allocation failed: ") + e.what();
            if (ctx) hmcgpu_ctx_destroy(ctx);
          }
        });
    }
    for (auto& t : th) t.join();
    int bad = 0;
    r->gpu_ms = 0; r->sweep_kernel_ms = 0; r->n_launches = 0; r->n_sweep_launches = 0; r->h2d_bytes = 0; r->d2h_bytes = 0; r->state_steps = 0;
    r->sweep_launch_ms_sum = 0; r->sweep_kernel = 0; r->n_tasks = 0;
    for (int d = 0; d < n_dev; ++d) {
        if (rcs[d] < 0) return fail(nullptr, rcs[d], "device %d: %s", devices[d], errs[d].c_str());
        bad += rcs[d];
        r->gpu_ms = std::max(r->gpu_ms, parts[d].gpu_ms);
        r->sweep_kernel_ms = std::max(r->sweep_kernel_ms, parts[d].sweep_kernel_ms);
        r->n_launches += parts[d].n_launches; r->n_sweep_launches += parts[d].n_sweep_launches;
        r->h2d_bytes += parts[d].h2d_bytes; r->d2h_bytes += parts[d].d2h_bytes; r->state_steps += parts[d].state_steps;
        r->sweep_launch_ms_sum += parts[d].sweep_launch_ms_sum; r->n_tasks += parts[d].n_tasks;
        if (shard[d].size()) r->sweep_kernel = parts[d].sweep_kernel;
    }
    return bad;
}
