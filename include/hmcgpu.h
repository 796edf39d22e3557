/*
 * hmcgpu.h — C ABI of the B200 (sm_100a) Gibbs/FFBS path that replaces the hot loop of joe5saia/Hmc.jl.
 *
 * Plain C: opaque handles, plain pointers and sizes, int return codes.  No C++ types, no exceptions,
 * no stdout, no exit() cross this boundary.  Julia binds it with `ccall` (hmc.jl_b200/julia/HmcGPU.jl),
 * the test harness with Python ctypes (hmc.jl_b200/binding.py); both see exactly these symbols.
 *
 * Reference interfaces replaced (paths under the reference checkout, src/Hmc.jl):
 *   hmcgpu_estimate / hmcgpu_plan_*  <- estimatemodel (:850-865) = makeParams (:161-195) + HyperParams (:132-142)
 *                                       + gibbssample! (:517-562, gibbssweep! :486-515) + forecast loop (:858-862);
 *                                       called from code/run_hmm.jl:119
 *   hmcgpu_filter / _filter_masked   <- forwardupdate_P! (:371-440)   (fixed parameters -> pif, totals, loglik; signal rows)
 *   hmcgpu_smooth                    <- backwardupdate_P! (:442-457)  (marginals pib)
 *   hmcgpu_sample_states             <- update_X! (:459-484)          (injected uniforms -> state path)
 *   hmcgpu_draw_params / _signals    <- update_μσ! draws (:302-335; with signal statistics :267-314), update_ρ! (:350-356),
 *                                       update_A! (:358-369)
 *   hmcgpu_forecast                  <- forecast (:658-667)
 *
 * Conventions
 *   - All host arrays are fp64 (int64 for states) whatever the device precision.
 *   - Batched deterministic calls use row-major [batch][...] arrays: A[b][r][s] = P(X_t=s|X_{t-1}=r),
 *     pif[b][t][s], sigma2 holds VARIANCES (as the reference's σ does).
 *   - hmcgpu_estimate outputs use Julia COLUMN-MAJOR layout per window so Julia can wrap them without
 *     a copy (see hmcgpu_result).
 *   - States are 1-based in X, windows are 1-based inclusive [start,end] like `sampleRange`.
 *   - Ownership: the caller owns every pointer it passes; the library copies what it needs before
 *     returning and never frees or retains host pointers.  Device memory belongs to ctx / plan.
 *   - Threading: a ctx is bound to one GPU and is not re-entrant; different ctxs may be driven from
 *     different host threads concurrently.
 *   - Return codes: 0 = OK; < 0 = error (message via hmcgpu_last_error); > 0 (estimate/plan_fetch only)
 *     = number of chains that saw a zero-normaliser / non-finite event (data still returned — mirrors the
 *     reference's warn-and-continue, :319-329, :435, :472-480).
 *   - There is no CPU fallback: without a CUDA device every compute entry point returns HMCGPU_ERR_NODEVICE.
 */
#ifndef HMCGPU_H
#define HMCGPU_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HMCGPU_OK 0
#define HMCGPU_ERR_ARG (-1)
#define HMCGPU_ERR_CUDA (-2)
#define HMCGPU_ERR_ALLOC (-3)
#define HMCGPU_ERR_UNSUPPORTED (-4)
#define HMCGPU_ERR_NODEVICE (-5)

/* hmcgpu_problem.flags */
#define HMCGPU_FLAG_REF_Q1 1u        /* reproduce :512-514 (X[N] drawn from the relabelled pif[N,:]); hosts set it by default */
#define HMCGPU_FLAG_DRAWS 2u         /* fill the per-draw arrays of hmcgpu_result */
#define HMCGPU_FLAG_SUMMARY 4u       /* fill per-window posterior mean / variance (pooled over chains and draws) */
#define HMCGPU_FLAG_SMOOTHED_MEAN 8u /* fill pib_mean: posterior mean of the smoothed state probabilities */
#define HMCGPU_FLAG_LOGLIK 16u       /* compute the per-draw log-likelihood sum_t log(total_t) */
#define HMCGPU_FLAG_FILTERED_MEAN 64u /* fill pib_mean / insample_forecast_mean with the posterior means of the FILTERED state
                                        probabilities pif[t,:] and of pif[t,:]' A^h mu (what the reference's published in-sample table
                                        data/output/official_insample/forecats_insample.csv holds); K <= 8, not with SMOOTHED_MEAN or signals */
#define HMCGPU_FLAG_DIAGNOSTICS  128u /* fill rhat / ess / ess_lag: split-R̂ and effective sample size per window and summary field,
                                        computed on the device from every saved draw; needs nrun >= 4 (see hmcgpu_result) */
#define HMCGPU_FLAG_PREDICTIVE  256u /* fill hmcgpu_predictive: posterior predictive CDF on pred_grid, PIT, log score and moments per
                                        window and horizon, computed on the device from every saved draw (see hmcgpu_predictive) */
#define HMCGPU_FLAG_RANKED  512u     /* keep every saved draw on the device so that hmcgpu_plan_fetch_ranked can compute exact quantiles,
                                        rank-normalised R̂ and bulk / tail ESS; needs nrun >= 4 and n_chains * nrun < 2^31 (see hmcgpu_ranked) */

typedef struct hmcgpu_ctx hmcgpu_ctx;
typedef struct hmcgpu_plan hmcgpu_plan;

/* One rolling-window estimation job = what code/run_hmm.jl builds in `opt` (:95-109), for many end dates at once. */
typedef struct hmcgpu_problem {
    const double* y;          /* series, COLUMN-major [y_len x n_series] (series s at y + s*y_len) = opt.rawdata */
    int64_t y_len;
    int32_t n_series;         /* >= 1 */
    int32_t n_windows;        /* independent estimation windows (end dates) */
    const int32_t* win_series;/* [n_windows] 0-based series index, NULL = all 0 */
    const int32_t* win_start; /* [n_windows] 1-based first index of sampleRange */
    const int32_t* win_end;   /* [n_windows] 1-based last index of sampleRange (= endIndex) */
    const int64_t* win_id;    /* [n_windows] global window id used in the RNG counter, NULL = 0..n_windows-1.
                                 Makes results independent of how windows are sharded over GPUs. */
    int32_t K;                /* number of states D */
    int32_t n_chains;         /* independent chains per window (reference: 1) */
    int64_t burnin, nrun;     /* opt.burnin, opt.Nrun */
    uint64_t seed;            /* opt.seed -> Philox key */
    const double* xi;         /* [K] prior mean; NULL = mean(Y_window) (:136) */
    const double* alpha;      /* [K] NULL = 1 (:137) */
    const double* nu;         /* [K] NULL = 1 (:140) */
    const double* beta0;      /* [K] β used by the first sweep; NULL = 1 (:179) */
    const double* beta;       /* [K] β afterwards; NULL = 2 (:347) */
    double kappa;             /* hp.κ = opt.noise (:116, :158): signals are emitted with sd*(1+κ) (:382) and weigh 1/(1+κ) in
                                 the statistics (:302, :314); only used with is_signal */
    const uint8_t* is_signal; /* [y_len] 1 = time index belongs to opt.signalRange (noisy signal), 0 = observation: one mask for
                                 every series, or [y_len x n_series] column-major like y when is_signal_per_series != 0.
                                 NULL = no signals (estimatemodel).  K <= 4, not with SMOOTHED_MEAN. */
    const int32_t* horizons;  /* [n_h] forecast horizons >= 0 from the window end (reference scripts: {12}); 0 = pi_end'mu */
    int32_t n_h;
    const int64_t* X0;        /* [sum_w T_w] initial state paths (1-based states), windows concatenated in caller order and
                                 shared by the window's chains; NULL = makeParams rule (:185-187) */
    int32_t precision;        /* 32 or 64: device arithmetic */
    uint32_t flags;
    /* ---- signals tier (estimatesignals!, :868-914); zero / NULL = estimatemodel behaviour */
    const int32_t* win_init_series; /* [n_windows] series the makeParams / HyperParams rules read (X0, default xi), while the
                                 chain itself runs on win_series: estimatesignals! initialises from the real data and
                                 estimates on the perturbed copy (:888-892).  NULL = win_series */
    int32_t pi_row_back;      /* pi_end (and its summary) = smoothed marginal pib[N - pi_row_back, :] instead of the last row:
                                 samples.πb[:, opt.endIndex, :] with signalLen rows after endIndex (:893).  K <= 4. */
    int32_t is_signal_per_series; /* 0: is_signal holds y_len flags; 1: y_len flags per series (many end dates, each with its
                                 own signalRange, in one call) */
    /* ---- appended in ABI version 400: read only with HMCGPU_FLAG_PREDICTIVE (older callers are never read past their end) */
    const double* pred_grid;  /* [n_grid] finite, strictly increasing points at which the predictive CDF is evaluated; shared by
                                 every window and horizon */
    int32_t n_grid;           /* 1..512 */
} hmcgpu_problem;

/* Caller-allocated outputs; any pointer may be NULL.  R = n_chains*nrun draws per window, draw index
 * d = chain*nrun + i (chain-major).  Per window w the arrays are Julia column-major, windows concatenated:
 *   mu[w*R*K + k*R + d], sigma2 likewise, pi_end likewise (= samples.πb[:,end,:], :744)
 *   A[w*R*K*K + (s*K + r)*R + d]            (reshape(A,R,:) gives trans columns as saveresults expects, :745)
 *   forecasts[w*R*2*n_h + (2*j+e)*R + d]    e=0 forecast, e=1 forecast error for horizons[j] (:858-862)
 *   loglik[w*R + d]
 * States are emitted in increasing-μ order (:501-513).
 * Summary fields per window, F = 3K + K*K + 2*n_h + 1 in the order
 *   mu[K], sigma2[K], A[K*K] (index s*K+r), pi_end[K], forecasts[2*n_h], loglik:
 *   summary_mean[w*F + f], summary_var[w*F + f]  (population variance over the R pooled draws; the loglik field is 0
 *   unless HMCGPU_FLAG_LOGLIK is set)
 * pib_mean: per window N_w x K column-major, concatenated: offset_w = K * sum_{v<w} N_v.
 * insample_forecast_mean: per window N_w x n_h column-major, concatenated (offset_w = n_h * sum_{v<w} N_v): the posterior
 *   mean of pib[t,:]' A^h mu for every date t of the window and every horizon (forecastinsample, src/Hmc.jl:683-699);
 *   the forecast error of date t is this minus y[t+h].  Needs HMCGPU_FLAG_SMOOTHED_MEAN (K <= 4).
 * status[w*n_chains + c]: event count of that chain.
 * rhat, ess, ess_lag [w*F + f] (HMCGPU_FLAG_DIAGNOSTICS; same fields and order as summary_mean): convergence diagnostics of each
 *   summary field over the window's chains.  Each chain's nrun saved draws are split into two sequences of n = floor(nrun/2)
 *   draws (the middle draw of an odd nrun is dropped), M = 2*n_chains sequences in all.  With W the mean of the sequences'
 *   variances (denominator n-1) and B/n the variance of their means (denominator M-1), var+ = (n-1)/n W + B/n and
 *   rhat = sqrt(var+ / W): the classic split-R̂ of BDA3, NOT rank-normalised.  ess = M n / tau with
 *   tau = max(-1 + 2 sum_k P_k, 1/log10(M n)), P_k = rho_2k + rho_2k+1 summed while positive and made non-increasing
 *   (Geyer's initial monotone sequence), rho_l = 1 - (W - mean_m gamma_m,l) / var+ from the sequences' autocovariances
 *   gamma_m,l (denominator n).  Lags are capped at 63 (32 pairs): ess_lag is the last lag summed, and ess_lag equal to the
 *   largest odd lag <= min(63, n-1) means the sum was cut at the cap and ess over-estimates the effective sample size.
 *   A field with a non-finite draw (e.g. the forecast error of a horizon past the end of the series) or W = 0 (a constant
 *   field), and the loglik field without HMCGPU_FLAG_LOGLIK, give rhat = ess = NaN and ess_lag = -1.  Bit-identical for a
 *   window however the windows are batched or sharded (given the same draws).
 *   These three pointers were appended in ABI version 300 and are read only when HMCGPU_FLAG_DIAGNOSTICS is set, so a caller
 *   built against the shorter struct is never read past its end. */
typedef struct hmcgpu_result {
    double* mu;
    double* sigma2;
    double* A;
    double* pi_end;
    double* forecasts;
    double* loglik;
    double* summary_mean;
    double* summary_var;
    double* pib_mean;
    double* insample_forecast_mean;
    int32_t* status;
    /* filled by the library */
    double gpu_ms;        /* device time of the whole run: chain init, every sweep launch, per-chunk post-processing (CUDA
                             events on the library's stream) */
    double sweep_kernel_ms; /* device time from the start of the first Gibbs sweep launch to the end of the last one (CUDA events
                             on the task-group streams; the launches of different groups overlap, so this is their enclosing
                             interval — it leaves out the init kernel and the post-processing after the last sweep) */
    int64_t n_launches;   /* kernels launched for this job */
    int64_t n_sweep_launches; /* launches of the Gibbs sweep kernel among them */
    int64_t h2d_bytes, d2h_bytes;
    int64_t state_steps;  /* sum_w T_w * n_chains * (burnin + nrun) */
    /* ---- appended in ABI version 200 (older callers that zero-initialise the struct keep working) */
    double sweep_launch_ms_sum; /* sum over the sweep-kernel launches of each launch's own duration (an event pair around every
                             launch on its stream); divided by n_sweep_launches = the average launch duration */
    int32_t sweep_kernel; /* which sweep kernel the plan chose: HMCGPU_KERNEL_* */
    int32_t n_tasks;      /* warp tasks of that kernel (32 lanes each) */
    /* ---- appended in ABI version 300 (read only with HMCGPU_FLAG_DIAGNOSTICS) */
    double* rhat;         /* [n_windows x F] split-R̂ */
    double* ess;          /* [n_windows x F] effective sample size */
    int32_t* ess_lag;     /* [n_windows x F] last autocorrelation lag in the ESS sum */
} hmcgpu_result;

/* Posterior predictive distribution (HMCGPU_FLAG_PREDICTIVE); caller-allocated, any pointer may be NULL.
 * Draw d of window w (emitted fields: mu_s, sigma2_s, A[r][s], pi = pi_end) gives for horizon h_j = horizons[j] the mixture
 *   weights v = pi' A^h_j (v_s = sum_r pi_r (A^h_j)[r][s], so sum_s v_s mu_s is the draw's forecast field),
 *   F_d(x) = sum_s v_s Phi((x - mu_s) / sqrt(sigma2_s)),   p_d(x) = sum_s v_s phi((x - mu_s) / sqrt(sigma2_s)) / sqrt(sigma2_s).
 * Pooled over the R = n_chains*nrun draws, with y+ = y[end_w + h_j] of the window's series (the value the forecast error uses,
 * fp64; NaN past the end of the series) and c_w = y[end_w]:
 *   cdf[(w*n_h + j)*n_grid + g] = (1/R) sum_d F_d(pred_grid[g])
 *   pit[w*n_h + j]              = (1/R) sum_d F_d(y+)            (NaN when y+ is NaN)
 *   log_score[w*n_h + j]        = log((1/R) sum_d p_d(y+))       (NaN when y+ is NaN)
 *   moments[(w*n_h + j)*3 + k]  = mean, variance, skewness of the pooled mixture, from the raw moments about c_w
 *                                 M1 = sum_s v_s (mu_s - c_w), M2 = sum_s v_s ((mu_s - c_w)^2 + sigma2_s),
 *                                 M3 = sum_s v_s ((mu_s - c_w)^3 + 3 (mu_s - c_w) sigma2_s) averaged over the draws
 * All predictive arithmetic is fp64 on the draws as the plan produced them, converted to double, whatever the precision.  A window
 * with a non-finite mu / sigma2 / A / pi_end draw gets NaN in every output.  Every sum runs in draw order, then chain order, with
 * no atomics: a window's outputs are bit-identical however the windows are batched, chunked or sharded.
 * Needs n_h >= 1, 1 <= n_grid <= 512 and pi_row_back == 0 (with pi_row_back the emitted pi_end is a smoothed row, not the vector
 * the forecasts are built from).  Device state: 8 * n_slots * n_h * (n_grid + 5) bytes (n_slots ~ n_windows * n_chains, e.g.
 * 0.85 GB for 128 000 chains, n_h = 12, n_grid = 64), allocated only with the flag. */
typedef struct hmcgpu_predictive {
    double* cdf;          /* [n_windows][n_h][n_grid] */
    double* pit;          /* [n_windows][n_h] */
    double* log_score;    /* [n_windows][n_h] */
    double* moments;      /* [n_windows][n_h][3] */
} hmcgpu_predictive;

/* Ranked outputs (HMCGPU_FLAG_RANKED); caller-allocated, any output pointer may be NULL.  Per window w and summary field f (the
 * fields and order of summary_mean), over the R = n_chains*nrun saved draws x_d converted to double (d = chain*nrun + i):
 *   quantiles[(w*F + f)*n_probs + k]  type 7 (numpy method="linear"): with h = (R-1) p_k and the sorted draws x_(j) (0-based),
 *                                     q(p) = x_(floor h) + (h - floor h) (x_(floor h + 1) - x_(floor h))
 *   ranks r_d                         1-based over the R draws, ties averaged, -0.0 and +0.0 tied; normal scores
 *                                     z_d = Phi^-1((r_d - 3/8) / (R + 1/4))
 *   bulk R̂ / ESS                      the split-R̂ and ESS of rhat / ess above: same split, Geyer's initial monotone sequence, lags
 *                                     capped at 63, applied to z
 *   folded R̂                          the same applied to the normal scores of |x - q(0.5)| (fold taken in fp64)
 *   rhat_rank[w*F + f]                max(bulk R̂, folded R̂)
 *   ess_bulk[w*F + f]                 the bulk ESS
 *   ess_tail[w*F + f]                 min(ESS of 1[x <= q(0.05)], ESS of 1[x <= q(0.95)])
 * A field with a non-finite draw, and the loglik field without HMCGPU_FLAG_LOGLIK, get NaN in every output, quantiles included.
 * R̂ and ESS are NaN where the split-R̂ definition gives NaN (W = 0: a constant field, a constant indicator); rhat_rank and
 * ess_tail are NaN when either of their parts is.  A constant field's quantiles are the constant.  Every sum runs in a fixed
 * order with no atomics: a window's outputs are bit-identical however the windows are batched, chunked or sharded.
 * Device memory: n_windows * F * n_chains * nrun * (precision / 8) bytes of retained draws (C2: 500 windows x 43 fields x 256
 * chains x 1000 draws in fp32 = 22 GB), checked against the device's total memory at hmcgpu_plan_create (HMCGPU_ERR_ALLOC when
 * they do not fit), plus about 2 GiB of scratch at fetch. */
typedef struct hmcgpu_ranked {
    const double* probs;  /* [n_probs] quantile probabilities, finite, in [0, 1] (input) */
    int32_t n_probs;      /* 0..64; 0 = no quantiles */
    double* quantiles;    /* [n_windows][F][n_probs] */
    double* rhat_rank;    /* [n_windows x F] rank-normalised split-R̂: max(bulk, folded) */
    double* ess_bulk;     /* [n_windows x F] */
    double* ess_tail;     /* [n_windows x F] */
} hmcgpu_ranked;

#define HMCGPU_KERNEL_THREAD 0  /* one thread per chain (gibbs_sweeps_kernel), wide batches, K <= 8 */
#define HMCGPU_KERNEL_SCAN 1    /* one warp per chain, time-parallel scans (gibbs_scan_kernel), narrow batches */
#define HMCGPU_KERNEL_LANE 2    /* one lane per state (gibbs_wide_kernel), K = 9..32 */
#define HMCGPU_KERNEL_PAIR 3    /* reserved (the two-chains-per-thread kernel of round 1 was removed: slower than the default at every width) */
#define HMCGPU_KERNEL_SEG 4     /* L lanes per chain, each lane a contiguous time segment (gibbs_seg_kernel), mid-width batches */

int hmcgpu_version(void);
/* "<abi version>;<hash of the CUDA/C sources the library was built from>" — hosts compare the hash with the sources next to
 * them and refuse (or rebuild) a stale library */
const char* hmcgpu_build_info(void);
/* number of CUDA devices visible (0 if none / no driver) */
int hmcgpu_device_count(void);
int hmcgpu_ctx_create(int device, hmcgpu_ctx** out);
void hmcgpu_ctx_destroy(hmcgpu_ctx* ctx);
/* message of the last error on this ctx (ctx may be NULL: last error of ctx_create on this thread) */
const char* hmcgpu_last_error(const hmcgpu_ctx* ctx);
/* blocks until all work queued by this ctx has finished */
int hmcgpu_ctx_sync(hmcgpu_ctx* ctx);
/* Releases the idle device buffers the context keeps for reuse between calls (bounded by HMCGPU_POOL_MAX_GB, default 16 GiB;
 * they are also released when an allocation on this context fails and at hmcgpu_ctx_destroy). */
int hmcgpu_ctx_trim(hmcgpu_ctx* ctx);

/* Whole estimation, host buffers in and out (H2D, all sweeps, D2H inside the call).  = hmcgpu_estimate_predictive(.., NULL) */
int hmcgpu_estimate(hmcgpu_ctx* ctx, const hmcgpu_problem* p, hmcgpu_result* r);
/* Same, windows sharded over several GPUs by sum of T_w (one host thread per device, no collectives).
 * = hmcgpu_estimate_multi_predictive(.., NULL) */
int hmcgpu_estimate_multi(const int* devices, int n_devices, const hmcgpu_problem* p, hmcgpu_result* r);
/* The same two calls filling the posterior predictive outputs too.  With HMCGPU_FLAG_PREDICTIVE, pr must not be NULL
 * (HMCGPU_ERR_ARG: the library does not compute what it would discard); without it pr is ignored.  The multi-GPU form
 * scatters each shard's rows into the caller's window order. */
int hmcgpu_estimate_predictive(hmcgpu_ctx* ctx, const hmcgpu_problem* p, hmcgpu_result* r, hmcgpu_predictive* pr);
int hmcgpu_estimate_multi_predictive(const int* devices, int n_devices, const hmcgpu_problem* p, hmcgpu_result* r,
                                     hmcgpu_predictive* pr);
/* The same filling the ranked outputs too (hmcgpu_estimate_predictive and hmcgpu_estimate_multi_predictive are these with
 * rk = NULL).  With HMCGPU_FLAG_RANKED, rk must not be NULL (HMCGPU_ERR_ARG); without it rk is ignored. */
int hmcgpu_estimate_ranked(hmcgpu_ctx* ctx, const hmcgpu_problem* p, hmcgpu_result* r, hmcgpu_predictive* pr, hmcgpu_ranked* rk);
int hmcgpu_estimate_multi_ranked(const int* devices, int n_devices, const hmcgpu_problem* p, hmcgpu_result* r,
                                 hmcgpu_predictive* pr, hmcgpu_ranked* rk);

/* Split form: create uploads inputs and allocates device state; run executes every sweep (inputs resident
 * in HBM, no host transfers); fetch copies the requested outputs back.  run may be repeated (it restarts
 * the chains from the initial state). */
int hmcgpu_plan_create(hmcgpu_ctx* ctx, const hmcgpu_problem* p, hmcgpu_plan** out);
int hmcgpu_plan_run(hmcgpu_plan* plan);
int hmcgpu_plan_fetch(hmcgpu_plan* plan, hmcgpu_result* r);
/* Posterior predictive outputs of the last run; HMCGPU_ERR_ARG on a plan without HMCGPU_FLAG_PREDICTIVE or before a run. */
int hmcgpu_plan_fetch_predictive(hmcgpu_plan* plan, hmcgpu_predictive* pr);
/* Ranked outputs of the last run, computed now from the retained draws; may be called again with other probs without running
 * the plan again.  HMCGPU_ERR_ARG on a plan without HMCGPU_FLAG_RANKED, before a run, with n_probs outside 0..64 or a
 * probability that is not finite or outside [0, 1]. */
int hmcgpu_plan_fetch_ranked(hmcgpu_plan* plan, hmcgpu_ranked* rk);
void hmcgpu_plan_destroy(hmcgpu_plan* plan);

/* Forward filter for fixed parameters.  y: [T] shared by the batch (y_batch_stride = 0) or [B][T]
 * (y_batch_stride = T).  totals [B][T] and loglik [B] may be NULL. */
int hmcgpu_filter(hmcgpu_ctx* ctx, int32_t precision, int32_t K, int64_t B, int64_t T,
                  const double* y, int64_t y_batch_stride,
                  const double* A, const double* mu, const double* sigma2, const double* rho,
                  double* pif, double* totals, double* loglik);
/* Same with the signal branch of forwardupdate_P! (:380-383, :396, :424): is_signal [T] flags the rows emitted with
 * sd*(1+kappa) (one mask for the whole batch; NULL = hmcgpu_filter).  K <= 4. */
int hmcgpu_filter_masked(hmcgpu_ctx* ctx, int32_t precision, int32_t K, int64_t B, int64_t T,
                         const double* y, int64_t y_batch_stride, const uint8_t* is_signal, double kappa,
                         const double* A, const double* mu, const double* sigma2, const double* rho,
                         double* pif, double* totals, double* loglik);
/* Smoothed marginals pib [B][T][K] from pif [B][T][K] and A [B][K][K]. */
int hmcgpu_smooth(hmcgpu_ctx* ctx, int32_t precision, int32_t K, int64_t B, int64_t T,
                  const double* A, const double* pif, double* pib);
/* Backward state sampling with injected uniforms u [B][T] in [0,1); fp64, bit-exact against the oracle's
 * pif form.  piN [B][K] (NULL = pif[:,T-1,:]) is what X[T] is drawn from.  X [B][T], 1-based. */
int hmcgpu_sample_states(hmcgpu_ctx* ctx, int32_t K, int64_t B, int64_t T,
                         const double* A, const double* pif, const double* piN, const double* u, int64_t* X);
/* Conjugate draws from sufficient statistics with the library's Philox streams (chain ids chain0..chain0+B-1).
 * Ni [B][K] counts, S [B][K] sums, S2 [B][K] centred sums of squares, trans [B][K][K] counts INCLUDING the +1 prior. */
int hmcgpu_draw_params(hmcgpu_ctx* ctx, int32_t precision, int32_t K, int64_t B,
                       const int64_t* Ni, const double* S, const double* S2, const int64_t* trans,
                       const double* xi, const double* alpha, const double* nu, const double* beta,
                       uint64_t seed, uint32_t chain0, uint32_t sweep,
                       double* sigma2, double* mu, double* rho, double* A);
/* Same with the noisy signals of update_μσ! (:267-314): Mi [B][K] signal counts, Sm [B][K] sums, Sm2 [B][K] centred sums of
 * squares of the signals of each state, kappa their relative imprecision (Ni / S / S2 then cover the observations only).  K <= 4. */
int hmcgpu_draw_params_signals(hmcgpu_ctx* ctx, int32_t precision, int32_t K, int64_t B,
                               const int64_t* Ni, const double* S, const double* S2,
                               const int64_t* Mi, const double* Sm, const double* Sm2, double kappa, const int64_t* trans,
                               const double* xi, const double* alpha, const double* nu, const double* beta,
                               uint64_t seed, uint32_t chain0, uint32_t sweep,
                               double* sigma2, double* mu, double* rho, double* A);
/* out [B][2*n_h]: forecast and error for each horizon; yreal [n_h]. */
int hmcgpu_forecast(hmcgpu_ctx* ctx, int32_t K, int64_t B, const double* mu, const double* A, const double* pi,
                    const int32_t* horizons, int32_t n_h, const double* yreal, double* out);
/* Raw Philox4x32-10 blocks (known-answer tests): ctr [n][4], key [n][2] -> out [n][4]. */
int hmcgpu_philox(hmcgpu_ctx* ctx, int64_t n, const uint32_t* ctr, const uint32_t* key, uint32_t* out);
/* Same with the round count of the stream: 10 = parameter draws, 7 = the backward sampler's state uniforms. */
int hmcgpu_philox_rounds(hmcgpu_ctx* ctx, int32_t rounds, int64_t n, const uint32_t* ctr, const uint32_t* key, uint32_t* out);

#ifdef __cplusplus
}
#endif
#endif
