/*
 * hmc_oracle.h — CPU fp64 restatement of the Gibbs/FFBS hot path of joe5saia/Hmc.jl.
 *
 * TEST INFRASTRUCTURE ONLY.  Nothing under oracle/ is part of the product: only tests/,
 * __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs may load it,
 * and only as the checker / reported CPU baseline.  The product path (hmc.jl_b200/) never
 * links, imports or falls back to this code.
 *
 * Parity status: deterministic pieces (filter, smoother, forecast) have NO known-answer vectors
 * in the reference (SURVEY.md §8c) — they are pinned by this restatement plus an independent
 * numpy/scipy log-space check (tests/test_oracle.py), and the filter + forecast also by the
 * reference's published in-sample table (data/output/official_insample/forecats_insample.csv =
 * posterior means of the filtered probabilities on 576 dates, tests/golden/official_insample.json).  Random draws are "parity unpinned" at the
 * bit level (Julia's MersenneTwister + Distributions.jl 0.21.8 samplers are not vendored and Julia
 * is absent); the full sampler is pinned distributionally against the reference's own golden
 * posterior summaries (data/output/official/<var>_summary.csv, copied to tests/golden/), the signal
 * tier (mask, kappa-weighted statistics, quirk Q3, HyperParams(opt) priors) against the reference's
 * noisy-signal outputs (data/output/signals_official_noise_<kappa>_allsignal/<var>_dispersion.csv,
 * tests/golden/signals_allsignal_subset.json), and against the reference's only test
 * (test/runtests.jl:56-57).
 *
 * Array conventions: row-major C arrays, 0-based in storage, states reported 1-based in X
 * exactly as the reference stores them.  A[r*K+s] = P(X_t=s | X_{t-1}=r); sigma2 holds variances.
 * pif[t*K+s], Pf[(t*K+r)*K+s].
 *
 * Random numbers: a counter-based Philox4x32 stream specification (10 rounds; 7 for the STATES stream) shared with the CUDA
 * product (documented in DESIGN.md §RNG).  The oracle has its own independent implementation.
 */
#ifndef HMC_ORACLE_H
#define HMC_ORACLE_H
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* flags */
#define ORC_FLAG_REF_Q1 1u      /* reproduce src/Hmc.jl:512-514: X[N] drawn from relabelled pif[N,:] */
#define ORC_FLAG_PIF_FORM 2u    /* backward sampler uses pif[k,r]*A[r,x] instead of the Pf column (SURVEY §3.2-8) */

/* purposes of a Philox block: counter = {block, purpose, sweep, chain}, key = seed */
#define ORC_KIND_STATES 0u
#define ORC_KIND_MU     1u
#define ORC_KIND_SIGMA  2u
#define ORC_KIND_RHO    3u
#define ORC_KIND_A      4u

void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
void orc_philox4x32(int rounds, const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]);
#define ORC_STATE_ROUNDS 7   /* rounds of the STATES stream (backward-sampler uniforms) */
double orc_u01(uint32_t w);
/* one standard normal pair from a block's words 0..3 (Box-Muller: words 0,1 -> cos branch z0; sin branch z1) */
void orc_normal_pair(const uint32_t w[4], double* z0, double* z1);
/* Marsaglia-Tsang gamma(shape, scale 1); purpose identifies the draw, attempts index the block */
double orc_gamma(double shape, uint64_t seed, uint32_t chain, uint32_t sweep, uint32_t purpose);

/* src/Hmc.jl:161-195 makeParams: initial X (1-based), returns mu0/sd0 if non-NULL */
void orc_make_params(const double* y, int N, int K, int64_t* X, double* mu0, double* sd0);
/* src/Hmc.jl:132-142 HyperParams(Y,D): xi=mean(Y), alpha=nu=1 */
void orc_hyper_defaults(const double* y, int N, int K, double* xi, double* alpha, double* nu);

/* src/Hmc.jl:371-440 forwardupdate_P!.  Pf may be NULL.  totals (N) and loglik optional. */
int orc_forward(const double* y, int N, int K, const uint8_t* is_signal, double kappa,
                const double* A, const double* mu, const double* sigma2, const double* rho,
                double* Pf, double* pif, double* totals, double* loglik);
/* src/Hmc.jl:442-457 backwardupdate_P!  (needs Pf) */
void orc_backward(int N, int K, const double* Pf, const double* pif, double* Pb, double* pib);
/* same smoothed marginals from pif and A only (the form the CUDA path uses) */
void orc_backward_pif(int N, int K, const double* A, const double* pif, double* pib);
/* src/Hmc.jl:459-484 update_X! with injected uniforms u[t] (u[N-1] used first).
 * form 0: literal Pf column; form 1: pif[k,r]*A[r,x].  piN = the K probabilities X[N] is drawn from. */
void orc_sample_states(int N, int K, const double* Pf, const double* pif, const double* A,
                       const double* piN, const double* u, int form, int64_t* X);
/* src/Hmc.jl:658-667 forecast: pib' * A^h * mu, and error vs yreal */
void orc_forecast(int K, const double* mu, const double* A, const double* pib, int h, double yreal,
                  double* fc, double* err);
/* conjugate draws given sufficient statistics (src/Hmc.jl:302-335, 350-369), Philox spec streams */
void orc_draw_params(int K, const int64_t* Ni, const int64_t* Mi, const double* S, const double* Sm,
                     const double* S2, const double* Sm2, const int64_t* trans /*K*K counts incl. the +1 prior*/,
                     const double* xi, const double* alpha, const double* nu, const double* beta, double kappa,
                     uint64_t seed, uint32_t chain, uint32_t sweep,
                     double* sigma2, double* mu, double* rho, double* A);

typedef struct {
    const double* y;          /* window observations Y = rawdata[sampleRange] (length N) */
    int32_t N, K;
    const uint8_t* is_signal; /* NULL = all observations (official config) */
    const double *xi, *alpha, *nu, *beta0, *beta; /* NULL -> reference defaults */
    double kappa;
    const int64_t* X0;        /* NULL -> makeParams rule */
    int64_t burnin, nrun;
    uint64_t seed; uint32_t chain; uint32_t flags;
    const int32_t* horizons; int32_t n_h;
    const double* y_future;   /* y_future[j] = rawdata[endIndex + horizons[j]] (may be NaN) */
} orc_problem;

typedef struct {              /* any pointer may be NULL; all [draw]-major row-major */
    double* mu;        /* nrun*K   */
    double* sigma2;    /* nrun*K   */
    double* A;         /* nrun*K*K */
    double* pi_end;    /* nrun*K  = pib[N,:] = pif[N,:] relabelled */
    double* forecasts; /* nrun*2*n_h  interleaved forecast,error (src/Hmc.jl:858-862) */
    double* loglik;    /* nrun */
    double* pib_mean;  /* N*K posterior mean of smoothed probabilities (relabelled per draw) */
    double* pib_full;  /* nrun*N*K */
    int64_t* X_final;  /* N */
    int64_t n_events;  /* zero-normaliser / non-finite events */
    /* Per sweep (burnin + nrun entries, indexed by sweep): how far the sweep's discrete decisions were from flipping.  A chain
     * run in lower precision on the same streams can leave this chain only through such a decision.
     * state_margin: min over t (X[N] included) of |u_t - nearest cumulative boundary| of the normalised p it was compared with.
     * gamma_margin: min over the sweep's gamma draws of the distance of each comparison from its threshold (see gamma_m). */
    double* state_margin;
    double* gamma_margin;
} orc_result;

/* src/Hmc.jl:517-562 gibbssample! + :850-865 estimatemodel glue, one chain */
int orc_gibbs(const orc_problem* p, orc_result* r);

/* pthread batch of independent chains (the CPU baseline): problems[i] -> results[i]; returns threads used */
int orc_gibbs_batch(const orc_problem* p, orc_result* r, int n, int n_threads);

#ifdef __cplusplus
}
#endif
#endif
