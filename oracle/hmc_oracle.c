/*
 * hmc_oracle.c — CPU fp64 restatement of the reference's Gibbs/FFBS path.  TEST INFRASTRUCTURE ONLY
 * (see hmc_oracle.h).  Each function cites the reference lines (under /root/reference) it follows.
 * Build: see oracle/Makefile (-O2 -ffp-contract=off: no FMA contraction, so fp64 results are
 * reproducible operation by operation and comparable bit-for-bit with the CUDA fp64 exact path).
 */
#include "hmc_oracle.h"
#include <math.h>
#include <stdlib.h>
#include <string.h>
#include <pthread.h>
#include <unistd.h>

#define MAXK 64
static const double INVSQRT2PI = 0.3989422804014327; /* StatsFuns.invsqrt2π */
static const double TWO_PI = 6.283185307179586;
static const double EPS64 = 2.220446049250313e-16;   /* Julia eps() */

/* ---------------------------------------------------------------- RNG spec (DESIGN.md §RNG) */
void orc_philox4x32(int rounds, const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) {
    uint32_t c0 = ctr[0], c1 = ctr[1], c2 = ctr[2], c3 = ctr[3], k0 = key[0], k1 = key[1];
    for (int round = 0; round < rounds; ++round) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

void orc_philox4x32_10(const uint32_t ctr[4], const uint32_t key[2], uint32_t out[4]) { orc_philox4x32(10, ctr, key, out); }

/* parameter draws: 10 rounds; the STATES stream (one uniform per time step and sweep): Philox4x32-7 */
static void orc_block(uint64_t seed, uint32_t chain, uint32_t sweep, uint32_t purpose, uint32_t block, uint32_t w[4]) {
    uint32_t ctr[4] = {block, purpose, sweep, chain};
    uint32_t key[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
    orc_philox4x32((purpose >> 16) == ORC_KIND_STATES ? ORC_STATE_ROUNDS : 10, ctr, key, w);
}

double orc_u01(uint32_t w) { return ((double)w + 0.5) * 2.3283064365386963e-10; /* 2^-32 */ }

void orc_normal_pair(const uint32_t w[4], double* z0, double* z1) {
    double r = sqrt(-2.0 * log(orc_u01(w[0])));
    double th = TWO_PI * orc_u01(w[1]);
    if (z0) *z0 = r * cos(th);
    if (z1) *z1 = r * sin(th);
}

/* *m = min(*m, d): the margin outputs of orc_result (NULL: not tracked) */
static void shrink(double* m, double d) { if (m && d < *m) *m = d; }

/* Marsaglia & Tsang (2000) for shape >= 1; shape < 1 boosted by U^(1/shape).  Attempt k uses block k:
 * words 0,1 -> normal (cos branch), word 2 -> acceptance uniform, word 3 -> boost uniform.
 * margin (may be NULL): lowered to the distance of every comparison made from its threshold — |v| for v <= 0, |u - s| for the
 * squeeze u < s, and |log u - r| / max(1, d) for the log test (its rounding error in a lower precision grows with d). */
static double gamma_m(double shape, uint64_t seed, uint32_t chain, uint32_t sweep, uint32_t purpose, double* margin) {
    double a = shape < 1.0 ? shape + 1.0 : shape;
    double d = a - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
    for (uint32_t k = 0;; ++k) {
        uint32_t w[4];
        orc_block(seed, chain, sweep, purpose, k, w);
        double z; orc_normal_pair(w, &z, NULL);
        double v = 1.0 + c * z;
        shrink(margin, fabs(v));
        if (v <= 0.0) continue;
        v = v * v * v;
        double u = orc_u01(w[2]);
        double z2 = z * z;
        double sq = 1.0 - 0.0331 * z2 * z2;
        shrink(margin, fabs(u - sq));
        int accept = u < sq;
        if (!accept) {
            double lu = log(u), r = 0.5 * z2 + d * (1.0 - v + log(v));
            shrink(margin, fabs(lu - r) / (d > 1.0 ? d : 1.0));
            accept = lu < r;
        }
        if (accept) {
            double g = d * v;
            if (shape < 1.0) g *= pow(orc_u01(w[3]), 1.0 / shape);
            return g;
        }
        if (k > 1000000u) return d; /* unreachable in practice */
    }
}

double orc_gamma(double shape, uint64_t seed, uint32_t chain, uint32_t sweep, uint32_t purpose) {
    return gamma_m(shape, seed, chain, sweep, purpose, NULL);
}

/* ---------------------------------------------------------------- initial state and priors */
static int cmp_double(const void* a, const void* b) {
    double x = *(const double*)a, y = *(const double*)b;
    return (x > y) - (x < y);
}

static double normpdf(double mu, double sd, double x) { /* StatsFuns 0.9 normpdf(μ,σ,x) */
    double z = (x - mu) / sd;
    return exp(-(z * z) / 2.0) * INVSQRT2PI / sd;
}

/* src/Hmc.jl:161-195 */
void orc_make_params(const double* y, int N, int K, int64_t* X, double* mu0, double* sd0) {
    double* tmp = (double*)malloc(sizeof(double) * (size_t)N);
    memcpy(tmp, y, sizeof(double) * (size_t)N);
    qsort(tmp, (size_t)N, sizeof(double), cmp_double);
    double med = (N & 1) ? tmp[N / 2] : 0.5 * (tmp[N / 2 - 1] + tmp[N / 2]);
    double R = tmp[N - 1] - tmp[0];
    free(tmp);
    double mean = 0.0;
    for (int i = 0; i < N; ++i) mean += y[i];
    mean /= N;
    double ss = 0.0;
    for (int i = 0; i < N; ++i) ss += (y[i] - mean) * (y[i] - mean);
    double sd = sqrt(ss / (N - 1));                    /* Statistics.std (corrected) :177 */
    double mu[MAXK];
    double lo = med - 0.25 * R, hi = med + 0.25 * R;   /* :176 */
    for (int k = 0; k < K; ++k) mu[k] = (K > 1) ? lo + (hi - lo) * ((double)k / (double)(K - 1)) : med;
    /* :185-187 findmax of pdf(Normal(mu_k, sd), y_i) -> FIRST maximum.  All states share sd, so the pdf is a decreasing
     * function of |y - mu_k| and the first maximum of the pdf is the first minimum of that distance.  Comparing distances
     * instead of exp(-z^2/2) makes the rule independent of the exp implementation and of the last bits of sd: with an odd
     * window length and an even K the median observation lies exactly between two grid points (a tie in exact arithmetic,
     * decided by the last bit of the grid arithmetic above), and libm / CUDA / Julia exponentials round such near-ties
     * differently.  Exact ties go to the lower state, as findmax does. */
    for (int i = 0; i < N; ++i) {
        int best = 0; double bv = fabs(y[i] - mu[0]);
        for (int k = 1; k < K; ++k) {
            double v = fabs(y[i] - mu[k]);
            if (v < bv) { bv = v; best = k; }
        }
        X[i] = best + 1;
    }
    if (mu0) memcpy(mu0, mu, sizeof(double) * (size_t)K);
    if (sd0) *sd0 = sd;
}

/* src/Hmc.jl:132-142 */
void orc_hyper_defaults(const double* y, int N, int K, double* xi, double* alpha, double* nu) {
    double mean = 0.0;
    for (int i = 0; i < N; ++i) mean += y[i];
    mean /= N;
    for (int k = 0; k < K; ++k) { xi[k] = mean; alpha[k] = 1.0; nu[k] = 1.0; }
}

/* ---------------------------------------------------------------- deterministic pieces */
/* src/Hmc.jl:371-440.  Loop order `for s, r` (s outer) as in the reference; pdf evaluated once per
 * state (a pure function of (s,t); the reference re-evaluates it K times, same value). */
int orc_forward(const double* y, int N, int K, const uint8_t* is_signal, double kappa,
                const double* A, const double* mu, const double* sigma2, const double* rho,
                double* Pf, double* pif, double* totals, double* loglik) {
    double sdo[MAXK], sds[MAXK], e[MAXK], P[MAXK * MAXK];
    int events = 0;
    double ll = 0.0;
    for (int s = 0; s < K; ++s) { sdo[s] = sqrt(sigma2[s]); sds[s] = (1.0 + kappa) * sqrt(sigma2[s]); } /* :380-383 */
    for (int t = 0; t < N; ++t) {
        const double* prev = (t == 0) ? rho : pif + (size_t)(t - 1) * K;   /* :390 / :415 */
        int sig = is_signal && is_signal[t];
        for (int s = 0; s < K; ++s) e[s] = normpdf(mu[s], sig ? sds[s] : sdo[s], y[t]);
        double total = 0.0;
        for (int s = 0; s < K; ++s)
            for (int r = 0; r < K; ++r) {
                double v = prev[r] * A[r * K + s] * e[s];
                P[r * K + s] = v;
                total += v;
            }
        double* pi = pif + (size_t)t * K;
        for (int s = 0; s < K; ++s) pi[s] = 0.0;
        for (int s = 0; s < K; ++s)
            for (int r = 0; r < K; ++r) {
                P[r * K + s] /= total;                                      /* :401 / :430 */
                pi[s] += P[r * K + s];
            }
        if (Pf) memcpy(Pf + (size_t)t * K * K, P, sizeof(double) * (size_t)(K * K));
        if (totals) totals[t] = total;
        ll += log(total);
        if (!(total > 0.0) || !isfinite(total)) ++events;                   /* :435 @warn */
    }
    if (loglik) *loglik = ll;
    return events;
}

/* src/Hmc.jl:442-457 */
void orc_backward(int N, int K, const double* Pf, const double* pif, double* Pb, double* pib) {
    size_t KK = (size_t)K * K;
    memset(pib, 0, sizeof(double) * (size_t)N * K);
    memcpy(Pb + (size_t)(N - 1) * KK, Pf + (size_t)(N - 1) * KK, sizeof(double) * KK);
    memcpy(pib + (size_t)(N - 1) * K, pif + (size_t)(N - 1) * K, sizeof(double) * (size_t)K);
    for (int t = N - 2; t >= 0; --t) {
        for (int s = 0; s < K; ++s)
            for (int r = 0; r < K; ++r) pib[(size_t)t * K + r] += Pb[(size_t)(t + 1) * KK + r * K + s];
        for (int s = 0; s < K; ++s)
            for (int r = 0; r < K; ++r)
                Pb[(size_t)t * KK + r * K + s] =
                    Pf[(size_t)t * KK + r * K + s] * pib[(size_t)t * K + s] / pif[(size_t)t * K + s];
    }
}

/* Same marginals without Pf: pib[t,r] = pif[t,r] * sum_s A[r,s] * pib[t+1,s] / pred[t+1,s],
 * pred[t+1,s] = sum_r pif[t,r] A[r,s]   (algebraically equal to the recursion above). */
void orc_backward_pif(int N, int K, const double* A, const double* pif, double* pib) {
    double w[MAXK];
    memcpy(pib + (size_t)(N - 1) * K, pif + (size_t)(N - 1) * K, sizeof(double) * (size_t)K);
    for (int t = N - 2; t >= 0; --t) {
        const double* f = pif + (size_t)t * K;
        const double* nb = pib + (size_t)(t + 1) * K;
        for (int s = 0; s < K; ++s) {
            double p = 0.0;
            for (int r = 0; r < K; ++r) p += f[r] * A[r * K + s];
            w[s] = (p > 0.0) ? nb[s] / p : 0.0;
        }
        for (int r = 0; r < K; ++r) {
            double acc = 0.0;
            for (int s = 0; s < K; ++s) acc += A[r * K + s] * w[s];
            pib[(size_t)t * K + r] = f[r] * acc;
        }
    }
}

/* Distributions 0.21 rand(Categorical(p)): i=1; c=p[1]; while c < u && i < n: c += p[i+=1]  (SURVEY §8c) */
static int64_t categorical(const double* p, int K, double u) {
    int i = 0;
    double c = p[0];
    while (c < u && i < K - 1) { ++i; c += p[i]; }
    return i + 1;
}

/* distance of u from the nearest of the K - 1 cumulative boundaries categorical() may compare it with */
static double categorical_margin(const double* p, int K, double u) {
    double c = 0.0, m = INFINITY;
    for (int j = 0; j < K - 1; ++j) { c += p[j]; if (fabs(u - c) < m) m = fabs(u - c); }
    return m;
}

/* src/Hmc.jl:459-484 */
/* margin (may be NULL): lowered to the categorical_margin of every draw */
static void sample_states_m(int N, int K, const double* Pf, const double* pif, const double* A,
                            const double* piN, const double* u, int form, int64_t* X, double* margin) {
    double p[MAXK];
    X[N - 1] = categorical(piN, K, u[N - 1]);                   /* :464 */
    if (margin) shrink(margin, categorical_margin(piN, K, u[N - 1]));
    for (int k = N - 2; k >= 0; --k) {
        int x = (int)X[k + 1] - 1;
        double total = 0.0;
        for (int r = 0; r < K; ++r) {
            p[r] = (form == 0) ? Pf[((size_t)(k + 1) * K + r) * K + x]      /* :469 */
                               : pif[(size_t)k * K + r] * A[r * K + x];
            total += p[r];
        }
        /* :472 tests total = sum_r Pf[k+1,r,x] = pif[k+1,x]; the pif form applies the same threshold to pif[k+1,x] (SURVEY Q5) */
        double gate = (form == 0) ? total : pif[(size_t)(k + 1) * K + x];
        if (gate > EPS64 && total > 0.0) for (int j = 0; j < K; ++j) p[j] /= total;
        else for (int j = 0; j < K; ++j) p[j] = 1.0 / K;
        X[k] = categorical(p, K, u[k]);
        if (margin) shrink(margin, categorical_margin(p, K, u[k]));
    }
}

void orc_sample_states(int N, int K, const double* Pf, const double* pif, const double* A,
                       const double* piN, const double* u, int form, int64_t* X) {
    sample_states_m(N, K, Pf, pif, A, piN, u, form, X, NULL);
}

static void matmul(int K, const double* a, const double* b, double* c) {
    for (int i = 0; i < K; ++i)
        for (int j = 0; j < K; ++j) {
            double acc = 0.0;
            for (int l = 0; l < K; ++l) acc += a[i * K + l] * b[l * K + j];
            c[i * K + j] = acc;
        }
}

/* src/Hmc.jl:658-667; A^h by repeated squaring like Julia's power_by_squaring */
void orc_forecast(int K, const double* mu, const double* A, const double* pib, int h, double yreal,
                  double* fc, double* err) {
    double base[MAXK * MAXK], acc[MAXK * MAXK], tmp[MAXK * MAXK];
    size_t KK = (size_t)K * K;
    memcpy(base, A, sizeof(double) * KK);
    int have = 0;
    for (int e = h; e > 0; e >>= 1) {
        if (e & 1) {
            if (!have) { memcpy(acc, base, sizeof(double) * KK); have = 1; }
            else { matmul(K, acc, base, tmp); memcpy(acc, tmp, sizeof(double) * KK); }
        }
        if (e > 1) { matmul(K, base, base, tmp); memcpy(base, tmp, sizeof(double) * KK); }
    }
    if (!have) { memset(acc, 0, sizeof(double) * KK); for (int i = 0; i < K; ++i) acc[i * K + i] = 1.0; }
    double f = 0.0;
    for (int s = 0; s < K; ++s) {
        double s1 = 0.0;
        for (int r = 0; r < K; ++r) s1 += pib[r] * acc[r * K + s];
        f += s1 * mu[s];
    }
    *fc = f;
    *err = f - yreal;
}

/* src/Hmc.jl:302-335 (sigma2, mu), :350-356 (rho), :358-369 (A) given the sufficient statistics */
/* margin (may be NULL): lowered by every gamma draw (gamma_m) */
static void draw_params_m(int K, const int64_t* Ni, const int64_t* Mi, const double* S, const double* Sm,
                          const double* S2, const double* Sm2, const int64_t* trans,
                          const double* xi, const double* alpha, const double* nu, const double* beta, double kappa,
                          uint64_t seed, uint32_t chain, uint32_t sweep,
                          double* sigma2, double* mu, double* rho, double* A, double* margin) {
    double Neff[MAXK], g[MAXK];
    for (int i = 0; i < K; ++i) {
        double mi = Mi ? (double)Mi[i] : 0.0, sm = Sm ? Sm[i] : 0.0, sm2 = Sm2 ? Sm2[i] : 0.0;
        double ni = (double)Ni[i];
        double totalbar = (ni + mi > 0.0) ? (S[i] + sm) / (ni + mi) : 0.0;       /* :282-288 */
        double Meff = mi / (1.0 + kappa);                                         /* :302 */
        Neff[i] = ni + Meff;                                                      /* :303 */
        double a = alpha[i] + 0.5 * ni + 0.5 * mi;                                /* :313 */
        double dev = totalbar - xi[i];
        double b = beta[i] + 0.5 * S2[i] + (0.5 / (1.0 + kappa)) * sm2
                 + 0.5 * Neff[i] * nu[i] / (Neff[i] + nu[i]) * (dev * dev);       /* :314 */
        if (a > 0.0 && b > 0.0) {
            double gm = gamma_m(a, seed, chain, sweep, (ORC_KIND_SIGMA << 16) | (uint32_t)i, margin);
            sigma2[i] = b / gm;                                                   /* :320 InverseGamma(a,b) */
        } /* else: reference's catch keeps the old value (:321-329) */
    }
    for (int i = 0; i < K; ++i) {
        double sm = Sm ? Sm[i] : 0.0;
        double m = (S[i] + sm + nu[i] * xi[i]) / (Neff[i] + nu[i]);               /* :331 */
        double s = sqrt(sigma2[i] / (Neff[i] + nu[i]));                           /* :332 */
        uint32_t w[4];
        orc_block(seed, chain, sweep, (ORC_KIND_MU << 16), (uint32_t)(i >> 1), w);
        double z0, z1;
        orc_normal_pair(w, &z0, &z1);
        /* state 2j uses the (w0,w1) cos branch of block j, state 2j+1 the (w2,w3) cos branch */
        if (i & 1) { uint32_t w2[4] = {w[2], w[3], 0, 0}; orc_normal_pair(w2, &z0, NULL); }
        mu[i] = m + s * z0;                                                       /* :334 */
    }
    double tot = 0.0;                                                              /* :354-355 Dirichlet(1..1) */
    for (int i = 0; i < K; ++i) { g[i] = gamma_m(1.0, seed, chain, sweep, (ORC_KIND_RHO << 16) | (uint32_t)i, margin); tot += g[i]; }
    for (int i = 0; i < K; ++i) rho[i] = g[i] / tot;
    for (int i = 0; i < K; ++i) {                                                  /* :366-368 */
        tot = 0.0;
        for (int j = 0; j < K; ++j) {
            g[j] = gamma_m((double)trans[i * K + j], seed, chain, sweep, (ORC_KIND_A << 16) | (uint32_t)(i * K + j), margin);
            tot += g[j];
        }
        for (int j = 0; j < K; ++j) A[i * K + j] = g[j] / tot;
    }
}

void orc_draw_params(int K, const int64_t* Ni, const int64_t* Mi, const double* S, const double* Sm,
                     const double* S2, const double* Sm2, const int64_t* trans,
                     const double* xi, const double* alpha, const double* nu, const double* beta, double kappa,
                     uint64_t seed, uint32_t chain, uint32_t sweep,
                     double* sigma2, double* mu, double* rho, double* A) {
    draw_params_m(K, Ni, Mi, S, Sm, S2, Sm2, trans, xi, alpha, nu, beta, kappa, seed, chain, sweep, sigma2, mu, rho, A, NULL);
}

/* ---------------------------------------------------------------- the sampler */
/* src/Hmc.jl:486-515 gibbssweep!, :517-562 gibbssample!, :850-865 estimatemodel */
int orc_gibbs(const orc_problem* p, orc_result* res) {
    const int N = p->N, K = p->K;
    const size_t KK = (size_t)K * K;
    if (K < 1 || K > MAXK || N < 2) return -1;
    double xi[MAXK], alpha[MAXK], nu[MAXK], beta[MAXK], beta_after[MAXK];
    orc_hyper_defaults(p->y, N, K, xi, alpha, nu);
    for (int k = 0; k < K; ++k) {
        if (p->xi) xi[k] = p->xi[k];
        if (p->alpha) alpha[k] = p->alpha[k];
        if (p->nu) nu[k] = p->nu[k];
        beta[k] = p->beta0 ? p->beta0[k] : 1.0;          /* makeParams β=1 (:179) */
        beta_after[k] = p->beta ? p->beta[k] : 2.0;      /* update_β! (:347) */
    }
    int64_t* X = (int64_t*)malloc(sizeof(int64_t) * (size_t)N);
    if (p->X0) memcpy(X, p->X0, sizeof(int64_t) * (size_t)N);
    else orc_make_params(p->y, N, K, X, NULL, NULL);
    double* Pf = (double*)malloc(sizeof(double) * (size_t)N * KK);
    double* Pb = (double*)malloc(sizeof(double) * (size_t)N * KK);
    double* pif = (double*)malloc(sizeof(double) * (size_t)N * K);
    double* pib = (double*)malloc(sizeof(double) * (size_t)N * K);
    double* u = (double*)malloc(sizeof(double) * (size_t)N);
    double mu[MAXK], sigma2[MAXK], rho[MAXK], A[MAXK * MAXK], Atmp[MAXK * MAXK], tmpv[MAXK], piN[MAXK];
    for (int k = 0; k < K; ++k) { mu[k] = 0.0; sigma2[k] = 1.0; }
    if (res->pib_mean) memset(res->pib_mean, 0, sizeof(double) * (size_t)N * K);
    res->n_events = 0;
    const int want_pib = res->pib_mean || res->pib_full;
    const int64_t total_sweeps = p->burnin + p->nrun;
    for (int64_t sw = 0; sw < total_sweeps; ++sw) {
        const uint32_t sweep = (uint32_t)sw;
        /* --- update_μσ! statistics (:243-300), two passes like the reference */
        int64_t Ni[MAXK], Mi[MAXK], trans[MAXK * MAXK];
        double S[MAXK], Sm[MAXK], S2[MAXK], Sm2[MAXK], ybar[MAXK], sbar[MAXK];
        for (int k = 0; k < K; ++k) { Ni[k] = Mi[k] = 0; S[k] = Sm[k] = S2[k] = Sm2[k] = 0.0; }
        for (int t = 0; t < N; ++t) {
            int i = (int)X[t] - 1;
            if (p->is_signal && p->is_signal[t]) { Mi[i] += 1; Sm[i] += p->y[t]; }
            else { Ni[i] += 1; S[i] += p->y[t]; }
        }
        for (int k = 0; k < K; ++k) {
            ybar[k] = Ni[k] > 0 ? S[k] / (double)Ni[k] : 0.0;
            sbar[k] = Mi[k] > 0 ? Sm[k] / (double)Mi[k] : 0.0;
        }
        for (int t = 0; t < N; ++t) {
            int i = (int)X[t] - 1;
            if (p->is_signal && p->is_signal[t]) { double d = p->y[t] - sbar[i]; Sm2[i] += d * d; }
            else { double d = p->y[t] - ybar[i]; S2[i] += d * d; }
        }
        /* --- update_A! counts (:362-365) */
        for (size_t j = 0; j < KK; ++j) trans[j] = 1;
        for (int t = 0; t + 1 < N; ++t) trans[((int)X[t] - 1) * K + ((int)X[t + 1] - 1)] += 1;
        /* --- draws: σ², μ (β of this sweep), then β .= 2 (:347), ρ, A */
        double* gmargin = res->gamma_margin ? res->gamma_margin + sw : NULL;
        if (gmargin) *gmargin = INFINITY;
        draw_params_m(K, Ni, Mi, S, Sm, S2, Sm2, trans, xi, alpha, nu, beta, p->kappa,
                      p->seed, p->chain, sweep, sigma2, mu, rho, A, gmargin);
        memcpy(beta, beta_after, sizeof(double) * (size_t)K);
        /* --- forward / backward (:498-499) */
        double ll;
        res->n_events += orc_forward(p->y, N, K, p->is_signal, p->kappa, A, mu, sigma2, rho, Pf, pif, NULL, &ll);
        if (want_pib) orc_backward(N, K, Pf, pif, Pb, pib);
        else memcpy(pib + (size_t)(N - 1) * K, pif + (size_t)(N - 1) * K, sizeof(double) * (size_t)K);
        /* --- relabel (:501-513): stable sortperm(μ) */
        int order[MAXK];
        for (int k = 0; k < K; ++k) order[k] = k;
        for (int i = 1; i < K; ++i) {
            int o = order[i], j = i - 1;
            while (j >= 0 && mu[order[j]] > mu[o]) { order[j + 1] = order[j]; --j; }
            order[j + 1] = o;
        }
        for (int k = 0; k < K; ++k) tmpv[k] = mu[order[k]];
        memcpy(mu, tmpv, sizeof(double) * (size_t)K);
        for (int k = 0; k < K; ++k) tmpv[k] = sigma2[order[k]];
        memcpy(sigma2, tmpv, sizeof(double) * (size_t)K);
        for (int k = 0; k < K; ++k) tmpv[k] = beta[order[k]];
        memcpy(beta, tmpv, sizeof(double) * (size_t)K);
        for (int k = 0; k < K; ++k) tmpv[k] = rho[order[k]];
        memcpy(rho, tmpv, sizeof(double) * (size_t)K);
        memcpy(Atmp, A, sizeof(double) * KK);
        for (int i = 0; i < K; ++i)
            for (int j = 0; j < K; ++j) A[i * K + j] = Atmp[order[i] * K + order[j]];
        /* πf, πb columns permuted; Pf, Pb, X are NOT (quirk Q1).  Only row N of πf is read again. */
        const double* fN = pif + (size_t)(N - 1) * K;
        for (int k = 0; k < K; ++k) piN[k] = (p->flags & ORC_FLAG_REF_Q1) ? fN[order[k]] : fN[k];
        if (want_pib)
            for (int t = 0; t < N; ++t) {
                double* row = pib + (size_t)t * K;
                for (int k = 0; k < K; ++k) tmpv[k] = row[order[k]];
                memcpy(row, tmpv, sizeof(double) * (size_t)K);
            }
        else {
            double* row = pib + (size_t)(N - 1) * K;
            for (int k = 0; k < K; ++k) tmpv[k] = row[order[k]];
            memcpy(row, tmpv, sizeof(double) * (size_t)K);
        }
        /* --- update_X! (:514): one uniform per t from the STATES stream, indexed in consumption order:
         *     the i-th uniform drawn (i = 0 for X[N], i = N-1-t for X[t]) is word i&3 of block i>>2 */
        for (int i = 0; i < N; i += 4) {
            uint32_t w[4];
            orc_block(p->seed, p->chain, sweep, (ORC_KIND_STATES << 16), (uint32_t)(i >> 2), w);
            for (int j = 0; j < 4 && i + j < N; ++j) u[N - 1 - (i + j)] = orc_u01(w[j]);
        }
        /* chain-label A for the pif form (Atmp is the un-permuted matrix) */
        double* smargin = res->state_margin ? res->state_margin + sw : NULL;
        if (smargin) *smargin = INFINITY;
        sample_states_m(N, K, Pf, pif, Atmp, piN, u, (p->flags & ORC_FLAG_PIF_FORM) ? 1 : 0, X, smargin);
        /* --- save (:554-560) + forecasts (:858-862) */
        if (sw >= p->burnin) {
            size_t d = (size_t)(sw - p->burnin);
            if (res->mu) memcpy(res->mu + d * K, mu, sizeof(double) * (size_t)K);
            if (res->sigma2) memcpy(res->sigma2 + d * K, sigma2, sizeof(double) * (size_t)K);
            if (res->A) memcpy(res->A + d * KK, A, sizeof(double) * KK);
            if (res->pi_end) memcpy(res->pi_end + d * K, pib + (size_t)(N - 1) * K, sizeof(double) * (size_t)K);
            if (res->loglik) res->loglik[d] = ll;
            if (res->forecasts)
                for (int j = 0; j < p->n_h; ++j)
                    orc_forecast(K, mu, A, pib + (size_t)(N - 1) * K, p->horizons[j],
                                 p->y_future ? p->y_future[j] : NAN,
                                 res->forecasts + d * 2 * p->n_h + 2 * j, res->forecasts + d * 2 * p->n_h + 2 * j + 1);
            if (res->pib_full) memcpy(res->pib_full + d * (size_t)N * K, pib, sizeof(double) * (size_t)N * K);
            if (res->pib_mean) for (size_t j = 0; j < (size_t)N * K; ++j) res->pib_mean[j] += pib[j];
        }
    }
    if (res->pib_mean && p->nrun > 0) for (size_t j = 0; j < (size_t)N * K; ++j) res->pib_mean[j] /= (double)p->nrun;
    if (res->X_final) memcpy(res->X_final, X, sizeof(int64_t) * (size_t)N);
    free(X); free(Pf); free(Pb); free(pif); free(pib); free(u);
    return 0;
}

typedef struct { const orc_problem* p; orc_result* r; int n; int next; pthread_mutex_t mu; } orc_pool;

static void* orc_worker(void* arg) {
    orc_pool* pool = (orc_pool*)arg;
    for (;;) {
        pthread_mutex_lock(&pool->mu);
        int i = pool->next++;
        pthread_mutex_unlock(&pool->mu);
        if (i >= pool->n) break;
        orc_gibbs(&pool->p[i], &pool->r[i]);
    }
    return NULL;
}

/* pthread pool over independent chains; n_threads <= 0 -> all online cores */
int orc_gibbs_batch(const orc_problem* p, orc_result* r, int n, int n_threads) {
    if (n_threads <= 0) n_threads = (int)sysconf(_SC_NPROCESSORS_ONLN);
    if (n_threads > n) n_threads = n;
    if (n_threads < 1) n_threads = 1;
    orc_pool pool = {p, r, n, 0, PTHREAD_MUTEX_INITIALIZER};
    pthread_t* th = (pthread_t*)malloc(sizeof(pthread_t) * (size_t)n_threads);
    for (int t = 0; t < n_threads; ++t) pthread_create(&th[t], NULL, orc_worker, &pool);
    for (int t = 0; t < n_threads; ++t) pthread_join(th[t], NULL);
    free(th);
    return n_threads;
}
