// lane_draws.cuh — the per-state conjugate posterior of draw_params (hmm_device.cuh, src/Hmc.jl:302-335) that the scan,
// segment and lane-per-state kernels share, and the chain state the scan and segment kernels keep between launches.  The
// expressions are draw_params' in the same order, so the compiler contracts them into the same FMAs and every kernel draws
// the same bits as the thread-per-chain kernel.
#pragma once
#include "gibbs_kernel.cuh"     // GibbsArgs; hmm_device.cuh (Hyper, SigStats), rng.cuh

namespace hmc {

// shape a and rate b of sigma2's inverse gamma (:313-314); Neff, and the sums over observations and signals that give the
// normal of mu (:331-332)
template <typename R> struct StatePosterior {
    R a, b, neff, sumd, ntot;
    __device__ __forceinline__ R mean(R c, R nu, R xi) const { return (sumd + ntot * c + nu * xi) / (neff + nu); }  // sumd: about c
    __device__ __forceinline__ R sd(R sig2, R nu) const { return M<R>::sqrt(sig2 / (neff + nu)); }
};

// one state from its statistics about the shift c (Sd = sum(y-c), Qd = sum((y-c)^2) over its cnt observations); with SIG
// also from those of its signals (m of them, Sm, Qm) at the relative precision k1 = 1/(1+kappa)
template <typename R, bool SIG = false>
__device__ __forceinline__ StatePosterior<R> state_posterior(int cnt, R Sd, R Qd, R c, R alpha, R beta, R nu, R xi,
                                                             int cm = 0, R Sm = R(0), R Qm = R(0), R k1 = R(0)) {
    StatePosterior<R> p;
    const R n = (R)cnt;
    const R dbar = cnt > 0 ? Sd / n : R(0);                          // ybar - c
    R s2 = Qd - n * dbar * dbar;                                     // sum (y - ybar)^2   (:291-294)
    s2 = s2 > R(0) ? s2 : R(0);
    R totalbar = cnt > 0 ? dbar + c : R(0);                          // :282-288
    R ne = n, extra = R(0);
    p.sumd = Sd; p.ntot = n;
    p.a = alpha + R(0.5) * n;                                        // :313
    if constexpr (SIG) {
        const R m = (R)cm;
        const R sbar = cm > 0 ? Sm / m : R(0);                       // sbar - c   (:272-278)
        R sm2 = Qm - m * sbar * sbar;                                // sum (signal - sbar)^2   (:297-300)
        sm2 = sm2 > R(0) ? sm2 : R(0);
        p.sumd = Sd + Sm; p.ntot = n + m;
        totalbar = (cnt + cm) > 0 ? p.sumd / p.ntot + c : R(0);
        ne = n + m * k1;                                             // Neff = Ni + Mi/(1+kappa)  (:302-303)
        p.a += R(0.5) * m;
        extra = R(0.5) * k1 * sm2;                                   // (0.5/(1+kappa)) Sm2  (:314)
    }
    const R dev = totalbar - xi;
    R b = beta + R(0.5) * s2;                                        // :314
    if constexpr (SIG) b += extra;
    b += R(0.5) * ne * nu / (ne + nu) * (dev * dev);
    p.b = b;
    p.neff = ne;
    return p;
}

// The chain state between launches (field f of a slot at [f * ns + slot], ns = a.n_slots) and the chain's priors.  With SIG
// also the statistics of the signals (cnt / Sd / Qd then count the observations only).
template <typename R, int K, bool SIG = false>
__device__ __forceinline__ void load_chain_stats(const GibbsArgs& a, const int ns, const int slot, int (&cnt)[K], R (&Sd)[K], R (&Qd)[K],
                                                 int (&trans)[K][K], Hyper<R, K>& hp, SigStats<R, K>* sg = nullptr) {
#pragma unroll
    for (int i = 0; i < K; ++i) {
        cnt[i] = a.cnt[i * ns + slot];
        Sd[i] = reinterpret_cast<const R*>(a.Sd)[i * ns + slot];
        Qd[i] = reinterpret_cast<const R*>(a.Qd)[i * ns + slot];
        hp.xi[i] = reinterpret_cast<const R*>(a.xi)[i * ns + slot];
        hp.alpha[i] = (R)a.alpha[i];
        hp.nu[i] = (R)a.nu[i];
#pragma unroll
        for (int j = 0; j < K; ++j) trans[i][j] = a.trans[(i * K + j) * ns + slot];
    }
    if constexpr (SIG) {
#pragma unroll
        for (int i = 0; i < K; ++i) {
            sg->m[i] = a.cntM[i * ns + slot];
            sg->Sm[i] = reinterpret_cast<const R*>(a.Sm)[i * ns + slot];
            sg->Qm[i] = reinterpret_cast<const R*>(a.Qm)[i * ns + slot];
        }
        sg->k1 = (R)(1.0 / (1.0 + a.kappa));
    }
}

// the chain's statistics back to GibbsArgs, and its events of this launch added to a.events (called by one lane of the chain)
template <typename R, int K, bool SIG = false>
__device__ __forceinline__ void store_chain_stats(const GibbsArgs& a, const int ns, const int slot, const int (&cnt)[K], const R (&Sd)[K],
                                                  const R (&Qd)[K], const int (&trans)[K][K], const int events,
                                                  const SigStats<R, K>* sg = nullptr) {
#pragma unroll
    for (int i = 0; i < K; ++i) {
        a.cnt[i * ns + slot] = cnt[i];
        reinterpret_cast<R*>(a.Sd)[i * ns + slot] = Sd[i];
        reinterpret_cast<R*>(a.Qd)[i * ns + slot] = Qd[i];
#pragma unroll
        for (int j = 0; j < K; ++j) a.trans[(i * K + j) * ns + slot] = trans[i][j];
        if constexpr (SIG) {
            a.cntM[i * ns + slot] = sg->m[i];
            reinterpret_cast<R*>(a.Sm)[i * ns + slot] = sg->Sm[i];
            reinterpret_cast<R*>(a.Qm)[i * ns + slot] = sg->Qm[i];
        }
    }
    a.events[slot] += events;
}

}  // namespace hmc
