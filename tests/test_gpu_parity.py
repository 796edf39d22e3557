"""GPU parity tests (run on the B200 box with -m gpu): every call goes through the C ABI (libhmcgpu.so via ctypes)
and is checked against the CPU oracle on the same seeded inputs, against the reference's golden posterior
summaries, or through size-independent properties at full size.

Tolerances (north_star): deterministic pieces 1e-5 relative in fp64 and 1e-3 in fp32; state paths under injected
uniforms bit-exact; full Gibbs posteriors within Monte-Carlo error.
"""
import json
import os

import numpy as np
import pytest

from conftest import dispersion_close, signals_golden_case, GOLDEN, K3_TRUTH, load_inflation, random_params, synth_hmm

pytestmark = pytest.mark.gpu

RTOL64, RTOL32 = 1e-5, 1e-3


@pytest.fixture(autouse=True, params=["auto", "thread", "seg"])
def _sweep_kernel_choice(request, monkeypatch):
    """Narrow batches (most tests) are served by the time-parallel warp-per-chain kernel; every test also runs with that
    kernel disabled so that the thread-per-chain kernels see the same small, ragged cases, and once more with the
    mid-width kernel forced (4 lanes per chain, one time segment each; it takes the plain sweep for K <= 4 — other
    problems fall through to the thread-per-chain kernels as in production)."""
    if request.param in ("thread", "seg"):
        monkeypatch.setenv("HMCGPU_SCAN_MAX_CHAINS", "0")
        # (HMC_TEST_SEG_LANES=2 / 8: the same suite on the other segment counts)
        monkeypatch.setenv("HMCGPU_SEG_LANES", os.environ.get("HMC_TEST_SEG_LANES", "4") if request.param == "seg" else "0")
    return request.param


def test_the_forced_sweep_kernel_is_the_one_that_ran(H, ctx, _sweep_kernel_choice):
    """hmcgpu_result.sweep_kernel reports the plan's choice: the three runs of every test really exercise three kernels."""
    y, _ = synth_hmm(80, **K3_TRUTH)
    o = _run(H, ctx, y, [1, 3], [70, 77], K=3, n_chains=3, burnin=2, nrun=2, seed=1, horizons=(1,), precision=32, flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS)
    assert o.sweep_kernel == {"auto": 1, "thread": 0, "seg": 4}[_sweep_kernel_choice]
    assert H.binding.KERNEL_NAMES[o.sweep_kernel].startswith({"auto": "gibbs_scan", "thread": "gibbs_sweeps", "seg": "gibbs_seg"}[_sweep_kernel_choice])


def test_native_library_is_loaded(H, ctx):
    tag = os.environ.get("HMC_TAG")            # A/B runs of a side library (scripts/ab_lib.sh) load lib/libhmcgpu_<tag>.so
    assert os.path.samefile(H.lib_path(), os.path.join(os.path.dirname(H.__file__), "lib", f"libhmcgpu_{tag}.so" if tag else "libhmcgpu.so"))
    assert H.load().hmcgpu_device_count() >= 1


def test_philox_known_answers_on_device(ctx, oracle):
    ctr = np.array([[0, 0, 0, 0], [0xffffffff] * 4, [0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344]], dtype=np.uint32)
    key = np.array([[0, 0], [0xffffffff] * 2, [0xa4093822, 0x299f31d0]], dtype=np.uint32)
    out = ctx.philox(ctr, key)
    assert out.tolist() == [[0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8], [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd],
                            [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]]
    rng = np.random.default_rng(0)
    ctr = rng.integers(0, 2**32, size=(1000, 4), dtype=np.uint64).astype(np.uint32)
    key = rng.integers(0, 2**32, size=(1000, 2), dtype=np.uint64).astype(np.uint32)
    out = ctx.philox(ctr, key)
    for i in range(0, 1000, 37):
        assert out[i].tolist() == oracle.philox(ctr[i], key[i])
    # the 7-round generator of the STATES stream (Random123 kat_vectors, philox4x32-7)
    out7 = ctx.philox(ctr[:3], key[:3], rounds=7)
    for i in range(3):
        assert out7[i].tolist() == oracle.philox(ctr[i], key[i], rounds=7)
    kat = ctx.philox(np.array([[0, 0, 0, 0], [0xffffffff] * 4], dtype=np.uint32), np.array([[0, 0], [0xffffffff] * 2], dtype=np.uint32), rounds=7)
    assert kat.tolist() == [[0x5f6fb709, 0x0d893f64, 0x4f121f81, 0x4f730a48], [0x5207ddc2, 0x45165e59, 0x4d8ee751, 0x8c52f662]]


@pytest.mark.parametrize("K", [2, 3, 4, 5, 8, 32])
@pytest.mark.parametrize("precision,rtol", [(64, RTOL64), (32, RTOL32)])
def test_filter_matches_oracle(ctx, oracle, K, precision, rtol):
    rng = np.random.default_rng(100 + K)
    B, T = 37, 700
    A, mu, s2, rho = random_params(rng, B, K)
    y = rng.normal(0, 3, size=(B, T))
    g = ctx.filter(y, A, mu, s2, rho, precision=precision)
    for b in range(B):
        f = oracle.forward(y[b], A[b], mu[b], s2[b], rho[b], want_Pf=False)
        # probabilities: relative on anything that matters, absolute floor for vanishing entries
        np.testing.assert_allclose(g.pif[b], f.pif, rtol=rtol, atol=rtol * 1e-3)
        assert abs(g.loglik[b] - f.loglik) <= rtol * abs(f.loglik)
        np.testing.assert_allclose(np.log(g.totals[b]), np.log(f.totals), rtol=0, atol=10 * rtol)
    if precision == 64:     # actual agreement is far tighter than the stated bar
        f = oracle.forward(y[0], A[0], mu[0], s2[0], rho[0], want_Pf=False)
        np.testing.assert_allclose(g.pif[0], f.pif, rtol=1e-10, atol=1e-200)


def test_filter_shared_series_and_extreme_observations(ctx, oracle):
    rng = np.random.default_rng(5)
    K, B, T = 3, 5, 400
    A, mu, s2, rho = random_params(rng, B, K)
    y = rng.normal(0, 3, size=T)
    y[50] = 40.0       # 13+ sigma from every state: the fp32 path must not underflow (hazard H1, scaled recursion)
    y[200] = -35.0
    for precision, rtol in ((64, RTOL64), (32, RTOL32)):
        g = ctx.filter(y, A, mu, s2, rho, precision=precision)
        assert np.isfinite(g.pif).all() and np.isfinite(g.loglik).all()
        for b in range(B):
            f = oracle.forward(y, A[b], mu[b], s2[b], rho[b], want_Pf=False)
            np.testing.assert_allclose(g.pif[b], f.pif, rtol=rtol, atol=rtol * 1e-3)
            assert abs(g.loglik[b] - f.loglik) <= rtol * abs(f.loglik)


@pytest.mark.parametrize("precision,rtol", [(64, RTOL64), (32, RTOL32)])
def test_filter_with_signal_rows_matches_oracle(ctx, oracle, precision, rtol):
    """hmcgpu_filter_masked: signal rows are emitted with sd*(1+kappa) (src/Hmc.jl:380-383), first row included."""
    rng = np.random.default_rng(77)
    K, B, T = 3, 11, 300
    A, mu, s2, rho = random_params(rng, B, K)
    y = rng.normal(0, 3, size=T)
    mask = (rng.random(T) < 0.3).astype(np.uint8); mask[0] = 1
    for kappa in (0.0, 0.6, 3.0):
        g = ctx.filter(y, A, mu, s2, rho, precision=precision, is_signal=mask, kappa=kappa)
        for b in range(B):
            f = oracle.forward(y, A[b], mu[b], s2[b], rho[b], is_signal=mask, kappa=kappa, want_Pf=False)
            np.testing.assert_allclose(g.pif[b], f.pif, rtol=rtol, atol=rtol * 1e-3)
            assert abs(g.loglik[b] - f.loglik) <= rtol * abs(f.loglik)
            np.testing.assert_allclose(np.log(g.totals[b]), np.log(f.totals), rtol=0, atol=10 * rtol)


@pytest.mark.parametrize("precision,rtol", [(64, RTOL64), (32, RTOL32)])
def test_smoother_matches_oracle(ctx, oracle, precision, rtol):
    rng = np.random.default_rng(21)
    K, B, T = 3, 9, 500
    A, mu, s2, rho = random_params(rng, B, K)
    y = rng.normal(0, 3, size=(B, T))
    pif = np.stack([oracle.forward(y[b], A[b], mu[b], s2[b], rho[b]).pif for b in range(B)])
    g = ctx.smooth(A, pif, precision=precision)
    for b in range(B):
        f = oracle.forward(y[b], A[b], mu[b], s2[b], rho[b])
        _, pib = oracle.backward(f.Pf, f.pif)        # the reference's literal Pb recursion
        np.testing.assert_allclose(g[b], pib, rtol=rtol, atol=rtol * 1e-3)


@pytest.mark.parametrize("K", [2, 3, 4, 8, 32])
def test_state_paths_bit_exact_under_injected_uniforms(ctx, oracle, K):
    rng = np.random.default_rng(31 + K)
    B, T = 64, 600
    A, mu, s2, rho = random_params(rng, B, K)
    y = rng.normal(0, 3, size=(B, T))
    pif = np.stack([oracle.forward(y[b], A[b], mu[b], s2[b], rho[b], want_Pf=False).pif for b in range(B)])
    u = rng.random((B, T))
    X = ctx.sample_states(A, pif, u)
    for b in range(B):
        Xo = oracle.sample_states(pif[b], A[b], u[b], form=1)
        np.testing.assert_array_equal(X[b], Xo)
    # edge cases: u = 0, u just below 1, and an explicit piN (quirk Q1 path)
    u0 = np.zeros((B, T)); u1 = np.full((B, T), np.nextafter(1.0, 0.0))
    piN = rng.dirichlet(np.ones(K), size=B)
    for uu in (u0, u1):
        X = ctx.sample_states(A, pif, uu, piN=piN)
        for b in range(0, B, 7):
            np.testing.assert_array_equal(X[b], oracle.sample_states(pif[b], A[b], uu[b], piN=piN[b], form=1))


def test_forecast_matches_oracle(ctx, oracle):
    rng = np.random.default_rng(41)
    K, B = 3, 50
    A, mu, s2, rho = random_params(rng, B, K)
    hs = list(range(1, 13))
    yreal = rng.normal(size=len(hs))
    g = ctx.forecast(mu, A, rho, hs, yreal)
    for b in range(B):
        for j, h in enumerate(hs):
            f, e = oracle.forecast(mu[b], A[b], rho[b], h, yreal[j])
            assert abs(g[b, j, 0] - f) <= 1e-12 * max(1, abs(f)) and abs(g[b, j, 1] - e) <= 1e-11 * max(1, abs(e))


def test_conjugate_draws_match_oracle_streams(ctx, oracle):
    """Same Philox streams on both sides: fp64 draws agree to rounding, fp32 to 1e-3 relative in distribution."""
    rng = np.random.default_rng(51)
    K, B = 3, 200
    Ni = rng.integers(0, 300, size=(B, K))
    ybar = rng.normal(3, 2, size=(B, K))
    S = Ni * ybar
    S2 = Ni * rng.uniform(0.3, 4.0, size=(B, K))
    trans = rng.integers(0, 200, size=(B, K, K)) + 1
    xi, one = np.full(K, 3.3), np.ones(K)
    s2, mu, rho, A = ctx.draw_params(Ni, S, S2, trans, xi, one, one, 2 * one, seed=1234, chain0=1000, sweep=17, precision=64)
    for b in range(B):
        o = oracle.draw_params(Ni[b], S[b], S2[b], trans[b], xi, one, one, 2 * one, 1234, 1000 + b, 17)
        np.testing.assert_allclose(s2[b], o[0], rtol=1e-9)
        np.testing.assert_allclose(mu[b], o[1], rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(rho[b], o[2], rtol=1e-9)
        np.testing.assert_allclose(A[b], o[3], rtol=1e-9)
    s2f, muf, rhof, Af = ctx.draw_params(Ni, S, S2, trans, xi, one, one, 2 * one, seed=1234, chain0=1000, sweep=17, precision=32)
    # fp32 follows the same streams; a rejection decision can flip only on a measure-~1e-6 set
    close = np.isclose(s2f, s2, rtol=2e-3).mean()
    assert close > 0.99
    assert np.isclose(Af, A, rtol=5e-3, atol=1e-5).mean() > 0.99


def test_conjugate_draws_with_signal_statistics_match_oracle_streams(ctx, oracle):
    """update_μσ! with noisy signals (src/Hmc.jl:267-314): Meff = Mi/(1+κ), a = α + ½Ni + ½Mi, b with ½Sm2/(1+κ), posterior mean
    (S + Sm + νξ)/(Neff + ν) — fp64 draws agree with the oracle's on the same Philox streams."""
    rng = np.random.default_rng(52)
    K, B = 3, 150
    Ni = rng.integers(0, 300, size=(B, K)); Mi = rng.integers(0, 40, size=(B, K))
    Mi[::7] = 0; Ni[3::11] = 0
    S = Ni * rng.normal(3, 2, size=(B, K)); Sm = Mi * rng.normal(3, 2, size=(B, K))
    S2 = Ni * rng.uniform(0.3, 4.0, size=(B, K)); Sm2 = Mi * rng.uniform(0.3, 6.0, size=(B, K))
    trans = rng.integers(0, 200, size=(B, K, K)) + 1
    xi, two = np.full(K, 3.3), np.full(K, 2.0)
    for kappa in (0.0, 0.6, 3.0):
        s2, mu, rho, A = ctx.draw_params(Ni, S, S2, trans, xi, two, two, two, seed=99, chain0=500, sweep=4, precision=64,
                                         Mi=Mi, Sm=Sm, Sm2=Sm2, kappa=kappa)
        for b in range(0, B, 3):
            o = oracle.draw_params(Ni[b], S[b], S2[b], trans[b], xi, two, two, two, 99, 500 + b, 4, kappa=kappa, Mi=Mi[b], Sm=Sm[b], Sm2=Sm2[b])
            np.testing.assert_allclose(s2[b], o[0], rtol=1e-9)
            np.testing.assert_allclose(mu[b], o[1], rtol=1e-9, atol=1e-9)
            np.testing.assert_allclose(rho[b], o[2], rtol=1e-9)
            np.testing.assert_allclose(A[b], o[3], rtol=1e-9)


def _run(H, ctx, y, ws, we, **kw):
    spec = H.ProblemSpec(y, ws, we, **kw)
    return H.estimate(ctx, spec)


def test_gibbs_first_sweeps_follow_the_oracle_chain(H, ctx, oracle):
    """fp64 device chain vs oracle chain on the same Philox streams: identical up to libm rounding for the first sweeps."""
    y, _ = synth_hmm(260, **K3_TRUTH)
    hs = (1, 12)
    for (s, e) in ((1, 200), (20, 248)):
        o = _run(H, ctx, y, [s], [e], K=3, n_chains=3, burnin=2, nrun=6, seed=77, horizons=hs, precision=64,
                 flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK)
        assert o.events == 0
        for c in range(3):
            yf = [y[e - 1 + h] for h in hs]
            r = oracle.gibbs(y[s - 1:e], 3, 2, 6, seed=77, chain=c, horizons=hs, y_future=yf,
                             flags=oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM)
            sl = slice(c * 6, (c + 1) * 6)
            np.testing.assert_allclose(o.mu[0][:, sl].T, r.mu, rtol=1e-8)
            np.testing.assert_allclose(o.sigma2[0][:, sl].T, r.sigma2, rtol=1e-8)
            np.testing.assert_allclose(np.transpose(o.A[0][:, :, sl], (2, 1, 0)), r.A, rtol=1e-8)
            np.testing.assert_allclose(o.pi_end[0][:, sl].T, r.pi_end, rtol=1e-7, atol=1e-12)
            np.testing.assert_allclose(o.forecasts[0][:, sl].T, r.forecasts, rtol=1e-8, atol=1e-9)
            np.testing.assert_allclose(o.loglik[0][sl], r.loglik, rtol=1e-9)


def test_mixed_segment_counts_follow_the_oracle_chain(H, ctx, oracle, monkeypatch):
    """Mid-width plans with thread slots to spare give their LONGEST windows 8 lanes per chain and the rest 4 (two slot ranges with
    their own warp-task tables, one stream group per class).  Forced here on a small ragged batch (HMCGPU_SEG_LONG = number of
    long windows): every chain of both classes must follow the oracle's chain, and the split must not move any window's results
    to another window (slot ranges, padding between the classes, summaries per window)."""
    monkeypatch.setenv("HMCGPU_SCAN_MAX_CHAINS", "0")
    monkeypatch.delenv("HMCGPU_SEG_LANES", raising=False)
    monkeypatch.setenv("HMCGPU_SEG_LONG", "5")
    y, _ = synth_hmm(420, seed=21, **K3_TRUTH)
    ends = [400, 160, 333, 250, 129, 380, 90, 301, 64, 222, 199, 147]          # 12 windows; the 5 longest (T >= 250) form the long class
    starts = [1, 3, 2, 1, 1, 9, 5, 1, 2, 4, 1, 1]
    nc = 7                                                                       # 35 long chains (padding inside the class), 49 others
    o = _run(H, ctx, y, starts, ends, K=3, n_chains=nc, burnin=1, nrun=3, seed=13, horizons=(1, 2), precision=64,
             flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK | H.FLAG_SUMMARY)
    assert o.events == 0 and o.sweep_kernel == 4
    for w, (s, e) in enumerate(zip(starts, ends)):
        for c in (0, nc - 1):
            r = oracle.gibbs(y[s - 1:e], 3, 1, 3, seed=13, chain=w * nc + c, horizons=(1, 2), y_future=[y[e], y[e + 1]],
                             flags=oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM)
            sl = slice(c * 3, (c + 1) * 3)
            np.testing.assert_allclose(o.mu[w][:, sl].T, r.mu, rtol=1e-7, atol=1e-9)
            np.testing.assert_allclose(o.sigma2[w][:, sl].T, r.sigma2, rtol=1e-7)
            np.testing.assert_allclose(np.transpose(o.A[w][:, :, sl], (2, 1, 0)), r.A, rtol=1e-7, atol=1e-12)
            np.testing.assert_allclose(o.loglik[w][sl], r.loglik, rtol=1e-8)
    # the same batch with one segment count for every window: same chains (fp64: to rounding), same per-window summaries
    monkeypatch.setenv("HMCGPU_SEG_MIXED", "0")
    monkeypatch.delenv("HMCGPU_SEG_LONG")
    u = _run(H, ctx, y, starts, ends, K=3, n_chains=nc, burnin=1, nrun=3, seed=13, horizons=(1, 2), precision=64,
             flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK | H.FLAG_SUMMARY)
    np.testing.assert_allclose(o.summary_mean, u.summary_mean, rtol=1e-7, atol=1e-9)
    for w in range(len(ends)):
        np.testing.assert_allclose(o.mu[w], u.mu[w], rtol=1e-7, atol=1e-9)


@pytest.mark.parametrize("K,T", [(2, 37), (3, 2), (3, 33), (3, 1500), (4, 334)])
def test_chunk_shapes_follow_the_oracle_chain(H, ctx, oracle, K, T):
    """Window lengths that stress the time-parallel kernel's chunking (idle lanes, one step per lane, chunks longer than
    the 32-step path record) and K = 2, 4; the same cases run on the thread-per-chain kernel through the module fixture.
    Even K with an odd window length is included: the median observation then lies exactly between the initial states K/2
    and K/2 + 1 of makeParams (src/Hmc.jl:175-187); device and oracle decide it with the same exact distance comparison
    (ties to the lower state, as findmax)."""
    tr = K3_TRUTH if K == 3 else _truth(K)
    y, _ = synth_hmm(T + 3, seed=9 + K, **tr)
    o = _run(H, ctx, y, [1, 2], [T, T + 1], K=K, n_chains=2, burnin=1, nrun=4, seed=5, horizons=(1, 2), precision=64,
             flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK)
    for w, (s, e) in enumerate(((1, T), (2, T + 1))):
        for c in range(2):
            r = oracle.gibbs(y[s - 1:e], K, 1, 4, seed=5, chain=w * 2 + c, horizons=(1, 2), y_future=[y[e], y[e + 1]],
                             flags=oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM)
            sl = slice(c * 4, (c + 1) * 4)
            np.testing.assert_allclose(o.mu[w][:, sl].T, r.mu, rtol=1e-7, atol=1e-9)
            np.testing.assert_allclose(o.sigma2[w][:, sl].T, r.sigma2, rtol=1e-7)
            np.testing.assert_allclose(np.transpose(o.A[w][:, :, sl], (2, 1, 0)), r.A, rtol=1e-7, atol=1e-12)
            np.testing.assert_allclose(o.pi_end[w][:, sl].T, r.pi_end, rtol=1e-6, atol=1e-12)
            np.testing.assert_allclose(o.forecasts[w][:, sl].T, r.forecasts, rtol=1e-7, atol=1e-8)
            np.testing.assert_allclose(o.loglik[w][sl], r.loglik, rtol=1e-8)


def test_gibbs_reference_integration_test(H, ctx):
    """The reference's only test (test/runtests.jl:20-57) through the estimatemodel mirror, fp64 and fp32."""
    y, _ = synth_hmm(500, [[0.5, 0.5], [0.2, 0.8]], [-5.0, 4.0], [1.0, 0.5], seed=123)
    for precision in (64, 32):
        opt = H.EstOpt(y, list(range(500)), sampleRange=range(1, 477), endIndex=476, horizons=[12], D=2, burnin=3000,
                       Nrun=1000, series="test", precision=precision)
        s = H.estimatemodel(opt, ctx)
        assert s.μ.shape == (1000, 2) and s.σ.shape == (1000, 2) and s.A.shape == (1000, 2, 2)
        assert s.πb.shape == (1000, 1, 2) and s.forecasts.shape == (1000, 2) and len(s.obsdates) == 1000
        assert np.all(np.abs(s.μ.mean(0) - [-5.0, 4.0]) < 0.3)          # runtests.jl:56
        assert np.all(np.abs(s.σ.mean(0) - [1.0, 0.5]) < 0.5)           # runtests.jl:57
        assert np.all(np.diff(s.μ, axis=1) > 0)
        np.testing.assert_allclose(s.A.sum(2), 1.0, atol=1e-5)
        np.testing.assert_allclose(s.πb[:, -1, :].sum(1), 1.0, atol=1e-5)
        np.testing.assert_allclose(s.forecasts[:, 1], s.forecasts[:, 0] - y[476 + 11], atol=1e-4)
        assert s.events == 0


@pytest.mark.parametrize("precision", [64, 32])
def test_gibbs_posterior_matches_oracle_posterior(H, ctx, oracle, precision):
    """Monte-Carlo parity on a synthetic series: pooled multi-chain posterior means/variances vs the oracle's."""
    y, _ = synth_hmm(412, **K3_TRUTH)
    hs = (1, 6, 12)
    nch, burn, nrun = 64, 500, 500
    o = _run(H, ctx, y, [1], [400], K=3, n_chains=nch, burnin=burn, nrun=nrun, seed=2024, horizons=hs, precision=precision,
             flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY)
    yf = [y[400 - 1 + h] for h in hs]
    outs, _ = oracle.gibbs_batch([dict(y=y[:400], K=3, burnin=burn, nrun=nrun, seed=4048, chain=c, horizons=hs, y_future=yf)
                                  for c in range(16)])
    cat = lambda k: np.concatenate([getattr(r, k) for r in outs])
    om, os2, oA, ope, ofc = cat("mu"), cat("sigma2"), cat("A"), cat("pi_end"), cat("forecasts")

    def close(g, ref, name):
        # standard error of the difference of two MC means; chains are autocorrelated -> inflate by 4, 5-sigma band
        se = 4 * np.sqrt(ref.var(0) / len(ref) + g.var(0) / len(g))
        d = np.abs(g.mean(0) - ref.mean(0))
        assert np.all(d <= 5 * se + 1e-4), (name, d, se)
        np.testing.assert_allclose(g.var(0), ref.var(0), rtol=0.35, atol=1e-5, err_msg=name)

    close(o.mu[0].T, om, "mu")
    close(o.sigma2[0].T, os2, "sigma2")
    close(np.transpose(o.A[0], (2, 1, 0)).reshape(-1, 9), oA.reshape(-1, 9), "A")
    close(o.pi_end[0].T, ope, "pi_end")
    close(o.forecasts[0].T, ofc, "forecasts")
    # device-side summary == moments of the returned draws
    F = np.concatenate([o.mu[0], o.sigma2[0], o.A[0].reshape(9, -1), o.pi_end[0], o.forecasts[0]])
    np.testing.assert_allclose(o.summary_mean[0][:-1], F.mean(1), rtol=1e-6, atol=1e-7)
    np.testing.assert_allclose(o.summary_var[0][:-1], F.var(1), rtol=1e-4, atol=1e-7)


@pytest.mark.parametrize("which", [0, 9, 18])
def test_gibbs_matches_reference_golden_summaries(H, ctx, which):
    """Real series, real end dates: posterior means vs data/output/official/*_summary.csv (MC tolerance)."""
    y, dates = load_inflation()
    g = json.load(open(os.path.join(GOLDEN, "official_summary_subset.json")))["windows"][which]
    idx = g["end_index"]
    o = _run(H, ctx, y, [1], [idx], K=3, n_chains=64, burnin=2000, nrun=1000, seed=1234, horizons=(12,), precision=32,
             flags=H.FLAG_REF_Q1 | H.FLAG_SUMMARY)
    m = o.summary_mean[0]
    np.testing.assert_allclose(m[0:3], g["filtered_means"], atol=0.08)
    np.testing.assert_allclose(m[3:6], g["filtered_variances"], rtol=0.06)
    np.testing.assert_allclose(m[6:15], g["filtered_trans_probs"], atol=0.01)     # summary A index s*K+r == trans_s_r column
    np.testing.assert_allclose(m[15:18], g["filtered_state_probs"], atol=0.01)
    if idx + 12 <= len(y):
        np.testing.assert_allclose(m[18:20], g["forecasts"], atol=0.06)


def test_smoothed_probability_means(H, ctx, oracle):
    y, _ = synth_hmm(300, **K3_TRUTH)
    o = _run(H, ctx, y, [1, 1], [300, 250], K=3, n_chains=32, burnin=300, nrun=300, seed=9, horizons=(), precision=32,
             flags=H.FLAG_REF_Q1 | H.FLAG_SMOOTHED_MEAN | H.FLAG_SUMMARY)
    for w, n in enumerate((300, 250)):
        outs, _ = oracle.gibbs_batch([dict(y=y[:n], K=3, burnin=300, nrun=600, seed=10, chain=c, horizons=(), want_pib_mean=True)
                                      for c in range(8)])
        ref = np.mean([r.pib_mean for r in outs], axis=0)
        pm = o.pib_mean[w]
        assert pm.shape == (n, 3)
        np.testing.assert_allclose(pm.sum(1), 1.0, atol=1e-4)
        assert np.abs(pm - ref).max() < 0.06 and np.abs(pm - ref).mean() < 0.004
        # last row = mean of pi_end
        np.testing.assert_allclose(pm[-1], o.summary_mean[w][15:18], atol=1e-5)


def test_expanding_windows_ragged_batch_and_sharding_invariance(H, ctx):
    """Ragged windows in one launch; results must not depend on batching/sharding (counter-based RNG + win_id)."""
    y, _ = synth_hmm(330, **K3_TRUTH)
    ws, we = H.expanding_windows(101, 140)
    kw = dict(K=3, n_chains=3, burnin=30, nrun=20, seed=5, horizons=(1, 12), precision=64, flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS)
    full = _run(H, ctx, y, ws, we, **kw)
    assert full.state_steps == int((we - ws + 1).sum()) * 3 * 50
    for shard in H.shard_windows(we - ws + 1, 3):
        part = _run(H, ctx, y, ws[shard], we[shard], win_id=shard, **kw)
        np.testing.assert_array_equal(part.mu, full.mu[shard])
        np.testing.assert_array_equal(part.A, full.A[shard])
        np.testing.assert_array_equal(part.forecasts, full.forecasts[shard])
    # a window estimated alone equals the same window inside the batch
    one = _run(H, ctx, y, ws[7:8], we[7:8], win_id=[7], **kw)
    np.testing.assert_array_equal(one.mu[0], full.mu[7])


def test_estimate_multi_shards_windows_and_gathers_on_the_host(H, ctx):
    """hmcgpu_estimate_multi: windows sharded over a device list (here device 0 twice: two host threads, two contexts), every
    per-window output scattered back into the caller's arrays — identical to the single-context call, with and without the
    signals-tier inputs (mask, X0, init series) and with the smoothed means."""
    rng = np.random.default_rng(2)
    y0, _ = synth_hmm(260, **K3_TRUTH)
    ys = np.stack([y0, y0 + rng.normal(0, 0.3, size=len(y0))])
    ws = np.array([1, 5, 2, 40, 1], dtype=np.int32); we = np.array([200, 180, 120, 240, 90], dtype=np.int32)
    mask = np.zeros(len(y0), dtype=np.uint8); mask[60:66] = 1
    X0 = [rng.integers(1, 4, int(e - s + 1)) for s, e in zip(ws, we)]
    cases = [dict(flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY | H.FLAG_LOGLIK),
             dict(flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY, is_signal=mask, kappa=0.7, X0=X0, win_init_series=[0] * 5, pi_row_back=2),
             dict(flags=H.FLAG_REF_Q1 | H.FLAG_SUMMARY | H.FLAG_SMOOTHED_MEAN)]
    for extra in cases:
        kw = dict(K=3, n_chains=2, burnin=3, nrun=5, seed=9, horizons=(1, 12), precision=64, win_series=[1, 0, 1, 1, 0], **extra)
        one = _run(H, ctx, ys, ws, we, **kw)
        multi = H.estimate_multi([0, 0], H.ProblemSpec(ys, ws, we, **kw))
        for k in ("mu", "sigma2", "A", "pi_end", "forecasts", "loglik", "summary_mean", "summary_var"):
            if getattr(one, k) is not None:
                np.testing.assert_array_equal(getattr(multi, k), getattr(one, k), err_msg=k)
        if one.pib_mean is not None:
            for a, b in zip(multi.pib_mean, one.pib_mean):
                np.testing.assert_array_equal(a, b)
            for a, b in zip(multi.insample_forecast_mean, one.insample_forecast_mean):
                np.testing.assert_array_equal(a, b)
        assert multi.state_steps == one.state_steps and multi.events == one.events


def test_multiple_series_time_major_layout(H, ctx):
    rng = np.random.default_rng(3)
    ys = np.stack([synth_hmm(150, seed=s, **K3_TRUTH)[0] for s in range(5)])
    kw = dict(K=3, n_chains=2, burnin=20, nrun=10, seed=1, horizons=(3,), precision=64, flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS)
    o = _run(H, ctx, ys, [1] * 5, [140] * 5, win_series=np.arange(5), **kw)
    for s in (0, 3):
        single = _run(H, ctx, ys[s], [1], [140], win_id=[s], **kw)
        np.testing.assert_array_equal(single.mu[0], o.mu[s])
        np.testing.assert_array_equal(single.forecasts[0], o.forecasts[s])


def test_staged_upload_of_large_series_is_bit_identical(H, ctx, monkeypatch):
    """Series uploads above two staging chunks go through pinned double buffers filled by several host threads
    (hmcgpu.cu::staged_upload); the results must not depend on the chunk size, the thread count or on staging at all.
    3000 series x 700 observations = 16.8 MB: staged with 1 MB chunks (odd tail chunk, uneven thread slices)."""
    rng = np.random.default_rng(11)
    base = np.stack([synth_hmm(700, seed=s, **K3_TRUTH)[0] for s in range(8)])
    ys = np.ascontiguousarray(np.tile(base, (375, 1)) + 1e-3 * rng.standard_normal((3000, 700)))
    kw = dict(K=3, n_chains=1, burnin=4, nrun=4, seed=5, horizons=(1,), precision=64, flags=H.FLAG_REF_Q1 | H.FLAG_SUMMARY,
              win_series=np.arange(3000))
    outs = []
    for mb, thr in (("0", "1"), ("1", "3"), ("1", "8"), ("5", "2")):
        monkeypatch.setenv("HMCGPU_STAGE_MB", mb)
        monkeypatch.setenv("HMCGPU_STAGE_THREADS", thr)
        outs.append(_run(H, ctx, ys, [1] * 3000, [690] * 3000, **kw))
    for o in outs[1:]:
        np.testing.assert_array_equal(o.summary_mean, outs[0].summary_mean)
        np.testing.assert_array_equal(o.summary_var, outs[0].summary_var)
    assert outs[0].h2d_bytes == outs[1].h2d_bytes


def test_plan_run_is_repeatable_and_device_resident(H, ctx):
    y, _ = synth_hmm(220, **K3_TRUTH)
    spec = H.ProblemSpec(y, [1, 1], [200, 150], K=3, n_chains=40, burnin=20, nrun=30, seed=3, horizons=(12,), precision=32,
                         flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY)
    plan = H.Plan(ctx, spec)
    plan.run(); a = plan.fetch()
    plan.run(); b = plan.fetch()
    plan.close()
    np.testing.assert_array_equal(a.mu, b.mu)
    np.testing.assert_array_equal(a.summary_mean, b.summary_mean)
    assert a.n_sweep_launches >= 2 and a.gpu_ms > 0 and a.sweep_kernel_ms > 0
    assert a.state_steps == (200 + 150) * 40 * 50


def test_warm_started_window_chaining(H, ctx, oracle):
    """api.sample_and_forecast_all (the intent of sampleAndForecastAll, src/Hmc.jl:584-638) on the device against the oracle run
    the same way: long burn-in on the first sample, then per end date a short burn-in from the carried state path (new dates
    by the makeParams rule, :610-620), beta0 = 2 (:347), posterior means per end date and forecasts from those means.  The two
    chains share the law, not the realisation (Julia's stream is unpinnable; the device re-draws the carried path from
    X | theta, y): agreement within the Monte-Carlo error of one chain."""
    y, _ = synth_hmm(262, **K3_TRUTH)
    dates = list(range(1, len(y) + 1))
    ends = list(range(240, 246))
    out = H.sample_and_forecast_all(y, dates, range(1, len(y) + 1), [1, 12], ends, D=3, burnin=150, Nrun=3000, initialburn=1500,
                                    initialNrun=50, seed=11, ctx=ctx)
    assert out["events"] == 0 and out["dates"] == ends
    # the oracle chained the same way (its own final state path is carried: X_final).  Oracle seed 13: with seed 12 the long
    # burn-in ends in the posterior's minority mode (mu_2 = 3.43, sigma2_2 = 0.70 over the first window's 3000 draws; seeds 13-15
    # give 0.533 +- 0.003) and leaves it only one end date later — the reference algorithm's own mixing, not a parity question.
    r = oracle.gibbs(y[:ends[0]], 3, 1500, 50, seed=13, chain=0, horizons=(1,))
    X = r.X_final
    two = np.full(3, 2.0)
    for i, j in enumerate(ends):
        X0 = oracle.make_params(y[:j], 3)[0]
        m = min(len(X0), len(X))
        X0[:m] = X[:m]
        np.testing.assert_array_equal(X0[m:], H.makeparams_states(y[:j], 3)[m:])       # host copy of the makeParams rule
        r = oracle.gibbs(y[:j], 3, 150, 3000, seed=13, chain=i + 1, horizons=(1,), X0=X0, beta0=two)
        X = r.X_final
        mu, A, pe = r.mu.mean(0), r.A.mean(0), r.pi_end.mean(0)
        np.testing.assert_allclose(out["μ"][i], mu, atol=0.12)
        np.testing.assert_allclose(out["σ"][i], r.sigma2.mean(0), rtol=0.12)
        np.testing.assert_allclose(out["A"][i], A, atol=0.02)
        np.testing.assert_allclose(out["πb"][i], pe, atol=0.03)
        for k, h in enumerate((1, 12)):
            f = float(pe @ np.linalg.matrix_power(A, h) @ mu)
            assert abs(out["forecasts"][i, 2 * k] - f) < 0.12
            assert abs(out["forecasts"][i, 2 * k + 1] - (out["forecasts"][i, 2 * k] - y[j + h - 1])) < 1e-12
    assert np.all(np.diff(out["μ"], axis=1) > 0)


def test_full_size_properties_fp32(H, ctx):
    """BASELINE config 2 shape (500 expanding windows, T=101..600), reduced sweeps: size-independent properties."""
    y, _ = synth_hmm(612, **K3_TRUTH)
    ws, we = H.expanding_windows(101, 600)
    o = _run(H, ctx, y, ws, we, K=3, n_chains=32, burnin=60, nrun=40, seed=1234, horizons=tuple(range(1, 13)), precision=32,
             flags=H.FLAG_REF_Q1 | H.FLAG_SUMMARY)
    m, v = o.summary_mean, o.summary_var
    assert np.isfinite(m).all() and np.isfinite(v).all() and (v >= 0).all()
    assert o.events == 0 and (o.status == 0).all()
    assert np.all(np.diff(m[:, 0:3], axis=1) > 0)                                  # increasing-mu order
    A = m[:, 6:15].reshape(-1, 3, 3)                                               # [s][r]
    np.testing.assert_allclose(A.sum(1), 1.0, atol=1e-4)                           # rows of the mean A sum to 1
    np.testing.assert_allclose(m[:, 15:18].sum(1), 1.0, atol=1e-4)                 # pi_end is a probability vector
    fc = m[:, 18:42].reshape(-1, 12, 2)
    yreal = np.array([[y[e - 1 + h] for h in range(1, 13)] for e in we])
    np.testing.assert_allclose(fc[:, :, 0] - fc[:, :, 1], yreal, atol=2e-4)        # error = forecast - realised
    assert (fc[:, :, 0] > m[:, 0:1] - 0.5).all() and (fc[:, :, 0] < m[:, 2:3] + 0.5).all()   # convex combination of mu
    # long windows recover the generating parameters
    big = we >= 500
    assert np.abs(m[big, 0:3] - K3_TRUTH["mu"]).max() < 1.2     # only 60 burn-in sweeps


def test_zero_normaliser_events_are_counted_and_survived(H, ctx, monkeypatch):
    """An observation so far out that every fp64 emission underflows (total = 0) — a tight variance prior (alpha = 1e4)
    keeps the sampler from absorbing the outlier into one state's variance: the reference only warns (src/Hmc.jl:435)
    and carries NaNs on; the device counts the event, resets that row to the uniform vector and goes on.  Both sweep
    kernels (time-parallel: serial checked fallback; thread-per-chain: checked re-run) must agree over the first sweeps
    (this posterior is degenerate — variances from 1e-4 to 800, probabilities of exactly 0 and 1 — so any last-bit
    difference eventually sends the two chains to different modes); the fp32 path rescales and sees no event at all."""
    y, _ = synth_hmm(212, **K3_TRUTH)
    y[120] = 4.0e3
    tight = np.full(3, 1.0e4)
    outs = {}
    for mode in ("scan", "thread"):
        monkeypatch.setenv("HMCGPU_SCAN_MAX_CHAINS", "100000" if mode == "scan" else "0")
        outs[mode] = _run(H, ctx, y, [1], [200], K=3, n_chains=3, burnin=0, nrun=3, seed=3, horizons=(1,), precision=64,
                          flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK, alpha=tight)
        o = outs[mode]
        assert o.events == 3 and (o.status > 0).all()                       # every chain hit it (every sweep)
        assert np.isfinite(o.mu).all() and np.isfinite(o.sigma2).all() and np.isfinite(o.A).all() and np.isfinite(o.pi_end).all()
    np.testing.assert_allclose(outs["scan"].mu, outs["thread"].mu, rtol=1e-7)
    np.testing.assert_allclose(outs["scan"].pi_end, outs["thread"].pi_end, rtol=1e-6, atol=1e-12)
    o32 = _run(H, ctx, y, [1], [200], K=3, n_chains=3, burnin=2, nrun=6, seed=3, horizons=(1,), precision=32,
               flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS, alpha=tight)
    assert o32.events == 0 and np.isfinite(o32.mu).all()


def test_error_paths(H, ctx):
    y = np.arange(50.0)
    with pytest.raises(H.HmcGpuError) as e:
        _run(H, ctx, y, [1], [60], K=3)
    assert e.value.code == -1
    with pytest.raises(H.HmcGpuError) as e:
        _run(H, ctx, y, [1], [40], K=40)
    assert e.value.code == -4
    with pytest.raises(H.HmcGpuError) as e:          # smoothing accumulators exist for the thread-per-chain kernels only (K <= 8)
        _run(H, ctx, y, [1], [40], K=12, flags=H.FLAG_SMOOTHED_MEAN)
    assert e.value.code == -4
    with pytest.raises(H.HmcGpuError):
        _run(H, ctx, y, [10], [10], K=3)
    with pytest.raises(H.HmcGpuError) as e:          # 32-bit chain slots: refused before anything is allocated
        H.Plan(ctx, H.ProblemSpec(y, [1] * 40000, [40] * 40000, K=3, n_chains=60000))
    assert e.value.code == -4
    with pytest.raises(H.HmcGpuError):
        H.Context(99)


# ---------------------------------------------------------------------------------------------------------------------
# K = 5..32: the lane-per-state kernel (gibbs_wide_kernel) and the runtime-K deterministic entry points

def _truth(K):
    A = np.full((K, K), 0.1 / (K - 1)) + np.eye(K) * (0.9 - 0.1 / (K - 1))
    return dict(A=A, mu=2.0 * np.arange(K), sigma2=np.full(K, 0.5))           # SURVEY section 8d: K=8/32 truth


@pytest.mark.parametrize("K", [5, 8, 32])
def test_wide_smoother_forecast_draws_match_oracle(ctx, oracle, K):
    rng = np.random.default_rng(200 + K)
    B, T = 6, 120
    A, mu, s2, rho = random_params(rng, B, K)
    y = rng.normal(0, 3, size=(B, T))
    pif = np.stack([oracle.forward(y[b], A[b], mu[b], s2[b], rho[b]).pif for b in range(B)])
    g = ctx.smooth(A, pif, precision=64)
    fc = ctx.forecast(mu, A, rho, [1, 12], [0.5, -0.25])
    for b in range(B):
        f = oracle.forward(y[b], A[b], mu[b], s2[b], rho[b])
        _, pib = oracle.backward(f.Pf, f.pif)
        np.testing.assert_allclose(g[b], pib, rtol=RTOL64, atol=1e-9)
        for j, h in enumerate((1, 12)):
            fo, eo = oracle.forecast(mu[b], A[b], rho[b], h, (0.5, -0.25)[j])
            assert abs(fc[b, j, 0] - fo) < 1e-11 * max(1, abs(fo)) and abs(fc[b, j, 1] - eo) < 1e-10 * max(1, abs(eo))
    Ni = rng.integers(0, 50, size=(B, K)); S = Ni * rng.normal(3, 2, size=(B, K)); S2 = Ni * rng.uniform(0.3, 2, size=(B, K))
    trans = rng.integers(0, 30, size=(B, K, K)) + 1
    xi, one = np.full(K, 3.0), np.ones(K)
    s2d, mud, rhod, Ad = ctx.draw_params(Ni, S, S2, trans, xi, one, one, 2 * one, seed=99, chain0=7, sweep=3, precision=64)
    for b in range(B):
        o = oracle.draw_params(Ni[b], S[b], S2[b], trans[b], xi, one, one, 2 * one, 99, 7 + b, 3)
        np.testing.assert_allclose(s2d[b], o[0], rtol=1e-9)
        np.testing.assert_allclose(mud[b], o[1], rtol=1e-9, atol=1e-9)
        np.testing.assert_allclose(rhod[b], o[2], rtol=1e-9)
        np.testing.assert_allclose(Ad[b], o[3], rtol=1e-9)


@pytest.mark.parametrize("K,T,lane", [(5, 150, 0), (6, 300, 0), (7, 700, 0), (8, 200, 0), (8, 900, 0), (5, 150, 1), (8, 200, 1),
                                      (16, 160, 0), (32, 260, 0)])
def test_wide_gibbs_first_sweeps_follow_the_oracle_chain(H, ctx, oracle, K, T, lane, monkeypatch):
    """fp64 chain vs the oracle chain on the same Philox streams for K > 4 (several chains: sub-warp groups).  K = 5..8
    run on the thread-per-chain kernel (packed transition counters flushed every 2^(64/K)-1 steps: T = 700 / 900 cross
    that bound) or, with HMCGPU_LANE_KERNEL=1, on the lane-per-state kernel that serves K = 9..32."""
    if lane:
        monkeypatch.setenv("HMCGPU_LANE_KERNEL", "1")
    y, _ = synth_hmm(T + 12, seed=5 + K, **_truth(K))
    hs = (1, 12)
    nch = 5
    o = _run(H, ctx, y, [1, 3], [T, T - 17], K=K, n_chains=nch, burnin=1, nrun=4, seed=31, horizons=hs, precision=64,
             flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK)
    assert o.events == 0
    for w, (s, e) in enumerate(((1, T), (3, T - 17))):
        for c in range(nch):
            r = oracle.gibbs(y[s - 1:e], K, 1, 4, seed=31, chain=w * nch + c, horizons=hs, y_future=[y[e - 1 + h] for h in hs],
                             flags=oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM)
            sl = slice(c * 4, (c + 1) * 4)
            np.testing.assert_allclose(o.mu[w][:, sl].T, r.mu, rtol=1e-7, atol=1e-9)
            np.testing.assert_allclose(o.sigma2[w][:, sl].T, r.sigma2, rtol=1e-7)
            np.testing.assert_allclose(np.transpose(o.A[w][:, :, sl], (2, 1, 0)), r.A, rtol=1e-7, atol=1e-12)
            np.testing.assert_allclose(o.pi_end[w][:, sl].T, r.pi_end, rtol=1e-6, atol=1e-12)
            np.testing.assert_allclose(o.forecasts[w][:, sl].T, r.forecasts, rtol=1e-7, atol=1e-8)
            np.testing.assert_allclose(o.loglik[w][sl], r.loglik, rtol=1e-8)


def test_wide_gibbs_fp32_posterior_matches_oracle(H, ctx, oracle):
    """fp32 thread-per-chain kernel at K = 8 (the default for K <= 8; the lane kernel's fp32 chains at K = 5..32 are checked
    draw by draw in test_fp32_chain_parity.py): pooled posterior means vs the oracle's under identical settings (K=8 mixes
    slowly from the makeParams start, so both are compared to each other, not to the generating truth)."""
    K = 8
    tr = _truth(K)
    y, _ = synth_hmm(612, seed=3, **tr)
    burn, nrun = 300, 200
    o = _run(H, ctx, y, [1], [600], K=K, n_chains=96, burnin=burn, nrun=nrun, seed=4, horizons=(1, 12), precision=32,
             flags=H.FLAG_REF_Q1 | H.FLAG_SUMMARY)
    m = o.summary_mean[0]
    assert o.events == 0 and np.isfinite(m).all()
    outs, _ = oracle.gibbs_batch([dict(y=y[:600], K=K, burnin=burn, nrun=nrun, seed=8, chain=c, horizons=(1, 12),
                                       y_future=[y[600], y[611]]) for c in range(48)])
    om = np.concatenate([r.mu for r in outs]).mean(0)
    os2 = np.concatenate([r.sigma2 for r in outs]).mean(0)
    oA = np.concatenate([r.A for r in outs]).mean(0)
    ofc = np.concatenate([r.forecasts for r in outs]).mean(0)
    assert np.all(np.diff(m[0:K]) > 0)
    np.testing.assert_allclose(m[0:K], om, atol=0.35)
    np.testing.assert_allclose(m[K:2 * K], os2, rtol=0.35, atol=0.15)
    A = m[2 * K:2 * K + K * K].reshape(K, K).T                 # summary index s*K+r -> A[r, s]
    np.testing.assert_allclose(A, oA, atol=0.06)
    np.testing.assert_allclose(A.sum(1), 1.0, atol=1e-4)
    np.testing.assert_allclose(m[3 * K + K * K:3 * K + K * K + 4], ofc, atol=0.3)


@pytest.mark.parametrize("K", [12, 20])
def test_lane_kernel_fp32_posterior_and_loglik(H, ctx, oracle, K):
    """fp32 lane-per-state kernel (W = 16 for K = 12, W = 32 with the max-rescaled recursion for K = 20): pooled posterior
    means and the per-draw log-likelihood vs the oracle's."""
    tr = _truth(K)
    y, _ = synth_hmm(312, seed=3, **tr)
    burn, nrun = 200, 100
    o = _run(H, ctx, y, [1], [300], K=K, n_chains=64, burnin=burn, nrun=nrun, seed=4, horizons=(1, 12), precision=32,
             flags=H.FLAG_REF_Q1 | H.FLAG_SUMMARY | H.FLAG_DRAWS | H.FLAG_LOGLIK)
    m = o.summary_mean[0]
    assert o.events == 0 and np.isfinite(m).all()
    outs, _ = oracle.gibbs_batch([dict(y=y[:300], K=K, burnin=burn, nrun=nrun, seed=8, chain=c, horizons=(1, 12),
                                       y_future=[y[300], y[311]]) for c in range(32)])
    om = np.concatenate([r.mu for r in outs]).mean(0)
    oA = np.concatenate([r.A for r in outs]).mean(0)
    ofc = np.concatenate([r.forecasts for r in outs]).mean(0)
    oll = np.concatenate([r.loglik for r in outs])
    np.testing.assert_allclose(m[0:K], om, atol=0.4)
    A = m[2 * K:2 * K + K * K].reshape(K, K).T
    np.testing.assert_allclose(A, oA, atol=0.06)
    np.testing.assert_allclose(A.sum(1), 1.0, atol=1e-4)
    np.testing.assert_allclose(o.pi_end[0].sum(0), 1.0, atol=1e-4)
    np.testing.assert_allclose(m[3 * K + K * K:3 * K + K * K + 4], ofc, atol=0.4)
    assert abs(o.loglik[0].mean() - oll.mean()) < 0.02 * abs(oll.mean())
    # the log-likelihood of a draw is a deterministic function of its parameters: re-filter a few draws with the oracle
    for d in (0, 17, 63 * nrun + 5):
        mu, s2 = o.mu[0][:, d], o.sigma2[0][:, d]
        Ad = o.A[0][:, :, d].T                     # stored [s][r] -> A[r, s]
        lls = []
        for _ in range(1):
            f = oracle.forward(y[:300], Ad, mu, s2, np.full(K, 1.0 / K), want_Pf=False)
            lls.append(f.loglik)
        # rho of the draw is not returned: the first step's prior differs, everything else is identical
        assert abs(o.loglik[0][d] - lls[0]) < 6.0


@pytest.mark.parametrize("K", [3, 5, 8])
def test_insample_forecast_means(H, ctx, oracle, K):
    """forecastinsample (src/Hmc.jl:683-699): per-date posterior mean of pib[j,t,:]' A_j^h mu_j.  fp64 device chain vs the
    oracle chain on the same Philox streams (pib_full + per-draw mu, A from the oracle), plus an fp32 Monte-Carlo check.
    K = 5 and 8: the smoothed means of the thread-per-chain kernels with flushed transition counters (:442-457 has no K limit)."""
    y, _ = synth_hmm(172, **(K3_TRUTH if K == 3 else _truth(K)))
    hs = (1, 12)
    wins = ((1, 160), (5, 140))
    o = _run(H, ctx, y, [w[0] for w in wins], [w[1] for w in wins], K=K, n_chains=2, burnin=2, nrun=5, seed=11, horizons=hs,
             precision=64, flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SMOOTHED_MEAN)
    for w, (s, e) in enumerate(wins):
        n = e - s + 1
        ref_fc, ref_pib = np.zeros((n, len(hs))), np.zeros((n, K))
        for c in range(2):
            r = oracle.gibbs(y[s - 1:e], K, 2, 5, seed=11, chain=w * 2 + c, horizons=hs, y_future=[y[e - 1 + h] for h in hs],
                             flags=oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM, want_pib_full=True)
            for j in range(5):
                for k, h in enumerate(hs):
                    ref_fc[:, k] += r.pib_full[j] @ np.linalg.matrix_power(r.A[j], h) @ r.mu[j]
                ref_pib += r.pib_full[j]
        assert o.insample_forecast_mean[w].shape == (n, len(hs))
        np.testing.assert_allclose(o.insample_forecast_mean[w], ref_fc / 10, rtol=1e-7, atol=1e-9)
        np.testing.assert_allclose(o.pib_mean[w], ref_pib / 10, rtol=1e-6, atol=1e-10)
        # the last date's in-sample forecast is the end-of-window forecast
        np.testing.assert_allclose(o.insample_forecast_mean[w][-1], o.forecasts[w][0::2].mean(1), rtol=1e-9)
    # fp32, pooled chains: same quantity within Monte-Carlo error of the fp64 run
    a = _run(H, ctx, y, [1], [160], K=3, n_chains=64, burnin=300, nrun=200, seed=12, horizons=hs, precision=32,
             flags=H.FLAG_REF_Q1 | H.FLAG_SMOOTHED_MEAN | H.FLAG_SUMMARY)
    b = _run(H, ctx, y, [1], [160], K=3, n_chains=64, burnin=300, nrun=200, seed=13, horizons=hs, precision=64,
             flags=H.FLAG_REF_Q1 | H.FLAG_SMOOTHED_MEAN | H.FLAG_SUMMARY)
    assert np.abs(a.insample_forecast_mean[0] - b.insample_forecast_mean[0]).max() < 0.15
    np.testing.assert_allclose(a.insample_forecast_mean[0][-1], a.summary_mean[0][18:22:2], rtol=1e-4)


def test_filtered_mean_accumulator_matches_the_filter_entry_point(H, ctx):
    """HMCGPU_FLAG_FILTERED_MEAN against hmcgpu_filter on the SAME parameter draws (FLAG_DRAWS of the same call): the device sums
    must equal the mean over draws of the filtered rows up to the flat-prior rho the sampler redraws every sweep (:350-356; it
    only touches the first few rows), and the forecast sums the mean of pif' A^h mu.  K = 3 and K = 5, fp64 and fp32."""
    for K, prec, tol in ((3, 64, 1e-9), (3, 32, 2e-4), (5, 64, 1e-9)):
        tr = K3_TRUTH if K == 3 else _truth(K)
        y, _ = synth_hmm(180, seed=4 + K, **tr)
        hs = (1, 12)
        o = _run(H, ctx, y, [1, 11], [160, 150], K=K, n_chains=3, burnin=40, nrun=30, seed=3, horizons=hs, precision=prec,
                 flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_FILTERED_MEAN)
        assert o.events == 0
        for w, (s, e) in enumerate(((1, 160), (11, 150))):
            yw = y[s - 1:e]
            mu, s2 = o.mu[w].T, o.sigma2[w].T
            A = np.transpose(o.A[w], (2, 1, 0))
            R = len(mu)
            rho = np.full((R, K), 1.0 / K)
            pif = ctx.filter(yw, A, mu, s2, rho, precision=64, want_totals=False).pif            # [R, T, K], states already sorted
            skip = 60                                                                             # rows where the sampler's random rho still matters
            np.testing.assert_allclose(o.pib_mean[w][skip:], pif.mean(0)[skip:], atol=max(tol, 1e-6), rtol=0)
            np.testing.assert_allclose(o.pib_mean[w].sum(1), 1.0, atol=1e-5)
            for k, h in enumerate(hs):
                wv = np.einsum("brs,bs->br", np.linalg.matrix_power(A, h), mu)
                f = np.einsum("btk,bk->t", pif, wv) / R
                np.testing.assert_allclose(o.insample_forecast_mean[w][skip:, k], f[skip:], atol=max(10 * tol, 1e-5), rtol=0)
    with pytest.raises(H.HmcGpuError):
        _run(H, ctx, y, [1], [100], K=3, n_chains=1, burnin=1, nrun=1, flags=H.FLAG_FILTERED_MEAN | H.FLAG_SMOOTHED_MEAN)


def test_insample_filtered_table_matches_reference_publication(H, ctx):
    """forecastinsample(probabilities="filtered") on the GPU — ONE hmcgpu_estimate call whose forward pass accumulates the filtered
    rows and their forecasts over every saved draw (HMCGPU_FLAG_FILTERED_MEAN) — against the reference's published in-sample
    table, data/output/official_insample/forecats_insample.csv: its s1..s3 are posterior means of the filtered probabilities
    (tests/test_oracle.py::test_golden_insample_table_is_filtered)."""
    y, dates = load_inflation()
    g = json.load(open(os.path.join(GOLDEN, "official_insample.json")))
    N = g["last_index"]
    opt = H.EstOpt(y, dates, sampleRange=range(1, N + 1), endIndex=N, horizons=[12], D=3, burnin=2000, Nrun=1500, n_chains=8,
                   precision=32)
    t = H.forecastinsample(opt, ctx=ctx, probabilities="filtered")
    p = np.stack([t["s1"], t["s2"], t["s3"]], axis=1)
    np.testing.assert_allclose(p.sum(1), 1.0, atol=1e-5)
    d = np.abs(p - np.array(g["probs"])).max(1)
    assert np.median(d) < 2e-3 and (d < 0.03).mean() > 0.85 and d.max() < 0.25, (np.median(d), (d < 0.03).mean(), d.max())
    df = np.abs(t["forecast"] - np.array(g["forecast"]))
    assert np.median(df) < 0.03 and np.quantile(df, 0.99) < 0.5, (np.median(df), np.quantile(df, 0.99))
    ts = H.forecastinsample(opt, ctx=ctx, probabilities="smoothed")              # the smoothed table is a different object
    ds = np.abs(np.stack([ts["s1"], ts["s2"], ts["s3"]], axis=1) - np.array(g["probs"])).max(1)
    assert ds.mean() > 2 * d.mean() and ds[-1] < 5e-3


def test_complete_official_run_against_reference_summaries(H, ctx):
    """All 460 end dates of the reference's published run (data/output/official/*_summary.csv, real series) in one call.
    Typical agreement is ~1e-3; a few end dates have a bimodal posterior (e.g. idx 479: mu_3 near 8.25 or 10.45 — the
    oracle's long chain wanders between the modes too), where the mean depends on mixing, so the test is on quantiles."""
    y, dates = load_inflation()
    g = json.load(open(os.path.join(GOLDEN, "official_summary_all.json")))
    ends = np.array(g["end_index"], dtype=np.int32)
    assert len(ends) == 460 and dates[ends[0] - 1] == g["date"][0]
    o = H.estimate_windows(y, np.ones_like(ends), ends, K=3, n_chains=64, burnin=1500, nrun=1000, horizons=(12,), precision=32, ctx=ctx)
    m = o.summary_mean
    assert o.events == 0 and np.isfinite(m).all()
    d_mu = np.abs(m[:, 0:3] - np.array(g["filtered_means"])).max(1)
    d_s2 = np.abs(m[:, 3:6] / np.array(g["filtered_variances"]) - 1).max(1)
    d_A = np.abs(m[:, 6:15] - np.array(g["filtered_trans_probs"])).max(1)
    d_pi = np.abs(m[:, 15:18] - np.array(g["filtered_state_probs"])).max(1)
    ok = ends + 12 <= len(y)
    d_fc = np.abs(m[ok, 18] - np.array(g["forecasts"])[ok, 0])
    assert np.median(d_mu) < 0.01 and np.median(d_s2) < 0.01 and np.median(d_A) < 1e-3 and np.median(d_pi) < 1e-3
    assert np.median(d_fc) < 0.01
    assert (d_mu < 0.1).mean() > 0.85 and (d_A < 0.01).mean() > 0.9 and (d_fc < 0.1).mean() > 0.85


# ---------------------------------------------------------------------------------------------------------------------
# signals tier (SURVEY section 8f-2): signal mask, kappa-weighted statistics, user X0, init series, pi_row_back

def _signal_case(T=180, extra=12):
    y, _ = synth_hmm(T + extra, **K3_TRUTH)
    mask = np.zeros(len(y), dtype=np.uint8)
    mask[T - 6:T] = 1            # a block of signals at the end of the window (run_hmm.jl:146-148) ...
    mask[[20, 21, 77]] = 1       # ... and a few inside it
    return y, mask


@pytest.mark.parametrize("kappa", [0.0, 0.6, 3.0])
def test_signals_first_sweeps_follow_the_oracle_chain(H, ctx, oracle, kappa):
    """fp64 device chain with a signal mask vs the oracle chain on the same Philox streams (src/Hmc.jl:267-314, :380-383),
    HyperParams(opt) priors (alpha = nu = 2, :148-159), and the smoothed row N - back as pi_end (:893)."""
    T = 180
    y, mask = _signal_case(T)
    hs = (0, 1, 6)
    two, xi = np.full(3, 2.0), np.full(3, 3.21)
    back = 6
    o = _run(H, ctx, y, [1], [T], K=3, n_chains=2, burnin=2, nrun=7, seed=99, horizons=hs, precision=64,
             flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK, is_signal=mask, kappa=kappa, alpha=two, nu=two, xi=xi,
             pi_row_back=back)
    assert o.events == 0
    for c in range(2):
        yf = [y[T - 1 + h] for h in hs]
        r = oracle.gibbs(y[:T], 3, 2, 7, seed=99, chain=c, horizons=hs, y_future=yf, is_signal=mask[:T], kappa=kappa,
                         alpha=two, nu=two, xi=xi, flags=oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM, want_pib_full=True)
        sl = slice(c * 7, (c + 1) * 7)
        np.testing.assert_allclose(o.mu[0][:, sl].T, r.mu, rtol=1e-8)
        np.testing.assert_allclose(o.sigma2[0][:, sl].T, r.sigma2, rtol=1e-8)
        np.testing.assert_allclose(np.transpose(o.A[0][:, :, sl], (2, 1, 0)), r.A, rtol=1e-8)
        np.testing.assert_allclose(o.pi_end[0][:, sl].T, r.pib_full[:, T - 1 - back, :], rtol=1e-7, atol=1e-12)
        np.testing.assert_allclose(o.forecasts[0][:, sl].T, r.forecasts, rtol=1e-8, atol=1e-9)
        np.testing.assert_allclose(o.loglik[0][sl], r.loglik, rtol=1e-9)
        # horizon 0 = pib[N,:]' mu
        np.testing.assert_allclose(o.forecasts[0][0, sl], (r.pi_end * r.mu).sum(1), rtol=1e-8)


def test_signals_every_step_a_signal_and_ragged_batch(H, ctx, oracle):
    """run_hmm.jl:170-172 (`Make everything a signal`) and windows of different lengths in one warp task."""
    y, _ = synth_hmm(160, **K3_TRUTH)
    mask = np.ones(len(y), dtype=np.uint8)
    ws, we = [1, 11, 3], [150, 120, 43]
    o = _run(H, ctx, y, ws, we, K=3, n_chains=1, burnin=1, nrun=5, seed=5, horizons=(1,), precision=64,
             flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS, is_signal=mask, kappa=0.6)
    for w, (s, e) in enumerate(zip(ws, we)):
        r = oracle.gibbs(y[s - 1:e], 3, 1, 5, seed=5, chain=w, horizons=(1,), y_future=[y[e]], is_signal=mask[s - 1:e],
                         kappa=0.6, flags=oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM)
        np.testing.assert_allclose(o.mu[w].T, r.mu, rtol=1e-8)
        np.testing.assert_allclose(o.sigma2[w].T, r.sigma2, rtol=1e-8)
        np.testing.assert_allclose(o.pi_end[w].T, r.pi_end, rtol=1e-7, atol=1e-12)


def test_signals_per_series_masks_and_long_window(H, ctx, oracle):
    """One mask per series (many end dates, each with its own signalRange, in one call: y is streamed per chain) and a
    window long enough for the 64-bit packed transition counters (T > 1023 at K = 3)."""
    rng = np.random.default_rng(3)
    y0, _ = synth_hmm(1312, **K3_TRUTH)
    ends = [1300, 1180, 90]
    ys = np.stack([y0 + (rng.normal(0, 0.7, size=len(y0)) if i else 0.0) for i in range(3)])
    mask = np.zeros_like(ys, dtype=np.uint8)
    for i, e in enumerate(ends):
        mask[i, e - 12:e] = 1
        mask[i, 5 + i] = 1
    two = np.full(3, 2.0)
    o = _run(H, ctx, ys, [1, 1, 1], ends, K=3, n_chains=2, burnin=1, nrun=3, seed=21, horizons=(0, 12), precision=64,
             flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK, win_series=[0, 1, 2], is_signal=mask, kappa=0.8, alpha=two, nu=two,
             pi_row_back=12)
    assert o.events == 0
    for w, e in enumerate(ends):
        for c in range(2):
            r = oracle.gibbs(ys[w, :e], 3, 1, 3, seed=21, chain=w * 2 + c, horizons=(0, 12), y_future=[ys[w, e - 1], ys[w, e + 11]],
                             is_signal=mask[w, :e], kappa=0.8, alpha=two, nu=two, flags=oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM,
                             want_pib_full=True)
            sl = slice(c * 3, (c + 1) * 3)
            np.testing.assert_allclose(o.mu[w][:, sl].T, r.mu, rtol=1e-7)
            np.testing.assert_allclose(o.sigma2[w][:, sl].T, r.sigma2, rtol=1e-7)
            np.testing.assert_allclose(np.transpose(o.A[w][:, :, sl], (2, 1, 0)), r.A, rtol=1e-7)
            np.testing.assert_allclose(o.pi_end[w][:, sl].T, r.pib_full[:, e - 13, :], rtol=1e-6, atol=1e-12)
            np.testing.assert_allclose(o.loglik[w][sl], r.loglik, rtol=1e-9)


def test_user_initial_states_and_init_series(H, ctx, oracle):
    """X0 supplied by the caller, and makeParams / HyperParams read from another series than the chain runs on
    (estimatesignals! initialises from the real sample and estimates on the perturbed copy, src/Hmc.jl:888-892)."""
    rng = np.random.default_rng(8)
    T = 140
    y, _ = synth_hmm(T + 2, **K3_TRUTH)
    X0 = rng.integers(1, 4, size=T)
    o = _run(H, ctx, y, [1], [T], K=3, n_chains=1, burnin=1, nrun=5, seed=11, horizons=(1,), precision=64,
             flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS, X0=X0)
    r = oracle.gibbs(y[:T], 3, 1, 5, seed=11, chain=0, horizons=(1,), y_future=[y[T]], X0=X0,
                     flags=oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM)
    np.testing.assert_allclose(o.mu[0].T, r.mu, rtol=1e-8)
    np.testing.assert_allclose(o.sigma2[0].T, r.sigma2, rtol=1e-8)
    # series 1 = perturbed copy; X0 and xi come from series 0
    yp = y.copy()
    yp[T - 5:T] += rng.normal(0, 1.5, size=5)
    mask = np.zeros(len(y), dtype=np.uint8); mask[T - 5:T] = 1
    o = _run(H, ctx, np.stack([y, yp]), [1], [T], K=3, n_chains=1, burnin=1, nrun=5, seed=11, horizons=(1,), precision=64,
             flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS, win_series=[1], win_init_series=[0], is_signal=mask, kappa=0.3)
    X0r, _, _ = oracle.make_params(y[:T], 3)
    r = oracle.gibbs(yp[:T], 3, 1, 5, seed=11, chain=0, horizons=(1,), y_future=[yp[T]], X0=X0r, xi=np.full(3, y[:T].mean()),
                     is_signal=mask[:T], kappa=0.3, flags=oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM)
    np.testing.assert_allclose(o.mu[0].T, r.mu, rtol=1e-8)
    np.testing.assert_allclose(o.sigma2[0].T, r.sigma2, rtol=1e-8)
    np.testing.assert_allclose(o.pi_end[0].T, r.pi_end, rtol=1e-7, atol=1e-12)
    with pytest.raises(H.HmcGpuError):
        _run(H, ctx, y, [1], [T], K=3, X0=np.full(T, 4))


@pytest.mark.parametrize("precision", [64, 32])
def test_signals_posterior_matches_oracle_posterior(H, ctx, oracle, precision):
    """Monte-Carlo parity of the signal-aware sampler: pooled posterior moments vs the oracle's, 12 signals at the end."""
    T = 300
    y, _ = synth_hmm(T + 12, **K3_TRUTH)
    mask = np.zeros(len(y), dtype=np.uint8); mask[T - 12:T] = 1
    two = np.full(3, 2.0)
    nch, burn, nrun = 64, 400, 400
    o = _run(H, ctx, y, [1], [T], K=3, n_chains=nch, burnin=burn, nrun=nrun, seed=7, horizons=(1, 12), precision=precision,
             flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY, is_signal=mask, kappa=1.0, alpha=two, nu=two, pi_row_back=12)
    assert o.events == 0
    outs, _ = oracle.gibbs_batch([dict(y=y[:T], K=3, burnin=burn, nrun=nrun, seed=70, chain=c, horizons=(1, 12),
                                       y_future=[y[T], y[T + 11]], is_signal=mask[:T], kappa=1.0, alpha=two, nu=two,
                                       want_pib_full=True) for c in range(12)])
    cat = lambda k: np.concatenate([getattr(r, k) for r in outs])
    om, os2, oA, ofc = cat("mu"), cat("sigma2"), cat("A"), cat("forecasts")
    opb = np.concatenate([r.pib_full[:, T - 13, :] for r in outs])

    def close(g, ref, name):
        se = 4 * np.sqrt(ref.var(0) / len(ref) + g.var(0) / len(g))
        d = np.abs(g.mean(0) - ref.mean(0))
        assert np.all(d <= 5 * se + 1e-4), (name, d, se)

    close(o.mu[0].T, om, "mu")
    close(o.sigma2[0].T, os2, "sigma2")
    close(np.transpose(o.A[0], (2, 1, 0)).reshape(-1, 9), oA.reshape(-1, 9), "A")
    close(o.pi_end[0].T, opb, "pib[N-12]")
    close(o.forecasts[0].T, ofc, "forecasts")
    F = np.concatenate([o.mu[0], o.sigma2[0], o.A[0].reshape(9, -1), o.pi_end[0], o.forecasts[0]])
    np.testing.assert_allclose(o.summary_mean[0][:-1], F.mean(1), rtol=1e-6, atol=1e-7)


def test_estimatesignals_mirror(H, ctx, tmp_path):
    """Hmc.estimatesignals! (src/Hmc.jl:868-914) through the host mirror: shapes, signal bookkeeping, forecast rules
    (:900-906) and the hassignals CSV layout (:707-721, :733-741)."""
    y, _ = synth_hmm(260, **K3_TRUTH)
    end, sigLen = 200, 12
    opt = H.EstOpt(y, list(range(1, 261)), sampleRange=range(1, end + sigLen + 1), signalRange=range(end + 1, end + sigLen + 1),
                   signalSave=range(end + 1, end + sigLen + 1), endIndex=end, horizons=[12, 24], D=3, burnin=300, Nrun=300,
                   signalburnin=300, signalNrun=200, noise=1.0, noiseSamples=16, precision=32, series="test")
    assert opt.σsignal == 0.0
    s = H.estimatesignals(opt, ctx)
    # :869-872: a zero σsignal is set IN PLACE to mean(σ²-draws of a plain estimatemodel run) x noise before anything else happens
    base = H.estimatemodel(H.EstOpt(y, list(range(1, 261)), sampleRange=range(1, end + sigLen + 1), signalRange=range(end + 1, end + sigLen + 1),
                                    signalSave=range(end + 1, end + sigLen + 1), endIndex=end, horizons=[12, 24], D=3, burnin=300, Nrun=300,
                                    signalburnin=300, signalNrun=200, noise=1.0, noiseSamples=16, precision=32, series="test"), ctx)
    assert opt.σsignal == float(base.σ.mean() * opt.noise) and s.σsignal == opt.σsignal
    n = 16 * 200
    assert s.μ.shape == (n, 3) and s.σ.shape == (n, 3) and s.πb.shape == (n, 3) and s.A.shape == (n, 3, 3)
    assert s.forecasts.shape == (n, 4) and s.signalvals.shape == (n, 12) and s.signalids.tolist() == np.repeat(np.arange(1, 17), 200).tolist()
    assert opt.σsignal > 0 and s.events == 0
    np.testing.assert_allclose(s.πb.sum(1), 1.0, atol=1e-4)
    assert np.all(np.diff(s.μ, axis=1) > 0)
    # signal values are the perturbed series, constant within a copy, different across copies
    assert np.ptp(s.signalvals[:200], axis=0).max() == 0 and np.ptp(s.signalvals[::200], axis=0).min() > 0
    sd = (s.signalvals[::200] - y[end:end + sigLen]).std()
    assert 0.6 * opt.σsignal < sd < 1.4 * opt.σsignal
    # h = 12 = sigLen: forecastsignal (:670-681) is an average of the signal and the state means
    a = (1 / opt.σsignal) / (1 + 1 / opt.σsignal)
    sig12 = s.signalvals[:, 11]
    f0 = (s.forecasts[:, 0] - a * sig12) / (1 - a)
    assert np.all(f0 > s.μ[:, 0] - 1e-3) and np.all(f0 < s.μ[:, 2] + 1e-3)
    np.testing.assert_allclose(s.forecasts[:, 1], s.forecasts[:, 0] - y[end + 12 - 1], atol=1e-4)
    # h = 24 > sigLen: 12 steps past the window end, scored against y[end + 24]
    np.testing.assert_allclose(s.forecasts[:, 3], s.forecasts[:, 2] - y[end + 24 - 1], atol=1e-4)
    paths = H.saveresults(s, opt, str(tmp_path), hassignals=True)
    head = open(paths["filtered_means"]).readline().strip().split(",")
    assert head == ["date", "signalid", "state_1", "state_2", "state_3"] + [f"signal_{i}" for i in range(1, 13)]
    row = open(paths["forecasts"]).readlines()[1].strip().split(",")
    assert row[1] == "1" and len(row) == 2 + 4 + 12


@pytest.mark.parametrize("noise", [0.1, 0.3, 0.6])
@pytest.mark.parametrize("end_index", [121, 200, 300, 450, 570])
def test_estimatesignals_matches_reference_golden_dispersion(H, ctx, end_index, noise):
    """The whole noisy-signal Monte Carlo through the host mirror (EstOpt -> estimatesignals -> calcdispersion) against
    the reference's OWN outputs, data/output/signals_official_noise_<noise>_allsignal/*_dispersion.csv (the "make
    everything a signal" block of code/run_hmm.jl:160-176: 100 perturbed copies per end date).  Same tolerances as the
    oracle's check of the same goldens (tests/test_oracle.py::test_golden_signal_dispersion); fp32 kernels."""
    y, dates, case, ssig = signals_golden_case(end_index, noise)
    rng_all = range(1, end_index + 1)
    opt = H.EstOpt(y, dates, sampleRange=rng_all, signalRange=rng_all, signalSave=range(end_index - 1, end_index + 1),
                   endIndex=end_index, horizons=[12], D=3, signalburnin=1500, signalNrun=500, noise=noise, noiseSamples=100,
                   σsignal=ssig, n_chains=8, precision=32)
    s = H.estimatesignals(opt, ctx, rng=np.random.default_rng(1234))
    assert s.events == 0 and s.μ.shape == (100 * 8 * 500, 3)
    assert abs(s.signalvals[::4000].std(0, ddof=1).mean() / ssig - 1) < 0.25          # the copies carry the injected noise level
    _, per_copy = H.signal_summaries(s)
    dispersion_close(per_copy["filtered_means"], case["filtered_means"], "mu", atol=0.02)
    dispersion_close(per_copy["filtered_variances"], case["filtered_variances"], "sigma2", atol=0.25 * ssig ** 2 / (1 + noise))
    dispersion_close(per_copy["filtered_state_probs"], case["filtered_state_probs"], "pi_end")
    dispersion_close(per_copy["filtered_trans_probs"], case["filtered_trans_probs"], "A")
    dispersion_close(per_copy["forecasts"], case["forecasts"], "forecasts", atol=0.02)
    disp = H.calcdispersion(s)                                                          # the table aggregate.jl writes
    np.testing.assert_allclose(disp["filtered_means"][0], per_copy["filtered_means"].mean(0))


def test_differential_fuzz_of_the_two_sweep_kernels():
    """Random shapes (K, ragged windows, chains, signal masks, kappa, pi_row_back, user X0) through the time-parallel and the
    thread-per-chain kernels in fp64: identical chains (scripts/fuzz_kernels.py; 300 cases were run when it was written)."""
    import subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "scripts", "fuzz_kernels.py"), "40", "7"], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
