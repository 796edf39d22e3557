"""CPU tests: the oracle (oracle/hmc_oracle.c) against known answers, an independent numpy/scipy restatement,
the reference's own test tolerances (test/runtests.jl:56-57) and the reference's golden posterior summaries."""
import json
import os

import numpy as np
import pytest
from scipy.special import logsumexp
from scipy.stats import norm

from conftest import GOLDEN, K3_TRUTH, dispersion_close, load_inflation, random_params, signals_golden_case, synth_hmm


def test_philox_known_answers(oracle):
    # Random123 kat_vectors for philox4x32-10
    assert oracle.philox([0, 0, 0, 0], [0, 0]) == [0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8]
    assert oracle.philox([0xffffffff] * 4, [0xffffffff] * 2) == [0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd]
    assert oracle.philox([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0]) == \
        [0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1]
    # Random123 kat_vectors for philox4x32-7: the round count of the STATES stream (backward-sampler uniforms)
    assert oracle.philox([0, 0, 0, 0], [0, 0], rounds=7) == [0x5f6fb709, 0x0d893f64, 0x4f121f81, 0x4f730a48]
    assert oracle.philox([0xffffffff] * 4, [0xffffffff] * 2, rounds=7) == [0x5207ddc2, 0x45165e59, 0x4d8ee751, 0x8c52f662]
    assert oracle.philox([0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344], [0xa4093822, 0x299f31d0], rounds=7) == \
        [0x4dfccaba, 0x190a87f0, 0xc47362ba, 0xb6b5242a]


def numpy_filter(y, A, mu, sigma2, rho):
    """Independent log-space forward filter (scipy.stats.norm.logpdf + logsumexp)."""
    T, K = len(y), len(mu)
    logp = norm.logpdf(y[:, None], mu[None, :], np.sqrt(sigma2)[None, :])
    la = np.log(A)
    pif = np.zeros((T, K))
    ll = 0.0
    prev = np.log(rho)
    for t in range(T):
        joint = prev[:, None] + la + logp[t][None, :]
        tot = logsumexp(joint)
        ll += tot
        prev = logsumexp(joint, axis=0) - tot
        pif[t] = np.exp(prev)
    return pif, ll


@pytest.mark.parametrize("K", [2, 3, 4])
def test_forward_matches_numpy(oracle, K):
    rng = np.random.default_rng(7 + K)
    A, mu, s2, rho = (v[0] for v in random_params(rng, 1, K))
    y = rng.normal(0, 3, size=300)
    f = oracle.forward(y, A, mu, s2, rho)
    pif, ll = numpy_filter(y, A, mu, s2, rho)
    np.testing.assert_allclose(f.pif, pif, rtol=1e-9, atol=1e-300)
    assert abs(f.loglik - ll) < 1e-8 * abs(ll)
    np.testing.assert_allclose(f.pif.sum(1), 1.0, atol=1e-12)
    np.testing.assert_allclose(f.Pf.sum((1, 2)), 1.0, atol=1e-12)
    assert abs(np.log(f.totals).sum() - f.loglik) < 1e-9


@pytest.mark.parametrize("kappa", [0.0, 0.6, 3.0])
def test_forward_signal_rows_match_numpy(oracle, kappa):
    """Signal rows are emitted with sd*(1+kappa) (src/Hmc.jl:382, :396, :424), observation rows with sd."""
    rng = np.random.default_rng(21)
    K = 3
    A, mu, s2, rho = (v[0] for v in random_params(rng, 1, K))
    y = rng.normal(0, 3, size=120)
    mask = np.zeros(len(y), dtype=np.uint8)
    mask[[0, 5, 6, 50]] = 1
    mask[-12:] = 1                                           # the reference's layout: signals after the end date (+ row 1)
    f = oracle.forward(y, A, mu, s2, rho, is_signal=mask, kappa=kappa)
    sd = np.sqrt(s2)[None, :] * np.where(mask[:, None] != 0, 1.0 + kappa, 1.0)
    logp = norm.logpdf(y[:, None], mu[None, :], sd)
    prev, ll, pif = np.log(rho), 0.0, np.zeros((len(y), K))
    for t in range(len(y)):
        joint = prev[:, None] + np.log(A) + logp[t][None, :]
        tot = logsumexp(joint)
        ll += tot
        prev = logsumexp(joint, axis=0) - tot
        pif[t] = np.exp(prev)
    np.testing.assert_allclose(f.pif, pif, rtol=1e-9, atol=1e-300)
    assert abs(f.loglik - ll) < 1e-8 * abs(ll)
    if kappa == 0.0:                                         # kappa = 0: a signal is an observation
        np.testing.assert_array_equal(f.pif, oracle.forward(y, A, mu, s2, rho).pif)


def test_shortest_window_and_single_step_filter(oracle):
    """Edge sizes: T = 1 for the deterministic pieces, T = 2 for a whole chain (the shortest window the library accepts)."""
    rng = np.random.default_rng(2)
    A, mu, s2, rho = (v[0] for v in random_params(rng, 1, 3))
    f = oracle.forward(np.array([0.7]), A, mu, s2, rho)
    joint = rho[:, None] * A * norm.pdf(0.7, mu, np.sqrt(s2))[None, :]
    np.testing.assert_allclose(f.Pf[0], joint / joint.sum(), rtol=1e-12)
    np.testing.assert_allclose(f.totals[0], joint.sum(), rtol=1e-12)
    X = oracle.sample_states(f.pif, A, np.array([0.999999]), form=1)
    assert X.tolist() == [3]
    o = oracle.gibbs(np.array([1.0, 4.0]), 2, 5, 20, seed=3, horizons=(0, 1), y_future=[4.0, np.nan])
    assert o.mu.shape == (20, 2) and np.isfinite(o.mu).all() and np.isfinite(o.sigma2).all() and (o.sigma2 > 0).all()
    np.testing.assert_allclose(o.A.sum(2), 1.0, atol=1e-12)
    np.testing.assert_allclose(o.pi_end.sum(1), 1.0, atol=1e-12)
    np.testing.assert_allclose(o.forecasts[:, 0], (o.pi_end * o.mu).sum(1), rtol=1e-12)      # horizon 0 = pi_end' mu
    assert np.isnan(o.forecasts[:, 3]).all()                                                   # no realised value: NaN error


def test_categorical_convention_and_zero_normaliser_fallback(oracle):
    """rand(Categorical(p)) = first i with cumsum_i >= u; rows whose normaliser is <= eps() fall back to 1/D (:472-480)."""
    K = 3
    A = np.array([[0.0, 0.5, 0.5], [0.0, 0.5, 0.5], [0.0, 0.5, 0.5]])      # no path INTO state 1
    pif = np.array([[0.2, 0.3, 0.5], [1.0, 0.0, 0.0]])                     # ... but X[2] = 1 is forced by piN
    for u0, want in ((0.0, 1), (0.3, 1), (0.34, 2), (0.66, 2), (0.67, 3), (0.999, 3)):
        X = oracle.sample_states(pif, A, np.array([u0, 0.5]), form=1)
        assert X.tolist() == [want, 1], (u0, X)
    # regular rows: boundaries of the cumulative sums of pif[0] * A[:, x] normalised
    A2 = np.array([[0.5, 0.25, 0.25], [0.1, 0.8, 0.1], [0.3, 0.3, 0.4]])
    pif2 = np.array([[0.2, 0.3, 0.5], [0.0, 1.0, 0.0]])
    w = pif2[0] * A2[:, 1]
    c = np.cumsum(w / w.sum())
    for u0 in (0.0, c[0] - 1e-9, c[0] + 1e-9, c[1] - 1e-9, c[1] + 1e-9, 0.999999):
        X = oracle.sample_states(pif2, A2, np.array([u0, 0.5]), form=1)
        assert X[1] == 2 and X[0] == 1 + int(np.searchsorted(c, u0, side="left")), (u0, X)


def test_backward_forms_agree_and_match_numpy(oracle):
    rng = np.random.default_rng(3)
    K = 3
    A, mu, s2, rho = (v[0] for v in random_params(rng, 1, K))
    y = rng.normal(0, 3, size=200)
    f = oracle.forward(y, A, mu, s2, rho)
    Pb, pib = oracle.backward(f.Pf, f.pif)
    pib2 = oracle.backward_pif(A, f.pif)
    np.testing.assert_allclose(pib, pib2, rtol=1e-9, atol=1e-14)
    # independent forward-backward: beta recursion
    logp = norm.pdf(y[:, None], mu[None, :], np.sqrt(s2)[None, :])
    T = len(y)
    beta = np.ones((T, K))
    for t in range(T - 2, -1, -1):
        beta[t] = A @ (logp[t + 1] * beta[t + 1])
        beta[t] /= beta[t].sum()
    sm = f.pif * beta
    sm /= sm.sum(1, keepdims=True)
    np.testing.assert_allclose(pib, sm, rtol=1e-8, atol=1e-13)


def test_sample_states_forms_give_same_paths(oracle):
    rng = np.random.default_rng(5)
    K = 3
    A, mu, s2, rho = (v[0] for v in random_params(rng, 1, K))
    y = rng.normal(0, 3, size=400)
    f = oracle.forward(y, A, mu, s2, rho)
    for rep in range(20):
        u = rng.random(len(y))
        X0 = oracle.sample_states(f.pif, A, u, Pf=f.Pf, form=0)
        X1 = oracle.sample_states(f.pif, A, u, form=1)
        assert X0.min() >= 1 and X0.max() <= K
        assert (X0 == X1).all()


def test_sample_states_distribution(oracle):
    # the marginal of many sampled paths must equal the smoothed probabilities
    rng = np.random.default_rng(11)
    K = 3
    A, mu, s2, rho = (v[0] for v in random_params(rng, 1, K))
    y = rng.normal(0, 3, size=30)
    f = oracle.forward(y, A, mu, s2, rho)
    pib = oracle.backward_pif(A, f.pif)
    n = 20000
    counts = np.zeros((len(y), K))
    for _ in range(n):
        X = oracle.sample_states(f.pif, A, rng.random(len(y)), form=1)
        counts[np.arange(len(y)), X - 1] += 1
    assert np.abs(counts / n - pib).max() < 4 * 0.5 / np.sqrt(n)


def test_forecast_matches_numpy(oracle):
    rng = np.random.default_rng(13)
    for K in (2, 3, 4):
        A, mu, s2, rho = (v[0] for v in random_params(rng, 1, K))
        for h in (1, 2, 5, 12, 13):
            f, e = oracle.forecast(mu, A, rho, h, 1.25)
            ref = rho @ np.linalg.matrix_power(A, h) @ mu
            assert abs(f - ref) < 1e-12 * max(1, abs(ref)) and abs(e - (ref - 1.25)) < 1e-12 * max(1, abs(ref))


def test_gamma_normal_moments(oracle):
    for shape in (0.5, 1.0, 2.5, 50.0):
        g = np.array([oracle.gamma(shape, 99, c, 3, (2 << 16)) for c in range(40000)])
        assert abs(g.mean() - shape) < 5 * np.sqrt(shape / len(g))
        assert abs(g.var() - shape) < 0.08 * shape


def test_draw_params_moments(oracle):
    K = 3
    Ni, S, S2 = np.array([50, 100, 10]), np.array([80.0, 350.0, 83.0]), np.array([40.0, 55.0, 79.0])
    trans = np.array([[45, 3, 2], [4, 90, 6], [2, 3, 5]]) + 1
    xi, one = np.full(K, 3.2), np.ones(K)
    n = 8000
    out = [oracle.draw_params(Ni, S, S2, trans, xi, one, one, 2 * one, 1234, c, 7) for c in range(n)]
    s2 = np.array([o[0] for o in out]); mu = np.array([o[1] for o in out]); rho = np.array([o[2] for o in out]); A = np.array([o[3] for o in out])
    ybar = S / Ni
    a = 1 + 0.5 * Ni
    b = 2 + 0.5 * S2 + 0.5 * Ni / (Ni + 1) * (ybar - xi) ** 2
    np.testing.assert_allclose(s2.mean(0), b / (a - 1), rtol=0.03)               # mean of InverseGamma(a,b)
    np.testing.assert_allclose(mu.mean(0), (S + xi) / (Ni + 1), atol=0.02)
    np.testing.assert_allclose(rho.mean(0), 1 / 3, atol=0.01)
    np.testing.assert_allclose(A.mean(0), trans / trans.sum(1, keepdims=True), atol=0.01)
    np.testing.assert_allclose(A.sum(2), 1.0, atol=1e-12)


def test_make_params_rule(oracle):
    y, _ = synth_hmm(300, **K3_TRUTH)
    X, mu0, sd0 = oracle.make_params(y, 3)
    R = y.max() - y.min()
    np.testing.assert_allclose(mu0, np.linspace(np.median(y) - 0.25 * R, np.median(y) + 0.25 * R, 3))
    assert abs(sd0 - y.std(ddof=1)) < 1e-12
    np.testing.assert_array_equal(X, np.argmin(np.abs(y[:, None] - mu0[None, :]), axis=1) + 1)


def test_reference_integration_test(oracle):
    """test/runtests.jl:20-57: D=2, T=500, sampleRange=1:476, burnin 3000, Nrun 1000; atol 0.3 (mu), 0.5 (sigma)."""
    y, _ = synth_hmm(500, [[0.5, 0.5], [0.2, 0.8]], [-5.0, 4.0], [1.0, 0.5], seed=123)
    o = oracle.gibbs(y[:476], 2, 3000, 1000, seed=1234, horizons=(12,), y_future=[y[476 + 11]])
    assert np.all(np.abs(o.mu.mean(0) - [-5.0, 4.0]) < 0.3)
    assert np.all(np.abs(o.sigma2.mean(0) - [1.0, 0.5]) < 0.5)
    assert o.n_events == 0
    assert np.all(np.diff(o.mu, axis=1) > 0)                 # draws are emitted in increasing-mu order (:501-513)
    np.testing.assert_allclose(o.A.sum(2), 1.0, atol=1e-12)
    np.testing.assert_allclose(o.forecasts[:, 1], o.forecasts[:, 0] - y[476 + 11], atol=1e-12)


def test_gibbs_deterministic_and_batch(oracle):
    y, _ = synth_hmm(200, **K3_TRUTH)
    a = oracle.gibbs(y, 3, 50, 50, seed=5, chain=3)
    b = oracle.gibbs(y, 3, 50, 50, seed=5, chain=3)
    c = oracle.gibbs(y, 3, 50, 50, seed=5, chain=4)
    np.testing.assert_array_equal(a.mu, b.mu)
    assert not np.array_equal(a.mu, c.mu)
    outs, used = oracle.gibbs_batch([dict(y=y, K=3, burnin=50, nrun=50, seed=5, chain=ch) for ch in (3, 4)], n_threads=2)
    np.testing.assert_array_equal(outs[0].mu, a.mu)
    np.testing.assert_array_equal(outs[1].mu, c.mu)
    assert used == 2
    # the pif form of the backward sampler follows the same chain (identical paths up to measure-zero rounding ties)
    d = oracle.gibbs(y, 3, 50, 50, seed=5, chain=3, flags=oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM)
    np.testing.assert_allclose(d.mu, a.mu, rtol=1e-9)


def test_state_margins_recomputed_from_the_first_sweep(oracle):
    """want_margins: state_margin[0] is the distance of the sweep-0 STATES uniforms from the nearest cumulative boundary of the
    categoricals they were compared with.  Recomputed here from the chain's own sweep-0 parameters (makeParams statistics ->
    draw_params in chain labels -> forward), the uniforms of the Philox-7 stream and the sampled path; moving every u by half
    the margin keeps the path, moving the closest one 1.5 margins towards its boundary changes it."""
    K, seed, chain = 3, 17, 5
    y, _ = synth_hmm(150, seed=2, **K3_TRUTH)
    N = len(y)
    flags = oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM
    r = oracle.gibbs(y, K, 0, 1, seed=seed, chain=chain, flags=flags, want_margins=True)
    assert oracle.gibbs(y, K, 0, 1, seed=seed, chain=chain, flags=flags).state_margin is None
    assert r.state_margin.shape == (1,) and r.gamma_margin.shape == (1,)
    assert 0 < r.gamma_margin[0] < np.inf
    # sweep 0 in chain labels, as the oracle computes it
    X0, _, _ = oracle.make_params(y, K)
    st = X0 - 1
    Ni = np.bincount(st, minlength=K)
    S = np.array([sum(y[st == k]) for k in range(K)])       # (sequential sums, as the oracle adds)
    ybar = np.where(Ni > 0, S / np.maximum(Ni, 1), 0.0)
    S2 = np.array([sum((y[st == k] - ybar[k]) ** 2) for k in range(K)])
    trans = np.ones((K, K), dtype=np.int64)
    np.add.at(trans, (st[:-1], st[1:]), 1)
    one = np.ones(K)
    s2, mu, rho, A = oracle.draw_params(Ni, S, S2, trans, np.full(K, sum(y) / N), one, one, one, seed, chain, 0)
    order = np.argsort(mu, kind="stable")
    np.testing.assert_array_equal(r.mu[0], mu[order])
    pif = oracle.forward(y, A, mu, s2, rho, want_Pf=False).pif
    piN = pif[-1][order]                                    # quirk Q1: X[N] drawn from the relabelled row
    u = np.zeros(N)
    for i in range(0, N, 4):
        w = oracle.philox([i >> 2, oracle.KIND_STATES << 16, 0, chain], [seed & 0xFFFFFFFF, seed >> 32], rounds=7)
        for j in range(min(4, N - i)):
            u[N - 1 - (i + j)] = (w[j] + 0.5) * 2.0 ** -32
    X = oracle.sample_states(pif, A, u, piN=piN, form=1)
    np.testing.assert_array_equal(X, r.X_final)
    m, side = np.zeros(N), np.zeros(N)                     # per-step margin and the direction of the nearest boundary
    for t in range(N - 1, -1, -1):
        if t == N - 1:
            p = piN
        else:
            x = X[t + 1] - 1
            p = pif[t] * A[:, x]
            p = p / p.sum() if pif[t + 1, x] > np.finfo(float).eps and p.sum() > 0 else np.full(K, 1.0 / K)
        d = u[t] - np.cumsum(p)[:K - 1]
        j = np.argmin(np.abs(d))
        m[t], side[t] = abs(d[j]), np.sign(d[j])
    np.testing.assert_allclose(m.min(), r.state_margin[0], rtol=1e-12)
    for s in (-0.5, 0.5):
        np.testing.assert_array_equal(oracle.sample_states(pif, A, u + s * m.min(), piN=piN, form=1), X)
    t = int(np.argmin(m))
    v = u.copy()
    v[t] -= side[t] * 1.5 * m[t]
    assert oracle.sample_states(pif, A, v, piN=piN, form=1)[t] != X[t]


@pytest.mark.parametrize("which", [0, 9, 18])
def test_golden_posterior_summaries(oracle, which):
    """The oracle reproduces the reference's own posterior means (data/output/official/*_summary.csv, 250k draws
    after 100k burn-in) on the real series within Monte-Carlo tolerance."""
    y, dates = load_inflation()
    g = json.load(open(os.path.join(GOLDEN, "official_summary_subset.json")))["windows"][which]
    idx = g["end_index"]
    assert dates[idx - 1] == g["date"]
    yf = [y[idx - 1 + 12]] if idx - 1 + 12 < len(y) else [np.nan]
    outs, _ = oracle.gibbs_batch([dict(y=y[:idx], K=3, burnin=3000, nrun=6000, seed=1234, chain=c, horizons=(12,), y_future=yf)
                                  for c in range(4)])
    mu = np.concatenate([o.mu for o in outs]).mean(0)
    s2 = np.concatenate([o.sigma2 for o in outs]).mean(0)
    A = np.concatenate([o.A for o in outs]).mean(0)
    pe = np.concatenate([o.pi_end for o in outs]).mean(0)
    fc = np.concatenate([o.forecasts for o in outs]).mean(0)
    np.testing.assert_allclose(mu, g["filtered_means"], atol=0.08)
    np.testing.assert_allclose(s2, g["filtered_variances"], rtol=0.06)
    np.testing.assert_allclose(A.T.ravel(), g["filtered_trans_probs"], atol=0.01)   # trans_a_b column = A[b,a]
    np.testing.assert_allclose(pe, g["filtered_state_probs"], atol=0.01)
    if np.isfinite(fc[1]):
        np.testing.assert_allclose(fc, g["forecasts"], atol=0.06)


@pytest.mark.parametrize("end_index,noise", [(121, 0.3), (200, 0.6), (300, 0.1), (450, 0.3), (570, 0.6)])
def test_golden_signal_dispersion(oracle, end_index, noise):
    """The signal tier (mask, sd*(1+kappa) emissions, kappa-weighted statistics incl. quirk Q3, HyperParams(opt) priors,
    estimatesignals! :868-914) against the reference's OWN outputs: data/output/signals_official_noise_<kappa>_allsignal
    (every observation a signal, 100 perturbed copies per end date).  sigma_signal is taken from the golden's realised
    signal spread (the reference derives it from a heavy-tailed mean of sigma^2 draws that no finite run pins down)."""
    y, dates, case, ssig = signals_golden_case(end_index, noise)
    Y = y[:end_index]
    mask, two, xi = np.ones(end_index, dtype=np.uint8), np.full(3, 2.0), np.full(3, Y.mean())
    X0, _, _ = oracle.make_params(Y, 3)                         # :888: initial states from the real data
    rng = np.random.default_rng(1234)
    S = 100
    outs, _ = oracle.gibbs_batch([dict(y=Y + rng.standard_normal(end_index) * ssig, K=3, burnin=1500, nrun=2500, seed=1234,
                                       chain=100 + s, horizons=(12,), y_future=[y[end_index - 1 + 12]], is_signal=mask, kappa=noise,
                                       alpha=two, nu=two, xi=xi, X0=X0) for s in range(S)])
    assert sum(o.n_events for o in outs) == 0
    pm = lambda k: np.array([getattr(o, k).mean(0) for o in outs])
    dispersion_close(pm("mu"), case["filtered_means"], "mu", atol=0.02)
    # the injected sigma_signal is itself an estimate from 2 x 100 values (+-5 %, so +-10 % on sigma_signal^2, which enters the
    # variance draws as Sm2 / (1 + kappa), :315): allow 2.5 sigma of that on top of the sampling error
    dispersion_close(pm("sigma2"), case["filtered_variances"], "sigma2", atol=0.25 * ssig ** 2 / (1 + noise))
    dispersion_close(pm("pi_end"), case["filtered_state_probs"], "pi_end")
    dispersion_close(np.transpose(pm("A"), (0, 2, 1)).reshape(S, 9), case["filtered_trans_probs"], "A")     # trans_a_b = A[b,a]
    dispersion_close(pm("forecasts"), case["forecasts"], "forecasts", atol=0.02)


def test_golden_insample_table_is_filtered(oracle):
    """The reference's published in-sample table (data/output/official_insample/forecats_insample.csv, 576 dates, one
    full-sample estimation) against the oracle: its state probabilities are the posterior mean of the FILTERED
    probabilities pif (median deviation < 2e-3) and not of the smoothed pib, which is far sharper in mid-sample; its
    12-month forecasts are pif[t,:]' A^12 mu.  This pins the forward filter (:371-440) to reference output on every date."""
    y, dates = load_inflation()
    g = json.load(open(os.path.join(GOLDEN, "official_insample.json")))
    N = g["last_index"]
    gp, gf = np.array(g["probs"]), np.array(g["forecast"])
    outs, _ = oracle.gibbs_batch([dict(y=y[:N], K=3, burnin=3000, nrun=3000, seed=1234, chain=c, horizons=(12,),
                                       y_future=[y[N - 1 + 12]], want_pib_mean=True) for c in range(8)])
    rng = np.random.default_rng(0)
    pf, fc, n = np.zeros((N, 3)), np.zeros(N), 0
    for o in outs:
        for j in range(0, 3000, 12):
            A, mu = o.A[j], o.mu[j]
            f = oracle.forward(y[:N], A, mu, o.sigma2[j], rng.dirichlet(np.ones(3)), want_Pf=False)     # rho ~ flat prior (:350-356)
            pf += f.pif
            fc += f.pif @ np.linalg.matrix_power(A, 12) @ mu
            n += 1
    pf /= n
    fc /= n
    pb = np.mean([o.pib_mean for o in outs], axis=0)
    d_f, d_b = np.abs(pf - gp).max(1), np.abs(pb - gp).max(1)
    assert np.median(d_f) < 2e-3 and (d_f < 0.03).mean() > 0.85 and d_f.max() < 0.25
    assert (d_b < 0.03).mean() < 0.8 and d_b.max() > 0.5 and d_b.mean() > 2 * d_f.mean()     # the smoothed rows are NOT what was published
    assert d_f[-1] < 5e-3 and d_b[-1] < 5e-3                                                  # last date: filtered = smoothed
    assert np.median(np.abs(fc - gf)) < 0.03 and np.quantile(np.abs(fc - gf), 0.99) < 0.5
