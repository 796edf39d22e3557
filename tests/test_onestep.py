"""One-step-ahead posterior predictive scores of every in-sample date (HMCGPU_FLAG_ONESTEP): the numpy definition the device
must match, its analytic cases, a mirror of the device's streaming fold, the host plumbing, and (with -m gpu) the device against
that definition applied to the same call's draws."""
import ctypes
import os
import re

import numpy as np
import pytest
from scipy.special import logsumexp, ndtr
from scipy.stats import kstest, norm

from conftest import ROOT, K3_TRUTH, synth_hmm


def onestep_terms(mu, sigma2, A, y):
    """ell [R, N] = log p(y_t | y_1..t-1, theta_d) and F [R, N] = the one-step-ahead CDF at y_t, from the forward filter started
    at the uniform distribution (include/hmcgpu.h, hmcgpu_onestep).  mu, sigma2 [R, K], A [R, K, K] with A[d, r, s] =
    P(X_t = s | X_t-1 = r), y [N]."""
    mu, sigma2, A, y = (np.asarray(a, dtype=np.float64) for a in (mu, sigma2, A, y))
    R, K = mu.shape
    sd = np.sqrt(sigma2)
    w = np.full((R, K), 1.0 / K)
    ell, F = np.empty((R, len(y))), np.empty((R, len(y)))
    for t, yt in enumerate(y):
        l = np.log(w) + norm.logpdf(yt, mu, sd)
        ell[:, t] = logsumexp(l, axis=1)
        F[:, t] = np.sum(w * ndtr((yt - mu) / sd), axis=1)
        alpha = np.exp(l - ell[:, t:t + 1])
        w = np.einsum("dr,drs->ds", alpha, A)
    return ell, F


def waic_row(lpd, lpd_var):
    e = lpd - lpd_var
    lppd, pw = lpd.sum(), lpd_var.sum()
    return np.array([lppd, pw, lppd - pw, np.sqrt(len(e) * np.var(e, ddof=1))])


def onestep_reference(mu, sigma2, A, y):
    """Definition of include/hmcgpu.h for one window (two passes over the R pooled draws).  Returns pit, lpd, lpd_var [N] and
    waic [4] (lppd, p_waic, elpd_waic, se); NaN everywhere when a draw is not finite."""
    N = len(y)
    if not all(np.all(np.isfinite(a)) for a in (mu, sigma2, A)):
        return np.full(N, np.nan), np.full(N, np.nan), np.full(N, np.nan), np.full(4, np.nan)
    ell, F = onestep_terms(mu, sigma2, A, y)
    R = ell.shape[0]
    lpd = logsumexp(ell, axis=0) - np.log(R)
    var = np.var(ell, axis=0, ddof=1)
    return F.mean(axis=0), lpd, var, waic_row(lpd, var)


def onestep_stream(ell, F, n_chains):
    """The device's order of operations: per chain and date a running log-sum-exp and Welford update in draw order, then the
    chains combined in chain order (log-sum-exp pairs, Chan's pairwise update).  ell, F [n_chains * nrun, N] chain-major."""
    R, N = ell.shape
    nrun = R // n_chains
    pit, lpd, var = np.empty(N), np.empty(N), np.empty(N)
    for t in range(N):
        states = []
        for c in range(n_chains):
            p, mx, sc, mean, m2 = 0.0, -np.inf, 0.0, 0.0, 0.0
            for i in range(nrun):
                x = ell[c * nrun + i, t]
                p += F[c * nrun + i, t]
                if x > mx:
                    sc, mx = sc * np.exp(mx - x) + 1.0, x
                else:
                    sc += np.exp(x - mx)
                dl = x - mean
                mean += dl / (i + 1)
                m2 += dl * (x - mean)
            states.append((p, mx, sc, mean, m2))
        mx = max(s[1] for s in states)
        sf = sum(s[0] for s in states)
        sc, na, mean, m2 = 0.0, 0.0, 0.0, 0.0
        for s in states:
            sc += s[2] * np.exp(s[1] - mx)
            n = na + nrun
            d = s[3] - mean
            mean += d * (nrun / n)
            m2 += s[4] + d * d * (na * nrun / n)
            na = n
        pit[t], lpd[t], var[t] = sf / R, mx + np.log(sc / R), m2 / (R - 1)
    return pit, lpd, var


def _draws(rng, R, K):
    mu = np.sort(rng.normal(0, 3, size=(R, K)), axis=1)
    sigma2 = rng.uniform(0.3, 3.0, size=(R, K))
    A = rng.dirichlet(np.ones(K) * 2.0, size=(R, K))
    return mu, sigma2, A


def test_equal_states_give_the_normal():
    """K states with one mu and sigma2: whatever the weights, p_t = phi and PIT = Phi(z); identical draws have no spread."""
    rng = np.random.default_rng(1)
    R, K = 6, 4
    y = rng.normal(1.0, 2.0, size=40)
    mu, s2 = np.full((R, K), 1.3), np.full((R, K), 2.5)
    A = np.repeat(rng.dirichlet(np.ones(K), size=(1, K)), R, axis=0)
    pit, lpd, var, waic = onestep_reference(mu, s2, A, y)
    np.testing.assert_allclose(lpd, norm.logpdf(y, 1.3, np.sqrt(2.5)), rtol=1e-13)
    np.testing.assert_allclose(pit, norm.cdf(y, 1.3, np.sqrt(2.5)), atol=1e-15)
    assert np.all(np.abs(var) < 1e-26) and abs(waic[1]) < 1e-24
    np.testing.assert_allclose(waic[[0, 2]], lpd.sum(), rtol=1e-13)


def test_observation_fifty_sd_out_stays_finite():
    """Two states at 0 and 1 (sd 1), rows of A = (1/2, 1/2): w_2 = (1/2, 1/2) whatever y_1, so
    ell_2 = log(phi(50; 0, 1) / 2 + phi(50; 1, 1) / 2) = -log 2 - log(2 pi) / 2 - 1200.5 + log1p(exp(-49.5)).  The direct pdf
    underflows to 0 in fp64 there."""
    mu, s2 = np.array([[0.0, 1.0]]), np.ones((1, 2))
    A = np.full((1, 2, 2), 0.5)
    y = np.array([0.2, 50.0, 0.3])
    ell, F = onestep_terms(mu, s2, A, y)
    want = -np.log(2.0) - 0.5 * np.log(2 * np.pi) - 1200.5 + np.log1p(np.exp(-49.5))
    assert np.exp(-0.5 * 49.0 ** 2) == 0.0
    np.testing.assert_allclose(ell[0, 1], want, rtol=1e-14)
    assert abs(F[0, 1] - 1.0) < 1e-15 and np.all(np.isfinite(ell))
    # whatever the filter holds after the outlier, the uniform rows of A score y_3 under (1/2, 1/2)
    np.testing.assert_allclose(ell[0, 2], np.log(0.5 * norm.pdf(0.3, 0, 1) + 0.5 * norm.pdf(0.3, 1, 1)), rtol=1e-13)


def test_streaming_fold_matches_two_passes():
    rng = np.random.default_rng(2)
    n_chains, nrun, K = 3, 57, 3
    mu, s2, A = _draws(rng, n_chains * nrun, K)
    y = rng.normal(0, 3, size=25)
    y[7] = 60.0                                                 # one far outlier: a wide spread of ell across draws
    ell, F = onestep_terms(mu, s2, A, y)
    pit, lpd, var, _ = onestep_reference(mu, s2, A, y)
    spit, slpd, svar = onestep_stream(ell, F, n_chains)
    np.testing.assert_allclose(spit, pit, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(slpd, lpd, rtol=1e-12)
    np.testing.assert_allclose(svar, var, rtol=1e-12)


def test_non_finite_draw_poisons_the_window():
    rng = np.random.default_rng(3)
    mu, s2, A = _draws(rng, 10, 3)
    A[4, 1, 2] = np.nan
    outs = onestep_reference(mu, s2, A, rng.normal(size=12))
    assert all(np.all(np.isnan(o)) for o in outs)


def test_flag_constant_struct_and_symbols_match_header(H, tmp_path):
    from hmc_jl_b200 import binding as B
    from test_host import _C2CTYPES, _C2JULIA, _c_offsets, _header_struct_fields
    header = open(os.path.join(ROOT, "include", "hmcgpu.h")).read()
    jl = open(os.path.join(ROOT, "hmc.jl_b200", "julia", "HmcGPU.jl")).read()
    assert int(re.search(r"#define HMCGPU_FLAG_ONESTEP\s+(\d+)u", header).group(1)) == B.FLAG_ONESTEP == H.FLAG_ONESTEP == 1024
    assert re.search(r"const FLAG_ONESTEP = UInt32\(1024\)", jl)
    for sym in ("hmcgpu_estimate_onestep", "hmcgpu_estimate_multi_onestep", "hmcgpu_plan_fetch_onestep"):
        assert sym in B.SYMBOLS and re.search(r"\b%s\(" % sym, header) and re.search(r":%s\b" % sym, jl)
    fields = _header_struct_fields("hmcgpu_onestep")
    off = _c_offsets(tmp_path, "hmcgpu_onestep", fields)
    assert [f for f, _ in B.Onestep._fields_] == [f for _, f in fields] == ["pit", "lpd", "lpd_var", "waic"]
    assert ctypes.sizeof(B.Onestep) == off["sizeof"]
    for (ctype, f), (_, pytype) in zip(fields, B.Onestep._fields_):
        assert getattr(B.Onestep, f).offset == off[f] and pytype.__name__ == _C2CTYPES[ctype], f
    body = re.search(r"struct Onestep\n(.*?)\nend", jl, re.S).group(1)
    jfields = [tuple(x.strip().split("::")) for ln in body.splitlines() for x in ln.split(";") if x.strip()]
    assert jfields == [(f, _C2JULIA[ctype]) for ctype, f in fields]
    assert H.load().hmcgpu_version() == 600


def test_binding_allocates_and_splits_per_window(H):
    y = np.random.default_rng(0).normal(size=60)
    spec = H.ProblemSpec(y, [1, 5, 2], [50, 30, 41], K=3, nrun=8, flags=H.FLAG_SUMMARY)
    o, _ = spec.alloc_result()
    assert spec.alloc_onestep(o) is None and not hasattr(o, "lpd")
    spec = H.ProblemSpec(y, [1, 5, 2], [50, 30, 41], K=3, nrun=8, flags=H.FLAG_ONESTEP)
    o, res = spec.alloc_result()
    os_ = spec.alloc_onestep(o)
    assert o.lpd.shape == o.lpd_var.shape == o.onestep_pit.shape == (50 + 26 + 40,) and o.waic.shape == (3, 4)
    assert os_.pit and os_.waic
    o.lpd[:] = np.arange(o.lpd.size)
    spec.finish(o, res, 0)
    assert [len(a) for a in o.lpd] == [50, 26, 40] and o.lpd[1][0] == 50 and o.lpd[2][-1] == 115


def _fake_fit(rng, lens, shift=0.0):
    from types import SimpleNamespace
    lpd = [rng.normal(-1.5, 0.4, size=n) + shift for n in lens]
    var = [rng.uniform(0.0, 0.05, size=n) for n in lens]
    waic = np.array([waic_row(a, b) for a, b in zip(lpd, var)])
    pit = [rng.uniform(size=n) for n in lens]
    return SimpleNamespace(lpd=lpd, lpd_var=var, waic=waic, onestep_pit=pit)


def test_compare_waic_and_pseudo_residuals(H):
    rng = np.random.default_rng(4)
    a, b = _fake_fit(rng, [30, 45]), _fake_fit(rng, [30, 45], shift=-0.2)
    c = H.compare_waic(a, b)
    for w in range(2):
        e = (a.lpd[w] - a.lpd_var[w]) - (b.lpd[w] - b.lpd_var[w])
        np.testing.assert_allclose(c.elpd_diff[w], e.sum(), rtol=1e-12)
        np.testing.assert_allclose(c.se_diff[w], np.sqrt(len(e) * np.var(e, ddof=1)), rtol=1e-12)
    assert np.all(c.elpd_diff > 0)
    with pytest.raises(ValueError, match="same windows"):
        H.compare_waic(a, _fake_fit(rng, [30, 44]))
    np.testing.assert_allclose(H.pseudo_residuals(np.array([0.5, 0.975, 0.025])), [0.0, 1.959963984540054, -1.959963984540054],
                               atol=1e-12)
    z = H.pseudo_residuals(a.onestep_pit)
    assert [len(x) for x in z] == [30, 45] and np.all(np.isinf(H.pseudo_residuals(np.array([0.0, 1.0]))))


def test_estimate_windows_flag_and_write_onestep(H, tmp_path, monkeypatch):
    from hmc_jl_b200 import api, binding as B
    seen = {}

    class FakeCtx:
        def close(self):
            pass

    def fake_estimate(ctx, spec):
        seen["spec"] = spec
        return None

    monkeypatch.setattr(B, "estimate", fake_estimate)
    y = np.random.default_rng(0).normal(size=40)
    api.estimate_windows(y, [1, 1], [30, 35], K=2, nrun=10, onestep=True, ctx=FakeCtx())
    assert seen["spec"].flags & B.FLAG_ONESTEP
    api.estimate_windows(y, [1], [30], K=2, nrun=10, ctx=FakeCtx())
    assert not seen["spec"].flags & B.FLAG_ONESTEP

    out = _fake_fit(np.random.default_rng(5), [3, 2])
    paths = H.write_onestep(out, ["2001-01", "2001-06"], str(tmp_path))
    lines = open(paths["scores"]).read().splitlines()
    assert lines[0] == "date,t,pit,pseudo_residual,lpd,lpd_var" and len(lines) == 1 + 5
    assert [ln.split(",")[:2] for ln in lines[1:]] == [["2001-01", "1"], ["2001-01", "2"], ["2001-01", "3"], ["2001-06", "1"], ["2001-06", "2"]]
    got = np.loadtxt(paths["scores"], delimiter=",", skiprows=1, usecols=(2, 3, 4, 5))
    want = np.column_stack([np.concatenate(v) for v in (out.onestep_pit, H.pseudo_residuals(out.onestep_pit), out.lpd, out.lpd_var)])
    np.testing.assert_array_equal(got, want)
    w = open(paths["waic"]).read().splitlines()
    assert w[0] == "date,lppd,p_waic,elpd_waic,se" and [ln.split(",")[0] for ln in w[1:]] == ["2001-01", "2001-06"]
    np.testing.assert_array_equal(np.loadtxt(paths["waic"], delimiter=",", skiprows=1, usecols=(1, 2, 3, 4)), out.waic)


def _oracle_fit(oracle, y, K, n_chains=4, burnin=1000, nrun=500):
    outs, _ = oracle.gibbs_batch([dict(y=y, K=K, burnin=burnin, nrun=nrun, seed=21, chain=c, horizons=(1,)) for c in range(n_chains)])
    mu = np.concatenate([o.mu for o in outs])
    s2 = np.concatenate([o.sigma2 for o in outs])
    A = np.concatenate([o.A for o in outs])
    pit, lpd, var, waic = onestep_reference(mu, s2, A, y)
    from types import SimpleNamespace
    return SimpleNamespace(onestep_pit=[pit], lpd=[lpd], lpd_var=[var], waic=waic[None])


def test_model_choice_margin_with_the_oracle_chain(H, oracle):
    """The margin the GPU model-choice test relies on, taken with the reference sampler (the oracle) and the numpy definition:
    on T = 1500 dates from the three-state truth, K = 3 beats K = 2 by far more than 4 se_diff; and the K = 3 PIT of T = 2000
    dates is uniform to a KS distance below 0.05."""
    y, _ = synth_hmm(1500, **K3_TRUTH, seed=31)
    c = H.compare_waic(_oracle_fit(oracle, y, 3), _oracle_fit(oracle, y, 2))
    assert c.elpd_diff[0] > 4 * c.se_diff[0], (c.elpd_diff, c.se_diff)
    y, _ = synth_hmm(2000, **K3_TRUTH, seed=32)
    assert kstest(_oracle_fit(oracle, y, 3).onestep_pit[0], "uniform").statistic < 0.05


# ---------------------------------------------------------------------------------------------------------------------------- GPU

def _series():
    y, _ = synth_hmm(90, **K3_TRUTH, seed=7)
    return y


_KERNELS = {"thread": 0, "scan": 1, "lane": 2, "seg": 4}


def _force(monkeypatch, kernel):
    for v in ("HMCGPU_SCAN_MAX_CHAINS", "HMCGPU_SEG_LANES", "HMCGPU_LANE_KERNEL"):
        monkeypatch.delenv(v, raising=False)
    if kernel == "scan":
        monkeypatch.setenv("HMCGPU_SCAN_MAX_CHAINS", "100000")
    else:
        monkeypatch.setenv("HMCGPU_SCAN_MAX_CHAINS", "0")
        monkeypatch.setenv("HMCGPU_SEG_LANES", "4" if kernel == "seg" else "0")
    if kernel == "lane":
        monkeypatch.setenv("HMCGPU_LANE_KERNEL", "1")


def _check_against_reference(o, spec, y_of_window):
    """Every output of every window against onestep_reference applied to the call's returned draws.  fp64: 1e-10 relative.
    fp32: the device filters in fp32 (series and draws as the chain saw them) against the fp64 definition, to about 8 times the
    largest error seen on a B200."""
    fp64 = spec.precision == 64
    for w in range(spec.n_windows):
        y = y_of_window(w)[spec.win_start[w] - 1:spec.win_end[w]]
        pit, lpd, var, waic = onestep_reference(o.mu[w].T, o.sigma2[w].T, o.A[w].transpose(2, 1, 0), y)
        n = len(y)
        msg = f"window {w}"
        if fp64:
            np.testing.assert_allclose(o.onestep_pit[w], pit, rtol=1e-10, atol=1e-13, err_msg=msg)
            np.testing.assert_allclose(o.lpd[w], lpd, rtol=1e-10, err_msg=msg)
            np.testing.assert_allclose(o.lpd_var[w], var, rtol=1e-10, atol=1e-15, err_msg=msg)
            np.testing.assert_allclose(o.waic[w], waic, rtol=1e-10, err_msg=msg)
        else:
            # observed on a B200 over these cases: pit 6e-8, lpd 7e-7 absolute; lpd_var 5e-7, p_waic 1e-7, se 8e-8 relative;
            # lppd 1.0e-5 absolute over 88 dates
            np.testing.assert_allclose(o.onestep_pit[w], pit, rtol=0, atol=5e-7, err_msg=msg)
            np.testing.assert_allclose(o.lpd[w], lpd, rtol=0, atol=5e-6, err_msg=msg)
            np.testing.assert_allclose(o.lpd_var[w], var, rtol=5e-6, atol=1e-9, err_msg=msg)
            np.testing.assert_allclose(o.waic[w, [0, 2]], waic[[0, 2]], rtol=0, atol=1e-6 * n, err_msg=msg)
            np.testing.assert_allclose(o.waic[w, [1, 3]], waic[[1, 3]], rtol=1e-6, err_msg=msg)
        assert np.all(np.isfinite(o.lpd[w])) and np.all((o.onestep_pit[w] >= 0) & (o.onestep_pit[w] <= 1))


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,precision,nrun,K", [
    ("thread", 32, 1501, 3), ("thread", 64, 2049, 3), ("scan", 32, 2049, 3), ("scan", 64, 1501, 3), ("seg", 32, 1501, 3),
    ("seg", 64, 2049, 3), ("thread", 32, 1501, 2), ("thread", 32, 1501, 5), ("thread", 64, 1501, 6), ("thread", 32, 2049, 8),
    ("thread", 64, 1501, 8), ("lane", 32, 1501, 5), ("lane", 64, 1501, 7), ("lane", 32, 2049, 8), ("lane", 64, 1501, 8)])
def test_device_matches_reference(H, ctx, monkeypatch, kernel, precision, nrun, K):
    """nrun = 1501 / 2049: two and three draw chunks; windows of 88, 66 and 41 dates."""
    _force(monkeypatch, kernel)
    y = _series()
    spec = H.ProblemSpec(y, [1, 5, 20], [88, 70, 60], K=K, n_chains=3, burnin=30, nrun=nrun, seed=11, horizons=(1,),
                         precision=precision, flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_ONESTEP)
    o = H.estimate(ctx, spec)
    assert o.sweep_kernel == _KERNELS[kernel]
    _check_against_reference(o, spec, lambda w: y)


@pytest.mark.gpu
def test_far_outlier_and_pi_row_back(H, ctx):
    """A window whose draws all sit far from one observation (y = 300 against states near 1.6 / 3.5 / 8.3 elsewhere) keeps every
    lpd finite on the device in fp64 and fp32; pi_row_back is accepted.  (fp32 carries ~1e-7 of the large log-density there.)"""
    y = _series()
    y[40] = 300.0
    for precision in (64, 32):
        spec = H.ProblemSpec(y, [1, 10], [88, 80], K=3, n_chains=2, burnin=30, nrun=300, seed=4, horizons=(1,), precision=precision,
                             pi_row_back=2, flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_ONESTEP)
        o = H.estimate(ctx, spec)
        assert all(np.all(np.isfinite(a)) for a in o.lpd + o.lpd_var) and np.all(np.isfinite(o.waic))
        for w in range(2):
            yw = y[spec.win_start[w] - 1:spec.win_end[w]]
            pit, lpd, var, waic = onestep_reference(o.mu[w].T, o.sigma2[w].T, o.A[w].transpose(2, 1, 0), yw)
            rtol = 1e-10 if precision == 64 else 1e-5
            np.testing.assert_allclose(o.lpd[w], lpd, rtol=rtol, atol=0 if precision == 64 else 2e-5)
            np.testing.assert_allclose(o.onestep_pit[w], pit, rtol=rtol, atol=1e-13 if precision == 64 else 2e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["thread", "seg", "lane"])
def test_flag_changes_nothing_else(H, ctx, monkeypatch, kernel):
    """Draws, summaries, diagnostics, predictive outputs and status are bit-identical with and without HMCGPU_FLAG_ONESTEP; the
    flag adds exactly one launch per draw chunk (nrun = 2049: three chunks)."""
    _force(monkeypatch, kernel)
    base = H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY | H.FLAG_LOGLIK | H.FLAG_DIAGNOSTICS | H.FLAG_PREDICTIVE
    outs = []
    for flag in (0, H.FLAG_ONESTEP):
        spec = H.ProblemSpec(_series(), [1, 9], [80, 61], K=5 if kernel == "lane" else 3, n_chains=5, burnin=20, nrun=2049, seed=3,
                             horizons=(2,), precision=32, flags=base | flag, pred_grid=np.linspace(0, 10, 20))
        outs.append(H.estimate(ctx, spec))
    a, b = outs
    assert b.sweep_kernel == _KERNELS[kernel]
    assert b.n_sweep_launches == a.n_sweep_launches and b.n_launches == a.n_launches + 3
    for name in ("mu", "sigma2", "A", "pi_end", "forecasts", "loglik", "summary_mean", "summary_var", "status", "rhat", "ess",
                 "ess_lag", "pred_cdf", "pit", "log_score", "pred_moments"):
        np.testing.assert_array_equal(getattr(a, name), getattr(b, name), err_msg=name)
    assert a.events == b.events and not hasattr(a, "lpd") and all(np.all(np.isfinite(x)) for x in b.lpd)


def _chunk(nw, nc, K, nh, nrun, precision=32):
    """plan_build's chunk rule for the thread-per-chain kernel: min(nrun, 1024, 2 GiB / n_bufs / per-draw bytes)."""
    n_slots = (nw * nc + 31) // 32 * 32
    tasks = n_slots // 32
    groups = 4 if tasks >= 1024 else (2 if tasks >= 256 else 1)
    n_bufs = 2 if groups > 1 else 1
    F = 3 * K + K * K + 2 * nh + 1
    return min(nrun, 1024, max(1, (2 << 30) // n_bufs // (F * n_slots * precision // 8)))


@pytest.mark.gpu
def test_batching_chunking_and_multi_invariance(H, ctx, monkeypatch):
    """A window's outputs are bit-identical alone, in a ragged batch, across two runs of one plan, through
    hmcgpu_estimate_multi_onestep on two contexts, and inside a batch wide enough for a different chunk size."""
    _force(monkeypatch, "thread")
    y = _series()
    names = ("onestep_pit", "lpd", "lpd_var")
    kw = dict(K=3, n_chains=4, burnin=20, nrun=2049, seed=9, horizons=(1, 12), precision=32, flags=H.FLAG_REF_Q1 | H.FLAG_ONESTEP)
    starts, ends = [1, 1, 30, 1, 12], [85, 40, 77, 66, 90]

    def same(a, wa, b, wb):
        for n in names:
            np.testing.assert_array_equal(getattr(a, n)[wa], getattr(b, n)[wb], err_msg=n)
        np.testing.assert_array_equal(a.waic[wa], b.waic[wb])

    batch = H.estimate(ctx, H.ProblemSpec(y, starts, ends, win_id=np.arange(5), **kw))
    for w in (0, 2, 4):
        same(H.estimate(ctx, H.ProblemSpec(y, [starts[w]], [ends[w]], win_id=[w], **kw)), 0, batch, w)
    spec = H.ProblemSpec(y, starts, ends, **kw)
    plan = H.Plan(ctx, spec)
    try:
        plan.run()
        first = plan.fetch()
        plan.run()
        again = plan.fetch()
    finally:
        plan.close()
    multi = H.estimate_multi([0, 0], spec)
    for w in range(5):
        same(first, w, batch, w)
        same(again, w, batch, w)
        same(multi, w, batch, w)
    nw = 3000
    assert _chunk(nw + 1, 4, 3, 2, 2049) != _chunk(5, 4, 3, 2, 2049) == 1024
    wide_s = np.concatenate([[starts[0]], 60 + np.arange(nw) % 10])
    wide_e = np.concatenate([[ends[0]], 80 + np.arange(nw) % 10])
    wide = H.estimate(ctx, H.ProblemSpec(y, wide_s, wide_e, win_id=np.arange(nw + 1) + 100000 * (np.arange(nw + 1) > 0), **kw))
    assert wide.sweep_kernel == 0
    same(wide, 0, batch, 0)


@pytest.mark.gpu
def test_refusals(H, ctx):
    import ctypes as C
    from hmc_jl_b200 import binding as B
    y = _series()
    kw = dict(K=3, n_chains=2, burnin=5, nrun=10, horizons=(1,), flags=H.FLAG_REF_Q1 | H.FLAG_ONESTEP)

    def message():
        return ctx.L.hmcgpu_last_error(ctx.h).decode()

    def code(spec, **override):
        prob = spec.struct()
        for k, v in override.items():
            setattr(prob, k, v)
        o, res = spec.alloc_result()
        os_ = spec.alloc_onestep(o)
        return ctx.L.hmcgpu_estimate_onestep(ctx.h, C.byref(prob), C.byref(res), None, None, C.byref(os_))

    ok = H.ProblemSpec(y, [1], [60], **kw)
    assert code(ok) >= 0
    assert code(ok, n_chains=1, nrun=1) == B.ERR_ARG and "n_chains * nrun >= 2" in message()
    assert code(H.ProblemSpec(y, [1], [60], **{**kw, "K": 9})) == B.ERR_UNSUPPORTED and "K <= 8" in message()
    mask = np.zeros(len(y), dtype=np.uint8)
    mask[50:55] = 1
    assert code(H.ProblemSpec(y, [1], [60], is_signal=mask, **kw)) == B.ERR_UNSUPPORTED and "is_signal" in message()
    # the flag through the entry points without one-step outputs
    prob, (o, res) = ok.struct(), ok.alloc_result()
    assert ctx.L.hmcgpu_estimate(ctx.h, C.byref(prob), C.byref(res)) == B.ERR_ARG and "hmcgpu_onestep" in message()
    assert ctx.L.hmcgpu_estimate_ranked(ctx.h, C.byref(prob), C.byref(res), None, None) == B.ERR_ARG and "hmcgpu_onestep" in message()
    dev = (C.c_int * 1)(0)
    assert ctx.L.hmcgpu_estimate_multi(dev, 1, C.byref(prob), C.byref(res)) == B.ERR_ARG
    assert "hmcgpu_onestep" in ctx.L.hmcgpu_last_error(None).decode()
    # fetch on a plan without the flag, and before a run
    plan = H.Plan(ctx, H.ProblemSpec(y, [1], [60], **{**kw, "flags": H.FLAG_REF_Q1}))
    os_ = B.Onestep()
    try:
        plan.run()
        assert ctx.L.hmcgpu_plan_fetch_onestep(plan.h, C.byref(os_)) == B.ERR_ARG and "without HMCGPU_FLAG_ONESTEP" in message()
    finally:
        plan.close()
    plan = H.Plan(ctx, ok)
    try:
        assert ctx.L.hmcgpu_plan_fetch_onestep(plan.h, C.byref(os_)) == B.ERR_ARG and "before plan_run" in message()
    finally:
        plan.close()


@pytest.mark.gpu
def test_calibration_and_model_choice(H, ctx):
    """K = 3 fitted to 2000 dates from the three-state truth: the one-step PIT is uniform (KS distance < 0.05).  On 1500 dates
    compare_waic(K = 3, K = 2) favours the true K by more than 4 se_diff (the margin test_model_choice_margin_with_the_oracle_chain
    takes with the reference sampler)."""
    kw = dict(n_chains=8, burnin=1000, nrun=500, seed=21, horizons=(1,), precision=32, summary=False, onestep=True, ctx=ctx)
    y, _ = synth_hmm(2000, **K3_TRUTH, seed=32)
    fit = H.estimate_windows(y, [1], [len(y)], K=3, **kw)
    assert kstest(fit.onestep_pit[0], "uniform").statistic < 0.05
    y, _ = synth_hmm(1500, **K3_TRUTH, seed=31)
    c = H.compare_waic(H.estimate_windows(y, [1], [len(y)], K=3, **kw), H.estimate_windows(y, [1], [len(y)], K=2, **kw))
    assert c.elpd_diff[0] > 4 * c.se_diff[0], (c.elpd_diff, c.se_diff)
