"""PSIS-LOO of every in-sample date (HMCGPU_FLAG_LOO): the numpy definition the device must match (exact leave-one-out terms of
the HMM, then Pareto-smoothed importance sampling as the R package loo 2.x does it), its analytic and brute-force cases, the
g++-compiled PSIS header (tests/psis_driver.cpp), the host plumbing, and (with -m gpu) the device against that definition
applied to the same call's draws."""
import ctypes
import itertools
import os
import re
import subprocess

import numpy as np
import pytest
from scipy.special import logsumexp, ndtr
from scipy.stats import kstest, norm

from conftest import ROOT, K3_TRUTH, synth_hmm
from test_onestep import onestep_terms

CSRC = os.path.join(ROOT, "hmc.jl_b200", "csrc")
DBL_EPS = np.finfo(np.float64).eps


# ------------------------------------------------------------------------------------------------------- numpy definition

def loo_terms(mu, sigma2, A, y):
    """ell [R, N] = log p(y_t | y_-t, theta_d) and F [R, N] = P(Y_t <= y_t | y_-t, theta_d), from the forward filter started at
    the uniform distribution and the backward recursion b_N = 1 (include/hmcgpu.h, hmcgpu_loo).  mu, sigma2 [R, K],
    A [R, K, K] with A[d, r, s] = P(X_t = s | X_t-1 = r), y [N]."""
    mu, sigma2, A, y = (np.asarray(a, dtype=np.float64) for a in (mu, sigma2, A, y))
    R, K = mu.shape
    N = len(y)
    sd = np.sqrt(sigma2)
    lphi = norm.logpdf(y[:, None, None], mu[None], sd[None])            # [N, R, K]
    cdf = ndtr((y[:, None, None] - mu[None]) / sd[None])
    logw = np.empty((N, R, K))
    w = np.full((R, K), 1.0 / K)
    for t in range(N):
        logw[t] = np.log(w)
        l = logw[t] + lphi[t]
        alpha = np.exp(l - logsumexp(l, axis=1, keepdims=True))
        w = np.einsum("dr,drs->ds", alpha, A)
    logb = np.zeros((N, R, K))
    logA = np.log(A)
    for t in range(N - 2, -1, -1):
        u = lphi[t + 1] + logb[t + 1]                                   # [R, K] over s
        logb[t] = logsumexp(logA + u[:, None, :], axis=2)
        logb[t] -= logb[t].max(axis=1, keepdims=True)
    num = logw + lphi + logb
    den = logw + logb
    ell = (logsumexp(num, axis=2) - logsumexp(den, axis=2)).T
    q = np.exp(den - logsumexp(den, axis=2, keepdims=True))
    F = np.sum(q * cdf, axis=2).T
    return ell, F


def psis_tail_len(R):
    return int(np.ceil(min(0.2 * R, 3 * np.sqrt(R))))


def k_threshold(R):
    return min(1 - 1 / np.log10(R), 0.7)


def gpdfit(x):
    """loo's gpdfit (Zhang & Stephens, wip = TRUE, min_grid_pts = 30, prior 3) of x sorted ascending: (k, sigma)."""
    M = len(x)
    m = 30 + int(np.floor(np.sqrt(M)))
    j = np.arange(1, m + 1)
    xstar = x[int(np.floor(M / 4 + 0.5)) - 1]
    theta = 1 / x[-1] + (1 - np.sqrt(m / (j - 0.5))) / 3 / xstar
    kk = np.array([np.mean(np.log1p(-t * x)) for t in theta])
    l_theta = M * (np.log(-theta / kk) - kk - 1)
    w = np.exp(l_theta - logsumexp(l_theta))
    theta_hat = np.sum(theta * w)
    k = np.mean(np.log1p(-theta_hat * x))
    sigma = -k / theta_hat
    k = k * M / (M + 10) + 10 * 0.5 / (M + 10)
    return (np.inf if np.isnan(k) else k), sigma


def psis(r):
    """loo 2.x's do_psis_i with r_eff = 1 on log ratios r [R]: (truncated log weights lw [R] relative to max r, k̂)."""
    r = np.asarray(r, dtype=np.float64)
    R = len(r)
    lw = r - r.max()
    M = psis_tail_len(R)
    k = np.inf
    if M >= 5:
        ord_ = np.lexsort((np.arange(R), lw))                          # ascending, ties by draw index
        tail = ord_[R - M:]
        if abs(lw[tail[-1]] - lw[tail[0]]) >= DBL_EPS / 100:
            cutoff = lw[ord_[R - M - 1]]
            k, sigma = gpdfit(np.exp(lw[tail]) - np.exp(cutoff))
            if np.isfinite(k):
                p = (np.arange(1, M + 1) - 0.5) / M
                q = sigma * np.expm1(-k * np.log1p(-p)) / k if sigma > 0 else np.full(M, np.nan)
                lw[tail] = np.log(q + np.exp(cutoff))
    return np.minimum(lw, 0.0), k


def loo_summary(elpd, lppd, k, R):
    N = len(elpd)
    return np.array([elpd.sum(), np.sqrt(N * np.var(elpd, ddof=1)), np.sum(lppd - elpd), lppd.sum(), k.max(),
                     float(np.sum(k > k_threshold(R)))])


def loo_reference(mu, sigma2, A, y):
    """Definition of include/hmcgpu.h for one window: elpd, lppd, pareto_k, pit [N] and the summary row [6]; NaN everywhere
    when a draw is not finite."""
    N = len(y)
    if not all(np.all(np.isfinite(a)) for a in (mu, sigma2, A)):
        return (*(np.full(N, np.nan) for _ in range(4)), np.full(6, np.nan))
    ell, F = loo_terms(mu, sigma2, A, y)
    R = ell.shape[0]
    elpd, lppd, pk, pit = np.array([loo_date(ell[:, t], F[:, t]) for t in range(N)]).T
    return elpd, lppd, pk, pit, loo_summary(elpd, lppd, pk, R)


def loo_date(ell, F):
    """elpd, lppd, pareto_k and pit of one date from its pointwise terms ell [R] and F [R]."""
    lw, k = psis(-ell)
    W = np.exp(lw - logsumexp(lw))
    return logsumexp(lw + ell) - logsumexp(lw), logsumexp(ell) - np.log(len(ell)), k, np.sum(W * F)


# ---------------------------------------------------------------------------------------------------------------- CPU tests

def _draws(rng, R, K):
    mu = np.sort(rng.normal(0, 3, size=(R, K)), axis=1)
    sigma2 = rng.uniform(0.3, 3.0, size=(R, K))
    A = rng.dirichlet(np.ones(K) * 2.0, size=(R, K))
    return mu, sigma2, A


def _brute(mu, s2, A, y):
    """log p(y_t | y_-t) and P(Y_t <= y_t | y_-t) of one draw by enumeration of all K^N paths from the uniform start."""
    K, N = len(mu), len(y)
    sd = np.sqrt(s2)
    phi = norm.pdf(y[:, None], mu[None], sd[None])                     # [N, K]
    cdf = norm.cdf(y[:, None], mu[None], sd[None])
    ell, F = np.empty(N), np.empty(N)
    paths = np.array(list(itertools.product(range(K), repeat=N)))
    prior = np.full(len(paths), 1.0 / K)
    for t in range(1, N):
        prior *= A[paths[:, t - 1], paths[:, t]]
    lik = np.prod(phi[np.arange(N), paths], axis=1)
    for t in range(N):
        rest = prior * lik / phi[t, paths[:, t]]                        # p(path, y_-t)
        ell[t] = np.log(np.sum(prior * lik)) - np.log(np.sum(rest))
        F[t] = np.sum(rest * cdf[t, paths[:, t]]) / np.sum(rest)
    return ell, F


@pytest.mark.parametrize("K,N", [(2, 6), (3, 5)])
def test_terms_match_brute_force_enumeration(K, N):
    rng = np.random.default_rng(10 + K)
    mu, s2, A = _draws(rng, 3, K)
    y = rng.normal(0, 3, size=N)
    ell, F = loo_terms(mu, s2, A, y)
    for d in range(3):
        be, bF = _brute(mu[d], s2[d], A[d], y)
        np.testing.assert_allclose(ell[d], be, rtol=1e-12, atol=1e-13)
        np.testing.assert_allclose(F[d], bF, rtol=1e-12, atol=1e-14)


def test_last_date_is_the_one_step_term():
    rng = np.random.default_rng(11)
    mu, s2, A = _draws(rng, 7, 3)
    y = rng.normal(0, 3, size=30)
    ell, F = loo_terms(mu, s2, A, y)
    oe, oF = onestep_terms(mu, s2, A, y)
    np.testing.assert_allclose(ell[:, -1], oe[:, -1], rtol=1e-13)
    np.testing.assert_allclose(F[:, -1], oF[:, -1], rtol=1e-13, atol=1e-15)
    assert np.max(np.abs(ell[:, :-1] - oe[:, :-1])) > 1e-3          # earlier dates are conditioned on later ones too


def test_equal_states_and_identical_draws():
    """K states with one mu and sigma2: the term is the normal density and the LOO-PIT Phi(z); identical draws give uniform
    weights (a constant tail: k̂ = inf, elpd = lppd)."""
    rng = np.random.default_rng(12)
    R, K = 40, 3
    y = rng.normal(1.0, 2.0, size=25)
    mu, s2 = np.full((R, K), 1.3), np.full((R, K), 2.5)
    A = np.repeat(rng.dirichlet(np.ones(K), size=(1, K)), R, axis=0)
    ell, F = loo_terms(mu, s2, A, y)
    np.testing.assert_allclose(ell, np.broadcast_to(norm.logpdf(y, 1.3, np.sqrt(2.5)), ell.shape), rtol=1e-13)
    np.testing.assert_allclose(F, np.broadcast_to(norm.cdf(y, 1.3, np.sqrt(2.5)), F.shape), atol=1e-14)
    lw, k = psis(-ell[:, 0])
    assert k == np.inf and np.all(lw == 0.0)
    elpd, lppd, pk, pit, summ = loo_reference(mu, s2, A, y)
    np.testing.assert_allclose(elpd, lppd, rtol=1e-13)
    assert np.all(np.isinf(pk)) and summ[5] == len(y)


def test_observation_fifty_sd_out_stays_finite():
    mu, s2 = np.array([[0.0, 1.0]]), np.ones((1, 2))
    A = np.array([[[0.9, 0.1], [0.2, 0.8]]])
    y = np.array([0.2, 0.5, 50.0, 0.3, 1.1])
    ell, F = loo_terms(mu, s2, A, y)
    assert np.all(np.isfinite(ell)) and np.all(np.isfinite(F))
    be, bF = _brute(mu[0], s2[0], A[0], np.array([0.2, 0.5, 5.0, 0.3, 1.1]))
    assert np.isfinite(be).all()
    assert ell[0, 2] < -1000 and abs(F[0, 2] - 1.0) < 1e-15


@pytest.mark.parametrize("k_true", [0.2, 0.5, 0.9])
def test_khat_on_exact_gpd_tails(k_true):
    """Ratios whose exponentials are generalised Pareto with shape k: k̂ lands within 0.06 of k (R = 100 000).  (The fit's spread
    over seeds is ~0.04 here, and the prior pulls k̂ towards 0.5; seed 0 gives 0.23 / 0.525 / 0.914.)"""
    rng = np.random.default_rng(0)
    u = rng.uniform(size=100_000)
    r = np.log(((1 - u) ** -k_true - 1) / k_true)
    _, k = psis(r)
    assert abs(k - k_true) < 0.06, k


def test_degenerate_branches():
    """M < 5 (R <= 24): no smoothing, k̂ = inf; a constant tail: no smoothing, k̂ = inf; both truncate nothing."""
    rng = np.random.default_rng(13)
    assert psis_tail_len(24) == 5 and psis_tail_len(20) == 4
    r = rng.normal(size=20)
    lw, k = psis(r)
    assert k == np.inf and np.array_equal(lw, r - r.max())
    r = np.concatenate([rng.normal(size=900), np.full(100, 10.0)])  # the M = 95 largest all equal
    lw, k = psis(r)
    assert k == np.inf and np.array_equal(lw, r - 10.0)


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    exe = tmp_path_factory.mktemp("psis") / "psis_driver"
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), "-I", CSRC,
                           "-o", str(exe), os.path.join(ROOT, "tests", "psis_driver.cpp")])
    return str(exe)


def _run_psis(driver, r):
    out = subprocess.run([driver, "psis"], input=f"{len(r)}\n" + "\n".join(repr(float(v)) for v in r), capture_output=True,
                         text=True, check=True, timeout=120).stdout.split()
    return np.array([float(v) for v in out[1:]]), float(out[0])


@pytest.mark.parametrize("case", ["normal", "student2", "heavy", "ties", "small"])
def test_header_matches_numpy(driver, case):
    rng = np.random.default_rng({"normal": 1, "student2": 2, "heavy": 3, "ties": 4, "small": 5}[case])
    r = {"normal": lambda: rng.normal(size=4000), "student2": lambda: rng.standard_t(2, size=3000),
         "heavy": lambda: np.log(rng.pareto(0.7, size=5000) + 1e-3), "ties": lambda: np.round(rng.normal(size=2000), 1),
         "small": lambda: rng.normal(size=30)}[case]()
    lw, k = psis(r)
    dlw, dk = _run_psis(driver, r)
    assert (np.isinf(k) and np.isinf(dk)) or abs(dk - k) < 1e-12 * max(1.0, abs(k)), (k, dk)   # (sums in another order)
    np.testing.assert_allclose(dlw, lw, rtol=1e-12, atol=1e-12)
    for R in (2, 24, 25, 2000, 1 << 24):
        M, m, thr = subprocess.run([driver, "params", str(R)], capture_output=True, text=True, check=True).stdout.split()
        assert int(M) == psis_tail_len(R) and int(m) == 30 + int(np.sqrt(int(M))) and abs(float(thr) - k_threshold(R)) < 1e-15
    assert psis_tail_len(1 << 24) == 12288


def test_non_finite_draw_poisons_the_window():
    rng = np.random.default_rng(14)
    mu, s2, A = _draws(rng, 30, 3)
    s2[4, 1] = np.inf
    assert all(np.all(np.isnan(o)) for o in loo_reference(mu, s2, A, rng.normal(size=12)))


def test_flag_constant_struct_and_symbols_match_header(H, tmp_path):
    from hmc_jl_b200 import binding as B
    from test_host import _C2CTYPES, _C2JULIA, _c_offsets, _header_struct_fields
    header = open(os.path.join(ROOT, "include", "hmcgpu.h")).read()
    jl = open(os.path.join(ROOT, "hmc.jl_b200", "julia", "HmcGPU.jl")).read()
    assert int(re.search(r"#define HMCGPU_FLAG_LOO\s+(\d+)u", header).group(1)) == B.FLAG_LOO == H.FLAG_LOO == 2048
    assert re.search(r"const FLAG_LOO = UInt32\(2048\)", jl)
    for sym in ("hmcgpu_estimate_loo", "hmcgpu_estimate_multi_loo", "hmcgpu_plan_fetch_loo"):
        assert sym in B.SYMBOLS and re.search(r"\b%s\(" % sym, header) and re.search(r":%s\b" % sym, jl)
    assert len(B.SYMBOLS) == len(set(B.SYMBOLS)) == 35
    fields = _header_struct_fields("hmcgpu_loo")
    off = _c_offsets(tmp_path, "hmcgpu_loo", fields)
    assert [f for f, _ in B.Loo._fields_] == [f for _, f in fields] == ["elpd", "lppd", "pareto_k", "pit", "summary"]
    assert ctypes.sizeof(B.Loo) == off["sizeof"]
    for (ctype, f), (_, pytype) in zip(fields, B.Loo._fields_):
        assert getattr(B.Loo, f).offset == off[f] and pytype.__name__ == _C2CTYPES[ctype], f
    body = re.search(r"struct Loo\n(.*?)\nend", jl, re.S).group(1)
    jfields = [tuple(x.strip().split("::")) for ln in body.splitlines() for x in ln.split(";") if x.strip()]
    assert jfields == [(f, _C2JULIA[ctype]) for ctype, f in fields]
    assert H.load().hmcgpu_version() == 600


def test_binding_allocates_and_splits_per_window(H):
    y = np.random.default_rng(0).normal(size=60)
    spec = H.ProblemSpec(y, [1, 5, 2], [50, 30, 41], K=3, nrun=8, flags=H.FLAG_SUMMARY)
    o, _ = spec.alloc_result()
    assert spec.alloc_loo(o) is None and not hasattr(o, "loo_elpd")
    spec = H.ProblemSpec(y, [1, 5, 2], [50, 30, 41], K=3, nrun=8, flags=H.FLAG_LOO)
    o, res = spec.alloc_result()
    lo = spec.alloc_loo(o)
    assert o.loo_elpd.shape == o.loo_lppd.shape == o.pareto_k.shape == o.loo_pit.shape == (50 + 26 + 40,)
    assert o.loo.shape == (3, 6) and lo.elpd and lo.summary
    o.pareto_k[:] = np.arange(o.pareto_k.size)
    spec.finish(o, res, 0)
    assert [len(a) for a in o.pareto_k] == [50, 26, 40] and o.pareto_k[1][0] == 50 and o.pareto_k[2][-1] == 115
    assert [len(a) for a in o.loo_pit] == [50, 26, 40]


def _fake_fit(rng, lens, shift=0.0):
    from types import SimpleNamespace
    elpd = [rng.normal(-1.5, 0.4, size=n) + shift for n in lens]
    lppd = [e + rng.uniform(0.0, 0.05, size=len(e)) for e in elpd]
    k = [rng.uniform(-0.2, 0.9, size=n) for n in lens]
    loo = np.array([loo_summary(e, l, kk, 2000) for e, l, kk in zip(elpd, lppd, k)])
    return SimpleNamespace(loo_elpd=elpd, loo_lppd=lppd, pareto_k=k, loo_pit=[rng.uniform(size=n) for n in lens], loo=loo)


def test_compare_loo_and_write_loo(H, tmp_path, monkeypatch):
    from hmc_jl_b200 import api, binding as B
    rng = np.random.default_rng(4)
    a, b = _fake_fit(rng, [30, 45]), _fake_fit(rng, [30, 45], shift=-0.2)
    c = H.compare_loo(a, b)
    for w in range(2):
        e = a.loo_elpd[w] - b.loo_elpd[w]
        np.testing.assert_allclose(c.elpd_diff[w], e.sum(), rtol=1e-12)
        np.testing.assert_allclose(c.elpd_diff[w], a.loo[w, 0] - b.loo[w, 0], rtol=1e-12)
        np.testing.assert_allclose(c.se_diff[w], np.sqrt(len(e) * np.var(e, ddof=1)), rtol=1e-12)
    assert np.all(c.elpd_diff > 0)
    with pytest.raises(ValueError, match="same windows"):
        H.compare_loo(a, _fake_fit(rng, [30, 44]))

    seen = {}

    class FakeCtx:
        def close(self):
            pass

    monkeypatch.setattr(B, "estimate", lambda ctx, spec: seen.setdefault("spec", spec))
    api.estimate_windows(rng.normal(size=40), [1], [30], K=2, nrun=10, loo=True, ctx=FakeCtx())
    assert seen["spec"].flags & B.FLAG_LOO

    out = _fake_fit(np.random.default_rng(5), [3, 2])
    paths = H.write_loo(out, ["2001-01", "2001-06"], str(tmp_path))
    lines = open(paths["scores"]).read().splitlines()
    assert lines[0] == "date,t,elpd,lppd,pareto_k,pit" and len(lines) == 1 + 5
    assert [ln.split(",")[:2] for ln in lines[1:]] == [["2001-01", "1"], ["2001-01", "2"], ["2001-01", "3"], ["2001-06", "1"], ["2001-06", "2"]]
    got = np.loadtxt(paths["scores"], delimiter=",", skiprows=1, usecols=(2, 3, 4, 5))
    want = np.column_stack([np.concatenate(v) for v in (out.loo_elpd, out.loo_lppd, out.pareto_k, out.loo_pit)])
    np.testing.assert_array_equal(got, want)
    w = open(paths["loo"]).read().splitlines()
    assert w[0] == "date,elpd_loo,se,p_loo,lppd,max_k,n_high_k" and [ln.split(",")[0] for ln in w[1:]] == ["2001-01", "2001-06"]
    np.testing.assert_array_equal(np.loadtxt(paths["loo"], delimiter=",", skiprows=1, usecols=range(1, 7)), out.loo)


OUTLIER_T, OUTLIER_AT, OUTLIER_SHIFT = 300, 150, 60.0


def _outlier_series():
    y, _ = synth_hmm(OUTLIER_T, **K3_TRUTH, seed=41)
    y[OUTLIER_AT] += OUTLIER_SHIFT
    return y


def _check_outlier(pk, pit, R):
    assert int(np.argmax(pk)) == OUTLIER_AT, (np.argmax(pk), np.sort(pk)[-3:])
    assert pk[OUTLIER_AT] > k_threshold(R), pk[OUTLIER_AT]
    assert pit[OUTLIER_AT] > 0.999, pit[OUTLIER_AT]


def test_outlier_margin_with_the_oracle_chain(oracle):
    """The margin the GPU outlier test relies on, taken with the reference sampler (the oracle) and the numpy definition: one
    date of T = 300 from the three-state truth shifted by +60 has the largest k̂, above the threshold, and a LOO-PIT above 0.999
    (K = 3, 4 chains x 500 draws).  Nothing is asserted about the other dates, whose largest k̂ sits near the threshold."""
    y = _outlier_series()
    outs, _ = oracle.gibbs_batch([dict(y=y, K=3, burnin=1000, nrun=500, seed=21, chain=c, horizons=(1,)) for c in range(4)])
    mu, s2, A = (np.concatenate([getattr(o, f) for o in outs]) for f in ("mu", "sigma2", "A"))
    elpd, lppd, pk, pit, _ = loo_reference(mu, s2, A, y)
    _check_outlier(pk, pit, len(mu))


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


def _window_reference(o, spec, y, w):
    yw = y[spec.win_start[w] - 1:spec.win_end[w]]
    return loo_reference(o.mu[w].T, o.sigma2[w].T, o.A[w].transpose(2, 1, 0), yw)


def _check_against_reference(o, spec, y):
    """Every output of every window against loo_reference applied to the call's returned draws.  fp64: 1e-9 relative, k̂ 1e-9
    absolute.  fp32: the device filters in fp32 against the fp64 definition; a near-tie can move a draw across the tail boundary,
    so k̂ is bounded separately."""
    fp64 = spec.precision == 64
    R = spec.n_chains * spec.nrun
    for w in range(spec.n_windows):
        elpd, lppd, pk, pit, summ = _window_reference(o, spec, y, w)
        msg = f"window {w}"
        if fp64:
            np.testing.assert_allclose(o.loo_elpd[w], elpd, rtol=1e-9, err_msg=msg)
            np.testing.assert_allclose(o.loo_lppd[w], lppd, rtol=1e-9, err_msg=msg)
            np.testing.assert_allclose(o.pareto_k[w], pk, rtol=0, atol=1e-9, err_msg=msg)
            np.testing.assert_allclose(o.loo_pit[w], pit, rtol=1e-9, atol=1e-12, err_msg=msg)
            np.testing.assert_allclose(o.loo[w], summ, rtol=1e-9, atol=1e-9, err_msg=msg)
        else:
            n = len(elpd)
            np.testing.assert_allclose(o.loo_elpd[w], elpd, rtol=0, atol=FP32_TOL["elpd"], err_msg=msg)
            np.testing.assert_allclose(o.loo_lppd[w], lppd, rtol=0, atol=FP32_TOL["lppd"], err_msg=msg)
            np.testing.assert_allclose(o.pareto_k[w], pk, rtol=0, atol=FP32_TOL["k"], err_msg=msg)
            np.testing.assert_allclose(o.loo_pit[w], pit, rtol=0, atol=FP32_TOL["pit"], err_msg=msg)
            np.testing.assert_allclose(o.loo[w, [0, 3]], summ[[0, 3]], rtol=0, atol=FP32_TOL["elpd"] * n, err_msg=msg)
            np.testing.assert_allclose(o.loo[w, 1], summ[1], rtol=1e-5, err_msg=msg)                          # se
            np.testing.assert_allclose(o.loo[w, 2], summ[2], rtol=0, atol=2 * FP32_TOL["elpd"] * n, err_msg=msg)  # p_loo
            np.testing.assert_allclose(o.loo[w, 4], summ[4], rtol=0, atol=FP32_TOL["k"], err_msg=msg)          # max k̂
            assert o.loo[w, 5] == np.sum(o.pareto_k[w] > k_threshold(R))
        assert np.all(np.isfinite(o.loo_elpd[w])) and np.all((o.loo_pit[w] >= 0) & (o.loo_pit[w] <= 1 + 1e-12))


# fp32 against the fp64 definition, absolute: about 8 times the largest error seen on a B200 over these cases (elpd 7.8e-7,
# lppd 6.0e-7, k̂ 1.0e-5, pit 1.3e-7)
FP32_TOL = dict(elpd=6e-6, lppd=5e-6, k=1e-4, pit=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,precision,nrun,K,ranked", [
    ("thread", 32, 1501, 3, False), ("thread", 64, 2049, 3, False), ("scan", 32, 2049, 3, False), ("scan", 64, 1501, 3, True),
    ("seg", 32, 1501, 3, True), ("seg", 64, 2049, 3, False), ("thread", 32, 1501, 2, False), ("thread", 32, 1501, 5, True),
    ("thread", 64, 1501, 6, False), ("thread", 32, 2049, 8, False), ("thread", 64, 1501, 8, True), ("lane", 32, 1501, 5, False),
    ("lane", 64, 1501, 7, False), ("lane", 32, 2049, 8, True), ("lane", 64, 1501, 8, False), ("thread", 64, 1501, 4, True)])
def test_device_matches_reference(H, ctx, monkeypatch, kernel, precision, nrun, K, ranked):
    """nrun = 1501 / 2049: two and three draw chunks; windows of 88, 66 and 41 dates; with and without HMCGPU_FLAG_RANKED."""
    _force(monkeypatch, kernel)
    y = _series()
    spec = H.ProblemSpec(y, [1, 5, 20], [88, 70, 60], K=K, n_chains=3, burnin=30, nrun=nrun, seed=11, horizons=(1,),
                         precision=precision, quantile_probs=[0.5] if ranked else None,
                         flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOO | (H.FLAG_RANKED if ranked else 0))
    o = H.estimate(ctx, spec)
    assert o.sweep_kernel == _KERNELS[kernel]
    _check_against_reference(o, spec, y)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["thread", "lane"])
def test_flag_changes_nothing_else(H, ctx, monkeypatch, kernel):
    """Every other output is bit-identical with and without HMCGPU_FLAG_LOO; the flag adds exactly one launch per draw chunk
    (nrun = 2049: three chunks), and none when HMCGPU_FLAG_RANKED keeps the draws already."""
    _force(monkeypatch, kernel)
    base = H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY | H.FLAG_LOGLIK | H.FLAG_DIAGNOSTICS | H.FLAG_ONESTEP
    K = 5 if kernel == "lane" else 3
    for extra in (0, H.FLAG_RANKED):
        outs = []
        for flag in (0, H.FLAG_LOO):
            spec = H.ProblemSpec(_series(), [1, 9], [80, 61], K=K, n_chains=5, burnin=20, nrun=2049, seed=3, horizons=(2,),
                                 precision=32, flags=base | extra | flag, quantile_probs=[0.1, 0.9] if extra else None)
            outs.append(H.estimate(ctx, spec))
        a, b = outs
        assert b.n_sweep_launches == a.n_sweep_launches and b.n_launches == a.n_launches + (0 if extra else 3)
        names = ["mu", "sigma2", "A", "pi_end", "forecasts", "loglik", "summary_mean", "summary_var", "status", "rhat", "ess",
                 "ess_lag", "onestep_pit", "lpd", "lpd_var", "waic"] + (["quantiles", "rhat_rank", "ess_bulk", "ess_tail"] if extra else [])
        for name in names:
            x, z = getattr(a, name), getattr(b, name)
            if isinstance(x, list):
                for u, v in zip(x, z):
                    np.testing.assert_array_equal(u, v, err_msg=name)
            else:
                np.testing.assert_array_equal(x, z, err_msg=name)
        assert a.events == b.events and not hasattr(a, "loo_elpd") and all(np.all(np.isfinite(x)) for x in b.loo_elpd)


@pytest.mark.gpu
def test_batching_chunking_and_multi_invariance(H, ctx, monkeypatch):
    """A window's outputs are bit-identical alone, in a ragged batch, across two runs of one plan (and a second fetch), through
    hmcgpu_estimate_multi_loo on two contexts, and when the fetch cuts the dates into batches of four (HMCGPU_LOO_SCRATCH_MB=1:
    R = 8196 draws x 28 bytes per date), which splits windows across batches."""
    _force(monkeypatch, "thread")
    y = _series()
    names = ("loo_elpd", "loo_lppd", "pareto_k", "loo_pit")
    kw = dict(K=3, n_chains=4, burnin=20, nrun=2049, seed=9, horizons=(1, 12), precision=32, flags=H.FLAG_REF_Q1 | H.FLAG_LOO)
    starts, ends = [1, 1, 30, 1, 12], [85, 40, 77, 66, 90]

    def same(a, wa, b, wb):
        for n in names:
            np.testing.assert_array_equal(getattr(a, n)[wa], getattr(b, n)[wb], err_msg=n)
        np.testing.assert_array_equal(a.loo[wa], b.loo[wb])

    batch = H.estimate(ctx, H.ProblemSpec(y, starts, ends, win_id=np.arange(5), **kw))
    for w in (0, 2, 4):
        same(H.estimate(ctx, H.ProblemSpec(y, [starts[w]], [ends[w]], win_id=[w], **kw)), 0, batch, w)
    spec = H.ProblemSpec(y, starts, ends, **kw)
    plan = H.Plan(ctx, spec)
    try:
        plan.run()
        first = plan.fetch()
        refetch = plan.fetch()
        plan.run()
        again = plan.fetch()
    finally:
        plan.close()
    multi = H.estimate_multi([0, 0], spec)
    monkeypatch.setenv("HMCGPU_LOO_SCRATCH_MB", "1")
    small = H.estimate(ctx, spec)
    monkeypatch.delenv("HMCGPU_LOO_SCRATCH_MB")
    for w in range(5):
        same(first, w, batch, w)
        same(refetch, w, batch, w)
        same(again, w, batch, w)
        same(multi, w, batch, w)
        same(small, w, batch, w)


@pytest.mark.gpu
def test_more_pieces_than_one_launch_holds(H, ctx, monkeypatch):
    """70 000 windows of a few draws fit one batch of dates: more pieces than one launch of loo_terms_kernel holds (65 535 grid
    rows).  Windows of the second launch are bit-identical to the same windows alone."""
    _force(monkeypatch, "thread")
    y = _series()
    nw = 70_000
    starts = 1 + np.arange(nw) % 40
    kw = dict(K=2, n_chains=1, burnin=5, nrun=4, seed=5, horizons=(1,), precision=32, flags=H.FLAG_REF_Q1 | H.FLAG_LOO)
    wide = H.estimate(ctx, H.ProblemSpec(y, starts, starts + 9, win_id=np.arange(nw), **kw))
    assert all(np.all(np.isfinite(x)) for x in wide.loo_elpd[::997])
    for w in (3, 65_534, 65_535, 65_536, nw - 1):
        alone = H.estimate(ctx, H.ProblemSpec(y, [starts[w]], [starts[w] + 9], win_id=[w], **kw))
        for n in ("loo_elpd", "loo_lppd", "pareto_k", "loo_pit"):
            np.testing.assert_array_equal(getattr(alone, n)[0], getattr(wide, n)[w], err_msg=f"{n} window {w}")


@pytest.fixture(scope="module")
def psis_device(tmp_path_factory):
    """tests/loo_psis_driver.cu built with nvcc for sm_100a: loo_psis_kernel on given pointwise terms."""
    from hmc_jl_b200 import build as Bld
    exe = tmp_path_factory.mktemp("loo_psis") / "loo_psis_driver"
    subprocess.check_call([Bld.NVCC, "-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-std=c++17", "-I", os.path.join(ROOT, "include"),
                           "-I", CSRC, "-o", str(exe), os.path.join(ROOT, "tests", "loo_psis_driver.cu")])

    def run(ell, F):
        n, R = ell.shape
        text = f"{R} {n}\n" + "\n".join(" ".join(repr(float(v)) for v in np.concatenate([ell[j], F[j]])) for j in range(n))
        out = subprocess.run([str(exe)], input=text, capture_output=True, text=True, check=True, timeout=300).stdout
        return np.array([[float(v) for v in ln.split()] for ln in out.splitlines()])
    return run


@pytest.mark.gpu
def test_psis_kernel_on_given_terms(psis_device):
    """loo_psis_kernel against loo_date on ratio sets chosen here: light and heavy tails, rounded values with ties, a constant
    tail, R < 25 (no smoothing), and a tail of which more than M/4 values tie with the cutoff while the rest spread above it
    (x* = 0: the fit gives NaN, k̂ = inf, and the tail keeps its own log ratios)."""
    rng = np.random.default_rng(8)
    R = 2000
    M = psis_tail_len(R)
    tie = np.concatenate([rng.normal(-3.0, 0.5, size=R - M - 25), np.full(60, -1.0), rng.uniform(-0.9, 2.0, size=M - 35)])
    assert np.sum(tie > -1.0) == M - 35 and 35 >= int(np.floor(M / 4 + 0.5))
    cases = [rng.normal(size=R), rng.standard_t(2, size=R), np.log(rng.pareto(0.7, size=R) + 1e-3), np.round(rng.normal(size=R), 1),
             np.concatenate([rng.normal(size=R - 200), np.full(200, 9.0)]), rng.permutation(tie)]
    ell = -np.array(cases)                                            # the kernel's log ratios are -ell
    F = rng.uniform(size=ell.shape)
    got = psis_device(ell, F)
    want = np.array([loo_date(e, f) for e, f in zip(ell, F)])
    assert np.isinf(want[-1, 2]) and np.isinf(got[-1, 2])
    np.testing.assert_array_equal(np.isinf(got[:, 2]), np.isinf(want[:, 2]))
    fin = np.isfinite(want[:, 2])
    np.testing.assert_allclose(got[fin, 2], want[fin, 2], rtol=0, atol=1e-9)
    np.testing.assert_allclose(got[:, [0, 1, 3]], want[:, [0, 1, 3]], rtol=1e-9, atol=1e-12)
    small = psis_device(-rng.normal(size=(3, 20)), rng.uniform(size=(3, 20)))
    assert np.all(np.isinf(small[:, 2]))


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [64, 32])
def test_fifty_sd_observation_on_the_device(H, ctx, precision):
    """One observation more than 50 sd from every state mean of every draw: every output stays finite and matches the numpy
    definition (fp64 to 1e-9; fp32 relative to the large log densities there, as test_onestep's far outlier).  Left to the data,
    the sampler widens a state to cover the outlier; strong priors (alpha = nu = 10^4 per state, beta = alpha sigma2 of the
    truth, xi its means) hold every draw near the three-state truth, ~100 sd from y = 300."""
    y = _series()
    y[40] = 300.0
    n = np.full(3, 1e4)
    spec = H.ProblemSpec(y, [1, 10], [88, 80], K=3, n_chains=2, burnin=30, nrun=300, seed=4, horizons=(1,), precision=precision,
                         xi=K3_TRUTH["mu"], alpha=n, nu=n, beta0=n * K3_TRUTH["sigma2"], beta=n * K3_TRUTH["sigma2"],
                         flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOO)
    o = H.estimate(ctx, spec)
    for w in range(2):
        mu, s2 = o.mu[w].T, o.sigma2[w].T
        assert np.all(np.abs(300.0 - mu) / np.sqrt(s2) > 50)
        assert all(np.all(np.isfinite(a[w])) for a in (o.loo_elpd, o.loo_lppd, o.loo_pit)) and np.all(np.isfinite(o.loo[w, :4]))
        elpd, lppd, pk, pit, summ = _window_reference(o, spec, y, w)
        if precision == 64:
            np.testing.assert_allclose(o.loo_elpd[w], elpd, rtol=1e-9)
            np.testing.assert_allclose(o.loo_lppd[w], lppd, rtol=1e-9)
            np.testing.assert_allclose(o.pareto_k[w], pk, rtol=0, atol=1e-9)
            np.testing.assert_allclose(o.loo_pit[w], pit, rtol=1e-9, atol=1e-12)
            np.testing.assert_allclose(o.loo[w], summ, rtol=1e-9, atol=1e-9)
        else:
            np.testing.assert_allclose(o.loo_elpd[w], elpd, rtol=1e-5, atol=2e-5)
            np.testing.assert_allclose(o.loo_lppd[w], lppd, rtol=1e-5, atol=2e-5)
            np.testing.assert_allclose(o.loo_pit[w], pit, rtol=0, atol=2e-5)
            np.testing.assert_allclose(o.pareto_k[w], pk, rtol=0, atol=0.05)


@pytest.mark.gpu
def test_refusals(H, ctx):
    import ctypes as C
    from hmc_jl_b200 import binding as B
    y = _series()
    kw = dict(K=3, n_chains=2, burnin=5, nrun=10, horizons=(1,), flags=H.FLAG_REF_Q1 | H.FLAG_LOO)

    def message():
        return ctx.L.hmcgpu_last_error(ctx.h).decode()

    def code(spec, **override):
        prob = spec.struct()
        for k, v in override.items():
            setattr(prob, k, v)
        o, res = spec.alloc_result()
        lo = spec.alloc_loo(o)
        return ctx.L.hmcgpu_estimate_loo(ctx.h, C.byref(prob), C.byref(res), None, None, None, C.byref(lo))

    ok = H.ProblemSpec(y, [1], [60], **kw)
    assert code(ok) >= 0
    assert code(ok, n_chains=1, nrun=1) == B.ERR_ARG and "n_chains * nrun >= 2" in message()
    assert code(ok, n_chains=2, nrun=(1 << 23) + 1) == B.ERR_ARG and "2^24" in message()
    assert code(H.ProblemSpec(y, [1], [60], **{**kw, "K": 9})) == B.ERR_UNSUPPORTED and "K <= 8" in message()
    mask = np.zeros(len(y), dtype=np.uint8)
    mask[50:55] = 1
    assert code(H.ProblemSpec(y, [1], [60], is_signal=mask, **kw)) == B.ERR_UNSUPPORTED and "is_signal" in message()
    assert code(H.ProblemSpec(y, [1], [60], pi_row_back=2, **kw)) >= 0
    # the kept draws of a shape far beyond the device: refused at plan_create, before anything is allocated
    big = H.ProblemSpec(y, [1] * 2000, [60] * 2000, **{**kw, "n_chains": 4096, "nrun": 4096})
    h = C.c_void_p()
    prob = big.struct()
    assert ctx.L.hmcgpu_plan_create(ctx.h, C.byref(prob), C.byref(h)) == B.ERR_ALLOC and "HMCGPU_FLAG_LOO" in message()
    # the flag through every entry point without LOO outputs
    prob, (o, res) = ok.struct(), ok.alloc_result()
    assert ctx.L.hmcgpu_estimate(ctx.h, C.byref(prob), C.byref(res)) == B.ERR_ARG and "hmcgpu_loo" in message()
    assert ctx.L.hmcgpu_estimate_predictive(ctx.h, C.byref(prob), C.byref(res), None) == B.ERR_ARG and "hmcgpu_loo" in message()
    assert ctx.L.hmcgpu_estimate_ranked(ctx.h, C.byref(prob), C.byref(res), None, None) == B.ERR_ARG and "hmcgpu_loo" in message()
    assert ctx.L.hmcgpu_estimate_onestep(ctx.h, C.byref(prob), C.byref(res), None, None, None) == B.ERR_ARG and "hmcgpu_loo" in message()
    dev = (C.c_int * 1)(0)
    for call in (lambda: ctx.L.hmcgpu_estimate_multi(dev, 1, C.byref(prob), C.byref(res)),
                 lambda: ctx.L.hmcgpu_estimate_multi_predictive(dev, 1, C.byref(prob), C.byref(res), None),
                 lambda: ctx.L.hmcgpu_estimate_multi_ranked(dev, 1, C.byref(prob), C.byref(res), None, None),
                 lambda: ctx.L.hmcgpu_estimate_multi_onestep(dev, 1, C.byref(prob), C.byref(res), None, None, None),
                 lambda: ctx.L.hmcgpu_estimate_multi_loo(dev, 1, C.byref(prob), C.byref(res), None, None, None, None)):
        assert call() == B.ERR_ARG and "hmcgpu_loo" in ctx.L.hmcgpu_last_error(None).decode()
    # fetch on a plan without the flag, and before a run
    plan = H.Plan(ctx, H.ProblemSpec(y, [1], [60], **{**kw, "flags": H.FLAG_REF_Q1}))
    lo = B.Loo()
    try:
        plan.run()
        assert ctx.L.hmcgpu_plan_fetch_loo(plan.h, C.byref(lo)) == B.ERR_ARG and "without HMCGPU_FLAG_LOO" in message()
    finally:
        plan.close()
    plan = H.Plan(ctx, ok)
    try:
        assert ctx.L.hmcgpu_plan_fetch_loo(plan.h, C.byref(lo)) == B.ERR_ARG and "before plan_run" in message()
    finally:
        plan.close()


@pytest.mark.gpu
@pytest.mark.parametrize("precision", [64, 32])
def test_outlier_on_the_device(H, ctx, precision):
    """The oracle-chain margin on the device: the shifted date has the largest k̂, above the threshold, and a LOO-PIT above
    0.999; every output stays finite next to an observation ~20 sd from every state."""
    y = _outlier_series()
    fit = H.estimate_windows(y, [1], [len(y)], K=3, n_chains=4, burnin=1000, nrun=500, seed=21, horizons=(1,), precision=precision,
                             summary=False, loo=True, ctx=ctx)
    _check_outlier(fit.pareto_k[0], fit.loo_pit[0], 2000)
    assert np.all(np.isfinite(fit.loo_elpd[0])) and np.all(np.isfinite(fit.loo))


@pytest.mark.gpu
def test_calibration_and_model_choice(H, ctx):
    """K = 3 fitted to 2000 dates from the three-state truth: the LOO-PIT is uniform (KS distance < 0.05).  On 1500 dates
    compare_loo(K = 3, K = 2) favours the true K by more than 4 se_diff."""
    kw = dict(n_chains=8, burnin=1000, nrun=500, seed=21, horizons=(1,), precision=32, summary=False, loo=True, ctx=ctx)
    y, _ = synth_hmm(2000, **K3_TRUTH, seed=32)
    fit = H.estimate_windows(y, [1], [len(y)], K=3, **kw)
    assert kstest(fit.loo_pit[0], "uniform").statistic < 0.05
    y, _ = synth_hmm(1500, **K3_TRUTH, seed=31)
    c = H.compare_loo(H.estimate_windows(y, [1], [len(y)], K=3, **kw), H.estimate_windows(y, [1], [len(y)], K=2, **kw))
    assert c.elpd_diff[0] > 4 * c.se_diff[0], (c.elpd_diff, c.se_diff)
