"""Posterior predictive distribution of every forecast (HMCGPU_FLAG_PREDICTIVE): the numpy definition the device must match,
its analytic cases, the host plumbing, and (with -m gpu) the device against that definition applied to the same call's draws."""
import ctypes
import os
import re

import numpy as np
import pytest
from scipy.special import ndtr
from scipy.stats import norm

from conftest import ROOT, K3_TRUTH, synth_hmm


def predictive_reference(mu, sigma2, A, pi_end, horizons, grid, y_plus, shift):
    """Definition of include/hmcgpu.h (hmcgpu_predictive) for one window.  mu, sigma2, pi_end [R, K], A [R, K, K] with
    A[d, r, s] = P(X_t = s | X_t-1 = r), y_plus [n_h] realised values (NaN past the series), shift = c_w.
    Returns cdf [n_h, n_grid], pit [n_h], log_score [n_h], moments [n_h, 3] (mean, variance, skewness)."""
    mu, sigma2, A, pi_end = (np.asarray(a, dtype=np.float64) for a in (mu, sigma2, A, pi_end))
    grid = np.asarray(grid, dtype=np.float64)
    sd = np.sqrt(sigma2)
    phi_grid = ndtr((grid[None, :, None] - mu[:, None, :]) / sd[:, None, :])         # [R, n_grid, K]
    nh = len(horizons)
    cdf, pit, ls, mom = np.empty((nh, len(grid))), np.empty(nh), np.empty(nh), np.empty((nh, 3))
    d = mu - shift
    for j, h in enumerate(horizons):
        v = pi_end.copy()
        for _ in range(int(h)):
            v = np.einsum("dr,drs->ds", v, A)
        cdf[j] = np.einsum("dgk,dk->g", phi_grid, v) / len(mu)
        pit[j] = np.mean(np.sum(v * ndtr((y_plus[j] - mu) / sd), axis=1))
        ls[j] = np.log(np.mean(np.sum(v * norm.pdf(y_plus[j], mu, sd), axis=1)))
        m1 = np.mean(np.sum(v * d, axis=1))
        m2 = np.mean(np.sum(v * (d * d + sigma2), axis=1))
        m3 = np.mean(np.sum(v * (d ** 3 + 3 * d * sigma2), axis=1))
        var = m2 - m1 * m1
        mom[j] = shift + m1, var, (m3 - 3 * m1 * m2 + 2 * m1 ** 3) / var ** 1.5
    return cdf, pit, ls, mom


def _draws(rng, R, K, level=0.0):
    mu = np.sort(level + rng.normal(0, 3, size=(R, K)), axis=1)
    sigma2 = rng.uniform(0.3, 3.0, size=(R, K))
    A = rng.dirichlet(np.ones(K) * 2.0, size=(R, K))
    pi = rng.dirichlet(np.ones(K), size=R)
    return mu, sigma2, A, pi


def test_one_state_is_a_normal():
    rng = np.random.default_rng(1)
    R, K = 1, 3
    mu, s2, A, _ = _draws(rng, R, K)
    A[:] = np.eye(K)                     # all weight stays on state 2 at every horizon
    pi = np.array([[0.0, 1.0, 0.0]])
    grid = np.linspace(-8, 8, 33)
    cdf, pit, ls, mom = predictive_reference(mu, s2, A, pi, [0, 3], grid, np.array([0.7, -1.2]), 0.0)
    sd = np.sqrt(s2[0, 1])
    np.testing.assert_allclose(cdf[1], norm.cdf(grid, mu[0, 1], sd), atol=1e-15)
    np.testing.assert_allclose(pit, norm.cdf([0.7, -1.2], mu[0, 1], sd), atol=1e-15)
    np.testing.assert_allclose(ls, norm.logpdf([0.7, -1.2], mu[0, 1], sd), rtol=1e-13)
    np.testing.assert_allclose(mom[0], [mu[0, 1], s2[0, 1], 0.0], atol=1e-12)


def test_identity_transition_keeps_pi_end():
    rng = np.random.default_rng(2)
    mu, s2, A, pi = _draws(rng, 50, 4)
    A[:] = np.eye(4)
    grid = np.linspace(-10, 10, 21)
    cdf, pit, ls, mom = predictive_reference(mu, s2, A, pi, [0, 7], grid, np.array([0.3, 0.3]), 0.5)
    np.testing.assert_array_equal(cdf[0], cdf[1])
    np.testing.assert_array_equal(mom[0], mom[1])
    direct = np.mean([np.sum(p * ndtr((grid[:, None] - m) / np.sqrt(s)), axis=1) for m, s, p in zip(mu, s2, pi)], axis=0)
    np.testing.assert_allclose(cdf[0], direct, atol=1e-15)


def test_mirror_symmetric_mixture_has_no_skew():
    mu = np.array([[-2.0, 2.0], [-1.0, 1.0]])
    s2 = np.array([[0.5, 0.5], [2.0, 2.0]])
    A = np.array([[[0.9, 0.1], [0.1, 0.9]]] * 2)
    pi = np.array([[0.5, 0.5], [0.5, 0.5]])
    cdf, _, _, mom = predictive_reference(mu, s2, A, pi, [0, 4], np.linspace(-3, 3, 7), np.array([0.0, 0.0]), 0.0)
    assert np.all(np.abs(mom[:, 2]) < 1e-14) and np.all(np.abs(mom[:, 0]) < 1e-15)
    np.testing.assert_allclose(cdf[:, 3], 0.5, atol=1e-15)            # symmetric about 0
    np.testing.assert_allclose(cdf[:, ::-1] + cdf, 1.0, atol=1e-14)


def test_moments_follow_the_law_of_total_variance():
    rng = np.random.default_rng(3)
    mu, s2, A, pi = _draws(rng, 400, 3)
    _, _, _, mom = predictive_reference(mu, s2, A, pi, [2], np.zeros(1), np.array([0.0]), 1.3)
    v = np.einsum("dr,drs->ds", np.einsum("dr,drs->ds", pi, A), A)
    cond_mean = np.sum(v * mu, axis=1)                                  # E[Y | draw, state mix]
    cond_var = np.sum(v * (s2 + mu ** 2), axis=1) - cond_mean ** 2
    np.testing.assert_allclose(mom[0, 0], cond_mean.mean(), rtol=1e-13)
    np.testing.assert_allclose(mom[0, 1], cond_var.mean() + cond_mean.var(), rtol=1e-12)
    # skewness of the pooled mixture from its exact central moments (two passes over every component)
    m = mom[0, 0]
    c3 = np.mean(np.sum(v * ((mu - m) ** 3 + 3 * (mu - m) * s2), axis=1))
    np.testing.assert_allclose(mom[0, 2], c3 / mom[0, 1] ** 1.5, rtol=1e-11)


def test_shift_keeps_level_series_exact():
    """Level 300 (the fp32 parity tests' 200/250/300 series): raw moments about c_w = 300 give the two-pass central moments to
    1e-12 (the skewness, near 0, to 1e-12 absolute); about 0 they cancel (mean and variance agree to 1e-9 only)."""
    rng = np.random.default_rng(4)
    mu, s2, A, pi = _draws(rng, 300, 3, level=300.0)
    mu = 300.0 + (mu - 300.0) * 0.3
    _, _, _, shifted = predictive_reference(mu, s2, A, pi, [1, 6], np.zeros(1), np.full(2, 300.0), 300.0)
    _, _, _, raw = predictive_reference(mu, s2, A, pi, [1, 6], np.zeros(1), np.full(2, 300.0), 0.0)
    for j, h in enumerate((1, 6)):
        v = pi
        for _ in range(h):
            v = np.einsum("dr,drs->ds", v, A)
        m = np.mean(np.sum(v * mu, axis=1))
        c2 = np.mean(np.sum(v * ((mu - m) ** 2 + s2), axis=1))
        c3 = np.mean(np.sum(v * ((mu - m) ** 3 + 3 * (mu - m) * s2), axis=1))
        np.testing.assert_allclose(shifted[j, :2], [m, c2], rtol=1e-12)
        np.testing.assert_allclose(shifted[j, 2], c3 / c2 ** 1.5, rtol=0, atol=1e-12)     # (a skewness near 0: absolute)
        np.testing.assert_allclose(raw[j, :2], shifted[j, :2], rtol=1e-9)


def test_flag_constant_matches_header_and_bindings(H):
    from hmc_jl_b200 import binding as B
    header = open(os.path.join(ROOT, "include", "hmcgpu.h")).read()
    jl = open(os.path.join(ROOT, "hmc.jl_b200", "julia", "HmcGPU.jl")).read()
    assert int(re.search(r"#define HMCGPU_FLAG_PREDICTIVE\s+(\d+)u", header).group(1)) == B.FLAG_PREDICTIVE == H.FLAG_PREDICTIVE == 256
    assert re.search(r"const FLAG_PREDICTIVE = UInt32\(256\)", jl)
    # the header's single-space constants (eleven of them, counted by test_host.py) do not include it
    single = dict(re.findall(r"#define HMCGPU_((?:FLAG|ERR)_\w+) \(?(-?\d+)u?\)?", header))
    assert "FLAG_PREDICTIVE" not in single and len(single) == 11
    for sym in ("hmcgpu_estimate_predictive", "hmcgpu_estimate_multi_predictive", "hmcgpu_plan_fetch_predictive"):
        assert sym in B.SYMBOLS and re.search(r"\b%s\(" % sym, header)


def test_predictive_struct_and_problem_tail_match_header(H, tmp_path):
    from hmc_jl_b200 import binding as B
    from test_host import _C2CTYPES, _C2JULIA, _c_offsets, _header_struct_fields
    jl = open(os.path.join(ROOT, "hmc.jl_b200", "julia", "HmcGPU.jl")).read()
    for cname, S in (("hmcgpu_predictive", B.Predictive), ("hmcgpu_problem", B.Problem)):
        fields = _header_struct_fields(cname)
        off = _c_offsets(tmp_path, cname, fields)
        assert [f for f, _ in S._fields_] == [f for _, f in fields]
        assert ctypes.sizeof(S) == off["sizeof"]
        for (ctype, f), (_, pytype) in zip(fields, S._fields_):
            assert getattr(S, f).offset == off[f], f
            assert pytype.__name__ == _C2CTYPES[ctype], f
        body = re.search(r"struct %s\n(.*?)\nend" % S.__name__, jl, re.S).group(1)
        jfields = [tuple(x.strip().split("::")) for ln in body.splitlines() for x in ln.split(";") if x.strip()]
        assert jfields == [(f, _C2JULIA[ctype]) for ctype, f in fields]
    assert [f for f, _ in B.Problem._fields_][-2:] == ["pred_grid", "n_grid"]
    assert [f for f, _ in B.Predictive._fields_] == ["cdf", "pit", "log_score", "moments"]


def test_binding_refuses_grid_without_flag_and_flag_without_grid(H):
    y = np.random.default_rng(0).normal(size=60)
    with pytest.raises(ValueError, match="without FLAG_PREDICTIVE"):
        H.ProblemSpec(y, [1], [50], K=3, nrun=8, flags=H.FLAG_SUMMARY, pred_grid=[0.0, 1.0])
    with pytest.raises(ValueError, match="needs pred_grid"):
        H.ProblemSpec(y, [1], [50], K=3, nrun=8, flags=H.FLAG_SUMMARY | H.FLAG_PREDICTIVE)
    spec = H.ProblemSpec(y, [1], [50], K=3, nrun=8, flags=H.FLAG_SUMMARY)
    o, _ = spec.alloc_result()
    assert spec.alloc_predictive(o) is None and spec.struct().n_grid == 0 and not spec.struct().pred_grid
    spec = H.ProblemSpec(y, [1, 2], [50, 55], K=3, nrun=8, horizons=(1, 12, 3), flags=H.FLAG_PREDICTIVE, pred_grid=np.arange(5.0))
    o, _ = spec.alloc_result()
    pr = spec.alloc_predictive(o)
    assert o.pred_cdf.shape == (2, 3, 5) and o.pit.shape == o.log_score.shape == (2, 3) and o.pred_moments.shape == (2, 3, 3)
    assert pr.cdf and pr.moments and spec.struct().n_grid == 5


def test_estimate_windows_and_write_predictive(H, tmp_path, monkeypatch):
    from hmc_jl_b200 import api, binding as B
    seen = {}

    class FakeCtx:
        def close(self):
            pass

    def fake_estimate(ctx, spec):
        seen["spec"] = spec
        o, _ = spec.alloc_result()
        spec.alloc_predictive(o)
        if spec.flags & B.FLAG_PREDICTIVE:
            for a in (o.pred_cdf, o.pit, o.log_score, o.pred_moments):
                a[:] = np.arange(a.size).reshape(a.shape) + 0.25
        return o

    monkeypatch.setattr(B, "estimate", fake_estimate)
    hz, grid = (1, 12), [-1.0, 0.5, 2.0]
    y = np.random.default_rng(0).normal(size=40)
    out = api.estimate_windows(y, [1, 1], [30, 35], K=2, n_chains=2, nrun=10, horizons=hz, predictive_grid=grid, ctx=FakeCtx())
    assert seen["spec"].flags & B.FLAG_PREDICTIVE and list(seen["spec"].pred_grid) == grid
    assert out.pred_cdf.shape == (2, 2, 3)
    api.estimate_windows(y, [1], [30], K=2, nrun=10, horizons=hz, ctx=FakeCtx())
    assert not seen["spec"].flags & B.FLAG_PREDICTIVE and seen["spec"].pred_grid is None

    dates = ["2001-01", "2001-06"]
    paths = H.write_predictive(out, hz, grid, dates, str(tmp_path))
    assert sorted(paths) == ["cdf_h1", "cdf_h12", "scores"]
    lines = open(paths["cdf_h12"]).read().splitlines()
    assert lines[0] == "date,-1.0,0.5,2.0" and [ln.split(",")[0] for ln in lines[1:]] == dates
    np.testing.assert_array_equal(np.loadtxt(paths["cdf_h12"], delimiter=",", skiprows=1, usecols=(1, 2, 3)), out.pred_cdf[:, 1, :])
    hdr = open(paths["scores"]).readline().strip().split(",")
    assert hdr == ["date"] + [f"{k}_{h}" for h in hz for k in ("pit", "log_score", "mean", "variance", "skewness")]
    got = np.loadtxt(paths["scores"], delimiter=",", skiprows=1, usecols=range(1, 11))
    for j in range(2):
        np.testing.assert_array_equal(got[:, 5 * j:5 * j + 5],
                                      np.column_stack([out.pit[:, j], out.log_score[:, j], out.pred_moments[:, j]]))
    # the gather of a per-window table across ranks is the summaries' gather
    flat = out.pred_cdf.reshape(2, -1)
    np.testing.assert_array_equal(H.gather_window_summaries(flat[::-1], np.array([1, 0]), 2), flat)


def test_predictive_quantiles_to_the_grid_spacing(H):
    grid = np.linspace(-9.0, 11.0, 401)
    step = grid[1] - grid[0]
    cdf = norm.cdf(grid, 1.0, 2.0)
    probs = np.array([0.01, 0.05, 0.25, 0.5, 0.75, 0.95, 0.99])
    q = H.predictive_quantiles(np.stack([cdf, cdf]), grid, probs)
    assert q.shape == (2, len(probs))
    assert np.all(np.abs(q - norm.ppf(probs, 1.0, 2.0)) < step)
    narrow = H.predictive_quantiles(norm.cdf(np.linspace(-1, 3, 41), 1.0, 2.0), np.linspace(-1, 3, 41), [0.05, 0.5, 0.95])
    assert np.isnan(narrow[0]) and np.isnan(narrow[2]) and abs(narrow[1] - 1.0) < 0.1
    assert np.all(np.isnan(H.predictive_quantiles(np.full(5, np.nan), np.arange(5.0), [0.5])))


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
    """Every output of every window equals predictive_reference applied to the call's returned draws."""
    K, hz, grid = spec.K, spec.horizons, spec.pred_grid
    for w in range(spec.n_windows):
        y = y_of_window(w)
        end = int(spec.win_end[w])
        yp = np.array([y[end + h - 1] if end + h <= len(y) else np.nan for h in hz])
        ref = predictive_reference(o.mu[w].T, o.sigma2[w].T, o.A[w].transpose(2, 1, 0), o.pi_end[w].T, hz, grid, yp, y[end - 1])
        np.testing.assert_allclose(o.pred_cdf[w], ref[0], atol=1e-10, rtol=0, err_msg=f"cdf window {w}")
        np.testing.assert_allclose(o.pit[w], ref[1], atol=1e-10, rtol=0, err_msg=f"pit window {w}")
        np.testing.assert_allclose(o.log_score[w], ref[2], rtol=1e-10, err_msg=f"log_score window {w}")
        np.testing.assert_allclose(o.pred_moments[w], ref[3], rtol=1e-10, atol=1e-13, err_msg=f"moments window {w}")
        assert np.all(np.isnan(o.pit[w]) == np.isnan(yp)) and np.all(np.isfinite(o.pred_cdf[w])) and np.all(np.isfinite(o.pred_moments[w]))


def _check_mean_against_summary(o, spec):
    """The predictive mean is the posterior mean of the forecast field (which the sweep kernel computes in the plan's
    precision: fp32 rounds each draw's forecast to ~1e-7)."""
    K, nh = spec.K, spec.n_h
    f0 = 3 * K + K * K
    rtol = 1e-12 if spec.precision == 64 else 1e-5
    np.testing.assert_allclose(o.pred_moments[:, :, 0], o.summary_mean[:, f0:f0 + 2 * nh:2], rtol=rtol)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,precision,nrun,K,n_grid", [
    ("thread", 32, 1501, 3, 40), ("thread", 64, 2049, 3, 300), ("scan", 32, 2049, 3, 40), ("scan", 64, 1501, 3, 64),
    ("seg", 32, 1501, 3, 33), ("seg", 64, 2049, 3, 40), ("thread", 32, 1501, 2, 40), ("lane", 32, 2049, 5, 64),
    ("lane", 64, 1501, 10, 17), ("lane", 32, 1501, 32, 40)])
def test_device_matches_reference(H, ctx, monkeypatch, kernel, precision, nrun, K, n_grid):
    """nrun = 1501 / 2049: two and three draw chunks.  The window ending at 88 has no y[88 + 12]: its h = 12 PIT and log score
    are NaN, its CDF and moments finite.  n_grid = 300 takes two grid points per thread.  The lane-per-state kernel runs K >= 5
    only (HMCGPU_LANE_KERNEL=1 moves K = 5..8 to it; K = 9..32 always use it), so K = 2 and 3 are covered by the other kernels."""
    _force(monkeypatch, kernel)
    y = _series()
    hz = (0, 1, 12)
    spec = H.ProblemSpec(y, [1, 5, 20], [88, 70, 60], K=K, n_chains=3, burnin=30, nrun=nrun, seed=11, horizons=hz,
                         precision=precision, pred_grid=np.linspace(-3.0, 14.0, n_grid),
                         flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY | H.FLAG_PREDICTIVE)
    o = H.estimate(ctx, spec)
    assert o.sweep_kernel == _KERNELS[kernel]
    assert np.isnan(o.pit[0, 2]) and np.isnan(o.log_score[0, 2]) and np.all(np.isfinite(o.pit[1:]))
    _check_against_reference(o, spec, lambda w: y)
    _check_mean_against_summary(o, spec)


@pytest.mark.gpu
def test_device_matches_reference_signals_tier(H, ctx):
    y = _series()
    mask = np.zeros(len(y), dtype=np.uint8)
    mask[80:86] = 1
    ys = np.stack([y, y + 0.01 * np.arange(len(y))])
    spec = H.ProblemSpec(ys, [1, 1], [86, 84], K=3, n_chains=4, burnin=30, nrun=1501, seed=5, horizons=(1, 4), precision=32,
                         win_series=[0, 1], win_init_series=[0, 0], is_signal=mask, kappa=0.5, pred_grid=np.linspace(-2, 12, 50),
                         flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY | H.FLAG_PREDICTIVE)
    o = H.estimate(ctx, spec)
    _check_against_reference(o, spec, lambda w: ys[w])
    _check_mean_against_summary(o, spec)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,extra", [("thread", "smoothed"), ("seg", "diagnostics"), ("lane", "diagnostics")])
def test_flag_changes_nothing_else(H, ctx, monkeypatch, kernel, extra):
    """Draws, summaries, diagnostics, pib_mean and status are bit-identical with and without HMCGPU_FLAG_PREDICTIVE."""
    _force(monkeypatch, kernel)
    base = H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY | H.FLAG_LOGLIK \
        | (H.FLAG_SMOOTHED_MEAN if extra == "smoothed" else H.FLAG_DIAGNOSTICS)
    outs = []
    for flag, grid in ((0, None), (H.FLAG_PREDICTIVE, np.linspace(0, 10, 20))):
        spec = H.ProblemSpec(_series(), [1, 9], [80, 61], K=5 if kernel == "lane" else 3, n_chains=5, burnin=20, nrun=300, seed=3,
                             horizons=(2,), precision=32, flags=base | flag, pred_grid=grid)
        outs.append(H.estimate(ctx, spec))
    a, b = outs
    assert b.sweep_kernel == _KERNELS[kernel] and b.n_launches > a.n_launches
    for name in ("mu", "sigma2", "A", "pi_end", "forecasts", "loglik", "summary_mean", "summary_var", "status", "rhat", "ess", "ess_lag"):
        if getattr(a, name) is not None:
            np.testing.assert_array_equal(getattr(a, name), getattr(b, name), err_msg=name)
    if extra == "smoothed":
        for pa, pb in zip(a.pib_mean, b.pib_mean):
            np.testing.assert_array_equal(pa, pb)
    assert not hasattr(a, "pred_cdf") and np.all(np.isfinite(b.pred_cdf))


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
    """A window's predictive outputs are bit-identical alone, in a ragged batch, across two runs of one plan, through
    hmcgpu_estimate_multi_predictive, and inside a batch wide enough for a different chunk size."""
    _force(monkeypatch, "thread")
    y = _series()
    names = ("pred_cdf", "pit", "log_score", "pred_moments")
    kw = dict(K=3, n_chains=4, burnin=20, nrun=2049, seed=9, horizons=(1, 12), precision=32, pred_grid=np.linspace(-2, 12, 24),
              flags=H.FLAG_REF_Q1 | H.FLAG_PREDICTIVE)
    starts, ends = [1, 1, 30, 1, 12], [85, 40, 77, 66, 90]
    batch = H.estimate(ctx, H.ProblemSpec(y, starts, ends, win_id=np.arange(5), **kw))
    for w in (0, 2, 4):
        alone = H.estimate(ctx, H.ProblemSpec(y, [starts[w]], [ends[w]], win_id=[w], **kw))
        for n in names:
            np.testing.assert_array_equal(getattr(alone, n)[0], getattr(batch, n)[w], err_msg=n)
    spec = H.ProblemSpec(y, starts, ends, **kw)
    plan = H.Plan(ctx, spec)
    try:
        plan.run()
        first = plan.fetch()
        plan.run()
        again = plan.fetch()
    finally:
        plan.close()
    multi = H.estimate_multi([0], spec)
    for n in names:
        np.testing.assert_array_equal(getattr(first, n), getattr(again, n), err_msg=n)
        np.testing.assert_array_equal(getattr(first, n), getattr(batch, n), err_msg=n)
        np.testing.assert_array_equal(getattr(multi, n), getattr(batch, n), err_msg=n)
    # wide batch: 3000 short windows x 4 chains -> another chunk size; window 0 is the long one of the batch above
    nw = 3000
    assert _chunk(nw + 1, 4, 3, 2, 2049) != _chunk(5, 4, 3, 2, 2049) == 1024
    wide_s = np.concatenate([[starts[0]], 60 + np.arange(nw) % 10])
    wide_e = np.concatenate([[ends[0]], 80 + np.arange(nw) % 10])
    wide = H.estimate(ctx, H.ProblemSpec(y, wide_s, wide_e, win_id=np.arange(nw + 1) + 100000 * (np.arange(nw + 1) > 0), **kw))
    assert wide.sweep_kernel == 0
    for n in names:
        np.testing.assert_array_equal(getattr(wide, n)[0], getattr(batch, n)[0], err_msg=n)


@pytest.mark.gpu
def test_refusals(H, ctx):
    import ctypes as C
    from hmc_jl_b200 import binding as B
    y = _series()
    kw = dict(K=3, n_chains=2, burnin=5, nrun=10, horizons=(1,), flags=H.FLAG_REF_Q1 | H.FLAG_PREDICTIVE)

    def code(spec, **override):
        prob = spec.struct()
        for k, v in override.items():
            setattr(prob, k, v)
        o, res = spec.alloc_result()
        pr = spec.alloc_predictive(o)
        return ctx.L.hmcgpu_estimate_predictive(ctx.h, C.byref(prob), C.byref(res), C.byref(pr))

    ok = H.ProblemSpec(y, [1], [60], pred_grid=[0.0, 1.0], **kw)
    assert code(ok) >= 0
    assert code(ok, n_grid=0) == B.ERR_ARG
    assert code(H.ProblemSpec(y, [1], [60], pred_grid=np.arange(513.0), **kw)) == B.ERR_ARG
    assert code(H.ProblemSpec(y, [1], [60], pred_grid=[0.0, np.inf], **kw)) == B.ERR_ARG
    assert code(H.ProblemSpec(y, [1], [60], pred_grid=[0.0, 1.0, 1.0], **kw)) == B.ERR_ARG
    assert code(H.ProblemSpec(y, [1], [60], pred_grid=[1.0, 0.0], **kw)) == B.ERR_ARG
    assert code(H.ProblemSpec(y, [1], [60], pred_grid=[0.0, np.nan], **kw)) == B.ERR_ARG
    assert code(H.ProblemSpec(y, [1], [60], pred_grid=[0.0, 1.0], **{**kw, "horizons": ()})) == B.ERR_ARG
    assert code(H.ProblemSpec(y, [1], [60], pred_grid=[0.0, 1.0], pi_row_back=2, **kw)) == B.ERR_UNSUPPORTED
    # the flag through the entry points without predictive outputs
    prob, (o, res) = ok.struct(), ok.alloc_result()
    assert ctx.L.hmcgpu_estimate(ctx.h, C.byref(prob), C.byref(res)) == B.ERR_ARG
    assert "hmcgpu_predictive" in ctx.L.hmcgpu_last_error(ctx.h).decode()
    dev = (C.c_int * 1)(0)
    assert ctx.L.hmcgpu_estimate_multi(dev, 1, C.byref(prob), C.byref(res)) == B.ERR_ARG
    # fetch on a plan without the flag, and before a run
    plain = H.ProblemSpec(y, [1], [60], **{**kw, "flags": H.FLAG_REF_Q1})
    plan = H.Plan(ctx, plain)
    pr = B.Predictive()
    try:
        plan.run()
        assert ctx.L.hmcgpu_plan_fetch_predictive(plan.h, C.byref(pr)) == B.ERR_ARG
    finally:
        plan.close()
    plan = H.Plan(ctx, ok)
    try:
        assert ctx.L.hmcgpu_plan_fetch_predictive(plan.h, C.byref(pr)) == B.ERR_ARG
    finally:
        plan.close()
