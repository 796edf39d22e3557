"""Exact quantiles, rank-normalised split-R̂ and bulk / tail ESS per (window, field) (HMCGPU_FLAG_RANKED).

`ranked_reference` is the definition the device matches (include/hmcgpu.h, hmcgpu_ranked); the CPU tests pin it on cases with
known answers.  The GPU tests compare the device's tables with `ranked_reference` applied to the draws the same call returns."""
import ctypes
import os
import re
import time

import numpy as np
import pytest
from scipy.stats import norm, rankdata

from conftest import ROOT, K3_TRUTH, synth_hmm
from test_diagnostics import split_rhat_ess


def _type7(s, p):
    """Type-7 quantile of sorted draws s: h = (R-1) p, q = s[floor h] + (h - floor h) (s[floor h + 1] - s[floor h])."""
    h = (len(s) - 1) * p
    i = int(np.floor(h))
    return s[i] if i + 1 >= len(s) else s[i] + (h - i) * (s[i + 1] - s[i])


def normal_scores(x):
    """z = Phi^-1((r - 3/8) / (R + 1/4)) of the 1-based average ranks r over all draws of x (-0.0 and +0.0 tie)."""
    x = np.asarray(x, dtype=np.float64)
    r = rankdata(x.ravel() + 0.0, method="average").reshape(x.shape)
    return norm.ppf((r - 0.375) / (x.size + 0.25))


def ranked_reference(x, probs):
    """Ranked outputs of one field of one window: x [n_chains, nrun] (draw d = chain*nrun + i), as doubles.
    Quantiles: type 7 (numpy method="linear").  Bulk: split_rhat_ess (the library's split-R̂ / ESS: same split, Geyer's initial
    monotone sequence, lags capped at 63) of the normal scores z.  Folded: the same of the normal scores of |x - q(0.5)|
    (fp64).  rhat_rank = max(bulk, folded); ess_tail = min(ESS of 1[x <= q(0.05)], ESS of 1[x <= q(0.95)]).  A non-finite
    draw gives NaN everywhere; rhat_rank / ess_tail are NaN when either part is.  Also returns the parts, and the
    Geyer stopping pair of each ESS (`stops`, for the comparison with the device)."""
    x = np.asarray(x, dtype=np.float64)
    nan = np.nan
    if not np.all(np.isfinite(x)):
        return dict(quantiles=np.full(len(probs), nan), rhat_rank=nan, ess_bulk=nan, ess_tail=nan, rhat_bulk=nan, rhat_fold=nan,
                    z=None, stops=())
    s = np.sort(x.ravel())
    q = lambda p: _type7(s, p)
    z = normal_scores(x)
    rb, eb, _, sb = split_rhat_ess(z, full=True)
    rf, _, _, _ = split_rhat_ess(normal_scores(np.abs(x - q(0.5))), full=True)
    _, e05, _, s05 = split_rhat_ess((x <= q(0.05)).astype(np.float64), full=True)
    _, e95, _, s95 = split_rhat_ess((x <= q(0.95)).astype(np.float64), full=True)
    return dict(quantiles=np.array([q(p) for p in probs]),
                rhat_rank=nan if np.isnan(rb) or np.isnan(rf) else max(rb, rf), ess_bulk=eb,
                ess_tail=nan if np.isnan(e05) or np.isnan(e95) else min(e05, e95),
                rhat_bulk=rb, rhat_fold=rf, z=z, stops=(sb, s05, s95))


def _ar1(rng, chains, nrun, phi=0.5):
    x = np.zeros((chains, nrun))
    e = rng.standard_normal((chains, nrun))
    x[:, 0] = e[:, 0]
    for t in range(1, nrun):
        x[:, t] = phi * x[:, t - 1] + np.sqrt(1 - phi * phi) * e[:, t]
    return x


def test_monotone_transform_leaves_ranks_unchanged():
    x = _ar1(np.random.default_rng(1), 6, 501)
    a, b = ranked_reference(x, [0.5]), ranked_reference(np.exp(x), [0.5])
    np.testing.assert_array_equal(a["z"], b["z"])
    for k in ("rhat_bulk", "ess_bulk", "ess_tail"):
        np.testing.assert_allclose(a[k], b[k], rtol=1e-12, err_msg=k)


def test_heavy_tails_mix():
    ref = ranked_reference(np.random.default_rng(2).standard_cauchy((8, 1000)), [0.05, 0.95])
    assert np.isfinite(ref["rhat_rank"]) and abs(ref["rhat_rank"] - 1.0) < 0.01
    assert ref["ess_bulk"] > 4000 and ref["ess_tail"] > 2000


def test_scale_difference_is_seen_by_the_folded_rhat():
    x = np.random.default_rng(1).normal(size=(8, 1000))
    x[4:] *= 3.0
    assert abs(split_rhat_ess(x)[0] - 1.0) < 0.01            # classic split-R̂: equal locations look mixed
    ref = ranked_reference(x, [])
    assert abs(ref["rhat_bulk"] - 1.0) < 0.01 and ref["rhat_fold"] > 1.05 and ref["rhat_rank"] == ref["rhat_fold"]


def test_ties_get_average_ranks():
    x = np.random.default_rng(3).integers(0, 4, size=(4, 50)).astype(np.float64)
    x[0, :3] = [-0.0, 0.0, -0.0]
    z = normal_scores(x)
    flat, R = x.ravel(), x.size
    for v in np.unique(flat):
        below, tied = np.sum(flat < v), np.sum(flat == v)
        r = below + (tied + 1) / 2.0                          # the mean of ranks below+1 .. below+tied
        np.testing.assert_allclose(z.ravel()[flat == v], norm.ppf((r - 0.375) / (R + 0.25)), rtol=1e-15)


@pytest.mark.parametrize("R_shape", [(3, 7), (4, 250), (5, 401)])
def test_quantiles_are_numpy_linear(R_shape):
    x = np.random.default_rng(4).normal(2.0, 5.0, size=R_shape)
    probs = np.array([0.0, 0.01, 0.05, 0.25, 0.5, 1 / 3, 0.95, 0.999, 1.0])
    got = ranked_reference(x, probs)["quantiles"]
    np.testing.assert_allclose(got, np.quantile(x.ravel(), probs, method="linear"), rtol=0, atol=1e-12 * np.abs(x).max())
    assert got[0] == x.min() and got[-1] == x.max()


def test_degenerate_fields():
    rng = np.random.default_rng(5)
    x = rng.normal(size=(4, 100))
    x[x > np.quantile(x, 0.9)] = 10.0                        # q(0.95) = the maximum: 1[x <= q(0.95)] is constant
    ref = ranked_reference(x, [0.5])
    assert np.isnan(ref["ess_tail"]) and np.isfinite(ref["ess_bulk"]) and np.isfinite(ref["rhat_rank"])
    x[1, 7] = np.inf
    ref = ranked_reference(x, [0.1, 0.5])
    assert all(np.all(np.isnan(ref[k])) for k in ("quantiles", "rhat_rank", "ess_bulk", "ess_tail"))
    ref = ranked_reference(np.full((3, 20), 2.5), [0.0, 0.3, 1.0])
    np.testing.assert_array_equal(ref["quantiles"], 2.5)
    assert np.isnan(ref["rhat_rank"]) and np.isnan(ref["ess_bulk"]) and np.isnan(ref["ess_tail"])


def test_flag_constant_matches_header_and_bindings(H):
    from hmc_jl_b200 import binding as B
    header = open(os.path.join(ROOT, "include", "hmcgpu.h")).read()
    jl = open(os.path.join(ROOT, "hmc.jl_b200", "julia", "HmcGPU.jl")).read()
    assert int(re.search(r"#define HMCGPU_FLAG_RANKED\s+(\d+)u", header).group(1)) == B.FLAG_RANKED == H.FLAG_RANKED == 512
    assert re.search(r"const FLAG_RANKED = UInt32\(512\)", jl)
    single = dict(re.findall(r"#define HMCGPU_((?:FLAG|ERR)_\w+) \(?(-?\d+)u?\)?", header))
    assert "FLAG_RANKED" not in single and len(single) == 11
    for sym in ("hmcgpu_estimate_ranked", "hmcgpu_estimate_multi_ranked", "hmcgpu_plan_fetch_ranked"):
        assert sym in B.SYMBOLS and re.search(r"\b%s\(" % sym, header)
        assert re.search(r":%s\b" % sym, jl), sym


def test_ranked_struct_matches_header(H, tmp_path):
    from hmc_jl_b200 import binding as B
    from test_host import _C2CTYPES, _C2JULIA, _c_offsets, _header_struct_fields
    fields = _header_struct_fields("hmcgpu_ranked")
    off = _c_offsets(tmp_path, "hmcgpu_ranked", fields)
    assert [f for f, _ in B.Ranked._fields_] == [f for _, f in fields] == \
        ["probs", "n_probs", "quantiles", "rhat_rank", "ess_bulk", "ess_tail"]
    assert ctypes.sizeof(B.Ranked) == off["sizeof"]
    for (ctype, f), (_, pytype) in zip(fields, B.Ranked._fields_):
        assert getattr(B.Ranked, f).offset == off[f], f
        assert pytype.__name__ == _C2CTYPES[ctype], f
    jl = open(os.path.join(ROOT, "hmc.jl_b200", "julia", "HmcGPU.jl")).read()
    body = re.search(r"struct Ranked\n(.*?)\nend", jl, re.S).group(1)
    jfields = [tuple(x.strip().split("::")) for ln in body.splitlines() for x in ln.split(";") if x.strip()]
    assert jfields == [(f, _C2JULIA[ctype]) for ctype, f in fields]


def test_binding_refuses_probs_without_flag_and_allocates(H):
    y = np.random.default_rng(0).normal(size=60)
    with pytest.raises(ValueError, match="without FLAG_RANKED"):
        H.ProblemSpec(y, [1], [50], K=3, nrun=8, flags=H.FLAG_SUMMARY, quantile_probs=[0.5])
    spec = H.ProblemSpec(y, [1], [50], K=3, nrun=8, flags=H.FLAG_SUMMARY)
    o, _ = spec.alloc_result()
    assert spec.alloc_ranked(o) is None
    spec = H.ProblemSpec(y, [1, 2], [50, 55], K=2, nrun=8, horizons=(1, 12), flags=H.FLAG_RANKED, quantile_probs=[0.05, 0.5, 0.95])
    o, _ = spec.alloc_result()
    rk = spec.alloc_ranked(o)
    F = 3 * 2 + 4 + 4 + 1
    assert o.quantiles.shape == (2, F, 3) and o.rhat_rank.shape == o.ess_bulk.shape == o.ess_tail.shape == (2, F)
    assert rk.n_probs == 3 and rk.probs[1] == 0.5 and rk.quantiles and rk.ess_tail
    rk = spec.alloc_ranked(o, probs=[0.25])
    assert rk.n_probs == 1 and o.quantiles.shape == (2, F, 1)
    rk = H.ProblemSpec(y, [1], [50], K=2, nrun=8, horizons=(1, 12), flags=H.FLAG_RANKED).alloc_ranked(o)
    assert rk.n_probs == 0 and o.quantiles.shape == (1, F, 0)


def test_estimate_windows_and_write_ranked(H, tmp_path, monkeypatch):
    from hmc_jl_b200 import api, binding as B
    seen = {}

    class FakeCtx:
        def close(self):
            pass

    def fake_estimate(ctx, spec):
        seen["spec"] = spec
        o, _ = spec.alloc_result()
        if spec.alloc_ranked(o) is not None:
            for a in (o.quantiles, o.rhat_rank, o.ess_bulk, o.ess_tail):
                a[:] = np.arange(a.size).reshape(a.shape) + 0.25
        return o

    monkeypatch.setattr(B, "estimate", fake_estimate)
    hz, K = (1, 12), 2
    y = np.random.default_rng(0).normal(size=40)
    out = api.estimate_windows(y, [1, 1], [30, 35], K=K, n_chains=2, nrun=10, horizons=hz, quantiles=(0.05, 0.5, 0.95), ctx=FakeCtx())
    assert seen["spec"].flags & B.FLAG_RANKED and list(seen["spec"].quantile_probs) == [0.05, 0.5, 0.95]
    api.estimate_windows(y, [1], [30], K=K, nrun=10, horizons=hz, rank_diagnostics=True, ctx=FakeCtx())
    assert seen["spec"].flags & B.FLAG_RANKED and seen["spec"].quantile_probs is None
    api.estimate_windows(y, [1], [30], K=K, nrun=10, horizons=hz, ctx=FakeCtx())
    assert not seen["spec"].flags & B.FLAG_RANKED

    dates = ["2001-01", "2001-06"]
    paths = H.write_ranked(out, K, hz, dates, str(tmp_path))
    kinds = ("q5", "q50", "q95", "rhat_rank", "ess_bulk", "ess_tail")
    names = ("filtered_means", "filtered_variances", "filtered_trans_probs", "filtered_state_probs", "forecasts")
    assert sorted(paths) == sorted(f"{n}_{k}" for n in names for k in kinds)
    assert os.path.basename(paths["filtered_means_q95"]) == "filtered_means_q95.csv"
    lines = open(paths["forecasts_q50"]).read().splitlines()
    assert lines[0] == "date,forecast_1_q50,forecast_error_1_q50,forecast_12_q50,forecast_error_12_q50"
    assert [ln.split(",")[0] for ln in lines[1:]] == dates
    f0 = 3 * K + K * K
    np.testing.assert_array_equal(np.loadtxt(paths["forecasts_q50"], delimiter=",", skiprows=1, usecols=range(1, 5)),
                                  out.quantiles[:, f0:f0 + 4, 1])
    np.testing.assert_array_equal(np.loadtxt(paths["filtered_variances_ess_tail"], delimiter=",", skiprows=1, usecols=(1, 2)),
                                  out.ess_tail[:, K:2 * K])
    assert open(paths["filtered_means_rhat_rank"]).readline().strip() == "date,state_1_rhat_rank,state_2_rhat_rank"


# ---------------------------------------------------------------------------------------------------------------------------- GPU

PROBS = np.array([0.0, 0.05, 0.25, 0.5, 0.95, 1.0, 1 / 3])


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


def _fields(o, w, K, nh, n_chains, nrun):
    """Draws of window w as [F, n_chains, nrun] in the summary field order (the loglik field: its draws, or zeros)."""
    ll = o.loglik[w][None] if o.loglik is not None else np.zeros((1, n_chains * nrun))
    parts = [o.mu[w], o.sigma2[w], o.A[w].reshape(K * K, -1), o.pi_end[w]] + ([o.forecasts[w]] if nh else []) + [ll]
    return np.concatenate(parts).reshape(-1, n_chains, nrun)


def _check_against_reference(o, spec, probs):
    """Quantiles to 1e-12 of the field's largest |draw| (exactly where (R-1)p is an integer), R̂ / ESS to 1e-9 relative.  An
    ESS may differ where the reference's Geyer sum stopped on a pair that is ~0 (the order of summation decides its sign)."""
    K, nh, nc, nrun = spec.K, spec.n_h, spec.n_chains, spec.nrun
    has_ll = bool(spec.flags & 16)
    R = nc * nrun
    exact = np.array([float((R - 1) * p).is_integer() for p in probs])
    n_stop = 0
    for w in range(spec.n_windows):
        x = _fields(o, w, K, nh, nc, nrun)
        for f in range(x.shape[0]):
            ref = ranked_reference(x[f], probs)
            if f == x.shape[0] - 1 and not has_ll:
                ref = ranked_reference(np.full_like(x[f], np.nan), probs)
            q = o.quantiles[w, f]
            if np.isnan(ref["rhat_rank"]) and np.all(np.isnan(ref["quantiles"])):
                assert np.all(np.isnan(q)) and np.isnan(o.rhat_rank[w, f]) and np.isnan(o.ess_bulk[w, f]) and np.isnan(o.ess_tail[w, f]), (w, f)
                continue
            np.testing.assert_array_equal(q[exact], ref["quantiles"][exact], err_msg=f"quantiles window {w} field {f}")
            np.testing.assert_allclose(q, ref["quantiles"], rtol=0, atol=1e-12 * np.abs(x[f]).max(), err_msg=f"quantiles {w} {f}")
            for k in ("rhat_rank", "ess_bulk", "ess_tail"):
                got, want = o.__dict__[k][w, f], ref[k]
                if np.isnan(want):
                    assert np.isnan(got), (k, w, f)
                    continue
                if k != "rhat_rank" and not np.isclose(got, want, rtol=1e-9, atol=0):
                    assert any(s is not None and abs(s) < 1e-9 for s in ref["stops"]), (k, w, f, got, want)
                    n_stop += 1
                    continue
                np.testing.assert_allclose(got, want, rtol=1e-9, err_msg=f"{k} window {w} field {f}")
    assert n_stop <= 1


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,precision,nrun", [("thread", 32, 1501), ("thread", 64, 1000), ("scan", 32, 1000), ("scan", 64, 1501),
                                                    ("seg", 32, 1000), ("seg", 64, 1501), ("lane", 32, 1501), ("lane", 64, 1000)])
def test_device_matches_reference(H, ctx, monkeypatch, kernel, precision, nrun):
    """Every ranked output of every (window, field) against ranked_reference of the returned draws.  nrun = 1501: odd (the
    middle draw is dropped) and two chunks; 1000: even.  The window ending at 88 has no y[88 + 12]: its h = 12 forecast error is
    NaN, so that field is NaN in every output.  Without HMCGPU_FLAG_LOGLIK the loglik field is NaN too (the lane run sets it)."""
    _force(monkeypatch, kernel)
    K = 5 if kernel == "lane" else 3
    loglik = 0 if kernel == "lane" else H.FLAG_LOGLIK
    spec = H.ProblemSpec(_series(), [1, 5, 20], [88, 70, 60], K=K, n_chains=3, burnin=30, nrun=nrun, seed=11, horizons=(1, 12),
                         precision=precision, quantile_probs=PROBS, flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | loglik | H.FLAG_RANKED)
    o = H.estimate(ctx, spec)
    assert o.sweep_kernel == _KERNELS[kernel]
    fe = 3 * K + K * K + 3
    assert np.all(np.isnan(o.quantiles[0, fe])) and np.isfinite(o.rhat_rank[1, fe]) and np.all(np.isfinite(o.quantiles[:, :3 * K]))
    assert np.all(np.isnan(o.rhat_rank[:, -1])) == (loglik == 0)
    _check_against_reference(o, spec, PROBS)


@pytest.mark.gpu
def test_device_matches_reference_signals_tier(H, ctx):
    y = _series()
    mask = np.zeros(len(y), dtype=np.uint8)
    mask[80:86] = 1
    ys = np.stack([y, y + 0.01 * np.arange(len(y))])
    spec = H.ProblemSpec(ys, [1, 1], [86, 84], K=3, n_chains=4, burnin=30, nrun=1001, seed=5, horizons=(1, 4), precision=32,
                         win_series=[0, 1], win_init_series=[0, 0], is_signal=mask, kappa=0.5, pi_row_back=2, quantile_probs=PROBS,
                         flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK | H.FLAG_RANKED)
    o = H.estimate(ctx, spec)
    _check_against_reference(o, spec, PROBS)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel", ["thread", "seg", "scan", "lane"])
def test_flag_changes_nothing_else(H, ctx, monkeypatch, kernel):
    """Draws, summaries, diagnostics, predictive outputs, pib_mean, status and the return value are bit-identical with and
    without HMCGPU_FLAG_RANKED; the flag adds one retention launch per draw chunk and nothing else."""
    _force(monkeypatch, kernel)
    base = H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY | H.FLAG_LOGLIK | H.FLAG_DIAGNOSTICS | H.FLAG_PREDICTIVE \
        | (H.FLAG_SMOOTHED_MEAN if kernel == "thread" else 0)
    outs = []
    for flag in (0, H.FLAG_RANKED):
        spec = H.ProblemSpec(_series(), [1, 9], [80, 61], K=5 if kernel == "lane" else 3, n_chains=5, burnin=20, nrun=1300, seed=3,
                             horizons=(2,), precision=32, flags=base | flag, pred_grid=np.linspace(0, 10, 20),
                             quantile_probs=[0.5] if flag else None)
        outs.append(H.estimate(ctx, spec))
    a, b = outs
    assert b.sweep_kernel == a.sweep_kernel == _KERNELS[kernel]
    assert b.n_launches == a.n_launches + 2 and b.events == a.events          # 1300 draws: two chunks
    for name in ("mu", "sigma2", "A", "pi_end", "forecasts", "loglik", "summary_mean", "summary_var", "status", "rhat", "ess", "ess_lag",
                 "pred_cdf", "pit", "log_score", "pred_moments"):
        np.testing.assert_array_equal(getattr(a, name), getattr(b, name), err_msg=name)
    if kernel == "thread":
        for pa, pb in zip(a.pib_mean, b.pib_mean):
            np.testing.assert_array_equal(pa, pb)
    assert not hasattr(a, "rhat_rank") and np.all(np.isfinite(b.rhat_rank[:, :-1]))


_NAMES = ("quantiles", "rhat_rank", "ess_bulk", "ess_tail")


@pytest.mark.gpu
def test_batching_chunking_runs_and_multi_invariance(H, ctx, monkeypatch):
    """A window's ranked outputs are bit-identical alone, in a ragged batch, across two runs of one plan, through
    hmcgpu_estimate_multi_ranked over two contexts on device 0, and in a batch wide enough for another chunk size.  nrun = 2049:
    the chunks of 1024 draws split the second half-chain ([1025, 2049))."""
    _force(monkeypatch, "thread")
    y = _series()
    kw = dict(K=3, n_chains=4, burnin=20, nrun=2049, seed=9, horizons=(1, 12), precision=32, quantile_probs=PROBS,
              flags=H.FLAG_REF_Q1 | H.FLAG_RANKED)
    starts, ends = [1, 1, 30, 1, 12], [85, 40, 77, 66, 90]
    batch = H.estimate(ctx, H.ProblemSpec(y, starts, ends, win_id=np.arange(5), **kw))
    for w in (0, 2, 4):
        alone = H.estimate(ctx, H.ProblemSpec(y, [starts[w]], [ends[w]], win_id=[w], **kw))
        for n in _NAMES:
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
    multi = H.estimate_multi([0, 0], spec)
    for n in _NAMES:
        np.testing.assert_array_equal(getattr(first, n), getattr(again, n), err_msg=n)
        np.testing.assert_array_equal(getattr(first, n), getattr(batch, n), err_msg=n)
        np.testing.assert_array_equal(getattr(multi, n), getattr(batch, n), err_msg=n)
    # wide batch: 3000 short windows x 4 chains -> chunks of fewer than 1024 draws; window 0 is the long one of the batch above
    nw = 3000
    wide_s = np.concatenate([[starts[0]], 60 + np.arange(nw) % 10])
    wide_e = np.concatenate([[ends[0]], 80 + np.arange(nw) % 10])
    wide = H.estimate(ctx, H.ProblemSpec(y, wide_s, wide_e, win_id=np.arange(nw + 1) + 100000 * (np.arange(nw + 1) > 0), **kw))
    assert wide.sweep_kernel == 0
    for n in _NAMES:
        np.testing.assert_array_equal(getattr(wide, n)[0], getattr(batch, n)[0], err_msg=n)


@pytest.mark.gpu
def test_repeated_fetch_with_other_probs(H, ctx):
    spec = H.ProblemSpec(_series(), [1, 20], [88, 70], K=3, n_chains=3, burnin=20, nrun=600, seed=4, horizons=(1,), precision=64,
                         quantile_probs=[0.1, 0.9], flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK | H.FLAG_RANKED)
    plan = H.Plan(ctx, spec)
    try:
        plan.run()
        o = plan.fetch()
        other = plan.fetch_ranked(probs=PROBS)
    finally:
        plan.close()
    _check_against_reference(o, spec, [0.1, 0.9])
    for n in ("rhat_rank", "ess_bulk", "ess_tail"):
        np.testing.assert_array_equal(getattr(other, n), getattr(o, n), err_msg=n)
    o.quantiles = other.quantiles
    _check_against_reference(o, spec, PROBS)


@pytest.mark.gpu
def test_refusals(H, ctx):
    import ctypes as C
    from hmc_jl_b200 import binding as B
    y = _series()
    kw = dict(K=3, n_chains=2, burnin=5, nrun=10, horizons=(1,), flags=H.FLAG_REF_Q1 | H.FLAG_RANKED)

    def code(spec, probs=(0.5,), **override):
        prob = spec.struct()
        for k, v in override.items():
            setattr(prob, k, v)
        o, res = spec.alloc_result()
        rk = spec.alloc_ranked(o, probs=probs)
        return ctx.L.hmcgpu_estimate_ranked(ctx.h, C.byref(prob), C.byref(res), None, C.byref(rk))

    def message():
        return ctx.L.hmcgpu_last_error(ctx.h).decode()

    ok = H.ProblemSpec(y, [1], [60], **kw)
    assert code(ok) >= 0 and code(ok, probs=np.linspace(0, 1, 64)) >= 0 and code(ok, probs=[]) >= 0
    assert code(ok, probs=np.linspace(0, 1, 65)) == B.ERR_ARG and "n_probs" in message()
    for bad in (-0.1, 1.5, np.nan, np.inf):
        assert code(ok, probs=[0.5, bad]) == B.ERR_ARG and "probs[1]" in message()
    assert code(ok, nrun=3) == B.ERR_ARG and "HMCGPU_FLAG_RANKED needs nrun >= 4" in message()
    assert code(ok, n_chains=2, nrun=1 << 30) == B.ERR_ARG and "n_chains * nrun" in message()
    # the flag without ranked outputs, one-shot and multi-device
    prob, (o, res) = ok.struct(), ok.alloc_result()
    assert ctx.L.hmcgpu_estimate(ctx.h, C.byref(prob), C.byref(res)) == B.ERR_ARG and "hmcgpu_ranked" in message()
    dev = (C.c_int * 1)(0)
    assert ctx.L.hmcgpu_estimate_multi_ranked(dev, 1, C.byref(prob), C.byref(res), None, None) == B.ERR_ARG
    assert "hmcgpu_ranked" in ctx.L.hmcgpu_last_error(None).decode()
    # fetch on a plan without the flag, and before a run
    rk = B.Ranked()
    plan = H.Plan(ctx, H.ProblemSpec(y, [1], [60], **{**kw, "flags": H.FLAG_REF_Q1}))
    try:
        plan.run()
        assert ctx.L.hmcgpu_plan_fetch_ranked(plan.h, C.byref(rk)) == B.ERR_ARG and "without HMCGPU_FLAG_RANKED" in message()
    finally:
        plan.close()
    plan = H.Plan(ctx, ok)
    try:
        assert ctx.L.hmcgpu_plan_fetch_ranked(plan.h, C.byref(rk)) == B.ERR_ARG and "before plan_run" in message()
    finally:
        plan.close()
    # retained draws larger than the device: refused before anything is allocated (2 windows x 13 fields x 256 chains x 8e6
    # draws x 4 bytes = 213 GB against 180 GB)
    import torch
    free0 = torch.cuda.mem_get_info(0)[0]
    big = H.ProblemSpec(y, [1, 2], [60, 61], K=2, n_chains=256, burnin=0, nrun=8_000_000, horizons=(1,), precision=32,
                        flags=H.FLAG_REF_Q1 | H.FLAG_RANKED)
    keep = 2 * (3 * 2 + 4 + 2 + 1) * 256 * 8_000_000 * 4
    assert keep > torch.cuda.get_device_properties(0).total_memory
    h = C.c_void_p()
    t0 = time.perf_counter()
    assert ctx.L.hmcgpu_plan_create(ctx.h, C.byref(big.struct()), C.byref(h)) == B.ERR_ALLOC
    assert time.perf_counter() - t0 < 5.0 and not h.value
    assert "HMCGPU_FLAG_RANKED" in message() and str(keep) in message()
    assert abs(torch.cuda.mem_get_info(0)[0] - free0) < (4 << 30)     # (other work may share the device)
