"""Split-R̂ and effective sample size per (window, field) (HMCGPU_FLAG_DIAGNOSTICS).

`split_rhat_ess` is the definition the device matches; the CPU tests pin it on cases with known answers, and check a numpy
mirror of the device's streaming algebra (diagnostics.cuh) against it before any GPU runs.  The GPU tests compare the
device's tables with `split_rhat_ess` applied to the draws the same call returns."""
import os
import re

import numpy as np
import pytest

from conftest import ROOT, K3_TRUTH, synth_hmm

LAG_CAP = 63          # autocovariance lags 0..63 (32 Geyer pairs), include/hmcgpu.h


def _split(x):
    """[n_chains, nrun] -> [2 n_chains, n]: first and last n = nrun // 2 draws of every chain (the middle one of an odd nrun
    is dropped)."""
    x = np.asarray(x, dtype=np.float64)
    n = x.shape[1] // 2
    return np.concatenate([x[:, :n], x[:, x.shape[1] - n:]])


def _geyer(rho, M, n):
    """Initial monotone sequence over the pairs P_k = rho_2k + rho_2k+1 (rho[l] for l = 0..L): (ESS, last lag summed,
    value of the pair that stopped the sum or None)."""
    total, prev, last, stop = 0.0, np.inf, -1, None
    for k in range(len(rho) // 2):
        p = rho[2 * k] + rho[2 * k + 1]
        if not p > 0:
            stop = p
            break
        p = min(p, prev)
        prev = p
        total += p
        last = 2 * k + 1
    tau = max(-1.0 + 2.0 * total, 1.0 / np.log10(M * n))
    return M * n / tau, last, stop


def split_rhat_ess(x, full=False):
    """Classic split-R̂ (BDA3, not rank-normalised) and ESS (Geyer's initial monotone sequence, lags <= 63) of one field of
    one window: x [n_chains, nrun].  Returns (rhat, ess, ess_lag); NaN, NaN, -1 when a draw used is non-finite or W = 0.
    full=True appends the value of the pair that stopped the autocorrelation sum (None if the cap did)."""
    s = _split(x)
    M, n = s.shape
    nan = (np.nan, np.nan, -1) + ((None,) if full else ())
    if not np.all(np.isfinite(s)):
        return nan
    d = s - s[:, :1]                                 # (shifted by each sequence's first value: a constant sequence has s2 = 0 exactly)
    d = d - d.mean(axis=1, keepdims=True)
    s2 = (d * d).sum(axis=1) / (n - 1)
    W = s2.mean()
    if not W > 0:
        return nan
    Bn = s.mean(axis=1).var(ddof=1)
    varp = (n - 1) / n * W + Bn
    L = min(LAG_CAP, n - 1)
    gamma = np.array([(d[:, :n - l] * d[:, l:]).sum(axis=1).mean() / n for l in range(L + 1)])
    rho = 1.0 - (W - gamma) / varp
    rho[0] = 1.0
    ess, lag, stop = _geyer(rho, M, n)
    out = (float(np.sqrt(varp / W)), float(ess), lag)
    return out + ((stop,) if full else ())


def streaming_mirror(x, chunk):
    """The device algebra in numpy: draws arrive in chunks of `chunk` (the per-chunk buffer); per chain and sequence the state
    is S1, the lag-product sums P_l of the values shifted by the sequence's first value, its first 64 values and a ring of
    its last 64; a sequence ends with the head / ring corrections that centre P_l, summed over the chains in chain order."""
    x = np.asarray(x, dtype=np.float64)
    C, nrun = x.shape
    n = nrun // 2
    starts = (0, nrun - n)
    means, s2, G = np.zeros((2, C)), np.zeros((2, C)), np.zeros(LAG_CAP + 1)
    for c in range(C):
        st = {}
        for d0 in range(0, nrun, chunk):
            for h, h0 in enumerate(starts):
                lo, hi = max(d0, h0), min(d0 + chunk, h0 + n)
                for d in range(lo, hi):
                    t = d - h0
                    if t == 0:
                        st = dict(c0=x[c, d], S1=0.0, P=np.zeros(LAG_CAP + 1), head=np.zeros(64), ring=np.zeros(64))
                    y = x[c, d] - st["c0"]
                    prev = np.array([st["ring"][(t - l) % 64] - st["c0"] if t - l >= 0 else 0.0 for l in range(1, LAG_CAP + 1)])
                    st["P"] += y * np.concatenate([[y], prev])
                    st["S1"] += y
                    if t < 64:
                        st["head"][t] = x[c, d]
                    st["ring"][t % 64] = x[c, d]
                if hi == h0 + n and lo < hi:          # the sequence ended in this chunk
                    ybar = st["S1"] / n
                    hy = st["head"][:min(64, n)] - st["c0"]
                    ty = np.array([st["ring"][t % 64] - st["c0"] for t in range(max(0, n - 64), n)])
                    means[h, c] = st["c0"] + ybar
                    s2[h, c] = (st["P"][0] - st["S1"] * ybar) / (n - 1)
                    for l in range(min(LAG_CAP, n - 1) + 1):
                        hs, ts = hy[:l].sum(), ty[len(ty) - l:].sum() if l else 0.0
                        G[l] += st["P"][l] - ybar * ((st["S1"] - ts) + (st["S1"] - hs)) + (n - l) * ybar * ybar
    M = 2 * C
    means, s2 = means.ravel(), s2.ravel()
    if not (np.all(np.isfinite(means)) and np.all(np.isfinite(s2))) or not s2.mean() > 0:
        return np.nan, np.nan, -1
    W, Bn = s2.mean(), means.var(ddof=1)
    varp = (n - 1) / n * W + Bn
    L = min(LAG_CAP, n - 1)
    rho = 1.0 - (W - G[:L + 1] / (M * n)) / varp
    rho[0] = 1.0
    ess, lag, _ = _geyer(rho, M, n)
    return float(np.sqrt(varp / W)), float(ess), lag


def _ar1(rng, chains, nrun, phi, offsets=None):
    e = rng.standard_normal((chains, nrun))
    x = np.empty_like(e)
    x[:, 0] = e[:, 0] / np.sqrt(1 - phi * phi)
    for t in range(1, nrun):
        x[:, t] = phi * x[:, t - 1] + e[:, t]
    return x if offsets is None else x + np.asarray(offsets, dtype=np.float64)[:, None]


# ---------------------------------------------------------------------------------------------------------------------------- CPU

def test_iid_chains_mix():
    x = np.random.default_rng(0).standard_normal((8, 4000))
    rhat, ess, lag = split_rhat_ess(x)
    assert rhat < 1.01
    assert 0.9 * x.size < ess < 1.1 * x.size and lag < 10


def test_ar1_ess_matches_theory():
    phi = 0.9
    x = _ar1(np.random.default_rng(1), 16, 20000, phi)
    rhat, ess, lag = split_rhat_ess(x)
    want = x.size * (1 - phi) / (1 + phi)
    assert rhat < 1.01
    assert abs(ess / want - 1) < 0.15, (ess, want)
    assert 1 <= lag <= LAG_CAP               # (rho_63 = 0.9^63 > 0: the sum reaches the cap, with a negligible bias here)


def test_offset_chains_do_not_mix():
    x = np.random.default_rng(2).standard_normal((4, 1000)) + np.array([0.0, 0.0, 3.0, 3.0])[:, None]
    assert split_rhat_ess(x)[0] > 1.5


def test_odd_nrun_drops_the_middle_draw():
    x = np.random.default_rng(3).standard_normal((3, 201))
    y = x.copy()
    y[:, 100] = 1e6                                          # the dropped draw changes nothing ...
    assert split_rhat_ess(x) == split_rhat_ess(y)
    y[:, 100] = np.nan                                       # ... not even when it is NaN
    assert split_rhat_ess(x) == split_rhat_ess(y)
    assert split_rhat_ess(x) == split_rhat_ess(np.delete(x, 100, axis=1))


def test_degenerate_fields_are_nan():
    assert split_rhat_ess(np.full((4, 100), 0.1))[2] == -1
    assert np.isnan(split_rhat_ess(np.full((4, 100), 0.1))[0])
    x = np.random.default_rng(4).standard_normal((4, 100))
    x[2, 7] = np.nan
    assert np.isnan(split_rhat_ess(x)[1])
    x[2, 7] = np.inf
    assert np.isnan(split_rhat_ess(x)[0])
    # constant within every chain, different between chains: W = 0
    assert np.isnan(split_rhat_ess(np.repeat(np.arange(4.0)[:, None], 50, axis=1))[0])


def test_short_sequences_cap_the_lags_at_n_minus_1():
    x = np.random.default_rng(5).standard_normal((2, 4))            # n = 2: one pair (lags 0, 1) at most
    rhat, ess, lag = split_rhat_ess(x)
    assert np.isfinite(rhat) and lag in (-1, 1)


@pytest.mark.parametrize("nrun,chunk", [(300, 1000), (300, 48), (301, 64), (257, 100), (131, 7), (9, 2), (4, 1), (2049, 1024)])
def test_streaming_mirror_equals_definition(nrun, chunk):
    """Chunked input, the shift, the head and ring corrections, the half boundary inside a chunk (nrun / 2 not a multiple of
    the chunk), odd nrun and sequences shorter than the lag cap: the device's algebra gives the definition's numbers."""
    rng = np.random.default_rng(nrun + chunk)
    for x in (_ar1(rng, 3, nrun, 0.95, offsets=[50.0, 50.5, 49.0]), rng.standard_normal((3, nrun)) * 1e-3 + 7.0,
              _ar1(rng, 2, nrun, -0.6)):
        want, got = split_rhat_ess(x), streaming_mirror(x, chunk)
        np.testing.assert_allclose(got[:2], want[:2], rtol=1e-12)
        assert got[2] == want[2]
    x = rng.standard_normal((3, nrun))
    x[1, 0] = np.nan
    assert np.isnan(streaming_mirror(x, chunk)[0]) and np.isnan(split_rhat_ess(x)[0])


def test_flag_constant_and_result_fields_match_header(H):
    from hmc_jl_b200 import binding as B
    header = open(os.path.join(ROOT, "include", "hmcgpu.h")).read()
    jl = open(os.path.join(ROOT, "hmc.jl_b200", "julia", "HmcGPU.jl")).read()
    assert int(re.search(r"#define HMCGPU_FLAG_DIAGNOSTICS\s+(\d+)u", header).group(1)) == B.FLAG_DIAGNOSTICS == H.FLAG_DIAGNOSTICS == 128
    assert re.search(r"const FLAG_DIAGNOSTICS = UInt32\(128\)", jl)
    assert [f for f, _ in B.Result._fields_][-3:] == ["rhat", "ess", "ess_lag"]


def test_binding_refuses_diagnostics_without_the_flag(H):
    y = np.random.default_rng(0).normal(size=60)
    spec = H.ProblemSpec(y, [1], [50], K=3, n_chains=2, nrun=8, flags=H.FLAG_SUMMARY)
    with pytest.raises(ValueError, match="FLAG_DIAGNOSTICS"):
        spec.alloc_result(diagnostics=True)
    o, res = spec.alloc_result()
    assert o.rhat is None and not res.rhat and not res.ess and not res.ess_lag
    spec = H.ProblemSpec(y, [1, 3], [50, 60], K=3, n_chains=2, nrun=8, horizons=(1, 12), flags=H.FLAG_SUMMARY | H.FLAG_DIAGNOSTICS)
    o, res = spec.alloc_result()
    F = 3 * 3 + 9 + 4 + 1
    assert o.rhat.shape == o.ess.shape == o.ess_lag.shape == (2, F) and o.ess_lag.dtype == np.int32 and res.rhat and res.ess_lag


def test_estimate_windows_and_write_diagnostics(H, tmp_path, monkeypatch):
    """Host side: estimate_windows(diagnostics=True) sets the flag and returns the tables; write_diagnostics writes them in the
    column layout of write_summaries (one helper builds both)."""
    from hmc_jl_b200 import api, binding as B
    seen = {}

    class FakeCtx:
        def close(self):
            pass

    def fake_estimate(ctx, spec):
        seen["spec"] = spec
        o, _ = spec.alloc_result()
        for a in (o.summary_mean, o.rhat, o.ess):
            if a is not None:
                a[:] = np.arange(a.size).reshape(a.shape) + 0.5
        return o

    monkeypatch.setattr(B, "estimate", fake_estimate)
    K, hz = 2, (1, 12)
    y = np.random.default_rng(0).normal(size=40)
    out = api.estimate_windows(y, [1, 1], [30, 35], K=K, n_chains=2, nrun=10, horizons=hz, diagnostics=True, ctx=FakeCtx())
    assert seen["spec"].flags & B.FLAG_DIAGNOSTICS and seen["spec"].flags & B.FLAG_SUMMARY
    F = 3 * K + K * K + 2 * len(hz) + 1
    assert out.rhat.shape == (2, F)
    api.estimate_windows(y, [1], [30], K=K, nrun=10, horizons=hz, ctx=FakeCtx())
    assert not seen["spec"].flags & B.FLAG_DIAGNOSTICS and seen["spec"].alloc_result()[0].rhat is None

    dates = ["2001-01", "2001-06"]
    summ = H.write_summaries(out, K, hz, dates, str(tmp_path))
    paths = H.write_diagnostics(out, K, hz, dates, str(tmp_path))
    assert sorted(paths) == sorted(f"{v}_{k}" for v in summ for k in ("rhat", "ess"))
    for var, p in summ.items():
        hdr = open(p).readline().strip().split(",")
        for kind, table in (("rhat", out.rhat), ("ess", out.ess)):
            lines = open(paths[f"{var}_{kind}"]).read().splitlines()
            assert lines[0].split(",") == [h[:-len("_mean")] + "_" + kind if h != "date" else h for h in hdr]
            assert [ln.split(",")[0] for ln in lines[1:]] == dates
    got = np.loadtxt(paths["forecasts_ess"], delimiter=",", skiprows=1, usecols=(1, 2, 3, 4))
    np.testing.assert_array_equal(got, out.ess[:, 3 * K + K * K:3 * K + K * K + 4])
    assert open(paths["filtered_trans_probs_rhat"]).readline().startswith("date,trans_1_1_rhat,trans_2_1_rhat,trans_1_2_rhat")
    # the gather of a diagnostics table across ranks is the summaries' gather
    full = H.gather_window_summaries(out.rhat[::-1], np.array([1, 0]), 2)
    np.testing.assert_array_equal(full, out.rhat)


# ---------------------------------------------------------------------------------------------------------------------------- GPU

def _fields(o, w, K, nh, n_chains, nrun):
    """Draws of window w as [F, n_chains, nrun] in the summary field order."""
    parts = [o.mu[w], o.sigma2[w], o.A[w].reshape(K * K, -1), o.pi_end[w]] + ([o.forecasts[w]] if nh else []) + [o.loglik[w][None]]
    return np.concatenate(parts).reshape(-1, n_chains, nrun)


def _check_against_reference(o, K, nh, n_chains, nrun):
    nw, F = o.rhat.shape
    n_lag_mismatch = 0
    for w in range(nw):
        x = _fields(o, w, K, nh, n_chains, nrun)
        for f in range(F):
            rhat, ess, lag, stop = split_rhat_ess(x[f], full=True)
            if np.isnan(rhat):
                assert np.isnan(o.rhat[w, f]) and np.isnan(o.ess[w, f]) and o.ess_lag[w, f] == -1, (w, f)
                continue
            np.testing.assert_allclose(o.rhat[w, f], rhat, rtol=1e-9, err_msg=f"rhat window {w} field {f}")
            if o.ess_lag[w, f] != lag:                       # only where the reference's stopping pair is ~0
                assert stop is not None and abs(stop) < 1e-9, (w, f, o.ess_lag[w, f], lag, stop)
                n_lag_mismatch += 1
                continue
            np.testing.assert_allclose(o.ess[w, f], ess, rtol=1e-9, err_msg=f"ess window {w} field {f}")
    assert n_lag_mismatch <= 1


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


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,precision,nrun", [("thread", 32, 1501), ("thread", 64, 2049), ("scan", 32, 2049), ("scan", 64, 1501),
                                                    ("seg", 32, 1501), ("seg", 64, 2049), ("lane", 32, 1501)])
def test_device_matches_reference(H, ctx, monkeypatch, kernel, precision, nrun):
    """R̂, ESS and ess_lag of every (window, field) equal split_rhat_ess of the returned draws (the values the device
    accumulated; only the order of summation differs).  nrun = 1501: odd, the half boundary inside the first chunk (chunks hold
    at most 1024 draws); 2049: three chunks, lags across chunk edges.  The window ending at 88 has no y[88 + 12]: its h = 12
    forecast error is NaN."""
    _force(monkeypatch, kernel)
    K = 5 if kernel == "lane" else 3
    nc, hz = 3, (1, 12)
    spec = H.ProblemSpec(_series(), [1, 5, 20], [88, 70, 60], K=K, n_chains=nc, burnin=30, nrun=nrun, seed=11, horizons=hz,
                         precision=precision, flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK | H.FLAG_DIAGNOSTICS)
    o = H.estimate(ctx, spec)
    assert o.sweep_kernel == _KERNELS[kernel]
    F = 3 * K + K * K + 2 * len(hz) + 1
    assert o.rhat.shape == (3, F)
    assert np.isnan(o.rhat[0, 3 * K + K * K + 3]) and np.isfinite(o.rhat[0, 3 * K + K * K + 2])     # forecast error / forecast, h = 12
    assert np.all(np.isfinite(o.rhat[1:, :3 * K]))
    _check_against_reference(o, K, len(hz), nc, nrun)


@pytest.mark.gpu
def test_device_matches_reference_signals_tier(H, ctx):
    y = _series()
    mask = np.zeros(len(y), dtype=np.uint8)
    mask[80:86] = 1
    nc, nrun = 4, 1501
    spec = H.ProblemSpec(np.stack([y, y + 0.01 * np.arange(len(y))]), [1, 1], [86, 86], K=3, n_chains=nc, burnin=30, nrun=nrun,
                         seed=5, horizons=(1,), precision=32, win_series=[0, 1], win_init_series=[0, 0], is_signal=mask, kappa=0.5,
                         pi_row_back=2, flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK | H.FLAG_DIAGNOSTICS)
    o = H.estimate(ctx, spec)
    _check_against_reference(o, 3, 1, nc, nrun)


@pytest.mark.gpu
@pytest.mark.parametrize("kernel,flags", [("thread", "smoothed"), ("seg", "loglik"), ("scan", "loglik")])
def test_flag_changes_nothing_else(H, ctx, monkeypatch, kernel, flags):
    """Draws, summaries, pib_mean and status are bit-identical with and without HMCGPU_FLAG_DIAGNOSTICS; without
    HMCGPU_FLAG_LOGLIK the log-likelihood field's diagnostics are NaN."""
    _force(monkeypatch, kernel)
    base = H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY | (H.FLAG_SMOOTHED_MEAN if flags == "smoothed" else H.FLAG_LOGLIK)
    outs = []
    for extra in (0, H.FLAG_DIAGNOSTICS):
        spec = H.ProblemSpec(_series(), [1, 9], [80, 61], K=3, n_chains=5, burnin=20, nrun=300, seed=3, horizons=(2,),
                             precision=32, flags=base | extra)
        outs.append(H.estimate(ctx, spec))
    a, b = outs
    assert b.sweep_kernel == _KERNELS[kernel]
    for name in ("mu", "sigma2", "A", "pi_end", "forecasts", "loglik", "summary_mean", "summary_var", "status"):
        if getattr(a, name) is not None:
            np.testing.assert_array_equal(getattr(a, name), getattr(b, name), err_msg=name)
    if flags == "smoothed":
        for pa, pb in zip(a.pib_mean, b.pib_mean):
            np.testing.assert_array_equal(pa, pb)
        assert np.all(np.isnan(b.rhat[:, -1])) and np.all(b.ess_lag[:, -1] == -1)
    assert a.rhat is None and np.all(np.isfinite(b.rhat[:, :9]))


@pytest.mark.gpu
def test_batching_invariance_and_multi(H, ctx, monkeypatch):
    """A window's diagnostics are bit-identical alone and inside a ragged batch (thread-per-chain kernel; same win_id, so the
    same chains), repeated plan runs give the same tables, and estimate_multi scatters the same tables as estimate."""
    _force(monkeypatch, "thread")
    y = _series()
    flags = H.FLAG_REF_Q1 | H.FLAG_SUMMARY | H.FLAG_LOGLIK | H.FLAG_DIAGNOSTICS
    kw = dict(K=3, n_chains=6, burnin=20, nrun=777, seed=9, horizons=(1, 3), precision=32, flags=flags)
    starts, ends = [1, 1, 30, 1, 12], [85, 40, 77, 66, 90]
    batch = H.estimate(ctx, H.ProblemSpec(y, starts, ends, win_id=np.arange(5), **kw))
    assert batch.sweep_kernel == 0
    for w in (0, 2, 4):
        alone = H.estimate(ctx, H.ProblemSpec(y, [starts[w]], [ends[w]], win_id=[w], **kw))
        for name in ("rhat", "ess", "ess_lag"):
            np.testing.assert_array_equal(getattr(alone, name)[0], getattr(batch, name)[w], err_msg=name)
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
    for name in ("rhat", "ess", "ess_lag"):
        np.testing.assert_array_equal(getattr(first, name), getattr(again, name), err_msg=name)
        np.testing.assert_array_equal(getattr(multi, name), getattr(batch, name), err_msg=name)


@pytest.mark.gpu
def test_diagnostics_need_four_draws(H, ctx):
    y = _series()
    spec = H.ProblemSpec(y, [1], [60], K=3, n_chains=2, burnin=5, nrun=3, flags=H.FLAG_SUMMARY | H.FLAG_DIAGNOSTICS)
    with pytest.raises(H.HmcGpuError) as e:
        H.estimate(ctx, spec)
    assert e.value.code == -1 and "nrun >= 4" in str(e.value)
    spec = H.ProblemSpec(y, [1], [60], K=3, n_chains=2, burnin=5, nrun=4, flags=H.FLAG_SUMMARY | H.FLAG_DIAGNOSTICS)
    o = H.estimate(ctx, spec)
    assert o.rhat.shape == (1, 3 * 3 + 9 + 2 + 1)
