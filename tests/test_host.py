"""CPU tests of the host logic and of the C-ABI library as a binary artefact (no compute calls without a GPU)."""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT


def test_library_exports_every_declared_symbol(H):
    header = open(os.path.join(ROOT, "include", "hmcgpu.h")).read()
    declared = set(re.findall(r"\b(hmcgpu_[a-z_]+)\s*\(", header))
    assert declared == set(H.SYMBOLS), declared ^ set(H.SYMBOLS)
    L = H.load()
    for s in declared:
        assert hasattr(L, s), s
    assert L.hmcgpu_version() >= 100


def _header_struct_fields(name):
    """(type, field) pairs of `typedef struct <name> {...}` in include/hmcgpu.h, in declaration order."""
    header = open(os.path.join(ROOT, "include", "hmcgpu.h")).read()
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (name, name), header, re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    out = []
    for decl in body.split(";"):
        decl = " ".join(decl.split())
        if not decl:
            continue
        m = re.match(r"(const )?(\w+)\s*(\*?)\s*(.+)$", decl)
        ctype = m.group(2) + m.group(3)
        for f in m.group(4).split(","):
            out.append((ctype, f.strip()))
    return out


def _c_offsets(tmp_path, name, fields):
    """offsetof of every field and sizeof the struct as gcc lays out include/hmcgpu.h."""
    import subprocess
    src = tmp_path / f"layout_{name}.c"
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "hmcgpu.h"', "int main(void) {"]
    lines += [f'  printf("{f} %zu\\n", offsetof({name}, {f}));' for _, f in fields]
    lines += [f'  printf("sizeof %zu\\n", sizeof({name}));', "  return 0; }"]
    src.write_text("\n".join(lines))
    exe = tmp_path / f"layout_{name}"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)])
    return {k: int(v) for k, v in (ln.split() for ln in subprocess.check_output([str(exe)], text=True).splitlines())}


_C2CTYPES = {"double*": "LP_c_double", "int32_t*": "LP_c_int", "int64_t*": "LP_c_long", "uint8_t*": "LP_c_ubyte",
             "double": "c_double", "int32_t": "c_int", "uint32_t": "c_uint", "int64_t": "c_long", "uint64_t": "c_ulong"}
_C2JULIA = {"double*": "Ptr{Float64}", "int32_t*": "Ptr{Int32}", "int64_t*": "Ptr{Int64}", "uint8_t*": "Ptr{UInt8}",
            "double": "Float64", "int32_t": "Int32", "uint32_t": "UInt32", "int64_t": "Int64", "uint64_t": "UInt64"}


@pytest.mark.parametrize("cname,pyname", [("hmcgpu_problem", "Problem"), ("hmcgpu_result", "Result")])
def test_struct_layout_matches_header(H, tmp_path, cname, pyname):
    """Both bindings mirror include/hmcgpu.h field by field: the ctypes Structure is compared with gcc's offsetof/sizeof
    of the header itself, the Julia struct (never executed here) by field name, order and type."""
    from hmc_jl_b200 import binding as B
    fields = _header_struct_fields(cname)
    off = _c_offsets(tmp_path, cname, fields)
    S = getattr(B, pyname)
    assert [f for f, _ in S._fields_] == [f for _, f in fields]
    assert ctypes.sizeof(S) == off["sizeof"]
    for (ctype, f), (_, pytype) in zip(fields, S._fields_):
        assert getattr(S, f).offset == off[f], f
        assert pytype.__name__ == _C2CTYPES[ctype], (f, pytype.__name__, ctype)
    jl = open(os.path.join(ROOT, "hmc.jl_b200", "julia", "HmcGPU.jl")).read()
    body = re.search(r"struct %s\n(.*?)\nend" % pyname, jl, re.S).group(1)
    jfields = [tuple(x.strip().split("::")) for ln in body.splitlines() for x in ln.split(";") if x.strip()]
    assert jfields == [(f, _C2JULIA[ctype]) for ctype, f in fields]


def test_flag_and_error_constants_match_header(H):
    from hmc_jl_b200 import binding as B
    header = open(os.path.join(ROOT, "include", "hmcgpu.h")).read()
    jl = open(os.path.join(ROOT, "hmc.jl_b200", "julia", "HmcGPU.jl")).read()
    defs = {k: int(v) for k, v in re.findall(r"#define HMCGPU_((?:FLAG|ERR)_\w+) \(?(-?\d+)u?\)?", header)}
    assert len(defs) == 11
    for k, v in defs.items():
        assert getattr(B, k) == v, k
        if k.startswith("FLAG_"):
            assert re.search(r"const %s = UInt32\(%d\)" % (k, v), jl), k


def test_no_device_fails_loudly(H):
    L = H.load()
    if L.hmcgpu_device_count() > 0:
        pytest.skip("a GPU is visible")
    with pytest.raises(H.HmcGpuError) as e:
        H.Context(0)
    assert e.value.code == -5 and "no CPU fallback" in str(e.value)


def test_product_never_imports_oracle():
    """The product path must not import, link, load or call anything under oracle/ (comments may mention it)."""
    pkg = os.path.join(ROOT, "hmc.jl_b200")
    bad = re.compile(r"import\s+oracle|from\s+oracle|libhmc_oracle|hmc_oracle\.h|\borc_[a-z_]+\s*\(")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".jl", ".h")):
                assert not bad.search(open(os.path.join(dp, f)).read()), f


def test_shard_windows_lpt_balance(H):
    starts, ends = H.expanding_windows(101, 600)
    T = ends - starts + 1
    for n in (1, 2, 4, 8):
        shards = H.shard_windows(T, n)
        assert sorted(np.concatenate(shards).tolist()) == list(range(len(T)))
        loads = np.array([T[s].sum() for s in shards])
        assert loads.max() - loads.min() <= T.max()
        assert loads.max() <= 1.01 * T.sum() / n + T.max()


def test_estopt_mirror_defaults_and_validation(H):
    y = np.arange(200.0)
    o = H.EstOpt(y, None)
    assert (o.D, o.burnin, o.Nrun, o.seed, list(o.horizons), o.endIndex) == (3, 1000, 1000, 1234, [12], 121)
    assert list(o.sampleRange)[:2] == [1, 2] and len(o.sampleRange) == 121 and len(o.signalRange) == 0
    o = H.EstOpt(y, None, sampleRange=range(1, 124), signalRange=range(122, 124), signalSave=range(123, 124))
    m = o.signal_mask()
    assert m.sum() == 2 and m[121] == 1 and m[122] == 1 and m[120] == 0                   # 1-based 122:123
    with pytest.raises(ValueError):                                                       # src/Hmc.jl:61
        H.EstOpt(y, None, signalRange=range(130, 132))
    with pytest.raises(ValueError):                                                       # src/Hmc.jl:62
        H.EstOpt(y, None, sampleRange=range(1, 124), signalRange=range(122, 124), signalSave=range(120, 123))
    with pytest.raises(ValueError):
        H.EstOpt(y, None, sampleRange=range(1, 300))
    # accessors (src/Hmc.jl:75-107): 1-based like the reference
    dates = [f"d{i}" for i in range(1, 201)]
    o = H.EstOpt(y, dates, sampleRange=range(3, 124), signalRange=range(122, 124), endIndex=121)
    assert o.obsRange == list(range(3, 122))
    np.testing.assert_array_equal(o.makey(), y[2:123])
    np.testing.assert_array_equal(o.makeysignals(), y[121:123])
    assert (o.enddate(), o.enddate(12), o.startdate()) == ("d121", "d133", "d3")
    assert (o.yobs(1), o.yend(), o.yend(12)) == (0.0, 120.0, 132.0)
    with pytest.raises(IndexError):
        o.yobs(201)
    with pytest.raises(IndexError):
        o.yobs(0)
    o.signalRange = range(130, 132)                                                      # edited by hand, then re-derived
    with pytest.raises(ValueError):
        o.update_itators()
    o.signalRange = range(123, 124)
    assert o.update_itators().obsRange == list(range(3, 123))


def test_problem_spec_layouts(H):
    y = np.random.default_rng(0).normal(size=(3, 50))
    spec = H.ProblemSpec(y, [1, 5], [40, 50], K=3, n_chains=2, burnin=1, nrun=4, horizons=(1, 12),
                         flags=H.FLAG_DRAWS | H.FLAG_SUMMARY | H.FLAG_SMOOTHED_MEAN)
    o, res = spec.alloc_result()
    assert o.mu.shape == (2, 3, 8) and o.A.shape == (2, 3, 3, 8) and o.forecasts.shape == (2, 4, 8)
    assert o.summary_mean.shape == (2, 3 * 3 + 9 + 4 + 1)
    assert o.pib_mean.size == (40 + 46) * 3
    st = spec.struct()
    assert st.y_len == 50 and st.n_series == 3 and st.n_windows == 2 and st.n_h == 2
    assert not st.is_signal and not st.X0 and not st.win_init_series and st.pi_row_back == 0
    mask = np.zeros(50, dtype=np.uint8); mask[45:] = 1
    X0 = [np.ones(40, dtype=np.int64), np.full(46, 2)]
    spec = H.ProblemSpec(y, [1, 5], [40, 50], K=3, is_signal=mask, kappa=0.5, X0=X0, win_init_series=[0, 0], pi_row_back=5)
    st = spec.struct()
    assert st.is_signal[47] == 1 and st.is_signal[3] == 0 and st.kappa == 0.5 and st.pi_row_back == 5
    assert st.X0[39] == 1 and st.X0[40] == 2 and st.win_init_series[1] == 0
    with pytest.raises(ValueError):
        H.ProblemSpec(y, [1, 5], [40, 50], K=3, X0=np.ones(10, dtype=np.int64))
    with pytest.raises(ValueError):
        H.ProblemSpec(y, [1, 5], [40, 50], K=3, is_signal=np.zeros(7))


def test_saveresults_csv_layout(H, tmp_path):
    """src/Hmc.jl:707-748: headers, 5-digit rounding, trans_i_j column order, piB[:, end, :]."""
    from types import SimpleNamespace
    rng = np.random.default_rng(0)
    R, D = 4, 3
    A = rng.dirichlet(np.ones(D), size=(R, D))
    s = SimpleNamespace(μ=rng.normal(size=(R, D)), σ=rng.uniform(1, 2, size=(R, D)), A=A,
                        πb=rng.dirichlet(np.ones(D), size=R)[:, None, :], forecasts=rng.normal(size=(R, 2)))
    dates = [f"2000-{m:02d}-01" for m in range(1, 13)]
    opt = H.EstOpt(np.arange(12.0), dates, sampleRange=range(1, 11), endIndex=10, horizons=[12], D=D)
    paths = H.saveresults(s, opt, str(tmp_path))
    lines = open(paths["filtered_trans_probs"]).read().splitlines()
    assert lines[0] == "date,trans_1_1,trans_2_1,trans_3_1,trans_1_2,trans_2_2,trans_3_2,trans_1_3,trans_2_3,trans_3_3"
    row = lines[1].split(",")
    assert row[0] == "2000-10-01" and len(lines) == R + 1
    np.testing.assert_allclose([float(v) for v in row[1:]], np.round(A[0].T.ravel(), 5))     # trans_i_j = A[i, j]
    assert open(paths["forecasts"]).readline().strip() == "date,forecast_12,forecast_error_12"
    assert open(paths["filtered_means"]).readline().strip() == "date,state_1,state_2,state_3"
    got = np.loadtxt(paths["filtered_state_probs"], delimiter=",", skiprows=1, usecols=(1, 2, 3))
    np.testing.assert_allclose(got, np.round(s.πb[:, -1, :], 5))


def test_write_summaries_matches_reference_summary_columns(H, tmp_path):
    import json
    from types import SimpleNamespace
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "official_summary_subset.json")))
    K, hs = 3, [12]
    F = 3 * K + K * K + 2 * len(hs) + 1
    m = np.arange(2 * F, dtype=float).reshape(2, F)
    paths = H.write_summaries(SimpleNamespace(summary_mean=m), K, hs, ["1979-12-01", "1980-01-01"], str(tmp_path))
    for name in ("filtered_means", "filtered_variances", "filtered_state_probs", "forecasts"):
        hdr = open(paths[name]).readline().strip().split(",")[1:]
        assert hdr == g["columns"][name], name
    hdr = open(paths["filtered_trans_probs"]).readline().strip().split(",")[1:]
    assert sorted(hdr) == sorted(g["columns"]["filtered_trans_probs"])          # same names (the goldens predate the :727 order)
    row = open(paths["filtered_means"]).read().splitlines()[2].split(",")
    assert row[0] == "1980-01-01" and [float(v) for v in row[1:]] == m[1, 0:3].tolist()


def test_dispersion_and_correlation_analytics(H):
    """calcdispersion / calccorr mirrors (src/Hmc.jl:1078-1129) on synthetic draw arrays."""
    from types import SimpleNamespace
    rng = np.random.default_rng(0)
    S, R, D = 5, 40, 3
    n = S * R
    mu = np.sort(rng.normal(size=(n, D)), axis=1) + np.repeat(np.arange(S), R)[:, None]
    s = SimpleNamespace(μ=mu, σ=rng.uniform(0.5, 2, size=(n, D)), πb=rng.dirichlet(np.ones(D), size=n),
                        A=rng.dirichlet(np.ones(D), size=(n, D)), forecasts=np.stack([mu.sum(1), rng.normal(size=n)], 1),
                        signalids=np.repeat(np.arange(1, S + 1), R))
    ids, per = H.signal_summaries(s)
    assert ids.tolist() == [1, 2, 3, 4, 5] and per["filtered_means"].shape == (S, D) and per["filtered_trans_probs"].shape == (S, 9)
    np.testing.assert_allclose(per["filtered_means"][2], mu[2 * R:3 * R].mean(0))
    disp = H.calcdispersion(s)
    m, sd = disp["filtered_means"]
    np.testing.assert_allclose(m, per["filtered_means"].mean(0))
    np.testing.assert_allclose(sd, per["filtered_means"].std(0, ddof=1))
    names, C = H.calccorr(s, D)
    assert len(names) == 3 * D + D * D + 1 and C.shape == (len(names), len(names)) and names[9] == "trans_1_1" and names[10] == "trans_2_1"
    np.testing.assert_allclose(np.diag(C), 1.0)
    assert C[names.index("μ1"), names.index("forecast")] > 0.5
    np.testing.assert_allclose(C[9, 0], np.corrcoef(s.A[:, 0, 0], mu[:, 0])[0, 1])      # trans_1_1 = A[1,1]
    np.testing.assert_allclose(C[10, 0], np.corrcoef(s.A[:, 1, 0], mu[:, 0])[0, 1])     # trans_2_1 = A[2,1]


def test_signal_summary_and_dispersion_csv_layout(H, tmp_path):
    """write_signal_summaries / write_dispersion produce the files of a signals directory (runaggregate with groups
    [:date, :signalid] + calcdispersion, src/Hmc.jl:1053-1090); headers as in data/output/signals_official_noise_*_allsignal."""
    from types import SimpleNamespace
    rng = np.random.default_rng(1)
    S, R, D = 4, 30, 3

    def fake(date, shift):
        n = S * R
        ids = np.repeat(np.arange(1, S + 1), R)
        return SimpleNamespace(μ=np.sort(rng.normal(size=(n, D)), axis=1) + shift + ids[:, None], σ=rng.uniform(0.5, 2, size=(n, D)),
                               πb=rng.dirichlet(np.ones(D), size=n), A=rng.dirichlet(np.ones(D), size=(n, D)),
                               forecasts=rng.normal(size=(n, 2)), signalids=ids, obsdates=np.array([date] * n, dtype=object),
                               signalvals=np.repeat(rng.normal(size=(S, 2)), R, axis=0))
    runs = [fake("1980-01-01", 0.0), fake("1980-02-01", 5.0)]
    sp = H.write_signal_summaries(runs, [12], str(tmp_path))
    dp = H.write_dispersion(runs, [12], str(tmp_path))
    # the reference's own headers (signals_official_noise_0.3_allsignal/forecasts_summary.csv, filtered_means_dispersion.csv)
    assert open(sp["forecasts"]).readline().strip() == "date,signalid,forecast_12_mean,forecast_error_12_mean,signal_1_mean,signal_2_mean"
    assert open(dp["filtered_means"]).readline().strip() == (
        "date,signalid_mean,state_1_mean,state_2_mean,state_3_mean,signal_1_mean,signal_2_mean,"
        "signalid_std,state_1_std,state_2_std,state_3_std,signal_1_std,signal_2_std")
    assert open(dp["forecasts"]).readline().strip() == (
        "date,signalid_mean,forecast_12_mean,forecast_error_12_mean,signal_1_mean,signal_2_mean,"
        "signalid_std,forecast_12_std,forecast_error_12_std,signal_1_std,signal_2_std")
    hdr = open(dp["filtered_trans_probs"]).readline().strip().split(",")
    assert len(hdr) == 1 + 2 * (1 + 9 + 2) and sorted(hdr[2:11]) == sorted(f"trans_{i}_{j}_mean" for i in (1, 2, 3) for j in (1, 2, 3))
    rows = [ln.split(",") for ln in open(sp["filtered_means"]).read().splitlines()[1:]]
    assert len(rows) == 2 * S and rows[S][0] == "1980-02-01" and rows[S][1] == "1"
    _, per = H.signal_summaries(runs[1])
    np.testing.assert_allclose([float(v) for v in rows[S][2:5]], per["filtered_means"][0])
    np.testing.assert_allclose(float(rows[S][5]), runs[1].signalvals[0, 0])
    d = [ln.split(",") for ln in open(dp["filtered_means"]).read().splitlines()[1:]]
    assert len(d) == 2 and d[1][0] == "1980-02-01" and float(d[1][1]) == 2.5                        # mean of signalid 1..4
    disp = H.calcdispersion(runs[1])
    np.testing.assert_allclose([float(v) for v in d[1][2:5]], disp["filtered_means"][0])
    np.testing.assert_allclose([float(v) for v in d[1][8:11]], disp["filtered_means"][1])
    np.testing.assert_allclose(float(d[1][7]), np.std([1, 2, 3, 4], ddof=1))


def test_insample_and_smoothed_writers_use_the_reference_headers(H, tmp_path):
    """saveinsampleforecasts (src/Hmc.jl:701-705, header of data/output/official_insample/forecats_insample.csv) and
    savesmoothresults (:750-758: Date,state_1..state_D)."""
    table = {"date": ["1970-01-01", "1970-02-01"], "forecast": np.array([6.4768, 6.1]), "forecasterror": np.array([1.18, -0.2]),
             "current": np.array([6.18, 6.0]), "future": np.array([5.29, 6.3]),
             "s1": np.array([1e-4, 0.2]), "s2": np.array([0.0489, 0.3]), "s3": np.array([0.951, 0.5])}
    f = H.saveinsampleforecasts(table, str(tmp_path / "insample" / "forecats_insample.csv"))
    lines = open(f).read().splitlines()
    assert lines[0] == "date,forecast,forecasterror,current,future,s1,s2,s3"
    assert lines[1].split(",")[0] == "1970-01-01" and float(lines[1].split(",")[1]) == 6.4768 and len(lines) == 3
    rows = [["1970-01-01", 0.25, 0.75], ["1970-02-01", 0.5, 0.5]]
    g = H.savesmoothresults(rows, str(tmp_path / "smooth"))
    lines = open(g).read().splitlines()
    assert os.path.basename(g) == "smoothed_state_probs.csv" and lines[0] == "Date,state_1,state_2"
    assert lines[2] == "1970-02-01,0.5,0.5"


def test_forecastinsample_filtered_host_logic(H, oracle, monkeypatch):
    """Host side of forecastinsample(probabilities="filtered"): one estimation call with HMCGPU_FLAG_FILTERED_MEAN, whose per-date
    means become the table.  The C-ABI call is replaced by an oracle-backed stand-in (no GPU here) that produces what the device
    accumulates — the mean over the saved draws of pif[t,:] and of pif[t,:]' A^12 mu — and the table is checked against the
    reference's published in-sample table.  The GPU run of the same function is a -m gpu test."""
    import json
    from types import SimpleNamespace
    from conftest import load_inflation
    from hmc_jl_b200 import binding as B
    y, dates = load_inflation()
    g = json.load(open(os.path.join(ROOT, "tests", "golden", "official_insample.json")))
    N = g["last_index"]

    def fake_estimate(ctx, spec):
        assert spec.flags & B.FLAG_FILTERED_MEAN and not spec.flags & B.FLAG_SMOOTHED_MEAN and list(spec.horizons) == [12] and spec.win_end[0] == N
        outs, _ = oracle.gibbs_batch([dict(y=spec.y[0, :N], K=spec.K, burnin=spec.burnin, nrun=spec.nrun, seed=spec.seed, chain=c,
                                           horizons=(12,), y_future=[spec.y[0, N - 1 + 12]]) for c in range(spec.n_chains)])
        cat = lambda k: np.concatenate([getattr(o, k) for o in outs])
        mu, s2, A = cat("mu"), cat("sigma2"), cat("A")
        pick = np.linspace(0, len(mu) - 1, 300).round().astype(np.int64)                 # a thinned sample of the draws keeps the CPU test short
        rng = np.random.default_rng(0)
        probs, fc = np.zeros((N, spec.K)), np.zeros(N)
        for j in pick:
            pif = oracle.forward(spec.y[0, :N], A[j], mu[j], s2[j], rng.dirichlet(np.ones(spec.K)), want_Pf=False).pif
            probs += pif
            fc += pif @ (np.linalg.matrix_power(A[j], 12) @ mu[j])
        return SimpleNamespace(pib_mean=[probs / len(pick)], insample_forecast_mean=[(fc / len(pick))[:, None]], events=0)

    class FakeCtx:
        def close(self):
            pass

    monkeypatch.setattr(B, "estimate", fake_estimate)
    opt = H.EstOpt(y, dates, sampleRange=range(1, N + 1), endIndex=N, horizons=[12], D=3, burnin=1500, Nrun=1500, n_chains=2)
    t = H.forecastinsample(opt, ctx=FakeCtx(), probabilities="filtered")
    assert t["date"][0] == dates[0] and len(t["forecast"]) == N
    p = np.stack([t["s1"], t["s2"], t["s3"]], axis=1)
    np.testing.assert_allclose(p.sum(1), 1.0, atol=1e-9)
    d = np.abs(p - np.array(g["probs"])).max(1)
    assert np.median(d) < 5e-3 and (d < 0.05).mean() > 0.85
    assert np.median(np.abs(t["forecast"] - np.array(g["forecast"]))) < 0.05
    np.testing.assert_allclose(t["forecasterror"][:N - 12], t["forecast"][:N - 12] - y[12:N], atol=1e-12)
    np.testing.assert_array_equal(t["current"], y[:N])
    with pytest.raises(ValueError):
        H.forecastinsample(opt, ctx=FakeCtx(), probabilities="both")


def test_warm_started_window_chaining_host_logic(H, oracle, monkeypatch):
    """sample_and_forecast_all (the intent of the stale sampleAndForecastAll, src/Hmc.jl:584-638): the carried state path, the
    makeParams rule for new dates, beta0 = 2 in chained windows, posterior-mean tables and forecasts — with the three C-ABI
    calls it makes replaced by oracle-backed stand-ins that check the argument shapes the real binding requires."""
    from types import SimpleNamespace
    from conftest import K3_TRUTH, synth_hmm
    from hmc_jl_b200 import binding as B
    y, _ = synth_hmm(260, **K3_TRUTH)
    for n in (150, 201):
        np.testing.assert_array_equal(H.makeparams_states(y[:n], 3), oracle.make_params(y[:n], 3)[0])
    seen = []

    def fake_estimate(ctx, spec):
        end = int(spec.win_end[0])
        X0 = None if spec.X0 is None else spec.X0.copy()
        seen.append(SimpleNamespace(end=end, X0=X0, beta0=spec.hp[3], burnin=spec.burnin, nrun=spec.nrun, wid=int(spec.win_id[0])))
        assert spec.n_chains == 1 and spec.flags & B.FLAG_DRAWS and (X0 is None or X0.shape == (end,))
        r = oracle.gibbs(spec.y[0, :end], spec.K, spec.burnin, spec.nrun, seed=spec.seed, chain=int(spec.win_id[0]), horizons=(12,),
                         y_future=[np.nan], X0=X0, beta0=spec.hp[3])
        return SimpleNamespace(mu=[r.mu.T], sigma2=[r.sigma2.T], A=[np.transpose(r.A, (2, 1, 0))], pi_end=[r.pi_end.T], events=0)

    class FakeCtx:
        def filter(self, yw, A, mu, s2, rho, precision=64, want_totals=True):
            assert A.shape == (1, 3, 3) and mu.shape == s2.shape == rho.shape == (1, 3) and yw.ndim == 1 and precision == 64
            return SimpleNamespace(pif=oracle.forward(yw, A[0], mu[0], s2[0], rho[0], want_Pf=False).pif[None])

        def sample_states(self, A, pif, u, piN=None):
            assert A.shape == (1, 3, 3) and pif.ndim == 3 and u.shape == pif.shape[:2] and (u >= 0).all() and (u < 1).all()
            return oracle.sample_states(pif[0], A[0], u[0], form=1)[None]

        def close(self):
            pass

    monkeypatch.setattr(B, "estimate", fake_estimate)
    dates = [f"d{i}" for i in range(1, 261)]
    out = H.sample_and_forecast_all(y, dates, range(1, 261), [1, 12], range(200, 204), D=3, burnin=60, Nrun=300, initialburn=800,
                                    initialNrun=50, ctx=FakeCtx())
    assert [s.end for s in seen] == [200, 200, 201, 202, 203] and [s.wid for s in seen] == [0, 1, 2, 3, 4]
    assert seen[0].X0 is None and seen[0].beta0 is None and (seen[0].burnin, seen[0].nrun) == (800, 50)
    for a, b in zip(seen[1:], seen[2:]):                               # chained windows: short burn-in, beta0 = 2, carried path
        assert (b.burnin, b.nrun) == (60, 300) and b.beta0.tolist() == [2.0, 2.0, 2.0] and len(b.X0) == len(a.X0) + 1
        assert b.X0[-1] == H.makeparams_states(y[:b.end], 3)[-1]       # the new date starts from the makeParams rule (:612-617)
    # the carried path is a draw of X | theta, y: overwhelmingly equal to the true regime on this well-separated series
    assert out["dates"] == ["d200", "d201", "d202", "d203"] and out["μ"].shape == (4, 3) and out["A"].shape == (4, 3, 3)
    np.testing.assert_allclose(out["A"].sum(2), 1.0, atol=1e-9)
    np.testing.assert_allclose(out["πb"].sum(1), 1.0, atol=1e-9)
    assert np.all(np.abs(out["μ"] - np.array(K3_TRUTH["mu"])) < 0.6)                         # warm start: 60 sweeps of burn-in suffice
    f12 = np.array([out["πb"][i] @ np.linalg.matrix_power(out["A"][i], 12) @ out["μ"][i] for i in range(4)])
    np.testing.assert_allclose(out["forecasts"][:, 2], f12, rtol=1e-12)
    np.testing.assert_allclose(out["forecasts"][:, 1], out["forecasts"][:, 0] - y[200:204], rtol=1e-12)
    with pytest.raises(ValueError):
        H.sample_and_forecast_all(y, dates, range(1, 261), [12], range(259, 263), D=3, ctx=FakeCtx())


def test_committed_bench_lines_carry_the_contract_keys():
    """profiles/r1_bench_n*.json are bench.py's own output lines: each parses and carries the measurement contract's keys."""
    import glob
    import json
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r1_bench_n*.json")))
    assert files
    for f in files:
        d = json.loads(open(f).read().strip().splitlines()[-1])
        for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
                  "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline"):
            assert k in d, (f, k)
        assert d["warmup"] >= 3 and d["gpu_launches"] > 0 and d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0
        assert d["roofline"]["bound"] == "hbm" and abs(d["roofline"]["frac"] - d["roofline"]["achieved"] / d["roofline"]["peak"]) < 1e-9
        assert not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
        if d["n_gpus"] == 1:
            assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1


def test_bench_issue_roofline_arithmetic():
    """bench.issue_roofline on the numbers of the committed bench line: nominal fraction as recorded, and the measured
    mixed-blend peak (profiles/r1_issue_peak.json) scaled to the sampled clock."""
    import importlib.util
    import json
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    r = b.issue_roofline(100.0, 3.2e11, 1.0, 148, 1500.0)
    assert abs(r["achieved"] - 1000.0) < 1e-9 and abs(r["peak"] - 888.0) < 1e-9 and abs(r["frac"] - 1000.0 / 888.0) < 1e-12
    m = json.load(open(os.path.join(ROOT, "profiles", "r1_issue_peak.json")))
    want = m["mix_gwarp_inst_s"] * 1500.0 / (m["nominal_issue_gwarp_inst_s_at_max_clock"] / (148 * 4) * 1e3)
    assert abs(r["measured_mixed_peak"] - want) < 1e-6 * want and r["frac_of_measured_mixed_peak"] > r["frac"]


def test_bench_dump_outputs_layout_and_sampling(H, tmp_path):
    """bench.dump_outputs writes the fetched per-window outputs in caller window order as float64 .npy files, and a fixed
    seeded sample of the windows when the whole set would exceed the size limit."""
    import importlib.util
    from types import SimpleNamespace
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    b = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(b)
    nw, F, chains = 50, 7, 3
    shard = np.random.default_rng(0).permutation(nw)
    res = SimpleNamespace(summary_mean=shard[:, None] + np.arange(F) / 10.0, summary_var=-shard[:, None] - np.arange(F) / 10.0,
                          status=np.tile(shard[:, None] % 2, (1, chains)).astype(np.int32))
    names = b.dump_outputs(str(tmp_path / "all"), res, shard, nw)
    assert names == ["status", "summary_mean", "summary_var", "window_index"]
    got = {n: np.load(tmp_path / "all" / f"{n}.npy") for n in names}
    assert all(a.dtype == np.float64 for a in got.values())
    np.testing.assert_array_equal(got["window_index"], np.arange(nw))
    np.testing.assert_array_equal(got["summary_mean"], np.arange(nw)[:, None] + np.arange(F) / 10.0)
    np.testing.assert_array_equal(got["summary_var"], -np.arange(nw)[:, None] - np.arange(F) / 10.0)
    np.testing.assert_array_equal(got["status"], np.tile(np.arange(nw)[:, None] % 2, (1, chains)))
    limit = 20 * (2 * F + chains + 1) * 8
    for d in ("s1", "s2"):
        b.dump_outputs(str(tmp_path / d), res, shard, nw, limit=limit)
    s1 = {n: np.load(tmp_path / "s1" / f"{n}.npy") for n in names}
    assert sum(a.nbytes for a in s1.values()) <= limit and len(s1["window_index"]) == 20
    idx = s1["window_index"].astype(np.int64)
    assert np.all(np.diff(idx) > 0) and idx.max() < nw
    np.testing.assert_array_equal(s1["summary_mean"], got["summary_mean"][idx])
    for n in names:                                                                      # the same sample every time
        np.testing.assert_array_equal(np.load(tmp_path / "s2" / f"{n}.npy"), s1[n])


def test_bench_reference_arm_prints_one_contract_line():
    """`bench.py --impl reference` (the CPU port on the host cores; no GPU involved): exactly one JSON line on stdout with
    the contract's keys, whatever the libraries print."""
    import json, subprocess, sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                        "--burnin", "2", "--nrun", "2"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
              "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["impl"] == "reference" and d["value"] > 0 and d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and "workload" in d["config"]


def test_committed_headline_profile_matches_kernel_sources():
    """bench.py's issue roofline takes warp-instructions per warp-step and DRAM bytes per state-step from the ncu capture in
    profiles/r2_headline_profile.json, and uses them only when the capture was taken from the kernel sources it runs
    (hot_source_hash = sha256 of gibbs_kernel.cuh, hmm_device.cuh, rng.cuh and the compiler flags).  A kernel edit without a new
    capture (scripts/profile_headline.sh on the GPU box) must not go unnoticed: the committed capture has to match the sources."""
    import json
    import sys
    sys.path.insert(0, os.path.join(ROOT, "hmc.jl_b200"))
    import build as hb
    prof = json.load(open(os.path.join(ROOT, "profiles", "r2_headline_profile.json")))
    assert prof["hot_source_hash"] == hb.hot_source_hash(), "kernel sources changed since the committed ncu capture: run scripts/profile_headline.sh"
    assert 60 < prof["warp_inst_per_warp_step"] < 130 and 10 < prof["dram_bytes_per_state_step"] < 40
