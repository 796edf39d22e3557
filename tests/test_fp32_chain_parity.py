"""fp32 sweep kernels, draw by draw, against the fp64 oracle chain on the same Philox streams and chain ids.

An fp32 chain can leave the fp64 chain only through a discrete decision that rounding flips: a categorical draw of the
backward sampler or an accept/reject test of a gamma draw.  The oracle reports, per sweep, how far those decisions were from
flipping (oracle.gibbs(want_margins=True): state_margin, gamma_margin).  Hence:

* draw 0 of every chain is a deterministic function of the makeParams states and the Philox streams; it must match the
  oracle's within the fp32 bar unless its sweep-0 gamma_margin is below DELTA_G;
* draws 1 and 2 of a chain are held to the same bar when the chain is certified: every earlier state_margin above DELTA_S and
  every gamma_margin up to that draw above DELTA_G.  This is what checks the fp32 backward sampler and the statistics it
  accumulates for the next sweep (shifted sums and the last state's complement, packed transition counters and their flushes,
  the segment kernel's composed products).

Tolerances (TOL): mu, sigma2, forecasts 1e-3 relative (mu and forecasts: relative to at
least a tenth of the window's range, i.e. 1e-4 x range absolute; a pi_end error of 1e-4 moves a forecast that much);
A, pi_end 1e-4 absolute; loglik 1e-4 relative.  Errors are reported as multiples of the tolerance.

Calibration (NVIDIA B200, 1000 W power limit; every case of this file).  Outside the statistics hazard below, the worst error of
a certified chain was 0.5 x the tolerance (loglik; every other quantity <= 0.3 x, typically 0.01 x), and no chain left the
oracle's through a discrete decision: the smallest margins passed without a flip were 1.9e-7 (states) and 6.7e-7 (gamma).  The
largest fp32 error in the probabilities the backward sampler compares against was 1.7e-6 (pi_end), so DELTA_S = 2e-5 is about
ten times it; DELTA_G = 1e-5 is about ten times the fp32 rounding of a gamma test (~1e-6).  A case must certify MIN_CERTIFIED
of its chains through the last draw; long windows and large K get an explicit lower floor, since each of the (K - 1) T
boundaries of a sweep lies within DELTA_S of its uniform with probability up to 2 DELTA_S, and each of the K^2 + 2K gamma
draws adds its own chance.

Statistics hazard (measured; a strict xfail until fixed): the K <= 4 kernels keep the state statistics as sums about one
per-window shift and form s2 = Qd - n dbar^2 in fp32 (hmm_device.cuh).  For tight states far from the window mean this
cancels: two states at 0 and 100 with variance 0.01 put sigma2 1.5 % off at draw 0 and 3-9 % off at draws 1-2 on the scan,
thread and segment kernels (loglik 0.7-1.6 %).  With the default prior (xi = window mean) the (ybar - xi)^2 term of b hides it;
with xi at the state means it reaches the sigma2 draw.  The levels series (200/250/300, variance 1) is at 1.3 x the
tolerance on the thread kernel at draw 2.

With FLAG_LOGLIK on and off (different template instantiations) every other output is bit-identical.
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import K3_TRUTH, synth_hmm

pytestmark = pytest.mark.gpu

DELTA_S, DELTA_G = 2e-5, 1e-5
MIN_CERTIFIED = 0.9
TOL = dict(mu=1e-3, sigma2=1e-3, forecasts=1e-3, A=1e-4, pi_end=1e-4, loglik=1e-4)

# kernel -> (environment, hmcgpu_result.sweep_kernel)
KERNELS = {
    "scan": ({"HMCGPU_SCAN_MAX_CHAINS": "1000000"}, 1),
    "thread": ({"HMCGPU_SCAN_MAX_CHAINS": "0", "HMCGPU_SEG_LANES": "0"}, 0),
    "seg2": ({"HMCGPU_SCAN_MAX_CHAINS": "0", "HMCGPU_SEG_LANES": "2"}, 4),
    "seg4": ({"HMCGPU_SCAN_MAX_CHAINS": "0", "HMCGPU_SEG_LANES": "4"}, 4),
    "seg8": ({"HMCGPU_SCAN_MAX_CHAINS": "0", "HMCGPU_SEG_LANES": "8"}, 4),
    "mixed": ({"HMCGPU_SCAN_MAX_CHAINS": "0", "HMCGPU_SEG_LONG": "4"}, 4),        # 4 windows x 8 chains on 8 lanes, the rest on 4
    "lane": ({"HMCGPU_LANE_KERNEL": "1"}, 2),
}
_SWITCHES = ("HMCGPU_SCAN_MAX_CHAINS", "HMCGPU_SEG_LANES", "HMCGPU_SEG_LONG", "HMCGPU_SEG_MIXED", "HMCGPU_LANE_KERNEL")


@pytest.fixture
def force(monkeypatch):
    """force(kernel): set that kernel's switches (and clear the others); returns the sweep_kernel it must report."""
    def f(kernel):
        for v in _SWITCHES:
            monkeypatch.delenv(v, raising=False)
        env, code = KERNELS[kernel]
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        return code
    return f


def truth(K, sep=2.0, s2=0.5, stay=0.9):
    A = np.full((K, K), (1 - stay) / (K - 1)) + np.eye(K) * (stay - (1 - stay) / (K - 1))
    return dict(A=A, mu=sep * np.arange(K), sigma2=np.full(K, s2))


def series(K, n, seed=1):
    return synth_hmm(n, seed=seed, **(K3_TRUTH if K == 3 else truth(K)))[0]


def ragged(T, short=True):
    """Window lengths T, T-1, T-2, T-3 (every residue mod 4) and, with short, windows of 3 and 2 steps."""
    lens = [T, T - 1, T - 2, T - 3] + ([3, 2] if short else [])
    return [1 + i for i in range(len(lens))], [1 + i + n - 1 for i, n in enumerate(lens)]


def check_chains(H, ctx, oracle, y, ws, we, K, nc, code, nrun=3, seed=7, hs=(1, 12), xi=None, alpha=None, nu=None,
                 is_signal=None, kappa=1.0, X0=None, pi_row_back=0, mean_flag=0, min_certified=MIN_CERTIFIED):
    """Run the batch in fp32 (FLAG_LOGLIK on and off) and every chain on the oracle; assert the draw-by-draw parity described
    in the module docstring.  Returns the oracle's outputs and the device's."""
    y = np.asarray(y, dtype=np.float64)
    flags = H.FLAG_REF_Q1 | H.FLAG_DRAWS | mean_flag
    kw = dict(K=K, n_chains=nc, burnin=0, nrun=nrun, seed=seed, horizons=hs, precision=32, xi=xi, alpha=alpha, nu=nu,
              is_signal=is_signal, kappa=kappa, X0=X0, pi_row_back=pi_row_back)
    o = H.estimate(ctx, H.ProblemSpec(y, ws, we, flags=flags | H.FLAG_LOGLIK, **kw))
    assert o.sweep_kernel == code, (H.binding.KERNEL_NAMES[o.sweep_kernel], code)
    assert o.events == 0
    q = H.estimate(ctx, H.ProblemSpec(y, ws, we, flags=flags, **kw))
    for k in ("mu", "sigma2", "A", "pi_end", "forecasts", "pib_mean", "insample_forecast_mean"):
        a, b = getattr(o, k), getattr(q, k)
        if a is not None:
            for w in range(len(ws)):
                np.testing.assert_array_equal(a[w], b[w], err_msg=f"{k}: FLAG_LOGLIK changed another output")
    jobs = []
    for w, (s, e) in enumerate(zip(ws, we)):
        for c in range(nc):
            jobs.append(dict(y=y[s - 1:e], K=K, burnin=0, nrun=nrun, seed=seed, chain=w * nc + c, horizons=hs,
                             y_future=[y[e - 1 + h] for h in hs], flags=oracle.FLAG_REF_Q1 | oracle.FLAG_PIF_FORM,
                             xi=xi, alpha=alpha, nu=nu, kappa=kappa, want_margins=True,
                             want_pib_full=bool(pi_row_back or mean_flag),
                             is_signal=None if is_signal is None else is_signal[s - 1:e],
                             X0=None if X0 is None else X0[w]))
    outs, _ = oracle.gibbs_batch(jobs)
    worst = {k: np.zeros(nrun) for k in TOL}
    n_cert = 0
    flips = []
    for w, (s, e) in enumerate(zip(ws, we)):
        T = e - s + 1
        floor = 0.1 * max(np.ptp(y[s - 1:e]), 1e-6)
        for c in range(nc):
            r = outs[w * nc + c]
            sl = slice(c * nrun, (c + 1) * nrun)
            ref_pi = r.pib_full[:, T - 1 - pi_row_back, :] if pi_row_back else r.pi_end
            got = dict(mu=o.mu[w][:, sl].T, sigma2=o.sigma2[w][:, sl].T, A=np.transpose(o.A[w][:, :, sl], (2, 1, 0)),
                       pi_end=o.pi_end[w][:, sl].T, forecasts=o.forecasts[w][0::2, sl].T, loglik=o.loglik[w][sl])
            ref = dict(mu=r.mu, sigma2=r.sigma2, A=r.A, pi_end=ref_pi, forecasts=r.forecasts[:, 0::2], loglik=r.loglik)
            for d in range(nrun):
                err = {}
                for k in TOL:
                    g, x = np.asarray(got[k][d], dtype=np.float64), np.asarray(ref[k][d], dtype=np.float64)
                    if k in ("A", "pi_end"):
                        den = 1.0
                    elif k == "sigma2":
                        den = np.abs(x)
                    else:
                        den = np.maximum(np.abs(x), floor if k != "loglik" else 0.0)
                    err[k] = float(np.max(np.abs(g - x) / den) / TOL[k]) if np.all(np.isfinite(g)) else np.inf
                cert = bool(np.all(r.state_margin[:d] > DELTA_S) and np.all(r.gamma_margin[:d + 1] > DELTA_G))
                if cert:
                    for k in TOL:
                        worst[k][d] = max(worst[k][d], err[k])
                if max(err.values()) > 1:          # the margins of every chain that left the oracle's: what DELTA_* rest on
                    flips.append((w, c, d, cert, float(np.min(r.state_margin[:d], initial=np.inf)), float(np.min(r.gamma_margin[:d + 1]))))
                if d == nrun - 1:
                    n_cert += cert
    frac = n_cert / (len(ws) * nc)
    print("FP32PARITY", os.environ.get("PYTEST_CURRENT_TEST", "").split(" ")[0], dict(cert=round(frac, 3), worst={k: [float(f"{v:.3g}") for v in worst[k]] for k in TOL},
                             min_state_margin=float(min(np.min(r.state_margin[:nrun - 1], initial=np.inf) for r in outs)),
                             min_gamma_margin=float(min(np.min(r.gamma_margin) for r in outs)), flips=flips[:8]))
    bad = {k: v.tolist() for k, v in worst.items() if np.max(v) > 1}
    assert not bad, f"certified chains off the oracle by these multiples of the tolerance (per draw): {bad}"
    assert frac >= min_certified, f"only {frac:.2f} of the chains certified"
    return outs, o


# ---------------------------------------------------------------------------------------------------- plain sweeps, K <= 4

@pytest.mark.parametrize("K", [2, 3, 4])
@pytest.mark.parametrize("kernel", ["scan", "thread", "seg2", "seg4", "seg8", "mixed"])
def test_plain_sweeps(H, ctx, oracle, force, kernel, K):
    """Ragged windows of every length mod 4 plus 3- and 2-step windows, 8 chains each."""
    code = force(kernel)
    y = series(K, 330, seed=10 + K)
    ws, we = ragged(300)
    check_chains(H, ctx, oracle, y, ws, we, K, 8, code)


@pytest.mark.parametrize("K", [2, 3, 4])
@pytest.mark.parametrize("kernel", ["scan", "thread"])
def test_user_initial_states(H, ctx, oracle, force, kernel, K):
    code = force(kernel)
    rng = np.random.default_rng(K)
    y = series(K, 260, seed=20 + K)
    ws, we = ragged(240, short=False)
    X0 = [rng.integers(1, K + 1, e - s + 1) for s, e in zip(ws, we)]
    check_chains(H, ctx, oracle, y, ws, we, K, 10, code, X0=X0)


@pytest.mark.parametrize("kappa", [0.0, 0.6, 3.0])
@pytest.mark.parametrize("K", [2, 3, 4])
@pytest.mark.parametrize("kernel", ["scan", "thread"])
def test_signals(H, ctx, oracle, force, kernel, K, kappa):
    """Signal mask (a block at the window ends and a few inside), kappa-weighted statistics, HyperParams(opt) priors and the
    smoothed row N - 6 as pi_end."""
    code = force(kernel)
    y = series(K, 220, seed=30 + K)
    ws, we = ragged(200, short=False)
    mask = np.zeros(len(y), dtype=np.uint8)
    mask[[20, 21, 77]] = 1
    for e in we:
        mask[e - 6:e] = 1
    two = np.full(K, 2.0)
    check_chains(H, ctx, oracle, y, ws, we, K, 10, code, is_signal=mask, kappa=kappa, alpha=two, nu=two,
                 xi=np.full(K, float(np.mean(y))), pi_row_back=6)


# ---------------------------------------------------------------------------------------------------- per-date means

@pytest.mark.parametrize("flag", ["smoothed", "filtered"])
@pytest.mark.parametrize("K", [3, 4, 5, 6, 7, 8])
def test_per_date_means_of_draw_zero(H, ctx, oracle, force, K, flag):
    """FLAG_SMOOTHED_MEAN / FLAG_FILTERED_MEAN with nrun = 1 and one chain per window: each window's means are its chain's
    draw 0.  Smoothed: the oracle's pib_full and pib' A^h mu.  Filtered: oracle.forward of the device's own draw with a flat
    rho (the sampler's rho is not returned), compared from row 60 on where rho no longer matters."""
    if K > 4 and flag == "filtered":
        pytest.skip("filtered means are a K <= 4 feature")
    code = force("thread")
    y = series(K, 200, seed=40 + K)
    ends = [180 - 2 * i for i in range(40)]
    ws = [1 + (i % 5) for i in range(40)]
    hs = (1, 12)
    mean_flag = H.FLAG_SMOOTHED_MEAN if flag == "smoothed" else H.FLAG_FILTERED_MEAN
    outs, o = check_chains(H, ctx, oracle, y, ws, ends, K, 1, code, nrun=1, hs=hs, mean_flag=mean_flag)
    worst = 0.0
    for w, (s, e) in enumerate(zip(ws, ends)):
        r = outs[w]
        if not r.gamma_margin[0] > DELTA_G:
            continue
        if flag == "smoothed":
            pib, skip = r.pib_full[0], 0
        else:
            A = o.A[w][:, :, 0].T
            pib = oracle.forward(y[s - 1:e], A, o.mu[w][:, 0], o.sigma2[w][:, 0], np.full(K, 1.0 / K), want_Pf=False).pif
            skip = 60
        mu, A = (r.mu[0], r.A[0]) if flag == "smoothed" else (o.mu[w][:, 0], o.A[w][:, :, 0].T)
        fc = np.stack([pib @ np.linalg.matrix_power(A, h) @ mu for h in hs], axis=1)
        np.testing.assert_allclose(o.pib_mean[w][skip:], pib[skip:], rtol=0, atol=TOL["pi_end"])
        scale = max(np.ptp(y[s - 1:e]), 1e-6)
        np.testing.assert_allclose(o.insample_forecast_mean[w][skip:], fc[skip:], rtol=TOL["forecasts"], atol=0.1 * scale * TOL["forecasts"])
        worst = max(worst, float(np.abs(o.pib_mean[w][skip:] - pib[skip:]).max()))
    print("FP32PARITY means", flag, K, worst)


# ---------------------------------------------------------------------------------------------------- kernel-internal bounds

@pytest.mark.parametrize("K,T", [(3, 1024), (3, 1025), (4, 256), (4, 257)])
def test_packed_transition_rows(H, ctx, oracle, force, K, T):
    """Both sides of the switch from 32- to 64-bit packed transition-counter rows (K = 3: T > 1024, K = 4: T > 256)."""
    code = force("thread")
    y = series(K, T + 12, seed=50 + K)
    check_chains(H, ctx, oracle, y, [1, 1], [T, T - 130], K, 16, code, min_certified=0.8)


@pytest.mark.parametrize("T,kernel", [(504, "seg2"), (505, "thread")])
def test_segment_length_bound(H, ctx, oracle, force, T, kernel):
    """K = 4 with 2 lanes: seg_max_T = 504.  A 504-step window runs on the segment kernel, a 505-step one falls back to the
    thread-per-chain kernel (and must say so)."""
    force("seg2")
    y = series(4, T + 12, seed=60)
    check_chains(H, ctx, oracle, y, [1, 1, 1], [T, T - 1, T - 2], 4, 12, KERNELS[kernel][1], min_certified=0.8)


@pytest.mark.parametrize("K,T", [(5, 4200), (6, 1100), (7, 600), (8, 300)])
@pytest.mark.parametrize("kernel", ["thread", "lane"])
def test_wide_k_across_the_counter_flush(H, ctx, oracle, force, kernel, K, T):
    """K = 5..8: windows past the thread kernel's flush bound of its packed counters, 2^(64/K) - 1 steps, next to one below it."""
    code = force(kernel)
    y = series(K, T + 12, seed=70 + K)
    bound = (1 << (64 // K)) - 1
    check_chains(H, ctx, oracle, y, [1, 1, 3], [T, min(bound - 5, T - 1), T - 17], K, 12, code, min_certified={5: 0.3, 6: 0.6}.get(K, 0.8))


@pytest.mark.parametrize("K", [9, 16, 17, 20, 32])
def test_lane_kernel_widths(H, ctx, oracle, force, K):
    """Lane-per-state kernel: W = 16 (K <= 16) and the max-rescaled W = 32 recursion (K > 16)."""
    code = force("lane")
    y = series(K, 312, seed=80 + K)
    check_chains(H, ctx, oracle, y, [1, 2, 5], [300, 280, 150], K, 12, code, min_certified=0.6)


# ---------------------------------------------------------------------------------------------------- numerical edges

def _edge(name):
    """(y, K, xi, lane_K): the edge series, its K, the prior mean (None = window mean) and the K to run on the lane kernel."""
    rng = np.random.default_rng(11)
    if name == "outliers":                      # 13+ sigma from every state
        y = series(3, 420, seed=5)
        y[50], y[200] = 40.0, -35.0
        return y, 3, None
    if name == "sticky":                        # well-separated sticky regimes: fp32 emission ratios underflow, A ~ 1e-4 entries
        return synth_hmm(620, seed=6, **truth(4, sep=20.0, s2=0.25, stay=0.995))[0], 4, None
    if name == "empty":                         # three clusters, K = 4: makeParams leaves a state empty
        X = rng.choice(3, size=330, p=[0.4, 0.3, 0.3])
        return np.array([0.0, 1.0, 20.0])[X] + 0.3 * rng.standard_normal(330), 4, None
    if name.startswith("levels"):               # a series in levels with a rare last state
        tr = dict(A=np.array([[0.97, 0.025, 0.005], [0.025, 0.97, 0.005], [0.05, 0.05, 0.9]]), mu=np.array([200.0, 250.0, 300.0]),
                  sigma2=np.ones(3))
        y = synth_hmm(620, seed=7, **tr)[0]
        return y, 3, (tr["mu"] if name.endswith("xi") else None)
    if name.startswith("separated"):            # two far-apart, tight states
        tr = dict(A=np.array([[0.95, 0.05], [0.05, 0.95]]), mu=np.array([0.0, 100.0]), sigma2=np.full(2, 0.01))
        y = synth_hmm(920, seed=8, **tr)[0]
        return y, 2, (tr["mu"] if name.endswith("xi") else None)
    raise ValueError(name)


EDGES = ["outliers", "sticky", "empty", "levels", "separated", "levels_xi", "separated_xi"]
# the statistics hazard of the module docstring: s2 = Qd - n dbar^2 about one per-window shift cancels in fp32 (hmm_device.cuh,
# draw_params), measured on a B200 as the largest sigma2 error over draws 0-2 (in units of the 1e-3 tolerance)
HAZARD = {("separated_xi", "scan"): "sigma2 off by 1.5 % at draw 0, 3.2 % at draw 2",
          ("separated_xi", "thread"): "sigma2 off by 1.5 % at draw 0, 9.0 % at draw 2",
          ("separated_xi", "seg4"): "sigma2 off by 1.5 % at draw 0, 5.6 % at draw 2",
          ("levels_xi", "thread"): "sigma2 off by 0.13 % at draw 2"}


@pytest.mark.parametrize("kernel", ["scan", "thread", "seg4"])
@pytest.mark.parametrize("edge", EDGES)
def test_numerical_edges(H, ctx, oracle, force, edge, kernel, request):
    if (edge, kernel) in HAZARD:
        request.applymarker(pytest.mark.xfail(strict=True, reason="fp32 state statistics about one per-window shift: "
                                              + HAZARD[(edge, kernel)]))
    y, K, xi = _edge(edge)
    if edge == "empty":
        X0, _, _ = oracle.make_params(y[:300], K)
        assert len(np.unique(X0)) < K
    code = force(kernel)
    T = len(y) - 20
    ws, we = ragged(T)
    check_chains(H, ctx, oracle, y, ws, we, K, 8, code, xi=xi, min_certified=0.8)


@pytest.mark.parametrize("edge", ["outliers", "sticky"])
def test_numerical_edges_lane(H, ctx, oracle, force, edge):
    """The outlier and sticky-regime series with K = 5 on the lane kernel."""
    y, _, _ = _edge(edge)
    code = force("lane")
    T = len(y) - 20
    check_chains(H, ctx, oracle, y, [1, 2, 3], [T, T - 1, T - 40], 5, 12, code, min_certified=0.8)


def test_fp32_differential_fuzz_against_the_oracle():
    """scripts/fuzz_kernels.py --precision 32: random shapes on every kernel, each against the oracle chain."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "scripts", "fuzz_kernels.py"), "12", "3", "--precision", "32"],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
