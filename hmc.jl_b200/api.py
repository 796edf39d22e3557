"""Host-side mirror of the reference's estimation interface (Julia is not installed here, so the host layer the
parity tests drive is Python; hmc.jl_b200/julia/HmcGPU.jl is the same thing for a Julia user).

  EstOpt           <- Hmc.estopt           (src/Hmc.jl:17-73)   same field names and defaults
  estimatemodel    <- Hmc.estimatemodel    (src/Hmc.jl:850-865) returns (μ, σ, πb, A, forecasts, obsdates)
  estimatesignals  <- Hmc.estimatesignals! (src/Hmc.jl:868-914) noisy-signal Monte Carlo, one chain per perturbed copy
  estimate_windows <- the SLURM array of run_hmm.jl jobs (slurmscripts/base_estimation.sh:5,17): many end dates at once
"""
from __future__ import annotations

from dataclasses import dataclass, field
from types import SimpleNamespace
from typing import Optional, Sequence

import numpy as np

from . import binding as B


@dataclass
class EstOpt:
    """Mirror of `mutable struct estopt` (src/Hmc.jl:17-60).  Ranges are 1-based inclusive like Julia's."""
    rawdata: np.ndarray
    dates: Sequence
    sampleRange: range = range(1, 122)          # 1:121
    signalRange: range = range(2, 2)            # 2:1 (empty)
    signalSave: range = range(2, 2)
    endIndex: int = 121
    horizons: Sequence[int] = (12,)
    D: int = 3
    burnin: int = 1000
    Nrun: int = 1000
    signalburnin: int = 1000
    signalNrun: int = 1000
    noise: float = 0.0
    noiseSamples: int = 1
    σsignal: float = 0.0
    series: str = "offical"
    seed: int = 1234
    # extensions of the GPU path (not in the reference)
    n_chains: int = 1
    precision: int = 64
    device: int = 0

    def __post_init__(self):
        sr = self.sampleRange
        if len(sr) < 2 or sr.step != 1:
            raise ValueError("sampleRange must be a contiguous range of at least 2 observations")
        if sr[0] < 1 or sr[-1] > len(self.rawdata):
            raise ValueError("sampleRange outside rawdata")
        # the reference only logs these two (@error, src/Hmc.jl:61-62) and carries on; here they are hard errors
        if not set(self.signalRange) <= set(sr):
            raise ValueError("signalRange is not a subset of sampleRange")
        if not set(self.signalSave) <= set(self.signalRange):
            raise ValueError("signalSave is not a subset of signalRange")

    # ---- accessors of the reference (src/Hmc.jl:75-107), same names and 1-based index meaning
    @property
    def obsRange(self):
        """setdiff(sampleRange, signalRange) (:63, :76), in sampleRange order."""
        sig = set(self.signalRange)
        return [i for i in self.sampleRange if i not in sig]

    def update_itators(self):
        """`update_itators!` (:75-83).  The reference caches six index vectors that must be rebuilt by hand after the
        ranges are edited (`code/run_hmm.jl` does so per end date); here every range-derived quantity (obsRange, the signal
        mask) is computed on access, so this only re-validates the ranges."""
        self.__post_init__()
        return self

    def makey(self):
        """rawdata[sampleRange] (:85-87)."""
        return np.asarray(self.rawdata, dtype=np.float64)[self.sampleRange[0] - 1:self.sampleRange[-1]]

    def makeysignals(self):
        """rawdata[signalRange] (:89-91)."""
        return np.asarray(self.rawdata, dtype=np.float64)[[i - 1 for i in self.signalRange]]

    def enddate(self, extra: int = 0):
        """dates[endIndex + extra] (:93-95)."""
        return self.dates[self.endIndex + extra - 1]

    def startdate(self):
        """dates[first(sampleRange)] (:97-99)."""
        return self.dates[self.sampleRange[0] - 1]

    def yobs(self, index: int):
        """rawdata[index], 1-based (:101-103)."""
        if index < 1:
            raise IndexError(index)                   # Julia's BoundsError; a negative numpy index would wrap silently
        return float(self.rawdata[index - 1])

    def yend(self, extra: int = 0):
        """rawdata[endIndex + extra] (:105-107)."""
        return self.yobs(self.endIndex + extra)

    def signal_mask(self):
        """uint8 flag per index of rawdata: 1 on opt.signalRange (obsRange = setdiff(sampleRange, signalRange), :63)."""
        m = np.zeros(len(self.rawdata), dtype=np.uint8)
        for i in self.signalRange:
            m[i - 1] = 1
        return m


def estimatemodel(opt: EstOpt, ctx: Optional[B.Context] = None):
    """GPU drop-in for Hmc.estimatemodel(opt) (src/Hmc.jl:850-865).

    Returns a namespace with the reference's NamedTuple fields and shapes:
      μ (Nrun, D), σ (Nrun, D) [variances], A (Nrun, D, D), forecasts (Nrun, 2*len(horizons)), obsdates (Nrun,),
      πb (Nrun, 1, D): only the end-of-window row is materialised — `saveresults` reads πb[:, end, :] (:744), which
      works unchanged on this array; the full Nrun x N x D tensor (3.5 GB per end date in production) is never built.
    With n_chains > 1 the draw axis is n_chains*Nrun (chain-major).
    """
    own = ctx is None
    ctx = ctx or B.Context(opt.device)
    try:
        sr = opt.sampleRange
        # With a non-empty signalRange the reference's estimatemodel still routes through the signal branches of
        # update_μσ! / forwardupdate_P! with hp = HyperParams(Y, D), i.e. κ = 1.0 (:132, :853) — mirrored here.
        sig = opt.signal_mask() if len(opt.signalRange) else None
        spec = B.ProblemSpec(np.asarray(opt.rawdata, dtype=np.float64), [sr[0]], [sr[-1]], K=opt.D, n_chains=opt.n_chains,
                             burnin=opt.burnin, nrun=opt.Nrun, seed=opt.seed, horizons=list(opt.horizons),
                             precision=opt.precision, flags=B.FLAG_REF_Q1 | B.FLAG_DRAWS, is_signal=sig, kappa=1.0)
        o = B.estimate(ctx, spec)
    finally:
        if own:
            ctx.close()
    R = opt.n_chains * opt.Nrun
    date = opt.dates[opt.endIndex - 1] if opt.dates is not None else None
    fc = o.forecasts[0].T.copy() if o.forecasts is not None else np.empty((R, 0))
    if sr[-1] != opt.endIndex:
        # :861 propagates πb[end] h steps from the END of the window but scores against yobs(endIndex + h)
        y = np.asarray(opt.rawdata, dtype=np.float64)
        for k, h in enumerate(opt.horizons):
            fc[:, 2 * k + 1] = fc[:, 2 * k] - (y[opt.endIndex + h - 1] if opt.endIndex + h <= len(y) else np.nan)
    return SimpleNamespace(
        μ=o.mu[0].T.copy(), σ=o.sigma2[0].T.copy(),
        A=np.transpose(o.A[0], (2, 1, 0)).copy(),            # stored [s][r][draw] -> (draw, r, s)
        πb=o.pi_end[0].T.copy()[:, None, :],
        forecasts=fc,
        obsdates=np.array([date] * R, dtype=object), events=o.events, gpu_ms=o.gpu_ms)


def estimatesignals(opt: EstOpt, ctx: Optional[B.Context] = None, rng: Optional[np.random.Generator] = None):
    """GPU drop-in for Hmc.estimatesignals!(opt) (src/Hmc.jl:868-914): the noisy-signal Monte Carlo.

    opt.noiseSamples perturbed copies of the sample (real data + N(0, σsignal²) noise on opt.signalRange, :890) are
    estimated with the signal-aware sampler: signals are emitted with sd·(1+κ) (:382) and enter the conjugate draws with
    weight 1/(1+κ) (:302-314), κ = opt.noise, priors HyperParams(opt) (α = ν = 2, ξ = mean of the real sample,
    :148-159); X0 comes from makeParams on the real data (:888).  As in the reference, a zero opt.σsignal is first set to
    mean(σ²-draws)·noise from a plain estimatemodel run (:869-872) — opt is updated in place like the `!` says.

    One difference, stated: the reference runs the copies one after the other on ONE chain (copy s starts from the final
    state of copy s−1, each with its own signalburnin); here every copy is an independent chain started from X0, all
    copies side by side on the GPU (× opt.n_chains chains per copy).  After burn-in the draws have the same distribution.
    The perturbations use numpy's Generator(seed) — Julia's MersenneTwister stream cannot be reproduced.

    Returns the reference's NamedTuple fields: μ, σ (Ndraws, D), πb (Ndraws, D) = smoothed probabilities at row
    opt.endIndex (:893), A (Ndraws, D, D), forecasts (Ndraws, 2|H|), obsdates, signalvals (Ndraws, |signalSave|),
    signalids; Ndraws = noiseSamples·n_chains·signalNrun, copy-major."""
    own = ctx is None
    ctx = ctx or B.Context(opt.device)
    try:
        if np.isclose(opt.σsignal, 0.0):                                      # :869-872
            base = estimatemodel(opt, ctx)
            opt.σsignal = float(base.σ.mean() * opt.noise)
        sr, D, S = opt.sampleRange, opt.D, opt.noiseSamples
        y = np.asarray(opt.rawdata, dtype=np.float64)
        rng = rng or np.random.default_rng(opt.seed)
        sig_idx = np.array(list(opt.signalRange), dtype=np.int64) - 1
        series = np.tile(y, (S + 1, 1))                                        # series 0 = real data, s = 1..S perturbed
        series[1:, sig_idx] += rng.standard_normal((S, len(sig_idx))) * opt.σsignal   # :890
        sigLen = (opt.signalRange[-1] if len(opt.signalRange) else opt.endIndex) - opt.endIndex     # :886
        hs = [max(h - sigLen, 0) for h in opt.horizons]                        # :901-905: horizon counted from the window end
        two = np.full(D, 2.0)
        xi = np.full(D, y[sr[0] - 1:sr[-1]].mean())                           # HyperParams(opt) :148-159
        spec = B.ProblemSpec(series, [sr[0]] * S, [sr[-1]] * S, K=D, n_chains=opt.n_chains, burnin=opt.signalburnin,
                             nrun=opt.signalNrun, seed=opt.seed, horizons=hs, precision=opt.precision,
                             flags=B.FLAG_REF_Q1 | B.FLAG_DRAWS, win_series=np.arange(1, S + 1), win_init_series=np.zeros(S),
                             xi=xi, alpha=two, nu=two, kappa=opt.noise, is_signal=opt.signal_mask(),
                             pi_row_back=sr[-1] - opt.endIndex)
        o = B.estimate(ctx, spec)
    finally:
        if own:
            ctx.close()
    R = opt.n_chains * opt.signalNrun
    cat = lambda a: np.concatenate([a[w].T for w in range(S)])                  # (S*R, ...) copy-major
    fc = cat(o.forecasts) if o.forecasts is not None else np.empty((S * R, 0))
    for k, h in enumerate(opt.horizons):
        yreal = y[opt.endIndex + h - 1] if opt.endIndex + h <= len(y) else np.nan
        if sigLen == h:                                                        # forecastsignal (:670-681), `noise` = σsignal (:904)
            a = (1.0 / opt.σsignal) / (1.0 + 1.0 / opt.σsignal)
            signal = np.repeat(series[1:, opt.endIndex + h - 1], R)
            fc[:, 2 * k] = a * signal + (1.0 - a) * fc[:, 2 * k]             # horizon 0 from the window end = πb_end'μ
            fc[:, 2 * k + 1] = fc[:, 2 * k] - yreal
        elif sigLen > h:                                                       # left unassigned by the reference (:900-906)
            fc[:, 2 * k:2 * k + 2] = np.nan
        else:
            fc[:, 2 * k + 1] = fc[:, 2 * k] - yreal                           # error against the REAL series (:902)
    date = opt.dates[opt.endIndex - 1] if opt.dates is not None else None
    save_idx = np.array(list(opt.signalSave), dtype=np.int64) - 1
    return SimpleNamespace(
        μ=cat(o.mu), σ=cat(o.sigma2), πb=cat(o.pi_end),
        A=np.concatenate([np.transpose(o.A[w], (2, 1, 0)) for w in range(S)]),
        forecasts=fc, obsdates=np.array([date] * (S * R), dtype=object),
        signalvals=np.repeat(series[1:, save_idx], R, axis=0), signalids=np.repeat(np.arange(1, S + 1), R),
        events=o.events, gpu_ms=o.gpu_ms, σsignal=opt.σsignal)


def expanding_windows(first_end: int, last_end: int, start: int = 1):
    """The reference's rolling scheme: sampleRange = startindex:dateindex for every end date (code/run_hmm.jl:80,98)."""
    ends = np.arange(first_end, last_end + 1, dtype=np.int32)
    return np.full_like(ends, start), ends


def shard_windows(T: Sequence[int], n_shards: int):
    """Longest-processing-time-first assignment of windows to shards by T_w (cost of a window is ∝ T_w).
    Returns a list of index arrays, one per shard (the same rule hmcgpu_estimate_multi applies)."""
    T = np.asarray(T)
    order = np.argsort(-T, kind="stable")
    load = np.zeros(n_shards, dtype=np.int64)
    out = [[] for _ in range(n_shards)]
    for w in order:
        d = int(np.argmin(load))
        out[d].append(int(w))
        load[d] += int(T[w])
    return [np.array(sorted(s), dtype=np.int64) for s in out]


def estimate_windows(y, win_start, win_end, *, K=3, n_chains=1, burnin=1000, nrun=1000, seed=1234, horizons=(12,),
                     precision=32, draws=False, summary=True, smoothed=False, loglik=False, win_id=None,
                     win_series=None, diagnostics=False, predictive_grid=None, quantiles=None, rank_diagnostics=False,
                     ctx: Optional[B.Context] = None, device: int = 0):
    """Many end-date windows in one call (what the SLURM job array does one process at a time).  `diagnostics=True` adds
    `rhat`, `ess` and `ess_lag` [n_windows, F] (split-R̂ and effective sample size per summary field; see write_diagnostics).
    `predictive_grid` (increasing points, shared by every window and horizon) adds the posterior predictive distribution of
    every forecast: `pred_cdf` [n_windows, n_h, n_grid], `pit` and `log_score` [n_windows, n_h] and `pred_moments`
    [n_windows, n_h, 3] (mean, variance, skewness); see write_predictive and include/hmcgpu.h.  `quantiles` (probabilities
    in [0, 1]) and / or `rank_diagnostics=True` keep every saved draw on the device (HMCGPU_FLAG_RANKED) and add the exact
    posterior `quantiles` [n_windows, F, n_probs], the rank-normalised split-R̂ `rhat_rank` and the bulk / tail effective
    sample sizes `ess_bulk` / `ess_tail` [n_windows, F]; see write_ranked."""
    ranked = quantiles is not None or rank_diagnostics
    flags = B.FLAG_REF_Q1 | (B.FLAG_DRAWS if draws else 0) | (B.FLAG_SUMMARY if summary else 0) \
        | (B.FLAG_SMOOTHED_MEAN if smoothed else 0) | (B.FLAG_LOGLIK if loglik else 0) \
        | (B.FLAG_DIAGNOSTICS if diagnostics else 0) | (B.FLAG_PREDICTIVE if predictive_grid is not None else 0) \
        | (B.FLAG_RANKED if ranked else 0)
    spec = B.ProblemSpec(y, win_start, win_end, K=K, n_chains=n_chains, burnin=burnin, nrun=nrun, seed=seed,
                         horizons=list(horizons), precision=precision, flags=flags, win_id=win_id, win_series=win_series,
                         pred_grid=predictive_grid, quantile_probs=quantiles)
    own = ctx is None
    ctx = ctx or B.Context(device)
    try:
        return B.estimate(ctx, spec)
    finally:
        if own:
            ctx.close()


def gather_window_summaries(local: np.ndarray, shard: np.ndarray, n_windows: int, dist=None, device=None):
    """Final host gather of per-window summaries (the only cross-rank step of the path; no data-path collective).

    `local` [len(shard), F] holds this rank's windows, `shard` their global indices.  Returns the full
    [n_windows, F] table on rank 0 (None elsewhere).  `dist` is torch.distributed (initialised: nccl on the
    GPU box, gloo in the CPU tests) or None for a single process."""
    local = np.ascontiguousarray(local, dtype=np.float64)
    if dist is None or dist.get_world_size() == 1:
        sh = np.asarray(shard)
        if len(sh) == n_windows and np.array_equal(sh, np.arange(n_windows)):
            return local                             # one process holding every window in order: nothing to move
        out = np.empty((n_windows, local.shape[1]))
        out[np.asarray(shard)] = local
        return out
    import torch
    world, rank = dist.get_world_size(), dist.get_rank()
    # shards are balanced by sum of T_w (LPT), not by window count: a shard of short windows can hold many more rows than
    # n_windows / world, so the padded payload is sized by the real maximum over the ranks
    rows = torch.tensor([len(shard)], dtype=torch.int64, device=device if device is not None else "cpu")
    dist.all_reduce(rows, op=dist.ReduceOp.MAX)
    max_rows = max(1, int(rows.item()))
    # payload rows: [global index, F values]; padded with index -1
    pad = torch.full((max_rows, local.shape[1] + 1), -1.0, dtype=torch.float64)
    pad[: len(shard), 0] = torch.as_tensor(np.asarray(shard), dtype=torch.float64)
    pad[: len(shard), 1:] = torch.from_numpy(local)
    if device is not None:
        pad = pad.to(device)
    parts = [torch.empty_like(pad) for _ in range(world)] if rank == 0 else None
    dist.gather(pad, parts, dst=0)
    if rank != 0:
        return None
    out = np.full((n_windows, local.shape[1]), np.nan)
    for t in parts:
        t = t.cpu().numpy()
        keep = t[:, 0] >= 0
        out[t[keep, 0].astype(np.int64)] = t[keep, 1:]
    return out


# ---------------------------------------------------------------------------------------------------------------------
# Output layer (SURVEY section 8f-1): the reference's per-end-date CSVs and the per-date means of code/aggregate.jl

def _fmt(v, digits=5):
    return repr(round(float(v), digits))


def saveresults(samples, opt: EstOpt, directory: str, precision: int = 5, hassignals: bool = False):
    """Mirror of Hmc.saveresults(samples, opt, dir; hassignals=false) (src/Hmc.jl:724-748 -> basicsave :707-722):
    five CSVs per end date, one row per draw, values rounded to `precision` digits (:719).  Headers as the current
    reference code builds them: state_i; trans_i_j in column-major order of (i, j) with column trans_i_j = A[i, j]
    (:727, :745); forecast_h, forecast_error_h (:729-732)."""
    import os
    os.makedirs(directory, exist_ok=True)
    D = opt.D
    date = str(opt.dates[opt.endIndex - 1])
    h1 = [f"state_{i}" for i in range(1, D + 1)]
    h2 = [f"trans_{i}_{j}" for j in range(1, D + 1) for i in range(1, D + 1)]
    h3 = []
    for h in opt.horizons:
        h3 += [f"forecast_{h}", f"forecast_error_{h}"]
    R = samples.μ.shape[0]
    tables = {
        "filtered_means": (h1, samples.μ),
        "filtered_variances": (h1, samples.σ),
        "filtered_state_probs": (h1, samples.πb if hassignals else samples.πb[:, -1, :]),    # :738 / :744
        "filtered_trans_probs": (h2, np.transpose(samples.A, (0, 2, 1)).reshape(R, D * D)),  # reshape(A, Nrun, :) column-major
        "forecasts": (h3, samples.forecasts),
    }
    paths = {}
    for name, (hdr, data) in tables.items():
        path = os.path.join(directory, f"{name}_{date}.csv")
        with open(path, "w") as f:
            if hassignals:   # basicsave with signal / signalids (:707-721): date, signalid, data..., signal_1..n
                nsig = samples.signalvals.shape[1]
                f.write(",".join(["date", "signalid"] + hdr + [f"signal_{i}" for i in range(1, nsig + 1)]) + "\n")
                for sid, row, sv in zip(samples.signalids, np.asarray(data), samples.signalvals):
                    f.write(",".join([date, str(int(sid))] + [_fmt(v, precision) for v in row] + [_fmt(v, 5) for v in sv]) + "\n")
            else:
                f.write(",".join(["date"] + hdr) + "\n")
                for row in np.asarray(data):
                    f.write(",".join([date] + [_fmt(v, precision) for v in row]) + "\n")
        paths[name] = path
    return paths


def _summary_tables(table, K: int, horizons: Sequence[int], suffix: str):
    """Splits an [n_windows, F] table in the summary field order (include/hmcgpu.h) into the reference's per-variable CSV
    tables: {name: (column names, [n_windows, n_cols] block)}; every column name ends in `suffix`."""
    m = np.asarray(table)
    nh = len(horizons)
    states = [f"state_{i}_{suffix}" for i in range(1, K + 1)]
    return {
        "filtered_means": (states, m[:, 0:K]),
        "filtered_variances": (states, m[:, K:2 * K]),
        # summary A index s*K + r = A[r, s]  ->  column-major (i, j) order with trans_i_j = A[i, j]
        "filtered_trans_probs": ([f"trans_{i}_{j}_{suffix}" for j in range(1, K + 1) for i in range(1, K + 1)], m[:, 2 * K:2 * K + K * K]),
        "filtered_state_probs": (states, m[:, 2 * K + K * K:3 * K + K * K]),
        "forecasts": (sum([[f"forecast_{h}_{suffix}", f"forecast_error_{h}_{suffix}"] for h in horizons], []),
                      m[:, 3 * K + K * K:3 * K + K * K + 2 * nh]),
    }


def _write_tables(tables, dates: Sequence, directory: str, file_suffix: str):
    import os
    os.makedirs(directory, exist_ok=True)
    paths = {}
    for name, (hdr, data) in tables.items():
        path = os.path.join(directory, f"{name}_{file_suffix}.csv")
        with open(path, "w") as f:
            f.write(",".join(["date"] + hdr) + "\n")
            for d, row in zip(dates, data):
                f.write(",".join([str(d)] + [repr(float(v)) for v in row]) + "\n")
        paths[name] = path
    return paths


def write_summaries(out, K: int, horizons: Sequence[int], dates: Sequence, directory: str):
    """Per-date posterior means in the layout of the reference's `<var>_summary.csv` (Hmc.runaggregate,
    src/Hmc.jl:1025-1051: group by date, mean -> columns `<col>_mean`), computed on the device
    (HMCGPU_FLAG_SUMMARY) instead of from 250 000-row draw files.  One row per window, in caller order."""
    return _write_tables(_summary_tables(out.summary_mean, K, horizons, "mean"), dates, directory, "summary")


def write_diagnostics(out, K: int, horizons: Sequence[int], dates: Sequence, directory: str):
    """Convergence diagnostics next to the summaries: `<var>_rhat.csv` (split-R̂, columns `<col>_rhat`) and `<var>_ess.csv`
    (effective sample size, columns `<col>_ess`), one row per window in the column layout of write_summaries; computed on the
    device (HMCGPU_FLAG_DIAGNOSTICS, estimate_windows(diagnostics=True)).  NaN marks a field with a non-finite draw (a forecast
    horizon past the end of the series) or no within-chain variation.  An ESS whose autocorrelation sum reached the lag cap
    (out.ess_lag, include/hmcgpu.h) over-estimates the effective sample size.  Returns {"<var>_rhat": path, "<var>_ess": path}."""
    paths = {}
    for kind, table in (("rhat", out.rhat), ("ess", out.ess)):
        for name, path in _write_tables(_summary_tables(table, K, horizons, kind), dates, directory, kind).items():
            paths[f"{name}_{kind}"] = path
    return paths


def write_ranked(out, K: int, horizons: Sequence[int], dates: Sequence, directory: str):
    """The ranked outputs of estimate_windows(quantiles=..., rank_diagnostics=True) in the column layout of write_summaries,
    one row per window in caller order: `<var>_q<pct>.csv` per quantile probability (columns `<col>_q<pct>`, e.g. `_q5` for
    0.05), `<var>_rhat_rank.csv` (rank-normalised split-R̂), `<var>_ess_bulk.csv` and `<var>_ess_tail.csv`.  NaN marks a field
    with a non-finite draw; R̂ / ESS are also NaN for a field (or a tail indicator) without within-chain variation.
    Returns {"<var>_<kind>": path}."""
    tables = [(f"q{100 * float(p):g}", np.asarray(out.quantiles)[:, :, j]) for j, p in enumerate(out.quantile_probs)]
    tables += [("rhat_rank", out.rhat_rank), ("ess_bulk", out.ess_bulk), ("ess_tail", out.ess_tail)]
    paths = {}
    for kind, table in tables:
        for name, path in _write_tables(_summary_tables(table, K, horizons, kind), dates, directory, kind).items():
            paths[f"{name}_{kind}"] = path
    return paths


def write_predictive(out, horizons: Sequence[int], grid: Sequence[float], dates: Sequence, directory: str):
    """The posterior predictive distributions of estimate_windows(predictive_grid=grid), one row per window in caller order:
    `predictive_cdf_h<h>.csv` per horizon (date, then the CDF at every grid point; columns named by the point) and
    `predictive_scores.csv` (date, then pit_<h>, log_score_<h>, mean_<h>, variance_<h>, skewness_<h> per horizon).  PIT and
    log score are NaN for a horizon past the end of the series.  Returns {"cdf_h<h>": path, ..., "scores": path}."""
    import os
    os.makedirs(directory, exist_ok=True)
    cdf, m = np.asarray(out.pred_cdf), np.asarray(out.pred_moments)
    grid = [float(g) for g in grid]
    tables = {f"cdf_h{h}": (f"predictive_cdf_h{h}.csv", [repr(g) for g in grid], cdf[:, j, :]) for j, h in enumerate(horizons)}
    hdr, cols = [], []
    for j, h in enumerate(horizons):
        hdr += [f"pit_{h}", f"log_score_{h}", f"mean_{h}", f"variance_{h}", f"skewness_{h}"]
        cols += [np.asarray(out.pit)[:, j], np.asarray(out.log_score)[:, j], m[:, j, 0], m[:, j, 1], m[:, j, 2]]
    tables["scores"] = ("predictive_scores.csv", hdr, np.stack(cols, axis=1))
    paths = {}
    for key, (fname, cols_hdr, data) in tables.items():
        path = os.path.join(directory, fname)
        with open(path, "w") as f:
            f.write(",".join(["date"] + cols_hdr) + "\n")
            for d, row in zip(dates, data):
                f.write(",".join([str(d)] + [repr(float(v)) for v in row]) + "\n")
        paths[key] = path
    return paths


def predictive_quantiles(cdf, grid, probs):
    """Quantiles of a predictive distribution from its CDF on a grid (out.pred_cdf[..., :] over `grid`), by linear
    interpolation between grid points: accurate to the grid spacing, not better.  `cdf` [..., n_grid] (non-decreasing along the
    last axis), `probs` [n_p]; returns [..., n_p], NaN where a probability lies outside [cdf[0], cdf[-1]] (the grid does not
    cover that quantile) or the CDF is NaN."""
    cdf = np.asarray(cdf, dtype=np.float64)
    grid = np.asarray(grid, dtype=np.float64)
    probs = np.atleast_1d(np.asarray(probs, dtype=np.float64))
    flat = cdf.reshape(-1, cdf.shape[-1])
    res = np.full((flat.shape[0], len(probs)), np.nan)
    for i, c in enumerate(flat):
        if not np.all(np.isfinite(c)):
            continue
        inside = (probs >= c[0]) & (probs <= c[-1])
        res[i, inside] = np.interp(probs[inside], c, grid)
    return res.reshape(cdf.shape[:-1] + (len(probs),))


def forecastinsample(opt: EstOpt, horizon_index: int = -1, ctx: Optional[B.Context] = None, probabilities: str = "smoothed"):
    """GPU version of the reference's in-sample table (forecastinsample + saveinsampleforecasts, src/Hmc.jl:683-705;
    the reference's own function is stale/un-callable): one full-sample estimation, then per date t of the sample the
    posterior means of the h-step forecast p[j,t,:]' A_j^h mu_j, its error vs y[t+h], y[t], y[t+h] and the state
    probabilities p.  Returns a dict of columns: date, forecast, forecasterror, current, future, s1..sD.

    probabilities="smoothed": p = pib, what `samples.πb[j,date,:]` holds in the current source (:689, :695); accumulated on the
        device inside the sweep kernel (HMCGPU_FLAG_SMOOTHED_MEAN).
    probabilities="filtered": p = pif, the real-time probabilities P(X_t | y_1..t, θ_j).  This is what the reference's PUBLISHED
        table data/output/official_insample/forecats_insample.csv contains (its code state stored the filtered rows: the
        published s1..s3 agree with the posterior mean of pif to a median 5e-4 and are far from pib in mid-sample,
        tests/test_oracle.py::test_golden_insample_table_is_filtered).  Accumulated on the device by the forward pass of the
        same estimation call, over every saved draw (HMCGPU_FLAG_FILTERED_MEAN); ρ is the sampler's own draw of each sweep
        (:350-356)."""
    if probabilities not in ("smoothed", "filtered"):
        raise ValueError("probabilities must be 'smoothed' or 'filtered'")
    own = ctx is None
    ctx = ctx or B.Context(opt.device)
    sr = opt.sampleRange
    y = np.asarray(opt.rawdata, dtype=np.float64)
    h = list(opt.horizons)[horizon_index]
    try:
        flag = B.FLAG_SMOOTHED_MEAN if probabilities == "smoothed" else B.FLAG_FILTERED_MEAN
        spec = B.ProblemSpec(y, [sr[0]], [sr[-1]], K=opt.D, n_chains=opt.n_chains, burnin=opt.burnin, nrun=opt.Nrun,
                             seed=opt.seed, horizons=list(opt.horizons), precision=opt.precision, flags=B.FLAG_REF_Q1 | flag)
        o = B.estimate(ctx, spec)
        fc = o.insample_forecast_mean[0][:, horizon_index]
        probs = o.pib_mean[0]
    finally:
        if own:
            ctx.close()
    idx = np.arange(sr[0], sr[-1] + 1)                       # 1-based dates of the sample
    fut = np.array([y[i - 1 + h] if i - 1 + h < len(y) else np.nan for i in idx])
    table = {"date": [opt.dates[i - 1] for i in idx] if opt.dates is not None else idx.tolist(),
             "forecast": fc, "forecasterror": fc - fut, "current": y[idx - 1], "future": fut}
    for k in range(opt.D):
        table[f"s{k + 1}"] = probs[:, k]
    return table


def saveinsampleforecasts(table, fname: str):
    """Mirror of Hmc.saveinsampleforecasts (src/Hmc.jl:701-705): the table of `forecastinsample` as CSV with the reference's
    header `date,forecast,forecasterror,current,future,s1..sD` (layout of data/output/official_insample/forecats_insample.csv;
    CSV.jl writes full-precision floats, `repr` does the same here)."""
    import os
    os.makedirs(os.path.dirname(os.path.abspath(fname)), exist_ok=True)
    D = sum(1 for k in table if k.startswith("s") and k[1:].isdigit())
    cols = ["date", "forecast", "forecasterror", "current", "future"] + [f"s{i}" for i in range(1, D + 1)]
    with open(fname, "w") as f:
        f.write(",".join(cols) + "\n")
        for i in range(len(table["forecast"])):
            f.write(",".join([str(table["date"][i])] + [repr(float(table[c][i])) for c in cols[1:]]) + "\n")
    return fname


def smoothStates(rawdata, dates, dataRange, *, D: int = 2, burnin: int = 1000, Nrun: int = 1000, n_chains: int = 1, seed: int = 1234,
                 precision: int = 64, ctx: Optional[B.Context] = None):
    """GPU version of Hmc.smoothStates (src/Hmc.jl:640-656): one estimation on rawdata[dataRange] and, per date of the sample, the
    posterior mean of the smoothed state probabilities πb[t, :] (`calcPostior`, :564-571), accumulated on the device
    (HMCGPU_FLAG_SMOOTHED_MEAN).  Returns the reference's table: a list of rows [date, p_1, ..., p_D]."""
    y = np.asarray(rawdata, dtype=np.float64)
    s, e = int(dataRange[0]), int(dataRange[-1])
    own = ctx is None
    ctx = ctx or B.Context(0)
    try:
        spec = B.ProblemSpec(y, [s], [e], K=D, n_chains=n_chains, burnin=burnin, nrun=Nrun, seed=seed, horizons=[], precision=precision,
                             flags=B.FLAG_REF_Q1 | B.FLAG_SMOOTHED_MEAN)
        o = B.estimate(ctx, spec)
    finally:
        if own:
            ctx.close()
    pm = o.pib_mean[0]
    return [[dates[j - 1] if dates is not None else j] + pm[i].tolist() for i, j in enumerate(range(s, e + 1))]


def savesmoothresults(πbresults, directory: str):
    """Mirror of Hmc.savesmoothresults (src/Hmc.jl:750-758): `smoothed_state_probs.csv` with the reference's header
    `Date,state_1,...,state_D` (its Dname vector is state_0..state_D with the first entry replaced by Date)."""
    import os
    os.makedirs(directory, exist_ok=True)
    path = os.path.join(directory, "smoothed_state_probs.csv")
    D = len(πbresults[0]) - 1
    with open(path, "w") as f:
        f.write(",".join(["Date"] + [f"state_{j}" for j in range(1, D + 1)]) + "\n")
        for row in πbresults:
            f.write(",".join([str(row[0])] + [repr(float(v)) for v in row[1:]]) + "\n")
    return path


def makeparams_states(Y, D: int):
    """The initial state path of `makeParams` (src/Hmc.jl:161-195, :185-187): X_i = argmax_s pdf(Normal(μ0_s, std(Y)), y_i) on the
    grid μ0 = range(median − 0.25R, median + 0.25R, length = D), first maximum on ties (`findmax`).  1-based states.
    (The library applies the same rule on the device when no X0 is passed; this host copy exists for window chaining.)"""
    Y = np.asarray(Y, dtype=np.float64)
    R = Y.max() - Y.min()
    med = float(np.median(Y))
    lo, hi = med - 0.25 * R, med + 0.25 * R
    mu0 = np.array([lo + (hi - lo) * (k / (D - 1)) for k in range(D)]) if D > 1 else np.array([med])
    # the pdfs share sd: first maximum of the pdf = first minimum of |y - mu0_k| (exact; the library and the oracle use the same form)
    return np.argmin(np.abs(Y[:, None] - mu0[None, :]), axis=1).astype(np.int64) + 1


def sample_and_forecast_all(rawdata, dates, dataRange, horizons, filterRange, *, D: int = 2, burnin: int = 1000, Nrun: int = 1000,
                            initialburn: int = 1000, initialNrun: int = 1000, seed: int = 1234, precision: int = 64,
                            ctx: Optional[B.Context] = None, rng: Optional[np.random.Generator] = None):
    """Warm-started rolling estimation: the intent of the reference's `sampleAndForecastAll` (src/Hmc.jl:584-638, stale — it calls
    helpers with signatures that no longer exist): one long burn-in on the first sample, then for every end date j of
    filterRange a SHORT burn-in started from the previous window's state path (new dates initialised by the makeParams rule,
    :613-617), posterior means per end date (`calcPostior`, :564-571) and forecasts from those means (:631-635).

    The device never materialises X, so the carried path is re-drawn: after each window the last parameter draw θ goes through
    the batched filter and the backward sampler (hmcgpu_filter + hmcgpu_sample_states with fresh uniforms), which is exactly the
    conditional X | θ, y the next sweep of that chain would have sampled — the chain continues with the same law, not the same
    realisation.  β stays at its post-first-sweep value 2 in the chained windows (:347).  End dates are serial by construction
    (the opposite of hmcgpu_estimate's all-end-dates-at-once batch); each call is a narrow batch on the time-parallel kernel.

    Returns a dict of tables with one row per end date: dates, μ [n, D], σ [n, D] (variances), A [n, D, D], πb [n, D] (last
    row), forecasts [n, 2|H|] (forecast, error vs rawdata[j + h]; NaN past the end of the data) and events."""
    y = np.asarray(rawdata, dtype=np.float64)
    start = int(dataRange[0])
    ends = [int(j) for j in filterRange]
    if not ends or start < 1 or ends[0] - start + 1 < 2 or ends[-1] > len(y):
        raise ValueError("filterRange must lie inside rawdata and leave at least 2 observations in the first sample")
    rng = rng or np.random.default_rng(seed)
    own = ctx is None
    ctx = ctx or B.Context(0)
    two = np.full(D, 2.0)
    hs = [int(h) for h in horizons] or [1]     # per-draw device forecasts are not used here (forecasts come from the posterior means)

    def run(end, X0, burn, nrun, beta0, wid):
        spec = B.ProblemSpec(y, [start], [end], K=D, n_chains=1, burnin=burn, nrun=nrun, seed=seed, horizons=hs, precision=precision,
                             flags=B.FLAG_REF_Q1 | B.FLAG_DRAWS, X0=None if X0 is None else [X0], beta0=beta0, win_id=[wid])
        o = B.estimate(ctx, spec)
        mu, s2 = o.mu[0][:, -1], o.sigma2[0][:, -1]
        A = np.ascontiguousarray(o.A[0][:, :, -1].T)                              # stored [s][r][draw] -> A[r, s] of the last draw
        Yw = y[start - 1:end]
        pif = ctx.filter(Yw, A[None], mu[None], s2[None], rng.dirichlet(np.ones(D))[None], precision=64, want_totals=False).pif
        X = ctx.sample_states(A[None], pif, rng.random((1, len(Yw))))[0]
        return o, X

    try:
        _, X = run(ends[0], None, initialburn, initialNrun, None, 0)             # :596-603 long burn-in on the first sample
        n, nh = len(ends), len(horizons)
        out = {"dates": [dates[j - 1] if dates is not None else j for j in ends], "μ": np.empty((n, D)), "σ": np.empty((n, D)),
               "A": np.empty((n, D, D)), "πb": np.empty((n, D)), "forecasts": np.full((n, 2 * nh), np.nan), "events": 0}
        for i, j in enumerate(ends):
            X0 = makeparams_states(y[start - 1:j], D)                             # :612 makeParams(Y, D) ...
            m = min(len(X0), len(X))
            X0[:m] = X[:m]                                                        # ... :613-615 copy over the previous states
            o, X = run(j, X0, burnin, Nrun, two, i + 1)
            mu, A = o.mu[0].mean(1), np.transpose(o.A[0], (2, 1, 0)).mean(0)      # calcPostior: means over the draws
            pe = o.pi_end[0].mean(1)
            out["μ"][i], out["σ"][i], out["A"][i], out["πb"][i] = mu, o.sigma2[0].mean(1), A, pe
            out["events"] += int(o.events)
            for k, h in enumerate(horizons):
                f = float(pe @ np.linalg.matrix_power(A, int(h)) @ mu)            # forecast (:658-667) at the posterior means
                out["forecasts"][i, 2 * k] = f
                if j + h <= len(y):
                    out["forecasts"][i, 2 * k + 1] = f - y[j + h - 1]
    finally:
        if own:
            ctx.close()
    return out


# ---------------------------------------------------------------------------------------------------------------------
# Offline analytics of the reference (SURVEY section 8f-4), on the arrays the GPU path returns instead of on CSV files

def signal_summaries(samples):
    """Per-signal posterior means — what Hmc.runaggregate produces for a signals directory (groups = [:date, :signalid],
    src/Hmc.jl:1062-1075).  Returns (signalids [S], dict name -> [S, columns])."""
    ids = np.unique(samples.signalids)
    R = samples.μ.shape[0]
    tabs = {"filtered_means": samples.μ, "filtered_variances": samples.σ, "filtered_state_probs": samples.πb,
            "filtered_trans_probs": np.transpose(samples.A, (0, 2, 1)).reshape(R, -1), "forecasts": samples.forecasts}
    return ids, {k: np.stack([v[samples.signalids == i].mean(0) for i in ids]) for k, v in tabs.items()}


def calcdispersion(samples):
    """Mirror of Hmc.calcdispersion (src/Hmc.jl:1078-1090) for one end date: mean and standard deviation (n-1, like
    Statistics.std) ACROSS the perturbed copies of the per-copy posterior means.  dict name -> (mean [cols], std [cols])."""
    _, per_signal = signal_summaries(samples)
    return {k: (v.mean(0), v.std(0, ddof=1) if len(v) > 1 else np.full(v.shape[1], np.nan)) for k, v in per_signal.items()}


def _signal_tables(samples, horizons: Sequence[int]):
    """name -> (column names without suffix, [S, columns]) per perturbed copy, incl. the saved signal values (constant within a
    copy, so their mean is the value itself), in the column order of the reference's signal CSVs (:707-721, :733-741)."""
    ids, per_signal = signal_summaries(samples)
    D = samples.μ.shape[1]
    vals = np.stack([samples.signalvals[samples.signalids == i].mean(0) for i in ids])
    sig_cols = [f"signal_{j}" for j in range(1, vals.shape[1] + 1)]
    state = [f"state_{i}" for i in range(1, D + 1)]
    heads = {"filtered_means": state, "filtered_variances": state, "filtered_state_probs": state,
             "filtered_trans_probs": [f"trans_{i}_{j}" for j in range(1, D + 1) for i in range(1, D + 1)],
             "forecasts": sum([[f"forecast_{h}", f"forecast_error_{h}"] for h in horizons], [])}
    return ids, {k: (heads[k] + sig_cols, np.concatenate([per_signal[k], vals], axis=1)) for k in heads}


def write_signal_summaries(samples_by_date, horizons: Sequence[int], directory: str):
    """`<var>_summary.csv` of a signals directory: Hmc.runaggregate with groups [:date, :signalid] (src/Hmc.jl:1053-1076),
    one row per (end date, perturbed copy) = that copy's posterior means, columns `<col>_mean`.
    samples_by_date: iterable of estimatesignals results (one per end date)."""
    import os
    os.makedirs(directory, exist_ok=True)
    paths, files = {}, {}
    for smp in samples_by_date:
        ids, tabs = _signal_tables(smp, horizons)
        for name, (hdr, data) in tabs.items():
            if name not in files:
                paths[name] = os.path.join(directory, f"{name}_summary.csv")
                files[name] = open(paths[name], "w")
                files[name].write(",".join(["date", "signalid"] + [h + "_mean" for h in hdr]) + "\n")
            for i, row in zip(ids, data):
                files[name].write(",".join([str(smp.obsdates[0]), str(int(i))] + [repr(float(v)) for v in row]) + "\n")
    for f in files.values():
        f.close()
    return paths


def write_dispersion(samples_by_date, horizons: Sequence[int], directory: str):
    """`<var>_dispersion.csv`: Hmc.calcdispersion (src/Hmc.jl:1078-1090) = per end date the mean and the standard deviation
    (n−1) over the perturbed copies of every column of `<var>_summary.csv` (signalid included, as DataFrames.aggregate does):
    `date, signalid_mean, <col>_mean…, signal_j_mean…, signalid_std, <col>_std…, signal_j_std…` — the layout of
    data/output/signals_official_noise_*_allsignal/*_dispersion.csv."""
    import os
    os.makedirs(directory, exist_ok=True)
    paths, files = {}, {}
    for smp in samples_by_date:
        ids, tabs = _signal_tables(smp, horizons)
        for name, (hdr, data) in tabs.items():
            full = np.concatenate([ids[:, None].astype(np.float64), data], axis=1)
            cols = ["signalid"] + hdr
            if name not in files:
                paths[name] = os.path.join(directory, f"{name}_dispersion.csv")
                files[name] = open(paths[name], "w")
                files[name].write(",".join(["date"] + [c + "_mean" for c in cols] + [c + "_std" for c in cols]) + "\n")
            sd = full.std(0, ddof=1) if len(full) > 1 else np.full(full.shape[1], np.nan)
            files[name].write(",".join([str(smp.obsdates[0])] + [repr(float(v)) for v in full.mean(0)] + [repr(float(v)) for v in sd]) + "\n")
    for f in files.values():
        f.close()
    return paths


def calccorr(samples, D: int):
    """Mirror of the per-date block of Hmc.calccorr (src/Hmc.jl:1092-1129): correlation matrix across draws of
    [μ_1..D, σ_1..D, π_1..D, trans_i_j (column-major), first forecast].  Returns (names, matrix)."""
    R = samples.μ.shape[0]
    pib = samples.πb if samples.πb.ndim == 2 else samples.πb[:, -1, :]
    cols = np.concatenate([samples.μ, samples.σ, pib, np.transpose(samples.A, (0, 2, 1)).reshape(R, D * D),
                           samples.forecasts[:, :1]], axis=1)
    names = [f"μ{i}" for i in range(1, D + 1)] + [f"σ{i}" for i in range(1, D + 1)] + [f"π{i}" for i in range(1, D + 1)] \
        + [f"trans_{i}_{j}" for j in range(1, D + 1) for i in range(1, D + 1)] + ["forecast"]
    return names, np.corrcoef(cols, rowvar=False)
