"""ctypes binding of libhmcgpu.so — the same C ABI (include/hmcgpu.h) Julia reaches with `ccall`.

No torch, no CPU fallback: if the library is missing or no B200 is visible the calls raise.
"""
from __future__ import annotations

import ctypes as C
import os
from types import SimpleNamespace

import numpy as np

from . import build as _build

FLAG_REF_Q1 = 1
FLAG_DRAWS = 2
FLAG_SUMMARY = 4
FLAG_SMOOTHED_MEAN = 8
FLAG_LOGLIK = 16
FLAG_FILTERED_MEAN = 64   # pib_mean / insample_forecast_mean carry the FILTERED means (the reference's published in-sample table)
FLAG_DIAGNOSTICS = 128    # rhat / ess / ess_lag per window and summary field (split-R̂ and ESS, include/hmcgpu.h)
FLAG_PREDICTIVE = 256     # posterior predictive CDF on a grid, PIT, log score and moments per window and horizon (hmcgpu_predictive)
FLAG_RANKED = 512         # keep every saved draw on the device: exact quantiles, rank-normalised R̂, bulk / tail ESS (hmcgpu_ranked)

ERR_ARG, ERR_CUDA, ERR_ALLOC, ERR_UNSUPPORTED, ERR_NODEVICE = -1, -2, -3, -4, -5

# every symbol include/hmcgpu.h declares
SYMBOLS = [
    "hmcgpu_version", "hmcgpu_device_count", "hmcgpu_ctx_create", "hmcgpu_ctx_destroy", "hmcgpu_last_error",
    "hmcgpu_ctx_sync", "hmcgpu_estimate", "hmcgpu_estimate_multi", "hmcgpu_plan_create", "hmcgpu_plan_run",
    "hmcgpu_plan_fetch", "hmcgpu_plan_destroy", "hmcgpu_filter", "hmcgpu_filter_masked", "hmcgpu_smooth", "hmcgpu_sample_states",
    "hmcgpu_draw_params", "hmcgpu_draw_params_signals", "hmcgpu_forecast", "hmcgpu_philox", "hmcgpu_philox_rounds",
    "hmcgpu_build_info", "hmcgpu_ctx_trim", "hmcgpu_estimate_predictive", "hmcgpu_estimate_multi_predictive",
    "hmcgpu_plan_fetch_predictive", "hmcgpu_estimate_ranked", "hmcgpu_estimate_multi_ranked", "hmcgpu_plan_fetch_ranked",
]
KERNEL_NAMES = {0: "gibbs_sweeps_kernel (thread per chain)", 1: "gibbs_scan_kernel (warp per chain, time-parallel)",
                2: "gibbs_wide_kernel (lane per state)", 3: "(reserved)",
                4: "gibbs_seg_kernel (L lanes per chain, one time segment per lane)"}

_dp = C.POINTER(C.c_double)
_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_u8p = C.POINTER(C.c_uint8)
_u32p = C.POINTER(C.c_uint32)


class Problem(C.Structure):
    _fields_ = [("y", _dp), ("y_len", C.c_int64), ("n_series", C.c_int32), ("n_windows", C.c_int32),
                ("win_series", _i32p), ("win_start", _i32p), ("win_end", _i32p), ("win_id", _i64p),
                ("K", C.c_int32), ("n_chains", C.c_int32), ("burnin", C.c_int64), ("nrun", C.c_int64),
                ("seed", C.c_uint64), ("xi", _dp), ("alpha", _dp), ("nu", _dp), ("beta0", _dp), ("beta", _dp),
                ("kappa", C.c_double), ("is_signal", _u8p), ("horizons", _i32p), ("n_h", C.c_int32),
                ("X0", _i64p), ("precision", C.c_int32), ("flags", C.c_uint32),
                ("win_init_series", _i32p), ("pi_row_back", C.c_int32), ("is_signal_per_series", C.c_int32),
                ("pred_grid", _dp), ("n_grid", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("mu", _dp), ("sigma2", _dp), ("A", _dp), ("pi_end", _dp), ("forecasts", _dp), ("loglik", _dp),
                ("summary_mean", _dp), ("summary_var", _dp), ("pib_mean", _dp), ("insample_forecast_mean", _dp), ("status", _i32p),
                ("gpu_ms", C.c_double), ("sweep_kernel_ms", C.c_double), ("n_launches", C.c_int64),
                ("n_sweep_launches", C.c_int64), ("h2d_bytes", C.c_int64), ("d2h_bytes", C.c_int64),
                ("state_steps", C.c_int64), ("sweep_launch_ms_sum", C.c_double), ("sweep_kernel", C.c_int32), ("n_tasks", C.c_int32),
                ("rhat", _dp), ("ess", _dp), ("ess_lag", _i32p)]


class Predictive(C.Structure):
    _fields_ = [("cdf", _dp), ("pit", _dp), ("log_score", _dp), ("moments", _dp)]


class Ranked(C.Structure):
    _fields_ = [("probs", _dp), ("n_probs", C.c_int32), ("quantiles", _dp), ("rhat_rank", _dp), ("ess_bulk", _dp), ("ess_tail", _dp)]


class HmcGpuError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"hmcgpu error {code}: {msg}")
        self.code = code


_lib = None


def lib_path() -> str:
    return _build.LIB


def load(build_if_missing: bool = True):
    """dlopen the in-tree library (building it with nvcc first if sources are newer)."""
    global _lib
    if _lib is not None:
        return _lib
    path = _build.build() if build_if_missing else _build.LIB
    if not os.path.exists(path):
        raise HmcGpuError(ERR_NODEVICE, f"{path} is missing: run `python __graft_entry__.py` / hmc.jl_b200/build.py (no CPU fallback exists)")
    L = C.CDLL(path)
    L.hmcgpu_last_error.restype = C.c_char_p
    L.hmcgpu_last_error.argtypes = [C.c_void_p]
    L.hmcgpu_ctx_create.argtypes = [C.c_int, C.POINTER(C.c_void_p)]
    L.hmcgpu_ctx_destroy.argtypes = [C.c_void_p]
    L.hmcgpu_ctx_destroy.restype = None
    L.hmcgpu_ctx_sync.argtypes = [C.c_void_p]
    L.hmcgpu_ctx_trim.argtypes = [C.c_void_p]
    L.hmcgpu_build_info.restype = C.c_char_p
    L.hmcgpu_build_info.argtypes = []
    # a library built from other sources than the ones next to it must never be measured or tested by mistake
    info = L.hmcgpu_build_info().decode()
    want = _build.source_hash()
    if want is not None and info.split(";")[1] != want:
        raise HmcGpuError(ERR_UNSUPPORTED, f"{path} was built from other sources (library {info}, sources {want}): rebuild with hmc.jl_b200/build.py --force")
    L.hmcgpu_estimate.argtypes = [C.c_void_p, C.POINTER(Problem), C.POINTER(Result)]
    L.hmcgpu_estimate_multi.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(Problem), C.POINTER(Result)]
    L.hmcgpu_plan_create.argtypes = [C.c_void_p, C.POINTER(Problem), C.POINTER(C.c_void_p)]
    L.hmcgpu_plan_run.argtypes = [C.c_void_p]
    L.hmcgpu_plan_fetch.argtypes = [C.c_void_p, C.POINTER(Result)]
    L.hmcgpu_estimate_predictive.argtypes = [C.c_void_p, C.POINTER(Problem), C.POINTER(Result), C.POINTER(Predictive)]
    L.hmcgpu_estimate_multi_predictive.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(Problem), C.POINTER(Result),
                                                   C.POINTER(Predictive)]
    L.hmcgpu_plan_fetch_predictive.argtypes = [C.c_void_p, C.POINTER(Predictive)]
    L.hmcgpu_estimate_ranked.argtypes = [C.c_void_p, C.POINTER(Problem), C.POINTER(Result), C.POINTER(Predictive), C.POINTER(Ranked)]
    L.hmcgpu_estimate_multi_ranked.argtypes = [C.POINTER(C.c_int), C.c_int, C.POINTER(Problem), C.POINTER(Result),
                                               C.POINTER(Predictive), C.POINTER(Ranked)]
    L.hmcgpu_plan_fetch_ranked.argtypes = [C.c_void_p, C.POINTER(Ranked)]
    L.hmcgpu_plan_destroy.argtypes = [C.c_void_p]
    L.hmcgpu_plan_destroy.restype = None
    L.hmcgpu_filter.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64, _dp, C.c_int64,
                                _dp, _dp, _dp, _dp, _dp, _dp, _dp]
    L.hmcgpu_filter_masked.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64, _dp, C.c_int64, _u8p, C.c_double,
                                       _dp, _dp, _dp, _dp, _dp, _dp, _dp]
    L.hmcgpu_smooth.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64, _dp, _dp, _dp]
    L.hmcgpu_sample_states.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.c_int64, _dp, _dp, _dp, _dp, _i64p]
    L.hmcgpu_draw_params.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, _i64p, _dp, _dp, _i64p,
                                     _dp, _dp, _dp, _dp, C.c_uint64, C.c_uint32, C.c_uint32, _dp, _dp, _dp, _dp]
    L.hmcgpu_draw_params_signals.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_int64, _i64p, _dp, _dp, _i64p, _dp, _dp, C.c_double,
                                             _i64p, _dp, _dp, _dp, _dp, C.c_uint64, C.c_uint32, C.c_uint32, _dp, _dp, _dp, _dp]
    L.hmcgpu_forecast.argtypes = [C.c_void_p, C.c_int32, C.c_int64, _dp, _dp, _dp, _i32p, C.c_int32, _dp, _dp]
    L.hmcgpu_philox.argtypes = [C.c_void_p, C.c_int64, _u32p, _u32p, _u32p]
    L.hmcgpu_philox_rounds.argtypes = [C.c_void_p, C.c_int32, C.c_int64, _u32p, _u32p, _u32p]
    _lib = L
    return L


def _f64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def _p(a, t=_dp):
    return None if a is None else a.ctypes.data_as(t)


def _ref(st):
    return None if st is None else C.byref(st)


class Context:
    """One GPU.  Not re-entrant; use one Context per host thread/GPU (include/hmcgpu.h threading note)."""

    def __init__(self, device: int = 0):
        self.L = load()
        h = C.c_void_p()
        rc = self.L.hmcgpu_ctx_create(device, C.byref(h))
        if rc != 0:
            raise HmcGpuError(rc, self.L.hmcgpu_last_error(None).decode())
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None):
            self.L.hmcgpu_ctx_destroy(self.h)
            self.h = None

    def trim(self):
        """Release the idle device buffers kept for reuse between calls (hmcgpu_ctx_trim)."""
        self._check(self.L.hmcgpu_ctx_trim(self.h))

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc < 0:
            raise HmcGpuError(rc, self.L.hmcgpu_last_error(self.h).decode())
        return rc

    # ---- deterministic pieces -------------------------------------------------------------------------------
    def filter(self, y, A, mu, sigma2, rho, precision=64, want_totals=True, is_signal=None, kappa=1.0):
        """Batched forward filter (forwardupdate_P!, src/Hmc.jl:371-440). A [B,K,K], mu/sigma2/rho [B,K];
        y [T] shared or [B,T]; is_signal [T] (optional) flags the rows emitted with sd*(1+kappa) (:382).
        Returns pif [B,T,K], totals [B,T], loglik [B]."""
        A, mu, sigma2, rho, y = map(_f64, (A, mu, sigma2, rho, y))
        B, K = mu.shape
        T = y.shape[-1]
        stride = T if y.ndim == 2 else 0
        pif = np.empty((B, T, K))
        totals = np.empty((B, T)) if want_totals else None
        ll = np.empty(B)
        if is_signal is None:
            self._check(self.L.hmcgpu_filter(self.h, precision, K, B, T, _p(y), stride, _p(A), _p(mu), _p(sigma2), _p(rho),
                                             _p(pif), _p(totals), _p(ll)))
        else:
            sig = np.ascontiguousarray(is_signal, dtype=np.uint8)
            if sig.shape != (T,):
                raise ValueError("is_signal must have one flag per time step")
            self._check(self.L.hmcgpu_filter_masked(self.h, precision, K, B, T, _p(y), stride, _p(sig, _u8p), float(kappa), _p(A), _p(mu),
                                                    _p(sigma2), _p(rho), _p(pif), _p(totals), _p(ll)))
        return SimpleNamespace(pif=pif, totals=totals, loglik=ll)

    def smooth(self, A, pif, precision=64):
        A, pif = _f64(A), _f64(pif)
        B, T, K = pif.shape
        pib = np.empty_like(pif)
        self._check(self.L.hmcgpu_smooth(self.h, precision, K, B, T, _p(A), _p(pif), _p(pib)))
        return pib

    def sample_states(self, A, pif, u, piN=None):
        """Backward state sampling with injected uniforms (update_X!, src/Hmc.jl:459-484); X is 1-based [B,T]."""
        A, pif, u, piN = _f64(A), _f64(pif), _f64(u), _f64(piN)
        B, T, K = pif.shape
        X = np.empty((B, T), dtype=np.int64)
        self._check(self.L.hmcgpu_sample_states(self.h, K, B, T, _p(A), _p(pif), _p(piN), _p(u), _p(X, _i64p)))
        return X

    def draw_params(self, Ni, S, S2, trans, xi, alpha, nu, beta, seed, chain0, sweep, precision=64, Mi=None, Sm=None, Sm2=None, kappa=1.0):
        Ni = np.ascontiguousarray(Ni, dtype=np.int64)
        trans = np.ascontiguousarray(trans, dtype=np.int64)
        S, S2, xi, alpha, nu, beta = map(_f64, (S, S2, xi, alpha, nu, beta))
        B, K = Ni.shape
        s2, mu, rho, A = np.empty((B, K)), np.empty((B, K)), np.empty((B, K)), np.empty((B, K, K))
        if Mi is None:
            self._check(self.L.hmcgpu_draw_params(self.h, precision, K, B, _p(Ni, _i64p), _p(S), _p(S2), _p(trans, _i64p),
                                                  _p(xi), _p(alpha), _p(nu), _p(beta), seed, chain0, sweep,
                                                  _p(s2), _p(mu), _p(rho), _p(A)))
        else:
            Mi = np.ascontiguousarray(Mi, dtype=np.int64)
            Sm, Sm2 = _f64(Sm), _f64(Sm2)
            self._check(self.L.hmcgpu_draw_params_signals(self.h, precision, K, B, _p(Ni, _i64p), _p(S), _p(S2), _p(Mi, _i64p), _p(Sm),
                                                          _p(Sm2), float(kappa), _p(trans, _i64p), _p(xi), _p(alpha), _p(nu), _p(beta),
                                                          seed, chain0, sweep, _p(s2), _p(mu), _p(rho), _p(A)))
        return s2, mu, rho, A

    def forecast(self, mu, A, pi, horizons, yreal):
        mu, A, pi, yreal = map(_f64, (mu, A, pi, yreal))
        h = np.ascontiguousarray(horizons, dtype=np.int32)
        B, K = mu.shape
        out = np.empty((B, len(h), 2))
        self._check(self.L.hmcgpu_forecast(self.h, K, B, _p(mu), _p(A), _p(pi), _p(h, _i32p), len(h), _p(yreal), _p(out)))
        return out

    def philox(self, ctr, key, rounds=10):
        ctr = np.ascontiguousarray(ctr, dtype=np.uint32)
        key = np.ascontiguousarray(key, dtype=np.uint32)
        out = np.empty_like(ctr)
        self._check(self.L.hmcgpu_philox_rounds(self.h, rounds, len(ctr), _p(ctr, _u32p), _p(key, _u32p), _p(out, _u32p)))
        return out


class ProblemSpec:
    """Owns the numpy buffers behind an hmcgpu_problem."""

    def __init__(self, y, win_start, win_end, K=3, n_chains=1, burnin=1000, nrun=1000, seed=1234, horizons=(12,),
                 precision=32, flags=FLAG_REF_Q1 | FLAG_DRAWS, win_series=None, win_id=None,
                 xi=None, alpha=None, nu=None, beta0=None, beta=None, kappa=1.0, is_signal=None, X0=None,
                 win_init_series=None, pi_row_back=0, pred_grid=None, quantile_probs=None):
        """`pred_grid`: the points of the posterior predictive CDF (FLAG_PREDICTIVE; one grid for every window and horizon).
        `quantile_probs`: the probabilities of the exact posterior quantiles of every summary field (FLAG_RANKED; passed at fetch)."""
        y = np.asarray(y, dtype=np.float64)
        if y.ndim == 1:
            y = y[None, :]
        self.y = np.ascontiguousarray(y)            # [n_series, y_len] == column-major [y_len x n_series]
        self.n_series, self.y_len = self.y.shape
        self.win_start = np.ascontiguousarray(win_start, dtype=np.int32)
        self.win_end = np.ascontiguousarray(win_end, dtype=np.int32)
        self.n_windows = len(self.win_start)
        self.win_series = None if win_series is None else np.ascontiguousarray(win_series, dtype=np.int32)
        self.win_id = None if win_id is None else np.ascontiguousarray(win_id, dtype=np.int64)
        self.K, self.n_chains, self.burnin, self.nrun, self.seed = K, n_chains, burnin, nrun, seed
        self.horizons = np.ascontiguousarray(horizons, dtype=np.int32)
        self.n_h = len(self.horizons)
        self.precision, self.flags, self.kappa = precision, flags, kappa
        self.hp = [_f64(v) for v in (xi, alpha, nu, beta0, beta)]
        self.T = (self.win_end - self.win_start + 1).astype(np.int64)
        self.is_signal = None if is_signal is None else np.ascontiguousarray(is_signal, dtype=np.uint8)
        if self.is_signal is not None and self.is_signal.shape not in ((self.y_len,), (self.n_series, self.y_len)):
            raise ValueError("is_signal must have one flag per time index of the series ([y_len] or [n_series, y_len])")
        self.sig_per_series = int(self.is_signal is not None and self.is_signal.ndim == 2)
        if X0 is not None and not isinstance(X0, np.ndarray):
            X0 = np.concatenate([np.asarray(x, dtype=np.int64) for x in X0])     # list of per-window paths
        self.X0 = None if X0 is None else np.ascontiguousarray(X0, dtype=np.int64)
        if self.X0 is not None and self.X0.shape != (int(self.T.sum()),):
            raise ValueError("X0 must hold sum_w T_w states")
        self.win_init_series = None if win_init_series is None else np.ascontiguousarray(win_init_series, dtype=np.int32)
        self.pi_row_back = int(pi_row_back)
        # the library reads the grid only with the flag, so a grid without it (or the flag without one) is refused here
        self.pred_grid = None if pred_grid is None else np.ascontiguousarray(np.ravel(pred_grid), dtype=np.float64)
        if self.pred_grid is not None and not flags & FLAG_PREDICTIVE:
            raise ValueError("pred_grid given without FLAG_PREDICTIVE")
        if flags & FLAG_PREDICTIVE and self.pred_grid is None:
            raise ValueError("FLAG_PREDICTIVE needs pred_grid")
        self.n_grid = 0 if self.pred_grid is None else len(self.pred_grid)
        # host-side only (hmcgpu_ranked carries them to the fetch); without the flag nothing would compute them
        self.quantile_probs = None if quantile_probs is None else np.ascontiguousarray(np.ravel(quantile_probs), dtype=np.float64)
        if self.quantile_probs is not None and not flags & FLAG_RANKED:
            raise ValueError("quantile_probs given without FLAG_RANKED")

    def struct(self) -> Problem:
        return Problem(_p(self.y), self.y_len, self.n_series, self.n_windows, _p(self.win_series, _i32p),
                       _p(self.win_start, _i32p), _p(self.win_end, _i32p), _p(self.win_id, _i64p), self.K, self.n_chains,
                       self.burnin, self.nrun, self.seed, *[_p(v) for v in self.hp], self.kappa, _p(self.is_signal, _u8p),
                       _p(self.horizons, _i32p), self.n_h, _p(self.X0, _i64p), self.precision, self.flags,
                       _p(self.win_init_series, _i32p), self.pi_row_back, self.sig_per_series, _p(self.pred_grid), self.n_grid)

    def alloc_result(self, diagnostics=None):
        """Output arrays for the flags of this problem.  `diagnostics=True` asks for rhat / ess / ess_lag, which the library
        fills only with FLAG_DIAGNOSTICS (it cannot tell whether a caller's struct has these fields, so it never checks them);
        default: whenever the flag is set."""
        if diagnostics is None:
            diagnostics = bool(self.flags & FLAG_DIAGNOSTICS)
        if diagnostics and not self.flags & FLAG_DIAGNOSTICS:
            raise ValueError("rhat / ess / ess_lag requested without FLAG_DIAGNOSTICS")
        K, nw, nh = self.K, self.n_windows, self.n_h
        R = self.n_chains * self.nrun
        F = 3 * K + K * K + 2 * nh + 1
        o = SimpleNamespace(mu=None, sigma2=None, A=None, pi_end=None, forecasts=None, loglik=None, summary_mean=None,
                            summary_var=None, pib_mean=None, insample_forecast_mean=None, status=np.zeros((nw, self.n_chains), dtype=np.int32),
                            rhat=None, ess=None, ess_lag=None)
        if self.flags & FLAG_DRAWS:
            # Julia column-major (R x K) per window == C arrays [window][k][draw]
            o.mu = np.empty((nw, K, R)); o.sigma2 = np.empty((nw, K, R)); o.A = np.empty((nw, K, K, R))
            o.pi_end = np.empty((nw, K, R))
            o.forecasts = np.empty((nw, 2 * nh, R)) if nh else None
            o.loglik = np.empty((nw, R)) if self.flags & FLAG_LOGLIK else None
        if self.flags & FLAG_SUMMARY:
            o.summary_mean = np.empty((nw, F)); o.summary_var = np.empty((nw, F))
        if self.flags & (FLAG_SMOOTHED_MEAN | FLAG_FILTERED_MEAN):
            o.pib_mean = np.empty(int(self.T.sum()) * K)
            o.insample_forecast_mean = np.empty(int(self.T.sum()) * nh) if nh else None
        if diagnostics:   # [n_windows, F] in the field order of summary_mean
            o.rhat = np.empty((nw, F)); o.ess = np.empty((nw, F)); o.ess_lag = np.empty((nw, F), dtype=np.int32)
        res = Result(_p(o.mu), _p(o.sigma2), _p(o.A), _p(o.pi_end), _p(o.forecasts), _p(o.loglik), _p(o.summary_mean),
                     _p(o.summary_var), _p(o.pib_mean), _p(o.insample_forecast_mean), _p(o.status, _i32p), 0, 0, 0, 0, 0, 0, 0, 0, 0, 0,
                     _p(o.rhat), _p(o.ess), _p(o.ess_lag, _i32p))
        return o, res

    def alloc_predictive(self, o):
        """Adds the predictive outputs to `o` (pred_cdf [nw, n_h, n_grid], pit / log_score [nw, n_h], pred_moments [nw, n_h, 3]:
        mean, variance, skewness) and returns the hmcgpu_predictive struct over them; None without FLAG_PREDICTIVE."""
        if not self.flags & FLAG_PREDICTIVE:
            return None
        nw, nh = self.n_windows, self.n_h
        o.pred_cdf = np.empty((nw, nh, self.n_grid)); o.pit = np.empty((nw, nh)); o.log_score = np.empty((nw, nh))
        o.pred_moments = np.empty((nw, nh, 3))
        return Predictive(_p(o.pred_cdf), _p(o.pit), _p(o.log_score), _p(o.pred_moments))

    def alloc_ranked(self, o, probs=None):
        """Adds the ranked outputs to `o` (quantiles [nw, F, n_probs] at `probs`, default quantile_probs; rhat_rank / ess_bulk /
        ess_tail [nw, F] in the field order of summary_mean) and returns the hmcgpu_ranked struct over them; None without
        FLAG_RANKED."""
        if not self.flags & FLAG_RANKED:
            return None
        probs = self.quantile_probs if probs is None else np.ascontiguousarray(np.ravel(probs), dtype=np.float64)
        probs = np.zeros(0) if probs is None else probs
        nw, F = self.n_windows, 3 * self.K + self.K * self.K + 2 * self.n_h + 1
        o.quantile_probs = probs
        o.quantiles = np.empty((nw, F, len(probs)))
        o.rhat_rank = np.empty((nw, F)); o.ess_bulk = np.empty((nw, F)); o.ess_tail = np.empty((nw, F))
        return Ranked(_p(probs), len(probs), _p(o.quantiles), _p(o.rhat_rank), _p(o.ess_bulk), _p(o.ess_tail))

    def finish(self, o, res, rc):
        o.events = rc
        o.gpu_ms, o.sweep_kernel_ms = res.gpu_ms, res.sweep_kernel_ms
        o.n_launches, o.n_sweep_launches = res.n_launches, res.n_sweep_launches
        o.h2d_bytes, o.d2h_bytes, o.state_steps = res.h2d_bytes, res.d2h_bytes, res.state_steps
        o.sweep_launch_ms_sum, o.sweep_kernel, o.n_tasks = res.sweep_launch_ms_sum, res.sweep_kernel, res.n_tasks
        if o.pib_mean is not None:   # split into per-window [N_w, K] (stored column-major N_w x K)
            K, off, parts = self.K, 0, []
            for n in self.T:
                parts.append(o.pib_mean[off:off + n * K].reshape(K, n).T)
                off += n * K
            o.pib_mean = parts
        if o.insample_forecast_mean is not None:   # per-window [N_w, n_h]
            nh, off, parts = self.n_h, 0, []
            for n in self.T:
                parts.append(o.insample_forecast_mean[off:off + n * nh].reshape(nh, n).T)
                off += n * nh
            o.insample_forecast_mean = parts
        return o


def estimate(ctx: Context, spec: ProblemSpec):
    """hmcgpu_estimate: host buffers in, all sweeps, host buffers out."""
    o, res = spec.alloc_result()
    pr = spec.alloc_predictive(o)
    rk = spec.alloc_ranked(o)
    prob = spec.struct()
    if rk is not None:
        rc = ctx._check(ctx.L.hmcgpu_estimate_ranked(ctx.h, C.byref(prob), C.byref(res), _ref(pr), C.byref(rk)))
    elif pr is None:
        rc = ctx._check(ctx.L.hmcgpu_estimate(ctx.h, C.byref(prob), C.byref(res)))
    else:
        rc = ctx._check(ctx.L.hmcgpu_estimate_predictive(ctx.h, C.byref(prob), C.byref(res), C.byref(pr)))
    return spec.finish(o, res, rc)


def estimate_multi(devices, spec: ProblemSpec):
    L = load()
    o, res = spec.alloc_result()
    pr = spec.alloc_predictive(o)
    rk = spec.alloc_ranked(o)
    prob = spec.struct()
    dev = (C.c_int * len(devices))(*devices)
    if rk is not None:
        rc = L.hmcgpu_estimate_multi_ranked(dev, len(devices), C.byref(prob), C.byref(res), _ref(pr), C.byref(rk))
    elif pr is None:
        rc = L.hmcgpu_estimate_multi(dev, len(devices), C.byref(prob), C.byref(res))
    else:
        rc = L.hmcgpu_estimate_multi_predictive(dev, len(devices), C.byref(prob), C.byref(res), C.byref(pr))
    if rc < 0:
        raise HmcGpuError(rc, L.hmcgpu_last_error(None).decode())
    return spec.finish(o, res, rc)


class Plan:
    """create (upload) / run (device only) / fetch (download) split of hmcgpu_estimate."""

    def __init__(self, ctx: Context, spec: ProblemSpec):
        self.ctx, self.spec = ctx, spec
        self._prob = spec.struct()
        h = C.c_void_p()
        ctx._check(ctx.L.hmcgpu_plan_create(ctx.h, C.byref(self._prob), C.byref(h)))
        self.h = h

    def run(self):
        self.ctx._check(self.ctx.L.hmcgpu_plan_run(self.h))

    def fetch(self):
        o, res = self.spec.alloc_result()
        rc = self.ctx._check(self.ctx.L.hmcgpu_plan_fetch(self.h, C.byref(res)))
        pr = self.spec.alloc_predictive(o)
        if pr is not None:
            self.ctx._check(self.ctx.L.hmcgpu_plan_fetch_predictive(self.h, C.byref(pr)))
        if self.spec.flags & FLAG_RANKED:
            self.fetch_ranked(out=o)
        return self.spec.finish(o, res, rc)

    def fetch_ranked(self, probs=None, out=None):
        """hmcgpu_plan_fetch_ranked: the ranked outputs of the last run (quantiles at `probs`, default the spec's
        quantile_probs), computed now from the retained draws; may be called again with other probabilities."""
        o = SimpleNamespace() if out is None else out
        rk = self.spec.alloc_ranked(o, probs)
        if rk is None:
            raise ValueError("fetch_ranked on a plan without FLAG_RANKED")
        self.ctx._check(self.ctx.L.hmcgpu_plan_fetch_ranked(self.h, C.byref(rk)))
        return o

    def close(self):
        if getattr(self, "h", None):
            self.ctx.L.hmcgpu_plan_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
