"""ctypes binding of the CPU oracle (oracle/hmc_oracle.c).

TEST INFRASTRUCTURE ONLY: imported by tests/, __graft_entry__.smoke() and bench.py's CPU-baseline
legs.  The product package (hmc.jl_b200/) must never import this module.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from types import SimpleNamespace

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libhmc_oracle.so")

FLAG_REF_Q1 = 1
FLAG_PIF_FORM = 2
KIND_STATES, KIND_MU, KIND_SIGMA, KIND_RHO, KIND_A = 0, 1, 2, 3, 4

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int64)
_i32p = C.POINTER(C.c_int32)
_u8p = C.POINTER(C.c_uint8)


class _Problem(C.Structure):
    _fields_ = [("y", _dp), ("N", C.c_int32), ("K", C.c_int32), ("is_signal", _u8p),
                ("xi", _dp), ("alpha", _dp), ("nu", _dp), ("beta0", _dp), ("beta", _dp),
                ("kappa", C.c_double), ("X0", _ip), ("burnin", C.c_int64), ("nrun", C.c_int64),
                ("seed", C.c_uint64), ("chain", C.c_uint32), ("flags", C.c_uint32),
                ("horizons", _i32p), ("n_h", C.c_int32), ("y_future", _dp)]


class _Result(C.Structure):
    _fields_ = [("mu", _dp), ("sigma2", _dp), ("A", _dp), ("pi_end", _dp), ("forecasts", _dp),
                ("loglik", _dp), ("pib_mean", _dp), ("pib_full", _dp), ("X_final", _ip),
                ("n_events", C.c_int64), ("state_margin", _dp), ("gamma_margin", _dp)]


def build(force: bool = False) -> str:
    """Compile the oracle with the committed Makefile (gcc, no external deps)."""
    src = os.path.join(_HERE, "hmc_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.run(["make", "-C", _HERE, "-B", "libhmc_oracle.so"], check=True, capture_output=True)
    return _LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        L.orc_u01.restype = C.c_double
        L.orc_u01.argtypes = [C.c_uint32]
        L.orc_gamma.restype = C.c_double
        L.orc_gamma.argtypes = [C.c_double, C.c_uint64, C.c_uint32, C.c_uint32, C.c_uint32]
        L.orc_forward.restype = C.c_int
        L.orc_gibbs.restype = C.c_int
        L.orc_gibbs_batch.restype = C.c_int
        _lib = L
    return _lib


def _d(a):
    return None if a is None else a.ctypes.data_as(_dp)


def _f64(a):
    return None if a is None else np.ascontiguousarray(a, dtype=np.float64)


def philox(ctr, key, rounds=10):
    c = (C.c_uint32 * 4)(*[int(x) & 0xFFFFFFFF for x in ctr])
    k = (C.c_uint32 * 2)(*[int(x) & 0xFFFFFFFF for x in key])
    o = (C.c_uint32 * 4)()
    lib().orc_philox4x32(C.c_int(rounds), c, k, o)
    return [int(x) for x in o]


def gamma(shape, seed, chain, sweep, purpose):
    return float(lib().orc_gamma(float(shape), int(seed), int(chain), int(sweep), int(purpose)))


def make_params(y, K):
    y = _f64(y)
    X = np.zeros(len(y), dtype=np.int64)
    mu0 = np.zeros(K)
    sd0 = C.c_double()
    lib().orc_make_params(_d(y), C.c_int(len(y)), C.c_int(K), X.ctypes.data_as(_ip), _d(mu0), C.byref(sd0))
    return X, mu0, sd0.value


def forward(y, A, mu, sigma2, rho, is_signal=None, kappa=1.0, want_Pf=True):
    y, A, mu, sigma2, rho = map(_f64, (y, A, mu, sigma2, rho))
    N, K = len(y), len(mu)
    Pf = np.zeros((N, K, K)) if want_Pf else None
    pif = np.zeros((N, K))
    totals = np.zeros(N)
    ll = C.c_double()
    sig = None if is_signal is None else np.ascontiguousarray(is_signal, dtype=np.uint8)
    ev = lib().orc_forward(_d(y), C.c_int(N), C.c_int(K),
                           None if sig is None else sig.ctypes.data_as(_u8p), C.c_double(kappa),
                           _d(A), _d(mu), _d(sigma2), _d(rho), _d(Pf), _d(pif), _d(totals), C.byref(ll))
    return SimpleNamespace(Pf=Pf, pif=pif, totals=totals, loglik=ll.value, events=ev)


def backward(Pf, pif):
    N, K = pif.shape
    Pb = np.zeros((N, K, K))
    pib = np.zeros((N, K))
    lib().orc_backward(C.c_int(N), C.c_int(K), _d(_f64(Pf)), _d(_f64(pif)), _d(Pb), _d(pib))
    return Pb, pib


def backward_pif(A, pif):
    N, K = pif.shape
    pib = np.zeros((N, K))
    lib().orc_backward_pif(C.c_int(N), C.c_int(K), _d(_f64(A)), _d(_f64(pif)), _d(pib))
    return pib


def sample_states(pif, A, u, Pf=None, piN=None, form=1):
    pif, A, u = map(_f64, (pif, A, u))
    N, K = pif.shape
    piN = _f64(pif[-1] if piN is None else piN)
    X = np.zeros(N, dtype=np.int64)
    lib().orc_sample_states(C.c_int(N), C.c_int(K), _d(_f64(Pf)), _d(pif), _d(A), _d(piN), _d(u),
                            C.c_int(form), X.ctypes.data_as(_ip))
    return X


def forecast(mu, A, pib, h, yreal):
    mu, A, pib = map(_f64, (mu, A, pib))
    f, e = C.c_double(), C.c_double()
    lib().orc_forecast(C.c_int(len(mu)), _d(mu), _d(A), _d(pib), C.c_int(h), C.c_double(yreal), C.byref(f), C.byref(e))
    return f.value, e.value


def draw_params(Ni, S, S2, trans, xi, alpha, nu, beta, seed, chain, sweep, kappa=1.0, Mi=None, Sm=None, Sm2=None):
    K = len(Ni)
    Ni = np.ascontiguousarray(Ni, dtype=np.int64)
    trans = np.ascontiguousarray(trans, dtype=np.int64)
    Mi_ = None if Mi is None else np.ascontiguousarray(Mi, dtype=np.int64)
    S, S2, xi, alpha, nu, beta, Sm, Sm2 = map(_f64, (S, S2, xi, alpha, nu, beta, Sm, Sm2))
    sigma2, mu, rho, A = np.ones(K), np.zeros(K), np.zeros(K), np.zeros((K, K))
    lib().orc_draw_params(C.c_int(K), Ni.ctypes.data_as(_ip), None if Mi_ is None else Mi_.ctypes.data_as(_ip),
                          _d(S), _d(Sm), _d(S2), _d(Sm2), trans.ctypes.data_as(_ip),
                          _d(xi), _d(alpha), _d(nu), _d(beta), C.c_double(kappa),
                          C.c_uint64(seed), C.c_uint32(chain), C.c_uint32(sweep),
                          _d(sigma2), _d(mu), _d(rho), _d(A))
    return sigma2, mu, rho, A


class _Job:
    """Owns the numpy buffers behind one orc_problem/orc_result pair."""

    def __init__(self, y, K, burnin, nrun, seed=1234, chain=0, flags=FLAG_REF_Q1, horizons=(12,), y_future=None,
                 X0=None, is_signal=None, xi=None, alpha=None, nu=None, beta0=None, beta=None, kappa=1.0,
                 want_pib_mean=False, want_pib_full=False, want_margins=False):
        self.y = _f64(y)
        N = len(self.y)
        self.N, self.K, self.nrun = N, K, nrun
        self.h = np.ascontiguousarray(horizons, dtype=np.int32)
        nh = len(self.h)
        self.yf = _f64(np.full(nh, np.nan) if y_future is None else y_future)
        self.X0 = None if X0 is None else np.ascontiguousarray(X0, dtype=np.int64)
        self.sig = None if is_signal is None else np.ascontiguousarray(is_signal, dtype=np.uint8)
        self.hp = [_f64(v) for v in (xi, alpha, nu, beta0, beta)]
        self.out = SimpleNamespace(
            mu=np.zeros((nrun, K)), sigma2=np.zeros((nrun, K)), A=np.zeros((nrun, K, K)),
            pi_end=np.zeros((nrun, K)), forecasts=np.zeros((nrun, 2 * nh)), loglik=np.zeros(nrun),
            pib_mean=np.zeros((N, K)) if want_pib_mean else None,
            pib_full=np.zeros((nrun, N, K)) if want_pib_full else None,
            X_final=np.zeros(N, dtype=np.int64), n_events=0,
            state_margin=np.zeros(burnin + nrun) if want_margins else None,
            gamma_margin=np.zeros(burnin + nrun) if want_margins else None)
        o = self.out
        self.problem = _Problem(_d(self.y), N, K, None if self.sig is None else self.sig.ctypes.data_as(_u8p),
                                *[_d(v) for v in self.hp], kappa,
                                None if self.X0 is None else self.X0.ctypes.data_as(_ip),
                                burnin, nrun, seed, chain, flags, self.h.ctypes.data_as(_i32p), nh, _d(self.yf))
        self.result = _Result(_d(o.mu), _d(o.sigma2), _d(o.A), _d(o.pi_end), _d(o.forecasts), _d(o.loglik),
                              _d(o.pib_mean), _d(o.pib_full), o.X_final.ctypes.data_as(_ip), 0,
                              _d(o.state_margin), _d(o.gamma_margin))


def gibbs(y, K, burnin, nrun, **kw):
    """One chain of the reference sampler (src/Hmc.jl:517-562 + :850-865). Returns draw-major arrays.
    want_margins=True adds state_margin / gamma_margin, one entry per sweep (burnin included): how close that sweep's
    categorical draws and gamma accept/reject tests came to the other outcome (hmc_oracle.h, orc_result)."""
    job = _Job(y, K, burnin, nrun, **kw)
    rc = lib().orc_gibbs(C.byref(job.problem), C.byref(job.result))
    if rc != 0:
        raise RuntimeError(f"orc_gibbs failed: {rc}")
    job.out.n_events = int(job.result.n_events)
    return job.out


def gibbs_batch(jobs_kwargs, n_threads=0):
    """Run many independent chains on host threads. jobs_kwargs: list of dicts for _Job. Returns (outs, threads)."""
    jobs = [_Job(**kw) for kw in jobs_kwargs]
    n = len(jobs)
    P = (_Problem * n)(*[j.problem for j in jobs])
    R = (_Result * n)(*[j.result for j in jobs])
    used = lib().orc_gibbs_batch(P, R, C.c_int(n), C.c_int(n_threads))
    for j, r in zip(jobs, R):
        j.out.n_events = int(r.n_events)
    return [j.out for j in jobs], int(used)
