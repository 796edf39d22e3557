"""Device-time cost of HMCGPU_FLAG_DIAGNOSTICS (split-R̂ / ESS per window and field) on the bench's C2 shape.

C2: 500 expanding windows T = 101..600 of bench.py's synthetic series, 256 chains per window, 1000 burn-in + 1000 saved
sweeps, horizons 1..12, fp32.  Two resident plans, FLAG_SUMMARY and FLAG_SUMMARY | FLAG_DIAGNOSTICS, each warmed up once and
then run alternately (--repeats times each); gpu_ms is the library's own device time of a plan run (CUDA events).  Writes one
JSON object to --out with the card's name and power limit read in the same process.

    python scripts/diag_overhead.py --out profiles/diag_overhead_c2.json
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (synthetic series and horizons of the C2 workload)
import hmc_jl_b200 as H  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm,driver_version"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, power, clock, driver = [v.strip() for v in out.stdout.strip().split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock, driver=driver)


def state_bytes(n_slots, n_windows, n_chains, F, precision):
    """Device memory of the diagnostics: per (slot, field) 64 fp64 lag sums, S1, 64 head and 64 ring values of the draw type;
    per (window, field) the 2 n_chains sequence means and variances and 64 fp64 lag sums (diagnostics.cuh)."""
    per_sf = 64 * 8 + 8 + 2 * 64 * (precision // 8)
    return dict(per_slot_field=per_sf, streaming=n_slots * F * per_sf,
                per_window=n_windows * F * (2 * n_chains * 2 * 8 + 64 * 8))


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--chains", type=int, default=256)
    args = ap.parse_args()
    y = bench.synth_series()
    ws, we = H.expanding_windows(101, 600)
    nw, nc, K, hz = len(ws), args.chains, bench.K, list(bench.HORIZONS)
    F = 3 * K + K * K + 2 * len(hz) + 1
    ctx = H.Context(0)

    def spec(flags):
        return H.ProblemSpec(y, ws, we, K=K, n_chains=nc, burnin=1000, nrun=1000, seed=1234, horizons=hz, precision=32,
                             flags=H.FLAG_REF_Q1 | flags, win_id=np.arange(nw))

    variants = {"summary": H.FLAG_SUMMARY, "summary+diagnostics": H.FLAG_SUMMARY | H.FLAG_DIAGNOSTICS}
    plans = {k: H.Plan(ctx, spec(f)) for k, f in variants.items()}
    info = {}
    for k, p in plans.items():                       # warm-up (module load, pool) of both shapes
        p.run()
        r = H.binding.Result()
        ctx._check(ctx.L.hmcgpu_plan_fetch(p.h, ctypes.byref(r)))
        info[k] = dict(kernel=H.binding.KERNEL_NAMES[r.sweep_kernel], launches=int(r.n_launches))
    runs = []
    for i in range(args.repeats):
        for k, p in plans.items():
            p.run()
            r = H.binding.Result()                   # timing fields only: no outputs copied
            ctx._check(ctx.L.hmcgpu_plan_fetch(p.h, ctypes.byref(r)))
            runs.append(dict(variant=k, rep=i, gpu_ms=r.gpu_ms, sweep_kernel_ms=r.sweep_kernel_ms))
    o = plans["summary+diagnostics"].fetch()
    med = {k: statistics.median(r["gpu_ms"] for r in runs if r["variant"] == k) for k in variants}
    n_slots = (nw * nc + 31) // 32 * 32
    fin = np.isfinite(o.rhat)
    res = dict(
        workload="C2: 500 expanding windows T=101..600, K=3, 256 chains x (1000 burn-in + 1000 saved), horizons 1..12, fp32",
        **gpu_info(), runs=runs, median_gpu_ms=med, launches=info,
        overhead_pct=100.0 * (med["summary+diagnostics"] / med["summary"] - 1.0),
        state_bytes=state_bytes(n_slots, nw, nc, F, 32),
        diagnostics=dict(finite_fields=int(fin.sum()), of=int(fin.size), rhat_max=float(o.rhat[fin].max()),
                         rhat_median=float(np.median(o.rhat[fin])), ess_min=float(o.ess[fin].min()),
                         ess_median=float(np.median(o.ess[fin])), ess_lag_at_cap=int((o.ess_lag == 63).sum())))
    for p in plans.values():
        p.close()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "power_limit", "median_gpu_ms", "overhead_pct", "state_bytes")}))


if __name__ == "__main__":
    main()
