"""Device-time cost of HMCGPU_FLAG_PREDICTIVE (posterior predictive CDF, PIT, log score, moments) on the bench's C2 shape.

C2: 500 expanding windows T = 101..600 of bench.py's synthetic series, 256 chains per window, 1000 burn-in + 1000 saved
sweeps, horizons 1..12, fp32.  Two resident plans, FLAG_SUMMARY and FLAG_SUMMARY | FLAG_PREDICTIVE with a 64-point grid, each
warmed up once and then run alternately (--repeats times each); gpu_ms is the library's own device time of a plan run (CUDA
events).  A last run of each plan under torch.profiler gives the device time per kernel name.  Writes one JSON object to --out
with the card's name and power limit read in the same process.

    python scripts/predictive_overhead.py --out profiles/predictive_overhead_c2.json
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
from collections import defaultdict

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


def kernel_ms(ctx, plan):
    """Device time per kernel name of one plan run (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        plan.run()
        torch.cuda.synchronize()
    tot = defaultdict(float)
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            tot[e.name.split("<")[0].split("(")[0]] += e.device_time_total / 1000.0
    return dict(sorted(((k, round(v, 3)) for k, v in tot.items()), key=lambda kv: -kv[1])[:8])


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--chains", type=int, default=256)
    ap.add_argument("--grid", type=int, default=64)
    args = ap.parse_args()
    y = bench.synth_series()
    ws, we = H.expanding_windows(101, 600)
    nw, nc, K, hz = len(ws), args.chains, bench.K, list(bench.HORIZONS)
    grid = np.linspace(np.min(y) - 3.0, np.max(y) + 3.0, args.grid)
    ctx = H.Context(0)

    def spec(flags):
        return H.ProblemSpec(y, ws, we, K=K, n_chains=nc, burnin=1000, nrun=1000, seed=1234, horizons=hz, precision=32,
                             flags=H.FLAG_REF_Q1 | flags, win_id=np.arange(nw),
                             pred_grid=grid if flags & H.FLAG_PREDICTIVE else None)

    variants = {"summary": H.FLAG_SUMMARY, "summary+predictive": H.FLAG_SUMMARY | H.FLAG_PREDICTIVE}
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
    o = plans["summary+predictive"].fetch()
    med = {k: statistics.median(r["gpu_ms"] for r in runs if r["variant"] == k) for k in variants}
    n_slots = (nw * nc + 31) // 32 * 32
    f0 = 3 * K + K * K
    res = dict(
        workload="C2: 500 expanding windows T=101..600, K=3, 256 chains x (1000 burn-in + 1000 saved), horizons 1..12, fp32",
        n_grid=args.grid, **gpu_info(), runs=runs, median_gpu_ms=med, launches=info,
        overhead_pct=100.0 * (med["summary+predictive"] / med["summary"] - 1.0),
        state_bytes=8 * n_slots * len(hz) * (args.grid + 5),
        predictive=dict(pit_finite=int(np.isfinite(o.pit).sum()), of=int(o.pit.size),
                        mean_vs_summary_max_rel=float(np.nanmax(np.abs(o.pred_moments[:, :, 0] / o.summary_mean[:, f0:f0 + 2 * len(hz):2] - 1))),
                        cdf_min=float(o.pred_cdf.min()), cdf_max=float(o.pred_cdf.max())),
        kernel_ms={k: kernel_ms(ctx, p) for k, p in plans.items()})
    for p in plans.values():
        p.close()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "power_limit", "median_gpu_ms", "overhead_pct", "state_bytes", "kernel_ms")}))


if __name__ == "__main__":
    main()
