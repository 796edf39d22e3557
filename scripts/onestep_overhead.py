"""Cost of HMCGPU_FLAG_ONESTEP (one-step-ahead PIT / log predictive density of every in-sample date, WAIC per window).

Three shapes of bench.py's synthetic series, K = 3, 1000 burn-in + 1000 saved sweeps, horizons 1..12:
  - C2 fp32 and C2 fp64: 500 expanding windows T = 101..600, 256 chains per window (sum_w T_w = 175 250 dates);
  - C1: one window T = 600, one chain (fp32).
Per shape two resident plans, FLAG_SUMMARY and FLAG_SUMMARY | FLAG_ONESTEP, each warmed up once and then run alternately
(--repeats times each).  gpu_ms is the library's own device time of a plan run (CUDA events); the difference is the
accumulation kernel.  fetch_onestep_ms is the host wall time of hmcgpu_plan_fetch_onestep after each one-step run (the finish
kernel plus the copy of the outputs; it synchronises).  A last run under torch.profiler gives the device time of the
accumulation kernel on its own.  Writes one JSON object to --out with the card's name and power limit read in the same process.

    python scripts/onestep_overhead.py --out profiles/onestep_overhead_c2.json
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time
from collections import defaultdict

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (synthetic series and horizons of the C1 / C2 workloads)
import hmc_jl_b200 as H  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm,driver_version"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, power, clock, driver = [v.strip() for v in out.stdout.strip().split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock, driver=driver)


def run_kernel_ms(plan):
    """Device time per kernel name of one plan run (torch.profiler, CUDA activities), top ten."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        plan.run()
        torch.cuda.synchronize()
    tot = defaultdict(float)
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            tot[e.name.split("<")[0].split("(")[0]] += e.device_time_total / 1000.0
    return dict(sorted(((k, round(v, 3)) for k, v in tot.items()), key=lambda kv: -kv[1])[:10])


def measure(ctx, y, ws, we, nc, precision, repeats):
    def spec(flags):
        return H.ProblemSpec(y, ws, we, K=bench.K, n_chains=nc, burnin=1000, nrun=1000, seed=1234, horizons=list(bench.HORIZONS),
                             precision=precision, flags=H.FLAG_REF_Q1 | flags, win_id=np.arange(len(ws)))

    variants = {"summary": H.FLAG_SUMMARY, "summary+onestep": H.FLAG_SUMMARY | H.FLAG_ONESTEP}
    plans = {k: H.Plan(ctx, spec(f)) for k, f in variants.items()}
    info = {}
    for k, p in plans.items():                       # warm-up (module load, pool) of both shapes and of the fetch
        p.run()
        r = H.binding.Result()
        ctx._check(ctx.L.hmcgpu_plan_fetch(p.h, ctypes.byref(r)))
        info[k] = dict(kernel=H.binding.KERNEL_NAMES[r.sweep_kernel], launches=int(r.n_launches))
    plans["summary+onestep"].fetch_onestep()
    runs = []
    for i in range(repeats):
        for k, p in plans.items():
            p.run()
            r = H.binding.Result()                   # timing fields only: no outputs copied
            ctx._check(ctx.L.hmcgpu_plan_fetch(p.h, ctypes.byref(r)))
            row = dict(variant=k, rep=i, gpu_ms=r.gpu_ms, sweep_kernel_ms=r.sweep_kernel_ms)
            if k == "summary+onestep":
                t0 = time.perf_counter()
                o = plans[k].fetch_onestep()
                row["fetch_onestep_ms"] = 1000.0 * (time.perf_counter() - t0)
            runs.append(row)
    med = {k: statistics.median(r["gpu_ms"] for r in runs if r["variant"] == k) for k in variants}
    res = dict(runs=runs, median_gpu_ms=med, launches=info,
               overhead_ms=med["summary+onestep"] - med["summary"],
               overhead_pct=100.0 * (med["summary+onestep"] / med["summary"] - 1.0),
               median_fetch_onestep_ms=statistics.median(r["fetch_onestep_ms"] for r in runs if "fetch_onestep_ms" in r),
               state_bytes=int(5 * 8 * nc * int((np.asarray(we) - np.asarray(ws) + 1).sum())),
               date_draw_pairs=int(nc * 1000 * int((np.asarray(we) - np.asarray(ws) + 1).sum())),
               lpd_finite=bool(np.all(np.isfinite(o.lpd))), waic_elpd_mean=float(np.mean(o.waic[:, 2])),
               kernel_ms=run_kernel_ms(plans["summary+onestep"]))
    for p in plans.values():
        p.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--chains", type=int, default=256)
    args = ap.parse_args()
    import torch
    torch.cuda.init()
    y = bench.synth_series()
    ws, we = H.expanding_windows(101, 600)
    ctx = H.Context(0)
    res = dict(workloads={
        "c2_fp32": "C2: 500 expanding windows T=101..600, K=3, 256 chains x (1000 burn-in + 1000 saved), horizons 1..12, fp32",
        "c2_fp64": "the same C2 job in fp64",
        "c1": "C1: one window T=600, K=3, one chain x (1000 burn-in + 1000 saved), horizons 1..12, fp32"}, **gpu_info())
    res["c2_fp32"] = measure(ctx, y, ws, we, args.chains, 32, args.repeats)
    res["c2_fp64"] = measure(ctx, y, ws, we, args.chains, 64, args.repeats)
    res["c1"] = measure(ctx, y, np.array([1], dtype=np.int32), np.array([600], dtype=np.int32), 1, 32, args.repeats)
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "power_limit": res["power_limit"],
                      **{k: dict(median_gpu_ms=res[k]["median_gpu_ms"], overhead_pct=res[k]["overhead_pct"],
                                 fetch_ms=res[k]["median_fetch_onestep_ms"]) for k in ("c2_fp32", "c2_fp64", "c1")}}))


if __name__ == "__main__":
    main()
