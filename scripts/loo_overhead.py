"""Cost of HMCGPU_FLAG_LOO (PSIS-LOO of every in-sample date: leave-one-out density, Pareto k̂, LOO-PIT).

Shapes of bench.py's synthetic series, K = 3, 1000 burn-in + 1000 saved sweeps, horizons 1..12:
  - C2 fp32 and C2 fp64: 500 expanding windows T = 101..600, 256 chains per window (sum_w T_w = 175 250 dates);
  - C2 x 32 chains (fp32);
  - C1: one window T = 600, one chain (fp32).
Per shape two resident plans, FLAG_SUMMARY and FLAG_SUMMARY | FLAG_LOO, each warmed up once and then run alternately
(--repeats times each).  gpu_ms is the library's own device time of a plan run (CUDA events); the difference is the retention
of the mu / sigma2 / A draws.  fetch_loo_ms is the host wall time of one hmcgpu_plan_fetch_loo (it ends in a stream
synchronise), and a second fetch under torch.profiler splits it by kernel.  Writes one JSON object to --out with the card's
name and power limit read in the same process.

    python scripts/loo_overhead.py --out profiles/loo_overhead_c2.json
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


def kernel_ms(fn):
    """Device time per kernel name of fn() (torch.profiler, CUDA activities), top ten."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
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

    variants = {"summary": H.FLAG_SUMMARY, "summary+loo": H.FLAG_SUMMARY | H.FLAG_LOO}
    plans = {k: H.Plan(ctx, spec(f)) for k, f in variants.items()}
    info = {}
    for k, p in plans.items():                       # warm-up (module load, pool) of both shapes
        p.run()
        r = H.binding.Result()
        ctx._check(ctx.L.hmcgpu_plan_fetch(p.h, ctypes.byref(r)))
        info[k] = dict(kernel=H.binding.KERNEL_NAMES[r.sweep_kernel], launches=int(r.n_launches))
    runs = []
    for i in range(repeats):
        for k, p in plans.items():
            p.run()
            r = H.binding.Result()                   # timing fields only: no outputs copied
            ctx._check(ctx.L.hmcgpu_plan_fetch(p.h, ctypes.byref(r)))
            runs.append(dict(variant=k, rep=i, gpu_ms=r.gpu_ms, sweep_kernel_ms=r.sweep_kernel_ms))
    t0 = time.perf_counter()
    o = plans["summary+loo"].fetch_loo()
    fetch_ms = 1000.0 * (time.perf_counter() - t0)
    med = {k: statistics.median(r["gpu_ms"] for r in runs if r["variant"] == k) for k in variants}
    dates = int((np.asarray(we) - np.asarray(ws) + 1).sum())
    R = nc * 1000
    res = dict(runs=runs, median_gpu_ms=med, launches=info,
               overhead_ms=med["summary+loo"] - med["summary"],
               overhead_pct=100.0 * (med["summary+loo"] / med["summary"] - 1.0),
               fetch_loo_ms=fetch_ms,
               kept_bytes=int(len(ws) * (2 * bench.K + bench.K ** 2) * R * precision // 8),
               date_draw_pairs=int(R * dates),
               scratch_bytes_moved=int(R * dates * (16 + bench.K * precision // 8)),
               elpd_finite=bool(np.all(np.isfinite(o.loo_elpd))), elpd_loo_mean=float(np.mean(o.loo[:, 0])),
               max_k=float(np.max(o.loo[:, 4])), dates_high_k=int(np.sum(o.loo[:, 5])),
               fetch_kernel_ms=kernel_ms(plans["summary+loo"].fetch_loo))
    for p in plans.values():
        p.close()
    return res


def main():
    ap = argparse.ArgumentParser(description=__doc__.splitlines()[0])
    ap.add_argument("--out", required=True)
    ap.add_argument("--repeats", type=int, default=3)
    args = ap.parse_args()
    import torch
    torch.cuda.init()
    y = bench.synth_series()
    ws, we = H.expanding_windows(101, 600)
    ctx = H.Context(0)
    res = dict(workloads={
        "c2_fp32": "C2: 500 expanding windows T=101..600, K=3, 256 chains x (1000 burn-in + 1000 saved), horizons 1..12, fp32",
        "c2_fp64": "the same C2 job in fp64",
        "c2_32chains": "the C2 windows with 32 chains per window, fp32",
        "c1": "C1: one window T=600, K=3, one chain x (1000 burn-in + 1000 saved), horizons 1..12, fp32"}, **gpu_info())
    res["c2_fp32"] = measure(ctx, y, ws, we, 256, 32, args.repeats)
    res["c2_fp64"] = measure(ctx, y, ws, we, 256, 64, args.repeats)
    res["c2_32chains"] = measure(ctx, y, ws, we, 32, 32, args.repeats)
    res["c1"] = measure(ctx, y, np.array([1], dtype=np.int32), np.array([600], dtype=np.int32), 1, 32, args.repeats)
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "power_limit": res["power_limit"],
                      **{k: dict(median_gpu_ms=res[k]["median_gpu_ms"], overhead_pct=res[k]["overhead_pct"],
                                 fetch_ms=res[k]["fetch_loo_ms"], fetch_kernel_ms=res[k]["fetch_kernel_ms"])
                         for k in ("c2_fp32", "c2_fp64", "c2_32chains", "c1")}}))


if __name__ == "__main__":
    main()
