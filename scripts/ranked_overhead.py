"""Cost of HMCGPU_FLAG_RANKED (exact quantiles, rank-normalised R̂, bulk / tail ESS) on the bench's C2 shape.

C2: 500 expanding windows T = 101..600 of bench.py's synthetic series, 256 chains per window, 1000 burn-in + 1000 saved
sweeps, horizons 1..12 (F = 43 fields), fp32, quantile probabilities (0.05, 0.5, 0.95).  Two resident plans, FLAG_SUMMARY and
FLAG_SUMMARY | FLAG_RANKED, each warmed up once and then run alternately (--repeats times each):
  - gpu_ms: the library's own device time of a plan run (CUDA events); the difference is the retention of the draws;
  - fetch_ranked_ms: host wall time of hmcgpu_plan_fetch_ranked after each ranked run, from the call to its return (it
    synchronises), i.e. the sorts, ranks and split statistics of all 500 x 43 fields plus the copy of the outputs;
  - device memory in use (cudaMemGetInfo) before the plans, with both plans resident, and after a fetch (the context keeps the
    fetch's scratch in its buffer pool, so this is the peak).
A last fetch under torch.profiler gives the device time per kernel name.  Writes one JSON object to --out with the card's name
and power limit read in the same process.

    python scripts/ranked_overhead.py --out profiles/ranked_overhead_c2.json
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

import bench  # noqa: E402  (synthetic series and horizons of the C2 workload)
import hmc_jl_b200 as H  # noqa: E402


def gpu_info():
    q = "name,power.limit,clocks.max.sm,driver_version"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    name, power, clock, driver = [v.strip() for v in out.stdout.strip().split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clock, driver=driver)


def used_bytes():
    import torch
    free, total = torch.cuda.mem_get_info(0)
    return total - free


def fetch_kernel_ms(plan):
    """Device time per kernel name of one hmcgpu_plan_fetch_ranked (torch.profiler, CUDA activities)."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        plan.fetch_ranked()
        torch.cuda.synchronize()
    tot = defaultdict(float)
    for e in prof.events():
        if e.device_type == torch.autograd.DeviceType.CUDA:
            tot[e.name.split("<")[0].split("(")[0]] += e.device_time_total / 1000.0
    return dict(sorted(((k, round(v, 3)) for k, v in tot.items()), key=lambda kv: -kv[1])[:10])


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
    nw, nc, K, hz = len(ws), args.chains, bench.K, list(bench.HORIZONS)
    probs = (0.05, 0.5, 0.95)
    F = 3 * K + K * K + 2 * len(hz) + 1
    mem = dict(before=used_bytes())
    ctx = H.Context(0)

    def spec(flags):
        return H.ProblemSpec(y, ws, we, K=K, n_chains=nc, burnin=1000, nrun=1000, seed=1234, horizons=hz, precision=32,
                             flags=H.FLAG_REF_Q1 | flags, win_id=np.arange(nw),
                             quantile_probs=probs if flags & H.FLAG_RANKED else None)

    variants = {"summary": H.FLAG_SUMMARY, "summary+ranked": H.FLAG_SUMMARY | H.FLAG_RANKED}
    plans = {k: H.Plan(ctx, spec(f)) for k, f in variants.items()}
    mem["plans_resident"] = used_bytes()
    info = {}
    for k, p in plans.items():                       # warm-up (module load, pool) of both shapes and of the fetch
        p.run()
        r = H.binding.Result()
        ctx._check(ctx.L.hmcgpu_plan_fetch(p.h, ctypes.byref(r)))
        info[k] = dict(kernel=H.binding.KERNEL_NAMES[r.sweep_kernel], launches=int(r.n_launches))
    plans["summary+ranked"].fetch_ranked()
    mem["after_fetch"] = used_bytes()
    runs = []
    for i in range(args.repeats):
        for k, p in plans.items():
            p.run()
            r = H.binding.Result()                   # timing fields only: no outputs copied
            ctx._check(ctx.L.hmcgpu_plan_fetch(p.h, ctypes.byref(r)))
            row = dict(variant=k, rep=i, gpu_ms=r.gpu_ms, sweep_kernel_ms=r.sweep_kernel_ms)
            if k == "summary+ranked":
                t0 = time.perf_counter()
                o = p.fetch_ranked()
                row["fetch_ranked_ms"] = 1000.0 * (time.perf_counter() - t0)
            runs.append(row)
    mem["after_fetch"] = max(mem["after_fetch"], used_bytes())
    med = {k: statistics.median(r["gpu_ms"] for r in runs if r["variant"] == k) for k in variants}
    fetch_med = statistics.median(r["fetch_ranked_ms"] for r in runs if "fetch_ranked_ms" in r)
    res = dict(
        workload="C2: 500 expanding windows T=101..600, K=3, 256 chains x (1000 burn-in + 1000 saved), horizons 1..12, fp32, "
                 "quantiles (0.05, 0.5, 0.95)",
        **gpu_info(), runs=runs, median_gpu_ms=med, launches=info,
        retention_overhead_pct=100.0 * (med["summary+ranked"] / med["summary"] - 1.0),
        median_fetch_ranked_ms=fetch_med, fetch_over_run=fetch_med / med["summary+ranked"],
        retained_bytes=nw * F * nc * 1000 * 4,
        device_bytes_in_use=mem, peak_bytes_over_before=max(mem["plans_resident"], mem["after_fetch"]) - mem["before"],
        ranked=dict(rhat_rank_finite=int(np.isfinite(o.rhat_rank).sum()), of=int(o.rhat_rank.size),
                    rhat_rank_max=float(np.nanmax(o.rhat_rank)), ess_bulk_min=float(np.nanmin(o.ess_bulk)),
                    ess_tail_min=float(np.nanmin(o.ess_tail))),
        fetch_kernel_ms=fetch_kernel_ms(plans["summary+ranked"]))
    for p in plans.values():
        p.close()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({k: res[k] for k in ("gpu", "power_limit", "median_gpu_ms", "retention_overhead_pct", "median_fetch_ranked_ms",
                                          "peak_bytes_over_before", "fetch_kernel_ms")}))


if __name__ == "__main__":
    main()
