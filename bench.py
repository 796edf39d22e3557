#!/usr/bin/env python
"""bench.py — HMM state-steps/sec of the rolling-window Gibbs/FFBS estimation (BASELINE.json metric).

One "step" = one whole estimation pass over the batch: every window x chain runs burnin + nrun Gibbs sweeps
(draws, forward filter, backward sampling, forecasts h=1..12, per-window posterior summaries).
Workload at N=1 = BASELINE.json configs[1] (SURVEY §8d "C2"): one synthetic K=3 series of length 612 (numpy
default_rng(1234)), 500 expanding windows T_w = 101..600, 1000 burn-in + 1000 saved sweeps, 256 chains per window.
N>1 (torchrun, one rank per GPU): end dates are sharded over the ranks (LPT on T_w) and the chains per window scale
with N so per-GPU work is fixed (weak scaling); no data-path collective, only a final gather of per-window summaries.

  value : state-steps / device time of the sweeps with inputs resident in HBM (hmcgpu_plan_run; CUDA events on the
          library's stream, max over ranks).
  e2e   : the same through the public call with HOST buffers (hmcgpu_estimate: H2D of the series, all sweeps, D2H of
          the summaries, device allocation included), wall clock between barriers.
  --impl reference : the CPU oracle (port of the reference's algorithm; Julia is not installed, so the reference's own
          implementation cannot run) on all host threads, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "HMM state-steps/sec (windows x chains x T per Gibbs sweep)"
UNIT = "state-steps/s"
K = 3
TRUTH = dict(A=np.array([[0.96, 0.02, 0.02], [0.02, 0.96, 0.02], [0.02, 0.02, 0.96]]),
             mu=np.array([1.6, 3.5, 8.3]), sigma2=np.array([0.8, 0.55, 7.9]))
HORIZONS = tuple(range(1, 13))


def synth_series(T=612, seed=1234):
    """generateData semantics (src/Hmc.jl:210-229) with numpy's default_rng(1234) (SURVEY §8d)."""
    rng = np.random.default_rng(seed)
    X = np.zeros(T, dtype=np.int64)
    for t in range(1, T):
        X[t] = rng.choice(K, p=TRUTH["A"][X[t - 1]])
    return TRUTH["mu"][X] + np.sqrt(TRUTH["sigma2"][X]) * rng.standard_normal(T)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
                for n, v in zip(names, r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        busy = [s for s, p in zip(sm, power) if p >= 0.5 * max(power)] or sm
        return {"sm_mhz": float(np.median(busy)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(power)),
                "samples": len(sm), "reasons": sorted(reasons)}


def issue_roofline(warp_inst_per_warp_step, state_steps, sweep_seconds, sms, sm_mhz):
    """Warp-instruction issue roofline of the sweep kernel: nominal peak = SMs x 4 schedulers x the SM clock sampled under
    load; next to it the MEASURED rate of a pure-arithmetic kernel with the sweep's instruction blend
    (scripts/issue_peak.cu -> profiles/r1_issue_peak.json: FFMA / MUFU.EX2 / IMAD.WIDE / integer folds), scaled to that clock."""
    ach = warp_inst_per_warp_step * (state_steps / 32.0) / sweep_seconds
    pk = sms * 4 * sm_mhz * 1e6
    out = {"bound": "issue", "achieved": ach / 1e9, "peak": pk / 1e9, "unit": "Gwarp-inst/s", "frac": ach / pk,
           "warp_inst_per_warp_step": warp_inst_per_warp_step, "mufu_per_state_step": 4, "peak_source": "SMs x 4 x sampled SM clock"}
    try:
        m = json.load(open(os.path.join(ROOT, "profiles", "r1_issue_peak.json")))
        mixed = float(m["mix_gwarp_inst_s"]) * 1e9 * (sm_mhz * 1e6 * 4 * int(m["sms"])) / (float(m["nominal_issue_gwarp_inst_s_at_max_clock"]) * 1e9)
        out["measured_mixed_peak"] = mixed / 1e9
        out["frac_of_measured_mixed_peak"] = ach / mixed
    except Exception:
        pass
    return out


# Rank 0 prints ONE JSON line on stdout.  Libraries (NCCL's version banner, ...) write to file descriptor 1 directly, so
# the descriptor is pointed at stderr for the whole run and the line goes to a private duplicate of the real stdout.
_REAL_STDOUT = None


def capture_stdout():
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_line(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, line)


def dist_setup(n_gpus):
    rank, world, local = int(os.environ.get("RANK", 0)), int(os.environ.get("WORLD_SIZE", 1)), int(os.environ.get("LOCAL_RANK", 0))
    dist = None
    if world > 1:
        # (NCCL prints its version banner on stdout from NCCL_DEBUG=VERSION upwards; stdout is redirected, see emit_line)
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    return rank, world, local, dist


def barrier_sync(dist, local):
    import torch
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize(local)


def all_max(dist, local, x):
    if dist is None:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def all_sum(dist, local, x):
    if dist is None:
        return x
    import torch
    t = torch.tensor([x], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


def cpu_baseline(y, ws, we, target_seconds=15.0, threads=0, burnin=1000, nrun=1000):
    """The oracle (kind "port") on all host cores over a bounded sample of the workload: every window with the
    workload's own burn-in + draws, and as many chains per window as fit ~target_seconds (calibrated on a short run)."""
    from oracle import oracle as O
    cores = threads or os.cpu_count() or 1
    T = (we - ws + 1).astype(np.int64)

    def jobs(burn, run, chains):
        out = []
        for c in range(chains):
            for w in range(len(T)):
                e = int(we[w])
                yf = [y[e - 1 + h] if e - 1 + h < len(y) else np.nan for h in HORIZONS]
                out.append(dict(y=y[int(ws[w]) - 1:e], K=K, burnin=burn, nrun=run, seed=1234, chain=w * 4096 + c,
                                horizons=HORIZONS, y_future=yf))
        return out

    t0 = time.perf_counter()
    O.gibbs_batch(jobs(16, 16, 1), n_threads=cores)
    cal = max(time.perf_counter() - t0, 1e-3)
    rate = T.sum() * 32 / cal
    sweeps = burnin + nrun
    chains = int(max(1, min(64, round(target_seconds * rate / (T.sum() * sweeps)))))
    if chains == 1 and T.sum() * sweeps / rate > 2 * target_seconds:     # slow host: fewer sweeps, same mix of windows
        sweeps = int(max(8, target_seconds * rate / T.sum()))
        burnin, nrun = sweeps // 2, sweeps - sweeps // 2
    t0 = time.perf_counter()
    _, used = O.gibbs_batch(jobs(burnin, nrun, chains), n_threads=cores)
    dt = time.perf_counter() - t0
    steps = int(T.sum()) * sweeps * chains
    return {"value": steps / dt, "unit": UNIT, "cores": used, "kind": "port", "chains_per_window": chains, "sweeps": sweeps,
            "sample": f"all {len(T)} windows (T=101..600) x {chains} chain(s), {burnin}+{nrun} sweeps, h=1..12 forecasts; "
                      f"{steps:.3e} state-steps in {dt:.1f}s; fp64 C port of src/Hmc.jl on {used} threads (Julia absent)"}, dt, steps


ALG_SLOTS_PER_STATE_STEP = 65.0     # SURVEY section 8d at K = 3: ~60 FP32/INT issue slots + 5 MUFU per state-step


def headline_profile():
    """profiles/r2_headline_profile.json (written by scripts/profile_headline.sh from an ncu --set full capture of the headline
    kernel): warp-instructions per warp-step and DRAM bytes per state-step of the kernel sources identified by `hot_source_hash`.
    None when the file is missing or was taken from other kernel sources than the ones being run."""
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "r2_headline_profile.json")))
        from hmc_jl_b200 import build as _b
        prof["matches_sources"] = prof.get("hot_source_hash") == _b.hot_source_hash()
        return prof
    except Exception:
        return None


def timed_plan(H, ctx, spec, steps, warmup, dist, local):
    """Device-resident timing of one problem: warm-up runs, then `steps` runs of hmcgpu_plan_run between barriers; device
    time from the library's CUDA events (max over ranks), state-steps summed over ranks."""
    plan = H.Plan(ctx, spec)
    for _ in range(warmup):
        plan.run()
    barrier_sync(dist, local)
    t0 = time.perf_counter()
    acc = dict(dev_ms=0.0, sweep_ms=0.0, launch_ms_sum=0.0, launches=0, sweep_launches=0)
    r = None
    for _ in range(steps):
        plan.run()
        r = H.binding.Result()                      # timing fields only (no output pointers -> no D2H)
        ctx._check(ctx.L.hmcgpu_plan_fetch(plan.h, ctypes.byref(r)))
        acc["dev_ms"] += r.gpu_ms; acc["sweep_ms"] += r.sweep_kernel_ms; acc["launch_ms_sum"] += r.sweep_launch_ms_sum
        acc["launches"] += r.n_launches; acc["sweep_launches"] += r.n_sweep_launches
    barrier_sync(dist, local)
    acc["wall_s"] = time.perf_counter() - t0
    acc["steps_per_run"] = int(r.state_steps)
    acc["kernel"] = int(r.sweep_kernel); acc["n_tasks"] = int(r.n_tasks)
    acc["dev_s"] = all_max(dist, local, acc["dev_ms"] / 1e3)
    acc["total_steps"] = all_sum(dist, local, float(r.state_steps) * steps)
    acc["value"] = acc["total_steps"] / acc["dev_s"]
    acc["plan"] = plan
    return acc


def timed_e2e(H, ctx, spec, steps, shard, n_windows, dist, local, total_steps):
    """The same through the public call with HOST buffers (hmcgpu_estimate: upload, all sweeps, download) plus the final gather
    of the per-window summaries on rank 0; wall clock between barriers, max over ranks."""
    dev = f"cuda:{local}" if dist is not None else None
    o = H.estimate(ctx, spec)                        # warm the allocator path and the gather's lazy NCCL connections once
    H.gather_window_summaries(np.concatenate([o.summary_mean, o.summary_var], axis=1), shard, n_windows, dist, device=dev)
    barrier_sync(dist, local)
    t0 = time.perf_counter()
    h2d = d2h = 0
    t_est = t_gat = 0.0
    for _ in range(steps):
        ta = time.perf_counter()
        o = H.estimate(ctx, spec)
        tb = time.perf_counter()
        h2d += o.h2d_bytes; d2h += o.d2h_bytes
        H.gather_window_summaries(np.concatenate([o.summary_mean, o.summary_var], axis=1), shard, n_windows, dist, device=dev)
        t_est += tb - ta; t_gat += time.perf_counter() - tb
    barrier_sync(dist, local)
    e2e_s = all_max(dist, local, time.perf_counter() - t0)
    return {"value": total_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d // steps, "d2h_bytes_per_step": d2h // steps,
            "ms_per_step": 1e3 * e2e_s / steps, "estimate_ms": 1e3 * t_est / steps, "gather_ms": 1e3 * t_gat / steps, "device_ms": o.gpu_ms}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, res, shard, n_windows, dist=None, device=None, limit=DUMP_LIMIT_BYTES):
    """Writes what the timed path returned in its last step (hmcgpu_plan_fetch: per-window posterior means and variances,
    per-chain status) as <out_dir>/<name>.npy in float64, windows in caller order, so that two builds can be compared output
    for output.  window_index.npy holds the windows written: all of them, or, when that would exceed `limit` bytes, a fixed
    seeded sample.  Every rank calls it (the windows are gathered to rank 0, which writes)."""
    import hmc_jl_b200 as H
    F = res.summary_mean.shape[1]
    rows = np.concatenate([res.summary_mean, res.summary_var, res.status.astype(np.float64)], axis=1)
    full = H.gather_window_summaries(rows, shard, n_windows, dist, device=device)
    if full is None:
        return None
    row_bytes = (full.shape[1] + 1) * 8                      # + the window index
    idx = np.arange(n_windows)
    if n_windows * row_bytes > limit:
        idx = np.sort(np.random.default_rng(1234).choice(n_windows, limit // row_bytes, replace=False))
    arrays = {"summary_mean": full[idx, :F], "summary_var": full[idx, F:2 * F], "status": full[idx, 2 * F:], "window_index": idx}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))
    return sorted(arrays)


def wide_series(n_ser, length, Kw=3, n_gen=2048):
    """C4 / C5 inputs (SURVEY section 8d): independent series from the truth parameters, numpy default_rng(1234); n_gen distinct
    series tiled to n_ser (device work does not depend on the values being distinct)."""
    truth = TRUTH if Kw == 3 else dict(A=np.full((Kw, Kw), 0.1 / (Kw - 1)) + np.eye(Kw) * (0.9 - 0.1 / (Kw - 1)),
                                       mu=2.0 * np.arange(Kw), sigma2=np.full(Kw, 0.5))
    n_gen = min(n_ser, n_gen)
    L = length + 12
    rng = np.random.default_rng(1234)
    X = np.zeros((n_gen, L), dtype=np.int64)
    u = rng.random((n_gen, L))
    cum = np.cumsum(truth["A"], axis=1)
    for t in range(1, L):
        X[:, t] = np.minimum((u[:, t, None] > cum[X[:, t - 1]]).sum(1), Kw - 1)
    y = truth["mu"][X] + np.sqrt(truth["sigma2"][X]) * rng.standard_normal((n_gen, L))
    return np.tile(y, ((n_ser + n_gen - 1) // n_gen, 1))[:n_ser]


def run_reference(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return
    y = synth_series()
    ws = np.ones(500, dtype=np.int32); we = np.arange(101, 601, dtype=np.int32)
    per = []
    base = None
    target = max(3.0, min(20.0, 120.0 / max(1, args.steps + args.warmup)))
    for i in range(args.warmup + args.steps):
        b, dt, steps = cpu_baseline(y, ws, we, target_seconds=target, burnin=args.burnin, nrun=args.nrun)
        if i >= args.warmup:
            per.append((dt, steps))
            base = b
    dt = sum(p[0] for p in per); steps = sum(p[1] for p in per)
    v = steps / dt
    base["value"] = v
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * dt / len(per), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, 1) | {"chains_per_window": base["chains_per_window"], "sharding": "none (host threads over windows x chains)",
                                                  "note": "reference arm = CPU port of the reference on host cores (Julia is not installed, so "
                                                          "the reference itself cannot run); a bounded sample of the workload: every window, "
                                                          "the workload's sweeps, as many chains per window as fit the time budget — the "
                                                          "metric is a rate, so it does not depend on the number of chains"},
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    emit_line(line)


def workload_config(args, world):
    if getattr(args, "workload", "c2") != "c2":
        return {"workload": {"c1": "C1: one window T=600, K=3, one chain (latency-bound by construction)",
                             "c4": "C4: independent series of T=2000, K=3, one chain each (wide batch)",
                             "c5": f"C5: independent series of T={args.length}, K={args.states}, one chain each",
                             "sig": "S1 noisy-signal Monte Carlo (estimatesignals!, src/Hmc.jl:868-914): 64 end dates x 100 perturbed "
                                    "copies, 12 signals after each end date (kappa = 1), smoothed state probabilities at the end date"}[args.workload],
                "K": getattr(args, "K_run", K), "chains": getattr(args, "chains_run", args.chains), "burnin": args.burnin, "nrun": args.nrun,
                "precision": f"fp{args.precision}", "l2": "pif spill working set exceeds the 126 MB L2; no flush needed"}
    return {"workload": "C2 rolling estimation: 500 expanding windows T=101..600 of one synthetic K=3 series (len 612, "
                        "default_rng(1234)), burnin+nrun Gibbs sweeps, forecasts h=1..12, per-window posterior summaries",
            "K": K, "windows": 500, "chains_per_window": args.chains * world, "burnin": args.burnin, "nrun": args.nrun,
            "precision": f"fp{args.precision}", "sharding": f"end dates over {world} rank(s) (LPT on T_w), no collective",
            "l2": "pif spill working set (sum_T*chains*12 B per rank) exceeds the 126 MB L2; no flush needed"}


def main():
    def count(least):
        def parse(s):
            v = int(s)
            if v < least:
                raise argparse.ArgumentTypeError(f"must be at least {least}")
            return v
        return parse

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=count(1), default=5, help="timed steps")
    ap.add_argument("--warmup", type=count(0), default=3)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what their last step computed as DIR/<name>.npy")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--chains", type=int, default=256, help="chains per window per GPU")
    ap.add_argument("--states", type=int, default=3, help="K for --workload c5 (K=3: SURVEY truth; otherwise mu_k=2k, sigma2=0.5)")
    ap.add_argument("--length", type=int, default=2000, help="T for --workload c4/c5")
    ap.add_argument("--workload", default="c2", choices=["c2", "c1", "c4", "c5", "sig"],
                    help="c2 (default, BASELINE configs[1]): 500 expanding windows; c1: one window T=600, one chain; "
                         "c4: --chains independent series (default 65536) of T=2000, K=3")
    ap.add_argument("--burnin", type=int, default=1000)
    ap.add_argument("--nrun", type=int, default=1000)
    ap.add_argument("--precision", type=int, default=32, choices=[32, 64])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-records", action="store_true", help="skip the mid-width / fp64 / C4 sub-records of the N=1 line")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    capture_stdout()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import hmc_jl_b200 as H
    rank, world, local, dist = dist_setup(args.gpus)
    torch.cuda.set_device(local)
    torch.zeros(1, device=f"cuda:{local}")          # create the primary context torch.cuda.synchronize() needs

    win_series = None
    sig_kw = {}
    if args.workload == "c2":
        y = synth_series()
        ws_all, we_all = H.expanding_windows(101, 600)
        n_chains = args.chains * world              # weak scaling: per-GPU work fixed
    elif args.workload == "c1":
        y = synth_series()
        ws_all, we_all = np.array([1], dtype=np.int32), np.array([600], dtype=np.int32)
        n_chains = 1
    elif args.workload == "sig":                    # SURVEY section 8f-2: signals_official_noise_* runs, many end dates per call
        y0 = synth_series()
        n_dates, n_copies, sig_len = 64, 100, 12
        ends = np.arange(600 - n_dates + 1 - sig_len, 600 - sig_len + 1)           # end dates; the window runs to end + 12
        rng = np.random.default_rng(1234)
        n_ser = n_dates * n_copies * world
        y = np.tile(y0, (n_ser + 1, 1))                                             # series 0 = the real data
        mask = np.zeros((n_ser + 1, len(y0)), dtype=np.uint8)
        we_all = np.tile(np.repeat(ends + sig_len, n_copies), world).astype(np.int32)
        for i in range(n_ser):
            e = we_all[i] - sig_len
            y[i + 1, e:e + sig_len] += rng.standard_normal(sig_len) * 0.8
            mask[i + 1, e:e + sig_len] = 1
        ws_all = np.ones(n_ser, dtype=np.int32)
        win_series = np.arange(1, n_ser + 1, dtype=np.int32)
        n_chains = args.chains if args.chains != 256 else 4
        sig_kw = dict(is_signal=mask, kappa=1.0, alpha=np.full(K, 2.0), nu=np.full(K, 2.0), pi_row_back=sig_len)
    else:                                           # c4 / c5: wide batch of independent series (SURVEY section 8d)
        Kw = args.states if args.workload == "c5" else 3
        n_ser = (args.chains if args.chains != 256 else 65536) * world
        y = wide_series(n_ser, args.length, Kw)
        ws_all, we_all = np.ones(n_ser, dtype=np.int32), np.full(n_ser, args.length, dtype=np.int32)
        win_series = np.arange(n_ser, dtype=np.int32)
        n_chains = 1
        args.K_run = Kw
    args.chains_run = int(len(ws_all) * n_chains)      # chains in the whole job
    Krun = getattr(args, "K_run", K)
    shard = H.shard_windows(we_all - ws_all + 1, world)[rank]
    ws, we = ws_all[shard], we_all[shard]

    def make_spec(chains, precision=args.precision, flags=H.FLAG_REF_Q1 | H.FLAG_SUMMARY):
        return H.ProblemSpec(y, ws, we, K=Krun, n_chains=chains, burnin=args.burnin, nrun=args.nrun, seed=1234, horizons=HORIZONS,
                             precision=precision, flags=flags, win_id=shard,
                             win_series=None if win_series is None else win_series[shard],
                             win_init_series=np.zeros(len(shard), dtype=np.int32) if sig_kw else None, **sig_kw)

    spec = make_spec(n_chains)
    ctx = H.Context(local)
    sampler = ClockSampler(local)
    sampler.start()
    m = timed_plan(H, ctx, spec, args.steps, args.warmup, dist, local)
    clocks = sampler.stop()
    plan = m.pop("plan")
    res = plan.fetch()
    plan.close()
    if args.dump_outputs:
        names = dump_outputs(args.dump_outputs, res, shard, len(we_all), dist, device=f"cuda:{local}" if dist is not None else None)
        if names:
            print(f"[bench] wrote {', '.join(names)} to {args.dump_outputs}", file=sys.stderr, flush=True)
    value, dev_s, total_steps, steps_per_run = m["value"], m["dev_s"], m["total_steps"], m["steps_per_run"]
    sweep_ms, dev_ms, sweep_launches = m["sweep_ms"], m["dev_ms"], m["sweep_launches"]
    kernel_name = H.binding.KERNEL_NAMES.get(m["kernel"], str(m["kernel"]))

    # ---- end to end through the public call with host buffers
    e2e = timed_e2e(H, ctx, spec, args.steps, shard, len(we_all), dist, local, total_steps)
    print(f"[bench rank {rank}] e2e per step: estimate {e2e['estimate_ms']:.1f} ms (device {e2e['device_ms']:.1f} ms), "
          f"gather {e2e['gather_ms']:.1f} ms", file=sys.stderr, flush=True)

    # ---- rooflines of the dominant kernel.  north_star: "the slower of HBM traffic and FP32/MUFU issue".  The sweep kernel is
    # bound by instruction issue, so `roofline` is the issue roofline; the HBM fractions (algorithmic bytes, and the DRAM bytes ncu
    # counted) stand beside it.  Instructions per warp-step and DRAM bytes per state-step come from the ncu capture recorded in
    # profiles/r2_headline_profile.json; they are only used when that capture was taken from the kernel sources being run.
    bpe = 4 if args.precision == 32 else 8
    alg_bytes_per_step = (2 * Krun + 2) * bpe
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "MEASURED_PEAKS.json (measured copy)" if peaks else "fallback 6650 (B200_PROFILING.md)"
    sweep_s = sweep_ms / 1e3
    rate = float(steps_per_run) * args.steps / sweep_s          # state-steps/s of this rank inside the sweeps
    hbm_alg = {"achieved": alg_bytes_per_step * rate / 1e9, "peak": peak, "unit": "GB/s", "frac": alg_bytes_per_step * rate / 1e9 / peak,
               "bytes_per_state_step": alg_bytes_per_step, "peak_source": peak_src}
    prof = headline_profile() if (args.workload == "c2" and args.precision == 32 and m["kernel"] == 0) else None
    usable = bool(prof and prof.get("matches_sources"))
    hbm_dram = None
    traffic = None
    if usable:
        bps = float(prof["dram_bytes_per_state_step"])
        hbm_dram = {"achieved": bps * rate / 1e9, "peak": peak, "unit": "GB/s", "frac": bps * rate / 1e9 / peak, "bytes_per_state_step": bps,
                    "source": prof.get("source")}
        traffic = bps * float(steps_per_run) * args.steps / max(1, sweep_launches)      # DRAM bytes per sweep-kernel launch
    common = {"kernel": kernel_name, "launches_timed": sweep_launches, "avg_launch_ms": m["launch_ms_sum"] / max(1, sweep_launches),
              "sweep_kernel_share_of_step": sweep_ms / dev_ms, "traffic": traffic, "hbm_algorithmic": hbm_alg, "hbm_dram": hbm_dram,
              "profile": None if prof is None else {k: prof.get(k) for k in ("source", "hot_source_hash", "matches_sources")},
              "note": "launches of the task groups overlap on separate streams: `achieved` uses the enclosing device time of all sweep "
                      "launches, avg_launch_ms is each launch's own event pair; traffic = ncu DRAM bytes per state-step x the "
                      "state-steps of an average launch"}
    if usable and clocks.get("sm_mhz"):
        sms = torch.cuda.get_device_properties(local).multi_processor_count
        iss = issue_roofline(float(prof["warp_inst_per_warp_step"]), float(steps_per_run) * args.steps, sweep_s, sms, clocks["sm_mhz"])
        iss["algorithmic_frac"] = ALG_SLOTS_PER_STATE_STEP * (rate / 32.0) / (iss["peak"] * 1e9)
        iss["algorithmic_slots_per_state_step"] = ALG_SLOTS_PER_STATE_STEP
        roofline = iss | common
    else:
        # no ncu capture of these kernel sources (or another kernel / workload): only the algorithmic HBM roofline is known
        roofline = {"bound": "hbm", "achieved": hbm_alg["achieved"], "peak": peak, "unit": "GB/s", "frac": hbm_alg["frac"]} | common

    extra = {}
    if args.workload == "c2":
        # ---- strong scaling: the FIXED job (500 end dates x args.chains chains) sharded over the ranks by end date, next to the
        # weak-scaling headline (per-GPU work fixed).  Efficiency against the whole job on ONE GPU (rank 0) in the same run.
        if world > 1:
            sspec = make_spec(args.chains)
            sm_ = timed_plan(H, ctx, sspec, args.steps, 1, dist, local)
            sm_.pop("plan").close()
            se2e = timed_e2e(H, ctx, sspec, args.steps, shard, len(we_all), dist, local, sm_["total_steps"])
            one = None
            if rank == 0:
                full = H.ProblemSpec(y, ws_all, we_all, K=K, n_chains=args.chains, burnin=args.burnin, nrun=args.nrun, seed=1234, horizons=HORIZONS,
                                     precision=args.precision, flags=H.FLAG_REF_Q1 | H.FLAG_SUMMARY)
                one = timed_plan(H, ctx, full, 2, 1, None, local)
                one.pop("plan").close()
            barrier_sync(dist, local)
            n1 = all_max(dist, local, one["value"] if one else 0.0)
            extra["strong"] = {"workload": f"the fixed job: 500 end dates x {args.chains} chains, end dates sharded over {world} ranks",
                               "value": sm_["value"], "unit": UNIT, "ms_per_step": 1e3 * sm_["dev_s"] / args.steps,
                               "e2e": se2e["value"], "e2e_ms_per_step": se2e["ms_per_step"], "kernel": H.binding.KERNEL_NAMES.get(sm_["kernel"]),
                               "warp_tasks_per_gpu": sm_["n_tasks"], "one_gpu_same_run": n1, "efficiency": sm_["value"] / (world * n1) if n1 else None}
        else:
            extra["strong"] = {"workload": f"the fixed job: 500 end dates x {args.chains} chains on one rank", "value": value, "unit": UNIT,
                               "e2e": e2e["value"], "efficiency": 1.0}
    literal = None
    if args.workload == "c2" and world == 1:
        # ---- the reference's own shape of the same job (BASELINE configs[1] read literally): ONE chain per end date (time-parallel
        # kernel), and the mid-width shapes in between: one GPU's share of the fixed job at 8 / 4 / 2 GPUs
        spec1 = H.ProblemSpec(y, ws, we, K=K, n_chains=1, burnin=args.burnin, nrun=args.nrun, seed=1234, horizons=HORIZONS,
                              precision=args.precision, flags=H.FLAG_REF_Q1 | H.FLAG_SUMMARY)
        H.estimate(ctx, spec1)
        t0 = time.perf_counter()
        for _ in range(3):
            o1 = H.estimate(ctx, spec1)
        dt1 = (time.perf_counter() - t0) / 3
        literal = {"workload": "500 end dates x ONE chain (the reference's configuration), same sweeps and outputs",
                   "value": float(o1.state_steps) / dt1, "unit": UNIT, "ms_per_pass_e2e": 1e3 * dt1, "device_ms": o1.gpu_ms,
                   "kernel": H.binding.KERNEL_NAMES.get(o1.sweep_kernel)}
        if not args.no_side_records:
            widths = []
            for c in (32, 64, 128):
                if c >= args.chains:
                    continue
                wm = timed_plan(H, ctx, make_spec(c), 2, 1, None, local)
                wm.pop("plan").close()
                widths.append({"chains_per_window": c, "chains": 500 * c, "value": wm["value"], "ms_per_step": 1e3 * wm["dev_s"] / 2,
                               "kernel": H.binding.KERNEL_NAMES.get(wm["kernel"]), "warp_tasks": wm["n_tasks"]})
            extra["mid_width"] = widths
            # ---- the reference computes in fp64 throughout (src/Hmc.jl:231 ff.): the same job in fp64
            if args.precision == 32:
                s64 = make_spec(n_chains, precision=64)
                m64 = timed_plan(H, ctx, s64, 2, 1, None, local)
                m64.pop("plan").close()
                e64 = timed_e2e(H, ctx, s64, 2, shard, len(we_all), None, local, m64["total_steps"])
                a64 = (2 * K + 2) * 8 * (m64["steps_per_run"] * 2 / (m64["sweep_ms"] / 1e3)) / 1e9
                extra["fp64"] = {"workload": "the same C2 job, every array and operation in fp64", "dtype": "f64", "value": m64["value"], "unit": UNIT,
                                 "ms_per_step": 1e3 * m64["dev_s"] / 2, "e2e": e64["value"],
                                 "roofline": {"bound": "hbm", "achieved": a64, "peak": peak, "unit": "GB/s", "frac": a64 / peak,
                                              "bytes_per_state_step": (2 * K + 2) * 8, "traffic": None}}
            # ---- C4 (BASELINE configs[3]): 65 536 independent series of T = 2000, K = 3, 10 + 100 sweeps, fp32 and fp64
            yc4 = wide_series(65536, 2000)
            # e2e: the 1 GB of series in PAGE-LOCKED host memory (the bench contract's host side; the library then copies it with
            # one DMA), e2e_pageable: the same from an ordinary numpy array (the library stages it through its own pinned buffers)
            try:
                yc4_pinned = torch.from_numpy(yc4).pin_memory().numpy()
            except Exception as exc:                   # (a host that refuses to page-lock 1 GB: both records then come from pageable memory)
                print(f"[bench] could not page-lock the C4 series ({exc}); e2e = e2e_pageable", file=sys.stderr, flush=True)
                yc4_pinned = yc4
            c4 = {}
            for prec in (32, 64):
                mk = lambda ysrc: H.ProblemSpec(ysrc, np.ones(65536, dtype=np.int32), np.full(65536, 2000, dtype=np.int32), K=3, n_chains=1,
                                                burnin=10, nrun=100, seed=1234, horizons=HORIZONS, precision=prec,
                                                flags=H.FLAG_REF_Q1 | H.FLAG_SUMMARY, win_series=np.arange(65536, dtype=np.int32))
                sc4 = mk(yc4_pinned)
                mc = timed_plan(H, ctx, sc4, 2, 1, None, local)
                mc.pop("plan").close()
                ec = timed_e2e(H, ctx, sc4, 2, np.arange(65536), 65536, None, local, mc["total_steps"])
                ep = timed_e2e(H, ctx, mk(yc4), 2, np.arange(65536), 65536, None, local, mc["total_steps"])
                ab = 8 * (prec // 8) * (mc["steps_per_run"] * 2 / (mc["sweep_ms"] / 1e3)) / 1e9
                c4[f"fp{prec}"] = {"value": mc["value"], "unit": UNIT, "ms_per_step": 1e3 * mc["dev_s"] / 2, "e2e": ec["value"],
                                   "e2e_pageable": ep["value"],
                                   "h2d_bytes_per_step": ec["h2d_bytes_per_step"], "kernel": H.binding.KERNEL_NAMES.get(mc["kernel"]),
                                   "roofline": {"bound": "hbm", "achieved": ab, "peak": peak, "unit": "GB/s", "frac": ab / peak,
                                                "bytes_per_state_step": 8 * (prec // 8), "traffic": None,
                                                "note": "every chain streams its own series: DRAM bytes = algorithmic bytes"}}
            del yc4, yc4_pinned
            extra["c4"] = {"workload": "C4: 65 536 independent series of T=2000, K=3, one chain each, 10+100 sweeps, h=1..12, summaries"} | c4
    if rank == 0:
        cb = None
        if not args.no_cpu_baseline and world == 1 and args.workload == "c2":
            cb, _, _ = cpu_baseline(y, ws_all, we_all, burnin=args.burnin, nrun=args.nrun)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * dev_s / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32" if args.precision == 32 else "f64", "data": "synthetic", "config": workload_config(args, world),
                "wall_ms_per_step": 1e3 * m["wall_s"] / args.steps, "clocks": clocks,
                "e2e": {k: e2e[k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "ms_per_step")},
                "gpu_launches": int(m["launches"]), "roofline": roofline, "one_chain_per_end_date": literal, "cpu_baseline": cb,
                "check": {"mu_mean_longest_window": res.summary_mean[int(np.argmax(we - ws))][0:Krun].tolist(),
                          "events": int(res.events)}} | extra
        emit_line(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    ctx.close()


if __name__ == "__main__":
    main()
