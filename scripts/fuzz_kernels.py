"""Differential fuzzing of the sweep kernels on the GPU box: random shapes (K, window lengths, ragged batches, chains,
signal masks, kappa, pi_row_back, user X0) are estimated in fp64 with two kernels that must produce the same chains (same
Philox streams): K = 2..4 time-parallel warp-per-chain vs thread-per-chain; K = 5..8 thread-per-chain vs lane-per-state; K = 2..4 plain sweeps also on the segment kernel
(2 / 4 / 8 lanes per chain, or mixed 8 + 4) vs thread-per-chain.
With --precision 32 the same shapes run in fp32 (burnin 0, 3 draws, one series), and each kernel is checked on its own against
the fp64 oracle chain with the certification of tests/test_fp32_chain_parity.py (fp32 kernels legitimately differ from each
other in the last bits).
python scripts/fuzz_kernels.py [n] [seed] [--precision 32]"""
import os, sys
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import hmc_jl_b200 as H

args = [a for a in sys.argv[1:]]
fp32 = "--precision" in args and args[args.index("--precision") + 1] == "32"
if "--precision" in args:
    i = args.index("--precision")
    if args[i + 1] not in ("32", "64"):
        sys.exit("--precision must be 32 or 64")
    del args[i:i + 2]
n_cases = int(args[0]) if len(args) > 0 else 100
rng = np.random.default_rng(int(args[1]) if len(args) > 1 else 0)
ctx = H.Context(0)
if fp32:
    from oracle import oracle as O
    from test_fp32_chain_parity import KERNELS, check_chains
bad = 0
for case in range(n_cases):
    K = int(rng.integers(2, 9))
    L = int(rng.integers(8, 900))
    mu = np.sort(rng.normal(0, 4, K)); s2 = rng.uniform(0.3, 2.0, K)
    A = rng.dirichlet(np.ones(K) * 0.5, K) * 0.3 + np.eye(K) * 0.7
    X = np.zeros(L + 14, dtype=int)
    for t in range(1, L + 14):
        X[t] = rng.choice(K, p=A[X[t - 1]])
    n_ser = int(rng.integers(1, 3))
    y = np.stack([mu[X] + np.sqrt(s2[X]) * rng.standard_normal(L + 14) for _ in range(n_ser)])
    nw = int(rng.integers(1, 5))
    ws = rng.integers(1, max(2, L // 3), nw)
    we = np.array([int(rng.integers(s + 1, L + 1)) for s in ws])
    kw = dict(K=K, n_chains=int(rng.integers(1, 4)), burnin=int(rng.integers(0, 2)), nrun=int(rng.integers(2, 5)), seed=int(rng.integers(1, 10**6)),
              horizons=tuple(sorted(set(rng.integers(0, 13, 2).tolist()))), precision=64,
              flags=H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_LOGLIK | H.FLAG_SUMMARY, win_series=rng.integers(0, n_ser, nw))
    if K <= 4 and rng.random() < 0.5:                           # signals tier
        per_series = rng.random() < 0.5 and n_ser > 1
        mask = (rng.random((n_ser, L + 14) if per_series else (L + 14,)) < rng.choice([0.02, 0.3, 1.0])).astype(np.uint8)
        kw.update(is_signal=mask, kappa=float(rng.choice([0.0, 0.5, 2.0])), pi_row_back=int(rng.integers(0, min(6, int((we - ws).min()) + 1))),
                  alpha=np.full(K, 2.0), nu=np.full(K, 2.0))
    if rng.random() < 0.3:
        kw.update(X0=[rng.integers(1, K + 1, int(e - s + 1)) for s, e in zip(ws, we)])
    for v in ("HMCGPU_SEG_LANES", "HMCGPU_SEG_LONG", "HMCGPU_SCAN_MAX_CHAINS", "HMCGPU_LANE_KERNEL"):
        os.environ.pop(v, None)
    if fp32:
        kernels = ["scan", "thread"] if K <= 4 else ["thread", "lane"]
        if K <= 4 and "is_signal" not in kw:
            lanes = int(rng.choice([2, 4, 8]))
            if (we - ws + 1).max() <= lanes * (((1 << (32 // K)) - 1) // 4 * 4):       # seg_max_T
                kernels.append(f"seg{lanes}")
        sig = kw.get("is_signal")
        for name in kernels:
            for v in ("HMCGPU_SEG_LANES", "HMCGPU_SEG_LONG", "HMCGPU_SCAN_MAX_CHAINS", "HMCGPU_LANE_KERNEL"):
                os.environ.pop(v, None)
            os.environ.update(KERNELS[name][0])
            try:
                check_chains(H, ctx, O, y[0], ws, we, K, kw["n_chains"], KERNELS[name][1], seed=kw["seed"], hs=kw["horizons"],
                             alpha=kw.get("alpha"), nu=kw.get("nu"), is_signal=None if sig is None else (sig[0] if sig.ndim == 2 else sig),
                             kappa=kw.get("kappa", 1.0), X0=kw.get("X0"), pi_row_back=kw.get("pi_row_back", 0), min_certified=0.0)
            except AssertionError as e:
                bad += 1
                print("MISMATCH case", case, name, dict(K=K, ws=ws.tolist(), we=we.tolist()), str(e)[:500], flush=True)
        continue
    outs = {}
    run = lambda: H.estimate(ctx, H.ProblemSpec(y, ws, we, **kw))
    if K <= 4:
        os.environ["HMCGPU_SCAN_MAX_CHAINS"] = "1000000"
        outs["scan"] = run()
        os.environ["HMCGPU_SCAN_MAX_CHAINS"] = "0"; os.environ["HMCGPU_SEG_LANES"] = "0"
        outs["thread"] = run()
        pairs = [(outs["scan"], outs["thread"])]
        if "is_signal" not in kw:              # plain sweep: the segment kernel with 2 / 4 / 8 lanes per chain, or mixed 8 + 4
            choice = str(rng.choice(["2", "4", "8", "mixed"]))
            if choice == "mixed":
                kw["n_chains"] = int(rng.integers(8, 36))          # (a long class needs at least 32 chains)
                ref = run()                                          # thread-per-chain, the same chains
                os.environ.pop("HMCGPU_SEG_LANES")
                os.environ["HMCGPU_SEG_LONG"] = str(int(rng.integers(1, nw + 1)))
                pairs.append((run(), ref))
            else:
                os.environ["HMCGPU_SEG_LANES"] = choice
                pairs.append((run(), outs["thread"]))
    else:
        os.environ["HMCGPU_LANE_KERNEL"] = "0"
        outs["thread"] = run()
        os.environ["HMCGPU_LANE_KERNEL"] = "1"
        outs["lane"] = run()
        pairs = [(outs["thread"], outs["lane"])]
    ok = True
    for a, b in pairs:
        ok = ok and a.events == b.events
        for k in ("mu", "sigma2", "A", "pi_end", "forecasts", "loglik"):
            for w in range(nw):
                x, z = np.asarray(getattr(a, k)[w]), np.asarray(getattr(b, k)[w])
                fin = np.isfinite(z)
                ok = ok and x.shape == z.shape and np.array_equal(np.isfinite(x), fin) and np.allclose(x[fin], z[fin], rtol=1e-6, atol=1e-9)
    if not ok:
        bad += 1
        print("MISMATCH case", case, dict(K=K, ws=ws.tolist(), we=we.tolist(), **{k: (v if np.isscalar(v) else "...") for k, v in kw.items()}), flush=True)
print(f"{n_cases} cases, {bad} mismatches")
sys.exit(1 if bad else 0)
