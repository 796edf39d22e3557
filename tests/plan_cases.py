"""The problems of the sweep-kernel choice table and what a B200 (148 SMs) plans for them: the kernel, the warp tasks it is
laid out in, and how the sweeps are cut into launches over the task groups.  test_plan_choice.py runs each problem on the GPU,
test_plan_policy.py computes the plan on the CPU."""

BURNIN, NRUN = 24, 24           # sweeps of every problem

# cleared before each problem; a problem sets its own
TUNING = ("HMCGPU_LANE_KERNEL", "HMCGPU_SCAN_MAX_CHAINS", "HMCGPU_SEG_LANES", "HMCGPU_SEG_MIXED", "HMCGPU_SEG_LONG",
          "HMCGPU_GROUPS", "HMCGPU_Y_SMEM", "HMCGPU_SEG_WARMUP", "HMCGPU_SEG_BARRIERS", "HMCGPU_SEG_THREADS",
          "HMCGPU_SWEEPS_PER_LAUNCH", "HMCGPU_LAUNCH_TIMING", "HMCGPU_VERBOSE")

MIXED_T = list(range(249, 149, -1))     # 100 windows of 150..249 steps: the longest tenth qualifies for 8 lanes per chain

# name -> (problem, environment).  Problem: nw windows x nc chains of length T (or the list of lengths), K states, on one
# series unless nser > 1 (windows alternate between the series); sig: every observation a noisy signal.
CASES = {
    # warp per chain up to 4096 chains (the plain sweep) ...
    "scan": (dict(nw=10, nc=16), {}),
    "scan_fp64": (dict(nw=10, nc=16, precision=64), {}),
    "scan_4096": (dict(nw=64, nc=64), {}),
    "scan_4160": (dict(nw=65, nc=64), {}),
    # ... scaled down when the window leaves room for fewer resident blocks (two here: bound 1638 chains) ...
    "scan_long_1500": (dict(nw=1, nc=1500, T=1560), {}),
    "scan_long_2000": (dict(nw=1, nc=2000, T=1560), {}),
    # ... and never past scan_max_T (3196 steps for fp32, K = 3)
    "scan_too_long": (dict(nw=1, nc=32, T=3300), {}),
    # the signals tier has no segment kernel: warp per chain up to 12 288 chains, then a thread per chain
    "sig_scan": (dict(nw=100, nc=120, sig=True), {}),
    "sig_thread": (dict(nw=100, nc=130, sig=True), {}),
    # segment kernel: 4 lanes per chain up to half a wave of thread slots, 2 lanes up to 5/4 of a wave on one shared series
    "seg4": (dict(nw=100, nc=64), {}),
    "seg2": (dict(nw=200, nc=256), {}),
    "seg2_distinct_series": (dict(nw=200, nc=256, nser=2), {}),
    "thread_wide": (dict(nw=400, nc=256), {}),
    "seg4_too_long": (dict(nw=100, nc=64, K=4, T=1100), {}),
    # the mixed long class (8 lanes for the longest tenth of the windows) and what turns it off
    "seg4_mixed": (dict(nw=100, nc=64, T=MIXED_T), {}),
    "seg4_mixed_off": (dict(nw=100, nc=64, T=MIXED_T), {"HMCGPU_SEG_MIXED": "0"}),
    "seg4_lanes_set": (dict(nw=100, nc=64, T=MIXED_T), {"HMCGPU_SEG_LANES": "4"}),
    "seg4_long_20": (dict(nw=100, nc=64, T=MIXED_T), {"HMCGPU_SEG_LONG": "20"}),
    # HMCGPU_SEG_LANES=0: no segment kernel, so the warp-per-chain kernel keeps the batch up to 12 288 chains
    "seg_lanes_0": (dict(nw=100, nc=64), {"HMCGPU_SEG_LANES": "0"}),
    # per-date means: thread per chain at any width
    "smoothed": (dict(nw=10, nc=16, smoothed=True), {}),
    "filtered": (dict(nw=10, nc=16, filtered=True), {}),
    # K = 5..8: thread per chain unless HMCGPU_LANE_KERNEL=1; K >= 9: lane per state
    "k6": (dict(nw=10, nc=16, K=6), {}),
    "k6_lane": (dict(nw=10, nc=16, K=6), {"HMCGPU_LANE_KERNEL": "1"}),
    "k12": (dict(nw=10, nc=16, K=12), {}),
    # task groups and launch length
    "groups_3": (dict(nw=100, nc=64), {"HMCGPU_GROUPS": "3"}),
    "sweeps_5": (dict(nw=100, nc=64), {"HMCGPU_SWEEPS_PER_LAUNCH": "5"}),
    "scan_sweeps_8": (dict(nw=10, nc=16), {"HMCGPU_SWEEPS_PER_LAUNCH": "8"}),
}

# (sweep_kernel, n_tasks, n_sweep_launches, n_launches)
EXPECTED = {
    "scan": (1, 5, 2, 4),
    "scan_fp64": (1, 5, 2, 4),
    "scan_4096": (1, 128, 2, 4),
    "scan_4160": (4, 520, 8, 10),
    "scan_long_1500": (1, 47, 2, 4),
    "scan_long_2000": (4, 252, 4, 6),
    "scan_too_long": (4, 4, 4, 6),
    "sig_scan": (1, 375, 2, 4),
    "sig_thread": (0, 407, 8, 10),
    "seg4": (4, 800, 8, 10),
    "seg2": (4, 3200, 17, 19),
    "seg2_distinct_series": (0, 1600, 17, 19),
    "thread_wide": (0, 3200, 17, 19),
    "seg4_too_long": (0, 200, 4, 6),
    "seg4_mixed": (4, 880, 13, 15),
    "seg4_mixed_off": (4, 800, 8, 10),
    "seg4_lanes_set": (4, 800, 8, 10),
    "seg4_long_20": (4, 960, 17, 19),
    "seg_lanes_0": (1, 200, 2, 4),
    "smoothed": (0, 5, 4, 8),
    "filtered": (0, 5, 4, 8),
    "k6": (0, 5, 4, 6),
    "k6_lane": (2, 5, 4, 6),
    "k12": (2, 5, 4, 6),
    "groups_3": (4, 800, 13, 15),
    "sweeps_5": (4, 800, 21, 23),
    "scan_sweeps_8": (1, 5, 6, 8),
}


def problem(name):
    """The problem of CASES[name] with the defaults filled in and T as the list of window lengths."""
    p = dict(T=60, K=3, precision=32, nser=1, sig=False, smoothed=False, filtered=False)
    p.update(CASES[name][0])
    if not isinstance(p["T"], list):
        p["T"] = [p["T"]] * p["nw"]
    assert len(p["T"]) == p["nw"]
    return p
