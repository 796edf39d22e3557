"""The host policy of a plan (hmc.jl_b200/csrc/plan_policy.cuh) on the CPU: the sweep-kernel choice and slot layout of the
choice table in plan_cases.py, and the rules of the launch schedule over a grid of run shapes.  tests/plan_policy_driver.cpp
is compiled with g++ and prints what the header decides."""
import itertools
import math
import os
import subprocess

import pytest

from conftest import ROOT
from plan_cases import BURNIN, CASES, EXPECTED, NRUN, TUNING, problem

CSRC = os.path.join(ROOT, "hmc.jl_b200", "csrc")
SUMMARY, SMOOTHED_MEAN, FILTERED_MEAN = 4, 8, 64       # HMCGPU_FLAG_* (include/hmcgpu.h)


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    exe = tmp_path_factory.mktemp("plan_policy") / "plan_policy_driver"
    subprocess.check_call(["g++", "-std=c++17", "-O2", "-I", os.path.join(ROOT, "include"), "-I", CSRC,
                           "-o", str(exe), os.path.join(ROOT, "tests", "plan_policy_driver.cpp")])
    return str(exe)


def run(driver, args, env=None, stdin=None):
    e = {k: v for k, v in os.environ.items() if k not in TUNING}
    e.update(env or {})
    return subprocess.run([driver, *args], env=e, input=stdin, capture_output=True, text=True, check=True, timeout=120).stdout


def parse_ops(lines):
    """The schedule in order: launches, and posts as {"post": chunk}."""
    ops = []
    for ln in lines:
        f = ln.split()
        if f[0] == "P":
            ops.append({"post": int(f[1])})
        else:
            g, s0, n, k, wait, closes, last = map(int, f[1:])
            ops.append(dict(g=g, s0=s0, n=n, k=k, wait=wait, closes=bool(closes), last=bool(last)))
    return ops


def plan(driver, name=None, sm=148, env=None, **prob):
    """(header values, schedule) the driver prints for a problem of plan_cases (by name) or given directly."""
    if name is not None:
        prob, env = problem(name), CASES[name][1]
    flags = 1 | SUMMARY | (SMOOTHED_MEAN if prob.get("smoothed") else 0) | (FILTERED_MEAN if prob.get("filtered") else 0)
    args = ["plan", f"sm={sm}", f"K={prob.get('K', 3)}", f"precision={prob.get('precision', 32)}", f"nc={prob['nc']}",
            f"nser={prob.get('nser', 1)}", f"sig={int(bool(prob.get('sig')))}", "n_h=1", f"flags={flags}",
            f"burnin={prob.get('burnin', BURNIN)}", f"nrun={prob.get('nrun', NRUN)}", "T=" + ",".join(map(str, prob["T"]))]
    out = run(driver, args, env).splitlines()
    if out[0].startswith("error"):
        return out[0], []
    head = {k: int(v) for k, v in (ln.split() for ln in out if ln[0].islower())}
    return head, parse_ops([ln for ln in out if ln[0] in "LP"])


@pytest.mark.parametrize("name", list(CASES))
def test_choice_table_on_148_sms(driver, name):
    head, ops = plan(driver, name)
    launches = [o for o in ops if "post" not in o]
    assert (head["kernel"], head["n_tasks"], len(launches)) == EXPECTED[name][:3]
    assert [o["post"] for o in ops if "post" in o] == list(range(math.ceil(NRUN / head["chunk"])))


def test_scan_and_segment_window_limits(driver):
    assert run(driver, ["limits", "32", "3", "8"]).split() == ["scan_max_T", "3196", "seg_max_T", "8160"]
    assert run(driver, ["limits", "64", "4", "2"]).split() == ["scan_max_T", "1278", "seg_max_T", "504"]


def test_bad_segment_lanes_is_an_argument_error(driver):
    err, _ = plan(driver, nc=64, T=[60] * 100, env={"HMCGPU_SEG_LANES": "3"})
    assert err == "error -1 HMCGPU_SEG_LANES must be 0, 2, 4 or 8"


def test_mixed_class_is_padded_to_whole_warps(driver):
    """The layout of test_status_is_read_through_the_slot_layout: 3 long windows x 24 chains = 72 slots, padded to 96, in
    96 / 4 tasks of 8 lanes per chain; the other 97 windows in 2336 / 8 tasks of 4 lanes."""
    head, _ = plan(driver, nc=24, T=list(range(249, 149, -1)), precision=64, nser=2, burnin=0, nrun=3,
                   env={"HMCGPU_SCAN_MAX_CHAINS": "0", "HMCGPU_SEG_LONG": "3"})
    assert (head["kernel"], head["n_long"], head["seg_lanes"], head["n_slots"], head["n_tasks"]) == (4, 3, 4, 96 + 2336, 316)


def check_schedule(ops, burnin, nrun, chunk, n_bufs, G, L):
    S, n_chunks = burnin + nrun, math.ceil(nrun / chunk)

    def limit(s0):                                       # the next boundary: end of burn-in or of the draw chunk
        return burnin if s0 < burnin else burnin + min(nrun, ((s0 - burnin) // chunk + 1) * chunk)

    next_s = [0] * G
    closed = [dict() for _ in range(G)]                  # group -> {chunk: position of its closing launch}
    post_at = {}
    for i, o in enumerate(ops):
        if "post" in o:
            k = o["post"]
            assert k == len(post_at), "chunks are posted once each, in order"
            assert all(k in c for c in closed), "a chunk is posted after every group has closed it"
            ready = max([c[k] for c in closed] + [post_at.get(k - 1, -1)])
            assert all("post" in ops[j] for j in range(ready + 1, i)), "posted as soon as every group has closed it"
            post_at[k] = i
            continue
        g, s0, n = o["g"], o["s0"], o["n"]
        assert s0 == next_s[g] and n >= 1, "a group's launches tile its sweeps in order"
        assert s0 + n <= limit(s0), "no launch crosses the end of burn-in or of a draw chunk"
        want = max(1, L * (g + 1) // G) if s0 == 0 and G > 1 else L    # first launch of a group: the stagger
        assert n == min(want, limit(s0) - s0)
        k = (s0 - burnin) // chunk if s0 >= burnin else -1
        assert o["k"] == k
        assert o["closes"] == (k >= 0 and s0 + n == limit(s0))
        if o["closes"]:
            closed[g][k] = i
        starts_chunk = k >= n_bufs and (s0 - burnin) % chunk == 0
        assert o["wait"] == (k - n_bufs if starts_chunk else -1)
        if starts_chunk:
            assert post_at.get(k - n_bufs, i) < i, "a chunk's buffer is reused only after the post of chunk k - n_bufs"
        assert o["last"] == (s0 + n == S)
        next_s[g] = s0 + n
    assert next_s == [S] * G
    assert sum(o.get("last", False) for o in ops) == G
    assert sorted(post_at) == list(range(n_chunks))
    assert all(sorted(c) == list(range(n_chunks)) for c in closed)


def test_launch_schedule_rules(driver):
    shapes = []
    for burnin, nrun, n_bufs, G, L in itertools.product((0, 1, 24, 1000), (1, 3, 24, 1025), (1, 2), (1, 2, 3, 4, 8), (1, 5, 16, 64)):
        for chunk in sorted({c for c in (1, 2, 7, 24, 1024) if c <= nrun} | {nrun}):
            shapes.append((burnin, nrun, chunk, n_bufs, G, L))
    out = run(driver, ["schedule"], stdin="".join("%d %d %d %d %d %d\n" % s for s in shapes))
    blocks = out.split("end\n")
    assert len(blocks) == len(shapes) + 1 and blocks[-1] == ""
    for shape, block in zip(shapes, blocks):
        check_schedule(parse_ops(block.splitlines()), *shape)
