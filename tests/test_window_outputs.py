"""The per-window outputs of hmcgpu_result and hmcgpu_predictive, as the single-device fetch, the multi-device scatter, the flag
checks and the pointer gating treat them.  The tests walk the pointer fields of the ctypes structs instead of naming outputs, so
an output added to the ABI is covered as soon as ProblemSpec.alloc_result / alloc_predictive allocate it."""
import ctypes as C

import numpy as np
import pytest

from conftest import K3_TRUTH, synth_hmm

pytestmark = pytest.mark.gpu

GATED = ("rhat", "ess", "ess_lag")        # appended in ABI version 300: read only with HMCGPU_FLAG_DIAGNOSTICS


def _pointer_fields(struct):
    return [name for name, t in struct._fields_ if issubclass(t, C._Pointer)]


def _call(ctx, spec, devices=None, res_fill=None):
    """One hmcgpu_estimate_predictive (devices None) or hmcgpu_estimate_multi_predictive call over the arrays ProblemSpec
    allocates.  res_fill(res) may repoint fields first.  Returns (rc, {pointer field: the array it points to, or None})."""
    from hmc_jl_b200 import binding as B
    o, res = spec.alloc_result()
    pr = spec.alloc_predictive(o)
    arrays = {a.ctypes.data: a for a in vars(o).values() if isinstance(a, np.ndarray)}
    if res_fill is not None:
        arrays.update(res_fill(res))
    prob = spec.struct()
    prp = None if pr is None else C.byref(pr)
    if devices is None:
        rc = ctx.L.hmcgpu_estimate_predictive(ctx.h, C.byref(prob), C.byref(res), prp)
    else:
        rc = ctx.L.hmcgpu_estimate_multi_predictive((C.c_int * len(devices))(*devices), len(devices), C.byref(prob), C.byref(res), prp)
    out = {}
    for struct, cls in ((res, B.Result), (pr, B.Predictive)):
        for name in _pointer_fields(cls):
            p = None if struct is None else C.cast(getattr(struct, name), C.c_void_p).value
            out[name] = None if p is None else arrays[p]
    return rc, out


def _ragged_spec(H, flags, horizons, **kw):
    y0, _ = synth_hmm(260, **K3_TRUTH)
    ys = np.stack([y0, y0 + np.random.default_rng(2).normal(0, 0.3, size=len(y0))])
    return H.ProblemSpec(ys, [1, 5, 2, 40, 1], [200, 180, 120, 240, 90], K=3, n_chains=3, burnin=10, nrun=8, seed=9,
                         horizons=horizons, precision=32, flags=flags, win_series=[1, 0, 1, 1, 0], **kw)


@pytest.mark.parametrize("case", ["all", "summary_filtered"])
def test_multi_device_outputs_equal_single_device(H, ctx, case):
    """Every output, the status of every chain and the return value: estimate_multi over two contexts (windows sharded, then
    scattered back per window) is bit-identical to one estimate, for ragged windows."""
    from hmc_jl_b200 import binding as B
    if case == "all":
        flags = H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY | H.FLAG_LOGLIK | H.FLAG_DIAGNOSTICS | H.FLAG_PREDICTIVE | H.FLAG_SMOOTHED_MEAN
        spec = _ragged_spec(H, flags, (1, 3), pred_grid=np.linspace(-2, 12, 17))
    else:
        spec = _ragged_spec(H, H.FLAG_REF_Q1 | H.FLAG_SUMMARY | H.FLAG_FILTERED_MEAN, (1, 4))
    rc1, one = _call(ctx, spec)
    rc2, two = _call(ctx, spec, devices=[0, 0])
    assert rc1 >= 0 and rc2 == rc1
    assert set(one) == set(_pointer_fields(B.Result) + _pointer_fields(B.Predictive))
    if case == "all":
        assert all(a is not None for a in one.values()), [k for k, a in one.items() if a is None]
    else:
        assert all(one[k] is not None for k in ("summary_mean", "summary_var", "pib_mean", "insample_forecast_mean", "status"))
    for name, a in one.items():
        if a is None:
            assert two[name] is None, name
        else:
            np.testing.assert_array_equal(two[name], a, err_msg=name)


def test_gated_fields_are_not_read_and_unflagged_requests_fail(H, ctx):
    from hmc_jl_b200 import binding as B
    spec = _ragged_spec(H, H.FLAG_REF_Q1 | H.FLAG_DRAWS | H.FLAG_SUMMARY, (1, 2))
    F = 3 * 3 + 9 + 2 * 2 + 1
    types = dict(B.Result._fields_)

    # without HMCGPU_FLAG_DIAGNOSTICS the diagnostics pointers are neither read nor written
    def sentinels(res):
        arrs = {}
        for name in GATED:
            a = np.full((spec.n_windows, F), -7, dtype=np.int32 if name == "ess_lag" else np.float64)
            setattr(res, name, C.cast(a.ctypes.data, types[name]))
            arrs[a.ctypes.data] = a
        return arrs
    for devices in (None, [0, 0]):
        rc, out = _call(ctx, spec, devices, sentinels)
        assert rc >= 0
        for name in GATED:
            assert (out[name] == -7).all(), name

    # an output requested without the flag that produces it: HMCGPU_ERR_ARG from hmcgpu_plan_fetch, naming the flag
    buf = np.zeros(1 << 16)
    plan = H.Plan(ctx, _ragged_spec(H, H.FLAG_REF_Q1, (1, 2)))
    draws = H.Plan(ctx, _ragged_spec(H, H.FLAG_REF_Q1 | H.FLAG_DRAWS, (1, 2)))
    try:
        plan.run()
        draws.run()
        checked = [n for n in _pointer_fields(B.Result) if n not in GATED and n != "status"]    # (status needs no flag)
        cases = [(plan, n, "HMCGPU_FLAG_") for n in checked] + [(draws, "loglik", "HMCGPU_FLAG_LOGLIK")]
        for pl, name, flag in cases:
            res = B.Result()
            setattr(res, name, C.cast(buf.ctypes.data, types[name]))
            assert ctx.L.hmcgpu_plan_fetch(pl.h, C.byref(res)) == B.ERR_ARG, name
            msg = ctx.L.hmcgpu_last_error(ctx.h).decode()
            assert name in msg and flag in msg, msg
        assert (buf == 0).all()
    finally:
        plan.close()
        draws.close()


def test_status_is_read_through_the_slot_layout(H, ctx, monkeypatch):
    """status and the return value (chains with events) read each window's chains where the slot layout put them.  In the
    mixed segment layout the long class is padded to a multiple of 32 slots (here 3 windows x 24 chains = 72 -> 96), so every
    later window starts 24 slots past j * n_chains.  The shortest window (last in length order) runs on a series of its own
    with an observation so far out that every fp64 emission underflows under a tight variance prior (as in
    test_zero_normaliser_events_are_counted_and_survived): each of its chains counts events at every sweep.  The other windows'
    series varies so little that no emission underflows."""
    monkeypatch.setenv("HMCGPU_SCAN_MAX_CHAINS", "0")   # (2400 chains would otherwise take the warp-per-chain kernel)
    monkeypatch.setenv("HMCGPU_SEG_LONG", "3")
    lens = list(range(249, 149, -1))                    # 100 windows of 150..249 steps
    nw, nc = len(lens), 24
    quiet = 0.05 + 0.01 * np.random.default_rng(5).standard_normal(max(lens) + 12)
    loud = quiet.copy()
    loud[120] = 4.0e3
    spec = H.ProblemSpec(np.stack([quiet, loud]), [1] * nw, lens, K=3, n_chains=nc, burnin=0, nrun=3, seed=3, horizons=(1,),
                         precision=64, flags=H.FLAG_REF_Q1 | H.FLAG_SUMMARY, win_series=[0] * (nw - 1) + [1],
                         alpha=np.full(3, 1.0e4))
    o = H.estimate(ctx, spec)
    # segment kernel with the long class: 96 / 4 + 2336 / 8 - 96 / 8 warp tasks (300 without it)
    assert (o.sweep_kernel, o.n_tasks) == (4, 316)
    assert np.flatnonzero(o.status.any(axis=1)).tolist() == [nw - 1]
    assert (o.status[nw - 1] > 0).all()
    assert o.events == np.count_nonzero(o.status) == nc
