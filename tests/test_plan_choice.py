"""Sweep-kernel selection by default, characterised.

The other GPU tests force each kernel through the HMCGPU_* tuning variables; this one pins what the plan chooses on its own,
at both sides of every threshold of the policy, and what a few overrides change.  For each problem of the table (short
windows, a few sweeps) one hmcgpu_estimate reports (sweep_kernel, n_tasks, n_sweep_launches, n_launches): the kernel, the
warp tasks it was laid out in, and how the sweeps were cut into launches over the task groups.

The thresholds scale with the SM count, so the expected values hold on a device with the 148 SMs of the B200 they were
recorded on (NVIDIA B200, 1000 W power limit)."""
import numpy as np
import pytest

from conftest import K3_TRUTH, synth_hmm
from plan_cases import BURNIN, CASES, EXPECTED, NRUN, TUNING, problem

pytestmark = pytest.mark.gpu


def spec_for(H, nw, nc, T, K, precision, nser, sig, smoothed, filtered):
    y_len = max(T) + 12
    y = np.stack([synth_hmm(y_len, seed=1 + s, **K3_TRUTH)[0] for s in range(nser)])
    flags = H.FLAG_REF_Q1 | H.FLAG_SUMMARY
    flags |= H.FLAG_SMOOTHED_MEAN if smoothed else 0
    flags |= H.FLAG_FILTERED_MEAN if filtered else 0
    return H.ProblemSpec(y, [1] * nw, T, K=K, n_chains=nc, burnin=BURNIN, nrun=NRUN, seed=11, precision=precision, flags=flags,
                         win_series=[w % nser for w in range(nw)] if nser > 1 else None,
                         is_signal=np.ones(y_len, dtype=np.uint8) if sig else None)


def observe(H, ctx, monkeypatch, name):
    for v in TUNING:
        monkeypatch.delenv(v, raising=False)
    for k, v in CASES[name][1].items():
        monkeypatch.setenv(k, v)
    o = H.estimate(ctx, spec_for(H, **problem(name)))
    assert o.events == 0
    return (o.sweep_kernel, o.n_tasks, o.n_sweep_launches, o.n_launches)


@pytest.fixture(scope="module")
def b200_sms():
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    if sms != 148:
        pytest.skip(f"the table was recorded on 148 SMs; this device has {sms}")


@pytest.mark.parametrize("name", list(CASES))
def test_default_kernel_choice(H, ctx, monkeypatch, b200_sms, name):
    assert observe(H, ctx, monkeypatch, name) == EXPECTED[name]
