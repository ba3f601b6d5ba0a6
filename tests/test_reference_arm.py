"""The CPU arm of bench.py computes what the UNMODIFIED reference computes.  The reference's own outputs on the bench
workload's rays (seed 0) and weights are stored in tests/golden/reference_arm_{xavier,trained_like}.npz
(tests/golden/make_golden.py); the oracle port, which bench.py times on the host, must reproduce them bit for bit."""
import importlib.util
import os

import pytest
import torch

from helpers import ROOT, golden, golden_levels, golden_rays, make_state_dict, oracle

FIELDS = ("comp_rgb", "distance", "acc", "weights", "t_samples")


def assert_equals_reference(got, g, what):
    want = golden_levels(g)
    assert len(got) == len(want) == 2
    for lvl in range(2):
        for k, name in enumerate(FIELDS):
            assert torch.equal(got[lvl][k], torch.from_numpy(want[lvl][k])), (what, lvl, name)


@pytest.mark.parametrize("kind", ["xavier", "trained_like"])
def test_port_equals_reference_bit_for_bit(kind):
    g = golden(f"reference_arm_{kind}.npz")
    sd = make_state_dict(seed=0, kind=kind)
    got = oracle.forward(sd, oracle.Rays(*golden_rays(g)), False, True)
    assert_equals_reference(got, g, kind)


def test_bench_cpu_arm_computes_the_references_outputs():
    spec = importlib.util.spec_from_file_location("bench_mod", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    kind, forward = bench._cpu_arm_setup()
    assert kind == "port"
    g = golden("reference_arm_xavier.npz")
    assert_equals_reference(forward(make_state_dict(seed=0), golden_rays(g)), g, "bench CPU arm")
