"""Curve points outside the prime-order subgroup (test_gpu_points.py) in the host-thread emulation of the product
sources (see test_emulated_pipeline.py), at small sizes: the curve and subgroup check against Python, the
parameters reader element by element, MSMs over small-order points under every form, and a proof with a key read
unchecked."""
import pytest

import bellman_b200 as bb

import test_gpu_points as GP
from test_emulated_pipeline import worker                       # noqa: F401  (the emulated-library fixture)


@pytest.mark.parametrize("group,n,sites", [(bb.G1, 1, (0,)), (bb.G1, 129, (0, 127, 128)), (bb.G2, 1, (0,)), (bb.G2, 129, (0, 128))])
def test_emulated_points_validate(worker, group, n, sites):
    GP.validation_case(worker, group, n, sites)


def test_emulated_points_validate_identity_and_subgroup(worker):
    GP.test_points_validate_identity_and_subgroup(worker)


def test_emulated_read_parameters_refuses_each_element(worker):
    GP.read_parameters_case(worker)


@pytest.mark.parametrize("group,n,windows,rounds", [(bb.G1, 100, (2, 8, 13, 16), (1, 3, 5)), (bb.G2, 12, (3, 8), (2, 5))])
def test_emulated_msm_outside_subgroup(worker, group, n, windows, rounds):
    GP.msm_outside_subgroup_case(worker, group, n, windows=windows, rounds=rounds)


def test_emulated_prove_with_unchecked_key(worker):
    GP.unchecked_key_prove_case(worker, rounds=30, shard_counts=(2, 8), pairs=2)
