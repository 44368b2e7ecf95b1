"""Host-side pose algebra (diffdrr_b200/pose.py) against the UNMODIFIED reference (diffdrr/pose.py), recorded in
tests/golden/pose_reference.npz by make_golden_pose.py, plus round trips: all nine parameterisations in BOTH directions
(se3_log_map / quaternion_adjugate / rotation_10d included in RigidTransform.convert)."""
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN
from diffdrr_b200.pose import PARAMETERIZATIONS, RigidTransform, convert


def _poses(B=6, seed=0):
    g = torch.Generator().manual_seed(seed)
    rot = (torch.rand(B, 3, generator=g) * 2 - 1) * 1.2
    xyz = (torch.rand(B, 3, generator=g) * 2 - 1) * 200.0
    return convert(rot, xyz, parameterization="euler_angles", convention="ZXY")


@pytest.mark.parametrize("param", [p for p in PARAMETERIZATIONS])
def test_convert_round_trip(param):
    pose = _poses()
    kw = dict(convention="ZYX") if param == "euler_angles" else {}
    back = pose.convert(param, **kw)
    again = convert(*back, parameterization=param, **kw) if param != "matrix" else RigidTransform(pose.matrix)
    assert torch.allclose(again.matrix, pose.matrix, atol=2e-4, rtol=1e-5), param


@pytest.fixture(scope="module")
def ref():
    return {k: torch.from_numpy(v) for k, v in np.load(os.path.join(GOLDEN, "pose_reference.npz")).items()}


@pytest.mark.parametrize("param", [p for p in PARAMETERIZATIONS if p != "matrix"])
def test_convert_matches_the_reference_both_ways(param, ref):
    pose = RigidTransform(ref["matrix"].clone())
    kw = dict(convention="ZXY") if param == "euler_angles" else {}
    ours = pose.convert(param, **kw)
    theirs = [ref[f"{param}_{i}"] for i in range(int(ref[f"{param}_n"]))]
    assert len(ours) == len(theirs), param
    for a, b in zip(ours, theirs):
        assert torch.allclose(a, b, atol=5e-4, rtol=1e-4), param
    fwd_ours = convert(*theirs, parameterization=param, **kw).matrix
    assert torch.allclose(fwd_ours, ref[f"{param}_fwd"], atol=5e-4, rtol=1e-4), param
    assert torch.allclose(pose.get_se3_log(), ref["se3_log"], atol=5e-4, rtol=1e-4)
