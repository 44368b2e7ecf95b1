#!/usr/bin/env python
"""Records the UNMODIFIED reference's pose algebra (diffdrr/pose.py: RigidTransform.convert, convert, get_se3_log) on six
random rigid poses, for every parameterisation but "matrix", into pose_reference.npz (read by tests/test_pose_cpu.py).
Needs the reference sources on sys.path; pass their root as the first argument:
    python tests/golden/make_golden_pose.py <DiffDRR checkout>"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(os.path.dirname(HERE), "_refshim"))
sys.path.insert(0, sys.argv[1])
import diffdrr.pose as ref  # noqa: E402  (the reference's own module)

PARAMS = ["axis_angle", "euler_angles", "quaternion", "quaternion_adjugate", "rotation_6d", "rotation_9d", "rotation_10d",
          "se3_log_map"]

g = torch.Generator().manual_seed(3)
rot = (torch.rand(6, 3, generator=g) * 2 - 1) * 1.2
xyz = (torch.rand(6, 3, generator=g) * 2 - 1) * 200.0
matrix = ref.convert(rot, xyz, parameterization="euler_angles", convention="ZXY").matrix.contiguous()
rec = {"matrix": matrix.numpy(), "se3_log": ref.RigidTransform(matrix.clone()).get_se3_log().numpy()}
for param in PARAMS:
    kw = dict(convention="ZXY") if param == "euler_angles" else {}
    theirs = ref.RigidTransform(matrix.clone()).convert(param, **kw)
    rec[f"{param}_n"] = np.array(len(theirs))
    for i, t in enumerate(theirs):
        rec[f"{param}_{i}"] = t.numpy()
    rec[f"{param}_fwd"] = ref.convert(*theirs, parameterization=param, **kw).matrix.numpy()
np.savez_compressed(os.path.join(HERE, "pose_reference.npz"), **rec)
print({k: v.shape for k, v in rec.items()})
