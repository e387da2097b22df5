"""Writes tests/golden/cameras.npz from the UNMODIFIED reference's camera_utils (CPU, a second):

    NFE_REFERENCE=/path/to/NeRFFaceEditing python tests/golden/make_golden_cameras.py [out.npz]

LookAtPoseSampler.sample for the two (horizontal, vertical) pairs of test_host_cpu.py's camera check (look-at point (0, 0, 0.2),
radius 2.7) and FOV_to_intrinsics(18.837), the cameras synth_inputs restates.
"""
import math
import os
import sys

import numpy as np
import torch

REFERENCE = os.environ.get("NFE_REFERENCE")
if not REFERENCE or not os.path.isfile(os.path.join(REFERENCE, "camera_utils.py")):
    raise SystemExit("set NFE_REFERENCE to a checkout of the original NeRFFaceEditing project")
sys.path.insert(0, REFERENCE)

import camera_utils  # noqa: E402

PAIRS = ((math.pi / 2, math.pi / 2), (math.pi / 2 - 0.4, math.pi / 2 + 0.25))

out = sys.argv[1] if len(sys.argv) > 1 else os.path.join(os.path.dirname(os.path.abspath(__file__)), "cameras.npz")
cam2world = torch.cat([camera_utils.LookAtPoseSampler.sample(h, v, torch.tensor([0, 0, 0.2]), radius=2.7) for h, v in PAIRS])
np.savez_compressed(out, pairs=np.array(PAIRS), cam2world=cam2world.numpy(), intrinsics=camera_utils.FOV_to_intrinsics(18.837).numpy(),
                    fov_degrees=np.float64(18.837))
print(out, cam2world.shape)
