"""Small golden fixtures made by running the reference's OWN code (BODYFIT_REFERENCE = a checkout of the reference project):

  reference_init_conversion.npz  utils/geometry.py:331-493 convert_hom_to_angle (incl. the NaN patch for the identity) and the
                                 world transform of the root orientation, smplify/body_fitting.py:70-73, on seeded rotations;
  reference_openpose_parse.npz   utils/io_utils.py:138-183 load_openpose on the reference's only real-data fixture,
                                 openpose/test.json (copied next to it as a data fixture: it is an OpenPose output file, not
                                 reference source).

    BODYFIT_REFERENCE=<reference checkout> python tests/golden/make_golden_aux.py
"""
import os
import shutil
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import ref_harness as rh          # noqa: E402


def main():
    rh.load_reference()                        # stubs + sys.path for the reference's top-level packages
    import utils.geometry as rg                # the reference's file, unmodified
    from scipy.spatial.transform import Rotation as Rot
    rng = np.random.RandomState(7)
    rv = rng.randn(2 * 24, 3) * 1.1
    rv[0] = 0.0                                # identity: the reference's converter yields NaN and patches it to 0
    rv[5] = [np.pi - 1e-3, 0.0, 0.0]
    R = torch.tensor(Rot.from_rotvec(rv).as_matrix(), dtype=torch.float32).reshape(2, 24, 3, 3)
    pose = rg.convert_hom_to_angle(R, 2, torch.device('cpu')).numpy()
    c2w = np.eye(4, dtype=np.float32)
    c2w[:3, :3] = Rot.from_rotvec([0.3, -0.8, 0.5]).as_matrix().astype(np.float32)
    c2w[:3, 3] = [0.1, 0.2, 2.5]
    Rw = R[:1].clone()
    Rw[0, 0] = torch.from_numpy(c2w)[:3, :3] @ Rw[0, 0]                          # body_fitting.py:70-72, verbatim ops
    pose_world = rg.convert_hom_to_angle(Rw, 1, torch.device('cpu')).numpy()
    np.savez_compressed(os.path.join(HERE, 'reference_init_conversion.npz'), rotmat=R.numpy(), pose=pose, c2w=c2w,
                        pose_world=pose_world)
    print('wrote reference_init_conversion.npz', pose.shape, pose_world.shape)

    import utils.io_utils as rio
    src = os.path.join(rh.REFERENCE_ROOT, 'openpose', 'test.json')
    dst = os.path.join(HERE, 'openpose_test.json')
    shutil.copyfile(src, dst)
    parsed = rio.load_openpose(src)
    np.savez_compressed(os.path.join(HERE, 'reference_openpose_parse.npz'), **{k: np.asarray(v) for k, v in parsed.items()})
    print('wrote reference_openpose_parse.npz', {k: np.asarray(v).shape for k, v in parsed.items()})


if __name__ == '__main__':
    main()
