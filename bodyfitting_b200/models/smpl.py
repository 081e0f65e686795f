"""``SMPL`` -- the reference's ``models/smpl.py:56-90`` wrapper (smplx SMPL + 9 regressed extra joints,
re-indexed to the 49-joint list) and ``create_smplx`` -- the ``smplx.create(model_type='smplx', ...)``
call of ``smplify/smplify.py:59-80`` -- as torch modules whose forward / backward run on the B200
all-vertex LBS kernels (bf_lbs_forward / bf_lbs_backward)."""
import os
from dataclasses import dataclass
from typing import NewType

import numpy as np
import torch
import torch.nn as nn

from .. import ops
from ..model import PreparedModel

Tensor = NewType('Tensor', torch.Tensor)


@dataclass
class ModelOutput:
    vertices: Tensor = None
    joints: Tensor = None
    full_pose: Tensor = None
    betas: Tensor = None
    expression: Tensor = None
    global_orient: Tensor = None
    body_pose: Tensor = None
    left_hand_pose: Tensor = None
    right_hand_pose: Tensor = None
    jaw_pose: Tensor = None
    joints_ori: Tensor = None

    def __getitem__(self, key):
        return getattr(self, key)


class SMPL(nn.Module):
    """Extension of the SMPL model to support more joints (reference: models/smpl.py:56-83)."""

    def __init__(self, model_path='data/smpl', batch_size=1, gender='neutral', create_transl=True, model_data=None,
                 J_regressor_extra=None, J_regressor_h36m=None, device='cuda', **kwargs):
        super().__init__()
        if model_data is None:
            model_data = model_path
        if J_regressor_extra is None:
            fn = os.path.join('data', 'J_regressor_extra.npy')                  # config.JOINT_REGRESSOR_TRAIN_EXTRA
            if not os.path.exists(fn):
                raise FileNotFoundError(fn)
            J_regressor_extra = np.load(fn)
        from ..model import load_model_data
        data = load_model_data(model_data, 'smpl', gender)
        self.prepared = PreparedModel('smpl', data, gmm=None, J_regressor_extra=J_regressor_extra, device=device)
        self.faces = self.prepared.faces
        self.joints = None
        if J_regressor_h36m is None:
            fn = os.path.join('data', 'J_regressor_h36m.npy')                   # config.JOINT_REGRESSOR_H36M (models/smpl.py:63)
            J_regressor_h36m = np.load(fn) if os.path.exists(fn) else None
        self._h36m = ops.SparseRegressor(J_regressor_h36m, self.prepared.device) if J_regressor_h36m is not None else None

    def get_joints_h36m(self, vertices):
        """models/smpl.py:85-87: the 17 Human3.6M joints regressed from the vertices [B,V,3] (differentiable)."""
        if self._h36m is None:
            raise FileNotFoundError('J_regressor_h36m was not given and data/J_regressor_h36m.npy does not exist')
        return ops.regress_joints(vertices, self._h36m)

    def forward(self, global_orient=None, body_pose=None, betas=None, transl=None, return_full_pose=False, **kwargs):
        pm = self.prepared
        theta = pm.pack_theta(global_orient, body_pose, betas)
        verts, joints_all, full_pose = ops.lbs(theta, pm)
        joints, joints_ori = joints_all[:, :pm.K_out], joints_all[:, pm.K_out:]
        if transl is not None:
            verts, joints, joints_ori = verts + transl[:, None], joints + transl[:, None], joints_ori + transl[:, None]
        self.joints = joints_ori
        return ModelOutput(vertices=verts, global_orient=global_orient, body_pose=body_pose, joints=joints,
                           joints_ori=joints_ori, betas=betas, full_pose=full_pose if return_full_pose else None)

    def get_joints_ori(self):
        return self.joints


class SMPLX(nn.Module):
    """SMPL-X as ``SMPLify.__init__`` builds it: 6 PCA hand components, 10 betas + 10 expression coefficients, contour
    landmarks, joints mapped to the 135 OpenPose keypoints (smplify.py:59-80).  Built as a face-parameter model, so
    ``forward`` takes ``jaw_pose`` and ``expression`` like ``smplx.SMPLX.forward``, with gradients (None = 0)."""

    def __init__(self, model_data, device='cuda', num_betas=10, num_expression=10, **kwargs):
        super().__init__()
        self.prepared = PreparedModel('smplx', model_data, gmm=None, device=device, num_betas=num_betas,
                                      num_expression=num_expression, face_params=True)
        self.faces = self.prepared.faces

    def forward(self, global_orient=None, body_pose=None, betas=None, jaw_pose=None, leye_pose=None, reye_pose=None,
                left_hand_pose=None, right_hand_pose=None, expression=None, return_full_pose=False, **kwargs):
        """``jaw_pose`` [B,3] or [B,1,3], ``expression`` [B,NE]; both differentiable, None = 0."""
        pm = self.prepared
        theta = pm.pack_theta(global_orient, body_pose, betas, leye=leye_pose, reye=reye_pose, lhand=left_hand_pose,
                              rhand=right_hand_pose, jaw=jaw_pose, expression=expression)
        verts, joints, full_pose = ops.lbs(theta, pm)
        return ModelOutput(vertices=verts, joints=joints, betas=betas, expression=expression, global_orient=global_orient,
                           body_pose=body_pose, left_hand_pose=left_hand_pose, right_hand_pose=right_hand_pose,
                           jaw_pose=jaw_pose, full_pose=full_pose if return_full_pose else None)


def create_smplx(model_path='data', gender='neutral', model_data=None, device='cuda', num_betas=10, num_expression=10,
                 **kwargs):
    from ..model import load_model_data
    data = model_data if model_data is not None else load_model_data(model_path, 'smplx', gender)
    return SMPLX(data, device=device, num_betas=num_betas, num_expression=num_expression)
