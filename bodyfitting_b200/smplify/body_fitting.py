"""Callers of the fitting path (SURVEY.md 8f rank 1): ``BodyFitting`` with the reference's call signature
(``smplify/body_fitting.py:78-107``: SMPLify construction, fit, ``{smpl_type}_parameter.npy`` + ``.obj`` output)
and ``fit_sequence`` -- the batched replacement of the per-frame loop of ``apps/genebody_fitting.py:183-192``:
all frames of a sequence go through ONE SMPLify call (the model is built once, not once per frame).

The HMR network itself (``run_hmr``'s ResNet-50 regressor) is out of scope: the initial (betas, poses) are an
argument (``net_output``), come from a user-supplied ``init_fn(image, c2w) -> (betas[1,10], poses[1,72])``, or -- keeping
the reference's conversion step (body_fitting.py:70-73) -- from ``regressor(image) -> (rotmat[1,24,3,3], betas[1,10], cam)``
whose root orientation is carried into world coordinates and converted to axis-angle here.
"""
import os

import numpy as np

from ..utils.io_utils import load_openpose, save_obj_mesh
from .smplify import SMPLify


class BodyFitting(object):
    def __init__(self, options=None, smpl_type=None, age='adult', use_mask=False, debug=False, init_fn=None, regressor=None,
                 face_params=False, **smplify_kw):
        """``face_params=True`` (SMPL-X): the fits also optimise jaw pose and expression (SMPLify(face_params=)); the results
        and the saved parameter file then hold ``jaw_pose`` and ``expression``.  The hand options ``num_pca_comps``,
        ``use_pca`` and ``flat_hand_mean`` pass through ``smplify_kw`` to SMPLify (or come from ``options``); the saved
        hand poses then have num_pca_comps (or 45) entries."""
        self.options = options
        self.smpl_type = smpl_type or getattr(options, 'smpl_type', 'smpl')
        self.age = getattr(options, 'age', age)
        self.use_mask = getattr(options, 'use_mask', use_mask)
        self.debug = debug
        self.use_hand_face = (self.smpl_type == 'smplx')
        self.init_fn = init_fn
        self.regressor = regressor
        self.face_params = bool(getattr(options, 'face_params', face_params))
        for k in ('num_pca_comps', 'use_pca', 'flat_hand_mean'):
            if hasattr(options, k):
                smplify_kw.setdefault(k, getattr(options, k))
        self.smplify_kw = smplify_kw
        self._smplify = {}

    def _fitter(self, gender, num_iters):
        key = (gender, num_iters)
        if key not in self._smplify:                       # built once per gender, not once per frame
            kw = dict(self.smplify_kw)
            if num_iters is not None:
                kw['num_iters'] = num_iters
            self._smplify[key] = SMPLify(smpl_type=self.smpl_type, age=self.age, gender=gender, use_mask=self.use_mask,
                                         debug=False, face_params=self.face_params, **kw)
        return self._smplify[key]

    def __call__(self, images, c2ws, Ks, keypoints, gender='male', keyframe=25, use_frames=list(range(48)),
                 use_mask=False, masks=None, mask_frames=None, render_skip=12, output_folder=None, use_mesh=False,
                 meshfile=None, disp=False, net_output=None, num_iters=None, imsize=None):
        if net_output is None and self.init_fn is None and self.regressor is not None:
            from ..utils.geometry import world_init_from_camera_rotmat
            pred_rotmat, pred_betas = self.regressor(images[keyframe])[:2]               # body_fitting.py:67
            net_output = (pred_betas, world_init_from_camera_rotmat(pred_rotmat, c2ws[keyframe]))   # :70-73
        if net_output is None:
            if self.init_fn is None:
                raise ValueError('pass net_output=(betas, poses) or construct BodyFitting(init_fn=...) '
                                 '(the HMR regressor of the reference is out of scope)')
            net_output = self.init_fn(images[keyframe], c2ws[keyframe])
        if imsize is None:
            imsize = images[0].shape[0] if images is not None else 512
        smplify = self._fitter(gender, num_iters)
        result = smplify(net_output, c2ws, Ks, keypoints, output_folder, use_mask=use_mask, masks=masks,
                         use_frames=use_frames, mask_frames=mask_frames, keyframe=keyframe, imsize=imsize,
                         use_mesh=use_mesh, meshfile=meshfile, displacement=disp)
        if output_folder is not None:
            write_result(output_folder, self.smpl_type, result, disp)
        return result


def write_result(output_folder, smpl_type, result, disp=False):
    """``{smpl_type}_parameter.npy`` (pickled dict) + ``{smpl_type}.obj`` (+ ``{smpl_type}+d.obj``), body_fitting.py:94-99.
    The parameter file holds every key of ``result``: ``jaw_pose`` / ``expression`` too when the fit optimised them, and
    the hand poses with as many entries as the fit's hand configuration has (num_pca_comps, or 45 without PCA)."""
    os.makedirs(output_folder, exist_ok=True)
    np.save(os.path.join(output_folder, '%s_parameter.npy' % smpl_type), result)
    save_obj_mesh(os.path.join(output_folder, '%s.obj' % smpl_type), result['vertices'], result['faces'])
    if disp and 'displacement' in result:
        save_obj_mesh(os.path.join(output_folder, '%s+d.obj' % smpl_type), result['vertices'] + result['displacement'],
                      result['faces'])


def read_openpose_views(json_paths):
    """One frame: list of per-view OpenPose JSON paths -> list of dicts / None (apps/genebody_fitting.py:157-163)."""
    return [load_openpose(p) if (p is not None and os.path.exists(p)) else None for p in json_paths]


def fit_sequence(fitter, net_outputs, c2ws, Ks, keypoints_per_frame, output_folders=None, imsize=512):
    """All frames of a sequence in one batched fit.
    fitter: SMPLify; net_outputs: (betas [F,10], poses [F,72]); keypoints_per_frame: list over frames of per-view
    OpenPose dict lists (None = view without detection) or of per-view JSON path lists; output_folders: optional list
    of F folders receiving the reference's per-frame files.  Returns the list of per-frame result dicts."""
    frames = []
    for views in keypoints_per_frame:
        if len(views) and isinstance(views[0], str):
            views = read_openpose_views(views)
        frames.append(list(views))
    F = len(frames)
    out = fitter(net_outputs, c2ws, Ks, frames, None, use_frames=list(range(len(c2ws))), imsize=imsize)
    results = []
    for f in range(F):
        r = {k: (np.array(v[f]) if (isinstance(v, np.ndarray) and k != 'faces' and F > 1) else v) for k, v in out.items()}
        results.append(r)
        if output_folders is not None and output_folders[f] is not None:
            write_result(output_folders[f], fitter.smpl_type, r)
    return results
