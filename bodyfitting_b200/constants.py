"""Static index tables consumed by the kernels (data, not arithmetic).

* ``SPIN_JOINT_MAP``: the 49-entry re-indexing that the reference's SMPL wrapper applies
  to ``cat(45 smplx joints, 9 J_regressor_extra joints)`` -- it is
  ``[constants.JOINT_MAP[n] for n in constants.JOINT_NAMES]`` of the reference
  (constants.py:13-89, models/smpl.py:61,74-75): 25 OpenPose joints then 24 GT joints.
* ``smpl_to_openpose``: OpenPose (coco25 / coco19) <- model joint tables of
  models/utils.py:32-141.
* loss constants of smplify/loss.py:17-20,139-141 and smplify/smplify.py:160.
"""
import numpy as np

SPIN_JOINT_MAP = [
    # 25 OpenPose joints
    24, 12, 17, 19, 21, 16, 18, 20, 0, 2, 5, 8, 1, 4, 7, 25, 26, 27, 28, 29, 30, 31, 32, 33, 34,
    # 24 ground-truth joints
    8, 5, 45, 46, 4, 7, 21, 19, 17, 16, 18, 20, 47, 48, 49, 50, 51, 52, 53, 24, 26, 25, 28, 27,
]

SKELETON_LENGTH = 25          # smplify/loss.py:17
HANDS_LENGTH = 42             # smplify/loss.py:18
FACE_LENGTH = 68              # smplify/loss.py:19
FACE_MAPPING = list(range(17, 17 + 51)) + list(range(0, 17))   # smplify/loss.py:20

GMOF_SIGMA = 100.0            # smplify/loss.py:139
SHAPE_PRIOR_WEIGHT = 5.0      # smplify/loss.py:140
EXPR_PRIOR_WEIGHT = 5.0       # expression L2 prior of face-parameter fits (this project's choice; not in the reference)
ANGLE_PRIOR_WEIGHT = 15.2     # smplify/loss.py:140
POSE_PRIOR_WEIGHT = 4.78      # smplify/loss.py:141
ANGLE_PRIOR_IDXS = [52, 55, 9, 12]            # smplify/loss.py:60-61 (into the 69-D body pose)
ANGLE_PRIOR_SIGNS = [1.0, -1.0, -1.0, -1.0]
CONSTANT_SCALE_NO_SCAN = 0.3  # smplify/smplify.py:160
LR_TRANSL_SCALE = 0.1         # smplify/smplify.py:167-168
LR_DEFAULT = 1e-2             # smplify/smplify.py:174
ADAM_BETAS = (0.9, 0.999)
ADAM_EPS = 1e-8

_BODY25 = {
    'smpl': [24, 12, 17, 19, 21, 16, 18, 20, 0, 2, 5, 8, 1, 4, 7] + list(range(25, 35)),
    'smplh': [52, 12, 17, 19, 21, 16, 18, 20, 0, 2, 5, 8, 1, 4, 7] + list(range(53, 63)),
    'smplx': [55, 12, 17, 19, 21, 16, 18, 20, 0, 2, 5, 8, 1, 4, 7] + list(range(56, 66)),
}
# (wrist, first finger joint of thumb/index/middle/ring/pinky in OpenPose order, first tip index)
_HANDS = {
    ('smplh', 25): ((20, (34, 22, 25, 31, 28), 63), (21, (49, 37, 40, 46, 43), 68)),
    ('smplx', 25): ((20, (37, 25, 28, 34, 31), 66), (21, (52, 40, 43, 49, 46), 71)),
    ('smplh', 19): ((20, (34, 22, 25, 31, 28), 57), (21, (49, 37, 40, 46, 43), 62)),
    ('smplx', 19): ((20, (37, 25, 28, 34, 31), 60), (21, (52, 40, 43, 49, 46), 65)),
}


def smpl_to_openpose(model_type='smplx', use_hands=True, use_face=True, use_face_contour=False,
                     openpose_format='coco25'):
    """Indices into the model's joint list for every OpenPose keypoint
    (same values as models/utils.py:32-141 of the reference)."""
    fmt = openpose_format.lower()
    if fmt not in ('coco25', 'coco19'):
        raise ValueError('Unknown joint format: {}'.format(openpose_format))
    if model_type not in _BODY25:
        raise ValueError('Unknown model type: {}'.format(model_type))
    n = 25 if fmt == 'coco25' else 19
    body = _BODY25[model_type][:n]
    if model_type == 'smpl':
        return np.array(body, dtype=np.int32)
    out = list(body)
    if use_hands:
        for wrist, firsts, tip0 in _HANDS[(model_type, n)]:
            out.append(wrist)
            for f, j0 in enumerate(firsts):
                out += [j0, j0 + 1, j0 + 2, tip0 + f]
    if use_face and model_type == 'smplx':
        start = 76 if n == 25 else 70
        out += list(range(start, start + 51 + 17 * int(bool(use_face_contour))))
    return np.array(out, dtype=np.int32)


# Vertex ids of the 21 vertex-picked joints (smplx.vertex_ids: nose, reye, leye, rear, lear, LBigToe, LSmallToe, LHeel,
# RBigToe, RSmallToe, RHeel, left thumb / index / middle / ring / pinky tips, right ...), in vertex_joint_selector order.
# The official model files do not carry them (smplx hard-codes the table), so the loader falls back to these.
EXTRA_VIDS = {
    'smpl': [332, 6260, 2800, 4071, 583, 3216, 3226, 3387, 6617, 6624, 6787,
             2746, 2319, 2445, 2556, 2673, 6191, 5782, 5905, 6016, 6133],
    'smplx': [9120, 9929, 9448, 616, 6, 5770, 5780, 8846, 8463, 8474, 8635,
              5361, 4933, 5058, 5169, 5286, 8079, 7669, 7794, 7905, 8022],
}
SHAPE_SPACE_DIM = 300          # official SMPL-X files: shapedirs [V,3,400] = 300 shape + 100 expression directions
