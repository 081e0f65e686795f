"""ORACLE -- TEST INFRASTRUCTURE ONLY.

Runs the reference's own, UNMODIFIED ``smplify/{smplify,loss,prior}.py`` and
``models/{smpl,utils}.py`` from a checkout of the reference project on the CPU
(SURVEY.md Appendix B).  The checkout is the directory named by the environment variable
BODYFIT_REFERENCE or, when that is unset, a directory ``reference`` beside this
repository.  Works only where such a checkout exists: it is used to generate the
committed golden vectors (tests/golden/make_golden*.py) and to validate the standalone
restatement ``oracle/fit_port.py`` live; without it those live tests skip and the
golden vectors stand in.  The product and the GPU tests never import this module.

Unrelated imports of the reference are stubbed (torchgeometry, trimesh,
neural_renderer, matplotlib.dviread, scipy.misc.face, utils.camera, mesh_grid);
``smplx`` is provided by oracle/shim/smplx (restated arithmetic, see smplx_port.py).
"""
import contextlib
import os
import sys
import types

_HERE = os.path.dirname(os.path.abspath(__file__))
REFERENCE_ROOT = os.path.abspath(os.environ.get('BODYFIT_REFERENCE') or os.path.join(_HERE, '..', '..', 'reference'))
_loaded = {}


def available():
    return os.path.isdir(os.path.join(REFERENCE_ROOT, 'smplify'))


def _stub(name, **attrs):
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def load_reference():
    """Import the verbatim reference modules; returns a namespace with
    ``smplify`` (module smplify.smplify), ``loss``, ``prior``, ``smpl`` (models.smpl)."""
    if _loaded:
        return _loaded['ns']
    if not available():
        raise RuntimeError('no reference checkout at %s (set BODYFIT_REFERENCE)' % REFERENCE_ROOT)
    repo = os.path.dirname(_HERE)
    for p in (repo, os.path.join(_HERE, 'shim'), REFERENCE_ROOT):
        if p not in sys.path:
            sys.path.insert(0, p)
    # our package also has sub-packages called models/utils/smplify *inside* bodyfitting_b200,
    # never top-level, so the reference's top-level names resolve to the reference checkout.
    nop = lambda *a, **k: None
    if 'torchgeometry' not in sys.modules:
        _stub('torchgeometry', angle_axis_to_rotation_matrix=nop)
    if 'trimesh' not in sys.modules:
        _stub('trimesh')
    if 'neural_renderer' not in sys.modules:
        _stub('neural_renderer')
    try:
        import matplotlib  # noqa: F401
        import matplotlib.dviread  # noqa: F401
    except Exception:
        mp = _stub('matplotlib')
        mp.dviread = _stub('matplotlib.dviread')
    import scipy.misc
    if not hasattr(scipy.misc, 'face'):
        scipy.misc.face = nop
    _stub('mesh_grid', insert_grid_surface=nop, cumsum=nop, search_nearest_point=nop,
          search_inside_mesh=nop, search_intersect=nop, search_nearest_point_backward=nop)
    import utils  # the reference's top-level package
    assert os.path.abspath(utils.__file__).startswith(REFERENCE_ROOT), utils.__file__
    cam = _stub('utils.camera')
    utils.camera = cam
    import smplx  # the shim
    assert 'oracle' in os.path.abspath(smplx.__file__), smplx.__file__
    import smplify.smplify as ref_smplify
    import smplify.loss as ref_loss
    import smplify.prior as ref_prior
    import models.smpl as ref_smpl
    import models.utils as ref_mutils
    ns = types.SimpleNamespace(smplify=ref_smplify, loss=ref_loss, prior=ref_prior, smpl=ref_smpl,
                               mutils=ref_mutils)
    _loaded['ns'] = ns
    return ns


@contextlib.contextmanager
def data_cwd(data_parent):
    """The reference resolves ``data/...`` relative to the cwd (config.py:1-6)."""
    old = os.getcwd()
    os.chdir(data_parent)
    try:
        yield
    finally:
        os.chdir(old)


class _Cv2ThreeReturn(object):
    """The reference calls OpenCV 3's ``_, contours, _ = cv2.findContours(...)`` (smplify/loss.py:79); OpenCV 4 returns
    (contours, hierarchy).  This adapter restores the three-value form and forwards everything else untouched."""

    def __init__(self, cv2):
        self._cv2 = cv2

    def __getattr__(self, name):
        return getattr(self._cv2, name)

    def findContours(self, *a, **k):
        res = self._cv2.findContours(*a, **k)
        return (None, res[0], res[1]) if len(res) == 2 else res


def run_reference_fit(data_parent, smpl_type, init_betas, init_poses, c2ws, Ks, keypoints, num_iters=100,
                      imsize=512, record=True, masks=None, mask_frames=None, age='adult'):
    """One frame through the verbatim ``SMPLify.__call__`` (smplify/smplify.py:84-250) on CPU.
    ``keypoints`` = list (per view) of OpenPose dicts.  Returns (result dict, per-iteration
    total-loss list, per-iteration loss-term dicts)."""
    import numpy as np
    import torch
    ns = load_reference()
    trace, terms = [], []
    orig = ns.smplify.multiview_keypoint_loss

    def recording(*a, **k):
        total, d = orig(*a, **k)
        trace.append(float(total.detach()))
        terms.append({kk: float(np.asarray(vv).sum()) for kk, vv in d.items()})
        return total, d

    with data_cwd(data_parent):
        if record:
            ns.smplify.multiview_keypoint_loss = recording
        try:
            fitter = ns.smplify.SMPLify(smpl_type=smpl_type, num_iters=num_iters, gender='neutral', age=age,
                                        device=torch.device('cpu'), debug=False)
            nv = len(c2ws)
            extra = {}
            if masks is not None:                       # silhouette term: masks [Nm,H,W] uint8 of the views mask_frames
                extra = dict(use_mask=True, masks=list(masks), mask_frames=list(mask_frames))
                ns.loss.cv2 = _Cv2ThreeReturn(ns.loss.cv2)
            res = fitter((torch.tensor(init_betas).float().reshape(1, -1).clone(),
                          torch.tensor(init_poses).float().reshape(1, -1).clone()),
                         [np.asarray(c, dtype=np.float32) for c in c2ws], [np.asarray(k) for k in Ks],
                         keypoints, None, use_frames=list(range(nv)), imsize=imsize, **extra)
        finally:
            ns.smplify.multiview_keypoint_loss = orig
            if isinstance(ns.loss.cv2, _Cv2ThreeReturn):
                ns.loss.cv2 = ns.loss.cv2._cv2
    return res, trace, terms, fitter
