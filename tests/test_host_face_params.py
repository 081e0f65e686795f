"""Face-parameter SMPL-X models (jaw pose + expression coefficients in theta) on the host: both model builders, the theta
layout, the blob round trip and pack_theta / split_theta.  No GPU needed."""
import ctypes

import numpy as np
import pytest
import torch

from bodyfitting_b200 import _lib
from bodyfitting_b200 import synthetic as syn
from bodyfitting_b200.model import PreparedModel, model_desc

from test_host import _FLOAT_FIELDS, _parse_blob

# (num_betas, num_expression): the default, another split of 20, no expression, and the longest row (1 + 19: 111 entries)
COUNTS = [(10, 10), (12, 8), (10, 0), (1, 19)]


def _c_blob(mt, data, gmm=None, **kw):
    d, keep = model_desc(mt, data, gmm=gmm, tensor_cores=True, **kw)
    blob, n = ctypes.c_void_p(), ctypes.c_int64()
    rc = _lib.lib().bf_model_build_blob(ctypes.byref(d), ctypes.byref(blob), ctypes.byref(n))
    if rc != 0:
        return rc, _lib.last_error()
    raw = ctypes.string_at(blob, n.value)
    _lib.lib().bf_blob_free(blob)
    return rc, raw


def _layout(nb, ne, face):
    """theta offsets of an SMPL-X row (include/bodyfit_b200.h)"""
    off_betas = 7 + 63
    off_leye = off_betas + nb
    off_jaw = off_leye + 18
    return dict(off_betas=off_betas, off_leye=off_leye, off_rh=off_leye + 12, off_jaw=off_jaw, off_expr=off_jaw + 3,
                np=off_jaw + (3 + ne if face else 0))


@pytest.mark.parametrize('nb,ne', COUNTS, ids=['nb%d-ne%d' % c for c in COUNTS])
def test_builders_agree_on_face_models(assets, nb, ne, tmp_path):
    """bf_model_build_blob (C++) and PreparedModel (Python) build the same face-parameter model: every table, NP, the flag."""
    data = syn.make_model('smplx', 0, nb, ne)
    gmm = assets('gmm')
    pm = PreparedModel('smplx', data, gmm=gmm, device='cpu', tensor_cores=True, num_betas=nb, num_expression=ne,
                       face_params=True)
    L = _layout(nb, ne, True)
    assert pm.NP == L['np'] and pm.NE == ne and pm.face_params
    img_p, arr_p = _parse_blob(open(pm.save_blob(str(tmp_path / 'py.blob')), 'rb').read())
    rc, raw = _c_blob('smplx', data, gmm=gmm, num_betas=nb, num_expression=ne, face_params=True)
    assert rc == 0, raw
    img_c, arr_c = _parse_blob(raw)
    assert img_c.face == img_p.face == 1 and img_c.NP == img_p.NP == L['np'], (img_c.NP, img_p.NP)
    for tag, a, b in (('m', img_p, img_c), ('full', img_p.full, img_c.full), ('act', img_p.act, img_c.act)):
        for name, typ in a._fields_:
            if typ is _lib._i32 and not name.startswith('_pad'):
                assert getattr(a, name) == getattr(b, name), (tag, name)
    assert set(arr_p) == set(arr_c)
    for key in sorted(arr_p):
        a, b = arr_p[key], arr_c[key]
        assert len(a) == len(b), key
        if key.split('_', 1)[1] in _FLOAT_FIELDS:
            fa, fb = np.frombuffer(a, np.float32), np.frombuffer(b, np.float32)
            tol = 1e-3 if 'gmm' in key else 1e-6
            assert np.abs(fa - fb).max() <= tol * max(1e-30, float(np.abs(fa).max())), key
        else:
            assert a == b, key
    # the face-off model of the same counts: the same tables, the row without the face block
    off = PreparedModel('smplx', data, gmm=gmm, device='cpu', tensor_cores=True, num_betas=nb, num_expression=ne)
    assert off.NP == _layout(nb, ne, False)['np'] and off.struct.face == 0
    _, arr_off = _parse_blob(open(off.save_blob(str(tmp_path / 'off.blob')), 'rb').read())
    assert arr_off == arr_p


def test_longest_face_row_is_111():
    pm = PreparedModel('smplx', syn.make_model('smplx', 0, 1, 19), device='cpu', tensor_cores=False, num_betas=1,
                       num_expression=19, face_params=True)
    assert pm.NP == 111


def test_builders_reject_face_params_on_smpl(assets):
    """Both builders refuse a face-parameter SMPL model, with the same text; the theta limit of the row without the face
    block stays as it is."""
    text = 'face parameters (jaw pose, expression) apply to SMPL-X only'
    rc, msg = _c_blob('smpl', assets('smpl'), face_params=True)
    assert rc != 0 and msg.endswith(text), msg
    with pytest.raises(ValueError) as e:
        PreparedModel('smpl', assets('smpl'), device='cpu', tensor_cores=False, face_params=True)
    assert str(e.value) == text
    data = syn.make_model('smplx', 0, 16, 4)
    rc, msg = _c_blob('smplx', data, num_betas=16, num_expression=4, face_params=True)
    assert rc != 0 and msg.endswith('104 theta entries exceed the limit of 100'), msg
    with pytest.raises(ValueError, match='104 theta entries exceed the limit of 100'):
        PreparedModel('smplx', data, device='cpu', tensor_cores=False, num_betas=16, num_expression=4, face_params=True)


def test_blob_keeps_face_flag(tmp_path):
    """save_blob / the C++ blob carry BfModel.face (the struct image is stored whole)."""
    data = syn.make_model('smplx', 0)
    pm = PreparedModel('smplx', data, device='cpu', tensor_cores=False, face_params=True)
    img, _ = _parse_blob(open(pm.save_blob(str(tmp_path / 'm.blob')), 'rb').read())
    assert img.face == 1 and img.NP == 111
    rc, raw = _c_blob('smplx', data, face_params=True)
    assert rc == 0
    img_c, _ = _parse_blob(raw)
    assert img_c.face == 1 and img_c.NP == 111
    rc, raw = _c_blob('smplx', data)
    assert _parse_blob(raw)[0].face == 0 and _parse_blob(raw)[0].NP == 98


@pytest.mark.parametrize('nb,ne', COUNTS, ids=['nb%d-ne%d' % c for c in COUNTS])
def test_pack_split_theta_inverse(nb, ne):
    pm = PreparedModel('smplx', syn.make_model('smplx', 0, nb, ne), device='cpu', tensor_cores=False, num_betas=nb,
                       num_expression=ne, face_params=True)
    B = 3
    g = torch.Generator().manual_seed(0)
    r = lambda n: torch.randn(B, n, generator=g)
    parts = dict(transl=r(3), scale=r(1), global_orient=r(3), body_pose=r(63), betas=r(nb), leye_pose=r(3),
                 reye_pose=r(3), left_hand_pose=r(6), right_hand_pose=r(6), jaw_pose=r(3), expression=r(ne))
    th = pm.pack_theta(parts['global_orient'], parts['body_pose'], parts['betas'], transl=parts['transl'],
                       scale=parts['scale'], leye=parts['leye_pose'], reye=parts['reye_pose'], lhand=parts['left_hand_pose'],
                       rhand=parts['right_hand_pose'], jaw=parts['jaw_pose'].reshape(B, 1, 3), expression=parts['expression'])
    assert th.shape == (B, pm.NP)
    L = _layout(nb, ne, True)
    assert torch.equal(th[:, L['off_jaw']:L['off_jaw'] + 3], parts['jaw_pose'])
    assert torch.equal(th[:, L['off_expr']:], parts['expression'])
    sp = pm.split_theta(th)
    assert set(sp) == set(parts)
    for k, v in parts.items():
        assert torch.equal(sp[k], v), k
    # None = 0 for the face block; a face-off model refuses face inputs
    th0 = pm.pack_theta(parts['global_orient'], parts['body_pose'], parts['betas'])
    assert not th0[:, L['off_jaw']:].any()
    off = PreparedModel('smplx', syn.make_model('smplx', 0, nb, ne), device='cpu', tensor_cores=False, num_betas=nb,
                        num_expression=ne)
    with pytest.raises(ValueError):
        off.pack_theta(parts['global_orient'], parts['body_pose'], parts['betas'], jaw=parts['jaw_pose'])
    assert 'jaw_pose' not in off.split_theta(off.pack_theta(parts['global_orient'], parts['body_pose'], parts['betas']))
