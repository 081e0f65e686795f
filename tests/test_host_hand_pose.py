"""SMPL-X hand options (smplx.create's num_pca_comps / use_pca / flat_hand_mean) on the host: both model builders, the theta
layout, the limits, the blob round trip and pack_theta / split_theta.  No GPU needed."""
import ctypes

import numpy as np
import pytest
import torch

from bodyfitting_b200 import _lib
from bodyfitting_b200 import synthetic as syn
from bodyfitting_b200.model import PreparedModel, model_desc

from test_host import _FLOAT_FIELDS, _parse_blob


def hand_model(seed=0, nb=10, ne=10):
    """the synthetic SMPL-X model with 45-row hand component tables: its own first 6 rows, then 39 rows drawn from an
    independent seed at the same scale (the synthetic generator's stream stays untouched)"""
    data = dict(syn.make_model('smplx', seed, nb, ne))
    rng = np.random.RandomState(4500 + seed)
    for k in ('hands_componentsl', 'hands_componentsr'):
        c = np.asarray(data[k], np.float32)
        extra = rng.standard_normal((45 - c.shape[0], 45)) * float(c.std())
        data[k] = np.concatenate([c, extra.astype(np.float32)], 0)
    return data


# (num_pca_comps, use_pca, flat_hand_mean): PCA with 6, 12, 1 and 45 components, with and without the hand mean, and
# axis-angle hands with and without it
HANDS = [(n, True, flat) for n in (6, 12, 1, 45) for flat in (False, True)] + [(6, False, False), (6, False, True)]
HAND_IDS = ['%s%s' % ('pca%d' % n if pca else 'aa', '-flat' if flat else '') for n, pca, flat in HANDS]


def n_hand(n, pca):
    return n if pca else 45


def _c_blob(data, **kw):
    d, keep = model_desc('smplx' if 'hands_meanl' in data else 'smpl', data, tensor_cores=False, **kw)
    blob, nb = ctypes.c_void_p(), ctypes.c_int64()
    rc = _lib.lib().bf_model_build_blob(ctypes.byref(d), ctypes.byref(blob), ctypes.byref(nb))
    if rc != 0:
        return rc, _lib.last_error()
    raw = ctypes.string_at(blob, nb.value)
    _lib.lib().bf_blob_free(blob)
    return rc, raw


def _py_blob(pm, path):
    return open(pm.save_blob(str(path)), 'rb').read()


@pytest.fixture(scope='module')
def data45():
    return hand_model(0)


@pytest.mark.parametrize('face', [False, True], ids=['face-off', 'face-on'])
@pytest.mark.parametrize('n,pca,flat', HANDS, ids=HAND_IDS)
def test_builders_agree_on_hand_models(data45, n, pca, flat, face, tmp_path):
    """bf_model_build_blob (C++) and PreparedModel (Python) build the same hand model table by table: n_hand, NP, the
    component rows (the identity for axis-angle hands) and the pose mean (no hand mean for flat_hand_mean)."""
    kw = dict(num_pca_comps=n, use_pca=pca, flat_hand_mean=flat, face_params=face)
    pm = PreparedModel('smplx', data45, device='cpu', tensor_cores=False, **kw)
    nh = n_hand(n, pca)
    assert pm.n_hand == nh and pm.NP == 86 + 2 * nh + (13 if face else 0)
    img_p, arr_p = _parse_blob(_py_blob(pm, tmp_path / 'py.blob'))
    rc, raw = _c_blob(data45, **kw)
    assert rc == 0, raw
    img_c, arr_c = _parse_blob(raw)
    assert img_c.n_hand == img_p.n_hand == nh and img_c.NP == img_p.NP == pm.NP and img_c.face == img_p.face == int(face)
    for tag, a, b in (('m', img_p, img_c), ('full', img_p.full, img_c.full), ('act', img_p.act, img_c.act)):
        for name, typ in a._fields_:
            if typ is _lib._i32:
                assert getattr(a, name) == getattr(b, name), (tag, name)
    assert set(arr_p) == set(arr_c)
    for key in sorted(arr_p):
        a, b = arr_p[key], arr_c[key]
        assert len(a) == len(b), key
        if key.split('_', 1)[1] in _FLOAT_FIELDS:
            fa, fb = np.frombuffer(a, np.float32), np.frombuffer(b, np.float32)
            tol = 0 if key in ('m_hand_l', 'm_hand_r', 'm_pose_mean') else 1e-6
            assert np.abs(fa - fb).max() <= tol * max(1e-30, float(np.abs(fa).max())), key
        else:
            assert a == b, key
    hl = np.frombuffer(arr_c['m_hand_l'], np.float32)[:nh * 45].reshape(nh, 45)
    want = np.asarray(data45['hands_componentsl'], np.float32)[:nh] if pca else np.eye(45, dtype=np.float32)
    assert np.array_equal(hl, want)
    pmean = np.frombuffer(arr_c['m_pose_mean'], np.float32)[:165]
    assert np.array_equal(pmean[75:120], np.zeros(45, np.float32) if flat else np.asarray(data45['hands_meanl'], np.float32))


def test_six_components_from_45_rows_is_the_default_model(data45, tmp_path):
    """num_pca_comps=6 on 45-row tables builds the default model byte for byte, in both builders."""
    default = PreparedModel('smplx', syn.make_model('smplx', 0), device='cpu', tensor_cores=False)
    six = PreparedModel('smplx', data45, device='cpu', tensor_cores=False, num_pca_comps=6)
    assert _py_blob(six, tmp_path / 'six.blob') == _py_blob(default, tmp_path / 'default.blob')
    assert default.n_hand == 6 and default.NP == 98
    rc0, raw0 = _c_blob(syn.make_model('smplx', 0))
    rc6, raw6 = _c_blob(data45, num_pca_comps=6)
    assert rc0 == rc6 == 0 and raw0 == raw6
    assert _parse_blob(raw0)[0].n_hand == 6


def test_builders_reject_bad_hand_options(assets):
    """Both builders refuse the same hand descriptions with the same text: hand options on SMPL, a component count
    outside 1..45 (in the C descriptor 0 means 6), and -- unchanged -- the existing over-limit rows."""
    L = _lib.lib()

    def both(mt, data, desc_kw, py_kw, nb=10, ne=10):
        d, keep = model_desc(mt, data, num_betas=nb, num_expression=ne, tensor_cores=False, **desc_kw)
        blob, n = ctypes.c_void_p(), ctypes.c_int64()
        rc = L.bf_model_build_blob(ctypes.byref(d), ctypes.byref(blob), ctypes.byref(n))
        if rc == 0:
            L.bf_blob_free(blob)
        cmsg = None if rc == 0 else _lib.last_error()
        try:
            PreparedModel(mt, data, device='cpu', tensor_cores=False, num_betas=nb, num_expression=ne, **py_kw)
            pmsg = None
        except ValueError as e:
            pmsg = str(e)
        return cmsg, pmsg

    smpl_text = 'hand options (num_pca_comps, use_pca, flat_hand_mean) apply to SMPL-X only'
    range_text = 'num_pca_comps must be between 1 and 45'
    x45 = hand_model(0)
    cases = [('smpl', assets('smpl'), dict(num_pca_comps=12), smpl_text),
             ('smpl', assets('smpl'), dict(use_pca=False), smpl_text),
             ('smpl', assets('smpl'), dict(flat_hand_mean=True), smpl_text),
             ('smplx', x45, dict(num_pca_comps=-1), range_text),
             ('smplx', x45, dict(num_pca_comps=46), range_text),
             ('smplx', x45, dict(num_pca_comps=46, use_pca=False), range_text)]
    for mt, data, kw, text in cases:
        cmsg, pmsg = both(mt, data, kw, kw)
        assert cmsg is not None and cmsg.endswith(text), (mt, kw, cmsg)
        assert pmsg == text, (mt, kw, pmsg)
    # num_pca_comps = 0: the descriptor's default (6), a ValueError in Python
    cmsg, _ = both('smplx', x45, dict(num_pca_comps=0), {})
    assert cmsg is None
    with pytest.raises(ValueError, match=range_text):
        PreparedModel('smplx', x45, device='cpu', tensor_cores=False, num_pca_comps=0)
    # the 100-entry limit is still computed with 6 hand parameters and keeps its text, whatever the hands
    data = syn.make_model('smplx', 0, 16, 4)
    for kw in (dict(num_pca_comps=1), dict(use_pca=False), dict(num_pca_comps=1, face_params=True)):
        cmsg, pmsg = both('smplx', data, kw, kw, nb=16, ne=4)
        assert cmsg.endswith('104 theta entries exceed the limit of 100') and pmsg == '104 theta entries exceed the limit of 100', kw
    cmsg, pmsg = both('smplx', syn.make_model('smplx', 0, 12, 9), dict(use_pca=False), dict(use_pca=False), nb=12, ne=9)
    text = '21 shape coefficients (betas + expression) exceed the limit of 20'
    assert cmsg.endswith(text) and pmsg == text
    # too few component rows: the Python builder says so
    with pytest.raises(ValueError, match='num_pca_comps=12 needs at least 12 hand component rows'):
        PreparedModel('smplx', syn.make_model('smplx', 0), device='cpu', tensor_cores=False, num_pca_comps=12)


def test_widest_row_is_189(data45):
    pm = PreparedModel('smplx', data45, device='cpu', tensor_cores=False, use_pca=False, face_params=True)
    assert pm.NP == 189 == 7 + 63 + 10 + 6 + 90 + 3 + 10


def test_blob_round_trip_hand_model(data45, tmp_path):
    """save_blob stores n_hand, NP and the [n_hand,45] tables; parsing the file gives them back, equal to the C++ blob."""
    for kw, nh in ((dict(num_pca_comps=12, flat_hand_mean=True), 12), (dict(use_pca=False, face_params=True), 45)):
        pm = PreparedModel('smplx', data45, device='cpu', tensor_cores=False, **kw)
        img, arr = _parse_blob(_py_blob(pm, tmp_path / 'm.blob'))
        assert img.n_hand == nh and img.NP == pm.NP
        hr = np.frombuffer(arr['m_hand_r'], np.float32)[:nh * 45].reshape(nh, 45)
        assert np.array_equal(hr, pm._dev['m_hand_r'].numpy())
        rc, raw = _c_blob(data45, **kw)
        img_c, arr_c = _parse_blob(raw)
        assert img_c.n_hand == nh and arr_c['m_hand_r'] == arr['m_hand_r'] and arr_c['m_pose_mean'] == arr['m_pose_mean']


@pytest.mark.parametrize('n,pca,face', [(12, True, False), (1, True, True), (6, False, False), (6, False, True)],
                         ids=['pca12', 'pca1-face', 'aa', 'aa-face'])
def test_pack_split_theta_inverse_hands(data45, n, pca, face):
    pm = PreparedModel('smplx', data45, device='cpu', tensor_cores=False, num_pca_comps=n, use_pca=pca, face_params=face)
    nh, B = n_hand(n, pca), 3
    g = torch.Generator().manual_seed(0)
    r = lambda k: torch.randn(B, k, generator=g)
    parts = dict(transl=r(3), scale=r(1), global_orient=r(3), body_pose=r(63), betas=r(10), leye_pose=r(3),
                 reye_pose=r(3), left_hand_pose=r(nh), right_hand_pose=r(nh))
    if face:
        parts.update(jaw_pose=r(3), expression=r(10))
    th = pm.pack_theta(parts['global_orient'], parts['body_pose'], parts['betas'], transl=parts['transl'],
                       scale=parts['scale'], leye=parts['leye_pose'], reye=parts['reye_pose'], lhand=parts['left_hand_pose'],
                       rhand=parts['right_hand_pose'], jaw=parts.get('jaw_pose'), expression=parts.get('expression'))
    assert th.shape == (B, pm.NP)
    o = 7 + 63 + 10 + 6
    assert torch.equal(th[:, o:o + nh], parts['left_hand_pose']) and torch.equal(th[:, o + nh:o + 2 * nh], parts['right_hand_pose'])
    sp = pm.split_theta(th)
    assert set(sp) == set(parts)
    for k, v in parts.items():
        assert torch.equal(sp[k], v), k
    with pytest.raises(RuntimeError):                   # a hand pose of the wrong width
        pm.pack_theta(parts['global_orient'], parts['body_pose'], parts['betas'], lhand=r(nh + 1))


@pytest.mark.parametrize('dtype', [torch.float32, torch.float64])
def test_identity_projection_is_exact(dtype):
    """The GPU test oracle expands axis-angle hands through the identity table, as the kernels do: x @ I is x itself, bit for
    bit (every product but one is an exact zero), so that oracle is smplx's direct path."""
    g = torch.Generator().manual_seed(3)
    x = torch.randn(64, 45, generator=g, dtype=dtype) * 0.3
    x[0, :5] = torch.tensor([0.0, 1e-30, -1e-30, 1e30, 3.0], dtype=dtype)
    eye = torch.eye(45, dtype=dtype)
    assert torch.equal(torch.einsum('bi,ij->bj', x, eye), x)
