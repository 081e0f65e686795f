"""CPU tests of the host logic: model tables (checked with a numpy interpreter of the tables
against the oracle's joints), theta packing, camera / keypoint packing, the C-ABI library's
exported symbols and struct layouts.  No kernel is launched here."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

from bodyfitting_b200 import _lib, constants as C, synthetic as syn
from bodyfitting_b200.engine import pack_cameras, pack_keypoints
from bodyfitting_b200.model import PreparedModel
from util import make_port, perturbed_params, relerr

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def prepared(assets):
    return {mt: PreparedModel(mt, assets(mt), gmm=assets('gmm'), J_regressor_extra=assets('jx'), device='cpu')
            for mt in ('smpl', 'smplx')}


def _vs_tables(pm, tag):
    return {k[len(tag) + 1:]: v.numpy() for k, v in pm._dev.items() if k.startswith(tag + '_')}


def _interp_joints(t, K_out, yaw, Jtr, verts):
    out = np.zeros((K_out, 3))
    for k in range(K_out):
        kind, src, w = t['kj_kind'][k], t['kj_src'][k], t['kj_w'][k]
        if kind == 0:
            out[k] = Jtr[src[0]]
        elif kind == 1:
            out[k] = sum(verts[src[i]] * w[i] for i in range(3))
        elif kind == 2:
            out[k] = sum(verts[t['dyn_src'][yaw, src[0], i]] * t['dyn_w'][yaw, src[0], i] for i in range(3))
        else:
            r = src[0]
            e0, e1 = t['xr_ptr'][r], t['xr_ptr'][r + 1]
            out[k] = (verts[t['xr_vid'][e0:e1]] * t['xr_w'][e0:e1, None]).sum(0)
    return out


@pytest.mark.parametrize('mt', ['smpl', 'smplx'])
def test_joint_tables_reproduce_oracle_joints(assets, prepared, mt):
    pm = prepared[mt]
    port = make_port(assets, mt, dtype=torch.float64)
    B = 3
    p = perturbed_params(mt, B, seed=9)
    p['global_orient'][1, 1] = 0.6           # exercise a non-zero contour-landmark row
    p['global_orient'][2, 1] = -0.5
    c2ws, Ks = syn.make_cameras(2)
    ev = port.loss_and_grads(p, c2ws, Ks, np.zeros((B, 2, pm.K_used, 3), np.float32))
    verts, joints = ev['model_vertices'], ev['model_joints']
    full = _vs_tables(pm, 'full')
    act = _vs_tables(pm, 'act')
    # chain joints = the oracle's first J pre-map joints; recover them through the mapped list
    Jtr = np.zeros((B, pm.J, 3))
    for k, (kind, src, _) in enumerate(pm.joint_table):
        if kind == 0:
            Jtr[:, src[0]] = joints[:, k]
    fp64 = torch.tensor(ev['full_pose'], dtype=torch.float64)
    for b in range(B):
        yaw = 0
        if mt == 'smplx':
            from oracle import smplx_port as sp
            m = port.model
            idx, _ = sp.find_dynamic_lmk_idx_and_bcoords(torch.zeros(1, pm.V, 3, dtype=torch.float64), fp64[b:b + 1],
                                                         torch.arange(79)[:, None].expand(79, 17), m.dynamic_lmk_bary_coords,
                                                         m.neck_kin_chain)
            yaw = int(idx[0, 0])
        jf = _interp_joints(full, pm.K_out, yaw, Jtr[b], verts[b])
        assert relerr(jf, joints[b]) < 1e-6
        ja = _interp_joints(act, pm.K_used, yaw, Jtr[b], verts[b][pm.active_vids])
        assert relerr(ja, joints[b, :pm.K_used]) < 1e-6
    assert pm.n_act == (11 if mt == 'smpl' else len(pm.active_vids)) and pm.n_act < 600


@pytest.mark.parametrize('mt', ['smpl', 'smplx'])
def test_target_lists_are_the_transpose_of_the_joint_table(prepared, mt):
    """d(sum_k g_k . joint_k)/d(target) through tg_* equals the direct transpose, for every yaw row."""
    pm = prepared[mt]
    for tag, K_out, n in (('act', pm.K_used, pm.n_act), ('full', pm.K_full, pm.V)):
        t = _vs_tables(pm, tag)
        rng = np.random.RandomState(1)
        g = rng.standard_normal((K_out, 3))
        for yaw in ((0, 17, 78) if mt == 'smplx' else (0,)):
            direct = np.zeros((pm.J + n, 3))
            for k in range(K_out):
                kind, src, w = t['kj_kind'][k], t['kj_src'][k], t['kj_w'][k]
                if kind == 0:
                    direct[src[0]] += g[k]
                elif kind == 1:
                    for i in range(3):
                        direct[pm.J + src[i]] += w[i] * g[k]
                elif kind == 2:
                    for i in range(3):
                        direct[pm.J + t['dyn_src'][yaw, src[0], i]] += t['dyn_w'][yaw, src[0], i] * g[k]
                else:
                    r = src[0]
                    for e in range(t['xr_ptr'][r], t['xr_ptr'][r + 1]):
                        direct[pm.J + t['xr_vid'][e]] += t['xr_w'][e] * g[k]
            via = np.zeros_like(direct)
            ptr = t['tg_ptr']
            assert ptr.shape[0] == pm.J + n + 1
            assert (t['tg_a'] < 0).all()                 # static entries only; contour landmarks go through dyn_*
            for tg in np.nonzero(np.diff(ptr))[0]:
                for e in range(ptr[tg], ptr[tg + 1]):
                    via[tg] += t['tg_w'][e] * g[t['tg_k'][e]]
            if 'dyn_k' in t:
                for s, k in enumerate(t['dyn_k']):
                    assert t['kj_kind'][k] == 2 and t['kj_src'][k][0] == s
                    for i in range(3):
                        via[pm.J + t['dyn_src'][yaw, s, i]] += t['dyn_w'][yaw, s, i] * g[k]
            assert np.abs(via - direct).max() < 1e-6


def test_gmm_gemm_operand(prepared):
    """The tensor-core form of the GMM prior: [pose | 1 | 0] @ [P_sym,m | -P_sym,m mu_m | 0]^T == P_sym,m (pose - mu_m)."""
    pm = prepared['smplx']
    bt = (pm._dev['m_gmm_bt_hi'] + pm._dev['m_gmm_bt_lo']).numpy().astype(np.float64)
    hi = pm._dev['m_gmm_bt_hi'].numpy()
    assert bt.shape == (pm.n_gmm * 72, 80) and ((hi.view(np.uint32) & 0x1FFF) == 0).all()     # hi parts are TF32 values
    psym, mu = pm._dev['m_gmm_psym'].numpy().astype(np.float64), pm._dev['m_gmm_mean'].numpy().astype(np.float64)
    x = np.random.RandomState(2).standard_normal(69) * 0.3
    a = np.zeros(80); a[:69] = x; a[69] = 1.0
    y = bt @ a
    for c in range(pm.n_gmm):
        ref = psym[c, :, :69] @ (x - mu[c])
        assert np.abs(y[c * 72:c * 72 + 69] - ref).max() < 1e-5 * max(1.0, np.abs(ref).max())
        assert not y[c * 72 + 69:c * 72 + 72].any()


@pytest.mark.parametrize('mt', ['smpl', 'smplx'])
def test_live_vertex_tables(assets, prepared, mt):
    """Per contour row: the live list is exactly the set of active vertices with a non-zero keypoint gradient, its gather
    lists reproduce the transposed joint table (static entries, then contour entries in slot order), and the restricted
    joint->vertex lists are the skinning weights of the live vertices."""
    pm = prepared[mt]
    t = _vs_tables(pm, 'act')
    W = assets(mt)['weights'][pm.active_vids]
    rows, lmax, n_nz = t['lv_n'].shape[0], t['lv_vid'].shape[1], len(t['jv_nz'])
    assert rows == (79 if mt == 'smplx' else 1) and pm.struct.act.lmax == lmax and pm.struct.act.n_rows == rows
    rng = np.random.RandomState(3)
    g = rng.standard_normal((pm.K_used, 3))
    for a in ((0, 11, 40, 78) if mt == 'smplx' else (0,)):
        direct = np.zeros((pm.n_act, 3))
        for k in range(pm.K_used):
            kind, src, w = t['kj_kind'][k], t['kj_src'][k], t['kj_w'][k]
            if kind == 1:
                for i in range(3):
                    direct[src[i]] += w[i] * g[k]
            elif kind == 2:
                for i in range(3):
                    direct[t['dyn_src'][a, src[0], i]] += t['dyn_w'][a, src[0], i] * g[k]
            elif kind == 3:
                for e in range(t['xr_ptr'][src[0]], t['xr_ptr'][src[0] + 1]):
                    direct[t['xr_vid'][e]] += t['xr_w'][e] * g[k]
        L = int(t['lv_n'][a])
        live = t['lv_vid'][a, :L]
        assert (np.diff(live) > 0).all() and L <= lmax
        touched = set(np.nonzero(np.abs(direct).sum(1))[0])
        assert touched <= set(live.tolist())                 # every vertex with a gradient is live
        via = np.zeros_like(direct)
        for i, v in enumerate(live):
            for e in range(t['lt_ptr'][a, i], t['lt_ptr'][a, i + 1]):
                via[v] += t['lt_w'][e] * g[t['lt_k'][e]]
        assert np.abs(via - direct).max() < 1e-6
        sub = np.zeros((pm.n_act, pm.J))
        for jn, j in enumerate(t['jv_nz']):
            for e in range(t['lj_ptr'][a, jn], t['lj_ptr'][a, jn + 1]):
                sub[live[t['lj_vid'][e]], j] = t['lj_w'][e]          # lj_vid indexes the row's live list
        ref = np.zeros_like(sub)
        ref[live] = W[live]
        assert np.array_equal(sub, ref.astype(np.float32))
        assert t['lj_ptr'].shape == (rows, n_nz + 1)


@pytest.mark.parametrize('mt', ['smpl', 'smplx'])
def test_blend_matrix_and_folded_regressor(assets, prepared, mt):
    pm, data = prepared[mt], assets(mt)
    full = _vs_tables(pm, 'full')
    Bm = full['Bm']
    V, P, NS = pm.V, pm.P, pm.NS
    assert Bm.shape == (pm.Kp, 3 * full['ell_j'].shape[0]) and pm.Kp % 16 == 0
    rng = np.random.RandomState(0)
    pf = np.zeros(pm.Kp); pf[:P] = rng.standard_normal(P) * 0.1; pf[P:P + NS] = rng.standard_normal(NS); pf[P + NS] = 1.0
    vp = (pf @ Bm.astype(np.float64))[:3 * V].reshape(V, 3)
    ref = data['v_template'] + np.einsum('l,vcl->vc', pf[P:P + NS], data['shapedirs'][:, :, :NS].astype(np.float64)) + \
        (pf[:P] @ np.reshape(data['posedirs'], [-1, P]).T.astype(np.float64)).reshape(V, 3)
    assert np.abs(vp - ref).max() < 1e-6
    assert (Bm[:, 3 * V:] == 0).all() and (Bm[P + NS + 1:] == 0).all()
    Jt, Jd = pm._dev['m_Jt'].numpy(), pm._dev['m_Jd'].numpy()
    Jref = data['J_regressor'].astype(np.float64) @ (data['v_template'] + np.einsum('l,vcl->vc', pf[P:P + NS], data['shapedirs'][:, :, :NS]))
    assert np.abs(Jt + Jd @ pf[P:P + NS] - Jref).max() < 1e-6
    # ELL weights reproduce the dense rows; CSR by joint is their transpose
    W = data['weights']
    dense = np.zeros_like(W)
    for k in range(full['ell_j'].shape[1]):
        np.add.at(dense, (np.arange(V), full['ell_j'][:V, k]), full['ell_w'][:V, k])
    assert np.array_equal(dense, W)
    jv = np.zeros_like(W)
    for j in range(pm.J):
        e0, e1 = full['jv_ptr'][j], full['jv_ptr'][j + 1]
        jv[full['jv_vid'][e0:e1], j] = full['jv_w'][e0:e1]
    assert np.array_equal(jv, W)
    act = _vs_tables(pm, 'act')
    assert np.array_equal(act['Bm'][:, :3 * pm.n_act].reshape(pm.Kp, pm.n_act, 3), Bm[:, :3 * V].reshape(pm.Kp, V, 3)[:, pm.active_vids])


def test_kinematic_tables(prepared):
    for mt, depth in (('smpl', 8), ('smplx', 10)):
        pm = prepared[mt]
        par, dep = pm._dev['m_parents'].numpy(), pm._dev['m_depth'].numpy()
        assert pm.max_depth == depth and dep[0] == 0 and par[0] == -1
        lp, lj = pm._dev['m_lvl_ptr'].numpy(), pm._dev['m_lvl_j'].numpy()
        assert lp[0] == 0 and lp[-1] == pm.J and sorted(lj.tolist()) == list(range(pm.J))
        assert all((dep[lj[lp[d]:lp[d + 1]]] == d).all() for d in range(depth + 1))
        assert all(dep[j] == dep[par[j]] + 1 for j in range(1, pm.J))
        cp, ci = pm._dev['m_child_ptr'].numpy(), pm._dev['m_child_idx'].numpy()
        for j in range(pm.J):
            assert sorted(ci[cp[j]:cp[j + 1]]) == [c for c in range(1, pm.J) if par[c] == j]


def test_theta_pack_roundtrip(prepared):
    for mt in ('smpl', 'smplx'):
        pm = prepared[mt]
        B = 4
        p = perturbed_params(mt, B, seed=2)
        T = lambda k: torch.as_tensor(p[k]) if k in p else None
        th = pm.pack_theta(T('global_orient'), T('body_pose'), T('betas'), transl=T('global_transl'), scale=T('body_scale'),
                           leye=T('leye_pose'), reye=T('reye_pose'), lhand=T('left_hand_pose'), rhand=T('right_hand_pose'))
        assert th.shape == (B, pm.NP) and pm.NP == (98 if mt == 'smplx' else 86)
        s = pm.split_theta(th)
        assert np.array_equal(s['body_pose'].numpy(), p['body_pose']) and np.array_equal(s['betas'].numpy(), p['betas'])
        assert np.array_equal(s['scale'].numpy(), p['body_scale'])
        if mt == 'smplx':
            assert np.array_equal(s['right_hand_pose'].numpy(), p['right_hand_pose'])


def test_smpl_to_openpose_tables():
    a = C.smpl_to_openpose('smplx', use_hands=True, use_face=True, use_face_contour=True, openpose_format='coco25')
    assert len(a) == 135 and list(a[:3]) == [55, 12, 17] and a[25] == 20 and a[29] == 66 and a[46] == 21 and a[-1] == 143
    assert list(C.smpl_to_openpose('smpl', openpose_format='coco25')) == [24, 12, 17, 19, 21, 16, 18, 20, 0, 2, 5, 8, 1, 4, 7] + list(range(25, 35))
    assert len(C.smpl_to_openpose('smplh', use_hands=True, openpose_format='coco19')) == 19 + 42
    assert len(C.SPIN_JOINT_MAP) == 49 and C.SPIN_JOINT_MAP[27] == 45
    with pytest.raises(ValueError):
        C.smpl_to_openpose('foo')


def test_pack_cameras_and_keypoints():
    c2ws, Ks = syn.make_cameras(3)
    M = pack_cameras(list(c2ws), list(Ks)).reshape(3, 3, 4)
    X = np.array([0.1, -0.2, 0.05, 1.0])
    for v in range(3):
        w2c = np.linalg.inv(c2ws[v].astype(np.float64))
        ref = Ks[v] @ (w2c[:3] @ X)
        assert np.abs(M[v] @ X - ref).max() < 1e-4
    kp = np.random.RandomState(0).rand(2, 3, 135, 3).astype(np.float32)
    out = pack_keypoints(kp, True)
    assert out.shape == (2, 135, 3, 3) and out.is_contiguous()         # device layout is joint-major [B,K,Nv,3]
    out = out.permute(0, 2, 1, 3).numpy()
    assert np.allclose(out[..., :25, 2], kp[..., :25, 2] ** 2)
    assert np.allclose(out[..., 30, 2], (kp[..., 25:46, 2] ** 2).sum(-1))
    assert np.allclose(out[..., 100, 2], (kp[..., 67:, 2] ** 2).sum(-1), rtol=1e-5)
    assert np.array_equal(out[..., :2], kp[..., :2])


def test_openpose_dict_roundtrip():
    kp = np.random.RandomState(1).rand(8, 135, 3).astype(np.float32)
    views = syn.keypoints_to_openpose(kp, 'smplx')
    assert views[0]['face'].shape == (70, 3) and views[0]['hand_left'].shape == (21, 3)
    assert np.array_equal(syn.openpose_to_keypoints(views, 'smplx'), kp)
    views[3] = None
    del views[4]['hand_right']
    back = syn.openpose_to_keypoints(views, 'smplx')
    assert (back[3] == 0).all() and (back[4, 46:67] == 0).all() and np.array_equal(back[4, :46], kp[4, :46])


def test_library_loads_and_exports_every_declared_symbol():
    L = _lib.lib()
    hdr = open(os.path.join(ROOT, 'include', 'bodyfit_b200.h')).read() + open(os.path.join(ROOT, 'include', 'bodyfit_b200_ops.h')).read() + \
        open(os.path.join(ROOT, 'include', 'bodyfit_b200_grid.h')).read() + open(os.path.join(ROOT, 'include', 'bodyfit_b200_mask.h')).read()
    declared = set(re.findall(r'^(?:int|int64_t|void|const char\*)\s+(bf_[a-z0-9_]+)\s*\(', hdr, re.M))
    assert declared, 'no declarations parsed'
    for name in sorted(declared):
        assert hasattr(L, name), 'symbol %s declared in the header but not exported' % name
    assert declared == set(_lib.EXPORTED) | set(_lib.EXPORTED_OPS) | set(_lib.EXPORTED_GRID) | set(_lib.EXPORTED_MASK)
    assert L.bf_abi_version() == _lib.ABI_VERSION
    for i, st in enumerate((_lib.BfVSet, _lib.BfModel, _lib.BfFrames, _lib.BfGrid, _lib.BfSmpld, _lib.BfMask)):
        assert L.bf_sizeof(i) == ctypes.sizeof(st), st.__name__


def test_no_gpu_means_loud_failure():
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    with pytest.raises(_lib.BodyfitError):
        _lib.require_device()
    from bodyfitting_b200.smplify.smplify import SMPLify
    fit = SMPLify(smpl_type='smpl', num_iters=2, model_data=syn.make_model('smpl', 0), gmm=syn.make_gmm(0), device='cpu')
    kp = np.zeros((1, 2, 25, 3), np.float32)
    c2ws, Ks = syn.make_cameras(2)
    with pytest.raises(_lib.BodyfitError):
        fit((np.zeros((1, 10), np.float32), np.zeros((1, 72), np.float32)), list(c2ws), list(Ks), kp, None)


def test_product_never_imports_oracle():
    pkg = os.path.join(ROOT, 'bodyfitting_b200')
    for dp, _, fns in os.walk(pkg):
        for fn in fns:
            if fn.endswith('.py'):
                src = open(os.path.join(dp, fn)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle', src, re.M), fn


def test_openpose_json_and_obj_formats(tmp_path):
    """load_openpose on an OpenPose-1.3 style file (25x3 body, confidences may exceed 1, empty hand arrays, a second
    weaker person), OBJ writer/reader round trip, parameter .npy schema."""
    import json
    from bodyfitting_b200.smplify.body_fitting import write_result
    from bodyfitting_b200.utils.io_utils import load_obj_mesh, load_openpose, save_obj_mesh
    rng = np.random.RandomState(0)
    body = np.concatenate([rng.rand(25, 2) * 500, rng.rand(25, 1) * 3.5], 1)
    hand = np.concatenate([rng.rand(21, 2) * 500, rng.rand(21, 1)], 1)
    doc = {'version': 1.3, 'people': [
        {'person_id': [-1], 'pose_keypoints_2d': (body * 0.1).reshape(-1).tolist(), 'face_keypoints_2d': [],
         'hand_left_keypoints_2d': [], 'hand_right_keypoints_2d': []},
        {'person_id': [-1], 'pose_keypoints_2d': body.reshape(-1).tolist(), 'face_keypoints_2d': np.zeros(210).tolist(),
         'hand_left_keypoints_2d': hand.reshape(-1).tolist(), 'hand_right_keypoints_2d': [], 'pose_keypoints_3d': []}]}
    fn = tmp_path / 'f_keypoints.json'
    fn.write_text(json.dumps(doc))
    d = load_openpose(str(fn))
    assert set(d) == {'pose', 'hand_left'} and d['pose'].shape == (25, 3) and d['hand_left'].shape == (21, 3)
    assert np.allclose(d['pose'], body)                      # the stronger person; all-zero face dropped
    assert len(load_openpose(str(fn), only_one=False)) == 2
    (tmp_path / 'empty.json').write_text(json.dumps({'people': []}))
    assert load_openpose(str(tmp_path / 'empty.json')) is None
    v = rng.rand(10, 3); f = rng.randint(0, 10, (6, 3))
    write_result(str(tmp_path / 'out'), 'smpl', dict(vertices=v, faces=f, pose=np.zeros(69)))
    v2, f2 = load_obj_mesh(str(tmp_path / 'out' / 'smpl.obj'))
    assert np.abs(v2 - v).max() < 1e-4 and np.array_equal(f2, f)
    back = np.load(str(tmp_path / 'out' / 'smpl_parameter.npy'), allow_pickle=True).item()
    assert set(back) == {'vertices', 'faces', 'pose'}
    (tmp_path / 'quad.obj').write_text('v 0 0 0\nv 1 0 0\nv 1 1 0\nv 0 1 0\nvn 0 0 1\nf 1/1/1 2/1/1 3/1/1 4/1/1\n')
    _, fq = load_obj_mesh(str(tmp_path / 'quad.obj'))
    assert fq.tolist() == [[0, 1, 2], [0, 2, 3]]


def test_rotation_matrix_to_axis_angle():
    from scipy.spatial.transform import Rotation as Rot
    from bodyfitting_b200.utils.geometry import convert_hom_to_angle, rotation_matrix_to_angle_axis
    rng = np.random.RandomState(3)
    rv = rng.randn(200, 3) * 1.2
    rv[0] = 0.0                                              # identity (the reference patches a NaN here)
    rv[1] = [np.pi - 1e-4, 0, 0]                             # near pi
    R = torch.tensor(Rot.from_rotvec(rv).as_matrix(), dtype=torch.float64)
    out = rotation_matrix_to_angle_axis(R).numpy()
    ref = Rot.from_matrix(R.numpy()).as_rotvec()
    assert np.abs(out - ref).max() < 1e-8 and (out[0] == 0).all()
    pose = convert_hom_to_angle(R[:48].reshape(2, 24, 3, 3).float(), 2)
    assert pose.shape == (2, 72) and np.abs(pose.numpy().reshape(-1, 3) - ref[:48]).max() < 1e-5


def test_staggered_ranges_partition_properties():
    """Part layout of large batches (engine.staggered_ranges): a partition of [0, B) into consecutive ranges of
    non-increasing size, GEMM-tile aligned, for every taper / lead setting."""
    from bodyfitting_b200.engine import staggered_ranges
    for B in (1, 100, 2047, 4096, 10000, 16384, 100001):
        for n_parts in (1, 2, 4, 6):
            for taper in (0.0, 0.5, 1.5):
                for lead in (0, 512):
                    rs = staggered_ranges(B, n_parts, taper=taper, lead=lead)
                    assert rs[0][0] == 0 and rs[-1][1] == B
                    assert all(rs[i][1] == rs[i + 1][0] for i in range(len(rs) - 1))
                    assert all(hi > lo for lo, hi in rs)
                    body = rs[1:] if (lead and len(rs) > 1 and rs[0][1] == lead) else rs
                    sizes = [hi - lo for lo, hi in body]
                    assert all(sizes[i] >= sizes[i + 1] - 128 for i in range(len(sizes) - 1))
                    assert all(lo % 128 == 0 for lo, _ in rs)
                    assert len(rs) <= n_parts + (1 if lead else 0)
    assert staggered_ranges(10000, 4) == [(0, 3584), (3584, 6400), (6400, 8576), (8576, 10000)]


def test_reference_mesh_grid_wrapper_binds_to_our_module():
    """The reference's own utils/mesh_grid_searcher.py imports `mesh_grid` by name and pulls its six native functions
    (mesh_grid_searcher.py:2); with bodyfitting_b200.compat.mesh_grid registered under that name the UNMODIFIED file imports
    and its classes resolve.  (Running them needs a GPU: tests/test_gpu_grid.py drives the same call protocol.)"""
    import importlib.util
    import sys
    import types
    from oracle import ref_harness as rh
    if not rh.available():
        pytest.skip('no reference checkout (BODYFIT_REFERENCE, or reference/ beside the repository)')
    ref = os.path.join(rh.REFERENCE_ROOT, 'utils', 'mesh_grid_searcher.py')
    import bodyfitting_b200.compat.mesh_grid as mg
    saved = {k: sys.modules.get(k) for k in ('mesh_grid', 'trimesh')}
    sys.modules['mesh_grid'] = mg
    sys.modules['trimesh'] = types.ModuleType('trimesh')            # imported by the wrapper, never used on this path
    try:
        spec = importlib.util.spec_from_file_location('ref_mesh_grid_searcher', ref)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        assert hasattr(mod, 'MeshGridSearcher') and hasattr(mod, 'SurfaceNearest')
        for name in ('insert_grid_surface', 'cumsum', 'search_nearest_point', 'search_inside_mesh', 'search_intersect',
                     'search_nearest_point_backward'):
            assert getattr(mod, name) is getattr(mg, name)
    finally:
        for k, v in saved.items():
            if v is None:
                sys.modules.pop(k, None)
            else:
                sys.modules[k] = v


def test_init_conversion_matches_reference_converter():
    """(f)3: rotmat -> axis-angle and the world transform of the root orientation against the REFERENCE'S OWN
    utils/geometry.py:331-493 + smplify/body_fitting.py:70-73 -- committed golden (tests/golden/make_golden_aux.py) and, where
    BODYFIT_REFERENCE names a reference checkout, the live reference functions."""
    from bodyfitting_b200.utils.geometry import convert_hom_to_angle, world_init_from_camera_rotmat
    g = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'reference_init_conversion.npz'))
    R = torch.tensor(g['rotmat'])
    pose = convert_hom_to_angle(R, 2).numpy()
    assert pose.shape == g['pose'].shape
    # axis-angle is unique up to fp32 conversion noise except at angle ~ pi (sign of the axis): compare as rotations
    from scipy.spatial.transform import Rotation as Rot
    def same_rot(a, b):
        return np.abs(Rot.from_rotvec(a.reshape(-1, 3)).as_matrix() - Rot.from_rotvec(b.reshape(-1, 3)).as_matrix()).max()
    assert same_rot(pose, g['pose']) < 2e-6
    far_from_pi = np.linalg.norm(g['pose'].reshape(-1, 3), axis=1) < 3.0
    assert np.abs(pose.reshape(-1, 3)[far_from_pi] - g['pose'].reshape(-1, 3)[far_from_pi]).max() < 2e-5
    assert (pose.reshape(-1, 3)[0] == 0).all() and (g['pose'].reshape(-1, 3)[0] == 0).all()       # identity
    before = R[:1].clone()
    pw = world_init_from_camera_rotmat(R[:1], g['c2w']).numpy()
    assert torch.equal(R[:1], before)                                  # input not modified
    assert same_rot(pw, g['pose_world']) < 2e-6 and np.abs(pw[0, 3:] - pose[0, 3:]).max() < 1e-6   # only the root changes
    assert np.abs(pw[0, :3] - pose[0, :3]).max() > 0.1
    from oracle import ref_harness as rh
    if rh.available():
        rh.load_reference()
        import utils.geometry as rg
        live = rg.convert_hom_to_angle(R, 2, torch.device('cpu')).numpy()
        assert np.array_equal(live, g['pose'])


def test_load_openpose_on_the_reference_fixture():
    """utils/io_utils.py:138-183 load_openpose on the reference's only real-data fixture (openpose/test.json, an OpenPose 1.3
    output with one person and confidences > 1): same dict as the reference's own parser (committed golden)."""
    from bodyfitting_b200.utils.io_utils import load_openpose
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
    got = load_openpose(os.path.join(here, 'openpose_test.json'))
    want = np.load(os.path.join(here, 'reference_openpose_parse.npz'))
    assert set(got) == set(want.files)
    for k in want.files:
        assert np.asarray(got[k]).shape == want[k].shape and np.allclose(np.asarray(got[k], dtype=np.float64), want[k], rtol=0, atol=1e-6), k


def test_loader_accepts_official_model_file_layout(assets, tmp_path):
    """Official SMPL / SMPL-X files carry no 'extra_vids' (smplx hard-codes the vertex ids of the 21 picked joints) and SMPL-X
    stores 300 shape + 100 expression directions (expression = columns 300..309, not 10..19).  A dict / .npz laid out like
    that must give exactly the tables of the synthetic layout, in the product loader AND in the oracle's restatement; the
    gendered file is resolved from the data folder (a missing gender falls back to NEUTRAL with a warning, never silently)."""
    import warnings
    from bodyfitting_b200 import constants as K
    from bodyfitting_b200.model import PreparedModel, load_model_data
    from oracle import smplx_port as sp
    for mt in ('smpl', 'smplx'):
        d = dict(assets(mt))
        assert list(d['extra_vids']) == K.EXTRA_VIDS[mt] == sp._EXTRA_VIDS[mt]      # product and oracle tables agree
        off = {k: v for k, v in d.items() if k != 'extra_vids'}
        if mt == 'smplx':
            rng = np.random.RandomState(0)
            sd = rng.standard_normal(d['shapedirs'].shape[:2] + (400,)).astype(np.float32)      # junk everywhere ...
            sd[:, :, :10] = d['shapedirs'][:, :, :10]                                            # ... except the columns in use
            sd[:, :, 300:310] = d['shapedirs'][:, :, 10:20]
            off['shapedirs'] = sd
        a = PreparedModel(mt, d, gmm=assets('gmm'), J_regressor_extra=assets('jx'), device='cpu', tensor_cores=False)
        b = PreparedModel(mt, off, gmm=assets('gmm'), J_regressor_extra=assets('jx'), device='cpu', tensor_cores=False)
        assert set(a._dev) == set(b._dev)
        for k in a._dev:
            assert torch.equal(a._dev[k], b._dev[k]), (mt, k)
        # the oracle's restatement reads the same layout
        la = sp.SMPLXLayer(d) if mt == 'smplx' else sp.SMPLLayer(d)
        lb = sp.SMPLXLayer(off) if mt == 'smplx' else sp.SMPLLayer(off)
        assert torch.equal(la.extra_joints_idxs, lb.extra_joints_idxs)
        if mt == 'smplx':
            assert torch.equal(la.expr_dirs, lb.expr_dirs)
    # gender resolution in a reference-style data folder
    folder = tmp_path / 'data' / 'smpl'
    folder.mkdir(parents=True)
    np.savez(str(folder / 'SMPL_NEUTRAL.npz'), **{k: v for k, v in assets('smpl').items() if k not in ('extra_vids', 'model_type')})
    np.savez(str(folder / 'SMPL_FEMALE.npz'), **{k: (v * 2 if k == 'v_template' else v) for k, v in assets('smpl').items()
                                                  if k not in ('extra_vids', 'model_type')})
    fem = load_model_data(str(tmp_path / 'data'), 'smpl', 'female')
    assert np.array_equal(fem['v_template'], assets('smpl')['v_template'] * 2)
    with warnings.catch_warnings(record=True) as w:
        warnings.simplefilter('always')
        male = load_model_data(str(tmp_path / 'data'), 'smpl', 'male')
    assert np.array_equal(male['v_template'], assets('smpl')['v_template']) and any('NEUTRAL' in str(x.message) for x in w)


# ---- bf_model_create: the C++ table builder against the Python one --------------------------------------------------
_FLOAT_FIELDS = {'Jt', 'Jd', 'pose_mean', 'hand_l', 'hand_r', 'gmm_mean', 'gmm_psym', 'gmm_logw', 'gmm_bt_hi', 'gmm_bt_lo',
                 'Bm', 'ell_w', 'jv_w', 'kj_w', 'dyn_w', 'tg_w', 'xr_w', 'Bt_hi', 'Bt_lo', 'Bm_hi', 'Bm_lo', 'lt_w', 'lj_w'}


def _parse_blob(raw):
    """blob bytes -> (BfModel image, {'m_x' / 'full_x' / 'act_x': raw bytes of the array, padding included})"""
    assert raw[:8] == b'BFMODEL1'
    abi, sz = np.frombuffer(raw[8:16], np.int32)
    assert abi == _lib.ABI_VERSION and sz == ctypes.sizeof(_lib.BfModel)
    img = _lib.BfModel.from_buffer_copy(raw[16:16 + sz])
    total = int(np.frombuffer(raw[16 + sz:24 + sz], np.int64)[0])
    sec = raw[24 + sz:24 + sz + total]
    offs = {}
    for tag, st in (('m', img), ('full', img.full), ('act', img.act)):
        for name, typ in st._fields_:
            if typ is _lib._fp and getattr(st, name):
                offs[tag + '_' + name] = getattr(st, name) - 1
    ends = sorted(set(offs.values()) | {total})
    return img, {k: sec[o:ends[ends.index(o) + 1]] for k, o in offs.items()}


# other shape-space sizes: (model type, num_betas, num_expression), the kid template adds one beta.  The same grid as
# tests/test_gpu_model_shapes.py: 1 / 16 / 17 / 20 betas, NS = 20 with NP = 100, no expression at all, Kp = 496 (NS <= 9)
_COUNTS = {'smpl_nb1': ('smpl', 1, 0), 'smpl_nb16': ('smpl', 16, 0), 'smpl_nb17': ('smpl', 17, 0), 'smpl_nb20': ('smpl', 20, 0),
           'smpl_kid_nb16': ('smpl', 16, 0), 'smplx_nb12_ne8': ('smplx', 12, 8), 'smplx_nb10_ne0': ('smplx', 10, 0),
           'smplx_nb5_ne4': ('smplx', 5, 4), 'smplx_nb1_ne0': ('smplx', 1, 0)}


@pytest.mark.parametrize('case', ['smpl', 'smplx', 'smpl_kid', 'smpl_plain', 'smplx_official'] + list(_COUNTS))
def test_bf_model_create_tables_match_python_builder(assets, case, tmp_path):
    """include/bodyfit_b200.h: bf_model_build_blob (what bf_model_create uploads) builds the SAME tables from the raw model
    arrays as bodyfitting_b200.model.PreparedModel: index tables bit for bit; folded / inverted float tables to rounding --
    for the default shape space and for other numbers of betas / expression coefficients."""
    mt = 'smplx' if case.startswith('smplx') else 'smpl'
    model = assets(mt)
    counts = {}
    if case in _COUNTS:
        _, nb, ne = _COUNTS[case]
        model = syn.make_model(mt, 0, nb, ne)
        counts = dict(num_betas=nb, num_expression=ne)
    if case == 'smplx_official':
        # the layout of the official files: no 'extra_vids' key (smplx hard-codes the ids), 300 shape + 100 expression directions
        model = {k: v for k, v in model.items() if k != 'extra_vids'}
        sd = np.asarray(model['shapedirs'], np.float32)
        wide = np.zeros(sd.shape[:2] + (400,), np.float32)
        wide[:, :, :10], wide[:, :, 300:310] = sd[:, :, :10], sd[:, :, 10:20]
        wide[:, :, 10:300] = 1e-3                                      # directions the fit must not pick up
        model['shapedirs'] = wide
    kid = case.startswith('smpl_kid')
    kw = dict(kid_template=syn.make_kid_template(0)) if kid else {}
    jx = assets('jx') if (mt == 'smpl' and case != 'smpl_plain') else None
    gmm = None if case == 'smpl_plain' else assets('gmm')
    pm = PreparedModel(mt, model, gmm=gmm, J_regressor_extra=jx, device='cpu', tensor_cores=True,
                       age='kid' if kid else 'adult', **kw, **counts)
    if counts:
        assert pm.NB == counts['num_betas'] + kid and pm.NS == pm.NB + (counts['num_expression'] if mt == 'smplx' else 0)
    path = pm.save_blob(str(tmp_path / 'py.blob'))
    img_p, arr_p = _parse_blob(open(path, 'rb').read())
    from bodyfitting_b200.model import model_desc
    d, keep = model_desc(mt, model, gmm=gmm, J_regressor_extra=jx, tensor_cores=True, **kw, **counts)
    assert (d.extra_vids is None) == (case == 'smplx_official')
    blob, n = ctypes.c_void_p(), ctypes.c_int64()
    rc = _lib.lib().bf_model_build_blob(ctypes.byref(d), ctypes.byref(blob), ctypes.byref(n))
    assert rc == 0, _lib.last_error()
    raw = ctypes.string_at(blob, n.value)
    _lib.lib().bf_blob_free(blob)
    img_c, arr_c = _parse_blob(raw)
    # scalar members
    for tag, a, b in (('m', img_p, img_c), ('full', img_p.full, img_c.full), ('act', img_p.act, img_c.act)):
        for name, typ in a._fields_:
            if typ is _lib._i32 and not name.startswith('_pad'):
                assert getattr(a, name) == getattr(b, name), (tag, name)
    assert set(arr_p) == set(arr_c), set(arr_p) ^ set(arr_c)
    worst = {}
    for key in sorted(arr_p):
        a, b = arr_p[key], arr_c[key]
        assert len(a) == len(b), (key, len(a), len(b))
        name = key.split('_', 1)[1]
        if name in _FLOAT_FIELDS:
            fa, fb = np.frombuffer(a, np.float32), np.frombuffer(b, np.float32)
            scale = max(1e-30, float(np.abs(fa).max()))
            worst[key] = float(np.abs(fa - fb).max()) / scale
        else:
            assert a == b, key
    # float tables: identical except where a reduction is folded (fp64 accumulation order) or a matrix inverted
    # (numpy inverts the float32 covariances in float32, the C++ builder in float64): measured <= 2e-7 / 3e-5
    loose = {k for k in worst if 'gmm' in k}
    assert max([v for k, v in worst.items() if k not in loose] + [0.0]) < 1e-6, {k: v for k, v in worst.items() if v > 0}
    assert max([worst[k] for k in loose] + [0.0]) < 1e-3, {k: worst[k] for k in loose}
    print(case, 'largest relative differences:', {k: '%.1e' % v for k, v in worst.items() if v > 0})


def test_bf_model_create_rejects_bad_descriptions(assets):
    """bf_model_build_blob fails loudly (negative code + bf_last_error) instead of building tables from inconsistent input."""
    from bodyfitting_b200.model import model_desc
    L = _lib.lib()

    def build(d):
        blob, n = ctypes.c_void_p(), ctypes.c_int64()
        rc = L.bf_model_build_blob(ctypes.byref(d), ctypes.byref(blob), ctypes.byref(n))
        if rc == 0:
            L.bf_blob_free(blob)
        return rc, _lib.last_error()

    rc, msg = build(_lib.BfModelDesc())
    assert rc != 0 and 'required' in msg
    # kinematic tree out of order
    d, keep = model_desc('smpl', assets('smpl'))
    par = np.ascontiguousarray(np.asarray(assets('smpl')['kintree_table'])[0].astype(np.int32))
    par[3] = 7
    d.parents = par.ctypes.data
    rc, msg = build(d)
    assert rc != 0 and 'topologically' in msg
    # SMPL-X without its landmark tables
    d, keep = model_desc('smplx', assets('smplx'))
    d.lmk_faces_idx = None
    rc, msg = build(d)
    assert rc != 0 and 'landmark' in msg
    # a landmark face index beyond the face list
    d, keep = model_desc('smplx', assets('smplx'))
    lf = np.ascontiguousarray(np.asarray(assets('smplx')['lmk_faces_idx']).astype(np.int32))
    lf[5] = d.F
    d.lmk_faces_idx = lf.ctypes.data
    rc, msg = build(d)
    assert rc != 0 and 'outside the face list' in msg
    # vertex-picked joint outside the mesh
    d, keep = model_desc('smpl', assets('smpl'))
    bad = np.full(21, 10 ** 6, np.int32)
    d.extra_vids, d.n_extra_vids = bad.ctypes.data, 21
    rc, msg = build(d)
    assert rc != 0 and 'outside the mesh' in msg
    # a covariance that is not positive definite
    g = {k: np.array(v, dtype=np.float32) for k, v in assets('gmm').items()}
    g['covars'][0] = -np.eye(69, dtype=np.float32)
    d, keep = model_desc('smpl', assets('smpl'), gmm=g)
    rc, msg = build(d)
    assert rc != 0 and 'positive definite' in msg
    # the kid template belongs to SMPL
    d, keep = model_desc('smplx', assets('smplx'))
    kid = np.zeros((d.V, 3), np.float32)
    d.kid_template = kid.ctypes.data
    rc, msg = build(d)
    assert rc != 0 and 'SMPL only' in msg


def test_builders_agree_on_shape_space_limits(assets):
    """Both model builders (bf_model_build_blob in C++ and PreparedModel in Python) reject, with the same text, shape spaces the
    kernels cannot run: more than 20 betas + expression coefficients (BF_MAXNS), more than 100 theta entries (BF_MAXNP), or
    fewer than one beta -- when the model is built, not at its first launch.  Zero expression coefficients are honoured by
    both (SMPL-X without expression directions)."""
    from bodyfitting_b200.model import model_desc
    L = _lib.lib()

    def both(mt, nb, ne, **kw):
        data = syn.make_model(mt, 0, max(nb, 1), max(ne, 0))
        d, keep = model_desc(mt, data, num_betas=nb, num_expression=ne, **kw)
        blob, n = ctypes.c_void_p(), ctypes.c_int64()
        rc = L.bf_model_build_blob(ctypes.byref(d), ctypes.byref(blob), ctypes.byref(n))
        img = None
        if rc == 0:
            img, _ = _parse_blob(ctypes.string_at(blob, n.value))
            L.bf_blob_free(blob)
        c = (rc, None if rc == 0 else _lib.last_error(), img)
        try:
            pm = PreparedModel(mt, data, device='cpu', tensor_cores=False, num_betas=nb, num_expression=ne,
                               age='kid' if 'kid_template' in kw else 'adult', **kw)
            return c, (None, pm)
        except ValueError as e:
            return c, (str(e), None)

    kid = dict(kid_template=syn.make_kid_template(0))
    for mt, nb, ne, kw, text in (('smplx', 16, 4, {}, '104 theta entries exceed the limit of 100'),      # NS = 20, NP = 104
                                 ('smplx', 12, 9, {}, '21 shape coefficients (betas + expression) exceed the limit of 20'),
                                 ('smpl', 21, 0, {}, '21 shape coefficients (betas + expression) exceed the limit of 20'),
                                 ('smpl', 20, 0, kid, '21 shape coefficients (betas + expression) exceed the limit of 20'),
                                 ('smpl', 0, 0, {}, 'num_betas must be at least 1 and num_expression not negative'),
                                 ('smplx', 0, 10, {}, 'num_betas must be at least 1 and num_expression not negative'),
                                 ('smplx', 10, -1, {}, 'num_betas must be at least 1 and num_expression not negative')):
        (rc, cmsg, _), (pmsg, _) = both(mt, nb, ne, **kw)
        assert rc != 0 and cmsg.endswith(text), (mt, nb, ne, cmsg)
        assert pmsg == text, (mt, nb, ne, pmsg)
    # the largest accepted shape spaces, and SMPL-X without expression: both builders take the counts as given
    for mt, nb, ne, kw, ns, np_ in (('smplx', 12, 8, {}, 20, 100), ('smpl', 20, 0, {}, 20, 96), ('smpl', 19, 0, kid, 20, 96),
                                    ('smplx', 10, 0, {}, 10, 98), ('smplx', 1, 0, {}, 1, 89)):
        (rc, cmsg, img), (pmsg, pm) = both(mt, nb, ne, **kw)
        assert rc == 0 and pmsg is None, (mt, nb, ne, cmsg, pmsg)
        assert (img.NS, img.NP) == (pm.NS, pm.NP) == (ns, np_), (mt, nb, ne)
