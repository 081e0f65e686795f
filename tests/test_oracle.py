"""CPU tests of the oracle (no GPU): the standalone port against the committed golden vectors
(tests/golden: produced by the verbatim reference; the kid and silhouette paths pinned where the live
tests held the port equal to it), against the verbatim reference itself where a checkout of it is at
hand (BODYFIT_REFERENCE, or reference/ beside the repository), fp32 vs fp64, batched vs per-frame, and
finite differences of the LBS restatement."""
import os

import numpy as np
import pytest
import torch

from bodyfitting_b200 import synthetic as syn
from oracle import fit_port as fp, ref_harness as rh, smplx_port as sp
from util import gt_param_dict, make_port, make_scene, relerr

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


@pytest.mark.parametrize('mt', ['smpl', 'smplx'])
def test_port_matches_golden_reference(assets, mt):
    g = np.load(os.path.join(GOLD, 'reference_fit_%s.npz' % mt))
    port = make_port(assets, mt)
    views = syn.keypoints_to_openpose(g['kp'][0], mt)
    if mt == 'smpl':
        views[2] = None
    res, trace = port.fit_frame(g['init_betas'][0], g['init_pose'][0], g['c2ws'], g['Ks'], views, num_iters=100)
    assert relerr(trace, g['trace']) < 1e-5
    for k in ('pose', 'betas', 'global_orient', 'global_transl', 'scale', 'joints', 'vertices', 'full_pose'):
        assert np.abs(res[k] - g['out_' + k]).max() < 1e-4, k


def test_golden_covers_missing_view_and_quirks():
    g = np.load(os.path.join(GOLD, 'reference_fit_smpl.npz'))
    assert (g['kp'][0, 2] == 0).all()              # the None view
    assert g['trace'].shape == (100,) and g['terms'].shape == (100, 4)
    assert g['out_joints'].shape == (49, 3) and g['out_vertices'].shape == (6890, 3)
    gx = np.load(os.path.join(GOLD, 'reference_fit_smplx.npz'))
    assert gx['out_joints'].shape == (135, 3) and gx['out_full_pose'].shape == (165,)


@pytest.mark.skipif(not rh.available(), reason='no reference checkout (BODYFIT_REFERENCE, or reference/ beside the repository)')
@pytest.mark.parametrize('mt,nv', [('smpl', 4), ('smplx', 8)])
def test_port_bit_exact_vs_verbatim_reference(assets, tmp_path, mt, nv):
    syn.write_data_dir(str(tmp_path / 'data'), seed=0, model_types=(mt,))
    port = make_port(assets, mt)
    sc = make_scene(port, mt, 1, nv, seed=31)
    views = syn.keypoints_to_openpose(sc['kp'][0], mt)
    N = 25
    res, trace, terms, _ = rh.run_reference_fit(str(tmp_path), mt, sc['init_betas'][0], sc['init_pose'][0], sc['c2ws'],
                                                sc['Ks'], views, num_iters=N)
    resp, trp = port.fit_frame(sc['init_betas'][0], sc['init_pose'][0], sc['c2ws'], sc['Ks'], views, num_iters=N)
    assert np.array_equal(np.asarray(trace), np.asarray(trp))
    for k in ('pose', 'betas', 'global_orient', 'global_transl', 'scale', 'joints', 'vertices', 'full_pose'):
        assert np.array_equal(res[k], resp[k]), k


@pytest.mark.skipif(not rh.available(), reason='no reference checkout (BODYFIT_REFERENCE, or reference/ beside the repository)')
def test_kid_model_port_bit_exact_vs_verbatim_reference(assets, tmp_path):
    """age='kid' (smplify/smplify.py:50-56,112-115): the verbatim reference builds SMPL(age='kid', kid_template_path=
    config.SMIL_MODEL_DIR) and starts from 11 zero betas; the restatement follows it bit for bit (the kid shape space itself is
    smplx's, restated in oracle/smplx_port.py)."""
    syn.write_data_dir(str(tmp_path / 'data'), seed=0, model_types=('smpl',))
    kid = syn.make_kid_template(0)
    port = fp.FitPort('smpl', assets('smpl'), assets('gmm'), assets('jx'), age='kid', kid_template=kid)
    adult = make_port(assets, 'smpl')
    sc = make_scene(adult, 'smpl', 1, 4, seed=37)
    views = syn.keypoints_to_openpose(sc['kp'][0], 'smpl')
    N = 15
    res, trace, terms, _ = rh.run_reference_fit(str(tmp_path), 'smpl', sc['init_betas'][0], sc['init_pose'][0], sc['c2ws'],
                                                sc['Ks'], views, num_iters=N, age='kid')
    resp, trp = port.fit_frame(sc['init_betas'][0], sc['init_pose'][0], sc['c2ws'], sc['Ks'], views, num_iters=N)
    assert res['betas'].shape == (11,) and np.abs(res['betas']).max() > 0
    assert np.array_equal(np.asarray(trace), np.asarray(trp))
    for k in ('pose', 'betas', 'global_orient', 'global_transl', 'scale', 'joints', 'vertices'):
        assert np.array_equal(res[k], resp[k]), k


@pytest.mark.skipif(not rh.available(), reason='no reference checkout (BODYFIT_REFERENCE, or reference/ beside the repository)')
def test_mask_term_port_bit_exact_vs_verbatim_reference(assets, tmp_path):
    """Silhouette term (use_mask=True, smplify/loss.py:73-130): the restatement run for one frame equals the verbatim
    reference bit for bit (cv2.findContours adapted to OpenCV 4's return arity in the harness)."""
    mt, nv, N = 'smpl', 4, 10
    syn.write_data_dir(str(tmp_path / 'data'), seed=0, model_types=(mt,))
    port = make_port(assets, mt)
    sc = make_scene(port, mt, 1, nv, seed=12)
    ev = port.loss_and_grads(gt_param_dict(sc['gt'], mt), sc['c2ws'], sc['Ks'], np.zeros((1, nv, 25, 3), np.float32))
    mask_frames = [1, 3]
    masks = syn.make_masks(ev['vertices'][0], port.faces, sc['c2ws'], sc['Ks'])[mask_frames]
    views = syn.keypoints_to_openpose(sc['kp'][0], mt)
    res, trace, terms, _ = rh.run_reference_fit(str(tmp_path), mt, sc['init_betas'][0], sc['init_pose'][0], sc['c2ws'],
                                                sc['Ks'], views, num_iters=N, masks=masks, mask_frames=mask_frames)
    resp, trp = port.fit_frame(sc['init_betas'][0], sc['init_pose'][0], sc['c2ws'], sc['Ks'], views, num_iters=N,
                               masks=masks, mask_frames=mask_frames)
    for k in ('pose', 'betas', 'global_orient', 'global_transl', 'scale', 'joints', 'vertices', 'full_pose'):
        assert np.array_equal(res[k], resp[k]), k
    # the harness records the keypoint objective alone; the port's trace includes 5 x the mask term from iteration N//3+1 on
    assert np.array_equal(np.asarray(trace[:N // 3 + 1]), np.asarray(trp[:N // 3 + 1]))
    assert all(t > 2 * r for t, r in zip(trp[N // 3 + 1:], trace[N // 3 + 1:]))
    # batched restatement (what the GPU tests compare against): same first iterations of the mask phase; afterwards the
    # objective's argmin / inside-outside switches make trajectories sensitive to the last bit
    resb, trb, mls = port.fit_batched_mask(sc['init_betas'][:1], sc['init_pose'][:1], sc['c2ws'], sc['Ks'], sc['kp'][:1],
                                           masks[None], mask_frames, num_iters=N)
    assert mls is not None and (mls > 0).all()
    assert relerr(trb[:N // 3 + 2, 0], np.asarray(trp[:N // 3 + 2])) < 1e-5
    assert relerr(trb[:N // 3 + 3, 0], np.asarray(trp[:N // 3 + 3])) < 1e-3


def _fit_golden(port, g, **kw):
    """One frame of a port_fit_*.npz scene on one torch thread, as the vectors were made (tests/golden/make_golden_port.py:
    in the mask phase the trajectory follows the last bit of every reduction, which depends on the thread count)."""
    views = syn.keypoints_to_openpose(g['kp'][0], 'smpl')
    n = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        return port.fit_frame(g['init_betas'][0], g['init_pose'][0], g['c2ws'], g['Ks'], views, num_iters=int(g['num_iters']), **kw)
    finally:
        torch.set_num_threads(n)


def test_kid_model_port_matches_golden(assets):
    """The kid path against tests/golden/port_fit_kid.npz: the scene of the live bit-exact test above, stored where that test
    held the restatement equal to the verbatim reference (tests/golden/make_golden_port.py)."""
    g = np.load(os.path.join(GOLD, 'port_fit_kid.npz'))
    port = fp.FitPort('smpl', assets('smpl'), assets('gmm'), assets('jx'), age='kid', kid_template=syn.make_kid_template(0))
    res, trace = _fit_golden(port, g)
    assert res['betas'].shape == (11,) and np.abs(res['betas']).max() > 0
    assert relerr(trace, g['trace']) < 1e-5
    for k in ('pose', 'betas', 'global_orient', 'global_transl', 'scale', 'joints', 'vertices'):
        assert np.abs(res[k] - g['out_' + k]).max() < 1e-4, k


def test_mask_term_port_matches_golden(assets):
    """The silhouette term against tests/golden/port_fit_mask.npz: the scene and masks of the live bit-exact test above
    (tests/golden/make_golden_port.py); the trace includes 5 x the mask term from iteration N//3+1 on."""
    g = np.load(os.path.join(GOLD, 'port_fit_mask.npz'))
    port = make_port(assets, 'smpl')
    res, trace = _fit_golden(port, g, masks=g['masks'], mask_frames=list(g['mask_frames']))
    assert relerr(trace, g['trace']) < 1e-5
    for k in ('pose', 'betas', 'global_orient', 'global_transl', 'scale', 'joints', 'vertices', 'full_pose'):
        assert np.abs(res[k] - g['out_' + k]).max() < 1e-4, k


@pytest.mark.parametrize('mt,nv', [('smpl', 4), ('smplx', 8)])
def test_batched_port_equals_per_frame(assets, mt, nv):
    port = make_port(assets, mt)
    B, N = 2, 12
    sc = make_scene(port, mt, B, nv, seed=8)
    resb, trb = port.fit_batched(sc['init_betas'], sc['init_pose'], sc['c2ws'], sc['Ks'], sc['kp'], num_iters=N)
    for f in range(B):
        views = syn.keypoints_to_openpose(sc['kp'][f], mt)
        res, tr = port.fit_frame(sc['init_betas'][f], sc['init_pose'][f], sc['c2ws'], sc['Ks'], views, num_iters=N)
        assert relerr(trb[:, f], tr) < 2e-6
        assert np.abs(res['pose'] - resb['pose'][f]).max() < 1e-5
        assert np.abs(res['vertices'] - resb['vertices'][f]).max() < 1e-5


def test_rodrigues_is_a_rotation_and_handles_zero():
    r = torch.tensor([[0.0, 0.0, 0.0], [0.3, -0.2, 0.9], [3.0, 0.1, -0.4]], dtype=torch.float64)
    R = sp.batch_rodrigues(r)
    assert torch.allclose(R[0], torch.eye(3, dtype=torch.float64), atol=1e-12)
    assert torch.allclose(R @ R.transpose(1, 2), torch.eye(3, dtype=torch.float64).expand(3, 3, 3), atol=1e-7)
    assert torch.allclose(torch.linalg.det(R), torch.ones(3, dtype=torch.float64), atol=1e-7)


def test_lbs_rest_pose_identity(assets):
    """zero pose, zero betas -> vertices == template, chain joints == regressed rest joints."""
    m = sp.SMPLLayer(assets('smpl'), dtype=torch.float64)
    out = m(betas=torch.zeros(1, 10, dtype=torch.float64), body_pose=torch.zeros(1, 69, dtype=torch.float64),
            global_orient=torch.zeros(1, 3, dtype=torch.float64))
    vt = torch.tensor(assets('smpl')['v_template'], dtype=torch.float64)
    assert torch.allclose(out.vertices[0], vt, atol=1e-9)
    J = torch.tensor(assets('smpl')['J_regressor'], dtype=torch.float64) @ vt
    assert torch.allclose(out.joints[0, :24], J, atol=1e-9)
    assert out.joints.shape == (1, 45, 3)


def test_dynamic_landmark_rows(assets):
    """yaw look-up: 0 rad -> row 0; +/- yaw maps into [0,39] / [40,78] as in smplx."""
    m = sp.SMPLXLayer(assets('smplx'), dtype=torch.float64)
    z = torch.zeros(1, 165, dtype=torch.float64)
    v = torch.zeros(1, 10475, 3, dtype=torch.float64)
    idx0, _ = sp.find_dynamic_lmk_idx_and_bcoords(v, z, m.dynamic_lmk_faces_idx, m.dynamic_lmk_bary_coords, m.neck_kin_chain)
    assert torch.equal(idx0[0], m.dynamic_lmk_faces_idx[0])
    for deg, row in ((20.0, 59), (-20.0, 20), (60.0, 78), (-60.0, 39)):
        p = z.clone()
        p[0, 1] = np.deg2rad(deg)                      # rotate the root about y
        idx, _ = sp.find_dynamic_lmk_idx_and_bcoords(v, p, m.dynamic_lmk_faces_idx, m.dynamic_lmk_bary_coords, m.neck_kin_chain)
        assert torch.equal(idx[0], m.dynamic_lmk_faces_idx[row]), (deg, row)


def test_hand_face_confidence_broadcast_quirk():
    """loss.py:134 with a [N,1] confidence: (sum_i c_i^2) * (sum_j rho_j), not sum_j c_j^2 rho_j."""
    rng = np.random.RandomState(0)
    cord, gt = torch.tensor(rng.rand(5, 2)), torch.tensor(rng.rand(5, 2) * 50)
    conf = torch.tensor(rng.rand(5, 1))
    val = fp.reprojection(cord, gt, conf, 0.5, 100.0)
    rho = fp.gmof((gt - cord) / 0.5, 100.0).sum(-1)
    assert val.shape == (5,)                       # one entry per confidence, each times the whole residual sum
    assert torch.allclose(val.sum(), (conf ** 2).sum() * rho.sum())
    assert torch.allclose(fp.reprojection(cord, gt, conf.squeeze(-1), 0.5, 100.0), ((conf.squeeze(-1) ** 2) * rho).sum())


def test_fp32_oracle_close_to_fp64(assets):
    mt, nv, B = 'smplx', 8, 2
    p32, p64 = make_port(assets, mt), make_port(assets, mt, dtype=torch.float64)
    sc = make_scene(p32, mt, B, nv, seed=3)
    from util import perturbed_params
    p = perturbed_params(mt, B, seed=4)
    a, b = p32.loss_and_grads(p, sc['c2ws'], sc['Ks'], sc['kp']), p64.loss_and_grads(p, sc['c2ws'], sc['Ks'], sc['kp'])
    assert relerr(a['loss'], b['loss']) < 1e-5
    assert relerr(a['model_vertices'], b['model_vertices']) < 1e-5
    for k in ('body_pose', 'betas', 'global_orient', 'left_hand_pose'):
        assert relerr(a['grads'][k], b['grads'][k]) < 1e-4, k
