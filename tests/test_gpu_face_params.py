"""GPU tests of face-parameter SMPL-X models: the jaw pose and the expression coefficients as inputs of the body-model
operator and, opt-in, as parameters of the fit (PreparedModel(face_params=True), SMPLify(face_params=True)).

Every case runs with and without tensor cores against the fp64 (and fp32) oracle extended by FaceFitPort below: the
reference's loop (oracle/fit_port.py::FitPort) plus the jaw / expression Adam groups and the expression prior
w_expr^2 sum psi^2.  A face model at zero face parameters must give the
face-off model's numbers bit for bit, and the fit's invariances (graph replay, row order, parts, dense iterations) hold
bit for bit on a face model too."""
import os

import numpy as np
import pytest
import torch

from bodyfitting_b200 import constants as K
from bodyfitting_b200 import synthetic as syn
from oracle import fit_port as fp
from util import relerr

pytestmark = pytest.mark.gpu


class FaceFitPort(fp.FitPort):
    """FitPort with the face parameters optimised: ``jaw_pose`` and ``expression`` as two more Adam groups at the default lr,
    and the expression prior w_expr^2 sum psi^2 added to every frame's loss (and to its shape-prior term).  The base loop
    is reused unchanged; the prior's value and gradient (2 w_expr^2 psi) are added around it."""

    def __init__(self, *a, w_expr=K.EXPR_PRIOR_WEIGHT, num_expression=10, **kw):
        super().__init__(*a, num_expression=num_expression, **kw)
        self.w_expr, self.num_expression = float(w_expr), int(num_expression)

    def _init_params(self, init_betas, init_poses, B):
        p = super()._init_params(init_betas, init_poses, B)
        p['expression'] = torch.zeros(B, self.num_expression, dtype=self.dtype, device=self.device, requires_grad=True)
        return p

    def _optimizer(self, p):
        opt = super()._optimizer(p)
        opt.add_param_group({'params': p['jaw_pose']})
        opt.add_param_group({'params': p['expression']})
        return opt

    def forward_model(self, p):
        return self.model(global_orient=p['global_orient'], body_pose=p['body_pose'], betas=p['betas'],
                          jaw_pose=p['jaw_pose'], leye_pose=p['leye_pose'], reye_pose=p['reye_pose'],
                          left_hand_pose=p['left_hand_pose'], right_hand_pose=p['right_hand_pose'],
                          expression=p['expression'].reshape(-1, self.num_expression), return_full_pose=True)

    def _prior(self, psi):
        return (self.w_expr ** 2) * (psi ** 2).sum(dim=-1)

    def _result(self, p, out, joints, verts, squeeze):
        r = super()._result(p, out, joints, verts, squeeze)
        sq = (lambda t: t.detach().cpu().squeeze(0).numpy()) if squeeze else (lambda t: t.detach().cpu().numpy())
        r.update(jaw_pose=sq(p['jaw_pose'].reshape(-1, 3)), expression=sq(p['expression']))
        return r

    def fit_batched(self, *a, **kw):
        priors = []

        def hook(it, p, out, joints, verts, per_frame):        # after backward, before the Adam step
            with torch.no_grad():
                psi = p['expression']
                priors.append(self._prior(psi).clone())
                psi.grad += (2.0 * self.w_expr ** 2) * psi
        res, trace = super().fit_batched(*a, hook=hook, **kw)
        return res, trace + torch.stack(priors).numpy()

    def loss_and_grads(self, params, c2ws, Ks, kp, imsize=512):
        params = dict(params)
        params.setdefault('expression', np.zeros((np.asarray(kp).shape[0], self.num_expression), np.float32))
        ev = super().loss_and_grads(params, c2ws, Ks, kp, imsize)
        psi = torch.as_tensor(params['expression'], dtype=self.dtype)
        pr = self._prior(psi).numpy()
        ev['loss'] = ev['loss'] + pr
        ev['terms']['shape_prior_loss'] = ev['terms']['shape_prior_loss'] + pr
        ev['grads']['expression'] = ev['grads']['expression'] + (2.0 * self.w_expr ** 2 * psi).numpy()
        return ev


TC = [pytest.param(True, id='tc'), pytest.param(False, id='ffma')]
MT = 'smplx'


@pytest.fixture(scope='module')
def face(assets):
    """models / oracles of this file, built once"""
    cache = {}

    def get(kind, *key):
        k = (kind,) + key
        if k not in cache:
            from bodyfitting_b200.model import PreparedModel
            if kind == 'model':
                tc, on = key
                cache[k] = PreparedModel(MT, assets(MT), gmm=assets('gmm'), device='cuda', tensor_cores=tc, face_params=on)
            elif kind == 'port':
                (dtype,) = key
                cache[k] = FaceFitPort(MT, assets(MT), assets('gmm'), dtype=dtype)
        return cache[k]
    return get


def _face_values(B, seed):
    rng = np.random.RandomState(1000 + seed)
    return dict(jaw_pose=(rng.standard_normal((B, 3)) * 0.2).astype(np.float32),
                expression=rng.standard_normal((B, 10)).astype(np.float32))


def _params(B, seed, with_face=True):
    gt, _ = syn.make_params(MT, B, seed=seed)
    p = dict(global_orient=gt['global_orient'], body_pose=gt['body_pose'], betas=gt['betas'], global_transl=gt['transl'],
             body_scale=gt['scale'])
    p.update({k: gt[k] for k in ('leye_pose', 'reye_pose', 'left_hand_pose', 'right_hand_pose')})
    if with_face:
        p.update(_face_values(B, seed))
    return p


def _theta(pm, p):
    T = lambda k: None if k not in p else torch.as_tensor(p[k])
    kw = dict(jaw=T('jaw_pose'), expression=T('expression')) if pm.face_params else {}
    return pm.pack_theta(T('global_orient'), T('body_pose'), T('betas'), transl=T('global_transl'), scale=T('body_scale'),
                         leye=T('leye_pose'), reye=T('reye_pose'), lhand=T('left_hand_pose'), rhand=T('right_hand_pose'), **kw)


def _check_columns(got, ref, bound, what):
    """each column against the group maximum and against its own maximum (as test_gpu_model_shapes._check_betas_columns)"""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    gmax = max(np.abs(ref).max(), 1e-30)
    err = np.abs(got - ref).max(0)
    own = err / np.maximum(np.abs(ref).max(0), 1e-30)
    bad = [c for c in range(ref.shape[1]) if err[c] > bound * gmax or own[c] > 10 * bound]
    print('   %s per column: max %.2e of the group max, %.2e of the column max' % (what, err.max() / gmax, own.max()))
    assert not bad, '%s: wrong columns %s' % (what, bad)


def _scene(port, B, nv, seed, gt_face=False):
    """cameras, init parameters and keypoints from the oracle's joints at GT parameters (with a non-zero jaw / expression
    when gt_face)"""
    c2ws, Ks = syn.make_cameras(nv, seed=seed)
    gt, init = syn.make_params(MT, B, seed=seed)
    gp = dict(global_orient=gt['global_orient'], body_pose=gt['body_pose'], betas=gt['betas'], global_transl=gt['transl'],
              body_scale=gt['scale'])
    gp.update({k: gt[k] for k in ('leye_pose', 'reye_pose', 'left_hand_pose', 'right_hand_pose')})
    if gt_face:
        fv = _face_values(B, seed)
        gp.update(jaw_pose=fv['jaw_pose'] * 2.0, expression=fv['expression'])
    ev = port.loss_and_grads(gp, c2ws, Ks, np.zeros((B, nv, 135, 3), np.float32))
    kp = syn.make_keypoints(ev['joints'][:, :135], c2ws, Ks, seed=seed)
    init_pose = np.concatenate([init['global_orient'], init['body_pose']], 1)
    return dict(c2ws=c2ws, Ks=Ks, kp=kp, init_pose=np.ascontiguousarray(init_pose, np.float32),
                init_betas=np.ascontiguousarray(init['betas'], np.float32))


# ---- 1. forward ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('tc', TC)
def test_forward_with_jaw_and_expression(face, tc):
    from bodyfitting_b200.engine import FrameBuffers
    pm, port = face('model', tc, True), face('port', torch.float64)
    c2ws, Ks = syn.make_cameras(1)
    for B in (1, 129):
        p = _params(B, seed=3)
        ev = port.loss_and_grads(p, c2ws, Ks, np.zeros((B, 1, pm.K_used, 3), np.float32))
        fb = FrameBuffers(pm, B, full=True, need_backward=False)
        fb.t['theta'].copy_(_theta(pm, p))
        fb.call('bf_lbs_forward')
        torch.cuda.synchronize()
        ev_ = relerr(fb.t['verts'].view(B, -1, 3).cpu().numpy(), ev['model_vertices'])
        ej = relerr(fb.t['joints'].cpu().numpy()[:, :pm.K_out], ev['model_joints'])
        ef = relerr(fb.t['full_pose'].cpu().numpy(), ev['full_pose'])
        print('B', B, 'verts rel %.2e joints rel %.2e full_pose rel %.2e' % (ev_, ej, ef))
        assert ev_ < 1e-5 and ej < 1e-5 and ef < 1e-5, B
        assert np.abs(ev['full_pose'][:, 66:69] - p['jaw_pose']).max() < 1e-6           # the jaw lands in entries 66..68


# ---- 2. zero face parameters == the face-off model, bit for bit ---------------------------------------------------------
@pytest.mark.parametrize('tc', TC)
def test_zero_face_parameters_match_face_off_model(face, tc):
    from bodyfitting_b200.engine import FrameBuffers, pack_cameras, pack_keypoints
    on, off = face('model', tc, True), face('model', tc, False)
    B, nv = 33, 8
    p = _params(B, seed=5, with_face=False)
    rng = np.random.RandomState(2)
    dV = torch.from_numpy(rng.standard_normal((B, on.V * 3)).astype(np.float32)).cuda()
    dJ = torch.from_numpy(rng.standard_normal((B, on.K_full, 3)).astype(np.float32)).cuda()
    res = {}
    for name, pm in (('on', on), ('off', off)):
        fb = FrameBuffers(pm, B, full=True)
        fb.t['theta'].copy_(_theta(pm, p))
        fb.call('bf_lbs_forward')
        fb.t['dverts'].copy_(dV)
        fb.bind('djoints', dJ)
        fb.call('bf_lbs_backward')
        res[name] = {k: fb.t[k].clone() for k in ('verts', 'joints', 'full_pose', 'grad')}
    NPo = off.NP
    for k in ('verts', 'joints', 'full_pose'):
        assert torch.equal(res['on'][k], res['off'][k]), k
    assert torch.equal(res['on']['grad'][:, :NPo], res['off']['grad']), 'operator backward'
    port = face('port', torch.float32)
    sc = _scene(port, B, nv, seed=1)
    kp = pack_keypoints(torch.as_tensor(sc['kp']).cuda(), True)
    cams = torch.from_numpy(pack_cameras(sc['c2ws'], sc['Ks'])).cuda()
    ev = {}
    for name, pm in (('on', on), ('off', off)):
        fb = FrameBuffers(pm, B, full=False, Nv=nv)
        fb.t['theta'].copy_(_theta(pm, p))
        fb.bind('kp', kp)
        fb.bind('cams', cams)
        for fn, extra in (('bf_pose_forward', ()), ('bf_skin_forward', (0,)), ('bf_keypoint_loss', (0,)),
                          ('bf_gmm_prior', ()), ('bf_skin_backward', (0,)), ('bf_pose_backward', (1 | 4,))):
            fb.call(fn, *extra)
        ev[name] = {k: fb.t[k].clone() for k in ('loss', 'loss_terms', 'grad')}
    assert torch.equal(ev['on']['loss'], ev['off']['loss'])
    assert torch.equal(ev['on']['loss_terms'], ev['off']['loss_terms'])
    assert torch.equal(ev['on']['grad'][:, :NPo], ev['off']['grad']), 'objective gradient'


# ---- 3. operator backward -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('tc', TC)
def test_operator_backward_jaw_and_expression(face, tc):
    from bodyfitting_b200.engine import FrameBuffers
    pm, port = face('model', tc, True), face('port', torch.float64)
    B = 129
    p = {k: v for k, v in _params(B, seed=7).items() if k not in ('global_transl', 'body_scale')}
    rng = np.random.RandomState(0)
    dV = rng.standard_normal((B, pm.V, 3)).astype(np.float32)
    dJ = rng.standard_normal((B, pm.K_out, 3)).astype(np.float32)
    pt = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in p.items()}
    full = dict(pt)
    for k in ('jaw_pose', 'leye_pose', 'reye_pose'):
        full[k] = pt[k].reshape(B, 1, 3)
    out = port.forward_model(full)
    ((out.vertices * torch.tensor(dV, dtype=torch.float64)).sum() +
     (out.joints * torch.tensor(dJ, dtype=torch.float64)).sum()).backward()
    fb = FrameBuffers(pm, B, full=True)
    fb.t['theta'].copy_(_theta(pm, p))
    fb.call('bf_lbs_forward')
    fb.t['dverts'].copy_(torch.from_numpy(dV).view(B, -1))
    dJfull = torch.zeros(B, pm.K_full, 3)
    dJfull[:, :pm.K_out] = torch.from_numpy(dJ)
    fb.bind('djoints', dJfull.cuda().contiguous())
    fb.call('bf_lbs_backward')
    torch.cuda.synchronize()
    g = pm.split_theta(fb.t['grad'])
    for k in ('global_orient', 'body_pose', 'betas', 'jaw_pose', 'expression'):
        got, ref = g[k].cpu().numpy(), pt[k].grad.reshape(B, -1).numpy()
        e = relerr(got, ref)
        print('operator grad %-12s %.2e' % (k, e))
        if k == 'expression':
            _check_columns(got, ref, 1e-4, 'operator expression')
        assert e < 1e-4, k


# ---- 4. objective and gradient ------------------------------------------------------------------------------------------
@pytest.mark.parametrize('tc', TC)
def test_objective_and_gradient_with_expression_prior(face, tc):
    from bodyfitting_b200.engine import FrameBuffers, pack_cameras, pack_keypoints
    B, nv = 33, 8
    pm = face('model', tc, True)
    port, port64 = face('port', torch.float32), face('port', torch.float64)
    sc = _scene(port, B, nv, seed=1)
    p = _params(B, seed=5)
    ev = port.loss_and_grads(p, sc['c2ws'], sc['Ks'], sc['kp'])
    ev64 = port64.loss_and_grads(p, sc['c2ws'], sc['Ks'], sc['kp'])
    fb = FrameBuffers(pm, B, full=False, Nv=nv)
    fb.t['theta'].copy_(_theta(pm, p))
    fb.bind('kp', pack_keypoints(torch.as_tensor(sc['kp']).cuda(), True))
    fb.bind('cams', torch.from_numpy(pack_cameras(sc['c2ws'], sc['Ks'])).cuda())
    for fn, extra in (('bf_pose_forward', ()), ('bf_skin_forward', (0,)), ('bf_keypoint_loss', (0,)),
                      ('bf_gmm_prior', ()), ('bf_skin_backward', (0,)), ('bf_pose_backward', (1 | 4,))):
        fb.call(fn, *extra)
    torch.cuda.synchronize()
    loss, terms = fb.t['loss'].cpu().numpy(), fb.t['loss_terms'].cpu().numpy()
    for i, k in enumerate(('reprojection_loss', 'pose_prior_loss', 'angle_prior_loss', 'shape_prior_loss')):
        assert relerr(terms[:, i], ev64['terms'][k]) < 2e-4, k
    assert relerr(loss, ev64['loss']) < 2e-4
    names = dict(transl='global_transl', scale='body_scale')
    for k, gv in pm.split_theta(fb.t['grad']).items():
        ok = names.get(k, k)
        ref64, ref32 = ev64['grads'][ok].reshape(B, -1), ev['grads'][ok].reshape(B, -1)
        got = gv.cpu().numpy()
        e, e32 = relerr(got, ref64), relerr(ref32, ref64)
        print('   grad %-16s cuda-vs-fp64 %.2e   fp32oracle-vs-fp64 %.2e' % (k, e, e32))
        bound = max(2e-4, 20 * e32)
        if k == 'expression':
            _check_columns(got, ref64, bound, 'objective expression')
        assert e < bound, k


# ---- 5. fit against the oracle ------------------------------------------------------------------------------------------
def _fit_vs_oracle(face, tc, B, nv, N, seed):
    from bodyfitting_b200.engine import FitSession, pack_cameras, pack_keypoints
    pm, port = face('model', tc, True), face('port', torch.float32)
    sc = _scene(port, B, nv, seed=seed)
    ref, trace = port.fit_batched(sc['init_betas'], sc['init_pose'], sc['c2ws'], sc['Ks'], sc['kp'], num_iters=N)
    sess = FitSession(pm, B, nv, N)
    sess.set_inputs(pack_keypoints(torch.as_tensor(sc['kp']).cuda(), True),
                    torch.from_numpy(pack_cameras(sc['c2ws'], sc['Ks'])).cuda())
    pose0 = torch.as_tensor(sc['init_pose'])
    sess.run(theta0=pm.pack_theta(pose0[:, :3], pose0[:, 3:3 + pm.nbody], torch.as_tensor(sc['init_betas'])))
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in sess.results().items()}
    rel = np.abs(sess.trace.cpu().numpy() - trace) / np.abs(trace)
    print('tc' if tc else 'ffma', 'N', N, 'fit: loss trace max rel %.2e' % rel.max())
    for k in ('pose', 'betas', 'global_orient', 'global_transl', 'scale', 'leye_pose', 'reye_pose', 'left_hand_pose',
              'right_hand_pose', 'jaw_pose', 'expression'):
        d = np.abs(out[k].reshape(B, -1) - np.asarray(ref[k]).reshape(B, -1)).max()
        print('   %-16s max abs diff %.3e' % (k, d))
        assert d < 2e-5, k
    assert np.abs(out['jaw_pose']).max() > 0 and np.abs(out['expression']).max() > 0
    assert rel.max() < 2e-5
    assert relerr(out['vertices'], ref['vertices']) < 1e-5


@pytest.mark.parametrize('tc', TC)
def test_fit_matches_oracle(face, tc):
    _fit_vs_oracle(face, tc, 5, 8, 20, seed=2)


def test_fit_matches_oracle_100_iterations(face):
    _fit_vs_oracle(face, True, 3, 8, 100, seed=4)


# ---- 6. property: the face parameters absorb face residuals --------------------------------------------------------------
def test_face_fit_lowers_the_data_term(face, assets):
    """On a scene made with a non-zero jaw and expression, the face-parameter fit ends with a lower data term than the
    face-off fit, frame by frame on average and in total."""
    from bodyfitting_b200.smplify.smplify import SMPLify
    B, nv, N = 6, 8, 100
    sc = _scene(face('port', torch.float32), B, nv, seed=8, gt_face=True)
    data = {}
    for on in (False, True):
        fit = SMPLify(smpl_type=MT, num_iters=N, gender='neutral', model_data=assets(MT), gmm=assets('gmm'), face_params=on)
        out = fit((sc['init_betas'], sc['init_pose']), list(sc['c2ws']), list(sc['Ks']), sc['kp'], None, imsize=512)
        data[on] = fit.last_loss_terms[:, 0].cpu().numpy().astype(np.float64)
        assert ('jaw_pose' in out) == on and ('expression' in out) == on
    print('data term: face off %.4g, face on %.4g' % (data[False].sum(), data[True].sum()))
    assert data[True].sum() < data[False].sum()


# ---- 7. invariances on a face model, bit for bit -------------------------------------------------------------------------
def _smplify_out(assets, sc, N, **kw):
    from bodyfitting_b200.smplify.smplify import SMPLify
    fit = SMPLify(smpl_type=MT, num_iters=N, gender='neutral', model_data=assets(MT), gmm=assets('gmm'), face_params=True,
                  **kw)
    o = fit((sc['init_betas'], sc['init_pose']), list(sc['c2ws']), list(sc['Ks']), sc['kp'], None, imsize=512)
    return {k: np.array(v) for k, v in o.items()}


_KEYS = ('pose', 'betas', 'global_orient', 'scale', 'jaw_pose', 'expression', 'vertices', 'joints', 'full_pose')


def test_face_fit_invariances(face, assets):
    """graph replay == direct launches, row-sorted + block-masked == plain order, two concurrent parts == one batch (B = 300);
    dense_every_iter == active set (B = 5)."""
    N = 12
    sc = _scene(face('port', torch.float32), 300, 8, seed=6)
    base = _smplify_out(assets, sc, N, graph=False, sort_frames=False, concurrent_parts=1)
    assert np.abs(base['expression']).max() > 0
    for name, kw in (('graph', dict(graph=True, sort_frames=False, concurrent_parts=1)),
                     ('sorted', dict(graph=False, sort_frames=True, concurrent_parts=1)),
                     ('parts', dict(concurrent_parts=2, concurrent_min_part=128))):
        o = _smplify_out(assets, sc, N, **kw)
        for k in _KEYS:
            assert np.array_equal(o[k], base[k]), (name, k)
    sc5 = {k: (v[:5] if k in ('kp', 'init_pose', 'init_betas') else v) for k, v in sc.items()}
    a = _smplify_out(assets, sc5, N)
    b = _smplify_out(assets, sc5, N, dense_every_iter=True)
    for k in _KEYS:
        assert np.array_equal(a[k], b[k]), ('dense', k)


# ---- 8. the SMPLX module ------------------------------------------------------------------------------------------------
def test_smplx_module_autograd_jaw_expression(face, assets):
    from bodyfitting_b200.models.smpl import create_smplx
    m = create_smplx(model_data=assets(MT), device='cuda')
    port = face('port', torch.float64)
    B = 4
    p = _params(B, seed=11)
    rng = np.random.RandomState(5)
    dV = rng.standard_normal((B, m.prepared.V, 3))
    dJ = rng.standard_normal((B, m.prepared.K_out, 3))
    names = ('global_orient', 'body_pose', 'betas', 'jaw_pose', 'expression', 'leye_pose', 'reye_pose', 'left_hand_pose',
             'right_hand_pose')
    tg = {k: torch.tensor(p[k], device='cuda', requires_grad=True) for k in names}
    kw = dict(tg)
    kw['jaw_pose'] = tg['jaw_pose'].reshape(B, 1, 3)
    out = m(**kw)
    assert out.expression is tg['expression'] and out.jaw_pose is not None
    ((out.vertices * torch.tensor(dV, device='cuda', dtype=torch.float32)).sum() +
     (out.joints * torch.tensor(dJ, device='cuda', dtype=torch.float32)).sum()).backward()
    to = {k: torch.tensor(p[k], dtype=torch.float64, requires_grad=True) for k in names}
    full = dict(to)
    for k in ('jaw_pose', 'leye_pose', 'reye_pose'):
        full[k] = to[k].reshape(B, 1, 3)
    ro = port.forward_model(full)
    assert relerr(out.vertices.detach().cpu().numpy(), ro.vertices.detach().numpy()) < 1e-5
    ((ro.vertices * torch.tensor(dV)).sum() + (ro.joints * torch.tensor(dJ)).sum()).backward()
    for k in ('jaw_pose', 'expression', 'betas', 'body_pose'):
        e = relerr(tg[k].grad.cpu().numpy(), to[k].grad.numpy())
        print('SMPLX module grad %-12s %.2e' % (k, e))
        assert e < 1e-4, k


# ---- 9. a host without Python -------------------------------------------------------------------------------------------
def test_c_host_program_face_model(face, assets, tmp_path):
    """tests/c_host/fit_host.cpp builds a face-parameter model with bf_model_create (face_params = 1), binds the frame buffers
    and runs bf_fit_run: the parameters it writes equal the Python-built model's bit for bit."""
    import shutil
    import struct
    import subprocess
    from bodyfitting_b200 import _lib
    from bodyfitting_b200.engine import FitSession, pack_cameras
    from bodyfitting_b200.model import model_desc
    if shutil.which('nvcc') is None:
        pytest.skip('nvcc not on PATH')
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = str(tmp_path / 'fit_host')
    libdir = os.path.join(root, 'bodyfitting_b200')
    r = subprocess.run(['nvcc', '-std=c++17', '-O2', '-I', os.path.join(root, 'include'), '-o', exe,
                        os.path.join(root, 'tests', 'c_host', 'fit_host.cpp'), '-L', libdir, '-lbodyfit_b200',
                        '-Xlinker', '-rpath', '-Xlinker', libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    nv, B, N = 4, 21, 12
    sc = _scene(face('port', torch.float32), B, nv, seed=91)
    pm = face('model', True, True)
    kp = np.ascontiguousarray(sc['kp'], np.float32)
    cams = pack_cameras(sc['c2ws'], sc['Ks']).astype(np.float32)
    poses, betas = np.ascontiguousarray(sc['init_pose'], np.float32), np.ascontiguousarray(sc['init_betas'], np.float32)
    sess = FitSession(pm, B, nv, N + 1, graph=False, trace=True)
    sess.load_inputs(torch.from_numpy(kp).cuda(), torch.from_numpy(cams).cuda(), torch.from_numpy(poses).cuda(),
                     torch.from_numpy(betas).cuda())
    sess.fb.t['theta'].copy_(sess.theta0); sess.fb.t['adam_m'].zero_(); sess.fb.t['adam_v'].zero_()
    sess.fb.struct.iter = 0
    sess.fb.call('bf_fit_run', N)
    torch.cuda.synchronize()
    perm = sess.perm0.cpu().numpy() if getattr(sess, 'sort_frames', False) else np.arange(B)
    want = np.empty((B, pm.NP), np.float32)
    want[perm] = sess.fb.t['theta'].cpu().numpy()
    assert np.abs(want[:, -10:]).max() > 0                          # the expression moved
    desc, keep = model_desc(MT, assets(MT), gmm=assets('gmm'), tensor_cores=pm.tensor_cores, face_params=True)
    by_ptr = {a.ctypes.data: a for a in keep}
    path = str(tmp_path / 'in.bin')
    with open(path, 'wb') as f:
        f.write(struct.pack('<I', 0xB200C057))
        for name, typ in _lib.BfModelDesc._fields_:
            if typ is _lib._fp:
                a = by_ptr.get(getattr(desc, name))
                f.write(struct.pack('<q', a.nbytes if a is not None else 0))
                if a is not None:
                    f.write(a.tobytes())
        f.write(struct.pack('<16i', *[getattr(desc, name) for name, typ in _lib.BfModelDesc._fields_ if typ is _lib._i32]))
        f.write(struct.pack('<6i', B, nv, pm.K_used, poses.shape[1], N, 1))
        for a in (kp, cams, poses, betas):
            f.write(a.tobytes())
    out = str(tmp_path / 'theta.bin')
    r = subprocess.run([exe, path, out], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    got = np.fromfile(out, np.float32).reshape(B, pm.NP)
    print('C++ host vs Python session (face model): max |d theta| %.2e' % np.abs(got - want).max())
    assert np.array_equal(got, want)
