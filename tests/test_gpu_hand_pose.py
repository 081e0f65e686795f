"""GPU tests of the SMPL-X hand options (PreparedModel / SMPLify / SMPLX num_pca_comps, use_pca, flat_hand_mean).

The model is the synthetic SMPL-X model with 45-row hand component tables (test_host_hand_pose.hand_model: its own first 6
rows, then rows from an independent seed).  Every comparison is against the fp64 (or fp32) oracle built with the same hand
options: oracle/fit_port.py::FitPort with its SMPL-X layer given smplx's hand options by HandFitPort below; cases run with and
without tensor cores.  Rows
longer than 112 entries (axis-angle hands, PCA-12 with face parameters) take the wide instantiation of the pose kernels;
the fit invariances are checked bit for bit on such a row."""
import os

import numpy as np
import pytest
import torch

from bodyfitting_b200 import constants as K
from bodyfitting_b200 import synthetic as syn
from oracle import fit_port as fp
from oracle import smplx_port as sp
from test_gpu_face_params import FaceFitPort, _check_columns
from test_host_hand_pose import hand_model
from util import relerr

pytestmark = pytest.mark.gpu


class HandSMPLXLayer(sp.SMPLXLayer):
    """oracle/smplx_port.SMPLXLayer with smplx's other hand options: ``num_pca_comps`` (the base layer's own argument),
    ``use_pca=False`` (hand poses are the 45 axis-angle entries; smplx skips the projection) and ``flat_hand_mean=True``
    (the hand mean is zero).  Without PCA the components become the identity: the base layer's einsum then returns each
    entry times 1 plus exact zeros, i.e. the input itself (test_host_hand_pose.py::test_identity_projection_is_exact)."""

    def __init__(self, data, num_pca_comps=6, use_pca=True, flat_hand_mean=False, **kw):
        super().__init__(data, num_pca_comps=num_pca_comps if use_pca else 6, **kw)
        if not use_pca:
            eye = torch.eye(45, dtype=self.left_hand_components.dtype)
            self.left_hand_components, self.right_hand_components = eye, eye.clone()
        if flat_hand_mean:
            pm = self.pose_mean.clone()
            pm[75:] = 0
            self.pose_mean = pm


class HandFitPort(fp.FitPort):
    """FitPort of an SMPL-X model with other hand options: the model is HandSMPLXLayer (joint map as fp.build_model), the
    hand parameters are [B, n_hand] and step in the same Adam groups as the reference's PCA-6 hands."""

    def __init__(self, smpl_type, model_data, gmm, num_pca_comps=6, use_pca=True, flat_hand_mean=False, dtype=torch.float32,
                 num_betas=10, num_expression=10, **kw):
        super().__init__(smpl_type, model_data, gmm, dtype=dtype, num_betas=num_betas, num_expression=num_expression, **kw)
        assert smpl_type == 'smplx'
        self.n_hand = num_pca_comps if use_pca else 45
        mapper = fp._Mapper(K.smpl_to_openpose('smplx', use_hands=True, use_face=True, use_face_contour=True,
                                               openpose_format='coco25'))
        self.model = HandSMPLXLayer(model_data, num_pca_comps=num_pca_comps, use_pca=use_pca, flat_hand_mean=flat_hand_mean,
                                    num_betas=num_betas, num_expression_coeffs=num_expression, joint_mapper=mapper,
                                    use_face_contour=True, create_transl=False, dtype=dtype).to(self.device)

    def _init_params(self, init_betas, init_poses, B):
        p = super()._init_params(init_betas, init_poses, B)
        for k in ('left_hand_pose', 'right_hand_pose'):
            p[k] = torch.zeros(B, self.n_hand, dtype=self.dtype, device=self.device, requires_grad=True)
        return p

    def loss_and_grads(self, params, c2ws, Ks, kp, imsize=512):
        """FitPort.loss_and_grads with [B, n_hand] hand parameters"""
        kp = torch.as_tensor(kp, dtype=self.dtype)
        B = kp.shape[0]
        p = {k: torch.as_tensor(v, dtype=self.dtype).clone() for k, v in params.items()}
        for k, shape in (('jaw_pose', (B, 1, 3)), ('leye_pose', (B, 1, 3)), ('reye_pose', (B, 1, 3)),
                         ('left_hand_pose', (B, self.n_hand)), ('right_hand_pose', (B, self.n_hand)), ('global_transl', (B, 3))):
            p[k] = p[k].reshape(shape) if k in p else torch.zeros(shape, dtype=self.dtype)
        if 'body_scale' not in p:
            p['body_scale'] = torch.ones(B, 1, dtype=self.dtype)
        for v in p.values():
            v.requires_grad_(True)
        w2cs = torch.inverse(torch.as_tensor(np.array(c2ws), dtype=self.dtype))
        Kt = torch.as_tensor(np.array(Ks), dtype=self.dtype)
        out = self.forward_model(p)
        joints, verts = self.world(out, p)
        per_frame, terms = fp.batched_objective(w2cs, Kt, kp, joints, p['body_pose'], p['betas'], self.prior, imsize,
                                                self.use_hand_face)
        per_frame.sum().backward()
        grads = {k: (v.grad.detach().numpy() if v.grad is not None else None) for k, v in p.items()}
        return dict(loss=per_frame.detach().numpy(), joints=joints.detach().numpy(), vertices=verts.detach().numpy(),
                    model_joints=out.joints.detach().numpy(), model_vertices=out.vertices.detach().numpy(),
                    full_pose=out.full_pose.detach().numpy(), grads=grads,
                    terms={k: v.detach().numpy() for k, v in terms.items()})


class HandFaceFitPort(FaceFitPort, HandFitPort):
    """hand options + the face parameters of test_gpu_face_params.FaceFitPort"""

TC = [pytest.param(True, id='tc'), pytest.param(False, id='ffma')]
MT = 'smplx'
# hand configurations under test: PCA with 12 components, axis-angle hands, the default PCA-6 with a flat hand mean
HANDS = {'pca12': dict(num_pca_comps=12), 'aa': dict(use_pca=False), 'flat': dict(flat_hand_mean=True)}


def _nh(cfg):
    return 45 if not cfg.get('use_pca', True) else cfg.get('num_pca_comps', 6)


@pytest.fixture(scope='module')
def hands(assets):
    """models / oracles of this file, built once"""
    cache = {}
    data = hand_model(0)

    def get(kind, *key):
        k = (kind,) + key
        if k not in cache:
            from bodyfitting_b200.model import PreparedModel
            if kind == 'data':
                return data
            if kind == 'model':
                tc, name, face = key
                cache[k] = PreparedModel(MT, data, gmm=assets('gmm'), device='cuda', tensor_cores=tc, face_params=face,
                                         **HANDS.get(name, {}))
            elif kind == 'port':
                dtype, name, face = key
                cls = HandFaceFitPort if face else HandFitPort
                cache[k] = cls(MT, data, assets('gmm'), dtype=dtype, **HANDS.get(name, {}))
        return cache[k]
    return get


def _hand_values(B, nh, seed, scale=None):
    rng = np.random.RandomState(2000 + seed)
    s = scale if scale is not None else (0.2 if nh == 45 else 0.5)
    return dict(left_hand_pose=(rng.standard_normal((B, nh)) * s).astype(np.float32),
                right_hand_pose=(rng.standard_normal((B, nh)) * s).astype(np.float32))


def _params(B, seed, nh, face=False, with_hands=True):
    gt, _ = syn.make_params(MT, B, seed=seed)
    p = dict(global_orient=gt['global_orient'], body_pose=gt['body_pose'], betas=gt['betas'], global_transl=gt['transl'],
             body_scale=gt['scale'], leye_pose=gt['leye_pose'], reye_pose=gt['reye_pose'])
    if with_hands:
        p.update(_hand_values(B, nh, seed))
    if face:
        rng = np.random.RandomState(1000 + seed)
        p.update(jaw_pose=(rng.standard_normal((B, 3)) * 0.2).astype(np.float32),
                 expression=rng.standard_normal((B, 10)).astype(np.float32))
    return p


def _theta(pm, p):
    T = lambda k: None if k not in p else torch.as_tensor(p[k])
    kw = dict(jaw=T('jaw_pose'), expression=T('expression')) if pm.face_params else {}
    return pm.pack_theta(T('global_orient'), T('body_pose'), T('betas'), transl=T('global_transl'), scale=T('body_scale'),
                         leye=T('leye_pose'), reye=T('reye_pose'), lhand=T('left_hand_pose'), rhand=T('right_hand_pose'), **kw)


def _scene(port, B, nv, seed, gt_hands=None):
    """cameras, init parameters and keypoints from the oracle's joints at GT parameters (``gt_hands``: hand poses of the
    port's hand configuration, else zero hands)"""
    c2ws, Ks = syn.make_cameras(nv, seed=seed)
    gt, init = syn.make_params(MT, B, seed=seed)
    gp = dict(global_orient=gt['global_orient'], body_pose=gt['body_pose'], betas=gt['betas'], global_transl=gt['transl'],
              body_scale=gt['scale'], leye_pose=gt['leye_pose'], reye_pose=gt['reye_pose'])
    if gt_hands is not None:
        gp.update(gt_hands)
    ev = port.loss_and_grads(gp, c2ws, Ks, np.zeros((B, nv, 135, 3), np.float32))
    kp = syn.make_keypoints(ev['joints'][:, :135], c2ws, Ks, seed=seed)
    init_pose = np.concatenate([init['global_orient'], init['body_pose']], 1)
    return dict(c2ws=c2ws, Ks=Ks, kp=kp, init_pose=np.ascontiguousarray(init_pose, np.float32),
                init_betas=np.ascontiguousarray(init['betas'], np.float32))


# ---- 1. forward ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('tc', TC)
@pytest.mark.parametrize('name', list(HANDS))
def test_forward_hand_options(hands, tc, name):
    from bodyfitting_b200.engine import FrameBuffers
    pm, port = hands('model', tc, name, False), hands('port', torch.float64, name, False)
    assert pm.n_hand == _nh(HANDS[name])
    c2ws, Ks = syn.make_cameras(1)
    for B in (1, 129):
        p = _params(B, 3, pm.n_hand)
        ev = port.loss_and_grads(p, c2ws, Ks, np.zeros((B, 1, pm.K_used, 3), np.float32))
        fb = FrameBuffers(pm, B, full=True, need_backward=False)
        fb.t['theta'].copy_(_theta(pm, p))
        fb.call('bf_lbs_forward')
        torch.cuda.synchronize()
        ev_ = relerr(fb.t['verts'].view(B, -1, 3).cpu().numpy(), ev['model_vertices'])
        ej = relerr(fb.t['joints'].cpu().numpy()[:, :pm.K_out], ev['model_joints'])
        ef = relerr(fb.t['full_pose'].cpu().numpy(), ev['full_pose'])
        print(name, 'B', B, 'NP', pm.NP, 'verts rel %.2e joints rel %.2e full_pose rel %.2e' % (ev_, ej, ef))
        assert ev_ < 1e-5 and ej < 1e-5 and ef < 1e-5, B


# ---- 2. zero hand parameters == the default model, bit for bit ----------------------------------------------------------
@pytest.mark.parametrize('tc', TC)
@pytest.mark.parametrize('name', ['pca12', 'aa'])
def test_zero_hands_match_default_model(hands, assets, tc, name):
    from bodyfitting_b200.engine import FrameBuffers
    from bodyfitting_b200.model import PreparedModel
    pm = hands('model', tc, name, False)
    default = PreparedModel(MT, assets(MT), gmm=assets('gmm'), device='cuda', tensor_cores=tc)
    B = 33
    p = _params(B, 5, 6, with_hands=False)
    res = {}
    for key, m in (('hands', pm), ('default', default)):
        fb = FrameBuffers(m, B, full=True, need_backward=False)
        fb.t['theta'].copy_(_theta(m, p))
        fb.call('bf_lbs_forward')
        res[key] = {k: fb.t[k].clone() for k in ('verts', 'joints', 'full_pose')}
    for k in ('verts', 'joints', 'full_pose'):
        assert torch.equal(res['hands'][k], res['default'][k]), k


# ---- 3. axis-angle hands = the PCA-6 expansion -------------------------------------------------------------------------
@pytest.mark.parametrize('tc', TC)
def test_axis_angle_reproduces_pca6(hands, assets, tc):
    from bodyfitting_b200.engine import FrameBuffers
    from bodyfitting_b200.model import PreparedModel
    aa = hands('model', tc, 'aa', False)
    pca6 = PreparedModel(MT, hands('data'), gmm=assets('gmm'), device='cuda', tensor_cores=tc)
    B = 17
    p = _params(B, 9, 6)
    data = hands('data')
    q = dict(p)
    for side, key in (('l', 'left_hand_pose'), ('r', 'right_hand_pose')):
        comp = np.asarray(data['hands_components' + side], np.float64)[:6]
        q[key] = (p[key].astype(np.float64) @ comp).astype(np.float32)
    res = {}
    for key, m, pp in (('aa', aa, q), ('pca6', pca6, p)):
        fb = FrameBuffers(m, B, full=True, need_backward=False)
        fb.t['theta'].copy_(_theta(m, pp))
        fb.call('bf_lbs_forward')
        torch.cuda.synchronize()
        res[key] = {k: fb.t[k].cpu().numpy() for k in ('verts', 'joints', 'full_pose')}
    for k in ('verts', 'joints', 'full_pose'):
        e = relerr(res['aa'][k], res['pca6'][k])
        print('axis-angle vs PCA-6 %-9s rel %.2e' % (k, e))
        assert e < 1e-6, k


# ---- 4. operator backward and objective gradient -----------------------------------------------------------------------
@pytest.mark.parametrize('tc', TC)
@pytest.mark.parametrize('name', list(HANDS))
def test_operator_backward_hands(hands, tc, name):
    from bodyfitting_b200.engine import FrameBuffers
    pm, port = hands('model', tc, name, False), hands('port', torch.float64, name, False)
    B = 129
    p = {k: v for k, v in _params(B, 7, pm.n_hand).items() if k not in ('global_transl', 'body_scale')}
    p['jaw_pose'] = np.zeros((B, 3), np.float32)
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
    for k in ('global_orient', 'body_pose', 'betas', 'left_hand_pose', 'right_hand_pose'):
        got, ref = g[k].cpu().numpy(), pt[k].grad.reshape(B, -1).numpy()
        e = relerr(got, ref)
        print('operator grad %-16s %.2e' % (k, e))
        if 'hand' in k:
            _check_columns(got, ref, 1e-4, 'operator ' + k)
        assert e < 1e-4, k


@pytest.mark.parametrize('tc', TC)
@pytest.mark.parametrize('name,face', [('pca12', False), ('aa', False), ('flat', False), ('aa', True)],
                         ids=['pca12', 'aa', 'flat', 'aa-face'])
def test_objective_and_gradient_hands(hands, tc, name, face):
    from bodyfitting_b200.engine import FrameBuffers, pack_cameras, pack_keypoints
    B, nv = 33, 8
    pm = hands('model', tc, name, face)
    port, port64 = hands('port', torch.float32, name, face), hands('port', torch.float64, name, face)
    sc = _scene(port, B, nv, seed=1)
    p = _params(B, 5, pm.n_hand, face=face)
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
        if 'hand' in k:
            _check_columns(got, ref64, bound, 'objective ' + k)
        assert e < bound, k


# ---- 5. fits against the oracle ---------------------------------------------------------------------------------------
def _fit_vs_oracle(hands, tc, name, face, B, nv, N, seed):
    from bodyfitting_b200.engine import FitSession, pack_cameras, pack_keypoints
    pm, port = hands('model', tc, name, face), hands('port', torch.float32, name, face)
    sc = _scene(port, B, nv, seed=seed, gt_hands=_hand_values(B, pm.n_hand, seed))
    ref, trace = port.fit_batched(sc['init_betas'], sc['init_pose'], sc['c2ws'], sc['Ks'], sc['kp'], num_iters=N)
    sess = FitSession(pm, B, nv, N)
    sess.set_inputs(pack_keypoints(torch.as_tensor(sc['kp']).cuda(), True),
                    torch.from_numpy(pack_cameras(sc['c2ws'], sc['Ks'])).cuda())
    pose0 = torch.as_tensor(sc['init_pose'])
    sess.run(theta0=pm.pack_theta(pose0[:, :3], pose0[:, 3:3 + pm.nbody], torch.as_tensor(sc['init_betas'])))
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in sess.results().items()}
    rel = np.abs(sess.trace.cpu().numpy() - trace) / np.abs(trace)
    print('tc' if tc else 'ffma', name, 'face' if face else '', 'NP', pm.NP, 'N', N, 'fit: loss trace max rel %.2e' % rel.max())
    keys = ['pose', 'betas', 'global_orient', 'global_transl', 'scale', 'leye_pose', 'reye_pose', 'left_hand_pose',
            'right_hand_pose'] + (['jaw_pose', 'expression'] if face else [])
    for k in keys:
        d = np.abs(out[k].reshape(B, -1) - np.asarray(ref[k]).reshape(B, -1)).max()
        print('   %-16s max abs diff %.3e' % (k, d))
        assert d < 2e-5, k
    assert out['left_hand_pose'].shape == (B, pm.n_hand) and np.abs(out['left_hand_pose']).max() > 0
    assert rel.max() < 2e-5
    assert relerr(out['vertices'], ref['vertices']) < 1e-5


@pytest.mark.parametrize('tc', TC)
@pytest.mark.parametrize('name', list(HANDS))
def test_fit_matches_oracle_hands(hands, tc, name):
    _fit_vs_oracle(hands, tc, name, False, 5, 8, 20, seed=2)


def test_fit_matches_oracle_widest_row_100_iterations(hands):
    assert hands('model', True, 'aa', True).NP == 189
    _fit_vs_oracle(hands, True, 'aa', True, 3, 8, 100, seed=4)


# ---- 6. invariances on a wide row, bit for bit -----------------------------------------------------------------------
def _smplify_out(hands, assets, sc, N, hand_kw, **kw):
    from bodyfitting_b200.smplify.smplify import SMPLify
    fit = SMPLify(smpl_type=MT, num_iters=N, gender='neutral', model_data=hands('data'), gmm=assets('gmm'), **hand_kw, **kw)
    o = fit((sc['init_betas'], sc['init_pose']), list(sc['c2ws']), list(sc['Ks']), sc['kp'], None, imsize=512)
    return fit, {k: np.array(v) for k, v in o.items()}


_KEYS = ('pose', 'betas', 'global_orient', 'scale', 'left_hand_pose', 'right_hand_pose', 'vertices', 'joints', 'full_pose')


def test_wide_row_fit_invariances(hands, assets):
    """axis-angle hands (NP = 176, the wide pose kernels): graph replay == direct launches, row-sorted + block-masked ==
    plain order, two concurrent parts == one batch (B = 300); dense_every_iter == active set (B = 5)."""
    N, hk = 12, dict(use_pca=False)
    sc = _scene(hands('port', torch.float32, 'aa', False), 300, 8, seed=6, gt_hands=_hand_values(300, 45, 6))
    fit, base = _smplify_out(hands, assets, sc, N, hk, graph=False, sort_frames=False, concurrent_parts=1)
    assert fit.model.NP == 176 and base['left_hand_pose'].shape == (300, 45) and np.abs(base['left_hand_pose']).max() > 0
    for name, kw in (('graph', dict(graph=True, sort_frames=False, concurrent_parts=1)),
                     ('sorted', dict(graph=False, sort_frames=True, concurrent_parts=1)),
                     ('parts', dict(concurrent_parts=2, concurrent_min_part=128))):
        _, o = _smplify_out(hands, assets, sc, N, hk, **kw)
        for k in _KEYS:
            assert np.array_equal(o[k], base[k]), (name, k)
    sc5 = {k: (v[:5] if k in ('kp', 'init_pose', 'init_betas') else v) for k, v in sc.items()}
    _, a = _smplify_out(hands, assets, sc5, N, hk)
    _, b = _smplify_out(hands, assets, sc5, N, hk, dense_every_iter=True)
    for k in _KEYS:
        assert np.array_equal(a[k], b[k]), ('dense', k)


# ---- 7. temporal term across shards of one GPU on a wide row ----------------------------------------------------------
def test_wide_row_nvlink_halo_shards_of_one_gpu(hands, assets):
    """The in-kernel halo of the temporal term with rows of 189 entries (the halo slots carry the first 128, which hold
    every entry the temporal term reads): three shards of one GPU == one session over the whole sequence, bit for bit."""
    from bodyfitting_b200.sharding import HaloLink, frame_range
    from bodyfitting_b200.smplify.smplify import SMPLify
    nv, B, N, w, G = 8, 11, 14, 300.0, 3
    sc = _scene(hands('port', torch.float32, 'aa', True), B, nv, seed=91, gt_hands=_hand_values(B, 45, 91))
    kw = dict(smpl_type=MT, num_iters=N, gender='neutral', model_data=hands('data'), gmm=assets('gmm'), temporal_weight=w,
              use_pca=False, face_params=True)
    one = SMPLify(**kw)
    assert one.model.NP == 189
    ref = one((sc['init_betas'], sc['init_pose']), list(sc['c2ws']), list(sc['Ks']), sc['kp'], None, imsize=512)
    ref = {k: np.array(v) for k, v in ref.items()}
    links = HaloLink.local_chain(G)
    fits = [SMPLify(halo=links[r], graph=False, **kw) for r in range(G)]
    streams = [torch.cuda.Stream() for _ in range(G)]
    outs = []
    for r in range(G):
        lo, hi = frame_range(B, r, G)
        with torch.cuda.stream(streams[r]):
            outs.append(fits[r]((sc['init_betas'][lo:hi], sc['init_pose'][lo:hi]), list(sc['c2ws']), list(sc['Ks']),
                                sc['kp'][lo:hi], None, imsize=512, as_numpy=False))
    torch.cuda.synchronize()
    for k in ('pose', 'betas', 'global_orient', 'global_transl', 'scale', 'left_hand_pose', 'expression', 'vertices'):
        got = torch.cat([o[k] for o in outs], 0).cpu().numpy()
        assert np.array_equal(got, ref[k]), k
    for l in links:
        l.close()


# ---- 8. property: axis-angle hands fit hands the PCA-6 span cannot represent ------------------------------------------
def test_axis_angle_fit_lowers_the_hand_keypoint_term(hands, assets):
    """Ground-truth hands drawn in axis-angle space (mostly outside the 6-component span): after the same 100 iterations
    the axis-angle fit's hand-keypoint term is lower than the PCA-6 fit's."""
    from bodyfitting_b200.smplify.smplify import SMPLify
    B, nv, N = 6, 8, 100
    port_aa = hands('port', torch.float32, 'aa', False)
    sc = _scene(port_aa, B, nv, seed=8, gt_hands=_hand_values(B, 45, 8, scale=0.3))
    hand_kp = np.array(sc['kp'])
    hand_kp[:, :, :25, 2] = 0
    hand_kp[:, :, 67:, 2] = 0                             # only the two hands' 42 keypoints carry weight
    term = {}
    for name, hk in (('pca6', {}), ('aa', dict(use_pca=False))):
        fit = SMPLify(smpl_type=MT, num_iters=N, gender='neutral', model_data=hands('data'), gmm=assets('gmm'), **hk)
        out = fit((sc['init_betas'], sc['init_pose']), list(sc['c2ws']), list(sc['Ks']), sc['kp'], None, imsize=512)
        port = port_aa if name == 'aa' else hands('port', torch.float32, 'pca6', False)
        p = dict(global_orient=out['global_orient'], body_pose=out['pose'], betas=out['betas'], body_scale=out['scale'],
                 global_transl=np.asarray(out['global_transl']) / np.asarray(out['scale']), leye_pose=out['leye_pose'],
                 reye_pose=out['reye_pose'], left_hand_pose=out['left_hand_pose'], right_hand_pose=out['right_hand_pose'])
        term[name] = float(port.loss_and_grads(p, sc['c2ws'], sc['Ks'], hand_kp)['terms']['reprojection_loss'].sum())
    print('hand-keypoint term after %d iterations: PCA-6 %.4g, axis-angle %.4g' % (N, term['pca6'], term['aa']))
    assert term['aa'] < term['pca6']


# ---- 9. the SMPLX module with [B,45] hands ----------------------------------------------------------------------------
def test_smplx_module_autograd_axis_angle_hands(hands):
    from bodyfitting_b200.models.smpl import create_smplx
    m = create_smplx(model_data=hands('data'), device='cuda', use_pca=False, flat_hand_mean=True)
    assert m.prepared.n_hand == 45
    port = HandFaceFitPort(MT, hands('data'), syn.make_gmm(0), dtype=torch.float64, use_pca=False, flat_hand_mean=True)
    B = 4
    p = _params(B, 11, 45, face=True)
    rng = np.random.RandomState(5)
    dV = rng.standard_normal((B, m.prepared.V, 3))
    dJ = rng.standard_normal((B, m.prepared.K_out, 3))
    names = ('global_orient', 'body_pose', 'betas', 'jaw_pose', 'expression', 'leye_pose', 'reye_pose', 'left_hand_pose',
             'right_hand_pose')
    tg = {k: torch.tensor(p[k], device='cuda', requires_grad=True) for k in names}
    out = m(**tg)
    assert out.left_hand_pose is tg['left_hand_pose']
    ((out.vertices * torch.tensor(dV, device='cuda', dtype=torch.float32)).sum() +
     (out.joints * torch.tensor(dJ, device='cuda', dtype=torch.float32)).sum()).backward()
    to = {k: torch.tensor(p[k], dtype=torch.float64, requires_grad=True) for k in names}
    full = dict(to)
    for k in ('jaw_pose', 'leye_pose', 'reye_pose'):
        full[k] = to[k].reshape(B, 1, 3)
    ro = port.forward_model(full)
    assert relerr(out.vertices.detach().cpu().numpy(), ro.vertices.detach().numpy()) < 1e-5
    ((ro.vertices * torch.tensor(dV)).sum() + (ro.joints * torch.tensor(dJ)).sum()).backward()
    for k in ('left_hand_pose', 'right_hand_pose', 'jaw_pose', 'body_pose'):
        e = relerr(tg[k].grad.cpu().numpy(), to[k].grad.numpy())
        print('SMPLX module grad %-16s %.2e' % (k, e))
        assert e < 1e-4, k


# ---- 10. a host without Python ----------------------------------------------------------------------------------------
@pytest.mark.parametrize('name,face', [('pca12', False), ('aa', True)], ids=['pca12', 'aa-face'])
def test_c_host_program_hand_model(hands, assets, tmp_path, name, face):
    """tests/c_host/fit_host.cpp with the hand options in BfModelDesc: the 16 int32 members it reads from its input file
    carry num_pca_comps; for the two flags after them this test writes a patched copy of the program's struct read.  The
    parameters it fits equal the Python-built model's bit for bit."""
    import shutil
    import struct
    import subprocess
    from bodyfitting_b200 import _lib
    from bodyfitting_b200.engine import FitSession, pack_cameras
    from bodyfitting_b200.model import model_desc
    if shutil.which('nvcc') is None:
        pytest.skip('nvcc not on PATH')
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    src = open(os.path.join(root, 'tests', 'c_host', 'fit_host.cpp')).read()
    old = 'if (!rd(f, &d.is_smplx, 16 * sizeof(int32_t))) return 1;'
    assert src.count(old) == 1
    src = src.replace(old, old + ' if (!rd(f, &d.hand_axis_angle, 2 * sizeof(uint32_t))) return 1;')
    cpp = tmp_path / 'fit_host_hands.cpp'
    cpp.write_text(src)
    exe = str(tmp_path / 'fit_host')
    libdir = os.path.join(root, 'bodyfitting_b200')
    r = subprocess.run(['nvcc', '-std=c++17', '-O2', '-I', os.path.join(root, 'include'), '-o', exe, str(cpp),
                        '-L', libdir, '-lbodyfit_b200', '-Xlinker', '-rpath', '-Xlinker', libdir], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-2000:]
    nv, B, N = 4, 21, 12
    pm = hands('model', True, name, face)
    sc = _scene(hands('port', torch.float32, name, face), B, nv, seed=91, gt_hands=_hand_values(B, pm.n_hand, 91))
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
    desc, keep = model_desc(MT, hands('data'), gmm=assets('gmm'), tensor_cores=pm.tensor_cores, face_params=face,
                            **HANDS[name])
    by_ptr = {a.ctypes.data: a for a in keep}
    path = str(tmp_path / 'in.bin')
    with open(path, 'wb') as f:
        f.write(struct.pack('<I', 0xB200C057))
        for fname, typ in _lib.BfModelDesc._fields_:
            if typ is _lib._fp:
                a = by_ptr.get(getattr(desc, fname))
                f.write(struct.pack('<q', a.nbytes if a is not None else 0))
                if a is not None:
                    f.write(a.tobytes())
        f.write(struct.pack('<16i', *[getattr(desc, n) for n, typ in _lib.BfModelDesc._fields_ if typ is _lib._i32]))
        f.write(struct.pack('<2I', desc.hand_axis_angle, desc.flat_hand_mean))
        f.write(struct.pack('<6i', B, nv, pm.K_used, poses.shape[1], N, 1))
        for a in (kp, cams, poses, betas):
            f.write(a.tobytes())
    out = str(tmp_path / 'theta.bin')
    r = subprocess.run([exe, path, out], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    got = np.fromfile(out, np.float32).reshape(B, pm.NP)
    print('C++ host vs Python session (%s): NP %d, max |d theta| %.2e' % (name, pm.NP, np.abs(got - want).max()))
    o = 7 + 63 + 10 + 6
    assert np.abs(want[:, o:o + 2 * pm.n_hand]).max() > 0                     # the hands moved
    assert np.array_equal(got, want)
