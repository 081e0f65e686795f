"""GPU parity across shape-space sizes: the number of betas (NB) and of expression coefficients (NE) is not fixed at 10 / 10.

The kernels have code that changes with these counts, and the other parity tests use one size per model family:
  * the rest-joint regression in k_pose_fwd (a vectorised path for NB == 10, a generic loop otherwise);
  * the rest-joint part of d loss / d betas in k_pose_bwd, split across warp lanes in 3, 2 or 1 parts by NB;
  * the theta layout: the eye and hand parameters of SMPL-X sit after the NB betas;
  * the column tile of the backward blend GEMM, chosen from Kp = round16(P + NS + 1) -- 496 for SMPL-X with NS <= 9.
Every configuration runs with and without tensor cores, against the fp64 (and fp32) oracle with the same counts.  The betas
gradient is checked column by column, so that a few wrong betas cannot hide inside the maximum of the group."""
import numpy as np
import pytest
import torch

from bodyfitting_b200 import synthetic as syn
from util import relerr

pytestmark = pytest.mark.gpu

# (model type, num_betas, num_expression, kid): NS = betas (+1 for the kid direction) + expression <= 20, NP <= 100
CONFIGS = [('smpl', 1, 0, False), ('smpl', 10, 0, False), ('smpl', 16, 0, False), ('smpl', 17, 0, False),
           ('smpl', 20, 0, False), ('smpl', 10, 0, True), ('smpl', 16, 0, True),
           ('smplx', 10, 10, False), ('smplx', 12, 8, False), ('smplx', 10, 0, False), ('smplx', 5, 4, False),
           ('smplx', 1, 0, False)]


def _cid(c):
    return ('kid' if c[3] else c[0]) + '-nb%d' % c[1] + ('-ne%d' % c[2] if c[0] == 'smplx' else '')


CASES = [pytest.param(c, tc, id=_cid(c) + ('-tc' if tc else '-ffma')) for c in CONFIGS for tc in (True, False)]


@pytest.fixture(scope='module')
def shapes(assets):
    """Models, oracles and oracle results of this file, built once per configuration (and per kernel family)."""
    cache = {}

    def get(kind, cfg, *key):
        k = (kind, cfg) + key
        if k not in cache:
            cache[k] = _make(get, assets, kind, cfg, *key)
        return cache[k]
    return get


def _make(get, assets, kind, cfg, *key):
    from bodyfitting_b200.model import PreparedModel
    from oracle import fit_port as fp
    mt, nb, ne, kid = cfg
    if kind == 'data':
        return syn.make_model(mt, 0, nb, ne)
    kw = dict(age='kid', kid_template=syn.make_kid_template(0)) if kid else {}
    if kind == 'model':
        (tc,) = key
        pm = PreparedModel(mt, get('data', cfg), gmm=assets('gmm'), J_regressor_extra=assets('jx'), device='cuda',
                           num_betas=nb, num_expression=ne, tensor_cores=tc, **kw)
        assert pm.NB == nb + kid and pm.NS == nb + kid + (ne if mt == 'smplx' else 0)
        return pm
    if kind == 'port':
        (dtype,) = key
        return fp.FitPort(mt, get('data', cfg), assets('gmm'), assets('jx'), dtype=dtype, num_betas=nb, num_expression=ne, **kw)
    if kind == 'fit':                                     # the oracle's fit, shared by both kernel families
        B, nv, N = key
        port = get('port', cfg, torch.float32)
        sc = _scene(port, cfg, B, nv, seed=2)
        ref, trace = port.fit_batched(sc['init_betas'], sc['init_pose'], sc['c2ws'], sc['Ks'], sc['kp'], num_iters=N)
        return ref, trace, sc
    raise KeyError(kind)


def _betas(betas10, n, seed):
    """[B, n] betas: the first columns of the synthetic 10, further columns drawn at the same scale."""
    rng = np.random.RandomState(seed)
    extra = rng.standard_normal((betas10.shape[0], max(0, n - 10))).astype(np.float32)
    return np.ascontiguousarray(np.concatenate([betas10[:, :n], extra], 1), dtype=np.float32)


def _params(cfg, B, seed):
    """Generic (non-zero everywhere) parameters with NB betas (the kid coefficient included)."""
    mt, nb, ne, kid = cfg
    gt, _ = syn.make_params(mt, B, seed=seed)
    p = dict(global_orient=gt['global_orient'], body_pose=gt['body_pose'], betas=_betas(gt['betas'], nb + kid, seed),
             global_transl=gt['transl'], body_scale=gt['scale'])
    if mt == 'smplx':
        p.update({k: gt[k] for k in ('leye_pose', 'reye_pose', 'left_hand_pose', 'right_hand_pose')})
    return p


def _theta(pm, p):
    T = lambda k: None if k not in p else torch.as_tensor(p[k])
    return pm.pack_theta(T('global_orient'), T('body_pose'), T('betas'), transl=T('global_transl'),
                         scale=T('body_scale'), leye=T('leye_pose'), reye=T('reye_pose'),
                         lhand=T('left_hand_pose'), rhand=T('right_hand_pose'))


def _groups(mt):
    return ('global_orient', 'body_pose', 'betas') + (('leye_pose', 'reye_pose', 'left_hand_pose', 'right_hand_pose')
                                                     if mt == 'smplx' else ())


def _check_betas_columns(got, ref, bound, what):
    """Every betas column on its own, against the largest reference entry of the group (the bound of the group check) and
    against its own largest entry (a wrong column is wrong by about its own size)."""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    gmax = max(np.abs(ref).max(), 1e-30)
    err = np.abs(got - ref).max(0)
    own = err / np.maximum(np.abs(ref).max(0), 1e-30)
    print('   %s betas per column: max %.2e of the group max, %.2e of the column max' % (what, err.max() / gmax, own.max()))
    bad = [c for c in range(ref.shape[1]) if err[c] > bound * gmax or own[c] > 10 * bound]
    assert not bad, '%s: wrong betas columns %s (error / group max %s)' % (what, bad, ['%.1e' % (err[c] / gmax) for c in bad])


@pytest.mark.parametrize('cfg,tc', CASES)
def test_dense_forward(shapes, cfg, tc):
    """bf_lbs_forward on all vertices at B = 1 and 129 (a second 128-frame tile): vertices, joints and full pose against the
    fp64 oracle, at the bounds of test_gpu_parity.py::test_lbs_forward."""
    from bodyfitting_b200.engine import FrameBuffers
    mt = cfg[0]
    pm, port = shapes('model', cfg, tc), shapes('port', cfg, torch.float64)
    c2ws, Ks = syn.make_cameras(1)
    for B in (1, 129):
        p = _params(cfg, B, seed=3)
        ev = port.loss_and_grads(p, c2ws, Ks, np.zeros((B, 1, pm.K_used, 3), np.float32))
        fb = FrameBuffers(pm, B, full=True, need_backward=False)
        fb.t['theta'].copy_(_theta(pm, p))
        fb.call('bf_lbs_forward')
        torch.cuda.synchronize()
        verts = fb.t['verts'].view(B, -1, 3).cpu().numpy()
        joints = fb.t['joints'].cpu().numpy()[:, :pm.K_out]
        fpose = fb.t['full_pose'].cpu().numpy()
        ev_, ej, ef = relerr(verts, ev['model_vertices']), relerr(joints, ev['model_joints']), relerr(fpose, ev['full_pose'])
        print(_cid(cfg), 'tc' if tc else 'ffma', 'B', B, 'verts rel %.2e joints rel %.2e full_pose rel %.2e' % (ev_, ej, ef))
        assert ev_ < 1e-5 and ej < 1e-5 and ef < 1e-6, B


@pytest.mark.parametrize('cfg,tc', CASES)
def test_dense_backward(shapes, cfg, tc):
    """bf_lbs_backward (the autograd of models.smpl.SMPL) at B = 129: random d(vertices), d(joints) -> d theta against fp64
    autograd of the oracle, every group <= 1e-4 and the betas column by column."""
    from bodyfitting_b200.engine import FrameBuffers
    mt, B = cfg[0], 129
    pm, port = shapes('model', cfg, tc), shapes('port', cfg, torch.float64)
    p = _params(cfg, B, seed=7)
    rng = np.random.RandomState(0)
    dV = rng.standard_normal((B, pm.V, 3)).astype(np.float32)
    dJ = rng.standard_normal((B, pm.K_out, 3)).astype(np.float32)
    dJfull = np.zeros((B, pm.K_full, 3), np.float32)
    dJfull[:, :pm.K_out] = dJ
    pt = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in p.items()
          if k not in ('global_transl', 'body_scale')}
    z = lambda *s: torch.zeros(*s, dtype=torch.float64)
    full = dict(jaw_pose=z(B, 1, 3), leye_pose=z(B, 1, 3), reye_pose=z(B, 1, 3), left_hand_pose=z(B, 6), right_hand_pose=z(B, 6))
    for k in list(full):
        if k in pt:
            full[k] = pt[k].reshape(full[k].shape)
    full.update(global_orient=pt['global_orient'], body_pose=pt['body_pose'], betas=pt['betas'])
    out = port.forward_model(full)
    (out.vertices * torch.tensor(dV, dtype=torch.float64)).sum().add((out.joints * torch.tensor(dJ, dtype=torch.float64)).sum()).backward()
    fb = FrameBuffers(pm, B, full=True)
    fb.t['theta'].copy_(_theta(pm, {k: v for k, v in p.items() if k not in ('global_transl', 'body_scale')}))
    fb.call('bf_lbs_forward')
    fb.t['dverts'].copy_(torch.from_numpy(dV).view(B, -1))
    fb.bind('djoints', torch.from_numpy(dJfull).cuda().contiguous())
    fb.call('bf_lbs_backward')
    torch.cuda.synchronize()
    g = pm.split_theta(fb.t['grad'])
    for k in _groups(mt):
        got, ref = g[k].cpu().numpy(), pt[k].grad.reshape(B, -1).numpy()
        e = relerr(got, ref)
        print(_cid(cfg), 'tc' if tc else 'ffma', 'operator grad %-16s %.2e' % (k, e))
        if k == 'betas':
            assert got.shape[1] == cfg[1] + cfg[3]
            _check_betas_columns(got, ref, 1e-4, 'operator')
        assert e < 1e-4, k


def _scene(port, cfg, B, nv, seed):
    """cameras, GT / init parameters (NB betas) and keypoints from the oracle's GT joints (tests/util.py::make_scene)."""
    mt, nb, ne, kid = cfg
    c2ws, Ks = syn.make_cameras(nv, seed=seed)
    gt, init = syn.make_params(mt, B, seed=seed)
    gp = _params(cfg, B, seed)
    gp.update(global_orient=gt['global_orient'], body_pose=gt['body_pose'], global_transl=gt['transl'], body_scale=gt['scale'])
    K = 135 if mt == 'smplx' else 25
    ev = port.loss_and_grads(gp, c2ws, Ks, np.zeros((B, nv, K, 3), np.float32))
    kp = syn.make_keypoints(ev['joints'][:, :K], c2ws, Ks, seed=seed)
    init_pose = np.concatenate([init['global_orient'], init['body_pose']], 1)
    init_betas = _betas(init['betas'], nb, seed + 1)
    return dict(c2ws=c2ws, Ks=Ks, kp=kp, init_pose=np.ascontiguousarray(init_pose, dtype=np.float32), init_betas=init_betas)


def _nviews(mt):
    return 8 if mt == 'smplx' else 4


@pytest.mark.parametrize('cfg,tc', CASES)
def test_objective_and_gradient(shapes, cfg, tc):
    """One evaluation of the objective on the active vertex set (test_gpu_parity.py::test_loss_and_gradients): per-frame loss,
    the four loss terms and d loss / d theta against the oracle in fp64 (and fp32), B = 33."""
    from bodyfitting_b200.engine import FrameBuffers, pack_cameras, pack_keypoints
    mt, B, nv = cfg[0], 33, _nviews(cfg[0])
    pm = shapes('model', cfg, tc)
    port, port64 = shapes('port', cfg, torch.float32), shapes('port', cfg, torch.float64)
    sc = _scene(port, cfg, B, nv, seed=1)
    p = _params(cfg, B, seed=5)
    ev = port.loss_and_grads(p, sc['c2ws'], sc['Ks'], sc['kp'])
    ev64 = port64.loss_and_grads(p, sc['c2ws'], sc['Ks'], sc['kp'])
    fb = FrameBuffers(pm, B, full=False, Nv=nv)
    fb.t['theta'].copy_(_theta(pm, p))
    fb.bind('kp', pack_keypoints(torch.as_tensor(sc['kp']).cuda(), mt == 'smplx'))
    fb.bind('cams', torch.from_numpy(pack_cameras(sc['c2ws'], sc['Ks'])).cuda())
    for fn, extra in (('bf_pose_forward', ()), ('bf_skin_forward', (0,)), ('bf_keypoint_loss', (0,)),
                      ('bf_gmm_prior', ()), ('bf_skin_backward', (0,)), ('bf_pose_backward', (1 | 4,))):
        fb.call(fn, *extra)
    torch.cuda.synchronize()
    loss = fb.t['loss'].cpu().numpy()
    terms = fb.t['loss_terms'].cpu().numpy()
    print(_cid(cfg), 'tc' if tc else 'ffma', 'loss rel vs fp64 %.2e' % relerr(loss, ev64['loss']))
    for i, k in enumerate(('reprojection_loss', 'pose_prior_loss', 'angle_prior_loss', 'shape_prior_loss')):
        assert relerr(terms[:, i], ev64['terms'][k]) < 1e-4, k
    assert relerr(loss, ev64['loss']) < 1e-4
    g = pm.split_theta(fb.t['grad'])
    names = dict(transl='global_transl', scale='body_scale')
    for k, gv in g.items():
        ok = names.get(k, k)
        ref64, ref32 = ev64['grads'][ok].reshape(B, -1), ev['grads'][ok].reshape(B, -1)
        got = gv.cpu().numpy()
        e, e32 = relerr(got, ref64), relerr(ref32, ref64)
        print('   grad %-16s cuda-vs-fp64 %.2e   fp32oracle-vs-fp64 %.2e' % (k, e, e32))
        bound = max(2e-4, 20 * e32)
        if k == 'betas':
            assert got.shape[1] == cfg[1] + cfg[3]
            _check_betas_columns(got, ref64, bound, 'objective')
        assert e < bound, k


@pytest.mark.parametrize('cfg', [pytest.param(c, id=_cid(c)) for c in CONFIGS])
def test_init_theta(shapes, cfg):
    """bf_init_theta takes the network's 10 betas whatever the model's count: the first NB of them when NB < 10 (the eye and
    hand parameters after them start at 0), all 10 and zeros beyond otherwise (the kid direction, betas past the 10th)."""
    from bodyfitting_b200 import _lib
    pm, B = shapes('model', cfg, True), 7
    rng = np.random.RandomState(3)
    poses = torch.from_numpy(rng.randn(B, 72).astype(np.float32)).cuda()
    betas = torch.from_numpy(rng.randn(B, 10).astype(np.float32)).cuda()
    theta = torch.full((B, pm.NP), 7.0, device='cuda')
    L, st = _lib.lib(), torch.cuda.current_stream().cuda_stream
    _lib.check(L.bf_init_theta(pm.struct, poses.data_ptr(), 72, betas.data_ptr(), theta.data_ptr(), B, None, st), 'bf_init_theta')
    assert torch.equal(theta, pm.pack_theta(poses[:, :3], poses[:, 3:3 + pm.nbody], betas[:, :min(pm.NB, 10)]))


@pytest.mark.parametrize('cfg,tc', CASES)
def test_fit(shapes, cfg, tc):
    """20 iterations through FitSession.run(theta0=...) against the oracle's batched loop with the same counts
    (test_gpu_parity.py::test_fit_trajectory bounds): per-iteration loss <= 2e-5 relative, parameters <= 2e-5 absolute --
    the eye and hand parameters of SMPL-X included, whose place in theta depends on NB.  theta0 is packed here: bf_init_theta
    takes exactly 10 betas."""
    from bodyfitting_b200.engine import FitSession, pack_cameras, pack_keypoints
    mt, nb, ne, kid = cfg
    B, nv, N = 5, _nviews(mt), 20
    pm = shapes('model', cfg, tc)
    ref, trace, sc = shapes('fit', cfg, B, nv, N)
    sess = FitSession(pm, B, nv, N)
    sess.set_inputs(pack_keypoints(torch.as_tensor(sc['kp']).cuda(), mt == 'smplx'),
                    torch.from_numpy(pack_cameras(sc['c2ws'], sc['Ks'])).cuda())
    betas0 = np.zeros((B, nb + 1), np.float32) if kid else sc['init_betas']        # the kid model starts from zero betas
    pose0 = torch.as_tensor(sc['init_pose'])
    theta0 = pm.pack_theta(pose0[:, :3], pose0[:, 3:3 + pm.nbody], torch.as_tensor(betas0))
    sess.run(theta0=theta0)
    torch.cuda.synchronize()
    out = {k: v.cpu().numpy() for k, v in sess.results().items()}
    tr = sess.trace.cpu().numpy()
    rel = np.abs(tr - trace) / np.abs(trace)
    print(_cid(cfg), 'tc' if tc else 'ffma', 'fit: loss trace max rel %.2e' % rel.max())
    keys = ('pose', 'betas', 'global_orient', 'global_transl', 'scale')
    if mt == 'smplx':
        keys += ('leye_pose', 'reye_pose', 'left_hand_pose', 'right_hand_pose')
    for k in keys:
        d = np.abs(out[k].reshape(B, -1) - np.asarray(ref[k]).reshape(B, -1))
        print('   %-16s max abs diff %.3e' % (k, d.max()))
        if k == 'betas':
            assert out[k].shape == (B, nb + kid)
            bad = [c for c in range(d.shape[1]) if d[:, c].max() >= 2e-5]
            assert not bad, 'fit: wrong betas columns %s' % bad
        assert d.max() < 2e-5, k
    assert rel.max() < 2e-5
    assert relerr(out['vertices'], ref['vertices']) < 1e-5
    assert relerr(out['joints'], ref['joints']) < 1e-5

