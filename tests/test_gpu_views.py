"""GPU parity across camera view counts, image sizes and the launch shapes of the fit's fused per-frame kernel.

The number of views is the input that moves k_frame_loss_bwd (bf_frame.cuh) between its code paths: the bulk-copy (TMA) or
plain staging chosen by bf_frame_use_tma, the 16-byte keypoint reads (Nv % 4 == 0) against the scalar tail, the staged
camera rows and the shared-memory layout (frame_smem_layout).  The unfused k_keypoint_loss, the operator surface (k_kp_world)
and the input packing (k_pack_keypoints) take the same views.  The C ABI accepts 1 to 64 views (BF_MAXVIEWS).

Launch shape of k_frame_loss_bwd the host picks (bf_api.cu, bf_frame_loss_backward) for the synthetic models, computed by
_frame_shape below and asserted by the launch-shape test:

    model (K_used)   views                                       < 2,048 frames   >= 2,048 frames
    SMPL-X (135)     4, 8, 12                                     <1,224>          <2,160>
    SMPL-X           not a multiple of 4, or >= 16 (the staged    <0,224>          <0,224>
                     keypoint row takes the kernel above 48 KB:
                     52.3 KB at 16 views)
    SMPL (25)        multiples of 4 up to 64                      <1,224>          <2,160>
    SMPL             others                                       <0,224>          <0,224>

<TMA, threads>: <1,224> stages the keypoint row by bulk copy, <2,160> reads it from global memory, <0,224> uses plain loads.

Every case runs with and without tensor cores, against the fp64 (and fp32) oracle (oracle/fit_port.py) at the bounds of
test_gpu_parity.py::test_loss_and_gradients.  Scenes carry frames with a view without detections, a whole view without
detections (views without detections still count in the 1 / Nv of the reference) and a joint without detections.
"""
import numpy as np
import pytest
import torch

from bodyfitting_b200 import synthetic as syn
from util import gt_param_dict, perturbed_params, relerr

pytestmark = pytest.mark.gpu

VIEWS = (1, 2, 3, 4, 5, 7, 8, 12, 13, 16, 30, 31, 48, 64)
GRID = [(mt, nv, 512) for mt in ('smpl', 'smplx') for nv in VIEWS] + \
       [(mt, nv, im) for mt in ('smpl', 'smplx') for nv in (8, 13) for im in (1000, 1024, 2048)]
TERMS = ('reprojection_loss', 'pose_prior_loss', 'angle_prior_loss', 'shape_prior_loss')
NB = 37                     # frames of the one-evaluation grid: a partial 128-frame tile, not a multiple of 4 or 8


@pytest.fixture(scope='module')
def views(assets):
    """Models, oracles, scenes and oracle results of this file, built once per key."""
    cache = {}

    def get(kind, *key):
        k = (kind,) + key
        if k not in cache:
            cache[k] = _make(get, assets, kind, *key)
        return cache[k]
    return get


def _make(get, assets, kind, *key):
    from bodyfitting_b200.model import PreparedModel
    from oracle import fit_port as fp
    if kind == 'model':
        mt, tc = key
        return PreparedModel(mt, assets(mt), gmm=assets('gmm'), J_regressor_extra=assets('jx'), device='cuda', tensor_cores=tc)
    if kind == 'port':
        mt, dtype = key
        return fp.FitPort(mt, assets(mt), assets('gmm'), assets('jx'), dtype=dtype)
    if kind == 'scene':
        mt, nv, imsize, B = key
        return _scene(get('port', mt, torch.float32), mt, B, nv, imsize, seed=nv)
    if kind == 'oracle':                         # one evaluation at generic parameters, fp32 and fp64
        mt, nv, imsize, B = key
        sc = get('scene', mt, nv, imsize, B)
        p = perturbed_params(mt, B, seed=5)
        ev = get('port', mt, torch.float32).loss_and_grads(p, sc['c2ws'], sc['Ks'], sc['kp'], imsize=imsize)
        ev64 = get('port', mt, torch.float64).loss_and_grads(p, sc['c2ws'], sc['Ks'], sc['kp'], imsize=imsize)
        return p, ev, ev64
    raise KeyError(kind)


def _scene(port, mt, B, nv, imsize, seed):
    """A ring of nv cameras whose focal length scales with the image (the body covers the same share of every image size),
    GT / init parameters and detections from the oracle's GT joints (tests/util.py::make_scene), and detections removed:
    frame 1 has none in view 0, no frame has any in the last view (nv >= 3), frame 2 has none of joint 3 in any view."""
    c2ws, Ks = syn.make_cameras(nv, focal=float(imsize), imsize=imsize, seed=seed)
    gt, init = syn.make_params(mt, B, seed=seed)
    K = 135 if mt == 'smplx' else 25
    ev = port.loss_and_grads(gt_param_dict(gt, mt), c2ws, Ks, np.zeros((B, nv, K, 3), np.float32), imsize=imsize)
    kp = syn.make_keypoints(ev['joints'][:, :K], c2ws, Ks, seed=seed)
    if B > 2:
        kp[1, 0] = 0.0
        kp[2, :, 3] = 0.0
    if nv >= 3:
        kp[:, nv - 1] = 0.0
    init_pose = np.concatenate([init['global_orient'], init['body_pose']], 1)
    if mt == 'smplx':
        init_pose = np.concatenate([init_pose, np.zeros((B, 6), np.float32)], 1)
    return dict(c2ws=c2ws, Ks=Ks, kp=np.ascontiguousarray(kp), init_pose=np.ascontiguousarray(init_pose, dtype=np.float32),
                init_betas=init['betas'])


def _theta(pm, p):
    T = lambda k: None if k not in p else torch.as_tensor(p[k])
    return pm.pack_theta(T('global_orient'), T('body_pose'), T('betas'), transl=T('global_transl'),
                         scale=T('body_scale'), leye=T('leye_pose'), reye=T('reye_pose'),
                         lhand=T('left_hand_pose'), rhand=T('right_hand_pose'))


def _frame_shape(pm, nv, B):
    """<TMA, threads> of k_frame_loss_bwd (bf_api.cu: bf_frame_use_tma, bf_frame_loss_backward) for 16-byte aligned buffers
    (torch allocations): frame_smem_layout of bf_frame.cuh restated."""
    a, K, J = pm.struct.act, pm.K_used, pm.J
    base = ((3 * K + 3) & ~3) + nv * 12 + 64 + ((J * 12 + 15) & ~15) + 2 * a.ldn + 12 * a.lmax
    staged = 4 * (base + ((K * nv * 3 + 3) & ~3) + 4)
    tma = (K * nv) % 4 == 0 and staged <= 48 * 1024
    return (2, 160) if tma and B >= 2048 else (1, 224) if tma else (0, 224)


def _evaluate(pm, theta, kp, cams, nv, imsize, fused):
    """One evaluation of the objective and d loss / d theta on the active vertex set, in a fresh FrameBuffers (the block
    masks of the tensor-core path and their parity follow the iteration).  fused: the calls of one fit iteration
    (bf_api.cu fit_iteration) without the Adam step -- pose forward, blend GEMM (tensor cores; the per-frame kernel skins)
    or blend + skinning (FFMA), k_frame_loss_bwd, GMM prior, blend backward GEMM, pose backward.  Otherwise the unfused
    path of the all-vertex loop: k_keypoint_loss and the separate skinning backward."""
    from bodyfitting_b200 import _lib
    from bodyfitting_b200.engine import FrameBuffers
    B = theta.shape[0]
    fb = FrameBuffers(pm, B, full=False, Nv=nv, imsize=imsize)
    fb.t['theta'].copy_(theta)
    fb.bind('kp', kp)
    fb.bind('cams', cams)
    fb.call('bf_pose_forward')
    if fused:
        if pm.tensor_cores:
            fb.call('bf_blend_forward', 0)
            fb.struct.flags |= _lib.F_SKIN_FUSED
        else:
            fb.call('bf_skin_forward', 0)
        fb.call('bf_frame_loss_backward')
        fb.struct.flags &= ~_lib.F_SKIN_FUSED
        fb.call('bf_gmm_prior')
        fb.call('bf_skin_backward_parts', 0, 4)
    else:
        fb.call('bf_skin_forward', 0)
        fb.call('bf_keypoint_loss', 0)
        fb.call('bf_gmm_prior')
        fb.call('bf_skin_backward', 0)
    fb.call('bf_pose_backward', 1 | 4)
    torch.cuda.synchronize()
    return {k: fb.t[k].cpu().numpy().copy() for k in ('loss', 'loss_terms', 'grad')}


def _inputs(sc, mt):
    from bodyfitting_b200.engine import pack_cameras, pack_keypoints
    return (pack_keypoints(torch.as_tensor(sc['kp']).cuda(), mt == 'smplx'),
            torch.from_numpy(pack_cameras(sc['c2ws'], sc['Ks'])).cuda())


def _check_oracle(pm, got, ev, ev64, rows, what):
    """Loss, the four terms and every theta group of split_theta(grad) against the oracle's rows."""
    loss, terms = got['loss'], got['loss_terms']
    ref_loss = ev64['loss'][rows]
    print(what, 'loss rel vs fp64 %.2e (fp32 oracle %.2e)' % (relerr(loss, ref_loss), relerr(ev['loss'][rows], ref_loss)))
    for i, k in enumerate(TERMS):
        assert relerr(terms[:, i], ev64['terms'][k][rows]) < 1e-4, (what, k)
    assert relerr(loss, ref_loss) < 1e-4, what
    names = dict(transl='global_transl', scale='body_scale')
    B = len(loss)
    for k, gv in pm.split_theta(torch.from_numpy(got['grad'])).items():
        ok = names.get(k, k)
        ref64, ref32 = ev64['grads'][ok][rows].reshape(B, -1), ev['grads'][ok][rows].reshape(B, -1)
        e, e32 = relerr(gv.numpy(), ref64), relerr(ref32, ref64)
        assert e < max(2e-4, 20 * e32), (what, k, e, e32)


@pytest.mark.parametrize('tc', [True, False], ids=['tc', 'ffma'])
@pytest.mark.parametrize('fused', [True, False], ids=['fused', 'unfused'])
@pytest.mark.parametrize('mt,nv,imsize', GRID, ids=['%s-nv%d-%dpx' % g for g in GRID])
def test_objective_and_gradient(views, mt, nv, imsize, fused, tc):
    """One evaluation of the fit's own objective (k_frame_loss_bwd, fused) or of the all-vertex loop's (k_keypoint_loss,
    unfused) against the oracle: per-frame loss, the four loss terms and every group of d loss / d theta."""
    pm = views('model', mt, tc)
    sc = views('scene', mt, nv, imsize, NB)
    p, ev, ev64 = views('oracle', mt, nv, imsize, NB)
    kp, cams = _inputs(sc, mt)
    got = _evaluate(pm, _theta(pm, p).cuda(), kp, cams, nv, imsize, fused)
    shape = _frame_shape(pm, nv, NB) if fused else 'k_keypoint_loss'
    _check_oracle(pm, got, ev, ev64, np.arange(NB), '%s nv=%d %dpx %s %s' % (mt, nv, imsize, 'tc' if tc else 'ffma', shape))


LAUNCH = [('smplx', 4), ('smplx', 8), ('smplx', 12), ('smplx', 6), ('smplx', 48), ('smpl', 4), ('smpl', 48)]


@pytest.mark.parametrize('tc', [True, False], ids=['tc', 'ffma'])
@pytest.mark.parametrize('mt,nv', LAUNCH, ids=['%s-nv%d' % c for c in LAUNCH])
def test_launch_shapes(views, mt, nv, tc):
    """24 distinct frames tiled into a 2,049-frame batch, copies on both sides of the 128-frame tile boundary (127 / 128) and of
    the 2,048-frame launch-shape boundary (2047 / 2048).  The big batch runs <2,160> where the small one runs <1,224>
    (bulk-copy staging) and <0,224> where neither can stage the keypoint row; every row equals the oracle's result for its
    frame and, bit for bit, the same frame evaluated in the 24-frame batch (both shapes run the same per-frame arithmetic in
    the same order)."""
    D, B = 24, 2049
    pm = views('model', mt, tc)
    sc = views('scene', mt, nv, 512, D)
    p, ev, ev64 = views('oracle', mt, nv, 512, D)
    kp, cams = _inputs(sc, mt)
    theta = _theta(pm, p).cuda()
    small = _evaluate(pm, theta, kp, cams, nv, 512, True)
    _check_oracle(pm, small, ev, ev64, np.arange(D), '%s nv=%d B=%d %s' % (mt, nv, D, _frame_shape(pm, nv, D)))
    src = (np.arange(B) * 7) % D                       # every frame in many places, neighbours differ
    src[127] = src[128] = src[2047] = src[2048] = 2     # frame 2 (a joint without detections) across both boundaries
    src[0] = src[2046] = 1                              # frame 1 (a view without detections)
    idx = torch.from_numpy(src).cuda()
    big = _evaluate(pm, theta[idx].contiguous(), kp[idx].contiguous(), cams, nv, 512, True)
    shapes = (_frame_shape(pm, nv, D), _frame_shape(pm, nv, B))
    want = {('smplx', 6): ((0, 224), (0, 224)), ('smplx', 48): ((0, 224), (0, 224))}.get((mt, nv), ((1, 224), (2, 160)))
    assert shapes == want, shapes
    _check_oracle(pm, big, ev, ev64, src, '%s nv=%d B=%d %s' % (mt, nv, B, shapes[1]))
    for k in ('loss', 'loss_terms', 'grad'):
        bad = np.nonzero((big[k] != small[k][src]).reshape(B, -1).any(1))[0]
        assert not len(bad), '%s: rows %s of the %d-frame batch differ from the %d-frame batch' % (k, bad[:10], B, D)


def test_fit_at_1000_pixels(assets):
    """20 iterations through the drop-in SMPLify class at imsize = 1000, where 1024 / imsize is not exact in fp32, against the
    oracle's batched loop at the bounds of test_gpu_parity.py::test_fit_trajectory."""
    from bodyfitting_b200.smplify.smplify import SMPLify
    from util import make_port
    mt, nv, B, N, imsize = 'smplx', 8, 3, 20, 1000
    port = make_port(assets, mt)
    sc = _scene(port, mt, B, nv, imsize, seed=3)
    ref, trace = port.fit_batched(sc['init_betas'], sc['init_pose'], sc['c2ws'], sc['Ks'], sc['kp'], num_iters=N, imsize=imsize)
    fit = SMPLify(smpl_type=mt, num_iters=N, gender='neutral', model_data=assets(mt), gmm=assets('gmm'),
                  J_regressor_extra=assets('jx'))
    out = fit((sc['init_betas'], sc['init_pose']), list(sc['c2ws']), list(sc['Ks']), sc['kp'], None,
              use_frames=list(range(nv)), imsize=imsize)
    rel = np.abs(fit.last_trace.cpu().numpy() - trace) / np.abs(trace)
    print('fit at %d px: loss trace max rel err %.2e' % (imsize, rel.max()))
    assert rel.max() < 2e-5
    for k in ('pose', 'betas', 'global_orient', 'global_transl', 'scale'):
        assert np.abs(np.asarray(out[k]).reshape(B, -1) - np.asarray(ref[k]).reshape(B, -1)).max() < 2e-5, k
    assert relerr(out['vertices'], ref['vertices']) < 1e-5
    assert relerr(out['joints'], ref['joints']) < 1e-5


@pytest.mark.parametrize('mt', ['smpl', 'smplx'])
def test_mask_term_at_1024_pixels(assets, mt):
    """The silhouette term (test_gpu_mask.py::test_mask_term_value_and_vertex_gradient) with 1024 x 1024 masks of four views
    picked non-contiguously from a 48-view ring: per-frame value and d/d(world vertices) against the oracle."""
    from bodyfitting_b200.engine import FrameBuffers, pack_cameras
    from bodyfitting_b200.model import PreparedModel
    from bodyfitting_b200.smplify.mask import SilhouetteTerm
    from oracle import fit_port as fp
    from util import make_port
    B, nv, imsize, mask_frames = 2, 48, 1024, [0, 7, 23, 40]
    port = make_port(assets, mt)
    c2ws, Ks = syn.make_cameras(nv, focal=float(imsize), imsize=imsize, seed=21)
    gt, init = syn.make_params(mt, B, seed=21)
    K = 135 if mt == 'smplx' else 25
    evg = port.loss_and_grads(gt_param_dict(gt, mt), c2ws, Ks, np.zeros((B, nv, K, 3), np.float32), imsize=imsize)
    masks = np.stack([syn.make_masks(evg['vertices'][b], port.faces, c2ws[mask_frames], Ks[mask_frames], imsize=imsize)
                      for b in range(B)])
    pm = PreparedModel(mt, assets(mt), gmm=assets('gmm'), J_regressor_extra=assets('jx'), device='cuda')
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    fb = FrameBuffers(pm, B, full=True, Nv=nv, imsize=imsize)
    fb.t['theta'].copy_(pm.pack_theta(T(init['global_orient']), T(init['body_pose']), T(init['betas'])))
    fb.call('bf_pose_forward')
    fb.call('bf_skin_forward', 1)
    fb.t['loss'].zero_(); fb.t['grad'].zero_(); fb.t['dverts'].zero_()
    cams = pack_cameras(list(c2ws), list(Ks))
    sil = SilhouetteTerm(pm, masks, cams[mask_frames], imsize=imsize)
    sil.add(fb, 1.0)
    torch.cuda.synchronize()
    p = dict(global_orient=init['global_orient'], body_pose=init['body_pose'], betas=init['betas'])
    ev = port.loss_and_grads(p, c2ws, Ks, np.zeros((B, nv, K, 3), np.float32), imsize=imsize)
    f64 = torch.float64
    w2cs = torch.inverse(torch.as_tensor(c2ws, dtype=f64))
    Kt = torch.as_tensor(Ks, dtype=f64)
    mk = torch.as_tensor((masks > 128).astype(np.float32))
    vals, grads, smooth = [], [], []
    for b in range(B):
        v = torch.tensor(ev['vertices'][b:b + 1], dtype=f64, requires_grad=True)
        cont = [c.to(f64) for c in fp.extract_contours(mk[b])]
        vw, vK = [w2cs[f] for f in mask_frames], [Kt[f] for f in mask_frames]
        val = fp.mask_objective(cont, mk[b].to(f64), v, vw, vK, imsize, exact_cdist=True)
        val.backward()
        vals.append(float(val)); grads.append(v.grad[0, ::4].numpy())
        smooth.append(_mask_term_smooth(v.detach()[0, ::4], cont, vw, vK, imsize))
    got = sil.mask_loss.cpu().numpy()
    print(mt, 'mask term at %d px' % imsize, got, 'oracle', vals)
    assert relerr(got, np.array(vals)) < 2e-5
    assert relerr(fb.t['loss'].cpu().numpy(), np.array(vals)) < 2e-5
    g, gref, smooth = sil.dPw.cpu().numpy(), np.stack(grads), np.stack(smooth)
    print(mt, 'vertex gradient rel err %.2e on %d of %d vertices (all: %.2e)' % (relerr(g[smooth], gref[smooth]), smooth.sum(),
                                                                                  smooth.size, relerr(g, gref)))
    assert smooth.mean() > 0.98
    assert relerr(g[smooth], gref[smooth]) < 1e-4


def _mask_term_smooth(sv, contours, w2cs, Ks, imsize, tol=3e-4):
    """[Nq] bool: the sampled vertices at which the silhouette term is differentiable with a margin of `tol` pixels in every
    mask view.  Its gradient jumps where a projected vertex crosses a pixel boundary (the bilinear cells of grid_sample, the
    truncated lookup of the outside penalty, the image border) and where two vertices tie for a contour point's arg-min; an
    fp32 projection about 1e-4 pixels away from the fp64 one can land on the other side of such an edge (the fp32 oracle
    itself does, for one SMPL vertex of this scene).  About 0.5 % of the sampled vertices lie this close to an edge here.
    The value is continuous there and is compared everywhere."""
    from oracle import fit_port as fp
    ok = np.ones(sv.shape[0], bool)
    for c, w2c, K in zip(contours, w2cs, Ks):
        uv = fp.project(sv[None], w2c[None, :3, :3], w2c[None, :3, 3], K)[0].numpy()
        ok &= (np.abs(uv - 0.5 - np.round(uv - 0.5)) > tol).all(1)       # bilinear cells: pixel centres (W == imsize)
        inside = ((uv >= 0) & (uv < imsize)).all(1)
        ok &= (np.abs(uv) > tol).all(1) & (np.abs(uv - imsize) > tol).all(1)
        iq = np.nonzero(inside)[0]
        d = np.sqrt(((c.numpy().reshape(-1, 1, 2) - uv[iq][None]) ** 2).sum(-1))      # [Nc, inside]
        two = np.argsort(d, 1)[:, :2]
        gap = np.take_along_axis(d, two, 1)
        tie = gap[:, 1] - gap[:, 0] < tol
        ok[iq[two[tie].ravel()]] = False
        win = iq[two[:, 0]]                                               # arg-min vertices: their pixel picks the penalty
        ok[win[(np.abs(uv[win] - np.round(uv[win])) <= tol).any(1)]] = False
    return ok


def test_multiview_keypoint_loss_48_views(assets):
    """smplify.loss.multiview_keypoint_loss (k_kp_world) for one SMPL-X frame at 48 views, five of them None (no detections:
    they still count in the 1 / Nv), against the reference-style objective of the oracle in fp64: value, terms, gradients
    (test_gpu_ops.py::test_multiview_keypoint_loss_composed at 8 views)."""
    from bodyfitting_b200.models.smpl import create_smplx
    from bodyfitting_b200.smplify.loss import multiview_keypoint_loss
    from bodyfitting_b200.smplify.prior import MaxMixturePrior
    from oracle import fit_port as fp
    from util import make_port
    mt, nv = 'smplx', 48
    port = make_port(assets, mt, dtype=torch.float64)
    sc = _scene(make_port(assets, mt), mt, 1, nv, 512, seed=17)
    views = syn.keypoints_to_openpose(sc['kp'][0], mt)
    for v in (0, 5, 6, 29, 47):
        views[v] = None
    p = perturbed_params(mt, 1, seed=18)
    pr = {k: torch.tensor(v, dtype=torch.float64, requires_grad=True) for k, v in p.items()}
    full = dict(pr)
    full['jaw_pose'] = torch.zeros(1, 1, 3, dtype=torch.float64)
    full['leye_pose'] = pr['leye_pose'].view(1, 1, 3); full['reye_pose'] = pr['reye_pose'].view(1, 1, 3)
    o = port.forward_model(full)
    jw = (o.joints + pr['global_transl']) * pr['body_scale'] * 0.3
    w2cs = torch.inverse(torch.tensor(np.array(sc['c2ws']), dtype=torch.float64))
    ref, terms = fp.keypoint_objective(w2cs, [np.asarray(k, np.float64) for k in sc['Ks']], views, jw, pr['body_pose'], pr['betas'],
                                       port.prior, 512, True)
    ref.backward()
    pg = {k: torch.tensor(v).cuda().requires_grad_(True) for k, v in p.items()}
    model = create_smplx(model_data=assets(mt))
    out = model(global_orient=pg['global_orient'], body_pose=pg['body_pose'], betas=pg['betas'], leye_pose=pg['leye_pose'],
                reye_pose=pg['reye_pose'], left_hand_pose=pg['left_hand_pose'], right_hand_pose=pg['right_hand_pose'])
    jwg = (out.joints + pg['global_transl'][:, None]) * pg['body_scale'][:, None] * 0.3
    prior = MaxMixturePrior(gmm=assets('gmm'))
    tot, losses = multiview_keypoint_loss(w2cs.float(), list(sc['Ks']), views, jwg, pg['body_pose'], pg['betas'], list(range(nv)),
                                          prior, imsize=512, use_hand_face=True)
    tot.backward()
    print('48 views: loss rel %.2e' % relerr(float(tot), float(ref)))
    assert relerr(float(tot), float(ref)) < 1e-5
    for k in TERMS:
        assert relerr(losses[k], terms[k].detach().numpy()) < 1e-5, k
    for k in p:
        e = relerr(pg[k].grad.cpu().numpy(), pr[k].grad.numpy())
        print('   grad %-16s %.2e' % (k, e))
        assert e < 2e-4, k
