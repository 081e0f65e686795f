"""ORACLE -- TEST INFRASTRUCTURE ONLY.  Never imported by the product path.

Standalone CPU (torch) restatement of the reference's multi-view SMPLify fitting path,
so that the GPU box (where /root/reference does not exist) has a checker and a CPU
baseline.  Each function cites the reference lines it follows:

  project()            smplify/loss.py:22-43    perspective_projection
  gmof()               smplify/loss.py:45-51
  angle_prior()        smplify/loss.py:54-61
  reprojection()       smplify/loss.py:132-136  (incl. the [N,1]x[N] broadcast of the
                                                 hand / face confidences at :168,:173,:179)
  keypoint_objective() smplify/loss.py:139-230  multiview_keypoint_loss
  GMMPrior             smplify/prior.py:100-196 MaxMixturePrior (merged likelihood)
  SpinSMPL             models/smpl.py:56-83     SMPL wrapper (+9 regressed joints, 49-joint map)
  FitPort.fit_frame()  smplify/smplify.py:84-226 SMPLify.__call__ for ONE frame, same op
                                                 sequence (per-view Python loop, 9-group Adam)
  extract_contours()   smplify/loss.py:73-83    extract_countours
  mask_objective()     smplify/loss.py:85-130   multview_mask_loss (silhouette term, use_mask=True)
  FitPort.fit_batched()the same objective for B independent frames at once (the
                       reference supports B=1 only, smplify/smplify.py:189-190); validated
                       against fit_frame per frame in tests/test_oracle.py

PARITY STATUS: pinned against the verbatim reference files run in the authoring
container (oracle/ref_harness.py -> tests/golden/*.npz, tests/test_oracle.py); the
LBS arithmetic underneath (oracle/smplx_port.py) restates the un-vendored third-party
``smplx`` package and is unpinned against it.
"""
import numpy as np
import torch
import torch.nn as nn

from bodyfitting_b200 import constants as C
from oracle import smplx_port as sp


def project(points, rotation, translation, K):
    """points [B,N,3], rotation [1|B,3,3], translation [1|B,3], K [3,3] -> [B,N,2];
    no epsilon, no clamp (loss.py:38-43)."""
    B = points.shape[0]
    if isinstance(K, np.ndarray):
        K = torch.tensor(K, dtype=points.dtype, device=points.device)
    K = K[None].expand(B, -1, -1)
    pc = torch.einsum('bij,bkj->bki', rotation.expand(B, -1, -1), points) + translation.unsqueeze(1)
    ph = torch.einsum('bij,bkj->bki', K, pc)
    return (ph / ph[:, :, -1].unsqueeze(-1))[:, :, :-1]


def gmof(x, sigma):
    x2, s2 = x ** 2, sigma ** 2
    return (s2 * x2) / (s2 + x2)


def angle_prior(pose):
    sign = torch.tensor(C.ANGLE_PRIOR_SIGNS, dtype=pose.dtype, device=pose.device)
    return torch.exp(pose[:, C.ANGLE_PRIOR_IDXS] * sign) ** 2


def reprojection(cord, cord_gt, conf, scale_coeff, sigma):
    """``conf`` is [N] for the body and [N,1] for hands / face, exactly as the reference
    passes it: the latter broadcasts to [N,N], i.e. (sum_i conf_i^2) * (sum_j rho_j)."""
    err = gmof((cord_gt - cord) / scale_coeff, sigma)
    return ((conf ** 2) * err.sum(dim=-1)).sum(dim=-1)


class GMMPrior(nn.Module):
    """min_m [ 0.5 d^T P_m d - log(nll_w_m) ],  nll_w = w / ((2 pi)^(69/2) sqrtdet/min sqrtdet)."""

    def __init__(self, gmm, dtype=torch.float32):
        super().__init__()
        npd = np.float32 if dtype == torch.float32 else np.float64
        means = np.asarray(gmm['means']).astype(npd)
        covs = np.asarray(gmm['covars']).astype(npd)
        self.register_buffer('means', torch.tensor(means, dtype=dtype))
        prec = np.stack([np.linalg.inv(c) for c in covs]).astype(npd)
        self.register_buffer('precisions', torch.tensor(prec, dtype=dtype))
        sqrdets = np.array([np.sqrt(np.linalg.det(c)) for c in gmm['covars']])
        const = (2 * np.pi) ** (69 / 2.)
        nllw = np.asarray(gmm['weights'] / (const * (sqrdets / sqrdets.min())))
        self.register_buffer('nll_weights', torch.tensor(nllw, dtype=dtype).unsqueeze(0))

    def forward(self, pose, betas=None):
        d = pose.unsqueeze(1) - self.means
        pd = torch.einsum('mij,bmj->bmi', self.precisions, d)
        ll = 0.5 * (pd * d).sum(-1) - torch.log(self.nll_weights)
        return torch.min(ll, dim=1)[0]


class SpinSMPL(sp.SMPLLayer):
    """models/smpl.py:56-83: 45 joints ++ J_regressor_extra @ vertices, re-indexed to 49."""

    def __init__(self, data, J_regressor_extra, **kw):
        super().__init__(data, create_transl=True, **kw)
        self.register_buffer('J_regressor_extra', torch.tensor(np.asarray(J_regressor_extra), dtype=torch.float32))
        self.joint_map = torch.tensor(C.SPIN_JOINT_MAP, dtype=torch.long)

    def forward(self, *a, **kw):
        out = super().forward(*a, **kw)
        extra = sp.vertices2joints(self.J_regressor_extra.to(out.vertices.dtype), out.vertices)
        out.joints_ori = out.joints
        out.joints = torch.cat([out.joints, extra], dim=1)[:, self.joint_map, :]
        return out


class _Mapper(nn.Module):
    def __init__(self, idx):
        super().__init__()
        self.register_buffer('idx', torch.tensor(np.asarray(idx), dtype=torch.long))

    def forward(self, joints, **kw):
        return torch.index_select(joints, 1, self.idx)


def build_model(smpl_type, model_data, J_regressor_extra=None, dtype=torch.float32, age='adult', kid_template='',
                num_betas=10, num_expression=10):
    """Body model exactly as SMPLify.__init__ builds it (smplify/smplify.py:50-80); ``num_betas`` / ``num_expression`` (SMPL-X)
    select other shape-space sizes (the reference uses smplx's defaults, 10 / 10)."""
    if smpl_type == 'smpl':
        m = SpinSMPL(model_data, J_regressor_extra, dtype=dtype, age=age, kid_template_path=kid_template, num_betas=num_betas)
    else:
        mapper = _Mapper(C.smpl_to_openpose('smplx', use_hands=True, use_face=True, use_face_contour=True,
                                            openpose_format='coco25'))
        m = sp.SMPLXLayer(model_data, num_betas=num_betas, num_expression_coeffs=num_expression, joint_mapper=mapper,
                          use_face_contour=True, create_transl=False, dtype=dtype)
    return m


def keypoint_objective(w2cs, Ks, views, model_joints, poses, betas, prior, imsize, use_hand_face,
                       sigma=C.GMOF_SIGMA):
    """One frame (B=1), per-view Python loop as in loss.py:156-217.  ``views`` = list of
    OpenPose dicts (or None).  Returns (scalar total, dict of the four terms)."""
    body, hand, face = [], [], []
    sc = imsize / 1024
    dev = model_joints.device
    for i in range(len(views)):
        if views[i] is None:
            continue
        w2c = w2cs[i]
        proj = project(model_joints, w2c[:3, :3].unsqueeze(0), w2c[:3, 3].unsqueeze(0), Ks[i])
        kp = torch.from_numpy(np.asarray(views[i]['pose'])).to(model_joints.dtype).to(dev)
        gt, conf = torch.split(kp, [2, 1], dim=-1)
        body.append(reprojection(proj[0, :25], gt, conf.squeeze(-1), sc, sigma))
        if use_hand_face:
            for key, lo, hi, dst in (('hand_left', 25, 46, hand), ('hand_right', 46, 67, hand)):
                if key in views[i]:
                    kp = torch.from_numpy(np.asarray(views[i][key])).to(model_joints.dtype).to(dev)
                    gt, conf = torch.split(kp, [2, 1], dim=-1)
                    dst.append(reprojection(proj[0, lo:hi], gt, conf, sc, sigma))
            if 'face' in views[i]:
                kp = torch.from_numpy(np.asarray(views[i]['face'])[C.FACE_MAPPING]).to(model_joints.dtype).to(dev)
                gt, conf = torch.split(kp, [2, 1], dim=-1)
                face.append(reprojection(proj[0, 67:], gt, conf, sc, sigma))
    nv = len(views)
    loss_2d = torch.sum(torch.stack(body, dim=0)) / nv
    if use_hand_face:
        loss_2d = loss_2d + torch.sum(torch.stack(hand, dim=0)) / nv
        loss_2d = loss_2d + torch.sum(torch.stack(face, dim=0)) / nv
        poses = torch.cat([poses, torch.zeros_like(poses[:, :6])], dim=-1)
    pose_l = (C.POSE_PRIOR_WEIGHT ** 2) * prior(poses, None)
    angle_l = (C.ANGLE_PRIOR_WEIGHT ** 2) * angle_prior(poses).sum(dim=-1)
    shape_l = (C.SHAPE_PRIOR_WEIGHT ** 2) * (betas ** 2).sum(dim=-1)
    total = loss_2d + pose_l + angle_l + shape_l
    return total.sum(), dict(reprojection_loss=loss_2d, pose_prior_loss=pose_l, angle_prior_loss=angle_l,
                             shape_prior_loss=shape_l)


def extract_contours(masks):
    """smplify/loss.py:73-83 extract_countours: per mask the longest external contour (cv2.RETR_EXTERNAL,
    CHAIN_APPROX_NONE) as a float tensor [Nc,1,2] of (x, y) pixels.  The reference unpacks OpenCV 3's three return
    values (:79); OpenCV 4 returns (contours, hierarchy) -- same contours."""
    import cv2
    out = []
    for mask in masks:
        res = cv2.findContours(mask.cpu().numpy().astype(np.uint8) * 255, cv2.RETR_EXTERNAL, cv2.CHAIN_APPROX_NONE)
        contour = res[-2]
        contour = contour[int(np.argmax(np.array([a.shape[1] for a in contour])))]
        out.append(torch.tensor(contour, dtype=torch.float32, device=masks.device))
    return out


def mask_objective(contours, masks, verts, w2cs, Ks, imsize=512, epsilon=10, exact_cdist=False):
    """smplify/loss.py:85-130 multview_mask_loss for ONE frame: ``verts`` [1,V,3] world vertices, ``masks`` [Nm,H,W]
    float 0/1, ``contours`` from extract_contours, ``w2cs`` / ``Ks`` of the mask views.
      * every 4th vertex is projected (:100,:105);
      * the contour is [Nc,1,2], so ``cdist(points[1,Np,2], contour[1,Nc,1,2])`` broadcasts to [Nc,Np,1] and ``min(dist, 1)``
        picks, for every CONTOUR point, the closest projected in-image vertex (:111-112);
      * that vertex's pixel decides the penalty: 10 x if it falls outside the mask, 1 x otherwise (:115-118);
      * plus 10 x the bilinear samples of (1 - mask) at every projected vertex (grid_sample, align_corners=False) (:124-128).
    ``exact_cdist``: direct |x - c| instead of torch's matmul-based expansion (what the CUDA kernel computes)."""
    scale_coeff = 1
    sv = verts.squeeze(0)[::4]
    losses, uvs = [], []
    for i in range(len(contours)):
        pose, K, contour, mask = w2cs[i], Ks[i], contours[i], masks[i]
        pp = project(sv.unsqueeze(0), pose[None, :3, :3], pose[None, :3, 3], K).squeeze(0)
        inside = torch.prod((pp < imsize) & (pp >= 0), dim=1).squeeze(0) > 0
        ip = pp[inside]
        uvs.append(pp)
        if exact_cdist:
            dist = torch.cdist(ip.unsqueeze(0) / scale_coeff, contour.unsqueeze(0) / scale_coeff,
                               compute_mode='donot_use_mm_for_euclid_dist').squeeze(0)
        else:
            dist = torch.cdist(ip.unsqueeze(0) / scale_coeff, contour.unsqueeze(0) / scale_coeff).squeeze(0)
        mindist, index = torch.min(dist, 1)
        cp = ip[index[:, 0]].long()
        outside = (mask[cp[:, 1], cp[:, 0]] < 0.1).to(verts.dtype)[:, None]
        coeff = outside * (epsilon - 1) + 1
        losses.append(torch.sum(mindist * coeff))
    total = torch.stack(losses).sum()
    uvs = torch.stack(uvs, dim=0).view(len(masks), -1, 1, 2) / imsize * 2 - 1
    binary = torch.nn.functional.grid_sample(1 - masks[:, None], uvs, align_corners=False)
    return total + torch.sum(binary) * epsilon


def effective_weights(kp, use_hand_face):
    """kp [B,Nv,K,3] -> w [B,Nv,K]: conf^2 for the body joints; for each hand / the face
    the reference's broadcast makes every joint of the group weigh sum_i conf_i^2."""
    c2 = kp[..., 2] ** 2
    w = c2.clone()
    if use_hand_face:
        for lo, hi in ((25, 46), (46, 67), (67, 135)):
            w[..., lo:hi] = c2[..., lo:hi].sum(-1, keepdim=True)
    return w


def batched_objective(w2cs, Ks, kp, model_joints, poses, betas, prior, imsize, use_hand_face,
                      sigma=C.GMOF_SIGMA):
    """B independent frames: per-frame loss [B] (data + priors) with the semantics of
    ``keypoint_objective`` applied to each frame separately."""
    B, Nv = kp.shape[:2]
    sc = imsize / 1024
    model_joints = model_joints[:, :kp.shape[2]]          # SMPL: 49 joints, the loss reads [:25]
    R, t = w2cs[:, :3, :3], w2cs[:, :3, 3]
    pc = torch.einsum('vij,bkj->bvki', R, model_joints) + t[None, :, None, :]
    ph = torch.einsum('vij,bvkj->bvki', Ks, pc)
    uv = ph[..., :2] / ph[..., 2:3]
    rho = gmof((kp[..., :2] - uv) / sc, sigma).sum(-1)                     # [B,Nv,K]
    data = (effective_weights(kp, use_hand_face) * rho).sum(dim=(1, 2)) / Nv
    if use_hand_face:
        poses = torch.cat([poses, torch.zeros_like(poses[:, :6])], dim=-1)
    pose_l = (C.POSE_PRIOR_WEIGHT ** 2) * prior(poses, None)
    angle_l = (C.ANGLE_PRIOR_WEIGHT ** 2) * angle_prior(poses).sum(dim=-1)
    shape_l = (C.SHAPE_PRIOR_WEIGHT ** 2) * (betas ** 2).sum(dim=-1)
    return data + pose_l + angle_l + shape_l, dict(reprojection_loss=data, pose_prior_loss=pose_l,
                                                   angle_prior_loss=angle_l, shape_prior_loss=shape_l)


class FitPort(object):
    def __init__(self, smpl_type, model_data, gmm, J_regressor_extra=None, dtype=torch.float32,
                 constant_scale=C.CONSTANT_SCALE_NO_SCAN, device='cpu', age='adult', kid_template='', num_betas=10,
                 num_expression=10):
        """``device='cuda'``: the same eager op sequence on the GPU (the reference's default device, smplify.py:29) --
        bench.py's second, non-target baseline; parity is always checked with the CPU path.  ``num_betas`` /
        ``num_expression``: shape-space sizes of the body model (build_model)."""
        self.smpl_type = smpl_type
        self.use_hand_face = smpl_type == 'smplx'
        self.dtype = dtype
        self.device = torch.device(device)
        self.prior = GMMPrior(gmm, dtype=dtype).to(self.device)
        self.age = age
        self.model = build_model(smpl_type, model_data, J_regressor_extra, dtype=dtype, age=age, kid_template=kid_template,
                                 num_betas=num_betas, num_expression=num_expression).to(self.device)
        self.num_betas = self.model.num_betas          # the kid model: num_betas + 1
        if hasattr(self.model, 'joint_map'):
            self.model.joint_map = self.model.joint_map.to(self.device)
        self.constant_scale = constant_scale
        self.faces = np.asarray(self.model.faces).astype(np.int32)

    # -- shared ---------------------------------------------------------------
    def _init_params(self, init_betas, init_poses, B):
        dt, dev = self.dtype, self.device
        init_poses = torch.as_tensor(init_poses, dtype=dt).reshape(B, -1).to(dev)
        nb = 69 if self.smpl_type == 'smpl' else 63
        p = dict(body_pose=init_poses[:, 3:3 + nb].detach().clone(),
                 betas=(torch.as_tensor(init_betas, dtype=dt).reshape(B, -1).to(dev).detach().clone() if self.age == 'adult'
                        else torch.zeros(B, self.num_betas, dtype=dt, device=dev)),     # smplify.py:112-115
                 global_orient=init_poses[:, :3].detach().clone(),
                 global_transl=torch.zeros(B, 3, dtype=dt, device=dev), body_scale=torch.ones(B, 1, dtype=dt, device=dev),
                 jaw_pose=torch.zeros(B, 1, 3, dtype=dt, device=dev), leye_pose=torch.zeros(B, 1, 3, dtype=dt, device=dev),
                 reye_pose=torch.zeros(B, 1, 3, dtype=dt, device=dev), left_hand_pose=torch.zeros(B, 6, dtype=dt, device=dev),
                 right_hand_pose=torch.zeros(B, 6, dtype=dt, device=dev))
        for v in p.values():
            v.requires_grad_(True)
        return p

    def _optimizer(self, p):
        groups = [{'params': p['global_transl'], 'lr': C.LR_TRANSL_SCALE},
                  {'params': p['body_scale'], 'lr': C.LR_TRANSL_SCALE},
                  {'params': p['body_pose']}, {'params': p['betas']}, {'params': p['global_orient']},
                  {'params': p['leye_pose']}, {'params': p['reye_pose']},
                  {'params': p['left_hand_pose']}, {'params': p['right_hand_pose']}]
        return torch.optim.Adam(groups, lr=C.LR_DEFAULT, betas=C.ADAM_BETAS)   # jaw_pose: not optimised (:118 vs :167-173)

    def forward_model(self, p):
        return self.model(global_orient=p['global_orient'], body_pose=p['body_pose'], betas=p['betas'],
                          jaw_pose=p['jaw_pose'], leye_pose=p['leye_pose'], reye_pose=p['reye_pose'],
                          left_hand_pose=p['left_hand_pose'], right_hand_pose=p['right_hand_pose'],
                          return_full_pose=True)

    def world(self, out, p):
        j = (out.joints + p['global_transl'].unsqueeze(1)) * p['body_scale'].unsqueeze(1) * self.constant_scale
        v = (out.vertices + p['global_transl'].unsqueeze(1)) * p['body_scale'].unsqueeze(1) * self.constant_scale
        return j, v

    def _result(self, p, out, joints, verts, squeeze):
        sq = (lambda t: t.detach().cpu().squeeze(0).numpy()) if squeeze else (lambda t: t.detach().cpu().numpy())
        return dict(vertices=sq(verts), joints=sq(joints), pose=sq(p['body_pose']), betas=sq(p['betas']),
                    global_orient=sq(p['global_orient']), faces=self.faces,
                    global_transl=sq(p['global_transl'] * p['body_scale']), scale=sq(p['body_scale']),
                    full_pose=sq(out.full_pose),
                    leye_pose=sq(p['leye_pose']), reye_pose=sq(p['reye_pose']),
                    left_hand_pose=sq(p['left_hand_pose']), right_hand_pose=sq(p['right_hand_pose']))

    # -- one frame, reference op sequence ---------------------------------------
    def fit_frame(self, init_betas, init_poses, c2ws, Ks, views, num_iters=100, imsize=512, masks=None, mask_frames=None):
        """``masks`` [Nm,H,W] uint8 + ``mask_frames``: also the silhouette term (use_mask=True, smplify.py:137-144,196-199)."""
        p = self._init_params(init_betas, init_poses, 1)
        w2cs = torch.inverse(torch.from_numpy(np.array(c2ws)).to(self.dtype).to(self.device))
        Ks = [np.asarray(k) for k in Ks]
        opt = self._optimizer(p)
        trace = []
        if masks is not None:
            mk = torch.from_numpy((np.array(masks) > 128).astype(np.float32)).to(self.dtype)
            use_frames = list(range(len(c2ws)))
            mask_w2cs = [w2cs[use_frames.index(f)] for f in mask_frames]
            mask_Ks = [Ks[use_frames.index(f)] for f in mask_frames]
            contours = extract_contours(mk)
        for i in range(num_iters):
            out = self.forward_model(p)
            # reference broadcasting for B=1: [1,K,3] + [1,3] and * [1,1]
            joints = (out.joints + p['global_transl']) * p['body_scale'] * self.constant_scale
            verts = (out.vertices + p['global_transl']) * p['body_scale'] * self.constant_scale
            loss, _ = keypoint_objective(w2cs, Ks, views, joints, p['body_pose'], p['betas'], self.prior,
                                         imsize, self.use_hand_face)
            if masks is not None and i > (num_iters // 3):
                loss = loss + 5 * mask_objective(contours, mk, verts, mask_w2cs, mask_Ks, imsize) + 5 * 0
            trace.append(float(loss.detach()))
            opt.zero_grad()
            loss.backward()
            opt.step()
        return self._result(p, out, joints, verts, True), trace

    # -- B frames at once ---------------------------------------------------------
    def fit_batched(self, init_betas, init_poses, c2ws, Ks, kp, num_iters=100, imsize=512, hook=None,
                    temporal_weight=0.0):
        kp = torch.as_tensor(kp, dtype=self.dtype)
        B = kp.shape[0]
        p = self._init_params(init_betas, init_poses, B)
        w2cs = torch.inverse(torch.as_tensor(np.array(c2ws), dtype=self.dtype))
        Kt = torch.as_tensor(np.array(Ks), dtype=self.dtype)
        opt = self._optimizer(p)
        trace = []
        for it in range(num_iters):
            out = self.forward_model(p)
            joints, verts = self.world(out, p)
            per_frame, _ = batched_objective(w2cs, Kt, kp, joints, p['body_pose'], p['betas'], self.prior,
                                             imsize, self.use_hand_face)
            if temporal_weight > 0 and B > 1:
                # builder-defined sequence term (BASELINE config 4, not in the reference): frame f pays the edge (f-1, f)
                pvec = torch.cat([p['global_transl'], p['global_orient'], p['body_pose']], dim=1)
                edge = temporal_weight * ((pvec[1:] - pvec[:-1]) ** 2).sum(dim=1)
                per_frame = per_frame + torch.cat([edge.new_zeros(1), edge])
            trace.append(per_frame.detach().clone())
            opt.zero_grad()
            per_frame.sum().backward()
            if hook is not None:
                hook(it, p, out, joints, verts, per_frame)
            opt.step()
        return self._result(p, out, joints, verts, False), torch.stack(trace).numpy()

    # -- keypoints + silhouette term (use_mask=True, smplify/smplify.py:137-144,196-199,210) ------------
    def fit_batched_mask(self, init_betas, init_poses, c2ws, Ks, kp, masks, mask_frames, num_iters=12, imsize=512,
                         exact_cdist=False):
        """B frames, each with its own masks [B,Nm,H,W] (uint8 0..255) of the views ``mask_frames`` (indices into the
        camera list; the reference looks them up through use_frames, smplify.py:141-142):
        loss_f = keypoint objective + 5 x mask objective for i > num_iters // 3."""
        kp = torch.as_tensor(kp, dtype=self.dtype)
        B = kp.shape[0]
        p = self._init_params(init_betas, init_poses, B)
        w2cs = torch.inverse(torch.as_tensor(np.array(c2ws), dtype=self.dtype))
        Kt = torch.as_tensor(np.array(Ks), dtype=self.dtype)
        mk = torch.as_tensor((np.asarray(masks) > 128).astype(np.float32)).to(self.dtype)          # smplify.py:139
        contours = [[c.to(self.dtype) for c in extract_contours(mk[b])] for b in range(B)]
        mw2c = [w2cs[f] for f in mask_frames]
        mK = [Kt[f] for f in mask_frames]
        opt = self._optimizer(p)
        trace, mls = [], []
        for it in range(num_iters):
            out = self.forward_model(p)
            joints, verts = self.world(out, p)
            per_frame, _ = batched_objective(w2cs, Kt, kp, joints, p['body_pose'], p['betas'], self.prior, imsize,
                                             self.use_hand_face)
            if it > (num_iters // 3):
                ml = torch.stack([mask_objective(contours[b], mk[b], verts[b:b + 1], mw2c, mK, imsize, exact_cdist=exact_cdist)
                                  for b in range(B)])
                per_frame = per_frame + 5 * ml
                mls.append(ml.detach().clone())
            trace.append(per_frame.detach().clone())
            opt.zero_grad()
            per_frame.sum().backward()
            opt.step()
        res = self._result(p, out, joints, verts, False)
        return res, torch.stack(trace).numpy(), (torch.stack(mls).numpy() if mls else None)

    # -- keypoints + point-to-scan term (use_mesh=True, smplify/smplify.py:146-156,205-210) ----------
    def fit_batched_scan(self, init_betas, init_poses, c2ws, Ks, kp, scan_verts, scan_faces, num_iters=12, imsize=512):
        """B frames against ONE scan; the CUDA-only mesh_grid closest point is replaced by the exact fp64
        brute force (oracle/geometry_port.py); per frame pc = |P - C.detach()|_F / scan_height * imsize,
        loss = body + 5 pc for i > num_iters // 3."""
        from oracle import geometry_port as gp
        kp = torch.as_tensor(kp, dtype=self.dtype)
        B = kp.shape[0]
        sv = np.asarray(scan_verts, dtype=np.float64)
        scan_height = float((sv.max(0) - sv.min(0))[1])
        cs = scan_height / 1.7
        p = self._init_params(init_betas, init_poses, B)
        w2cs = torch.inverse(torch.as_tensor(np.array(c2ws), dtype=self.dtype))
        Kt = torch.as_tensor(np.array(Ks), dtype=self.dtype)
        opt = self._optimizer(p)
        trace, pcs = [], []
        for it in range(num_iters):
            out = self.forward_model(p)
            joints = (out.joints + p['global_transl'].unsqueeze(1)) * p['body_scale'].unsqueeze(1) * cs
            verts = (out.vertices + p['global_transl'].unsqueeze(1)) * p['body_scale'].unsqueeze(1) * cs
            per_frame, _ = batched_objective(w2cs, Kt, kp, joints, p['body_pose'], p['betas'], self.prior, imsize,
                                             self.use_hand_face)
            if it > (num_iters // 3):
                cp, _, _ = gp.closest_points_bruteforce(verts.detach().reshape(-1, 3).numpy(), sv, scan_faces)
                cp = torch.as_tensor(cp.reshape(B, -1, 3), dtype=self.dtype)
                pc = torch.sqrt(((verts - cp) ** 2).sum(dim=(1, 2))) / scan_height * imsize
                per_frame = per_frame + 5 * pc
                pcs.append(pc.detach().clone())
            trace.append(per_frame.detach().clone())
            opt.zero_grad()
            per_frame.sum().backward()
            opt.step()
        res = self._result(p, out, joints, verts, False)
        return res, torch.stack(trace).numpy(), (torch.stack(pcs).numpy() if pcs else None)

    # -- single evaluation: loss + grads (for kernel gradient parity) ---------------
    def loss_and_grads(self, params, c2ws, Ks, kp, imsize=512):
        kp = torch.as_tensor(kp, dtype=self.dtype)
        B = kp.shape[0]
        p = {}
        for k, v in params.items():
            p[k] = torch.as_tensor(v, dtype=self.dtype).clone().requires_grad_(True)
        for k, shape in (('jaw_pose', (B, 1, 3)), ('leye_pose', (B, 1, 3)), ('reye_pose', (B, 1, 3)),
                         ('left_hand_pose', (B, 6)), ('right_hand_pose', (B, 6)),
                         ('global_transl', (B, 3))):
            if k not in p:
                p[k] = torch.zeros(shape, dtype=self.dtype, requires_grad=True)
            else:
                p[k] = p[k].reshape(shape).detach().clone().requires_grad_(True)
        if 'body_scale' not in p:
            p['body_scale'] = torch.ones(B, 1, dtype=self.dtype, requires_grad=True)
        w2cs = torch.inverse(torch.as_tensor(np.array(c2ws), dtype=self.dtype))
        Kt = torch.as_tensor(np.array(Ks), dtype=self.dtype)
        out = self.forward_model(p)
        joints, verts = self.world(out, p)
        per_frame, terms = batched_objective(w2cs, Kt, kp, joints, p['body_pose'], p['betas'], self.prior,
                                             imsize, self.use_hand_face)
        per_frame.sum().backward()
        grads = {k: (v.grad.detach().numpy() if v.grad is not None else None) for k, v in p.items()}
        return dict(loss=per_frame.detach().numpy(), joints=joints.detach().numpy(), vertices=verts.detach().numpy(),
                    model_joints=out.joints.detach().numpy(), model_vertices=out.vertices.detach().numpy(),
                    full_pose=out.full_pose.detach().numpy(), grads=grads,
                    terms={k: v.detach().numpy() for k, v in terms.items()})
