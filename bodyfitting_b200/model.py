"""Host-side preparation of the body-model tables the kernels consume.

Everything here runs once per model (numpy, fp64 where a reduction is pre-folded) and
produces device tensors plus the ``BfModel`` struct handed to the C ABI:

* ``Bm`` -- ONE blend matrix [Kp, 3 n_pad] whose rows are posedirs (P), shapedirs^T (NS) and
  v_template (1), so that v_posed = [pose_feature | shape | 1] @ Bm is a single dense
  contraction (smplx.lbs: blend_shapes + pose_offsets matmul + template add).
* ``Jt`` / ``Jd`` -- J_regressor folded into the template / shape directions
  (J_regressor @ (v_template + S beta) == Jt + Jd beta).
* ELL skinning weights, CSR joint->vertex lists (for dA), the output-joint table
  (chain joints, vertex picks, barycentric landmarks, yaw-dependent contour landmarks,
  regressed extra joints) and its inverse, CSR by target, used by the atomics-free backward.
* the *active vertex set*: the union of vertices the keypoint loss can ever touch
  (21 picked + 51x3 static + all 79x17x3 contour candidates for SMPL-X, 11 for SMPL).
  Gradients of the keypoint objective are exactly zero on every other vertex, so the
  fitting loop runs blend + skinning only on this set; the full set is used for the
  operator surface (SMPL.forward) and for the final vertices.

Reference: models/smpl.py:56-83, models/utils.py:32-141, smplify/prior.py:127-174,
smplx (un-vendored) as restated in oracle/smplx_port.py.
"""
import ctypes as C
import os
import warnings

import numpy as np
import torch

from . import _lib
from . import constants as K


MAX_NS = 20         # betas + expression coefficients per frame (BF_MAXNS, csrc/bf_common.cuh)
MAX_NP = 100        # theta entries per frame without the face block, counted with 6 hand components (BF_MAXNP)


def _round_up(x, m):
    return (x + m - 1) // m * m


def split_tf32(x):
    """x = hi + lo with hi the round-to-nearest TF32 value (low 13 mantissa bits zero, what
    ``cvt.rna.tf32.f32`` produces) and lo the exact fp32 remainder: operands of the 3xTF32 GEMMs."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    u = x.view(np.uint32)
    hi = ((u + np.uint32(0x1000)) & np.uint32(0xFFFFE000)).view(np.float32)
    return hi, (x - hi).astype(np.float32)


def load_model_data(path_or_dict, model_type=None, gender='neutral'):
    """Accepts a dict (e.g. synthetic.make_model) or a path: a ``.npz``/``.pkl`` file, or a
    folder laid out like the reference's ``data/`` (data/smpl/SMPL_NEUTRAL.npz ...)."""
    if isinstance(path_or_dict, dict):
        return path_or_dict
    path = path_or_dict
    if os.path.isdir(path):
        mt = model_type or 'smpl'
        base = os.path.basename(os.path.normpath(path))
        folder = path if base == mt else os.path.join(path, mt)
        want = [os.path.join(folder, '%s_%s.%s' % (mt.upper(), str(gender).upper(), ext)) for ext in ('npz', 'pkl')]
        cands = want + [os.path.join(folder, '%s_NEUTRAL.%s' % (mt.upper(), ext)) for ext in ('npz', 'pkl')]
        found = [c for c in cands if os.path.exists(c)]
        if not found:
            raise FileNotFoundError('no %s model file under %s (tried %s)' % (mt, path, cands))
        path = found[0]
        if path not in want:        # the reference would fail here (SMPL(gender=...) / smplx.create(gender=...)); say so loudly
            warnings.warn('no %s model for gender %r under %s: using %s' % (mt, gender, folder, os.path.basename(path)))
    if path.endswith('.pkl'):
        import pickle
        with open(path, 'rb') as f:
            d = pickle.load(f, encoding='latin1')
        return {k: (np.asarray(v.todense()) if 'scipy.sparse' in str(type(v)) else v) for k, v in d.items()}
    d = np.load(path, allow_pickle=True)
    return {k: d[k] for k in d.files}


def model_desc(smpl_type, data, gmm=None, J_regressor_extra=None, num_betas=10, num_expression=10, tensor_cores=True,
               gender='neutral', kid_template=None, face_params=False, num_pca_comps=6, use_pca=True, flat_hand_mean=False):
    """``(BfModelDesc, keepalive)`` for ``bf_model_create`` / ``bf_model_build_blob``: the raw model arrays as the C ABI
    takes them (what a non-Python host would pass after reading the model file itself).  The hand options are passed as
    given; the C++ builder validates them."""
    data = load_model_data(data, smpl_type, gender)
    keep = []

    def arr(x, dt):
        a = np.ascontiguousarray(np.asarray(x), dtype=dt)
        keep.append(a)
        return a.ctypes.data

    d = _lib.BfModelDesc()
    vt = np.asarray(data['v_template'])
    W = np.asarray(data['weights'])
    sd = np.asarray(data['shapedirs'])
    if sd.ndim == 2:
        sd = sd[:, :, None]
    faces = np.asarray(data['f'])
    d.v_template, d.shapedirs, d.posedirs = arr(vt, np.float32), arr(sd, np.float32), arr(data['posedirs'], np.float32)
    d.J_regressor, d.weights = arr(data['J_regressor'], np.float32), arr(W, np.float32)
    d.parents, d.faces = arr(np.asarray(data['kintree_table'])[0].astype(np.int64), np.int32), arr(faces, np.int32)
    d.is_smplx, d.V, d.J, d.F, d.n_shape_dirs = int(smpl_type == 'smplx'), vt.shape[0], W.shape[1], faces.shape[0], sd.shape[2]
    d.num_betas, d.num_expression, d.tensor_cores = num_betas, num_expression, int(bool(tensor_cores))
    d.face_params = int(bool(face_params))
    d.num_pca_comps, d.hand_axis_angle, d.flat_hand_mean = int(num_pca_comps), int(not use_pca), int(bool(flat_hand_mean))
    if smpl_type == 'smplx':
        d.hands_meanl, d.hands_meanr = arr(data['hands_meanl'], np.float32), arr(data['hands_meanr'], np.float32)
        d.hands_componentsl, d.hands_componentsr = arr(data['hands_componentsl'], np.float32), arr(data['hands_componentsr'], np.float32)
        d.lmk_faces_idx, d.lmk_bary_coords = arr(data['lmk_faces_idx'], np.int32), arr(data['lmk_bary_coords'], np.float32)
        dyn = np.asarray(data['dynamic_lmk_faces_idx'])
        d.dynamic_lmk_faces_idx, d.dynamic_lmk_bary_coords = arr(dyn, np.int32), arr(data['dynamic_lmk_bary_coords'], np.float32)
        d.n_lmk, d.n_dyn_rows, d.n_dyn = len(np.asarray(data['lmk_faces_idx'])), dyn.shape[0], dyn.shape[1]
    if 'extra_vids' in data:
        d.extra_vids, d.n_extra_vids = arr(data['extra_vids'], np.int32), len(np.asarray(data['extra_vids']))
    if J_regressor_extra is not None:
        d.J_regressor_extra, d.n_regressor_extra = arr(J_regressor_extra, np.float32), np.asarray(J_regressor_extra).shape[0]
    if kid_template is not None:
        d.kid_template = arr(kid_template, np.float32)
    if gmm is not None:
        d.gmm_means, d.gmm_covars, d.gmm_weights = arr(gmm['means'], np.float32), arr(gmm['covars'], np.float32), arr(gmm['weights'], np.float32)
        d.n_gmm = np.asarray(gmm['means']).shape[0]
    return d, keep


class PreparedModel(object):
    """numpy tables -> device tensors -> BfModel struct (kept alive by this object).

    ``face_params=True`` (SMPL-X only) builds a face-parameter model: theta rows end with [jaw 3 | expression NE], which the
    operator takes as inputs and the fit optimises.  Without it the jaw and the expression stay at zero, as in the reference.

    Hands (SMPL-X only; smplx.create's options and defaults): ``num_pca_comps`` PCA components per hand (1..45, the first rows
    of the model's component tables), ``use_pca=False`` for 45 axis-angle entries per hand instead, ``flat_hand_mean=True``
    to leave the hand mean out of the full pose.  ``n_hand`` is the number of hand parameters per hand in theta."""

    def __init__(self, smpl_type, data, gmm=None, J_regressor_extra=None, device='cuda', num_betas=10,
                 num_expression=10, tensor_cores=None, gender='neutral', age='adult', kid_template=None, face_params=False,
                 num_pca_comps=6, use_pca=True, flat_hand_mean=False):
        assert smpl_type in ('smpl', 'smplx')
        self.smpl_type = smpl_type
        self.is_smplx = smpl_type == 'smplx'
        if tensor_cores is None:                     # BODYFIT_TC=0 selects the FP32 FFMA contraction kernels
            tensor_cores = os.environ.get('BODYFIT_TC', '1') != '0'
        self.tensor_cores = bool(tensor_cores)
        self.device = torch.device(device)
        data = load_model_data(data, smpl_type, gender)
        self.gender = gender
        self.faces = np.asarray(data['f']).astype(np.int64)
        vt = np.asarray(data['v_template'], dtype=np.float32)
        V = vt.shape[0]
        kt = np.asarray(data['kintree_table'])[0].astype(np.int64)
        parents = kt.copy()
        parents[0] = -1
        J = len(parents)
        assert all(parents[j] < j for j in range(1, J)), 'kinematic tree must be topologically sorted'
        P = (J - 1) * 9
        if num_betas < 1 or (self.is_smplx and num_expression < 0):
            raise ValueError('num_betas must be at least 1 and num_expression not negative')
        if face_params and not self.is_smplx:
            raise ValueError('face parameters (jaw pose, expression) apply to SMPL-X only')
        self.face_params = bool(face_params)
        if not self.is_smplx and (num_pca_comps != 6 or not use_pca or flat_hand_mean):
            raise ValueError('hand options (num_pca_comps, use_pca, flat_hand_mean) apply to SMPL-X only')
        if not 1 <= num_pca_comps <= 45:
            raise ValueError('num_pca_comps must be between 1 and 45')
        self.num_pca_comps, self.use_pca, self.flat_hand_mean = int(num_pca_comps), bool(use_pca), bool(flat_hand_mean)
        self.n_hand = (self.num_pca_comps if self.use_pca else 45) if self.is_smplx else 0
        NB = num_betas
        sd_all = np.asarray(data['shapedirs'], dtype=np.float32)
        if sd_all.ndim == 2:
            sd_all = sd_all[:, :, None]
        self.age = age
        if age == 'kid':
            # smplx's kid model (reference call site smplify/smplify.py:50-56: age=, kid_template_path=): the mean-centred SMIL
            # template minus the adult template becomes an extra, 11th shape direction; betas are then [B,11]
            assert not self.is_smplx, "age='kid' is passed to the SMPL branch only (smplify.py:50-56)"
            if kid_template is None:
                raise FileNotFoundError("age='kid' needs the SMIL template (kid_template= array or path; reference: config.SMIL_MODEL_DIR)")
            kt_ = kid_template
            if isinstance(kt_, (str, os.PathLike)):
                kt_ = np.load(kt_, allow_pickle=True)
                kt_ = kt_.item()['v_template'] if getattr(kt_, 'dtype', None) == object else kt_
            kt_ = np.array(kt_, dtype=np.float32)
            assert kt_.shape == vt.shape, 'kid template has %s vertices, model %s' % (kt_.shape, vt.shape)
            kt_ = kt_ - kt_.mean(axis=0)
            sd_all = np.concatenate([sd_all[:, :, :NB], (kt_ - vt)[:, :, None]], axis=2)
            NB = NB + 1
        elif age != 'adult':
            raise ValueError("age must be 'adult' or 'kid'")
        NS = NB + (num_expression if self.is_smplx else 0)
        NP = 7 + (63 if self.is_smplx else 69) + NB + (18 if self.is_smplx else 0)      # 98 / 86 (87 for the kid model)
        # the kernels' per-frame limits, checked when the model is built rather than at its first launch (same text as the
        # C++ builder, csrc/bf_model_build.cuh)
        if NS > MAX_NS:
            raise ValueError('%d shape coefficients (betas + expression) exceed the limit of %d' % (NS, MAX_NS))
        if NP > MAX_NP:
            raise ValueError('%d theta entries exceed the limit of %d' % (NP, MAX_NP))
        self.NE = NS - NB
        if self.is_smplx:
            NP += 2 * (self.n_hand - 6)             # the limit above counts 6 hand parameters; at most 189 entries
        if self.face_params:
            NP += 3 + self.NE                       # [jaw 3 | expression NE]; bounded by MAX_NS
        if self.is_smplx and sd_all.shape[-1] >= K.SHAPE_SPACE_DIM + num_expression:
            # official files: the expression directions follow the 300 shape directions (smplx: SHAPE_SPACE_DIM)
            sd = np.concatenate([sd_all[:, :, :NB], sd_all[:, :, K.SHAPE_SPACE_DIM:K.SHAPE_SPACE_DIM + num_expression]], -1)
        else:
            sd = sd_all[:, :, :NS]                  # 10 shape (+ 10 expression) directions stored back to back
        sd = np.ascontiguousarray(sd)
        assert sd.shape == (V, 3, NS), sd.shape
        pdirs = np.asarray(data['posedirs'], dtype=np.float32)
        PD = np.reshape(pdirs, [-1, P]).T                                   # [P, 3V]
        Jreg = np.asarray(data['J_regressor'], dtype=np.float32)
        W = np.asarray(data['weights'], dtype=np.float32)
        self.V, self.J, self.P, self.NB, self.NS = V, J, P, NB, NS
        self.Kdim = P + NS + 1
        self.Kp = _round_up(self.Kdim, 16)
        self.NP = NP
        self.nbody = 63 if self.is_smplx else 69
        self.parents = parents

        depth = np.zeros(J, dtype=np.int32)
        for j in range(1, J):
            depth[j] = depth[parents[j]] + 1
        child_ptr = np.zeros(J + 1, dtype=np.int32)
        child_idx = []
        for j in range(J):
            ch = [c for c in range(1, J) if parents[c] == j]
            child_idx += ch
            child_ptr[j + 1] = len(child_idx)
        Jt = (Jreg.astype(np.float64) @ vt.astype(np.float64)).astype(np.float32)
        Jd = np.einsum('jv,vcl->jcl', Jreg.astype(np.float64), sd.astype(np.float64)).astype(np.float32)

        pose_mean = np.zeros(3 * J, dtype=np.float32)
        hand_l = hand_r = None
        if self.is_smplx:
            if not self.flat_hand_mean:
                pose_mean[75:120] = np.asarray(data['hands_meanl'], dtype=np.float32)
                pose_mean[120:165] = np.asarray(data['hands_meanr'], dtype=np.float32)
            if self.use_pca:
                hand_l = np.asarray(data['hands_componentsl'], dtype=np.float32)[:self.n_hand]
                hand_r = np.asarray(data['hands_componentsr'], dtype=np.float32)[:self.n_hand]
                if hand_l.shape != (self.n_hand, 45) or hand_r.shape != (self.n_hand, 45):
                    raise ValueError('num_pca_comps=%d needs at least %d hand component rows of 45 entries (the model has %s / %s)'
                                     % (self.n_hand, self.n_hand, hand_l.shape, hand_r.shape))
            else:                                   # axis-angle hands: the identity, so the kernels keep one hand loop
                hand_l = hand_r = np.eye(45, dtype=np.float32)

        # ---- output joint table (pre-map list, then the reference's joint map) --------------------
        # vertex-picked joints: the official files do not list them (smplx hard-codes the ids)
        extra_vids = np.asarray(data['extra_vids'] if 'extra_vids' in data else K.EXTRA_VIDS[smpl_type]).astype(np.int64)
        assert extra_vids.max() < V, 'vertex-picked joint ids outside the mesh'
        self.extra_vids = extra_vids
        pre = [(0, (j, 0, 0), (1.0, 0.0, 0.0)) for j in range(J)]
        pre += [(1, (int(v), int(v), int(v)), (1.0, 0.0, 0.0)) for v in extra_vids]
        dyn_faces = dyn_bary = None
        xr = None
        if self.is_smplx:
            lf = self.faces[np.asarray(data['lmk_faces_idx']).astype(np.int64)]
            lb = np.asarray(data['lmk_bary_coords'], dtype=np.float32)
            pre += [(1, tuple(int(x) for x in lf[i]), tuple(float(x) for x in lb[i])) for i in range(lf.shape[0])]
            dyn_faces = self.faces[np.asarray(data['dynamic_lmk_faces_idx']).astype(np.int64)]      # [79,17,3]
            dyn_bary = np.asarray(data['dynamic_lmk_bary_coords'], dtype=np.float32)
            pre += [(2, (s, 0, 0), (0.0, 0.0, 0.0)) for s in range(dyn_faces.shape[1])]
            jmap = K.smpl_to_openpose('smplx', use_hands=True, use_face=True, use_face_contour=True,
                                      openpose_format='coco25')
            K_used = len(jmap)
        else:
            if J_regressor_extra is not None:
                xr = np.asarray(J_regressor_extra, dtype=np.float32)
                pre += [(3, (r, 0, 0), (0.0, 0.0, 0.0)) for r in range(xr.shape[0])]
                jmap = np.asarray(K.SPIN_JOINT_MAP)
            else:
                jmap = K.smpl_to_openpose('smpl', openpose_format='coco25')
            K_used = 25
        self.K_used = K_used
        self.joint_table = [pre[int(i)] for i in jmap]
        self.K_out = len(self.joint_table)
        # SMPL wrapper also returns the 45 un-mapped smplx joints as ``joints_ori`` (models/smpl.py:73,80):
        # appended to the all-vertex joint table so that one kernel produces (and back-propagates) both
        self.ori_table = pre[:J + len(extra_vids)] if not self.is_smplx else []
        self.K_full = self.K_out + len(self.ori_table)
        self._dyn_faces, self._dyn_bary, self._xr = dyn_faces, dyn_bary, xr

        # ---- GMM prior (smplify/prior.py:127-160) ------------------------------------------------
        g = {}
        if gmm is not None:
            means = np.asarray(gmm['means']).astype(np.float32)
            covs = np.asarray(gmm['covars']).astype(np.float32)
            prec = np.stack([np.linalg.inv(c) for c in covs]).astype(np.float32)
            sqrdets = np.array([np.sqrt(np.linalg.det(c)) for c in np.asarray(gmm['covars'])])
            const = (2 * np.pi) ** (69 / 2.)
            nllw = np.asarray(np.asarray(gmm['weights']) / (const * (sqrdets / sqrdets.min()))).astype(np.float32)
            psym = np.zeros((means.shape[0], 69, 72), dtype=np.float32)      # (P + P^T)/2, rows padded to 72
            psym[:, :, :69] = (prec + np.transpose(prec, (0, 2, 1))) * np.float32(0.5)
            g = dict(gmm_mean=means, gmm_psym=psym, gmm_logw=np.log(nllw).astype(np.float32))
            if self.tensor_cores and means.shape[0] * 72 % 192 == 0:
                # tensor-core form of the prior: y_m = P_sym,m (x - mu_m) for all components at once is ONE GEMM
                # [pose69 | 1 | 0..] (K = 80) @ [P_sym,m | -P_sym,m mu_m] -> [B, n_gmm * 72]; K-major operand, 3xTF32 split
                bt = np.zeros((means.shape[0] * 72, 80), dtype=np.float32)
                for c in range(means.shape[0]):
                    bt[c * 72:c * 72 + 69, :69] = psym[c, :, :69]
                    bt[c * 72:c * 72 + 69, 69] = -(psym[c, :, :69].astype(np.float64) @ means[c].astype(np.float64)).astype(np.float32)
                g['gmm_bt_hi'], g['gmm_bt_lo'] = split_tf32(bt)
            self.n_gmm = means.shape[0]
            assert means.shape[1] == 69
        else:
            self.n_gmm = 0

        # ---- vertex sets -------------------------------------------------------------------------
        Bm_rows = np.zeros((self.Kp, 3 * V), dtype=np.float32)
        Bm_rows[:P] = PD
        Bm_rows[P:P + NS] = sd.reshape(V * 3, NS).T
        Bm_rows[P + NS] = vt.reshape(-1)
        # Active set order: first the vertices every frame uses (picked joints, static landmarks, regressed extra joints; ascending
        # id), then the contour candidates in the order of the first yaw row that uses them.  A frame on row `a` then touches the
        # static 16-vertex blocks plus a handful of contour blocks (the rows' vertex sets slide with the yaw angle), which is
        # what lets the blend GEMMs skip whole blocks for frame tiles that hold few rows (lv_blk below, csrc/bf_blend_tc.cuh).
        static, first_row = set(), {}
        for kind, src, w in self.joint_table[:K_used]:
            if kind == 1:
                static.update(int(s) for s, ww in zip(src, w) if ww != 0.0)
            elif kind == 3:
                static.update(int(x) for x in np.nonzero(xr[src[0]])[0])
        for kind, src, w in self.joint_table[:K_used]:
            if kind == 2:
                for a in range(dyn_faces.shape[0]):
                    for x in dyn_faces[a, src[0], :].reshape(-1):
                        if int(x) not in static:
                            first_row[int(x)] = min(first_row.get(int(x), a), a)
        self.active_vids = np.array(sorted(static) + sorted(first_row, key=lambda v: (first_row[v], v)), dtype=np.int64)
        self.n_static = len(static)
        # joints grouped by tree level: the chain kernels walk one level at a time with lane = joint of that level
        lvl_j = np.argsort(depth, kind='stable').astype(np.int32)
        lvl_ptr = np.zeros(int(depth.max()) + 2, dtype=np.int32)
        np.add.at(lvl_ptr, depth + 1, 1)
        lvl_ptr = np.cumsum(lvl_ptr).astype(np.int32)
        self._host = dict(parents=parents.astype(np.int32), depth=depth, lvl_ptr=lvl_ptr, lvl_j=lvl_j, child_ptr=child_ptr,
                          child_idx=np.array(child_idx + [0], dtype=np.int32), Jt=Jt, Jd=Jd, pose_mean=pose_mean,
                          hand_l=hand_l, hand_r=hand_r, **g)
        self.max_depth = int(depth.max())
        full_h = self._build_vset(np.arange(V, dtype=np.int64), Bm_rows, W, self.joint_table + self.ori_table)
        act_h = self._build_vset(self.active_vids, Bm_rows, W, self.joint_table[:K_used], build_live=True)
        del Bm_rows

        # ---- upload ----------------------------------------------------------------------------
        self._dev = {}
        self.struct = _lib.BfModel()
        for k, v in self._host.items():
            setattr(self.struct, k, self._up('m_' + k, v))
        self._fill_vset(self.struct.full, 'full', full_h)
        self._fill_vset(self.struct.act, 'act', act_h)
        for k, v in dict(J=J, P=P, NS=NS, NB=NB, Kp=self.Kp, NP=self.NP, is_smplx=int(self.is_smplx),
                         max_depth=self.max_depth, K_used=K_used, n_gmm=self.n_gmm, face=int(self.face_params),
                         n_hand=self.n_hand).items():
            setattr(self.struct, k, v)
        self.n_act = int(act_h['n'])
        self.n_pad_full = int(full_h['n_pad'])
        self.ld_act = 3 * int(act_h['n_pad'])
        self.n_act_pad = int(act_h['n_pad'])
        self.K_out_act = int(act_h['K_out'])
        self._host = None

    # ------------------------------------------------------------------------------------------
    def _up(self, name, arr):
        if arr is None:
            return None
        t = torch.from_numpy(np.ascontiguousarray(arr)).to(self.device)
        self._dev[name] = t
        return t.data_ptr()

    def _fill_vset(self, vs, tag, h):
        for k, v in h.items():
            if isinstance(v, np.ndarray):
                setattr(vs, k, self._up(tag + '_' + k, v))
            else:
                setattr(vs, k, int(v))

    def _build_vset(self, vids, Bm_rows, W, table, build_live=False):
        """Tables for the vertex set ``vids`` (distinct global vertex ids, in the set's column order)."""
        J = self.J
        n = len(vids)
        n_pad = _round_up(max(n, 1), 32)
        pos = -np.ones(self.V, dtype=np.int64)
        pos[vids] = np.arange(n)
        cols = (3 * vids[:, None] + np.arange(3)[None]).reshape(-1)
        Bm = np.zeros((self.Kp, 3 * n_pad), dtype=np.float32)
        Bm[:, :3 * n] = Bm_rows[:, cols]
        Ws = W[vids]                                                        # [n, J]
        nnz = max(1, int((Ws != 0).sum(1).max()))
        ell_j = np.zeros((n_pad, nnz), dtype=np.int32)
        ell_w = np.zeros((n_pad, nnz), dtype=np.float32)
        order = np.argsort(-(Ws != 0).astype(np.int8), axis=1, kind='stable')[:, :nnz]     # non-zeros first, joint order kept
        ell_j[:n] = order
        ell_w[:n] = np.take_along_axis(Ws, order, 1)
        ell_j[:n][ell_w[:n] == 0] = 0
        vv, jj = np.nonzero(Ws)
        o = np.lexsort((vv, jj))
        vv, jj = vv[o], jj[o]
        jv_ptr = np.zeros(J + 1, dtype=np.int32)
        np.add.at(jv_ptr, jj + 1, 1)
        jv_ptr = np.cumsum(jv_ptr).astype(np.int32)
        jv_vid = vv.astype(np.int32)
        jv_w = Ws[vv, jj].astype(np.float32)

        K_out = len(table)
        kj_kind = np.zeros(K_out, dtype=np.int32)
        kj_src = np.zeros((K_out, 3), dtype=np.int32)
        kj_w = np.zeros((K_out, 3), dtype=np.float32)
        entries = []                                                        # (target, k, a, w)
        dyn_src = dyn_w = None
        n_dyn = 0
        if self._dyn_faces is not None:
            n_dyn = self._dyn_faces.shape[1]
            dyn_src = pos[self._dyn_faces].astype(np.int32)                 # [79, n_dyn, 3]
            dyn_w = self._dyn_bary.astype(np.float32)
        xr_ptr = xr_vid = xr_w = None
        n_extra = 0
        if self._xr is not None and any(kind == 3 for kind, _, _ in table):
            n_extra = self._xr.shape[0]
            ptr, vidl, wl = [0], [], []
            for r in range(n_extra):
                nzv = np.nonzero(self._xr[r])[0]
                assert (pos[nzv] >= 0).all()
                vidl += [int(pos[x]) for x in nzv]
                wl += [float(self._xr[r, x]) for x in nzv]
                ptr.append(len(vidl))
            xr_ptr, xr_vid, xr_w = np.array(ptr, np.int32), np.array(vidl, np.int32), np.array(wl, np.float32)
        for k, (kind, src, w) in enumerate(table):
            kj_kind[k] = kind
            if kind == 0:
                kj_src[k] = (src[0], 0, 0)
                entries.append((src[0], k, -1, 1.0))
            elif kind == 1:
                p = [int(pos[s]) for s in src]
                assert min(p) >= 0, 'joint %d references a vertex outside the set' % k
                kj_src[k] = p
                kj_w[k] = w
                for pi, wi in zip(p, w):
                    if wi != 0.0:
                        entries.append((J + pi, k, -1, float(wi)))
            elif kind == 2:
                s = src[0]
                kj_src[k] = (s, 0, 0)
                assert (dyn_src[:, s, :] >= 0).all()
                for a in range(dyn_src.shape[0]):
                    for i in range(3):
                        entries.append((J + int(dyn_src[a, s, i]), k, a, float(dyn_w[a, s, i])))
            else:
                r = src[0]
                kj_src[k] = (r, 0, 0)
                for e in range(xr_ptr[r], xr_ptr[r + 1]):
                    entries.append((J + int(xr_vid[e]), k, -1, float(xr_w[e])))
        dyn_k = [k for k, (kind, _, _) in enumerate(table) if kind == 2]
        entries = [e for e in entries if e[2] < 0]        # contour landmarks are scattered directly from dyn_src (yaw-dependent)
        entries.sort(key=lambda t: (t[0], t[1], t[2]))
        ntg = J + n
        tg_ptr = np.zeros(ntg + 1, dtype=np.int32)
        for t, _, _, _ in entries:
            tg_ptr[t + 1] += 1
        tg_ptr = np.cumsum(tg_ptr).astype(np.int32)
        pad1 = lambda a, dt: np.array(a if len(a) else [0], dtype=dt)
        h = dict(Bm=Bm, ell_j=ell_j, ell_w=ell_w, jv_ptr=jv_ptr, jv_vid=pad1(jv_vid, np.int32), jv_w=pad1(jv_w, np.float32),
                 kj_kind=kj_kind, kj_src=kj_src, kj_w=kj_w, tg_ptr=tg_ptr,
                 tg_k=pad1([e[1] for e in entries], np.int32), tg_a=pad1([e[2] for e in entries], np.int32),
                 tg_w=pad1([e[3] for e in entries], np.float32),
                 n=n, n_pad=n_pad, ldn=3 * n_pad, nnz=nnz, K_out=K_out, n_dyn=n_dyn, n_extra=n_extra)
        if self.tensor_cores:
            h['Bm_hi'], h['Bm_lo'] = split_tf32(Bm)
            h['Bt_hi'], h['Bt_lo'] = split_tf32(np.ascontiguousarray(Bm.T))
        if dyn_src is not None and dyn_k:
            assert [table[k][1][0] for k in dyn_k] == list(range(n_dyn))
            h['dyn_src'] = np.ascontiguousarray(dyn_src)
            h['dyn_w'] = np.ascontiguousarray(dyn_w)
            h['dyn_k'] = np.array(dyn_k, dtype=np.int32)
        else:
            h['n_dyn'] = 0
        nzj = np.nonzero(np.diff(jv_ptr))[0].astype(np.int32)
        h['jv_nz'] = nzj if len(nzj) else np.zeros(1, np.int32)
        h['n_nz'] = len(nzj)
        if build_live:
            h.update(self._build_live_tables(J, n, entries, dyn_src if h['n_dyn'] else None, dyn_w, dyn_k, Ws, nzj))
        if xr_ptr is not None:
            h.update(xr_ptr=xr_ptr, xr_vid=xr_vid, xr_w=xr_w)
        return h

    @staticmethod
    def _build_live_tables(J, n, entries, dyn_src, dyn_w, dyn_k, Ws, nzj):
        """Per contour row (79 yaw rows for SMPL-X, one row otherwise): the vertices of the set that carry a
        non-zero keypoint gradient for a frame on that row (static picks / landmarks + the 17 x 3 contour vertices
        of the row), the keypoint-gradient gather lists of those vertices (static entries first, then the contour
        entries in slot order -- the accumulation order of the unfused kernels) and the joint->vertex skinning lists
        restricted to them.  The fused per-frame kernel walks only these lists (k_frame_loss_bwd)."""
        rows = dyn_src.shape[0] if dyn_src is not None else 1
        static = {}
        for t, k, a, w in entries:                                          # already sorted by (target, k)
            if t >= J:
                static.setdefault(t - J, []).append((k, w))
        per_row = []
        for a in range(rows):
            ent = {v: list(e) for v, e in static.items()}
            if dyn_src is not None:
                for s_, k in enumerate(dyn_k):
                    for i in range(3):
                        ent.setdefault(int(dyn_src[a, s_, i]), []).append((k, float(dyn_w[a, s_, i])))
            per_row.append(ent)
        lmax = _round_up(max(len(e) for e in per_row), 32)
        lv_n = np.zeros(rows, np.int32)
        lv_vid = np.zeros((rows, lmax), np.int32)
        lt_ptr = np.zeros((rows, lmax + 1), np.int32)
        lt_k, lt_w = [], []
        nnzj = max(1, len(nzj))
        lj_ptr = np.zeros((rows, nnzj + 1), np.int32)
        lj_vid, lj_w = [], []
        for a, ent in enumerate(per_row):
            live = sorted(ent)
            lv_n[a] = len(live)
            lv_vid[a, :len(live)] = live
            for i, v in enumerate(live):
                lt_ptr[a, i] = len(lt_k)
                lt_k += [k for k, _ in ent[v]]
                lt_w += [w for _, w in ent[v]]
            lt_ptr[a, len(live):] = len(lt_k)
            sub = Ws[live]                                                  # [L, J]
            for jn, j in enumerate(nzj):
                lj_ptr[a, jn] = len(lj_vid)
                nzv = np.nonzero(sub[:, j])[0]
                lj_vid += [int(x) for x in nzv]                             # index into this row's live list
                lj_w += [float(sub[x, j]) for x in nzv]
            lj_ptr[a, len(nzj):] = len(lj_vid)
        pad1 = lambda x, dt: np.array(x if len(x) else [0], dtype=dt)
        # 16-vertex blocks a frame on row `a` needs (bit i = block i of the set); all ones where the set has > 32 blocks
        lv_blk = np.zeros(rows, dtype=np.uint32)
        for a in range(rows):
            blocks = np.unique(lv_vid[a, :lv_n[a]] // 16)
            lv_blk[a] = np.uint32(0xFFFFFFFF) if (n + 15) // 16 > 32 else np.bitwise_or.reduce((np.uint32(1) << blocks.astype(np.uint32)))
        return dict(lv_n=lv_n, lv_vid=lv_vid, lt_ptr=lt_ptr, lt_k=pad1(lt_k, np.int32), lt_w=pad1(lt_w, np.float32),
                    lj_ptr=lj_ptr, lj_vid=pad1(lj_vid, np.int32), lj_w=pad1(lj_w, np.float32), lv_blk=lv_blk.view(np.int32),
                    lmax=lmax, n_rows=rows)

    # ------------------------------------------------------------------------------------------
    def save_blob(self, path):
        """Serialise the prepared tables for hosts that do not run Python: ``bf_model_load(path, &model)`` of the C ABI maps
        the file, uploads the array section with one copy and patches the pointers (include/bodyfit_b200.h).
        Layout: 16-byte header ("BFMODEL1", ABI version, sizeof(BfModel)), the BfModel struct image with every pointer field
        replaced by (offset into the array section + 1), 0 = NULL, then the array section (each array 16-byte aligned)."""
        import struct as _st
        img = _lib.BfModel()
        C.memmove(C.byref(img), C.byref(self.struct), C.sizeof(_lib.BfModel))
        blobs, off = [], 0

        def put(t):
            nonlocal off
            a = t.detach().cpu().contiguous().numpy().tobytes()
            pad = (-len(a)) % 16
            blobs.append(a + b'\0' * pad)
            o = off
            off += len(a) + pad
            return o + 1

        def patch(st, tag):
            for name, typ in st._fields_:
                if typ is _lib._fp:
                    t = self._dev.get(tag + '_' + name)
                    setattr(st, name, put(t) if t is not None else None)
        patch(img, 'm')
        patch(img.full, 'full')
        patch(img.act, 'act')
        with open(path, 'wb') as f:
            f.write(b'BFMODEL1' + _st.pack('<ii', _lib.ABI_VERSION, C.sizeof(_lib.BfModel)))
            f.write(bytes(img))
            f.write(_st.pack('<q', off))
            for b in blobs:
                f.write(b)
        return path

    def pack_theta(self, global_orient, body_pose, betas, transl=None, scale=None, leye=None, reye=None,
                   lhand=None, rhand=None, jaw=None, expression=None):
        """Assemble [B, NP] theta rows (layout in include/bodyfit_b200.h).  ``lhand`` / ``rhand`` are [B, n_hand] (PCA
        coefficients, or 45 axis-angle entries).  ``jaw`` [B,3] / ``expression`` [B,NE] belong to a face-parameter model
        (None = 0); a face-off model accepts them only as None."""
        B = global_orient.shape[0]
        dev, dt = self.device, torch.float32
        z = lambda n: torch.zeros(B, n, device=dev, dtype=dt)
        f = lambda t, n: z(n) if t is None else t.reshape(B, n).to(device=dev, dtype=dt)
        bt = betas.reshape(B, -1).to(device=dev, dtype=dt)
        if bt.shape[1] < self.NB:                       # kid model: 11 betas, the network gives 10
            bt = torch.cat([bt, torch.zeros(B, self.NB - bt.shape[1], device=dev, dtype=dt)], dim=1)
        parts = [f(transl, 3), torch.ones(B, 1, device=dev, dtype=dt) if scale is None else f(scale, 1),
                 f(global_orient, 3), f(body_pose, self.nbody), bt]
        if self.is_smplx:
            parts += [f(leye, 3), f(reye, 3), f(lhand, self.n_hand), f(rhand, self.n_hand)]
        if self.face_params:
            parts += [f(jaw, 3), f(expression, self.NE)]
        elif jaw is not None or expression is not None:
            raise ValueError('jaw / expression need a face-parameter SMPL-X model (face_params=True)')
        return torch.cat(parts, dim=1).contiguous()

    def split_theta(self, theta):
        nb = self.nbody
        out = dict(transl=theta[:, 0:3], scale=theta[:, 3:4], global_orient=theta[:, 4:7],
                   body_pose=theta[:, 7:7 + nb], betas=theta[:, 7 + nb:7 + nb + self.NB])
        if self.is_smplx:
            o, nh = 7 + nb + self.NB, self.n_hand
            out.update(leye_pose=theta[:, o:o + 3], reye_pose=theta[:, o + 3:o + 6],
                       left_hand_pose=theta[:, o + 6:o + 6 + nh], right_hand_pose=theta[:, o + 6 + nh:o + 6 + 2 * nh])
            o += 6 + 2 * nh
            if self.face_params:
                out.update(jaw_pose=theta[:, o:o + 3], expression=theta[:, o + 3:o + 3 + self.NE])
        return out
