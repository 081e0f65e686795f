"""``SMPLify`` -- multi-view SMPL / SMPL-X fitting, same constructor / call signature and
result dict as the reference's ``smplify/smplify.py:19-254``, running on the B200 kernels.

Extensions over the reference (which supports one frame per call, smplify.py:189-190):
``__call__`` also accepts B frames at once -- ``net_output`` = ([B,10], [B,72]) and
``keypoints`` either a list over frames of per-view OpenPose dict lists, or a packed
[B,Nv,K,3] array in model joint order -- each frame being an independent fit with its
own Adam state, exactly as B separate reference calls.

``use_mask=True`` (silhouette term) and ``use_mesh=True`` (point-to-scan term, SMPL+D) run the all-vertex loop
(``_fit_dense``); the keypoint-only objective runs the fused active-set loop.
"""
import os
import pickle

import numpy as np
import torch

from .. import constants as K
from ..engine import ConcurrentFitSession, FitSession, pack_cameras, pack_keypoints, staggered_ranges  # noqa: F401
from ..model import PreparedModel
from ..synthetic import openpose_to_keypoints


def _mark_event():
    e = torch.cuda.Event(enable_timing=True)
    e.record(torch.cuda.current_stream())
    return e


class SMPLify(object):
    """Implementation of multiview SMPLify (reference: smplify/smplify.py:19-82)."""

    def __init__(self, smpl_type='smpl', age='adult', step_size=1e-2, batch_size=1, num_iters=600,
                 gender='male', use_mask=False, device=torch.device('cuda'), debug=True,
                 model_data=None, gmm=None, J_regressor_extra=None, data_root='data', dense_every_iter=False,
                 concurrent_parts=None, concurrent_min_part=512, temporal_weight=0.0, halo_exchange=None, halo=None,
                 copy_outputs=None, graph=None, sort_frames=None, kid_template=None, face_params=False,
                 expr_prior_weight=K.EXPR_PRIOR_WEIGHT):
        """``face_params=True`` (SMPL-X only): the fit also optimises the jaw pose and the expression coefficients, with the
        expression prior ``expr_prior_weight^2 * sum psi^2`` (the reference optimises neither, smplify.py:118,167-173; no jaw
        prior).  The result dict then also holds ``jaw_pose`` and ``expression``."""
        if age not in ('adult', 'kid'):
            raise ValueError("age must be 'adult' or 'kid' (smplify.py:23,112-115)")
        if age == 'kid' and smpl_type != 'smpl':
            raise ValueError("age='kid' exists for smpl_type='smpl' only: the reference passes it to the SMPL branch (smplify.py:50-56)")
        if face_params and smpl_type != 'smplx':
            raise ValueError("face_params=True needs smpl_type='smplx': SMPL has no jaw / expression parameters")
        self.face_params, self.expr_prior_weight = bool(face_params), float(expr_prior_weight)
        self.device = torch.device(device)
        self.debug = debug
        self.gender = gender
        self.smpl_type = smpl_type
        self.use_hand_face = (smpl_type == 'smplx')
        self.age = age
        self.use_mask = use_mask
        self.batch_size = batch_size
        self.num_iters = num_iters
        if gmm is None:                                   # smplify.py:46-48 -> prior.py:119-128
            fn = os.path.join(data_root, 'gmm_08.pkl')
            if not os.path.exists(fn):
                raise FileNotFoundError('The path to the mixture prior "%s" does not exist' % fn)
            with open(fn, 'rb') as f:
                gmm = pickle.load(f, encoding='latin1')
        if model_data is None:                            # smplify.py:51,63
            model_data = os.path.join(data_root, smpl_type)
        if smpl_type == 'smpl' and J_regressor_extra is None:
            fn = os.path.join(data_root, 'J_regressor_extra.npy')      # config.py:1, models/smpl.py:62
            J_regressor_extra = np.load(fn) if os.path.exists(fn) else None
        if age == 'kid' and kid_template is None:
            kid_template = os.path.join(data_root, 'smil', 'smil_web.pkl')           # config.SMIL_MODEL_DIR (config.py:5)
        self.model = PreparedModel(smpl_type, model_data, gmm=gmm, J_regressor_extra=J_regressor_extra,
                                   device=self.device, gender=gender, age=age, kid_template=kid_template,
                                   face_params=self.face_params)
        self.smpl_faces = self.model.faces.astype(np.int32).reshape(1, -1, 3)
        self.last_trace = None
        self.dense_every_iter = dense_every_iter
        # temporal smoothness between consecutive frames of the batch (not in the reference; BASELINE config 4)
        # halo: a sharding.HaloLink (boundary rows by in-kernel NVLink stores, graph-capturable) or halo_exchange: a host
        # callback (sharding.exchange_halo, one NCCL send/recv pair per iteration) -- the tested fallback
        self.temporal_weight, self.halo_exchange, self.halo = float(temporal_weight), halo_exchange, halo
        # Results on the host: the reference returns fresh arrays.  True = always copy out of the pinned staging buffers,
        # False = return views of them (valid until the next call with the same shapes), None = copy unless the results
        # exceed 32 MB (~250 SMPL-X frames; fresh pages cost ~0.2 ms per MB: the 160 MB of a 1,250-frame shard took 36 ms to copy,
        # 2.5x the fit itself -- large batches get views, and the docstring of __call__ says so)
        self.copy_outputs = copy_outputs
        self.sort_frames = sort_frames    # None: SMPL-X batches are processed in contour-row order (engine.FitSession), False: as given
        self.graph = graph            # None: CUDA-graph replay of the whole fit unless BODYFIT_GRAPH=0; False: direct launches
        # batches of >= 4096 frames are fitted as up to this many staggered parts on their own streams (1 = one batch)
        if concurrent_parts is None:
            concurrent_parts = int(os.environ.get('BODYFIT_PARTS', '4'))
        self.concurrent_parts = max(1, int(concurrent_parts))
        self.device_parts = int(os.environ.get('BODYFIT_DEVICE_PARTS', '2'))
        self.concurrent_min_part = int(os.environ.get('BODYFIT_MIN_PART', concurrent_min_part))
        self.concurrent_lead = int(os.environ.get('BODYFIT_LEAD', '0'))
        self.concurrent_taper = float(os.environ.get('BODYFIT_TAPER', '0.5'))
        self._pinned = {}
        self.last_loss_terms = None

    # ------------------------------------------------------------------------------------------
    def _pack_inputs(self, net_output, keypoints):
        init_betas, init_poses = net_output
        init_betas = torch.as_tensor(init_betas, dtype=torch.float32).reshape(-1, 10)
        if self.age == 'kid':                                  # the kid model starts from zero betas (11 of them, smplify.py:114-115)
            init_betas = torch.zeros_like(init_betas)
        init_poses = torch.as_tensor(init_poses, dtype=torch.float32)
        init_poses = init_poses.reshape(init_betas.shape[0], -1)
        B = init_poses.shape[0]
        if isinstance(keypoints, (np.ndarray, torch.Tensor)):
            kp = torch.as_tensor(keypoints, dtype=torch.float32)
            if kp.dim() == 3:
                kp = kp[None]
        else:
            frames = keypoints if (len(keypoints) and isinstance(keypoints[0], (list, tuple))) else [keypoints]
            kp = torch.from_numpy(np.stack([openpose_to_keypoints(v, self.smpl_type) for v in frames]))
        assert kp.shape[0] == B, 'keypoints for %d frames, parameters for %d' % (kp.shape[0], B)
        return init_betas, init_poses, kp

    def __call__(self, *args, **kwargs):
        """Same signature and result dict as the reference's SMPLify.__call__ (smplify/smplify.py:84-86,216-226); see _fit.
        Runs with ``self.device`` as the current CUDA device (the library launches on the current device's streams), whatever
        device the caller has selected.  Host results: fresh numpy arrays, except for batches whose results exceed 32 MB,
        which are returned as views of session-owned pinned buffers valid until the next call (``copy_outputs``)."""
        if self.device.type == 'cuda':
            with torch.cuda.device(self.device):
                return self._fit(*args, **kwargs)
        return self._fit(*args, **kwargs)

    def _fit(self, net_output, c2ws, Ks, keypoints, output_folder=None, use_mask=False, masks=None,
             use_frames=[0], mask_frames=[0], keyframe=6, imsize=512, use_mesh=False, meshfile=None,
             displacement=False, return_vertices=True, as_numpy=True):
        if use_mask or use_mesh:
            return self._fit_dense(net_output, c2ws, Ks, keypoints, imsize, as_numpy, use_mesh=use_mesh, meshfile=meshfile,
                                   displacement=displacement, use_mask=use_mask, masks=masks, use_frames=use_frames,
                                   mask_frames=mask_frames)
        m, dev = self.model, self.device
        init_betas, init_poses, kp = self._pack_inputs(net_output, keypoints)
        B, Nv = kp.shape[0], kp.shape[1]
        assert kp.shape[2] == m.K_used, 'expected %d keypoints per view, got %d' % (m.K_used, kp.shape[2])
        assert len(c2ws) == Nv and len(Ks) == Nv
        sess = self.session(B, Nv, imsize, return_vertices, host_io=bool(as_numpy))
        self.h2d_bytes = int(kp.numel() + init_poses.numel() + init_betas.numel() + 12 * Nv) * 4
        if isinstance(sess, ConcurrentFitSession):
            return self._call_concurrent(sess, init_betas, init_poses, kp, c2ws, Ks, as_numpy)

        # host -> device (pinned staging so the copies are asynchronous DMA), then two packing kernels of the library
        with torch.cuda.device(dev):
            kp_dev = self._h2d('kp', kp)
            poses_dev = self._h2d('poses', init_poses)
            betas_dev = self._h2d('betas', init_betas)
            cams = self._h2d('cams', torch.from_numpy(pack_cameras(c2ws, Ks)))
            # init: body pose / betas / global orient from the network, transl 0, scale 1, rest 0 (smplify.py:103-128)
            sess.load_inputs(kp_dev, cams, poses_dev, betas_dev)
            sess.run()
            out = sess.results()
            self.last_trace = sess.trace
            self.last_loss_terms = sess.loss_terms
            if as_numpy:
                out = self._d2h(out)
        out['faces'] = self.smpl_faces[0]
        return out

    def _call_concurrent(self, sess, init_betas, init_poses, kp, c2ws, Ks, as_numpy):
        """Large batches: staggered parts on their own streams (engine.ConcurrentFitSession).  Each part's inputs go up,
        its frames are fitted and its results come down on the part's stream, so the device->host copy of an early
        part (126 KB of vertices per SMPL-X frame) overlaps the fitting of the later ones.  Results are bit-identical to
        the single-batch path (frames are independent)."""
        m = self.model
        B = kp.shape[0]
        with torch.cuda.device(self.device):
            cur = torch.cuda.current_stream()
            cams = self._h2d('cams', torch.from_numpy(pack_cameras(c2ws, Ks)))
            ready = torch.cuda.Event()
            ready.record(cur)
            host, nbytes = {}, 0
            streams = sess.prio_streams                            # decreasing priority: parts finish in launch order
            trace_ev = [] if os.environ.get('BODYFIT_E2E_TRACE') else None      # per part: start, inputs up, fit done, results down
            mark = (lambda: trace_ev[-1].append(_mark_event())) if trace_ev is not None else (lambda: None)
            for k, ((lo, hi), part, st) in enumerate(zip(sess.ranges, sess.parts, streams)):
                with torch.cuda.stream(st):
                    st.wait_event(ready)
                    if trace_ev is not None:
                        trace_ev.append([])
                    mark()
                    kp_dev = self._h2d(('kp', k), kp[lo:hi])
                    poses_dev = self._h2d(('poses', k), init_poses[lo:hi])
                    betas_dev = self._h2d(('betas', k), init_betas[lo:hi])
                    part.load_inputs(kp_dev, cams, poses_dev, betas_dev)
                    mark()
                    part.run(priority=st.priority)
                    mark()
                    if as_numpy:
                        for name, v in part.results().items():
                            pbuf = self._pinned.get(('out', name))
                            if pbuf is None or pbuf.shape != (B,) + tuple(v.shape[1:]):
                                pbuf = torch.empty((B,) + tuple(v.shape[1:]), dtype=v.dtype, pin_memory=True)
                                self._pinned[('out', name)] = pbuf
                            host[name] = pbuf
                            pbuf[lo:hi].copy_(v, non_blocking=True)
                            nbytes += int(v.numel() * v.element_size())
                    mark()
            if as_numpy:
                for st in streams:
                    st.synchronize()
                if trace_ev is not None:
                    t0 = trace_ev[0][0]
                    self.last_e2e_timeline = [[round(t0.elapsed_time(e), 3) for e in evs] for evs in trace_ev]
                self.d2h_bytes = nbytes
                out = self._host_results(host, nbytes)
            else:
                for st in streams:
                    cur.wait_stream(st)
                out = sess.results()
        self.last_trace, self.last_loss_terms = sess.trace, sess.loss_terms
        out['faces'] = self.smpl_faces[0]
        return out

    # ------------------------------------------------------------------------------------------
    def _fit_dense(self, net_output, c2ws, Ks, keypoints, imsize, as_numpy, use_mesh=False, meshfile=None, displacement=False,
                   use_mask=False, masks=None, use_frames=None, mask_frames=None):
        """The objectives that need ALL vertices in every iteration (dense LBS backward):
        ``use_mesh=True`` (smplify.py:146-156,205-210,228-247): keypoints + 5 x point-to-scan term from iteration N//3+1 on,
        then the optional SMPL+D displacement loop; ``meshfile`` = path of an OBJ or a (vertices, faces) pair;
        ``use_mask=True`` (smplify.py:137-144,196-199,210): keypoints + 5 x silhouette term from iteration N//3+1 on;
        ``masks`` = [Nm,H,W] (one frame) or [B,Nm,H,W] uint8 images of the views ``mask_frames`` (ids looked up in
        ``use_frames``, the ids of the cameras passed in, :141-142)."""
        import ctypes as C
        from .. import _lib
        from ..engine import FrameBuffers, _stream
        m, dev, N = self.model, self.device, int(self.num_iters)
        init_betas, init_poses, kp = self._pack_inputs(net_output, keypoints)
        B, Nv = kp.shape[0], kp.shape[1]
        constant_scale = K.CONSTANT_SCALE_NO_SCAN
        searcher = scan_height = None
        if use_mesh:
            from ..utils.io_utils import load_obj_mesh
            from ..utils.mesh_grid_searcher import MeshGridSearcher
            scan_verts, scan_faces = load_obj_mesh(meshfile) if isinstance(meshfile, str) else meshfile
            scan_verts, scan_faces = np.asarray(scan_verts), np.asarray(scan_faces)
            tris = scan_verts[scan_faces]
            face_norms = np.cross(tris[:, 1] - tris[:, 0], tris[:, 2] - tris[:, 0])
            scan_height = float((scan_verts.max(0) - scan_verts.min(0))[1])
            constant_scale = scan_height / 1.7                                            # smplify.py:156
            searcher = MeshGridSearcher(verts=scan_verts, faces=scan_faces, device=dev)
        fb = FrameBuffers(m, B, full=True, Nv=Nv, n_trace=N, imsize=imsize, constant_scale=constant_scale,
                          expr_weight=self.expr_prior_weight)
        kp_dev = self._h2d('kp', kp)
        poses_dev, betas_dev = self._h2d('poses', init_poses), self._h2d('betas', init_betas)
        fb.bind('kp', pack_keypoints(kp_dev, self.use_hand_face))
        cams_np = pack_cameras(c2ws, Ks)
        fb.bind('cams', self._h2d('cams', torch.from_numpy(cams_np)))
        fb.t['theta'].copy_(m.pack_theta(poses_dev[:, :3], poses_dev[:, 3:3 + m.nbody], betas_dev))
        sil = None
        if use_mask:
            from .mask import SilhouetteTerm
            use_frames = list(use_frames) if use_frames is not None and len(use_frames) == Nv else list(range(Nv))
            idx = [use_frames.index(f) for f in mask_frames]
            sil = SilhouetteTerm(m, masks, cams_np[idx], imsize=imsize, device=dev)
            assert sil.B == B, 'masks for %d frames, parameters for %d' % (sil.B, B)
        if use_mesh:
            Pw = torch.empty(B, m.V, 3, device=dev)
            near = torch.empty(B, m.V, 3, device=dev)
            near_f = torch.empty(B, m.V, dtype=torch.int32, device=dev)
            pc = torch.zeros(B, device=dev)
        L = _lib.lib()
        for i in range(N):
            fb.struct.iter = i
            fb.call('bf_pose_forward')
            fb.call('bf_skin_forward', 1)
            fb.call('bf_keypoint_loss', 1)
            if i > (N // 3):
                if sil is not None:
                    sil.add(fb, 5.0)
                if use_mesh:
                    _lib.check(L.bf_pc_loss(C.byref(searcher.grid), m.struct, fb.struct, float(imsize / scan_height), 5.0,
                                            Pw.data_ptr(), near.data_ptr(), near_f.data_ptr(), pc.data_ptr(), _stream()), 'bf_pc_loss')
            fb.call('bf_gmm_prior')
            if i == N - 1:
                theta_prev = fb.t['theta'].clone()
            fb.call('bf_skin_backward', 1)
            fb.call('bf_pose_backward', 1 | 2 | 4)
        fb.call('bf_joints_forward', 1)                                   # joints of the last forward pass
        sp, sn = m.split_theta(theta_prev), m.split_theta(fb.t['theta'])
        t, s = sp['transl'][:, None, :], sp['scale'][:, None, :]
        verts = (fb.t['verts'].view(B, m.V, 3) + t) * s * constant_scale
        out = dict(vertices=verts, joints=(fb.t['joints'][:, :m.K_out] + t) * s * constant_scale, pose=sn['body_pose'],
                   betas=sn['betas'], global_orient=sn['global_orient'], global_transl=sn['transl'] * sn['scale'],
                   scale=sn['scale'], full_pose=fb.t['full_pose'])
        if m.is_smplx:
            out.update(leye_pose=sn['leye_pose'], reye_pose=sn['reye_pose'],
                       left_hand_pose=sn['left_hand_pose'], right_hand_pose=sn['right_hand_pose'])
        if m.face_params:
            out.update(jaw_pose=sn['jaw_pose'], expression=sn['expression'])
        self.last_trace, self.last_loss_terms = fb.t['trace'], fb.t['loss_terms']
        self.last_pc_loss = pc if use_mesh else None
        self.last_mask_loss = sil.mask_loss if sil is not None else None
        if displacement:
            assert use_mesh, 'the displacement fit needs a scan (use_mesh=True)'
            assert B == 1, 'the displacement fit takes one subject per call (smplify.py:229-247)'
            from .smpld import DisplacementFitter
            fitter = DisplacementFitter(searcher, face_norms, m.faces, m.V, constant_scale, device=dev)
            disp, dtrace = fitter.run(verts[0], N)
            out['displacement'] = disp[None]
            self.last_disp_trace = dtrace
        if as_numpy:
            out = {k: v.detach().cpu().squeeze(0).numpy() for k, v in out.items()}
        out['faces'] = self.smpl_faces[0]
        return out

    def session(self, B, Nv, imsize=512, return_vertices=True, host_io=None):
        """Device state for B frames, cached across calls of the same shape: a ConcurrentFitSession (staggered parts on
        their own streams) for large batches, a plain FitSession otherwise / when the temporal term couples the frames.
        ``host_io=True``: results go back to host memory (__call__ with as_numpy): up to ``concurrent_parts`` (4) parts whose
        graphs run at decreasing priority, so that an early part's 126 KB of vertices per frame travel while the later parts
        are still being fitted; ``False``: device-resident runs use at most 2 parts (measured: 48.6 ms per 10,000 frames with
        2 parts, 54.7 with 4 -- the GEMM CTAs of four parts crowd each other); ``None``: whichever was used last for this
        shape (device-resident if none yet)."""
        base = (int(B), int(Nv), int(self.num_iters), float(imsize), bool(return_vertices))
        cache = self.__dict__.setdefault('_sessions', {})
        if host_io is None:
            host_io = cache.get(('last', base), False)
        key = base + (bool(host_io),)
        if key not in cache:
            for k in [k for k in cache if k[0] != 'last' and k[:5] != base]:       # another shape: drop the old buffers
                del cache[k]
            n_parts = 1 if self.temporal_weight > 0 else self.concurrent_parts
            if not host_io and 'BODYFIT_PARTS' not in os.environ:
                n_parts = min(n_parts, self.device_parts)
            # host results: even a small batch (one rank's shard of a strong-scaled sequence) is cut into parts, because the
            # copy of its vertices is the expensive step there -- eight ranks share ~90 GB/s of host ingest (measured:
            # the end-to-end overhead over the device time is ~14 ms for 10,000 frames whether 1 or 8 GPUs produce them), so a
            # shard's copy takes as long as its fit and has to overlap it.  Single process, 1,250 frames: 17.4 ms as one part,
            # 16.4 ms as four (profiles/r2_e2e_parts_sweep.log).
            min_part = self.concurrent_min_part
            if host_io and 'BODYFIT_MIN_PART' not in os.environ:
                min_part = min(min_part, 256)
            if n_parts > 1 and len(staggered_ranges(B, n_parts, min_part=min_part)) > 1:
                cache[key] = ConcurrentFitSession(self.model, B, Nv, self.num_iters, imsize=imsize, return_vertices=return_vertices,
                                                  dense_every_iter=self.dense_every_iter, n_parts=n_parts,
                                                  min_part=min_part, lead=self.concurrent_lead,
                                                  taper=self.concurrent_taper, graph=self.graph, sort_frames=self.sort_frames,
                                                  expr_weight=self.expr_prior_weight)
            else:
                cache[key] = FitSession(self.model, B, Nv, self.num_iters, imsize=imsize,
                                        return_vertices=return_vertices, dense_every_iter=self.dense_every_iter,
                                        temporal_weight=self.temporal_weight, halo_exchange=self.halo_exchange, halo=self.halo,
                                        expr_weight=self.expr_prior_weight,
                                        graph=self.graph, sort_frames=self.sort_frames)
        cache[('last', base)] = bool(host_io)
        return cache[key]

    def _h2d(self, name, t):
        """Host tensor -> device.  Page-locked sources (torch pinned tensors, cudaHostRegister'ed numpy arrays) are copied
        by ONE asynchronous DMA straight from the caller's memory; pageable sources go through a pinned staging buffer
        (re-used across calls; an event guards the previous DMA out of it)."""
        t = t.contiguous()
        if t.is_cuda:
            return t
        if t.is_pinned():
            return t.to(self.device, non_blocking=True)
        p = self._pinned.get(('in', name))
        if p is None or p.shape != t.shape or p.dtype != t.dtype:
            p = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            self._pinned[('in', name)] = p
        ev = self._pinned.get(('ev', name))
        if ev is not None:
            ev.synchronize()                                   # the previous DMA out of this staging buffer is done
        p.copy_(t)
        d = p.to(self.device, non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream())
        self._pinned[('ev', name)] = ev
        return d

    def _host_results(self, host, nbytes):
        """Pinned staging buffers -> the arrays handed to the caller; a batch dimension of 1 is squeezed as the reference's
        ``cpu()`` does (smplify.py:252-254).  See ``copy_outputs`` in __init__."""
        copy = self.copy_outputs if self.copy_outputs is not None else nbytes <= (32 << 20)
        if copy:
            return {k: np.array(p.squeeze(0).numpy()) for k, p in host.items()}
        return {k: p.squeeze(0).numpy() for k, p in host.items()}

    def _d2h(self, out):
        """Device results -> numpy via pinned buffers (one async copy each, one sync)."""
        host = {}
        nbytes = 0
        for k, v in out.items():
            v = v.detach()
            p = self._pinned.get(('out', k))
            if p is None or p.shape != v.shape:
                p = torch.empty(v.shape, dtype=v.dtype, pin_memory=True)
                self._pinned[('out', k)] = p
            p.copy_(v, non_blocking=True)
            nbytes += int(v.numel() * v.element_size())
            host[k] = p
        torch.cuda.current_stream().synchronize()
        self.d2h_bytes = nbytes
        return self._host_results(host, nbytes)

    def cpu(self, tensor):
        return tensor.detach().cpu().squeeze(0).numpy()
