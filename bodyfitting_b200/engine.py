"""Per-batch device buffers and the calls into the C ABI.

Torch is used for device memory, the current stream and autograd plumbing only; every
arithmetic step of the path is a kernel in ``libbodyfit_b200.so``.
"""
import os

import numpy as np
import torch

from . import _lib
from . import constants as K
from .model import PreparedModel


def _stream():
    return torch.cuda.current_stream().cuda_stream


class FrameBuffers(object):
    """Device buffers for B frames on one vertex set (``full=True``: all V vertices,
    else the active set).  Owns the ``BfFrames`` struct passed to the library."""

    def __init__(self, model: PreparedModel, B, full=False, Nv=0, need_backward=True, n_trace=0,
                 imsize=512.0, constant_scale=K.CONSTANT_SCALE_NO_SCAN, ext=None, temporal_weight=0.0,
                 expr_weight=K.EXPR_PRIOR_WEIGHT):
        _lib.require_device()
        self.model, self.B, self.full = model, int(B), bool(full)
        dev = model.device
        J, Kp, NP = model.J, model.Kp, model.NP
        self.ld_v = 3 * model.V if full else model.ld_act
        self.K_out = model.K_full if full else model.K_out_act
        f32 = dict(device=dev, dtype=torch.float32)
        t = {}
        ext = ext or {}

        def buf(name, *shape, zero=False, dtype=None):
            if name in ext and ext[name] is not None:
                t[name] = ext[name]
                return
            kw = dict(f32)
            if dtype is not None:
                kw['dtype'] = dtype
            t[name] = (torch.zeros if zero else torch.empty)(*shape, **kw)

        buf('theta', B, NP, zero=True)
        buf('pf', B, Kp)
        tc = model.tensor_cores
        if tc:
            buf('pf_hi', B, Kp)
            buf('pf_lo', B, Kp)
        buf('A', B, J, 12)
        buf('Jtr', B, J, 3)
        buf('full_pose', B, 3 * J)
        buf('yaw', B, dtype=torch.int32, zero=True)
        buf('verts', B, self.ld_v)
        buf('joints', B, self.K_out, 3)
        buf('loss', B, zero=True)
        if need_backward:
            buf('grad', B, NP, zero=True)
            buf('adam_m', B, NP, zero=True)
            buf('adam_v', B, NP, zero=True)
            buf('dpf', B, Kp)
            buf('dA', B, J, 12)
            buf('dJtr', B, J, 3)
            buf('vposed', B, self.ld_v)
            buf('dverts', B, self.ld_v, zero=True)
            buf('dvp', B, self.ld_v)
            if tc:                                 # 3xTF32 split of dvp, TMA-friendly padded rows, pad stays 0
                ldn = 3 * model.n_pad_full if full else model.ld_act
                buf('dvp_hi', B, ldn, zero=True)
                buf('dvp_lo', B, ldn, zero=True)
                nsplit = (ldn // 32 + 63) // 64          # accuracy: <= 2048 coordinates per accumulation run
                if nsplit > 1:
                    # + room to cut the reduction further when the tile grid alone would leave SMs idle (BODYFIT_BWD_FILL=1)
                    sms = torch.cuda.get_device_properties(dev).multi_processor_count
                    tiles = ((B + 127) // 128) * max(1, Kp // 256)
                    buf('ws', max(nsplit, min(64, sms // tiles)), B, Kp)
            buf('loss_terms', B, 4, zero=True)
            if tc and model.n_gmm and model.n_gmm * 72 % 192 == 0:
                buf('gmm_ws', B, model.n_gmm * 72 + 160)
            buf('gmm_grad', B, 69, zero=True)
            buf('gmm_loss', B, zero=True)
            buf('fwd_state', B, 24 * J)
            if tc and not full and model.n_act_pad <= 512:
                # per 128-frame tile the 16-vertex blocks of the active set its frames need (two buffers: iteration parity)
                buf('blk_mask', 2, (B + 127) // 128, zero=True, dtype=torch.int32)
                buf('dpf2', B, Kp, zero=True)            # second half-reduction of the masked backward GEMM
            if temporal_weight > 0:
                buf('tgrad', B, NP, zero=True)
                buf('tloss', B, zero=True)
        if n_trace:
            buf('trace', n_trace, B, zero=True)
        self.t = t
        s = _lib.BfFrames()
        for name, ten in t.items():
            setattr(s, name, ten.data_ptr())
        s.B, s.Nv, s.ld_v, s.iter = self.B, int(Nv), self.ld_v, 0
        s.flags = _lib.F_TC if tc else 0
        s.ws_floats = t['ws'].numel() if 'ws' in t else 0
        s.imsize, s.constant_scale, s.sigma = float(imsize), float(constant_scale), K.GMOF_SIGMA
        s.w_pose, s.w_angle, s.w_shape = K.POSE_PRIOR_WEIGHT, K.ANGLE_PRIOR_WEIGHT, K.SHAPE_PRIOR_WEIGHT
        s.lr_ts, s.lr = K.LR_TRANSL_SCALE, K.LR_DEFAULT
        s.beta1, s.beta2, s.eps = K.ADAM_BETAS[0], K.ADAM_BETAS[1], K.ADAM_EPS
        s.w_temporal = float(temporal_weight)
        s.w_expr = float(expr_weight)              # read by face-parameter models only
        self.struct = s

    def bind(self, name, tensor):
        """Point a struct field at an externally owned tensor (kept alive here)."""
        self.t[name] = tensor
        setattr(self.struct, name, tensor.data_ptr() if tensor is not None else None)

    def call(self, fn_name, *extra):
        L = _lib.lib()
        rc = getattr(L, fn_name)(self.model.struct, self.struct, *extra, _stream())
        _lib.check(rc, fn_name)


def pack_cameras(c2ws, Ks):
    """c2w [Nv,4,4], K [Nv,3,3] -> [Nv,12] fp32 rows of K @ inv(c2w)[:3] (smplify/smplify.py:131-135,
    smplify/loss.py:38-41 pre-composed in fp64 on the host)."""
    c2ws = np.asarray([np.asarray(c.detach().cpu() if torch.is_tensor(c) else c, dtype=np.float64) for c in c2ws])
    Ks = np.asarray([np.asarray(k.detach().cpu() if torch.is_tensor(k) else k, dtype=np.float64) for k in Ks])
    w2c = np.linalg.inv(c2ws.astype(np.float32)).astype(np.float64)         # the reference inverts in fp32
    M = np.einsum('vij,vjk->vik', Ks, w2c[:, :3, :])
    return np.ascontiguousarray(M.reshape(len(c2ws), 12).astype(np.float32))


def pack_keypoints(kp, use_hand_face):
    """[B,Nv,K,3] (x, y, conf) -> device layout [B,K,Nv,3] (x, y, effective weight), joint-major: the Nv views of
    one joint are 12*Nv contiguous bytes, so the (joint, view) lanes of the loss kernels read whole cache lines.
    Body joints weigh conf^2; the reference passes hand / face confidences as [N,1], which broadcasts against the
    [N] residuals, so every joint of such a group weighs sum_i conf_i^2 of that group and view
    (smplify/loss.py:134 with :168,:173,:179)."""
    kp = torch.as_tensor(kp, dtype=torch.float32)
    out = kp.clone()
    c2 = kp[..., 2] ** 2
    w = c2.clone()
    if use_hand_face:
        for lo, hi in ((25, 46), (46, 67), (67, 135)):
            w[..., lo:hi] = c2[..., lo:hi].sum(-1, keepdim=True)
    out[..., 2] = w
    return out.permute(0, 2, 1, 3).contiguous()


class FitSession(object):
    """All device state of a B-frame fit, allocated once and reusable across calls
    (smplify/smplify.py:84-226 for B frames in flight).

    ``run(theta0)`` = N iterations on the active vertex set; the reference returns the
    vertices / joints / full_pose of the LAST forward pass (parameters before the final
    Adam step) next to the parameters after it (smplify.py:216-226), so the all-vertex
    forward runs once, between iteration N-1 and N, writing world-space outputs directly.
    """

    def __init__(self, model: PreparedModel, B, Nv, num_iters, imsize=512, return_vertices=True,
                 chunk=4096, trace=True, dense_every_iter=False, temporal_weight=0.0, halo_exchange=None, out=None,
                 halo=None, graph=None, sort_frames=None, expr_weight=K.EXPR_PRIOR_WEIGHT):
        """``out`` (optional): externally owned result buffers for these B frames -- ``theta`` [B,NP], ``verts`` [B,V,3],
        ``joints`` [B,K_full,3], ``full_pose`` [B,3J] (contiguous row slices of a larger batch: ConcurrentFitSession).
        ``halo``: a sharding.HaloLink -- boundary rows of the temporal term travel by in-kernel NVLink stores (graph-capturable);
        ``halo_exchange``: the host-driven fallback (a callable, one NCCL send/recv pair per iteration).
        ``graph``: capture the whole run (N iterations + the all-vertex forward) in ONE CUDA graph on first use and replay it
        afterwards (default on; BODYFIT_GRAPH=0 or a host halo callback turn it off).  Inputs live in session-owned static
        buffers (``kp``, ``cams``, ``theta0``), so the captured pointers never change.
        ``sort_frames``: process the frames in the order of their contour (head-yaw) row at the initial pose, so that a
        128-frame tile of the blend GEMMs holds few rows and touches ~16 of the 30 vertex blocks of the SMPL-X active set
        (BfFrames.blk_mask).  Frames are independent fits, so the order is free; inputs are gathered and results scattered back
        by the packing kernels, all result tensors stay in the caller's frame order.  Default: on for SMPL-X batches of more
        than one tile without the temporal term (which couples neighbours); BODYFIT_SORT=0 turns it off.
        ``expr_weight``: weight of the expression prior of a face-parameter model (ignored otherwise)."""
        self.model, self.B, self.Nv, self.N = model, int(B), int(Nv), int(num_iters)
        assert self.N >= 1
        dev = model.device
        out = out or {}
        self.fb = FrameBuffers(model, B, full=False, Nv=Nv, n_trace=(self.N if trace else 0), imsize=imsize,
                               temporal_weight=temporal_weight, expr_weight=expr_weight)
        if sort_frames is None:
            sort_frames = os.environ.get('BODYFIT_SORT', '1') != '0'
        self.sort_frames = bool(sort_frames) and model.is_smplx and temporal_weight <= 0 and self.B > 128 and 'blk_mask' in self.fb.t
        # rows move during a fit (the pose converges: ~12 rows on the synthetic workload), so the order is renewed before a few
        # iterations: only theta / adam_m / adam_v rows are permuted, the keypoint rows stay behind `frame_index`
        self.resort_at, self.perm = [], None
        if self.sort_frames:
            self.perm = torch.arange(B, dtype=torch.int32, device=dev)          # current: sorted position -> caller's frame
            self.perm0 = self.perm.clone()                                      # order at the start of a run (initial poses)
            want = [int(x) for x in os.environ.get('BODYFIT_RESORT', '6,16,36').split(',') if x.strip()]
            self.resort_at = sorted(set(r for r in want if 0 < r < self.N - 1)) if not dense_every_iter else []
            self.perm_hist = torch.zeros(len(self.resort_at) + 1, B, dtype=torch.int32, device=dev)
            self._rows_tmp = torch.empty(B, model.NP, device=dev)
            self.fb.bind('frame_index', self.perm)
        self.theta_out = out['theta'] if out.get('theta') is not None else torch.zeros(B, model.NP, device=dev)
        # static inputs of the captured run
        self.kp = torch.zeros(B, model.K_used, Nv, 3, device=dev)
        self.cams = torch.zeros(Nv, 12, device=dev)
        self.theta0 = torch.zeros(B, model.NP, device=dev)
        self.fb.bind('kp', self.kp)
        self.fb.bind('cams', self.cams)
        # halo_exchange(first_row, last_row) -> (prev_row | None, next_row | None): boundary frames of the
        # neighbouring ranks, called before every iteration when the temporal term couples frames across shards
        self.halo = halo if temporal_weight > 0 else None
        self.halo_exchange = halo_exchange if (temporal_weight > 0 and self.halo is None) else None
        if self.halo is not None:
            self.fb.struct.halo_buf = self.halo.buf
            self.fb.struct.halo_peer_prev = self.halo.peer_prev
            self.fb.struct.halo_peer_next = self.halo.peer_next
            self.fb.struct.halo_iters = self.N
        self.theta_prev = torch.empty(B, model.NP, device=dev)
        self.verts = (out['verts'] if out.get('verts') is not None else torch.empty(B, model.V, 3, device=dev)) if return_vertices else None
        self.joints = out['joints'] if out.get('joints') is not None else torch.empty(B, model.K_full, 3, device=dev)
        self.full_pose = out['full_pose'] if out.get('full_pose') is not None else torch.empty(B, 3 * model.J, device=dev)
        self.dense_every_iter = bool(dense_every_iter)
        c = min(int(chunk), self.B)
        scratch = dict(pf=torch.empty(c, model.Kp, device=dev), pf_hi=torch.empty(c, model.Kp, device=dev),
                       pf_lo=torch.empty(c, model.Kp, device=dev), A=torch.empty(c, model.J, 12, device=dev),
                       Jtr=torch.empty(c, model.J, 3, device=dev), yaw=torch.zeros(c, dtype=torch.int32, device=dev),
                       loss=torch.zeros(c, device=dev))
        if not return_vertices:
            scratch['verts'] = torch.empty(c, 3 * model.V, device=dev)
        self.chunks = []
        for lo in range(0, self.B, c):
            hi = min(self.B, lo + c)
            ext = {k: v[:hi - lo] for k, v in scratch.items()}
            ext.update(theta=self.theta_prev[lo:hi], joints=self.joints[lo:hi], full_pose=self.full_pose[lo:hi])
            if return_vertices:
                ext['verts'] = self.verts[lo:hi].view(hi - lo, -1)
            fbf = FrameBuffers(model, hi - lo, full=True, need_backward=False, ext=ext)
            fbf.struct.flags |= _lib.F_WORLD
            self.chunks.append(fbf)
        self.kernel_launches = 0
        if graph is None:
            graph = os.environ.get('BODYFIT_GRAPH', '1') != '0'
        self.use_graph = bool(graph) and self.halo_exchange is None
        self.graph = None
        self.graphs = {}
        self._aligned = False

    def set_inputs(self, kp_packed, cams):
        """kp_packed [B,K_used,Nv,3] (x, y, effective weight; pack_keypoints) and cams [Nv,12], device tensors: copied into
        the session's static input buffers."""
        assert kp_packed.shape == (self.B, self.model.K_used, self.Nv, 3)
        if self.sort_frames:                              # theta0 arrives in the caller's order too
            self.perm0.copy_(torch.arange(self.B, dtype=torch.int32, device=self.perm.device))
        if kp_packed.data_ptr() != self.kp.data_ptr():
            self.kp.copy_(kp_packed)
        if cams.data_ptr() != self.cams.data_ptr():
            self.cams.copy_(cams)

    def load_inputs(self, kp_raw, cams, poses, betas):
        """Device tensors in the caller's layout -> the static input buffers, by two small kernels (no torch arithmetic):
        kp_raw [B,Nv,K,3] (x, y, conf), cams [Nv,12], poses [B,>=3+nbody], betas [B,10] (smplify.py:103-128)."""
        m = self.model
        assert kp_raw.shape == (self.B, self.Nv, m.K_used, 3) and kp_raw.is_contiguous() and kp_raw.dtype == torch.float32
        assert poses.is_contiguous() and betas.is_contiguous() and betas.shape == (self.B, 10)
        L, st = _lib.lib(), _stream()
        n = 2
        perm = None
        if self.sort_frames:
            # contour row of every frame at its initial pose -> stable argsort -> the packing kernels gather by it
            _lib.check(L.bf_init_theta(m.struct, poses.data_ptr(), int(poses.shape[1]), betas.data_ptr(), self.fb.t['theta'].data_ptr(),
                                       self.B, None, st), 'bf_init_theta')
            self.fb.struct.iter = 0
            self.fb.call('bf_pose_forward')
            self.perm0.copy_(torch.argsort(self.fb.t['yaw'], stable=True))
            perm = self.perm0.data_ptr()
            n += 2
        _lib.check(L.bf_pack_keypoints(kp_raw.data_ptr(), self.kp.data_ptr(), self.B, self.Nv, m.K_used, int(m.is_smplx), None, st),
                   'bf_pack_keypoints')                   # keypoint rows stay in the caller's order (frame_index)
        _lib.check(L.bf_init_theta(m.struct, poses.data_ptr(), int(poses.shape[1]), betas.data_ptr(), self.theta0.data_ptr(),
                                   self.B, perm, st), 'bf_init_theta')
        self.cams.copy_(cams, non_blocking=True)
        return n

    def _exchange(self):
        th = self.fb.t['theta']
        prev, nxt = self.halo_exchange(th[0], th[-1])
        self.fb.bind('halo_prev', prev)
        self.fb.bind('halo_next', nxt)

    def _dense_forward(self):
        n = 0
        sms = torch.cuda.get_device_properties(self.model.device).multi_processor_count
        for fbf in self.chunks:
            fbf.call('bf_lbs_forward')
            # pose, blend GEMM, per-frame skinning with the output joints fused in (a separate joints kernel when the frames
            # alone do not fill the SMs and the vertex range is cut into slabs)
            n += (3 if fbf.B >= 24 * sms else 4) if self.model.tensor_cores else 3
        return n

    def _body(self):
        """Every launch of one run, on the current stream (captured once, or issued directly)."""
        fb, N = self.fb, self.N
        fb.t['theta'].copy_(self.theta0)
        fb.t['adam_m'].zero_()
        fb.t['adam_v'].zero_()
        if 'blk_mask' in fb.t:
            fb.t['blk_mask'].zero_()
        if self.sort_frames:
            self.perm.copy_(self.perm0)
            self.perm_hist[0].copy_(self.perm0)
        launches = 0
        if self.halo is not None:
            fb.struct.iter = 0
            fb.call('bf_halo_begin', N)
            launches += 1
        # kernels of one iteration: blend GEMM, per-frame loss/backward, GMM prior (pack + GEMM + select on tensor cores,
        # one FFMA kernel otherwise), blend backward GEMM, pose backward (+ next pose forward); + temporal term if on
        per_it = 4 + (3 if 'gmm_ws' in fb.t else 1) + (1 if 'tgrad' in fb.t else 0)
        if self.dense_every_iter:
            # materialise all V vertices in every iteration, as the reference's model call does
            for it in range(N - 1):
                self._to_caller_order(fb.t['theta'], self.theta_prev)
                launches += self._dense_forward()
                fb.struct.iter = it
                fb.call('bf_fit_step')
                launches += per_it + 1
        elif self.halo_exchange is not None:
            for it in range(N - 1):
                self._exchange()
                fb.struct.iter = it
                fb.call('bf_fit_iteration', 1 if it == 0 else 0, 1)
                launches += per_it + (1 if it == 0 else 0)
        else:
            it = 0
            for k, stop in enumerate(self.resort_at + [N - 1]):
                if stop > it:
                    fb.struct.iter = it
                    fb.call('bf_fit_run', stop - it)
                    launches += per_it * (stop - it) + 1     # + the pose forward of the segment's first iteration
                it = stop
                if stop != N - 1:
                    launches += self._resort(it, k + 1)
        self._to_caller_order(fb.t['theta'], self.theta_prev)
        launches += self._dense_forward()
        fb.struct.iter = N - 1
        if self.halo_exchange is not None:
            self._exchange()
        fb.call('bf_fit_step')
        self._to_caller_order(fb.t['theta'], self.theta_out)
        launches += per_it + 1 + (2 if self.sort_frames else 0)
        self.kernel_launches = launches

    def _resort(self, it, k):
        """Renew the processing order before iteration ``it``: contour rows at the current iterate (one extra pose forward),
        stable argsort, theta / Adam rows permuted; the next segment starts with a pose forward in the new order."""
        fb = self.fb
        fb.struct.iter = it
        fb.call('bf_pose_forward')
        order = torch.argsort(fb.t['yaw'], stable=True)
        for name in ('theta', 'adam_m', 'adam_v'):
            torch.index_select(fb.t[name], 0, order, out=self._rows_tmp)
            fb.t[name].copy_(self._rows_tmp)
        self.perm.copy_(self.perm[order])
        self.perm_hist[k].copy_(self.perm)
        fb.t['blk_mask'][it & 1].zero_()                 # the forward above OR-ed the old order's rows into it
        return 1

    def _to_caller_order(self, src, dst):
        """rows of the (possibly row-sorted) batch -> the caller's frame order: dst[perm[r]] = src[r]"""
        if self.sort_frames:
            _lib.check(_lib.lib().bf_scatter_rows(src.data_ptr(), self.perm.data_ptr(), dst.data_ptr(), self.B, int(src.shape[1]),
                                                  _stream()), 'bf_scatter_rows')
        else:
            dst.copy_(src)

    def _capture(self, priority):
        """One uncaptured run on a capture stream (one-time setup of kernel attributes / side streams happens outside the
        capture), then the same launches recorded into a CUDA graph; the library's fork / join events to its side stream
        become graph edges.  A session keeps one graph per priority it is run with: the priority is written into the graph's
        kernel nodes (ConcurrentFitSession: decreasing priorities make the parts finish in order, so that the device->host
        copy of an early part overlaps the fitting of the later ones)."""
        dev = self.model.device
        cur = torch.cuda.current_stream(dev)
        gs = torch.cuda.Stream(device=dev) if priority is None else torch.cuda.Stream(device=dev, priority=priority)
        gs.wait_stream(cur)
        with torch.cuda.stream(gs):
            self._body()
        gs.synchronize()
        g = torch.cuda.CUDAGraph(keep_graph=priority is not None)
        with torch.cuda.graph(g, stream=gs, capture_error_mode='thread_local'):
            self._body()
        if priority is not None:
            # the launch stream's priority does not reach the kernels of a replayed graph: write it into the kernel nodes
            n = _lib.lib().bf_graph_set_kernel_priority(g.raw_cuda_graph(), int(priority))
            if n < 0:
                _lib.check(n, 'bf_graph_set_kernel_priority')
            g.instantiate()
        cur.wait_stream(gs)
        self.graphs[priority] = (g, gs)
        self.graph = g

    def run(self, theta0=None, priority=None):
        """N iterations from ``theta0`` ([B,NP] device tensor; None = whatever load_inputs / a previous call left in the
        static ``theta0`` buffer).  ``priority``: stream priority the graph's kernels run at (None = default)."""
        if theta0 is not None and theta0.data_ptr() != self.theta0.data_ptr():
            self.theta0.copy_(theta0)
        if self.halo is not None and not self._aligned:
            self.halo.align()
            self._aligned = True
        if self.use_graph:
            if priority not in self.graphs:
                self._capture(priority)
            self.graphs[priority][0].replay()
        else:
            self._body()
        return self.theta_out

    @property
    def theta(self):
        return self.theta_out

    def _unsorted(self, t, dim):
        """per-frame rows of the sorted batch -> the caller's order (diagnostics: loss trace / loss terms)"""
        if t is None or not self.sort_frames:
            return t
        out = torch.empty_like(t)
        out.index_copy_(dim, self.perm.long(), t)
        return out

    @property
    def trace(self):
        tr = self.fb.t.get('trace')
        if tr is None or not self.sort_frames:
            return tr
        out = torch.empty_like(tr)
        bounds = [0] + list(self.resort_at) + [self.N]           # iterations [bounds[k], bounds[k+1]) ran in order perm_hist[k]
        for k in range(len(bounds) - 1):
            out[bounds[k]:bounds[k + 1]].index_copy_(1, self.perm_hist[k].long(), tr[bounds[k]:bounds[k + 1]])
        return out

    @property
    def loss_terms(self):
        return self._unsorted(self.fb.t['loss_terms'], 0)

    def results(self):
        """Device tensors with the reference's result-dict keys (smplify.py:216-226)."""
        m = self.model
        sn = m.split_theta(self.theta_out)
        out = {}
        if self.verts is not None:
            out['vertices'] = self.verts
        out.update(joints=self.joints[:, :m.K_out], pose=sn['body_pose'], betas=sn['betas'], global_orient=sn['global_orient'],
                   global_transl=sn['transl'] * sn['scale'], scale=sn['scale'], full_pose=self.full_pose)
        if m.is_smplx:
            out.update(leye_pose=sn['leye_pose'], reye_pose=sn['reye_pose'],
                       left_hand_pose=sn['left_hand_pose'], right_hand_pose=sn['right_hand_pose'])
        if m.face_params:
            out.update(jaw_pose=sn['jaw_pose'], expression=sn['expression'])
        return out


def staggered_ranges(B, n_parts, grain=128, min_part=2048, lead=0, taper=0.5):
    """``lead`` > 0: a small first part of that many frames in front of the staggered ones -- its inputs are staged and
    uploaded quickly, so the GPU starts working while the host is still staging the large parts (end-to-end path only).

    Cut B frames into ``n_parts`` consecutive ranges of linearly shrinking size (multiples of ``grain`` frames = one
    GEMM row tile): run on streams of decreasing priority they finish in this order, so the results of the early, large
    parts travel to the host while the later parts are still being fitted and the last -- exposed -- copy is the smallest."""
    lead = (int(lead) // grain) * grain if min_part >= grain else int(lead)
    if lead > 0 and n_parts > 1 and B - lead >= 2 * min_part:
        rest = staggered_ranges(B - lead, n_parts, grain=grain, min_part=min_part, taper=taper)
        return [(0, lead)] + [(lo + lead, hi + lead) for lo, hi in rest]
    n_parts = max(1, min(int(n_parts), B // max(1, int(min_part))))   # a part should still fill the GPU a few times over
    grain = grain if min_part >= grain else 1
    if n_parts == 1:
        return [(0, B)]
    w = np.array([1.0 + float(taper) * k for k in range(n_parts)])[::-1]     # sizes shrink linearly; the last part weighs 1
    edges = np.round(np.cumsum(w) / w.sum() * B / grain).astype(np.int64) * grain
    edges[-1] = B
    lo, out = 0, []
    for hi in edges:
        hi = int(min(max(hi, lo + grain), B))
        out.append((lo, hi))
        lo = hi
    out[-1] = (out[-1][0], B)
    return [r for r in out if r[1] > r[0]]


class ConcurrentFitSession(object):
    """The B-frame fit as a few parts, each a FitSession on its own CUDA stream (frames are independent fits,
    smplify/body_fitting.py:82-91, so any partition gives bit-identical results).  Why: the per-frame kernels of one
    part fill the bubbles of the other parts' latency-bound ones (measured: 10,000 frames in 77 ms instead of 82 ms), and
    when the parts finish one after the other, the device->host copy of an early part's vertices (126 KB per SMPL-X
    frame) overlaps the remaining fitting instead of trailing it (SMPLify.__call__ uses ``prio_streams``: decreasing
    priority = finishing order = launch order, sizes shrinking so that the exposed last copy is the smallest;
    measured 112 -> 90 ms end to end per 10,000 frames).  ``run`` uses equal-priority streams (best device throughput).
    Same interface as FitSession (set_inputs / run / results)."""

    def __init__(self, model: PreparedModel, B, Nv, num_iters, imsize=512, return_vertices=True, dense_every_iter=False,
                 n_parts=4, trace=True, min_part=2048, lead=0, taper=0.5, graph=None, sort_frames=None,
                 expr_weight=K.EXPR_PRIOR_WEIGHT):
        self.model, self.B, self.Nv, self.N = model, int(B), int(Nv), int(num_iters)
        dev = model.device
        self.ranges = staggered_ranges(self.B, n_parts, min_part=min_part, lead=lead, taper=taper)
        self.theta = torch.zeros(B, model.NP, device=dev)
        self.verts = torch.empty(B, model.V, 3, device=dev) if return_vertices else None
        self.joints = torch.empty(B, model.K_full, 3, device=dev)
        self.full_pose = torch.empty(B, 3 * model.J, device=dev)
        self.parts, self.streams, self.prio_streams = [], [], []
        lowest, highest = 0, -3
        try:
            lowest, highest = torch.cuda.Stream.priority_range()
        except Exception:
            pass
        for k, (lo, hi) in enumerate(self.ranges):
            out = dict(theta=self.theta[lo:hi], joints=self.joints[lo:hi], full_pose=self.full_pose[lo:hi],
                       verts=self.verts[lo:hi] if return_vertices else None)
            self.parts.append(FitSession(model, hi - lo, Nv, num_iters, imsize=imsize, return_vertices=return_vertices,
                                         dense_every_iter=dense_every_iter, trace=trace, out=out, graph=graph, sort_frames=sort_frames,
                                         expr_weight=expr_weight))
            self.streams.append(torch.cuda.Stream(device=dev))
            self.prio_streams.append(torch.cuda.Stream(device=dev, priority=min(lowest, max(highest, highest + k))))
        self.kernel_launches = 0

    def set_inputs(self, kp_packed, cams):
        assert kp_packed.shape[0] == self.B
        for (lo, hi), p in zip(self.ranges, self.parts):
            p.set_inputs(kp_packed[lo:hi], cams)

    def load_inputs(self, kp_raw, cams, poses, betas):
        n = 0
        for (lo, hi), p in zip(self.ranges, self.parts):
            n += p.load_inputs(kp_raw[lo:hi], cams, poses[lo:hi], betas[lo:hi])
        return n

    def run(self, theta0=None):
        cur = torch.cuda.current_stream()
        ready = torch.cuda.Event()
        ready.record(cur)
        for (lo, hi), p, st in zip(self.ranges, self.parts, self.streams):
            st.wait_event(ready)
            with torch.cuda.stream(st):
                p.run(None if theta0 is None else theta0[lo:hi])
        for st in self.streams:
            cur.wait_stream(st)
        self.kernel_launches = sum(p.kernel_launches for p in self.parts)
        return self.theta

    @property
    def trace(self):
        ts = [p.trace for p in self.parts]
        return None if ts[0] is None else torch.cat(ts, dim=1)

    @property
    def loss_terms(self):
        return torch.cat([p.loss_terms for p in self.parts], dim=0)

    def results(self):
        m = self.model
        sn = m.split_theta(self.theta)
        out = {}
        if self.verts is not None:
            out['vertices'] = self.verts
        out.update(joints=self.joints[:, :m.K_out], pose=sn['body_pose'], betas=sn['betas'], global_orient=sn['global_orient'],
                   global_transl=sn['transl'] * sn['scale'], scale=sn['scale'], full_pose=self.full_pose)
        if m.is_smplx:
            out.update(leye_pose=sn['leye_pose'], reye_pose=sn['reye_pose'],
                       left_hand_pose=sn['left_hand_pose'], right_hand_pose=sn['right_hand_pose'])
        if m.face_params:
            out.update(jaw_pose=sn['jaw_pose'], expression=sn['expression'])
        return out
