#!/usr/bin/env python
"""Headline benchmark: fitted frames/s (SMPL-X, 8 views, 100 iters), BASELINE.json's metric.

  python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --steps K --warmup W    (CPU port of the reference path, rank 0 only)
  python bench.py --steps K --warmup W --dump-outputs DIR  (also writes the results of the last timed step to DIR/*.npy;
                                                            the inputs are seeded, so two builds can be compared file by file)

One *step* = one complete 100-iteration multi-view SMPLify fit of ONE synthetic sequence of ``--frames`` frames
(default 10,000 = BASELINE config 3).  STRONG scaling: the sequence is cut into contiguous frame ranges, one per rank
(``sharding.frame_range``); frames are independent fits, so no collective runs during the fit and one all_gather of the
fitted parameters ends the step.  ``--scaling weak`` gives every rank its own ``--frames`` frames instead (reported as the
extra key ``weak`` at N>1 in the default run).

  value : frames/s with inputs (keypoints, cameras, initial parameters) resident in HBM; every step is timed with its
          own CUDA-event pair on the launching stream, L2 flushed (a 256 MB fill) between steps, summed over the K steps
          after a barrier, max over ranks.
  e2e   : the same through the reference-facing API ``SMPLify.__call__`` with HOST (page-locked numpy) inputs and HOST
          numpy outputs (vertices included) -- H2D / D2H inside the timed region.
  roofline / kernels : per-kernel CUDA-event durations of one iteration and the algorithmic bytes of each kernel
          (DESIGN.md "Kernels"), for the dominant kernel of the step.
  lbs_dense : all-vertex LBS operator forward / backward (BASELINE config 2) against the HBM roofline.
  config4 : the same sequence with the temporal smoothness term; boundary rows cross GPUs by in-kernel NVLink stores
          (sharding.HaloLink) -- frames/s, halo cost per iteration, host-driven NCCL fallback beside it.
  config5 : SMPL+D scan path: uniform-grid build + closest-point search on 100k-vertex scans, subjects round-robin over
          the ranks; the reference's own mesh_grid kernel (oracle/_ref, compiled for sm_100a) timed on the same GPU.
  cpu_baseline : the oracle's single-frame restatement of the reference loop (oracle/fit_port.py, validated bit-for-bit
          against the verbatim reference in the authoring container) on the box's host cores; gpu_eager_baseline: the same
          eager op sequence on the B200 (the reference's default device) -- both reported, neither is the target.
"""
import argparse
import glob
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

METRIC = 'fitted frames/s (SMPL-X, 8 views, 100 iters)'
MT, NV, ITERS = 'smplx', 8, 100
TEMPORAL_W = 300.0


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--frames', type=int, default=10000, help='frames of the sequence (strong) / per GPU (weak)')
    ap.add_argument('--scaling', default='strong', choices=['strong', 'weak'])
    ap.add_argument('--iters', type=int, default=ITERS)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-dense', action='store_true')
    ap.add_argument('--no-extras', action='store_true', help='skip config4 / config5 / weak / GPU-eager legs')
    ap.add_argument('--cpu-frames', type=int, default=8)
    ap.add_argument('--weak', action='store_true', help='at N>1 also time the weak-scaling run (--frames on every rank)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps write the results of the last one as DIR/<name>.npy (at most 64 MB)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs writes the results of --impl ours; the reference leg times single-frame fits only')
    return args


def peaks():
    fn = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(fn):
        with open(fn) as f:
            d = json.load(f)
        return float(d['hbm_gbs']), 'measured (MEASURED_PEAKS.json)'
    return 6650.0, 'fallback (B200_PROFILING.md)'


def measured_traffic(kernel, frames):
    """dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed `ncu --set full` capture
    (profiles/r2_traffic.json, else r1_traffic.json; taken at 10,000 frames); None if this kernel / size was not captured."""
    for name in ('r2_traffic.json', 'r1_traffic.json'):
        fn = os.path.join(ROOT, 'profiles', name)
        if not os.path.exists(fn):
            continue
        with open(fn) as f:
            d = json.load(f).get(kernel)
        if d and d.get('frames') == frames:
            return d['dram_bytes_read'] + d['dram_bytes_write']
    return None


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.idx), '--query-gpu=' + self.Q,
                                          '--format=csv,noheader,nounits', '-lms', '200'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except Exception:
                continue
            for name, col in (('hw_slowdown', 5), ('hw_thermal_slowdown', 6), ('sw_thermal_slowdown', 7), ('sw_power_cap', 8)):
                if len(r) > col and r[col].lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': float(np.median(sm)) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'reasons': sorted(reasons), 'samples': len(sm)}


# ---------------------------------------------------------------------------------------------
def host_threads(share=1):
    """torchrun exports OMP_NUM_THREADS=1; the CPU legs use every core this process may run on (1/share of them when
    ``share`` ranks work side by side)."""
    import torch
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    torch.set_num_threads(max(1, n // max(1, share)))
    return torch.get_num_threads()


def cpu_reference_fit(n_frames, iters, warm=1, device='cpu'):
    """Reference-style single-frame fits (oracle port): on the host cores, or eagerly on the GPU. Returns s/frame list."""
    import torch
    from bodyfitting_b200 import synthetic as syn
    from oracle import fit_port as fp
    from util import make_scene
    cores = host_threads()
    model, gmm = syn.make_model(MT, 0), syn.make_gmm(0)
    port = fp.FitPort(MT, model, gmm)
    sc = make_scene(port, MT, n_frames + warm, NV, seed=11)
    if device != 'cpu':
        port = fp.FitPort(MT, model, gmm, device=device)
    times = []
    for f in range(n_frames + warm):
        views = syn.keypoints_to_openpose(sc['kp'][f], MT)
        if device != 'cpu':
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        port.fit_frame(sc['init_betas'][f], sc['init_pose'][f], sc['c2ws'], sc['Ks'], views, num_iters=iters)
        if device != 'cpu':
            torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if f >= warm:
            times.append(dt)
    return times, cores


def run_reference(args):
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    times, cores = cpu_reference_fit(args.steps, args.iters, warm=args.warmup)
    fps = len(times) / sum(times)
    line = {'impl': 'reference', 'metric': METRIC, 'value': fps, 'unit': 'frames/s', 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * sum(times) / len(times),
            'higher_is_better': True, 'scaling': args.scaling, 'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
            'config': {'workload': 'SMPL-X (10475 verts, 55 joints) 8-view 135-keypoint fit, %d Adam iterations, '
                                   '1 frame per step (the reference fits one frame per call)' % args.iters},
            'cpu_baseline': {'value': fps, 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                             'sample': '%d single-frame fits after %d warm-up, torch CPU fp32, oracle/fit_port.py '
                                       'FitPort.fit_frame (bit-exact restatement of smplify/smplify.py:84-226)' % (args.steps, args.warmup)},
            'e2e': {'value': fps, 'unit': 'frames/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
            'gpu_launches': 0}
    print(json.dumps(line))


# ---------------------------------------------------------------------------------------------
def build_workload(pm, F, seed, lo=0, hi=None):
    """Frames [lo, hi) of the synthetic F-frame scene ``seed``: GT joints from the CUDA forward, 2-D detections on the
    host.  Every rank draws the whole sequence's parameters (cheap) and keeps its own range, so the sequence does not
    depend on how it is sharded."""
    import torch
    from bodyfitting_b200 import synthetic as syn, _lib
    from bodyfitting_b200.engine import FrameBuffers
    hi = F if hi is None else hi
    c2ws, Ks = syn.make_cameras(NV, seed=0)
    gt, init = syn.make_params(MT, F, seed=seed)
    gt = {k: v[lo:hi] for k, v in gt.items()}
    init = {k: v[lo:hi] for k, v in init.items()}
    n = hi - lo
    T = lambda a: torch.from_numpy(np.ascontiguousarray(a))
    theta_gt = pm.pack_theta(T(gt['global_orient']), T(gt['body_pose']), T(gt['betas']), transl=T(gt['transl']),
                             scale=T(gt['scale']), leye=T(gt['leye_pose']), reye=T(gt['reye_pose']),
                             lhand=T(gt['left_hand_pose']), rhand=T(gt['right_hand_pose']))
    joints = torch.empty(n, pm.K_full, 3, device='cuda')
    chunk = 2048
    for a in range(0, n, chunk):
        b = min(n, a + chunk)
        fb = FrameBuffers(pm, b - a, full=True, need_backward=False,
                          ext=dict(theta=theta_gt[a:b].contiguous(), joints=joints[a:b]))
        fb.struct.flags |= _lib.F_WORLD
        fb.call('bf_lbs_forward')
    torch.cuda.synchronize()
    # detections: the noise stream is drawn per frame index so that a shard sees the frames of the whole sequence
    kp = syn.make_keypoints(joints[:, :pm.K_used].cpu().numpy(), c2ws, Ks, seed=seed + 7919 * lo)
    init_pose = np.concatenate([init['global_orient'], init['body_pose'], np.zeros((n, 6), np.float32)], 1)
    return dict(c2ws=c2ws, Ks=Ks, kp=kp, init_pose=np.ascontiguousarray(init_pose.astype(np.float32)),
                init_betas=np.ascontiguousarray(init['betas']))


def time_events(fn, reps):
    import torch
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(reps + 1)]
    ev[0].record()
    for i in range(reps):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    return [ev[i].elapsed_time(ev[i + 1]) for i in range(reps)]


DUMP_BYTES = 64 * 1000 * 1000


def frame_sample(n_frames, n, seed):
    """Frames kept in a dump: all of them, or a fixed, seeded sample of ``n`` in frame order."""
    if n >= n_frames:
        return np.arange(n_frames)
    return np.sort(np.random.RandomState(seed).choice(n_frames, max(1, n), replace=False))


def dump_outputs(out_dir, arrays):
    """``arrays``: name -> device tensor [frames, ...] of a fit's results, in frame order.  Writes out_dir/<name>.npy in
    float32 / float64, at most DUMP_BYTES in all: the parameters and joints of every frame while they fit into three
    quarters of it (else a seeded sample of frames), the vertices (126 KB per SMPL-X frame) as a seeded sample of frames in
    the rest.  frame_index.npy / vertices_frame_index.npy list the frames kept.  Returns the bytes written."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    n_frames = len(next(iter(arrays.values())))

    def write(names, budget, seed, index_name):
        row = sum(arrays[k][0].numel() * arrays[k].element_size() for k in names) + 8      # + the float64 index entry
        keep = frame_sample(n_frames, budget // row, seed)
        idx = torch.from_numpy(keep).to(arrays[names[0]].device)
        out = {index_name: keep.astype(np.float64)}
        out.update({k: arrays[k].index_select(0, idx).cpu().numpy() for k in names})
        n = 0
        for k, a in out.items():
            if a.dtype not in (np.float32, np.float64):
                a = a.astype(np.float64)
            fn = os.path.join(out_dir, k + '.npy')
            np.save(fn, a)
            n += os.path.getsize(fn)
        return n
    used = write(sorted(k for k in arrays if k != 'vertices'), DUMP_BYTES * 3 // 4, 0, 'frame_index')
    if 'vertices' in arrays:
        used += write(['vertices'], DUMP_BYTES - used - 4096, 1, 'vertices_frame_index')      # 4 KB: the two .npy headers
    return used


def kernel_breakdown(pm, sess, F, hbm_peak):
    """Per-kernel durations of ONE fit iteration (CUDA events, mean of 20) + algorithmic bytes."""
    fb = sess.fb
    m = pm
    nS3 = 3 * m.n_act
    J, Kp, NP, K, Nv = m.J, m.Kp, m.NP, m.K_used, sess.Nv
    bm_act = 4 * Kp * m.ld_act
    per_frame = {   # algorithmic bytes per frame (fp32), see DESIGN.md "Kernels"
        'k_pose_fwd': 4 * (NP + Kp * (3 if m.tensor_cores else 1) + J * 12 + J * 3 + 3 * J + 1),
        # tensor-core mode: the GEMM kernel only blends (pf -> v_posed) and the per-frame kernel skins its live vertices
        # from v_posed; FFMA mode: blend + skinning fused (v_posed and verts written, both read by the per-frame kernel)
        'k_skin_fwd': 4 * (Kp + nS3) if m.tensor_cores else 4 * (Kp + J * 12 + 2 * nS3),
        'k_frame_loss_bwd': 4 * (Nv * K * 3 + (1 if m.tensor_cores else 2) * nS3 + J * 3 + J * 12 + 4 + (2 if m.tensor_cores else 1) * nS3 + J * 12 + J * 3 + 4 + 1),
        'k_blend_bwd': 4 * (nS3 + Kp),
        'k_gmm_prior': 4 * (NP + 69 + 1),
        'k_pose_bwd': 4 * (NP * 7 + J * 12 + J * 3 + Kp + 2 + 70) + 4 * (Kp * (3 if m.tensor_cores else 1) + J * 12 + J * 3 + 3 * J + 1),
    }
    once = {'k_skin_fwd': bm_act, 'k_blend_bwd': bm_act}
    from bodyfitting_b200 import _lib

    def frame_kernel():
        if m.tensor_cores:
            fb.struct.flags |= _lib.F_SKIN_FUSED
        fb.call('bf_frame_loss_backward')
        fb.struct.flags &= ~_lib.F_SKIN_FUSED
    calls = [('k_pose_fwd', lambda: fb.call('bf_pose_forward')),
             ('k_skin_fwd', lambda: fb.call('bf_blend_forward' if m.tensor_cores else 'bf_skin_forward', 0)),
             ('k_frame_loss_bwd', frame_kernel),
             ('k_blend_bwd', lambda: fb.call('bf_skin_backward_parts', 0, 4)),
             ('k_gmm_prior', lambda: fb.call('bf_gmm_prior')),
             ('k_pose_bwd', lambda: fb.call('bf_pose_backward', 1 | 2 | 4 | 8))]   # incl. Adam + next iteration's pose forward
    out = []
    in_loop = {'k_pose_fwd': 0.0}            # fused into k_pose_bwd inside bf_fit_run (runs once per fit)
    for name, fn in calls:
        fn()
    for name, fn in calls:
        ms = float(np.mean(time_events(fn, 20)))
        by = per_frame[name] * F + once.get(name, 0)
        out.append({'kernel': name, 'ms': ms, 'bytes': by, 'gbs': by / ms / 1e6, 'frac_hbm': by / ms / 1e6 / hbm_peak,
                    'launches_per_iteration': in_loop.get(name, 1.0)})
    return out


def dense_lbs_bench(assets_seed, hbm_peak):
    """BASELINE config 2: SMPL, 1024 frames, all 6890 vertices: LBS forward / backward operator."""
    import torch
    from bodyfitting_b200 import synthetic as syn
    from bodyfitting_b200.engine import FrameBuffers
    from bodyfitting_b200.model import PreparedModel
    B = 1024
    pm = PreparedModel('smpl', syn.make_model('smpl', assets_seed), gmm=syn.make_gmm(assets_seed),
                       J_regressor_extra=syn.make_J_regressor_extra(seed=assets_seed), device='cuda')
    gt, _ = syn.make_params('smpl', B, seed=5)
    T = lambda a: torch.from_numpy(a)
    fb = FrameBuffers(pm, B, full=True)
    fb.t['theta'].copy_(pm.pack_theta(T(gt['global_orient']), T(gt['body_pose']), T(gt['betas'])))
    fb.bind('djoints', torch.randn(B, pm.K_full, 3, device='cuda'))
    fb.t['dverts'].normal_()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')

    def timed(fn, reps=10):
        ts = []
        for _ in range(reps):
            flush.zero_()                                  # evict L2 (126 MB) between timed launches
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record(); fn(); e.record(); torch.cuda.synchronize()
            ts.append(s.elapsed_time(e))
        return float(np.mean(ts))
    fb.call('bf_lbs_forward'); fb.call('bf_lbs_backward')
    V, J, Kout = pm.V, pm.J, pm.K_out
    alg = 4 * (3 * V + 3 * Kout + 72 + 10 + 4) * B            # SURVEY.md 8d: 83,612 B per frame
    fwd = timed(lambda: fb.call('bf_lbs_forward'))
    bwd = timed(lambda: fb.call('bf_lbs_backward'))
    # the blend GEMM alone against a TF32 peak measured the way MEASURED_PEAKS.json measures bf16 (cuBLAS, 8192^3, best of 5)
    gemm = {}
    try:
        fb.call('bf_pose_forward')
        g_ms = timed(lambda: fb.call('bf_blend_forward', 1)) if pm.tensor_cores else None
        old = torch.backends.cuda.matmul.allow_tf32
        torch.backends.cuda.matmul.allow_tf32 = True
        a, bm = torch.randn(8192, 8192, device='cuda'), torch.randn(8192, 8192, device='cuda')
        torch.matmul(a, bm)
        tf = max(2 * 8192 ** 3 / (t * 1e-3) / 1e12 for t in time_events(lambda: torch.matmul(a, bm), 5))
        torch.backends.cuda.matmul.allow_tf32 = old
        del a, bm
        gemm = {'tf32_cublas_tflops_measured': tf}
        if g_ms:
            fl = 3 * 2.0 * B * pm.Kp * 3 * pm.n_pad_full            # three TF32 MMAs per product (hi*hi + lo*hi + hi*lo)
            gemm.update(blend_gemm_ms=g_ms, blend_gemm_tf32_tflops=fl / (g_ms * 1e-3) / 1e12,
                        blend_gemm_frac_of_tf32_peak=fl / (g_ms * 1e-3) / 1e12 / tf,
                        note='3xTF32: the GEMM issues 3 MMAs per product, so at 100 %% of the TF32 peak it would still take '
                             '%.0f us, i.e. cap the forward at %.2f of the HBM roofline' % (fl / (tf * 1e12) * 1e6, alg / (fl / (tf * 1e12)) / 1e9 / hbm_peak))
    except Exception as ex:
        gemm = {'error': repr(ex)}
    return {'config': 'SMPL 6890 verts, 1024 frames (BASELINE config 2), L2 flushed between launches', 'gemm': gemm,
            'alg_bytes_per_frame': alg // B, 'design': 'v_posed and dv_posed are materialised (+12V B written and read each way); '
            'achieved uses the minimal algorithmic bytes of SURVEY.md 8d',
            'fwd_ms': fwd, 'bwd_ms': bwd, 'fwd_gbs': alg / fwd / 1e6, 'bwd_gbs': alg / bwd / 1e6,
            'fwd_frac_hbm': alg / fwd / 1e6 / hbm_peak, 'bwd_frac_hbm': alg / bwd / 1e6 / hbm_peak}


def config2_fit_bench():
    """BASELINE config 2 as a fit: SMPL, 1024 frames, 4 views, 25 keypoints, 100 iterations on one GPU (device-resident)."""
    import torch
    from bodyfitting_b200 import synthetic as syn
    from bodyfitting_b200.engine import FitSession, pack_cameras, pack_keypoints
    from bodyfitting_b200.model import PreparedModel
    B, nv, N = 1024, 4, 100
    pm = PreparedModel('smpl', syn.make_model('smpl', 0), gmm=syn.make_gmm(0),
                       J_regressor_extra=syn.make_J_regressor_extra(seed=0), device='cuda')
    gt, init = syn.make_params('smpl', B, seed=9)
    c2ws, Ks = syn.make_cameras(nv, seed=0)
    rng = np.random.RandomState(9)
    kp = np.concatenate([rng.rand(B, nv, 25, 2).astype(np.float32) * 512, rng.rand(B, nv, 25, 1).astype(np.float32)], -1)
    sess = FitSession(pm, B, nv, N)
    sess.set_inputs(pack_keypoints(torch.from_numpy(kp).cuda(), False), torch.from_numpy(pack_cameras(c2ws, Ks)).cuda())
    T = lambda a: torch.from_numpy(a).cuda()
    theta0 = pm.pack_theta(T(init['global_orient']), T(init['body_pose']), T(init['betas']))
    for _ in range(3):
        sess.run(theta0)
    ms = float(np.median(time_events(lambda: sess.run(theta0), 5)))
    return {'config': 'SMPL 6890 verts, 1024 frames, 4 views x 25 keypoints, 100 iterations (BASELINE config 2), one batch, '
                      'one CUDA graph' if sess.use_graph else 'one stream',
            'ms_per_fit': ms, 'frames_per_s': B / ms * 1e3, 'active_vertices': int(pm.n_act)}


def config5_bench(rank, world, n_subjects=8, searches=100):
    """BASELINE config 5 (SMPL+D scan path): per subject a 100k-vertex / 200k-face scan -> uniform-grid build, then
    ``searches`` closest-point searches of the 10,475 SMPL-X vertices (what the displacement loop does once per
    iteration).  Subjects round-robin over the ranks, no collective.  Rank 0 also times the reference's own mesh_grid
    kernel (oracle/_ref, compiled for sm_100a) on the first subject."""
    import torch
    from bodyfitting_b200 import synthetic as syn
    from bodyfitting_b200.utils.mesh_grid_searcher import MeshGridSearcher
    mine = list(range(rank, n_subjects, world))
    body, _ = syn.make_template(10475, 0)
    scans = {}
    for s in mine:
        v, f = syn.make_template(100000, 9 + s)
        scans[s] = ((v * 0.6).astype(np.float32), f.astype(np.int32))
    rng = np.random.RandomState(0)
    q = torch.from_numpy((body * 0.6 * 1.02 + rng.randn(*body.shape) * 0.004).astype(np.float32)).cuda()
    MeshGridSearcher(scans[mine[0]][0][:3000], scans[mine[0]][1][:10]) if mine else None      # warm-up
    torch.cuda.synchronize()
    build_ms, search_ms = [], []
    t_all = time.perf_counter()
    for s in mine:
        v, f = scans[s]
        vd, fd = torch.from_numpy(v).cuda(), torch.from_numpy(f).cuda()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        g = MeshGridSearcher(vd, fd)                       # on the rank's own GPU (the tensors' device)
        torch.cuda.synchronize()
        build_ms.append(1e3 * (time.perf_counter() - t0))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(searches):
            g.nearest_points(q)
        e1.record()
        torch.cuda.synchronize()
        search_ms.append(e0.elapsed_time(e1) / searches)
    wall = time.perf_counter() - t_all
    out = {'subjects': n_subjects, 'subjects_this_rank': len(mine), 'scan_verts': 100000, 'scan_faces': 200000, 'queries': 10475,
           'searches_per_subject': searches, 'grid_build_ms': float(np.mean(build_ms)) if build_ms else None,
           'nearest_ms': float(np.mean(search_ms)) if search_ms else None, 'rank_wall_s': wall}
    so = glob.glob(os.path.join(ROOT, 'oracle', '_ref', 'mesh_grid*.so'))
    if rank == 0 and so and mine:
        try:
            spec = importlib.util.spec_from_file_location('mesh_grid', so[0])
            mg = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(mg)
            v, f = scans[mine[0]]
            g = MeshGridSearcher(v, f)
            verts, fa = torch.from_numpy(v).cuda(), torch.from_numpy(f).cuda()
            num = torch.tensor(g.num, dtype=torch.int32).cuda()
            minmax = torch.from_numpy(np.asarray(g.minmax, np.float32)).cuda()
            tri_num = torch.zeros(g.num[3], dtype=torch.int32).cuda()
            tri_idx = torch.zeros(1, dtype=torch.int32).cuda()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            mg.insert_grid_surface(verts, fa, minmax, num, g.step, tri_num, tri_idx)
            torch.cuda.synchronize()
            out['reference_kernel_grid_build_ms'] = 1e3 * (time.perf_counter() - t0)
            nf = torch.zeros(len(q), dtype=torch.int32).cuda()
            co, npts = torch.zeros(len(q), 3).cuda(), torch.zeros(len(q), 3).cuda()
            fn = lambda: mg.search_nearest_point(q, verts, fa, tri_num, tri_idx, num, minmax, g.step, nf, npts, co)
            fn()
            out['reference_kernel_nearest_ms'] = float(np.median(time_events(fn, 5)))
            out['nearest_speedup_vs_reference_kernel'] = out['reference_kernel_nearest_ms'] / out['nearest_ms']
        except Exception as ex:
            out['reference_kernel'] = 'failed: %r' % (ex,)
    elif rank == 0:
        out['reference_kernel'] = 'oracle/_ref not built'
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist
    from bodyfitting_b200 import synthetic as syn
    from bodyfitting_b200.engine import FitSession
    from bodyfitting_b200.sharding import HaloLink, exchange_halo, frame_range
    from bodyfitting_b200.smplify.smplify import SMPLify
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        # NCCL announces its version on stdout when the first communicator is created; stdout must carry the ONE JSON
        # line only, so file descriptor 1 points at stderr while the communicator comes up
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', device_id=torch.device('cuda', local))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    host_threads(world)                                     # pinned staging / numpy of this rank may use its share of the cores
    t_start = time.perf_counter()

    def log(msg):
        sys.stderr.write('[bench rank %d +%.1fs] %s\n' % (rank, time.perf_counter() - t_start, msg))
        sys.stderr.flush()
    N = args.iters
    hbm_peak, peak_src = peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed_region(fn, K, W):
        """W untimed steps, barrier, K steps each bracketed by its own event pair with an L2 flush in front (not timed),
        barrier; the step times are summed per rank and the MAX over ranks is returned (plus the wall-clock maximum)."""
        for _ in range(W):
            fn()
        barrier()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
        wall = 0.0
        for s, e in ev:
            flush.zero_()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            s.record()
            fn()
            e.record()
            torch.cuda.synchronize()
            wall += time.perf_counter() - t0
        barrier()
        ms = sum(s.elapsed_time(e) for s, e in ev)
        if world > 1:
            t = torch.tensor([ms, wall * 1e3], device='cuda', dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1]) / 1e3
        return ms, wall

    def make_leg(F_total, lo, hi, temporal=0.0, halo=None, halo_exchange=None):
        """A fitter + device-resident session + pinned host inputs for frames [lo, hi) of the F_total-frame sequence."""
        fit = SMPLify(smpl_type=MT, num_iters=N, gender='neutral', model_data=model_data, gmm=gmm, temporal_weight=temporal,
                      halo=halo, halo_exchange=halo_exchange)
        wl = build_workload(fit.model, F_total, 100, lo, hi)
        pin = {k: torch.from_numpy(wl[k]).pin_memory() for k in ('kp', 'init_pose', 'init_betas')}
        from bodyfitting_b200.engine import pack_cameras
        sess = fit.session(hi - lo, NV, 512, True)
        cams = torch.from_numpy(pack_cameras(wl['c2ws'], wl['Ks'])).cuda()
        sess.load_inputs(pin['kp'].cuda(), cams, pin['init_pose'].cuda(), pin['init_betas'].cuda())
        torch.cuda.synchronize()
        host_args = ((pin['init_betas'].numpy(), pin['init_pose'].numpy()), list(wl['c2ws']), list(wl['Ks']), pin['kp'].numpy(), None)
        return fit, sess, host_args, pin

    model_data, gmm = syn.make_model(MT, 0), syn.make_gmm(0)
    if args.scaling == 'strong':
        F_total = args.frames
        lo, hi = frame_range(F_total, rank, world)
    else:
        F_total = args.frames * world
        lo, hi = rank * args.frames, (rank + 1) * args.frames
    F = hi - lo
    fit, sess, host_args, pin = make_leg(F_total, lo, hi)
    pm = fit.model
    from bodyfitting_b200.sharding import gather_frames

    def run_sess(s):
        return s.run()

    def step_device():
        theta = run_sess(sess)
        if world > 1:                                       # final gather of the fitted parameters
            gather_frames(theta, F_total)

    def step_e2e():
        out = fit(*host_args, use_frames=list(range(NV)), imsize=512)
        if world > 1:
            gather_frames(fit.session(F, NV, 512, True, host_io=True).theta, F_total)
        return out

    sampler = ClockSampler(local)
    sampler.start()
    ms_dev, wall_dev = timed_region(step_device, args.steps, max(args.warmup, 3))
    clocks = sampler.stop()
    if args.dump_outputs:
        # what a caller of the timed path holds after its last step: the fitted parameters run() returns and the session's
        # result tensors (the reference's result-dict keys), every frame of the sequence in frame order
        res = dict(sess.results(), theta=sess.theta)
        res = {k: gather_frames(v.contiguous(), F_total) for k, v in res.items()}
        if rank == 0:
            nb = dump_outputs(args.dump_outputs, res)
            log('results of the last timed step: %.1f MB written to %s' % (nb / 1e6, args.dump_outputs))
        del res
    launches = sess.kernel_launches * args.steps
    ms_e2e, wall_e2e = timed_region(step_e2e, args.steps, max(1, min(args.warmup, 3)))
    h2d, d2h = fit.h2d_bytes, fit.d2h_bytes
    if world > 1:
        t = torch.tensor([h2d, d2h, launches], device='cuda', dtype=torch.float64)
        dist.all_reduce(t)
        h2d, d2h, launches = (int(x) for x in t.tolist())

    # what the host link gives each rank while all ranks copy at once (pinned memory, 256 MB each way): the end-to-end path
    # moves 126 KB of vertices per fitted frame, so at several ranks this -- not the GPUs -- bounds `e2e`
    def link_gbs():
        nb = 256 << 20
        hbuf = torch.empty(nb, dtype=torch.uint8, pin_memory=True)
        dbuf = torch.empty(nb, dtype=torch.uint8, device='cuda')
        res = []
        for src, dst in ((dbuf, hbuf), (hbuf, dbuf)):
            dst.copy_(src, non_blocking=True)
            barrier()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            for _ in range(4):
                dst.copy_(src, non_blocking=True)
            e.record()
            torch.cuda.synchronize()
            res.append(4 * nb / (s.elapsed_time(e) / 1e3) / 1e9)
        t = torch.tensor(res, device='cuda', dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        return float(t[0]), float(t[1])
    d2h_gbs, h2d_gbs = link_gbs()

    frames_done = F_total * args.steps
    value = frames_done / (ms_dev / 1e3)
    e2e = frames_done / (max(ms_e2e / 1e3, wall_e2e))
    log('headline measured: %.0f frames/s device-resident, %.0f end to end' % (value, e2e))

    # ---- rank 0: per-kernel times, all-vertex operator, config 2 (single-GPU measurements; the other ranks wait) --------
    line = None
    if rank == 0:
        plain = FitSession(pm, F, NV, N, graph=False)       # one batch on one stream: per-kernel times of one iteration
        plain.load_inputs(pin['kp'].cuda(), sess.parts[0].cams if hasattr(sess, 'parts') else sess.cams, pin['init_pose'].cuda(),
                          pin['init_betas'].cuda())
        plain.run()
        kern = kernel_breakdown(pm, plain, F, hbm_peak)
        del plain
        iter_ms = sum(k['ms'] * k['launches_per_iteration'] for k in kern)
        dom = max(kern, key=lambda k: k['ms'] * k['launches_per_iteration'])
        kp_mb = F * pm.K_used * NV * 12 / 1e6
        state_mb = F * (2 * pm.Kp + 4 * pm.ld_act + 24 * pm.J + 4 * pm.NP) * 4 / 1e6
        line = {
            'metric': METRIC, 'value': value, 'unit': 'frames/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': max(args.warmup, 3), 'ms_per_step': ms_dev / args.steps, 'higher_is_better': True, 'scaling': args.scaling,
            'vs_baseline': None, 'dtype': 'fp32', 'data': 'synthetic',
            'config': {'workload': 'SMPL-X (10475 verts, 55 joints, random-init tensors) 8-view fit of ONE %d-frame sequence, '
                                   '135 OpenPose-layout keypoints per view, %d Adam iterations (BASELINE config 3), frame-sharded over '
                                   '%d GPU(s)' % (F_total, N, world),
                       'frames_total': F_total, 'frames_per_gpu': F, 'views': NV, 'iters': N, 'active_vertices': int(pm.n_act),
                       'design': 'fit loop runs blend+skinning on the %d vertices the keypoint loss can touch (exact: all other '
                                 'vertex gradients are zero); all 10475 vertices are produced once for the returned mesh' % pm.n_act,
                       'l2': 'L2 flushed (256 MB fill) before every timed step; per step %.0f MB of keypoints + %.0f MB of '
                             'per-frame state per rank' % (kp_mb, state_mb),
                       'parallelism': 'frames sharded, %d rank(s), no collective during the fit; final all_gather of parameters' % world,
                       'streams': 'per GPU the shard runs as %d part(s), each ONE CUDA graph (N iterations + all-vertex forward) on '
                                  'its own stream (bit-identical results); kernels[] / roofline are timed on one batch on one stream'
                                  % (len(getattr(sess, 'ranges', [0])))},
            'clocks': clocks,
            'e2e': {'value': e2e, 'unit': 'frames/s', 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h),
                    'ms_per_step': 1e3 * max(ms_e2e / 1e3, wall_e2e) / args.steps,
                    'host_link': {'d2h_gbs_per_rank_all_ranks_copying': d2h_gbs, 'h2d_gbs_per_rank_all_ranks_copying': h2d_gbs,
                                  'd2h_bound_frames_per_s': world * d2h_gbs * 1e9 / (d2h / max(1, world) / max(1, F)) if d2h else None},
                    'api': 'bodyfitting_b200.smplify.smplify.SMPLify.__call__ (page-locked numpy in, numpy out incl. vertices)'},
            'gpu_launches': int(launches),
            'roofline': {'bound': 'hbm', 'kernel': dom['kernel'], 'achieved': dom['gbs'], 'peak': hbm_peak, 'unit': 'GB/s',
                         'frac': dom['frac_hbm'], 'traffic': measured_traffic(dom['kernel'], F), 'peak_source': peak_src,
                         'share_of_iteration': dom['ms'] / iter_ms},
            'kernels': kern, 'iter_ms_sum_of_kernels': iter_ms,
        }
        if not args.no_dense:
            try:
                line['lbs_dense'] = dense_lbs_bench(0, hbm_peak)
            except Exception as ex:                          # report, never hide
                line['lbs_dense'] = {'error': repr(ex)}
            try:
                line['config2_fit'] = config2_fit_bench()
            except Exception as ex:
                line['config2_fit'] = {'error': repr(ex)}
        log('rank-0 kernel / operator measurements done')

    # ---- extra legs (configs 4 / 5, weak scaling).  They run under an emergency timer: if one of them blocks, rank 0 prints
    # the line it already holds (marked) and every rank leaves -- the headline is never hostage to an extra leg.
    extras = {}
    printed = threading.Event()

    def emit():
        if printed.is_set():
            return
        printed.set()
        if rank == 0:
            line.update(extras)
            sys.stdout.write(json.dumps(line) + '\n')
            sys.stdout.flush()

    def emergency():
        import faulthandler
        log('extra legs exceeded their time budget: printing what is there and leaving')
        faulthandler.dump_traceback(file=sys.stderr)
        extras['extras_timed_out'] = True
        emit()
        os._exit(0)
    timer = None
    if not args.no_extras:
        timer = threading.Timer(240.0 if world > 1 else 900.0, emergency)
        timer.daemon = True
        timer.start()
        barrier()
        # config 4: temporal term, boundary rows by in-kernel NVLink stores
        try:
            log('config4: temporal fit, NVLink halo')
            link = HaloLink()
            fit_t, sess_t, _, _ = make_leg(F_total, lo, hi, temporal=TEMPORAL_W, halo=link)
            k4 = max(2, min(args.steps, 5))
            ms_t, _ = timed_region(lambda: run_sess(sess_t), k4, 2)
            c4 = {'workload': 'config 3 + temporal smoothness term (weight %.0f) coupling consecutive frames; %d-frame sequence over '
                              '%d rank(s)' % (TEMPORAL_W, F_total, world), 'halo': 'in-kernel NVLink peer stores + flag (HaloLink)' if world > 1 else 'none (one rank)',
                  'frames_per_s': F_total * k4 / (ms_t / 1e3), 'ms_per_fit': ms_t / k4, 'graph': bool(sess_t.use_graph)}
            if world > 1:
                # the same shards without the link (every shard its own sequence): the difference is what the halo costs
                log('config4: same shards without the link')
                fit_u, sess_u, _, _ = make_leg(F_total, lo, hi, temporal=TEMPORAL_W)
                ms_u, _ = timed_region(lambda: run_sess(sess_u), k4, 2)
                c4['ms_per_fit_without_halo'] = ms_u / k4
                c4['halo_us_per_iteration'] = 1e3 * (ms_t - ms_u) / k4 / N
                log('config4: host NCCL fallback')
                fit_h, sess_h, _, _ = make_leg(F_total, lo, hi, temporal=TEMPORAL_W, halo_exchange=exchange_halo)
                ms_h, _ = timed_region(lambda: run_sess(sess_h), 2, 1)
                c4['host_nccl_fallback_ms_per_fit'] = ms_h / 2
                c4['host_nccl_fallback_halo_us_per_iteration'] = 1e3 * (ms_h / 2 - ms_u / k4) / N
                del fit_u, sess_u, fit_h, sess_h
            extras['config4'] = c4
            del fit_t, sess_t
        except Exception as ex:                              # report, never hide
            log('config4 failed: %r' % (ex,))
            extras['config4'] = {'error': repr(ex)}
        try:
            log('config5: scan path')
            c5 = config5_bench(rank, world)
            if world > 1:
                t = torch.tensor([c5['rank_wall_s']], device='cuda', dtype=torch.float64)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                c5['wall_s_max_over_ranks'] = float(t[0])
            else:
                c5['wall_s_max_over_ranks'] = c5['rank_wall_s']
            c5['subjects_per_s'] = c5['subjects'] / c5['wall_s_max_over_ranks']
            extras['config5'] = c5
        except Exception as ex:
            log('config5 failed: %r' % (ex,))
            extras['config5'] = {'error': repr(ex)}
        if world > 1 and args.scaling == 'strong' and args.weak:
            try:                                             # weak scaling beside it: --frames frames on EVERY rank
                log('weak leg: %d frames on every rank' % args.frames)
                fit_w, sess_w, _, _ = make_leg(args.frames * world, rank * args.frames, (rank + 1) * args.frames)
                log('weak leg: session ready')
                ms_w, _ = timed_region(lambda: run_sess(sess_w), 3, 2)
                extras['weak'] = {'frames_per_gpu': args.frames, 'value': args.frames * world * 3 / (ms_w / 1e3), 'unit': 'frames/s',
                                  'ms_per_step': ms_w / 3}
                del fit_w, sess_w
            except Exception as ex:
                log('weak leg failed: %r' % (ex,))
                extras['weak'] = {'error': repr(ex)}
        log('extra legs done')

    if world > 1:
        barrier()
    if timer is not None:
        timer.cancel()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if world > 1:
        dist.destroy_process_group()
    if world == 1 and not args.no_extras:
        try:
            times, _ = cpu_reference_fit(2, N, warm=1, device='cuda')
            extras['gpu_eager_baseline'] = {'value': len(times) / sum(times), 'unit': 'frames/s', 'kind': 'port on device=cuda',
                                            'sample': '2 single-frame SMPL-X 8-view %d-iteration fits after 1 warm-up: the reference\'s '
                                                      'eager torch op sequence (oracle/fit_port.py) on the B200 -- launch-bound, not the target' % N}
        except Exception as ex:
            extras['gpu_eager_baseline'] = {'error': repr(ex)}
    if world == 1 and not args.no_cpu_baseline:
        times, cores = cpu_reference_fit(args.cpu_frames, N, warm=1)
        extras['cpu_baseline'] = {'value': len(times) / sum(times), 'unit': 'frames/s', 'cores': cores, 'kind': 'port',
                                  'sample': '%d single-frame SMPL-X 8-view %d-iteration fits after 1 warm-up (oracle/fit_port.py '
                                            'FitPort.fit_frame, torch CPU fp32, %d host cpus)' % (len(times), N, os.cpu_count())}
    emit()


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
