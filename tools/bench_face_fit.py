#!/usr/bin/env python
"""Cost of optimising the SMPL-X jaw pose and expression coefficients (SMPLify(face_params=True)).

Times bench.py's headline workload -- SMPL-X, 8 views, 10,000 frames, 100 iterations, inputs resident on the device -- with
face parameters off and on, in alternating runs in one process, each timed with its own CUDA-event pair after an L2 flush
(a 256 MB fill).  Prints the card name and power limit with the numbers, and one JSON line.

  python tools/bench_face_fit.py [--frames 10000] [--rounds 5] [--warmup 2]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))


def card():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit', '--format=csv,noheader', '-i', '0'],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out.splitlines()[0] if out else 'unknown'
    except Exception as e:                          # the numbers stay valid; say that the card could not be read
        return 'unknown (%s)' % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--frames', type=int, default=10000)
    ap.add_argument('--iters', type=int, default=100)
    ap.add_argument('--rounds', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=2)
    args = ap.parse_args()
    import torch
    from bench import MT, NV, build_workload
    from bodyfitting_b200 import synthetic as syn
    from bodyfitting_b200.engine import pack_cameras
    from bodyfitting_b200.smplify.smplify import SMPLify
    torch.cuda.set_device(0)
    model_data, gmm = syn.make_model(MT, 0), syn.make_gmm(0)
    F = args.frames
    sessions = {}
    for on in (False, True):
        fit = SMPLify(smpl_type=MT, num_iters=args.iters, gender='neutral', model_data=model_data, gmm=gmm, face_params=on)
        wl = build_workload(fit.model, F, 100)
        sess = fit.session(F, NV, 512, True)
        cams = torch.from_numpy(pack_cameras(wl['c2ws'], wl['Ks'])).cuda()
        sess.load_inputs(torch.from_numpy(wl['kp']).cuda(), cams, torch.from_numpy(wl['init_pose']).cuda(),
                         torch.from_numpy(wl['init_betas']).cuda())
        sessions[on] = (fit, sess)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    for _ in range(args.warmup):
        for on in (False, True):
            sessions[on][1].run()
    torch.cuda.synchronize()
    ms = {False: [], True: []}
    for _ in range(args.rounds):
        for on in (False, True):
            flush.zero_()
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            sessions[on][1].run()
            e.record()
            torch.cuda.synchronize()
            ms[on].append(s.elapsed_time(e))
    dev = card()
    off_med, on_med = float(np.median(ms[False])), float(np.median(ms[True]))
    print('card: %s' % dev)
    print('SMPL-X, %d views, %d frames, %d iterations, device-resident; alternating runs (ms per fit):' % (NV, F, args.iters))
    print('  face parameters off: %s  median %.2f' % (' '.join('%.2f' % x for x in ms[False]), off_med))
    print('  face parameters on : %s  median %.2f  (%+.1f %%)' % (' '.join('%.2f' % x for x in ms[True]), on_med,
                                                                   100.0 * (on_med / off_med - 1.0)))
    print(json.dumps(dict(card=dev, frames=F, iters=args.iters, views=NV, off_ms=ms[False], on_ms=ms[True],
                          off_median_ms=off_med, on_median_ms=on_med)))


if __name__ == '__main__':
    main()
