#!/usr/bin/env python
"""Cost of wider SMPL-X hands (SMPLify(num_pca_comps=, use_pca=)).

Times bench.py's headline workload -- SMPL-X, 8 views, 10,000 frames, 100 iterations, inputs resident on the device -- with
the default hands (6 PCA components, theta rows of 98 entries), 12 PCA components (110 entries) and axis-angle hands (176
entries: the wide pose kernels), in alternating runs in one process, each timed with its own CUDA-event pair after an L2
flush (a 256 MB fill).  The model is the synthetic one with 45-row hand component tables (tests/test_host_hand_pose.py);
with num_pca_comps=6 it is the default model byte for byte.  Prints the card name and power limit with the numbers, and one
JSON line.

  python tools/bench_hand_fit.py [--frames 10000] [--rounds 5] [--warmup 2]
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
    from test_host_hand_pose import hand_model
    torch.cuda.set_device(0)
    model_data, gmm = hand_model(0), syn.make_gmm(0)
    F = args.frames
    configs = {'pca6': {}, 'pca12': dict(num_pca_comps=12), 'axis-angle': dict(use_pca=False)}
    sessions, wl = {}, None
    for name, hk in configs.items():
        fit = SMPLify(smpl_type=MT, num_iters=args.iters, gender='neutral', model_data=model_data, gmm=gmm, **hk)
        if wl is None:                              # one set of inputs (made with the default hands) for every configuration
            wl = build_workload(fit.model, F, 100)
        sess = fit.session(F, NV, 512, True)
        cams = torch.from_numpy(pack_cameras(wl['c2ws'], wl['Ks'])).cuda()
        sess.load_inputs(torch.from_numpy(wl['kp']).cuda(), cams, torch.from_numpy(wl['init_pose']).cuda(),
                         torch.from_numpy(wl['init_betas']).cuda())
        sessions[name] = (fit, sess)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device='cuda')
    for _ in range(args.warmup):
        for name in configs:
            sessions[name][1].run()
    torch.cuda.synchronize()
    ms = {name: [] for name in configs}
    for _ in range(args.rounds):
        for name in configs:
            flush.zero_()
            torch.cuda.synchronize()
            s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            s.record()
            sessions[name][1].run()
            e.record()
            torch.cuda.synchronize()
            ms[name].append(s.elapsed_time(e))
    dev = card()
    med = {name: float(np.median(v)) for name, v in ms.items()}
    print('card: %s' % dev)
    print('SMPL-X, %d views, %d frames, %d iterations, device-resident; alternating runs (ms per fit):' % (NV, F, args.iters))
    for name in configs:
        print('  %-10s NP %3d: %s  median %.2f  (%+.1f %%)' % (name, sessions[name][0].model.NP, ' '.join('%.2f' % x for x in ms[name]),
                                                               med[name], 100.0 * (med[name] / med['pca6'] - 1.0)))
    print(json.dumps(dict(card=dev, frames=F, iters=args.iters, views=NV, ms=ms, median_ms=med)))


if __name__ == '__main__':
    main()
