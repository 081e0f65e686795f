"""Generates tests/golden/*.npz by running the reference's OWN, unmodified
smplify/smplify.py (SMPLify.__call__) + smplify/loss.py + smplify/prior.py + models/smpl.py
from a checkout of the reference project on the CPU (oracle/ref_harness.py; smplx arithmetic from the shim):
    BODYFIT_REFERENCE=<reference checkout> python tests/golden/make_golden.py
Inputs are the seeded synthetic model / scene of bodyfitting_b200.synthetic (seed 0), so the
fixtures stay small: only scene inputs and reference outputs are stored, never model tensors.
"""
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))


def main():
    import torch
    from bodyfitting_b200 import synthetic as syn
    from oracle import fit_port as fp, ref_harness as rh
    from util import make_scene
    assert rh.available(), 'needs a checkout of the reference project (BODYFIT_REFERENCE, or reference/ beside the repository)'
    tmp = tempfile.mkdtemp(prefix='bf_golden_')
    syn.write_data_dir(os.path.join(tmp, 'data'), seed=0)
    gmm, jx = syn.make_gmm(0), syn.make_J_regressor_extra(seed=0)
    for mt, nv, seed in (('smpl', 4, 21), ('smplx', 8, 22)):
        port = fp.FitPort(mt, syn.make_model(mt, 0), gmm, jx)
        sc = make_scene(port, mt, 1, nv, seed=seed)
        views = syn.keypoints_to_openpose(sc['kp'][0], mt)
        if mt == 'smpl':
            views[2] = None                     # a view without detection (smplify/loss.py:157)
            sc['kp'][0, 2] = 0.0
        res, trace, terms, _ = rh.run_reference_fit(tmp, mt, sc['init_betas'][0], sc['init_pose'][0], sc['c2ws'],
                                                    sc['Ks'], views, num_iters=100)
        out = {('out_' + k): np.asarray(v) for k, v in res.items() if k != 'faces'}
        out.update(c2ws=sc['c2ws'], Ks=sc['Ks'], kp=sc['kp'], init_pose=sc['init_pose'], init_betas=sc['init_betas'],
                   trace=np.asarray(trace, dtype=np.float64),
                   terms=np.asarray([[t[k] for k in ('reprojection_loss', 'pose_prior_loss', 'angle_prior_loss',
                                                     'shape_prior_loss')] for t in terms], dtype=np.float64),
                   torch_version=np.array(torch.__version__))
        fn = os.path.join(HERE, 'reference_fit_%s.npz' % mt)
        np.savez_compressed(fn, **out)
        print('wrote', fn, os.path.getsize(fn) // 1024, 'KiB', 'loss', trace[0], '->', trace[-1])


if __name__ == '__main__':
    main()
