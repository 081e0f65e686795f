"""Golden vectors of the two reference paths that reference_fit_{smpl,smplx}.npz do not cover, for machines without a checkout
of the reference project:

  port_fit_kid.npz   age='kid' (smplify/smplify.py:50-56,112-115), the scene of
                     tests/test_oracle.py::test_kid_model_port_bit_exact_vs_verbatim_reference (seed 37, 4 views, 15 iterations);
  port_fit_mask.npz  the silhouette term (use_mask=True, smplify/loss.py:73-130), the scene of
                     tests/test_oracle.py::test_mask_term_port_bit_exact_vs_verbatim_reference (seed 12, 4 views, masks of
                     views 1 and 3, 10 iterations).

They hold the output of the oracle's restatement (oracle/fit_port.py FitPort.fit_frame), not of the reference itself: those
two live tests hold the restatement equal to the verbatim reference bit for bit on exactly these scenes, and the restatement
reproduces the reference-made reference_fit_*.npz bit for bit.  Made on one torch thread: once the silhouette term is on,
the contour argmin / inside-outside switches make the trajectory follow the last bit of every reduction, and those bits
depend on how many threads share a reduction.  Regenerate only after both live tests pass against a reference checkout:

    python tests/golden/make_golden_port.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, 'tests'))

KEYS = ('pose', 'betas', 'global_orient', 'global_transl', 'scale', 'joints', 'vertices', 'full_pose')


def kid_scene():
    from bodyfitting_b200 import synthetic as syn
    from oracle import fit_port as fp
    from util import make_scene
    model, gmm, jx = syn.make_model('smpl', 0), syn.make_gmm(0), syn.make_J_regressor_extra(seed=0)
    port = fp.FitPort('smpl', model, gmm, jx, age='kid', kid_template=syn.make_kid_template(0))
    sc = make_scene(fp.FitPort('smpl', model, gmm, jx), 'smpl', 1, 4, seed=37)
    return port, sc, dict(num_iters=15)


def mask_scene():
    from bodyfitting_b200 import synthetic as syn
    from oracle import fit_port as fp
    from util import gt_param_dict, make_scene
    mt, nv = 'smpl', 4
    port = fp.FitPort(mt, syn.make_model(mt, 0), syn.make_gmm(0), syn.make_J_regressor_extra(seed=0))
    sc = make_scene(port, mt, 1, nv, seed=12)
    ev = port.loss_and_grads(gt_param_dict(sc['gt'], mt), sc['c2ws'], sc['Ks'], np.zeros((1, nv, 25, 3), np.float32))
    mask_frames = [1, 3]
    masks = syn.make_masks(ev['vertices'][0], port.faces, sc['c2ws'], sc['Ks'])[mask_frames]
    return port, sc, dict(num_iters=10, masks=masks, mask_frames=mask_frames)


def main():
    import torch
    from bodyfitting_b200 import synthetic as syn
    torch.set_num_threads(1)
    for name, scene in (('kid', kid_scene), ('mask', mask_scene)):
        port, sc, kw = scene()
        views = syn.keypoints_to_openpose(sc['kp'][0], 'smpl')
        res, trace = port.fit_frame(sc['init_betas'][0], sc['init_pose'][0], sc['c2ws'], sc['Ks'], views, **kw)
        out = {('out_' + k): np.asarray(res[k]) for k in KEYS if k in res}
        out.update(c2ws=sc['c2ws'], Ks=sc['Ks'], kp=sc['kp'], init_pose=sc['init_pose'], init_betas=sc['init_betas'],
                   trace=np.asarray(trace, dtype=np.float64), num_iters=np.array(kw['num_iters']))
        if 'masks' in kw:
            out.update(masks=kw['masks'], mask_frames=np.array(kw['mask_frames']))
        fn = os.path.join(HERE, 'port_fit_%s.npz' % name)
        np.savez_compressed(fn, **out)
        print('wrote', fn, os.path.getsize(fn) // 1024, 'KiB', 'loss', trace[0], '->', trace[-1])


if __name__ == '__main__':
    main()
