#!/usr/bin/env python3
"""Cost of the left-right consistency check (s3d_upsample_disp_eval with lr_mask, forward(..., lr_check=True)), in one run,
CUDA events, the arms alternating:

  1. the upsample kernel alone in its four forms -- plain (s3d_upsample_disp), eval (s3d_upsample_disp_eval with GT), lr and
     lr + eval (s3d_upsample_disp_eval with lr_mask, without / with GT) -- at B = 64, 256 x 256, D = 32 (1/4-res input
     64 x 64).  Four
     buffer sets are rotated (more than the 126 MB L2), so every launch writes its 33.5 MB of disparity (+ 8.4 MB of mask)
     to HBM and the GT arms read their 33.5 MB of GT from there;
  2. the default Stereo2Voxel forward replayed from its CUDA graph, model.graphed(left, right, gt) against the same call
     with lr_check=True, at the same shape.

Also records the launches per forward (lib.launches()) and the torch.profiler kernel list of one eager forward with and
without lr_check, and the GPU name and power limit beside the numbers.

    python scripts/lr_check_time.py [--reps 20] [--out profiles/lr_check_time.json]
"""
import argparse
import json
import os
import statistics
import sys

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from config import cfg as default_cfg                              # noqa: E402
from disp_eval_time import gpu_info, kernel_list, summary, time_alternating   # noqa: E402
from stereo_3d_reconstruction_b200 import lib, models as M, ops    # noqa: E402
from stereo_3d_reconstruction_b200.utils import synthetic          # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {'gpu': gpu_info()}
    dev = 'cuda'
    cfg = default_cfg.clone()
    B, H, W, D = 64, cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.NETWORK.MAX_DISP
    h, w = H // 4, W // 4
    th = list(cfg.TEST.DISP_THRESH)
    tau = cfg.TEST.LR_THRESH
    max_gt = 4.0 * D

    # 1. the kernel alone
    g = torch.Generator().manual_seed(0)
    sets = []
    for s in range(4):
        q = (torch.rand(2 * B, h, w, generator=g) * (D - 1)).to(dev)
        d = torch.randint(0, 2 * D, (B, H), generator=g)
        sets.append(dict(q=q, out=torch.empty(2 * B, H, W, device=dev), gt=synthetic.disparity_gt(d, H, W).to(dev),
                         st=torch.zeros(B, 2, 2 + len(th), dtype=torch.int64, device=dev),
                         mask=torch.empty(B, 2, H, W, dtype=torch.uint8, device=dev),
                         ls=torch.zeros(B, 2, 3 + len(th), dtype=torch.int64, device=dev)))

    def S(k):
        return sets[k % 4]
    arms = {
        'plain': lambda k: ops.upsample_disp(S(k)['q'], H, W, 4.0, out=S(k)['out']),
        'eval': lambda k: ops.upsample_disp_eval(S(k)['q'], H, W, 4.0, S(k)['gt'], th, max_gt, S(k)['st'], out=S(k)['out']),
        'lr': lambda k: ops.upsample_disp_eval(S(k)['q'], H, W, 4.0, thresholds=th, lr_thresh=tau, mask=S(k)['mask'],
                                               lr_stats=S(k)['ls'], out=S(k)['out']),
        'lr_eval': lambda k: ops.upsample_disp_eval(S(k)['q'], H, W, 4.0, S(k)['gt'], th, max_gt, S(k)['st'], lr_thresh=tau,
                                                    mask=S(k)['mask'], lr_stats=S(k)['ls'], out=S(k)['out']),
    }
    time_alternating(arms, 8, 3)                                    # warm-up
    k = time_alternating(arms, 200, args.reps)
    disp_bytes, mask_bytes = 2 * B * H * W * 4, 2 * B * H * W
    hbm = {'plain': disp_bytes, 'eval': 2 * disp_bytes, 'lr': disp_bytes + mask_bytes, 'lr_eval': 2 * disp_bytes + mask_bytes}
    res['kernel'] = {'shape': 'B=%d (2B=%d images) %dx%d from %dx%d, D=%d, T=%d, tau=%g' % (B, 2 * B, H, W, h, w, D, len(th), tau),
                     'buffer_sets': 4, 'calls_per_sample': 200, 'samples': args.reps, 'hbm_bytes': hbm}
    for name in arms:
        m = statistics.median(k[name])
        res['kernel'][name] = dict(summary(k[name]), TBps=hbm[name] / (m * 1e-3) / 1e12)
    med = {n: res['kernel'][n]['median_ms'] for n in arms}
    res['kernel']['lr_minus_plain_ms'] = med['lr'] - med['plain']
    res['kernel']['lr_eval_minus_eval_ms'] = med['lr_eval'] - med['eval']
    # the mask the timed arms wrote, as a sanity figure: the share of kept pixels of random, unrelated views
    res['kernel']['lr_density_last_set'] = float(sets[0]['mask'].float().mean().item())
    del sets

    # 2. the graphed forward
    model = M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * D, seed=1)
    left, right = left.to(dev), right.to(dev)
    gt = synthetic.gt_volume(B, seed=2).to(dev)
    with torch.no_grad():
        arms = {'graphed': lambda k: model.graphed(left, right, gt),
                'graphed_lr_check': lambda k: model.graphed(left, right, gt, lr_check=True)}
        time_alternating(arms, 3, 2)
        f = time_alternating(arms, 10, args.reps)
        m_p, m_l = statistics.median(f['graphed']), statistics.median(f['graphed_lr_check'])
        res['graphed_forward'] = {'shape': 'Stereo2Voxel default config, %s, B=%d, %dx%d, D=%d' % (cfg.NETWORK.PRECISION, B, H, W, D),
                                  'calls_per_sample': 10, 'samples': args.reps,
                                  'graphed': summary(f['graphed']), 'graphed_lr_check': summary(f['graphed_lr_check']),
                                  'added_ms': m_l - m_p, 'added_pct': 100.0 * (m_l - m_p) / m_p,
                                  'pairs_per_s': B / (m_p * 1e-3), 'pairs_per_s_lr_check': B / (m_l * 1e-3)}
        out = model.graphed(left, right, gt, lr_check=True)
        res['graphed_forward']['lr_density'] = float(out[-2].float().mean().item())
        # launches and kernels of one eager forward, with and without the check
        n0 = lib.launches(); model(left, right, gt); n1 = lib.launches()
        model(left, right, gt, lr_check=True); n2 = lib.launches()
        plain = kernel_list(lambda: model(left, right, gt))
        lr = kernel_list(lambda: model(left, right, gt, lr_check=True))
    res['launches'] = {'forward': n1 - n0, 'forward_lr_check': n2 - n1}
    res['kernels'] = {'forward': plain, 'forward_lr_check': lr}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            fh.write(txt + '\n')


if __name__ == '__main__':
    main()
