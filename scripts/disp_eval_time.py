#!/usr/bin/env python3
"""Cost of the disparity evaluation (s3d_upsample_disp_eval, forward(..., disp_gt=...)), in one run, CUDA events, the two
arms alternating:

  1. the upsample kernel alone, s3d_upsample_disp against s3d_upsample_disp_eval, at B = 64, 256 x 256, D = 32 (1/4-res
     input 64 x 64).  Four disparity / GT / stats buffer sets are rotated (268 MB of outputs and GT, more than the 126 MB
     L2), so every launch writes its 33.5 MB of disparity to HBM and the eval arm also reads 33.5 MB of GT from there;
  2. the default Stereo2Voxel forward replayed from its CUDA graph, model.graphed(left, right, gt) against the same call
     with disp_gt, at the same shape.

Also prints the launches per forward (lib.launches()) and the torch.profiler kernel list of one eager forward with and
without disp_gt.  Prints the GPU name and power limit beside the numbers.

    python scripts/disp_eval_time.py [--reps 20] [--out FILE]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from config import cfg as default_cfg                              # noqa: E402
from stereo_3d_reconstruction_b200 import lib, models as M, ops    # noqa: E402
from stereo_3d_reconstruction_b200.utils import synthetic          # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:                                          # noqa: BLE001
        q = 'nvidia-smi unavailable (%s)' % e
    return {'device': torch.cuda.get_device_name(0), 'nvidia_smi': q}


def time_alternating(arms, inner, reps):
    """arms: {name: fn(k)}; each rep times `inner` calls of every arm in turn -> {name: [ms per call]}."""
    ev = {n: [] for n in arms}
    for _ in range(reps):
        for name, fn in arms.items():
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for k in range(inner):
                fn(k)
            b.record()
            b.synchronize()
            ev[name].append(a.elapsed_time(b) / inner)
    return ev


def summary(ms):
    return {'median_ms': statistics.median(ms), 'min_ms': min(ms), 'max_ms': max(ms)}


def kernel_list(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type.name == 'CUDA']


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
    max_gt = 4.0 * D

    # 1. the kernel alone
    g = torch.Generator().manual_seed(0)
    sets = []
    for s in range(4):
        q = (torch.rand(2 * B, h, w, generator=g) * (D - 1)).to(dev)
        d = torch.randint(0, 2 * D, (B, H), generator=g)
        sets.append(dict(q=q, out=torch.empty(2 * B, H, W, device=dev), gt=synthetic.disparity_gt(d, H, W).to(dev),
                         st=torch.zeros(B, 2, 2 + len(th), dtype=torch.int64, device=dev)))
    arms = {
        'upsample_disp': lambda k: ops.upsample_disp(sets[k % 4]['q'], H, W, 4.0, out=sets[k % 4]['out']),
        'upsample_disp_eval': lambda k: ops.upsample_disp_eval(sets[k % 4]['q'], H, W, 4.0, sets[k % 4]['gt'], th, max_gt,
                                                               sets[k % 4]['st'], out=sets[k % 4]['out']),
    }
    time_alternating(arms, 8, 3)                                    # warm-up
    k = time_alternating(arms, 200, args.reps)
    bytes_plain = 2 * B * H * W * 4
    res['kernel'] = {'shape': 'B=%d (2B=%d images) %dx%d from %dx%d, D=%d, T=%d' % (B, 2 * B, H, W, h, w, D, len(th)),
                     'buffer_sets': 4, 'calls_per_sample': 200, 'samples': args.reps,
                     'upsample_disp': summary(k['upsample_disp']), 'upsample_disp_eval': summary(k['upsample_disp_eval']),
                     'hbm_bytes_plain': bytes_plain, 'hbm_bytes_eval': 2 * bytes_plain}
    m_p, m_e = res['kernel']['upsample_disp']['median_ms'], res['kernel']['upsample_disp_eval']['median_ms']
    res['kernel']['added_ms'] = m_e - m_p
    res['kernel']['eval_TBps'] = 2 * bytes_plain / (m_e * 1e-3) / 1e12
    del sets

    # 2. the graphed forward
    model = M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * D, seed=1)
    left, right = left.to(dev), right.to(dev)
    gt = synthetic.gt_volume(B, seed=2).to(dev)
    dgt = synthetic.disparity_gt(d, H, W).to(dev)
    with torch.no_grad():
        arms = {'graphed': lambda k: model.graphed(left, right, gt),
                'graphed_disp_gt': lambda k: model.graphed(left, right, gt, disp_gt=dgt)}
        time_alternating(arms, 3, 2)
        f = time_alternating(arms, 10, args.reps)
        m_p, m_e = statistics.median(f['graphed']), statistics.median(f['graphed_disp_gt'])
        res['graphed_forward'] = {'shape': 'Stereo2Voxel default config, %s, B=%d, %dx%d, D=%d' % (cfg.NETWORK.PRECISION, B, H, W, D),
                                  'calls_per_sample': 10, 'samples': args.reps,
                                  'graphed': summary(f['graphed']), 'graphed_disp_gt': summary(f['graphed_disp_gt']),
                                  'added_ms': m_e - m_p, 'added_pct': 100.0 * (m_e - m_p) / m_p,
                                  'pairs_per_s': B / (m_p * 1e-3), 'pairs_per_s_disp_gt': B / (m_e * 1e-3)}
        # launches and kernels of one eager forward, with and without the evaluation
        n0 = lib.launches(); model(left, right, gt); n1 = lib.launches()
        model(left, right, gt, disp_gt=dgt); n2 = lib.launches()
        plain = kernel_list(lambda: model(left, right, gt))
        ev = kernel_list(lambda: model(left, right, gt, disp_gt=dgt))
    res['launches'] = {'forward': n1 - n0, 'forward_disp_gt': n2 - n1}
    res['kernels'] = {'forward': plain, 'forward_disp_gt': ev}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            fh.write(txt + '\n')


if __name__ == '__main__':
    main()
