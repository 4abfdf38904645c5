#!/usr/bin/env python3
"""Cost of the speckle filter (s3d_speckle_filter, forward(..., speckle=True)), in one run:

  1. the four kernels alone at B = 64, 256 x 256, through the C entry point into preallocated buffers, on
     - the disparity maps of one default Stereo2Voxel forward of the synthetic pairs (lr_check=True, with the GT disparity),
       without and with the LR mask and the GT;
     - a constant map (one region per map), a map of isolated pixels (a checkerboard of two values 2 * max_diff apart: every
       pixel its own region) and a serpentine region (full rows joined at alternating ends: one region per map that crosses
       every tile border and makes the longest union chains);
     L2 is overwritten (256 MB write) before every call: CUDA events around each single call (the arms alternating), and
     torch.profiler device times of each kernel in a run of their own, flushed the same way;
  2. the default Stereo2Voxel forward replayed from its CUDA graph at B = 64, model.graphed(left, right) against
     model.graphed(left, right, speckle=True), alternating, with the launches per eager forward of each.

Also records the kept fraction, the removed regions and pixels of every arm, and the GPU name and power limit beside the
numbers.

    python scripts/speckle_time.py [--reps 20] [--out profiles/speckle_time.json]
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
from disp_eval_time import gpu_info, summary, time_alternating     # noqa: E402
from point_eval_time import flushed_alternating                    # noqa: E402
from stereo_3d_reconstruction_b200 import lib, models as M, ops    # noqa: E402
from stereo_3d_reconstruction_b200.utils import synthetic          # noqa: E402

_KERNELS = ('speckle_local_kernel', 'speckle_border_kernel', 'speckle_size_kernel', 'speckle_finish_kernel')


def kernels_device_us(fn, flush, calls):
    """Mean device time per call of each speckle kernel over `calls` calls of fn, each after an L2 flush (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            flush.zero_()
            fn()
        torch.cuda.synchronize()
    out = {}
    for k in _KERNELS:
        ts = [e.device_time_total if hasattr(e, 'device_time_total') else e.cuda_time_total
              for e in prof.events() if e.device_type.name == 'CUDA' and k in e.name]
        out[k] = {'launches_seen': len(ts), 'mean_us': sum(ts) / len(ts) if ts else None}
    if all(out[k]['mean_us'] is not None for k in _KERNELS):
        out['all_us'] = sum(out[k]['mean_us'] for k in _KERNELS)
    return out


def synthetic_maps(kind, B, H, W, max_diff):
    """[2B,H,W] fp32 maps of the synthetic arms (module docstring)."""
    if kind == 'constant':
        return torch.full((2 * B, H, W), 7.0)
    if kind == 'isolated':
        y, x = torch.meshgrid(torch.arange(H), torch.arange(W), indexing='ij')
        return (((x + y) % 2).float() * (2 * max_diff + 1)).expand(2 * B, H, W).contiguous()
    d = torch.full((H, W), float('nan'))                               # serpentine
    d[0::2] = 3.0
    for y in range(1, H, 2):
        d[y, W - 1 if (y // 2) % 2 == 0 else 0] = 3.0
    return d.expand(2 * B, H, W).contiguous()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {'gpu': gpu_info()}
    dev = 'cuda'
    cfg = default_cfg.clone()
    B, H, W, D = cfg.CONST.BATCH_SIZE, cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.NETWORK.MAX_DISP
    max_size, max_diff = M.speckle_params(cfg)
    th = [float(t) for t in cfg.TEST.DISP_THRESH]
    T, max_gt = len(th), 4.0 * D
    model = M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()
    left, right, dg = synthetic.stereo_pair(B, H, W, 2 * D, seed=1)
    left, right = left.to(dev).contiguous(), right.to(dev).contiguous()
    disp_gt = synthetic.disparity_gt(dg, H, W).to(dev).contiguous()

    # 1. the kernels alone
    with torch.no_grad():
        o = dict(zip(M.Stereo2Voxel.output_names(disp_gt=True, lr_check=True),
                     model(left, right, disp_gt=disp_gt, lr_check=True)))
        fwd = torch.cat([o['disp_left'][:, 0], o['disp_right'][:, 0]]).contiguous()
        lr_mask = o['lr_mask'].clone()
    mask = torch.empty(B, 2, H, W, dtype=torch.uint8, device=dev)
    stats = torch.zeros(B, 2, 5 + T, dtype=torch.int64, device=dev)
    nb = ops.speckle_filter_workspace_bytes(B, H, W)
    ws = torch.empty(nb, dtype=torch.uint8, device=dev)
    L = lib.load()
    st = torch.cuda.current_stream().cuda_stream
    import ctypes
    tc = (ctypes.c_float * T)(*th)
    maps = {'forward': fwd}
    for kind in ('constant', 'isolated', 'serpentine'):
        maps[kind] = synthetic_maps(kind, B, H, W, max_diff).to(dev)
    arms = {}
    for name, dm, lr, gt in (('forward', fwd, None, None), ('forward_lr', fwd, lr_mask, None),
                             ('forward_gt', fwd, None, disp_gt), ('forward_lr_gt', fwd, lr_mask, disp_gt),
                             ('constant', maps['constant'], None, None), ('isolated', maps['isolated'], None, None),
                             ('serpentine', maps['serpentine'], None, None)):
        def call(dm=dm, lr=lr, gt=gt):                  # ops.speckle_filter's call, without its Python checks
            lib.check(L.s3d_speckle_filter(dm.data_ptr(), B, H, W, None if lr is None else lr.data_ptr(), max_size, max_diff,
                                           None if gt is None else gt.data_ptr(), tc, T, max_gt, mask.data_ptr(),
                                           stats.data_ptr(), ws.data_ptr(), nb, st), 's3d_speckle_filter')
        arms[name] = call
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    for fn in arms.values():
        for _ in range(3):
            fn()
    k = flushed_alternating(arms, flush, args.reps * 5)
    res['kernels'] = {'shape': 'B=%d, %dx%d (%d maps), max_size %d, max_diff %g, T = %d, max_gt %g; forward maps: default '
                               'Stereo2Voxel, %s, LR_THRESH %g' % (B, H, W, 2 * B, max_size, max_diff, T, max_gt,
                                                                   cfg.NETWORK.PRECISION, cfg.TEST.LR_THRESH),
                      'flushed_single_calls': args.reps * 5}
    pix = 2 * B * H * W
    for name, fn in arms.items():
        stats.zero_()
        fn()
        s = stats.sum((0, 1)).tolist()
        prof = kernels_device_us(fn, flush, 20)
        res['kernels'][name] = {'events_flushed': summary(k[name]), 'profiler': prof, 'kept_fraction': s[0] / pix,
                                'n_speckles': s[3 + T], 'speckle_pixels': s[4 + T]}
    del flush, ws, maps

    # 2. the graphed forward
    with torch.no_grad():
        f_arms = {'graphed': lambda i: model.graphed(left, right),
                  'graphed_speckle': lambda i: model.graphed(left, right, speckle=True)}
        time_alternating(f_arms, 3, 2)
        f = time_alternating(f_arms, 10, args.reps)
        m_p, m_s = statistics.median(f['graphed']), statistics.median(f['graphed_speckle'])
        res['graphed_forward'] = {'shape': 'Stereo2Voxel default config, %s, B=%d, %dx%d, D=%d, no gt'
                                           % (cfg.NETWORK.PRECISION, B, H, W, D),
                                  'calls_per_sample': 10, 'samples': args.reps,
                                  'graphed': summary(f['graphed']), 'graphed_speckle': summary(f['graphed_speckle']),
                                  'added_ms': m_s - m_p, 'added_pct': 100.0 * (m_s - m_p) / m_p}
        s = model.graphed(left, right, speckle=True)[-1].sum((0, 1)).tolist()
        res['graphed_forward'].update(kept_fraction=s[0] / pix, n_speckles=s[3 + T], speckle_pixels=s[4 + T])
        n0 = lib.launches(); model(left, right); n1 = lib.launches()
        model(left, right, speckle=True); n2 = lib.launches()
    res['launches'] = {'forward': n1 - n0, 'forward_speckle': n2 - n1}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            fh.write(txt + '\n')


if __name__ == '__main__':
    main()
