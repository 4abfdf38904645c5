#!/usr/bin/env python3
"""Cost of the WLS filter (s3d_disp_wls, forward(..., wls=True)), in one run:

  1. the six kernels alone at B = 64, 256 x 256, through the C entry point into preallocated buffers, on the disparity maps
     of one default Stereo2Voxel forward of the synthetic pairs (lr_check=True, speckle=True, with the GT disparity), with no
     mask and with the speckle mask, for uint8 HWC and fp32 NCHW guides.  L2 is overwritten (256 MB write) before every call:
     CUDA events around each single call (the arms alternating), and torch.profiler device times of each kernel in a run of
     their own, flushed the same way;
  2. the default Stereo2Voxel forward replayed from its CUDA graph at B = 64, model.graphed(left, right) against
     model.graphed(left, right, wls=True), alternating, with the launches per eager forward of each.

Also records the confident and finite fractions of every arm, and the GPU name and power limit beside the numbers.

    python scripts/wls_time.py [--reps 20] [--out profiles/wls_time.json]
"""
import argparse
import ctypes
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

_KERNELS = ('wls_row_kernel', 'wls_col_kernel')


def kernels_device_us(fn, flush, calls):
    """Mean device time per call of the row and column kernels (three launches each per call) over `calls` calls of fn, each
    after an L2 flush (torch.profiler)."""
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
        out[k] = {'launches_seen': len(ts), 'per_call_us': sum(ts) / calls if ts else None}
    if all(out[k]['per_call_us'] is not None for k in _KERNELS):
        out['all_us'] = sum(out[k]['per_call_us'] for k in _KERNELS)
    return out


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
    lam, sigma = M.wls_params(cfg)
    th = [float(t) for t in cfg.TEST.DISP_THRESH]
    T, max_gt = len(th), 4.0 * D
    model = M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()
    left, right, dg = synthetic.stereo_pair(B, H, W, 2 * D, seed=1)
    left, right = left.to(dev).contiguous(), right.to(dev).contiguous()
    disp_gt = synthetic.disparity_gt(dg, H, W).to(dev).contiguous()
    imgs = {'u8': [(x.permute(0, 2, 3, 1) * 255).round().clamp(0, 255).to(torch.uint8).contiguous() for x in (left, right)],
            'f32': [left, right]}

    # 1. the kernels alone
    with torch.no_grad():
        o = dict(zip(M.Stereo2Voxel.output_names(disp_gt=True, lr_check=True, speckle=True),
                     model(left, right, disp_gt=disp_gt, lr_check=True, speckle=True)))
        fwd = torch.cat([o['disp_left'][:, 0], o['disp_right'][:, 0]]).contiguous()
        spk = o['speckle_mask'].clone()
    lut = torch.from_numpy(ops.wls_weight_lut(sigma)).to(dev)
    out = torch.empty(2 * B, H, W, device=dev)
    stats = torch.zeros(B, 2, 4 + T, dtype=torch.int64, device=dev)
    nb = ops.disp_wls_workspace_bytes(B, H, W)
    ws = torch.empty(nb, dtype=torch.uint8, device=dev)
    L = lib.load()
    st = torch.cuda.current_stream().cuda_stream
    tc = (ctypes.c_float * T)(*th)
    arms = {}
    for g in ('u8', 'f32'):
        for mname, mask in (('no_mask', None), ('speckle_mask', spk)):
            def call(g=g, mask=mask):                   # ops.disp_wls's call, without its Python checks
                lib.check(L.s3d_disp_wls(fwd.data_ptr(), B, H, W, imgs[g][0].data_ptr(), imgs[g][1].data_ptr(),
                                         int(g == 'u8'), None if mask is None else mask.data_ptr(), lut.data_ptr(), lam,
                                         disp_gt.data_ptr(), tc, T, max_gt, out.data_ptr(), stats.data_ptr(), ws.data_ptr(),
                                         nb, st), 's3d_disp_wls')
            arms['%s_%s' % (g, mname)] = call
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    for fn in arms.values():
        for _ in range(3):
            fn()
    k = flushed_alternating(arms, flush, args.reps * 5)
    res['kernels'] = {'shape': 'B=%d, %dx%d (%d maps), lambda %g, sigma %g, T = %d, max_gt %g; forward maps: default '
                               'Stereo2Voxel, %s, LR_THRESH %g, speckle (%d, %g)'
                               % (B, H, W, 2 * B, lam, sigma, T, max_gt, cfg.NETWORK.PRECISION, cfg.TEST.LR_THRESH,
                                  *M.speckle_params(cfg)),
                      'flushed_single_calls': args.reps * 5}
    pix = 2 * B * H * W
    for name, fn in arms.items():
        stats.zero_()
        fn()
        s = stats.sum((0, 1)).tolist()
        prof = kernels_device_us(fn, flush, 20)
        res['kernels'][name] = {'events_flushed': summary(k[name]), 'profiler': prof, 'confident_fraction': s[3 + T] / pix,
                                'finite_fraction': s[0] / pix}
    del flush, ws

    # 2. the graphed forward
    with torch.no_grad():
        f_arms = {'graphed': lambda i: model.graphed(left, right),
                  'graphed_wls': lambda i: model.graphed(left, right, wls=True)}
        time_alternating(f_arms, 3, 2)
        f = time_alternating(f_arms, 10, args.reps)
        m_p, m_w = statistics.median(f['graphed']), statistics.median(f['graphed_wls'])
        res['graphed_forward'] = {'shape': 'Stereo2Voxel default config, %s, B=%d, %dx%d, D=%d, no gt'
                                           % (cfg.NETWORK.PRECISION, B, H, W, D),
                                  'calls_per_sample': 10, 'samples': args.reps,
                                  'graphed': summary(f['graphed']), 'graphed_wls': summary(f['graphed_wls']),
                                  'added_ms': m_w - m_p, 'added_pct': 100.0 * (m_w - m_p) / m_p}
        n0 = lib.launches(); model(left, right); n1 = lib.launches()
        model(left, right, wls=True); n2 = lib.launches()
    res['launches'] = {'forward': n1 - n0, 'forward_wls': n2 - n1}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            fh.write(txt + '\n')


if __name__ == '__main__':
    main()
