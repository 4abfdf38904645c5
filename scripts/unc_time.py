#!/usr/bin/env python3
"""Cost of the disparity uncertainty (disp_std_q set, forward(..., uncertainty=True)), in one run, CUDA events, the
arms alternating, at B = 64, 256 x 256, D = 32 (1/4-res 64 x 64, 2B = 128 images):

  1. each soft-argmin kernel without and with the standard deviation: the bf16 chain (s3d_conv_cls_soft_argmin: cls_a +
     classifier + partials_soft_argmin_kernel), cls_fused_kernel, tap_gather_soft_argmin_kernel, corr_tc_kernel and the SIMT
     corr_soft_argmin_kernel (fp32 features).  Their inputs are 2.1 GB volumes, or four rotated feature sets of more than the
     126 MB L2 for the corr kernels;
  2. the upsample kernel plain (s3d_upsample_disp), with the standard deviation (s3d_upsample_disp_eval) and with it plus GT
     evaluation and the LR check, four rotated buffer sets;
  3. the default Stereo2Voxel forward replayed from its CUDA graph, with and without uncertainty=True.

Records the GPU name and power limit beside the numbers, and the launches per forward with and without the flag.

    python scripts/unc_time.py [--reps 20] [--out profiles/unc_time.json]
"""
import argparse
import json
import os
import statistics
import sys

import torch
import torch.nn as nn

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, HERE)

from config import cfg as default_cfg                              # noqa: E402
from disp_eval_time import gpu_info, summary, time_alternating     # noqa: E402
from stereo_3d_reconstruction_b200 import lib, models as M, ops    # noqa: E402
from stereo_3d_reconstruction_b200.layers import PackedConv        # noqa: E402
from stereo_3d_reconstruction_b200.utils import synthetic          # noqa: E402


def pair(arms_plain, arms_std, calls, reps):
    """Time {name: fn(k)} plain / std arms alternating -> {name: {plain, std, added_ms, added_pct}}."""
    arms = {}
    for n in arms_plain:
        arms[n] = arms_plain[n]
        arms[n + '_std'] = arms_std[n]
    time_alternating(arms, 2, 2)                                    # warm-up
    t = time_alternating(arms, calls, reps)
    out = {}
    for n in arms_plain:
        a, b = statistics.median(t[n]), statistics.median(t[n + '_std'])
        out[n] = {'plain': summary(t[n]), 'std': summary(t[n + '_std']), 'added_ms': b - a, 'added_pct': 100.0 * (b - a) / a}
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
    B, H, W, D = 64, cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.NETWORK.MAX_DISP
    h, w, N = H // 4, W // 4, 2 * B
    g = torch.Generator(device=dev).manual_seed(0)
    sq = [torch.empty(N, h, w, device=dev) for _ in range(4)]
    dq = [torch.empty(N, h, w, device=dev) for _ in range(4)]

    # 1. the soft-argmin kernels
    with torch.no_grad():
        conv = nn.Conv3d(64, 64, 3, 1, 1, bias=True)
        conv.weight.mul_(0.5)
        pc = PackedConv.from_conv(conv, None, lib.ACT_RELU, lib.DTYPE_BF16, dev)
    x = torch.randn(N, D, h, w, 64, device=dev, generator=g).to(torch.bfloat16)        # 2.1 GB
    w_taps = (torch.randn(32, 64, device=dev, generator=g) * 0.1).to(torch.bfloat16)
    w_taps[27:] = 0
    ws = torch.empty(ops.conv_cls_workspace_bytes(N, D, h, w), dtype=torch.uint8, device=dev)
    vol = {
        'conv_cls_chain': (lambda k, s: ops.conv_cls_soft_argmin(pc, x, w_taps, -1.0, out=dq[k % 4], workspace=ws, std_out=s)),
        'cls_fused': (lambda k, s: ops.cls_soft_argmin(x, w_taps, -1.0, out=dq[k % 4], std_out=s)),
    }
    k_vol = pair({n: (lambda k, f=f: f(k, None)) for n, f in vol.items()},
                 {n: (lambda k, f=f: f(k, sq[k % 4])) for n, f in vol.items()}, 10, args.reps)
    del x
    taps = torch.randn(N, D, h, 32, w, device=dev, generator=g)                         # 2.1 GB
    k_tap = pair({'tap_gather': lambda k: ops.tap_gather_soft_argmin(taps, -1.0, out=dq[k % 4])},
                 {'tap_gather': lambda k: ops.tap_gather_soft_argmin(taps, -1.0, out=dq[k % 4], std_out=sq[k % 4])}, 10, args.reps)
    del taps
    fb = [torch.randn(N, 1, h, w, 32, device=dev, generator=g).to(torch.bfloat16) for _ in range(4)]   # 4 x 33.5 MB
    ff = [torch.randn(N, 1, h, w, 32, device=dev, generator=g) for _ in range(4)]                       # 4 x 67 MB
    k_corr = pair({'corr_tc': lambda k: ops.corr_soft_argmin(fb[k % 4], B, D, out=dq[k % 4]),
                   'corr_simt_fp32': lambda k: ops.corr_soft_argmin(ff[k % 4], B, D, out=dq[k % 4])},
                  {'corr_tc': lambda k: ops.corr_soft_argmin(fb[k % 4], B, D, out=dq[k % 4], std_out=sq[k % 4]),
                   'corr_simt_fp32': lambda k: ops.corr_soft_argmin(ff[k % 4], B, D, out=dq[k % 4], std_out=sq[k % 4])},
                  50, args.reps)
    del fb, ff
    res['soft_argmin'] = dict(k_vol, **k_tap, **k_corr)
    res['soft_argmin']['shape'] = '2B=%d images, %dx%d, D=%d; volumes 2.1 GB, corr features 4 rotated sets' % (N, h, w, D)

    # 2. the upsample kernel
    th, ut = list(cfg.TEST.DISP_THRESH), list(cfg.TEST.UNC_THRESH)
    sets = []
    for s in range(4):
        d = torch.randint(0, 2 * D, (B, H))
        sets.append(dict(q=torch.rand(N, h, w, device=dev, generator=g) * (D - 1), s=torch.rand(N, h, w, device=dev, generator=g),
                         out=torch.empty(N, H, W, device=dev), sd=torch.empty(B, 2, H, W, device=dev),
                         gt=synthetic.disparity_gt(d, H, W).to(dev),
                         st=torch.zeros(B, 2, 2 + len(th), dtype=torch.int64, device=dev),
                         mask=torch.empty(B, 2, H, W, dtype=torch.uint8, device=dev),
                         ls=torch.zeros(B, 2, 3 + len(th), dtype=torch.int64, device=dev),
                         us=torch.zeros(B, 2, len(ut), 3 + len(th), dtype=torch.int64, device=dev),
                         us0=torch.zeros(B, 2, len(ut), 3, dtype=torch.int64, device=dev)))

    def S(k):
        return sets[k % 4]
    arms = {
        'plain': lambda k: ops.upsample_disp(S(k)['q'], H, W, 4.0, out=S(k)['out']),
        'std': lambda k: ops.upsample_disp_eval(S(k)['q'], H, W, 4.0, std_q=S(k)['s'], unc_thresh=ut, unc_stats=S(k)['us0'],
                                                std_out=S(k)['sd'], out=S(k)['out']),
        'std_eval_lr': lambda k: ops.upsample_disp_eval(S(k)['q'], H, W, 4.0, S(k)['gt'], th, 4.0 * D, S(k)['st'],
                                                        lr_thresh=cfg.TEST.LR_THRESH, mask=S(k)['mask'], lr_stats=S(k)['ls'],
                                                        std_q=S(k)['s'], unc_thresh=ut, unc_stats=S(k)['us'],
                                                        std_out=S(k)['sd'], out=S(k)['out']),
    }
    time_alternating(arms, 8, 3)
    t = time_alternating(arms, 200, args.reps)
    res['upsample'] = {'shape': '2B=%d images %dx%d from %dx%d, K=%d, T=%d' % (N, H, W, h, w, len(ut), len(th)),
                       'buffer_sets': 4, 'calls_per_sample': 200, 'samples': args.reps}
    for n in arms:
        res['upsample'][n] = summary(t[n])
    res['upsample']['std_minus_plain_ms'] = statistics.median(t['std']) - statistics.median(t['plain'])
    del sets

    # 3. the graphed forward
    model = M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()
    left, right, _ = synthetic.stereo_pair(B, H, W, 2 * D, seed=1)
    left, right = left.to(dev), right.to(dev)
    gt = synthetic.gt_volume(B, seed=2).to(dev)
    with torch.no_grad():
        arms = {'graphed': lambda k: model.graphed(left, right, gt),
                'graphed_uncertainty': lambda k: model.graphed(left, right, gt, uncertainty=True)}
        time_alternating(arms, 3, 2)
        f = time_alternating(arms, 10, args.reps)
        m_p, m_u = statistics.median(f['graphed']), statistics.median(f['graphed_uncertainty'])
        res['graphed_forward'] = {'shape': 'Stereo2Voxel default config, %s, B=%d, %dx%d, D=%d' % (cfg.NETWORK.PRECISION, B, H, W, D),
                                  'calls_per_sample': 10, 'samples': args.reps,
                                  'graphed': summary(f['graphed']), 'graphed_uncertainty': summary(f['graphed_uncertainty']),
                                  'added_ms': m_u - m_p, 'added_pct': 100.0 * (m_u - m_p) / m_p}
        out = model.graphed(left, right, gt, uncertainty=True)
        res['graphed_forward']['disp_std_median_px'] = float(out[-2].median().item())
        n0 = lib.launches(); model(left, right, gt); n1 = lib.launches()
        model(left, right, gt, uncertainty=True); n2 = lib.launches()
    res['launches'] = {'forward': n1 - n0, 'forward_uncertainty': n2 - n1}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            fh.write(txt + '\n')


if __name__ == '__main__':
    main()
