#!/usr/bin/env python3
"""Cost of the nearest-neighbour distance histograms (s3d_chamfer_eval_hist, s3d_voxel_surface_eval_hist; forward(...,
fscore_curves=True) of both models), in one run:

  1. chamfer_eval_kernel at B = 32, 2048 predicted vs 16384 GT points (the default Stereo2Point shape), without the
     histogram and with K = 128 and K = 1024 edges.  The kernel runs after the Chamfer search inside one C call, so its own
     device time comes from torch.profiler, with L2 overwritten (256 MB write) before every call; the arms alternate over
     three rounds and the median of the rounds' means is reported;
  2. surface_count_kernel at B = 64, n = 32, T = 4 the same way, without the histogram and with K = 128 and 1024, on a noisy
     field (uniform in [0, 1]: many surface points) and on a smooth one (another GT volume as the prediction);
  3. the default graphed forwards with gt, CUDA events, the arms alternating: Stereo2Point model.graphed(left, right, gt)
     against (..., fscore_curves=True), and Stereo2Voxel (..., surface=True) against (..., surface=True,
     fscore_curves=True).

Also records the launches per eager forward with and without the flag, and the GPU name and power limit beside the numbers.

    python scripts/fscore_curves_time.py [--reps 20] [--out profiles/fscore_curves_time.json]
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
from stereo_3d_reconstruction_b200 import lib, models as M, ops    # noqa: E402
from stereo_3d_reconstruction_b200.utils import synthetic          # noqa: E402


def kernel_us(fn, flush, calls, kernel):
    """Mean device time (us) of `kernel` over `calls` calls of fn, each after an L2 flush, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            flush.zero_()
            fn()
        torch.cuda.synchronize()
    ts = [e.device_time_total if hasattr(e, 'device_time_total') else e.cuda_time_total
          for e in prof.events() if e.device_type.name == 'CUDA' and kernel in e.name]
    assert len(ts) == calls, (kernel, len(ts), calls)
    return sum(ts) / len(ts)


def alternating_kernel_us(arms, flush, calls, kernel, rounds=3):
    """arms: {name: fn()} -> {name: {'median_us', 'rounds_us'}}: per round, every arm's mean kernel time in turn."""
    got = {n: [] for n in arms}
    for _ in range(rounds):
        for name, fn in arms.items():
            got[name].append(kernel_us(fn, flush, calls, kernel))
    return {n: {'median_us': statistics.median(v), 'rounds_us': v} for n, v in got.items()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {'gpu': gpu_info()}
    dev = 'cuda'
    cfg = default_cfg.clone()
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)

    # 1. the point kernel
    B, N, Mg = 32, 2048, 16384
    a, b = synthetic.point_clouds(B, N, Mg, seed=8, duplicates=True)
    a, b = a.to(dev), b.to(dev)
    th = M.fscore_thresholds(cfg)
    st = torch.zeros(B, 2, 3 + len(th), dtype=torch.int64, device=dev)
    ws = torch.empty(max(ops.chamfer_workspace_bytes(B, N, Mg), 1), dtype=torch.uint8, device=dev)
    out = tuple(torch.empty(s, dtype=d, device=dev) for s, d in (((B, N), torch.float32), ((B, Mg), torch.float32),
                                                                  ((B, N), torch.int32), ((B, Mg), torch.int32)))
    arms, hists = {}, {}
    for K in (0, 128, 1024):
        e = M.dist_edges(cfg) if K == 128 else (None if K == 0 else [0.128 * k / K for k in range(1, K + 1)])
        h = hists[K] = None if K == 0 else torch.zeros(B, 2, K + 1, dtype=torch.int64, device=dev)
        arms['K=%d' % K if K else 'no_hist'] = (lambda e=e, h=h: ops.chamfer_eval(a, b, th, st, workspace=ws, out=out,
                                                                                  edges=e, hist=h))
    for fn in arms.values():
        fn()
    res['point_kernel'] = {'shape': 'B=%d, N=%d, M=%d, T=%d' % (B, N, Mg, len(th)), 'calls_per_round': args.reps,
                           'l2': 'overwritten before every call'}
    res['point_kernel'].update(alternating_kernel_us(arms, flush, args.reps, 'chamfer_eval_kernel'))
    base = res['point_kernel']['no_hist']['median_us']
    for K in (128, 1024):
        r = res['point_kernel']['K=%d' % K]
        r['added_us'] = r['median_us'] - base
        r['bins_hit_per_row'] = (hists[K] > 0).sum(-1).double().mean().item()

    # 2. the surface count kernel
    B, n, vt = 64, cfg.CONST.N_VOX, list(cfg.TEST.VOXEL_THRESH)
    fth = M.fscore_thresholds(cfg)
    gt = torch.cat([synthetic.gt_volume(1, n, seed=100000 + i) for i in range(B)]).to(dev).reshape(B, -1).to(torch.uint8)
    fields = {'noisy': torch.rand(B, n ** 3, generator=torch.Generator().manual_seed(1)).to(dev),
              'smooth': torch.cat([synthetic.gt_volume(1, n, seed=300000 + i) for i in range(B)]).to(dev)
              .reshape(B, -1).float()}
    sst = torch.zeros(B, len(vt), 2, 3 + len(fth), dtype=torch.int64, device=dev)
    sws = torch.empty(ops.voxel_surface_workspace_bytes(B, len(vt), n), dtype=torch.uint8, device=dev)
    res['surface_kernel'] = {'shape': 'B=%d, n=%d, T=%d, F=%d' % (B, n, len(vt), len(fth)), 'calls_per_round': args.reps,
                             'l2': 'overwritten before every call'}
    for fname, fused in fields.items():
        arms, hists = {}, {}
        for K in (0, 128, 1024):
            e = M.dist_edges(cfg) if K == 128 else (None if K == 0 else [0.128 * k / K for k in range(1, K + 1)])
            h = hists[K] = None if K == 0 else torch.zeros(B, len(vt), 2, K + 1, dtype=torch.int64, device=dev)
            arms['K=%d' % K if K else 'no_hist'] = (
                lambda e=e, h=h, fused=fused: ops.voxel_surface_eval(fused, gt, vt, fth, sst, workspace=sws, edges=e, hist=h))
        for fn in arms.values():
            fn()
        r = alternating_kernel_us(arms, flush, args.reps, 'surface_count_kernel')
        base = r['no_hist']['median_us']
        for K in (128, 1024):
            r['K=%d' % K]['added_pct'] = 100.0 * (r['K=%d' % K]['median_us'] - base) / base
            r['K=%d' % K]['bins_hit_per_row'] = (hists[K] > 0).sum(-1).double().mean().item()
        res['surface_kernel'][fname] = r
    del flush

    # 3. the graphed default forwards
    res['graphed_forward'] = {}
    res['launches'] = {}
    for name in ('Stereo2Point', 'Stereo2Voxel'):
        model = M.build_model(name, cfg, seed=0).cuda().pack()
        Bm, H, W, D = cfg.CONST.BATCH_SIZE, cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.NETWORK.MAX_DISP
        left, right, _ = synthetic.stereo_pair(Bm, H, W, 2 * D, seed=1)
        left, right = left.to(dev), right.to(dev)
        if name == 'Stereo2Point':
            g = synthetic.point_clouds(Bm, 1, cfg.CONST.N_GT_POINTS, seed=51)[1].to(dev)
            kw = {}
        else:
            g = synthetic.gt_volume(Bm, n, seed=51).to(dev)
            kw = dict(surface=True)
        with torch.no_grad():
            arms = {'graphed': lambda i: model.graphed(left, right, g, **kw),
                    'graphed_fscore_curves': lambda i: model.graphed(left, right, g, fscore_curves=True, **kw)}
            time_alternating(arms, 3, 2)
            f = time_alternating(arms, 10, args.reps)
            m0, m1 = statistics.median(f['graphed']), statistics.median(f['graphed_fscore_curves'])
            res['graphed_forward'][name] = {
                'shape': '%s default config, %s, B=%d, %dx%d, D=%d, with gt%s, K=%d'
                         % (name, cfg.NETWORK.PRECISION, Bm, H, W, D, ', surface' if kw else '', cfg.TEST.DIST_BINS),
                'calls_per_sample': 10, 'samples': args.reps, 'graphed': summary(f['graphed']),
                'graphed_fscore_curves': summary(f['graphed_fscore_curves']),
                'added_ms': m1 - m0, 'added_pct': 100.0 * (m1 - m0) / m0}
            n0 = lib.launches(); model(left, right, g, **kw); n1 = lib.launches()
            model(left, right, g, fscore_curves=True, **kw); n2 = lib.launches()
        res['launches'][name] = {'forward_gt': n1 - n0, 'forward_gt_fscore_curves': n2 - n1}
        del model
        torch.cuda.empty_cache()
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            fh.write(txt + '\n')


if __name__ == '__main__':
    main()
