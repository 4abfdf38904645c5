#!/usr/bin/env python3
"""Cost of the threshold-free occupancy evaluation (s3d_occupancy_curves, Stereo2Voxel forward(left, right, gt,
curves=True)), in one run, CUDA events, the arms alternating:

  1. the kernel alone at B = 64, n = 32, K = TEST.CURVE_BINS, through the C entry point into preallocated buffers, on a spread
     field (uniform in [0, 1]: every bin is hit) and on a field where every voxel is in one bin (0.5, as the untrained
     synthetic-weight predictions nearly are).  L2 is overwritten (256 MB write) before every single timed call: CUDA events
     around each call, and torch.profiler's device time of the kernel alone with the same flush before each call; a second
     measurement times 20 back-to-back calls (L2 warm, launch gaps hidden);
  2. the default Stereo2Voxel forward with gt replayed from its CUDA graph at B = 64, model.graphed(left, right, gt) against
     model.graphed(left, right, gt, curves=True).

Also records the launches per eager forward with and without the flag, and the GPU name and power limit beside the numbers.

    python scripts/curves_time.py [--reps 20] [--out profiles/curves_time.json]
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
from stereo_3d_reconstruction_b200 import lib, models as M         # noqa: E402
from stereo_3d_reconstruction_b200.utils import synthetic          # noqa: E402


def kernel_device_ms(fn, flush, calls):
    """Mean device time per call of occupancy_curves_kernel over `calls` calls of fn, each after an L2 flush, from
    torch.profiler (a run of its own)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            flush.zero_()
            fn()
        torch.cuda.synchronize()
    ts = [e.device_time_total if hasattr(e, 'device_time_total') else e.cuda_time_total
          for e in prof.events() if e.device_type.name == 'CUDA' and 'occupancy_curves_kernel' in e.name]
    return {'launches_seen': len(ts), 'mean_us': sum(ts) / len(ts) if ts else None,
            'max_us': max(ts) if ts else None, 'min_us': min(ts) if ts else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {'gpu': gpu_info()}
    dev = 'cuda'
    cfg = default_cfg.clone()
    B, n, K = cfg.CONST.BATCH_SIZE, cfg.CONST.N_VOX, M.curve_bins(cfg)
    nvox = n ** 3

    # 1. the kernel alone
    gt = torch.cat([synthetic.gt_volume(1, n, seed=100000 + i) for i in range(B)]).to(dev).reshape(B, -1).to(torch.uint8)
    fields = {'spread': torch.rand(B, nvox, generator=torch.Generator().manual_seed(1)).to(dev),
              'one_bin': torch.full((B, nvox), 0.5, device=dev)}
    hist = torch.empty(B, 3, K, dtype=torch.int64, device=dev)
    loss = torch.empty(B, 2, dtype=torch.int64, device=dev)
    L = lib.load()
    st = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    res['kernel'] = {'shape': 'B=%d, n=%d (nvox=%d), K=%d' % (B, n, nvox, K),
                     'input_bytes': B * nvox * 5, 'output_bytes': (hist.numel() + loss.numel()) * 8}
    for name, vol in fields.items():
        def curves():                               # ops.occupancy_curves's call, without its Python checks
            lib.check(L.s3d_occupancy_curves(vol.data_ptr(), gt.data_ptr(), B, nvox, K, hist.data_ptr(), loss.data_ptr(), st),
                      's3d_occupancy_curves')
        for _ in range(3):
            curves()
        k = flushed_alternating({name: curves}, flush, args.reps * 5)
        loop = time_alternating({name: lambda i: curves()}, 20, args.reps)
        prof = kernel_device_ms(curves, flush, args.reps)
        res['kernel'][name] = {'flushed_single_calls': args.reps * 5, 'loop_calls_per_sample': 20, 'loop_samples': args.reps,
                               'flushed_events': summary(k[name]), 'loop': summary(loop[name]),
                               'profiler_flushed': prof,
                               'bins_hit_per_sample': (hist[:, :2].sum(1) > 0).sum(1).double().mean().item()}
    del flush

    # 2. the graphed forward with gt
    model = M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()
    H, W, D = cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.NETWORK.MAX_DISP
    left, right, _ = synthetic.stereo_pair(B, H, W, 2 * D, seed=1)
    left, right = left.to(dev), right.to(dev)
    gtv = synthetic.gt_volume(B, n, seed=51).to(dev)
    with torch.no_grad():
        arms = {'graphed_gt': lambda i: model.graphed(left, right, gtv),
                'graphed_gt_curves': lambda i: model.graphed(left, right, gtv, curves=True)}
        time_alternating(arms, 3, 2)
        f = time_alternating(arms, 10, args.reps)
        m_p, m_s = statistics.median(f['graphed_gt']), statistics.median(f['graphed_gt_curves'])
        res['graphed_forward'] = {'shape': 'Stereo2Voxel default config, %s, B=%d, %dx%d, D=%d, with gt, K=%d'
                                           % (cfg.NETWORK.PRECISION, B, H, W, D, K),
                                  'calls_per_sample': 10, 'samples': args.reps,
                                  'graphed_gt': summary(f['graphed_gt']), 'graphed_gt_curves': summary(f['graphed_gt_curves']),
                                  'added_ms': m_s - m_p, 'added_pct': 100.0 * (m_s - m_p) / m_p}
        h = model.graphed(left, right, gtv, curves=True)[-2]
        res['graphed_forward']['bins_hit_per_sample'] = (h[:, :2].sum(1) > 0).sum(1).double().mean().item()
        n0 = lib.launches(); model(left, right, gtv); n1 = lib.launches()
        model(left, right, gtv, curves=True); n2 = lib.launches()
    res['launches'] = {'forward_gt': n1 - n0, 'forward_gt_curves': n2 - n1}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            fh.write(txt + '\n')


if __name__ == '__main__':
    main()
