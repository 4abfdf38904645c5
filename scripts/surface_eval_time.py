#!/usr/bin/env python3
"""Cost of the voxel-surface evaluation (s3d_voxel_surface_eval, Stereo2Voxel forward(left, right, gt, surface=True)), in
one run, CUDA events, the arms alternating:

  1. the two kernels alone at B = 64, n = 32, the default TEST.VOXEL_THRESH (T = 4) and TEST.FSCORE_THRESH, on the synthetic
     GT volumes and a prediction derived from them, called through the C entry point into preallocated buffers.  L2 is
     overwritten (256 MB write) before every single timed call; a second measurement times 20 back-to-back calls (L2 warm,
     launch gaps hidden), and torch.profiler gives the device time of each kernel;
  2. the default Stereo2Voxel forward replayed from its CUDA graph at B = 64, model.graphed(left, right, gt) against
     model.graphed(left, right, gt, surface=True).

Also records the launches per eager forward (lib.launches()) with and without surface, and the GPU name and power limit
beside the numbers.

    python scripts/surface_eval_time.py [--reps 20] [--out profiles/surface_eval_time.json]
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


def kernels_device_ms(fn, calls):
    """Mean device time per call of each surface kernel over `calls` calls of fn, from torch.profiler (a run of its own)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for k in ('surface_plane_kernel', 'surface_count_kernel'):
        ts = [e.device_time_total if hasattr(e, 'device_time_total') else e.cuda_time_total
              for e in prof.events() if e.device_type.name == 'CUDA' and k in e.name]
        out[k] = {'launches_seen': len(ts), 'mean_ms': sum(ts) / len(ts) / 1e3 if ts else None}
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
    B, n = cfg.CONST.BATCH_SIZE, cfg.CONST.N_VOX
    vth, fth = list(cfg.TEST.VOXEL_THRESH), M.fscore_thresholds(cfg)
    T, F = len(vth), len(fth)

    # 1. the kernels alone
    gt = torch.cat([synthetic.gt_volume(1, n, seed=100000 + i) for i in range(B)]).to(dev)
    noise = torch.rand(B, n, n, n, generator=torch.Generator().manual_seed(1)).to(dev)
    fused = (0.6 * gt.float() + 0.5 * noise).clamp_(0, 1).contiguous()
    nb = ops.voxel_surface_workspace_bytes(B, T, n)
    ws = torch.empty(nb, dtype=torch.uint8, device=dev)
    stats = torch.zeros(B, T, 2, 3 + F, dtype=torch.int64, device=dev)
    L = lib.load()
    st = torch.cuda.current_stream().cuda_stream
    th = (ctypes.c_float * T)(*vth)
    kb = (ctypes.c_int * max(F, 1))(*[ops.voxel_kbound(t, n) for t in fth])

    def surf():                                     # ops.voxel_surface_eval's call, without its Python checks
        lib.check(L.s3d_voxel_surface_eval(fused.data_ptr(), gt.data_ptr(), B, n, th, T, kb, F, stats.data_ptr(),
                                           ws.data_ptr(), nb, st), 's3d_voxel_surface_eval')
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    for _ in range(3):
        surf()
    k = flushed_alternating({'surface_eval': surf}, flush, args.reps * 5)
    loop = time_alternating({'surface_eval': lambda i: surf()}, 20, args.reps)
    stats.zero_()
    surf()
    c = stats.cpu()
    res['kernels'] = {'shape': 'B=%d, n=%d, T=%d %s, F=%d %s' % (B, n, T, vth, F, fth), 'workspace_bytes': nb,
                      'flushed_single_calls': args.reps * 5, 'loop_calls_per_sample': 20, 'loop_samples': args.reps,
                      'flushed': summary(k['surface_eval']), 'loop': summary(loop['surface_eval']),
                      'profiler': kernels_device_ms(surf, 20),
                      'mean_points_per_sample_and_direction': (c[:, :, :, 0].double().mean((0, 1))).tolist()}
    del ws, flush

    # 2. the graphed forward
    model = M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()
    H, W, D = cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.NETWORK.MAX_DISP
    left, right, _ = synthetic.stereo_pair(B, H, W, 2 * D, seed=1)
    left, right = left.to(dev), right.to(dev)
    with torch.no_grad():
        arms = {'graphed_gt': lambda i: model.graphed(left, right, gt),
                'graphed_gt_surface': lambda i: model.graphed(left, right, gt, surface=True)}
        time_alternating(arms, 3, 2)
        f = time_alternating(arms, 10, args.reps)
        m_p, m_s = statistics.median(f['graphed_gt']), statistics.median(f['graphed_gt_surface'])
        res['graphed_forward'] = {'shape': 'Stereo2Voxel default config, %s, B=%d, %dx%d, D=%d, with gt'
                                           % (cfg.NETWORK.PRECISION, B, H, W, D),
                                  'calls_per_sample': 10, 'samples': args.reps,
                                  'graphed_gt': summary(f['graphed_gt']), 'graphed_gt_surface': summary(f['graphed_gt_surface']),
                                  'added_ms': m_s - m_p, 'added_pct': 100.0 * (m_s - m_p) / m_p}
        out = model.graphed(left, right, gt, surface=True)
        res['graphed_forward']['surf_stats_sum'] = out[-1].sum(0).tolist()
        n0 = lib.launches(); model(left, right, gt); n1 = lib.launches()
        model(left, right, gt, surface=True); n2 = lib.launches()
    res['launches'] = {'forward_gt': n1 - n0, 'forward_gt_surface': n2 - n1}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            fh.write(txt + '\n')


if __name__ == '__main__':
    main()
