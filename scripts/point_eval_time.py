#!/usr/bin/env python3
"""Cost of the point-cloud evaluation (s3d_chamfer_eval, Stereo2Point forward(left, right, gt)), in one run, CUDA events,
the arms alternating:

  1. the Chamfer search alone (s3d_chamfer_forward_ws, what ops.chamfer_forward calls) against the search + metric
     counters (s3d_chamfer_eval, what ops.chamfer_eval calls) at B = 32, 2048 predicted vs 16384 GT points, the default
     TEST.FSCORE_THRESH.  Both arms call the C entry points directly, into the same preallocated buffers.  As in bench.py,
     L2 is flushed (256 MB write) before every single timed call; a second pair of arms times 50 back-to-back calls each
     (L2 warm, launch gaps hidden), and torch.profiler gives the device time of chamfer_eval_kernel itself;
  2. the default Stereo2Point forward replayed from its CUDA graph at B = 32, model.graphed(left, right) against
     model.graphed(left, right, gt).

Also records the launches per eager forward (lib.launches()) with and without gt, and the GPU name and power limit beside
the numbers.

    python scripts/point_eval_time.py [--reps 20] [--out profiles/point_eval_time.json]
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
from stereo_3d_reconstruction_b200 import lib, models as M, ops    # noqa: E402
from stereo_3d_reconstruction_b200.utils import synthetic          # noqa: E402


def flushed_alternating(arms, flush, reps):
    """arms: {name: fn()}; per rep, every arm once: L2 flush, then CUDA events around the one call -> {name: [ms]}."""
    ev = {n: [] for n in arms}
    for _ in range(reps):
        for name, fn in arms.items():
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            b.synchronize()
            ev[name].append(a.elapsed_time(b))
    return ev


def eval_kernel_device_ms(fn, calls):
    """Mean device time of chamfer_eval_kernel over `calls` calls of fn, from torch.profiler (a run of its own)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    ts = [e.device_time_total if hasattr(e, 'device_time_total') else e.cuda_time_total
          for e in prof.events() if e.device_type.name == 'CUDA' and 'chamfer_eval_kernel' in e.name]
    return {'launches_seen': len(ts), 'mean_ms': sum(ts) / len(ts) / 1e3 if ts else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=20)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    res = {'gpu': gpu_info()}
    dev = 'cuda'
    cfg = default_cfg.clone()
    B, N, Mg = 32, cfg.CONST.N_POINTS, cfg.CONST.N_GT_POINTS
    th = M.fscore_thresholds(cfg)

    # 1. the search alone against search + counters
    pts = (torch.rand(B, N, 3, generator=torch.Generator().manual_seed(0)) - 0.5).to(dev)
    gt = synthetic.point_clouds(B, 1, Mg, seed=3)[1].to(dev)
    nb = ops.chamfer_workspace_bytes(B, N, Mg)
    ws = torch.empty(max(nb, 1), dtype=torch.uint8, device=dev)
    bufs = (torch.empty(B, N, device=dev), torch.empty(B, Mg, device=dev), torch.empty(B, N, dtype=torch.int32, device=dev),
            torch.empty(B, Mg, dtype=torch.int32, device=dev))
    stats = torch.zeros(B, 2, 3 + len(th), dtype=torch.int64, device=dev)
    L = lib.load()
    st = torch.cuda.current_stream().cuda_stream
    d1, d2, i1, i2 = (t.data_ptr() for t in bufs)

    def search():                                   # the entry point chamfer_forward calls, into the same buffers
        lib.check(L.s3d_chamfer_forward_ws(pts.data_ptr(), gt.data_ptr(), d1, i1, d2, i2, B, N, Mg, ws.data_ptr() if nb else None,
                                           nb, st), 's3d_chamfer_forward_ws')

    tau = (ctypes.c_float * len(th))(*th)

    def search_eval():                              # ops.chamfer_eval's call, without its Python checks (as search())
        lib.check(L.s3d_chamfer_eval(pts.data_ptr(), gt.data_ptr(), d1, i1, d2, i2, B, N, Mg, tau, len(th), stats.data_ptr(),
                                     ws.data_ptr() if nb else None, nb, st), 's3d_chamfer_eval')
    arms = {'chamfer_forward': search, 'chamfer_eval': search_eval}
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    for fn in arms.values():                                        # warm-up
        for _ in range(3):
            fn()
    k = flushed_alternating(arms, flush, args.reps * 5)
    loop = time_alternating({n: (lambda i, f=f: f()) for n, f in arms.items()}, 50, args.reps)
    res['chamfer'] = {'shape': 'B=%d, N=%d predicted, M=%d GT points, T=%d (%s)' % (B, N, Mg, len(th), th),
                      'workspace_bytes': nb, 'search_path': 'one-pass (chamfer_sym_kernel)' if nb else 'one search per direction',
                      'flushed_single_calls': args.reps * 5, 'loop_calls_per_sample': 50, 'loop_samples': args.reps}
    for n in arms:
        res['chamfer'][n + '_flushed'] = summary(k[n])
        res['chamfer'][n + '_loop'] = summary(loop[n])
    res['chamfer']['added_ms_flushed'] = statistics.median(k['chamfer_eval']) - statistics.median(k['chamfer_forward'])
    res['chamfer']['added_ms_loop'] = statistics.median(loop['chamfer_eval']) - statistics.median(loop['chamfer_forward'])
    res['chamfer']['eval_kernel_profiler'] = eval_kernel_device_ms(search_eval, 20)
    res['chamfer']['eval_kernel_bytes_read'] = B * (N + Mg) * 4
    del ws, bufs, flush

    # 2. the graphed forward
    model = M.build_model('Stereo2Point', cfg, seed=0).cuda().pack()
    H, W, D = cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.NETWORK.MAX_DISP
    left, right, _ = synthetic.stereo_pair(B, H, W, 2 * D, seed=1)
    left, right = left.to(dev), right.to(dev)
    with torch.no_grad():
        arms = {'graphed': lambda i: model.graphed(left, right),
                'graphed_gt': lambda i: model.graphed(left, right, gt)}
        time_alternating(arms, 3, 2)
        f = time_alternating(arms, 10, args.reps)
        m_p, m_g = statistics.median(f['graphed']), statistics.median(f['graphed_gt'])
        res['graphed_forward'] = {'shape': 'Stereo2Point default config, %s, B=%d, %dx%d, D=%d, %d vs %d points'
                                           % (cfg.NETWORK.PRECISION, B, H, W, D, N, Mg),
                                  'calls_per_sample': 10, 'samples': args.reps,
                                  'graphed': summary(f['graphed']), 'graphed_gt': summary(f['graphed_gt']),
                                  'added_ms': m_g - m_p, 'added_pct': 100.0 * (m_g - m_p) / m_p}
        out = model.graphed(left, right, gt)
        s = out[3].sum(0)
        res['graphed_forward']['point_stats_sum'] = s.tolist()
        n0 = lib.launches(); model(left, right); n1 = lib.launches()
        model(left, right, gt); n2 = lib.launches()
    res['launches'] = {'forward': n1 - n0, 'forward_gt': n2 - n1}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            fh.write(txt + '\n')


if __name__ == '__main__':
    main()
