#!/usr/bin/env python3
"""Gain of the constant-region skip of the aggregation layers (include/s3d.h dz_nref; A/B knob no_dz_skip), CUDA events,
the two arms alternating:

  the default bf16 Stereo2Voxel forward at B = 64, 256 x 256, D = 32, eager (so that each of dres0b / dres1a / dres1b is
  bracketed by its own events).  Four input sets are rotated (4 x 50 MB of fp32 images, more than the 126 MB L2).  Each
  rep runs `--steps` resident forwards per arm; the step time is the events around a whole forward, the layer times the
  events around the layer's launch.

Also records the input planes the plane-scatter kernel marched per layer (executed MMA planes, the library's dz_planes
counter) against the algorithmic count (2B x ceil(h/32) x ceil(w/8) columns x D planes), and the GPU name and power limit
beside the numbers.

    python scripts/dz_skip_time.py [--reps 5] [--steps 20] [--out profiles/dz_skip_time.json]
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
from disp_eval_time import gpu_info                                # noqa: E402
from stereo_3d_reconstruction_b200 import layers, lib, models as M   # noqa: E402
from stereo_3d_reconstruction_b200.utils import synthetic          # noqa: E402

LAYERS = ('dres0b', 'dres1a', 'dres1b')


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--reps', type=int, default=5)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--batch', type=int, default=64)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    cfg = default_cfg.clone()
    B, D = args.batch, cfg.NETWORK.MAX_DISP
    model = M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()
    sets = []
    for s in range(4):
        left, right, _ = synthetic.stereo_pair(B, cfg.CONST.IMG_H, cfg.CONST.IMG_W, 2 * D, seed=100 + s)
        sets.append((left.cuda(), right.cuda(), synthetic.gt_volume(B, seed=200 + s).cuda()))

    marks = {}                                          # layer -> (start event, end event) of the current forward
    conv = model._conv

    def timed_conv(name, x, **kw):
        if name not in LAYERS:
            return conv(name, x, **kw)
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = conv(name, x, **kw)
        b.record()
        marks[name] = (a, b)
        return out
    model._conv = timed_conv

    arms = {'skip': 0, 'no_dz_skip': 1}
    step = {n: [] for n in arms}
    layer = {n: {l: [] for l in LAYERS} for n in arms}
    with torch.no_grad():
        for n, v in arms.items():                       # warm-up: both arms' tensor maps, schedules and workspaces
            lib.set_knob('no_dz_skip', v)
            for k in range(3):
                model(*sets[k % 4])
        torch.cuda.synchronize()
        for _ in range(args.reps):
            for n, v in arms.items():
                lib.set_knob('no_dz_skip', v)
                for k in range(args.steps):
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                    model(*sets[k % 4])
                    b.record()
                    b.synchronize()
                    step[n].append(a.elapsed_time(b))
                    for l in LAYERS:
                        layer[n][l].append(marks[l][0].elapsed_time(marks[l][1]))

        # planes marched per layer (one forward per arm, the counter attached to one layer at a time)
        h, w = cfg.CONST.IMG_H // 4, cfg.CONST.IMG_W // 4
        algo = 2 * B * -(-h // 32) * -(-w // 8) * D
        planes = {n: {} for n in arms}
        counter = torch.zeros(1, dtype=torch.int64, device='cuda')
        for n, v in arms.items():
            lib.set_knob('no_dz_skip', v)
            for l in LAYERS:
                def one(name, x, _l=l, **kw):
                    layers.plane_counter = counter if name == _l else None
                    try:
                        return conv(name, x, **kw)
                    finally:
                        layers.plane_counter = None
                model._conv = one
                counter.zero_()
                model(*sets[0])
                torch.cuda.synchronize()
                planes[n][l] = int(counter.item())
        lib.set_knob('no_dz_skip', 0)

    def summ(v):
        return {'median': statistics.median(v), 'min': min(v), 'max': max(v), 'n': len(v)}
    res = {
        'what': 'default bf16 Stereo2Voxel forward, eager, B = %d, %dx%d, D = %d; arms alternate %d x %d steps' % (
            B, cfg.CONST.IMG_H, cfg.CONST.IMG_W, D, args.reps, args.steps),
        'gpu': gpu_info(),
        'step_ms': {n: summ(step[n]) for n in arms},
        'layer_ms': {n: {l: summ(layer[n][l]) for l in LAYERS} for n in arms},
        'planes_marched': planes,
        'planes_algorithmic': algo,
    }
    s0, s1 = res['step_ms']['skip']['median'], res['step_ms']['no_dz_skip']['median']
    res['step_gain'] = 1 - s0 / s1
    res['layer_gain'] = {l: 1 - res['layer_ms']['skip'][l]['median'] / res['layer_ms']['no_dz_skip'][l]['median'] for l in LAYERS}
    res['planes_saved'] = {l: 1 - planes['skip'][l] / planes['no_dz_skip'][l] for l in LAYERS}
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            f.write(text + '\n')


if __name__ == '__main__':
    main()
