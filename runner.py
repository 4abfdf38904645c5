#!/usr/bin/env python3
# -*- coding: utf-8 -*-
"""CLI entry, same contract as the reference's runner.py (README.md:85,91):

    python3 runner.py --test --weights=/path/to/pretrained/model.pth

Only the inference (`--test`) path is built (training is out of scope, SURVEY.md 2 row 12).
StereoShapeNet and the pretrained .pth files are unavailable offline, so without --weights the
model gets seeded synthetic weights and the test set is synthetic (config.py shapes).
Multi-GPU: launch with torchrun (one process per GPU); shards are contiguous by rank and the
IoU / Chamfer statistics are reduced with one NCCL all-reduce.
"""
import argparse
import json
import os
import sys

import torch


def get_args():
    p = argparse.ArgumentParser(description='Stereo 3D reconstruction (B200 inference path)')
    p.add_argument('--test', action='store_true', help='run the test (inference) path')
    p.add_argument('--weights', default=None, help='checkpoint (.pth) with a state_dict or {"model": state_dict}')
    p.add_argument('--model', default='Stereo2Voxel', choices=['Stereo2Voxel', 'Stereo2Point'])
    p.add_argument('--precision', default=None, choices=['bf16', 'bf16x3', 'tf32', 'tf32x3', 'fp32'])
    p.add_argument('--batch-size', type=int, default=None)
    p.add_argument('--n-samples', type=int, default=None, help='synthetic test-set size (default: one batch per rank)')
    p.add_argument('--lr-check', action='store_true',
                   help='also run the left-right disparity consistency check and report it as lr_consistency')
    p.add_argument('--uncertainty', action='store_true',
                   help='also compute the per-pixel disparity uncertainty and report the confidence-filtered metrics as uncertainty')
    p.add_argument('--surface', action='store_true',
                   help='Stereo2Voxel: also evaluate the voxel-face surfaces against GT and report Chamfer L2 / L1 and '
                        'F-score as surface')
    p.add_argument('--save-meshes', metavar='DIR', default=None,
                   help='Stereo2Voxel: also write the marching-cubes mesh of each prediction (at TEST.MESH_THRESH) and of its '
                        'GT occupancy as DIR/%%06d.obj and DIR/%%06d_gt.obj, numbered by sample')
    p.add_argument('--curves', action='store_true',
                   help='Stereo2Voxel: also evaluate the occupancy probabilities in TEST.CURVE_BINS bins and report the IoU '
                        'and precision-recall curves over every bin threshold, BCE, Brier and calibration as occupancy_curves')
    return p.parse_args()


def flatten_checkpoint(ckpt, prefixes=()):
    """-> flat {key: tensor}.  Accepts a plain state_dict, {'model' | 'state_dict': sd}, or a checkpoint holding one
    state_dict PER SUB-NETWORK ({'dispnet': sd, 'decoder_state_dict': sd, ...}: the sub-dict's name, minus a
    '_state_dict' suffix, becomes the key prefix); DataParallel 'module.' prefixes are stripped at every level.
    (The upstream checkpoint layout is not on disk -- README.md:35-36 only names the files -- so nothing here maps
    upstream LAYER names; a mismatch is reported key by key instead of a bare strict-load failure.)"""
    flat = {}
    for k, v in ckpt.items():
        name = k[len('module.'):] if k.startswith('module.') else k
        if torch.is_tensor(v):
            flat['.'.join(prefixes + (name,))] = v
        elif isinstance(v, dict) and v and all(isinstance(kk, str) for kk in v):
            if name in ('model', 'state_dict') and not prefixes:
                flat.update(flatten_checkpoint(v))
            elif any(torch.is_tensor(t) or isinstance(t, dict) for t in v.values()) and 'optim' not in name and 'solver' not in name:
                sub = name[:-len('_state_dict')] if name.endswith('_state_dict') else name
                flat.update(flatten_checkpoint(v, prefixes + (sub,)))
    return {k.replace('.module.', '.'): v for k, v in flat.items()}


def load_checkpoint(model, path):
    ckpt = torch.load(path, map_location='cpu')
    if not isinstance(ckpt, dict):
        sys.exit('--weights: %s does not hold a state_dict' % path)
    sd = flatten_checkpoint(ckpt)
    own = model.state_dict()
    missing = sorted(k for k in own if k not in sd)
    unexpected = sorted(k for k in sd if k not in own)
    shape = sorted(k for k in own if k in sd and tuple(own[k].shape) != tuple(sd[k].shape))
    if missing or unexpected or shape:
        def head(keys):
            return ', '.join(keys[:8]) + (' ... (+%d)' % (len(keys) - 8) if len(keys) > 8 else '')
        sys.exit('--weights: %s does not match %s (this build defines its own [SPEC] layer names, DESIGN.md section 3; '
                 'upstream .pth files need a key map that cannot be written without the upstream source).\n'
                 '  missing    (%d): %s\n  unexpected (%d): %s\n  shape      (%d): %s'
                 % (path, type(model).__name__, len(missing), head(missing), len(unexpected), head(unexpected),
                    len(shape), head(shape)))
    model.load_state_dict(sd)


def main():
    args = get_args()
    from config import cfg
    if not args.test:
        sys.exit('Only `runner.py --test` is implemented: this is the inference-tier build (training is out of scope).')
    if args.surface and args.model != 'Stereo2Voxel':
        sys.exit('--surface evaluates voxel surfaces: Stereo2Voxel only')
    if args.save_meshes is not None and args.model != 'Stereo2Voxel':
        sys.exit('--save-meshes meshes the voxel occupancy: Stereo2Voxel only')
    if args.curves and args.model != 'Stereo2Voxel':
        sys.exit('--curves evaluates the voxel occupancy: Stereo2Voxel only')
    if not torch.cuda.is_available():
        sys.exit('runner.py --test needs a CUDA device (sm_100a); there is no CPU fallback.')
    from stereo_3d_reconstruction_b200 import models
    from stereo_3d_reconstruction_b200.core import test as T
    import torch.distributed as dist
    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    if args.precision:
        cfg.NETWORK.PRECISION = args.precision
    bs = args.batch_size or cfg.CONST.BATCH_SIZE
    n = args.n_samples or bs * world
    model = models.build_model(args.model, cfg, seed=None if args.weights else cfg.CONST.SEED)
    if args.weights:
        load_checkpoint(model, args.weights)
    model.cuda().pack()
    # one stats vector: the head's statistics, then the disparity counters of the same forwards (core/test.py::stats_layout)
    ev = dict(eval_disp=True, eval_lr=args.lr_check, eval_unc=args.uncertainty)
    if args.model == 'Stereo2Voxel':
        ev.update(eval_surface=args.surface, eval_curves=args.curves)
        stats = T.test_voxel(cfg, model, n, bs, rank, world, mesh_dir=args.save_meshes, **ev).cpu()
    else:
        ev.update(eval_points=True)
        stats = T.test_point(cfg, model, n, bs, rank, world, **ev).cpu()
    b = T.split_stats(stats, T.stats_layout(cfg, args.model, **ev))
    res = T.iou_summary(b['iou'], cfg.TEST.VOXEL_THRESH) if 'iou' in b else T.chamfer_summary(b['chamfer'])
    npix = res['n_samples'] * cfg.CONST.IMG_H * cfg.CONST.IMG_W
    res['disparity'] = T.disp_summary(b['disparity'], cfg.TEST.DISP_THRESH)
    if 'lr_consistency' in b:
        res['lr_consistency'] = T.lr_summary(b['lr_consistency'], cfg.TEST.DISP_THRESH, npix, b['disparity'])
        res['lr_consistency']['lr_thresh'] = float(cfg.TEST.LR_THRESH)
    if 'uncertainty' in b:
        res['uncertainty'] = T.unc_summary(b['uncertainty'], cfg.TEST.UNC_THRESH, cfg.TEST.DISP_THRESH, npix, b['disparity'])
    if 'surface' in b:
        res['surface'] = T.surface_summary(b['surface'], cfg.TEST.VOXEL_THRESH, cfg.TEST.FSCORE_THRESH, res['n_samples'])
    if 'curves' in b:
        res['occupancy_curves'] = T.curves_summary(b['curves'], cfg.TEST.CURVE_BINS, res['n_samples'])
    if 'points' in b:
        res['points'] = T.points_summary(b['points'], cfg.TEST.FSCORE_THRESH, res['n_samples'], cfg.CONST.N_POINTS,
                                         cfg.CONST.N_GT_POINTS)
    if rank == 0:
        res.update(model=args.model, precision=cfg.NETWORK.PRECISION, world_size=world, data='synthetic')
        print(json.dumps(res))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
