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
import math
import os
import sys

import torch


def camera_arg(text):
    """--camera f,cx,cy,baseline[,doffs] -> [5 floats]: finite, f > 0, baseline > 0 (doffs defaults to 0)."""
    try:
        c = [float(v) for v in text.split(',')]
    except ValueError:
        raise argparse.ArgumentTypeError('expected f,cx,cy,baseline[,doffs] as numbers, got %r' % text) from None
    if len(c) not in (4, 5) or not all(math.isfinite(v) for v in c) or not (c[0] > 0 and c[3] > 0):
        raise argparse.ArgumentTypeError('expected 4 or 5 finite numbers f,cx,cy,baseline[,doffs] with f > 0 and baseline > 0, '
                                         'got %r' % text)
    return c + [0.0] * (5 - len(c))


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
    p.add_argument('--speckle', action='store_true',
                   help='also remove the small connected regions of each disparity map (OpenCV\'s filterSpeckles with '
                        'TEST.SPECKLE_MAX_SIZE / SPECKLE_MAX_DIFF, after the LR check with --lr-check) and report the kept '
                        'pixels as speckle; with --save-clouds the clouds keep only those pixels')
    p.add_argument('--wls', action='store_true',
                   help='also fill each disparity map with the confidence-weighted WLS filter (OpenCV\'s DisparityWLSFilter '
                        'with TEST.WLS_LAMBDA / WLS_SIGMA; confident where --speckle / --lr-check keep a pixel, else where it '
                        'is finite) and report it as wls; with --save-clouds the clouds come from the filtered maps')
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
    p.add_argument('--fscore-curves', action='store_true',
                   help='also histogram the nearest-neighbour distances over TEST.DIST_BINS edges up to TEST.DIST_MAX and '
                        'report precision, recall and F-score at every edge, accuracy and completeness as point_curves '
                        '(Stereo2Point) or surface_curves (Stereo2Voxel, with --surface)')
    p.add_argument('--save-clouds', metavar='DIR', default=None,
                   help='also back-project both disparity maps of each pair into one coloured point cloud (filtered by '
                        '--lr-check / --uncertainty when given) and write it, with the cloud of its GT disparity, as '
                        'DIR/%%06d.ply and DIR/%%06d_gt.ply (binary PLY), numbered by sample; reports the points as cloud')
    p.add_argument('--camera', metavar='F,CX,CY,BASELINE[,DOFFS]', type=camera_arg, default=None,
                   help='camera of --save-clouds (default CONST.CAMERA): focal length and principal point in px, baseline in '
                        'the clouds\' units, principal-point offset between the views in px')
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
    if args.fscore_curves and args.model == 'Stereo2Voxel' and not args.surface:
        sys.exit('--fscore-curves evaluates the voxel surfaces for Stereo2Voxel: add --surface')
    if args.camera is not None and args.save_clouds is None:
        sys.exit('--camera sets the camera of --save-clouds: add --save-clouds DIR')
    if args.camera is not None:
        cfg.CONST.CAMERA = args.camera
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
    if args.save_clouds is not None:
        ev.update(eval_cloud=True)
    if args.speckle:
        ev.update(eval_speckle=True)
    if args.wls:
        ev.update(eval_wls=True)
    if args.fscore_curves:
        ev.update(eval_fscore_curves=True)
    if args.model == 'Stereo2Voxel':
        ev.update(eval_surface=args.surface, eval_curves=args.curves)
        stats = T.test_voxel(cfg, model, n, bs, rank, world, mesh_dir=args.save_meshes, cloud_dir=args.save_clouds, **ev).cpu()
    else:
        ev.update(eval_points=True)
        stats = T.test_point(cfg, model, n, bs, rank, world, cloud_dir=args.save_clouds, **ev).cpu()
    b = T.split_stats(stats, T.stats_layout(cfg, args.model, **ev))
    res = T.iou_summary(b['iou'], cfg.TEST.VOXEL_THRESH) if 'iou' in b else T.chamfer_summary(b['chamfer'])
    npix = res['n_samples'] * cfg.CONST.IMG_H * cfg.CONST.IMG_W
    res['disparity'] = T.disp_summary(b['disparity'], cfg.TEST.DISP_THRESH)
    if 'lr_consistency' in b:
        res['lr_consistency'] = T.lr_summary(b['lr_consistency'], cfg.TEST.DISP_THRESH, npix, b['disparity'])
        res['lr_consistency']['lr_thresh'] = float(cfg.TEST.LR_THRESH)
    if 'speckle' in b:
        res['speckle'] = T.speckle_summary(b['speckle'], cfg.TEST.DISP_THRESH, npix, b['disparity'])
        max_size, max_diff = models.speckle_params(cfg)
        res['speckle'].update(max_size=max_size, max_diff=max_diff, after_lr_check=args.lr_check)
    if 'wls' in b:
        res['wls'] = T.wls_summary(b['wls'], cfg.TEST.DISP_THRESH, npix, b['disparity'])
        lam, sigma = models.wls_params(cfg)
        res['wls'].update({'lambda': lam, 'sigma': sigma,
                           'confidence': 'speckle' if args.speckle else 'lr_check' if args.lr_check else 'finite'})
    if 'uncertainty' in b:
        res['uncertainty'] = T.unc_summary(b['uncertainty'], cfg.TEST.UNC_THRESH, cfg.TEST.DISP_THRESH, npix, b['disparity'])
    if 'cloud' in b:
        res['cloud'] = T.cloud_summary(b['cloud'], res['n_samples'], cfg.CONST.IMG_H, cfg.CONST.IMG_W)
        res['cloud'].update(camera=models.camera_values(cfg), min_disp=models.cloud_min_disp(cfg),
                            max_std=models.cloud_max_std(cfg) if args.uncertainty and not args.wls else None)
        if args.speckle:
            res['cloud'].update(speckle=dict(max_size=max_size, max_diff=max_diff))
        if args.wls:
            res['cloud'].update(wls={'lambda': lam, 'sigma': sigma})
    if 'surface' in b:
        res['surface'] = T.surface_summary(b['surface'], cfg.TEST.VOXEL_THRESH, cfg.TEST.FSCORE_THRESH, res['n_samples'])
    if 'curves' in b:
        res['occupancy_curves'] = T.curves_summary(b['curves'], cfg.TEST.CURVE_BINS, res['n_samples'])
    if 'points' in b:
        res['points'] = T.points_summary(b['points'], cfg.TEST.FSCORE_THRESH, res['n_samples'], cfg.CONST.N_POINTS,
                                         cfg.CONST.N_GT_POINTS)
    if 'surface_curves' in b:
        res['surface_curves'] = T.surface_curves_summary(b['surface_curves'], cfg.TEST.VOXEL_THRESH, models.dist_edges(cfg),
                                                         res['n_samples'])
    if 'point_curves' in b:
        res['point_curves'] = T.point_curves_summary(b['point_curves'], models.dist_edges(cfg), res['n_samples'])
    if rank == 0:
        res.update(model=args.model, precision=cfg.NETWORK.PRECISION, world_size=world, data='synthetic')
        print(json.dumps(res))
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
