#!/usr/bin/env python3
"""Cost of the stereo point clouds (s3d_disp_cloud, forward(..., camera=...)), in one run:

  1. the two kernels alone at B = 64, 256 x 256 on the disparity maps, LR mask and spread of one default Stereo2Voxel
     forward (lr_check=True with a 1000 px tolerance, uncertainty=True) of the synthetic pairs, with fp32 NCHW and uint8 HWC
     images, without a filter and with both (the spread threshold at the median spread), through the C entry point into
     preallocated buffers.  L2 is overwritten (256 MB write) before every
     timed call: CUDA events around each single call (the arms alternating), and torch.profiler device times of
     cloud_count_kernel and cloud_write_kernel in a run of their own, flushed the same way;
  2. the default Stereo2Voxel forward replayed from its CUDA graph at B = 64, model.graphed(left, right) against
     model.graphed(left, right, camera=camera).

Also records the kept points, the bytes each arm must move at least (reads of disp twice, of the filters twice, of the
kept pixels' colours, writes of the points) and the rate that gives, the launches per eager forward with and without the
camera, and the GPU name and power limit beside the numbers.

    python scripts/cloud_time.py [--reps 20] [--out profiles/cloud_time.json]
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

_KERNELS = ('cloud_count_kernel', 'cloud_write_kernel')


def kernels_device_ms(fn, flush, calls):
    """Mean device time per call of each cloud kernel over `calls` calls of fn, each after an L2 flush, from torch.profiler."""
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
        out['both_us'] = sum(out[k]['mean_us'] for k in _KERNELS)
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
    # the synthetic weights' maps are not left-right consistent: for the filtered arms, a wide LR tolerance keeps the pixels
    # whose match lies in the image, and the spread threshold is the median spread, so that each filter drops some pixels
    cfg.TEST.LR_THRESH = 1000.0
    model = M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()
    left, right, _ = synthetic.stereo_pair(B, H, W, 2 * D, seed=1)
    left, right = left.to(dev).contiguous(), right.to(dev).contiguous()
    camera = torch.tensor([M.camera_values(cfg)] * B, dtype=torch.float32, device=dev)
    min_disp = M.cloud_min_disp(cfg)

    # 1. the kernels alone, on the forward's own maps
    with torch.no_grad():
        o = dict(zip(M.Stereo2Voxel.output_names(lr_check=True, uncertainty=True),
                     model(left, right, lr_check=True, uncertainty=True)))
        disp = torch.cat([o['disp_left'][:, 0], o['disp_right'][:, 0]]).contiguous()
        mask, std = o['lr_mask'].clone(), o['disp_std'].clone()
        max_std = float(std[torch.isfinite(std)].median())
    u8 = {'left': (left * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous(),
          'right': (right * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous()}
    out = (torch.empty(B, 2 * H * W, 3, device=dev), torch.empty(B, 2 * H * W, 3, dtype=torch.uint8, device=dev),
           torch.empty(B, 2, dtype=torch.int32, device=dev))
    nb = ops.disp_cloud_workspace_bytes(B, H)
    ws = torch.empty(nb, dtype=torch.uint8, device=dev)
    L = lib.load()
    st = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    arms = {}
    for img in ('fp32', 'uint8'):
        lt, rt = (left, right) if img == 'fp32' else (u8['left'], u8['right'])
        for filt in ('none', 'lr_std'):
            mp, sp = (None, None) if filt == 'none' else (mask.data_ptr(), std.data_ptr())

            def cloud(lt=lt, rt=rt, mp=mp, sp=sp, u=int(img == 'uint8')):   # ops.disp_cloud's call, without its Python checks
                lib.check(L.s3d_disp_cloud(disp.data_ptr(), B, H, W, lt.data_ptr(), rt.data_ptr(), u, mp, sp, max_std,
                                           camera.data_ptr(), min_disp, out[0].data_ptr(), out[1].data_ptr(),
                                           out[2].data_ptr(), ws.data_ptr(), nb, st), 's3d_disp_cloud')
            arms['%s_%s' % (img, filt)] = (cloud, img, filt)
    for fn, _, _ in arms.values():
        for _ in range(3):
            fn()
    k = flushed_alternating({n: a[0] for n, a in arms.items()}, flush, args.reps * 5)
    res['kernels'] = {'shape': 'B=%d, %dx%d, camera %s, min_disp %g; lr_std arms: LR_THRESH %g, max_std %g (the median '
                               'spread)' % (B, H, W, M.camera_values(cfg), min_disp, cfg.TEST.LR_THRESH, max_std),
                      'flushed_single_calls': args.reps * 5}
    pix = 2 * B * H * W
    for name, (fn, img, filt) in arms.items():
        fn()
        c = out[2].to(torch.int64).sum().item()
        prof = kernels_device_ms(fn, flush, 20)
        filt_bytes = 0 if filt == 'none' else pix * (1 + 4)
        img_bytes = c * 3 * (4 if img == 'fp32' else 1)
        nbytes = 2 * (pix * 4 + filt_bytes) + img_bytes + c * 15
        e = {'events_flushed': summary(k[name]), 'profiler': prof, 'kept_points': c, 'kept_fraction': c / pix,
             'min_bytes': nbytes}
        if 'both_us' in prof:
            e['min_bytes_over_profiler_time_GBps'] = nbytes / prof['both_us'] / 1e3
        res['kernels'][name] = e
    del flush, out, ws

    # 2. the graphed forward
    with torch.no_grad():
        f_arms = {'graphed': lambda i: model.graphed(left, right),
                  'graphed_camera': lambda i: model.graphed(left, right, camera=camera)}
        time_alternating(f_arms, 3, 2)
        f = time_alternating(f_arms, 10, args.reps)
        m_p, m_c = statistics.median(f['graphed']), statistics.median(f['graphed_camera'])
        res['graphed_forward'] = {'shape': 'Stereo2Voxel default config, %s, B=%d, %dx%d, D=%d, no gt'
                                           % (cfg.NETWORK.PRECISION, B, H, W, D),
                                  'calls_per_sample': 10, 'samples': args.reps,
                                  'graphed': summary(f['graphed']), 'graphed_camera': summary(f['graphed_camera']),
                                  'added_ms': m_c - m_p, 'added_pct': 100.0 * (m_c - m_p) / m_p}
        c = model.graphed(left, right, camera=camera)[-1].to(torch.int64).sum().item()
        res['graphed_forward']['kept_fraction'] = c / pix
        n0 = lib.launches(); model(left, right); n1 = lib.launches()
        model(left, right, camera=camera); n2 = lib.launches()
    res['launches'] = {'forward': n1 - n0, 'forward_camera': n2 - n1}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            fh.write(txt + '\n')


if __name__ == '__main__':
    main()
