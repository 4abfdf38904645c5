#!/usr/bin/env python3
"""Cost of the marching-cubes mesh (s3d_voxel_mesh, Stereo2Voxel forward(left, right, mesh=True)), in one run, CUDA events,
the arms alternating:

  1. the kernel alone at B = 64, n = 32, t = TEST.MESH_THRESH, on a prediction-like field (the synthetic GT volumes blended
     with noise, as in surface_eval_time.py) and on smooth balls, through the C entry point into preallocated buffers.  L2 is
     overwritten (256 MB write) before every single timed call; a second measurement times 20 back-to-back calls (L2 warm,
     launch gaps hidden), and torch.profiler gives the kernel's device time;
  2. the default Stereo2Voxel forward replayed from its CUDA graph at B = 64, model.graphed(left, right) against
     model.graphed(left, right, mesh=True).

Also records the launches per eager forward with and without the flag, the mean mesh sizes, and the GPU name and power limit
beside the numbers.

    python scripts/mesh_time.py [--reps 20] [--out profiles/mesh_time.json]
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


def kernel_device_ms(fn, calls):
    """Mean device time per call of voxel_mesh_kernel over `calls` calls of fn, from torch.profiler (a run of its own)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    ts = [e.device_time_total if hasattr(e, 'device_time_total') else e.cuda_time_total
          for e in prof.events() if e.device_type.name == 'CUDA' and 'voxel_mesh_kernel' in e.name]
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
    B, n, t = cfg.CONST.BATCH_SIZE, cfg.CONST.N_VOX, M.mesh_thresh(cfg)

    # 1. the kernel alone
    gt = torch.cat([synthetic.gt_volume(1, n, seed=100000 + i) for i in range(B)]).to(dev)
    noise = torch.rand(B, n, n, n, generator=torch.Generator().manual_seed(1)).to(dev)
    fields = {'noisy_gt': (0.6 * gt.float() + 0.5 * noise).clamp_(0, 1).contiguous()}
    g = (torch.arange(n, device=dev, dtype=torch.float32) + 0.5) / n - 0.5
    z, y, x = torch.meshgrid(g, g, g, indexing='ij')
    r = torch.linspace(0.1, 0.45, B, device=dev).view(B, 1, 1, 1)
    fields['balls'] = (0.5 + (r - torch.sqrt(x * x + y * y + z * z)) * n).clamp_(0, 1).contiguous()
    mv, mf = ops.voxel_mesh_bounds(n)
    out = (torch.empty(B, mv, 3, device=dev), torch.empty(B, mf, 3, dtype=torch.int32, device=dev),
           torch.empty(B, 2, dtype=torch.int32, device=dev))
    L = lib.load()
    st = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    res['kernel'] = {'shape': 'B=%d, n=%d, t=%g' % (B, n, t), 'max_verts': mv, 'max_faces': mf,
                     'output_bytes': sum(o.numel() * o.element_size() for o in out)}
    for name, vol in fields.items():
        def mesh():                                 # ops.voxel_mesh's call, without its Python checks
            lib.check(L.s3d_voxel_mesh(vol.data_ptr(), B, n, t, out[0].data_ptr(), mv, out[1].data_ptr(), mf,
                                       out[2].data_ptr(), st), 's3d_voxel_mesh')
        for _ in range(3):
            mesh()
        k = flushed_alternating({name: mesh}, flush, args.reps * 5)
        loop = time_alternating({name: lambda i: mesh()}, 20, args.reps)
        mesh()
        c = out[2].cpu().double()
        res['kernel'][name] = {'flushed_single_calls': args.reps * 5, 'loop_calls_per_sample': 20, 'loop_samples': args.reps,
                               'flushed': summary(k[name]), 'loop': summary(loop[name]), 'profiler': kernel_device_ms(mesh, 20),
                               'mean_verts_per_sample': c[:, 0].mean().item(), 'mean_faces_per_sample': c[:, 1].mean().item(),
                               'max_faces_per_sample': c[:, 1].max().item()}
    del flush, out

    # 2. the graphed forward
    model = M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()
    H, W, D = cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.NETWORK.MAX_DISP
    left, right, _ = synthetic.stereo_pair(B, H, W, 2 * D, seed=1)
    left, right = left.to(dev), right.to(dev)
    with torch.no_grad():
        arms = {'graphed': lambda i: model.graphed(left, right),
                'graphed_mesh': lambda i: model.graphed(left, right, mesh=True)}
        time_alternating(arms, 3, 2)
        f = time_alternating(arms, 10, args.reps)
        m_p, m_s = statistics.median(f['graphed']), statistics.median(f['graphed_mesh'])
        res['graphed_forward'] = {'shape': 'Stereo2Voxel default config, %s, B=%d, %dx%d, D=%d, no gt'
                                           % (cfg.NETWORK.PRECISION, B, H, W, D),
                                  'calls_per_sample': 10, 'samples': args.reps,
                                  'graphed': summary(f['graphed']), 'graphed_mesh': summary(f['graphed_mesh']),
                                  'added_ms': m_s - m_p, 'added_pct': 100.0 * (m_s - m_p) / m_p}
        c = model.graphed(left, right, mesh=True)[-1].cpu().double()
        res['graphed_forward']['mean_verts_faces_per_sample'] = c.mean(0).tolist()
        n0 = lib.launches(); model(left, right); n1 = lib.launches()
        model(left, right, mesh=True); n2 = lib.launches()
    res['launches'] = {'forward': n1 - n0, 'forward_mesh': n2 - n1}
    txt = json.dumps(res, indent=1)
    print(txt)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as fh:
            fh.write(txt + '\n')


if __name__ == '__main__':
    main()
