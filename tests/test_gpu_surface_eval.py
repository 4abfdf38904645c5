"""Voxel-surface evaluation inside the forward (s3d_voxel_surface_eval): the integer counters equal the reference statement
(tests/surface_oracle.py) exactly, on hand-built and random grids and on the very voxels the forward returns; every other
output of the forward is unchanged."""
import ctypes
import json
import sys

import numpy as np
import pytest
import torch

from stereo_3d_reconstruction_b200 import lib, models as M, ops
from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.utils import synthetic
from tests.common import small_cfg
from tests.surface_oracle import surface_block, surface_stats

pytestmark = pytest.mark.gpu
LEVELS = np.array([0.1, 0.25, 0.5, 0.75, 0.9], np.float32)
VTH8 = [0.25, 0.5, 0.75, 0.9, 0.1, 0.3, 0.6, 0.95]               # the first five are values present in fused: >= at equality
FTH8 = [0.01, 0.02, 0.03, 0.05, 0.08, 0.12, 0.3, 1.8]


def _grids(B, n, seed, p_gt=0.2):
    rng = np.random.default_rng(seed)
    fused = LEVELS[rng.integers(0, len(LEVELS), (B, n, n, n))]
    fused[rng.random((B, n, n, n)) < 0.02] = np.nan
    gt = (rng.random((B, n, n, n)) < p_gt).astype(np.uint8) * rng.integers(1, 256, (B, n, n, n)).astype(np.uint8)
    return fused, gt


def _run(fused, gt, vth, fth, stats=None):
    B = fused.shape[0]
    f, g = torch.from_numpy(np.ascontiguousarray(fused)).cuda(), torch.from_numpy(np.ascontiguousarray(gt)).cuda()
    if stats is None:
        stats = torch.zeros(B, len(vth), 2, 3 + len(fth), dtype=torch.int64, device='cuda')
    n0 = lib.launches()
    ops.voxel_surface_eval(f, g, vth, fth, stats)
    assert lib.launches() - n0 == 2
    return stats


def _check(fused, gt, vth, fth):
    want = surface_stats(fused, gt, vth, fth)
    st = _run(fused, gt, vth, fth)
    assert np.array_equal(st.cpu().numpy(), want)
    _run(fused, gt, vth, fth, stats=st)                             # ADDED to: a second call doubles every counter
    assert np.array_equal(st.cpu().numpy(), 2 * want)
    return want


@pytest.mark.parametrize('n,B,T_,F', [(4, 3, 4, 8), (8, 3, 4, 8), (32, 3, 4, 8), (64, 1, 8, 8),
                                      (8, 1, 1, 1), (8, 64, 4, 1), (8, 3, 8, 1), (8, 3, 1, 8), (32, 64, 4, 1)])
def test_kernel_matches_oracle(n, B, T_, F):
    fused, gt = _grids(B, n, seed=n * 1000 + B * 10 + T_ + F)
    want = _check(fused, gt, VTH8[:T_], FTH8[:F])
    assert (want[:, :, 1, 0] > 0).all() and (want[:, :, :, 1] > 0).any()    # (t = 0.95 is above every value: an empty prediction)
    if n >= 8:
        assert (want[:, :, :, 3 + F - 1] > 0).any()


def test_kernel_one_and_odd_sizes():
    for n in (1, 2, 3, 5, 17, 63):
        fused, gt = _grids(2, n, seed=n, p_gt=0.5)
        _check(fused, gt, [0.25, 0.75], [0.02, 0.2])


def test_kernel_empty_and_full():
    n = 8
    fused = np.stack([np.zeros((n,) * 3), np.ones((n,) * 3), np.full((n,) * 3, np.nan), np.ones((n,) * 3)]).astype(np.float32)
    gt = np.stack([np.ones((n,) * 3), np.zeros((n,) * 3), np.ones((n,) * 3), np.ones((n,) * 3)]).astype(np.uint8)
    gt[3, 2:5, 1:7, 3] = 0                                          # a full prediction against a GT with a hole
    want = _check(fused, gt, [0.5, 2.0], [0.05, 0.5])
    assert want[0, 0, 0, 0] == 0 and want[0, 0, 1].tolist() == [6 * n * n, 0, 0, 0, 0]       # empty prediction
    assert want[1, 0, 0].tolist() == [6 * n * n, 0, 0, 0, 0] and want[1, 0, 1, 0] == 0        # empty GT
    assert want[1, 1].tolist() == [[0] * 5, [0] * 5]                                          # both empty
    assert want[3, 0, 1, 1] > 0


def test_kernel_synthetic_gt_density():
    g = synthetic.gt_volume(4, 32, seed=100000).numpy()
    fused = np.where(synthetic.gt_volume(4, 32, seed=7).numpy() != 0, 0.8, 0.2).astype(np.float32)
    want = _check(fused, g, [0.5], [0.01, 0.03])
    assert all(17000 < c < 19000 for c in want[:, 0, 1, 0])


def test_kernel_bad_arguments():
    L = lib.load()
    B, n = 2, 8
    f = torch.rand(B, n, n, n, device='cuda')
    g = torch.zeros(B, n, n, n, dtype=torch.uint8, device='cuda')
    st = torch.zeros(B, 8, 2, 11, dtype=torch.int64, device='cuda')
    need = ops.voxel_surface_workspace_bytes(B, 8, 64)
    ws = torch.empty(need, dtype=torch.uint8, device='cuda')
    s = torch.cuda.current_stream().cuda_stream

    def th(*v):
        return (ctypes.c_float * max(len(v), 1))(*v)

    def kb(*v):
        return (ctypes.c_int * max(len(v), 1))(*v)

    def call(B_=B, n_=n, th_=th(0.5), T_=1, kb_=kb(1), F_=1, st_=st.data_ptr(), ws_=ws.data_ptr(), wsb=need, f_=f.data_ptr(),
             g_=g.data_ptr()):
        return L.s3d_voxel_surface_eval(f_, g_, B_, n_, th_, T_, kb_, F_, st_, ws_, wsb, s)
    assert call() == 0 and call(B_=0) == 0 and call(T_=8, th_=th(*[0.5] * 8), kb_=kb(*[1] * 8), F_=8) == 0
    assert call(F_=0, kb_=None) == 0 and call(kb_=kb(3 * 16 * 16 + 1)) == 0
    for bad in (dict(n_=65), dict(n_=0), dict(T_=9, th_=th(*[0.5] * 9)), dict(F_=9, kb_=kb(*[1] * 9)), dict(T_=-1),
                dict(B_=-1), dict(st_=None), dict(ws_=None), dict(wsb=ops.voxel_surface_workspace_bytes(B, 1, n) - 1),
                dict(f_=None), dict(g_=None), dict(th_=None), dict(kb_=None), dict(kb_=kb(-1)), dict(kb_=kb(3 * 16 * 16 + 2))):
        rc = call(**bad)
        assert rc == -1, bad
        with pytest.raises(lib.S3dError):
            lib.check(rc, 's3d_voxel_surface_eval')
    assert L.s3d_voxel_surface_workspace_bytes(1, 1, 65) < 0
    torch.cuda.synchronize()
    for bad in (dict(stats=st[:, :1, :, :3].contiguous()), dict(fused=f.double()), dict(gt8=g.float()), dict(gt8=g[:1]),
                dict(fused=f.reshape(B, -1)[:, 1:].contiguous(), gt8=g.reshape(B, -1)[:, 1:].contiguous()),
                dict(workspace=ws[:10])):
        kw = dict(fused=f, gt8=g, stats=st[:, :1, :, :4].contiguous(), workspace=None)
        kw.update(bad)
        with pytest.raises(ValueError):
            ops.voxel_surface_eval(kw['fused'], kw['gt8'], [0.5], [0.01], kw['stats'], workspace=kw['workspace'])


# ---- the model ------------------------------------------------------------------------------------------------------------
FTH = [0.01, 0.05, 0.1]


def _model(prec, default=False, **kw):
    kw.setdefault('TEST__FSCORE_THRESH', FTH)
    if default:
        from config import cfg as dcfg
        cfg = dcfg.clone()
        cfg.NETWORK.PRECISION = prec
        for k, v in kw.items():
            sec, key = k.split('__')
            cfg[sec][key] = v
    else:
        cfg = small_cfg(NETWORK__PRECISION=prec, **kw)
    return cfg, M.build_model('Stereo2Voxel', cfg, seed=3).cuda().pack()


def _inputs(cfg, B, seed):
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=seed)
    gt = synthetic.gt_volume(B, cfg.CONST.N_VOX, seed=seed + 50)
    return (left.cuda(), right.cuda()), gt.cuda(), synthetic.disparity_gt(d, H, W).cuda()


def _check_model(cfg, vox, gt, ss):
    want = surface_stats(vox.cpu().numpy(), gt.cpu().numpy(), list(cfg.TEST.VOXEL_THRESH), list(cfg.TEST.FSCORE_THRESH))
    assert ss.dtype == torch.int64 and np.array_equal(ss.cpu().numpy(), want)
    return want


@pytest.mark.parametrize('default', [False, True])
@pytest.mark.parametrize('prec', ['bf16', 'bf16x3'])
def test_model_surface_stats_exact_and_outputs_unchanged(prec, default):
    cfg, model = _model(prec, default)
    args, gt, _ = _inputs(cfg, 2, seed=1)
    with torch.no_grad():
        n0 = lib.launches()
        plain = [t.clone() for t in model(*args, gt)]
        n1 = lib.launches()
        surf = [t.clone() for t in model(*args, gt, surface=True)]
        n2 = lib.launches()
    assert (n2 - n1) - (n1 - n0) == 2                               # surface_plane_kernel + surface_count_kernel
    assert len(plain) == 4 and len(surf) == 5
    for a, b in zip(plain, surf):
        assert torch.equal(a, b)
    want = _check_model(cfg, surf[2], gt, surf[4])
    assert (want[:, :, :, 0] > 0).any()


def test_model_launches_unchanged_without_flag():
    cfg, model = _model('bf16')
    args, gt, dgt = _inputs(cfg, 2, seed=0)
    with torch.no_grad():
        counts = []
        for kw in (dict(), dict(surface=False), dict(surface=True)):
            n0 = lib.launches()
            model(*args, gt, disp_gt=dgt, **kw)
            counts.append(lib.launches() - n0)
    assert counts[0] == counts[1] and counts[2] == counts[0] + 2


def test_model_tuple_positions_with_every_option():
    cfg, model = _model('bf16')
    args, gt, dgt = _inputs(cfg, 2, seed=4)
    with torch.no_grad():
        base = [t.clone() for t in model(*args, gt, disp_gt=dgt, lr_check=True, uncertainty=True)]
        full = [t.clone() for t in model(*args, gt, disp_gt=dgt, lr_check=True, uncertainty=True, surface=True)]
    assert len(base) == 9 and len(full) == 10
    for a, b in zip(base, full):
        assert torch.equal(a, b)
    _check_model(cfg, full[2], gt, full[-1])


def test_graphed_matches_eager():
    cfg, model = _model('bf16')
    seen = []
    for seed in (0, 1):
        args, gt, dgt = _inputs(cfg, 2, seed=seed)
        with torch.no_grad():
            eager = [t.clone() for t in model(*args, gt, disp_gt=dgt, surface=True)]
            graphed = [t.clone() for t in model.graphed(*args, gt, disp_gt=dgt, surface=True)]
        assert len(graphed) == 6
        for a, b in zip(eager, graphed):
            assert torch.equal(a, b)
        seen.append(eager[-1])
    assert not torch.equal(seen[0], seen[1])
    with torch.no_grad():
        assert len(model.graphed(*args, gt, disp_gt=dgt)) == 5
    assert len(model._graphs) == 2                                  # surface is part of the graph key


def test_micro_batch_concatenates_chunks():
    cfg, model = _model('bf16', CONST__MICRO_BATCH=2)
    args, gt, dgt = _inputs(cfg, 5, seed=6)
    with torch.no_grad():
        full = [t.clone() for t in model(*args, gt, disp_gt=dgt, surface=True)]
        parts = [[t.clone() for t in model(args[0][s:s + 2], args[1][s:s + 2], gt[s:s + 2], disp_gt=dgt[s:s + 2], surface=True)]
                 for s in range(0, 5, 2)]
    for i, t in enumerate(full):
        assert torch.equal(t, torch.cat([p[i] for p in parts]))
    _check_model(cfg, full[2], gt, full[-1])


def test_value_errors_before_any_launch():
    cfg, model = _model('bf16')
    args, gt, _ = _inputs(cfg, 2, seed=0)
    model(*args)                                                    # packed, workspace built
    n0 = lib.launches()
    with pytest.raises(ValueError):
        model(*args, surface=True)
    with pytest.raises(ValueError):
        model.graphed(*args, surface=True)
    for bad in ([-0.1], [float('nan')], [0.1] * 9):
        cfg.TEST.FSCORE_THRESH = bad
        with pytest.raises(ValueError):
            model(*args, gt, surface=True)
        with pytest.raises(ValueError):
            model.graphed(*args, gt, surface=True)
    assert lib.launches() == n0
    pcfg = small_cfg(NETWORK__PRECISION='bf16')
    pm = M.build_model('Stereo2Point', pcfg, seed=0).cuda().pack()
    with pytest.raises(ValueError):
        pm.graphed(*args, surface=True)
    with pytest.raises(TypeError):
        pm(*args, surface=True)
    assert lib.launches() == n0


def test_driver_eval_surface():
    cfg, model = _model('bf16')
    n, bs = 3, 2
    base = T.test_voxel(cfg, model, n, bs, eval_disp=True, eval_lr=True).cpu()
    full = T.test_voxel(cfg, model, n, bs, eval_disp=True, eval_lr=True, eval_surface=True).cpu()
    assert torch.equal(full[:base.numel()], base)
    H, W, nv = cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.CONST.N_VOX
    want = 0
    for s in range(0, n, bs):
        ids = range(s, min(s + bs, n))
        pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in ids]
        gt = torch.cat([synthetic.gt_volume(1, nv, seed=100000 + i) for i in ids])
        with torch.no_grad():
            vox = model(torch.cat([p[0] for p in pairs]).cuda(), torch.cat([p[1] for p in pairs]).cuda())[2]
        want = want + surface_block(surface_stats(vox.cpu().numpy(), gt.numpy(), list(cfg.TEST.VOXEL_THRESH), FTH), nv).flatten()
    assert np.array_equal(full[base.numel():].numpy(), want)


def test_runner_prints_surface_block(monkeypatch, capsys):
    import runner
    from config import cfg as dcfg
    n, bs = 2, 2
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--batch-size', str(bs), '--n-samples', str(n), '--surface'])
    runner.main()
    res = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    cfg = dcfg.clone()
    model = M.build_model('Stereo2Voxel', cfg, seed=cfg.CONST.SEED).cuda().pack()
    old = T.test_voxel(cfg, model, n, bs, eval_disp=True).cpu()
    nh = 2 * len(cfg.TEST.VOXEL_THRESH) + 1
    assert res['iou'] == json.loads(json.dumps(T.iou_summary(old[:nh], cfg.TEST.VOXEL_THRESH)))['iou']
    full = T.test_voxel(cfg, model, n, bs, eval_disp=True, eval_surface=True).cpu()
    want = T.surface_summary(full[old.numel():], cfg.TEST.VOXEL_THRESH, cfg.TEST.FSCORE_THRESH, n)
    assert res['surface'] == json.loads(json.dumps(want))
    assert len(res['surface']['by_thresh']) == len(cfg.TEST.VOXEL_THRESH)
