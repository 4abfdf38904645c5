"""Stereo point clouds on the GPU (s3d_disp_cloud): bit-exact against the numpy statement (tests/cloud_oracle.py) for fp32 and
uint8 images, every filter, odd and unaligned sizes, non-finite disparities and the all-rejected / all-kept edges; rows past
the counts stay untouched.  Inside both models the cloud is the op applied to the forward's own maps, every other output is
unchanged, graphed() equals forward(), micro-batches concatenate, and runner.py --test --save-clouds writes the same points."""
import json
import os
import sys

import numpy as np
import pytest
import torch

from stereo_3d_reconstruction_b200 import lib, models as M, ops
from stereo_3d_reconstruction_b200.utils import synthetic
from tests import cloud_oracle as O
from tests.common import small_cfg

pytestmark = pytest.mark.gpu

_POISON = -7.0


def _camera(B, seed, doffs=True):
    rng = np.random.default_rng(seed)
    cam = np.stack([rng.uniform(50, 400, B), rng.uniform(-5, 40, B), rng.uniform(-5, 40, B), rng.uniform(0.05, 2.0, B),
                    rng.uniform(-3, 3, B) if doffs else np.zeros(B)], 1).astype(np.float32)
    return cam


def _disp(B, H, W, seed, special=True):
    rng = np.random.default_rng(seed)
    d = rng.uniform(-4, 40, (2 * B, H, W)).astype(np.float32)
    if special:
        sel = rng.random(d.shape)
        d[sel < 0.05] = np.nan
        d[(sel >= 0.05) & (sel < 0.08)] = np.inf
        d[(sel >= 0.08) & (sel < 0.11)] = -np.inf
        d[(sel >= 0.11) & (sel < 0.14)] = 0.0
    return d


def _images(B, H, W, seed, u8):
    rng = np.random.default_rng(seed)
    if u8:
        return [rng.integers(0, 256, (B, H, W, 3), dtype=np.uint8) for _ in range(2)]
    out = []
    for _ in range(2):
        x = rng.uniform(-0.2, 1.2, (B, 3, H, W)).astype(np.float32)
        sel = rng.random(x.shape)
        x[sel < 0.02] = np.nan
        x[(sel >= 0.02) & (sel < 0.03)] = np.inf
        x[(sel >= 0.03) & (sel < 0.05)] = 0.5                      # 127.5: half to even
        out.append(x)
    return out


def _filters(B, H, W, seed, which):
    rng = np.random.default_rng(seed)
    mask = std = None
    if which in ('lr', 'both'):
        mask = (rng.random((B, 2, H, W)) < 0.7).astype(np.uint8)
        mask[rng.random(mask.shape) < 0.02] = 2                    # only 1 keeps
    if which in ('std', 'both'):
        std = rng.uniform(0, 4, (B, 2, H, W)).astype(np.float32)
        std[rng.random(std.shape) < 0.03] = np.nan
        std[rng.random(std.shape) < 0.02] = 2.0                    # == max_std: kept
    return mask, std


def _cuda(a, offset=0):
    """a as a CUDA tensor; offset > 0: a view that starts `offset` elements into its storage (an unaligned pointer)."""
    if a is None:
        return None
    t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
    if not offset:
        return t
    buf = torch.empty(t.numel() + offset, dtype=t.dtype, device='cuda')
    v = buf[offset:].view(t.shape)
    v.copy_(t)
    return v


def _run(disp, B, left, right, cam, min_disp, mask=None, std=None, max_std=2.0, u8=False, offset=0):
    H, W = disp.shape[1:]
    out = (torch.full((B, 2 * H * W, 3), _POISON, device='cuda'), torch.full((B, 2 * H * W, 3), 77, dtype=torch.uint8,
                                                                            device='cuda'),
           torch.full((B, 2), -7, dtype=torch.int32, device='cuda'))
    n0 = lib.launches()
    got = ops.disp_cloud(_cuda(disp, offset), B, _cuda(left), _cuda(right), _cuda(cam), min_disp, lr_mask=_cuda(mask, offset),
                         disp_std=_cuda(std, offset), max_std=max_std if std is not None else None, out=out)
    assert lib.launches() - n0 == (2 if B else 0)
    assert all(a is b for a, b in zip(got, out))
    xyz, rgb, c = (o.cpu().numpy() for o in out)
    want = O.disp_cloud(disp, B, left, right, cam, min_disp, mask, std, max_std, u8)
    for b, (wx, wc, n) in enumerate(want):
        assert tuple(c[b]) == n, b
        k = n[0] + n[1]
        assert np.array_equal(xyz[b, :k].view(np.uint32), wx.view(np.uint32)), b
        assert np.array_equal(rgb[b, :k], wc), b
        assert (xyz[b, k:] == _POISON).all() and (rgb[b, k:] == 77).all(), b     # rows past the counts are not written
    return want


@pytest.mark.parametrize('u8', [False, True])
@pytest.mark.parametrize('which', ['none', 'lr', 'std', 'both'])
@pytest.mark.parametrize('B,H,W', [(2, 7, 13), (3, 5, 36), (1, 9, 130), (2, 3, 1031), (1, 256, 256)])
def test_random_maps_match_oracle(B, H, W, which, u8):
    seed = B * 1000 + H * 10 + W
    d = _disp(B, H, W, seed)
    left, right = _images(B, H, W, seed + 1, u8)
    mask, std = _filters(B, H, W, seed + 2, which)
    _run(d, B, left, right, _camera(B, seed + 3), 1.5, mask, std, 2.0, u8)


@pytest.mark.parametrize('which', ['none', 'both'])
@pytest.mark.parametrize('u8', [False, True])
def test_batch_64_full_size(which, u8):
    B, H, W = 64, 256, 256
    d = _disp(B, H, W, 11)
    left, right = _images(B, H, W, 12, u8)
    mask, std = _filters(B, H, W, 13, which)
    _run(d, B, left, right, _camera(B, 14), 1.0, mask, std, 2.0, u8)


@pytest.mark.parametrize('which', ['none', 'both'])
def test_unaligned_pointers(which):
    B, H, W = 2, 6, 40                                              # W % 4 == 0 but the maps start off a 16-byte boundary
    d = _disp(B, H, W, 21)
    left, right = _images(B, H, W, 22, False)
    mask, std = _filters(B, H, W, 23, which)
    _run(d, B, left, right, _camera(B, 24), 1.0, mask, std, 2.0, False, offset=1)


def test_all_rejected_and_all_kept():
    B, H, W = 3, 8, 24
    left, right = _images(B, H, W, 31, False)
    cam = _camera(B, 32, doffs=False)
    want = _run(np.full((2 * B, H, W), np.nan, np.float32), B, left, right, cam, 1.0)
    assert all(n == (0, 0) for _, _, n in want)
    want = _run(np.full((2 * B, H, W), 0.5, np.float32), B, left, right, cam, 1.0)     # below min_disp
    assert all(n == (0, 0) for _, _, n in want)
    want = _run(np.full((2 * B, H, W), 4.0, np.float32), B, left, right, cam, 1.0)
    assert all(n == (H * W, H * W) for _, _, n in want)
    mask = np.ones((B, 2, H, W), np.uint8)
    std = np.zeros((B, 2, H, W), np.float32)
    want = _run(_disp(B, H, W, 33, special=False) + 50, B, left, right, cam, 1.0, mask, std, 0.0)
    assert all(n == (H * W, H * W) for _, _, n in want)
    want = _run(np.full((2 * B, H, W), 4.0, np.float32), B, left, right, cam, 1.0, mask * 0, std)
    assert all(n == (0, 0) for _, _, n in want)


def test_counts_do_not_depend_on_the_batch():
    B, H, W = 5, 16, 20
    d = _disp(B, H, W, 41)
    left, right = _images(B, H, W, 42, True)
    cam = _camera(B, 43)
    full = ops.disp_cloud(_cuda(d), B, _cuda(left), _cuda(right), _cuda(cam), 1.0)
    for b in range(B):
        one = ops.disp_cloud(_cuda(d[[b, B + b]]), 1, _cuda(left[b:b + 1]), _cuda(right[b:b + 1]), _cuda(cam[b:b + 1]), 1.0)
        k = int(one[2].sum())
        assert torch.equal(one[2][0], full[2][b])
        assert torch.equal(one[0][0, :k], full[0][b, :k]) and torch.equal(one[1][0, :k], full[1][b, :k])


def test_bad_arguments_rejected_before_any_launch():
    B, H, W = 2, 4, 8
    d, cam = _cuda(_disp(B, H, W, 51)), _cuda(_camera(B, 52))
    left, right = (_cuda(x) for x in _images(B, H, W, 53, False))
    n0 = lib.launches()
    bad = [dict(disp=d[:3]), dict(B=3), dict(left=left.to(torch.uint8)), dict(camera=cam[:1]), dict(camera=cam.double()),
           dict(min_disp=0.0), dict(min_disp=float('nan')), dict(min_disp=1e-50), dict(lr_mask=torch.ones(B, 2, H, W, device='cuda')),
           dict(disp_std=torch.zeros(B, 2, H, W, device='cuda')), dict(disp_std=torch.zeros(B, 2, H, W, device='cuda'), max_std=-1.0),
           dict(disp_std=torch.zeros(B, 2, H, W, device='cuda'), max_std=float('inf')),
           dict(workspace=torch.empty(ops.disp_cloud_workspace_bytes(B, H) - 1, dtype=torch.uint8, device='cuda')),
           dict(out=(torch.empty(B, 2 * H * W, 3, device='cuda'),) * 3)]
    for kw in bad:
        args = dict(disp=d, B=B, left=left, right=right, camera=cam, min_disp=1.0)
        args.update(kw)
        with pytest.raises(ValueError):
            ops.disp_cloud(**args)
    assert lib.launches() == n0
    # the C entry point checks on its own
    L = lib.load()
    xyz = torch.empty(B, 2 * H * W, 3, device='cuda')
    rgb = torch.empty(B, 2 * H * W, 3, dtype=torch.uint8, device='cuda')
    cnt = torch.empty(B, 2, dtype=torch.int32, device='cuda')
    nb = ops.disp_cloud_workspace_bytes(B, H)
    assert nb == B * 2 * H * 4
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    s = torch.cuda.current_stream().cuda_stream

    def call(H_=H, W_=W, u8=0, min_disp=1.0, std=None, max_std=0.0, nbytes=nb, disp=d.data_ptr()):
        return L.s3d_disp_cloud(disp, B, H_, W_, left.data_ptr(), right.data_ptr(), u8, None, std, max_std, cam.data_ptr(),
                                min_disp, xyz.data_ptr(), rgb.data_ptr(), cnt.data_ptr(), ws.data_ptr(), nbytes, s)
    for kw in (dict(H_=0), dict(W_=0), dict(u8=2), dict(min_disp=0.0), dict(min_disp=float('inf')), dict(nbytes=nb - 1),
               dict(std=d.data_ptr(), max_std=float('nan')), dict(disp=None), dict(H_=1 << 16, W_=1 << 15)):
        assert call(**kw) == -1, kw
        assert L.s3d_last_error()
    assert call() == 0
    torch.cuda.synchronize()
    assert L.s3d_disp_cloud(d.data_ptr(), 0, H, W, left.data_ptr(), right.data_ptr(), 0, None, None, 0.0, cam.data_ptr(), 1.0,
                            xyz.data_ptr(), rgb.data_ptr(), cnt.data_ptr(), None, 0, s) == 0


# ---- the models -----------------------------------------------------------------------------------------------------------
def _model(name='Stereo2Voxel', prec='bf16', **kw):
    cfg = small_cfg(NETWORK__PRECISION=prec, **kw)
    return cfg, M.build_model(name, cfg, seed=3).cuda().pack()


def _inputs(cfg, B, seed, u8=False):
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=seed)
    if u8:
        left, right = ((x * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous() for x in (left, right))
    gt = synthetic.gt_volume(B, cfg.CONST.N_VOX, seed=seed + 50)
    cam = torch.tensor(_camera(B, seed + 60, doffs=False))
    cam[:, 1:3] = 31.5                                              # a 64 x 64 image's centre
    return (left.cuda(), right.cuda()), gt.cuda(), synthetic.disparity_gt(d, H, W).cuda(), cam.cuda()


def _check_model_cloud(cfg, names, out, left, right, cam):
    """The forward's cloud equals the op applied to its own disp_left / disp_right, lr_mask and disp_std."""
    o = dict(zip(names, out))
    B = left.shape[0]
    disp = torch.cat([o['disp_left'][:, 0], o['disp_right'][:, 0]]).contiguous()
    std = o.get('disp_std')
    ref = ops.disp_cloud(disp, B, left, right, cam, M.cloud_min_disp(cfg), lr_mask=o.get('lr_mask'), disp_std=std,
                         max_std=None if std is None else M.cloud_max_std(cfg))
    assert torch.equal(ref[2], o['cloud_counts'])
    for b in range(B):
        k = int(ref[2][b].sum())
        assert torch.equal(ref[0][b, :k], o['cloud_xyz'][b, :k]) and torch.equal(ref[1][b, :k], o['cloud_rgb'][b, :k])
    # and the oracle on the same maps
    want = O.disp_cloud(disp.cpu().numpy(), B, left.cpu().numpy(), right.cpu().numpy(), cam.cpu().numpy(),
                        M.cloud_min_disp(cfg), None if o.get('lr_mask') is None else o['lr_mask'].cpu().numpy(),
                        None if std is None else std.cpu().numpy(), M.cloud_max_std(cfg), left.dtype == torch.uint8)
    for b, (wx, _, n) in enumerate(want):
        assert tuple(o['cloud_counts'][b].tolist()) == n
        assert np.array_equal(o['cloud_xyz'][b, :len(wx)].cpu().numpy().view(np.uint32), wx.view(np.uint32))
    return o


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
@pytest.mark.parametrize('u8', [False, True])
def test_model_cloud_is_the_op_on_its_own_maps(name, u8):
    # the synthetic weights' maps are not left-right consistent: a wide tolerance keeps the pixels whose match lies in the
    # image, and the spread threshold is set to the median spread, so that both filters keep some pixels and drop others
    cfg, model = _model(name, TEST__LR_THRESH=1000.0)
    args, gt, dgt, cam = _inputs(cfg, 2, seed=1, u8=u8)
    with torch.no_grad():
        for kw in (dict(), dict(lr_check=True), dict(uncertainty=True), dict(lr_check=True, uncertainty=True, disp_gt=dgt)):
            n0 = lib.launches()
            plain = [t.clone() for t in model(*args, **kw)]
            n1 = lib.launches()
            if 'uncertainty' in kw:
                std = dict(zip(type(model).output_names(**{k: True for k in kw}), plain))['disp_std']
                cfg.TEST.CLOUD_MAX_STD = float(std[torch.isfinite(std)].median())
            full = [t.clone() for t in model(*args, camera=cam, **kw)]
            n2 = lib.launches()
            assert (n2 - n1) - (n1 - n0) == 2                       # cloud_count_kernel + cloud_write_kernel
            names = type(model).output_names(camera=True, **{k: True for k in kw})
            assert len(full) == len(plain) + 3 and len(names) == len(full)
            o = _check_model_cloud(cfg, names, full, *args, cam)
            for n, t in zip(type(model).output_names(**{k: True for k in kw}), plain):
                assert torch.equal(t, o[n]), n
            kept = int(o['cloud_counts'].sum())
            assert 0 < kept < 2 * 2 * cfg.CONST.IMG_H * cfg.CONST.IMG_W if kw else kept > 0


def test_model_launches_unchanged_without_camera():
    cfg, model = _model()
    args, gt, dgt, cam = _inputs(cfg, 2, seed=0)
    with torch.no_grad():
        counts = []
        for kw in (dict(), dict(camera=None), dict(camera=cam)):
            n0 = lib.launches()
            model(*args, gt, disp_gt=dgt, **kw)
            counts.append(lib.launches() - n0)
    assert counts[0] == counts[1] and counts[2] == counts[0] + 2


def test_model_every_option():
    cfg, model = _model()
    args, gt, dgt, cam = _inputs(cfg, 2, seed=4)
    kw = dict(disp_gt=dgt, lr_check=True, uncertainty=True, surface=True, mesh=True, curves=True, fscore_curves=True)
    with torch.no_grad():
        base = [t.clone() for t in model(*args, gt, **kw)]
        full = [t.clone() for t in model(*args, gt, camera=cam, **kw)]
    names = M.Stereo2Voxel.output_names(gt=True, camera=True, **{k: True for k in kw if k != 'disp_gt'}, disp_gt=True)
    o = _check_model_cloud(cfg, names, full, *args, cam)
    for n, t in zip(M.Stereo2Voxel.output_names(gt=True, **{k: True for k in kw if k != 'disp_gt'}, disp_gt=True), base):
        if n.startswith('mesh_'):
            continue                                                # rows past the counts are not written
        assert torch.equal(t, o[n]), n


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_graphed_matches_eager(name):
    cfg, model = _model(name)
    seen = []
    for seed in (0, 1):
        args, gt, dgt, cam = _inputs(cfg, 2, seed=seed)
        with torch.no_grad():
            for kw in (dict(lr_check=True, uncertainty=True), {}):
                eager = [t.clone() for t in model(*args, camera=cam, **kw)]
                graphed = [t.clone() for t in model.graphed(*args, camera=cam, **kw)]
                assert len(graphed) == len(eager)
                c = eager[-1]
                for i, (a, b) in enumerate(zip(eager, graphed)):
                    if i in (len(eager) - 3, len(eager) - 2):       # compare the clouds up to the counts
                        for s in range(2):
                            k = int(c[s].sum())
                            assert torch.equal(a[s, :k], b[s, :k])
                    else:
                        assert torch.equal(a, b)
        seen.append(eager[-3])
    assert not torch.equal(seen[0], seen[1])
    with torch.no_grad():
        assert len(model.graphed(*args)) == 3
    assert len(model._graphs) == 3                                  # the camera is part of the graph key


def test_micro_batch_concatenates_chunks():
    cfg, model = _model(CONST__MICRO_BATCH=2)
    args, gt, dgt, cam = _inputs(cfg, 5, seed=6)
    with torch.no_grad():
        full = [t.clone() for t in model(*args, uncertainty=True, camera=cam)]
        parts = [[t.clone() for t in model(args[0][s:s + 2], args[1][s:s + 2], uncertainty=True, camera=cam[s:s + 2])]
                 for s in range(0, 5, 2)]
    for i, t in enumerate(full[:-3]):
        assert torch.equal(t, torch.cat([p[i] for p in parts]))
    c = torch.cat([p[-1] for p in parts])
    assert torch.equal(full[-1], c)
    for b in range(5):
        k, p = int(c[b].sum()), parts[b // 2]
        assert torch.equal(full[-3][b, :k], p[-3][b % 2, :k]) and torch.equal(full[-2][b, :k], p[-2][b % 2, :k])
    _check_model_cloud(cfg, M.Stereo2Voxel.output_names(uncertainty=True, camera=True), full, *args, cam)


def test_value_errors_before_any_launch():
    cfg, model = _model()
    args, gt, _, cam = _inputs(cfg, 2, seed=0)
    model(*args)
    n0 = lib.launches()
    for bad in (cam[:1], cam.double(), cam.cpu(), cam[:, :4].contiguous(), [1.0, 2.0, 3.0, 4.0, 5.0]):
        with pytest.raises(ValueError, match='camera'):
            model(*args, camera=bad)
        with pytest.raises(ValueError, match='camera'):
            model.graphed(*args, camera=bad)
    cfg.TEST.CLOUD_MIN_DISP = 0.0
    with pytest.raises(ValueError, match='CLOUD_MIN_DISP'):
        model(*args, camera=cam)
    cfg.TEST.CLOUD_MIN_DISP = 1.0
    cfg.TEST.CLOUD_MAX_STD = float('nan')
    with pytest.raises(ValueError, match='CLOUD_MAX_STD'):
        model.graphed(*args, uncertainty=True, camera=cam)
    assert lib.launches() == n0
    with torch.no_grad():
        model(*args, camera=cam)                                    # the spread threshold only matters with uncertainty=True


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_runner_save_clouds(name, monkeypatch, capsys, tmp_path):
    import runner
    from config import cfg as dcfg
    n, bs = 3, 2
    out_dir = str(tmp_path / 'clouds')
    cam = [200.0, 128.0, 120.0, 0.25, 0.5]
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--model', name, '--batch-size', str(bs), '--n-samples', str(n),
                                      '--lr-check', '--save-clouds', out_dir, '--camera', ','.join(map(str, cam))])
    runner.main()
    res = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    assert sorted(os.listdir(out_dir)) == sorted(['%06d.ply' % i for i in range(n)] + ['%06d_gt.ply' % i for i in range(n)])
    cfg = dcfg.clone()
    model = M.build_model(name, cfg, seed=cfg.CONST.SEED).cuda().pack()
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    tot = np.zeros(2, np.int64)
    for s in range(0, n, bs):
        ids = list(range(s, min(s + bs, n)))
        pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in ids]
        left, right = torch.cat([p[0] for p in pairs]).cuda(), torch.cat([p[1] for p in pairs]).cuda()
        camera = torch.tensor([cam] * len(ids), device='cuda')
        with torch.no_grad():
            out = model(left, right, lr_check=True, camera=camera)
        xyz, rgb, c = (t.cpu().numpy() for t in out[-3:])
        dgt = torch.cat([synthetic.disparity_gt(p[2], H, W) for p in pairs]).numpy()
        gwant = O.disp_cloud(dgt.transpose(1, 0, 2, 3).reshape(2 * len(ids), H, W), len(ids), left.cpu().numpy(),
                             right.cpu().numpy(), np.asarray([cam] * len(ids), np.float32), 1.0)
        for b, i in enumerate(ids):
            k = int(c[b].sum())
            tot += c[b]
            rec = O.read_ply(os.path.join(out_dir, '%06d.ply' % i))
            assert len(rec) == k
            got = np.stack([rec['x'], rec['y'], rec['z']], 1)
            assert np.array_equal(got.view(np.uint32), xyz[b, :k].view(np.uint32))
            assert np.array_equal(np.stack([rec['red'], rec['green'], rec['blue']], 1), rgb[b, :k])
            g = O.read_ply(os.path.join(out_dir, '%06d_gt.ply' % i))
            gx, gc, gn = gwant[b]
            assert len(g) == sum(gn) > 0
            assert np.array_equal(np.stack([g['x'], g['y'], g['z']], 1).view(np.uint32), gx.view(np.uint32))
            assert np.array_equal(np.stack([g['red'], g['green'], g['blue']], 1), gc)
    assert res['cloud']['left']['n_points'] == tot[0] and res['cloud']['right']['n_points'] == tot[1]
    assert res['cloud']['camera'] == cam and res['cloud']['n_samples'] == n
