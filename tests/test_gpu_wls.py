"""WLS filter on the GPU (s3d_disp_wls): maps and counters bit-exact against the numpy statement (tests/wls_oracle.py) on random
maps with NaN / +-inf holes, with and without mask and GT, fp32 and uint8 guides, several lambda and sigma, degenerate, odd
and unaligned shapes and B = 64 at 256^2; run to run identical; the counters accumulate; bad arguments rejected.  Inside both
models the WLS outputs are the op on the forward's own maps and mask, every other output is unchanged, the launch count grows
by 6, graphed() equals forward() without accumulating, micro-batches concatenate, the cloud back-projects the WLS maps, and
runner.py --test --wls --save-clouds writes those clouds."""
import ctypes
import json
import os
import sys

import numpy as np
import pytest
import torch

from stereo_3d_reconstruction_b200 import lib, models as M, ops
from stereo_3d_reconstruction_b200.utils import synthetic
from tests import cloud_oracle as CO
from tests import wls_oracle as O
from tests.common import small_cfg

pytestmark = pytest.mark.gpu

_TH = (0.5, 1.0, 3.0)
_LUTS = {}


def _lut(sigma):
    if sigma not in _LUTS:
        _LUTS[sigma] = ops.wls_weight_lut(sigma)
    return _LUTS[sigma]


def _maps(B, H, W, seed, special=True):
    """Random view-major maps [2B,H,W], smooth plus noise, with NaN / +inf / -inf holes."""
    rng = np.random.default_rng(seed)
    d = (rng.random((2 * B, H, W)) * 30).astype(np.float32)
    if special:
        sel = rng.random(d.shape)
        d[sel < 0.3] = np.nan
        d[(sel >= 0.3) & (sel < 0.33)] = np.inf
        d[(sel >= 0.33) & (sel < 0.36)] = -np.inf
    return d


def _images(B, H, W, seed, u8):
    """Blocky random guides (flat patches with edges between them), uint8 HWC or fp32 NCHW with values outside [0, 1] and NaN."""
    rng = np.random.default_rng(seed)
    c = rng.integers(0, 256, (2, B, H // 4 + 2, W // 4 + 2, 3))
    img = np.repeat(np.repeat(c, 4, 2), 4, 3)[:, :, :H, :W]
    img = np.clip(img + rng.integers(-2, 3, img.shape), 0, 255)
    if u8:
        return [x.astype(np.uint8) for x in img]
    f = (img / 255.0).astype(np.float32).transpose(0, 1, 4, 2, 3).copy()
    sel = rng.random(f.shape)
    f[sel < 0.01] = np.nan
    f[(sel >= 0.01) & (sel < 0.02)] = 1.5
    f[(sel >= 0.02) & (sel < 0.03)] = -0.5
    return list(f)


def _gt(d, B, seed):
    rng = np.random.default_rng(seed)
    H, W = d.shape[1:]
    g = (rng.random((B, 2, H, W)) * 30).astype(np.float32)
    sel = rng.random(g.shape)
    g[sel < 0.05] = np.nan
    g[(sel >= 0.05) & (sel < 0.07)] = -1.0
    g[(sel >= 0.07) & (sel < 0.09)] = 40.0
    return g


def _dev(a, offset=0):
    """A CUDA copy of numpy a; offset > 0 places it offset elements into its buffer (an unaligned data pointer)."""
    t = torch.from_numpy(np.ascontiguousarray(a))
    buf = torch.empty(t.numel() + offset, dtype=t.dtype, device='cuda')
    v = buf[offset:].view(t.shape)
    v.copy_(t)
    return v


def _same(a, b):
    """Bitwise equality of fp32 arrays (signed zeros told apart), NaN in the same places."""
    a, b = np.asarray(a, np.float32), np.asarray(b, np.float32)
    na, nb = np.isnan(a), np.isnan(b)
    return np.array_equal(na, nb) and np.array_equal(a[~na].view(np.uint32), b[~nb].view(np.uint32))


def _check(d, B, imgs, lam, sigma, mask=None, gt=None, th=_TH, max_gt=32.0, offset=0):
    lut = _lut(sigma)
    got = ops.disp_wls(_dev(d, offset), B, _dev(imgs[0], offset), _dev(imgs[1], offset), _dev(lut), lam,
                       mask=None if mask is None else _dev(mask, offset), disp_gt=None if gt is None else _dev(gt, offset),
                       thresholds=th, max_gt=None if gt is None else max_gt)
    want = O.disp_wls(d, B, imgs[0], imgs[1], lut, lam, mask, gt, th, max_gt)
    assert _same(got[0].cpu().numpy(), want[0])
    assert np.array_equal(got[1].cpu().numpy(), want[1])
    return want


@pytest.mark.parametrize('u8', [True, False])
@pytest.mark.parametrize('shape', [(1, 64, 64), (2, 33, 65), (1, 95, 130), (3, 31, 31)])
def test_random_maps_match_oracle(shape, u8):
    B, H, W = shape
    d = _maps(B, H, W, seed=H * W)
    imgs = _images(B, H, W, seed=H + W, u8=u8)
    want = _check(d, B, imgs, 8000.0, 1.5, th=())
    assert np.isfinite(want[0]).sum() > 0
    rng = np.random.default_rng(5)
    mask = rng.integers(0, 3, (B, 2, H, W)).astype(np.uint8)
    _check(d, B, imgs, 8000.0, 1.5, mask=mask, gt=_gt(d, B, 1))
    _check(d, B, imgs, 8000.0, 1.5, gt=_gt(d, B, 2))


@pytest.mark.parametrize('lam, sigma', [(1.0, 1.5), (100.0, 0.5), (8000.0, 5.0), (1e5, 20.0), (0.01, 1.5)])
def test_lambda_and_sigma(lam, sigma):
    B, H, W = 2, 40, 57
    d = _maps(B, H, W, seed=7)
    _check(d, B, _images(B, H, W, 8, u8=True), lam, sigma, gt=_gt(d, B, 3))
    _check(d, B, _images(B, H, W, 9, u8=False), lam, sigma)


@pytest.mark.parametrize('shape', [(1, 1, 1), (1, 1, 37), (2, 37, 1), (1, 1, 100), (2, 100, 1), (1, 3, 5), (2, 17, 33)])
@pytest.mark.parametrize('offset', [0, 1, 3])
def test_small_odd_and_unaligned(shape, offset):
    B, H, W = shape
    d = _maps(B, H, W, seed=H * 7 + W)
    for u8 in (True, False):
        imgs = _images(B, H, W, seed=W, u8=u8)
        _check(d, B, imgs, 8000.0, 1.5, mask=np.ones((B, 2, H, W), np.uint8), gt=_gt(d, B, 4), offset=offset)


def test_benchmark_size():
    B, H, W = 64, 256, 256
    d = _maps(B, H, W, seed=11)
    mask = (np.random.default_rng(12).random((B, 2, H, W)) < 0.2).astype(np.uint8)
    _check(d, B, _images(B, H, W, 13, u8=True), 8000.0, 1.5, mask=mask, gt=_gt(d, B, 14))


def test_runs_are_identical_and_batch_split():
    B, H, W = 8, 128, 128
    d = _dev(_maps(B, H, W, seed=31))
    imgs = [_dev(x) for x in _images(B, H, W, 32, u8=False)]
    gt = _dev(_gt(d.cpu().numpy(), B, 33))
    lut = _dev(_lut(1.5))
    a = [t.clone() for t in ops.disp_wls(d, B, *imgs, lut, 8000.0, disp_gt=gt, thresholds=_TH, max_gt=32.0)]
    for _ in range(2):
        b = ops.disp_wls(d, B, *imgs, lut, 8000.0, disp_gt=gt, thresholds=_TH, max_gt=32.0)
        assert _same(a[0].cpu(), b[0].cpu()) and torch.equal(a[1], b[1])
    h = B // 2
    half = torch.cat([d[:h], d[B:B + h]]).contiguous()
    r = ops.disp_wls(half, h, imgs[0][:h].contiguous(), imgs[1][:h].contiguous(), lut, 8000.0, disp_gt=gt[:h].contiguous(),
                     thresholds=_TH, max_gt=32.0)
    assert _same(r[0][:h].cpu(), a[0][:h].cpu()) and _same(r[0][h:].cpu(), a[0][B:B + h].cpu())
    assert torch.equal(r[1], a[1][:h])


def test_stats_accumulate_and_out_buffers():
    B, H, W = 2, 40, 40
    d = _dev(_maps(B, H, W, seed=41))
    imgs = [_dev(x) for x in _images(B, H, W, 42, u8=True)]
    out = torch.full((2 * B, H, W), 7.0, device='cuda')
    stats = torch.zeros(B, 2, 4, dtype=torch.int64, device='cuda')
    ws = torch.empty(ops.disp_wls_workspace_bytes(B, H, W), dtype=torch.uint8, device='cuda')
    assert ws.numel() == 2 * B * H * W * 16
    lut = _dev(_lut(1.5))
    n0 = lib.launches()
    ops.disp_wls(d, B, *imgs, lut, 8000.0, out=(out, stats), workspace=ws)
    assert lib.launches() - n0 == 6
    once = stats.clone()
    ops.disp_wls(d, B, *imgs, lut, 8000.0, out=(out, stats), workspace=ws)
    assert torch.equal(stats, 2 * once)
    empty = ops.disp_wls(torch.empty(0, H, W, device='cuda'), 0, imgs[0][:0], imgs[1][:0], lut, 8000.0)
    assert empty[0].shape == (0, H, W) and lib.launches() - n0 == 12


def test_bad_arguments():
    B, H, W = 2, 16, 16
    d = torch.zeros(2 * B, H, W, device='cuda')
    img = torch.zeros(B, H, W, 3, dtype=torch.uint8, device='cuda')
    out = torch.empty(2 * B, H, W, device='cuda')
    stats = torch.zeros(B, 2, 4, dtype=torch.int64, device='cuda')
    lut = _dev(_lut(1.5))
    nb = ops.disp_wls_workspace_bytes(B, H, W)
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    L = lib.load()
    s = torch.cuda.current_stream().cuda_stream
    th = (ctypes.c_float * 9)(*([1.0] * 9))

    def call(B_=B, H_=H, W_=W, lam=8000.0, gt=None, T=0, max_gt=0.0, nbytes=nb, disp=d.data_ptr(), o=out.data_ptr(),
             lt=lut.data_ptr(), w=ws.data_ptr(), u8=1):
        return L.s3d_disp_wls(disp, B_, H_, W_, img.data_ptr(), img.data_ptr(), u8, None, lt, lam, gt, th, T, max_gt, o,
                              stats.data_ptr(), w, nbytes, s)
    for kw in (dict(H_=0), dict(W_=0), dict(B_=-1), dict(B_=1 << 15), dict(lam=0.0), dict(lam=-1.0), dict(lam=float('nan')),
               dict(lam=float('inf')), dict(T=9), dict(T=-1), dict(nbytes=nb - 1), dict(gt=d.data_ptr(), max_gt=0.0),
               dict(gt=d.data_ptr(), max_gt=float('nan')), dict(disp=None), dict(o=None), dict(lt=None), dict(u8=2),
               dict(o=d.data_ptr()), dict(H_=1 << 16, W_=1 << 15), dict(w=ws.data_ptr() + 2)):
        assert call(**kw) == -1, kw
        assert L.s3d_last_error()
    assert call() == 0
    n0 = lib.launches()
    for kw in (dict(lam=0.0), dict(lam=-1.0), dict(lam=float('nan')), dict(lam=1e39), dict(lam='a'), dict(lam=True),
               dict(thresholds=[1.0] * 9), dict(disp_gt=d.view(B, 2, H, W)), dict(disp_gt=d.view(B, 2, H, W), max_gt=0.0),
               dict(mask=d.view(B, 2, H, W)), dict(mask=stats.to(torch.uint8)), dict(out=(out, stats[..., :3])),
               dict(out=(d, stats)), dict(workspace=ws[:-1]), dict(B=3), dict(B=True), dict(lut=lut[:-1]),
               dict(lut=lut.double()), dict(lut=None), dict(right=img.float())):
        args = dict(lam=8000.0, lut=lut, right=img)
        args.update(kw)
        B_ = args.pop('B', B)
        with pytest.raises(ValueError):
            ops.disp_wls(d, B_, img, args.pop('right'), args.pop('lut'), args.pop('lam'), **args)
    assert lib.launches() == n0
    for bad in (0.0, -1.0, float('nan'), float('inf'), 'a', True):
        with pytest.raises(ValueError):
            ops.wls_weight_lut(bad)


# ---- the models -----------------------------------------------------------------------------------------------------------
def _model(name='Stereo2Voxel', **kw):
    cfg = small_cfg(NETWORK__PRECISION='bf16', **kw)
    return cfg, M.build_model(name, cfg, seed=3).cuda().pack()


def _inputs(cfg, B, seed):
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=seed)
    gt = synthetic.gt_volume(B, cfg.CONST.N_VOX, seed=seed + 50)
    cam = torch.tensor([[64.0, 31.5, 31.5, 0.5, 0.0]] * B)
    return (left.cuda(), right.cuda()), gt.cuda(), synthetic.disparity_gt(d, H, W).cuda(), cam.cuda()


def _check_model_wls(cfg, args, names, out, dgt=None):
    """wls_left / wls_right / wls_stats equal the op (and the oracle) on the forward's own disp, images and mask."""
    o = dict(zip(names, out))
    B = o['disp_left'].shape[0]
    disp = torch.cat([o['disp_left'][:, 0], o['disp_right'][:, 0]]).contiguous()
    mask = o['speckle_mask'] if 'speckle_mask' in o else o.get('lr_mask')
    lam, sigma = M.wls_params(cfg)
    th = list(cfg.TEST.DISP_THRESH)
    ref = ops.disp_wls(disp, B, *args, _dev(_lut(sigma)), lam, mask=mask, disp_gt=dgt, thresholds=th,
                       max_gt=4.0 * cfg.NETWORK.MAX_DISP)
    got = torch.cat([o['wls_left'][:, 0], o['wls_right'][:, 0]])
    assert _same(ref[0].cpu(), got.cpu()) and torch.equal(ref[1], o['wls_stats'])
    want = O.disp_wls(disp.cpu().numpy(), B, args[0].cpu().numpy(), args[1].cpu().numpy(), _lut(sigma), lam,
                      None if mask is None else mask.cpu().numpy(), None if dgt is None else dgt.cpu().numpy(), th,
                      4.0 * cfg.NETWORK.MAX_DISP)
    assert _same(got.cpu(), want[0]) and np.array_equal(o['wls_stats'].cpu().numpy(), want[1])
    return o


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_model_wls_is_the_op_on_its_own_maps(name):
    cfg, model = _model(name, TEST__LR_THRESH=1000.0, TEST__SPECKLE_MAX_SIZE=20, TEST__SPECKLE_MAX_DIFF=0.25)
    args, gt, dgt, cam = _inputs(cfg, 2, seed=1)
    with torch.no_grad():
        for kw in (dict(), dict(lr_check=True), dict(disp_gt=dgt, speckle=True),
                   dict(lr_check=True, speckle=True, uncertainty=True, disp_gt=dgt)):
            on = {k: True for k in kw if k != 'disp_gt'}
            n0 = lib.launches()
            plain = [t.clone() for t in model(*args, **kw)]
            n1 = lib.launches()
            full = [t.clone() for t in model(*args, wls=True, **kw)]
            n2 = lib.launches()
            assert (n2 - n1) - (n1 - n0) == 6
            names = type(model).output_names(wls=True, disp_gt='disp_gt' in kw, **on)
            assert len(full) == len(plain) + 3 and len(names) == len(full)
            o = _check_model_wls(cfg, args, names, full, kw.get('disp_gt'))
            assert o['wls_left'].shape == o['disp_left'].shape and o['wls_right'].shape == o['disp_right'].shape
            for n, t in zip(type(model).output_names(disp_gt='disp_gt' in kw, **on), plain):
                assert torch.equal(t, o[n]), n


def test_model_launches_unchanged_without_wls():
    cfg, model = _model()
    args, gt, dgt, cam = _inputs(cfg, 2, seed=0)
    with torch.no_grad():
        counts, outs = [], []
        for kw in (dict(), dict(wls=False), dict(wls=True)):
            n0 = lib.launches()
            outs.append([t.clone() for t in model(*args, gt, disp_gt=dgt, lr_check=True, **kw)])
            counts.append(lib.launches() - n0)
    assert counts[0] == counts[1] and counts[2] == counts[0] + 6
    assert all(torch.equal(a, b) for a, b in zip(outs[0], outs[1]))


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_graphed_matches_eager_and_does_not_accumulate(name):
    cfg, model = _model(name)
    seen = []
    for seed in (0, 1):
        args, gt, dgt, cam = _inputs(cfg, 2, seed=seed)
        with torch.no_grad():
            for kw in (dict(lr_check=True, disp_gt=dgt), {}):
                eager = [t.clone() for t in model(*args, wls=True, **kw)]
                for _ in range(2):                                   # a second replay gives the same counters
                    graphed = [t.clone() for t in model.graphed(*args, wls=True, **kw)]
                    assert len(graphed) == len(eager) and all(_same(a.float().cpu(), b.float().cpu()) if a.is_floating_point()
                                                              else torch.equal(a, b) for a, b in zip(eager, graphed))
        seen.append(eager[0])
    assert not torch.equal(seen[0], seen[1])
    with torch.no_grad():
        model.graphed(*args)
    assert len(model._graphs) == 3                                   # wls is part of the graph key


def test_micro_batch_concatenates_chunks():
    cfg, model = _model(CONST__MICRO_BATCH=2)
    args, gt, dgt, cam = _inputs(cfg, 5, seed=6)
    with torch.no_grad():
        full = [t.clone() for t in model(*args, disp_gt=dgt, lr_check=True, wls=True)]
        parts = [[t.clone() for t in model(args[0][s:s + 2], args[1][s:s + 2], disp_gt=dgt[s:s + 2], lr_check=True,
                                           wls=True)] for s in range(0, 5, 2)]
    for i, t in enumerate(full):
        assert _same(t.float().cpu(), torch.cat([p[i] for p in parts]).float().cpu())
    _check_model_wls(cfg, args, M.Stereo2Voxel.output_names(disp_gt=True, lr_check=True, wls=True), full, dgt)


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_cloud_takes_the_wls_maps(name):
    cfg, model = _model(name, TEST__LR_THRESH=1000.0)
    args, gt, dgt, cam = _inputs(cfg, 2, seed=2)
    with torch.no_grad():
        for kw in (dict(), dict(lr_check=True, uncertainty=True), dict(lr_check=True, speckle=True)):
            names = type(model).output_names(wls=True, camera=True, **kw)
            o = dict(zip(names, [t.clone() for t in model(*args, wls=True, camera=cam, **kw)]))
            w = torch.cat([o['wls_left'][:, 0], o['wls_right'][:, 0]]).contiguous()
            ref = ops.disp_cloud(w, 2, *args, cam, M.cloud_min_disp(cfg))
            assert torch.equal(ref[2], o['cloud_counts'])
            for b in range(2):
                k = int(ref[2][b].sum())
                assert torch.equal(ref[0][b, :k], o['cloud_xyz'][b, :k]) and torch.equal(ref[1][b, :k], o['cloud_rgb'][b, :k])


def test_value_errors_before_any_launch():
    cfg, model = _model()
    args, gt, _, cam = _inputs(cfg, 2, seed=0)
    model(*args)
    n0 = lib.launches()
    for key, bad in (('WLS_LAMBDA', 0.0), ('WLS_LAMBDA', True), ('WLS_LAMBDA', float('nan')), ('WLS_SIGMA', -1.0),
                     ('WLS_SIGMA', 'a'), ('WLS_SIGMA', float('inf'))):
        old = cfg.TEST[key]
        cfg.TEST[key] = bad
        with pytest.raises(ValueError, match=key):
            model(*args, wls=True)
        with pytest.raises(ValueError, match=key):
            model.graphed(*args, wls=True)
        cfg.TEST[key] = old
    assert lib.launches() == n0


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_runner_wls_with_clouds(name, monkeypatch, capsys, tmp_path):
    import runner
    from config import cfg as dcfg
    n, bs = 3, 2
    out_dir = str(tmp_path / 'clouds')
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--model', name, '--batch-size', str(bs), '--n-samples', str(n),
                                      '--wls', '--save-clouds', out_dir])
    runner.main()
    res = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    cfg = dcfg.clone()
    lam, sigma = M.wls_params(cfg)
    assert res['wls']['lambda'] == lam and res['wls']['sigma'] == sigma and res['wls']['confidence'] == 'finite'
    assert res['cloud']['wls'] == {'lambda': lam, 'sigma': sigma}
    model = M.build_model(name, cfg, seed=cfg.CONST.SEED).cuda().pack()
    H, W, T = cfg.CONST.IMG_H, cfg.CONST.IMG_W, len(cfg.TEST.DISP_THRESH)
    cam = torch.tensor([M.camera_values(cfg)], device='cuda')
    tot = torch.zeros(2, 4 + T, dtype=torch.int64)
    for s in range(0, n, bs):
        ids = list(range(s, min(s + bs, n)))
        pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in ids]
        left, right = torch.cat([p[0] for p in pairs]).cuda(), torch.cat([p[1] for p in pairs]).cuda()
        dgt = torch.cat([synthetic.disparity_gt(p[2], H, W) for p in pairs]).cuda()
        with torch.no_grad():
            o = dict(zip(type(model).output_names(disp_gt=True, wls=True, camera=True),
                         model(left, right, disp_gt=dgt, wls=True, camera=cam.repeat(len(ids), 1))))
        tot += o['wls_stats'].sum(0).cpu()
        xyz, c = o['cloud_xyz'].cpu().numpy(), o['cloud_counts'].cpu().numpy()
        for b, i in enumerate(ids):
            k = int(c[b].sum())
            rec = CO.read_ply(os.path.join(out_dir, '%06d.ply' % i))
            assert len(rec) == k
            assert np.array_equal(np.stack([rec['x'], rec['y'], rec['z']], 1).view(np.uint32), xyz[b, :k].view(np.uint32))
            assert len(CO.read_ply(os.path.join(out_dir, '%06d_gt.ply' % i))) > 0
    for v, view in enumerate(('left', 'right')):
        r = res['wls'][view]
        assert r['n_finite'] == tot[v, 0] and r['n_valid_finite'] == tot[v, 1]
        assert r['filled'] == tot[v, 0] - tot[v, 3 + T]
