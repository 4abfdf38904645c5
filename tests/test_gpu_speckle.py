"""Speckle filter on the GPU (s3d_speckle_filter): mask and counters bit-exact against the numpy / scipy statement
(tests/speckle_oracle.py) on random maps at several max_diff, non-finite values, LR masks holding 0 / 1 / 2, the constant,
isolated-pixel and serpentine maps, stripes and regions on tile borders, degenerate, odd and unaligned shapes and B = 64 at
256^2, with and without GT; equal to cv2.filterSpeckles on 1/16-px maps; run to run identical; bad arguments rejected.
Inside both models the speckle outputs are the op on the forward's own maps, every other output is unchanged, graphed()
equals forward() without accumulating, micro-batches concatenate, the cloud takes the speckle mask, max_size 0 reproduces the
LR check, and runner.py --test --speckle writes the filtered clouds."""
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
from tests import speckle_oracle as O
from tests.common import small_cfg

pytestmark = pytest.mark.gpu

_TH = (0.5, 1.0, 3.0)


def _maps(B, H, W, seed, levels=24, step=0.125, special=True):
    """Random view-major maps [2B,H,W] with values on a coarse grid (so that equal and near neighbours form regions of every
    size) and, with special, NaN / +inf / -inf holes."""
    rng = np.random.default_rng(seed)
    # blocky values: a coarse random field upsampled, plus per-pixel jitter, gives regions from 1 px to large
    c = rng.integers(0, levels, (2 * B, H // 4 + 2, W // 4 + 2))
    d = np.repeat(np.repeat(c, 4, 1), 4, 2)[:, :H, :W].astype(np.float32) * np.float32(step)
    d += (rng.random(d.shape) < 0.15).astype(np.float32) * np.float32(step) * rng.integers(-3, 4, d.shape).astype(np.float32)
    if special:
        sel = rng.random(d.shape)
        d[sel < 0.05] = np.nan
        d[(sel >= 0.05) & (sel < 0.07)] = np.inf
        d[(sel >= 0.07) & (sel < 0.09)] = -np.inf
    return d


def _gt(d, B, seed):
    """GT [B,2,H,W] near the maps, with invalid pixels (NaN, negative, >= max_gt)."""
    rng = np.random.default_rng(seed)
    H, W = d.shape[1:]
    g = np.nan_to_num(d.reshape(2, B, H, W).transpose(1, 0, 2, 3), nan=1.0, posinf=2.0, neginf=0.5)
    g = (g + rng.normal(0, 1.5, g.shape)).astype(np.float32)
    sel = rng.random(g.shape)
    g[sel < 0.05] = np.nan
    g[(sel >= 0.05) & (sel < 0.07)] = -1.0
    g[(sel >= 0.07) & (sel < 0.09)] = 40.0
    return g


def _dev(a, offset=0, dtype=None):
    """A CUDA copy of numpy a; offset > 0 places it offset elements into its buffer (an unaligned data pointer)."""
    t = torch.from_numpy(np.ascontiguousarray(a))
    buf = torch.empty(t.numel() + offset, dtype=t.dtype, device='cuda')
    v = buf[offset:].view(t.shape)
    v.copy_(t)
    return v


def _check(d, B, max_size, max_diff, lr=None, gt=None, th=_TH, max_gt=32.0, offset=0):
    H, W = d.shape[1:]
    got = ops.speckle_filter(_dev(d, offset), B, max_size, max_diff, lr_mask=None if lr is None else _dev(lr, offset),
                             disp_gt=None if gt is None else _dev(gt, offset), thresholds=th,
                             max_gt=None if gt is None else max_gt)
    want = O.speckle_filter(d, B, max_size, max_diff, lr, gt, th, max_gt)
    assert np.array_equal(got[0].cpu().numpy(), want[0])
    assert np.array_equal(got[1].cpu().numpy(), want[1])
    return want


@pytest.mark.parametrize('max_diff', [0.0, 0.125, 0.5, 1.0, 3.0])
@pytest.mark.parametrize('shape', [(1, 64, 64), (2, 33, 65), (1, 95, 130), (3, 31, 31)])
def test_random_maps_match_oracle(shape, max_diff):
    B, H, W = shape
    d = _maps(B, H, W, seed=H * W + int(8 * max_diff))
    for max_size in (0, 1, 7, 40):
        want = _check(d, B, max_size, max_diff, th=())
        if max_size == 7:
            assert want[0].sum() > 0 and (max_diff > 1 or want[1][..., 3].sum() > 0)     # kept pixels and speckles
    _check(d, B, 7, max_diff, gt=_gt(d, B, 1))


def test_lr_mask_values_and_gt():
    B, H, W = 2, 48, 70
    d = _maps(B, H, W, seed=5)
    rng = np.random.default_rng(6)
    lr = rng.choice(np.array([0, 1, 1, 1, 2], np.uint8), (B, 2, H, W))    # only 1 is a candidate
    for max_size in (0, 3, 20):
        _check(d, B, max_size, 0.25, lr=lr, gt=_gt(d, B, 7))
        _check(d, B, max_size, 0.25, lr=lr)


def _serpentine(H, W):
    d = np.full((H, W), np.nan, np.float32)
    d[0::2] = 3.0
    for y in range(1, H, 2):
        d[y, W - 1 if (y // 2) % 2 == 0 else 0] = 3.0
    return d


@pytest.mark.parametrize('H, W', [(64, 64), (70, 97), (256, 256)])
def test_structured_maps(H, W):
    y, x = np.mgrid[:H, :W]
    cases = {
        'constant': np.full((H, W), 7.0, np.float32),
        'isolated': ((x + y) % 2 * 3.0).astype(np.float32),
        'serpentine': _serpentine(H, W),
        'vertical_stripes': (x // 3 % 2 * 5.0).astype(np.float32),
        'stripes_on_tile_borders': np.where((x % 32 == 31) | (x % 32 == 0) | (y % 32 == 0), 1.0, 9.0).astype(np.float32),
        # 2 x 2 squares astride the tile corners, isolated by NaN: regions of exactly 4 px split over four tiles
        'tile_corner_squares': np.where(((x % 32 == 31) | (x % 32 == 0)) & ((y % 32 == 31) | (y % 32 == 0)), 2.0,
                                        np.nan).astype(np.float32),
        'ramp': (x * 0.5 + y * 0.25).astype(np.float32),
    }
    for name, m in cases.items():
        d = np.stack([m, m[::-1, ::-1].copy()])                            # B = 1: view 0, view 1
        for max_size in (0, 3, 4, 5, H * W - 1, H * W):
            want = _check(d, 1, max_size, 1.0, th=())
            if name == 'constant':
                assert want[1][0, :, 3].tolist() == ([1, 1] if max_size >= H * W else [0, 0])
            if name == 'serpentine':
                n = int(np.isfinite(m).sum())
                assert want[1][0, 0, 0] == (n if max_size < n else 0)       # one region
            if name == 'isolated':
                assert want[1][0, 0, 3] == (H * W if max_size >= 1 else 0)


def test_regions_of_exactly_max_size():
    H, W = 40, 72
    d = np.full((H, W), np.nan, np.float32)
    d[3, 29:34] = 1.0                                                      # 5 px across a vertical tile border
    d[30:33, 10] = 2.0
    d[33:35, 10] = 2.5                                                     # 5 px across a horizontal one, steps of 0.5
    d[10, 50:56] = 4.0                                                     # 6 px
    m = np.stack([d, d])
    for max_size, kept in ((4, 16), (5, 6), (6, 0)):
        want = _check(m, 1, max_size, 0.5, th=())
        assert want[1][0, 0, 0] == kept
    want = _check(m, 1, 5, 0.25, th=())                                        # the 0.5 step splits the column: 3 + 2
    assert want[1][0, 0, 3] == 3


@pytest.mark.parametrize('shape', [(1, 1, 1), (1, 1, 37), (2, 37, 1), (1, 1, 100), (2, 100, 1), (1, 3, 5), (2, 17, 33)])
@pytest.mark.parametrize('offset', [0, 1, 3])
def test_small_odd_and_unaligned(shape, offset):
    B, H, W = shape
    d = _maps(B, H, W, seed=H + 7 * W + offset, levels=4)
    lr = np.random.default_rng(offset).integers(0, 3, (B, 2, H, W)).astype(np.uint8)
    for max_size in (0, 2, 5):
        _check(d, B, max_size, 0.125, lr=lr, gt=_gt(d, B, 2), offset=offset)
        _check(d, B, max_size, 0.125, offset=offset)


def test_benchmark_size_with_gt_and_lr():
    B, H, W = 64, 256, 256
    d = _maps(B, H, W, seed=11, levels=48)
    lr = (np.random.default_rng(12).random((B, 2, H, W)) < 0.9).astype(np.uint8)
    want = _check(d, B, 100, 1.0, lr=lr, gt=_gt(d, B, 13), th=(1.0, 3.0), max_gt=32.0)
    assert 0 < want[0].sum() < d.size and want[1][..., 5].sum() > 0


def test_equals_cv2_filter_speckles():
    cv2 = pytest.importorskip('cv2')
    rng = np.random.default_rng(21)
    for it in range(12):
        H, W = (int(v) for v in rng.integers(1, 90, 2))
        d = (rng.integers(-60, 60, (2, H, W)) // 4 * 4 / 16).astype(np.float32)     # multiples of 1/4 on a 1/16 grid
        d[rng.random(d.shape) < 0.1] = np.nan
        max_size, md16 = int(rng.integers(0, 30)), int(rng.integers(0, 20))
        mask, _ = ops.speckle_filter(_dev(d), 1, max_size, md16 / 16)
        for v in range(2):
            img = np.where(np.isfinite(d[v]), np.nan_to_num(d[v]) * 16, -32768).astype(np.int16)
            ref, _ = cv2.filterSpeckles(img, -32768, max_size, md16)
            assert np.array_equal(mask[0, v].cpu().numpy(), (ref != -32768).astype(np.uint8)), (it, v)


def test_runs_are_identical():
    B, H, W = 8, 256, 256
    d = _dev(_maps(B, H, W, seed=31, levels=8))
    d[:, ::2, :] = 2.0                                                     # big regions with many concurrent unions
    gt = _dev(_gt(d.cpu().numpy(), B, 32))
    a = [t.clone() for t in ops.speckle_filter(d, B, 50, 0.5, disp_gt=gt, thresholds=_TH, max_gt=32.0)]
    for _ in range(3):
        b = ops.speckle_filter(d, B, 50, 0.5, disp_gt=gt, thresholds=_TH, max_gt=32.0)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    # the batch split does not matter: each half alone gives its rows
    half = torch.cat([d[:B // 2], d[B:B + B // 2]]).contiguous()
    h = ops.speckle_filter(half, B // 2, 50, 0.5, disp_gt=gt[:B // 2].contiguous(), thresholds=_TH, max_gt=32.0)
    assert torch.equal(h[0], a[0][:B // 2]) and torch.equal(h[1], a[1][:B // 2])


def test_stats_accumulate_and_out_buffers():
    B, H, W = 2, 40, 40
    d = _dev(_maps(B, H, W, seed=41))
    mask = torch.full((B, 2, H, W), 9, dtype=torch.uint8, device='cuda')
    stats = torch.zeros(B, 2, 5, dtype=torch.int64, device='cuda')
    ws = torch.empty(ops.speckle_filter_workspace_bytes(B, H, W), dtype=torch.uint8, device='cuda')
    assert ws.numel() == 2 * B * H * W * 8
    n0 = lib.launches()
    ops.speckle_filter(d, B, 3, 0.25, out=(mask, stats), workspace=ws)
    assert lib.launches() - n0 == 4
    once = stats.clone()
    ops.speckle_filter(d, B, 3, 0.25, out=(mask, stats), workspace=ws)
    assert torch.equal(stats, 2 * once) and int(mask.max()) <= 1
    empty = ops.speckle_filter(torch.empty(0, H, W, device='cuda'), 0, 3, 0.25)
    assert empty[0].shape == (0, 2, H, W) and lib.launches() - n0 == 8


def test_bad_arguments():
    B, H, W = 2, 16, 16
    d = torch.zeros(2 * B, H, W, device='cuda')
    mask = torch.empty(B, 2, H, W, dtype=torch.uint8, device='cuda')
    stats = torch.zeros(B, 2, 5, dtype=torch.int64, device='cuda')
    nb = ops.speckle_filter_workspace_bytes(B, H, W)
    ws = torch.empty(nb, dtype=torch.uint8, device='cuda')
    L = lib.load()
    s = torch.cuda.current_stream().cuda_stream
    th = (ctypes.c_float * 9)(*([1.0] * 9))

    def call(B_=B, H_=H, W_=W, max_size=3, max_diff=1.0, gt=None, T=0, max_gt=0.0, nbytes=nb, disp=d.data_ptr(),
             m=mask.data_ptr(), w=ws.data_ptr()):
        return L.s3d_speckle_filter(disp, B_, H_, W_, None, max_size, max_diff, gt, th, T, max_gt, m, stats.data_ptr(), w,
                                    nbytes, s)
    for kw in (dict(H_=0), dict(W_=0), dict(B_=-1), dict(B_=1 << 15), dict(max_size=-1), dict(max_diff=-0.5),
               dict(max_diff=float('nan')), dict(max_diff=float('inf')), dict(T=9), dict(T=-1), dict(nbytes=nb - 1),
               dict(gt=d.data_ptr(), max_gt=0.0), dict(gt=d.data_ptr(), max_gt=float('nan')), dict(disp=None), dict(m=None),
               dict(H_=1 << 16, W_=1 << 15), dict(w=ws.data_ptr() + 2)):
        assert call(**kw) == -1, kw
        assert L.s3d_last_error()
    assert call() == 0
    n0 = lib.launches()
    for kw in (dict(max_size=-1), dict(max_size=1.5), dict(max_size=True), dict(max_diff=-1.0), dict(max_diff=float('nan')),
               dict(max_diff=1e39), dict(max_diff='a'), dict(thresholds=[1.0] * 9), dict(disp_gt=d.view(B, 2, H, W)),
               dict(disp_gt=d.view(B, 2, H, W), max_gt=0.0), dict(lr_mask=mask.float()), dict(lr_mask=mask[:1]),
               dict(disp_gt=d.view(B, 2, H, W).double(), max_gt=1.0), dict(out=(mask, stats[..., :4])),
               dict(workspace=ws[:-1]), dict(B=3), dict(B=True)):
        args = dict(max_size=3, max_diff=1.0)
        args.update(kw)
        B_ = args.pop('B', B)
        with pytest.raises(ValueError):
            ops.speckle_filter(d, B_, **args)
    with pytest.raises(ValueError):
        ops.speckle_filter(d.double(), B, 3, 1.0)
    with pytest.raises(ValueError):
        ops.speckle_filter(d[None], B, 3, 1.0)
    assert lib.launches() == n0


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


def _check_model_speckle(cfg, names, out, dgt=None):
    """speckle_mask / speckle_stats equal the op (and the oracle) on the forward's own disp and lr_mask."""
    o = dict(zip(names, out))
    B = o['disp_left'].shape[0]
    disp = torch.cat([o['disp_left'][:, 0], o['disp_right'][:, 0]]).contiguous()
    max_size, max_diff = M.speckle_params(cfg)
    th = list(cfg.TEST.DISP_THRESH)
    ref = ops.speckle_filter(disp, B, max_size, max_diff, lr_mask=o.get('lr_mask'), disp_gt=dgt, thresholds=th,
                             max_gt=4.0 * cfg.NETWORK.MAX_DISP)
    assert torch.equal(ref[0], o['speckle_mask']) and torch.equal(ref[1], o['speckle_stats'])
    want = O.speckle_filter(disp.cpu().numpy(), B, max_size, max_diff,
                            None if o.get('lr_mask') is None else o['lr_mask'].cpu().numpy(),
                            None if dgt is None else dgt.cpu().numpy(), th, 4.0 * cfg.NETWORK.MAX_DISP)
    assert np.array_equal(o['speckle_mask'].cpu().numpy(), want[0])
    assert np.array_equal(o['speckle_stats'].cpu().numpy(), want[1])
    return o


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_model_speckle_is_the_op_on_its_own_maps(name):
    # the synthetic weights' maps are not left-right consistent: a wide LR tolerance keeps the pixels whose match lies in the
    # image
    cfg, model = _model(name, TEST__LR_THRESH=1000.0, TEST__SPECKLE_MAX_SIZE=20, TEST__SPECKLE_MAX_DIFF=0.25)
    args, gt, dgt, cam = _inputs(cfg, 2, seed=1)
    with torch.no_grad():
        for kw in (dict(), dict(lr_check=True), dict(disp_gt=dgt), dict(lr_check=True, uncertainty=True, disp_gt=dgt)):
            on = {k: True for k in kw if k != 'disp_gt'}
            n0 = lib.launches()
            plain = [t.clone() for t in model(*args, **kw)]
            n1 = lib.launches()
            full = [t.clone() for t in model(*args, speckle=True, **kw)]
            n2 = lib.launches()
            assert (n2 - n1) - (n1 - n0) == 4
            names = type(model).output_names(speckle=True, disp_gt='disp_gt' in kw, **on)
            assert len(full) == len(plain) + 2 and len(names) == len(full)
            o = _check_model_speckle(cfg, names, full, kw.get('disp_gt'))
            for n, t in zip(type(model).output_names(disp_gt='disp_gt' in kw, **on), plain):
                assert torch.equal(t, o[n]), n


def test_model_launches_unchanged_without_speckle():
    cfg, model = _model()
    args, gt, dgt, cam = _inputs(cfg, 2, seed=0)
    with torch.no_grad():
        counts, outs = [], []
        for kw in (dict(), dict(speckle=False), dict(speckle=True)):
            n0 = lib.launches()
            outs.append([t.clone() for t in model(*args, gt, disp_gt=dgt, lr_check=True, **kw)])
            counts.append(lib.launches() - n0)
    assert counts[0] == counts[1] and counts[2] == counts[0] + 4
    assert all(torch.equal(a, b) for a, b in zip(outs[0], outs[1]))


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_graphed_matches_eager_and_does_not_accumulate(name):
    cfg, model = _model(name, TEST__SPECKLE_MAX_SIZE=20, TEST__SPECKLE_MAX_DIFF=0.25)
    seen = []
    for seed in (0, 1):
        args, gt, dgt, cam = _inputs(cfg, 2, seed=seed)
        with torch.no_grad():
            for kw in (dict(lr_check=True, disp_gt=dgt), {}):
                eager = [t.clone() for t in model(*args, speckle=True, **kw)]
                for _ in range(2):                                   # a second replay gives the same counters
                    graphed = [t.clone() for t in model.graphed(*args, speckle=True, **kw)]
                    assert len(graphed) == len(eager) and all(torch.equal(a, b) for a, b in zip(eager, graphed))
        seen.append(eager[0])
    assert not torch.equal(seen[0], seen[1])
    with torch.no_grad():
        model.graphed(*args)
    assert len(model._graphs) == 3                                   # speckle is part of the graph key


def test_micro_batch_concatenates_chunks():
    cfg, model = _model(CONST__MICRO_BATCH=2, TEST__SPECKLE_MAX_SIZE=20)
    args, gt, dgt, cam = _inputs(cfg, 5, seed=6)
    with torch.no_grad():
        full = [t.clone() for t in model(*args, disp_gt=dgt, lr_check=True, speckle=True)]
        parts = [[t.clone() for t in model(args[0][s:s + 2], args[1][s:s + 2], disp_gt=dgt[s:s + 2], lr_check=True,
                                           speckle=True)] for s in range(0, 5, 2)]
    for i, t in enumerate(full):
        assert torch.equal(t, torch.cat([p[i] for p in parts]))
    _check_model_speckle(cfg, M.Stereo2Voxel.output_names(disp_gt=True, lr_check=True, speckle=True), full, dgt)


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_cloud_takes_the_speckle_mask(name):
    cfg, model = _model(name, TEST__LR_THRESH=1000.0, TEST__SPECKLE_MAX_SIZE=20, TEST__SPECKLE_MAX_DIFF=0.25)
    args, gt, dgt, cam = _inputs(cfg, 2, seed=2)
    with torch.no_grad():
        for kw in (dict(), dict(lr_check=True)):
            names = type(model).output_names(speckle=True, camera=True, **kw)
            o = dict(zip(names, [t.clone() for t in model(*args, speckle=True, camera=cam, **kw)]))
            disp = torch.cat([o['disp_left'][:, 0], o['disp_right'][:, 0]]).contiguous()
            ref = ops.disp_cloud(disp, 2, *args, cam, M.cloud_min_disp(cfg), lr_mask=o['speckle_mask'])
            assert torch.equal(ref[2], o['cloud_counts'])
            for b in range(2):
                k = int(ref[2][b].sum())
                assert torch.equal(ref[0][b, :k], o['cloud_xyz'][b, :k]) and torch.equal(ref[1][b, :k], o['cloud_rgb'][b, :k])
            plain = dict(zip(type(model).output_names(camera=True, **kw), model(*args, camera=cam, **kw)))
            assert int(o['cloud_counts'].sum()) <= int(plain['cloud_counts'].sum())


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_max_size_zero_is_the_lr_check(name):
    cfg, model = _model(name, TEST__LR_THRESH=2.0, TEST__SPECKLE_MAX_SIZE=0)
    args, gt, dgt, cam = _inputs(cfg, 2, seed=3)
    T = len(cfg.TEST.DISP_THRESH)
    with torch.no_grad():
        o = dict(zip(type(model).output_names(disp_gt=True, lr_check=True, speckle=True),
                     model(*args, disp_gt=dgt, lr_check=True, speckle=True)))
    assert torch.equal(o['speckle_mask'], o['lr_mask'])
    assert torch.equal(o['speckle_stats'][..., :3 + T], o['lr_stats'])
    assert int(o['speckle_stats'][..., 3 + T:].abs().sum()) == 0


def test_value_errors_before_any_launch():
    cfg, model = _model()
    args, gt, _, cam = _inputs(cfg, 2, seed=0)
    model(*args)
    n0 = lib.launches()
    for key, bad in (('SPECKLE_MAX_SIZE', -1), ('SPECKLE_MAX_SIZE', True), ('SPECKLE_MAX_SIZE', 2.0),
                     ('SPECKLE_MAX_DIFF', float('nan')), ('SPECKLE_MAX_DIFF', -1.0)):
        old = cfg.TEST[key]
        cfg.TEST[key] = bad
        with pytest.raises(ValueError, match=key):
            model(*args, speckle=True)
        with pytest.raises(ValueError, match=key):
            model.graphed(*args, speckle=True)
        cfg.TEST[key] = old
    assert lib.launches() == n0


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_runner_speckle_with_clouds(name, monkeypatch, capsys, tmp_path):
    import runner
    from config import cfg as dcfg
    n, bs = 3, 2
    out_dir = str(tmp_path / 'clouds')
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--model', name, '--batch-size', str(bs), '--n-samples', str(n),
                                      '--lr-check', '--speckle', '--save-clouds', out_dir])
    runner.main()
    res = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    cfg = dcfg.clone()
    max_size, max_diff = M.speckle_params(cfg)
    assert res['speckle']['max_size'] == max_size and res['speckle']['max_diff'] == max_diff
    assert res['speckle']['after_lr_check'] is True
    assert res['cloud']['speckle'] == {'max_size': max_size, 'max_diff': max_diff}
    model = M.build_model(name, cfg, seed=cfg.CONST.SEED).cuda().pack()
    H, W, T = cfg.CONST.IMG_H, cfg.CONST.IMG_W, len(cfg.TEST.DISP_THRESH)
    cam = torch.tensor([M.camera_values(cfg)], device='cuda')
    tot = torch.zeros(2, 5 + T, dtype=torch.int64)
    for s in range(0, n, bs):
        ids = list(range(s, min(s + bs, n)))
        pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in ids]
        left, right = torch.cat([p[0] for p in pairs]).cuda(), torch.cat([p[1] for p in pairs]).cuda()
        dgt = torch.cat([synthetic.disparity_gt(p[2], H, W) for p in pairs]).cuda()
        with torch.no_grad():
            o = dict(zip(type(model).output_names(disp_gt=True, lr_check=True, speckle=True, camera=True),
                         model(left, right, disp_gt=dgt, lr_check=True, speckle=True, camera=cam.repeat(len(ids), 1))))
        tot += o['speckle_stats'].sum(0).cpu()
        xyz, c = o['cloud_xyz'].cpu().numpy(), o['cloud_counts'].cpu().numpy()
        for b, i in enumerate(ids):
            k = int(c[b].sum())
            rec = CO.read_ply(os.path.join(out_dir, '%06d.ply' % i))
            assert len(rec) == k
            assert np.array_equal(np.stack([rec['x'], rec['y'], rec['z']], 1).view(np.uint32), xyz[b, :k].view(np.uint32))
            assert len(CO.read_ply(os.path.join(out_dir, '%06d_gt.ply' % i))) > 0
    for v, view in enumerate(('left', 'right')):
        r = res['speckle'][view]
        assert r['n_kept'] == tot[v, 0] and r['n_valid_kept'] == tot[v, 1]
        assert r['n_speckles'] == tot[v, 3 + T] and r['speckle_pixels'] == tot[v, 4 + T]
        assert res['cloud'][view]['n_points'] <= r['n_kept']
