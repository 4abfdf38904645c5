"""Threshold-free occupancy evaluation on the GPU (s3d_occupancy_curves): histograms and Brier sums bit-exact against the
reference statement (tests/curves_oracle.py), the BCE sums within 2 units per sample (an fp64 log may differ by an ulp at a
rounding tie), on random, special-valued, single-bin, empty-GT and full-GT fields of cube and non-cube sizes; the forward's
curves=True option, its graph, its micro-batches, its launch count and its errors; and runner.py --test --curves."""
import ctypes
import json
import sys

import numpy as np
import pytest
import torch

from stereo_3d_reconstruction_b200 import lib, models as M, ops
from stereo_3d_reconstruction_b200.utils import synthetic
from tests import curves_oracle as O
from tests.common import small_cfg

pytestmark = pytest.mark.gpu


def _field(shape, seed, K, special=True, p=0.3):
    rng = np.random.default_rng(seed)
    v = rng.random(shape).astype(np.float32)
    if special:
        sel = rng.random(shape)
        v[sel < 0.1] = (rng.integers(0, K + 1, (sel < 0.1).sum()) / K).astype(np.float32)   # on bin edges
        for lo, x in ((0.1, np.nan), (0.12, -0.25), (0.14, 1.5), (0.16, np.inf), (0.17, -np.inf), (0.18, 0.0),
                      (0.2, 1.0), (0.22, 1e-30), (0.24, np.float32(1) - np.float32(2 ** -24))):
            v[(sel >= lo) & (sel < lo + 0.02)] = x
    gt = ((rng.random(shape) < p) * rng.integers(1, 256, shape)).astype(np.uint8)
    return v, gt


def _check(v, gt, K, hist, loss):
    wh, wl = O.occupancy_curves(v, gt, K)
    assert np.array_equal(hist, wh)
    assert np.array_equal(loss[:, 1], wl[:, 1])
    assert np.abs(loss[:, 0] - wl[:, 0]).max() <= 2
    return wh, wl


def _run(v, gt, K):
    x, g = torch.from_numpy(np.ascontiguousarray(v)).cuda(), torch.from_numpy(np.ascontiguousarray(gt)).cuda()
    B = v.shape[0]
    out = (torch.full((B, 3, K), -7, dtype=torch.int64, device='cuda'), torch.full((B, 2), -7, dtype=torch.int64, device='cuda'))
    n0 = lib.launches()
    got = ops.occupancy_curves(x, g, K, out=out)
    assert lib.launches() - n0 == (1 if B else 0)
    assert all(a is b for a, b in zip(got, out))
    return _check(v, gt, K, out[0].cpu().numpy(), out[1].cpu().numpy())


@pytest.mark.parametrize('n,B', [(1, 3), (2, 64), (5, 17), (13, 4), (32, 64), (64, 2)])
@pytest.mark.parametrize('K', [2, 16, 256, 1024])
def test_random_fields_match_oracle(n, B, K):
    v, gt = _field((B, n, n, n), seed=n * 1000 + B + K, K=K)
    _run(v, gt, K)


@pytest.mark.parametrize('shape', [(3, 7, 11), (5, 1), (2, 10001), (4, 6), (64, 32768 + 3)])
def test_non_cube_and_unaligned_sizes(shape):
    """nvox not a multiple of 4 (scalar loads), a multiple of 4 that is not a cube, and a single voxel."""
    v, gt = _field(shape, seed=sum(shape), K=256)
    _run(v, gt, 256)


def test_unaligned_pointers_take_the_scalar_path():
    B, nvox, K = 6, 4096, 64
    v, gt = _field((B, nvox), seed=5, K=K)
    xs = torch.zeros(B * nvox + 1, device='cuda')
    gs = torch.zeros(B * nvox + 1, dtype=torch.uint8, device='cuda')
    x = xs[1:].view(B, nvox)                                         # 4 bytes past a 16-byte boundary
    g = gs[1:].view(B, nvox)
    x.copy_(torch.from_numpy(v))
    g.copy_(torch.from_numpy(gt))
    hist, loss = ops.occupancy_curves(x, g, K)
    _check(v, gt, K, hist.cpu().numpy(), loss.cpu().numpy())


@pytest.mark.parametrize('K', [2, 16, 256, 1024])
def test_every_voxel_in_one_bin(K):
    """The untrained network's predictions sit near 0.5: one bin holds every voxel (the warp-aggregated update path)."""
    B, n = 64, 32
    for val in (0.5, np.float32(0.5) - np.float32(2 ** -24), 0.0, 1.0):
        v = np.full((B, n, n, n), val, np.float32)
        gt = _field((B, n, n, n), seed=K, K=K, special=False)[1]
        hist, _ = _run(v, gt, K)
        k = int(O.bins(np.float32(val), K))
        assert (hist[:, :2, k].sum(1) == n ** 3).all()


def test_empty_and_full_gt():
    B, n, K = 4, 16, 256
    v, _ = _field((B, n, n, n), seed=9, K=K)
    for gt in (np.zeros((B, n, n, n), np.uint8), np.full((B, n, n, n), 255, np.uint8)):
        hist, _ = _run(v, gt, K)
        assert (hist[:, 1 if gt.any() else 0].sum(1) == n ** 3).all()


def test_bad_arguments():
    L = lib.load()
    B, nvox, K = 2, 64, 16
    x = torch.rand(B, nvox, device='cuda')
    g = torch.zeros(B, nvox, dtype=torch.uint8, device='cuda')
    h = torch.full((B, 3, K), -5, dtype=torch.int64, device='cuda')
    lo = torch.full((B, 2), -5, dtype=torch.int64, device='cuda')
    s = torch.cuda.current_stream().cuda_stream

    def call(x_=x.data_ptr(), g_=g.data_ptr(), B_=B, n_=nvox, K_=K, h_=h.data_ptr(), l_=lo.data_ptr()):
        return L.s3d_occupancy_curves(x_, g_, B_, n_, K_, h_, l_, s)
    assert call(B_=0) == 0
    torch.cuda.synchronize()
    for bad in (dict(x_=None), dict(g_=None), dict(h_=None), dict(l_=None), dict(B_=-1), dict(B_=1 << 29), dict(n_=0),
                dict(n_=(1 << 24) + 1), dict(n_=-4), dict(K_=0), dict(K_=1), dict(K_=3), dict(K_=48), dict(K_=2048),
                dict(K_=-16)):
        rc = call(**bad)
        assert rc == -1, bad
        with pytest.raises(lib.S3dError):
            lib.check(rc, 's3d_occupancy_curves')
    torch.cuda.synchronize()
    assert (h == -5).all() and (lo == -5).all()                      # nothing ran
    n0 = lib.launches()
    for bx, bg, k in ((x.double(), g, K), (x, g.bool(), K), (x, g.float(), K), (x, g[:, :-1].contiguous(), K), (x[0], g[0], K),
                      (x, g, 3), (x, g, 1), (x, g, 2048), (x, g, 16.0), (x, g, True), (x, g, '16'),
                      (torch.rand(1, (1 << 24) + 4, device='cuda'), torch.zeros(1, (1 << 24) + 4, dtype=torch.uint8, device='cuda'), K)):
        with pytest.raises(ValueError):
            ops.occupancy_curves(bx, bg, k)
    for bad_out in ((h,), (h, lo, lo), (h[:, :2].contiguous(), lo), (h, lo.int()), (h.float(), lo), (h, lo[:1].contiguous()),
                    (torch.zeros(B, 3, 2 * K, dtype=torch.int64, device='cuda'), lo)):
        with pytest.raises(ValueError):
            ops.occupancy_curves(x, g, K, out=bad_out)
    with pytest.raises(lib.S3dError):
        ops.occupancy_curves(x, g, K, out=(h.cpu(), lo))
    with pytest.raises((ValueError, lib.S3dError)):
        ops.occupancy_curves(x, g.cpu(), K)
    with pytest.raises(lib.S3dError):
        ops.occupancy_curves(x.cpu(), g.cpu(), K)
    assert lib.launches() == n0


# ---- the model ------------------------------------------------------------------------------------------------------------
def _model(default=False, **kw):
    if default:
        from config import cfg as dcfg
        cfg = dcfg.clone()
        for k, v in kw.items():
            sec, key = k.split('__')
            cfg[sec][key] = v
    else:
        cfg = small_cfg(NETWORK__PRECISION='bf16', **kw)
    return cfg, M.build_model('Stereo2Voxel', cfg, seed=3).cuda().pack()


def _inputs(cfg, B, seed):
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=seed)
    gt = synthetic.gt_volume(B, cfg.CONST.N_VOX, seed=seed + 50)
    return (left.cuda(), right.cuda()), gt.cuda(), synthetic.disparity_gt(d, H, W).cuda()


def _check_model(cfg, vox, gt, hist, loss):
    K = cfg.TEST.CURVE_BINS
    _check(vox.cpu().numpy(), gt.cpu().numpy().astype(np.uint8), K, hist.cpu().numpy(), loss.cpu().numpy())


@pytest.mark.parametrize('default', [False, True])
def test_model_curves_exact_and_outputs_unchanged(default):
    cfg, model = _model(default)
    args, gt, dgt = _inputs(cfg, 2, seed=1)
    K = cfg.TEST.CURVE_BINS
    with torch.no_grad():
        for kw in (dict(), dict(disp_gt=dgt, lr_check=True, uncertainty=True, surface=True, mesh=True)):
            n0 = lib.launches()
            plain = [t.clone() for t in model(*args, gt, **kw)]
            n1 = lib.launches()
            off = [t.clone() for t in model(*args, gt, curves=False, **kw)]
            n2 = lib.launches()
            full = [t.clone() for t in model(*args, gt, curves=True, **kw)]
            n3 = lib.launches()
            assert n2 - n1 == n1 - n0 and (n3 - n2) - (n1 - n0) == 1      # occupancy_curves_kernel
            assert len(off) == len(plain) and len(full) == len(plain) + 2
            for a, b, c in zip(plain, off, full):
                assert torch.equal(a, b) and torch.equal(a, c)
            hist, loss = full[-2:]
            assert hist.shape == (2, 3, K) and loss.shape == (2, 2)
            _check_model(cfg, full[2], gt, hist, loss)
            # the pooled counts at bin K/2 are the IoU counts at t = 0.5 (a TEST.VOXEL_THRESH value)
            ti = list(cfg.TEST.VOXEL_THRESH).index(0.5)
            inter = hist[:, 1, K // 2:].sum(1)
            union = hist[:, :2, K // 2:].sum((1, 2)) + hist[:, 1].sum(1) - inter
            assert torch.equal(full[3][:, ti, 0], inter) and torch.equal(full[3][:, ti, 1], union)


def test_graphed_matches_eager_and_replays_do_not_accumulate():
    cfg, model = _model()
    with torch.no_grad():
        eager = []
        for seed in (0, 1):
            args, gt, dgt = _inputs(cfg, 2, seed=seed)
            eager.append([t.clone() for t in model(*args, gt, disp_gt=dgt, surface=True, curves=True)])
        for rep in range(2):
            for seed in (0, 1):
                args, gt, dgt = _inputs(cfg, 2, seed=seed)
                graphed = [t.clone() for t in model.graphed(*args, gt, disp_gt=dgt, surface=True, curves=True)]
                assert len(graphed) == len(eager[seed])
                for a, b in zip(eager[seed], graphed):
                    assert torch.equal(a, b)
        assert not torch.equal(eager[0][-2], eager[1][-2])
        args, gt, _ = _inputs(cfg, 2, seed=0)
        assert len(model.graphed(*args, gt)) == 4
    assert len(model._graphs) == 2                                   # curves is part of the graph key


def test_micro_batch_concatenates_chunks():
    cfg, model = _model(CONST__MICRO_BATCH=2)
    args, gt, _ = _inputs(cfg, 5, seed=6)
    with torch.no_grad():
        full = [t.clone() for t in model(*args, gt, curves=True)]
        parts = [[t.clone() for t in model(args[0][s:s + 2], args[1][s:s + 2], gt[s:s + 2], curves=True)]
                 for s in range(0, 5, 2)]
    for i, t in enumerate(full):
        assert torch.equal(t, torch.cat([p[i] for p in parts]))
    _check_model(cfg, full[2], gt, *full[-2:])


def test_other_curve_bins():
    cfg, model = _model(TEST__CURVE_BINS=1024)
    args, gt, _ = _inputs(cfg, 3, seed=2)
    with torch.no_grad():
        out = model(*args, gt, curves=True)
        assert out[-2].shape == (3, 3, 1024)
        _check_model(cfg, out[2], gt, *out[-2:])
        cfg.TEST.CURVE_BINS = 4
        out = model.graphed(*args, gt, curves=True)
        assert out[-2].shape == (3, 3, 4)
        _check_model(cfg, out[2], gt, *out[-2:])


def test_value_errors_before_any_launch():
    cfg, model = _model()
    args, gt, _ = _inputs(cfg, 2, seed=0)
    model(*args)                                                    # packed, workspace built
    n0 = lib.launches()
    with pytest.raises(ValueError, match='needs the GT'):
        model(*args, curves=True)
    with pytest.raises(ValueError, match='needs the GT'):
        model.graphed(*args, curves=True)
    for bad in (0, 3, 2048, 256.0, True, None, '256'):
        cfg.TEST.CURVE_BINS = bad
        with pytest.raises(ValueError, match='CURVE_BINS'):
            model(*args, gt, curves=True)
        with pytest.raises(ValueError, match='CURVE_BINS'):
            model.graphed(*args, gt, curves=True)
    assert lib.launches() == n0
    pcfg = small_cfg(NETWORK__PRECISION='bf16')
    pm = M.build_model('Stereo2Point', pcfg, seed=0).cuda().pack()
    pts = torch.rand(2, 64, 3, device='cuda')
    for g in (None, pts):
        with pytest.raises(ValueError, match='Stereo2Voxel only'):
            pm(*args, g, curves=True)
        with pytest.raises(ValueError, match='Stereo2Voxel only'):
            pm.graphed(*args, g, curves=True)
    assert lib.launches() == n0


def test_runner_curves(monkeypatch, capsys):
    import runner

    def run(*flags):
        monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--n-samples', '128'] + list(flags))
        runner.main()
        return capsys.readouterr().out.strip().splitlines()[-1]
    base, line = run(), run('--curves')
    res = json.loads(line)
    c = res.pop('occupancy_curves')
    assert json.dumps(res) == base                                  # every other key byte-identical
    from config import cfg
    K = cfg.TEST.CURVE_BINS
    assert c['n_samples'] == 128 and c['bins'] == K and len(c['iou']) == K and len(c['mean_iou']) == K
    assert c['n_voxels'] == 128 * cfg.CONST.N_VOX ** 3 and len(c['reliability']) == 16
    # the pooled curve at t = 0.5 is the IoU the runner reports there
    assert abs(c['iou'][K // 2] - res['iou'][list(cfg.TEST.VOXEL_THRESH).index(0.5)]) < 1e-12
    assert 0 <= c['ap'] <= 1 and c['bce'] > 0 and 0 <= c['brier'] <= 1 and 0 <= c['ece'] <= 1
    assert c['best']['iou'] == max(c['iou'])
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--model', 'Stereo2Point', '--curves'])
    with pytest.raises(SystemExit) as e:
        runner.main()
    assert 'Stereo2Voxel only' in str(e.value)
