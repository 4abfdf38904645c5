"""Speckle filter, host side: the numpy / scipy statement of s3d_speckle_filter (tests/speckle_oracle.py) against OpenCV's
filterSpeckles and on hand-built cases, the validation of the config keys, the forward's output order with speckle=True, the
test driver's 'speckle' block and summary, driver runs through a fake forward (also through a gloo world-2 all-reduce) and
runner.py's argument."""
import itertools
import os
import socket
import sys

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import runner
from stereo_3d_reconstruction_b200 import models
from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.models import Stereo2Point, Stereo2Voxel
from stereo_3d_reconstruction_b200.utils import synthetic
from tests import speckle_oracle as O
from tests.common import small_cfg

f32 = np.float32
_NAN = float('nan')


# ---- the rule against OpenCV ----------------------------------------------------------------------------------------------
def _cv2_mask(cv2, d, max_size, md16):
    """cv2.filterSpeckles on int16(16 d) with the non-finite pixels set to a newVal no candidate holds -> kept mask."""
    img = np.where(np.isfinite(d), np.nan_to_num(d) * 16, -32768).astype(np.int16)
    out, _ = cv2.filterSpeckles(img, -32768, max_size, md16)
    return (out != -32768).astype(np.uint8)


def _rand_map(rng, H, W, hole):
    d = (rng.integers(-40, 40, (H, W)) / 16).astype(f32)
    if hole:
        d[rng.random((H, W)) < 0.2] = np.nan
    return d


def test_oracle_equals_cv2_on_random_maps():
    cv2 = pytest.importorskip('cv2')
    rng = np.random.default_rng(0)
    for it in range(60):
        H, W = (int(v) for v in rng.integers(1, 40, 2))
        d = np.stack([_rand_map(rng, H, W, it % 2 == 0), _rand_map(rng, H, W, it % 3 == 0)])
        max_size, md16 = int(rng.integers(0, 12)), int(rng.integers(0, 40))
        mask, _ = O.speckle_filter(d, 1, max_size, md16 / 16)
        for v in range(2):
            assert np.array_equal(mask[0, v], _cv2_mask(cv2, d[v], max_size, md16)), (it, v)


@pytest.mark.parametrize('max_size', [0, 1, 4, 5, 6, 1000])
@pytest.mark.parametrize('md16', [0, 8, 16])
def test_oracle_equals_cv2_on_edges(max_size, md16):
    cv2 = pytest.importorskip('cv2')
    H, W = 12, 20
    d = np.full((H, W), np.nan, f32)
    d[1, 2:7] = 1.0                                              # 5 px
    d[3, 2:8] = 2.0                                              # 6 px
    d[5:9, 3] = 3.0                                              # 4 px
    d[5:8, 10] = [4.0, 4.5, 5.0]                                 # 3 px in steps of 8/16
    d[9:12, 12:19] = 0.0                                         # 21 px, a flat patch
    d[10, 15] = 1.0                                              # a step of 16/16 inside it
    m = np.stack([d, np.full((H, W), 7.0, f32)])                 # view 1: one region of H W = 240 px
    mask, st = O.speckle_filter(m, 1, max_size, md16 / 16)
    for v in range(2):
        assert np.array_equal(mask[0, v], _cv2_mask(cv2, m[v], max_size, md16))
    assert st[0, 1, 0] == (H * W if max_size < H * W else 0)


def test_oracle_counters_by_hand():
    d = np.full((2, 3, 4), np.nan, f32)
    d[0, 0, :2] = [1.0, 1.5]                                     # one region of 2 at max_diff 0.5
    d[0, 2, :] = [5.0, 5.0, 5.0, 9.0]                            # a region of 3 and one of 1
    d[1, 1, 1] = 2.0
    g = np.full((1, 2, 3, 4), np.nan, f32)
    g[0, 0, 2, :] = [4.0, 5.25, -1.0, 8.0]                       # errors 1, 0.25, invalid, 1
    g[0, 0, 0, 0] = 100.0                                        # >= max_gt: invalid
    mask, st = O.speckle_filter(d, 1, 1, 0.5, disp_gt=g, thresholds=(0.5, 1.0), max_gt=64.0)
    assert mask[0, 0].tolist() == [[1, 1, 0, 0], [0, 0, 0, 0], [1, 1, 1, 0]] and mask[0, 1].sum() == 0
    # [n_kept, n_valid_kept, q, bad(0.5), bad(1.0), n_speckles, n_speckle_px]
    assert st[0, 0].tolist() == [5, 2, 65536 + 16384, 1, 0, 1, 1]
    assert st[0, 1].tolist() == [0, 0, 0, 0, 0, 1, 1]
    lr = np.ones((1, 2, 3, 4), np.uint8)
    lr[0, 0, 2, 1] = 2                                           # breaks the region of 3 into two of 1
    mask, st = O.speckle_filter(d, 1, 1, 0.5, lr_mask=lr)
    assert mask[0, 0, 2].tolist() == [0, 0, 0, 0] and st[0, 0].tolist() == [2, 0, 0, 3, 3]


# ---- config -------------------------------------------------------------------------------------------------------------
def _cfg(**kw):
    return small_cfg(TEST__VOXEL_THRESH=[0.2, 0.4, 0.6, 0.8], TEST__DISP_THRESH=[1.0, 3.0], TEST__UNC_THRESH=[1.0, 2.0, 4.0],
                     TEST__FSCORE_THRESH=[0.05, 0.3], CONST__N_VOX=6, CONST__N_POINTS=4, CONST__N_GT_POINTS=8, **kw)


def test_config_defaults():
    from config import cfg
    assert models.speckle_params(cfg) == (100, 1.0)
    assert models.speckle_params(_cfg(TEST__SPECKLE_MAX_SIZE=0, TEST__SPECKLE_MAX_DIFF=0)) == (0, 0.0)


@pytest.mark.parametrize('v', [-1, True, False, 1.0, '5', None, 2 ** 31])
def test_speckle_max_size_rejects(v):
    with pytest.raises(ValueError, match='SPECKLE_MAX_SIZE'):
        models.speckle_params(_cfg(TEST__SPECKLE_MAX_SIZE=v))


@pytest.mark.parametrize('v', [-0.5, float('nan'), float('inf'), 1e39, 'a', None, True])
def test_speckle_max_diff_rejects(v):
    with pytest.raises(ValueError, match='SPECKLE_MAX_DIFF'):
        models.speckle_params(_cfg(TEST__SPECKLE_MAX_DIFF=v))


def test_forward_rejects_bad_speckle_config_before_any_launch():
    x = torch.zeros(1, 3, 64, 64)
    for name in ('Stereo2Voxel', 'Stereo2Point'):
        m = models.build_model(name, _cfg(TEST__SPECKLE_MAX_SIZE=-1))
        with pytest.raises(ValueError, match='SPECKLE_MAX_SIZE'):
            m(x, x, speckle=True)
        with pytest.raises(ValueError, match='SPECKLE_MAX_SIZE'):
            m.graphed(x, x, lr_check=True, speckle=True)


# ---- the forward's output order -------------------------------------------------------------------------------------------
@pytest.mark.parametrize('flags', list(itertools.product([False, True], repeat=5)))
def test_output_names_with_speckle(flags):
    gt, disp_gt, lr_check, uncertainty, camera = flags
    for cls in (Stereo2Voxel, Stereo2Point):
        kw = dict(gt=gt, disp_gt=disp_gt, lr_check=lr_check, uncertainty=uncertainty, camera=camera)
        off = cls.output_names(**kw)
        on = cls.output_names(speckle=True, **kw)
        i = off.index('lr_stats') + 1 if lr_check else len(cls.HEAD_OUTPUTS) + gt + disp_gt
        assert on == off[:i] + ('speckle_mask', 'speckle_stats') + off[i:]
        assert cls.output_names(speckle=False, **kw) == off


def test_speckle_in_the_declared_orders():
    names = [o for o, _ in models.OPTIONAL_OUTPUTS]
    assert names.index('speckle') == names.index('lr_check') + 1 and names.index('camera') == names.index('uncertainty') + 1
    assert dict(models.OPTIONAL_OUTPUTS)['speckle'] == ('speckle_mask', 'speckle_stats')
    f = models.Options._fields
    assert f.index('speckle') == f.index('lr_check') + 1 and f[-1] == 'fscore_curves'
    assert 'speckle' in Stereo2Voxel.OPTIONS and 'speckle' in Stereo2Point.OPTIONS
    assert Stereo2Point.output_names(gt=True, disp_gt=True, lr_check=True, speckle=True, uncertainty=True, camera=True,
                                     fscore_curves=True) == (
        'disp_left', 'disp_right', 'points', 'point_stats', 'disp_stats', 'lr_mask', 'lr_stats', 'speckle_mask',
        'speckle_stats', 'disp_std', 'unc_stats', 'cloud_xyz', 'cloud_rgb', 'cloud_counts', 'dist_hist')


# ---- stats block and summary ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('model', ['Stereo2Voxel', 'Stereo2Point'])
def test_speckle_block(model):
    tail = {'eval_surface': True} if model == 'Stereo2Voxel' else {'eval_points': True}
    cfg = _cfg()
    for lr in (False, True):
        ev = dict(eval_disp=True, eval_lr=lr, eval_unc=True, eval_cloud=True, **tail)
        on = T.stats_layout(cfg, model, eval_speckle=True, **ev)
        off = T.stats_layout(cfg, model, **ev)
        names = [b for b, _ in on]
        assert names.index('speckle') == names.index('lr_consistency' if lr else 'disparity') + 1
        assert names.index('uncertainty') == names.index('speckle') + 1 and dict(on)['speckle'] == 2 * (5 + 2)
        assert [b for b in on if b[0] != 'speckle'] == off
        assert T.stats_layout(cfg, model, **ev, eval_speckle=False) == off
    with pytest.raises(ValueError, match='eval_speckle=True needs eval_disp'):
        T.stats_layout(cfg, model, eval_speckle=True)
    with pytest.raises(ValueError, match='SPECKLE_MAX_DIFF'):
        T.stats_layout(_cfg(TEST__SPECKLE_MAX_DIFF=-1.0), model, eval_disp=True, eval_speckle=True)


def test_speckle_summary():
    # per view [n_kept, n_valid_kept, q, bad(1), bad(3), n_speckles, n_speckle_px]; T = 2
    block = torch.tensor([80, 40, 40 << 16, 10, 4, 5, 20, 60, 30, 60 << 16, 6, 0, 0, 0])
    disp = torch.tensor([50, 0, 0, 0, 50, 0, 0, 0])
    s = T.speckle_summary(block, [1.0, 3.0], 100, disp)
    lr = T.lr_summary(torch.tensor([80, 40, 40 << 16, 10, 4, 60, 30, 60 << 16, 6, 0]), [1.0, 3.0], 100, disp)
    for v in ('left', 'right', 'all'):
        for k, x in lr[v].items():
            assert s[v][k] == x
    assert s['left']['n_speckles'] == 5 and s['left']['speckle_pixels'] == 20 and s['left']['mean_speckle_size'] == 4.0
    assert s['right']['n_speckles'] == 0 and s['right']['mean_speckle_size'] == 0.0
    assert s['all']['n_speckles'] == 5 and s['all']['speckle_pixels'] == 20 and s['all']['density'] == 140 / 200
    assert s['left']['epe'] == 1.0 and s['all']['bad'] == [16 / 70, 4 / 70] and s['thresholds'] == [1.0, 3.0]


# ---- driver runs through a fake forward -----------------------------------------------------------------------------------
_H = _W = 2


def _sample(i):
    g = torch.Generator().manual_seed(7000 + i)

    def r(*shape, hi=1 << 20):
        return torch.randint(0, hi, (1,) + shape, generator=g)
    return {'disp_left': torch.full((1, 1, _H, _W), float(i)), 'disp_right': torch.zeros(1, 1, _H, _W),
            'voxels': torch.rand(1, 6, 6, 6, generator=g), 'iou_counts': r(4, 2, hi=1 << 15),
            'points': torch.full((1, 4, 3), float(i)), 'point_stats': torch.cat([r(2, 3), r(2, 2, hi=5)], -1),
            'disp_stats': r(2, 4), 'lr_mask': r(2, _H, _W, hi=2).to(torch.uint8), 'lr_stats': r(2, 5),
            'speckle_mask': r(2, _H, _W, hi=2).to(torch.uint8), 'speckle_stats': r(2, 7),
            'disp_std': torch.rand(1, 2, _H, _W, generator=g), 'unc_stats': r(2, 3, 5),
            'cloud_xyz': torch.rand(1, 2 * _H * _W, 3, generator=g), 'cloud_rgb': r(2 * _H * _W, 3, hi=256).to(torch.uint8),
            'cloud_counts': r(2, hi=_H * _W + 1).to(torch.int32), 'surf_stats': r(4, 2, 5, hi=50)}


class _Fake:
    """A forward that returns its outputs in the order output_names gives for the keywords it is called with."""

    def __init__(self, cls):
        self.cls, self.calls = cls, []

    def __call__(self, left, right, gt=None, **kw):
        self.calls.append(set(kw))
        on = {k: True for k in ('lr_check', 'speckle', 'uncertainty', 'surface') if kw.get(k)}
        names = self.cls.output_names(gt=gt is not None, disp_gt='disp_gt' in kw, camera='camera' in kw, **on)
        smp = [_sample(int(v)) for v in left[:, 0, 0, 0].tolist()]
        return tuple(torch.cat([s[n] for s in smp]) for n in names)


def _patch(mp_):
    def pair(B, H, W, dmax, seed):
        x = torch.full((1, 3, _H, _W), float(seed))
        return x, x, torch.zeros(1, _H)
    mp_.setattr(synthetic, 'stereo_pair', pair)
    mp_.setattr(synthetic, 'gt_volume', lambda B, n, seed: torch.zeros(1, n, n, n, dtype=torch.uint8))
    mp_.setattr(synthetic, 'point_clouds', lambda B, n, m, seed: (None, torch.zeros(1, m, 3)))
    mp_.setattr(T, '_disp_gt', lambda pairs, H, W, device: torch.zeros(len(pairs), 2, _H, _W))
    from stereo_3d_reconstruction_b200.extensions import chamfer_dist
    mp_.setattr(chamfer_dist, 'chamfer_per_sample', lambda a, b: a.double().mean((1, 2)) / 4)


@pytest.fixture
def patched(monkeypatch):
    _patch(monkeypatch)


def _run(model, n, bs, rank=0, world=1, **ev):
    cfg = _cfg(CONST__IMG_H=_H, CONST__IMG_W=_W)
    fn = T.test_voxel if model == 'Stereo2Voxel' else T.test_point
    cls = Stereo2Voxel if model == 'Stereo2Voxel' else Stereo2Point
    fake = _Fake(cls)
    return fn(cfg, fake, n, bs, rank, world, device='cpu', **ev), fake, cfg


@pytest.mark.parametrize('model', ['Stereo2Voxel', 'Stereo2Point'])
def test_driver_with_speckle(patched, model):
    n, bs = 7, 3
    ev = dict(eval_disp=True, eval_lr=True, eval_unc=True, eval_cloud=True)
    ev.update({'eval_surface': True} if model == 'Stereo2Voxel' else {'eval_points': True})
    got, fake, cfg = _run(model, n, bs, eval_speckle=True, **ev)
    assert all('speckle' in c for c in fake.calls) and len(fake.calls) == 3
    b = T.split_stats(got, T.stats_layout(cfg, model, eval_speckle=True, **ev))
    assert torch.equal(b['speckle'], sum(_sample(i)['speckle_stats'][0] for i in range(n)).flatten())
    off, fake_off, _ = _run(model, n, bs, **ev)
    assert all('speckle' not in c for c in fake_off.calls)
    assert torch.equal(torch.cat([v for k, v in b.items() if k != 'speckle']), off)


def _worker(rank, world, port, model, n, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    mpatch = pytest.MonkeyPatch()
    _patch(mpatch)
    ev = dict(eval_disp=True, eval_lr=True, eval_speckle=True)
    s, _, _ = _run(model, n, 2, rank, world, **ev)
    if rank == 0:
        q.put(s.tolist())
    dist.destroy_process_group()


@pytest.mark.parametrize('model', ['Stereo2Voxel', 'Stereo2Point'])
def test_gloo_world2_speckle_vector_matches_single_process(patched, model):
    n = 9
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker, args=(r, 2, port, model, n, q)) for r in range(2)]
    [p.start() for p in ps]
    got = q.get(timeout=120)
    [p.join(60) for p in ps]
    assert all(p.exitcode == 0 for p in ps)
    ref, _, cfg = _run(model, n, 2, eval_disp=True, eval_lr=True, eval_speckle=True)
    assert got == ref.tolist()
    b = T.split_stats(torch.tensor(got), T.stats_layout(cfg, model, eval_disp=True, eval_lr=True, eval_speckle=True))
    s = T.speckle_summary(b['speckle'], cfg.TEST.DISP_THRESH, n * _H * _W, b['disparity'])
    assert s['all']['n_speckles'] == s['left']['n_speckles'] + s['right']['n_speckles']


# ---- runner ---------------------------------------------------------------------------------------------------------------
def test_runner_speckle_argument(monkeypatch):
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--speckle'])
    assert runner.get_args().speckle is True
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test'])
    assert runner.get_args().speckle is False
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--speckle=1'])
    with pytest.raises(SystemExit):
        runner.get_args()
