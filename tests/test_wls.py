"""WLS filter, host side: the numpy statement of s3d_disp_wls (tests/wls_oracle.py) against scipy's banded solver in fp64 and
on exact cases, the weight table, the validation of the config keys, the forward's output order with wls=True, the test
driver's 'wls' block and summary, driver runs through a fake forward (also through a gloo world-2 all-reduce) and
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
from scipy.linalg import solve_banded

import runner
from stereo_3d_reconstruction_b200 import models, ops
from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.models import Stereo2Point, Stereo2Voxel
from tests import test_speckle as S
from tests import wls_oracle as O

f32 = np.float32
_LUT = ops.wls_weight_lut(1.5)


# ---- the rule ---------------------------------------------------------------------------------------------------------------
def test_weight_lut():
    assert _LUT.dtype == np.float32 and _LUT.shape == (3 * 255 ** 2 + 1,)
    assert _LUT[0] == 1.0 and _LUT[9] == np.float32(np.exp(-3.0 / 1.5))
    assert (_LUT[24323:] == 0).all() and _LUT[24322] > 0                   # strong edges decouple exactly at sigma = 1.5
    assert (np.diff(_LUT.astype(np.float64)) <= 0).all()
    for bad in (0, -1.0, float('nan'), float('inf'), 'a', None, True):
        with pytest.raises(ValueError):
            ops.wls_weight_lut(bad)


def test_one_pass_equals_the_banded_solve():
    # measured: over these lines the fp32 elimination is within 2.4e-4 of fp64, relative to the largest |u|; 5e-4 is the bound
    rng = np.random.default_rng(0)
    n, worst = 256, 0.0
    for lam in (1.0, 100.0, 8000.0):
        w = rng.random((8, n - 1)).astype(f32)
        w[:, rng.random(n - 1) < 0.1] = 0
        k = (f32(lam) * w).astype(f32)
        f = (rng.random((8, n)) * 30).astype(f32)
        c = (rng.random((8, n)) < 0.5).astype(f32)
        uf, uc = O.solve_lines(f, c, k)
        for li in range(8):
            kk = k[li].astype(np.float64)
            kl, kr = np.r_[0, kk], np.r_[kk, 0]
            ab = np.zeros((3, n))
            ab[0, 1:], ab[1], ab[2, :-1] = -kk, 1 + kl + kr, -kk
            for got, rhs in ((uf[li], f[li]), (uc[li], c[li])):
                ref = solve_banded((1, 1), ab, rhs.astype(np.float64))
                worst = max(worst, np.abs(got - ref).max() / max(np.abs(ref).max(), 1e-30))
    assert worst < 5e-4, worst


def _flat(H, W, value=100):
    return np.full((1, H, W, 3), value, np.uint8)


def test_zero_weights_return_d_on_confident_pixels():
    # a guide whose every edge has s >= 24323 (a checkerboard of 0 and 255 in every channel) has every weight exactly 0
    H, W = 6, 9
    img = np.where((np.indices((H, W)).sum(0) % 2 == 0)[..., None], 255, 0).astype(np.uint8)[None].repeat(3, -1)[..., :3]
    rng = np.random.default_rng(1)
    d = (rng.random((2, H, W)) * 20).astype(f32)
    d[0, 1, 2], d[1, 3, 3], d[0, 4, 4] = np.nan, np.inf, -np.inf
    out, st = O.disp_wls(d, 1, img, img, _LUT, 8000.0)
    conf = np.isfinite(d)
    assert np.array_equal(out[conf], d[conf]) and np.isnan(out[~conf]).all()
    assert st[0, :, 0].tolist() == [H * W - 2, H * W - 1] and st[0, :, 3].tolist() == st[0, :, 0].tolist()


def test_zero_weight_edge_separates_the_halves():
    H, W = 8, 12
    img = np.zeros((1, H, W, 3), np.uint8)
    img[:, :, W // 2:] = 255                                                # a vertical edge of weight 0 across the image
    rng = np.random.default_rng(2)
    d = (rng.random((2, H, W)) * 20).astype(f32)
    d[:, rng.random((H, W)) < 0.3] = np.nan
    e = d.copy()
    e[:, :, :W // 2] = (rng.random((2, H, W // 2)) * 50).astype(f32)       # other values on the left half
    a, _ = O.disp_wls(d, 1, img, img, _LUT, 8000.0)
    b, _ = O.disp_wls(e, 1, img, img, _LUT, 8000.0)
    assert np.array_equal(a[:, :, W // 2:], b[:, :, W // 2:], equal_nan=True)
    assert not np.array_equal(a[:, :, :W // 2], b[:, :, :W // 2], equal_nan=True)


def test_no_confident_pixel_is_nan_everywhere():
    d = np.full((2, 5, 7), np.nan, f32)
    d[1, 2, 3] = np.inf
    mask = np.zeros((1, 2, 5, 7), np.uint8)
    for m in (None, mask):
        out, st = O.disp_wls(d if m is None else np.ones_like(d), 1, _flat(5, 7), _flat(5, 7), _LUT, 8000.0, mask=m)
        assert np.isnan(out).all() and st.sum() == 0


def test_counters_by_hand():
    # a flat guide and one confident pixel per map: every pixel is reached, and the fill is the pixel's value
    H, W = 3, 4
    d = np.full((2, H, W), np.nan, f32)
    d[0, 1, 1], d[1, 0, 0] = 2.0, 5.0
    g = np.full((1, 2, H, W), np.nan, f32)
    g[0, 0, 0, :] = [1.0, 2.5, -1.0, 100.0]                                # errors 1, 0.5, invalid, invalid
    g[0, 1, 2, 3] = 5.0                                                     # error 0
    out, st = O.disp_wls(d, 1, _flat(H, W), _flat(H, W), _LUT, 8000.0, disp_gt=g, thresholds=(0.5, 0.75), max_gt=64.0)
    assert np.isfinite(out).all()
    assert np.abs(out[0] - 2.0).max() < 1e-5 and np.abs(out[1] - 5.0).max() < 1e-5
    e0 = np.abs(out[0, 0, :2] - g[0, 0, 0, :2]).astype(f32)
    q0 = int(np.rint(e0.astype(np.float64) * 65536).sum())
    e1 = np.abs(out[1, 2, 3] - f32(5.0))
    # [n_finite, n_valid_finite, q, bad(0.5), bad(0.75), n_conf]
    assert st[0, 0].tolist() == [12, 2, q0, int((e0 > 0.5).sum()), int((e0 > 0.75).sum()), 1]
    assert st[0, 1].tolist() == [12, 1, int(np.rint(np.float64(e1) * 65536)), int(e1 > 0.5), int(e1 > 0.75), 1]
    mask = np.ones((1, 2, H, W), np.uint8)
    mask[0, 1, 0, 0] = 2                                                    # the only confident pixel of view 1 is masked
    out, st = O.disp_wls(d, 1, _flat(H, W), _flat(H, W), _LUT, 8000.0, mask=mask)
    assert np.isnan(out[1]).all() and st[0, 1].tolist() == [0, 0, 0, 0] and st[0, 0].tolist() == [12, 0, 0, 1]


def test_fp32_guides_use_the_cloud_colour_rule():
    rng = np.random.default_rng(3)
    H, W = 5, 6
    f = rng.random((1, 3, H, W)).astype(f32)
    f[0, 0, 1, 1], f[0, 1, 2, 2], f[0, 2, 3, 3] = np.nan, 2.0, -1.0
    u = np.stack([O.colour(f[0], False)]).astype(np.uint8)
    d = (rng.random((2, H, W)) * 10).astype(f32)
    d[:, rng.random((H, W)) < 0.4] = np.nan
    a, sa = O.disp_wls(d, 1, f, f, _LUT, 8000.0)
    b, sb = O.disp_wls(d, 1, u, u, _LUT, 8000.0)
    assert np.array_equal(a, b, equal_nan=True) and np.array_equal(sa, sb)


# ---- config -------------------------------------------------------------------------------------------------------------
def test_config_defaults():
    from config import cfg
    assert models.wls_params(cfg) == (8000.0, 1.5)
    assert models.wls_params(S._cfg(TEST__WLS_LAMBDA=1, TEST__WLS_SIGMA=0.25)) == (1.0, 0.25)


@pytest.mark.parametrize('key', ['WLS_LAMBDA', 'WLS_SIGMA'])
@pytest.mark.parametrize('v', [0, -0.5, float('nan'), float('inf'), 1e39, 1e-50, 'a', None, True])
def test_wls_params_reject(key, v):
    with pytest.raises(ValueError, match=key):
        models.wls_params(S._cfg(**{'TEST__' + key: v}))


def test_forward_rejects_bad_wls_config_before_any_launch():
    x = torch.zeros(1, 3, 64, 64)
    for name in ('Stereo2Voxel', 'Stereo2Point'):
        m = models.build_model(name, S._cfg(TEST__WLS_LAMBDA=-1.0))
        with pytest.raises(ValueError, match='WLS_LAMBDA'):
            m(x, x, wls=True)
        with pytest.raises(ValueError, match='WLS_LAMBDA'):
            m.graphed(x, x, lr_check=True, wls=True)


# ---- the forward's output order -------------------------------------------------------------------------------------------
@pytest.mark.parametrize('flags', list(itertools.product([False, True], repeat=6)))
def test_output_names_with_wls(flags):
    gt, disp_gt, lr_check, speckle, uncertainty, camera = flags
    for cls in (Stereo2Voxel, Stereo2Point):
        kw = dict(gt=gt, disp_gt=disp_gt, lr_check=lr_check, speckle=speckle, uncertainty=uncertainty, camera=camera)
        off = cls.output_names(**kw)
        on = cls.output_names(wls=True, **kw)
        i = (off.index('speckle_stats') + 1 if speckle else off.index('lr_stats') + 1 if lr_check
             else len(cls.HEAD_OUTPUTS) + gt + disp_gt)
        assert on == off[:i] + ('wls_left', 'wls_right', 'wls_stats') + off[i:]
        assert cls.output_names(wls=False, **kw) == off


def test_wls_in_the_declared_orders():
    names = [o for o, _ in models.OPTIONAL_OUTPUTS]
    assert names.index('wls') == names.index('speckle') + 1 and names.index('camera') == names.index('uncertainty') + 1
    assert dict(models.OPTIONAL_OUTPUTS)['wls'] == ('wls_left', 'wls_right', 'wls_stats')
    f = models.Options._fields
    assert f.index('wls') == f.index('speckle') + 1 and f[-1] == 'fscore_curves'
    assert 'wls' in Stereo2Voxel.OPTIONS and 'wls' in Stereo2Point.OPTIONS
    assert Stereo2Point.output_names(gt=True, disp_gt=True, lr_check=True, speckle=True, wls=True, uncertainty=True,
                                     camera=True, fscore_curves=True) == (
        'disp_left', 'disp_right', 'points', 'point_stats', 'disp_stats', 'lr_mask', 'lr_stats', 'speckle_mask',
        'speckle_stats', 'wls_left', 'wls_right', 'wls_stats', 'disp_std', 'unc_stats', 'cloud_xyz', 'cloud_rgb',
        'cloud_counts', 'dist_hist')


# ---- stats block and summary ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize('model', ['Stereo2Voxel', 'Stereo2Point'])
def test_wls_block(model):
    tail = {'eval_surface': True} if model == 'Stereo2Voxel' else {'eval_points': True}
    cfg = S._cfg()
    for lr, spk in itertools.product((False, True), repeat=2):
        ev = dict(eval_disp=True, eval_lr=lr, eval_speckle=spk, eval_unc=True, eval_cloud=True, **tail)
        on = T.stats_layout(cfg, model, eval_wls=True, **ev)
        off = T.stats_layout(cfg, model, **ev)
        names = [b for b, _ in on]
        assert names.index('wls') == names.index('speckle' if spk else 'lr_consistency' if lr else 'disparity') + 1
        assert names.index('uncertainty') == names.index('wls') + 1 and dict(on)['wls'] == 2 * (4 + 2)
        assert [b for b in on if b[0] != 'wls'] == off
        assert T.stats_layout(cfg, model, **ev, eval_wls=False) == off
    with pytest.raises(ValueError, match='eval_wls=True needs eval_disp'):
        T.stats_layout(cfg, model, eval_wls=True)
    with pytest.raises(ValueError, match='WLS_SIGMA'):
        T.stats_layout(S._cfg(TEST__WLS_SIGMA=0.0), model, eval_disp=True, eval_wls=True)


def test_wls_summary():
    # per view [n_finite, n_valid_finite, q, bad(1), bad(3), n_conf]; T = 2
    block = torch.tensor([90, 40, 40 << 16, 10, 4, 30, 100, 50, 100 << 16, 5, 0, 100])
    disp = torch.tensor([50, 0, 0, 0, 80, 0, 0, 0])
    s = T.wls_summary(block, [1.0, 3.0], 100, disp)
    assert s['thresholds'] == [1.0, 3.0]
    assert s['left'] == {'n_finite': 90, 'density': 0.9, 'filled': 60, 'n_valid_finite': 40, 'valid_covered': 0.8,
                         'epe': 1.0, 'bad': [0.25, 0.1]}
    assert s['right'] == {'n_finite': 100, 'density': 1.0, 'filled': 0, 'n_valid_finite': 50, 'valid_covered': 50 / 80,
                          'epe': 2.0, 'bad': [0.1, 0.0]}
    assert s['all'] == {'n_finite': 190, 'density': 0.95, 'filled': 60, 'n_valid_finite': 90, 'valid_covered': 90 / 130,
                        'epe': 140 / 90, 'bad': [15 / 90, 4 / 90]}


# ---- driver runs through a fake forward -----------------------------------------------------------------------------------
def _sample(i):
    s = S._sample(i)
    g = torch.Generator().manual_seed(9000 + i)
    s.update(wls_left=torch.rand(1, 1, S._H, S._W, generator=g), wls_right=torch.rand(1, 1, S._H, S._W, generator=g),
             wls_stats=torch.randint(0, 1 << 20, (1, 2, 6), generator=g))
    return s


class _Fake(S._Fake):
    def __call__(self, left, right, gt=None, **kw):
        self.calls.append(set(kw))
        on = {k: True for k in ('lr_check', 'speckle', 'wls', 'uncertainty', 'surface') if kw.get(k)}
        names = self.cls.output_names(gt=gt is not None, disp_gt='disp_gt' in kw, camera='camera' in kw, **on)
        smp = [_sample(int(v)) for v in left[:, 0, 0, 0].tolist()]
        return tuple(torch.cat([s[n] for s in smp]) for n in names)


def _run(model, n, bs, rank=0, world=1, **ev):
    cfg = S._cfg(CONST__IMG_H=S._H, CONST__IMG_W=S._W)
    fn = T.test_voxel if model == 'Stereo2Voxel' else T.test_point
    fake = _Fake(Stereo2Voxel if model == 'Stereo2Voxel' else Stereo2Point)
    return fn(cfg, fake, n, bs, rank, world, device='cpu', **ev), fake, cfg


@pytest.mark.parametrize('model', ['Stereo2Voxel', 'Stereo2Point'])
def test_driver_with_wls(monkeypatch, model):
    S._patch(monkeypatch)
    n, bs = 7, 3
    ev = dict(eval_disp=True, eval_lr=True, eval_speckle=True, eval_unc=True, eval_cloud=True)
    ev.update({'eval_surface': True} if model == 'Stereo2Voxel' else {'eval_points': True})
    got, fake, cfg = _run(model, n, bs, eval_wls=True, **ev)
    assert all('wls' in c for c in fake.calls) and len(fake.calls) == 3
    b = T.split_stats(got, T.stats_layout(cfg, model, eval_wls=True, **ev))
    assert torch.equal(b['wls'], sum(_sample(i)['wls_stats'][0] for i in range(n)).flatten())
    off, fake_off, _ = _run(model, n, bs, **ev)
    assert all('wls' not in c for c in fake_off.calls)
    assert torch.equal(torch.cat([v for k, v in b.items() if k != 'wls']), off)


def _worker(rank, world, port, model, n, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    mpatch = pytest.MonkeyPatch()
    S._patch(mpatch)
    s, _, _ = _run(model, n, 2, rank, world, eval_disp=True, eval_wls=True)
    if rank == 0:
        q.put(s.tolist())
    dist.destroy_process_group()


@pytest.mark.parametrize('model', ['Stereo2Voxel', 'Stereo2Point'])
def test_gloo_world2_wls_vector_matches_single_process(monkeypatch, model):
    S._patch(monkeypatch)
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
    ref, _, cfg = _run(model, n, 2, eval_disp=True, eval_wls=True)
    assert got == ref.tolist()
    b = T.split_stats(torch.tensor(got), T.stats_layout(cfg, model, eval_disp=True, eval_wls=True))
    s = T.wls_summary(b['wls'], cfg.TEST.DISP_THRESH, n * S._H * S._W, b['disparity'])
    assert s['all']['filled'] == s['left']['filled'] + s['right']['filled']


# ---- runner ---------------------------------------------------------------------------------------------------------------
def test_runner_wls_argument(monkeypatch):
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--wls'])
    assert runner.get_args().wls is True
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test'])
    assert runner.get_args().wls is False
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--wls=1'])
    with pytest.raises(SystemExit):
        runner.get_args()
