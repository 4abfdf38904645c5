"""Stereo point clouds, host side: the numpy statement of s3d_disp_cloud (tests/cloud_oracle.py) on hand-built cases, the
forward's output order with camera= on, the test driver's 'cloud' block and summary, the PLY writer, the validation of the
config keys and of runner.py's arguments, and driver runs through a fake forward."""
import itertools
import sys

import numpy as np
import pytest
import torch

import runner
from stereo_3d_reconstruction_b200 import models
from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.models import Stereo2Point, Stereo2Voxel
from stereo_3d_reconstruction_b200.utils import synthetic
from tests import cloud_oracle as O
from tests.common import small_cfg

f32 = np.float32
_NAN = float('nan')


def _one(disp, cam, min_disp=1.0, **kw):
    """Oracle on a single sample: disp fp32 [2,H,W] (view 0, view 1), fp32 zero images."""
    H, W = disp.shape[1:]
    img = np.zeros((1, 3, H, W), f32)
    return O.disp_cloud(disp, 1, img, img, np.asarray([cam], f32), min_disp, **kw)[0]


# ---- the rule on hand-built cases ---------------------------------------------------------------------------------------
def test_view1_point_is_view0_point_of_the_same_surface_point():
    # f * baseline = 128, d = 8: z = 16, s = 1/16, every value exact.  The surface point seen at x = 100 in the left image is at
    # x - d = 92 in the right one: the view-1 point is its view-0 point, the baseline added back exactly.
    cam = (256.0, 64.0, 32.0, 0.5, 0.0)
    disp = np.full((2, 48, 128), _NAN, f32)
    disp[0, 40, 100] = 8.0
    disp[1, 40, 92] = 8.0
    xyz, _, n = _one(disp, cam)
    assert n == (1, 1)
    assert xyz[0].tolist() == [2.25, 0.5, 16.0] and xyz[1].tolist() == xyz[0].tolist()
    # the baseline: the view-1 X minus the baseline is the plain back-projection of x = 92
    assert xyz[1, 0] - f32(0.5) == f32((92 - 64) / 16.0)


def test_doffs_shifts_the_disparity():
    cam0, cam2 = (256.0, 64.0, 32.0, 0.5, 0.0), (256.0, 64.0, 32.0, 0.5, 2.0)
    a = np.full((2, 4, 8), _NAN, f32)
    b = a.copy()
    a[0, 1, 3] = 8.0
    b[0, 1, 3] = 6.0                                       # 6 + doffs 2 = 8: the same depth
    assert np.array_equal(_one(a, cam0)[0], _one(b, cam2)[0])
    assert _one(b, cam2)[0][0, 2] == 16.0
    # doffs also moves the min_disp edge: 6 + 2 >= 8 is kept, 6 + 0 is not
    assert _one(b, cam2, min_disp=8.0)[2] == (1, 0) and _one(b, cam0, min_disp=8.0)[2] == (0, 0)


def test_min_disp_edge():
    cam = (100.0, 1.0, 1.0, 0.1, 0.25)
    md = f32(2.0)
    d = np.full((2, 1, 4), _NAN, f32)
    d[0, 0] = [md - f32(0.25), np.nextafter(md - f32(0.25), f32(0)), 0.0, -1.0]
    d[1, 0] = [np.inf, -np.inf, 5.0, md]
    xyz, _, n = _one(d, cam, min_disp=md)
    assert n == (1, 2)                                     # den == min_disp kept; one ulp below, 0, < 0, inf not
    assert xyz[0, 2] == f32(f32(f32(100.0) * f32(0.1)) / md)


def test_raster_order_and_views():
    cam = (1.0, 0.0, 0.0, 1.0, 0.0)                        # z = 1 / d, X = x z (+ 1 for view 1), Y = y z
    d = np.full((2, 3, 5), _NAN, f32)
    kept = [(0, 2, 4), (0, 0, 3), (1, 1, 0), (0, 2, 0), (1, 0, 1), (0, 1, 1)]
    for v, y, x in kept:
        d[v, y, x] = 1.0
    xyz, _, n = _one(d, cam)
    assert n == (4, 2)
    want = [[x + v, y, 1.0] for v, y, x in sorted(kept)]
    assert xyz.tolist() == want


def test_filters():
    cam = (2.0, 0.0, 0.0, 1.0, 0.0)
    d = np.full((2, 2, 3), 4.0, f32)
    mask = np.ones((1, 2, 2, 3), np.uint8)
    mask[0, 0, 0, 1] = 0
    mask[0, 1, 1, 2] = 2                                   # only 1 keeps
    std = np.zeros((1, 2, 2, 3), f32)
    std[0, 0, 1, 0] = _NAN                                 # never kept
    std[0, 1, 0, 0] = 0.5                                  # == max_std: kept
    std[0, 1, 0, 1] = np.nextafter(f32(0.5), f32(1))       # just above: not
    std[0, 0, 0, 2] = np.inf
    base = _one(d, cam)[2]
    assert base == (6, 6)
    assert _one(d, cam, lr_mask=mask)[2] == (5, 5)
    assert _one(d, cam, disp_std=std, max_std=0.5)[2] == (4, 5)
    assert _one(d, cam, lr_mask=mask, disp_std=std, max_std=0.5)[2] == (3, 4)
    # NaN and inf disparities are never kept, whatever the filters say
    d[0, 0, 0] = _NAN
    d[1, 0, 0] = -np.inf
    assert _one(d, cam)[2] == (5, 5)


def test_colours():
    v = np.array([_NAN, -1.0, 0.0, 0.5, 1.0, 2.0, np.inf, -np.inf, 0.25], f32)
    img = np.stack([v, v[::-1], v]).reshape(3, 1, 9)
    c = O.colour(img, False)
    assert c[0, :, 0].tolist() == [0, 0, 0, 128, 255, 255, 255, 0, 64]   # 127.5 -> 128 and 63.75 -> 64 (half to even, nearest)
    assert c[0, :, 1].tolist() == c[0, ::-1, 0].tolist()
    u = np.arange(27, dtype=np.uint8).reshape(1, 9, 3)
    assert np.array_equal(O.colour(u, True), u)


def test_colours_of_each_view():
    cam = (1.0, 0.0, 0.0, 1.0, 0.0)
    d = np.full((2, 1, 2), 1.0, f32)
    left = np.array([[[[0.0, 1.0]], [[0.5, 0.5]], [[1.0, 0.0]]]], f32)
    right = 1.0 - left
    _, rgb, n = O.disp_cloud(d, 1, left, right, np.asarray([cam], f32), 1.0)[0]
    assert n == (2, 2)
    assert rgb.tolist() == [[0, 128, 255], [255, 128, 0], [255, 128, 0], [0, 128, 255]]


# ---- the forward's output order -----------------------------------------------------------------------------------------
def _order(head, gt_out, gt, disp_gt, lr_check, uncertainty, camera, surface=False, mesh=False):
    """The tuple order of INTEGRATION.md with the stereo clouds right after the uncertainty outputs."""
    return (('disp_left', 'disp_right', head) + ((gt_out,) if gt else ()) + (('disp_stats',) if disp_gt else ()) +
            (('lr_mask', 'lr_stats') if lr_check else ()) + (('disp_std', 'unc_stats') if uncertainty else ()) +
            (('cloud_xyz', 'cloud_rgb', 'cloud_counts') if camera else ()) + (('surf_stats',) if surface else ()) +
            (('mesh_verts', 'mesh_faces', 'mesh_counts') if mesh else ()))


@pytest.mark.parametrize('flags', [f for f in itertools.product([False, True], repeat=6) if f[0] or not f[4]])
def test_voxel_output_names_with_camera(flags):
    gt, disp_gt, lr_check, uncertainty, surface, mesh = flags
    got = Stereo2Voxel.output_names(gt=gt, disp_gt=disp_gt, lr_check=lr_check, uncertainty=uncertainty, surface=surface,
                                    mesh=mesh, camera=True)
    assert got == _order('voxels', 'iou_counts', gt, disp_gt, lr_check, uncertainty, True, surface, mesh)
    off = Stereo2Voxel.output_names(gt=gt, disp_gt=disp_gt, lr_check=lr_check, uncertainty=uncertainty, surface=surface,
                                    mesh=mesh)
    assert off == _order('voxels', 'iou_counts', gt, disp_gt, lr_check, uncertainty, False, surface, mesh)


@pytest.mark.parametrize('flags', list(itertools.product([False, True], repeat=4)))
def test_point_output_names_with_camera(flags):
    got = Stereo2Point.output_names(**dict(zip(('gt', 'disp_gt', 'lr_check', 'uncertainty'), flags)), camera=True)
    assert got == _order('points', 'point_stats', *flags, True)


def test_every_option_with_camera():
    assert Stereo2Voxel.output_names(gt=True, disp_gt=True, lr_check=True, uncertainty=True, camera=True, surface=True,
                                     mesh=True, curves=True, fscore_curves=True) == (
        'disp_left', 'disp_right', 'voxels', 'iou_counts', 'disp_stats', 'lr_mask', 'lr_stats', 'disp_std', 'unc_stats',
        'cloud_xyz', 'cloud_rgb', 'cloud_counts', 'surf_stats', 'mesh_verts', 'mesh_faces', 'mesh_counts', 'occ_hist',
        'occ_loss', 'dist_hist')
    assert Stereo2Point.output_names(gt=True, disp_gt=True, lr_check=True, uncertainty=True, camera=True,
                                     fscore_curves=True) == (
        'disp_left', 'disp_right', 'points', 'point_stats', 'disp_stats', 'lr_mask', 'lr_stats', 'disp_std', 'unc_stats',
        'cloud_xyz', 'cloud_rgb', 'cloud_counts', 'dist_hist')
    names = [o for o, _ in models.OPTIONAL_OUTPUTS]
    assert names.index('camera') == names.index('uncertainty') + 1
    f = models.Options._fields
    assert f.index('camera') == f.index('uncertainty') + 1 and f[-1] == 'fscore_curves'


# ---- stats block, summary, PLY ------------------------------------------------------------------------------------------
def _cfg(**kw):
    return small_cfg(TEST__VOXEL_THRESH=[0.2, 0.4, 0.6, 0.8], TEST__DISP_THRESH=[1.0, 3.0], TEST__UNC_THRESH=[1.0, 2.0, 4.0],
                     TEST__FSCORE_THRESH=[0.05, 0.3], CONST__N_VOX=6, CONST__N_POINTS=4, CONST__N_GT_POINTS=8, **kw)


@pytest.mark.parametrize('model', ['Stereo2Voxel', 'Stereo2Point'])
def test_cloud_block_follows_uncertainty(model):
    tail = {'eval_surface': True} if model == 'Stereo2Voxel' else {'eval_points': True}
    on = T.stats_layout(_cfg(), model, eval_disp=True, eval_lr=True, eval_unc=True, eval_cloud=True, **tail)
    off = T.stats_layout(_cfg(), model, eval_disp=True, eval_lr=True, eval_unc=True, **tail)
    names = [b for b, _ in on]
    assert names.index('cloud') == names.index('uncertainty') + 1 and dict(on)['cloud'] == 2
    assert [b for b in on if b[0] != 'cloud'] == off
    assert T.stats_layout(_cfg(), model, eval_cloud=True)[1] == ('cloud', 2)


def test_cloud_summary():
    s = T.cloud_summary(torch.tensor([30, 10]), 4, 2, 5)
    assert s['n_samples'] == 4
    assert s['left'] == {'n_points': 30, 'per_sample': 7.5, 'kept_fraction': 0.75}
    assert s['right'] == {'n_points': 10, 'per_sample': 2.5, 'kept_fraction': 0.25}
    assert s['all'] == {'n_points': 40, 'per_sample': 10.0, 'kept_fraction': 0.5}
    assert T.cloud_summary(torch.tensor([0, 0]), 0, 2, 5)['all'] == {'n_points': 0, 'per_sample': 0.0, 'kept_fraction': 0.0}


def test_ply_round_trip(tmp_path):
    rng = np.random.default_rng(0)
    xyz = rng.standard_normal((37, 3)).astype(f32)
    xyz[0] = [np.float32(1e-38), -0.0, np.float32(3.4e38)]
    rgb = rng.integers(0, 256, (37, 3), dtype=np.uint8)
    T.write_ply(str(tmp_path / 'a.ply'), xyz, rgb)
    rec = O.read_ply(str(tmp_path / 'a.ply'))
    assert rec.dtype.names == ('x', 'y', 'z', 'red', 'green', 'blue')
    got = np.stack([rec['x'], rec['y'], rec['z']], 1)
    assert got.tobytes() == xyz.tobytes()
    assert np.array_equal(np.stack([rec['red'], rec['green'], rec['blue']], 1), rgb)
    assert (tmp_path / 'a.ply').stat().st_size == len((tmp_path / 'a.ply').read_bytes().split(b'end_header\n')[0]) + 11 + 37 * 15
    T.write_ply(str(tmp_path / 'e.ply'), np.zeros((0, 3), f32), np.zeros((0, 3), np.uint8))
    assert len(O.read_ply(str(tmp_path / 'e.ply'))) == 0


# ---- config and runner validation ---------------------------------------------------------------------------------------
def test_config_defaults():
    from config import cfg
    assert models.cloud_min_disp(cfg) == 1.0 and models.cloud_max_std(cfg) == 2.0
    assert models.camera_values(cfg) == [256.0, 127.5, 127.5, 0.1, 0.0]


@pytest.mark.parametrize('v', [0.0, -1.0, float('nan'), float('inf'), 'a', None, 1e-50])
def test_cloud_min_disp_rejects(v):
    with pytest.raises(ValueError, match='CLOUD_MIN_DISP'):
        models.cloud_min_disp(_cfg(TEST__CLOUD_MIN_DISP=v))


@pytest.mark.parametrize('v', [-0.5, float('nan'), float('inf'), 'a', None])
def test_cloud_max_std_rejects(v):
    with pytest.raises(ValueError, match='CLOUD_MAX_STD'):
        models.cloud_max_std(_cfg(TEST__CLOUD_MAX_STD=v))
    assert models.cloud_max_std(_cfg(TEST__CLOUD_MAX_STD=0)) == 0.0


@pytest.mark.parametrize('v', [[1.0, 2.0, 3.0], [1, 2, 3, 4, 5, 6], [0.0, 1, 1, 1], [1.0, 1, 1, -1], [1.0, 1, float('nan'), 1],
                               None, ['a', 1, 1, 1]])
def test_camera_values_rejects(v):
    with pytest.raises(ValueError, match='CONST.CAMERA'):
        models.camera_values(_cfg(CONST__CAMERA=v))
    assert models.camera_values(_cfg(CONST__CAMERA=[2, 3, 4, 5])) == [2.0, 3.0, 4.0, 5.0, 0.0]


def test_forward_rejects_bad_cloud_config_before_any_launch():
    m = models.build_model('Stereo2Point', _cfg(TEST__CLOUD_MIN_DISP=0.0))
    x = torch.zeros(1, 3, 64, 64)
    with pytest.raises(ValueError, match='CLOUD_MIN_DISP'):
        m(x, x, camera=torch.zeros(1, 5))
    m = models.build_model('Stereo2Voxel', _cfg(TEST__CLOUD_MAX_STD=-1.0))
    with pytest.raises(ValueError, match='CLOUD_MAX_STD'):
        m(x, x, uncertainty=True, camera=torch.zeros(1, 5))


def test_runner_camera_argument(monkeypatch):
    assert runner.camera_arg('256,127.5,127.5,0.1') == [256.0, 127.5, 127.5, 0.1, 0.0]
    assert runner.camera_arg('1,2,3,4,5') == [1.0, 2.0, 3.0, 4.0, 5.0]
    for bad in ('1,2,3', '1,2,3,4,5,6', '0,1,1,1', '1,1,1,0', '1,x,1,1', '1,nan,1,1', '1,1,1,inf'):
        with pytest.raises(Exception, match='f,cx,cy,baseline'):
            runner.camera_arg(bad)
        monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--save-clouds', 'd', '--camera', bad])
        with pytest.raises(SystemExit):
            runner.get_args()
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--camera', '1,2,3,4'])
    with pytest.raises(SystemExit, match='--save-clouds'):
        runner.main()


# ---- driver runs through a fake forward ---------------------------------------------------------------------------------
_H = _W = 2


def _sample(i):
    g = torch.Generator().manual_seed(9000 + i)

    def r(*shape, hi=1 << 20):
        return torch.randint(0, hi, (1,) + shape, generator=g)
    return {'disp_left': torch.full((1, 1, _H, _W), float(i)), 'disp_right': torch.zeros(1, 1, _H, _W),
            'voxels': torch.rand(1, 6, 6, 6, generator=g), 'iou_counts': r(4, 2, hi=1 << 15),
            'points': torch.full((1, 4, 3), float(i)), 'point_stats': torch.cat([r(2, 3), r(2, 2, hi=5)], -1),
            'disp_stats': r(2, 4), 'lr_mask': r(2, _H, _W, hi=2).to(torch.uint8), 'lr_stats': r(2, 5),
            'disp_std': torch.rand(1, 2, _H, _W, generator=g), 'unc_stats': r(2, 3, 5),
            'cloud_xyz': torch.rand(1, 2 * _H * _W, 3, generator=g), 'cloud_rgb': r(2 * _H * _W, 3, hi=256).to(torch.uint8),
            'cloud_counts': r(2, hi=_H * _W + 1).to(torch.int32), 'surf_stats': r(4, 2, 5, hi=50),
            'mesh_verts': torch.rand(1, 5, 3, generator=g), 'mesh_faces': r(4, 3, hi=5).to(torch.int32),
            'mesh_counts': r(2, hi=5).to(torch.int32)}


class _Fake:
    """A forward in the order of _order for the keywords it is given; records them and the cameras."""

    def __init__(self, head, gt_out):
        self.head, self.gt_out, self.calls, self.cameras = head, gt_out, [], []

    def __call__(self, left, right, gt=None, **kw):
        self.calls.append(set(kw))
        if 'camera' in kw:
            self.cameras.append(kw['camera'])
        ids = [int(v) for v in left[:, 0, 0, 0].tolist()]
        smp = [_sample(i) for i in ids]
        names = _order(self.head, self.gt_out, gt is not None, 'disp_gt' in kw, kw.get('lr_check', False),
                       kw.get('uncertainty', False), 'camera' in kw, kw.get('surface', False), kw.get('mesh', False))
        return tuple(torch.cat([s[n] for s in smp]) for n in names)


@pytest.fixture
def patched(monkeypatch):
    def pair(B, H, W, dmax, seed):
        x = torch.full((1, 3, _H, _W), float(seed))
        return x, x, torch.zeros(1, _H)
    monkeypatch.setattr(synthetic, 'stereo_pair', pair)
    monkeypatch.setattr(synthetic, 'gt_volume', lambda B, n, seed: torch.zeros(1, n, n, n, dtype=torch.uint8))
    monkeypatch.setattr(synthetic, 'point_clouds', lambda B, n, m, seed: (None, torch.zeros(1, m, 3)))
    monkeypatch.setattr(T, '_disp_gt', lambda pairs, H, W, device: torch.zeros(len(pairs), 2, _H, _W))
    saved = []
    monkeypatch.setattr(T, 'save_clouds', lambda cloud_dir, ids, cloud, left, right, camera, disp_gt, min_disp:
                        saved.append((cloud_dir, list(ids), cloud, camera, min_disp)))
    monkeypatch.setattr(T, 'save_meshes', lambda mesh_dir, ids, mesh, gt: None)
    from stereo_3d_reconstruction_b200.extensions import chamfer_dist
    monkeypatch.setattr(chamfer_dist, 'chamfer_per_sample', lambda a, b: a.double().mean((1, 2)) / 4)
    return saved


def _check_saved(saved, cloud_dir, n, bs, cam):
    assert [ids for _, ids, _, _, _ in saved] == [list(range(s, min(s + bs, n))) for s in range(0, n, bs)]
    for d, ids, (xyz, rgb, c), camera, md in saved:
        assert d == cloud_dir and md == 1.0
        assert torch.equal(camera, torch.tensor([cam] * len(ids), dtype=torch.float32))
        assert torch.equal(xyz, torch.cat([_sample(i)['cloud_xyz'] for i in ids]))
        assert torch.equal(rgb, torch.cat([_sample(i)['cloud_rgb'] for i in ids]))
        assert torch.equal(c, torch.cat([_sample(i)['cloud_counts'] for i in ids]))


def test_voxel_driver_with_clouds(patched, tmp_path):
    n, bs = 7, 3
    cam = [100.0, 1.0, 2.0, 0.5, 0.25]
    cfg = _cfg(CONST__IMG_H=_H, CONST__IMG_W=_W, CONST__CAMERA=cam)
    model = _Fake('voxels', 'iou_counts')
    ev = dict(eval_disp=True, eval_lr=True, eval_unc=True, eval_surface=True)
    got = T.test_voxel(cfg, model, n, bs, device='cpu', mesh_dir=str(tmp_path / 'm'), cloud_dir=str(tmp_path / 'c'),
                       eval_cloud=True, **ev)
    assert model.calls == [{'disp_gt', 'lr_check', 'uncertainty', 'camera', 'surface', 'mesh'}] * 3
    b = T.split_stats(got, T.stats_layout(cfg, 'Stereo2Voxel', eval_cloud=True, **ev))
    want = sum(_sample(i)['cloud_counts'][0].to(torch.int64) for i in range(n))
    assert torch.equal(b['cloud'], want)
    # every other block is what the same run without the clouds gives
    off = T.test_voxel(cfg, _Fake('voxels', 'iou_counts'), n, bs, device='cpu', **ev)
    assert torch.equal(torch.cat([v for k, v in b.items() if k != 'cloud']), off)
    _check_saved(patched, str(tmp_path / 'c'), n, bs, cam)
    assert (tmp_path / 'c').is_dir()


def test_point_driver_with_clouds(patched, tmp_path):
    n, bs = 5, 2
    cfg = _cfg(CONST__IMG_H=_H, CONST__IMG_W=_W)
    model = _Fake('points', 'point_stats')
    got = T.test_point(cfg, model, n, bs, device='cpu', eval_cloud=True, cloud_dir=str(tmp_path), eval_points=True)
    assert model.calls == [{'camera'}] * 3
    b = T.split_stats(got, T.stats_layout(cfg, 'Stereo2Point', eval_cloud=True, eval_points=True))
    assert list(b) == ['chamfer', 'cloud', 'points']
    assert torch.equal(b['cloud'], sum(_sample(i)['cloud_counts'][0].to(torch.int64) for i in range(n)))
    _check_saved(patched, str(tmp_path), n, bs, [256.0, 127.5, 127.5, 0.1, 0.0])
    # the clouds alone: evaluated, nothing written
    patched.clear()
    T.test_point(cfg, _Fake('points', 'point_stats'), n, bs, device='cpu', eval_cloud=True)
    assert patched == []


def test_driver_rejects_bad_cloud_arguments(patched, tmp_path):
    with pytest.raises(ValueError, match='cloud_dir needs eval_cloud'):
        T.test_voxel(_cfg(), _Fake('voxels', 'iou_counts'), 1, 1, device='cpu', cloud_dir=str(tmp_path))
    with pytest.raises(ValueError, match='CONST.CAMERA'):
        T.test_point(_cfg(CONST__CAMERA=[1.0]), _Fake('points', 'point_stats'), 1, 1, device='cpu', eval_cloud=True)
    with pytest.raises(ValueError, match='CLOUD_MAX_STD'):
        T.test_point(_cfg(TEST__CLOUD_MAX_STD=-1), _Fake('points', 'point_stats'), 1, 1, device='cpu', eval_disp=True,
                     eval_unc=True, eval_cloud=True)
