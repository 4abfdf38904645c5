"""The two declared layouts, host side: the forward's output order (models.py, output_names) for every supported set of
options against the order INTEGRATION.md states, the test driver's stats blocks (core/test.py, stats_layout) against the
block formulas, and one driver run per model with every evaluation on through a fake forward that returns that order."""
import itertools

import pytest
import torch

from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.models import Stereo2Point, Stereo2Voxel
from stereo_3d_reconstruction_b200.utils import synthetic
from tests.common import small_cfg


def _order(head, gt_out, gt, disp_gt, lr_check, uncertainty, surface=False, mesh=False):
    """The tuple order of INTEGRATION.md: the head, its GT output, disp_stats, lr_mask / lr_stats, disp_std / unc_stats,
    surf_stats, then the mesh."""
    return (('disp_left', 'disp_right', head) + ((gt_out,) if gt else ()) + (('disp_stats',) if disp_gt else ()) +
            (('lr_mask', 'lr_stats') if lr_check else ()) + (('disp_std', 'unc_stats') if uncertainty else ()) +
            (('surf_stats',) if surface else ()) + (('mesh_verts', 'mesh_faces', 'mesh_counts') if mesh else ()))


@pytest.mark.parametrize('flags', [f for f in itertools.product([False, True], repeat=6) if f[0] or not f[4]])
def test_voxel_output_names(flags):                                 # every supported set: surface=True needs gt
    gt, disp_gt, lr_check, uncertainty, surface, mesh = flags
    got = Stereo2Voxel.output_names(gt=gt, disp_gt=disp_gt, lr_check=lr_check, uncertainty=uncertainty, surface=surface,
                                    mesh=mesh)
    assert got == _order('voxels', 'iou_counts', *flags)


@pytest.mark.parametrize('flags', list(itertools.product([False, True], repeat=4)))
def test_point_output_names(flags):
    gt, disp_gt, lr_check, uncertainty = flags
    got = Stereo2Point.output_names(gt=gt, disp_gt=disp_gt, lr_check=lr_check, uncertainty=uncertainty)
    assert got == _order('points', 'point_stats', *flags)
    with pytest.raises(ValueError, match='Stereo2Voxel only'):
        Stereo2Point.output_names(gt=gt, surface=True)
    with pytest.raises(ValueError, match='Stereo2Voxel only'):
        Stereo2Point.output_names(gt=gt, mesh=True)


def test_full_voxel_tuple():
    assert Stereo2Voxel.output_names(gt=True, disp_gt=True, lr_check=True, uncertainty=True, surface=True, mesh=True) == (
        'disp_left', 'disp_right', 'voxels', 'iou_counts', 'disp_stats', 'lr_mask', 'lr_stats', 'disp_std', 'unc_stats',
        'surf_stats', 'mesh_verts', 'mesh_faces', 'mesh_counts')


# ---- the stats vector ---------------------------------------------------------------------------------------------------
_TV, _TD, _K, _F, _N = 4, 2, 3, 2, 6
_NH, _ND, _NL, _NU = 2 * _TV + 1, 2 * (2 + _TD), 2 * (3 + _TD), 2 * _K * (3 + _TD)
_NS, _NP = _TV * (3 + 3 * _F), 2 * (3 + _F) + _F
_NPTS, _M = 4, 8


def _cfg():
    return small_cfg(TEST__VOXEL_THRESH=[0.2, 0.4, 0.6, 0.8], TEST__DISP_THRESH=[1.0, 3.0], TEST__UNC_THRESH=[1.0, 2.0, 4.0],
                     TEST__FSCORE_THRESH=[0.05, 0.3], CONST__N_VOX=_N, CONST__N_POINTS=_NPTS, CONST__N_GT_POINTS=_M)


@pytest.mark.parametrize('flags', list(itertools.product([False, True], repeat=4)))
def test_stats_layout(flags):
    disp, lr, unc, last = flags
    for model, head, tail in (('Stereo2Voxel', ('iou', _NH), ('surface', _NS)), ('Stereo2Point', ('chamfer', 2), ('points', _NP))):
        ev = dict(eval_disp=disp, eval_lr=lr, eval_unc=unc)
        ev['eval_surface' if model == 'Stereo2Voxel' else 'eval_points'] = last
        if (lr or unc) and not disp:
            with pytest.raises(ValueError, match='needs eval_disp=True'):
                T.stats_layout(_cfg(), model, **ev)
            continue
        want = [head] + [b for b, on in ((('disparity', _ND), disp), (('lr_consistency', _NL), lr),
                                         (('uncertainty', _NU), unc), (tail, last)) if on]
        assert T.stats_layout(_cfg(), model, **ev) == want


def test_split_stats_gives_views_in_order():
    layout = [('iou', 3), ('disparity', 2), ('surface', 4)]
    s = torch.arange(9)
    b = T.split_stats(s, layout)
    assert list(b) == ['iou', 'disparity', 'surface']
    assert b['iou'].tolist() == [0, 1, 2] and b['disparity'].tolist() == [3, 4] and b['surface'].tolist() == [5, 6, 7, 8]
    b['disparity'] += 10
    assert s[3:5].tolist() == [13, 14]


# ---- one driver run per model with every evaluation on, through fakes in the forward's order -------------------------
def _sample(i):
    """Seeded outputs of sample i, batch dim 1, keyed by output name."""
    g = torch.Generator().manual_seed(7000 + i)

    def r(*shape, hi=1 << 20):
        return torch.randint(0, hi, (1,) + shape, generator=g)
    return {'disp_left': torch.full((1, 1, 2, 2), float(i)), 'disp_right': torch.zeros(1, 1, 2, 2),
            'voxels': torch.rand(1, _N, _N, _N, generator=g), 'iou_counts': r(_TV, 2, hi=1 << 15),
            'points': torch.full((1, _NPTS, 3), float(i)), 'point_stats': torch.cat([r(2, 3), r(2, _F, hi=_NPTS + 1)], -1),
            'disp_stats': r(2, 2 + _TD), 'lr_mask': r(2, 2, 2, hi=2).to(torch.uint8), 'lr_stats': r(2, 3 + _TD),
            'disp_std': torch.rand(1, 2, 2, 2, generator=g), 'unc_stats': r(2, _K, 3 + _TD),
            'surf_stats': r(_TV, 2, 3 + _F, hi=50), 'mesh_verts': torch.rand(1, 5, 3, generator=g),
            'mesh_faces': r(4, 3, hi=5).to(torch.int32), 'mesh_counts': r(2, hi=5).to(torch.int32)}


class _Fake:
    """A forward in the tuple order of INTEGRATION.md (_order, written out independently of output_names) for the keywords
    it is given; records them."""

    def __init__(self, head, gt_out):
        self.head, self.gt_out, self.calls = head, gt_out, []

    def __call__(self, left, right, gt=None, **kw):
        self.calls.append(set(kw))
        ids = [int(v) for v in left[:, 0, 0, 0].tolist()]
        smp = [_sample(i) for i in ids]
        names = _order(self.head, self.gt_out, gt is not None, 'disp_gt' in kw, kw.get('lr_check', False),
                       kw.get('uncertainty', False), kw.get('surface', False), kw.get('mesh', False))
        return tuple(torch.cat([s[n] for s in smp]) for n in names)


@pytest.fixture
def patched(monkeypatch):
    def pair(B, H, W, dmax, seed):
        x = torch.full((1, 3, 2, 2), float(seed))
        return x, x, torch.zeros(1, 2, 2)
    monkeypatch.setattr(synthetic, 'stereo_pair', pair)
    monkeypatch.setattr(synthetic, 'gt_volume', lambda B, n, seed: torch.zeros(1, n, n, n, dtype=torch.uint8))
    monkeypatch.setattr(synthetic, 'point_clouds', lambda B, n, m, seed: (None, torch.zeros(1, m, 3)))
    monkeypatch.setattr(T, '_disp_gt', lambda pairs, H, W, device: torch.zeros(len(pairs), 2, 2, 2))
    saved = []
    monkeypatch.setattr(T, 'save_meshes', lambda mesh_dir, ids, mesh, gt: saved.append((list(ids), mesh)))
    from stereo_3d_reconstruction_b200.extensions import chamfer_dist
    # the Chamfer of sample i is i / 4: a multiple of 2^-40, so the driver's per-batch rounding is exact
    monkeypatch.setattr(chamfer_dist, 'chamfer_per_sample', lambda a, b: a.double().mean((1, 2)) / 4)
    return saved


def test_voxel_driver_every_option(patched, tmp_path):
    n, bs = 7, 3
    model = _Fake('voxels', 'iou_counts')
    got = T.test_voxel(_cfg(), model, n, bs, device='cpu', eval_disp=True, eval_lr=True, eval_unc=True,
                       eval_surface=True, mesh_dir=str(tmp_path))
    assert model.calls == [{'disp_gt', 'lr_check', 'uncertainty', 'surface', 'mesh'}] * 3
    want = torch.zeros(_NH + _ND + _NL + _NU + _NS, dtype=torch.int64)
    for i in range(n):
        s = _sample(i)
        want[:_TV] += s['iou_counts'][0, :, 0]
        want[_TV:2 * _TV] += s['iou_counts'][0, :, 1]
        want[2 * _TV] += 1
        want[_NH:_NH + _ND] += s['disp_stats'].flatten()
        want[_NH + _ND:_NH + _ND + _NL] += s['lr_stats'].flatten()
        want[_NH + _ND + _NL:_NH + _ND + _NL + _NU] += s['unc_stats'].flatten()
        want[-_NS:] += T.surface_block(s['surf_stats'], _N)
    assert torch.equal(got, want)
    assert [ids for ids, _ in patched] == [[0, 1, 2], [3, 4, 5], [6]]
    for ids, (v, f, c) in patched:
        assert torch.equal(v, torch.cat([_sample(i)['mesh_verts'] for i in ids]))
        assert torch.equal(f, torch.cat([_sample(i)['mesh_faces'] for i in ids]))
        assert torch.equal(c, torch.cat([_sample(i)['mesh_counts'] for i in ids]))
    # the uncertainty and surface blocks without the LR block: the keywords of exactly the evaluations that are on
    model = _Fake('voxels', 'iou_counts')
    part = T.test_voxel(_cfg(), model, n, 2, device='cpu', eval_disp=True, eval_unc=True, eval_surface=True)
    assert model.calls == [{'disp_gt', 'uncertainty', 'surface'}] * 4
    assert torch.equal(part, torch.cat([want[:_NH + _ND], want[_NH + _ND + _NL:]]))


def test_point_driver_every_option(patched):
    n, bs = 7, 3
    model = _Fake('points', 'point_stats')
    got = T.test_point(_cfg(), model, n, bs, device='cpu', eval_disp=True, eval_lr=True, eval_points=True, eval_unc=True)
    assert model.calls == [{'disp_gt', 'lr_check', 'uncertainty'}] * 3
    want = torch.zeros(2 + _ND + _NL + _NU + _NP, dtype=torch.int64)
    for i in range(n):
        s = _sample(i)
        want[0] += i << 38                                          # i / 4 in 2^-40 units
        want[1] += 1
        want[2:2 + _ND] += s['disp_stats'].flatten()
        want[2 + _ND:2 + _ND + _NL] += s['lr_stats'].flatten()
        want[2 + _ND + _NL:2 + _ND + _NL + _NU] += s['unc_stats'].flatten()
        want[-_NP:] += T.point_block(s['point_stats'], _NPTS, _M)
    assert torch.equal(got, want)
