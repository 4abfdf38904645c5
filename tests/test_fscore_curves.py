"""Nearest-neighbour distance histograms, host side: the reference statement in tests/fscore_curves_oracle.py against the
existing point / surface counters, tie handling at the edges, TEST.DIST_BINS / DIST_MAX validation, the point_curves /
surface_curves blocks of the stats vector (layout, block and summary arithmetic), a driver run per model through a fake
forward, and a gloo world-2 all-reduce."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from stereo_3d_reconstruction_b200 import models
from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.models import Stereo2Point, Stereo2Voxel, dist_edges
from stereo_3d_reconstruction_b200.utils import synthetic
from tests import fscore_curves_oracle as O
from tests import point_oracle as PO
from tests import surface_oracle as SO
from tests.common import small_cfg

FX = 1 << 32


def _dists(B, n, seed):
    """Squared distances with NaN, +-inf, values >= 2^8, exact squares of edges and zeros among random ones."""
    rng = np.random.default_rng(seed)
    d = (rng.random((B, n)) ** 3 * 0.03).astype(np.float32)
    sel = rng.random(d.shape)
    for lo, x in ((0.02, np.nan), (0.04, np.inf), (0.05, -np.inf), (0.06, 256.0), (0.07, 1e6), (0.1, 0.0)):
        d[(sel >= lo - 0.01) & (sel < lo)] = x
    return d


# ---- the histogram rule against the existing counters --------------------------------------------------------------------
@pytest.mark.parametrize('K', [1, 2, 16, 128, 1024])
def test_point_cumulative_counts_equal_the_tau_counters(K):
    e = O.edges(0.128, K)
    d1, d2 = _dists(3, 50, K), _dists(3, 70, K + 1)
    d1[0, :5] = e[:5] ** 2 if K >= 5 else d1[0, :5]               # squares of edges: sqrt_rn lands on or next to them
    h = O.point_hist_of_dists(d1, d2, e)
    assert h[:, 0].sum(-1).tolist() == [50] * 3 and h[:, 1].sum(-1).tolist() == [70] * 3
    counts = PO.point_counts(d1, d2, [float(x) for x in e])       # count(sqrt_rn(d) < tau) at tau = every fp32 edge
    assert np.array_equal(np.cumsum(h[..., :K], -1), counts[..., 3:])
    assert (h[..., K] >= counts[..., 2]).all()                   # every out-of-range point is in bin K


def test_surface_cumulative_counts_equal_the_surface_counters():
    rng = np.random.default_rng(3)
    n, e = 6, O.edges(0.5, 20)
    fused = rng.random((4, n, n, n)).astype(np.float32)
    gt = (rng.random((4, n, n, n)) < 0.4).astype(np.uint8)
    gt[1] = 0                                                     # empty GT: predicted points all in bin K
    fused[2] = 0.0                                                # empty prediction
    vt = [0.3, 0.7]
    h = O.surface_hist(fused, gt, vt, e)
    st = SO.surface_stats(fused, gt, vt, [float(x) for x in e])
    assert np.array_equal(h.sum(-1), st[..., 0])                  # rows sum to n_pts
    cum = np.cumsum(h[..., :len(e)], -1)
    assert np.array_equal(cum, st[..., 3:])                       # = count(s < voxel_kbound(e_k))
    assert (h[1, :, 0, :len(e)] == 0).all() and (h[1, :, 0, len(e)] == st[1, :, 0, 0]).all()


def test_ties_go_to_the_bin_above():
    e = np.array([0.25, 0.5, 0.75], np.float32)
    d = np.array([[0.0625, 0.25, 0.5625, 0.0624, 1.0, np.nan]], np.float32)   # sqrt = e_1, e_2, e_3 exactly
    assert O.point_bins(d, e).tolist() == [[1, 2, 3, 0, 3, 3]]
    assert np.sqrt(np.float32(0.5625)) == np.float32(0.75)
    kb = O.kbounds(np.array([0.25, 0.5], np.float32), 2)          # (4 * 0.25)^2 = 1, (4 * 0.5)^2 = 4
    assert kb.tolist() == [1, 4]
    assert np.searchsorted(kb, np.array([0, 1, 3, 4, 5]), side='right').tolist() == [0, 1, 1, 2, 2]


def test_repeated_bounds_give_empty_bins():
    kb = O.kbounds(O.edges(0.01, 8), 2)                           # 2n e <= 0.04: every bound is 1
    assert kb.tolist() == [1] * 8
    assert np.bincount(np.searchsorted(kb, np.array([0, 1, 2]), side='right'), minlength=9).tolist() == \
        [1, 0, 0, 0, 0, 0, 0, 0, 2]


# ---- configuration ------------------------------------------------------------------------------------------------------
def test_default_edges():
    e = dist_edges(small_cfg())
    assert e.dtype == np.float32 and len(e) == 128
    assert e[9] == np.float32(0.01) and e[-1] == np.float32(0.128) and (np.diff(e) > 0).all()
    assert np.array_equal(e, O.edges(0.128, 128))


@pytest.mark.parametrize('bins,dmax', [(True, 0.1), (0, 0.1), (1025, 0.1), (2.0, 0.1), ('8', 0.1), (None, 0.1),
                                       (8, float('nan')), (8, -0.1), (8, 0.0), (8, float('inf')), (8, 'x'),
                                       (1024, 1e-42), (1024, 1e39)])
def test_dist_edges_rejects(bins, dmax):
    with pytest.raises(ValueError, match='TEST.DIST_'):
        dist_edges(small_cfg(TEST__DIST_BINS=bins, TEST__DIST_MAX=dmax))


def test_dist_edges_rejects_colliding_edges():
    # 1024 edges below 1e-40 are fp32 subnormals 2^-149 apart at best: consecutive edges round to one value
    with pytest.raises(ValueError, match='strictly increasing'):
        dist_edges(small_cfg(TEST__DIST_BINS=1024, TEST__DIST_MAX=1e-42))
    assert len(dist_edges(small_cfg(TEST__DIST_BINS=1, TEST__DIST_MAX=3.0))) == 1


# ---- blocks and summaries -----------------------------------------------------------------------------------------------
def test_point_block_and_summary():
    K, N, M = 16, 50, 70
    e = O.edges(0.02, K)
    h = O.point_hist_of_dists(_dists(5, N, 1), _dists(5, M, 2), e)
    blk = T.point_curves_block(torch.from_numpy(h), N, M)
    assert blk.tolist() == O.point_curves_block(h, N, M).tolist()
    s = T.point_curves_summary(blk, e, 5)
    prf = O.point_curves_block(h, N, M)[2 * (K + 1):].reshape(K, 3)
    ref = O.curves(h[:, 0].sum(0), h[:, 1].sum(0), prf, e, 5)
    for k in ref:
        assert s[k] == ref[k], k
    assert s['thresholds'] == [float(x) for x in e] and s['n_samples'] == 5
    assert s['hist_pred'] == h[:, 0].sum(0).tolist() and s['hist_gt'] == h[:, 1].sum(0).tolist()
    # the F-score at e_k equals the existing per-sample F-score at tau = e_k
    counts = PO.point_counts(*[_dists(5, n, sd) for n, sd in ((N, 1), (M, 2))], [float(x) for x in e])
    assert prf[:, 2].tolist() == PO.fscore_fx(counts, N, M).tolist()


def test_surface_block_and_summary():
    rng = np.random.default_rng(5)
    n, e, vt = 5, O.edges(0.6, 12), [0.2, 0.5, 0.9]
    fused = rng.random((3, n, n, n)).astype(np.float32)
    gt = (rng.random((3, n, n, n)) < 0.5).astype(np.uint8)
    gt[0] = 0
    h = O.surface_hist(fused, gt, vt, e)
    blk = T.surface_curves_block(torch.from_numpy(h))
    assert blk.tolist() == O.surface_curves_block(h).tolist()
    # the per-edge F-score sums equal the surface block's at tau = e_k
    st = SO.surface_stats(fused, gt, vt, [float(x) for x in e])
    sb = SO.surface_block(st, n)                                  # [T, 3 + 3F]
    w = 2 * 13 + 3 * 12
    for t in range(3):
        assert blk[t * w + 26:(t + 1) * w].tolist() == sb[t, 3:].tolist()
    s = T.surface_curves_summary(blk, vt, e, 3)
    assert [x['voxel_thresh'] for x in s['by_thresh']] == vt and s['thresholds'] == [float(x) for x in e]
    for t in range(3):
        r = O.surface_curves_block(h)[t * w:(t + 1) * w]
        ref = O.curves(r[:13], r[13:26], r[26:].reshape(12, 3), e, 3)
        for k in ref:
            assert s['by_thresh'][t][k] == ref[k], (t, k)


def test_accuracy_completeness_hand_built():
    e = np.array([1.0, 2.0, 3.0, 4.0], np.float32)
    # predicted: 10 points, 5 below e_1, 4 more below e_3, 1 beyond; GT: 10 points, 2 below e_4, 8 beyond
    h = torch.tensor([[[5, 0, 4, 0, 1], [0, 0, 0, 2, 8]]])
    s = T.point_curves_summary(T.point_curves_block(h, 10, 10), e, 1)
    assert s['accuracy'] == {'p50': 1.0, 'p90': 3.0}
    assert s['completeness'] == {'p50': None, 'p90': None}
    assert s['pooled_precision'] == [0.5, 0.5, 0.9, 0.9] and s['pooled_recall'] == [0.0, 0.0, 0.0, 0.2]
    def q(x):
        return round(x * FX) / FX
    assert s['precision'] == [0.5, 0.5, q(0.9), q(0.9)] and s['recall'] == [0.0, 0.0, 0.0, q(0.2)]
    f4 = round(2 * 0.9 * 0.2 / 1.1 * FX) / FX
    assert s['fscore'] == [0.0, 0.0, 0.0, f4] and s['fscore_auc'] == f4 / 4
    # 0.9 reached exactly (9 of 10): integer comparison, no rounding
    h = torch.tensor([[[0, 9, 0, 0, 1], [10, 0, 0, 0, 0]]])
    s = T.point_curves_summary(T.point_curves_block(h, 10, 10), e, 1)
    assert s['accuracy'] == {'p50': 2.0, 'p90': 2.0} and s['completeness'] == {'p50': 1.0, 'p90': 1.0}


def test_summary_of_nothing():
    e = O.edges(0.1, 4)
    s = T.point_curves_summary(torch.zeros(2 * 5 + 12, dtype=torch.int64), e, 0)
    assert s['fscore'] == [0.0] * 4 and s['accuracy'] == {'p50': None, 'p90': None} and s['fscore_auc'] == 0.0
    s = T.surface_curves_summary(torch.zeros(2 * (2 * 5 + 12), dtype=torch.int64), [0.3, 0.5], e, 0)
    assert len(s['by_thresh']) == 2 and s['by_thresh'][1]['completeness'] == {'p50': None, 'p90': None}


# ---- the stats vector ---------------------------------------------------------------------------------------------------
_TV, _TD, _F, _N, _NPTS, _M, _KB = 4, 2, 2, 6, 4, 8, 10
_NH, _ND = 2 * _TV + 1, 2 * (2 + _TD)
_NS, _NP = _TV * (3 + 3 * _F), 2 * (3 + _F) + _F
_NSC, _NPC = _TV * (2 * (_KB + 1) + 3 * _KB), 2 * (_KB + 1) + 3 * _KB


def _cfg():
    return small_cfg(TEST__VOXEL_THRESH=[0.2, 0.4, 0.6, 0.8], TEST__DISP_THRESH=[1.0, 3.0], TEST__FSCORE_THRESH=[0.05, 0.3],
                     TEST__DIST_BINS=_KB, TEST__DIST_MAX=0.5, CONST__N_VOX=_N, CONST__N_POINTS=_NPTS,
                     CONST__N_GT_POINTS=_M)


def test_stats_layout_with_fscore_curves():
    c = _cfg()
    assert T.stats_layout(c, 'Stereo2Voxel', eval_surface=True, eval_fscore_curves=True) == \
        [('iou', _NH), ('surface', _NS), ('surface_curves', _NSC)]
    assert T.stats_layout(c, 'Stereo2Voxel', eval_disp=True, eval_surface=True, eval_curves=True,
                          eval_fscore_curves=True)[-3:] == [('surface', _NS), ('curves', 4 * 256 + 2), ('surface_curves', _NSC)]
    assert T.stats_layout(c, 'Stereo2Point', eval_disp=True, eval_points=True, eval_fscore_curves=True) == \
        [('chamfer', 2), ('disparity', _ND), ('points', _NP), ('point_curves', _NPC)]
    assert T.stats_layout(small_cfg(), 'Stereo2Point', eval_points=True, eval_fscore_curves=True)[-1] == \
        ('point_curves', 2 * 129 + 3 * 128)
    with pytest.raises(ValueError, match='needs eval_surface=True'):
        T.stats_layout(c, 'Stereo2Voxel', eval_fscore_curves=True)
    with pytest.raises(ValueError, match='needs eval_points=True'):
        T.stats_layout(c, 'Stereo2Point', eval_fscore_curves=True)
    with pytest.raises(ValueError, match='TEST.DIST_BINS'):
        T.stats_layout(small_cfg(TEST__DIST_BINS=0), 'Stereo2Point', eval_points=True, eval_fscore_curves=True)
    assert T.stats_layout(small_cfg(TEST__DIST_BINS=0), 'Stereo2Point', eval_points=True) == [('chamfer', 2), ('points', 9)]


def test_output_names_put_dist_hist_last():
    assert Stereo2Voxel.output_names(gt=True, disp_gt=True, lr_check=True, uncertainty=True, surface=True, mesh=True,
                                     curves=True, fscore_curves=True)[-4:] == ('mesh_counts', 'occ_hist', 'occ_loss',
                                                                               'dist_hist')
    assert Stereo2Point.output_names(gt=True, disp_gt=True, lr_check=True, uncertainty=True, fscore_curves=True) == (
        'disp_left', 'disp_right', 'points', 'point_stats', 'disp_stats', 'lr_mask', 'lr_stats', 'disp_std', 'unc_stats',
        'dist_hist')
    assert models.OPTIONAL_OUTPUTS[-1] == ('fscore_curves', ('dist_hist',))
    assert models.Options._fields[-1] == 'fscore_curves'


# ---- driver runs through fake forwards ----------------------------------------------------------------------------------
def _sample(i):
    """Seeded outputs of sample i, batch dim 1, keyed by name; dist_hist rows sum to the point counts."""
    g = torch.Generator().manual_seed(9000 + i)

    def r(*shape, hi=1 << 20):
        return torch.randint(0, hi, (1,) + shape, generator=g)

    def hist(*lead, total):
        cut = torch.sort(torch.randint(0, total + 1, (1,) + lead + (_KB,), generator=g), -1).values
        z = torch.zeros((1,) + lead + (1,), dtype=torch.int64)
        return torch.diff(torch.cat([z, cut, z + total], -1), dim=-1)
    sh = hist(_TV, 2, total=40)
    if i % 4 == 0:
        sh[0, :, 1] = 0                                            # an empty row: P or R is 0 there
    return {'disp_left': torch.full((1, 1, 2, 2), float(i)), 'disp_right': torch.zeros(1, 1, 2, 2),
            'voxels': torch.rand(1, _N, _N, _N, generator=g), 'iou_counts': r(_TV, 2, hi=1 << 15),
            'points': torch.full((1, _NPTS, 3), float(i)), 'point_stats': torch.cat([r(2, 3), r(2, _F, hi=_NPTS + 1)], -1),
            'disp_stats': r(2, 2 + _TD), 'surf_stats': r(_TV, 2, 3 + _F, hi=50),
            'point_hist': torch.cat([hist(1, total=_NPTS), hist(1, total=_M)], 1), 'surf_hist': sh}


class _Fake:
    """A forward in the tuple order written out independently: head, GT output, disp_stats, surf_stats, then dist_hist."""

    def __init__(self, head, gt_out, hist):
        self.head, self.gt_out, self.hist, self.calls = head, gt_out, hist, []

    def __call__(self, left, right, gt=None, **kw):
        self.calls.append(set(kw))
        ids = [int(v) for v in left[:, 0, 0, 0].tolist()]
        smp = [_sample(i) for i in ids]
        for s in smp:
            s['dist_hist'] = s[self.hist]
        names = ('disp_left', 'disp_right', self.head) + ((self.gt_out,) if gt is not None else ()) + \
            (('disp_stats',) if 'disp_gt' in kw else ()) + (('surf_stats',) if kw.get('surface') else ()) + \
            (('dist_hist',) if kw.get('fscore_curves') else ())
        return tuple(torch.cat([s[n] for s in smp]) for n in names)


def _patch(mpatch):
    def pair(B, H, W, dmax, seed):
        x = torch.full((1, 3, 2, 2), float(seed))
        return x, x, torch.zeros(1, 2, 2)
    mpatch.setattr(synthetic, 'stereo_pair', pair)
    mpatch.setattr(synthetic, 'gt_volume', lambda B, n, seed: torch.zeros(1, n, n, n, dtype=torch.uint8))
    mpatch.setattr(synthetic, 'point_clouds', lambda B, n, m, seed: (None, torch.zeros(1, m, 3)))
    mpatch.setattr(T, '_disp_gt', lambda pairs, H, W, device: torch.zeros(len(pairs), 2, 2, 2))
    from stereo_3d_reconstruction_b200.extensions import chamfer_dist
    mpatch.setattr(chamfer_dist, 'chamfer_per_sample', lambda a, b: a.double().mean((1, 2)) / 4)


def _want_voxel(ids):
    return torch.from_numpy(O.surface_curves_block(torch.cat([_sample(i)['surf_hist'] for i in ids]).numpy()))


def _want_point(ids):
    return torch.from_numpy(O.point_curves_block(torch.cat([_sample(i)['point_hist'] for i in ids]).numpy(), _NPTS, _M))


def test_voxel_driver_fscore_curves(monkeypatch):
    _patch(monkeypatch)
    n = 7
    model = _Fake('voxels', 'iou_counts', 'surf_hist')
    got = T.test_voxel(_cfg(), model, n, 3, device='cpu', eval_disp=True, eval_surface=True, eval_fscore_curves=True)
    assert model.calls == [{'disp_gt', 'surface', 'fscore_curves'}] * 3
    base = T.test_voxel(_cfg(), _Fake('voxels', 'iou_counts', 'surf_hist'), n, 3, device='cpu', eval_disp=True,
                        eval_surface=True)
    assert got.numel() == base.numel() + _NSC and torch.equal(got[:base.numel()], base)
    assert torch.equal(got[-_NSC:], _want_voxel(range(n)))
    other = T.test_voxel(_cfg(), _Fake('voxels', 'iou_counts', 'surf_hist'), n, 2, device='cpu', eval_surface=True,
                         eval_fscore_curves=True)
    assert torch.equal(other[-_NSC:], got[-_NSC:])                 # another batch split: the same integers
    with pytest.raises(ValueError, match='needs eval_surface'):
        T.test_voxel(_cfg(), model, n, 3, device='cpu', eval_fscore_curves=True)
    assert len(model.calls) == 3                                   # raised before any forward


def test_point_driver_fscore_curves(monkeypatch):
    _patch(monkeypatch)
    n = 7
    model = _Fake('points', 'point_stats', 'point_hist')
    got = T.test_point(_cfg(), model, n, 3, device='cpu', eval_disp=True, eval_points=True, eval_fscore_curves=True)
    assert model.calls == [{'disp_gt', 'fscore_curves'}] * 3
    base = T.test_point(_cfg(), _Fake('points', 'point_stats', 'point_hist'), n, 3, device='cpu', eval_disp=True,
                        eval_points=True)
    assert got.numel() == base.numel() + _NPC and torch.equal(got[:base.numel()], base)
    assert torch.equal(got[-_NPC:], _want_point(range(n)))
    with pytest.raises(ValueError, match='needs eval_points'):
        T.test_point(_cfg(), model, n, 3, device='cpu', eval_fscore_curves=True)
    assert len(model.calls) == 3


def _worker(rank, world, port, n, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    mp_patch = pytest.MonkeyPatch()
    _patch(mp_patch)
    v = T.test_voxel(_cfg(), _Fake('voxels', 'iou_counts', 'surf_hist'), n, 2, rank, world, device='cpu', eval_surface=True,
                     eval_fscore_curves=True)
    p = T.test_point(_cfg(), _Fake('points', 'point_stats', 'point_hist'), n, 2, rank, world, device='cpu',
                     eval_points=True, eval_fscore_curves=True)
    if rank == 0:
        q.put((v.tolist(), p.tolist()))
    dist.destroy_process_group()


def test_gloo_world2_fscore_curves_vectors_match_single_process(monkeypatch):
    n = 9
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0)); port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker, args=(r, 2, port, n, q)) for r in range(2)]
    [p.start() for p in ps]
    got_v, got_p = q.get(timeout=120)
    [p.join(60) for p in ps]
    assert all(p.exitcode == 0 for p in ps)
    _patch(monkeypatch)
    ref_v = T.test_voxel(_cfg(), _Fake('voxels', 'iou_counts', 'surf_hist'), n, 4, device='cpu', eval_surface=True,
                         eval_fscore_curves=True)
    ref_p = T.test_point(_cfg(), _Fake('points', 'point_stats', 'point_hist'), n, 4, device='cpu', eval_points=True,
                         eval_fscore_curves=True)
    assert got_v == ref_v.tolist() and got_p == ref_p.tolist()
    assert torch.equal(torch.tensor(got_v[-_NSC:]), _want_voxel(range(n)))
    assert torch.equal(torch.tensor(got_p[-_NPC:]), _want_point(range(n)))
