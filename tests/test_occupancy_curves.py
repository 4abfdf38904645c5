"""Threshold-free occupancy evaluation, host side: the reference statement in tests/curves_oracle.py against direct
thresholding and a sort-based AP, TEST.CURVE_BINS validation, the curves block of the stats vector (layout, block and summary
arithmetic), a driver run with every Stereo2Voxel evaluation through a fake forward, and a gloo world-2 all-reduce."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.models import Stereo2Voxel, curve_bins
from stereo_3d_reconstruction_b200.utils import synthetic
from tests import curves_oracle as O
from tests.common import small_cfg
from tests.test_output_layout import _order, _sample

FX20, FX32 = 1 << 20, 1 << 32


def _field(B, n, seed, K):
    """Random occupancy with values on bin edges, 0, 1, NaN, +-inf, negatives and values > 1, and a random GT."""
    rng = np.random.default_rng(seed)
    v = rng.random((B, n, n, n)).astype(np.float32)
    sel = rng.random(v.shape)
    v[sel < 0.1] = (rng.integers(0, K + 1, (sel < 0.1).sum()) / K).astype(np.float32)
    for lo, x in ((0.1, np.nan), (0.12, -0.25), (0.14, 1.5), (0.16, np.inf), (0.17, -np.inf), (0.18, 0.0), (0.2, 1.0)):
        v[(sel >= lo) & (sel < lo + 0.02)] = x
    gt = (rng.random(v.shape) < 0.3).astype(np.uint8) * rng.integers(1, 255, v.shape).astype(np.uint8)
    return v, gt


@pytest.mark.parametrize('K', [2, 16, 256])
def test_histogram_curves_equal_direct_thresholding(K):
    v, gt = _field(5, 6, seed=K, K=K)
    gt[1] = 0                                                     # an empty GT
    v[2] = 0.0                                                    # an empty prediction above t = 1/K
    gt[3] = 1                                                     # a full GT
    hist, loss = O.occupancy_curves(v, gt, K)
    assert hist[:, :2].sum((1, 2)).tolist() == [v[0].size] * 5
    blk = T.curves_block(torch.from_numpy(hist), torch.from_numpy(loss))
    assert blk.tolist() == O.curves_block(v, gt, K).tolist()      # per-sample IoUs: the histogram's equal direct ones
    s = T.curves_summary(blk, K, 5)
    ref = O.summary(v, gt, K)
    assert s['iou'] == ref['iou']
    assert np.allclose(s['mean_iou'], ref['mean_iou'], rtol=0, atol=1e-9)
    assert abs(s['ap'] - ref['ap']) < 1e-12
    assert abs(s['bce'] - ref['bce']) < 1e-6 and abs(s['brier'] - ref['brier']) < 1e-6
    assert abs(s['ece'] - ref['ece']) < 1e-6
    assert s['thresholds'] == [k / K for k in range(K)] and s['n_voxels'] == v.size
    assert sum(r['count'] for r in s['reliability']) == v.size and len(s['reliability']) == min(K, 16)


def test_empty_gt_and_empty_prediction_count_as_iou_one():
    K = 8
    v = np.zeros((2, 2, 2, 2), np.float32)
    gt = np.zeros((2, 2, 2, 2), np.uint8)
    v[1, 0, 0, 0] = 0.5                                           # sample 1: one voxel predicted up to t = 0.5
    blk = T.curves_block(*map(torch.from_numpy, O.occupancy_curves(v, gt, K)))
    miou = blk[3 * K + 2:].tolist()
    # t = 0: every voxel is predicted, IoU 0; above it sample 0 predicts nothing (IoU 1), sample 1 one voxel up to bin 4
    assert miou == [0] + [FX32] * 4 + [2 * FX32] * 3
    s = T.curves_summary(blk, K, 2)
    assert s['ap'] is None and s['iou'] == [0.0] * 5 + [1.0] * 3
    assert s['mean_iou'] == [0.0] + [0.5] * 4 + [1.0] * 3
    assert O.summary(v, gt, K)['iou'] == s['iou']


def test_ap_equals_sort_based_on_ties():
    K = 4
    v = np.array([[0.9, 0.9, 0.8, 0.6, 0.3, 0.1, 0.0, 0.74]], np.float32)
    gt = np.array([[1, 0, 1, 0, 1, 0, 0, 1]], np.uint8)
    blk = T.curves_block(*map(torch.from_numpy, O.occupancy_curves(v, gt, K)))
    ap = T.curves_summary(blk, K, 1)['ap']
    # G = 4; bin 3: 2 of 3 occupied (R 1/2, P 2/3), bin 2: 1 of 2 (R 3/4, P 3/5), bin 1: 1 of 1 (R 1, P 4/6), bin 0: none
    assert abs(ap - (0.5 * 2 / 3 + 0.25 * 3 / 5 + 0.25 * 4 / 6)) < 1e-12
    assert abs(ap - O.average_precision(O.clamp(v[0]), gt[0] != 0, K)) < 1e-12


def test_losses_and_calibration_hand_built():
    K = 2
    v = np.array([[0.0, 1.0, 0.25, 0.75]], np.float32)
    gt = np.array([[1, 1, 0, 1]], np.uint8)
    hist, loss = O.occupancy_curves(v, gt, K)
    assert hist[0].tolist() == [[1, 0], [1, 2], [FX20 // 4, FX20 + 3 * FX20 // 4]]
    bce = [100.0, 0.0, -np.log(0.75), -np.log(0.75)]
    assert loss[0].tolist() == [sum(int(np.rint(x * FX20)) for x in bce), FX20 + FX20 // 16 * 2]
    s = T.curves_summary(T.curves_block(torch.from_numpy(hist), torch.from_numpy(loss)), K, 1)
    assert abs(s['bce'] - sum(bce) / 4) < 1e-6 and s['brier'] == (1 + 1 / 16 + 1 / 16) / 4
    # bin 0: values 0, 0.25 against 1 occupied; bin 1: 1, 0.75 against 2
    assert s['reliability'] == [{'count': 2, 'confidence': 0.125, 'frequency': 0.5},
                                {'count': 2, 'confidence': 0.875, 'frequency': 1.0}]
    assert s['ece'] == (0.75 + 0.25) / 4
    # IoU 3/4 at t = 0 (everything predicted), 2/3 at t = 0.5
    assert s['iou'] == [0.75, 2 / 3]
    assert s['best'] == {'threshold': 0.0, 'iou': 0.75} and s['best_mean'] == {'threshold': 0.0, 'mean_iou': 0.75}


def test_ece_merges_bins():
    K = 64
    v, gt = _field(3, 5, seed=11, K=K)
    s = T.curves_summary(torch.from_numpy(O.curves_block(v, gt, K)), K, 3)
    assert len(s['reliability']) == 16 and abs(s['ece'] - O.summary(v, gt, K)['ece']) < 1e-6
    vc = O.clamp(v).reshape(-1)
    m = O.bins(vc, K) // 4
    assert [r['count'] for r in s['reliability']] == np.bincount(m, minlength=16).tolist()


def test_summary_of_nothing():
    s = T.curves_summary(torch.zeros(4 * 4 + 2, dtype=torch.int64), 4, 0)
    assert s['ap'] is None and s['bce'] == 0.0 and s['ece'] == 0.0 and s['mean_iou'] == [0.0] * 4
    assert all(r['confidence'] is None for r in s['reliability'])


@pytest.mark.parametrize('k', [2, 4, 16, 256, 1024])
def test_curve_bins_accepts(k):
    assert curve_bins(small_cfg(TEST__CURVE_BINS=k)) == k


@pytest.mark.parametrize('bad', [0, 1, 3, 6, 255, 2048, -4, 256.0, True, '256', None, [256]])
def test_curve_bins_rejects(bad):
    with pytest.raises(ValueError, match='CURVE_BINS'):
        curve_bins(small_cfg(TEST__CURVE_BINS=bad))
    with pytest.raises(ValueError, match='CURVE_BINS'):
        T.stats_layout(small_cfg(TEST__CURVE_BINS=bad), 'Stereo2Voxel', eval_curves=True)
    with pytest.raises(ValueError, match='CURVE_BINS'):
        T.test_voxel(small_cfg(TEST__CURVE_BINS=bad), None, 1, 1, device='cpu', eval_curves=True)
    assert T.stats_layout(small_cfg(TEST__CURVE_BINS=bad), 'Stereo2Voxel', eval_surface=True)[-1][0] == 'surface'


def test_output_names_put_curves_last():
    names = Stereo2Voxel.output_names(gt=True, disp_gt=True, lr_check=True, uncertainty=True, surface=True, mesh=True,
                                      curves=True)
    assert names == _order('voxels', 'iou_counts', True, True, True, True, True, True) + ('occ_hist', 'occ_loss')
    assert Stereo2Voxel.output_names(gt=True, curves=True) == ('disp_left', 'disp_right', 'voxels', 'iou_counts',
                                                               'occ_hist', 'occ_loss')
    from stereo_3d_reconstruction_b200.models import Stereo2Point
    with pytest.raises(ValueError, match='Stereo2Voxel only'):
        Stereo2Point.output_names(gt=True, curves=True)


# ---- the stats vector ---------------------------------------------------------------------------------------------------
_TV, _TD, _K, _F, _N, _BINS = 4, 2, 3, 2, 6, 16
_NH, _ND, _NL, _NU = 2 * _TV + 1, 2 * (2 + _TD), 2 * (3 + _TD), 2 * _K * (3 + _TD)
_NS, _NC = _TV * (3 + 3 * _F), 4 * _BINS + 2


def _cfg():
    return small_cfg(TEST__VOXEL_THRESH=[0.2, 0.4, 0.6, 0.8], TEST__DISP_THRESH=[1.0, 3.0], TEST__UNC_THRESH=[1.0, 2.0, 4.0],
                     TEST__FSCORE_THRESH=[0.05, 0.3], TEST__CURVE_BINS=_BINS, CONST__N_VOX=_N)


def test_stats_layout_with_curves():
    assert T.stats_layout(_cfg(), 'Stereo2Voxel', eval_curves=True) == [('iou', _NH), ('curves', _NC)]
    assert T.stats_layout(_cfg(), 'Stereo2Voxel', eval_disp=True, eval_lr=True, eval_unc=True, eval_surface=True,
                          eval_curves=True) == [('iou', _NH), ('disparity', _ND), ('lr_consistency', _NL),
                                                ('uncertainty', _NU), ('surface', _NS), ('curves', _NC)]
    assert T.stats_layout(small_cfg(), 'Stereo2Voxel', eval_curves=True)[-1] == ('curves', 4 * 256 + 2)


def _curves_sample(i):
    """Seeded occ_hist / occ_loss of sample i from the oracle (every fifth sample with an empty GT)."""
    v, gt = _field(1, _N, seed=500 + i, K=_BINS)
    if i % 5 == 0:
        gt[:] = 0
    return [torch.from_numpy(t) for t in O.occupancy_curves(v, gt, _BINS)]


class _Fake:
    """Stereo2Voxel's forward in the tuple order written out independently (_order, then occ_hist / occ_loss last) for the
    keywords it is given; records them."""

    def __init__(self):
        self.calls = []

    def __call__(self, left, right, gt=None, curves=False, **kw):
        self.calls.append(set(kw) | ({'curves'} if curves else set()))
        ids = [int(v) for v in left[:, 0, 0, 0].tolist()]
        smp = [_sample(i) for i in ids]
        for s, i in zip(smp, ids):
            s['occ_hist'], s['occ_loss'] = _curves_sample(i)
        names = _order('voxels', 'iou_counts', gt is not None, 'disp_gt' in kw, kw.get('lr_check', False),
                       kw.get('uncertainty', False), kw.get('surface', False), kw.get('mesh', False))
        names += ('occ_hist', 'occ_loss') if curves else ()
        return tuple(torch.cat([s[n] for s in smp]) for n in names)


def _patch(monkeypatch):
    def pair(B, H, W, dmax, seed):
        x = torch.full((1, 3, 2, 2), float(seed))
        return x, x, torch.zeros(1, 2, 2)
    monkeypatch.setattr(synthetic, 'stereo_pair', pair)
    monkeypatch.setattr(synthetic, 'gt_volume', lambda B, n, seed: torch.zeros(1, n, n, n, dtype=torch.uint8))
    monkeypatch.setattr(T, '_disp_gt', lambda pairs, H, W, device: torch.zeros(len(pairs), 2, 2, 2))
    monkeypatch.setattr(T, 'save_meshes', lambda mesh_dir, ids, mesh, gt: None)


def _want_curves(ids):
    return sum(T.curves_block(*_curves_sample(i)) for i in ids)


def test_voxel_driver_every_option_and_curves(monkeypatch, tmp_path):
    _patch(monkeypatch)
    n, bs = 7, 3
    model = _Fake()
    got = T.test_voxel(_cfg(), model, n, bs, device='cpu', eval_disp=True, eval_lr=True, eval_unc=True, eval_surface=True,
                       mesh_dir=str(tmp_path), eval_curves=True)
    assert model.calls == [{'disp_gt', 'lr_check', 'uncertainty', 'surface', 'mesh', 'curves'}] * 3
    base = T.test_voxel(_cfg(), _Fake(), n, bs, device='cpu', eval_disp=True, eval_lr=True, eval_unc=True,
                        eval_surface=True)
    assert got.numel() == base.numel() + _NC and torch.equal(got[:base.numel()], base)
    assert torch.equal(got[-_NC:], _want_curves(range(n)))
    model = _Fake()
    alone = T.test_voxel(_cfg(), model, n, 2, device='cpu', eval_curves=True)   # another batch split, no other block
    assert model.calls == [{'curves'}] * 4
    assert torch.equal(alone[_NH:], got[-_NC:]) and torch.equal(alone[:_NH], got[:_NH])


def _worker(rank, world, port, n, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    mp_patch = pytest.MonkeyPatch()
    _patch(mp_patch)
    s = T.test_voxel(_cfg(), _Fake(), n, 2, rank, world, device='cpu', eval_disp=True, eval_surface=True, eval_curves=True)
    if rank == 0:
        q.put(s.tolist())
    dist.destroy_process_group()


def test_gloo_world2_curves_vector_matches_single_process(monkeypatch):
    n = 9
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0)); port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker, args=(r, 2, port, n, q)) for r in range(2)]
    [p.start() for p in ps]
    got = q.get(timeout=120)
    [p.join(60) for p in ps]
    assert all(p.exitcode == 0 for p in ps)
    _patch(monkeypatch)
    ref = T.test_voxel(_cfg(), _Fake(), n, 4, device='cpu', eval_disp=True, eval_surface=True, eval_curves=True)
    assert got == ref.tolist()
    assert torch.equal(torch.tensor(got[-_NC:]), _want_curves(range(n)))
    s = T.curves_summary(torch.tensor(got[-_NC:]), _BINS, n)
    assert s['n_samples'] == n and s['n_voxels'] == n * _N ** 3
    assert 0 <= s['ap'] <= 1 and all(0 <= x <= 1 for x in s['iou'] + s['mean_iou'])
