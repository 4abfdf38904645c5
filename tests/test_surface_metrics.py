"""Voxel-surface evaluation, host side: the reference statement in tests/surface_oracle.py against scipy's exact Euclidean
distance transform, hand-built grids, the F-score bound k, the driver's surface block and summary arithmetic, the vector
layout, and the stats vector extended by the surface block through a gloo world-2 all-reduce."""
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp
from scipy import ndimage

from stereo_3d_reconstruction_b200 import ops
from stereo_3d_reconstruction_b200.core import test as T
from tests.surface_oracle import direction_counts, faces, kbound, nearest_sq, surface_block, surface_stats

FX = 1 << 32


def _edt_sq(a, b, n):
    """Squared distance of each site of a to the nearest site of b, from scipy's EDT on the (2n+1)^3 lattice."""
    m = np.zeros((2 * n + 1,) * 3, dtype=bool)
    m[tuple(b.T)] = True
    d = ndimage.distance_transform_edt(~m)
    return np.rint(d[tuple(a.T)] ** 2).astype(np.int64)


@pytest.mark.parametrize('n', [4, 7, 12, 16])
def test_oracle_matches_scipy_edt(n):
    rng = np.random.default_rng(n)
    for p, q in ((0.1, 0.3), (0.5, 0.05), (0.9, 0.5)):
        a, b = faces(rng.random((n,) * 3) < p), faces(rng.random((n,) * 3) < q)
        if not (len(a) and len(b)):
            continue
        assert np.array_equal(nearest_sq(a, b), _edt_sq(a, b, n))
        assert np.array_equal(nearest_sq(b, a), _edt_sq(b, a, n))
        # every surface point is a lattice site with exactly one even coordinate
        assert ((a % 2 == 0).sum(1) == 1).all() and a.min() >= 0 and a.max() <= 2 * n
        assert len(np.unique(a, axis=0)) == len(a)


def test_single_voxel():
    n = 5
    occ = np.zeros((n,) * 3, bool)
    occ[2, 1, 3] = True
    f = faces(occ)
    assert len(f) == 6
    centre = np.array([5, 3, 7])
    assert sorted(((f - centre) ** 2).sum(1).tolist()) == [1] * 6
    assert direction_counts(f, f, [1]).tolist() == [6, 0, 0, 6]                  # s = 0 against itself


def test_shifted_voxel():
    n = 4
    a = np.zeros((n,) * 3, bool)
    b = a.copy()
    a[1, 1, 1] = True
    b[1, 1, 2] = True                                             # one voxel over along the last axis: one shared face
    fa, fb = faces(a), faces(b)
    s = nearest_sq(fa, fb)
    # the shared face: 0; each side face: the shared face, one unit along two axes (s = 2); the far face: 2 away (s = 4)
    assert sorted(s.tolist()) == [0, 2, 2, 2, 2, 4]
    q2 = int(np.rint(np.float64(np.sqrt(np.float32(2))) * FX))
    c = direction_counts(fa, fb, [1, 3, 5])
    assert c.tolist() == [6, 12, 4 * q2 + 2 * FX, 1, 5, 6]


@pytest.mark.parametrize('n', [1, 3, 8])
def test_full_grid_and_empty(n):
    full = np.ones((n,) * 3, bool)
    assert len(faces(full)) == 6 * n * n
    assert len(faces(~full)) == 0
    fused = np.ones((1, n, n, n), np.float32)
    gt = np.zeros((1, n, n, n), np.uint8)
    st = surface_stats(fused, gt, [0.5, 2.0], [0.1])
    # t = 0.5: full prediction against an empty GT; t = 2.0: empty prediction (both surfaces empty)
    assert st[0, 0, 0].tolist() == [6 * n * n, 0, 0, 0] and st[0, 0, 1].tolist() == [0, 0, 0, 0]
    assert st[0, 1].tolist() == [[0, 0, 0, 0], [0, 0, 0, 0]]
    st = surface_stats(np.zeros((1, n, n, n), np.float32), full[None].astype(np.uint8), [0.5], [0.1])
    assert st[0, 0, 0].tolist() == [0, 0, 0, 0] and st[0, 0, 1].tolist() == [6 * n * n, 0, 0, 0]


def test_prediction_equal_to_gt():
    n = 8
    rng = np.random.default_rng(3)
    gt = (rng.random((2, n, n, n)) < 0.2).astype(np.uint8)
    fused = gt.astype(np.float32) * 0.75
    st = surface_stats(fused, gt, [0.5], [0.01, 0.2])
    assert (st[:, :, :, 1:3] == 0).all() and (st[:, :, :, 3:] == st[:, :, :, :1]).all()
    blk = surface_block(st, n)
    assert blk[0, 0] == 2 and blk[0, 1] == 0 and blk[0, 2] == 0
    assert blk[0, 3:].tolist() == [2 * FX] * 6                     # P = R = F = 1 per sample
    s = T.surface_summary(torch.from_numpy(blk.flatten()), [0.5], [0.01, 0.2], 2)['by_thresh'][0]
    assert s['chamfer_l2'] == 0 and s['chamfer_l1'] == 0 and s['fscore'] == [1.0, 1.0]


def test_threshold_at_nan_and_boundary():
    n = 3
    fused = np.full((1, n, n, n), np.nan, np.float32)
    fused[0, 1, 1, 1] = 0.25
    gt = np.zeros((1, n, n, n), np.uint8)
    gt[0, 1, 1, 1] = 1
    st = surface_stats(fused, gt, [0.25, np.nextafter(np.float32(0.25), np.float32(1))], [0.01])
    assert st[0, 0, 0].tolist() == [6, 0, 0, 6]                    # fused >= t at equality; NaN is empty
    assert st[0, 1, 0, 0] == 0 and st[0, 1, 1, 0] == 6


def test_kbound_on_lattice_distances():
    n = 32
    assert kbound(0.01, n) == 1                                   # F-Score@1 %: only coinciding faces at 32^3
    # tau exactly sqrt(k) / (2n) lands on a lattice distance: a point at that distance is not within tau (strict)
    for k in (1, 4, 16, 64, 4096):
        tau = math.sqrt(k) / (2 * n)
        assert kbound(tau, n) == k, k
        assert ops.voxel_kbound(tau, n) == k
    assert kbound(1.0 / (2 * n) + 1e-12, n) == 2
    assert kbound(10.0, n) == 3 * (2 * n) ** 2 + 1                # every distance counts
    assert kbound(math.sqrt(3), n) == 3 * (2 * n) ** 2             # the cube diagonal itself is not within sqrt(3)
    for tau in (0.003, 0.01, 0.05, 0.2, 0.77):
        assert ops.voxel_kbound(tau, 16) == kbound(tau, 16)
        k = kbound(tau, 16)
        # the rule: s counts exactly when sqrt(s) / (2n) < tau
        for s in range(max(0, k - 3), k + 3):
            assert (s < k) == (math.sqrt(s) / 32 < tau), (tau, s)


def test_synthetic_gt_surface_size():
    from stereo_3d_reconstruction_b200.utils import synthetic
    g = synthetic.gt_volume(4, 32, seed=100000).numpy()
    cnt = [len(faces(g[b] != 0)) for b in range(4)]
    assert all(17000 < c < 19000 for c in cnt)
    assert 3 * 33 * 32 * 32 == 101376


def test_surface_block_matches_oracle_and_splits():
    rng = np.random.default_rng(7)
    n = 6
    fused = rng.random((5, n, n, n)).astype(np.float32)
    gt = (rng.random((5, n, n, n)) < 0.3).astype(np.uint8)
    gt[3] = 0                                                     # an empty GT: n_both drops, P = R = 0 there
    st = surface_stats(fused, gt, [0.1, 0.5, 0.99], [0.05, 0.2])
    blk = T.surface_block(torch.from_numpy(st), n)
    assert blk.dtype == torch.int64 and blk.shape == (3 * (3 + 3 * 2),)
    assert blk.tolist() == surface_block(st, n).flatten().tolist()
    assert blk[0] == 4
    parts = sum(T.surface_block(torch.from_numpy(st[i:i + 1]), n) for i in range(5))
    assert torch.equal(parts, blk)                                # any batch split: the same sums


def test_surface_summary_arithmetic():
    n = 4
    st = np.zeros((2, 1, 2, 4), np.int64)
    st[0, 0, 0] = [10, 20, 10 * FX, 5]                            # s = 2 on each of 10 points; sqrt 2 rounded to q in sum
    st[0, 0, 1] = [5, 5, 5 * FX, 5]
    st[1, 0, 0] = [4, 0, 0, 4]                                    # sample 1: GT empty
    blk = T.surface_block(torch.from_numpy(st), n)
    r = blk.tolist()
    assert r[0] == 1
    assert r[1] == round((20 / 10 + 5 / 5) / 64 * FX)
    assert r[2] == FX // 8                                        # (1 + 1) / 2 / 2n
    assert r[3:] == [3 * FX // 2, FX, round(2 * 0.5 / 1.5 * FX)]      # P: 0.5 + 1 (sample 1: R = 0, F = 0)
    s = T.surface_summary(blk, [0.4], [0.01], 2)
    b = s['by_thresh'][0]
    assert s['n_samples'] == 2 and s['thresholds'] == [0.4] and b['n_both'] == 1
    assert abs(b['chamfer_l2'] - 3 / 64) < 1e-12 and abs(b['chamfer_l1'] - 1 / 8) < 1e-12
    assert b['precision'] == [0.75] and b['recall'] == [0.5] and abs(b['fscore'][0] - 1 / 3) < 1e-9
    z = T.surface_summary(torch.zeros(6, dtype=torch.int64), [0.4], [0.01], 3)['by_thresh'][0]
    assert z['chamfer_l2'] == float('inf') and z['chamfer_l1'] == float('inf') and z['fscore'] == [0.0]


@pytest.mark.parametrize('bad', [[-0.01], [0.0], [float('nan')], [0.01] * 9, None])
def test_driver_rejects_bad_thresholds(bad):
    from tests.common import small_cfg
    cfg = small_cfg(TEST__FSCORE_THRESH=bad)
    with pytest.raises(ValueError):
        T.test_voxel(cfg, None, 1, 1, device='cpu', eval_surface=True)


# ---- the stats vector with the surface block through the single all-reduce ---------------------------------------------
_TV, _TD, _F, _N = 4, 2, 2, 6
_ND, _NL = 2 * (2 + _TD), 2 * (3 + _TD)
_NS = _TV * (3 + 3 * _F)


class _FakeVoxel:
    """Stands in for Stereo2Voxel in test_voxel: seeded per-sample outputs in the forward's tuple layout for the keywords
    it is given (disp_stats when disp_gt= is passed at all: the driver's synthetic GT disparity is stubbed out)."""

    def __call__(self, left, right, gt, lr_check=False, surface=False, **kw):
        assert set(kw) <= {'disp_gt'}
        B = left.shape[0]
        ids = [int(v) for v in left[:, 0, 0, 0].tolist()]
        g = [torch.Generator().manual_seed(9000 + i) for i in ids]
        iou = torch.stack([torch.randint(0, 1 << 15, (_TV, 2), generator=x) for x in g])
        ds = torch.stack([torch.randint(0, 1 << 20, (2, 2 + _TD), generator=x) for x in g])
        ls = torch.stack([torch.randint(0, 1 << 20, (2, 3 + _TD), generator=x) for x in g])
        out = (None, None, None) + ((iou,) if gt is not None else ()) + ((ds,) if 'disp_gt' in kw else ())
        out += (None, ls) if lr_check else ()
        if surface:
            ss = []
            for i, x in zip(ids, g):
                fused = torch.rand(_N, _N, _N, generator=x).numpy()
                gv = (torch.rand(_N, _N, _N, generator=x) < 0.2).numpy().astype(np.uint8)
                if i % 5 == 0:
                    gv[:] = 0
                ss.append(torch.from_numpy(surface_stats(fused[None], gv[None], [0.2, 0.4, 0.6, 0.8], [0.05, 0.3])[0]))
            out += (torch.stack(ss),)
        assert B == len(ids)
        return out


def _cfg():
    from tests.common import small_cfg
    return small_cfg(TEST__VOXEL_THRESH=[0.2, 0.4, 0.6, 0.8], TEST__DISP_THRESH=[1.0, 3.0], TEST__FSCORE_THRESH=[0.05, 0.3],
                     CONST__N_VOX=_N)


def _patch_inputs(monkeypatch):
    from stereo_3d_reconstruction_b200.utils import synthetic

    def pair(B, H, W, dmax, seed):
        x = torch.full((1, 3, 2, 2), float(seed))
        return x, x, torch.zeros(1, 2, 2)
    monkeypatch.setattr(synthetic, 'stereo_pair', pair)
    monkeypatch.setattr(synthetic, 'gt_volume', lambda B, n, seed: torch.zeros(1, n, n, n, dtype=torch.uint8))
    monkeypatch.setattr(T, '_disp_gt', lambda pairs, H, W, device: None)


def test_driver_vector_layout_in_forward_order(monkeypatch):
    _patch_inputs(monkeypatch)
    cfg, model = _cfg(), _FakeVoxel()
    base = T.test_voxel(cfg, model, 7, 3, device='cpu', eval_disp=True, eval_lr=True)
    full = T.test_voxel(cfg, model, 7, 3, device='cpu', eval_disp=True, eval_lr=True, eval_surface=True)
    assert full.numel() == base.numel() + _NS and torch.equal(full[:base.numel()], base)
    want = sum(T.surface_block(model(torch.full((1, 3, 2, 2), float(i)), None, None, surface=True)[-1], _N)
               for i in range(7))
    assert torch.equal(full[base.numel():], want)
    alone = T.test_voxel(cfg, model, 7, 2, device='cpu', eval_surface=True)
    assert torch.equal(alone[2 * _TV + 1:], want)                  # another batch split, no disparity blocks


def _worker(rank, world, port, n, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    mp_patch = pytest.MonkeyPatch()
    _patch_inputs(mp_patch)
    s = T.test_voxel(_cfg(), _FakeVoxel(), n, 2, rank, world, device='cpu', eval_disp=True, eval_lr=True, eval_surface=True)
    if rank == 0:
        q.put(s.tolist())
    dist.destroy_process_group()


def test_gloo_world2_surface_vector_matches_single_process(monkeypatch):
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
    _patch_inputs(monkeypatch)
    ref = T.test_voxel(_cfg(), _FakeVoxel(), n, 4, device='cpu', eval_disp=True, eval_lr=True, eval_surface=True)
    assert got == ref.tolist()
    summ = T.surface_summary(torch.tensor(got)[-_NS:], [0.2, 0.4, 0.6, 0.8], [0.05, 0.3], n)
    assert summ['n_samples'] == n
    for b in summ['by_thresh']:
        assert 0 < b['n_both'] <= n and b['chamfer_l2'] > 0
        assert all(0 <= v <= 1 for v in b['precision'] + b['recall'] + b['fscore'])
