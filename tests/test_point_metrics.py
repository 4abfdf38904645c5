"""Point-cloud evaluation, host side: the reference statement in tests/point_oracle.py (half-even fixed point, strict
thresholds, out-of-range points), the driver's F-score block and summary arithmetic, threshold validation, and the stats
vector extended by the point counters through a gloo world-2 all-reduce."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle.chamfer import chamfer_c, chamfer_distance
from stereo_3d_reconstruction_b200 import models as M
from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.utils import synthetic
from tests.point_oracle import fscore_fx, point_counts, point_stats

NAN, INF = float('nan'), float('inf')
F32 = np.float32


def _one_to_one(offsets):
    """B single-point pairs: prediction at the origin, GT at offsets[b] -> (xyz1 [B,1,3], xyz2 [B,1,3])."""
    b = np.asarray(offsets, dtype=np.float32).reshape(-1, 1, 3)
    return np.zeros_like(b), b


def test_fixed_point_rounds_half_to_even():
    e = 2.0 ** -17                                                 # e^2 = 2^-34, so d is a small integer times 2^-34
    # (e, e, 0): d = 2 * 2^-34 = 2^-33 -> q = rint(0.5) = 0;  (2e, e, e): 6 * 2^-34 = 3 * 2^-33 -> rint(1.5) = 2;
    # (3e, e, 0): 5 * 2^-33 -> rint(2.5) = 2;  (3e, 2e, e): 7 * 2^-33 -> rint(3.5) = 4
    a, b = _one_to_one([(e, e, 0), (2 * e, e, e), (3 * e, e, 0), (3 * e, 2 * e, e)])
    d1, d2, _, _ = chamfer_c(a, b)
    want_d = [k * 2.0 ** -33 for k in (1, 3, 5, 7)]
    assert d1[:, 0].tolist() == want_d and d2[:, 0].tolist() == want_d
    c = point_stats(a, b, [])
    assert c[:, 0, 0].tolist() == [0, 2, 2, 4] and c[:, 1, 0].tolist() == [0, 2, 2, 4]
    # q(sqrt d): the float32 square root, then the same rounding
    s = np.sqrt(np.float32(2.0 ** -33))
    assert c[0, 0, 1] == int(np.rint(np.float64(s) * 2.0 ** 32)) and c[0, 0, 2] == 0


def test_threshold_is_strict():
    a, b = _one_to_one([(0.5, 0, 0)])                              # d = 0.25, sqrt_rn(d) = 0.5 exactly
    lo, hi = np.nextafter(F32(0.5), F32(-INF)), np.nextafter(F32(0.5), F32(INF))
    c = point_stats(a, b, [lo, 0.5, hi, 1.0])
    assert c[0, 0, 3:].tolist() == [0, 0, 1, 1] and c[0, 1, 3:].tolist() == [0, 0, 1, 1]
    # a point one ulp beyond tau in distance is not counted at tau, and is at the next float up
    d = np.array([[hi * hi]], F32)
    assert np.sqrt(d)[0, 0] == hi
    assert point_counts(d, d, [0.5, hi, np.nextafter(hi, F32(INF))])[0, 0, 3:].tolist() == [0, 0, 1]


def test_out_of_range_points():
    below = np.nextafter(F32(16.0), F32(0))
    a = np.array([[[0, 0, 0], [NAN, 0, 0], [0, 0, 0]]], F32)
    b = np.array([[[0, 0, 0.5], [16, 0, 0], [below, 0, 0]]], F32)
    d1, d2, _, _ = chamfer_c(a, b)
    assert d1[0, 1] == INF and d2[0, 1] == 256.0 and d2[0, 2] < 256.0
    c = point_stats(a, b, [1.0])
    # prediction: the NaN point is out; GT: d = 256 is out, d just below 2^8 is in (and not within 1.0)
    assert c[0, 0, 2] == 1 and c[0, 0, 3] == 2
    assert c[0, 1, 2] == 1 and c[0, 1, 3] == 1
    assert c[0, 1, 0] == int(np.rint(0.25 * 2.0 ** 32)) + int(np.rint(np.float64(d2[0, 2]) * 2.0 ** 32))
    # the rule on hand-made distances: NaN, inf and >= 2^8 go to n_out and count nowhere else
    d = np.array([[NAN, INF, 256.0, 1e30, np.nextafter(F32(256), F32(0)), 0.0]], F32)
    c = point_counts(d, d[:, 5:], [20.0])
    assert c[0, 0, 2] == 4 and c[0, 0, 3] == 2 and c[0, 0, 0] == int(np.rint(np.float64(d[0, 4]) * 2.0 ** 32))
    assert c[0, 1].tolist() == [0, 0, 0, 1]


def test_oracle_on_random_clouds_matches_float_chamfer():
    a, b = synthetic.point_clouds(3, 200, 700, seed=5, duplicates=True)
    th = [0.01, 0.03, 0.1]
    c = point_stats(a.numpy(), b.numpy(), th)
    d1, d2, _, _ = chamfer_c(a.numpy(), b.numpy())
    assert (c[:, :, 2] == 0).all()
    for t, tau in enumerate(th):
        assert (c[:, 0, 3 + t] == (np.sqrt(d1) < F32(tau)).sum(-1)).all()
        assert (c[:, 1, 3 + t] == (np.sqrt(d2) < F32(tau)).sum(-1)).all()
    assert 0 < c[:, :, 3].sum() < c[:, :, 5].sum()
    # the fixed-point sums against the float64 means: each of the N + M roundings is off by at most 2^-33
    cd = chamfer_distance(a.numpy(), b.numpy())
    l2 = (c[:, 0, 0] / 200 + c[:, 1, 0] / 700) / 2.0 ** 32
    assert np.abs(l2 - cd).max() <= 2.0 ** -32 + 1e-15
    l1 = 0.5 * (c[:, 0, 1] / 200 + c[:, 1, 1] / 700) / 2.0 ** 32
    ref = 0.5 * (np.sqrt(d1.astype(np.float64)).mean(1) + np.sqrt(d2.astype(np.float64)).mean(1))
    assert np.abs(l1 - ref).max() < 1e-7


def test_point_block_fscore():
    g = torch.Generator().manual_seed(2)
    N_, M_ = 50, 400
    c = torch.zeros(6, 2, 5, dtype=torch.int64)
    c[:, 0, 3:] = torch.randint(0, N_ + 1, (6, 2), generator=g)
    c[:, 1, 3:] = torch.randint(0, M_ + 1, (6, 2), generator=g)
    c[:, :, :2] = torch.randint(0, 1 << 40, (6, 2, 2), generator=g)
    c[0, :, 3:] = 0                                                # P = R = 0: F = 0
    c[1, 0, 3] = 0                                                 # P = 0 < R: F = 0
    c[2, :, 3] = torch.tensor([N_, M_])                            # P = R = 1: F = 1
    blk = T.point_block(c, N_, M_)
    assert blk.dtype == torch.int64 and blk.shape == (2 * 5 + 2,)
    assert torch.equal(blk[:10], c.sum(0).flatten())
    assert blk[10:].tolist() == fscore_fx(c.numpy(), N_, M_).tolist()
    one = [T.point_block(c[i:i + 1], N_, M_)[10:] for i in range(6)]
    assert one[0].tolist() == [0, 0] and one[1][0] == 0 and one[2][0] == 1 << 32
    p, r = c[3, 0, 4].item() / N_, c[3, 1, 4].item() / M_
    assert one[3][1] == round(2 * p * r / (p + r) * 2.0 ** 32)
    assert torch.equal(sum(one), blk[10:])                          # any batch split: the same sums


def test_points_summary_arithmetic():
    th = [0.01, 0.02]
    N_, M_, n = 4, 8, 2
    fx = 1 << 32
    blk = torch.tensor([6 * fx, 2 * fx, 0, 4, 8,                    # predicted -> GT: sum d = 6, sum sqrt d = 2
                        4 * fx, 8 * fx, 0, 2, 16,                   # GT -> predicted
                        fx // 2, 3 * fx // 2], dtype=torch.int64)   # sum of F-scores: 0.5, 1.5
    s = T.points_summary(blk, th, n, N_, M_)
    assert s['thresholds'] == th and s['n_samples'] == 2 and s['n_pred'] == 4 and s['n_gt'] == 8 and s['n_out'] == 0
    assert s['chamfer_l2'] == (6 / 4 + 4 / 8) / 2 and s['chamfer_l1'] == 0.5 * (2 / 4 + 8 / 8) / 2
    assert s['precision'] == [0.5, 1.0] and s['recall'] == [0.125, 1.0] and s['fscore'] == [0.25, 0.75]
    blk[7] = 1                                                      # one GT point out of range
    s = T.points_summary(blk, th, n, N_, M_)
    assert s['n_out'] == 1 and s['chamfer_l2'] == INF and s['chamfer_l1'] == INF and s['precision'] == [0.5, 1.0]
    z = T.points_summary(torch.zeros(12, dtype=torch.int64), th, 3, N_, M_)            # P = R = 0
    assert z['chamfer_l2'] == 0.0 and z['precision'] == [0.0, 0.0] and z['recall'] == [0.0, 0.0] and z['fscore'] == [0.0, 0.0]
    e = T.points_summary(torch.zeros(12, dtype=torch.int64), th, 0, N_, M_)            # no samples
    assert e['chamfer_l2'] == 0.0 and e['fscore'] == [0.0, 0.0]


@pytest.mark.parametrize('bad', [[-0.01], [0.0], [NAN], [INF], [0.01] * 9, ['x'], None, 0.01])
def test_driver_rejects_bad_thresholds(bad):
    from tests.common import small_cfg
    cfg = small_cfg(TEST__FSCORE_THRESH=bad)
    with pytest.raises(ValueError):
        M.fscore_thresholds(cfg)
    with pytest.raises(ValueError):
        T.test_point(cfg, None, 1, 1, device='cpu', eval_points=True)


def test_threshold_defaults():
    from config import cfg
    assert M.fscore_thresholds(cfg) == [0.01]
    from tests.common import small_cfg
    assert M.fscore_thresholds(small_cfg(TEST__FSCORE_THRESH=[0.5] * 8)) == [0.5] * 8
    assert M.fscore_thresholds(small_cfg(TEST__FSCORE_THRESH=[])) == []


# ---- the stats vector with the point counters through the single all-reduce ----------------------------------------------
_TD, _TF = 2, 3
_ND, _NL, _NP = 2 * (2 + _TD), 2 * (3 + _TD), 2 * (3 + _TF) + _TF
_N, _M = 2048, 16384


def _fake_sample(i):
    g = torch.Generator().manual_seed(5000 + i)
    head = torch.randint(0, 1 << 30, (1,), generator=g)
    ds = torch.randint(0, 1 << 20, (_ND,), generator=g)
    ls = torch.randint(0, 1 << 20, (_NL,), generator=g)
    ps = torch.zeros(1, 2, 3 + _TF, dtype=torch.int64)
    ps[0, :, :2] = torch.randint(0, 1 << 50, (2, 2), generator=g)
    ps[0, 0, 3:] = torch.randint(0, _N + 1, (_TF,), generator=g)
    ps[0, 1, 3:] = torch.randint(0, _M + 1, (_TF,), generator=g)
    if i % 7 == 0:
        ps[0, :, 3:] = 0                                            # P = R = 0
    return head, ds, ls, ps


def _local_stats(n, rank, world, batch):
    s = torch.zeros(2 + _ND + _NL + _NP, dtype=torch.int64)
    lo, hi = T.shard_range(n, rank, world)
    for b0 in range(lo, hi, batch):
        smp = [_fake_sample(i) for i in range(b0, min(b0 + batch, hi))]
        s[0] += sum(x[0] for x in smp)[0]
        s[1] += len(smp)
        s[2:2 + _ND] += sum(x[1] for x in smp)
        s[2 + _ND:2 + _ND + _NL] += sum(x[2] for x in smp)
        s[2 + _ND + _NL:] += T.point_block(torch.cat([x[3] for x in smp]), _N, _M)
    return s


def _worker(rank, world, port, n, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    s = T.reduce_stats(_local_stats(n, rank, world, batch=4))
    if rank == 0:
        q.put(s.tolist())
    dist.destroy_process_group()


def test_gloo_world2_point_vector_matches_single_process():
    n = 31
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0)); port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker, args=(r, 2, port, n, q)) for r in range(2)]
    [p.start() for p in ps]
    got = q.get(timeout=120)
    [p.join(60) for p in ps]
    assert all(p.exitcode == 0 for p in ps)
    ref = _local_stats(n, 0, 1, batch=5)                            # one process, another batch split
    assert got == ref.tolist()
    got = torch.tensor(got)
    summ = T.points_summary(got[2 + _ND + _NL:], [0.01, 0.02, 0.05], n, _N, _M)
    assert summ['n_samples'] == n and summ['n_out'] == 0
    assert all(0 <= v <= 1 for v in summ['precision'] + summ['recall'] + summ['fscore'])
