"""Disparity uncertainty, host side: the reference statement in tests/unc_oracle.py (fp64 moments of the soft-argmin
distribution, the inclusive fp32 confidence rule and the GT columns), TEST.UNC_THRESH validation, the summary arithmetic, and
the stats vector extended by the uncertainty counters through a gloo world-2 all-reduce."""
import math
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from stereo_3d_reconstruction_b200 import models as M
from stereo_3d_reconstruction_b200.core import test as T
from tests.common import small_cfg
from tests.disp_oracle import disp_error_counts
from tests.unc_oracle import soft_argmin_moments, unc_counts

NAN, INF = float('nan'), float('inf')


def _cost(planes):
    """One pixel: [1, D, 1, 1] from a list of D costs."""
    return torch.tensor(planes, dtype=torch.float64).view(1, -1, 1, 1)


def test_moments_uniform_and_two_minima():
    D = 32
    mu, sd = soft_argmin_moments(_cost([0.0] * D))
    assert mu.item() == pytest.approx((D - 1) / 2) and sd.item() == pytest.approx(math.sqrt((D * D - 1) / 12))
    c = [50.0] * D
    c[3] = c[11] = 0.0                                               # two equal minima: a Bernoulli on {3, 11}
    mu, sd = soft_argmin_moments(_cost(c))
    assert mu.item() == pytest.approx(7.0) and sd.item() == pytest.approx(4.0)


def test_moments_sharp_peak_and_sign():
    D = 128
    c = np.full(D, 60.0)
    c[120], c[119], c[121] = 0.0, 6.5, 6.5                          # p(119) = p(121) = e^-6.5 / Z
    mu, sd = soft_argmin_moments(_cost(list(c)))
    p = math.exp(-6.5) / (1 + 2 * math.exp(-6.5))
    assert mu.item() == pytest.approx(120.0, abs=1e-12) and sd.item() == pytest.approx(math.sqrt(2 * p), rel=1e-9)
    assert 0.05 < sd.item() < 0.06
    # the naive running sums of e, e d and e d^2 in fp32, then sum e d^2 / sum e - mu^2, miss 1e-4 * (1 + sigma) on this
    # pixel: the kernels must not compute it so
    f32 = np.float32
    s = t = t2 = f32(0)
    for d in range(D):
        e = f32(math.exp(-c[d]))
        s, t, t2 = s + e, t + e * f32(d), t2 + e * f32(d) * f32(d)
    naive = math.sqrt(max(float(t2 / s - (t / s) * (t / s)), 0.0))
    assert abs(naive - sd.item()) > 1e-4 * (1 + sd.item())
    # sign = +1 takes the maximum
    mu2, _ = soft_argmin_moments(-_cost(list(c)), sign=1.0)
    assert mu2.item() == pytest.approx(mu.item())


def test_moments_axis_and_shape():
    g = torch.Generator().manual_seed(0)
    cost = torch.randn(2, 8, 3, 5, generator=g)
    mu, sd = soft_argmin_moments(cost)
    assert mu.shape == (2, 3, 5) and sd.shape == (2, 3, 5) and (sd > 0).all() and (sd < 8).all()
    p = torch.softmax(-cost.double(), 1)
    d = torch.arange(8, dtype=torch.float64).view(1, 8, 1, 1)
    assert np.allclose(mu, (p * d).sum(1).numpy()) and np.allclose(sd ** 2, (p * d * d).sum(1).numpy() - mu ** 2)


def test_counts_threshold_inclusive_and_non_finite():
    up = torch.nextafter(torch.tensor(1.0), torch.tensor(INF)).item()
    disp = torch.zeros(1, 2, 1, 6)
    std = torch.tensor([[[[1.0, up, 0.0, NAN, INF, 0.5]], [[2.0, 2.0, 2.0, 2.0, 2.0, 2.0]]]])
    c = unc_counts(disp, std, [1.0, 0.0, 2.0])
    assert c.shape == (1, 2, 3, 3)
    assert c[0, 0, :, 0].tolist() == [3, 1, 4] and c[0, 1, :, 0].tolist() == [0, 0, 6]
    assert (c[..., 1:] == 0).all()                                   # no GT: column 0 only
    assert unc_counts(disp, std, []).shape == (1, 2, 0, 3)


def test_counts_gt_columns_equal_disp_oracle_on_the_confident_pixels():
    g = torch.Generator().manual_seed(1)
    disp = torch.rand(3, 2, 5, 16, generator=g) * 6
    std = torch.rand(disp.shape, generator=g) * 3
    gt = disp + (torch.rand(disp.shape, generator=g) - 0.5) * 6
    gt[0, 0, 0, :4] = NAN
    gt[1, 1, 2, :3] = -1.0
    th, ut, max_gt = [1.0, 2.0], [0.5, 1.5, 2.5], 8.0
    c = unc_counts(disp, std, ut, gt, th, max_gt)
    assert c.shape == (3, 2, 3, 5)
    for k, tau in enumerate(ut):
        conf = std <= tau
        assert torch.equal(c[:, :, k, 0], conf.sum((-2, -1)))
        want = disp_error_counts(disp, torch.where(conf, gt, torch.full_like(gt, NAN)), th, max_gt)
        assert torch.equal(c[:, :, k, 1:], want)
    # more confident pixels at a larger threshold; at tau >= max std all of them
    assert (c[:, :, 0, 0] <= c[:, :, 1, 0]).all() and (c[:, :, 1, 0] <= c[:, :, 2, 0]).all()
    assert torch.equal(unc_counts(disp, std, [3.0], gt, th, max_gt)[:, :, 0, 1:], disp_error_counts(disp, gt, th, max_gt))


def test_unc_thresh_validation():
    cfg = small_cfg()
    assert M.unc_thresholds(cfg) == [1.0, 2.0, 4.0]
    for good in ([], [0.0], [0, 1, 2, 3.5]):
        cfg.TEST.UNC_THRESH = good
        assert M.unc_thresholds(cfg) == [float(t) for t in good]
    for bad in ([1, 2, 3, 4, 5], [-0.5], [NAN], [INF], ['x'], None, 3.0):
        cfg.TEST.UNC_THRESH = bad
        with pytest.raises(ValueError):
            M.unc_thresholds(cfg)


def test_forward_rejects_bad_unc_thresh_before_anything_runs():
    cfg = small_cfg()
    cfg.TEST.UNC_THRESH = [1.0, NAN]
    model = M.build_model('Stereo2Voxel', cfg)
    with pytest.raises(ValueError):                                  # not the "needs CUDA" error of the input check
        model(torch.zeros(1, 3, 64, 64), torch.zeros(1, 3, 64, 64), uncertainty=True)
    with pytest.raises(ValueError):
        model.graphed(torch.zeros(1, 3, 64, 64), torch.zeros(1, 3, 64, 64), uncertainty=True)
    with pytest.raises(ValueError):
        T.test_voxel(cfg, model, 1, 1, device='cpu', eval_disp=True, eval_unc=True)


def test_driver_rejects_unc_without_disp():
    for fn in (T.test_voxel, T.test_point):
        with pytest.raises(ValueError):
            fn(small_cfg(), None, 1, 1, device='cpu', eval_disp=False, eval_unc=True)


def test_unc_summary_arithmetic():
    th, ut = [1.0, 3.0], [1.0, 4.0]
    disp = torch.tensor([8, 0, 0, 0,  5, 0, 0, 0], dtype=torch.int64)          # n_valid 8 (left), 5 (right)
    unc = torch.tensor([6, 4, 6 * 65536, 2, 1,    10, 8, 8 * 65536, 3, 0,        # left: tau 1, tau 4
                        2, 1, 65536, 0, 0,         4, 5, 15 * 65536, 5, 1],      # right
                       dtype=torch.int64)
    s = T.unc_summary(unc, ut, th, 20, disp)
    assert s['unc_thresh'] == ut and s['thresholds'] == th and len(s['left']) == 2
    l0, l1, r0, a1 = s['left'][0], s['left'][1], s['right'][0], s['all'][1]
    assert l0 == {'n_conf': 6, 'density': 0.3, 'n_valid_conf': 4, 'conf_of_valid': 0.5, 'epe': 1.5, 'bad': [0.5, 0.25]}
    assert l1['density'] == 0.5 and l1['epe'] == 1.0 and l1['bad'] == [3 / 8, 0.0]
    assert r0['conf_of_valid'] == 0.2 and r0['epe'] == 1.0
    assert a1 == {'n_conf': 14, 'density': 14 / 40, 'n_valid_conf': 13, 'conf_of_valid': 1.0, 'epe': 23 / 13,
                  'bad': [8 / 13, 1 / 13]}
    z = T.unc_summary(torch.zeros(2 * 2 * 5, dtype=torch.int64), ut, th, 0, torch.zeros(8, dtype=torch.int64))
    assert z['all'][0] == {'n_conf': 0, 'density': 0.0, 'n_valid_conf': 0, 'conf_of_valid': 0.0, 'epe': 0.0, 'bad': [0.0, 0.0]}


# ---- the stats vector with the uncertainty counters through the single all-reduce -------------------------------------
_T, _TD, _K = 4, 2, 3
_NH, _ND, _NU = 2 * _T + 1, 2 * (2 + _TD), 2 * _K * (3 + _TD)


def _fake_sample(i):
    g = torch.Generator().manual_seed(5000 + i)
    inter = torch.randint(0, 2000, (_T,), generator=g)
    union = inter + torch.randint(1, 3000, (_T,), generator=g)
    nval = torch.randint(100, 65536, (2,), generator=g)
    epe = nval * torch.randint(0, 40 << 16, (2,), generator=g)
    bad = torch.stack([torch.randint(0, int(n) + 1, (_TD,), generator=g) for n in nval])
    ds = torch.cat([nval.view(2, 1), epe.view(2, 1), bad], 1)
    rows = []
    for v in range(2):
        for _ in range(_K):
            nvc = torch.randint(0, int(nval[v]) + 1, (1,), generator=g)
            nc = nvc + torch.randint(0, 65536, (1,), generator=g)
            epec = nvc * torch.randint(0, 40 << 16, (1,), generator=g)
            badc = torch.randint(0, int(nvc) + 1, (_TD,), generator=g)
            rows.append(torch.cat([nc, nvc, epec, badc]))
    return inter, union, ds, torch.stack(rows).view(2, _K, 3 + _TD)


def _local_stats(n, rank, world):
    s = torch.zeros(_NH + _ND + _NU, dtype=torch.int64)
    lo, hi = T.shard_range(n, rank, world)
    for i in range(lo, hi):
        a, u, ds, us = _fake_sample(i)
        s[:_T] += a; s[_T:2 * _T] += u; s[2 * _T] += 1
        s[_NH:_NH + _ND] += ds.flatten()
        s[_NH + _ND:] += us.flatten()
    return s


def _worker(rank, world, port, n, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    s = T.reduce_stats(_local_stats(n, rank, world))
    if rank == 0:
        q.put(s.tolist())
    dist.destroy_process_group()


def test_gloo_world2_unc_vector_matches_single_process():
    n = 23
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0)); port = s.getsockname()[1]
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    ps = [ctx.Process(target=_worker, args=(r, 2, port, n, q)) for r in range(2)]
    [p.start() for p in ps]
    got = q.get(timeout=120)
    [p.join(60) for p in ps]
    assert all(p.exitcode == 0 for p in ps)
    ref = _local_stats(n, 0, 1)
    assert got == ref.tolist()
    got = torch.tensor(got)
    assert T.iou_summary(got[:_NH], [0.2, 0.3, 0.4, 0.5])['n_samples'] == n
    summ = T.unc_summary(got[_NH + _ND:], [1.0, 2.0, 4.0], [1.0, 3.0], n * 64 * 64, got[_NH:_NH + _ND])
    for k in range(_K):
        assert summ['all'][k]['n_conf'] == summ['left'][k]['n_conf'] + summ['right'][k]['n_conf']
        assert all(0 <= v <= 1 for v in summ['all'][k]['bad']) and 0 <= summ['all'][k]['conf_of_valid'] <= 1
