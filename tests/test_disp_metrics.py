"""Disparity evaluation, host side: the reference statement of the counters in tests/disp_oracle.py (validity rule, strict
'>', half-even fixed point), the synthetic GT disparity, the summary arithmetic, and the extended stats vector through a
gloo world-2 all-reduce."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.utils import synthetic
from tests.disp_oracle import disp_error_counts

NAN, INF = float('nan'), float('inf')


def test_validity_rule():
    max_gt = 128.0
    gt = torch.tensor([[[NAN, INF, -INF, -1.0, -1e-30, max_gt, 127.99999, 0.0, -0.0, 5.0]]])     # one 1 x 10 image
    disp = torch.full_like(gt, 7.0)
    got = disp_error_counts(disp, gt, [1.0], max_gt)
    # valid: 127.99999, 0.0, -0.0 (== 0), 5.0
    e_big = (torch.tensor(7.0) - torch.tensor(127.99999)).abs().item()          # fp32 subtraction
    assert got.tolist() == [[4, round(e_big * 65536) + 3 * 65536 * 7 - 65536 * 5, 4]]


def test_threshold_is_strict():
    gt = torch.tensor([[[2.0, 2.0, 2.0, 10.0]]])
    up = torch.nextafter(torch.tensor(3.0), torch.tensor(INF)).item()
    disp = torch.tensor([[[3.0, up, 1.0, 13.0]]])                    # errors 1, 1 + ulp, 1, 3: above 1 twice, above 3 never
    got = disp_error_counts(disp, gt, [1.0, 3.0], 100.0)[0].tolist()
    assert got[0] == 4 and got[2] == 2 and got[3] == 0


def test_fixed_point_rounds_half_to_even():
    k = 2.0 ** -17                                                  # q(e) = e * 2^16 = 0.5, 1.5, 2.5, 3.5
    gt = torch.zeros(1, 1, 4)
    disp = torch.tensor([[[1 * k, 3 * k, 5 * k, 7 * k]]])
    assert disp_error_counts(disp, gt, [], 1.0)[0].tolist() == [4, 0 + 2 + 2 + 4]
    # one pixel at a time: the rounding is per pixel, before the sum
    for v, q in zip(disp[0, 0].tolist(), (0, 2, 2, 4)):
        assert disp_error_counts(torch.tensor([[v]]), torch.zeros(1, 1), [], 1.0).tolist() == [1, q]


def test_counts_shape_per_image():
    g = torch.Generator().manual_seed(3)
    disp = torch.rand(3, 2, 5, 7, generator=g) * 20
    gt = torch.rand(3, 2, 5, 7, generator=g) * 20
    gt[0, 1, 2, 3] = NAN
    c = disp_error_counts(disp, gt, [1.0, 3.0], 16.0)
    assert c.shape == (3, 2, 4) and c.dtype == torch.int64
    ok = torch.isfinite(gt) & (gt >= 0) & (gt < 16.0)
    assert torch.equal(c[..., 0], ok.flatten(2).sum(-1))
    assert torch.equal(c[..., 3], (ok & ((disp - gt).abs() > 3.0)).flatten(2).sum(-1))


@pytest.mark.parametrize('B,H,W,maxd', [(2, 9, 13, 8), (1, 4, 5, 16), (3, 16, 40, 12)])
def test_disparity_gt_marks_unmatched_columns(B, H, W, maxd):
    left, right, d = synthetic.stereo_pair(B, H, W, maxd, seed=5)
    gt = synthetic.disparity_gt(d, H, W)
    assert gt.shape == (B, 2, H, W) and gt.dtype == torch.float32
    for b in range(B):
        for y in range(H):
            dy = int(d[b, y])
            for x in range(W):
                gl, gr = gt[b, 0, y, x].item(), gt[b, 1, y, x].item()
                if x - dy >= 0:
                    assert gl == dy and torch.equal(left[b, :, y, x], right[b, :, y, x - dy])
                else:
                    assert gl != gl
                if x + dy < W:
                    assert gr == dy and torch.equal(right[b, :, y, x], left[b, :, y, x + dy])
                else:
                    assert gr != gr and (right[b, :, y, x] == 0).all()


def test_disp_summary_arithmetic():
    th = [1.0, 3.0]
    block = torch.tensor([4, 6 * 65536, 2, 1,              # left: 4 valid, EPE 1.5, bad-1 0.5, bad-3 0.25
                          0, 0, 0, 0], dtype=torch.int64)   # right: no valid pixel
    s = T.disp_summary(block, th)
    assert s['thresholds'] == th
    assert s['left'] == {'n_valid': 4, 'epe': 1.5, 'bad': [0.5, 0.25]}
    assert s['right'] == {'n_valid': 0, 'epe': 0.0, 'bad': [0.0, 0.0]}
    assert s['all'] == {'n_valid': 4, 'epe': 1.5, 'bad': [0.5, 0.25]}
    block[4:] = torch.tensor([4, 2 * 65536 + 32768, 1, 0])
    s = T.disp_summary(block, th)
    assert s['right']['epe'] == 0.625 and s['all']['n_valid'] == 8
    assert s['all']['epe'] == (6 + 2.5) / 8 and s['all']['bad'] == [3 / 8, 1 / 8]


# ---- the extended stats vector through the single all-reduce -----------------------------------------------------------
_T, _TD = 4, 2


def _fake_sample(i):
    g = torch.Generator().manual_seed(2000 + i)
    inter = torch.randint(0, 2000, (_T,), generator=g)
    union = inter + torch.randint(1, 3000, (_T,), generator=g)
    nval = torch.randint(100, 65536, (2,), generator=g)
    epe = nval * torch.randint(0, 40 << 16, (2,), generator=g)      # large fixed-point sums
    bad = torch.stack([torch.randint(0, int(n) + 1, (_TD,), generator=g) for n in nval])
    return inter, union, torch.cat([nval.view(2, 1), epe.view(2, 1), bad], 1)


def _local_stats(n, rank, world):
    s = torch.zeros(2 * _T + 1 + 2 * (2 + _TD), dtype=torch.int64)
    lo, hi = T.shard_range(n, rank, world)
    for i in range(lo, hi):
        a, u, ds = _fake_sample(i)
        s[:_T] += a; s[_T:2 * _T] += u; s[2 * _T] += 1
        s[2 * _T + 1:] += ds.flatten()
    return s


def _worker(rank, world, port, n, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    s = T.reduce_stats(_local_stats(n, rank, world))
    if rank == 0:
        q.put(s.tolist())
    dist.destroy_process_group()


def test_gloo_world2_extended_vector_matches_single_process():
    n = 37
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
    assert T.iou_summary(got[:2 * _T + 1], [0.2, 0.3, 0.4, 0.5])['n_samples'] == n
    summ = T.disp_summary(got[2 * _T + 1:], [1.0, 3.0])
    assert summ['all']['n_valid'] == summ['left']['n_valid'] + summ['right']['n_valid']
    assert all(0 <= v <= 1 for v in summ['all']['bad'])
