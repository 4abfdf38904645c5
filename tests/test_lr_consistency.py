"""Left-right consistency check, host side: the reference statement in tests/lr_oracle.py (half-even rounding of the
match column, non-strict tolerance, range and non-finite rules), perfect prediction on the synthetic GT, the summary
arithmetic, and the stats vector extended by the LR counters through a gloo world-2 all-reduce."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.utils import synthetic
from tests.lr_oracle import lr_consistency

NAN, INF = float('nan'), float('inf')
W = 8


def _pair(left_row, right_row):
    """One sample, one row: [1, 2, 1, W] from the two views' rows (lists of W floats)."""
    return torch.tensor([[[left_row], [right_row]]], dtype=torch.float32)


def _kept(disp, tau=1.0):
    return lr_consistency(disp, tau)[0][0, :, 0].tolist()


def test_match_column_rounds_half_to_even():
    # view 0 at x = 6: d = 2.5 -> k = 2 -> xo = 4; d = 3.5 -> k = 4 -> xo = 2.  Only the right-view pixel the rounding
    # picks holds a value within tau.
    far = 100.0
    for d, xo in ((2.5, 4), (3.5, 2), (1.5, 4), (0.5, 6)):
        left = [far] * W
        left[6] = d
        right = [-far] * W
        right[xo] = d
        assert _kept(_pair(left, right))[0][6] == 1, (d, xo)
        right = [-far] * W
        right[xo - 1] = d
        right[xo + 1 if xo + 1 < W else xo - 2] = d
        assert _kept(_pair(left, right))[0][6] == 0, (d, xo)


def test_tolerance_is_inclusive():
    up = torch.nextafter(torch.tensor(4.0), torch.tensor(INF)).item()
    for other, tau, want in ((4.0, 1.0, 1), (up, 1.0, 0), (2.0, 1.0, 1), (3.0, 0.0, 1), (4.0, 0.0, 0)):
        left = [50.0] * W
        left[5] = 3.0                                                    # xo = 2
        right = [-50.0] * W
        right[2] = other
        assert _kept(_pair(left, right), tau)[0][5] == want, (other, tau)


def test_match_column_range():
    # view 0: xo = x - k; view 1: xo = x + k.  xo = -1 and W are out of range, 0 and W - 1 are in.
    for x, d, want in ((2, 3.0, 0), (2, 2.0, 1), (0, -(W - 1.0), 1), (0, -float(W), 0), (3, 3.0, 1), (3, 4.0, 0)):
        left = [1000.0] * W
        left[x] = d
        right = [d] * W
        assert _kept(_pair(left, right))[0][x] == want, (x, d)
    for x, d, want in ((W - 3, 2.0, 1), (W - 3, 3.0, 0), (1, -1.0, 1), (1, -2.0, 0)):
        right = [1000.0] * W
        right[x] = d
        left = [d] * W
        assert _kept(_pair(left, right))[1][x] == want, (x, d)


def test_non_finite_and_negative():
    left = [NAN, INF, -INF, 1e30, -1e30, -1.0, 0.0, 2.0]
    right = [0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, NAN]
    k = _kept(_pair(left, right))
    # own NaN / inf / huge: never; d = -1 at x = 5 -> xo = 6 (right 0.0, |-1 - 0| = 1): kept; d = 0 at x = 6 -> itself: kept
    # d = 2 at x = 7 -> xo = 5 (0.0): |2 - 0| = 2 > 1
    assert k[0] == [0, 0, 0, 0, 0, 1, 1, 0]
    # view 1, d = 0 everywhere finite -> xo = x: kept where the left value is within 1 of 0; x = 7 is NaN
    assert k[1] == [0, 0, 0, 0, 0, 1, 1, 0]
    # NaN on the OTHER side only: view 0 at x = 4 (d = 1) looks at right[3]; view 1 at x = 2 looks at left[3]
    k = _kept(_pair([1.0] * W, [1.0] * 3 + [NAN] + [1.0] * 4))
    assert k[0][4] == 0 and k[0][5] == 1 and k[1][3] == 0 and k[1][2] == 1
    k = _kept(_pair([1.0] * 3 + [NAN] + [1.0] * 4, [1.0] * W))
    assert k[1][2] == 0 and k[1][1] == 1 and k[0][3] == 0 and k[0][4] == 1


def test_counts_and_gt_columns():
    g = torch.Generator().manual_seed(1)
    disp = torch.rand(3, 2, 5, 16, generator=g) * 6
    gt = disp + (torch.rand(disp.shape, generator=g) - 0.5) * 6
    gt[0, 0, 0, :4] = NAN
    mask, c = lr_consistency(disp, 1.0, gt, [1.0, 3.0], 16.0)
    assert mask.shape == disp.shape and mask.dtype == torch.uint8 and c.shape == (3, 2, 5) and c.dtype == torch.int64
    kept = mask.bool()
    valid = torch.isfinite(gt) & (gt >= 0) & (gt < 16.0)
    e = (disp - gt).abs()
    assert torch.equal(c[..., 0], kept.flatten(2).sum(-1))
    assert torch.equal(c[..., 1], (kept & valid).flatten(2).sum(-1))
    assert torch.equal(c[..., 4], (kept & valid & (e > 3.0)).flatten(2).sum(-1))
    assert 0 < c[..., 0].sum() < disp.numel()
    _, c0 = lr_consistency(disp, 1.0, thresholds=[1.0, 3.0])                   # without GT: the GT columns stay zero
    assert torch.equal(c0[..., 0], c[..., 0]) and (c0[..., 1:] == 0).all()


@pytest.mark.parametrize('B,H,W_,maxd', [(2, 9, 13, 8), (3, 16, 40, 12), (1, 4, 5, 16)])
def test_perfect_prediction_keeps_exactly_the_pixels_with_gt(B, H, W_, maxd):
    _, _, d = synthetic.stereo_pair(B, H, W_, maxd, seed=7)
    gt = synthetic.disparity_gt(d, H, W_)
    mask, c = lr_consistency(gt, 0.0, gt, [1.0], 4.0 * maxd)
    assert torch.equal(mask.bool(), torch.isfinite(gt))
    n = torch.isfinite(gt).flatten(2).sum(-1)
    assert torch.equal(c[..., 0], n) and torch.equal(c[..., 1], n) and (c[..., 2:] == 0).all()


def test_lr_summary_arithmetic():
    th = [1.0, 3.0]
    disp = torch.tensor([8, 0, 0, 0,  5, 0, 0, 0], dtype=torch.int64)          # n_valid 8 (left), 5 (right)
    lr = torch.tensor([10, 4, 6 * 65536, 2, 1,                                   # left: 10 kept, 4 valid, EPE 1.5
                       6, 0, 0, 0, 0], dtype=torch.int64)                        # right: 6 kept, none valid
    s = T.lr_summary(lr, th, 20, disp)
    assert s['thresholds'] == th
    assert s['left'] == {'n_kept': 10, 'density': 0.5, 'n_valid_kept': 4, 'kept_of_valid': 0.5, 'epe': 1.5, 'bad': [0.5, 0.25]}
    assert s['right'] == {'n_kept': 6, 'density': 0.3, 'n_valid_kept': 0, 'kept_of_valid': 0.0, 'epe': 0.0, 'bad': [0.0, 0.0]}
    assert s['all'] == {'n_kept': 16, 'density': 0.4, 'n_valid_kept': 4, 'kept_of_valid': 4 / 13, 'epe': 1.5,
                        'bad': [0.5, 0.25]}
    lr[5:] = torch.tensor([6, 4, 2 * 65536 + 32768, 1, 0])
    s = T.lr_summary(lr, th, 20, disp)
    assert s['right']['epe'] == 0.625 and s['right']['kept_of_valid'] == 0.8
    assert s['all']['epe'] == (6 + 2.5) / 8 and s['all']['bad'] == [3 / 8, 1 / 8]


def test_driver_rejects_lr_without_disp():
    from tests.common import small_cfg
    for fn in (T.test_voxel, T.test_point):
        with pytest.raises(ValueError):
            fn(small_cfg(), None, 1, 1, device='cpu', eval_disp=False, eval_lr=True)


# ---- the stats vector with the LR counters through the single all-reduce ------------------------------------------------
_T, _TD = 4, 2
_NH, _ND, _NL = 2 * _T + 1, 2 * (2 + _TD), 2 * (3 + _TD)


def _fake_sample(i):
    g = torch.Generator().manual_seed(3000 + i)
    inter = torch.randint(0, 2000, (_T,), generator=g)
    union = inter + torch.randint(1, 3000, (_T,), generator=g)
    nval = torch.randint(100, 65536, (2,), generator=g)
    epe = nval * torch.randint(0, 40 << 16, (2,), generator=g)
    bad = torch.stack([torch.randint(0, int(n) + 1, (_TD,), generator=g) for n in nval])
    nvk = torch.stack([torch.randint(0, int(n) + 1, (1,), generator=g) for n in nval]).view(2)
    nk = nvk + torch.randint(0, 65536, (2,), generator=g)
    epek = nvk * torch.randint(0, 40 << 16, (2,), generator=g)
    badk = torch.stack([torch.randint(0, int(n) + 1, (_TD,), generator=g) for n in nvk])
    ds = torch.cat([nval.view(2, 1), epe.view(2, 1), bad], 1)
    ls = torch.cat([nk.view(2, 1), nvk.view(2, 1), epek.view(2, 1), badk], 1)
    return inter, union, ds, ls


def _local_stats(n, rank, world):
    s = torch.zeros(_NH + _ND + _NL, dtype=torch.int64)
    lo, hi = T.shard_range(n, rank, world)
    for i in range(lo, hi):
        a, u, ds, ls = _fake_sample(i)
        s[:_T] += a; s[_T:2 * _T] += u; s[2 * _T] += 1
        s[_NH:_NH + _ND] += ds.flatten()
        s[_NH + _ND:] += ls.flatten()
    return s


def _worker(rank, world, port, n, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    s = T.reduce_stats(_local_stats(n, rank, world))
    if rank == 0:
        q.put(s.tolist())
    dist.destroy_process_group()


def test_gloo_world2_lr_vector_matches_single_process():
    n = 29
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
    summ = T.lr_summary(got[_NH + _ND:], [1.0, 3.0], n * 64 * 64, got[_NH:_NH + _ND])
    assert summ['all']['n_kept'] == summ['left']['n_kept'] + summ['right']['n_kept']
    assert all(0 <= v <= 1 for v in summ['all']['bad']) and 0 <= summ['all']['kept_of_valid'] <= 1
