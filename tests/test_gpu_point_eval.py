"""Point-cloud evaluation inside the forward (s3d_chamfer_eval): the distances and indices are bit-identical to
s3d_chamfer_forward_ws, and the integer counters equal the reference statement (tests/point_oracle.py) on the C oracle's
distances of the very points the forward returns."""
import ctypes
import json
import sys

import numpy as np
import pytest
import torch

from config import cfg as default_cfg
from oracle.chamfer import chamfer_c
from stereo_3d_reconstruction_b200 import lib, models as M, ops
from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.utils import synthetic
from tests.common import small_cfg
from tests.point_oracle import fscore_fx, point_counts, point_stats

pytestmark = pytest.mark.gpu
TH = [0.005, 0.01, 0.03, 0.1]
NAN, INF = float('nan'), float('inf')


def _eval(a, b, th=TH, stats=None):
    B = a.shape[0]
    if stats is None:
        stats = torch.zeros(B, 2, 3 + len(th), dtype=torch.int64, device='cuda')
    return ops.chamfer_eval(a, b, th, stats), stats


def _bits(t):
    return t.view(torch.int32).cpu().numpy()


def _check(a, b, th=TH):
    """a [B,N,3], b [B,M,3] CPU: dist / idx against chamfer_forward (bit for bit) and the C oracle, stats against the
    reference statement; the stats accumulate.  -> the expected stats (numpy)."""
    ac, bc = a.cuda(), b.cuda()
    ref = ops.chamfer_forward(ac, bc)
    got, st = _eval(ac, bc, th)
    for x, y in zip(got, ref):
        assert np.array_equal(_bits(x), _bits(y))
    rd1, rd2, ri1, ri2 = chamfer_c(a.numpy(), b.numpy())
    assert np.array_equal(_bits(got[0]), rd1.view(np.int32)) and np.array_equal(_bits(got[1]), rd2.view(np.int32))
    assert np.array_equal(got[2].cpu().numpy(), ri1) and np.array_equal(got[3].cpu().numpy(), ri2)
    want = point_counts(rd1, rd2, th)
    assert np.array_equal(st.cpu().numpy(), want)
    _eval(ac, bc, th, stats=st)                                     # ADDED to: a second call doubles every counter
    assert np.array_equal(st.cpu().numpy(), 2 * want)
    return want


SIZES = [
    (3, 300, 1000, False),       # N < M
    (2, 1000, 300, True),        # N > M, exact ties
    (5, 1023, 2049, False),      # ragged: neither a multiple of 32 nor of the kernel's 1024-point blocks
    (1, 1, 513, False),          # N = 1, B = 1
    (4, 777, 1, False),          # M = 1
    (2, 2048, 4096, True),
]


@pytest.mark.parametrize('sym,R', [(-1, 0), (1, 4), (1, 8)])
@pytest.mark.parametrize('B,N,M_,dup', SIZES)
def test_kernel_matches_search_and_oracle(B, N, M_, dup, sym, R, knobs):
    knobs('chamfer_sym', sym)                                       # -1: one search per direction; 1: the one-pass kernel
    knobs('chamfer_sym_r', R)
    if sym == 1:
        assert ops.chamfer_workspace_bytes(B, N, M_) == 8 * B * min(N, M_)
    a, b = synthetic.point_clouds(B, N, M_, seed=B * 100 + N + M_, duplicates=dup)
    want = _check(a, b)
    assert (want[:, :, 2] == 0).all() and (want[:, :, 0] > 0).any()
    if min(N, M_) > 100:
        assert (want[:, :, 3 + 2] > 0).all()                        # the thresholds are not vacuous


def test_kernel_threshold_count_edges():
    a, b = synthetic.point_clouds(2, 600, 900, seed=4, duplicates=True)
    _check(a, b, [0.02 * (k + 1) for k in range(8)])                # eight thresholds
    _check(a, b, [])                                                # none
    _check(a, b, [1e-30, 10.0])                                     # only exact duplicates / every point


def test_kernel_full_size():
    """The default Stereo2Point shape: 32 x 2048 predicted vs 16384 GT points (the one-pass search at this size)."""
    assert ops.chamfer_workspace_bytes(32, 2048, 16384) > 0
    a, b = synthetic.point_clouds(32, 2048, 16384, seed=8, duplicates=True)
    want = _check(a, b, [0.01, 0.02])
    assert (want[:, :, 3] > 0).all()


@pytest.mark.parametrize('sym', [-1, 1])
def test_kernel_non_finite_and_out_of_range(sym, knobs):
    knobs('chamfer_sym', sym)
    a, b = synthetic.point_clouds(3, 300, 500, seed=6)
    a[0, 5] = torch.tensor([NAN, 0.0, 0.0])                         # NaN points: d = +inf
    b[0, 7] = torch.tensor([0.0, NAN, 0.0])
    a[0, 9] = torch.tensor([30.0, 0.0, 0.0])                        # far away: d >= 2^8
    b[1, :4] = torch.tensor([[20.0, 0, 0], [-20.0, 0, 0], [0, 20.0, 0], [0, 0, -17.0]])
    b[2] = NAN                                                      # a sample with no usable GT at all
    th = [0.5, float(np.nextafter(np.float32(0.5), np.float32(INF))), 0.05]
    want = _check(a, b, th)
    edge = _check(torch.zeros(1, 1, 3), torch.tensor([[[0.5, 0.0, 0.0]]]), th)
    assert edge[0, :, 3:].tolist() == [[0, 1, 0], [0, 1, 0]]       # strictly less than tau, in fp32
    assert want[0, 0, 2] == 2 and want[0, 1, 2] == 1 and want[1, 1, 2] >= 4
    assert (want[2, :, 2] == [300, 500]).all() and (want[2, :, [0, 1, 3]] == 0).all()


def test_kernel_bad_arguments():
    L = lib.load()
    B, N, M_ = 2, 64, 96
    a = torch.rand(B, N, 3, device='cuda')
    b = torch.rand(B, M_, 3, device='cuda')
    d1, i1 = torch.empty(B, N, device='cuda'), torch.empty(B, N, dtype=torch.int32, device='cuda')
    d2, i2 = torch.empty(B, M_, device='cuda'), torch.empty(B, M_, dtype=torch.int32, device='cuda')
    st = torch.zeros(B, 2, 3 + 8, dtype=torch.int64, device='cuda')
    s = torch.cuda.current_stream().cuda_stream
    ptr = dict(a=a.data_ptr(), b=b.data_ptr(), d1=d1.data_ptr(), i1=i1.data_ptr(), d2=d2.data_ptr(), i2=i2.data_ptr(),
               st=st.data_ptr())

    def th(*v):
        return (ctypes.c_float * max(len(v), 1))(*v)

    def call(T_=2, th_=th(0.1, 0.2), B_=B, N_=N, M__=M_, **kw):
        p = dict(ptr, **kw)
        return L.s3d_chamfer_eval(p['a'], p['b'], p['d1'], p['i1'], p['d2'], p['i2'], B_, N_, M__, th_, T_, p['st'], None, 0, s)
    assert call() == 0
    assert call(T_=0, th_=None) == 0 and call(T_=8, th_=th(*[0.1] * 8)) == 0 and call(B_=0) == 0
    for bad in (dict(st=None), dict(th_=None), dict(T_=9, th_=th(*[0.1] * 9)), dict(T_=-1),
                dict(th_=th(0.1, NAN)), dict(th_=th(INF, 0.1)), dict(th_=th(0.1, 0.0)), dict(th_=th(-0.1, 0.1)),
                dict(N_=1 << 22), dict(M__=1 << 22), dict(N_=0), dict(M__=0), dict(B_=-1),
                dict(a=None), dict(b=None), dict(d1=None), dict(i2=None)):
        rc = call(**bad)
        assert rc == -1, bad
        with pytest.raises(lib.S3dError):
            lib.check(rc, 's3d_chamfer_eval')
    torch.cuda.synchronize()
    with pytest.raises(ValueError):                                 # the Python wrapper checks shapes and dtypes
        ops.chamfer_eval(a, b, [0.1], torch.zeros(B, 2, 3, dtype=torch.int64, device='cuda'))
    with pytest.raises(ValueError):
        ops.chamfer_eval(a.double(), b, [0.1], st[..., :4].contiguous())


# ---- the model ------------------------------------------------------------------------------------------------------------
PT_TH = [0.05, 0.1, 0.2]


def _model(cv, prec, seed=3, **kw):
    kw.setdefault('TEST__FSCORE_THRESH', PT_TH)
    cfg = small_cfg(NETWORK__PRECISION=prec, NETWORK__COST_VOLUME=cv, **kw)
    return cfg, M.build_model('Stereo2Point', cfg, seed=seed).cuda().pack()


def _inputs(cfg, B, seed, n_gt=1000):
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=seed)
    gt = synthetic.point_clouds(B, 1, n_gt, seed=seed + 50)[1]
    return (left.cuda(), right.cuda()), gt.cuda(), synthetic.disparity_gt(d, H, W).cuda()


def _check_points(cfg, points, gt, ps):
    th = list(cfg.TEST.FSCORE_THRESH)
    assert ps.dtype == torch.int64 and ps.shape == (points.shape[0], 2, 3 + len(th))
    want = point_stats(points.cpu(), gt.cpu(), th)
    assert np.array_equal(ps.cpu().numpy(), want)
    return want


@pytest.mark.parametrize('prec', ['bf16', 'fp32', 'bf16x3'])
@pytest.mark.parametrize('cv', ['concat', 'corr'])
def test_model_outputs_unchanged_and_point_stats_exact(cv, prec):
    cfg, model = _model(cv, prec)
    args, gt, dgt = _inputs(cfg, 2, seed=0)
    with torch.no_grad():
        n0 = lib.launches()
        plain = [t.clone() for t in model(*args)]
        n1 = lib.launches()
        pt = [t.clone() for t in model(*args, gt)]
        n2 = lib.launches()
        ev = [t.clone() for t in model(*args, disp_gt=dgt, lr_check=True)]
        full = [t.clone() for t in model(*args, gt, disp_gt=dgt, lr_check=True)]
    assert (n2 - n1) - (n1 - n0) == 3                               # the two search kernels + chamfer_eval_kernel
    assert len(plain) == 3 and len(pt) == 4 and len(ev) == 6 and len(full) == 7
    for a, b in zip(plain, pt):
        assert torch.equal(a, b)
    for a, b in zip(ev, full[:3] + full[4:]):                       # disparities, points, disp_stats, lr_mask, lr_stats
        assert torch.equal(a, b)
    assert torch.equal(full[3], pt[3])
    want = _check_points(cfg, pt[2], gt, pt[3])
    assert (want[:, :, 2] == 0).all() and want[:, :, 3:].sum() > 0


def test_model_padded_points_row():
    """N_POINTS = 100: the fc2 output row (300 values) is padded to 304, so the points are copied out before the search."""
    cfg, model = _model('concat', 'bf16', CONST__N_POINTS=100)
    args, gt, _ = _inputs(cfg, 3, seed=2, n_gt=257)
    with torch.no_grad():
        plain = [t.clone() for t in model(*args)]
        out = model(*args, gt)
    assert not out[2].is_contiguous()
    for a, b in zip(plain, out):
        assert torch.equal(a, b)
    _check_points(cfg, out[2], gt, out[3])


def test_model_gt_validation():
    cfg, model = _model('concat', 'bf16')
    args, gt, _ = _inputs(cfg, 2, seed=0)
    for bad in (gt[:1], gt[..., :2], gt[0], gt.double(), gt.cpu(), gt[:, :0], gt.tolist()):
        with pytest.raises(ValueError):
            model(*args, bad)
        with pytest.raises(ValueError):
            model.graphed(*args, bad)
    n0 = lib.launches()
    for bad in ([-0.1], [NAN], [INF], [0.1] * 9):
        cfg.TEST.FSCORE_THRESH = bad
        with pytest.raises(ValueError):
            model(*args, gt)
        with pytest.raises(ValueError):
            model.graphed(*args, gt)
    assert lib.launches() == n0                                     # rejected before anything is launched
    cfg.TEST.FSCORE_THRESH = [0.5] * 5
    with torch.no_grad():
        assert model(*args)[2].shape == (2, cfg.CONST.N_POINTS, 3)
        assert model(*args, gt)[3].shape == (2, 2, 8)


def test_graphed_with_gt_matches_eager():
    cfg, model = _model('concat', 'bf16')
    seen = []
    for seed in (0, 1):
        args, gt, dgt = _inputs(cfg, 2, seed=seed)
        with torch.no_grad():
            eager = [t.clone() for t in model(*args, gt)]
            graphed = [t.clone() for t in model.graphed(*args, gt)]
        assert len(model._graphs) == 1
        assert len(graphed) == 4
        for a, b in zip(eager, graphed):
            assert torch.equal(a, b)
        _check_points(cfg, graphed[2], gt, graphed[3])
        seen.append(eager[3])
    assert not torch.equal(seen[0], seen[1])
    with torch.no_grad():                                           # gt binds to the point cloud, disp_gt stays keyword-only
        full = [t.clone() for t in model(*args, gt, disp_gt=dgt, lr_check=True)]
        g = [t.clone() for t in model.graphed(*args, gt, disp_gt=dgt, lr_check=True)]
        assert len(model._graphs) == 2 and len(g) == 7
        for a, b in zip(full, g):
            assert torch.equal(a, b)
        assert len(model.graphed(*args)) == 3 and len(model._graphs) == 3


def test_driver_eval_points():
    cfg, model = _model('concat', 'bf16', CONST__N_GT_POINTS=1000)
    n, bs = 3, 2
    base = T.test_point(cfg, model, n, bs, eval_disp=True, eval_lr=True).cpu()
    full = T.test_point(cfg, model, n, bs, eval_disp=True, eval_lr=True, eval_points=True).cpu()
    assert torch.equal(full[:base.numel()], base)
    assert torch.equal(T.test_point(cfg, model, n, bs, eval_points=True).cpu()[2:], full[base.numel():])
    H, W, N = cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.CONST.N_POINTS
    Mg = cfg.CONST.N_GT_POINTS
    want = np.zeros(2 * (3 + len(PT_TH)) + len(PT_TH), dtype=np.int64)
    for s in range(0, n, bs):                                       # the same batches, the model's own points
        ids = range(s, min(s + bs, n))
        pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in ids]
        gt = torch.cat([synthetic.point_clouds(1, 1, Mg, seed=200000 + i)[1] for i in ids])
        with torch.no_grad():
            pts = model(torch.cat([p[0] for p in pairs]).cuda(), torch.cat([p[1] for p in pairs]).cuda())[2]
        c = point_stats(pts.cpu(), gt, PT_TH)
        want += np.concatenate([c.sum(0).flatten(), fscore_fx(c, N, Mg)])
    assert np.array_equal(full[base.numel():].numpy(), want)
    summ = T.points_summary(full[base.numel():], PT_TH, n, N, Mg)
    cd = T.chamfer_summary(base[:2])['chamfer_distance']
    assert summ['n_out'] == 0 and abs(summ['chamfer_l2'] - cd) <= 2.0 ** -31       # the fixed-point bound: 2^-33 a point
    assert 0 < summ['chamfer_l1'] < 1 and all(0 <= f <= 1 for f in summ['fscore']) and summ['fscore'][-1] > 0


def test_runner_adds_points_and_keeps_every_key(monkeypatch, capsys):
    import runner
    n, bs = 3, 2
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test', '--model', 'Stereo2Point', '--batch-size', str(bs),
                                      '--n-samples', str(n), '--lr-check'])
    runner.main()
    res = json.loads(capsys.readouterr().out.strip().splitlines()[-1])
    cfg = default_cfg.clone()
    model = M.build_model('Stereo2Point', cfg, seed=cfg.CONST.SEED).cuda().pack()
    old = T.test_point(cfg, model, n, bs, eval_disp=True, eval_lr=True).cpu()      # what the runner reported before
    nd = 2 * (2 + len(cfg.TEST.DISP_THRESH))
    want = T.chamfer_summary(old[:2])
    want['disparity'] = T.disp_summary(old[2:2 + nd], cfg.TEST.DISP_THRESH)
    want['lr_consistency'] = T.lr_summary(old[2 + nd:], cfg.TEST.DISP_THRESH, n * cfg.CONST.IMG_H * cfg.CONST.IMG_W, old[2:2 + nd])
    want['lr_consistency']['lr_thresh'] = float(cfg.TEST.LR_THRESH)
    for k, v in want.items():
        assert res[k] == json.loads(json.dumps(v)), k
    full = T.test_point(cfg, model, n, bs, eval_disp=True, eval_lr=True, eval_points=True).cpu()
    pts = T.points_summary(full[old.numel():], cfg.TEST.FSCORE_THRESH, n, cfg.CONST.N_POINTS, cfg.CONST.N_GT_POINTS)
    assert res['points'] == json.loads(json.dumps(pts))
    assert res['points']['thresholds'] == [0.01] and res['points']['n_out'] == 0
    assert abs(res['points']['chamfer_l2'] - res['chamfer_distance']) <= 2.0 ** -31
