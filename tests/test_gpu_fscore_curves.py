"""Nearest-neighbour distance histograms inside the forward (s3d_chamfer_eval_hist, s3d_voxel_surface_eval_hist): the
histograms equal the reference statement (tests/fscore_curves_oracle.py) bit for bit, on hand-built and random inputs and on
the very points / voxels the forward returns; every other output, the launch count and the existing entry points are
unchanged."""
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
from tests import fscore_curves_oracle as O
from tests.common import small_cfg

pytestmark = pytest.mark.gpu
TH = [0.005, 0.01, 0.03]
NAN, INF = float('nan'), float('inf')


def _bits(t):
    return t.view(torch.int32).cpu().numpy()


# ---- the point kernel ---------------------------------------------------------------------------------------------------
def _point_check(a, b, e, th=TH):
    """a [B,N,3], b [B,M,3] CPU: dist / idx / stats of the histogram call bit-identical to the plain call, the histogram
    equal to the oracle's on the C oracle's distances, and ADDED to.  -> the expected histogram."""
    ac, bc = a.cuda(), b.cuda()
    B, K = a.shape[0], len(e)
    st0 = torch.zeros(B, 2, 3 + len(th), dtype=torch.int64, device='cuda')
    ref = [t.clone() for t in ops.chamfer_eval(ac, bc, th, st0)]
    st = torch.zeros_like(st0)
    hist = torch.zeros(B, 2, K + 1, dtype=torch.int64, device='cuda')
    n0 = lib.launches()
    got = ops.chamfer_eval(ac, bc, th, st, edges=e, hist=hist)
    assert lib.launches() - n0 == 3                                  # no launch added
    for x, y in zip(got, ref):
        assert np.array_equal(_bits(x), _bits(y))
    assert torch.equal(st, st0)
    d1, d2, _, _ = chamfer_c(a.numpy(), b.numpy())
    want = O.point_hist_of_dists(d1, d2, e)
    assert np.array_equal(hist.cpu().numpy(), want)
    assert (want[:, 0].sum(-1) == a.shape[1]).all() and (want[:, 1].sum(-1) == b.shape[1]).all()
    ops.chamfer_eval(ac, bc, th, st, edges=e, hist=hist)             # a second call doubles the histograms
    assert np.array_equal(hist.cpu().numpy(), 2 * want)
    return want


SIZES = [(3, 300, 1000, False), (2, 1000, 300, True), (5, 1023, 2049, False), (1, 1, 513, False), (4, 777, 1, False),
         (2, 2048, 4096, True)]


@pytest.mark.parametrize('sym,R', [(-1, 0), (1, 4), (1, 8)])
@pytest.mark.parametrize('B,N,M_,dup', SIZES)
def test_point_hist_matches_oracle(B, N, M_, dup, sym, R, knobs):
    knobs('chamfer_sym', sym)
    knobs('chamfer_sym_r', R)
    a, b = synthetic.point_clouds(B, N, M_, seed=B * 100 + N + M_, duplicates=dup)
    want = _point_check(a, b, O.edges(0.128, 128))
    if min(N, M_) > 100:
        assert (want[..., :128].sum(-1) > 0).all()                   # the edges are not vacuous


@pytest.mark.parametrize('K,dmax', [(1, 0.05), (2, 0.05), (128, 0.128), (1024, 0.5), (1024, 0.002)])
def test_point_hist_bin_counts(K, dmax):
    a, b = synthetic.point_clouds(3, 600, 900, seed=K, duplicates=True)
    _point_check(a, b, O.edges(dmax, K))


def test_point_hist_full_size():
    a, b = synthetic.point_clouds(32, 2048, 16384, seed=8, duplicates=True)
    for K in (128, 1024):
        want = _point_check(a, b, O.edges(0.128, K), th=[0.01])
        assert (want[:, :, 1:K].sum(-1) > 0).all()


@pytest.mark.parametrize('sym', [-1, 1])
def test_point_hist_non_finite_ties_and_out_of_range(sym, knobs):
    knobs('chamfer_sym', sym)
    a, b = synthetic.point_clouds(3, 300, 500, seed=6)
    a[0, 5] = torch.tensor([NAN, 0.0, 0.0])
    b[0, 7] = torch.tensor([0.0, INF, 0.0])
    a[0, 9] = torch.tensor([30.0, 0.0, 0.0])
    b[1, :4] = torch.tensor([[20.0, 0, 0], [-20.0, 0, 0], [0, 20.0, -INF], [0, 0, -17.0]])
    b[2] = NAN
    want = _point_check(a, b, O.edges(0.128, 128))
    assert want[2, 0, 128] == 300 and want[2, 1, 128] == 500 and want[0, 0, 128] >= 2
    e = np.array([0.25, 0.5, 0.75], np.float32)                      # distances exactly on the edges: the bin above
    tie = _point_check(torch.zeros(1, 1, 3), torch.tensor([[[0.25, 0, 0], [0.5, 0, 0], [0.0, 0.75, 0], [0.1, 0, 0]]]), e)
    assert tie[0, 1].tolist() == [1, 1, 1, 1] and tie[0, 0].tolist() == [1, 0, 0, 0]


def _abi_point(L, B, N, M_, edges, K, hist_ptr, stats):
    a = torch.rand(max(B, 1), N, 3, device='cuda')
    b = torch.rand(max(B, 1), M_, 3, device='cuda')
    d1, i1 = torch.empty(max(B, 1), N, device='cuda'), torch.empty(max(B, 1), N, dtype=torch.int32, device='cuda')
    d2, i2 = torch.empty(max(B, 1), M_, device='cuda'), torch.empty(max(B, 1), M_, dtype=torch.int32, device='cuda')
    th = (ctypes.c_float * 1)(0.1)
    ed = None if edges is None else (ctypes.c_float * max(len(edges), 1))(*edges)
    return L.s3d_chamfer_eval_hist(a.data_ptr(), b.data_ptr(), d1.data_ptr(), i1.data_ptr(), d2.data_ptr(), i2.data_ptr(),
                                   B, N, M_, th, 1, stats.data_ptr(), None, 0, torch.cuda.current_stream().cuda_stream,
                                   ed, K, hist_ptr)


def test_point_hist_bad_arguments_and_empty_batch():
    L = lib.load()
    B, N, M_ = 2, 64, 96
    st = torch.zeros(B, 2, 4, dtype=torch.int64, device='cuda')
    hist = torch.zeros(B, 2, 1025, dtype=torch.int64, device='cuda')
    e = [0.01 * (k + 1) for k in range(8)]
    assert _abi_point(L, B, N, M_, e, 8, hist.data_ptr(), st) == 0
    assert _abi_point(L, B, N, M_, None, 0, None, st) == 0           # K = 0: the plain evaluation
    assert _abi_point(L, B, N, M_, [0.001 * (k + 1) for k in range(1024)], 1024, hist.data_ptr(), st) == 0
    for edges, K, hp in ((e, -1, hist.data_ptr()), ([0.001 * (k + 1) for k in range(1025)], 1025, hist.data_ptr()),
                         (None, 8, hist.data_ptr()), (e, 8, None), ([0.1, NAN], 2, hist.data_ptr()),
                         ([0.1, INF], 2, hist.data_ptr()), ([0.0, 0.1], 2, hist.data_ptr()),
                         ([-0.1, 0.1], 2, hist.data_ptr()), ([0.1, 0.1], 2, hist.data_ptr()),
                         ([0.2, 0.1], 2, hist.data_ptr())):
        rc = _abi_point(L, B, N, M_, edges, K, hp, st)
        assert rc == -1, (edges, K)
        with pytest.raises(lib.S3dError):
            lib.check(rc, 's3d_chamfer_eval_hist')
    torch.cuda.synchronize()
    sentinel = torch.full((1, 2, 9), 7, dtype=torch.int64, device='cuda')
    st1 = torch.full((1, 2, 4), 7, dtype=torch.int64, device='cuda')
    assert _abi_point(L, 0, N, M_, e, 8, sentinel.data_ptr(), st1) == 0  # B = 0: nothing launched, nothing written
    torch.cuda.synchronize()
    assert (sentinel == 7).all() and (st1 == 7).all()
    a, b = torch.rand(B, N, 3, device='cuda'), torch.rand(B, M_, 3, device='cuda')
    good = torch.zeros(B, 2, 9, dtype=torch.int64, device='cuda')
    for kw in (dict(edges=e), dict(hist=good), dict(edges=e, hist=good[..., :8]), dict(edges=e, hist=good.int()),
               dict(edges=e, hist=good.cpu()), dict(edges=e[:1] * 2, hist=good[..., :3].contiguous()),
               dict(edges=[NAN] + e[1:], hist=good), dict(edges=[], hist=good[..., :1].contiguous()),
               dict(edges=[1e-3] * 1025, hist=torch.zeros(B, 2, 1026, dtype=torch.int64, device='cuda')),
               dict(edges='abc', hist=good), dict(edges=[1.0, 1.0 + 1e-9], hist=good[..., :3].contiguous())):
        with pytest.raises(ValueError):
            ops.chamfer_eval(a, b, [0.1], st, **kw)


# ---- the surface kernel -------------------------------------------------------------------------------------------------
LEVELS = np.array([0.1, 0.25, 0.5, 0.75, 0.9], np.float32)
VTH8 = [0.25, 0.5, 0.75, 0.9, 0.1, 0.3, 0.6, 0.95]
FTH = [0.01, 0.05]


def _grids(B, n, seed, p_gt=0.2):
    rng = np.random.default_rng(seed)
    fused = LEVELS[rng.integers(0, len(LEVELS), (B, n, n, n))]
    fused[rng.random((B, n, n, n)) < 0.02] = np.nan
    gt = (rng.random((B, n, n, n)) < p_gt).astype(np.uint8) * rng.integers(1, 256, (B, n, n, n)).astype(np.uint8)
    return fused, gt


def _surface_check(fused, gt, vth, e, fth=FTH):
    B, K = fused.shape[0], len(e)
    f, g = torch.from_numpy(np.ascontiguousarray(fused)).cuda(), torch.from_numpy(np.ascontiguousarray(gt)).cuda()
    st0 = torch.zeros(B, len(vth), 2, 3 + len(fth), dtype=torch.int64, device='cuda')
    ops.voxel_surface_eval(f, g, vth, fth, st0)
    st = torch.zeros_like(st0)
    hist = torch.zeros(B, len(vth), 2, K + 1, dtype=torch.int64, device='cuda')
    n0 = lib.launches()
    ops.voxel_surface_eval(f, g, vth, fth, st, edges=e, hist=hist)
    assert lib.launches() - n0 == (2 if B and vth else 0)
    assert torch.equal(st, st0)
    want = O.surface_hist(fused, gt, vth, e)
    assert np.array_equal(hist.cpu().numpy(), want)
    assert np.array_equal(want.sum(-1), st0[..., 0].cpu().numpy())  # rows sum to n_pts
    ops.voxel_surface_eval(f, g, vth, fth, st, edges=e, hist=hist)
    assert np.array_equal(hist.cpu().numpy(), 2 * want)
    return want


@pytest.mark.parametrize('n,B,T_,K', [(1, 3, 2, 4), (2, 3, 4, 16), (4, 3, 4, 128), (8, 3, 8, 128), (32, 3, 4, 128),
                                      (64, 1, 2, 1024), (8, 64, 4, 1), (32, 8, 4, 1024), (5, 2, 3, 2)])
def test_surface_hist_matches_oracle(n, B, T_, K):
    fused, gt = _grids(B, n, seed=n * 1000 + B * 10 + T_ + K)
    want = _surface_check(fused, gt, VTH8[:T_], O.edges(1.0 if n < 4 else 0.128, K))
    assert want.sum() > 0


def test_surface_hist_empty_and_full_grids():
    n = 8
    fused, gt = _grids(4, n, seed=11)
    gt[0] = 0                                                          # empty GT: the predicted points all in bin K
    fused[1] = 0.0                                                     # empty prediction at every t
    gt[2] = 1                                                          # full GT: its surface is the grid's boundary
    fused[3] = 1.0                                                     # full prediction
    e = O.edges(0.128, 128)
    want = _surface_check(fused, gt, [0.25, 0.5, 0.9], e)
    assert (want[0, :, 0, :128] == 0).all() and (want[0, :, 0, 128] > 0).all()
    assert (want[1, :, 1, :128] == 0).all() and (want[1, :, 0].sum(-1) == 0).all()
    assert (want[3, :, 0, 0] > 0).all()
    # repeated bounds (edges closer than one lattice step): empty bins between them
    want = _surface_check(*_grids(2, 4, seed=12), [0.5], O.edges(0.01, 16))
    assert (want[..., 1:16] == 0).all()


def _abi_surface(L, B, n, kb, K, hist_ptr):
    f = torch.rand(max(B, 1), n ** 3, device='cuda')
    g = torch.zeros(max(B, 1), n ** 3, dtype=torch.uint8, device='cuda')
    st = torch.zeros(max(B, 1), 1, 2, 3, dtype=torch.int64, device='cuda')
    need = ops.voxel_surface_workspace_bytes(max(B, 1), 1, n)
    ws = torch.empty(need, dtype=torch.uint8, device='cuda')
    th = (ctypes.c_float * 1)(0.5)
    kbp = None if kb is None else (ctypes.c_int * max(len(kb), 1))(*kb)
    return L.s3d_voxel_surface_eval_hist(f.data_ptr(), g.data_ptr(), B, n, th, 1, None, 0, st.data_ptr(), ws.data_ptr(),
                                         need, torch.cuda.current_stream().cuda_stream, kbp, K, hist_ptr)


def test_surface_hist_bad_arguments():
    L = lib.load()
    n, kmax = 4, 3 * 8 ** 2 + 1
    hist = torch.zeros(2, 1, 2, 1025, dtype=torch.int64, device='cuda')
    assert _abi_surface(L, 2, n, [0, 1, 1, 5, kmax], 5, hist.data_ptr()) == 0
    assert _abi_surface(L, 2, n, None, 0, None) == 0
    assert _abi_surface(L, 2, n, [1] * 1024, 1024, hist.data_ptr()) == 0
    for kb, K, hp in (([1], -1, hist.data_ptr()), ([1] * 1025, 1025, hist.data_ptr()), (None, 2, hist.data_ptr()),
                      ([1, 2], 2, None), ([2, 1], 2, hist.data_ptr()), ([-1, 2], 2, hist.data_ptr()),
                      ([1, kmax + 1], 2, hist.data_ptr())):
        rc = _abi_surface(L, 2, n, kb, K, hp)
        assert rc == -1, (kb, K)
        with pytest.raises(lib.S3dError):
            lib.check(rc, 's3d_voxel_surface_eval_hist')
    sentinel = torch.full((1, 1, 2, 3), 7, dtype=torch.int64, device='cuda')
    assert _abi_surface(L, 0, n, [1, 2], 2, sentinel.data_ptr()) == 0      # B = 0: nothing launched, nothing written
    torch.cuda.synchronize()
    assert (sentinel == 7).all()
    f = torch.rand(2, n, n, n, device='cuda')
    g = torch.zeros(2, n, n, n, dtype=torch.uint8, device='cuda')
    st = torch.zeros(2, 1, 2, 4, dtype=torch.int64, device='cuda')
    good = torch.zeros(2, 1, 2, 3, dtype=torch.int64, device='cuda')
    for kw in (dict(edges=[0.1, 0.2]), dict(hist=good), dict(edges=[0.1, 0.2], hist=good[..., :2]),
               dict(edges=[0.2, 0.1], hist=good), dict(edges=[0.1, INF], hist=good),
               dict(edges=[0.1, 0.2], hist=torch.zeros(2, 2, 2, 3, dtype=torch.int64, device='cuda'))):
        with pytest.raises(ValueError):
            ops.voxel_surface_eval(f, g, [0.5], [0.1], st, **kw)


# ---- the models ---------------------------------------------------------------------------------------------------------
def _inputs(cfg, B, seed, name):
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=seed)
    if name == 'Stereo2Point':
        gt = synthetic.point_clouds(B, 1, 1000, seed=seed + 50)[1]
    else:
        gt = synthetic.gt_volume(B, cfg.CONST.N_VOX, seed=seed + 50)
    return (left.cuda(), right.cuda()), gt.cuda(), synthetic.disparity_gt(d, H, W).cuda()


def _model(name, prec='bf16', **kw):
    kw.setdefault('TEST__FSCORE_THRESH', [0.05, 0.1])
    kw.setdefault('TEST__DIST_MAX', 0.5)
    cfg = small_cfg(NETWORK__PRECISION=prec, **kw)
    return cfg, M.build_model(name, cfg, seed=3).cuda().pack()


def _want_hist(cfg, name, out, gt):
    e = M.dist_edges(cfg)
    if name == 'Stereo2Point':
        return O.point_hist(out[2].cpu(), gt.cpu(), e)
    return O.surface_hist(out[2].cpu().numpy(), gt.cpu().numpy(), list(cfg.TEST.VOXEL_THRESH), e)


@pytest.mark.parametrize('name', ['Stereo2Point', 'Stereo2Voxel'])
@pytest.mark.parametrize('prec', ['bf16', 'fp32'])
def test_model_outputs_unchanged_and_hist_exact(name, prec):
    cfg, model = _model(name, prec)
    args, gt, dgt = _inputs(cfg, 2, 0, name)
    kw = dict(surface=True) if name == 'Stereo2Voxel' else {}
    with torch.no_grad():
        n0 = lib.launches()
        base = [t.clone() for t in model(*args, gt, **kw)]
        n1 = lib.launches()
        full = [t.clone() for t in model(*args, gt, fscore_curves=True, **kw)]
        n2 = lib.launches()
        eg = [t.clone() for t in model.graphed(*args, gt, fscore_curves=True, **kw)]
        eg2 = [t.clone() for t in model.graphed(*args, gt, fscore_curves=True, **kw)]   # a replay does not accumulate
    assert n2 - n1 == n1 - n0
    assert len(full) == len(base) + 1
    for a, b in zip(base, full):
        assert torch.equal(a, b)
    for a, b, c in zip(full, eg, eg2):
        assert torch.equal(a, b) and torch.equal(a, c)
    K = len(M.dist_edges(cfg))
    h = full[-1]
    assert h.dtype == torch.int64
    assert h.shape == ((2, 2, K + 1) if name == 'Stereo2Point' else (2, len(cfg.TEST.VOXEL_THRESH), 2, K + 1))
    want = _want_hist(cfg, name, full, gt)
    assert np.array_equal(h.cpu().numpy(), want)
    assert want[..., :K].sum() > 0


@pytest.mark.parametrize('name', ['Stereo2Point', 'Stereo2Voxel'])
def test_model_flag_last_with_every_option(name):
    cfg, model = _model(name)
    args, gt, dgt = _inputs(cfg, 2, 1, name)
    kw = dict(disp_gt=dgt, lr_check=True, uncertainty=True)
    if name == 'Stereo2Voxel':
        kw.update(surface=True, mesh=True, curves=True)
    with torch.no_grad():
        base = [t.clone() for t in model(*args, gt, **kw)]
        full = [t.clone() for t in model(*args, gt, fscore_curves=True, **kw)]
        g = [t.clone() for t in model.graphed(*args, gt, fscore_curves=True, **kw)]
    names = type(model).output_names(gt=True, fscore_curves=True, **{k: True for k in kw})
    assert names[-1] == 'dist_hist' and len(full) == len(names) == len(base) + 1
    for a, b in zip(base, full):
        assert torch.equal(a, b)
    for a, b in zip(full, g):
        assert torch.equal(a, b)
    assert np.array_equal(full[-1].cpu().numpy(), _want_hist(cfg, name, full, gt))


def test_model_micro_batch():
    cfg, model = _model('Stereo2Voxel', CONST__MICRO_BATCH=2)
    args, gt, _ = _inputs(cfg, 5, 2, 'Stereo2Voxel')
    with torch.no_grad():
        out = [t.clone() for t in model(*args, gt, surface=True, fscore_curves=True)]
        cfg.CONST.MICRO_BATCH = 0
        whole = [t.clone() for t in model(*args, gt, surface=True, fscore_curves=True)]
    assert out[-1].shape[0] == 5
    for a, b in zip(out, whole):
        assert torch.equal(a, b)
    assert np.array_equal(out[-1].cpu().numpy(), _want_hist(cfg, 'Stereo2Voxel', out, gt))


def test_model_errors_before_any_launch():
    pcfg, pm = _model('Stereo2Point')
    vcfg, vm = _model('Stereo2Voxel')
    pargs, pgt, _ = _inputs(pcfg, 2, 0, 'Stereo2Point')
    vargs, vgt, _ = _inputs(vcfg, 2, 0, 'Stereo2Voxel')
    n0 = lib.launches()
    for fn in (pm, pm.graphed):
        with pytest.raises(ValueError, match='needs the GT'):
            fn(*pargs, fscore_curves=True)
    for fn in (vm, vm.graphed):
        with pytest.raises(ValueError, match='needs the GT'):
            fn(*vargs, fscore_curves=True)
        with pytest.raises(ValueError, match='surface=True'):
            fn(*vargs, vgt, fscore_curves=True)
    for bins, dmax in ((0, 0.5), (True, 0.5), (1025, 0.5), (8, NAN), (8, -1.0), (1024, 1e-42)):
        for cfg, m, args, gt, kw in ((pcfg, pm, pargs, pgt, {}), (vcfg, vm, vargs, vgt, dict(surface=True))):
            cfg.TEST.DIST_BINS, cfg.TEST.DIST_MAX = bins, dmax
            for fn in (m, m.graphed):
                with pytest.raises(ValueError, match='TEST.DIST_'):
                    fn(*args, gt, fscore_curves=True, **kw)
    assert lib.launches() == n0


# ---- the driver and the runner ------------------------------------------------------------------------------------------
def _runner(monkeypatch, capsys, argv):
    import runner
    monkeypatch.setattr(sys, 'argv', ['runner.py', '--test'] + argv)
    runner.main()
    return json.loads(capsys.readouterr().out.strip().splitlines()[-1])


def test_runner_point_curves(monkeypatch, capsys):
    n, bs = 3, 2
    common = ['--model', 'Stereo2Point', '--batch-size', str(bs), '--n-samples', str(n)]
    old = _runner(monkeypatch, capsys, common)
    new = _runner(monkeypatch, capsys, common + ['--fscore-curves'])
    assert set(new) == set(old) | {'point_curves'}
    for k in old:
        assert json.dumps(new[k]) == json.dumps(old[k]), k
    cfg = default_cfg.clone()
    model = M.build_model('Stereo2Point', cfg, seed=cfg.CONST.SEED).cuda().pack()
    e = M.dist_edges(cfg)
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    blk = 0
    for s in range(0, n, bs):                                          # the runner's batches, the model's own points
        ids = range(s, min(s + bs, n))
        pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in ids]
        gt = torch.cat([synthetic.point_clouds(1, 1, cfg.CONST.N_GT_POINTS, seed=200000 + i)[1] for i in ids])
        with torch.no_grad():
            pts = model(torch.cat([p[0] for p in pairs]).cuda(), torch.cat([p[1] for p in pairs]).cuda())[2]
        blk = blk + O.point_curves_block(O.point_hist(pts.cpu(), gt, e), cfg.CONST.N_POINTS, cfg.CONST.N_GT_POINTS)
    want = T.point_curves_summary(torch.from_numpy(blk), e, n)
    assert new['point_curves'] == json.loads(json.dumps(want))
    assert len(new['point_curves']['fscore']) == cfg.TEST.DIST_BINS
    assert new['point_curves']['fscore'][9] == new['points']['fscore'][0]     # e_10 = the default F-Score@1 % threshold


def test_runner_surface_curves(monkeypatch, capsys):
    n, bs = 2, 2
    common = ['--batch-size', str(bs), '--n-samples', str(n), '--surface']
    with pytest.raises(SystemExit):
        _runner(monkeypatch, capsys, common[:-1] + ['--fscore-curves'])
    old = _runner(monkeypatch, capsys, common)
    new = _runner(monkeypatch, capsys, common + ['--fscore-curves'])
    assert set(new) == set(old) | {'surface_curves'}
    for k in old:
        assert json.dumps(new[k]) == json.dumps(old[k]), k
    cfg = default_cfg.clone()
    model = M.build_model('Stereo2Voxel', cfg, seed=cfg.CONST.SEED).cuda().pack()
    e = M.dist_edges(cfg)
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in range(n)]
    gt = torch.cat([synthetic.gt_volume(1, cfg.CONST.N_VOX, seed=100000 + i) for i in range(n)])
    with torch.no_grad():
        vox = model(torch.cat([p[0] for p in pairs]).cuda(), torch.cat([p[1] for p in pairs]).cuda())[2]
    h = O.surface_hist(vox.cpu().numpy(), gt.numpy(), list(cfg.TEST.VOXEL_THRESH), e)
    want = T.surface_curves_summary(torch.from_numpy(O.surface_curves_block(h)), cfg.TEST.VOXEL_THRESH, e, n)
    assert new['surface_curves'] == json.loads(json.dumps(want))
    for t, entry in enumerate(new['surface_curves']['by_thresh']):
        assert entry['fscore'][9] == new['surface']['by_thresh'][t]['fscore'][0]
