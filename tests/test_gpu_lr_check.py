"""Left-right consistency check inside the forward (s3d_upsample_disp_eval with lr_mask): the disparity and the disparity
stats are bit-identical to s3d_upsample_disp / s3d_upsample_disp_eval with GT only, and the mask and integer counters equal
the reference
statement (tests/lr_oracle.py) on the very disparities the kernel returns."""
import ctypes

import pytest
import torch

from config import cfg as default_cfg
from stereo_3d_reconstruction_b200 import lib, models as M, ops
from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.utils import synthetic
from tests.common import small_cfg
from tests.disp_oracle import disp_error_counts
from tests.lr_oracle import lr_consistency
from tests.test_gpu_disp_eval import _gt_like, _views

pytestmark = pytest.mark.gpu
TH = [1.0, 3.0]
NAN, INF = float('nan'), float('inf')


def _lr(q, H, W, scale, tau, gt=None, th=TH, max_gt=32.0, out=None):
    B = q.shape[0] // 2
    mask = torch.full((B, 2, H, W), 7, dtype=torch.uint8, device='cuda')      # every byte must be written
    ls = torch.zeros(B, 2, 3 + len(th), dtype=torch.int64, device='cuda')
    st = None if gt is None else torch.zeros(B, 2, 2 + len(th), dtype=torch.int64, device='cuda')
    out = ops.upsample_disp_eval(q, H, W, scale, gt, th, max_gt, st, lr_thresh=tau, mask=mask, lr_stats=ls, out=out)
    return out, mask, ls, st


@pytest.mark.parametrize('N,h,w,H,W', [
    (2, 16, 16, 64, 64),        # B = 1, 16-byte path
    (4, 64, 64, 256, 256),      # the default input size
    (4, 17, 26, 70, 101),       # W = 101: scalar path
    (6, 13, 13, 50, 50),        # W = 50: scalar path
    (2, 9, 25, 37, 101),
])
def test_lr_group_matches_upsample_eval_and_oracle(N, h, w, H, W):
    B = N // 2
    g = torch.Generator().manual_seed(N * 1000 + W + 1)
    # both views near one smooth per-row level: about half the pixels agree within tau after the x4 scale
    base = torch.rand(B, h, 1, generator=g) * 4 + 1
    q = torch.cat([base + torch.rand(B, h, w, generator=g) * 0.6, base + torch.rand(B, h, w, generator=g) * 0.6]).cuda()
    q[0, 0, 0] = -2.0                                                  # negative disparities in range
    ref = ops.upsample_disp(q, H, W, 4.0).clone()
    max_gt = 32.0
    gt = _gt_like(_views(ref, B), max_gt, TH, seed=W).cuda()
    st_ref = torch.zeros(B, 2, 2 + len(TH), dtype=torch.int64, device='cuda')
    ops.upsample_disp_eval(q, H, W, 4.0, gt, TH, max_gt, st_ref)
    tau = 1.0
    out, mask, ls, st = _lr(q, H, W, 4.0, tau, gt)
    assert torch.equal(out, ref) and torch.equal(st, st_ref)
    want_mask, want = lr_consistency(_views(out, B), tau, gt, TH, max_gt)
    assert torch.equal(mask.cpu(), want_mask) and torch.equal(ls.cpu(), want)
    n_img = H * W
    assert 0.1 * n_img < want[..., 0].min() and want[..., 0].max() < 0.95 * n_img          # neither vacuous nor trivial
    assert (want[..., 1] > 0).all() and (want[..., 1] < want[..., 0]).all() and (want[..., 3] > 0).all()
    # accumulate contract
    ops.upsample_disp_eval(q, H, W, 4.0, gt, TH, max_gt, st, lr_thresh=tau, mask=mask, lr_stats=ls, out=out)
    assert torch.equal(ls.cpu(), 2 * want) and torch.equal(st, 2 * st_ref) and torch.equal(out, ref)
    # no GT: same mask, column 0 only, the rest of the row untouched
    out0, mask0, ls0, _ = _lr(q, H, W, 4.0, tau)
    assert torch.equal(out0, ref) and torch.equal(mask0.cpu(), want_mask)
    assert torch.equal(ls0[..., 0].cpu(), want[..., 0]) and (ls0[..., 1:] == 0).all()
    # eight thresholds, none
    th8 = [0.25 * (k + 1) for k in range(8)]
    _, _, ls8, st8 = _lr(q, H, W, 4.0, tau, gt, th8)
    assert torch.equal(ls8.cpu(), lr_consistency(_views(ref, B), tau, gt, th8, max_gt)[1])
    assert torch.equal(st8.cpu(), disp_error_counts(_views(ref, B), gt, th8, max_gt))
    _, _, l0, s0 = _lr(q, H, W, 4.0, tau, gt, [])
    assert torch.equal(l0.cpu(), want[..., :3]) and torch.equal(s0, st_ref[..., :2])
    # another tolerance moves the mask the way the oracle says
    _, m2, l2, _ = _lr(q, H, W, 4.0, 0.25, gt)
    w2 = lr_consistency(_views(ref, B), 0.25, gt, TH, max_gt)
    assert torch.equal(m2.cpu(), w2[0]) and torch.equal(l2.cpu(), w2[1]) and (w2[1][..., 0] < want[..., 0]).all()


@pytest.mark.parametrize('W', [64, 61])                                # 16-byte and scalar path
def test_lr_group_hand_built_cases(W):
    """Identity scale (H = h, W = w, scale 1): a pixel stores q itself while its right and lower neighbours are finite.
    Row y of sample 0 carries one planted case; each is checked in the returned disparity, and the kernel's mask equals the
    oracle everywhere."""
    B, H = 2, 12
    big = 1000.0
    ql = torch.full((B, H, W), big)
    qr = torch.full((B, H, W), -big)
    up = torch.nextafter(torch.tensor(4.0), torch.tensor(INF)).item()
    # (y, view of the pixel, x, d, other value, expected kept); the other value goes to x - k (view 0) / x + k (view 1)
    cases = [
        (0, 0, 10, 3.0, 4.0, 1),          # |d - d_o| == tau: kept
        (1, 0, 10, 3.0, up, 0),           # one ulp above tau
        (2, 0, 10, 2.5, 2.5, 1),          # half-integer: k = 2
        (3, 0, 10, 3.5, 3.5, 1),          # k = 4
        (4, 0, 2, 3.0, None, 0),          # xo = -1
        (5, 0, 3, 3.0, 3.0, 1),           # xo = 0
        (6, 1, W - 3, 2.0, 2.0, 1),       # xo = W - 1
        (7, 1, W - 3, 3.0, None, 0),      # xo = W
        (8, 0, 5, -2.0, -2.0, 1),         # negative d: xo = x + 2
        (9, 1, 5, -2.0, -2.0, 1),         # negative d, view 1: xo = x - 2
        (10, 0, 10, 2e9, None, 0),        # |d| >= W + 1
    ]
    for y, v, x, d, other, _ in cases:
        own, oth = (ql, qr) if v == 0 else (qr, ql)
        own[0, y, x] = d
        if other is not None:
            k = int(torch.tensor(d).round().item())                      # torch.round: half to even
            oth[0, y, x - k if v == 0 else x + k] = other
    # non-finite: own NaN / inf (sample 1, row 0; the pixel to the left and the row above pick the NaN up too), and a NaN on
    # the other side (sample 1, row 4)
    ql[1, 0, 20], ql[1, 0, 30], qr[1, 0, 40] = NAN, INF, -INF
    ql[1, 4, 10] = 1.0
    qr[1, 4, 9] = NAN
    q = torch.cat([ql, qr]).cuda()
    out, mask, ls, _ = _lr(q, H, W, 1.0, 1.0, th=[])
    assert torch.equal(out.view(torch.int32), ops.upsample_disp(q, H, W, 1.0).view(torch.int32))     # NaNs too, bit for bit
    disp = _views(out, B).cpu()
    want_mask, want = lr_consistency(disp, 1.0)
    assert torch.equal(mask.cpu(), want_mask) and torch.equal(ls.cpu(), want)
    for y, v, x, d, other, kept in cases:
        assert disp[0, v, y, x].item() == d, (y, v, x)                    # the case is in the returned disparity
        if other is not None:
            k = int(torch.tensor(d).round().item())
            assert disp[0, 1 - v, y, x - k if v == 0 else x + k].item() == other, (y, v, x)
        assert want_mask[0, v, y, x].item() == kept, (y, v, x, d)
    assert torch.isnan(disp[1, 0, 0, 20]) and disp[1, 0, 0, 30] == INF and disp[1, 1, 0, 40] == -INF
    assert torch.isnan(disp[1, 0, 0, 19]) and torch.isnan(disp[1, 0, 0, 29])       # 0 * inf in the left neighbour
    assert want_mask[1, 0, 0, 20] == 0 and want_mask[1, 0, 0, 30] == 0 and want_mask[1, 1, 0, 40] == 0
    assert disp[1, 0, 4, 10] == 1.0 and disp[1, 1, 4, 9] != disp[1, 1, 4, 9] and want_mask[1, 0, 4, 10] == 0


def test_lr_group_bad_arguments():
    L = lib.load()
    B, h, w, H, W = 1, 8, 8, 32, 32
    q = torch.rand(2 * B, h, w, device='cuda')
    out = torch.empty(2 * B, H, W, device='cuda')
    mask = torch.empty(B, 2, H, W, dtype=torch.uint8, device='cuda')
    gt = torch.zeros(B, 2, H, W, device='cuda')
    st = torch.zeros(B, 2, 10 + 1, dtype=torch.int64, device='cuda')
    ls = torch.zeros(B, 2, 11 + 1, dtype=torch.int64, device='cuda')
    th = (ctypes.c_float * 9)(*range(9))
    s = torch.cuda.current_stream().cuda_stream
    ptr = dict(q=q.data_ptr(), out=out.data_ptr(), mask=mask.data_ptr(), gt=gt.data_ptr(), st=st.data_ptr(),
               ls=ls.data_ptr())

    def call(T_=2, max_gt=32.0, th_=th, B_=B, tau=1.0, H_=H, **kw):
        p = dict(ptr, **kw)
        return L.s3d_upsample_disp_eval(p['q'], p['out'], B_, h, w, H_, W, 4.0, p['gt'], th_, T_, max_gt, p['st'],
                                        p['mask'], tau, p['ls'], None, None, None, 0, None, s)
    assert call() == 0
    assert call(gt=None, st=None) == 0
    assert call(tau=0.0) == 0 and call(tau=INF) == 0
    for bad in (dict(q=None), dict(out=None), dict(mask=None), dict(ls=None), dict(th_=None),
                dict(tau=-1.0), dict(tau=NAN), dict(T_=9), dict(T_=-1),
                dict(gt=None), dict(st=None),
                dict(B_=0), dict(B_=40000), dict(H_=0), dict(H_=1 << 26),
                dict(max_gt=0.0), dict(max_gt=NAN)):
        rc = call(**bad)
        assert rc == -1, bad
        with pytest.raises(lib.S3dError):
            lib.check(rc, 's3d_upsample_disp_eval')
    torch.cuda.synchronize()


CASES = [('Stereo2Voxel', 'concat'), ('Stereo2Voxel', 'corr'), ('Stereo2Point', 'concat'), ('Stereo2Point', 'corr')]


def _model(name, cv, prec, seed=3, **kw):
    cfg = small_cfg(NETWORK__PRECISION=prec, NETWORK__COST_VOLUME=cv, **kw)
    return cfg, M.build_model(name, cfg, seed=seed).cuda().pack()


def _inputs(cfg, name, B, seed):
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=seed)
    args = (left.cuda(), right.cuda())
    if name == 'Stereo2Voxel':
        args += (synthetic.gt_volume(B, seed=seed).cuda(),)
    return args, synthetic.disparity_gt(d, H, W).cuda()


def _check_lr(cfg, out, B, dgt):
    """The last two outputs against the oracle on the returned disparities (out[0], out[1])."""
    mask, ls = out[-2], out[-1]
    T_ = len(cfg.TEST.DISP_THRESH)
    assert mask.shape == (B, 2, cfg.CONST.IMG_H, cfg.CONST.IMG_W) and mask.dtype == torch.uint8
    assert ls.shape == (B, 2, 3 + T_) and ls.dtype == torch.int64
    want_mask, want = lr_consistency(_views((out[0], out[1]), B), cfg.TEST.LR_THRESH, dgt, cfg.TEST.DISP_THRESH,
                                     4.0 * cfg.NETWORK.MAX_DISP)
    assert torch.equal(mask.cpu(), want_mask) and torch.equal(ls.cpu(), want)
    return want


@pytest.mark.parametrize('prec', ['bf16', 'fp32', 'bf16x3'])
@pytest.mark.parametrize('name,cv', CASES)
def test_model_outputs_unchanged_and_lr_exact(name, cv, prec):
    cfg, model = _model(name, cv, prec)
    args, dgt = _inputs(cfg, name, 2, seed=0)
    with torch.no_grad():
        n0 = lib.launches()
        plain = [t.clone() for t in model(*args)]
        n1 = lib.launches()
        lr = [t.clone() for t in model(*args, lr_check=True)]
        n2 = lib.launches()
        ev = [t.clone() for t in model(*args, disp_gt=dgt)]
        evlr = [t.clone() for t in model(*args, disp_gt=dgt, lr_check=True)]
        n3 = lib.launches()
    assert n2 - n1 == n1 - n0 and n3 - n2 == 2 * (n1 - n0)          # the LR kernel replaces the plain / eval upsample
    assert len(lr) == len(plain) + 2 and len(evlr) == len(ev) + 2
    for a, b in zip(plain, lr):
        assert torch.equal(a, b)
    for a, b in zip(ev, evlr):                                       # disparities, head outputs, IoU counts, disp_stats
        assert torch.equal(a, b)
    want = _check_lr(cfg, lr, 2, None)
    assert want[..., 0].sum() > 0 and (want[..., 1:] == 0).all()
    want = _check_lr(cfg, evlr, 2, dgt)
    assert want[..., 1].sum() > 0


@pytest.mark.parametrize('name,cv', CASES[:3])
def test_graphed_with_lr_check_matches_eager(name, cv):
    cfg, model = _model(name, cv, 'bf16')
    seen = []
    for seed in (0, 1):
        args, dgt = _inputs(cfg, name, 2, seed=seed)
        with torch.no_grad():
            eager = [t.clone() for t in model(*args, disp_gt=dgt, lr_check=True)]
            graphed = [t.clone() for t in model.graphed(*args, disp_gt=dgt, lr_check=True)]
        assert len(model._graphs) == 1
        for a, b in zip(eager, graphed):
            assert torch.equal(a, b)
        seen.append(eager[-1])
    assert not torch.equal(seen[0], seen[1])
    args, dgt = _inputs(cfg, name, 2, seed=0)
    with torch.no_grad():                                            # separate graphs without the check
        assert len(model.graphed(*args, disp_gt=dgt)) == len(eager) - 2
        g = [t.clone() for t in model.graphed(*args, lr_check=True)]
    assert len(model._graphs) == 3
    _check_lr(cfg, g, 2, None)


def test_micro_batched_lr_matches_unsplit():
    cfg, model = _model('Stereo2Voxel', 'concat', 'bf16', CONST__MICRO_BATCH=2)
    args, dgt = _inputs(cfg, 'Stereo2Voxel', 5, seed=4)
    with torch.no_grad():
        out = [t.clone() for t in model(*args, disp_gt=dgt, lr_check=True)]
    cfg.CONST.MICRO_BATCH = 0
    with torch.no_grad():
        whole = [t.clone() for t in model(*args, disp_gt=dgt, lr_check=True)]
    assert len(out) == len(whole) == 7
    for a, b in zip(out, whole):
        assert a.shape == b.shape and torch.equal(a, b)
    _check_lr(cfg, out, 5, dgt)


def test_lr_thresh_validation():
    cfg, model = _model('Stereo2Voxel', 'concat', 'bf16')
    args, _ = _inputs(cfg, 'Stereo2Voxel', 1, seed=0)
    n0 = lib.launches()
    for bad in (-0.5, NAN, INF):
        cfg.TEST.LR_THRESH = bad
        with pytest.raises(ValueError):
            model(*args, lr_check=True)
        with pytest.raises(ValueError):
            model.graphed(*args, lr_check=True)
    assert lib.launches() == n0                                     # rejected before anything is launched


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_driver_eval_lr(name):
    cfg, model = _model(name, 'concat', 'bf16')
    n, bs = 3, 2
    run = T.test_voxel if name == 'Stereo2Voxel' else T.test_point
    base = run(cfg, model, n, bs, eval_disp=True).cpu()
    full = run(cfg, model, n, bs, eval_disp=True, eval_lr=True).cpu()
    assert torch.equal(full[:base.numel()], base)
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    want = torch.zeros(2, 3 + len(cfg.TEST.DISP_THRESH), dtype=torch.int64)
    for s in range(0, n, bs):                                        # the same batches, the model's own disparities
        ids = range(s, min(s + bs, n))
        pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in ids]
        with torch.no_grad():
            dl, dr = model(torch.cat([p[0] for p in pairs]).cuda(), torch.cat([p[1] for p in pairs]).cuda())[:2]
        dgt = torch.cat([synthetic.disparity_gt(p[2], H, W) for p in pairs])
        want += lr_consistency(_views((dl, dr), len(ids)), cfg.TEST.LR_THRESH, dgt, cfg.TEST.DISP_THRESH,
                               4.0 * cfg.NETWORK.MAX_DISP)[1].sum(0)
    assert torch.equal(full[base.numel():], want.flatten())
    nd = 2 * (2 + len(cfg.TEST.DISP_THRESH))
    summ = T.lr_summary(full[base.numel():], cfg.TEST.DISP_THRESH, n * H * W, base[-nd:])
    assert 0 < summ['all']['density'] <= 1 and 0 < summ['all']['kept_of_valid'] <= 1


def test_default_network_matches_oracle():
    """Default network (256 x 256, D = 32), B = 2: the mask and counters of the forward against the oracle on its own
    disparities, with and without GT, and the disparities unchanged by the check."""
    cfg = default_cfg.clone()
    model = M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()
    B, H, W = 2, cfg.CONST.IMG_H, cfg.CONST.IMG_W
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=11)
    dgt = synthetic.disparity_gt(d, H, W).cuda()
    with torch.no_grad():
        ev = [t.clone() for t in model(left.cuda(), right.cuda(), disp_gt=dgt)]
        out = [t.clone() for t in model(left.cuda(), right.cuda(), disp_gt=dgt, lr_check=True)]
        out0 = [t.clone() for t in model(left.cuda(), right.cuda(), lr_check=True)]
    for a, b in zip(ev, out):
        assert torch.equal(a, b)
    want = _check_lr(cfg, out, B, dgt)
    assert want[..., 1].sum() > 0
    _check_lr(cfg, out0, B, None)
