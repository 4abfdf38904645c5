"""Disparity evaluation inside the forward (s3d_upsample_disp_eval): the disparity is bit-identical to s3d_upsample_disp and
the integer counters equal the reference statement (tests/disp_oracle.py) on the very disparities the kernel returns."""
import ctypes

import pytest
import torch

from config import cfg as default_cfg
from oracle import models as O
from stereo_3d_reconstruction_b200 import lib, models as M, ops
from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.utils import synthetic
from tests.common import small_cfg
from tests.disp_oracle import disp_error_counts

pytestmark = pytest.mark.gpu
TH = [1.0, 3.0]


def _views(disp, B):
    """[2B,H,W] (left-referenced first) or (disp_left, disp_right) [B,1,H,W] -> [B,2,H,W], the GT orientation."""
    if isinstance(disp, tuple):
        return torch.cat(disp, 1)
    return torch.stack([disp[:B], disp[B:]], 1)


def _gt_like(ref, max_gt, th, seed):
    """GT near the disparity `ref` [B,2,H,W] with ~20 % invalid entries of every kind and some at exactly ref -/+ t."""
    g = torch.Generator().manual_seed(seed)
    r = ref.cpu()
    gt = r + (torch.rand(r.shape, generator=g) - 0.5) * 8
    sel = torch.rand(r.shape, generator=g)
    for k, v in enumerate((float('nan'), float('inf'), -float('inf'), -0.5, max_gt, max_gt + 3)):
        gt[(sel >= 0.8 + k * 0.03) & (sel < 0.8 + (k + 1) * 0.03)] = v
    for k, t in enumerate(th):
        gt[(sel >= 0.1 * k) & (sel < 0.1 * k + 0.03)] = (r - t)[(sel >= 0.1 * k) & (sel < 0.1 * k + 0.03)]
        gt[(sel >= 0.1 * k + 0.03) & (sel < 0.1 * k + 0.06)] = (r + t)[(sel >= 0.1 * k + 0.03) & (sel < 0.1 * k + 0.06)]
    gt[0, 0, 0, 0] = float('nan')
    return gt.contiguous()


@pytest.mark.parametrize('N,h,w,H,W', [
    (2, 16, 16, 64, 64),        # B = 1, 16-byte path
    (4, 64, 64, 256, 256),      # the default input size
    (4, 17, 26, 70, 101),       # W = 101: scalar path
    (6, 13, 13, 50, 50),        # W = 50: scalar path
    (2, 9, 25, 37, 101),
])
def test_kernel_matches_upsample_and_oracle(N, h, w, H, W):
    B = N // 2
    g = torch.Generator().manual_seed(N * 1000 + W)
    q = (torch.rand(N, h, w, generator=g) * 8).cuda()
    ref = ops.upsample_disp(q, H, W, 4.0).clone()
    max_gt = 32.0
    gt = _gt_like(_views(ref, B), max_gt, TH, seed=W).cuda()
    stats = torch.zeros(B, 2, 2 + len(TH), dtype=torch.int64, device='cuda')
    out = ops.upsample_disp_eval(q, H, W, 4.0, gt, TH, max_gt, stats)
    assert torch.equal(out, ref)
    want = disp_error_counts(_views(out, B), gt, TH, max_gt)
    assert torch.equal(stats.cpu(), want)
    n_img = H * W
    assert 0.6 * n_img < want[..., 0].min() and want[..., 0].max() < 0.9 * n_img       # invalid entries were excluded
    assert (want[..., 2] > want[..., 3]).all() and (want[..., 3] > 0).all()
    ops.upsample_disp_eval(q, H, W, 4.0, gt, TH, max_gt, stats, out=out)              # accumulate contract
    assert torch.equal(stats.cpu(), 2 * want) and torch.equal(out, ref)
    # eight thresholds, none
    th8 = [0.25 * (k + 1) for k in range(8)]
    s8 = torch.zeros(B, 2, 10, dtype=torch.int64, device='cuda')
    ops.upsample_disp_eval(q, H, W, 4.0, gt, th8, max_gt, s8)
    assert torch.equal(s8.cpu(), disp_error_counts(_views(ref, B), gt, th8, max_gt))
    s0 = torch.zeros(B, 2, 2, dtype=torch.int64, device='cuda')
    ops.upsample_disp_eval(q, H, W, 4.0, gt, [], max_gt, s0)
    assert torch.equal(s0.cpu(), want[..., :2])


def test_gt_group_bad_arguments():
    L = lib.load()
    B, h, w, H, W = 1, 8, 8, 32, 32
    q = torch.rand(2 * B, h, w, device='cuda')
    out = torch.empty(2 * B, H, W, device='cuda')
    gt = torch.zeros(B, 2, H, W, device='cuda')
    st = torch.zeros(B, 2, 10 + 1, dtype=torch.int64, device='cuda')
    th = (ctypes.c_float * 9)(*range(9))
    s = torch.cuda.current_stream().cuda_stream
    ptr = dict(q=q.data_ptr(), out=out.data_ptr(), gt=gt.data_ptr(), st=st.data_ptr())

    def call(T_=2, max_gt=32.0, th_=th, B_=B, **kw):
        p = dict(ptr, **kw)
        return L.s3d_upsample_disp_eval(p['q'], p['out'], B_, h, w, H, W, 4.0, p['gt'], th_, T_, max_gt, p['st'],
                                        None, 0.0, None, None, None, None, 0, None, s)
    assert call() == 0
    for bad in (dict(q=None), dict(out=None), dict(gt=None), dict(st=None), dict(th_=None), dict(T_=9), dict(T_=-1),
                dict(max_gt=0.0), dict(max_gt=-1.0), dict(max_gt=float('nan')), dict(B_=0),
                dict(gt=None, st=None)):                                     # no group on: the plain call is s3d_upsample_disp
        rc = call(**bad)
        assert rc == -1, bad
        with pytest.raises(lib.S3dError):
            lib.check(rc, 's3d_upsample_disp_eval')
    torch.cuda.synchronize()


CASES = [('Stereo2Voxel', 'concat'), ('Stereo2Voxel', 'corr'), ('Stereo2Point', 'concat')]


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


@pytest.mark.parametrize('prec', ['bf16', 'fp32', 'bf16x3'])
@pytest.mark.parametrize('name,cv', CASES)
def test_model_outputs_unchanged_and_stats_exact(name, cv, prec):
    cfg, model = _model(name, cv, prec)
    args, dgt = _inputs(cfg, name, 2, seed=0)
    with torch.no_grad():
        n0 = lib.launches()
        plain = [t.clone() for t in model(*args)]
        n1 = lib.launches()
        ev = [t.clone() for t in model(*args, disp_gt=dgt)]
        n2 = lib.launches()
    assert n2 - n1 == n1 - n0                                  # the eval kernel replaces the plain upsample
    assert len(ev) == len(plain) + 1
    for a, b in zip(plain, ev):
        assert torch.equal(a, b)
    stats = ev[-1]
    assert stats.shape == (2, 2, 2 + len(cfg.TEST.DISP_THRESH)) and stats.dtype == torch.int64
    want = disp_error_counts(_views((ev[0], ev[1]), 2), dgt, cfg.TEST.DISP_THRESH, 4.0 * cfg.NETWORK.MAX_DISP)
    assert torch.equal(stats.cpu(), want)
    assert (want[..., 0] > 0).all()


@pytest.mark.parametrize('name,cv', CASES)
def test_graphed_with_disp_gt_matches_eager(name, cv):
    cfg, model = _model(name, cv, 'bf16')
    seen = []
    for seed in (0, 1):
        args, dgt = _inputs(cfg, name, 2, seed=seed)
        with torch.no_grad():
            eager = [t.clone() for t in model(*args, disp_gt=dgt)]
            graphed = [t.clone() for t in model.graphed(*args, disp_gt=dgt)]
        assert len(model._graphs) == 1
        for a, b in zip(eager, graphed):
            assert torch.equal(a, b)
        seen.append(eager[-1])
    assert not torch.equal(seen[0], seen[1])
    args, _ = _inputs(cfg, name, 2, seed=0)
    with torch.no_grad():                                      # a separate graph without the evaluation
        assert len(model.graphed(*args)) == len(eager) - 1
    assert len(model._graphs) == 2


def test_micro_batched_stats():
    cfg, model = _model('Stereo2Voxel', 'concat', 'bf16', CONST__MICRO_BATCH=2)
    args, dgt = _inputs(cfg, 'Stereo2Voxel', 5, seed=4)
    with torch.no_grad():
        out = model(*args, disp_gt=dgt)
    stats = out[-1]
    assert stats.shape == (5, 2, 2 + len(cfg.TEST.DISP_THRESH))
    want = disp_error_counts(_views((out[0], out[1]), 5), dgt, cfg.TEST.DISP_THRESH, 4.0 * cfg.NETWORK.MAX_DISP)
    assert torch.equal(stats.cpu(), want)


def test_disp_gt_validation():
    cfg, model = _model('Stereo2Voxel', 'concat', 'bf16')
    args, dgt = _inputs(cfg, 'Stereo2Voxel', 2, seed=0)
    for bad in (dgt[:1], dgt[:, :1], dgt.double(), dgt.cpu(), dgt[..., :-1]):
        with pytest.raises(ValueError):
            model(*args, disp_gt=bad)


def test_driver_eval_disp():
    cfg, model = _model('Stereo2Voxel', 'concat', 'bf16')
    n, bs = 3, 2
    base = T.test_voxel(cfg, model, n, bs, eval_disp=False).cpu()
    full = T.test_voxel(cfg, model, n, bs, eval_disp=True).cpu()
    assert torch.equal(full[:base.numel()], base)
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    want = torch.zeros(2, 2 + len(cfg.TEST.DISP_THRESH), dtype=torch.int64)
    for s in range(0, n, bs):                                  # the same batches, the model's own disparities
        ids = range(s, min(s + bs, n))
        pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in ids]
        with torch.no_grad():
            dl, dr = model(torch.cat([p[0] for p in pairs]).cuda(), torch.cat([p[1] for p in pairs]).cuda())[:2]
        dgt = torch.cat([synthetic.disparity_gt(p[2], H, W) for p in pairs])
        want += disp_error_counts(_views((dl, dr), len(ids)), dgt, cfg.TEST.DISP_THRESH, 4.0 * cfg.NETWORK.MAX_DISP).sum(0)
    assert torch.equal(full[base.numel():], want.flatten())
    summ = T.disp_summary(full[base.numel():], cfg.TEST.DISP_THRESH)
    assert summ['all']['n_valid'] > 0 and summ['all']['epe'] > 0


def test_default_network_epe_matches_oracle():
    """Default network, B = 2, 'bf16x3': the EPE from the kernel's counters against the EPE of the CPU oracle's disparities
    under the same validity rule.  |EPE - EPE_oracle| <= mean |d - d_oracle| <= the disparity tolerance of
    tests/test_gpu_baseline_configs.py for 'bf16x3' (1e-3 of the oracle's max disparity), plus 2^-17 px of fixed-point
    rounding per pixel."""
    cfg = default_cfg.clone()
    cfg.NETWORK.PRECISION = 'bf16x3'
    oracle = O.make_model('Stereo2Voxel', cfg, seed=0)
    model = M.build_model('Stereo2Voxel', cfg)
    model.load_state_dict(oracle.state_dict())
    model.cuda().pack()
    B, H, W = 2, cfg.CONST.IMG_H, cfg.CONST.IMG_W
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=11)
    dgt = synthetic.disparity_gt(d, H, W)
    with torch.no_grad():
        rdl, rdr, _ = oracle(left, right)
        out = model(left.cuda(), right.cuda(), disp_gt=dgt.cuda())
    max_gt = 4.0 * cfg.NETWORK.MAX_DISP
    s = out[-1].cpu().sum((0, 1))
    epe = s[1].item() / 65536.0 / s[0].item()
    ref = torch.cat([rdl, rdr], 1)
    valid = torch.isfinite(dgt) & (dgt >= 0) & (dgt < max_gt)
    assert s[0].item() == valid.sum().item()
    epe_ref = (ref - dgt).abs()[valid].double().mean().item()
    dmax = ref.abs().max().item()
    assert abs(epe - epe_ref) <= 1e-3 * dmax + 2.0 ** -17, (epe, epe_ref, dmax)
