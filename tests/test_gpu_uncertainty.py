"""Disparity uncertainty inside the forward: every soft-argmin kernel's standard deviation against the fp64 reference on costs
the test knows (tests/unc_oracle.py), disp_q unchanged by it, the upsampled map bit-identical to s3d_upsample_disp and the
confidence-filtered counters equal to the reference statement on the very tensors the kernel returns, and the model outputs
unchanged by uncertainty=True."""
import math

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from config import cfg as default_cfg
from oracle import models as O
from stereo_3d_reconstruction_b200 import lib, models as M, ops
from stereo_3d_reconstruction_b200.core import test as T
from stereo_3d_reconstruction_b200.layers import PackedConv
from stereo_3d_reconstruction_b200.utils import synthetic
from tests.common import small_cfg
from tests.disp_oracle import disp_error_counts
from tests.lr_oracle import lr_consistency
from tests.test_gpu_disp_eval import _gt_like, _views
from tests.unc_oracle import soft_argmin_moments, unc_counts

pytestmark = pytest.mark.gpu
NAN, INF = float('nan'), float('inf')
UT, TH = [0.5, 1.0, 2.0, 4.0], [1.0, 3.0]


def _bar(sd, ref):
    """|sigma_q - sigma_ref| <= 1e-4 (1 + sigma_ref) everywhere (include/s3d.h)."""
    sd = sd.detach().cpu().double().numpy()
    assert np.isfinite(sd).all() and (sd >= 0).all()
    err = np.abs(sd - ref) / (1 + ref)
    assert err.max() <= 1e-4, err.max()


def _close(sd, ref, atol):
    sd = sd.detach().cpu().double().numpy()
    assert np.isfinite(sd).all() and (sd >= 0).all()
    assert np.abs(sd - ref).max() <= atol, np.abs(sd - ref).max()


# ---- soft-argmin kernels ------------------------------------------------------------------------------------------------
def _taps_of(cost):
    """Line-planar taps [N,D,h,32,w] whose gather is exactly `cost` [N,D,h,w]: the centre tap (kz = ky = kx = 1) holds it."""
    N, D, h, w = cost.shape
    taps = torch.zeros(N, D, h, 32, w)
    taps[:, :, :, 13, :] = cost
    return taps.cuda()


@pytest.mark.parametrize('N,D,h,w', [(2, 8, 16, 16), (3, 32, 7, 13), (1, 128, 4, 33)])
def test_tap_gather_std_matches_fp64_oracle(N, D, h, w):
    g = torch.Generator().manual_seed(21)
    taps = (torch.randn(N, D, h, 32, w, generator=g) * 0.7).cuda()
    disp0 = ops.tap_gather_soft_argmin(taps, -1.0)
    sd = torch.full((N, h, w), 7.0, device='cuda')
    disp, cost = ops.tap_gather_soft_argmin(taps, -1.0, want_cost=True, std_out=sd)
    assert torch.equal(disp, disp0)
    mu, ref = soft_argmin_moments(cost)
    _bar(sd, ref)
    assert np.abs(disp.cpu().double().numpy() - mu).max() < 1e-3 * D


def _hand_costs():
    """[5, 128, 1, 4]: uniform; two equal minima at 3 and 100; the sharp peak at 120 (sigma 0.055); the same peak at 5;
    a peak on the last plane."""
    D = 128
    c = torch.full((5, D, 1, 4), 60.0)
    c[0] = 0.0
    c[1, 3] = c[1, 100] = 0.0
    c[2, 120], c[2, 119], c[2, 121] = 0.0, 6.5, 6.5
    c[3, 5], c[3, 4], c[3, 6] = 0.0, 6.5, 6.5
    c[4, D - 1], c[4, D - 2] = 0.0, 3.0
    return c


def _check_hand(sd):
    D = 128
    p = math.exp(-6.5) / (1 + 2 * math.exp(-6.5))
    want = [math.sqrt((D * D - 1) / 12), 48.5, math.sqrt(2 * p), math.sqrt(2 * p)]
    for i, wv in enumerate(want):
        assert abs(sd[i].max().item() - wv) <= 1e-4 * (1 + wv) and abs(sd[i].min().item() - wv) <= 1e-4 * (1 + wv), (i, sd[i])
    assert 0.05 < want[2] < 0.06


def test_tap_gather_std_hand_built():
    c = _hand_costs()
    sd = torch.empty(5, 1, 4, device='cuda')
    disp = ops.tap_gather_soft_argmin(_taps_of(c), -1.0, std_out=sd)
    _check_hand(sd.cpu())
    _bar(sd, soft_argmin_moments(c)[1])
    assert abs(disp[2].mean().item() - 120.0) < 1e-3
    # non-finite costs: NaN sigma where the mean is not finite
    c2 = torch.zeros(2, 8, 1, 1)
    c2[0, 3] = NAN
    c2[1, 2] = -INF
    sd2 = torch.empty(2, 1, 1, device='cuda')
    d2 = ops.tap_gather_soft_argmin(_taps_of(c2), -1.0, std_out=sd2)
    assert not torch.isfinite(d2).any() and torch.isnan(sd2).all()


def test_cls_fused_std_hand_built():
    """cls_fused.cu with the centre tap = channel 0: cost = x[..., 0] exactly (bf16 values)."""
    c = _hand_costs()                                               # 0, 3, 6.5, 60: exact in bf16
    N, D, h, w = c.shape
    x = torch.zeros(N, D, h, w, 16, dtype=torch.bfloat16)
    x[..., 0] = c.to(torch.bfloat16)
    w_taps = torch.zeros(32, 16, dtype=torch.bfloat16)
    w_taps[13, 0] = 1.0
    sd = torch.empty(N, h, w, device='cuda')
    disp = ops.cls_soft_argmin(x.cuda(), w_taps.cuda(), -1.0, std_out=sd)
    assert torch.equal(disp, ops.cls_soft_argmin(x.cuda(), w_taps.cuda(), -1.0))
    _check_hand(sd.cpu())


@pytest.mark.parametrize('N,C,D,h,w', [(2, 16, 8, 9, 13), (1, 64, 32, 16, 16), (3, 64, 5, 40, 21), (2, 32, 9, 64, 64)])
def test_cls_fused_std_matches_conv3d_costs(N, C, D, h, w):
    g = torch.Generator().manual_seed(13)
    x = torch.randn(N, C, D, h, w, generator=g).to(torch.bfloat16)
    wt = (torch.randn(1, C, 3, 3, 3, generator=g) * 0.3).to(torch.bfloat16)
    _, ref = soft_argmin_moments(F.conv3d(x.float(), wt.float(), padding=1).squeeze(1))
    w_taps = torch.zeros(32, C, dtype=torch.bfloat16)
    w_taps[:27] = wt[0].reshape(C, 27).t()
    xc = x.permute(0, 2, 3, 4, 1).contiguous().cuda()
    sd = torch.empty(N, h, w, device='cuda')
    disp = ops.cls_soft_argmin(xc, w_taps.cuda(), -1.0, std_out=sd)
    assert torch.equal(disp, ops.cls_soft_argmin(xc, w_taps.cuda(), -1.0))
    _close(sd, ref, 2e-4 * D)                                       # the disparity's tolerance class (test_gpu_ops.py)


@pytest.mark.parametrize('N,D,h,w', [(2, 8, 32, 16), (1, 5, 40, 21), (3, 32, 64, 64), (20, 4, 64, 64)])
def test_conv_cls_chain_std(N, D, h, w):
    g = torch.Generator().manual_seed(17)
    conv = nn.Conv3d(64, 64, 3, 1, 1, bias=True)
    with torch.no_grad():
        conv.weight.copy_((torch.randn(conv.weight.shape, generator=g) * 0.04).to(torch.bfloat16).float())
        conv.bias.copy_(torch.randn(64, generator=g) * 0.1)
    pc = PackedConv.from_conv(conv, None, lib.ACT_RELU, lib.DTYPE_BF16, 'cuda')
    x = torch.randn(N, 64, D, h, w, generator=g).to(torch.bfloat16)
    wt = (torch.randn(1, 64, 3, 3, 3, generator=g) * 0.3).to(torch.bfloat16)
    w_taps = torch.zeros(32, 64, dtype=torch.bfloat16)
    w_taps[:27] = wt[0].reshape(64, 27).t()
    xc = x.permute(0, 2, 3, 4, 1).contiguous().cuda()
    sd = torch.empty(N, h, w, device='cuda')
    got = ops.conv_cls_soft_argmin(pc, xc, w_taps.cuda(), -1.0, std_out=sd)
    assert torch.equal(got, ops.conv_cls_soft_argmin(pc, xc, w_taps.cuda(), -1.0))
    # the one-pass classifier on the stored bf16 Y: same costs up to the fp32 order of the 27 taps
    y = pc(xc, engine='igemm')
    sd2 = torch.empty(N, h, w, device='cuda')
    ops.cls_soft_argmin(y, w_taps.cuda(), -1.0, std_out=sd2)
    _close(sd, sd2.cpu().double().numpy(), 2e-4 * D)
    with torch.no_grad():
        yr = F.relu(conv(x.float())).to(torch.bfloat16).float()
        _, ref = soft_argmin_moments(F.conv3d(yr, wt.float(), padding=1).squeeze(1))
    _close(sd, ref, 5e-3 * D)


@pytest.mark.parametrize('dtype', [torch.float32, torch.bfloat16])
@pytest.mark.parametrize('B,C,h,w,D', [(2, 32, 8, 64, 32), (1, 16, 5, 21, 8), (1, 64, 3, 35, 64), (1, 32, 2, 40, 128)])
def test_corr_simt_std_matches_fp64_oracle(dtype, B, C, h, w, D):
    """SIMT kernel (cost_out forces it): its own costs, cost-0 planes where the window leaves the image included."""
    g = torch.Generator().manual_seed(2)
    f = torch.randn(2 * B, C, h, w, generator=g).to(dtype).float()
    feat = f.permute(0, 2, 3, 1).unsqueeze(1).contiguous().to(dtype).cuda()
    disp0, _ = ops.corr_soft_argmin(feat, B, D, want_cost=True)
    sd = torch.empty(2 * B, h, w, device='cuda')
    disp, cost = ops.corr_soft_argmin(feat, B, D, want_cost=True, std_out=sd)
    assert torch.equal(disp, disp0)
    _, ref = soft_argmin_moments(cost, sign=1.0)
    _bar(sd, ref)


@pytest.mark.parametrize('B,C,h,w,D', [(2, 32, 8, 64, 32), (1, 16, 5, 21, 8), (1, 64, 3, 35, 64), (1, 32, 2, 40, 128),
                                       (3, 32, 16, 64, 32)])
def test_corr_tc_std(B, C, h, w, D):
    """Tensor-core kernel (bf16, w <= 64): against the fp64 moments of the SIMT kernel's costs on the same features (the two
    sum the channels in different orders), with the zero-cost tail in closed form."""
    g = torch.Generator().manual_seed(3)
    feat = torch.randn(2 * B, 1, h, w, C, generator=g).to(torch.bfloat16).cuda()
    sd = torch.empty(2 * B, h, w, device='cuda')
    disp = ops.corr_soft_argmin(feat, B, D, std_out=sd)
    assert torch.equal(disp, ops.corr_soft_argmin(feat, B, D))
    _, cost = ops.corr_soft_argmin(feat, B, D, want_cost=True)
    _, ref = soft_argmin_moments(cost, sign=1.0)
    _close(sd, ref, 1e-3 * (1 + ref.max()))
    lib.set_knob('no_corr_tc', 1)
    try:
        sd2 = torch.empty(2 * B, h, w, device='cuda')
        ops.corr_soft_argmin(feat, B, D, std_out=sd2)
    finally:
        lib.set_knob('no_corr_tc', 0)
    _close(sd, sd2.cpu().double().numpy(), 1e-3 * (1 + ref.max()))


# ---- upsampling ---------------------------------------------------------------------------------------------------------
def _std_up(q, sq, H, W, scale, ut=UT, gt=None, th=TH, max_gt=32.0, lr=None):
    B = q.shape[0] // 2
    us = torch.zeros(B, 2, len(ut), 3 + len(th), dtype=torch.int64, device='cuda')
    st = None if gt is None else torch.zeros(B, 2, 2 + len(th), dtype=torch.int64, device='cuda')
    mask = ls = None
    if lr is not None:
        mask = torch.full((B, 2, H, W), 7, dtype=torch.uint8, device='cuda')
        ls = torch.zeros(B, 2, 3 + len(th), dtype=torch.int64, device='cuda')
    sd = torch.full((B, 2, H, W), 7.0, device='cuda')                      # every element must be written
    out = ops.upsample_disp_eval(q, H, W, scale, gt, th, max_gt, st, lr_thresh=lr or 0.0, mask=mask, lr_stats=ls, std_q=sq,
                                 unc_thresh=ut, unc_stats=us, std_out=sd)
    return out, sd, us, st, mask, ls


@pytest.mark.parametrize('N,h,w,H,W', [
    (2, 16, 16, 64, 64),        # 16-byte path
    (4, 64, 64, 256, 256),      # the default input size
    (4, 17, 26, 70, 101),       # scalar path
    (2, 9, 25, 37, 101),
])
def test_std_group_matches_upsample_and_oracle(N, h, w, H, W):
    B = N // 2
    g = torch.Generator().manual_seed(N * 100 + W)
    base = torch.rand(B, h, 1, generator=g) * 4 + 1
    q = torch.cat([base + torch.rand(B, h, w, generator=g) * 0.6, base + torch.rand(B, h, w, generator=g) * 0.6]).cuda()
    sq = (torch.rand(N, h, w, generator=g) * 0.8).cuda()             # x4: 0 .. 3.2 px, across the thresholds
    sq[0, 0, :3] = torch.tensor([NAN, INF, 0.0])
    ref = ops.upsample_disp(q, H, W, 4.0).clone()
    ref_sd = _views(ops.upsample_disp(sq, H, W, 4.0).clone(), B)
    gt = _gt_like(_views(ref, B), 32.0, TH, seed=W).cuda()
    st_ref = torch.zeros(B, 2, 2 + len(TH), dtype=torch.int64, device='cuda')
    ops.upsample_disp_eval(q, H, W, 4.0, gt, TH, 32.0, st_ref)
    m_ref, ls_ref = lr_consistency(_views(ref, B), 1.0, gt, TH, 32.0)
    for with_gt in (False, True):
        for lr in (None, 1.0):
            out, sd, us, st, mask, ls = _std_up(q, sq, H, W, 4.0, gt=gt if with_gt else None, lr=lr)
            assert torch.equal(out, ref)
            assert torch.equal(sd.view(torch.int32), ref_sd.contiguous().view(torch.int32))     # NaN / inf too
            want = unc_counts(_views(out, B), sd, UT, gt if with_gt else None, TH, 32.0)
            assert torch.equal(us.cpu(), want), (with_gt, lr)
            if with_gt:
                assert torch.equal(st, st_ref)
                assert (want[..., 1] > 0).all() and (want[..., 1] < want[..., 0]).all()
            else:
                assert (us[..., 1:] == 0).all()
            if lr is not None:
                assert torch.equal(mask.cpu(), m_ref)
                assert torch.equal(ls.cpu(), ls_ref if with_gt else torch.cat([ls_ref[..., :1], 0 * ls_ref[..., 1:]], -1))
    n_img = H * W
    assert 0 < want[..., 0, 0].min() and want[..., 0, 0].max() < n_img and (want[..., 3, 0] > want[..., 0, 0]).all()
    # accumulate contract, fewer thresholds, none
    out, sd, us, st, _, _ = _std_up(q, sq, H, W, 4.0, gt=gt)
    ops.upsample_disp_eval(q, H, W, 4.0, gt, TH, 32.0, st, std_q=sq, unc_thresh=UT, unc_stats=us, std_out=sd)
    assert torch.equal(us.cpu(), 2 * want) and torch.equal(st, 2 * st_ref)
    _, _, u1, _, _, _ = _std_up(q, sq, H, W, 4.0, ut=[1.0], gt=gt)
    assert torch.equal(u1.cpu(), want[:, :, 1:2])
    _, sd0, u0, _, _, _ = _std_up(q, sq, H, W, 4.0, ut=[], gt=gt)
    assert u0.numel() == 0 and torch.equal(sd0.view(torch.int32), ref_sd.contiguous().view(torch.int32))


def test_std_group_bad_arguments():
    L = lib.load()
    B, h, w, H, W = 1, 8, 8, 32, 32
    q = torch.rand(2 * B, h, w, device='cuda')
    out = torch.empty(2 * B, H, W, device='cuda')
    sd = torch.empty(B, 2, H, W, device='cuda')
    us = torch.zeros(B, 2, 5, 11, dtype=torch.int64, device='cuda')
    import ctypes
    ut = (ctypes.c_float * 5)(1, 2, 3, 4, 5)
    th = (ctypes.c_float * 2)(1, 3)
    s = torch.cuda.current_stream().cuda_stream

    def call(K=2, ut_=ut, sq=q.data_ptr(), so=sd.data_ptr(), u=us.data_ptr(), B_=B):
        return L.s3d_upsample_disp_eval(q.data_ptr(), out.data_ptr(), B_, h, w, H, W, 4.0, None, th, 2, 0.0, None,
                                        None, 0.0, None, sq, so, ut_, K, u, s)
    assert call() == 0 and call(K=0, u=None) == 0 and call(K=4) == 0
    for bad in (dict(K=5), dict(K=-1), dict(sq=None), dict(so=None), dict(u=None), dict(B_=0),
                dict(ut_=(ctypes.c_float * 2)(1, NAN)), dict(ut_=(ctypes.c_float * 2)(-1, 2)), dict(ut_=(ctypes.c_float * 2)(1, INF))):
        assert call(**bad) == -1, bad
    torch.cuda.synchronize()


# ---- models -------------------------------------------------------------------------------------------------------------
CASES = [('Stereo2Voxel', 'concat'), ('Stereo2Voxel', 'corr'), ('Stereo2Point', 'concat'), ('Stereo2Point', 'corr')]


def _model(name, cv, prec, seed=3, **kw):
    # D = 8: a near-uniform distribution has sigma = 9.2 px, so the last threshold takes every pixel
    cfg = small_cfg(NETWORK__PRECISION=prec, NETWORK__COST_VOLUME=cv, TEST__UNC_THRESH=[1.0, 4.0, 8.0, 32.0], **kw)
    return cfg, M.build_model(name, cfg, seed=seed).cuda().pack()


def _inputs(cfg, name, B, seed):
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    left, right, d = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=seed)
    args = (left.cuda(), right.cuda())
    if name == 'Stereo2Voxel':
        args += (synthetic.gt_volume(B, seed=seed).cuda(),)
    return args, synthetic.disparity_gt(d, H, W).cuda()


def _check_unc(cfg, out, B, dgt):
    """The last two outputs against the oracle on the returned disparities and standard deviations."""
    sd, us = out[-2], out[-1]
    K, T_ = len(cfg.TEST.UNC_THRESH), len(cfg.TEST.DISP_THRESH)
    assert sd.shape == (B, 2, cfg.CONST.IMG_H, cfg.CONST.IMG_W) and sd.dtype == torch.float32
    assert us.shape == (B, 2, K, 3 + T_) and us.dtype == torch.int64
    assert torch.isfinite(sd).all() and (sd >= 0).all()
    want = unc_counts(_views((out[0], out[1]), B), sd, cfg.TEST.UNC_THRESH, dgt, cfg.TEST.DISP_THRESH,
                      4.0 * cfg.NETWORK.MAX_DISP)
    assert torch.equal(us.cpu(), want)
    return want


@pytest.mark.parametrize('prec', ['bf16', 'fp32', 'bf16x3'])
@pytest.mark.parametrize('name,cv', CASES)
def test_model_outputs_unchanged_and_unc_exact(name, cv, prec):
    cfg, model = _model(name, cv, prec)
    args, dgt = _inputs(cfg, name, 2, seed=0)
    with torch.no_grad():
        n0 = lib.launches()
        plain = [t.clone() for t in model(*args)]
        n1 = lib.launches()
        unc = [t.clone() for t in model(*args, uncertainty=True)]
        n2 = lib.launches()
        full = [t.clone() for t in model(*args, disp_gt=dgt, lr_check=True)]
        fullu = [t.clone() for t in model(*args, disp_gt=dgt, lr_check=True, uncertainty=True)]
        n3 = lib.launches()
    assert n2 - n1 == n1 - n0 and n3 - n2 == 2 * (n1 - n0)
    assert len(unc) == len(plain) + 2 and len(fullu) == len(full) + 2
    for a, b in zip(plain + full, unc[:-2] + fullu[:-2]):
        assert torch.equal(a, b)
    want = _check_unc(cfg, unc, 2, None)
    assert (want[..., 1:] == 0).all() and (want[..., -1, 0] == 64 * 64).all()
    want = _check_unc(cfg, fullu, 2, dgt)
    assert want[..., 1].sum() > 0
    assert torch.equal(unc[-2], fullu[-2])
    # disp_std = the 1/4-res map the soft-argmin kernel wrote, upsampled as disp is
    B = 2
    sq = model._buf('disp_std_q', (2 * B, cfg.CONST.IMG_H // 4, cfg.CONST.IMG_W // 4), torch.float32)
    up = _views(ops.upsample_disp(sq, cfg.CONST.IMG_H, cfg.CONST.IMG_W, 4.0), B)
    assert torch.equal(up, fullu[-2])


@pytest.mark.parametrize('name,cv', CASES[:3])
def test_graphed_with_uncertainty_matches_eager(name, cv):
    cfg, model = _model(name, cv, 'bf16')
    seen = []
    for seed in (0, 1):
        args, dgt = _inputs(cfg, name, 2, seed=seed)
        with torch.no_grad():
            eager = [t.clone() for t in model(*args, disp_gt=dgt, lr_check=True, uncertainty=True)]
            graphed = [t.clone() for t in model.graphed(*args, disp_gt=dgt, lr_check=True, uncertainty=True)]
        assert len(model._graphs) == 1
        for a, b in zip(eager, graphed):
            assert torch.equal(a, b)
        seen.append(eager[-1])
    assert not torch.equal(seen[0], seen[1])
    args, dgt = _inputs(cfg, name, 2, seed=0)
    with torch.no_grad():
        g = [t.clone() for t in model.graphed(*args, uncertainty=True)]
    assert len(model._graphs) == 2
    _check_unc(cfg, g, 2, None)


def test_micro_batched_unc_matches_unsplit():
    cfg, model = _model('Stereo2Voxel', 'concat', 'bf16', CONST__MICRO_BATCH=2)
    args, dgt = _inputs(cfg, 'Stereo2Voxel', 5, seed=4)
    with torch.no_grad():
        out = [t.clone() for t in model(*args, disp_gt=dgt, lr_check=True, uncertainty=True)]
    cfg.CONST.MICRO_BATCH = 0
    with torch.no_grad():
        whole = [t.clone() for t in model(*args, disp_gt=dgt, lr_check=True, uncertainty=True)]
    assert len(out) == len(whole) == 9
    for a, b in zip(out, whole):
        assert a.shape == b.shape and torch.equal(a, b)
    _check_unc(cfg, out, 5, dgt)


@pytest.mark.parametrize('knob,prec,cv', [(None, 'bf16', 'concat'), ('no_cls_chain', 'bf16', 'concat'), (None, 'fp32', 'concat'),
                                          ('no_corr_tc', 'bf16', 'corr'), (None, 'bf16', 'corr')])
def test_each_kernel_runs_in_the_default_network(knob, prec, cv):
    """Default network (256 x 256, D = 32), B = 3: the chain (conv_scatter_cls, 96 columns > 74 pairs), cls_fused
    (no_cls_chain), tap_gather (fp32), corr_tc and the SIMT corr (no_corr_tc): outputs unchanged, counters exact."""
    cfg = default_cfg.clone()
    cfg.NETWORK.PRECISION = prec
    cfg.NETWORK.COST_VOLUME = cv
    cfg.TEST.UNC_THRESH = [1.0, 4.0, 16.0, 128.0]                   # sigma <= 9.2 planes = 37 px: the last takes every pixel
    if knob:
        lib.set_knob(knob, 1)
    try:
        model = M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()
        B, H, W = 3, cfg.CONST.IMG_H, cfg.CONST.IMG_W
        left, right, d = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=11)
        dgt = synthetic.disparity_gt(d, H, W).cuda()
        with torch.no_grad():
            ev = [t.clone() for t in model(left.cuda(), right.cuda(), disp_gt=dgt)]
            out = [t.clone() for t in model(left.cuda(), right.cuda(), disp_gt=dgt, uncertainty=True)]
    finally:
        if knob:
            lib.set_knob(knob, 0)
    for a, b in zip(ev, out):
        assert torch.equal(a, b)
    want = _check_unc(cfg, out, B, dgt)
    assert (want[..., -1, 0] == H * W).all() and want[..., -1, 1].sum() > 0


def test_default_network_fp32_std_matches_oracle_cost_volume():
    """fp32: disp_std against 4 * bilinear(sigma) of the oracle's own cost volume (oracle/models.py), with the tolerance the
    fp32 disparity meets against the oracle."""
    cfg = default_cfg.clone()
    cfg.NETWORK.PRECISION = 'fp32'
    B, H, W = 1, cfg.CONST.IMG_H, cfg.CONST.IMG_W
    oracle = O.make_model('Stereo2Voxel', cfg, seed=0)
    model = M.build_model('Stereo2Voxel', cfg)
    model.load_state_dict(oracle.state_dict())
    model.cuda().pack()
    left, right, _ = synthetic.stereo_pair(B, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=5)
    D = cfg.NETWORK.MAX_DISP
    with torch.no_grad():
        out = model(left.cuda(), right.cuda(), uncertainty=True)
        dn = oracle.dispnet                                          # oracle/models.py, DispNet.forward up to its cost volume
        feats = dn.encoder(torch.cat([left, right], 0))
        fl, fr = feats[:B], feats[B:]
        vol = torch.cat([O.build_concat_volume(fl, fr, D, -1), O.build_concat_volume(fr, fl, D, +1)], 0)
        cost = dn.aggregation(vol)
        rdl = dn(left, right)[0]
    mu, sd = soft_argmin_moments(cost, axis=1)
    up = F.interpolate(4.0 * torch.from_numpy(sd).float().unsqueeze(1), size=(H, W), mode='bilinear',
                       align_corners=False).squeeze(1)
    dmax = rdl.abs().max().item()
    assert (out[0].cpu() - rdl).abs().max().item() <= 1e-4 * dmax           # test_gpu_model.py's fp32 tolerance
    for v in range(2):
        err = (out[-2][:, v].cpu() - up[v * B:(v + 1) * B]).abs().max().item()
        assert err <= 1e-4 * dmax, (v, err, dmax)


@pytest.mark.parametrize('name', ['Stereo2Voxel', 'Stereo2Point'])
def test_driver_eval_unc(name):
    cfg, model = _model(name, 'concat', 'bf16')
    n, bs = 3, 2
    run = T.test_voxel if name == 'Stereo2Voxel' else T.test_point
    kw = {'eval_points': True} if name == 'Stereo2Point' else {}
    base = run(cfg, model, n, bs, eval_disp=True, eval_lr=True, **kw).cpu()
    full = run(cfg, model, n, bs, eval_disp=True, eval_lr=True, eval_unc=True, **kw).cpu()
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    K, T_ = len(cfg.TEST.UNC_THRESH), len(cfg.TEST.DISP_THRESH)
    nu = 2 * K * (3 + T_)
    npt = 2 * (3 + len(cfg.TEST.FSCORE_THRESH)) + len(cfg.TEST.FSCORE_THRESH) if name == 'Stereo2Point' else 0
    head = base.numel() - npt
    assert torch.equal(full[:head], base[:head]) and torch.equal(full[head + nu:], base[head:])     # point block stays last
    want = torch.zeros(2, K, 3 + T_, dtype=torch.int64)
    for s in range(0, n, bs):
        ids = range(s, min(s + bs, n))
        pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in ids]
        with torch.no_grad():
            o = model(torch.cat([p[0] for p in pairs]).cuda(), torch.cat([p[1] for p in pairs]).cuda(), uncertainty=True)
        dgt = torch.cat([synthetic.disparity_gt(p[2], H, W) for p in pairs])
        want += unc_counts(_views((o[0], o[1]), len(ids)), o[-2], cfg.TEST.UNC_THRESH, dgt, cfg.TEST.DISP_THRESH,
                           4.0 * cfg.NETWORK.MAX_DISP).sum(0)
    assert torch.equal(full[head:head + nu], want.flatten())
    nd = 2 * (2 + T_)
    nl = 2 * (3 + T_)
    summ = T.unc_summary(full[head:head + nu], cfg.TEST.UNC_THRESH, cfg.TEST.DISP_THRESH, n * H * W,
                         full[head - nl - nd:head - nl])
    assert 0 < summ['all'][-1]['density'] <= 1 and 0 < summ['all'][-1]['conf_of_valid'] <= 1


@pytest.mark.parametrize('model_name', ['Stereo2Voxel', 'Stereo2Point'])
def test_runner_prints_uncertainty(model_name, tmp_path):
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, 'runner.py'), '--test', '--model', model_name, '--batch-size', '2',
                        '--uncertainty', '--lr-check'], cwd=root, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-2000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    u = res['uncertainty']
    assert u['unc_thresh'] == default_cfg.TEST.UNC_THRESH and len(u['all']) == len(u['unc_thresh'])
    assert 'lr_consistency' in res and 'disparity' in res
    assert all(0 <= x['density'] <= 1 for x in u['all'])
