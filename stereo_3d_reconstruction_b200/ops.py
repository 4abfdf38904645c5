# -*- coding: utf-8 -*-
"""Python wrappers over the non-conv C-ABI entry points (include/s3d.h).  Every wrapper validates
device / dtype / contiguity, allocates outputs with torch, passes raw pointers and the current
CUDA stream, and raises on a non-zero return code.  None of them computes anything in Python."""
import ctypes
import math

import torch

from . import lib as _lib


def _code(t):
    if t.dtype == torch.bfloat16:
        return _lib.DTYPE_BF16
    if t.dtype == torch.float32:
        return _lib.DTYPE_F32
    raise TypeError('unsupported dtype %s' % t.dtype)


def _code_like(t, split):
    """dtype code of an activation tensor; split=True: bf16 pairs [hi(C) | lo(C)] (include/s3d.h, S3D_DTYPE_BF16X2)."""
    if split:
        assert t.dtype == torch.bfloat16 and t.shape[-1] % 2 == 0
        return _lib.DTYPE_BF16X2
    return _code(t)


def _chk(*ts):
    for t in ts:
        if t is None:
            continue
        if not t.is_cuda:
            raise _lib.S3dError('s3d ops need CUDA tensors (there is no CPU fallback)')
        if not t.is_contiguous():
            raise ValueError('tensor must be contiguous')


def _stream():
    return torch.cuda.current_stream().cuda_stream


def pack_image(img, disp=None, disp_scale=1.0, cpad=16, dtype=torch.bfloat16, out=None):
    """img fp32 NCHW [B,3,H,W], or uint8 HWC [B,H,W,3] (decoded PNG; scaled by 1/255), (+ disp fp32 [B,H,W])
    -> channels-last [B,1,H,W,cpad]."""
    _chk(img, disp, out)
    if img.dtype == torch.uint8:
        B, H, W, C = img.shape
        assert C == 3
        if out is None:
            out = torch.empty((B, 1, H, W, cpad), dtype=dtype, device=img.device)
        rc = _lib.load().s3d_pack_image_u8(img.data_ptr(), disp.data_ptr() if disp is not None else None,
                                           float(disp_scale), 1.0 / 255.0, out.data_ptr(), B, H, W, cpad, _code(out),
                                           _stream())
        _lib.check(rc, 's3d_pack_image_u8')
        _lib.count_launch()
        return out
    B, C, H, W = img.shape
    assert C == 3 and img.dtype == torch.float32
    if out is None:
        out = torch.empty((B, 1, H, W, cpad), dtype=dtype, device=img.device)
    rc = _lib.load().s3d_pack_image(img.data_ptr(), disp.data_ptr() if disp is not None else None, float(disp_scale),
                                    out.data_ptr(), B, H, W, cpad, _code(out), _stream())
    _lib.check(rc, 's3d_pack_image')
    _lib.count_launch()
    return out


def cost_volume_concat(feat, B, D, C=None, out=None, split=False):
    """feat [2B,1,h,w,C] -> vol [2B,D,h,w,2C].  split: feat [.., hi(C) | lo(C)] -> vol [.., hi(2C) | lo(2C)]."""
    _chk(feat, out)
    n2, one, h, w, Cf = feat.shape
    C = Cf if C is None else C
    assert n2 == 2 * B and one == 1 and C == Cf
    if out is None:
        out = torch.empty((2 * B, D, h, w, 2 * C), dtype=feat.dtype, device=feat.device)
    assert out.shape == (2 * B, D, h, w, 2 * C) and out.dtype == feat.dtype
    rc = _lib.load().s3d_cost_volume_concat(feat.data_ptr(), out.data_ptr(), B, h, w, C // 2 if split else C, D,
                                            _code_like(feat, split), _stream())
    _lib.check(rc, 's3d_cost_volume_concat')
    _lib.count_launch()
    return out


def soft_argmin(cost, sign=-1.0, out=None):
    """cost fp32 [N,D,h,w] -> disp fp32 [N,h,w] = sum_d d * softmax_d(sign*cost)."""
    _chk(cost, out)
    assert cost.dtype == torch.float32
    N, D, h, w = cost.shape
    if out is None:
        out = torch.empty((N, h, w), dtype=torch.float32, device=cost.device)
    rc = _lib.load().s3d_soft_argmin(cost.data_ptr(), out.data_ptr(), N, D, h, w, float(sign), _stream())
    _lib.check(rc, 's3d_soft_argmin')
    _lib.count_launch()
    return out


def _std_buf(std_out, like):
    """std_out (the soft-argmin calls' disp_std_q) must be an fp32 tensor shaped like the disparity `like`."""
    _chk(std_out)
    if std_out.dtype != torch.float32 or std_out.shape != like.shape:
        raise ValueError('std_out must be float32 %s, got %s %s' % (tuple(like.shape), std_out.dtype, tuple(std_out.shape)))
    return std_out


def tap_gather_soft_argmin(taps, sign=-1.0, out=None, want_cost=False, std_out=None):
    """taps fp32, line-planar [N,D,h,S>=27,w] (per-tap projections) -> disp fp32 [N,h,w]; see include/s3d.h.
    std_out: fp32 [N,h,w] that receives the standard deviation of each pixel's distribution (disp_std_q)."""
    _chk(taps, out)
    assert taps.dtype == torch.float32 and taps.dim() == 5
    N, D, h, S, w = taps.shape
    if out is None:
        out = torch.empty((N, h, w), dtype=torch.float32, device=taps.device)
    cost = torch.empty((N, D, h, w), dtype=torch.float32, device=taps.device) if want_cost else None
    std = None if std_out is None else _std_buf(std_out, out).data_ptr()
    rc = _lib.load().s3d_tap_gather_soft_argmin(taps.data_ptr(), out.data_ptr(), std, cost.data_ptr() if want_cost else None,
                                                N, D, h, w, S, float(sign), _stream())
    _lib.check(rc, 's3d_tap_gather_soft_argmin')
    _lib.count_launch()
    return (out, cost) if want_cost else out


def split_tf32(x, hi=None, lo=None):
    """fp32 x -> (hi, lo): hi representable in TF32 (low 13 mantissa bits cleared), lo = x - hi (include/s3d.h)."""
    _chk(x, hi, lo)
    assert x.dtype == torch.float32 and x.is_contiguous() and x.numel() % 4 == 0
    hi = torch.empty_like(x) if hi is None else hi
    lo = torch.empty_like(x) if lo is None else lo
    rc = _lib.load().s3d_split_tf32(x.data_ptr(), hi.data_ptr(), lo.data_ptr(), x.numel(), _stream())
    _lib.check(rc, 's3d_split_tf32')
    _lib.count_launch()
    return hi, lo


def split_bf16(x, out=None):
    """fp32 [..., C] -> bf16 pairs [..., hi(C) | lo(C)] (include/s3d.h, S3D_DTYPE_BF16X2)."""
    _chk(x, out)
    assert x.dtype == torch.float32 and x.is_contiguous()
    C = x.shape[-1]
    if out is None:
        out = torch.empty(x.shape[:-1] + (2 * C,), dtype=torch.bfloat16, device=x.device)
    rc = _lib.load().s3d_split_bf16(x.data_ptr(), out.data_ptr(), x.numel() // C, C, _stream())
    _lib.check(rc, 's3d_split_bf16')
    _lib.count_launch()
    return out


def unsplit_bf16(x, out=None):
    """bf16 pairs [..., hi(C) | lo(C)] -> fp32 [..., C] = hi + lo."""
    _chk(x, out)
    assert x.dtype == torch.bfloat16 and x.is_contiguous() and x.shape[-1] % 2 == 0
    C = x.shape[-1] // 2
    if out is None:
        out = torch.empty(x.shape[:-1] + (C,), dtype=torch.float32, device=x.device)
    rc = _lib.load().s3d_unsplit_bf16(x.data_ptr(), out.data_ptr(), x.numel() // (2 * C), C, _stream())
    _lib.check(rc, 's3d_unsplit_bf16')
    _lib.count_launch()
    return out


def depth_to_space(x, cpad=16, proj_w=None, proj_act=0, out=None, split=False):
    """x [N,d,h,w,64] (channel = parity class * 8 + c, from PackedConv.from_deconv_k4s2p1_blocked) -> [N,2d,2h,2w,cpad];
    optional projection of the 8 features into channel 8 (include/s3d.h, s3d_depth_to_space)."""
    _chk(x, proj_w, out)
    m = 2 if split else 1                                       # split: [.., hi(64) | lo(64)] -> [.., hi(cpad) | lo(cpad)]
    assert x.dim() == 5 and x.shape[-1] == 64 * m and x.is_contiguous()
    N, d, h, w, _ = x.shape
    if out is None:
        out = torch.empty((N, 2 * d, 2 * h, 2 * w, cpad * m), dtype=x.dtype, device=x.device)
    assert out.dtype == x.dtype and out.is_contiguous() and out.shape == (N, 2 * d, 2 * h, 2 * w, cpad * m)
    if proj_w is not None:
        assert proj_w.dtype == torch.float32 and proj_w.numel() >= 8
    rc = _lib.load().s3d_depth_to_space(x.data_ptr(), out.data_ptr(), proj_w.data_ptr() if proj_w is not None else None,
                                        int(proj_act), N, d, h, w, cpad, _code_like(x, split), _stream())
    _lib.check(rc, 's3d_depth_to_space')
    _lib.count_launch()
    return out


def conv_first(img, pc, disp=None, disp_scale=1.0, out=None):
    """First encoder layer straight from the raw image: img fp32 NCHW [B,3,H,W] or uint8 HWC [B,H,W,3] (+ disp fp32 [B,H,W]
    as a 4th channel) through PackedConv `pc` (3x3, stride 2, pad 1) -> channels-last [B,1,oH,oW,cout_pad]."""
    _chk(img, disp, out)
    u8 = img.dtype == torch.uint8
    if u8:
        B, H, W, C = img.shape
    else:
        B, C, H, W = img.shape
        assert img.dtype == torch.float32
    assert C == 3 and img.is_contiguous()
    assert pc.ksize == (1, 3, 3) and pc.stride == (1, 2, 2) and pc.pad == (0, 1, 1) and pc.n_classes == 1
    cin = 4 if disp is not None else 3
    assert pc.cin == cin, (pc.cin, cin)
    oH, oW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
    dt = pc.weight.dtype
    co = pc.cout_pad * (2 if pc.dtype_code == _lib.DTYPE_BF16X2 else 1)      # split layer: [.., hi | lo]
    if out is None:
        out = torch.empty((B, 1, oH, oW, co), dtype=dt, device=img.device)
    assert out.dtype == dt and out.is_contiguous() and out.shape[-1] == co
    rc = _lib.load().s3d_conv_first(img.data_ptr(), 1 if u8 else 0, disp.data_ptr() if disp is not None else None,
                                    float(disp_scale), pc.weight.data_ptr(), pc.bias.data_ptr(), out.data_ptr(), B, H, W, cin,
                                    pc.cin_pad, pc.cout_pad, pc.dtype_code, pc.act, pc.act_param, _stream())
    _lib.check(rc, 's3d_conv_first')
    _lib.count_launch()
    return out


def conv_concat_volume(pc, featp, B, D, pad, out=None, ref_once=False):
    """Concat cost volume + the 3x3x3 conv `pc` (PackedConv over 2C channels) in one kernel, the volume never written.
    featp: [2B,1,h,pitch,C] feature maps stored with `pad` >= D-1 ZERO pixels on both sides of every row (real pixels in
    columns pad .. pitch-pad-1), left images first.  -> [2B,D,h,w,cout_pad].  include/s3d.h, s3d_conv_concat_volume.
    ref_once: the reference-once form (s3d_conv_concat_volume_ro: half the tensor-core work, not bit-identical)."""
    import ctypes
    from .layers import is_split
    _chk(featp, out)
    split = is_split(pc.dtype_code)              # 'bf16x3': featp / out rows are [hi(C) | lo(C)] bf16 pairs, reference-once form only
    cm = 2 if split else 1
    n2, one, h, pitch, C = featp.shape
    C //= cm
    assert n2 == 2 * B and one == 1 and featp.is_contiguous() and pc.cin_pad == 2 * C and pad >= D - 1
    assert not split or ref_once, 'split (BF16X2) operands: reference-once form only'
    w = pitch - 2 * pad
    assert w > 0
    Co = cm * pc.cout_pad
    if out is None:
        out = torch.empty((2 * B, D, h, w, Co), dtype=featp.dtype, device=featp.device)
    assert out.is_contiguous() and out.shape == (2 * B, D, h, w, Co)
    p = pc.params(2 * B, D, h, w, (D * h * w * Co, h * w * Co, w * Co, Co), _code_like(out, split), pc.cout_pad)
    if ref_once:
        rc = _lib.load().s3d_conv_concat_volume_ro(ctypes.byref(p), featp.data_ptr(), pitch, pad, pc.refonce_weights(C).data_ptr(),
                                                   pc.bias.data_ptr(), out.data_ptr(), _stream())
        _lib.check(rc, 's3d_conv_concat_volume_ro')
    else:
        rc = _lib.load().s3d_conv_concat_volume(ctypes.byref(p), featp.data_ptr(), pitch, pad, pc.bias.data_ptr(), out.data_ptr(),
                                                _stream())
        _lib.check(rc, 's3d_conv_concat_volume')
    _lib.count_launch()
    return out


def conv_concat_volume_sheared(pc, featp, B, D, pad, out=None, bufs=None):
    """Concat cost volume + the 3x3x3 layer `pc` in SHEARED form (bf16, Cout 64, ReLU): four 2-D map convolutions on the
    tensor cores (1/14 of the layer's MMAs) + one streaming pass that writes the volume (include/s3d.h,
    s3d_concat_gonce_assemble; layers.py, PackedConv.gonce_convs).  featp as for conv_concat_volume.  bufs: optional dict of
    persistent fp32 workspaces {'maps_l', 'maps_r': [B,1,h,w+4,384], 'edge_l', 'edge_r': [B,1,h,D,256]}."""
    from .layers import is_split
    _chk(featp, out)
    split = is_split(pc.dtype_code)              # 'bf16x3': featp rows and the output are bf16 pairs [hi | lo], three MMAs per product
    cm = 2 if split else 1
    n2, one, h, pitch, C = featp.shape
    C //= cm
    assert n2 == 2 * B and one == 1 and featp.is_contiguous() and featp.dtype == torch.bfloat16
    assert pc.cin_pad == 2 * C and pc.cout_pad == 64 and pc.act == _lib.ACT_RELU and pad >= D - 1 and D >= 2
    w = pitch - 2 * pad
    g = pc.gonce_convs(C, pad, w, D)
    bufs = {} if bufs is None else bufs
    res = {}
    use_mc = C == 32 and not _lib.KNOBS['no_map_conv']       # the halo-once map engine (csrc/map_conv.cu): 32 feature channels
    for name, key, sl in (('left', 'maps_l', slice(0, B)), ('right', 'maps_r', slice(B, 2 * B)),
                          ('edge_left', 'edge_l', slice(0, B)), ('edge_right', 'edge_r', slice(B, 2 * B))):
        conv = g[name]
        off, ntx, ow = g[name + '_geom']
        o = bufs.get(key)
        if o is None:
            o = torch.empty((B, 1, h, ow, conv.cout_pad), dtype=torch.float32, device=featp.device)
        assert o.shape == (B, 1, h, ow, conv.cout_pad) and o.dtype == torch.float32 and o.is_contiguous()
        if use_mc:
            x = featp[sl]
            rc = _lib.load().s3d_map_conv(x.data_ptr(), conv.weight.data_ptr(), o.data_ptr(), B, h, pitch, ow, off, ntx,
                                          conv.cout_pad, pc.dtype_code, _stream())
            _lib.check(rc, 's3d_map_conv')
            _lib.count_launch()
            res[key] = o
        else:
            res[key] = conv(featp[sl], out=o)
    Co = cm * 64
    if out is None:
        out = torch.empty((2 * B, D, h, w, Co), dtype=torch.bfloat16, device=featp.device)
    assert out.is_contiguous() and out.shape == (2 * B, D, h, w, Co) and out.dtype == torch.bfloat16
    rc = _lib.load().s3d_concat_gonce_assemble(res['maps_l'].data_ptr(), res['maps_r'].data_ptr(), res['edge_l'].data_ptr(),
                                               res['edge_r'].data_ptr(), pc.bias.data_ptr(), out.data_ptr(), B, D, h, w, w + 4,
                                               _lib.DTYPE_BF16X2 if split else _lib.DTYPE_BF16, _stream())
    _lib.check(rc, 's3d_concat_gonce_assemble')
    _lib.count_launch()
    return out


def cls_soft_argmin(x, w_taps, sign=-1.0, out=None, std_out=None):
    """x bf16 [N,D,h,w,C] (aggregated volume), w_taps bf16 [32,C] (27 classifier taps) -> disp fp32 [N,h,w]: the Cout=1
    3x3x3 classifier and the soft-argmin in one pass (include/s3d.h, s3d_cls_soft_argmin).  std_out: as for
    tap_gather_soft_argmin."""
    _chk(x, w_taps, out)
    assert x.dtype == torch.bfloat16 and w_taps.dtype == torch.bfloat16 and x.dim() == 5 and x.is_contiguous()
    N, D, h, w, C = x.shape
    assert w_taps.numel() == 32 * C and w_taps.is_contiguous()
    if out is None:
        out = torch.empty((N, h, w), dtype=torch.float32, device=x.device)
    std = None if std_out is None else _std_buf(std_out, out).data_ptr()
    rc = _lib.load().s3d_cls_soft_argmin(x.data_ptr(), w_taps.data_ptr(), out.data_ptr(), std, N, D, h, w, C, float(sign),
                                         _stream())
    _lib.check(rc, 's3d_cls_soft_argmin')
    _lib.count_launch()
    return out


def conv_cls_workspace_bytes(N, D, h, w):
    return int(_lib.load().s3d_conv_cls_workspace_bytes(N, D, h, w))


def conv_cls_soft_argmin(pc, x, w_taps, sign=-1.0, out=None, workspace=None, std_out=None):
    """The last aggregation layer `pc` (PackedConv, bf16 3x3x3 64 -> 64 + ReLU) over x [N,D,h,w,64], the Cout = 1 classifier
    (w_taps bf16 [32,64]) and the soft-argmin, the layer's output volume never written (include/s3d.h,
    s3d_conv_cls_soft_argmin; csrc/conv_scatter_cls.cu).  workspace: >= conv_cls_workspace_bytes(N, D, h, w) bytes.
    std_out: as for tap_gather_soft_argmin.  -> disp fp32 [N,h,w]."""
    import ctypes
    _chk(x, w_taps, out, workspace)
    assert x.dtype == torch.bfloat16 and w_taps.dtype == torch.bfloat16 and x.dim() == 5 and x.is_contiguous()
    N, D, h, w, C = x.shape
    assert C == 64 and pc.cin_pad == 64 and pc.cout_pad == 64 and w_taps.numel() == 32 * 64 and w_taps.is_contiguous()
    need = conv_cls_workspace_bytes(N, D, h, w)
    if workspace is None:
        workspace = torch.empty(need, dtype=torch.uint8, device=x.device)
    assert workspace.is_contiguous() and workspace.numel() * workspace.element_size() >= need
    if out is None:
        out = torch.empty((N, h, w), dtype=torch.float32, device=x.device)
    p = pc.params(N, D, h, w, (D * h * w * 64, h * w * 64, w * 64, 64), _lib.DTYPE_BF16, 64)
    std = None if std_out is None else _std_buf(std_out, out).data_ptr()
    rc = _lib.load().s3d_conv_cls_soft_argmin(ctypes.byref(p), x.data_ptr(), pc.bias.data_ptr(), w_taps.data_ptr(),
                                              workspace.data_ptr(), out.data_ptr(), std, float(sign), _stream())
    _lib.check(rc, 's3d_conv_cls_soft_argmin')
    _lib.count_launch(2)
    return out


def corr_soft_argmin(feat, B, D, out=None, want_cost=False, c_real=None, std_out=None):
    """feat [2B,1,h,w,C] -> disp fp32 [2B,h,w] (fused correlation + soft-argmax).  c_real: number of REAL feature
    channels when C is a padded pitch (the correlation is a mean over the real channels; padded ones are zero).
    std_out: as for tap_gather_soft_argmin."""
    _chk(feat, out)
    n2, one, h, w, C = feat.shape
    assert n2 == 2 * B and one == 1
    if out is None:
        out = torch.empty((2 * B, h, w), dtype=torch.float32, device=feat.device)
    cost = torch.empty((2 * B, D, h, w), dtype=torch.float32, device=feat.device) if want_cost else None
    std = None if std_out is None else _std_buf(std_out, out).data_ptr()
    rc = _lib.load().s3d_corr_soft_argmin(feat.data_ptr(), out.data_ptr(), std, cost.data_ptr() if want_cost else None,
                                          B, h, w, C, int(c_real or 0), D, _code(feat), _stream())
    _lib.check(rc, 's3d_corr_soft_argmin')
    _lib.count_launch()
    return (out, cost) if want_cost else out


def upsample_disp(disp_q, H, W, scale, out=None):
    _chk(disp_q, out)
    assert disp_q.dtype == torch.float32
    N, h, w = disp_q.shape
    if out is None:
        out = torch.empty((N, H, W), dtype=torch.float32, device=disp_q.device)
    rc = _lib.load().s3d_upsample_disp(disp_q.data_ptr(), out.data_ptr(), N, h, w, H, W, float(scale), _stream())
    _lib.check(rc, 's3d_upsample_disp')
    _lib.count_launch()
    return out


def upsample_disp_eval(disp_q, H, W, scale, gt=None, thresholds=(), max_gt=0.0, stats=None, *, lr_thresh=0.0, mask=None,
                       lr_stats=None, std_q=None, unc_thresh=(), unc_stats=None, std_out=None, out=None):
    """upsample_disp + per-pixel evaluation in one launch (include/s3d.h, s3d_upsample_disp_eval).  disp_q fp32 [2B,h,w] (left-
    referenced first) -> disp fp32 [2B,H,W], bit-identical to upsample_disp.  At least one of three groups is on; every stats
    tensor is ADDED to, and T = len(thresholds) sets the row length of each (without gt only column 0 of lr_stats / unc_stats):
      gt fp32 [B,2,H,W] (NaN = no GT), stats int64 [B,2,2+T]: per image [n_valid, sum of |disp - gt| in 2^-16 px,
        count(|disp - gt| > t) per threshold];
      mask uint8 [B,2,H,W] <- 1 where the left-right consistency check keeps the pixel (tolerance lr_thresh px), lr_stats int64
        [B,2,3+T] += [n_kept, n_valid_kept, sum of |disp - gt| in 2^-16 px over valid & kept, count(|disp - gt| > t) over
        valid & kept];
      std_q fp32 [2B,h,w] (from a soft-argmin wrapper's std_out) -> std_out fp32 [B,2,H,W] (view 0 = left-referenced, allocated
        by the caller), unc_stats int64 [B,2,K,3+T] (K = len(unc_thresh) <= 4) += per view and threshold k, over the pixels with
        disp_std <= unc_thresh[k]: [n_conf, n_valid_conf, sum of |disp - gt| in 2^-16 px over valid & confident,
        count(|disp - gt| > t) over valid & confident]."""
    _chk(disp_q, gt, stats, mask, lr_stats, std_q, unc_stats, std_out, out)
    assert disp_q.dtype == torch.float32
    N, h, w = disp_q.shape
    B, T, K = N // 2, len(thresholds), len(unc_thresh)
    assert N == 2 * B
    assert (gt is None) == (stats is None) and (mask is None) == (lr_stats is None) and (std_q is None) == (std_out is None)
    if gt is not None:
        assert gt.dtype == torch.float32 and stats.dtype == torch.int64
        assert tuple(gt.shape) == (B, 2, H, W) and tuple(stats.shape) == (B, 2, 2 + T)
    if mask is not None:
        assert mask.dtype == torch.uint8 and lr_stats.dtype == torch.int64
        assert tuple(mask.shape) == (B, 2, H, W) and tuple(lr_stats.shape) == (B, 2, 3 + T)
    if std_q is not None:
        assert std_q.dtype == torch.float32 and std_q.shape == disp_q.shape
        assert unc_stats.dtype == torch.int64 and tuple(unc_stats.shape) == (B, 2, K, 3 + T)
        assert std_out.dtype == torch.float32 and tuple(std_out.shape) == (B, 2, H, W)
    if out is None:
        out = torch.empty((N, H, W), dtype=torch.float32, device=disp_q.device)
    th = (ctypes.c_float * max(T, 1))(*[float(t) for t in thresholds])
    ut = (ctypes.c_float * max(K, 1))(*[float(t) for t in unc_thresh])
    ptr = lambda t: None if t is None else t.data_ptr()
    rc = _lib.load().s3d_upsample_disp_eval(disp_q.data_ptr(), out.data_ptr(), B, h, w, H, W, float(scale),
                                            ptr(gt), th, T, float(max_gt), ptr(stats),
                                            ptr(mask), float(lr_thresh), ptr(lr_stats),
                                            ptr(std_q), ptr(std_out), ut, K, ptr(unc_stats), _stream())
    _lib.check(rc, 's3d_upsample_disp_eval')
    _lib.count_launch()
    return out


def latent_to_vox(x, L, out=None, split=False):
    """[N,1,H,W,C] -> pooled to LxL -> [N,2,2,2,C*L*L/8] (oracle's NCHW .view order).  split: hi | lo pairs in and out."""
    _chk(x, out)
    N, one, H, W, C = x.shape
    if out is None:
        out = torch.empty((N, 2, 2, 2, C * L * L // 8), dtype=x.dtype, device=x.device)
    assert out.shape[-1] == C * L * L // 8, 'latent_to_vox writes K = C*L*L/8 channels densely'
    rc = _lib.load().s3d_latent_to_vox(x.data_ptr(), out.data_ptr(), N, H, W, C // 2 if split else C, L,
                                       _code_like(x, split), _stream())
    _lib.check(rc, 's3d_latent_to_vox')
    _lib.count_launch()
    return out


def avg_pool(x, L, out=None, split=False):
    _chk(x, out)
    N, one, H, W, C = x.shape
    if out is None:
        out = torch.empty((N, 1, L, L, C), dtype=x.dtype, device=x.device)
    rc = _lib.load().s3d_avg_pool(x.data_ptr(), out.data_ptr(), N, H, W, C // 2 if split else C, L, _code_like(x, split),
                                  _stream())
    _lib.check(rc, 's3d_avg_pool')
    _lib.count_launch()
    return out


def fuse_views(score, score_off, score_stride, vol, vol_off, vol_stride, B, V, nvox, gt=None, thresholds=None,
               iou=None, out=None, score_lo=0, vol_lo=0):
    """Context-aware fusion epilogue (+ IoU counts).  score/vol: tensors holding [V*B, nvox] planes
    at element offset *_off with element stride *_stride between voxels.  score_lo / vol_lo > 0: split (hi | lo) tensors,
    the lo part of a value sits that many elements after its hi part."""
    _chk(score, vol, gt, iou, out)
    assert score.dtype == vol.dtype
    if out is None:
        out = torch.empty((B, nvox), dtype=torch.float32, device=score.device)
    T = 0
    th = None
    if gt is not None:
        assert gt.dtype == torch.uint8 and iou is not None and iou.dtype == torch.int64
        T = len(thresholds)
        th = (ctypes.c_float * T)(*[float(t) for t in thresholds])
    esz = score.element_size()
    rc = _lib.load().s3d_fuse_views(score.data_ptr() + score_off * esz, score_stride,
                                    vol.data_ptr() + vol_off * esz, vol_stride,
                                    _lib.DTYPE_BF16X2 if score_lo else _code(score), out.data_ptr(), B, V,
                                    nvox, gt.data_ptr() if gt is not None else None, th, T,
                                    iou.data_ptr() if iou is not None else None, int(score_lo), int(vol_lo), _stream())
    _lib.check(rc, 's3d_fuse_views')
    _lib.count_launch()
    return out


def chamfer_forward(xyz1, xyz2, workspace=None):
    """xyz1 [B,N,3], xyz2 [B,M,3] fp32 -> dist1 [B,N], dist2 [B,M], idx1 [B,N], idx2 [B,M] (int32).
    Large problems take the symmetric one-pass kernel (s3d_chamfer_forward_ws: every pair evaluated once for both
    directions), which needs a device workspace of s3d_chamfer_workspace_bytes(B, N, M) bytes; it is allocated here
    unless the caller passes one (uint8 tensor)."""
    _chk(xyz1, xyz2)
    assert xyz1.dtype == torch.float32 and xyz2.dtype == torch.float32
    B, N, three = xyz1.shape
    B2, M, three2 = xyz2.shape
    if three != 3 or three2 != 3 or B != B2:
        raise ValueError('chamfer: expected [B,N,3] and [B,M,3]')
    dev = xyz1.device
    dist1 = torch.empty((B, N), dtype=torch.float32, device=dev)
    dist2 = torch.empty((B, M), dtype=torch.float32, device=dev)
    idx1 = torch.empty((B, N), dtype=torch.int32, device=dev)
    idx2 = torch.empty((B, M), dtype=torch.int32, device=dev)
    L = _lib.load()
    need = chamfer_workspace_bytes(B, N, M)
    if need and (workspace is None or workspace.numel() * workspace.element_size() < need):
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    rc = L.s3d_chamfer_forward_ws(xyz1.data_ptr(), xyz2.data_ptr(), dist1.data_ptr(), idx1.data_ptr(),
                                  dist2.data_ptr(), idx2.data_ptr(), B, N, M,
                                  workspace.data_ptr() if need else None, need, _stream())
    _lib.check(rc, 's3d_chamfer_forward_ws')
    _lib.count_launch(2)
    return dist1, dist2, idx1, idx2


def chamfer_workspace_bytes(B, N, M):
    return int(_lib.load().s3d_chamfer_workspace_bytes(B, N, M)) if min(B, N, M) > 0 else 0


def _dist_hist_args(what, edges, hist, shape, dev):
    """Validate the optional distance-histogram arguments -> (edges as fp32 Python floats, K).  edges: a sequence of 1 to
    1024 values that are finite, > 0 and strictly increasing once rounded to fp32; hist: int64 `shape` + (K + 1,) on dev."""
    if edges is None and hist is None:
        return [], 0
    if edges is None or hist is None:
        raise ValueError('%s: edges and hist go together' % what)
    try:
        e = [float(ctypes.c_float(float(x)).value) for x in edges]
    except (TypeError, ValueError):
        raise ValueError('%s: edges must be a sequence of numbers, got %r' % (what, edges)) from None
    K = len(e)
    if not 1 <= K <= 1024:
        raise ValueError('%s: 1 to 1024 edges, got %d' % (what, K))
    if not all(math.isfinite(x) and x > 0.0 for x in e) or any(b <= a for a, b in zip(e, e[1:])):
        raise ValueError('%s: edges must be finite, > 0 and strictly increasing in fp32, got %r' % (what, e))
    want = tuple(shape) + (K + 1,)
    if not isinstance(hist, torch.Tensor) or hist.dtype != torch.int64 or tuple(hist.shape) != want or hist.device != dev:
        raise ValueError('%s: hist must be int64 %s on %s' % (what, want, dev))
    _chk(hist)
    return e, K


def chamfer_eval(xyz1, xyz2, tau, stats, workspace=None, out=None, edges=None, hist=None):
    """chamfer_forward + per-sample point-cloud metrics (include/s3d.h, s3d_chamfer_eval).  xyz1 = predicted [B,N,3], xyz2 =
    GT [B,M,3], fp32.  stats int64 [B,2,3+T] (T = len(tau)) += per direction (0: xyz1 -> xyz2, 1: xyz2 -> xyz1)
    [sum q(d), sum q(sqrt d), n_out, count(sqrt d < tau_t) per t], q(x) = round-half-even(x * 2^32), over the points with
    finite d < 2^8 (the others are n_out).  out: optional (dist1 [B,N], dist2 [B,M], idx1 [B,N], idx2 [B,M]) buffers (fp32,
    fp32, int32, int32) to write into.  -> (dist1, dist2, idx1, idx2), bit-identical to chamfer_forward.
    edges (K fp32 distances, strictly increasing) with hist int64 [B,2,K+1]: hist += per direction the number of points in
    each bin = the number of edges <= sqrt(d), out-of-range points in bin K (s3d_chamfer_eval_hist; same launches)."""
    _chk(xyz1, xyz2, stats, workspace)
    if xyz1.dtype != torch.float32 or xyz2.dtype != torch.float32:
        raise ValueError('chamfer_eval: point clouds must be float32')
    B, N, three = xyz1.shape
    B2, M, three2 = xyz2.shape
    if three != 3 or three2 != 3 or B != B2:
        raise ValueError('chamfer_eval: expected [B,N,3] and [B,M,3]')
    T = len(tau)
    if stats.dtype != torch.int64 or tuple(stats.shape) != (B, 2, 3 + T):
        raise ValueError('chamfer_eval: stats must be int64 [%d, 2, %d]' % (B, 3 + T))
    dev = xyz1.device
    e, K = _dist_hist_args('chamfer_eval', edges, hist, (B, 2), dev)
    if out is None:
        out = (torch.empty((B, N), dtype=torch.float32, device=dev), torch.empty((B, M), dtype=torch.float32, device=dev),
               torch.empty((B, N), dtype=torch.int32, device=dev), torch.empty((B, M), dtype=torch.int32, device=dev))
    dist1, dist2, idx1, idx2 = out
    _chk(dist1, dist2, idx1, idx2)
    for t, shape, dt in ((dist1, (B, N), torch.float32), (dist2, (B, M), torch.float32), (idx1, (B, N), torch.int32),
                         (idx2, (B, M), torch.int32)):
        if tuple(t.shape) != shape or t.dtype != dt:
            raise ValueError('chamfer_eval: out buffer %s %s, expected %s %s' % (tuple(t.shape), t.dtype, shape, dt))
    need = chamfer_workspace_bytes(B, N, M)
    if need and (workspace is None or workspace.numel() * workspace.element_size() < need):
        workspace = torch.empty(need, dtype=torch.uint8, device=dev)
    th = (ctypes.c_float * max(T, 1))(*[float(t) for t in tau])
    ed = (ctypes.c_float * max(K, 1))(*e)
    rc = _lib.load().s3d_chamfer_eval_hist(xyz1.data_ptr(), xyz2.data_ptr(), dist1.data_ptr(), idx1.data_ptr(),
                                           dist2.data_ptr(), idx2.data_ptr(), B, N, M, th, T, stats.data_ptr(),
                                           workspace.data_ptr() if need else None, need, _stream(), ed, K,
                                           hist.data_ptr() if K else None)
    _lib.check(rc, 's3d_chamfer_eval_hist')
    _lib.count_launch(3)                       # the two search kernels + chamfer_eval_kernel
    return dist1, dist2, idx1, idx2


def voxel_kbound(tau, n):
    """F-score threshold tau (Euclidean distance in unit-cube units; the n^3 grid spans the unit cube) -> the integer bound
    k of s3d_voxel_surface_eval, in float64: a surface point counts when its squared distance s in doubled lattice units is
    < k, i.e. exactly when sqrt(s) / (2n) < tau."""
    return min(math.ceil((2 * n * float(tau)) ** 2), 3 * (2 * n) ** 2 + 1)


def voxel_surface_workspace_bytes(B, T, n):
    return int(_lib.load().s3d_voxel_surface_workspace_bytes(B, T, n))


def voxel_surface_eval(fused, gt8, voxel_thresh, fscore_thresh, stats, workspace=None, edges=None, hist=None):
    """Voxel-face surface metrics (include/s3d.h, s3d_voxel_surface_eval).  fused fp32 [B,n,n,n] or [B,n^3], gt8 uint8 of the
    same shape (nonzero = occupied), 1 <= n <= 64.  stats int64 [B,T,2,3+F] (T = len(voxel_thresh), F = len(fscore_thresh))
    += per sample, threshold and direction (0: predicted -> GT, 1: GT -> predicted) [n_pts, sum s, sum q(sqrt s),
    count(s < voxel_kbound(tau)) per tau], s the squared distance in doubled lattice units.  workspace: optional uint8
    buffer of at least voxel_surface_workspace_bytes(B, T, n) bytes.  Two kernel launches.
    edges (K fp32 distances in unit-cube units, strictly increasing) with hist int64 [B,T,2,K+1]: hist += per sample,
    threshold and direction the number of surface points in each bin = the number of voxel_kbound(e_j, n) <= s; the points
    of a direction whose other surface is empty go to bin K (s3d_voxel_surface_eval_hist; same launches)."""
    _chk(fused, gt8, stats, workspace)
    if fused.dtype != torch.float32 or gt8.dtype != torch.uint8:
        raise ValueError('voxel_surface_eval: fused must be float32 and gt8 uint8, got %s / %s' % (fused.dtype, gt8.dtype))
    if fused.shape != gt8.shape or fused.dim() not in (2, 4):
        raise ValueError('voxel_surface_eval: expected fused and gt8 of one shape [B,n,n,n] or [B,n^3], got %s / %s'
                         % (tuple(fused.shape), tuple(gt8.shape)))
    B = fused.shape[0]
    nvox = fused[0].numel()
    n = round(nvox ** (1.0 / 3.0))
    if n ** 3 != nvox or (fused.dim() == 4 and tuple(fused.shape[1:]) != (n, n, n)) or not 1 <= n <= 64:
        raise ValueError('voxel_surface_eval: a sample must be an n^3 grid with 1 <= n <= 64, got %s' % (tuple(fused.shape),))
    T, F = len(voxel_thresh), len(fscore_thresh)
    if T > 8 or F > 8:
        raise ValueError('voxel_surface_eval: at most 8 voxel and 8 F-score thresholds, got %d / %d' % (T, F))
    if stats.dtype != torch.int64 or tuple(stats.shape) != (B, T, 2, 3 + F):
        raise ValueError('voxel_surface_eval: stats must be int64 [%d, %d, 2, %d]' % (B, T, 3 + F))
    for t in (gt8, stats, workspace):
        if t is not None and t.device != fused.device:
            raise ValueError('voxel_surface_eval: every tensor must be on %s' % fused.device)
    e, K = _dist_hist_args('voxel_surface_eval', edges, hist, (B, T, 2), fused.device)
    need = voxel_surface_workspace_bytes(B, T, n)
    if workspace is None:
        workspace = torch.empty(max(need, 1), dtype=torch.uint8, device=fused.device)
    elif workspace.numel() * workspace.element_size() < need:
        raise ValueError('voxel_surface_eval: workspace of %d bytes, need %d' % (workspace.numel() * workspace.element_size(), need))
    th = (ctypes.c_float * max(T, 1))(*[float(t) for t in voxel_thresh])
    kb = (ctypes.c_int * max(F, 1))(*[voxel_kbound(t, n) for t in fscore_thresh])
    hkb = (ctypes.c_int * max(K, 1))(*[voxel_kbound(x, n) for x in e])
    rc = _lib.load().s3d_voxel_surface_eval_hist(fused.data_ptr(), gt8.data_ptr(), B, n, th, T, kb, F, stats.data_ptr(),
                                                 workspace.data_ptr(), need, _stream(), hkb, K,
                                                 hist.data_ptr() if K else None)
    _lib.check(rc, 's3d_voxel_surface_eval_hist')
    if B and T:
        _lib.count_launch(2)                   # surface_plane_kernel + surface_count_kernel
    return stats


def voxel_mesh_bounds(n):
    """-> (max_verts, max_faces) of an n^3 grid: 3 (n+1)(n+2)^2 and 5 (n+1)^3, the worst case (include/s3d.h)."""
    mv, mf = ctypes.c_int(), ctypes.c_int()
    _lib.check(_lib.load().s3d_voxel_mesh_bounds(int(n), ctypes.byref(mv), ctypes.byref(mf)), 's3d_voxel_mesh_bounds')
    return mv.value, mf.value


def voxel_mesh(vol, t, out=None):
    """Marching-cubes mesh of each sample of vol fp32 [B,n,n,n] or [B,n^3] (1 <= n <= 64) at iso-level t (finite, 0 < t <= 1)
    -> (verts fp32 [B,max_verts,3], faces int32 [B,max_faces,3], counts int32 [B,2] = (n_verts, n_faces)) with
    (max_verts, max_faces) = voxel_mesh_bounds(n); only the first counts rows of each sample are written.  Vertices are xyz in
    the unit cube the grid spans, faces 0-based per-sample ids oriented outwards (include/s3d.h, s3d_voxel_mesh).  out: the
    three output tensors.  One kernel launch."""
    _chk(vol)
    if vol.dtype != torch.float32 or vol.dim() not in (2, 4):
        raise ValueError('voxel_mesh: expected vol float32 [B,n,n,n] or [B,n^3], got %s %s' % (vol.dtype, tuple(vol.shape)))
    B = vol.shape[0]
    nvox = vol[0].numel() if B else (vol.shape[1] if vol.dim() == 2 else vol.shape[1] * vol.shape[2] * vol.shape[3])
    n = round(nvox ** (1.0 / 3.0))
    if n ** 3 != nvox or (vol.dim() == 4 and tuple(vol.shape[1:]) != (n, n, n)) or not 1 <= n <= 64:
        raise ValueError('voxel_mesh: a sample must be an n^3 grid with 1 <= n <= 64, got %s' % (tuple(vol.shape),))
    try:
        t = float(t)
    except (TypeError, ValueError):
        raise ValueError('voxel_mesh: t must be a number, got %r' % (t,)) from None
    if not (math.isfinite(t) and 0.0 < t <= 1.0):
        raise ValueError('voxel_mesh: t must be finite and in (0, 1], got %r' % t)
    if float(ctypes.c_float(t).value) <= 0.0:
        raise ValueError('voxel_mesh: t = %r rounds to 0 in fp32' % t)
    mv, mf = voxel_mesh_bounds(n)
    want = ((torch.float32, (B, mv, 3)), (torch.int32, (B, mf, 3)), (torch.int32, (B, 2)))
    if out is None:
        out = tuple(torch.empty(s, dtype=d, device=vol.device) for d, s in want)
    else:
        out = tuple(out)
        if len(out) != 3:
            raise ValueError('voxel_mesh: out must hold (verts, faces, counts)')
        _chk(*out)
        for o, (d, s) in zip(out, want):
            if o.dtype != d or tuple(o.shape) != s or o.device != vol.device:
                raise ValueError('voxel_mesh: out tensors must be %s on %s, got %s'
                                 % ([(str(d), s) for d, s in want], vol.device, [(str(o.dtype), tuple(o.shape)) for o in out]))
    verts, faces, counts = out
    rc = _lib.load().s3d_voxel_mesh(vol.data_ptr(), B, n, t, verts.data_ptr(), mv, faces.data_ptr(), mf, counts.data_ptr(),
                                    _stream())
    _lib.check(rc, 's3d_voxel_mesh')
    if B:
        _lib.count_launch(1)                   # voxel_mesh_kernel
    return verts, faces, counts


def occupancy_curves(fused, gt8, K, out=None):
    """Threshold-free occupancy evaluation (include/s3d.h, s3d_occupancy_curves).  fused fp32 and gt8 uint8 (nonzero =
    occupied) of one shape [B, ...], a sample holding 1 to 2^24 voxels; K a power of two in [2, 1024].  -> (hist int64
    [B,3,K], loss int64 [B,2]): per sample the voxels with gt = 0 / gt = 1 in each bin k = min(floor(v * K), K - 1) of the
    clamped fused value v and sum q(v) per bin, then sum q(bce) and sum q((v - g)^2), q(x) = round-half-even(x * 2^20).  out:
    the two output tensors, written (not added to).  One kernel launch."""
    _chk(fused, gt8)
    if fused.dtype != torch.float32 or gt8.dtype != torch.uint8:
        raise ValueError('occupancy_curves: fused must be float32 and gt8 uint8, got %s / %s' % (fused.dtype, gt8.dtype))
    if fused.shape != gt8.shape or fused.dim() < 2:
        raise ValueError('occupancy_curves: expected fused and gt8 of one shape [B, ...], got %s / %s'
                         % (tuple(fused.shape), tuple(gt8.shape)))
    if gt8.device != fused.device:
        raise ValueError('occupancy_curves: gt8 must be on %s, got %s' % (fused.device, gt8.device))
    B = fused.shape[0]
    nvox = math.prod(fused.shape[1:])
    if not 1 <= nvox <= 1 << 24:
        raise ValueError('occupancy_curves: a sample must hold 1 to 2^24 voxels, got %d' % nvox)
    if not (isinstance(K, int) and not isinstance(K, bool) and 2 <= K <= 1024 and K & (K - 1) == 0):
        raise ValueError('occupancy_curves: K must be a power of two in [2, 1024], got %r' % (K,))
    want = ((B, 3, K), (B, 2))
    if out is None:
        out = tuple(torch.empty(s, dtype=torch.int64, device=fused.device) for s in want)
    else:
        out = tuple(out)
        if len(out) != 2:
            raise ValueError('occupancy_curves: out must hold (hist, loss)')
        _chk(*out)
        for o, s in zip(out, want):
            if o.dtype != torch.int64 or tuple(o.shape) != s or o.device != fused.device:
                raise ValueError('occupancy_curves: out tensors must be int64 %s on %s, got %s'
                                 % (list(want), fused.device, [(str(o.dtype), tuple(o.shape), str(o.device)) for o in out]))
    hist, loss = out
    rc = _lib.load().s3d_occupancy_curves(fused.data_ptr(), gt8.data_ptr(), B, nvox, K, hist.data_ptr(), loss.data_ptr(),
                                          _stream())
    _lib.check(rc, 's3d_occupancy_curves')
    if B:
        _lib.count_launch(1)                   # occupancy_curves_kernel
    return hist, loss


def disp_cloud_workspace_bytes(B, H):
    """Bytes of the workspace of disp_cloud: the int32 row counts [B, 2H]."""
    return int(_lib.load().s3d_disp_cloud_workspace_bytes(int(B), int(H)))


def disp_cloud(disp, B, left, right, camera, min_disp, lr_mask=None, disp_std=None, max_std=None, out=None, workspace=None):
    """Coloured point clouds of the two disparity maps (include/s3d.h, s3d_disp_cloud).  disp fp32 [2B,H,W], view-major (the
    forward's buffer: left-referenced maps first); left / right the images, both fp32 NCHW [B,3,H,W] or both uint8 HWC
    [B,H,W,3]; camera fp32 [B,5] = (f, cx, cy, baseline, doffs) on the same device; min_disp finite and > 0.  Filters:
    lr_mask uint8 [B,2,H,W] (kept where 1) and disp_std fp32 [B,2,H,W] (kept where <= max_std, finite and >= 0; needed with
    disp_std, ignored without it).
    -> (xyz fp32 [B,2HW,3], rgb uint8 [B,2HW,3], counts int32 [B,2]): per sample the kept points of view 0 in raster order,
    then those of view 1, in the left camera's frame; only the first counts[b,0] + counts[b,1] rows are written.  out: the
    three output tensors; workspace: uint8 of at least disp_cloud_workspace_bytes(B, H) bytes.  Two kernel launches."""
    _chk(disp, left, right, camera, lr_mask, disp_std, workspace)
    if disp.dtype != torch.float32 or disp.dim() != 3:
        raise ValueError('disp_cloud: expected disp float32 [2B,H,W], got %s %s' % (disp.dtype, tuple(disp.shape)))
    if not isinstance(B, int) or B < 0 or disp.shape[0] != 2 * B:
        raise ValueError('disp_cloud: disp must hold 2B = %r maps, got %s' % (2 * B if isinstance(B, int) else B,
                                                                             tuple(disp.shape)))
    H, W = disp.shape[1], disp.shape[2]
    dev = disp.device
    if left.dtype == torch.uint8 and right.dtype == torch.uint8:
        u8, want = 1, (B, H, W, 3)
    elif left.dtype == torch.float32 and right.dtype == torch.float32:
        u8, want = 0, (B, 3, H, W)
    else:
        raise ValueError('disp_cloud: left / right must be both float32 or both uint8, got %s / %s' % (left.dtype, right.dtype))
    for name, t, d, s in (('left', left, None, want), ('right', right, None, want), ('camera', camera, torch.float32, (B, 5)),
                          ('lr_mask', lr_mask, torch.uint8, (B, 2, H, W)), ('disp_std', disp_std, torch.float32, (B, 2, H, W))):
        if t is None:
            continue
        if (d is not None and t.dtype != d) or tuple(t.shape) != s or t.device != dev:
            raise ValueError('disp_cloud: expected %s %s %s on %s, got %s %s on %s'
                             % (name, '' if d is None else d, s, dev, t.dtype, tuple(t.shape), t.device))
    try:
        min_disp = float(min_disp)
        max_std = 0.0 if disp_std is None else float(max_std)
    except (TypeError, ValueError):
        raise ValueError('disp_cloud: min_disp and max_std must be numbers, got %r / %r' % (min_disp, max_std)) from None
    if not (math.isfinite(min_disp) and min_disp > 0) or float(ctypes.c_float(min_disp).value) <= 0.0:
        raise ValueError('disp_cloud: min_disp must be finite and > 0, got %r' % min_disp)
    if not (math.isfinite(max_std) and max_std >= 0):
        raise ValueError('disp_cloud: max_std must be finite and >= 0, got %r' % max_std)
    shapes = ((torch.float32, (B, 2 * H * W, 3)), (torch.uint8, (B, 2 * H * W, 3)), (torch.int32, (B, 2)))
    if out is None:
        out = tuple(torch.empty(s, dtype=d, device=dev) for d, s in shapes)
    else:
        out = tuple(out)
        if len(out) != 3:
            raise ValueError('disp_cloud: out must hold (xyz, rgb, counts)')
        _chk(*out)
        for o, (d, s) in zip(out, shapes):
            if o.dtype != d or tuple(o.shape) != s or o.device != dev:
                raise ValueError('disp_cloud: out tensors must be %s on %s, got %s'
                                 % ([(str(d), s) for d, s in shapes], dev, [(str(o.dtype), tuple(o.shape)) for o in out]))
    nb = disp_cloud_workspace_bytes(B, H)
    if workspace is None:
        workspace = torch.empty(max(nb, 1), dtype=torch.uint8, device=dev)
    elif workspace.dtype != torch.uint8 or workspace.numel() < nb or workspace.device != dev:
        raise ValueError('disp_cloud: workspace must be uint8 of at least %d bytes on %s' % (nb, dev))
    xyz, rgb, counts = out
    ptr = lambda t: None if t is None else t.data_ptr()
    rc = _lib.load().s3d_disp_cloud(disp.data_ptr(), B, H, W, left.data_ptr(), right.data_ptr(), u8, ptr(lr_mask),
                                    ptr(disp_std), max_std, camera.data_ptr(), min_disp, xyz.data_ptr(), rgb.data_ptr(),
                                    counts.data_ptr(), workspace.data_ptr(), workspace.numel(), _stream())
    _lib.check(rc, 's3d_disp_cloud')
    if B:
        _lib.count_launch(2)                   # cloud_count_kernel + cloud_write_kernel
    return xyz, rgb, counts


def speckle_filter_workspace_bytes(B, H, W):
    """Bytes of the workspace of speckle_filter: int32 labels and region sizes, 8 bytes per pixel of the 2B maps."""
    return int(_lib.load().s3d_speckle_filter_workspace_bytes(int(B), int(H), int(W)))


def speckle_filter(disp, B, max_size, max_diff, lr_mask=None, disp_gt=None, thresholds=(), max_gt=None, out=None,
                   workspace=None):
    """Speckle filter of the two disparity maps (include/s3d.h, s3d_speckle_filter), OpenCV's filterSpeckles on the GPU.  disp
    fp32 [2B,H,W], view-major (the forward's buffer: left-referenced maps first).  A pixel is a candidate where d is finite
    and, with lr_mask uint8 [B,2,H,W], lr_mask is 1; two 4-neighbour candidates are adjacent when |d_p - d_q| <= max_diff
    (finite, >= 0, input px); a region (connected component) of at most max_size pixels (an int >= 0) is a speckle.
    -> (mask uint8 [B,2,H,W]: 1 where a candidate's region is larger than max_size, stats int64 [B,2,5+T] ADDED to:
    [n_kept, n_valid_kept, sum of |disp - gt| in 2^-16 px and count(|disp - gt| > t) per threshold over the kept pixels with
    valid GT (disp_gt fp32 [B,2,H,W], valid where finite and 0 <= gt < max_gt; zero without it), n_speckles,
    n_speckle_px]).  T = len(thresholds) <= 8.  out: (mask, stats), else a new mask and zeroed stats; workspace: uint8 of
    at least speckle_filter_workspace_bytes(B, H, W) bytes.  Four kernel launches."""
    _chk(disp, lr_mask, disp_gt, workspace)
    if disp.dtype != torch.float32 or disp.dim() != 3:
        raise ValueError('speckle_filter: expected disp float32 [2B,H,W], got %s %s' % (disp.dtype, tuple(disp.shape)))
    if not isinstance(B, int) or isinstance(B, bool) or B < 0 or disp.shape[0] != 2 * B:
        raise ValueError('speckle_filter: disp must hold 2B maps for an int B >= 0, got B = %r and %s' % (B, tuple(disp.shape)))
    H, W = disp.shape[1], disp.shape[2]
    dev = disp.device
    for name, t, d in (('lr_mask', lr_mask, torch.uint8), ('disp_gt', disp_gt, torch.float32)):
        if t is not None and (t.dtype != d or tuple(t.shape) != (B, 2, H, W) or t.device != dev):
            raise ValueError('speckle_filter: expected %s %s %s on %s, got %s %s on %s'
                             % (name, d, (B, 2, H, W), dev, t.dtype, tuple(t.shape), t.device))
    if not isinstance(max_size, int) or isinstance(max_size, bool) or not 0 <= max_size < 2 ** 31:
        raise ValueError('speckle_filter: max_size must be an int in [0, 2^31), got %r' % (max_size,))
    try:
        max_diff = float(max_diff)
        th = [float(t) for t in thresholds]
        max_gt = None if max_gt is None else float(max_gt)
    except (TypeError, ValueError):
        raise ValueError('speckle_filter: max_diff, thresholds and max_gt must be numbers, got %r / %r / %r'
                         % (max_diff, thresholds, max_gt)) from None
    if not (math.isfinite(max_diff) and max_diff >= 0 and math.isfinite(ctypes.c_float(max_diff).value)):
        raise ValueError('speckle_filter: max_diff must be finite and >= 0 (also in fp32), got %r' % max_diff)
    if len(th) > 8:
        raise ValueError('speckle_filter: at most 8 thresholds, got %d' % len(th))
    if disp_gt is not None and not (max_gt is not None and max_gt > 0 and ctypes.c_float(max_gt).value > 0):
        raise ValueError('speckle_filter: disp_gt needs max_gt > 0, got %r' % (max_gt,))
    T = len(th)
    shapes = ((torch.uint8, (B, 2, H, W)), (torch.int64, (B, 2, 5 + T)))
    if out is None:
        out = (torch.empty(shapes[0][1], dtype=torch.uint8, device=dev), torch.zeros(shapes[1][1], dtype=torch.int64, device=dev))
    else:
        out = tuple(out)
        if len(out) != 2:
            raise ValueError('speckle_filter: out must hold (mask, stats)')
        _chk(*out)
        for o, (d, s) in zip(out, shapes):
            if o.dtype != d or tuple(o.shape) != s or o.device != dev:
                raise ValueError('speckle_filter: out tensors must be %s on %s, got %s'
                                 % ([(str(d), s) for d, s in shapes], dev, [(str(o.dtype), tuple(o.shape)) for o in out]))
    nb = speckle_filter_workspace_bytes(B, H, W)
    if workspace is None:
        workspace = torch.empty(max(nb, 1), dtype=torch.uint8, device=dev)
    elif workspace.dtype != torch.uint8 or workspace.numel() < nb or workspace.device != dev:
        raise ValueError('speckle_filter: workspace must be uint8 of at least %d bytes on %s' % (nb, dev))
    mask, stats = out
    if B == 0:                                 # no maps (and empty tensors may hold no data pointer)
        return mask, stats
    ptr = lambda t: None if t is None else t.data_ptr()
    tc = (ctypes.c_float * max(T, 1))(*th)
    rc = _lib.load().s3d_speckle_filter(disp.data_ptr(), B, H, W, ptr(lr_mask), max_size, max_diff, ptr(disp_gt), tc, T,
                                        0.0 if max_gt is None else max_gt, mask.data_ptr(), stats.data_ptr(),
                                        workspace.data_ptr(), workspace.numel(), _stream())
    if rc == -1:                               # S3D_ERR_INVALID: an argument the checks above let through (H W >= 2^31, ...)
        raise ValueError('speckle_filter: %s' % _lib.load().s3d_last_error().decode('utf-8', 'replace'))
    _lib.check(rc, 's3d_speckle_filter')
    _lib.count_launch(4)                       # speckle_local / border / size / finish kernels
    return mask, stats


def wls_weight_lut(sigma):
    """Edge-weight table of disp_wls for the colour scale sigma (finite and > 0, 8-bit colour units): float32 numpy
    [3 * 255^2 + 1], entry s = fp32(exp(-sqrt(s) / sigma)) computed in fp64, s the summed squared colour difference of two
    neighbours (OpenCV's DisparityWLSFilter table).  ValueError on a bad sigma."""
    import numpy as np
    try:
        s = float(sigma)
    except (TypeError, ValueError):
        raise ValueError('wls_weight_lut: sigma must be a number, got %r' % (sigma,)) from None
    if isinstance(sigma, bool) or not (math.isfinite(s) and s > 0):
        raise ValueError('wls_weight_lut: sigma must be finite and > 0, got %r' % (sigma,))
    return np.exp(-np.sqrt(np.arange(3 * 255 * 255 + 1, dtype=np.float64)) / s).astype(np.float32)


def disp_wls_workspace_bytes(B, H, W):
    """Bytes of the workspace of disp_wls: U(c), the elimination's g and the two edge weights, 16 bytes per pixel of the
    2B maps."""
    return int(_lib.load().s3d_disp_wls_workspace_bytes(int(B), int(H), int(W)))


def disp_wls(disp, B, left, right, lut, lam, mask=None, disp_gt=None, thresholds=(), max_gt=None, out=None, workspace=None):
    """Confidence-weighted WLS filter of the two disparity maps (include/s3d.h, s3d_disp_wls), OpenCV's DisparityWLSFilter
    fill on the GPU.  disp fp32 [2B,H,W], view-major (the forward's buffer: left-referenced maps first); left / right the
    guides, both fp32 NCHW [B,3,H,W] or both uint8 HWC [B,H,W,3]; lut fp32 [3 * 255^2 + 1] on the device (wls_weight_lut);
    lam (lambda) finite and > 0.  A pixel is confident where d is finite and, with mask uint8 [B,2,H,W], mask is 1.
    -> (out fp32 [2B,H,W]: U(d c) / U(c), NaN where no confident pixel reaches, stats int64 [B,2,4+T] ADDED to: [n_finite,
    n_valid_finite, sum of |out - gt| in 2^-16 px and count(|out - gt| > t) per threshold over the finite pixels with valid
    GT (disp_gt fp32 [B,2,H,W], valid where finite and 0 <= gt < max_gt; zero without it), n_conf]).  T = len(thresholds)
    <= 8.  out: (out, stats), else a new map and zeroed stats (out must not be disp); workspace: uint8 of at least
    disp_wls_workspace_bytes(B, H, W) bytes.  Six kernel launches."""
    _chk(disp, left, right, lut, mask, disp_gt, workspace)
    if disp.dtype != torch.float32 or disp.dim() != 3:
        raise ValueError('disp_wls: expected disp float32 [2B,H,W], got %s %s' % (disp.dtype, tuple(disp.shape)))
    if not isinstance(B, int) or isinstance(B, bool) or B < 0 or disp.shape[0] != 2 * B:
        raise ValueError('disp_wls: disp must hold 2B maps for an int B >= 0, got B = %r and %s' % (B, tuple(disp.shape)))
    H, W = disp.shape[1], disp.shape[2]
    dev = disp.device
    if left.dtype == torch.uint8 and right.dtype == torch.uint8:
        u8, want = 1, (B, H, W, 3)
    elif left.dtype == torch.float32 and right.dtype == torch.float32:
        u8, want = 0, (B, 3, H, W)
    else:
        raise ValueError('disp_wls: left / right must be both float32 or both uint8, got %s / %s' % (left.dtype, right.dtype))
    for name, t, d, s in (('left', left, None, want), ('right', right, None, want),
                          ('lut', lut, torch.float32, (3 * 255 * 255 + 1,)), ('mask', mask, torch.uint8, (B, 2, H, W)),
                          ('disp_gt', disp_gt, torch.float32, (B, 2, H, W))):
        if t is not None and ((d is not None and t.dtype != d) or tuple(t.shape) != s or t.device != dev):
            raise ValueError('disp_wls: expected %s %s %s on %s, got %s %s on %s'
                             % (name, '' if d is None else d, s, dev, t.dtype, tuple(t.shape), t.device))
    if lut is None:
        raise ValueError('disp_wls: lut is required (wls_weight_lut)')
    try:
        lam_v = float(lam)
        th = [float(t) for t in thresholds]
        max_gt = None if max_gt is None else float(max_gt)
    except (TypeError, ValueError):
        raise ValueError('disp_wls: lam, thresholds and max_gt must be numbers, got %r / %r / %r'
                         % (lam, thresholds, max_gt)) from None
    if isinstance(lam, bool) or not (math.isfinite(lam_v) and lam_v > 0 and math.isfinite(ctypes.c_float(lam_v).value) and
                                     ctypes.c_float(lam_v).value > 0):
        raise ValueError('disp_wls: lam must be finite and > 0 (also in fp32), got %r' % (lam,))
    if len(th) > 8:
        raise ValueError('disp_wls: at most 8 thresholds, got %d' % len(th))
    if disp_gt is not None and not (max_gt is not None and max_gt > 0 and ctypes.c_float(max_gt).value > 0):
        raise ValueError('disp_wls: disp_gt needs max_gt > 0, got %r' % (max_gt,))
    T = len(th)
    shapes = ((torch.float32, (2 * B, H, W)), (torch.int64, (B, 2, 4 + T)))
    if out is None:
        out = (torch.empty(shapes[0][1], dtype=torch.float32, device=dev),
               torch.zeros(shapes[1][1], dtype=torch.int64, device=dev))
    else:
        out = tuple(out)
        if len(out) != 2:
            raise ValueError('disp_wls: out must hold (out, stats)')
        _chk(*out)
        for o, (d, s) in zip(out, shapes):
            if o.dtype != d or tuple(o.shape) != s or o.device != dev:
                raise ValueError('disp_wls: out tensors must be %s on %s, got %s'
                                 % ([(str(d), s) for d, s in shapes], dev, [(str(o.dtype), tuple(o.shape)) for o in out]))
        if B and out[0].untyped_storage().data_ptr() == disp.untyped_storage().data_ptr():
            raise ValueError('disp_wls: out must not share memory with disp')
    nb = disp_wls_workspace_bytes(B, H, W)
    if workspace is None:
        workspace = torch.empty(max(nb, 1), dtype=torch.uint8, device=dev)
    elif workspace.dtype != torch.uint8 or workspace.numel() < nb or workspace.device != dev:
        raise ValueError('disp_wls: workspace must be uint8 of at least %d bytes on %s' % (nb, dev))
    res, stats = out
    if B == 0:                                 # no maps (and empty tensors may hold no data pointer)
        return res, stats
    ptr = lambda t: None if t is None else t.data_ptr()
    tc = (ctypes.c_float * max(T, 1))(*th)
    rc = _lib.load().s3d_disp_wls(disp.data_ptr(), B, H, W, left.data_ptr(), right.data_ptr(), u8, ptr(mask), lut.data_ptr(),
                                  lam_v, ptr(disp_gt), tc, T, 0.0 if max_gt is None else max_gt, res.data_ptr(),
                                  stats.data_ptr(), workspace.data_ptr(), workspace.numel(), _stream())
    if rc == -1:                               # S3D_ERR_INVALID: an argument the checks above let through (H W >= 2^31, ...)
        raise ValueError('disp_wls: %s' % _lib.load().s3d_last_error().decode('utf-8', 'replace'))
    _lib.check(rc, 's3d_disp_wls')
    _lib.count_launch(6)                       # wls_row_kernel / wls_col_kernel x 3 iterations
    return res, stats
