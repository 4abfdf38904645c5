# -*- coding: utf-8 -*-
"""Stereo2Voxel / Stereo2Point inference modules on the B200 kernels.

Drop-in boundary (SURVEY.md 8(b)): `nn.Module`s with `forward(left, right)` and a `state_dict`
whose keys and shapes are exactly those of the stock-PyTorch restatement of the north_star
(oracle/models.py), so a checkpoint round-trips with `load_state_dict`.  The reference's own module
code lives on branches that are not on disk (/root/reference/README.md:5,56,62); the only attested
contract is `runner.py --test --weights=...` (README.md:91) and `cfg.SECTION.KEY` (README.md:68-78).

The torch.nn layers below are PARAMETER CONTAINERS only -- their forward is never called.  `pack()`
folds BatchNorm and re-lays every weight for the tcgen05 implicit-GEMM engine once; `forward()` is a
sequence of C-ABI calls (include/s3d.h) on the current CUDA stream, with no torch math on the path.
"""
import collections
import ctypes
import math
import os

import numpy as np
import torch
import torch.nn as nn

from . import lib as _lib
from . import ops
from .layers import PackedConv, SplitConv, pad_to, torch_dtype, cmult, more_columns_than_pairs

A = _lib  # activation / dtype codes

# NETWORK.PRECISION.  'bf16x3': every activation and weight is a bf16 pair v = hi + lo and every tensor-core product runs as
# hi*hi + lo*hi + hi*lo on kind::f16 MMAs into one fp32 accumulator (include/s3d.h, S3D_DTYPE_BF16X2): the FAST mode that
# meets the north_star's 1e-3 fp32 tolerance.  'tf32x3' does the same with three kind::tf32 passes per layer through HBM.
PRECISIONS = ('bf16', 'bf16x3', 'tf32', 'tf32x3', 'fp32')

# The forward's optional output groups, in tuple order after the head's outputs and the gt output (iou_counts /
# point_stats): (keyword that turns the group on, its outputs).  output_names() derives every tuple layout from this.
OPTIONAL_OUTPUTS = (('disp_gt', ('disp_stats',)),
                    ('lr_check', ('lr_mask', 'lr_stats')),
                    ('speckle', ('speckle_mask', 'speckle_stats')),
                    ('wls', ('wls_left', 'wls_right', 'wls_stats')),
                    ('uncertainty', ('disp_std', 'unc_stats')),
                    ('camera', ('cloud_xyz', 'cloud_rgb', 'cloud_counts')),
                    ('surface', ('surf_stats',)),
                    ('mesh', ('mesh_verts', 'mesh_faces', 'mesh_counts')),
                    ('curves', ('occ_hist', 'occ_loss')),
                    ('fscore_curves', ('dist_hist',)))
_VOXEL_ONLY = {'surface': 'surface=True evaluates voxel surfaces: Stereo2Voxel only',
               'mesh': 'mesh=True meshes the voxel occupancy: Stereo2Voxel only',
               'curves': 'curves=True evaluates the voxel occupancy: Stereo2Voxel only'}

# The options of one forward, checked (_StereoBase._check_args): what the stages branch on and part of the graph key.
Options = collections.namedtuple('Options', 'gt disp_gt lr_check speckle wls uncertainty camera surface mesh curves '
                                              'fscore_curves')


def _conv_bn2d(cin, cout, k, s, p):
    return nn.Sequential(nn.Conv2d(cin, cout, k, s, p, bias=False), nn.BatchNorm2d(cout))


def _conv_bn3d(cin, cout):
    return nn.Sequential(nn.Conv3d(cin, cout, 3, 1, 1, bias=False), nn.BatchNorm3d(cout))


class _FeatureEncoder(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        c1, c2 = cfg.NETWORK.ENC_CHANNELS
        cf = cfg.NETWORK.FEAT_CHANNELS
        self.conv0 = _conv_bn2d(3, c1, 3, 2, 1)
        self.conv1 = _conv_bn2d(c1, c1, 3, 1, 1)
        self.conv2 = _conv_bn2d(c1, c2, 3, 2, 1)
        self.conv3 = _conv_bn2d(c2, c2, 3, 1, 1)
        self.conv4 = _conv_bn2d(c2, c2, 3, 1, 1)
        self.conv5 = nn.Conv2d(c2, cf, 3, 1, 1, bias=True)


class _CostAggregation(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        cin, a = 2 * cfg.NETWORK.FEAT_CHANNELS, cfg.NETWORK.AGG_CHANNELS
        self.dres0a = _conv_bn3d(cin, a)
        self.dres0b = _conv_bn3d(a, a)
        self.dres1a = _conv_bn3d(a, a)
        self.dres1b = _conv_bn3d(a, a)
        self.cls_a = _conv_bn3d(a, a)
        self.cls_b = nn.Conv3d(a, 1, 3, 1, 1, bias=False)


class _DispNet(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        self.encoder = _FeatureEncoder(cfg)
        if cfg.NETWORK.COST_VOLUME == 'concat':
            self.aggregation = _CostAggregation(cfg)


class _RGBDEncoder(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        ch = [4] + list(cfg.NETWORK.REC_CHANNELS)
        self.layers = nn.ModuleList([_conv_bn2d(ch[i], ch[i + 1], 3, 2, 1) for i in range(len(ch) - 1)])


class _VoxelDecoder(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        ch = list(cfg.NETWORK.DEC_CHANNELS)
        self.layers = nn.ModuleList([
            nn.Sequential(nn.ConvTranspose3d(ch[i], ch[i + 1], 4, 2, 1, bias=False), nn.BatchNorm3d(ch[i + 1]))
            for i in range(len(ch) - 1)])
        self.out = nn.ConvTranspose3d(ch[-1], 1, 1, bias=False)


class _Merger(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        ch = list(cfg.NETWORK.MERGER_CHANNELS)
        self.layers = nn.ModuleList([_conv_bn3d(ch[i], ch[i + 1]) for i in range(len(ch) - 1)])


class _PointDecoder(nn.Module):
    def __init__(self, cfg):
        super().__init__()
        c, L = cfg.NETWORK.REC_CHANNELS[-1], cfg.NETWORK.LATENT_HW
        self.conv = _conv_bn2d(2 * c, 2 * c, 3, 2, 1)
        self.fc1 = nn.Linear(2 * c * (L // 2) * (L // 2), cfg.NETWORK.POINT_FC)
        self.fc2 = nn.Linear(cfg.NETWORK.POINT_FC, cfg.CONST.N_POINTS * 3)


def init_synthetic_weights(model, seed=0):
    """Seeded He-normal weights + randomised eval-mode BN statistics (pretrained weights are not
    available offline, BASELINE.json north_star).  Same recipe as the oracle's initialiser."""
    g = torch.Generator().manual_seed(seed + 12345)
    gains = {'decoder.out': 3.0, 'merger.layers.4.0': 4.0, 'point_decoder.fc2': 2.0}
    with torch.no_grad():
        for name, m in model.named_modules():
            if isinstance(m, (nn.Conv2d, nn.Conv3d, nn.Linear, nn.ConvTranspose3d)):
                w = m.weight
                if isinstance(m, nn.ConvTranspose3d):
                    taps = 1
                    for k, s in zip(m.kernel_size, m.stride):
                        taps *= max(k // s, 1)
                    fan_in = w.shape[0] * taps
                else:
                    fan_in = w[0].numel()
                std = (2.0 / fan_in) ** 0.5 * gains.get(name, 1.0)
                w.copy_((torch.randn(w.shape, generator=g) * std).to(w.device))
                if m.bias is not None:
                    m.bias.copy_((torch.randn(m.bias.shape, generator=g) * 0.1).to(w.device))
            elif isinstance(m, (nn.BatchNorm2d, nn.BatchNorm3d)):
                n, dev = m.num_features, m.weight.device
                m.running_mean.copy_((torch.randn(n, generator=g) * 0.1).to(dev))
                m.running_var.copy_((torch.rand(n, generator=g) + 0.5).to(dev))
                m.weight.copy_((torch.rand(n, generator=g) * 0.4 + 0.8).to(dev))
                m.bias.copy_((torch.randn(n, generator=g) * 0.1).to(dev))
    return model.eval()


class _GraphedForward:
    """One captured forward: static input buffers, a torch.cuda.CUDAGraph of the model's launch sequence, static outputs."""

    def __init__(self, model, left, right, gt, disp_gt, camera, opts):
        self.left, self.right = torch.empty_like(left), torch.empty_like(right)
        self.gt = None if gt is None else torch.empty_like(gt)
        self.disp_gt = None if disp_gt is None else torch.empty_like(disp_gt)
        self.camera = None if camera is None else torch.empty_like(camera)
        self._copy_in(left, right, gt, disp_gt, camera)

        def run():                                    # zeroes its IoU / disparity / LR / uncertainty / surface counters itself: inside the graph
            return model._forward_impl(self.left, self.right, self.gt, self.disp_gt, self.camera, opts)
        side = torch.cuda.Stream(device=left.device)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):                 # warm-up: workspace buffers and tensor maps exist before capture
            for _ in range(2):
                run()
        torch.cuda.current_stream().wait_stream(side)
        self.graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self.graph):
            self.out = run()

    def _copy_in(self, left, right, gt, disp_gt, camera):
        self.left.copy_(left, non_blocking=True)
        self.right.copy_(right, non_blocking=True)
        if self.gt is not None:
            self.gt.copy_(gt, non_blocking=True)
        if self.disp_gt is not None:
            self.disp_gt.copy_(disp_gt, non_blocking=True)
        if self.camera is not None:
            self.camera.copy_(camera, non_blocking=True)

    def __call__(self, left, right, gt, disp_gt=None, camera=None):
        self._copy_in(left, right, gt, disp_gt, camera)
        self.graph.replay()
        return self.out


class _StereoBase(nn.Module):
    """Shared disparity stage (rows E, V, A, S) and RGB-D encoder (row X)."""

    def __init__(self, cfg):
        super().__init__()
        self.cfg = cfg
        self.dispnet = _DispNet(cfg)
        self.rgbd_encoder = _RGBDEncoder(cfg)
        self._packed = None
        self._ws = {}
        self._graphs = {}
        self._packed_prec = None
        # the nn layers are parameter containers: anything that changes them (load_state_dict, .to / .cuda / .half,
        # init_synthetic_weights writes in place and calls eval()) must drop the folded copies, workspaces and graphs
        self.register_load_state_dict_post_hook(lambda module, incompatible: module._invalidate())

    def _invalidate(self):
        self._packed = None
        self._ws = {}
        self._graphs = {}

    def _apply(self, fn, *args, **kwargs):
        r = super()._apply(fn, *args, **kwargs)
        self._invalidate()
        return r

    def train(self, mode=True):
        # init_synthetic_weights() / a user's model.eval() after editing parameters in place: re-pack on the next forward
        self._invalidate()
        return super().train(mode)

    # ---- packing ---------------------------------------------------------------------------
    @property
    def precision(self):
        return self.cfg.NETWORK.PRECISION

    def _dtype_code(self):
        if self.precision not in PRECISIONS:
            raise ValueError('NETWORK.PRECISION must be one of %s, got %r' % (PRECISIONS, self.precision))
        return {'bf16': A.DTYPE_BF16, 'bf16x3': A.DTYPE_BF16X2}.get(self.precision, A.DTYPE_F32)

    @property
    def _split(self):
        return self.precision == 'bf16x3'

    def _engine(self):
        return 'direct' if self.precision == 'fp32' else 'igemm'

    def pack(self):
        """Fold BN + re-lay weights for the conv engine.  Call after load_state_dict / .cuda()."""
        cfgn = self.cfg.NETWORK
        if cfgn.DEC_CHANNELS[0] % 16 or cfgn.REC_CHANNELS[-1] % 16:
            # latent_to_vox writes [.., C*L*L/8] densely; dec0 reads it with its padded channel pitch
            raise ValueError('NETWORK.DEC_CHANNELS[0] and NETWORK.REC_CHANNELS[-1] must be multiples of 16')
        dev = next(self.parameters()).device
        if dev.type != 'cuda':
            raise _lib.S3dError('Stereo2Voxel/Stereo2Point run on CUDA only (no CPU fallback); call .cuda() first')
        _lib.load()
        dc = self._dtype_code()
        P = {}
        e = self.dispnet.encoder
        for i in range(5):
            seq = getattr(e, 'conv%d' % i)
            P['enc%d' % i] = PackedConv.from_conv(seq[0], seq[1], A.ACT_NONE if i == 4 else A.ACT_RELU, dc, dev)
        P['enc5'] = PackedConv.from_conv(e.conv5, None, A.ACT_NONE, dc, dev)
        if self.cfg.NETWORK.COST_VOLUME == 'concat':
            ag = self.dispnet.aggregation
            for n in ('dres0a', 'dres0b', 'dres1a', 'dres1b', 'cls_a'):
                seq = getattr(ag, n)
                P[n] = PackedConv.from_conv(seq[0], seq[1], A.ACT_NONE if n == 'dres1b' else A.ACT_RELU, dc, dev)
            # Cout = 1: per-tap projections (pointwise GEMM, 27 "channels") + gather/soft-argmin kernel
            wb = ag.cls_b.weight                                      # [1, A, 3, 3, 3]
            P['cls_b'] = PackedConv.from_pointwise(wb[0].reshape(wb.shape[1], 27).t(), None, None, A.ACT_NONE, dc, dev)
        for i, seq in enumerate(self.rgbd_encoder.layers):
            P['rec%d' % i] = PackedConv.from_conv(seq[0], seq[1], A.ACT_RELU, dc, dev)
        self._pack_head(P, dc, dev)
        if self.precision == 'tf32x3':
            # every conv as three TF32 passes over split operands (layers.py::SplitConv): fp32 accuracy on the tensor cores
            P = {k: SplitConv(v) for k, v in P.items()}
        self._packed = P
        self._packed_prec = self.precision
        self._ws = {}
        self._graphs = {}
        return self

    def _pack_head(self, P, dc, dev):
        raise NotImplementedError

    def _buf(self, name, shape, dtype, zero=False):
        key = (name, tuple(shape), dtype)
        t = self._ws.get(key)
        if t is None:
            dev = next(self.parameters()).device
            t = (torch.zeros if zero else torch.empty)(shape, dtype=dtype, device=dev)
            self._ws[key] = t
        return t

    def _conv(self, name, x, **kw):
        return self._packed[name](x, engine=self._engine(), **kw)

    # ---- stages ----------------------------------------------------------------------------
    @staticmethod
    def _bhw(img):
        return (img.shape[0], img.shape[1], img.shape[2]) if img.dtype == torch.uint8 else (img.shape[0], img.shape[2], img.shape[3])

    def _disparity(self, left, right, disp_gt=None, lr_check=False, uncertainty=False):
        """-> (disp fp32 [2B,H,W] (left-referenced first) in input pixels, the dict of named evaluation outputs of
        _upsample_disp)."""
        cfg = self.cfg
        B, H, W = self._bhw(left)
        D = cfg.NETWORK.MAX_DISP
        dt = torch_dtype(self._dtype_code())
        x = self._first('enc0', 'e0', 'img', left, right, None, 1.0)
        x = self._conv('enc1', x, out=self._bufo('e1', 'enc1', x))
        x = self._conv('enc2', x, out=self._bufo('e2', 'enc2', x))
        y = self._conv('enc3', x, out=self._bufo('e3', 'enc3', x))
        x = self._conv('enc4', y, residual=x, out=self._bufo('e4', 'enc4', y))
        h, w = x.shape[2], x.shape[3]
        C = cfg.NETWORK.FEAT_CHANNELS
        p5, p0 = self._packed['enc5'], self._packed.get('dres0a')
        # 'bf16x3' (split operands): the reference-once kernel only (C = 32 feature channels, 64-wide first layer)
        ro_split = (self._split and C == 32 and isinstance(p0, PackedConv) and p0.cout_pad == 64 and p0.act == _lib.ACT_RELU and
                    not _lib.KNOBS['no_ref_once'])
        # SHEARED form of the cost volume + first aggregation layer (bf16 and the bf16 pairs of 'bf16x3', 32 feature channels,
        # 64-wide ReLU layer): 2-D map convolutions + one streaming pass; its kernels fill the chip at every batch size
        sheared = (cfg.NETWORK.COST_VOLUME == 'concat' and (self.precision == 'bf16' or ro_split) and C == 32 and p5.cout_pad == C and
                   isinstance(p0, PackedConv) and p0.weight_ns is not None and p0.cout_pad == 64 and p0.act == _lib.ACT_RELU and
                   D >= 4 and w + 2 <= 127 and not _lib.KNOBS['no_sheared'] and not _lib.KNOBS['no_concat_fuse'] and
                   not _lib.KNOBS['no_scatter'])
        fuse_volume = (cfg.NETWORK.COST_VOLUME == 'concat' and (self.precision in ('bf16', 'tf32') or ro_split) and p5.cout_pad == C and
                       isinstance(p0, PackedConv) and p0.weight_ns is not None and
                       (ro_split or C * x.element_size() in (32, 64)) and
                       not _lib.KNOBS['no_concat_fuse'] and not _lib.KNOBS['no_scatter'] and
                       # small batches: fewer columns than SMs -> unfused volume + the z-split plane-scatter kernel (a column of
                       # D planes would be a serial chain on a fraction of the chip; csrc/conv_scatter.cuh, ScArgs::nz)
                       (sheared or more_columns_than_pairs(2 * B, h, w)))
        cm = cmult(self._dtype_code())                           # physical channels per logical channel (2 when split)
        if fuse_volume:
            # features go into rows with D zero pixels on both sides: the fused cost-volume + dres0a kernel reads the shifted
            # target view of every disparity plane straight out of them (csrc/conv_scatter_concat.cu), no volume is written
            pad, P = D, w + 2 * D
            Cp = cm * C                                              # physical channels of a feature row ([hi | lo] when split)
            featp = self._buf('featp', (2 * B, 1, h, P, Cp), dt, zero=True)
            self._conv('enc5', x, out=featp, out_view=(pad * Cp, (h * P * Cp, h * P * Cp, P * Cp, Cp), C if self._split else 0),
                       cout_store=C)
            feat = None
        else:
            feat = self._conv('enc5', x, out=self._bufo('e5', 'enc5', x))
        disp_q = self._buf('disp_q', (2 * B, h, w), torch.float32)
        # the standard deviation of each pixel's soft-argmin distribution, from the same kernel as disp_q
        std_q = self._buf('disp_std_q', (2 * B, h, w), torch.float32) if uncertainty else None
        std_kw = {} if std_q is None else {'std_out': std_q}           # the plain calls keep their plain signature
        if cfg.NETWORK.COST_VOLUME == 'concat':
            if fuse_volume:
                # bf16: reference-once form -- the d-independent reference half is convolved once per column, the planes run
                # on the target half only (half the tensor-core work of this layer; csrc/conv_scatter_concat.cu)
                ro = ro_split or (self.precision == 'bf16' and p0.cout_pad == 64 and p0.act == _lib.ACT_RELU and
                                  not _lib.KNOBS['no_ref_once'])
                if sheared:
                    # SHEARED form: in u = x -/+ d the target half of the volume is the same map on every plane, so the layer is
                    # four 2-D map convolutions (csrc/map_conv.cu: 1/14 of the layer's MMAs) + one streaming pass that adds two
                    # maps per output element and writes the volume (csrc/concat_gonce.cu): 0.79 ms against 1.15 ms for the
                    # reference-once kernel at batch 64 (A/B knob no_sheared)
                    bufs = {'maps_l': self._buf('sh_ml', (B, 1, h, w + 4, 384), torch.float32),
                            'maps_r': self._buf('sh_mr', (B, 1, h, w + 4, 384), torch.float32),
                            'edge_l': self._buf('sh_el', (B, 1, h, D, 256), torch.float32),
                            'edge_r': self._buf('sh_er', (B, 1, h, D, 256), torch.float32)}
                    a = ops.conv_concat_volume_sheared(p0, featp, B, D, pad, out=self._buf('a0', (2 * B, D, h, w, cm * 64), dt), bufs=bufs)
                else:
                    a = ops.conv_concat_volume(p0, featp, B, D, pad, out=self._buf('a0', (2 * B, D, h, w, cm * p0.cout_pad), dt),
                                               ref_once=ro)
            else:
                assert feat.shape[-1] == cm * C, 'FEAT_CHANNELS must be a multiple of 16'
                vol = ops.cost_volume_concat(feat, B, D, out=self._buf('vol', (2 * B, D, h, w, 2 * cm * C), dt), split=self._split)
                a = self._conv('dres0a', vol, out=self._bufo('a0', 'dres0a', vol))
            # Where the target half of the concat volume is zero around a pixel (d > x + 1 left-referenced, d > w - 2 - x
            # right-referenced), a0 is the same on every plane up to D - 2: the layers below compute such planes once
            # (include/s3d.h dz_nref).  Each 3x3x3 layer moves the region one plane in from both ends.  bf16 only.
            bf = self.precision == 'bf16'
            a = self._conv('dres0b', a, out=self._bufo('a1', 'dres0b', a), dz=(B, 3, 1) if bf else None)
            y = self._conv('dres1a', a, out=self._bufo('a2', 'dres1a', a), dz=(B, 5, 2) if bf else None)
            a = self._conv('dres1b', y, residual=a, out=self._bufo('a3', 'dres1b', y), dz=(B, 7, 3) if bf else None)
            S = self._packed['cls_b'].cout_pad                      # 27 taps padded to 32 planes
            pa = self._packed['cls_a']
            if (self.precision == 'bf16' and isinstance(pa, PackedConv) and pa.weight_ns is not None and pa.cin_pad == 64 and
                    pa.cout_pad == 64 and pa.act == _lib.ACT_RELU and S == 32 and a.shape[-1] == 64 and
                    more_columns_than_pairs(2 * B, h, w) and
                    not _lib.KNOBS['no_cls_chain'] and not _lib.KNOBS['no_cls_fused'] and not _lib.KNOBS['no_scatter']):
                # cls_a + classifier + soft-argmin in one march, cls_a's 2.1 GB output never written (csrc/conv_scatter_cls.cu)
                nb = ops.conv_cls_workspace_bytes(2 * B, D, h, w)
                ops.conv_cls_soft_argmin(pa, a, self._packed['cls_b'].weight, -1.0, out=disp_q,
                                         workspace=self._buf('cls_ws', (nb,), torch.uint8), **std_kw)
                return self._upsample_disp(disp_q, H, W, disp_gt, lr_check, std_q)
            c = self._conv('cls_a', a, out=self._bufo('a0', 'cls_a', a))
            if self.precision == 'bf16' and c.shape[-1] in (16, 32, 64) and S == 32 and not _lib.KNOBS['no_cls_fused']:
                # classifier + soft-argmin in one pass over the volume (csrc/cls_fused.cu)
                ops.cls_soft_argmin(c, self._packed['cls_b'].weight, -1.0, out=disp_q, **std_kw)
            else:
                taps = self._buf('taps', (2 * B, D, h, S, w), torch.float32)   # line-planar: [.., y, tap, x]
                self._conv('cls_b', c, out=taps, out_view=(0, (D * h * S * w, h * S * w, S * w, 1, w)), cout_store=S)
                ops.tap_gather_soft_argmin(taps, -1.0, out=disp_q, **std_kw)
        else:
            if self._split:                                               # exact fp32 correlation on hi + lo
                feat = ops.unsplit_bf16(feat, out=self._buf('feat32', feat.shape[:-1] + (feat.shape[-1] // 2,), torch.float32))
            ops.corr_soft_argmin(feat, B, D, out=disp_q, c_real=C, **std_kw)        # mean over the REAL channels (feat is padded)
        return self._upsample_disp(disp_q, H, W, disp_gt, lr_check, std_q)

    def _upsample_disp(self, disp_q, H, W, disp_gt, lr_check=False, std_q=None):
        """Last kernel of the disparity stage: 1/4-res disparity -> input pixels [2B,H,W].  With disp_gt [B,2,H,W] the same
        kernel also counts, per sample and view, [n_valid, sum |disp - gt| in 2^-16 px, count(|disp - gt| > t) for t in
        TEST.DISP_THRESH] over the pixels with 0 <= gt < 4 * MAX_DISP -> disp_stats int64 [B,2,2+T].  With lr_check it
        also runs the left-right consistency check (include/s3d.h, s3d_upsample_disp_eval; tolerance TEST.LR_THRESH px) ->
        lr_mask uint8 [B,2,H,W], lr_stats int64 [B,2,3+T]: [n_kept, n_valid_kept, sum |disp - gt| in 2^-16 px and
        count(|disp - gt| > t) over the kept valid pixels]; GT columns zero without disp_gt.  With std_q (the 1/4-res
        standard deviation) the same kernel also upsamples it and counts the confident pixels (thresholds TEST.UNC_THRESH
        px) -> disp_std fp32 [B,2,H,W], unc_stats int64 [B,2,K,3+T]: per threshold [n_conf, n_valid_conf, sum |disp - gt| in
        2^-16 px and count(|disp - gt| > t) over the confident valid pixels]; GT columns zero without disp_gt.
        -> (disp, {name: tensor} of the outputs above that were computed)."""
        B = disp_q.shape[0] // 2
        out = self._buf('disp', (2 * B, H, W), torch.float32)
        if disp_gt is None and not lr_check and std_q is None:
            return ops.upsample_disp(disp_q, H, W, 4.0, out=out), {}
        th = list(self.cfg.TEST.DISP_THRESH)
        ev = {}
        if disp_gt is not None:
            ev['disp_stats'] = self._buf('disp_stats', (B, 2, 2 + len(th)), torch.int64).zero_()
        max_gt = 4.0 * self.cfg.NETWORK.MAX_DISP
        tau = 0.0
        if lr_check:
            tau = lr_thresh(self.cfg)
            ev['lr_mask'] = self._buf('lr_mask', (B, 2, H, W), torch.uint8)
            ev['lr_stats'] = self._buf('lr_stats', (B, 2, 3 + len(th)), torch.int64).zero_()
        ut = ()
        if std_q is not None:
            ut = unc_thresholds(self.cfg)
            ev['unc_stats'] = self._buf('unc_stats', (B, 2, len(ut), 3 + len(th)), torch.int64).zero_()
            ev['disp_std'] = self._buf('disp_std', (B, 2, H, W), torch.float32)
        ops.upsample_disp_eval(disp_q, H, W, 4.0, disp_gt, th, max_gt, ev.get('disp_stats'), lr_thresh=tau,
                               mask=ev.get('lr_mask'), lr_stats=ev.get('lr_stats'), std_q=std_q, unc_thresh=ut,
                               unc_stats=ev.get('unc_stats'), std_out=ev.get('disp_std'), out=out)
        return out, ev

    def _bufo(self, name, layer, x):
        """Output buffer of `layer` for input x (channels-last, padded channels)."""
        pc = self._packed[layer]
        N, iD, iH, iW, _ = x.shape
        oD, oH, oW = pc.out_grid(iD, iH, iW)
        m = pc.out_mult
        return self._buf(name, (N, oD * m[0], oH * m[1], oW * m[2], pc.cout_pad * cmult(pc.dtype_code)), x.dtype)

    def _latent(self, left, right, disp):
        """RGB-D encoder on both views -> [2B,1,h',w',C_last] (before pooling)."""
        B, H, W = self._bhw(left)
        dt = torch_dtype(self._dtype_code())
        scale = 1.0 / (4.0 * self.cfg.NETWORK.MAX_DISP)
        x = self._first('rec0', 'r0', 'rgbd', left, right, disp, scale)
        for i in range(1, len(self.rgbd_encoder.layers)):
            x = self._conv('rec%d' % i, x, out=self._bufo('r%d' % i, 'rec%d' % i, x))
        return x

    def _first(self, layer, out_name, stage_name, left, right, disp, scale):
        """First layer of an encoder on both views: straight from the raw images (csrc/conv_first.cu) when it is the
        3x3 stride-2 layer that kernel implements, else staged channels-last copy + the general conv engine."""
        B, H, W = self._bhw(left)
        pc = self._packed[layer]
        dt = torch_dtype(self._dtype_code())
        if pc.ksize == (1, 3, 3) and pc.stride == (1, 2, 2) and pc.pad == (0, 1, 1) and pc.cout_pad in (16, 32, 64) and \
                not _lib.KNOBS['no_conv_first']:
            oH, oW = (H - 1) // 2 + 1, (W - 1) // 2 + 1
            out = self._buf(out_name, (2 * B, 1, oH, oW, pc.cout_pad * cmult(pc.dtype_code)), dt)
            ops.conv_first(left, pc, None if disp is None else disp[:B], scale, out=out[:B])
            ops.conv_first(right, pc, None if disp is None else disp[B:], scale, out=out[B:])
            return out
        if self._split:
            raise _lib.S3dError("'bf16x3' needs the direct first layer (3x3 stride-2 conv, <= 64 output channels)")
        x = self._buf(stage_name, (2 * B, 1, H, W, 16), dt)
        ops.pack_image(left, None if disp is None else disp[:B], scale, out=x[:B])
        ops.pack_image(right, None if disp is None else disp[B:], scale, out=x[B:])
        return self._conv(layer, x, out=self._bufo(out_name, layer, x))

    # ---- CUDA-graph replay (SURVEY.md 8(f) item 3) ---------------------------------------------
    def graphed(self, left, right, gt=None, *, disp_gt=None, lr_check=False, speckle=False, wls=False, uncertainty=False,
                camera=None, surface=False, mesh=False, curves=False, fscore_curves=False):
        """Same results as forward(), replayed from a CUDA graph captured on first use for this input signature: one
        graph launch instead of ~35 kernel launches + torch glue.  Measured (scripts/graph_latency.py): B = 1 1.23 -> 1.19 ms,
        B = 8 2.40 -> 2.37 ms -- the forward is GPU-bound even at batch 1 (a column of 32 planes is a serial chain of
        ~0.12 ms per aggregation layer), so the graph only removes the launch gaps.
        Inputs are copied into the graph's static buffers; the returned tensors are the graph's static outputs and
        are overwritten by the next call with the same signature."""
        left, right, gt, disp_gt, camera, opts = self._check_args(left, right, gt, disp_gt, lr_check, uncertainty, camera,
                                                                  surface, mesh, curves, fscore_curves, speckle, wls)
        mb = int(self.cfg.CONST.get('MICRO_BATCH', 0) or 0)
        if mb and left.shape[0] > mb:
            raise ValueError('graphed(): batch %d exceeds CONST.MICRO_BATCH = %d; use forward()' % (left.shape[0], mb))
        key = (tuple(left.shape), left.dtype, None if gt is None else (tuple(gt.shape), gt.dtype),
               None if disp_gt is None else (tuple(disp_gt.shape), disp_gt.dtype),
               None if camera is None else (tuple(camera.shape), camera.dtype), opts)
        g = self._graphs.get(key)
        if g is None:
            g = self._graphs[key] = _GraphedForward(self, left, right, gt, disp_gt, camera, opts)
        return g(left, right, gt, disp_gt, camera)

    # ---- outputs and their checks --------------------------------------------------------------
    @classmethod
    def output_names(cls, gt=False, disp_gt=False, lr_check=False, uncertainty=False, surface=False, mesh=False,
                     curves=False, fscore_curves=False, camera=False, speckle=False, wls=False):
        """Names of the forward's outputs, in tuple order, for these options (gt / disp_gt / camera: whether the tensor is given):
        the head's outputs, the gt output, then the groups of OPTIONAL_OUTPUTS that are on.  ValueError on an option the
        class does not have."""
        on = {'disp_gt': disp_gt, 'lr_check': lr_check, 'speckle': speckle, 'wls': wls, 'uncertainty': uncertainty,
              'camera': camera, 'surface': surface, 'mesh': mesh, 'curves': curves, 'fscore_curves': fscore_curves}
        names = cls.HEAD_OUTPUTS + ((cls.GT_OUTPUT,) if gt else ())
        for opt, outs in OPTIONAL_OUTPUTS:
            if on[opt]:
                if opt not in cls.OPTIONS:
                    raise ValueError(_VOXEL_ONLY[opt])
                names += outs
        return names

    def _check_args(self, left, right, gt, disp_gt, lr_check, uncertainty, camera, surface, mesh, curves, fscore_curves,
                    speckle=False, wls=False):
        """The one check of forward() / graphed()'s arguments, before anything is launched: first the options (which the
        class has, what they need), then the cfg.TEST thresholds of the enabled outputs, then the tensors.
        -> (left, right, gt, disp_gt, camera) as the forward takes them and the options value: an Options of bools."""
        opts = Options(gt is not None, disp_gt is not None, bool(lr_check), bool(speckle), bool(wls), bool(uncertainty),
                       camera is not None, bool(surface), bool(mesh), bool(curves), bool(fscore_curves))
        self.output_names(**opts._asdict())                   # ValueError on an option this class does not have
        if opts.surface and not opts.gt:
            raise ValueError('surface=True needs the GT occupancy gt')
        if opts.curves and not opts.gt:
            raise ValueError('curves=True needs the GT occupancy gt')
        if opts.fscore_curves and not opts.gt:
            raise ValueError('fscore_curves=True needs the GT %s gt' % ('point cloud' if self.GT_OUTPUT == 'point_stats'
                                                                          else 'occupancy'))
        if opts.fscore_curves and 'surface' in self.OPTIONS and not opts.surface:
            raise ValueError('fscore_curves=True evaluates the voxel surfaces: it needs surface=True')
        if opts.uncertainty:
            unc_thresholds(self.cfg)
        if opts.surface or (opts.gt and self.GT_OUTPUT == 'point_stats'):     # the surface and point-cloud F-scores
            fscore_thresholds(self.cfg)
        if opts.mesh:
            mesh_thresh(self.cfg)
        if opts.curves:
            curve_bins(self.cfg)
        if opts.lr_check:
            lr_thresh(self.cfg)
        if opts.speckle:
            speckle_params(self.cfg)
        if opts.wls:
            wls_params(self.cfg)
        if opts.fscore_curves:
            dist_edges(self.cfg)
        if opts.camera:
            cloud_min_disp(self.cfg)
            if opts.uncertainty:
                cloud_max_std(self.cfg)
        left, right = self._check_inputs(left, right)
        if opts.wls:
            self._wls_lut(wls_params(self.cfg)[1])         # built here, outside the forward (and outside a graph capture)
        return (left, right, self._check_gt(gt, left), self._check_disp_gt(disp_gt, left), self._check_camera(camera, left),
                opts)

    def _forward_impl(self, left, right, gt, disp_gt, camera, opts):
        """The forward of checked arguments: the stages fill one dict of named outputs, returned in output_names order."""
        B = left.shape[0]
        disp, out = self._disparity(left, right, disp_gt, opts.lr_check, opts.uncertainty)
        out.update(disp_left=disp[:B].unsqueeze(1), disp_right=disp[B:].unsqueeze(1))
        if opts.speckle:
            out['speckle_mask'], out['speckle_stats'] = self._speckle(disp, disp_gt, out.get('lr_mask'))
        if opts.wls:
            out['wls_left'], out['wls_right'], out['wls_stats'] = self._wls(left, right, disp, disp_gt, out)
        if camera is not None:
            out['cloud_xyz'], out['cloud_rgb'], out['cloud_counts'] = self._cloud(left, right, disp, camera, out)
        self._head(left, right, gt, disp, opts, out)
        return tuple(out[n] for n in self.output_names(**opts._asdict()))

    def _check_inputs(self, left, right):
        if self._packed is None or self._packed_prec != self.precision:
            self.pack()
        if not (left.is_cuda and right.is_cuda):
            raise _lib.S3dError('inputs must be CUDA tensors (no CPU fallback)')
        if left.dtype == torch.uint8 and right.dtype == torch.uint8:
            # decoded 8-bit images, HWC [B,H,W,3]: converted (x/255) inside the staging kernel, 4x less H2D traffic
            if left.shape != right.shape or left.dim() != 4 or left.shape[3] != 3:
                raise ValueError('expected uint8 left/right of shape [B,H,W,3], got %s / %s' % (tuple(left.shape), tuple(right.shape)))
            return left.contiguous(), right.contiguous()
        if left.shape != right.shape or left.dim() != 4 or left.shape[1] != 3:
            raise ValueError('expected left/right of shape [B,3,H,W], got %s / %s' % (tuple(left.shape), tuple(right.shape)))
        return left.contiguous().float(), right.contiguous().float()

    def _check_gt(self, gt, left):
        """The head's GT as the head takes it (Stereo2Point validates its point cloud)."""
        return gt

    def _check_disp_gt(self, disp_gt, left):
        """GT disparity of (checked) inputs `left`: fp32 [B,2,H,W] on their device, in input pixels, view 0 = left-referenced
        (as disp_left), 1 = right-referenced; NaN marks pixels without GT."""
        if disp_gt is None:
            return None
        B, H, W = self._bhw(left)
        if not isinstance(disp_gt, torch.Tensor):
            raise ValueError('disp_gt must be a tensor, got %s' % type(disp_gt).__name__)
        if tuple(disp_gt.shape) != (B, 2, H, W):
            raise ValueError('expected disp_gt of shape %s, got %s' % ((B, 2, H, W), tuple(disp_gt.shape)))
        if disp_gt.dtype != torch.float32:
            raise ValueError('disp_gt must be float32, got %s' % disp_gt.dtype)
        if disp_gt.device != left.device:
            raise ValueError('disp_gt must be on %s (the images\' device), got %s' % (left.device, disp_gt.device))
        return disp_gt.contiguous()

    def _check_camera(self, camera, left):
        """Camera of (checked) inputs `left`: fp32 [B,5] = (f, cx, cy, baseline, doffs) per sample on their device (include/s3d.h,
        s3d_disp_cloud).  Its values stay on the device and are not checked."""
        if camera is None:
            return None
        B = left.shape[0]
        if not isinstance(camera, torch.Tensor):
            raise ValueError('camera must be a tensor, got %s' % type(camera).__name__)
        if tuple(camera.shape) != (B, 5):
            raise ValueError('expected camera of shape %s, got %s' % ((B, 5), tuple(camera.shape)))
        if camera.dtype != torch.float32:
            raise ValueError('camera must be float32, got %s' % camera.dtype)
        if camera.device != left.device:
            raise ValueError('camera must be on %s (the images\' device), got %s' % (left.device, camera.device))
        return camera.contiguous()

    def _speckle(self, disp, disp_gt, lr_mask):
        """Speckle filter of disp [2B,H,W] (include/s3d.h, s3d_speckle_filter; TEST.SPECKLE_MAX_SIZE / SPECKLE_MAX_DIFF), after
        the LR check when lr_mask is given -> (speckle_mask uint8 [B,2,H,W], speckle_stats int64 [B,2,5+T]): the counters of
        lr_stats over the kept pixels against disp_gt (TEST.DISP_THRESH, valid below 4 * MAX_DISP; zero without it), then
        n_speckles, n_speckle_px.  The stats are zeroed here, so a graph replay starts from zero; every buffer comes from the
        workspace: no allocation on this path."""
        B, H, W = disp.shape[0] // 2, disp.shape[1], disp.shape[2]
        max_size, max_diff = speckle_params(self.cfg)
        th = list(self.cfg.TEST.DISP_THRESH)
        nb = ops.speckle_filter_workspace_bytes(B, H, W)
        return ops.speckle_filter(disp, B, max_size, max_diff, lr_mask=lr_mask, disp_gt=disp_gt, thresholds=th,
                                  max_gt=4.0 * self.cfg.NETWORK.MAX_DISP,
                                  out=(self._buf('speckle_mask', (B, 2, H, W), torch.uint8),
                                       self._buf('speckle_stats', (B, 2, 5 + len(th)), torch.int64).zero_()),
                                  workspace=self._buf('speckle_ws', (max(nb, 1),), torch.uint8))

    def _wls_lut(self, sigma):
        """The edge-weight table of sigma on the module's device (ops.wls_weight_lut), built once per sigma and kept with
        the workspace."""
        key = ('wls_lut', sigma)
        t = self._ws.get(key)
        if t is None:
            t = self._ws[key] = torch.from_numpy(ops.wls_weight_lut(sigma)).to(next(self.parameters()).device)
        return t

    def _wls(self, left, right, disp, disp_gt, ev):
        """WLS filter of disp [2B,H,W] guided by each view's image (include/s3d.h, s3d_disp_wls; TEST.WLS_LAMBDA / WLS_SIGMA),
        confident where `ev` holds the speckle mask, else the LR mask, else where d is finite -> (wls_left fp32 [B,1,H,W],
        wls_right fp32 [B,1,H,W], views of one view-major buffer, wls_stats int64 [B,2,4+T]): the lr_stats counters over
        the finite output pixels against disp_gt (TEST.DISP_THRESH, valid below 4 * MAX_DISP; zero without it), then n_conf.
        The stats are zeroed here, so a graph replay starts from zero; the table was built by _check_args and every buffer
        comes from the workspace: no allocation and no host copy on this path."""
        B, H, W = disp.shape[0] // 2, disp.shape[1], disp.shape[2]
        lam, sigma = wls_params(self.cfg)
        th = list(self.cfg.TEST.DISP_THRESH)
        mask = ev['speckle_mask'] if 'speckle_mask' in ev else ev.get('lr_mask')
        nb = ops.disp_wls_workspace_bytes(B, H, W)
        w, stats = ops.disp_wls(disp, B, left, right, self._wls_lut(sigma), lam, mask=mask, disp_gt=disp_gt, thresholds=th,
                                max_gt=4.0 * self.cfg.NETWORK.MAX_DISP,
                                out=(self._buf('wls', (2 * B, H, W), torch.float32),
                                     self._buf('wls_stats', (B, 2, 4 + len(th)), torch.int64).zero_()),
                                workspace=self._buf('wls_ws', (max(nb, 1),), torch.uint8))
        return w[:B].unsqueeze(1), w[B:].unsqueeze(1), stats

    def _cloud(self, left, right, disp, camera, ev):
        """Coloured point clouds of disp [2B,H,W] with the camera -> (cloud_xyz fp32 [B,2HW,3], cloud_rgb uint8 [B,2HW,3],
        cloud_counts int32 [B,2]), filtered by the speckle mask (which includes the LR check) or else the LR mask, and by the
        disparity spread (TEST.CLOUD_MAX_STD), when the forward computed them in `ev` (include/s3d.h, s3d_disp_cloud;
        TEST.CLOUD_MIN_DISP).  When `ev` holds the WLS maps, those are back-projected instead, with no mask and no spread
        filter: the confidence already went into the filter.  The kernels write every output (nothing to zero) into workspace
        buffers: no allocation on this path."""
        B, H, W = disp.shape[0] // 2, disp.shape[1], disp.shape[2]
        std = ev.get('disp_std')
        nb = ops.disp_cloud_workspace_bytes(B, H)
        mask = ev['speckle_mask'] if 'speckle_mask' in ev else ev.get('lr_mask')
        if 'wls_stats' in ev:
            disp, mask, std = self._buf('wls', (2 * B, H, W), torch.float32), None, None
        return ops.disp_cloud(disp, B, left, right, camera, cloud_min_disp(self.cfg), lr_mask=mask, disp_std=std,
                              max_std=None if std is None else cloud_max_std(self.cfg),
                              out=(self._buf('cloud_xyz', (B, 2 * H * W, 3), torch.float32),
                                   self._buf('cloud_rgb', (B, 2 * H * W, 3), torch.uint8),
                                   self._buf('cloud_counts', (B, 2), torch.int32)),
                              workspace=self._buf('cloud_ws', (max(nb, 1),), torch.uint8))


class Stereo2Voxel(_StereoBase):
    """forward(left, right[, gt][, disp_gt=][, lr_check=][, speckle=][, wls=][, uncertainty=][, camera=]) -> (disp_left
    [B,1,H,W], disp_right [B,1,H,W], voxels [B,32,32,32][, iou_counts int64 [B,T,2]][, disp_stats int64 [B,2,2+T']][, lr_mask
    uint8 [B,2,H,W], lr_stats int64 [B,2,3+T']][, speckle_mask uint8 [B,2,H,W], speckle_stats int64 [B,2,5+T']][, wls_left
    fp32 [B,1,H,W], wls_right fp32 [B,1,H,W], wls_stats int64 [B,2,4+T']][, disp_std fp32
    [B,2,H,W], unc_stats int64 [B,2,K,3+T']][, cloud_xyz fp32 [B,2HW,3], cloud_rgb
    uint8 [B,2HW,3], cloud_counts int32 [B,2]][, surf_stats int64 [B,T,2,3+F]][, mesh_verts fp32
    [B,max_verts,3], mesh_faces int32 [B,max_faces,3], mesh_counts int32 [B,2]][, occ_hist int64 [B,3,K], occ_loss int64
    [B,2]]).
    Outputs are views of the module's workspace: clone to keep them.  disp_gt: fp32 [B,2,H,W] GT disparity of the two views
    (NaN = none); lr_check=True: left-right consistency check of the two disparity maps; uncertainty=True: the standard
    deviation of each pixel's soft-argmin distribution in input pixels, and counters over the pixels it marks as confident
    (K = len(TEST.UNC_THRESH)); disp_stats, lr_mask, lr_stats, disp_std, unc_stats: _StereoBase._upsample_disp.
    speckle=True: OpenCV's speckle filter of the two disparity maps (after the LR check with lr_check=True): speckle_mask is 1
    where a pixel's region of finite disparities whose 4-neighbours differ by at most TEST.SPECKLE_MAX_DIFF px has more than
    TEST.SPECKLE_MAX_SIZE pixels; speckle_stats = the lr_stats counters over those pixels, then the number of removed regions
    and their pixels (_StereoBase._speckle; include/s3d.h, s3d_speckle_filter; four more launches).  With camera= as well the
    cloud keeps only the pixels of speckle_mask.
    wls=True: OpenCV's WLS fill of the two disparity maps, guided by each view's image and weighted by the confidence
    (speckle_mask with speckle=True, else lr_mask with lr_check=True, else the finite pixels): wls_left / wls_right fp32
    [B,1,H,W] (NaN where no confident pixel reaches) and wls_stats int64 [B,2,4+T'] = the lr_stats counters over the finite
    output pixels, then the confident input pixels (_StereoBase._wls; include/s3d.h, s3d_disp_wls; TEST.WLS_LAMBDA /
    WLS_SIGMA; six more launches), right after the speckle outputs.  With camera= as well the cloud back-projects the WLS
    maps with no mask and no spread filter.
    camera=(fp32 [B,5] = (f, cx, cy, baseline, doffs) per sample on the images' device, with or without gt): the coloured
    point clouds of the two disparity maps in the left camera's frame, one per sample: the kept pixels of disp_left in raster
    order, then those of disp_right, each at depth f * baseline / (d + doffs) and coloured from its own image; a pixel is kept
    when d is finite and d + doffs >= TEST.CLOUD_MIN_DISP, with lr_check=True only where lr_mask is 1 and with
    uncertainty=True only where disp_std <= TEST.CLOUD_MAX_STD; cloud_counts = kept points per view and only the first
    cloud_counts[b,0] + cloud_counts[b,1] rows are written (include/s3d.h, s3d_disp_cloud; two more launches).
    surface=True (needs gt): the voxel-face surfaces of the prediction at each t in TEST.VOXEL_THRESH and of gt, evaluated
    against each other; surf_stats per sample, t and direction (0: predicted -> GT, 1: GT -> predicted) = [n_pts, sum s,
    sum q(sqrt s), count(s < k) per tau in TEST.FSCORE_THRESH] with s the exact squared distance to the other surface in
    doubled lattice units (include/s3d.h, s3d_voxel_surface_eval; two more launches).
    mesh=True (with or without gt): the marching-cubes mesh of voxels at the iso-level TEST.MESH_THRESH, a closed,
    outward-oriented triangle mesh in the unit cube the grid spans; per sample mesh_counts = (n_verts, n_faces) and only the
    first rows of mesh_verts / mesh_faces (0-based ids) are written; (max_verts, max_faces) = ops.voxel_mesh_bounds(N_VOX)
    (include/s3d.h, s3d_voxel_mesh; one more launch).
    curves=True (needs gt): the threshold-free evaluation of voxels against gt in K = TEST.CURVE_BINS probability bins; per
    sample occ_hist = [voxels with gt = 0 per bin, voxels with gt != 0 per bin, sum q(v) per bin] and occ_loss = [sum q(BCE),
    sum q(Brier)], q(x) = round-half-even(x * 2^20): the IoU and precision-recall curves at the thresholds k / K, the
    calibration and the test losses follow from them (include/s3d.h, s3d_occupancy_curves; one more launch).
    fscore_curves=True (needs gt and surface=True): dist_hist int64 [B,T,2,K+1], the histogram of the surface points'
    distances over the K = TEST.DIST_BINS edges of dist_edges (unit-cube units) per sample, t and direction, from the same
    kernel that counts surf_stats (include/s3d.h, s3d_voxel_surface_eval_hist; no more launches)."""

    HEAD_OUTPUTS = ('disp_left', 'disp_right', 'voxels')
    GT_OUTPUT = 'iou_counts'
    OPTIONS = ('disp_gt', 'lr_check', 'speckle', 'wls', 'uncertainty', 'camera', 'surface', 'mesh', 'curves', 'fscore_curves')

    def __init__(self, cfg):
        super().__init__(cfg)
        self.decoder = _VoxelDecoder(cfg)
        self.merger = _Merger(cfg)
        assert cfg.NETWORK.MERGER_CHANNELS[0] == cfg.NETWORK.DEC_CHANNELS[-1] + 1

    def _pack_head(self, P, dc, dev):
        for i, seq in enumerate(self.decoder.layers):
            P['dec%d' % i] = PackedConv.from_deconv_k4s2p1(seq[0], seq[1], A.ACT_RELU, dc, dev)
        w = self.decoder.out.weight            # [Cin, 1, 1,1,1]
        nl = len(self.decoder.layers)
        last = P['dec%d' % (nl - 1)]
        # last deconv (8 output channels): one blocked 3x3x3 conv on the plane-scatter kernel + depth-to-space, which
        # also applies the final 1x1x1 transposed conv + sigmoid (coarse volume -> channel 8)
        self._d2s = None
        self._fused_out = False
        row_bytes = last.cin_pad * (4 if dc == A.DTYPE_F32 else 2) * cmult(dc)
        seq = self.decoder.layers[nl - 1]
        if last.cout == 8 and row_bytes in ((64, 128, 256) if self._split else (32, 64, 128)) and self.precision != 'fp32' and \
                not _lib.KNOBS['no_d2s']:
            P['dec%d' % (nl - 1)] = PackedConv.from_deconv_k4s2p1_blocked(seq[0], seq[1], A.ACT_RELU, dc, dev)
            pw = torch.zeros(8, dtype=torch.float32)
            pw[:] = w.detach().float().cpu().view(-1)[:8]
            self._d2s = pw.to(dev)
            self._fused_out = True
        elif self._split:
            raise _lib.S3dError("'bf16x3' needs DEC_CHANNELS[-1] == 8 and DEC_CHANNELS[-2] in (16, 32, 64) (blocked last deconv)")
        elif last.cout_pad == 16 and last.cout < 16 and self.precision != 'tf32x3':     # (a projection epilogue cannot be split)
            self._fused_out = True
            # 1x1x1 transposed conv + sigmoid folded into the last deconv's epilogue: coarse volume -> channel `cout`
            last.set_projection(w.view(-1), last.cout, A.ACT_SIGMOID)
        else:
            P['dec_out'] = PackedConv.from_pointwise(w.view(w.shape[0], 1).t(), None, None, A.ACT_SIGMOID, dc, dev)
        for i, seq in enumerate(self.merger.layers):
            P['mrg%d' % i] = PackedConv.from_conv(seq[0], seq[1], A.ACT_LEAKY, dc, dev,
                                                  act_param=self.cfg.NETWORK.LEAKY_VALUE)

    def forward(self, left, right, gt=None, *, disp_gt=None, lr_check=False, speckle=False, wls=False, uncertainty=False,
                camera=None, surface=False, mesh=False, curves=False, fscore_curves=False):
        left, right, gt, disp_gt, camera, opts = self._check_args(left, right, gt, disp_gt, lr_check, uncertainty, camera,
                                                                  surface, mesh, curves, fscore_curves, speckle, wls)
        mb = int(self.cfg.CONST.get('MICRO_BATCH', 0) or 0)
        B = left.shape[0]
        if mb and B > mb:
            outs = []
            for s in range(0, B, mb):
                o = self._forward_impl(left[s:s + mb], right[s:s + mb], None if gt is None else gt[s:s + mb],
                                       None if disp_gt is None else disp_gt[s:s + mb],
                                       None if camera is None else camera[s:s + mb], opts)
                outs.append(tuple(t.clone() for t in o))
            return tuple(torch.cat(ts, 0) for ts in zip(*outs))
        return self._forward_impl(left, right, gt, disp_gt, camera, opts)

    def _head(self, left, right, gt, disp, opts, out):
        """The voxel head: adds voxels, iou_counts (with gt), surf_stats (surface), the mesh (mesh) and occ_hist / occ_loss
        (curves) to `out`."""
        cfg = self.cfg
        B, H, W = self._bhw(left)
        nv = cfg.CONST.N_VOX
        x = self._latent(left, right, disp)
        L = cfg.NETWORK.LATENT_HW
        k0 = cfg.NETWORK.DEC_CHANNELS[0]
        km = cmult(self._dtype_code())                             # physical channels per logical channel
        assert x.shape[-1] // km * L * L == k0 * 8, 'REC_CHANNELS[-1]*LATENT_HW^2 must equal DEC_CHANNELS[0]*8'
        x = ops.latent_to_vox(x, L, out=self._buf('lat', (2 * B, 2, 2, 2, km * pad_to(k0)), x.dtype, zero=True), split=self._split)
        nl = len(self.decoder.layers)
        for i in range(nl):
            x = self._conv('dec%d' % i, x, out=self._bufo('d%d' % i, 'dec%d' % i, x))
        if self._d2s is not None:
            # x is the blocked output [2B,16,16,16,8 classes x 8]: depth-to-space + coarse-volume projection
            n2, dd, hh, ww, _ = x.shape
            x = ops.depth_to_space(x, 16, self._d2s, A.ACT_SIGMOID, split=self._split,
                                   out=self._buf('d2s', (n2, 2 * dd, 2 * hh, 2 * ww, 16 * km), x.dtype))
        m_in = x                                                   # [2B,32,32,32,16]: ch 0-7 raw, 8 coarse volume, 9.. zero
        split_lo = m_in.shape[-1] // 2 if self._split else 0       # split: [.., hi(16) | lo(16)]
        cm = m_in.shape[-1]
        craw = cfg.NETWORK.DEC_CHANNELS[-1]
        assert m_in.shape[1] == nv and cm > craw
        # coarse volume = sigmoid(1x1x1 transposed conv) lives in channel `craw` of the same buffer: normally
        # produced by the last deconv's fused projection epilogue; otherwise by a pointwise launch (its weights
        # are zero for input channels >= craw, so the in-place write of channel `craw` cannot feed back).
        if not self._fused_out:
            self._conv('dec_out', m_in, out=m_in, out_view=(craw, (nv ** 3 * cm, nv * nv * cm, nv * cm, cm)), cout_store=1)
        s = m_in
        for i in range(len(self.merger.layers)):
            s = self._conv('mrg%d' % i, s, out=self._bufo('m%d' % (i % 2), 'mrg%d' % i, s))
        fused = self._buf('fused', (B, nv ** 3), torch.float32)
        iou = None
        gt8 = None
        if gt is not None:
            th = list(cfg.TEST.VOXEL_THRESH)
            iou = self._buf('iou', (B, len(th), 2), torch.int64)
            iou.zero_()
            gt8 = gt.reshape(B, -1).to(torch.uint8).contiguous()
        ops.fuse_views(s, 0, s.shape[-1], m_in, craw, cm, B, 2, nv ** 3, gt=gt8,
                       thresholds=list(cfg.TEST.VOXEL_THRESH) if gt is not None else None, iou=iou, out=fused,
                       score_lo=s.shape[-1] // 2 if self._split else 0, vol_lo=split_lo)
        out['voxels'] = fused.view(B, nv, nv, nv)
        if gt is not None:
            out['iou_counts'] = iou
        if opts.surface:
            out['surf_stats'], hist = self._surface_stats(fused, gt8, opts.fscore_curves)
            if opts.fscore_curves:
                out['dist_hist'] = hist
        if opts.mesh:
            out['mesh_verts'], out['mesh_faces'], out['mesh_counts'] = self._mesh(fused)
        if opts.curves:
            out['occ_hist'], out['occ_loss'] = self._occupancy_curves(fused, gt8)

    def _occupancy_curves(self, fused, gt8):
        """Probability histograms and loss sums of fused [B,n^3] against gt8 [B,n^3] -> (occ_hist int64 [B,3,K], occ_loss int64
        [B,2]), K = TEST.CURVE_BINS.  The kernel writes every counter (nothing to zero) into workspace buffers: no allocation on
        this path."""
        K, B = curve_bins(self.cfg), fused.shape[0]
        return ops.occupancy_curves(fused, gt8, K, out=(self._buf('occ_hist', (B, 3, K), torch.int64),
                                                        self._buf('occ_loss', (B, 2), torch.int64)))

    def _mesh(self, fused):
        """Marching-cubes mesh of fused [B,n^3] at TEST.MESH_THRESH -> (mesh_verts, mesh_faces, mesh_counts).  Every buffer
        comes from the workspace: no allocation on this path."""
        B, nv = fused.shape[0], self.cfg.CONST.N_VOX
        mv, mf = ops.voxel_mesh_bounds(nv)
        return ops.voxel_mesh(fused, mesh_thresh(self.cfg), out=(self._buf('mesh_verts', (B, mv, 3), torch.float32),
                                                                  self._buf('mesh_faces', (B, mf, 3), torch.int32),
                                                                  self._buf('mesh_counts', (B, 2), torch.int32)))

    def _surface_stats(self, fused, gt8, want_hist=False):
        """Voxel-surface counters of fused [B,n^3] against gt8 [B,n^3] -> (surf_stats int64 [B,T,2,3+F], dist_hist int64
        [B,T,2,K+1] if want_hist else None), both zeroed here (so a graph replay starts from zero) and filled by one call.
        Every buffer comes from the workspace: no allocation on this path."""
        th, fth = list(self.cfg.TEST.VOXEL_THRESH), fscore_thresholds(self.cfg)
        B, nv = fused.shape[0], self.cfg.CONST.N_VOX
        stats = self._buf('surf_stats', (B, len(th), 2, 3 + len(fth)), torch.int64)
        stats.zero_()
        e, hist = None, None
        if want_hist:
            e = dist_edges(self.cfg)
            hist = self._buf('dist_hist', (B, len(th), 2, len(e) + 1), torch.int64).zero_()
        nb = ops.voxel_surface_workspace_bytes(B, len(th), nv)
        ops.voxel_surface_eval(fused, gt8, th, fth, stats, workspace=self._buf('surf_ws', (max(nb, 1),), torch.uint8),
                               edges=e, hist=hist)
        return stats, hist


def unc_thresholds(cfg):
    """TEST.UNC_THRESH as floats: at most 4 (the kernel's limit) standard deviations in input pixels, each finite and >= 0 (a
    pixel with disp_std <= t counts as confident at t); anything else is a ValueError."""
    th = cfg.TEST.get('UNC_THRESH')
    try:
        th = [float(t) for t in th]
    except (TypeError, ValueError):
        raise ValueError('TEST.UNC_THRESH must be a list of numbers, got %r' % (th,)) from None
    if len(th) > 4 or not all(math.isfinite(t) and t >= 0 for t in th):
        raise ValueError('TEST.UNC_THRESH must hold at most 4 finite values >= 0, got %r' % (cfg.TEST.UNC_THRESH,))
    return th


def lr_thresh(cfg):
    """TEST.LR_THRESH as a float: the left-right consistency tolerance in input pixels, finite and >= 0; anything else is a
    ValueError."""
    tau = float(cfg.TEST.LR_THRESH)
    if not (math.isfinite(tau) and tau >= 0):
        raise ValueError('TEST.LR_THRESH must be finite and >= 0, got %r' % cfg.TEST.LR_THRESH)
    return tau


def mesh_thresh(cfg):
    """TEST.MESH_THRESH as a float: the iso-level of the exported mesh, finite and in (0, 1] (a voxel is inside when its
    occupancy is >= it, as for the IoU); anything else is a ValueError."""
    t = cfg.TEST.get('MESH_THRESH')
    try:
        t = float(t)
    except (TypeError, ValueError):
        raise ValueError('TEST.MESH_THRESH must be a number, got %r' % (t,)) from None
    if not (math.isfinite(t) and 0.0 < t <= 1.0) or float(ctypes.c_float(t).value) <= 0.0:
        raise ValueError('TEST.MESH_THRESH must be finite and in (0, 1], got %r' % (cfg.TEST.MESH_THRESH,))
    return t


def speckle_params(cfg):
    """(TEST.SPECKLE_MAX_SIZE, TEST.SPECKLE_MAX_DIFF) of the speckle filter: the largest region (px) that is removed, an int
    >= 0 and not a bool (OpenCV's maxSpeckleSize), and the largest disparity step (input px) inside a region, finite and >= 0
    also in fp32 (StereoSGBM's speckleRange); anything else is a ValueError."""
    n, t = cfg.TEST.get('SPECKLE_MAX_SIZE'), cfg.TEST.get('SPECKLE_MAX_DIFF')
    if not (isinstance(n, int) and not isinstance(n, bool) and 0 <= n < 2 ** 31):
        raise ValueError('TEST.SPECKLE_MAX_SIZE must be an int >= 0, got %r' % (n,))
    try:
        t = float(t)
    except (TypeError, ValueError):
        raise ValueError('TEST.SPECKLE_MAX_DIFF must be a number, got %r' % (t,)) from None
    if isinstance(cfg.TEST.SPECKLE_MAX_DIFF, bool) or not (math.isfinite(t) and t >= 0) or \
            not math.isfinite(ctypes.c_float(t).value):
        raise ValueError('TEST.SPECKLE_MAX_DIFF must be finite and >= 0, got %r' % (cfg.TEST.SPECKLE_MAX_DIFF,))
    return n, t


def wls_params(cfg):
    """(TEST.WLS_LAMBDA, TEST.WLS_SIGMA) of the WLS filter: the smoothness weight lambda and the colour scale sigma of the
    edge weights exp(-|colour difference| / sigma) in 8-bit colour units (OpenCV's DisparityWLSFilter lambda and
    sigmaColor), each a number (not a bool), finite and > 0 also in fp32; anything else is a ValueError."""
    out = []
    for key in ('WLS_LAMBDA', 'WLS_SIGMA'):
        v = cfg.TEST.get(key)
        try:
            t = float(v)
        except (TypeError, ValueError):
            raise ValueError('TEST.%s must be a number, got %r' % (key, v)) from None
        if isinstance(v, bool) or not (math.isfinite(t) and t > 0) or not (math.isfinite(ctypes.c_float(t).value) and
                                                                             ctypes.c_float(t).value > 0):
            raise ValueError('TEST.%s must be finite and > 0, got %r' % (key, v))
        out.append(t)
    return tuple(out)


def cloud_min_disp(cfg):
    """TEST.CLOUD_MIN_DISP as a float: the smallest disparity + doffs (input px) a stereo cloud back-projects, which bounds
    the depth at f * baseline / CLOUD_MIN_DISP; finite and > 0 (also in fp32); anything else is a ValueError."""
    t = cfg.TEST.get('CLOUD_MIN_DISP')
    try:
        t = float(t)
    except (TypeError, ValueError):
        raise ValueError('TEST.CLOUD_MIN_DISP must be a number, got %r' % (t,)) from None
    if not (math.isfinite(t) and t > 0) or float(ctypes.c_float(t).value) <= 0.0:
        raise ValueError('TEST.CLOUD_MIN_DISP must be finite and > 0, got %r' % (cfg.TEST.CLOUD_MIN_DISP,))
    return t


def cloud_max_std(cfg):
    """TEST.CLOUD_MAX_STD as a float: with uncertainty=True a stereo cloud keeps only the pixels whose disparity standard
    deviation is <= it (input px); finite and >= 0; anything else is a ValueError."""
    t = cfg.TEST.get('CLOUD_MAX_STD')
    try:
        t = float(t)
    except (TypeError, ValueError):
        raise ValueError('TEST.CLOUD_MAX_STD must be a number, got %r' % (t,)) from None
    if not (math.isfinite(t) and t >= 0):
        raise ValueError('TEST.CLOUD_MAX_STD must be finite and >= 0, got %r' % (cfg.TEST.CLOUD_MAX_STD,))
    return t


def camera_values(cfg):
    """CONST.CAMERA as 5 floats (f, cx, cy, baseline, doffs): 4 or 5 finite numbers (doffs defaults to 0) with f > 0 and
    baseline > 0, the camera the test driver and runner.py hand to forward(..., camera=); anything else is a ValueError."""
    c = cfg.CONST.get('CAMERA')
    try:
        c = [float(v) for v in c]
    except (TypeError, ValueError):
        raise ValueError('CONST.CAMERA must be a list of numbers (f, cx, cy, baseline[, doffs]), got %r' % (c,)) from None
    if len(c) not in (4, 5) or not all(math.isfinite(v) for v in c) or not (c[0] > 0 and c[3] > 0):
        raise ValueError('CONST.CAMERA must hold 4 or 5 finite numbers (f, cx, cy, baseline[, doffs]) with f > 0 and '
                         'baseline > 0, got %r' % (cfg.CONST.CAMERA,))
    return c + [0.0] * (5 - len(c))


def curve_bins(cfg):
    """TEST.CURVE_BINS: the bins of the threshold-free occupancy evaluation, an int (not a bool) that is a power of two in
    [2, 1024] (the curves are exact at the thresholds k / CURVE_BINS); anything else is a ValueError."""
    k = cfg.TEST.get('CURVE_BINS')
    if not (isinstance(k, int) and not isinstance(k, bool) and 2 <= k <= 1024 and k & (k - 1) == 0):
        raise ValueError('TEST.CURVE_BINS must be an int, a power of two in [2, 1024], got %r' % (k,))
    return k


def dist_edges(cfg):
    """The edges of the nearest-neighbour distance histograms (fscore_curves=True): e_k = fp32(TEST.DIST_MAX * k /
    TEST.DIST_BINS) for k = 1..DIST_BINS, computed in fp64 and rounded once -> float32 numpy array.  DIST_BINS must be an int
    (not a bool) in [1, 1024] and DIST_MAX finite and > 0, and the rounded edges must be finite, > 0 and strictly
    increasing; anything else is a ValueError."""
    K, dmax = cfg.TEST.get('DIST_BINS'), cfg.TEST.get('DIST_MAX')
    if not (isinstance(K, int) and not isinstance(K, bool) and 1 <= K <= 1024):
        raise ValueError('TEST.DIST_BINS must be an int in [1, 1024], got %r' % (K,))
    try:
        dmax = float(dmax)
    except (TypeError, ValueError):
        raise ValueError('TEST.DIST_MAX must be a number, got %r' % (dmax,)) from None
    if not (math.isfinite(dmax) and dmax > 0):
        raise ValueError('TEST.DIST_MAX must be finite and > 0, got %r' % (cfg.TEST.DIST_MAX,))
    with np.errstate(over='ignore'):                          # an edge beyond fp32 becomes inf: rejected below
        e = np.array([dmax * k / K for k in range(1, K + 1)], dtype=np.float64).astype(np.float32)
    if not (np.isfinite(e).all() and (e > 0).all() and (np.diff(e) > 0).all()):
        raise ValueError('TEST.DIST_MAX = %r over TEST.DIST_BINS = %d gives edges that are not finite, > 0 and strictly '
                         'increasing in fp32' % (cfg.TEST.DIST_MAX, K))
    return e


def fscore_thresholds(cfg):
    """TEST.FSCORE_THRESH as floats: at most 8 (the kernel's limit) Euclidean distances in the points' units, each finite
    and > 0; anything else is a ValueError."""
    th = cfg.TEST.get('FSCORE_THRESH')
    try:
        th = [float(t) for t in th]
    except (TypeError, ValueError):
        raise ValueError('TEST.FSCORE_THRESH must be a list of numbers, got %r' % (th,)) from None
    if len(th) > 8 or not all(math.isfinite(t) and t > 0 for t in th):
        raise ValueError('TEST.FSCORE_THRESH must hold at most 8 finite distances > 0, got %r' % (cfg.TEST.FSCORE_THRESH,))
    return th


class Stereo2Point(_StereoBase):
    """forward(left, right[, gt][, disp_gt=][, lr_check=][, speckle=][, wls=][, uncertainty=][, camera=]) -> (disp_left,
    disp_right, points [B,N_POINTS,3][, point_stats int64 [B,2,3+T]][, disp_stats int64 [B,2,2+T']][, lr_mask, lr_stats]
    [, speckle_mask, speckle_stats][, wls_left, wls_right, wls_stats][, disp_std, unc_stats][, cloud_xyz, cloud_rgb,
    cloud_counts][, dist_hist]) (disp_gt, lr_check, speckle, wls, uncertainty, camera and their outputs as for
    Stereo2Voxel: the stereo clouds are the dense counterpart of the decoder's points).  gt: fp32 [B,M,3] GT point cloud; with it the same forward runs the Chamfer search of
    `points` against it and counts, per sample and direction (0: predicted -> GT, 1: GT -> predicted), [sum of squared
    distances and sum of distances in 2^-32 units, points out of range, points closer than t for t in TEST.FSCORE_THRESH]
    (include/s3d.h, s3d_chamfer_eval).  fscore_curves=True (needs gt): dist_hist int64 [B,2,K+1], the histogram of the
    points' nearest-neighbour distances over the K = TEST.DIST_BINS edges of dist_edges per sample and direction, from the
    same kernel that counts point_stats (include/s3d.h, s3d_chamfer_eval_hist; no more launches)."""

    HEAD_OUTPUTS = ('disp_left', 'disp_right', 'points')
    GT_OUTPUT = 'point_stats'
    OPTIONS = ('disp_gt', 'lr_check', 'speckle', 'wls', 'uncertainty', 'camera', 'fscore_curves')

    def __init__(self, cfg):
        super().__init__(cfg)
        self.point_decoder = _PointDecoder(cfg)

    def _check_gt(self, gt, left):
        """GT point cloud of (checked) inputs `left`: fp32 [B,M,3], M >= 1, on their device."""
        if gt is None:
            return None
        B = left.shape[0]
        if not isinstance(gt, torch.Tensor):
            raise ValueError('gt must be a tensor, got %s' % type(gt).__name__)
        if gt.dim() != 3 or gt.shape[0] != B or gt.shape[1] < 1 or gt.shape[2] != 3:
            raise ValueError('expected gt of shape [%d, M, 3], got %s' % (B, tuple(gt.shape)))
        if gt.dtype != torch.float32:
            raise ValueError('gt must be float32, got %s' % gt.dtype)
        if gt.device != left.device:
            raise ValueError('gt must be on %s (the images\' device), got %s' % (left.device, gt.device))
        return gt.contiguous()

    def _pack_head(self, P, dc, dev):
        pd = self.point_decoder
        c, L = self.cfg.NETWORK.REC_CHANNELS[-1], self.cfg.NETWORK.LATENT_HW
        P['pt_conv'] = PackedConv.from_conv(pd.conv[0], pd.conv[1], A.ACT_RELU, dc, dev)
        P['pt_fc1'] = PackedConv.from_linear_over_map(pd.fc1, 2 * c, L // 2, L // 2, A.ACT_RELU, dc, dev)
        P['pt_fc2'] = PackedConv.from_pointwise(pd.fc2.weight, pd.fc2.bias, None, A.ACT_TANH, dc, dev, act_param=0.5)

    def forward(self, left, right, gt=None, *, disp_gt=None, lr_check=False, speckle=False, wls=False, uncertainty=False,
                camera=None, mesh=False, curves=False, fscore_curves=False):
        return self._forward_impl(*self._check_args(left, right, gt, disp_gt, lr_check, uncertainty, camera, False, mesh,
                                                    curves, fscore_curves, speckle, wls))

    def _head(self, left, right, gt, disp, opts, out):
        """The point head: adds points and point_stats (with gt) to `out`."""
        cfg = self.cfg
        B = left.shape[0]
        x = self._latent(left, right, disp)
        L = cfg.NETWORK.LATENT_HW
        if x.shape[2] != L or x.shape[3] != L:
            x = ops.avg_pool(x, L, out=self._buf('pool', (2 * B, 1, L, L, x.shape[-1]), x.dtype), split=self._split)
        c = x.shape[-1]
        cat = self._buf('latcat', (B, 1, L, L, 2 * c), x.dtype)
        if self._split:                    # [hi(left, right) | lo(left, right)]
            h = c // 2
            cat[..., :h].copy_(x[:B, ..., :h]);  cat[..., h:c].copy_(x[B:, ..., :h])
            cat[..., c:c + h].copy_(x[:B, ..., h:]);  cat[..., c + h:].copy_(x[B:, ..., h:])
        else:
            cat[..., :c].copy_(x[:B])          # channel concat of the two views' latents (tiny copy)
            cat[..., c:].copy_(x[B:])
        y = self._conv('pt_conv', cat, out=self._bufo('p0', 'pt_conv', cat))
        y = self._conv('pt_fc1', y, out=self._bufo('p1', 'pt_fc1', y))
        npts = cfg.CONST.N_POINTS
        pts = self._buf('pts', (B, 1, 1, 1, pad_to(npts * 3)), torch.float32)
        self._conv('pt_fc2', y, out=pts)
        points = pts.view(B, -1)[:, :npts * 3].reshape(B, npts, 3)
        out['points'] = points
        if gt is not None:
            out['point_stats'], hist = self._point_stats(points, gt, opts.fscore_curves)
            if opts.fscore_curves:
                out['dist_hist'] = hist

    def _point_stats(self, points, gt, want_hist=False):
        """Chamfer search of points [B,N,3] against gt [B,M,3] + the metric counters -> (point_stats int64 [B,2,3+T],
        dist_hist int64 [B,2,K+1] if want_hist else None), both zeroed here (so a graph replay starts from zero) and filled
        by one call.  Every buffer comes from the workspace: no allocation on this path."""
        th = fscore_thresholds(self.cfg)
        B, N, M = points.shape[0], points.shape[1], gt.shape[1]
        if not points.is_contiguous():                 # the fc2 output row is padded: copy the points out of it
            points = self._buf('pts_xyz', (B, N, 3), torch.float32).copy_(points)
        stats = self._buf('point_stats', (B, 2, 3 + len(th)), torch.int64)
        stats.zero_()
        e, hist = None, None
        if want_hist:
            e = dist_edges(self.cfg)
            hist = self._buf('dist_hist', (B, 2, len(e) + 1), torch.int64).zero_()
        nb = ops.chamfer_workspace_bytes(B, N, M)
        ops.chamfer_eval(points, gt, th, stats, workspace=self._buf('cd_ws', (nb,), torch.uint8) if nb else None,
                         out=(self._buf('cd_d1', (B, N), torch.float32), self._buf('cd_d2', (B, M), torch.float32),
                              self._buf('cd_i1', (B, N), torch.int32), self._buf('cd_i2', (B, M), torch.int32)),
                         edges=e, hist=hist)
        return stats, hist


def build_model(name, cfg, seed=None):
    m = {'Stereo2Voxel': Stereo2Voxel, 'Stereo2Point': Stereo2Point}[name](cfg)
    if seed is not None:
        init_synthetic_weights(m, seed)
    return m.eval()
