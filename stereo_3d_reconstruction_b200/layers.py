# -*- coding: utf-8 -*-
"""Host-side layer packing for the implicit-GEMM conv engine (s3d_conv_igemm / s3d_conv_direct).

At weight-load time every conv-like layer is folded and packed ONCE (SURVEY.md 8(f).1):
  * eval-mode BatchNorm is folded into the weights (scale) and a fp32 bias (shift);
  * weights are re-laid out as [class*taps][Cout_pad][Cin_pad] (K-major rows, what the TMA box of
    the B operand reads) in the compute dtype;
  * the tap table (input offset per tap) is built: ordinary convs, the 8 sub-pixel classes of a
    stride-2 ConvTranspose3d(k4,p1), 1x1x1 transposed convs, and Linear layers seen as a conv whose
    taps cover the whole input map.
The forward then has zero layout work: one C-ABI call per layer.
"""
import ctypes
import os
import itertools

import torch

from . import lib as _lib

PAD = 16   # channel padding granule (bf16: 32 B rows = one UMMA K step)


def pad_to(c, m=PAD):
    return (c + m - 1) // m * m


def torch_dtype(code):
    return torch.float32 if code == _lib.DTYPE_F32 else torch.bfloat16


def is_split(code):
    return code == _lib.DTYPE_BF16X2


def cmult(code):
    """Physical channels per logical channel: split (BF16X2) tensors are [hi(C) | lo(C)]."""
    return 2 if code == _lib.DTYPE_BF16X2 else 1


def to_storage(w, code):
    """fp32 [..., C] -> the storage form of `code`: fp32, bf16, or the bf16 pair [hi(C) | lo(C)] with hi = bf16(w),
    lo = bf16(w - hi) (include/s3d.h, S3D_DTYPE_BF16X2)."""
    if code == _lib.DTYPE_F32:
        return w.float()
    hi = w.to(torch.bfloat16)
    if code == _lib.DTYPE_BF16:
        return hi
    lo = (w.float() - hi.float()).to(torch.bfloat16)
    return torch.cat([hi, lo], -1)


def from_storage(t, code):
    """Inverse of to_storage (fp32 values of a stored tensor)."""
    if code != _lib.DTYPE_BF16X2:
        return t.float()
    c = t.shape[-1] // 2
    return t[..., :c].float() + t[..., c:].float()


def _fold_bn(w_out_first, bias, bn):
    """w_out_first: weight with the output channel as dim 0.  Returns folded (w, bias) in fp32."""
    w = w_out_first.detach().float()
    cout = w.shape[0]
    b = bias.detach().float() if bias is not None else torch.zeros(cout, device=w.device)
    if bn is not None:
        scale = bn.weight.detach().float() / torch.sqrt(bn.running_var.detach().float() + bn.eps)
        shift = bn.bias.detach().float() - bn.running_mean.detach().float() * scale
        w = w * scale.view(-1, *([1] * (w.dim() - 1)))
        b = b * scale + shift
    return w, b


def _choose_tile(N, oD, oH, oW, sx, sy, sz):
    """(tw, th, td, tn): powers of two, product 128, minimising padded work; ties -> wide tw."""
    best = None
    for lw, lh, ld in itertools.product(range(8), repeat=3):
        ln = 7 - lw - lh - ld
        if ln < 0:
            continue
        tw, th, td, tn = 1 << lw, 1 << lh, 1 << ld, 1 << ln
        if tw * sx > 256 or th * sy > 256 or td * sz > 256:
            continue
        waste = (-(-oW // tw) * tw) * (-(-oH // th) * th) * (-(-oD // td) * td) * (-(-N // tn) * tn)
        key = (waste, -lw, -lh, -ld)
        if best is None or key < best[0]:
            best = (key, (tw, th, td, tn))
    return best[1]


def _choose_bn(cout_pad, m_tiles=None, n_sms=148):
    """GEMM N tile of the generic engine: the widest divisor of Cout (<= 256) -- unless that leaves most of the chip idle:
    with few M tiles (small batches: dec0 at batch 1 is ONE 128-row tile x 8 classes streaming 134 MB of weights) the tile
    is narrowed until there are about as many tiles as SMs, so that the weight stream is spread over all of them."""
    divs = [bn for bn in range(min(256, cout_pad), 15, -16) if cout_pad % bn == 0]
    if not divs:
        raise ValueError('no N tile for Cout=%d' % cout_pad)
    if m_tiles is None:
        return divs[0]
    for bn in divs:
        if m_tiles * (cout_pad // bn) >= n_sms * 3 // 4:
            return bn
    return divs[-1]


# ---- constant-region skip of the plane-scatter kernel (include/s3d.h dz_nref, csrc/conv_scatter.cuh Item) ------------
# A column is a 32 x 8 pixel patch of one volume marching over the D planes.  Its output planes [zs, zs + J] repeat: the
# kernel marches the input planes dz_march(zs, J, D) and stores out plane zs J more times.  These functions mirror the
# kernel's arithmetic so that the schedule (and the tests) can reason about it without a GPU.

plane_counter = None      # int64 CUDA tensor [1] or None: every conv launch ADDS the input planes its scatter CTAs marched


def dz_first(col, N, nref, oH, oW, c):
    """First output plane of the repeating run of column `col` (conv_scatter.cuh dz_first); 0 for an empty column."""
    cy, cx = -(-oH // 32), -(-oW // 8)
    if col >= N * cy * cx:
        return 0
    n, x0 = col // (cy * cx), (col % cx) * 8
    xr = min(x0 + 7, oW - 1) if n < nref else oW - 1 - x0
    return xr + c + 2


def dz_jump(zs, D, e):
    """Planes skipped by a run starting at zs: the largest multiple of 3 <= (D - 2 - e) - zs (0 below 3)."""
    ze = D - 2 - e
    return (ze - zs) // 3 * 3 if ze - zs >= 3 else 0


def dz_march(zs, J, D):
    """Input planes a work item marches, in order (conv_scatter.cuh next_plane)."""
    out, p = [], 0
    while p < D:
        out.append(p)
        p = p + 1 + J if p == zs + 1 else p + 1
    return out


def dz_schedule(N, nref, oH, oW, D, c, e, npairs):
    """Pairing + balance table of the CTA pairs (include/s3d.h dz_sched) -> (int32 list, planes marched per pair).

    Partners issue the same MMAs, so they walk the intersection of their runs: columns are sorted by their first repeating
    plane and paired neighbour by neighbour (equal runs except at group borders; an odd column gets an empty partner).
    The pairs of columns are then dealt out longest first, each to the least loaded CTA pair."""
    total = N * -(-oH // 32) * -(-oW // 8)
    first = [dz_first(k, N, nref, oH, oW, c) for k in range(total)]
    cols = sorted(range(total), key=lambda k: (first[k], k))
    items = [(cols[i], cols[i + 1] if i + 1 < total else total) for i in range(0, total, 2)]
    cost = [D - dz_jump(max(first[a], first[b] if b < total else 0), D, e) for a, b in items]
    load, lists = [0] * npairs, [[] for _ in range(npairs)]
    for i in sorted(range(len(items)), key=lambda i: (-cost[i], i)):
        q = min(range(npairs), key=lambda q: (load[q], q))
        load[q] += cost[i]
        lists[q].append(items[i])
    offs, ent = [0], []
    for lst in lists:
        offs.append(offs[-1] + len(lst))
        for a, b in lst:
            ent += [a, b]
    return offs + ent, load


class PackedConv:
    """One folded + packed conv-like layer.  `taps`: list (per class) of lists of (dz,dy,dx)."""

    def __init__(self, w_rows, bias, taps, stride, out_mult, cin, cout, act, act_param, dtype_code, device,
                 ksize=(1, 1, 1), pad=(0, 0, 0)):
        # w_rows: fp32 [n_classes*ntaps, cout, cin]
        self._ctor = (w_rows.detach().float().cpu(), bias.detach().float().cpu(), taps, stride, out_mult, cin,
                      cout, act, act_param, dtype_code, device, tuple(ksize), tuple(pad))      # for derive()
        self.n_classes = len(taps)
        self.ntaps = len(taps[0])
        assert self.n_classes * self.ntaps <= _lib.S3D_MAX_TAPS
        self.cin, self.cout = cin, cout
        self.cin_pad, self.cout_pad = pad_to(cin), pad_to(cout)
        self.stride = stride              # (sz, sy, sx)
        self.out_mult = out_mult          # (omz, omy, omx)
        self.act, self.act_param = act, float(act_param)
        self.dtype_code = dtype_code
        wp = torch.zeros(self.n_classes * self.ntaps, self.cout_pad, self.cin_pad, dtype=torch.float32)
        wp[:, :cout, :cin] = w_rows.cpu()
        self.weight = to_storage(wp, dtype_code).to(device).contiguous()      # split: [rows, Cout_pad, hi(Cin_pad) | lo(Cin_pad)]
        bp = torch.zeros(self.cout_pad, dtype=torch.float32)
        bp[:cout] = bias.cpu()
        self.bias = bp.to(device)
        self.taps = taps
        self.ksize, self.pad = tuple(ksize), tuple(pad)
        # stride-1 3x3x3 layers with Cout <= 64: the three kz slices stacked on the output side in four rotations for
        # the plane-scatter kernel (csrc/conv_scatter.cuh, include/s3d.h w_nstack)
        self.weight_ns = None
        if tuple(ksize) == (3, 3, 3) and tuple(pad) == (1, 1, 1) and tuple(stride) == (1, 1, 1) and \
                self.n_classes == 1 and self.cout_pad <= 64:
            w3 = wp.view(3, 9, self.cout_pad, self.cin_pad)
            self.weight_ns = to_storage(self.pack_nstack(w3), dtype_code).to(device).contiguous()
        self.bn = _choose_bn(self.cout_pad)
        self.proj = None                 # optional fused 1x1 projection: (fp32[16] device tensor, channel, act)
        self._cache = {}
        # stride-1 3x3 2-D layers with Cout <= 64: a batch of images is a VOLUME whose kz = 0 / 2 weight slices are zero,
        # so the plane-scatter kernel (csrc/conv_scatter.cu: pixel-major, coalesced epilogue, marches over the images
        # of a column without per-image pipeline bubbles) runs them; its zero N blocks are free while N <= 96 (an MMA
        # costs ~51 cycles for its A operand anyway).  `vol` is the 27-tap twin of this layer.
        self.vol = None
        row_bytes = self.cin_pad * (4 if dtype_code == _lib.DTYPE_F32 else 2) * cmult(dtype_code)
        if tuple(ksize) == (1, 3, 3) and tuple(pad) == (0, 1, 1) and tuple(stride) == (1, 1, 1) and \
                self.n_classes == 1 and self.cout_pad <= 64 and \
                row_bytes in ((64, 128, 256) if is_split(dtype_code) else (32, 64, 128)) and \
                (not is_split(dtype_code) or self.cout_pad in (16, 32, 64)) and \
                [tuple(t) for t in taps[0]] == [(0, dy, dx) for dy in (-1, 0, 1) for dx in (-1, 0, 1)]:
            w27 = torch.zeros(27, cout, cin, dtype=torch.float32)
            w27[9:18] = w_rows.cpu()
            taps27 = [[(dz, dy, dx) for dz in (-1, 0, 1) for dy in (-1, 0, 1) for dx in (-1, 0, 1)]]
            self.vol = PackedConv(w27, bias, taps27, (1, 1, 1), (1, 1, 1), cin, cout, act, act_param, dtype_code, device,
                                  ksize=(3, 3, 3), pad=(1, 1, 1))

    def derive(self, w_rows, bias, act):
        """The same layer geometry with other weights / bias / activation (used by SplitConv)."""
        _, _, taps, stride, out_mult, cin, cout, _, act_param, dtype_code, device, ksize, pad = self._ctor
        pc = PackedConv(w_rows, bias, taps, stride, out_mult, cin, cout, act, act_param, dtype_code, device, ksize=ksize, pad=pad)
        for k in ('ntaps_algo', 'block_cout'):
            if hasattr(self, k):
                setattr(pc, k, getattr(self, k))
        return pc

    @staticmethod
    def pack_nstack(w3):
        """[3(kz), 9(kyx), Cout_pad, Cin_pad] -> [4, 9, 3*Cout_pad, Cin_pad]: the three kz slices stacked on the output
        side in the four rotations of include/s3d.h (w_nstack): rotation r, block s = W[kz = (r + 1 - s) mod 3]."""
        _, _, co, ci = w3.shape
        ns = torch.zeros(4, 9, 3 * co, ci, dtype=torch.float32)
        for r in range(4):
            for s in range(3):
                if r == 3 and s == 2:
                    continue                      # input plane 0 has no output plane -1
                ns[r, :, s * co:(s + 1) * co] = w3[((r % 3) + 1 - s) % 3]
        return ns.view(36, 3 * co, ci)

    def refonce_weights(self, C):
        """Special weight sets of the reference-once concat kernel (include/s3d.h, s3d_conv_concat_volume_ro) for a 3x3x3 layer
        over [ref(C) | tgt(C)] channels: [3, 9, Cout_pad, C] = [sum_kz W[kz] | -W[kz=0] | -W[kz=2]] on the reference channels."""
        key = ('refonce', C)
        if key not in self._cache:
            assert self.ntaps == 27 and self.n_classes == 1 and self.cin_pad == 2 * C
            w3 = self._ctor[0].view(3, 9, self.cout, self.cin)
            ro = torch.zeros(3, 9, self.cout_pad, C, dtype=torch.float32)
            cr = min(C, self.cin)
            ro[0, :, :self.cout, :cr] = w3[:, :, :, :cr].sum(0)
            ro[1, :, :self.cout, :cr] = -w3[0, :, :, :cr]
            ro[2, :, :self.cout, :cr] = -w3[2, :, :, :cr]
            self._cache[key] = to_storage(ro.view(27, self.cout_pad, C), self.dtype_code).to(self.weight.device).contiguous()
        return self._cache[key]

    def gonce_convs(self, C, pad, w, D):
        """The 2-D map convolutions of the SHEARED form of the concat cost volume + this 3x3x3 layer (bf16, include/s3d.h,
        s3d_concat_gonce_assemble).  With u = x - d (left reference; x + d for the right one) the target half of the volume is
        tgt[y, u] on EVERY disparity plane, so its contribution is a 2-D map G[a, y, u] = sum_{dz,dy,dx,c} W[a, C+c, dz, dy, dx]
        tgt[c, y+dy, u+dx-dz] read at a position that slides with d, and the reference half is the same map P on every plane:
            out[a, d, y, x] = relu(bias + P[y, x] + G[y, x -/+ d])        (+ border-plane and edge-column maps)
        i.e. the layer is a handful of 2-D convolutions (1/14 of its MMAs) plus a streaming pass that writes the volume.
        Returns {'left', 'right': map convs over the zero-margined feature rows of the left / right images
        -> fp32 [B,1,h,w+4,384] = [Psum | -P(dz=-1) | -P(dz=+1) | G | -H(dz=-1) | -H(dz=+1)], map column j <-> u = j - 2;
        'edge_left', 'edge_right': -> fp32 [B,1,h,D,256] = [Ge | +Ge(dz=-1) | +Ge(dz=+1) | 0], the in-plane taps that reach
        past the image edge (x' = w for the left-referenced volumes, -1 for the right-referenced ones): the volume is zero
        there but the sheared map reads a real target pixel}.  Weights are summed in fp32 and rounded to bf16 ONCE (like the
        reference-once kernel's sum over kz): same result as the fused layer up to that rounding and the summation order."""
        key = ('gonce', C, pad, w, D)
        if key in self._cache:
            return self._cache[key]
        assert self.ntaps == 27 and self.n_classes == 1 and self.cin == 2 * C and self.dtype_code in (_lib.DTYPE_BF16, _lib.DTYPE_BF16X2)
        A = self.cout
        Ap = self.cout_pad
        W = self._ctor[0].view(3, 3, 3, A, 2 * C)                 # [kz, ky, kx, a, c]
        Wl, Wr = W[..., :C], W[..., C:]
        dev = self.weight.device
        P = w + 2 * pad
        assert pad >= 2 and pad + w - D + 2 <= 127, 'tap offsets are int8'
        out = {}
        es = (-2, -1, 0, 1, 2)
        for name, sgn in (('left', 1), ('right', -1)):            # left images are the targets of the right-referenced volumes
            rows = torch.zeros(15, 6 * Ap, C)
            for iy in range(3):
                for ie, e in enumerate(es):
                    r = rows[iy * 5 + ie]
                    if -1 <= e <= 1:                              # reference maps: plain 3x3, dx = e
                        r[0 * Ap:0 * Ap + A] = Wl[:, iy, e + 1].sum(0)
                        r[1 * Ap:1 * Ap + A] = -Wl[0, iy, e + 1]
                        r[2 * Ap:2 * Ap + A] = -Wl[2, iy, e + 1]
                    for kz in range(3):                           # target maps: tap (dz, dx) lands on e = dx + sgn * dz
                        dx = e - sgn * (kz - 1)
                        if -1 <= dx <= 1:
                            r[3 * Ap:3 * Ap + A] += Wr[kz, iy, dx + 1]
                            if kz == 0:
                                r[4 * Ap:4 * Ap + A] -= Wr[kz, iy, dx + 1]
                            if kz == 2:
                                r[5 * Ap:5 * Ap + A] -= Wr[kz, iy, dx + 1]
            taps = [[(0, dy, e + pad - 2) for dy in (-1, 0, 1) for e in es]]
            out[name + '_geom'] = (pad - 4, 5, w + 4)             # (input column of output column 0 / tap 0, taps per row, output width)
            out[name] = PackedConv(rows, torch.zeros(6 * Ap), taps, (1, 1, 1), (1, 1, 1), C, 6 * Ap, _lib.ACT_NONE, 0.0,
                                   self.dtype_code, dev, ksize=(1, 3, P - (w + 4) + 1), pad=(0, 1, 0))
            # edge column: left-referenced volumes (targets = RIGHT images, sgn = -1): x = w-1, dx = +1, u = w-1-d;
            #              right-referenced volumes (targets = LEFT images, sgn = +1): x = 0, dx = -1, u = d
            dxe = -1 if name == 'left' else 1
            rows = torch.zeros(9, 4 * Ap, C)                      # 4th block zero: s3d_map_conv works in chunks of 128 channels
            for iy in range(3):
                for kz in range(3):
                    e = dxe + sgn * (kz - 1)                      # left images: e in {-2,-1,0}; right images: e in {0,1,2}
                    ie = e + 2 if name == 'left' else e
                    r = rows[iy * 3 + ie]
                    r[0:A] -= Wr[kz, iy, dxe + 1]
                    if kz == 0:
                        r[Ap:Ap + A] += Wr[kz, iy, dxe + 1]
                    if kz == 2:
                        r[2 * Ap:2 * Ap + A] += Wr[kz, iy, dxe + 1]
            # output column j <-> u = j (left images) / u = w - D + j (right images); strip tap ie reads u + ie - 2 / u + ie
            off = (pad - 2) if name == 'left' else (pad + w - D)
            taps = [[(0, dy, ie + off) for dy in (-1, 0, 1) for ie in range(3)]]
            out['edge_' + name + '_geom'] = (off, 3, D)
            out['edge_' + name] = PackedConv(rows, torch.zeros(4 * Ap), taps, (1, 1, 1), (1, 1, 1), C, 4 * Ap, _lib.ACT_NONE, 0.0,
                                             self.dtype_code, dev, ksize=(1, 3, P - D + 1), pad=(0, 1, 0))
        self._cache[key] = out
        return out

    # ---- constructors ------------------------------------------------------------------
    @classmethod
    def from_conv(cls, conv, bn, act, dtype_code, device, act_param=0.0):
        """nn.Conv2d / nn.Conv3d, odd kernel, symmetric padding, stride 1 or 2."""
        w, b = _fold_bn(conv.weight, conv.bias, bn)
        if w.dim() == 4:
            w = w.unsqueeze(2)
            ks, st, pd = (1,) + tuple(conv.kernel_size), (1,) + tuple(conv.stride), (0,) + tuple(conv.padding)
        else:
            ks, st, pd = tuple(conv.kernel_size), tuple(conv.stride), tuple(conv.padding)
        cout, cin = w.shape[0], w.shape[1]
        taps, rows = [], []
        for kz, ky, kx in itertools.product(range(ks[0]), range(ks[1]), range(ks[2])):
            taps.append((kz - pd[0], ky - pd[1], kx - pd[2]))
            rows.append(w[:, :, kz, ky, kx])
        return cls(torch.stack(rows), b, [taps], st, (1, 1, 1), cin, cout, act, act_param, dtype_code, device,
                   ksize=ks, pad=pd)

    @classmethod
    def from_deconv_k4s2p1(cls, deconv, bn, act, dtype_code, device, act_param=0.0):
        """nn.ConvTranspose3d(k=4, s=2, p=1): out o = 2i - 1 + k.  Output parity a uses, per dim,
        a=0: (input offset 0, k=1), (-1, k=3);  a=1: (+1, k=0), (0, k=2)."""
        assert tuple(deconv.kernel_size) == (4, 4, 4) and tuple(deconv.stride) == (2, 2, 2) and \
            tuple(deconv.padding) == (1, 1, 1) and tuple(deconv.output_padding) == (0, 0, 0)
        w, b = _fold_bn(deconv.weight.transpose(0, 1), deconv.bias, bn)   # -> [Cout, Cin, 4,4,4]
        cout, cin = w.shape[0], w.shape[1]
        per_dim = {0: [(0, 1), (-1, 3)], 1: [(1, 0), (0, 2)]}
        taps, rows = [], []
        for cz, cy, cx in itertools.product(range(2), repeat=3):      # class index = cz*4 + cy*2 + cx
            ct = []
            for (oz, kz), (oy, ky), (ox, kx) in itertools.product(per_dim[cz], per_dim[cy], per_dim[cx]):
                ct.append((oz, oy, ox))
                rows.append(w[:, :, kz, ky, kx])
            taps.append(ct)
        return cls(torch.stack(rows), b, taps, (1, 1, 1), (2, 2, 2), cin, cout, act, act_param, dtype_code, device)

    @classmethod
    def from_deconv_k4s2p1_blocked(cls, deconv, bn, act, dtype_code, device, act_param=0.0):
        """The same transposed conv as ONE stride-1 3x3x3 conv over the INPUT grid with 8*Cout output channels: channel
        (class, co) of input position j is output voxel 2j + class (class = (cz,cy,cx) parity) -- a depth-to-space
        layout.  Each class uses 2 of the 3 offsets per dimension, so 8 of its 27 taps are non-zero; as a dense
        3x3x3 layer it runs on the plane-scatter kernel (every input plane fetched once, N = 3*8*Cout) instead of
        8 classes x 8 re-fetched taps in the generic engine.  ops.depth_to_space() restores [.., 2d, 2h, 2w, C]."""
        assert tuple(deconv.kernel_size) == (4, 4, 4) and tuple(deconv.stride) == (2, 2, 2) and \
            tuple(deconv.padding) == (1, 1, 1) and tuple(deconv.output_padding) == (0, 0, 0)
        w, b = _fold_bn(deconv.weight.transpose(0, 1), deconv.bias, bn)   # -> [Cout, Cin, 4,4,4]
        cout, cin = w.shape[0], w.shape[1]
        kof = {0: {0: 1, -1: 3}, 1: {1: 0, 0: 2}}                    # parity -> {input offset: kernel index}
        taps, rows = [], []
        for dz, dy, dx in itertools.product((-1, 0, 1), repeat=3):
            m = torch.zeros(8 * cout, cin, dtype=w.dtype)
            for cz, cy, cx in itertools.product(range(2), repeat=3):
                if dz in kof[cz] and dy in kof[cy] and dx in kof[cx]:
                    c = (cz * 2 + cy) * 2 + cx
                    m[c * cout:(c + 1) * cout] = w[:, :, kof[cz][dz], kof[cy][dy], kof[cx][dx]]
            taps.append((dz, dy, dx))
            rows.append(m)
        pc = cls(torch.stack(rows), b.repeat(8), [taps], (1, 1, 1), (1, 1, 1), cin, 8 * cout, act, act_param, dtype_code,
                 device, ksize=(3, 3, 3), pad=(1, 1, 1))
        pc.ntaps_algo = 8                                          # non-zero taps per output channel (for flops())
        pc.block_cout = cout
        return pc

    @classmethod
    def from_pointwise(cls, w_out_in, bias, bn, act, dtype_code, device, act_param=0.0):
        """1x1(x1) conv / transposed conv given as a [Cout, Cin] matrix."""
        w, b = _fold_bn(w_out_in, bias, bn)
        return cls(w.unsqueeze(0), b, [[(0, 0, 0)]], (1, 1, 1), (1, 1, 1), w.shape[1], w.shape[0], act, act_param,
                   dtype_code, device)

    @classmethod
    def from_linear_over_map(cls, linear, C, h, w_, act, dtype_code, device, act_param=0.0):
        """nn.Linear over a flattened NCHW map [C,h,w] == conv with h*w taps, no padding, 1x1 output."""
        w, b = _fold_bn(linear.weight, linear.bias, None)
        w = w.view(w.shape[0], C, h, w_)
        taps, rows = [], []
        for y, x in itertools.product(range(h), range(w_)):
            taps.append((0, y, x))
            rows.append(w[:, :, y, x])
        return cls(torch.stack(rows), b, [taps], (1, 1, 1), (1, 1, 1), C, w.shape[0], act, act_param, dtype_code,
                   device, ksize=(1, h, w_), pad=(0, 0, 0))

    def set_projection(self, w_vec, channel, act):
        """Fuse a 1x1 projection of this layer's (activated) outputs into channel `channel` of its own output
        (include/s3d.h, proj_w).  Needs a single 16-channel accumulator group."""
        assert self.cout_pad == 16 and self.cout <= channel < 16, (self.cout_pad, self.cout, channel)
        v = torch.zeros(16, dtype=torch.float32)
        v[:self.cout] = w_vec.detach().float().cpu().flatten()[:self.cout]
        self.proj = (v.to(self.weight.device), int(channel), int(act))
        self._cache = {}
        return self

    # ---- launch ------------------------------------------------------------------------
    def out_grid(self, iD, iH, iW):
        """Logical output grid per class for an input of the given size."""
        if self.n_classes == 8:
            return iD, iH, iW
        return tuple((i + 2 * p - k) // s + 1 for i, k, p, s in zip((iD, iH, iW), self.ksize, self.pad, self.stride))

    def params(self, N, iD, iH, iW, out_strides, out_dtype_code, cout_store=None, os_lo=0, region=None):
        key = (N, iD, iH, iW, tuple(out_strides), out_dtype_code, cout_store, os_lo, region)
        p = self._cache.get(key)
        if p is not None:
            return p
        oD, oH, oW = self.out_grid(iD, iH, iW)
        p = _lib.S3dConvParams()
        p.N, p.iD, p.iH, p.iW, p.Cin = N, iD, iH, iW, self.cin_pad
        p.oD, p.oH, p.oW, p.Cout = oD, oH, oW, self.cout_pad
        p.sz, p.sy, p.sx = self.stride
        p.ntaps, p.n_classes = self.ntaps, self.n_classes
        i = 0
        for ct in self.taps:
            for (dz, dy, dx) in ct:
                p.dz[i], p.dy[i], p.dx[i] = dz, dy, dx
                i += 1
        p.osN, p.osD, p.osH, p.osW = out_strides[:4]
        p.osC = out_strides[4] if len(out_strides) > 4 else 1
        p.os_lo = os_lo
        p.omz, p.omy, p.omx = self.out_mult
        p.cout_store = self.cout_pad if cout_store is None else cout_store
        p.in_dtype, p.out_dtype = self.dtype_code, out_dtype_code
        p.act, p.act_param = self.act, self.act_param
        p.tw, p.th, p.td, p.tn = _choose_tile(N, oD, oH, oW, self.stride[2], self.stride[1], self.stride[0])
        m_tiles = self.n_classes * -(-oW // p.tw) * -(-oH // p.th) * -(-oD // p.td) * -(-N // p.tn)
        p.bn = _choose_bn(self.cout_pad, m_tiles)
        p.w_nstack = self.weight_ns.data_ptr() if self.weight_ns is not None else None
        if self.proj is not None:
            p.proj_w, p.proj_channel, p.proj_act = self.proj[0].data_ptr(), self.proj[1], self.proj[2]
        if region is not None:
            # the table lives as long as the cached params (built once per shape: graph replay reuses it)
            p.dz_nref, p.dz_c, p.dz_e = region
            dev = self.weight.device
            ncols = N * -(-oH // 32) * -(-oW // 8)
            p.dz_pairs = max(1, min(torch.cuda.get_device_properties(dev).multi_processor_count // 2, -(-ncols // 2)))
            table, _ = dz_schedule(N, p.dz_nref, oH, oW, oD, p.dz_c, p.dz_e, p.dz_pairs)
            sched = torch.tensor(table, dtype=torch.int32).to(dev)
            p.dz_sched, p.dz_sched_keep = sched.data_ptr(), sched
        self._cache[key] = p
        return p

    def __call__(self, x, out=None, residual=None, out_dtype=None, cout_store=None, out_view=None, engine='igemm', dz=None):
        """x: channels-last [N,D,H,W,Cin_pad] contiguous CUDA tensor ([.., hi(Cin_pad) | lo(Cin_pad)] for a split layer).

        dz: None or (nref, c, e): x is N = 2 * nref volumes whose plane z is the same for z in [xr + c, D - 1 - e]
        (include/s3d.h dz_nref; xr = x for the first nref volumes, W - 1 - x for the others).  Only a hint: the
        plane-scatter kernel computes the repeating output planes once, every other engine ignores it.

        out: destination tensor (allocated if None) -- `out_view` optionally gives
        (data_ptr_offset_elems, (osN, osD, osH, osW[, osC])) to write into a channel slice of a wider buffer
        or (osC != 1) a planar layout.  A split (BF16X2) layer writes a split output unless `out` is fp32."""
        cm = cmult(self.dtype_code)
        assert x.is_cuda and x.is_contiguous() and x.dim() == 5 and x.shape[-1] == cm * self.cin_pad, \
            (tuple(x.shape), self.cin_pad)
        assert x.dtype == torch_dtype(self.dtype_code)
        N, iD, iH, iW, _ = x.shape
        oD, oH, oW = self.out_grid(iD, iH, iW)
        m = self.out_mult
        odt = x.dtype if out_dtype is None else out_dtype
        if out is None:
            out = torch.empty((N, oD * m[0], oH * m[1], oW * m[2], self.cout_pad * (cm if odt == torch.bfloat16 else 1)),
                              dtype=odt, device=x.device)
        if out.dtype == torch.float32:
            code = _lib.DTYPE_F32
        else:
            code = _lib.DTYPE_BF16X2 if is_split(self.dtype_code) else _lib.DTYPE_BF16
        if self._halo2d_ok(x, out, residual, cout_store, out_view, engine):
            return self._call_halo2d(x, out, residual, out_view)
        if self.vol is not None and engine == 'igemm' and iD == 1 and self.proj is None and \
                (out_view is None or len(out_view[1]) == 4) and (out.dtype == x.dtype or not is_split(self.dtype_code)) and not _lib.KNOBS['no_vol2d'] and not _lib.KNOBS['no_scatter']:
            return self._call_as_volume(x, out, residual, cout_store, out_view)
        if out_view is None:
            assert out.is_contiguous() and out.dim() == 5
            C = out.shape[-1]
            strides = (out.shape[1] * out.shape[2] * out.shape[3] * C, out.shape[2] * out.shape[3] * C,
                       out.shape[3] * C, C)
            off = 0
            if cout_store is None:
                cout_store = min(self.cout_pad, C)
            if code == _lib.DTYPE_BF16X2:
                assert C == 2 * self.cout_pad, 'split output: [.., hi(Cout_pad) | lo(Cout_pad)]'
            os_lo = 0                                   # = Cout_pad
        else:
            off, strides = out_view[:2]
            os_lo = out_view[2] if len(out_view) > 2 else 0
            assert code != _lib.DTYPE_BF16X2 or os_lo > 0, 'a split output view needs its hi -> lo offset'
        p = self.params(N, iD, iH, iW, strides, code, cout_store, os_lo, dz)
        p.dz_planes = None if plane_counter is None else plane_counter.data_ptr()
        L = _lib.load()
        fn = L.s3d_conv_igemm if engine == 'igemm' else L.s3d_conv_direct
        esz = out.element_size()
        rptr = None
        if residual is not None:
            assert residual.dtype == out.dtype and residual.shape == out.shape and residual.is_contiguous()
            rptr = residual.data_ptr() + off * esz
        rc = fn(ctypes.byref(p), x.data_ptr(), self.weight.data_ptr(), self.bias.data_ptr(), rptr,
                out.data_ptr() + off * esz, torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, 's3d_conv_%s' % engine)
        _lib.count_launch()
        return out

    def _halo2d_ok(self, x, out, residual, cout_store, out_view, engine):
        """Stride-1 3x3 2-D layers, bf16, 32 / 64 channels in and out, ReLU or no activation: the halo-once engine
        (csrc/conv2d_halo.cu; A/B knob no_conv2d_halo falls back to the plane-scatter / generic engines).  Measured per 128
        images: conv3 0.078 -> 0.037 ms, conv4 (residual) 0.084 -> 0.056, conv5 0.056 -> 0.035 (64 x 64 pixels), conv1
        (32 -> 32 channels, 128 x 128 pixels: 18 small MMAs per tile) 0.078 -> 0.074."""
        return (engine == 'igemm' and x.shape[1] == 1 and self.dtype_code == _lib.DTYPE_BF16 and out.dtype == torch.bfloat16 and
                self.ksize == (1, 3, 3) and self.pad == (0, 1, 1) and tuple(self.stride) == (1, 1, 1) and self.n_classes == 1 and
                self.cin_pad in (32, 64) and self.cout_pad in (32, 64) and
                self.act in (_lib.ACT_NONE, _lib.ACT_RELU) and
                self.proj is None and (cout_store is None or cout_store == self.cout_pad) and
                (out_view is None or (len(out_view[1]) == 4 and (len(out_view) < 3 or not out_view[2]))) and
                [tuple(t) for t in self.taps[0]] == [(0, dy, dx) for dy in (-1, 0, 1) for dx in (-1, 0, 1)] and
                not _lib.KNOBS['no_conv2d_halo'] and not _lib.KNOBS['no_scatter'])

    def _call_halo2d(self, x, out, residual, out_view):
        N, _, H, W, _ = x.shape
        if out_view is None:
            assert out.is_contiguous() and out.dim() == 5 and out.shape[-1] >= self.cout_pad
            Co = out.shape[-1]
            off, sN, sH, sW = 0, out.shape[2] * out.shape[3] * Co, out.shape[3] * Co, Co
        else:
            off, (sN, _, sH, sW) = out_view[:2]
        rptr = None
        if residual is not None:
            assert residual.dtype == out.dtype and residual.shape == out.shape and residual.is_contiguous()
            rptr = residual.data_ptr() + off * 2
        rc = _lib.load().s3d_conv2d_halo(x.data_ptr(), self.weight.data_ptr(), self.bias.data_ptr(), rptr, out.data_ptr() + off * 2,
                                         N, H, W, self.cin_pad, self.cout_pad, sN, sH, sW, int(self.act == _lib.ACT_RELU),
                                         torch.cuda.current_stream().cuda_stream)
        _lib.check(rc, 's3d_conv2d_halo')
        _lib.count_launch()
        return out

    def _call_as_volume(self, x, out, residual, cout_store, out_view):
        """Run a batch of images [N,1,H,W,C] through the 27-tap twin as G volumes of N/G planes (see __init__)."""
        N, _, H, W, C = x.shape
        patches = -(-H // 32) * -(-W // 8)                     # columns per volume in conv_scatter.cu
        # G volumes of N/G images: minimise waves x (planes per column + pipeline fill/drain), 148 columns per wave
        G = min((g for g in range(1, N + 1) if N % g == 0),
                key=lambda g: (-(-g * patches // 148) * (N // g + 2), g))
        Dv = N // G
        if out_view is None:
            assert out.is_contiguous() and out.dim() == 5
            Co = out.shape[-1]
            sN, sH, sW = out.shape[2] * out.shape[3] * Co, out.shape[3] * Co, Co
            off = 0
            if cout_store is None:
                cout_store = min(self.cout_pad, Co)
            os_lo = self.cout_pad
        else:
            off, (sN, _, sH, sW) = out_view[:2]
            os_lo = out_view[2] if len(out_view) > 2 else 0
        self.vol(x.view(G, Dv, H, W, C), out=out, residual=residual, cout_store=cout_store,
                 out_view=(off, (Dv * sN, sN, sH, sW), os_lo))
        return out

    def flops(self, N, iD, iH, iW):
        """Algorithmic (unpadded) FLOPs: 2 * outputs * Cout * Cin * taps-that-hit."""
        oD, oH, oW = self.out_grid(iD, iH, iW)
        return 2.0 * N * oD * oH * oW * self.n_classes * self.cout * self.cin * getattr(self, 'ntaps_algo', self.ntaps)


class SplitConv:
    """'tf32x3' precision: fp32 accuracy from TF32 tensor cores.  Weights and activations are split into a part that is
    exactly representable in TF32 and the remainder (w = w_hi + w_lo, x = x_hi + x_lo; include/s3d.h, s3d_split_tf32), and

        conv(x, w) ~= conv(x_hi, w_hi) + conv(x_lo, w_hi) + conv(x_hi, w_lo)            (the lo*lo term is ~2^-22)

    runs as three passes of the same kernels, accumulating in fp32 IN the output tensor through the engines' residual
    input (pass 1 adds the layer's own residual; bias and activation are applied by pass 3 only)."""

    def __init__(self, pc):
        assert pc.dtype_code == _lib.DTYPE_F32 and pc.proj is None
        w, b = pc._ctor[0], pc._ctor[1]
        w_hi = (w.view(torch.int32) & -8192).view(torch.float32)          # clear the low 13 mantissa bits
        self.full = pc                                                     # geometry, flops()
        self.hi = pc.derive(w_hi, torch.zeros_like(b), _lib.ACT_NONE)
        self.lo = pc.derive(w - w_hi, b, pc.act)
        for k in ('cin', 'cout', 'cin_pad', 'cout_pad', 'ksize', 'stride', 'pad', 'n_classes', 'out_mult', 'act', 'act_param',
                  'dtype_code', 'weight', 'bias', 'proj'):
            setattr(self, k, getattr(pc, k))

    def out_grid(self, *a):
        return self.full.out_grid(*a)

    def flops(self, *a):
        return self.full.flops(*a)

    def __call__(self, x, out=None, residual=None, engine='igemm', **kw):
        from . import ops
        assert engine == 'igemm' and x.dtype == torch.float32
        x_hi, x_lo = ops.split_tf32(x)
        out = self.hi(x_hi, out=out, residual=residual, **kw)
        self.hi(x_lo, out=out, residual=out, **kw)
        self.lo(x_hi, out=out, residual=out, **kw)
        return out
