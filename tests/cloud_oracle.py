"""Stereo point clouds (s3d_disp_cloud, include/s3d.h) in plain numpy float32: every operation a single fp32 rounding, so the
kernel's points, colours and counts must equal these bit for bit."""
import numpy as np

f32 = np.float32


def colour(img, u8):
    """Colours of one image as uint8 [H,W,3]: the bytes of a uint8 HWC image, rint(clamp(v, 0, 1) * 255) with NaN -> 0 of an fp32
    CHW one (fp32 product, round half to even)."""
    img = np.asarray(img)
    if u8:
        return img.astype(np.uint8)
    v = np.nan_to_num(img.astype(f32).transpose(1, 2, 0), nan=0.0, posinf=1.0, neginf=0.0)
    v = np.clip(v, f32(0), f32(1)).astype(f32)
    return np.rint((v * f32(255)).astype(f32)).astype(np.uint8)


def keep_mask(d, doffs, min_disp, mask=None, std=None, max_std=0.0):
    """Kept pixels of one map d fp32 [H,W]."""
    d = np.asarray(d, f32)
    with np.errstate(invalid='ignore', over='ignore'):
        den = (d + f32(doffs)).astype(f32)
        k = np.isfinite(d) & (den >= f32(min_disp))
        if mask is not None:
            k &= np.asarray(mask) == 1
        if std is not None:
            k &= np.asarray(std, f32) <= f32(max_std)
    return k


def points(d, v, cam):
    """Points of all pixels of one map d fp32 [H,W] of view v with cam = (f, cx, cy, baseline, doffs) -> fp32 [H,W,3]."""
    f, cx, cy, bl, doffs = (f32(c) for c in cam)
    d = np.asarray(d, f32)
    H, W = d.shape
    with np.errstate(all='ignore'):
        den = (d + doffs).astype(f32)
        fb = f32(f * bl)
        z = (fb / den).astype(f32)
        s = (z / f).astype(f32)
        xs = np.arange(W, dtype=f32)[None, :]
        ys = np.arange(H, dtype=f32)[:, None]
        X = ((xs - cx).astype(f32) * s).astype(f32)
        if v == 1:
            X = (X + bl).astype(f32)
        Y = ((ys - cy).astype(f32) * s).astype(f32)
    return np.stack([X, np.broadcast_to(Y, X.shape), z], -1).astype(f32)


def disp_cloud(disp, B, left, right, camera, min_disp, lr_mask=None, disp_std=None, max_std=0.0, u8=False):
    """disp fp32 [2B,H,W] view-major, left / right [B,3,H,W] fp32 or [B,H,W,3] uint8, camera [B,5] -> list over samples of
    (xyz fp32 [n,3], rgb uint8 [n,3], (n0, n1))."""
    disp = np.asarray(disp, f32)
    out = []
    for b in range(B):
        xs, cs, ns = [], [], []
        for v, img in ((0, left), (1, right)):
            d = disp[v * B + b]
            k = keep_mask(d, camera[b][4], min_disp, None if lr_mask is None else lr_mask[b, v],
                          None if disp_std is None else disp_std[b, v], max_std)
            xs.append(points(d, v, camera[b])[k])
            cs.append(colour(img[b], u8)[k])
            ns.append(int(k.sum()))
        out.append((np.concatenate(xs).reshape(-1, 3), np.concatenate(cs).reshape(-1, 3), tuple(ns)))
    return out


def read_ply(path):
    """A PLY reader written from the format: parses the header and reads the vertex records it declares."""
    types = {'float': '<f4', 'uchar': 'u1'}
    with open(path, 'rb') as fh:
        assert fh.readline() == b'ply\n'
        props, n = [], None
        while True:
            line = fh.readline().decode('ascii').split()
            if line == ['end_header']:
                break
            if line[0] == 'format':
                assert line[1:] == ['binary_little_endian', '1.0']
            elif line[0] == 'element':
                assert line[1] == 'vertex'
                n = int(line[2])
            elif line[0] == 'property':
                props.append((line[2], types[line[1]]))
        rec = np.frombuffer(fh.read(), dtype=np.dtype(props))
    assert len(rec) == n
    return rec
