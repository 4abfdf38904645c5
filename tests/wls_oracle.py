"""Confidence-weighted WLS filter (s3d_disp_wls, include/s3d.h) in plain numpy float32, vectorised across the lines of a pass:
every operation a single fp32 rounding (numpy float32 neither contracts to FMA nor flushes denormals), so the kernels' maps
and counters must equal these bit for bit."""
import numpy as np

from tests.cloud_oracle import colour

f32 = np.float32


def weights(colours, lut):
    """Edge weights of guides with 8-bit colours [N,H,W,3] -> (wh fp32 [N,H,W-1] between (y,x) and (y,x+1), wv fp32
    [N,H-1,W] between (y,x) and (y+1,x)): lut[s], s the summed squared colour difference."""
    c = np.asarray(colours).astype(np.int64)
    sh = ((c[:, :, 1:] - c[:, :, :-1]) ** 2).sum(-1)
    sv = ((c[:, 1:] - c[:, :-1]) ** 2).sum(-1)
    lut = np.asarray(lut, f32)
    return lut[sh], lut[sv]


def solve_lines(f, c, k):
    """One pass over independent lines: f, c fp32 [L,n] (the two streams), k fp32 [L,n-1] the coupling coefficients ->
    (U(f), U(c)) by the Thomas elimination of include/s3d.h with g_{-1} = y_{-1} = 0."""
    L, n = f.shape
    z = np.zeros(L, f32)
    kl, g, yf, yc = z, z, z, z
    G, YF, YC = np.empty((L, n), f32), np.empty((L, n), f32), np.empty((L, n), f32)
    for i in range(n):
        kr = k[:, i] if i < n - 1 else z
        den = ((f32(1) + kl) + kr) - kl * g
        r = f32(1) / den
        g = kr * r
        yf = (f[:, i] + kl * yf) * r
        yc = (c[:, i] + kl * yc) * r
        G[:, i], YF[:, i], YC[:, i] = g, yf, yc
        kl = kr
    uf, uc = YF.copy(), YC.copy()
    for i in range(n - 2, -1, -1):
        uf[:, i] = YF[:, i] + G[:, i] * uf[:, i + 1]
        uc[:, i] = YC[:, i] + G[:, i] * uc[:, i + 1]
    return uf, uc


def lambdas(lam):
    """lam_t = fp32(lambda * 0.25^t), t = 0, 1, 2, computed in fp64."""
    return [f32(float(f32(lam)) * 0.25 ** t) for t in range(3)]


def filter_maps(d, colours, lut, lam, mask=None):
    """Maps d fp32 [N,H,W] with their guides' 8-bit colours [N,H,W,3] (cloud_oracle.colour) -> (out fp32 [N,H,W], conf bool
    [N,H,W])."""
    d = np.asarray(d, f32)
    N, H, W = d.shape
    conf = np.isfinite(d)
    if mask is not None:
        conf &= np.asarray(mask) == 1
    f = np.where(conf, d, f32(0)).astype(f32)
    c = conf.astype(f32)
    wh, wv = weights(colours, lut)
    with np.errstate(over='ignore', under='ignore'):
        for lt in lambdas(lam):
            f, c = (u.reshape(N, H, W) for u in solve_lines(f.reshape(N * H, W), c.reshape(N * H, W),
                                                             (lt * wh).reshape(N * H, W - 1)))
            tr = lambda a: np.ascontiguousarray(a.transpose(0, 2, 1))
            f, c = (tr(u.reshape(N, W, H)) for u in solve_lines(tr(f).reshape(N * W, H), tr(c).reshape(N * W, H),
                                                                tr(lt * wv).reshape(N * W, H - 1)))
        with np.errstate(invalid='ignore', divide='ignore'):
            out = np.where(c > 0, f / np.where(c > 0, c, f32(1)), f32(np.nan)).astype(f32)
    return out, conf


def disp_wls(disp, B, left, right, lut, lam, mask=None, disp_gt=None, thresholds=(), max_gt=None):
    """-> (out fp32 [2B,H,W], stats int64 [B,2,4+T]) of include/s3d.h, s3d_disp_wls.  left / right: uint8 HWC [B,H,W,3] or
    fp32 NCHW [B,3,H,W]."""
    disp = np.asarray(disp, f32)
    H, W = disp.shape[1:]
    left, right = np.asarray(left), np.asarray(right)
    u8 = left.dtype == np.uint8
    T = len(thresholds)
    cols = np.stack([colour(img[b], u8) for img in (left, right) for b in range(B)])      # view-major, as disp
    m = None if mask is None else np.asarray(mask).transpose(1, 0, 2, 3).reshape(2 * B, H, W)
    out, conf = filter_maps(disp, cols, lut, lam, m)
    stats = np.zeros((B, 2, 4 + T), np.int64)
    for v in range(2):
        for b in range(B):
            o = out[v * B + b]
            fin = np.isfinite(o)
            stats[b, v, 0] = fin.sum()
            stats[b, v, 3 + T] = conf[v * B + b].sum()
            if disp_gt is not None:
                g = np.asarray(disp_gt[b, v], f32)
                with np.errstate(invalid='ignore', over='ignore'):
                    valid = fin & np.isfinite(g) & (g >= 0) & (g < f32(max_gt))
                    e = np.abs(o - g).astype(f32)
                e = np.where(valid, e, f32(0))
                stats[b, v, 1] = valid.sum()
                stats[b, v, 2] = np.rint(e.astype(np.float64) * 65536.0).astype(np.int64).sum()
                for t, th in enumerate(thresholds):
                    stats[b, v, 3 + t] = (valid & (e > f32(th))).sum()
    return out, stats
