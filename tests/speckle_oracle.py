"""numpy / scipy statement of s3d_speckle_filter (include/s3d.h): candidates, 4-neighbour adjacency in float32, connected
components with scipy.sparse.csgraph, the mask and the per-(sample, view) counters."""
import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

f32 = np.float32


def regions(disp, B, max_diff, lr_mask=None):
    """disp fp32 [2B,H,W] (view-major) -> (cand bool [B,2,H,W], label int [B,2,H,W] of the connected component of every
    pixel (non-candidates are components of their own), size int [B,2,H,W] of each pixel's component)."""
    disp = np.asarray(disp, f32)
    H, W = disp.shape[1:]
    d = disp.reshape(2, B, H, W).transpose(1, 0, 2, 3)             # [B,2,H,W]
    cand = np.isfinite(d)
    if lr_mask is not None:
        cand &= np.asarray(lr_mask) == 1
    md = f32(max_diff)
    idx = np.arange(d.size).reshape(d.shape)
    with np.errstate(over='ignore', invalid='ignore'):
        # float32 subtraction: one rounding, as __fsub_rn (an overflow to inf is not adjacent)
        right = cand[..., :, 1:] & cand[..., :, :-1] & (np.abs(d[..., :, 1:] - d[..., :, :-1]) <= md)
        down = cand[..., 1:, :] & cand[..., :-1, :] & (np.abs(d[..., 1:, :] - d[..., :-1, :]) <= md)
    r = np.concatenate([idx[..., :, :-1][right], idx[..., :-1, :][down]])
    c = np.concatenate([idx[..., :, 1:][right], idx[..., 1:, :][down]])
    g = coo_matrix((np.ones(len(r), np.int8), (r, c)), shape=(d.size, d.size))
    _, lab = connected_components(g, directed=False)
    size = np.bincount(lab)[lab]
    return cand, lab.reshape(d.shape), size.reshape(d.shape)


def speckle_filter(disp, B, max_size, max_diff, lr_mask=None, disp_gt=None, thresholds=(), max_gt=None):
    """-> (mask uint8 [B,2,H,W], stats int64 [B,2,5+T]) of include/s3d.h, s3d_speckle_filter."""
    disp = np.asarray(disp, f32)
    H, W = disp.shape[1:]
    T = len(thresholds)
    cand, lab, size = regions(disp, B, max_diff, lr_mask)
    kept = cand & (size > max_size)
    small = cand & (size <= max_size)
    d = disp.reshape(2, B, H, W).transpose(1, 0, 2, 3)
    stats = np.zeros((B, 2, 5 + T), np.int64)
    stats[..., 0] = kept.sum((2, 3))
    if disp_gt is not None:
        g = np.asarray(disp_gt, f32)
        with np.errstate(invalid='ignore', over='ignore'):
            valid = kept & np.isfinite(g) & (g >= 0) & (g < f32(max_gt))
            e = np.abs(d - g)                                         # float32
        e = np.where(valid, e, f32(0))
        stats[..., 1] = valid.sum((2, 3))
        stats[..., 2] = np.where(valid, np.rint(e.astype(np.float64) * 65536.0), 0).astype(np.int64).sum((2, 3))
        for t, th in enumerate(thresholds):
            stats[..., 3 + t] = (valid & (e > f32(th))).sum((2, 3))
    # a region is counted once, at its first pixel; regions never span two maps
    first = np.unique(lab.ravel(), return_index=True)[1]
    img = first // (H * W)
    sm = small.ravel()[first]
    stats.reshape(2 * B, 5 + T)[:, 3 + T] = np.bincount(img[sm], minlength=2 * B)
    stats[..., 4 + T] = small.sum((2, 3))
    return kept.astype(np.uint8), stats
