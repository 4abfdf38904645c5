"""Reference statement of the threshold-free occupancy evaluation (include/s3d.h, s3d_occupancy_curves; core/test.py,
curves_block / curves_summary) in numpy.  The histogram follows the definitions voxel by voxel; the curves are computed from
the voxels themselves, not from a histogram: the IoU by thresholding v >= k / K directly, AP by sorting the voxels by bin."""
import numpy as np

FX20 = 1 << 20
FX32 = 1 << 32


def clamp(fused):
    """NaN -> 0, then [0, 1], in fp32."""
    v = np.nan_to_num(np.asarray(fused, np.float32), nan=0.0, posinf=1.0, neginf=0.0)
    return np.clip(v, np.float32(0), np.float32(1)).astype(np.float32)


def bins(v, K):
    """k = min(floor(v * K), K - 1), v * K in fp32 (exact for a power of two K)."""
    return np.minimum(np.floor(v * np.float32(K)).astype(np.int64), K - 1)


def q20(x):
    return np.rint(np.asarray(x, np.float64) * FX20).astype(np.int64)


def losses(v, g):
    """Per-voxel BCE (PyTorch's clamp at log = -100, fp64 log of the fp32 value; 1 - v in fp64) and squared error."""
    v = v.astype(np.float64)
    x = np.where(g, v, 1.0 - v)
    with np.errstate(divide='ignore'):
        bce = -np.maximum(np.log(x), -100.0)
    return bce, (v - g) ** 2


def occupancy_curves(fused, gt, K):
    """fused float [B, ...], gt [B, ...] (nonzero = occupied) -> (hist int64 [B,3,K], loss int64 [B,2])."""
    B = fused.shape[0]
    v = clamp(fused).reshape(B, -1)
    g = np.asarray(gt).reshape(B, -1) != 0
    hist = np.zeros((B, 3, K), np.int64)
    loss = np.zeros((B, 2), np.int64)
    for b in range(B):
        k = bins(v[b], K)
        hist[b, 0] = np.bincount(k[~g[b]], minlength=K)
        hist[b, 1] = np.bincount(k[g[b]], minlength=K)
        np.add.at(hist[b, 2], k, q20(v[b]))
        bce, sq = losses(v[b], g[b])
        loss[b] = [q20(bce).sum(), q20(sq).sum()]
    return hist, loss


def iou_direct(v, g, t):
    """IoU of (v >= t) against g; 1 when both are empty."""
    p = v >= np.float32(t)
    u = (p | g).sum()
    return (p & g).sum() / u if u else 1.0


def curves_block(fused, gt, K):
    """The driver's curves block [4K + 2] of one batch, with the per-sample IoUs from direct thresholding."""
    B = fused.shape[0]
    hist, loss = occupancy_curves(fused, gt, K)
    v = clamp(fused).reshape(B, -1)
    g = np.asarray(gt).reshape(B, -1) != 0
    miou = [sum(int(np.rint(np.float64(iou_direct(v[b], g[b], k / K)) * FX32)) for b in range(B)) for k in range(K)]
    return np.concatenate([hist.sum(0).reshape(-1), loss.sum(0), np.array(miou, np.int64)])


def average_precision(v, g, K):
    """AP of the voxels ranked by their bin (ties share a rank): walk the voxels sorted by bin, descending, and add the
    precision at each new recall level where the bin changes.  None when nothing is occupied."""
    G = int(g.sum())
    if G == 0:
        return None
    k = bins(v, K)
    order = np.argsort(-k, kind='stable')
    ks, gs = k[order], g[order]
    ap, tp, prev_r = 0.0, 0, 0.0
    for i in range(len(ks)):
        tp += int(gs[i])
        if i + 1 == len(ks) or ks[i + 1] != ks[i]:                # end of a tie group: one point of the curve
            r = tp / G
            ap += (r - prev_r) * (tp / (i + 1))
            prev_r = r
    return ap


def summary(fused, gt, K):
    """The statistics of curves_summary over all voxels of the batch, from the voxels themselves."""
    B = fused.shape[0]
    v = clamp(fused).reshape(-1)
    g = np.asarray(gt).reshape(-1) != 0
    vb = clamp(fused).reshape(B, -1)
    gb = np.asarray(gt).reshape(B, -1) != 0
    bce, sq = losses(v, g)
    M = min(K, 16)
    m = bins(v, K) // (K // M)
    ece = sum(abs(v[m == i].astype(np.float64).sum() - g[m == i].sum()) for i in range(M)) / v.size
    return {'iou': [iou_direct(v, g, k / K) for k in range(K)],
            'mean_iou': [np.mean([iou_direct(vb[b], gb[b], k / K) for b in range(B)]) for k in range(K)],
            'ap': average_precision(v, g, K), 'bce': bce.mean(), 'brier': sq.mean(), 'ece': ece}
