"""Reference statement of the nearest-neighbour distance histograms (test infrastructure): plain numpy, the rules of
s3d_chamfer_eval_hist and s3d_voxel_surface_eval_hist (include/s3d.h) applied to the distances of the C Chamfer oracle and
of tests/surface_oracle.py, and the driver's point_curves / surface_curves blocks and summaries written out independently
of core/test.py.  The kernels' histograms must equal it exactly."""
import math

import numpy as np

from oracle.chamfer import chamfer_c
from tests import surface_oracle as SO

FX = 2.0 ** 32


def edges(dist_max, K):
    """e_k = fp32(dist_max * k / K), k = 1..K, computed in fp64 and rounded once."""
    return np.array([float(dist_max) * k / K for k in range(1, K + 1)], dtype=np.float64).astype(np.float32)


def point_bins(d, e):
    """Squared distances d (float32, any shape) -> int64 bins: searchsorted(e, sqrt_rn(d), 'right') for d finite and
    < 2^8, K (= len(e)) for every other point."""
    d = np.asarray(d, dtype=np.float32)
    with np.errstate(invalid='ignore'):
        ok = np.isfinite(d) & (d < np.float32(256.0))
    s = np.sqrt(np.where(ok, d, np.float32(0)))                     # float32 sqrt: correctly rounded
    return np.where(ok, np.searchsorted(np.asarray(e, np.float32), s, side='right'), len(e)).astype(np.int64)


def point_hist_of_dists(dist1, dist2, e):
    """dist1 [B,N], dist2 [B,M] -> int64 [B,2,K+1]."""
    K = len(e)
    B = np.asarray(dist1).shape[0]
    out = np.zeros((B, 2, K + 1), dtype=np.int64)
    for k, d in enumerate((dist1, dist2)):
        bins = point_bins(d, e)
        for b in range(B):
            out[b, k] = np.bincount(bins[b], minlength=K + 1)
    return out


def point_hist(xyz1, xyz2, e):
    """xyz1 [B,N,3] predicted, xyz2 [B,M,3] GT -> int64 [B,2,K+1] of their C-oracle distances."""
    d1, d2, _, _ = chamfer_c(np.asarray(xyz1, dtype=np.float32), np.asarray(xyz2, dtype=np.float32))
    return point_hist_of_dists(d1, d2, e)


def kbounds(e, n):
    """Edges in unit-cube units -> the integer bounds voxel_kbound(e_k, n) of an n^3 grid."""
    return np.array([min(math.ceil((2 * n * float(x)) ** 2), 3 * (2 * n) ** 2 + 1) for x in e], dtype=np.int64)


def surface_hist(fused, gt, voxel_thresh, e):
    """fused fp32 [B,n,n,n] (or [B,n^3]), gt (nonzero = occupied) -> int64 [B,T,2,K+1]: per sample, threshold and direction
    the surface points binned by searchsorted(kbounds, s, 'right'); all in bin K when the other surface is empty."""
    fused = np.asarray(fused, dtype=np.float32)
    B = fused.shape[0]
    n = round(fused[0].size ** (1 / 3))
    fused = fused.reshape(B, n, n, n)
    gt = np.asarray(gt).reshape(B, n, n, n) != 0
    kb = kbounds(e, n)
    K = len(e)
    out = np.zeros((B, len(voxel_thresh), 2, K + 1), dtype=np.int64)

    def one(a, b):
        s = SO.nearest_sq(a, b)
        if s is None:
            h = np.zeros(K + 1, dtype=np.int64)
            h[K] = len(a)
            return h
        return np.bincount(np.searchsorted(kb, s, side='right'), minlength=K + 1)
    for b in range(B):
        fg = SO.faces(gt[b])
        for t, th in enumerate(voxel_thresh):
            with np.errstate(invalid='ignore'):
                fp = SO.faces(fused[b] >= np.float32(th))
            out[b, t, 0] = one(fp, fg)
            out[b, t, 1] = one(fg, fp)
    return out


def _prf(h0, h1, n0, n1):
    """One sample's rows -> float64 [K,3] (P, R, F) at every edge."""
    K = len(h0) - 1
    rows = []
    for k in range(1, K + 1):
        p = sum(int(x) for x in h0[:k]) / n0 if n0 else 0.0
        r = sum(int(x) for x in h1[:k]) / n1 if n1 else 0.0
        f = 2 * p * r / (p + r) if p + r > 0 else 0.0
        rows.append((p, r, f))
    return np.array(rows, dtype=np.float64).reshape(K, 3)


def point_curves_block(hist, N, M):
    """hist int64 [B,2,K+1] -> int64 [2(K+1) + 3K]: summed histograms, then per k sum_b q(P_b), q(R_b), q(F_b)."""
    hist = np.asarray(hist)
    q = sum(np.rint(_prf(h[0], h[1], N, M) * FX).astype(np.int64) for h in hist)
    return np.concatenate([hist.sum(0).reshape(-1), np.asarray(q, dtype=np.int64).reshape(-1)])


def surface_curves_block(hist):
    """hist int64 [B,T,2,K+1] -> int64 [T * (2(K+1) + 3K)], denominators the row sums."""
    hist = np.asarray(hist)
    out = []
    for t in range(hist.shape[1]):
        q = sum(np.rint(_prf(h[0], h[1], int(h[0].sum()), int(h[1].sum())) * FX).astype(np.int64) for h in hist[:, t])
        out.append(np.concatenate([hist[:, t].sum(0).reshape(-1), np.asarray(q, dtype=np.int64).reshape(-1)]))
    return np.concatenate(out)


def curves(h0, h1, prf_sum, e, n):
    """Summary of one block's numbers: summed rows h0 / h1, per-edge sums prf_sum [K,3] (q units), edges e, n samples."""
    K = len(e)
    e = [float(x) for x in e]
    c0, c1 = np.cumsum(h0[:K]), np.cumsum(h1[:K])
    t0, t1 = int(np.sum(h0)), int(np.sum(h1))
    f = [int(x) / FX / n if n else 0.0 for x in prf_sum[:, 2]]

    def first(c, t, frac_num, frac_den):
        for k in range(K):
            if t and c[k] * frac_den >= frac_num * t:
                return e[k]
        return None
    return {'precision': [int(x) / FX / n if n else 0.0 for x in prf_sum[:, 0]],
            'recall': [int(x) / FX / n if n else 0.0 for x in prf_sum[:, 1]], 'fscore': f,
            'pooled_precision': [int(c) / t0 if t0 else 0.0 for c in c0],
            'pooled_recall': [int(c) / t1 if t1 else 0.0 for c in c1],
            'fscore_auc': sum(f) / K,
            'accuracy': {'p50': first(c0, t0, 1, 2), 'p90': first(c0, t0, 9, 10)},
            'completeness': {'p50': first(c1, t1, 1, 2), 'p90': first(c1, t1, 9, 10)}}
