"""Reference statement of the voxel-surface counters (test infrastructure): plain numpy + scipy, the definition of
s3d_voxel_surface_eval (include/s3d.h).  The kernel's counters must equal it exactly.

Surface of an occupancy grid [n,n,n] = the centres of the faces between an occupied and an empty voxel (outside the grid is
empty), in doubled integer coordinates: a voxel centre is 2i+1, a face is at an even coordinate on its axis."""
import math

import numpy as np
from scipy.spatial import cKDTree

FX = 2.0 ** 32


def faces(occ):
    """occ bool [n,n,n] -> int64 [P,3] doubled coordinates of its surface points (axis order as the array's)."""
    occ = np.asarray(occ, dtype=bool)
    n = occ.shape[0]
    p = np.zeros((n + 2,) * 3, dtype=np.int8)
    p[1:-1, 1:-1, 1:-1] = occ
    pts = []
    for ax in range(3):
        d = np.diff(p, axis=ax) != 0                      # face between padded cells c and c + 1 along ax: index c = 0..n
        sl = [slice(1, -1)] * 3
        sl[ax] = slice(None)
        idx = np.argwhere(d[tuple(sl)]).astype(np.int64)
        c = 2 * idx + 1
        c[:, ax] -= 1                                     # the face's own axis: even 2c
        pts.append(c)
    return np.concatenate(pts)


def nearest_sq(a, b):
    """a [P,3], b [Q,3] int64 sites -> int64 [P] squared distance of each a to its nearest b (None when b is empty); the
    match comes from a KD-tree, the value is recomputed exactly from the integer coordinates."""
    if len(b) == 0:
        return None
    if len(a) == 0:
        return np.zeros(0, dtype=np.int64)
    _, j = cKDTree(b).query(a)
    return ((a - b[j]) ** 2).sum(1)


def kbound(tau, n):
    """F-score threshold tau (unit-cube units) -> k: a point counts when s < k, i.e. sqrt(s) / (2n) < tau."""
    return min(math.ceil((2 * n * float(tau)) ** 2), 3 * (2 * n) ** 2 + 1)


def _q_sqrt(s):
    return np.rint(np.sqrt(s.astype(np.float32)).astype(np.float64) * FX).astype(np.int64)


def direction_counts(a, b, ks):
    """Counters of surface a searched in surface b: [n_pts, sum s, sum q(sqrt_rn(s)), count(s < k) per k]."""
    s = nearest_sq(a, b)
    out = np.zeros(3 + len(ks), dtype=np.int64)
    out[0] = len(a)
    if s is None:
        return out
    out[1] = s.sum()
    out[2] = _q_sqrt(s).sum()
    for f, k in enumerate(ks):
        out[3 + f] = (s < k).sum()
    return out


def surface_stats(fused, gt, voxel_thresh, fscore_thresh):
    """fused fp32 [B,n,n,n] (or [B,n^3]), gt [B,...] (nonzero = occupied) -> int64 [B,T,2,3+F]: per sample, threshold t and
    direction (0: predicted -> GT, 1: GT -> predicted) the counters of direction_counts."""
    fused = np.asarray(fused, dtype=np.float32)
    B = fused.shape[0]
    n = round(fused[0].size ** (1 / 3))
    fused = fused.reshape(B, n, n, n)
    gt = np.asarray(gt).reshape(B, n, n, n) != 0
    ks = [kbound(t, n) for t in fscore_thresh]
    out = np.zeros((B, len(voxel_thresh), 2, 3 + len(ks)), dtype=np.int64)
    for b in range(B):
        fg = faces(gt[b])
        for t, th in enumerate(voxel_thresh):
            with np.errstate(invalid='ignore'):
                fp = faces(fused[b] >= np.float32(th))
            out[b, t, 0] = direction_counts(fp, fg, ks)
            out[b, t, 1] = direction_counts(fg, fp, ks)
    return out


def surface_block(stats, n):
    """stats int64 [B,T,2,3+F] -> int64 [T, 3 + 3F]: per t [n_both, sum_b q(CD_L2_b), sum_b q(CD_L1_b), then per tau
    sum_b q(P_b), sum_b q(R_b), sum_b q(F_b)], q(x) = round-half-even(x * 2^32), in float64 (core/test.py::surface_block)."""
    c = np.asarray(stats).astype(np.float64)
    n0, n1 = c[:, :, 0, 0], c[:, :, 1, 0]
    both = (n0 > 0) & (n1 > 0)
    with np.errstate(invalid='ignore', divide='ignore'):
        l2 = np.where(both, (c[:, :, 0, 1] / n0 + c[:, :, 1, 1] / n1) / (2 * n) ** 2, 0.0)
        l1 = np.where(both, (c[:, :, 0, 2] / n0 + c[:, :, 1, 2] / n1) / 2 / FX / (2 * n), 0.0)
        p = np.where(n0[..., None] > 0, c[:, :, 0, 3:] / n0[..., None], 0.0)
        r = np.where(n1[..., None] > 0, c[:, :, 1, 3:] / n1[..., None], 0.0)
        f = np.where(p + r > 0, 2 * p * r / (p + r), 0.0)

    def q(x):
        return np.rint(x * FX).astype(np.int64).sum(0)
    B, T, F = c.shape[0], c.shape[1], c.shape[3] - 3
    prf = np.stack([q(p), q(r), q(f)], -1).reshape(T, 3 * F)
    return np.concatenate([both.sum(0)[:, None].astype(np.int64), q(l2)[:, None], q(l1)[:, None], prf], 1)
