"""Reference statement of the point-cloud counters (test infrastructure): plain numpy, the rule of s3d_chamfer_eval
(include/s3d.h) applied to the distances of the C oracle (oracle/chamfer.py::chamfer_c).  The kernel's counters must equal
it exactly."""
import numpy as np

from oracle.chamfer import chamfer_c

FX = 2.0 ** 32


def _q(x):
    """round-half-even(x * 2^32) as int64; x float32, the product exact in float64."""
    return np.rint(x.astype(np.float64) * FX).astype(np.int64)


def point_counts(dist1, dist2, thresholds):
    """dist1 [B,N], dist2 [B,M] squared distances (float32) -> int64 [B,2,3+T]: per direction
    [sum q(d), sum q(sqrt_rn(d)), n_out, count(sqrt_rn(d) < t) per t] over the points with d finite and d < 2^8 (the others
    are n_out only); sqrt_rn = np.sqrt on float32 (correctly rounded), the comparison in float32 and strict."""
    T = len(thresholds)
    B = dist1.shape[0]
    out = np.zeros((B, 2, 3 + T), dtype=np.int64)
    for k, d in enumerate((dist1, dist2)):
        d = np.asarray(d, dtype=np.float32)
        with np.errstate(invalid='ignore'):
            ok = np.isfinite(d) & (d < np.float32(256.0))
        d = np.where(ok, d, np.float32(0))
        s = np.sqrt(d)
        out[:, k, 0] = np.where(ok, _q(d), 0).sum(-1)
        out[:, k, 1] = np.where(ok, _q(s), 0).sum(-1)
        out[:, k, 2] = (~ok).sum(-1)
        for t, tau in enumerate(thresholds):
            out[:, k, 3 + t] = (ok & (s < np.float32(tau))).sum(-1)
    return out


def point_stats(xyz1, xyz2, thresholds):
    """xyz1 [B,N,3] predicted, xyz2 [B,M,3] GT (float32 arrays or CPU tensors) -> point_counts of their C-oracle distances
    (a NaN point gets d = +inf there)."""
    d1, d2, _, _ = chamfer_c(np.asarray(xyz1, dtype=np.float32), np.asarray(xyz2, dtype=np.float32))
    return point_counts(d1, d2, thresholds)


def fscore_fx(counts, N, M):
    """counts int64 [B,2,3+T] -> int64 [T]: sum_b round-half-even(F_b * 2^32), F_b = 2 P R / (P + R) (0 when both are 0),
    P = count_pred / N, R = count_gt / M, in float64."""
    c = np.asarray(counts)[:, :, 3:].astype(np.float64)
    p, r = c[:, 0] / N, c[:, 1] / M
    with np.errstate(invalid='ignore'):
        f = np.where(p + r > 0, 2 * p * r / (p + r), 0.0)
    return np.rint(f * FX).astype(np.int64).sum(0)
