"""Reference statement of the left-right consistency check (test infrastructure): plain numpy fp32, the rule of
s3d_upsample_disp_eval (include/s3d.h).  The kernel's mask and integers must equal it exactly when both see the same disparity
maps."""
import numpy as np
import torch

from tests.disp_oracle import disp_error_counts


def lr_consistency(disp, tau, gt=None, thresholds=(), max_gt=None):
    """disp fp32 [..., 2, H, W] (view 0 = left-referenced, 1 = right-referenced), as the forward returns them.
    View v, pixel (y, x), d = disp[v, y, x]: not kept unless d is finite; k = round-half-even(d) (np.rint), xo = x - k for
    view 0 and x + k for view 1 (|d| >= W + 1 is out of range); kept iff 0 <= xo < W and |d - disp[1 - v, y, xo]| <= tau in
    fp32 (a NaN there is not kept).
    -> (mask uint8 [..., 2, H, W], counts int64 [..., 2, 3 + T]):
       [n_kept, n_valid_kept, sum_{valid & kept} q(|d - gt|), count_{valid & kept}(|d - gt| > t) per t], the last three as in
       disp_oracle.disp_error_counts (valid, q); zero without gt."""
    d = disp.detach().cpu().numpy().astype(np.float32)
    assert d.shape[-3] == 2
    W = d.shape[-1]
    x = np.arange(W)
    tau = np.float32(tau)
    kept = np.zeros(d.shape, dtype=bool)
    for v, sgn in ((0, -1), (1, 1)):
        dv, do = d[..., v, :, :], d[..., 1 - v, :, :]
        with np.errstate(invalid='ignore'):
            ok = np.abs(dv) < np.float32(W + 1)                            # False for NaN / inf
            k = np.rint(np.where(ok, dv, np.float32(0))).astype(np.int64)
            xo = x + sgn * k
            ok &= (xo >= 0) & (xo < W)
            other = np.take_along_axis(do, np.clip(xo, 0, W - 1), axis=-1)
            ok &= np.abs(dv - other) <= tau                                # fp32 subtraction, one rounding
        kept[..., v, :, :] = ok
    mask = torch.from_numpy(kept.astype(np.uint8))
    T = len(thresholds)
    counts = np.zeros(d.shape[:-2] + (3 + T,), dtype=np.int64)
    counts[..., 0] = kept.sum((-2, -1))
    if gt is not None:
        g = gt.detach().cpu().numpy().astype(np.float32)
        g = np.where(kept, g, np.float32(np.nan))                          # not kept = not valid
        counts[..., 1:] = disp_error_counts(disp.detach().cpu(), torch.from_numpy(g), thresholds, max_gt).numpy()
    return mask, torch.from_numpy(counts)
