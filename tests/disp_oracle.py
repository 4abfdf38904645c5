"""Reference statement of the disparity evaluation counters (test infrastructure): plain numpy fp32, the same validity rule,
strict '>' and half-even fixed point as s3d_upsample_disp_eval (include/s3d.h).  The kernel's integers must equal it exactly
when both see the same disparity tensor."""
import numpy as np
import torch


def disp_error_counts(disp, gt, thresholds, max_gt):
    """Per image, integer [n_valid, sum_valid q(|disp - gt|), count_valid(|disp - gt| > t) per t].
    disp, gt: fp32 [..., H, W] (same shape).  valid: gt finite and 0 <= gt < max_gt.  e = |disp - gt| in fp32 and
    q(e) = round-half-even(e * 2^16) (the scaling is exact).  Returns int64 [..., 2 + T]."""
    d = disp.detach().cpu().numpy().astype(np.float32)
    g = gt.detach().cpu().numpy().astype(np.float32)
    assert d.shape == g.shape
    with np.errstate(invalid='ignore'):
        valid = np.isfinite(g) & (g >= np.float32(0)) & (g < np.float32(max_gt))
        e = np.abs(d - g)                                                  # fp32 subtraction, one rounding
    e = np.where(valid, e, np.float32(0)).astype(np.float32)
    q = np.rint(e * np.float32(65536)).astype(np.int64)                    # np.rint: round half to even
    ax = (-2, -1)
    cols = [valid.sum(ax).astype(np.int64), q.sum(ax)]
    cols += [(valid & (e > np.float32(t))).sum(ax).astype(np.int64) for t in thresholds]
    return torch.from_numpy(np.stack(cols, -1))
