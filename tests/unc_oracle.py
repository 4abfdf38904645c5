"""Reference statement of the disparity uncertainty (test infrastructure): the soft-argmin mean and standard deviation in fp64
from a cost tensor, and the confidence-filtered counters of s3d_upsample_disp_eval (include/s3d.h) in plain numpy fp32, whose
integers the kernel must equal exactly when both see the same disparity and standard-deviation maps."""
import numpy as np
import torch

from tests.disp_oracle import disp_error_counts


def soft_argmin_moments(cost, sign=-1.0, axis=-3):
    """cost [..., D, h, w] (planes along `axis`) -> (mu, sigma) fp64 numpy: p_d = softmax_d(sign * cost_d),
    mu = sum p_d d, sigma = sqrt(sum p_d (d - mu)^2)."""
    c = np.moveaxis(np.asarray(cost.detach().cpu().numpy() if torch.is_tensor(cost) else cost, dtype=np.float64), axis, -1)
    v = sign * c
    e = np.exp(v - v.max(-1, keepdims=True))
    p = e / e.sum(-1, keepdims=True)
    d = np.arange(c.shape[-1], dtype=np.float64)
    mu = (p * d).sum(-1)
    sigma = np.sqrt((p * (d - mu[..., None]) ** 2).sum(-1))
    return mu, sigma


def unc_counts(disp, disp_std, unc_thresh, gt=None, thresholds=(), max_gt=None):
    """disp, disp_std fp32 [..., 2, H, W] as the forward returns them.  Per image and threshold k, the confident pixels are
    those with disp_std <= unc_thresh[k] in fp32 (NaN / inf never are).
    -> counts int64 [..., 2, K, 3 + T]: [n_conf, n_valid_conf, sum_{valid & conf} q(|d - gt|), count_{valid & conf}(|d - gt| > t)
    per t], the last three as in disp_oracle.disp_error_counts (valid, q); zero without gt."""
    s = disp_std.detach().cpu().numpy().astype(np.float32)
    K, T = len(unc_thresh), len(thresholds)
    counts = np.zeros(s.shape[:-2] + (K, 3 + T), dtype=np.int64)
    for k, tau in enumerate(unc_thresh):
        with np.errstate(invalid='ignore'):
            conf = s <= np.float32(tau)
        counts[..., k, 0] = conf.sum((-2, -1))
        if gt is not None:
            g = gt.detach().cpu().numpy().astype(np.float32)
            g = np.where(conf, g, np.float32(np.nan))                     # not confident = not valid
            counts[..., k, 1:] = disp_error_counts(disp.detach().cpu(), torch.from_numpy(g), thresholds, max_gt).numpy()
    return torch.from_numpy(counts)
