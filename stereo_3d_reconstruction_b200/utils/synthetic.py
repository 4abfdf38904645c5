# -*- coding: utf-8 -*-
"""Synthetic inputs of the config.py shape (StereoShapeNet is unavailable offline; BASELINE.json
north_star and SURVEY.md 8(d) 'synthetic data')."""
import torch


def stereo_pair(B, H, W, max_disp_px, seed=0, device='cpu'):
    """left = uniform noise in [0,1]; right = left shifted left by a per-row-constant integer disparity
    in [0, max_disp_px) (so that left[y, x] == right[y, x - d(y)]) -- a non-degenerate soft-argmin target."""
    g = torch.Generator().manual_seed(seed)
    left = torch.rand(B, 3, H, W, generator=g)
    d = torch.randint(0, max(1, max_disp_px), (B, H), generator=g)
    xs = torch.arange(W).view(1, 1, W) + d.view(B, H, 1)            # right[x] = left[x + d]
    valid = xs < W
    xs = xs.clamp(max=W - 1)
    right = torch.gather(left, 3, xs.unsqueeze(1).expand(B, 3, H, W))
    right = right * valid.unsqueeze(1)
    return left.to(device), right.to(device), d.to(device)


def disparity_gt(d, H, W):
    """GT disparity fp32 [B,2,H,W] of a stereo_pair with per-row disparity d [B,H], in the orientation of the models'
    disp_left / disp_right; NaN where a pixel has no match in the other view:
      view 0 (left-referenced):  left[y, x] == right[y, x - d], valid where x - d >= 0;
      view 1 (right-referenced): right[y, x] == left[y, x + d], valid where x + d < W (stereo_pair zeroes the other pixels)."""
    B = d.shape[0]
    assert tuple(d.shape) == (B, H)
    dd = d.to(torch.float32).view(B, H, 1).expand(B, H, W)
    x = torch.arange(W, device=d.device).view(1, 1, W)
    dv = d.view(B, H, 1)
    nan = torch.full_like(dd, float('nan'))
    return torch.stack([torch.where(x - dv >= 0, dd, nan), torch.where(x + dv < W, dd, nan)], 1)


def gt_volume(B, n_vox=32, p=0.1, seed=1, device='cpu'):
    g = torch.Generator().manual_seed(seed)
    return (torch.rand(B, n_vox, n_vox, n_vox, generator=g) < p).to(torch.uint8).to(device)


def point_clouds(B, N, M, seed=2, duplicates=False, device='cpu'):
    """Uniform points in [-0.5,0.5]^3.  duplicates=True repeats a block of points inside both sets so that
    exact ties exercise the lowest-index rule."""
    g = torch.Generator().manual_seed(seed)
    a = torch.rand(B, N, 3, generator=g) - 0.5
    b = torch.rand(B, M, 3, generator=g) - 0.5
    if duplicates:
        k = max(1, M // 8)
        b[:, M - k:] = b[:, :k]
        ka = max(1, N // 8)
        a[:, N - ka:] = a[:, :ka]
        b[:, k:2 * k][:, :min(k, ka)] = a[:, :min(k, ka)]
    return a.to(device), b.to(device)
