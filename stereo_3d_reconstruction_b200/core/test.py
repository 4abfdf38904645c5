# -*- coding: utf-8 -*-
"""Test driver: loop batches -> model forward -> IoU (Stereo2Voxel) / Chamfer (Stereo2Point)
statistics, sharded across ranks with ONE all-reduce of a small stats vector at the end
(SURVEY.md 8(e); the reference's `runner.py --test` path, README.md:91 -- its core/test.py is not
on disk).  Statistics are integer sums so that an N-GPU run is bit-identical to the 1-GPU run:
    per threshold t:  sum_b intersection(b,t), sum_b union(b,t)   (int64)
    n_samples                                                    (int64)
Chamfer: sum_b CD(b) is accumulated in fp64 and reduced as a fixed-point int64 (2^-40 units).
With eval_disp=True the same vector carries, per view (left-referenced, then right-referenced), the disparity counters the
forward computes against the synthetic GT disparity (models.py, _StereoBase._upsample_disp):
    n_valid, sum |disp - gt| in 2^-16 px, count(|disp - gt| > t) per t in TEST.DISP_THRESH   (int64)
With eval_lr=True (needs eval_disp) the left-right consistency counters of the same forwards follow, per view:
    n_kept, n_valid_kept, sum |disp - gt| in 2^-16 px and count(|disp - gt| > t) over the kept valid pixels  (int64)
With eval_speckle=True (needs eval_disp) the speckle-filter counters of the same forwards follow (models.py,
_StereoBase._speckle, after the LR check when eval_lr), per view:
    n_kept, n_valid_kept, sum |disp - gt| in 2^-16 px and count(|disp - gt| > t) over the kept valid pixels, n_speckles,
    n_speckle_px                                                                                     (int64)
With eval_wls=True (needs eval_disp) the WLS-filter counters of the same forwards follow (models.py, _StereoBase._wls,
confident where the speckle / LR mask keeps a pixel when eval_speckle / eval_lr, else where it is finite), per view:
    n_finite, n_valid_finite, sum |wls - gt| in 2^-16 px and count(|wls - gt| > t) over the finite valid pixels, n_conf
                                                                                                     (int64)
With eval_unc=True (needs eval_disp) the uncertainty counters of the same forwards follow, per view, then per threshold k in
TEST.UNC_THRESH (models.py, _StereoBase._upsample_disp):
    n_conf, n_valid_conf, sum |disp - gt| in 2^-16 px and count(|disp - gt| > t) over the confident valid pixels  (int64)
With eval_points=True (test_point) the point-cloud counters of the same forwards come last (models.py,
Stereo2Point._point_stats), per direction (predicted -> GT, then GT -> predicted), then per threshold t in
TEST.FSCORE_THRESH:
    sum q(d), sum q(sqrt d), n_out, count(sqrt d < t) per t                                    (int64)
    sum_b q(F_b(t)),  F_b = 2 P R / (P + R) (0 when both are 0), P = count_pred / N, R = count_gt / M   (int64)
with q(x) = round-half-even(x * 2^32); F_b is computed elementwise in fp64 on the device, so the vector stays integer.
With eval_surface=True (test_voxel) the voxel-surface counters of the same forwards follow (models.py,
Stereo2Voxel._surface_stats), per t in TEST.VOXEL_THRESH (surface_block):
    n_both, sum_b q(CD_L2_b), sum_b q(CD_L1_b), then per tau in TEST.FSCORE_THRESH sum_b q(P_b), sum_b q(R_b), sum_b q(F_b)
                                                                                               (int64)
again computed per batch in fp64 on the device.
With eval_curves=True (test_voxel) the threshold-free occupancy counters of the same forwards follow (models.py,
Stereo2Voxel._occupancy_curves; K = TEST.CURVE_BINS, curves_block):
    n_empty per bin (K), n_occ per bin (K), sum q20(v) per bin (K), sum q20(BCE), sum q20(Brier),
    sum_b q(IoU_b(k / K)) per k (K)                                                           (int64)
with q20(x) = round-half-even(x * 2^20) (include/s3d.h, s3d_occupancy_curves) and the per-sample IoU at every bin threshold
computed per batch in fp64 on the device; a sample whose GT and prediction are both empty at t has IoU 1 there.
With eval_fscore_curves=True (test_voxel with eval_surface, test_point with eval_points) the nearest-neighbour distance
histograms of the same forwards come last (models.py, _surface_stats / _point_stats; K = TEST.DIST_BINS edges e_k of
models.dist_edges, surface_curves_block per t in TEST.VOXEL_THRESH / point_curves_block):
    the histogram per direction (2 (K+1)), then per k sum_b q(P_b(e_k)), sum_b q(R_b(e_k)), sum_b q(F_b(e_k))   (int64)
with P_b, R_b the fractions of the predicted / GT points closer than e_k (the denominators of the surface / points blocks),
computed per batch in fp64 on the device.
stats_layout() declares these blocks and their order, split_stats() cuts a vector into them.
With eval_cloud=True (test_voxel / test_point) the same forwards also return the stereo point clouds (models.py,
_StereoBase._cloud, with the camera CONST.CAMERA), and their block follows the uncertainty one:
    kept points of view 0 (left-referenced), kept points of view 1, summed over the samples        (int64)
With cloud_dir (needs eval_cloud) each sample's cloud is also written as cloud_dir/%06d.ply and the GT disparity's cloud
(the same op without filters) as %06d_gt.ply, numbered by global sample id (save_clouds).
With mesh_dir (test_voxel) the same forwards also return the marching-cubes mesh of the prediction (models.py,
Stereo2Voxel._mesh), and each sample of the rank's shard is written as mesh_dir/%06d.obj (predicted) and %06d_gt.obj (the GT
occupancy, meshed by the same kernel at t = 0.5), numbered by global sample id; the stats vector does not change.
"""
import os

import numpy as np
import torch
import torch.distributed as dist

from .. import ops
from ..models import (Stereo2Point, Stereo2Voxel, camera_values, cloud_max_std, cloud_min_disp, curve_bins, dist_edges,
                      fscore_thresholds, mesh_thresh, speckle_params, unc_thresholds, wls_params)
from ..utils import synthetic

_FX = float(1 << 40)
_DISP_FX = float(1 << 16)
_PT_FX = float(1 << 32)
_OCC_FX = float(1 << 20)


def shard_range(n_total, rank, world):
    """Contiguous shard [lo, hi) of n_total samples for `rank` (first ranks take the remainder)."""
    base, rem = divmod(n_total, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def reduce_stats(stats):
    """SUM all-reduce of an int64 stats tensor over the default process group (no-op without one)."""
    if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    return stats


def iou_summary(stats, thresholds):
    """stats int64 [2T+1] -> dict.  IoU(t) = sum intersection / sum union."""
    T = len(thresholds)
    inter, union, n = stats[:T].double(), stats[T:2 * T].double(), int(stats[2 * T].item())
    return {'n_samples': n, 'thresholds': list(thresholds),
            'iou': [(i / u).item() if u > 0 else 0.0 for i, u in zip(inter, union)],
            'intersection': [int(v) for v in stats[:T].tolist()], 'union': [int(v) for v in stats[T:2 * T].tolist()]}


def disp_summary(stats_block, thresholds):
    """Disparity counters [n_valid, epe_fx, bad_t...] x 2 views (int64 [2 * (2 + T)]) -> dict: end-point error
    EPE = sum epe_fx / 2^16 / sum n_valid (px) and bad-pixel fractions, per view and over both views."""
    T = len(thresholds)
    v = [int(x) for x in stats_block.tolist()]
    assert len(v) == 2 * (2 + T)

    def one(n, epe_fx, bad):
        return {'n_valid': n, 'epe': epe_fx / _DISP_FX / n if n else 0.0, 'bad': [b / n if n else 0.0 for b in bad]}
    views = [v[:2 + T], v[2 + T:]]
    out = {'thresholds': list(thresholds)}
    for name, c in zip(('left', 'right'), views):
        out[name] = one(c[0], c[1], c[2:])
    out['all'] = one(views[0][0] + views[1][0], views[0][1] + views[1][1], [a + b for a, b in zip(views[0][2:], views[1][2:])])
    return out


def lr_summary(stats_block, thresholds, n_pixels, disp_block):
    """LR-check counters [n_kept, n_valid_kept, epe_fx, bad_t...] x 2 views (int64 [2 * (3 + T)]) -> dict, per view and over
    both views: density = n_kept / n_pixels (n_pixels: pixels of one view over the run), kept_of_valid = n_valid_kept /
    n_valid (n_valid from the disparity counters `disp_block`, as for disp_summary), and EPE / bad-pixel fractions over the
    kept valid pixels."""
    T = len(thresholds)
    v = [int(x) for x in stats_block.tolist()]
    nv = [int(x) for x in disp_block.tolist()]
    assert len(v) == 2 * (3 + T) and len(nv) == 2 * (2 + T)

    def one(pix, n_valid, c):
        nk, nvk, epe_fx, bad = c[0], c[1], c[2], c[3:]
        return {'n_kept': nk, 'density': nk / pix if pix else 0.0, 'n_valid_kept': nvk,
                'kept_of_valid': nvk / n_valid if n_valid else 0.0, 'epe': epe_fx / _DISP_FX / nvk if nvk else 0.0,
                'bad': [b / nvk if nvk else 0.0 for b in bad]}
    views = [v[:3 + T], v[3 + T:]]
    valid = [nv[0], nv[2 + T]]
    out = {'thresholds': list(thresholds)}
    for name, c, n in zip(('left', 'right'), views, valid):
        out[name] = one(n_pixels, n, c)
    out['all'] = one(2 * n_pixels, valid[0] + valid[1], [a + b for a, b in zip(views[0], views[1])])
    return out


def speckle_summary(stats_block, thresholds, n_pixels, disp_block):
    """Speckle-filter counters [n_kept, n_valid_kept, epe_fx, bad_t..., n_speckles, n_speckle_px] x 2 views (int64
    [2 * (5 + T)]) -> dict, per view and over both views: the lr_summary fields of the first 3 + T counters (density,
    kept_of_valid, EPE and bad-pixel fractions over the kept pixels), n_speckles (removed regions), speckle_pixels (their
    pixels) and mean_speckle_size = speckle_pixels / n_speckles."""
    T = len(thresholds)
    v = stats_block.reshape(2, 5 + T)
    out = lr_summary(v[:, :3 + T].reshape(-1), thresholds, n_pixels, disp_block)
    spk = [int(x) for x in v[:, 3 + T].tolist()]
    px = [int(x) for x in v[:, 4 + T].tolist()]
    for name, n, p in (('left', spk[0], px[0]), ('right', spk[1], px[1]), ('all', spk[0] + spk[1], px[0] + px[1])):
        out[name].update(n_speckles=n, speckle_pixels=p, mean_speckle_size=p / n if n else 0.0)
    return out


def wls_summary(stats_block, thresholds, n_pixels, disp_block):
    """WLS-filter counters [n_finite, n_valid_finite, epe_fx, bad_t..., n_conf] x 2 views (int64 [2 * (4 + T)]) -> dict, per
    view and over both views: n_finite, density = n_finite / n_pixels (n_pixels: pixels of one view over the run), filled =
    n_finite - n_conf (the pixels the filter filled in), n_valid_finite, valid_covered = n_valid_finite / n_valid (n_valid
    from the disparity counters `disp_block`), and EPE / bad-pixel fractions over the finite valid pixels."""
    T = len(thresholds)
    v = stats_block.reshape(2, 4 + T)
    lr = lr_summary(v[:, :3 + T].reshape(-1), thresholds, n_pixels, disp_block)
    conf = [int(x) for x in v[:, 3 + T].tolist()]
    out = {'thresholds': list(thresholds)}
    for name, nc in (('left', conf[0]), ('right', conf[1]), ('all', conf[0] + conf[1])):
        r = lr[name]
        out[name] = {'n_finite': r['n_kept'], 'density': r['density'], 'filled': r['n_kept'] - nc,
                     'n_valid_finite': r['n_valid_kept'], 'valid_covered': r['kept_of_valid'], 'epe': r['epe'],
                     'bad': r['bad']}
    return out


def unc_summary(stats_block, unc_thresh, thresholds, n_pixels, disp_block):
    """Uncertainty counters [n_conf, n_valid_conf, epe_fx, bad_t...] x K thresholds x 2 views (int64 [2 * K * (3 + T)]) -> dict,
    per view and over both views a list over the K thresholds tau (the sparsification curve at those points): density =
    n_conf / n_pixels (n_pixels: pixels of one view over the run), conf_of_valid = n_valid_conf / n_valid (n_valid from the
    disparity counters `disp_block`, as for lr_summary), and EPE / bad-pixel fractions over the confident valid pixels."""
    K, T = len(unc_thresh), len(thresholds)
    v = [int(x) for x in stats_block.tolist()]
    nv = [int(x) for x in disp_block.tolist()]
    assert len(v) == 2 * K * (3 + T) and len(nv) == 2 * (2 + T)

    def one(pix, n_valid, c):
        nc, nvc, epe_fx, bad = c[0], c[1], c[2], c[3:]
        return {'n_conf': nc, 'density': nc / pix if pix else 0.0, 'n_valid_conf': nvc,
                'conf_of_valid': nvc / n_valid if n_valid else 0.0, 'epe': epe_fx / _DISP_FX / nvc if nvc else 0.0,
                'bad': [b / nvc if nvc else 0.0 for b in bad]}
    r = 3 + T
    views = [[v[(vi * K + k) * r:(vi * K + k + 1) * r] for k in range(K)] for vi in range(2)]
    valid = [nv[0], nv[2 + T]]
    out = {'unc_thresh': list(unc_thresh), 'thresholds': list(thresholds)}
    for name, rows, n in zip(('left', 'right'), views, valid):
        out[name] = [one(n_pixels, n, c) for c in rows]
    out['all'] = [one(2 * n_pixels, valid[0] + valid[1], [a + b for a, b in zip(views[0][k], views[1][k])]) for k in range(K)]
    return out


def point_block(point_stats, N, M):
    """Per-batch increment of the point block from the forward's point_stats int64 [B,2,3+T] (N predicted, M GT points per
    sample): the counters summed over the batch, then sum_b round-half-even(F_b(t) * 2^32) per threshold, in fp64."""
    c = point_stats[:, :, 3:].double()
    p, r = c[:, 0] / N, c[:, 1] / M
    f = torch.where(p + r > 0, 2 * p * r / (p + r), torch.zeros_like(p))
    return torch.cat([point_stats.sum(0).flatten(), torch.round(f * _PT_FX).to(torch.int64).sum(0)])


def points_summary(block, thresholds, n_samples, N, M):
    """Point counters (int64 [2 * (3 + T) + T], as point_block sums them) -> dict:
    chamfer_l2 = (sum q(d1) / N + sum q(d2) / M) / 2^32 / n (squared distances: GRNet's ChamferDistance, the mean of dist1
    plus the mean of dist2), chamfer_l1 = (sum q(sqrt d1) / N + sum q(sqrt d2) / M) / 2 / 2^32 / n (GRNet's
    ChamferDistanceL1), both inf when a point was out of range (n_out > 0); per threshold the precision (predicted points
    within t of the GT), recall (GT points within t of the prediction) and the mean per-sample F-score."""
    T = len(thresholds)
    v = [int(x) for x in block.tolist()]
    assert len(v) == 2 * (3 + T) + T
    pred, gt, f = v[:3 + T], v[3 + T:2 * (3 + T)], v[2 * (3 + T):]
    n = n_samples
    n_out = pred[2] + gt[2]
    if n_out:
        l2 = l1 = float('inf')
    elif n:
        l2 = (pred[0] / N + gt[0] / M) / _PT_FX / n
        l1 = 0.5 * (pred[1] / N + gt[1] / M) / _PT_FX / n
    else:
        l2 = l1 = 0.0
    return {'n_samples': n, 'n_pred': N, 'n_gt': M, 'thresholds': list(thresholds), 'chamfer_l2': l2, 'chamfer_l1': l1,
            'n_out': n_out, 'precision': [c / (N * n) if n else 0.0 for c in pred[3:]],
            'recall': [c / (M * n) if n else 0.0 for c in gt[3:]], 'fscore': [x / _PT_FX / n if n else 0.0 for x in f]}


def surface_block(surf_stats, n):
    """Per-batch increment of the surface block from the forward's surf_stats int64 [B,T,2,3+F] (n = N_VOX) -> int64
    [T * (3 + 3F)]: per t [n_both, sum_b q(CD_L2_b), sum_b q(CD_L1_b), then per tau sum_b q(P_b), sum_b q(R_b), sum_b q(F_b)],
    q(x) = round-half-even(x * 2^32), in fp64.  Direction 0 = predicted -> GT (n_0 points), 1 = GT -> predicted (n_1):
    CD_L2_b = (sum s_0 / n_0 + sum s_1 / n_1) / (2n)^2 and CD_L1_b = (sum q_0 / n_0 + sum q_1 / n_1) / 2 / 2^32 / (2n), both
    over the n_both samples where both surfaces are non-empty (0 elsewhere); P_b = count_0 / n_0, R_b = count_1 / n_1 (0 when
    the denominator is 0), F_b = 2 P R / (P + R) (0 when P + R = 0)."""
    c = surf_stats.double()
    n0, n1 = c[:, :, 0, 0], c[:, :, 1, 0]
    both = (n0 > 0) & (n1 > 0)
    z = torch.zeros_like(n0)
    l2 = torch.where(both, (c[:, :, 0, 1] / n0 + c[:, :, 1, 1] / n1) / (2 * n) ** 2, z)
    l1 = torch.where(both, (c[:, :, 0, 2] / n0 + c[:, :, 1, 2] / n1) / 2 / _PT_FX / (2 * n), z)
    p = torch.where(n0[..., None] > 0, c[:, :, 0, 3:] / n0[..., None], torch.zeros_like(c[:, :, 0, 3:]))
    r = torch.where(n1[..., None] > 0, c[:, :, 1, 3:] / n1[..., None], torch.zeros_like(c[:, :, 1, 3:]))
    f = torch.where(p + r > 0, 2 * p * r / (p + r), torch.zeros_like(p))

    def q(x):
        return torch.round(x * _PT_FX).to(torch.int64).sum(0)
    T = c.shape[1]
    prf = torch.stack([q(p), q(r), q(f)], -1).reshape(T, -1)
    return torch.cat([both.sum(0, dtype=torch.int64)[:, None], q(l2)[:, None], q(l1)[:, None], prf], 1).flatten()


def surface_summary(block, voxel_thresh, fscore_thresh, n_samples):
    """Surface counters (int64 [T * (3 + 3F)], as surface_block sums them) -> dict with one entry per t in voxel_thresh:
    n_both, chamfer_l2 / chamfer_l1 (means over the n_both samples whose two surfaces are non-empty, in unit-cube units;
    inf when n_both = 0) and per tau the precision, recall and F-score as means over all n_samples."""
    T, F = len(voxel_thresh), len(fscore_thresh)
    v = [int(x) for x in block.tolist()]
    assert len(v) == T * (3 + 3 * F)
    n = n_samples
    per = []
    for t in range(T):
        r = v[t * (3 + 3 * F):(t + 1) * (3 + 3 * F)]
        nb = r[0]
        per.append({'voxel_thresh': float(voxel_thresh[t]), 'n_both': nb,
                    'chamfer_l2': r[1] / _PT_FX / nb if nb else float('inf'),
                    'chamfer_l1': r[2] / _PT_FX / nb if nb else float('inf'),
                    'precision': [r[3 + 3 * f] / _PT_FX / n if n else 0.0 for f in range(F)],
                    'recall': [r[4 + 3 * f] / _PT_FX / n if n else 0.0 for f in range(F)],
                    'fscore': [r[5 + 3 * f] / _PT_FX / n if n else 0.0 for f in range(F)]})
    return {'n_samples': n, 'thresholds': [float(t) for t in voxel_thresh], 'fscore_thresh': list(fscore_thresh),
            'by_thresh': per}


def curves_block(occ_hist, occ_loss):
    """Per-batch increment of the curves block from the forward's occ_hist int64 [B,3,K] and occ_loss int64 [B,2] -> int64
    [4K + 2]: the histogram rows and the loss sums summed over the batch, then per k sum_b q(IoU_b(k / K)), q(x) =
    round-half-even(x * 2^32), in fp64.  IoU_b(t_k) = I / U with I = sum_{j >= k} n_occ_j, U = sum_{j >= k} (n_empty_j +
    n_occ_j) + G_b - I, G_b the sample's occupied voxels; U = 0 (GT and prediction both empty) counts as IoU 1."""
    empty, occ = occ_hist[:, 0], occ_hist[:, 1]
    inter = occ.flip(1).cumsum(1).flip(1)
    union = (empty + occ).flip(1).cumsum(1).flip(1) + occ.sum(1, keepdim=True) - inter
    iou = torch.where(union > 0, inter.double() / union.clamp(min=1).double(), torch.ones_like(inter, dtype=torch.float64))
    return torch.cat([occ_hist.sum(0).flatten(), occ_loss.sum(0), torch.round(iou * _PT_FX).to(torch.int64).sum(0)])


def curves_summary(block, K, n_samples):
    """Curves counters (int64 [4K + 2], as curves_block sums them) -> dict.  thresholds t_k = k / K; iou: the pooled IoU
    sum I_k / sum U_k at every t_k (1 where U = 0, as per sample) and mean_iou: the mean of the per-sample IoUs; best /
    best_mean: the first t_k of the largest iou / mean_iou; ap = sum_k (R_k - R_{k+1}) P_k with R_k = I_k / G, P_k = I_k /
    Pred_k, R_K = 0 (average precision over the voxels' scores quantised to the bins; None when the GT is empty); bce and
    brier: means per voxel; ece = sum_m |S_m - O_m| / N over M = min(K, 16) equal-width bins merging K / M histogram bins
    (S_m the summed predictions, O_m the occupied voxels, N all voxels) and reliability: per merged bin {count, confidence
    S_m / count, frequency O_m / count} (None for an empty bin)."""
    v = [int(x) for x in block.tolist()]
    assert len(v) == 4 * K + 2
    empty, occ, sq, (bce, brier), miou = v[:K], v[K:2 * K], v[2 * K:3 * K], v[3 * K:3 * K + 2], v[3 * K + 2:]
    inter, pred = [0] * (K + 1), [0] * (K + 1)
    for k in range(K - 1, -1, -1):
        inter[k], pred[k] = inter[k + 1] + occ[k], pred[k + 1] + empty[k] + occ[k]
    G, N, n = inter[0], pred[0], n_samples
    thresholds = [k / K for k in range(K)]
    iou = [inter[k] / (pred[k] + G - inter[k]) if pred[k] + G - inter[k] else 1.0 for k in range(K)]
    mean_iou = [m / _PT_FX / n if n else 0.0 for m in miou]
    kb, km = max(range(K), key=iou.__getitem__), max(range(K), key=mean_iou.__getitem__)
    ap = sum(occ[k] / G * (inter[k] / pred[k]) for k in range(K) if occ[k]) if G else None
    M = min(K, 16)
    w = K // M
    ece, rel = 0.0, []
    for m in range(M):
        bins = range(m * w, (m + 1) * w)
        cnt = sum(empty[k] + occ[k] for k in bins)
        conf, obs = sum(sq[k] for k in bins) / _OCC_FX, sum(occ[k] for k in bins)
        ece += abs(conf - obs)
        rel.append({'count': cnt, 'confidence': conf / cnt if cnt else None, 'frequency': obs / cnt if cnt else None})
    return {'n_samples': n, 'n_voxels': N, 'bins': K, 'thresholds': thresholds, 'iou': iou, 'mean_iou': mean_iou,
            'best': {'threshold': thresholds[kb], 'iou': iou[kb]},
            'best_mean': {'threshold': thresholds[km], 'mean_iou': mean_iou[km]}, 'ap': ap,
            'bce': bce / _OCC_FX / N if N else 0.0, 'brier': brier / _OCC_FX / N if N else 0.0,
            'ece': ece / N if N else 0.0, 'reliability': rel}


def _prf_curves(hist, n0, n1):
    """hist int64 [..., 2, K+1] (direction 0: predicted -> GT, 1: GT -> predicted), n0 / n1 the denominators broadcastable to
    [...] -> int64 [K, 3]: per edge e_k (k = 1..K) sum over the leading dims of q(P), q(R), q(F) in fp64, P = (points of
    direction 0 in bins < k) / n0, R likewise for direction 1 over n1 (0 when the denominator is 0), F = 2 P R / (P + R)
    (0 when P + R = 0), q(x) = round-half-even(x * 2^32)."""
    K = hist.shape[-1] - 1
    cum = hist[..., :K].double().cumsum(-1)                   # [..., 2, K]: points closer than e_1 .. e_K
    n0 = torch.as_tensor(n0, dtype=torch.float64, device=hist.device)[..., None].expand_as(cum[..., 0, :])
    n1 = torch.as_tensor(n1, dtype=torch.float64, device=hist.device)[..., None].expand_as(cum[..., 1, :])
    z = torch.zeros_like(cum[..., 0, :])
    p = torch.where(n0 > 0, cum[..., 0, :] / n0.clamp(min=1), z)
    r = torch.where(n1 > 0, cum[..., 1, :] / n1.clamp(min=1), z)
    f = torch.where(p + r > 0, 2 * p * r / (p + r), z)
    q = torch.stack([p, r, f], -1)                            # [..., K, 3]
    return torch.round(q * _PT_FX).to(torch.int64).reshape(-1, K, 3).sum(0)


def point_curves_block(dist_hist, N, M):
    """Per-batch increment of the point_curves block from the forward's dist_hist int64 [B,2,K+1] (N predicted, M GT points
    per sample) -> int64 [2 (K+1) + 3K]: the histograms summed over the batch, then per edge e_k sum_b q(P_b), q(R_b),
    q(F_b) with P_b = (predicted points closer than e_k) / N and R_b = (GT points closer than e_k) / M, as point_block."""
    return torch.cat([dist_hist.sum(0).flatten(), _prf_curves(dist_hist, N, M).flatten()])


def surface_curves_block(dist_hist):
    """Per-batch increment of the surface_curves block from the forward's dist_hist int64 [B,T,2,K+1] -> int64
    [T * (2 (K+1) + 3K)]: per t the histograms summed over the batch, then per edge e_k sum_b q(P_b), q(R_b), q(F_b) with
    P_b = count_0(< e_k) / n_0 and R_b = count_1(< e_k) / n_1, n_d the row sums (the surface block's n_pts; 0 when empty)."""
    n = dist_hist.sum(-1).double()                            # [B,T,2]
    T = dist_hist.shape[1]
    per_t = [torch.cat([dist_hist[:, t].sum(0).flatten(), _prf_curves(dist_hist[:, t], n[:, t, 0], n[:, t, 1]).flatten()])
             for t in range(T)]
    return torch.cat(per_t) if per_t else torch.zeros(0, dtype=torch.int64, device=dist_hist.device)


def _first_reaching(cum, total, num, den):
    """The smallest k (0-based) with cum[k] / total >= num / den, in integers; None if none (or total = 0)."""
    if total <= 0:
        return None
    return next((k for k, c in enumerate(cum) if den * c >= num * total), None)


def _curves_summary(hist0, hist1, prf, edges, n_samples):
    """Summed histograms hist0 / hist1 (K+1 ints each) and the per-edge sums prf [K][3] -> the curves dict of one block."""
    K, n = len(edges), n_samples
    cum0, cum1, c0, c1 = [], [], 0, 0
    for k in range(K):
        c0 += hist0[k]
        c1 += hist1[k]
        cum0.append(c0)
        cum1.append(c1)
    t0, t1 = sum(hist0), sum(hist1)
    fscore = [prf[k][2] / _PT_FX / n if n else 0.0 for k in range(K)]

    def at(cum, total, num, den):
        k = _first_reaching(cum, total, num, den)
        return None if k is None else edges[k]
    return {'precision': [prf[k][0] / _PT_FX / n if n else 0.0 for k in range(K)],
            'recall': [prf[k][1] / _PT_FX / n if n else 0.0 for k in range(K)],
            'fscore': fscore,
            'pooled_precision': [c / t0 if t0 else 0.0 for c in cum0],
            'pooled_recall': [c / t1 if t1 else 0.0 for c in cum1],
            'fscore_auc': sum(fscore) / K,
            'accuracy': {'p50': at(cum0, t0, 1, 2), 'p90': at(cum0, t0, 9, 10)},
            'completeness': {'p50': at(cum1, t1, 1, 2), 'p90': at(cum1, t1, 9, 10)},
            'hist_pred': hist0, 'hist_gt': hist1}


def point_curves_summary(block, edges, n_samples):
    """point_curves counters (int64 [2 (K+1) + 3K], as point_curves_block sums them) -> dict over the K edges e_k
    (`thresholds`): precision / recall / fscore, the means of the per-sample values at every e_k; pooled_precision /
    pooled_recall, the fractions of all predicted / GT points closer than e_k; fscore_auc, the mean of the F-score curve over
    the K edges; accuracy / completeness {p50, p90}, the smallest e_k at which the pooled fraction of predicted / GT points
    closer than e_k reaches 0.5 / 0.9 (None if e_K does not); hist_pred / hist_gt, the summed histograms (bin K: beyond e_K
    or out of range)."""
    edges = [float(e) for e in edges]
    K = len(edges)
    v = [int(x) for x in block.tolist()]
    assert len(v) == 2 * (K + 1) + 3 * K
    prf = [v[2 * (K + 1) + 3 * k:2 * (K + 1) + 3 * k + 3] for k in range(K)]
    out = {'n_samples': n_samples, 'thresholds': edges}
    out.update(_curves_summary(v[:K + 1], v[K + 1:2 * (K + 1)], prf, edges, n_samples))
    return out


def surface_curves_summary(block, voxel_thresh, edges, n_samples):
    """surface_curves counters (int64 [T * (2 (K+1) + 3K)], as surface_curves_block sums them) -> dict with one entry per t
    in voxel_thresh holding the curves of point_curves_summary over the surface points (unit-cube units); a direction whose
    other surface is empty counts its points in bin K."""
    edges = [float(e) for e in edges]
    K, T = len(edges), len(voxel_thresh)
    v = [int(x) for x in block.tolist()]
    w = 2 * (K + 1) + 3 * K
    assert len(v) == T * w
    per = []
    for t in range(T):
        r = v[t * w:(t + 1) * w]
        prf = [r[2 * (K + 1) + 3 * k:2 * (K + 1) + 3 * k + 3] for k in range(K)]
        e = {'voxel_thresh': float(voxel_thresh[t])}
        e.update(_curves_summary(r[:K + 1], r[K + 1:2 * (K + 1)], prf, edges, n_samples))
        per.append(e)
    return {'n_samples': n_samples, 'thresholds': edges, 'by_thresh': per}


def write_obj(path, verts, faces):
    """Plain OBJ of verts fp32 [V,3] and 0-based faces int [F,3]: `v x y z` with %.9g (an fp32 value reads back exactly),
    then `f a b c` with 1-based ids."""
    with open(path, 'w') as fh:
        np.savetxt(fh, np.asarray(verts, np.float32).reshape(-1, 3), fmt='v %.9g %.9g %.9g')
        np.savetxt(fh, np.asarray(faces, np.int64).reshape(-1, 3) + 1, fmt='f %d %d %d')


def save_meshes(mesh_dir, ids, mesh, gt):
    """Writes the predicted meshes mesh = (verts, faces, counts) of samples `ids` (global ids) and the meshes of their GT
    occupancy gt [B,n,n,n] (nonzero = occupied, meshed at t = 0.5) as mesh_dir/%06d.obj and %06d_gt.obj."""
    gmesh = ops.voxel_mesh((gt != 0).to(torch.float32).contiguous(), 0.5)
    for name, (v, f, c) in (('%06d.obj', mesh), ('%06d_gt.obj', gmesh)):
        c = c.cpu()
        for b, i in enumerate(ids):
            nv, nf = int(c[b, 0]), int(c[b, 1])
            write_obj(os.path.join(mesh_dir, name % i), v[b, :nv].cpu().numpy(), f[b, :nf].cpu().numpy())


def cloud_summary(block, n_samples, H, W):
    """Cloud counters [kept points of view 0, of view 1] (int64 [2], summed over n_samples samples of H x W pairs) -> dict:
    per view and over both views the kept points, their mean per sample and the kept fraction of the view's pixels."""
    v = [int(x) for x in block.tolist()]
    assert len(v) == 2
    n, pix = n_samples, H * W

    def one(k, views):
        return {'n_points': k, 'per_sample': k / n if n else 0.0, 'kept_fraction': k / (views * n * pix) if n * pix else 0.0}
    return {'n_samples': n, 'left': one(v[0], 1), 'right': one(v[1], 1), 'all': one(v[0] + v[1], 2)}


_PLY_DTYPE = np.dtype([('x', '<f4'), ('y', '<f4'), ('z', '<f4'), ('red', 'u1'), ('green', 'u1'), ('blue', 'u1')])


def write_ply(path, xyz, rgb):
    """Binary little-endian PLY of points xyz fp32 [N,3] with colours rgb uint8 [N,3]: one vertex element with float x, y, z
    and uchar red, green, blue, 15 bytes per point."""
    xyz = np.asarray(xyz, np.float32).reshape(-1, 3)
    rgb = np.asarray(rgb, np.uint8).reshape(-1, 3)
    assert len(xyz) == len(rgb)
    rec = np.empty(len(xyz), _PLY_DTYPE)
    for i, k in enumerate(('x', 'y', 'z')):
        rec[k] = xyz[:, i]
    for i, k in enumerate(('red', 'green', 'blue')):
        rec[k] = rgb[:, i]
    head = ('ply\nformat binary_little_endian 1.0\nelement vertex %d\nproperty float x\nproperty float y\nproperty float z\n'
            'property uchar red\nproperty uchar green\nproperty uchar blue\nend_header\n' % len(rec))
    with open(path, 'wb') as fh:
        fh.write(head.encode('ascii'))
        fh.write(rec.tobytes())


def save_clouds(cloud_dir, ids, cloud, left, right, camera, disp_gt, min_disp):
    """Writes the forward's clouds cloud = (xyz, rgb, counts) of samples `ids` (global ids) as cloud_dir/%06d.ply, and the
    clouds of their GT disparity disp_gt fp32 [B,2,H,W] (NaN = none), back-projected by the same op with the same camera and
    min_disp and no other filter, as %06d_gt.ply."""
    B = disp_gt.shape[0]
    gcloud = ops.disp_cloud(disp_gt.transpose(0, 1).reshape(2 * B, disp_gt.shape[2], disp_gt.shape[3]).contiguous(), B,
                            left, right, camera, min_disp)
    for name, (xyz, rgb, c) in (('%06d.ply', cloud), ('%06d_gt.ply', gcloud)):
        n = c.to(torch.int64).sum(1).cpu()
        for b, i in enumerate(ids):
            write_ply(os.path.join(cloud_dir, name % i), xyz[b, :int(n[b])].cpu().numpy(), rgb[b, :int(n[b])].cpu().numpy())


def _camera(cfg, B, device):
    return torch.tensor([camera_values(cfg)], dtype=torch.float32).repeat(B, 1).to(device)


def _check_cloud(cfg, eval_cloud, eval_unc, cloud_dir):
    """ValueError on a bad cloud configuration, before any forward; creates cloud_dir."""
    if cloud_dir is not None and not eval_cloud:
        raise ValueError('cloud_dir needs eval_cloud=True')
    if eval_cloud:
        camera_values(cfg)
        cloud_min_disp(cfg)
        if eval_unc:
            cloud_max_std(cfg)
    if cloud_dir is not None:
        os.makedirs(cloud_dir, exist_ok=True)


def _disp_gt(pairs, H, W, device):
    return torch.cat([synthetic.disparity_gt(p[2], H, W) for p in pairs]).to(device)


def stats_layout(cfg, model, eval_disp=False, eval_lr=False, eval_unc=False, eval_surface=False, eval_points=False,
                 eval_curves=False, eval_fscore_curves=False, eval_cloud=False, eval_speckle=False, eval_wls=False):
    """The driver's int64 stats vector for `model` ('Stereo2Voxel' / 'Stereo2Point') as ordered blocks [(name, length)]: the
    head block ('iou' [2T+1] / 'chamfer' [2]), then 'disparity', 'lr_consistency', 'speckle', 'wls', 'uncertainty', 'cloud' [2],
    then 'surface',
    'curves' and 'surface_curves' (Stereo2Voxel) / 'points' and 'point_curves' (Stereo2Point), each present when its
    evaluation is on (module docstring).  ValueError on an evaluation without the counters it needs or on a bad cfg.TEST
    threshold: raised before any forward."""
    if eval_lr and not eval_disp:
        raise ValueError('eval_lr=True needs eval_disp=True')
    if eval_unc and not eval_disp:
        raise ValueError('eval_unc=True needs eval_disp=True')
    if eval_speckle and not eval_disp:
        raise ValueError('eval_speckle=True needs eval_disp=True')
    if eval_wls and not eval_disp:
        raise ValueError('eval_wls=True needs eval_disp=True')
    if eval_fscore_curves and model == 'Stereo2Voxel' and not eval_surface:
        raise ValueError('eval_fscore_curves=True for Stereo2Voxel needs eval_surface=True')
    if eval_fscore_curves and model != 'Stereo2Voxel' and not eval_points:
        raise ValueError('eval_fscore_curves=True for Stereo2Point needs eval_points=True')
    T = len(cfg.TEST.DISP_THRESH)
    blocks = [('iou', 2 * len(cfg.TEST.VOXEL_THRESH) + 1) if model == 'Stereo2Voxel' else ('chamfer', 2)]
    if eval_disp:
        blocks.append(('disparity', 2 * (2 + T)))
    if eval_lr:
        blocks.append(('lr_consistency', 2 * (3 + T)))
    if eval_speckle:
        speckle_params(cfg)
        blocks.append(('speckle', 2 * (5 + T)))
    if eval_wls:
        wls_params(cfg)
        blocks.append(('wls', 2 * (4 + T)))
    if eval_unc:
        blocks.append(('uncertainty', 2 * len(unc_thresholds(cfg)) * (3 + T)))
    if eval_cloud:
        blocks.append(('cloud', 2))
    if eval_surface:
        blocks.append(('surface', len(cfg.TEST.VOXEL_THRESH) * (3 + 3 * len(fscore_thresholds(cfg)))))
    if eval_curves:
        blocks.append(('curves', 4 * curve_bins(cfg) + 2))
    if eval_points:
        F = len(fscore_thresholds(cfg))
        blocks.append(('points', 2 * (3 + F) + F))
    if eval_fscore_curves:
        K = len(dist_edges(cfg))
        if model == 'Stereo2Voxel':
            blocks.append(('surface_curves', len(cfg.TEST.VOXEL_THRESH) * (2 * (K + 1) + 3 * K)))
        else:
            blocks.append(('point_curves', 2 * (K + 1) + 3 * K))
    return blocks


def split_stats(stats, layout):
    """{name: slice of the 1-D stats vector} for the blocks of `layout` (stats_layout); the slices are views."""
    out, lo = {}, 0
    for name, n in layout:
        out[name] = stats[lo:lo + n]
        lo += n
    return out


def _add_disp_blocks(blocks, out):
    """Adds the batch's disparity, LR-check, speckle-filter, WLS-filter, uncertainty and cloud counters of the named forward
    outputs `out` to their blocks."""
    for block, name in (('disparity', 'disp_stats'), ('lr_consistency', 'lr_stats'), ('speckle', 'speckle_stats'),
                        ('wls', 'wls_stats'), ('uncertainty', 'unc_stats'), ('cloud', 'cloud_counts')):
        if block in blocks:
            blocks[block] += out[name].sum(0).flatten()


def test_voxel(cfg, model, n_samples, batch_size, rank=0, world=1, device='cuda', eval_disp=False, eval_lr=False,
               eval_unc=False, eval_surface=False, mesh_dir=None, eval_curves=False, eval_fscore_curves=False, cloud_dir=None,
               eval_cloud=False, eval_speckle=False, eval_wls=False):
    """Synthetic StereoShapeNet stand-in: sample i is generated from seed i, so every rank can
    materialise exactly its own shard and the union over ranks is independent of `world`.
    eval_disp: the same forward also evaluates the disparities; their counters follow the IoU ones (module docstring).
    eval_lr: the same forward also runs the left-right consistency check; its counters follow the disparity ones.
    eval_speckle: the same forward also runs the speckle filter (after the LR check with eval_lr); its counters follow the LR
    ones, and with eval_cloud the clouds keep only the pixels it keeps.
    eval_wls: the same forward also runs the WLS filter (confident where the speckle / LR mask keeps a pixel, else where it
    is finite); its counters follow the speckle ones, and with eval_cloud the clouds are the WLS maps' (no other filter).
    eval_unc: the same forward also returns the disparity uncertainty; its counters follow the LR ones.
    eval_surface: the same forward also evaluates the voxel surfaces; their block follows the uncertainty one.
    eval_curves: the same forward also returns the occupancy histograms and loss sums; their block follows the surface one.
    eval_fscore_curves (needs eval_surface): the same call that counts the surface metrics also returns the surface distance
    histograms; their block comes last.
    mesh_dir: the same forward also meshes the prediction; the meshes and the GT's are written there (module docstring).
    eval_cloud: the same forward also returns the stereo point clouds (camera CONST.CAMERA); their counters follow the
    uncertainty ones.  cloud_dir (needs eval_cloud): the clouds and the GT disparity's are written there as PLY.
    The vector's blocks: stats_layout(cfg, 'Stereo2Voxel', ...)."""
    layout = stats_layout(cfg, 'Stereo2Voxel', eval_disp, eval_lr, eval_unc, eval_surface, eval_curves=eval_curves,
                          eval_fscore_curves=eval_fscore_curves, eval_cloud=eval_cloud, eval_speckle=eval_speckle,
                          eval_wls=eval_wls)
    _check_cloud(cfg, eval_cloud, eval_unc, cloud_dir)
    if mesh_dir is not None:
        mesh_thresh(cfg)                                # ValueError on a bad TEST.MESH_THRESH, before any forward
        os.makedirs(mesh_dir, exist_ok=True)
    kw = {k: True for k, on in (('lr_check', eval_lr), ('speckle', eval_speckle), ('wls', eval_wls), ('uncertainty', eval_unc),
                                ('surface', eval_surface), ('mesh', mesh_dir is not None), ('curves', eval_curves),
                                ('fscore_curves', eval_fscore_curves)) if on}    # the options that are on
    names = Stereo2Voxel.output_names(gt=True, disp_gt=eval_disp, camera=eval_cloud, **kw)
    stats = torch.zeros(sum(n for _, n in layout), dtype=torch.int64, device=device)
    blocks = split_stats(stats, layout)
    T = len(cfg.TEST.VOXEL_THRESH)
    lo, hi = shard_range(n_samples, rank, world)
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    with torch.no_grad():
        for s in range(lo, hi, batch_size):
            ids = range(s, min(s + batch_size, hi))
            pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in ids]
            left = torch.cat([p[0] for p in pairs]).to(device)
            right = torch.cat([p[1] for p in pairs]).to(device)
            gt = torch.cat([synthetic.gt_volume(1, cfg.CONST.N_VOX, seed=100000 + i) for i in ids]).to(device)
            dgt = _disp_gt(pairs, H, W, device) if eval_disp or cloud_dir is not None else None
            if eval_disp:
                kw['disp_gt'] = dgt
            if eval_cloud:
                kw['camera'] = _camera(cfg, len(ids), device)
            out = dict(zip(names, model(left, right, gt, **kw)))
            _add_disp_blocks(blocks, out)
            if cloud_dir is not None:
                save_clouds(cloud_dir, ids, (out['cloud_xyz'], out['cloud_rgb'], out['cloud_counts']), left, right,
                            kw['camera'], dgt, cloud_min_disp(cfg))
            if eval_surface:
                blocks['surface'] += surface_block(out['surf_stats'], cfg.CONST.N_VOX)
            if eval_curves:
                blocks['curves'] += curves_block(out['occ_hist'], out['occ_loss'])
            if eval_fscore_curves:
                blocks['surface_curves'] += surface_curves_block(out['dist_hist'])
            if mesh_dir is not None:
                save_meshes(mesh_dir, ids, (out['mesh_verts'], out['mesh_faces'], out['mesh_counts']), gt)
            iou = out['iou_counts']
            blocks['iou'][:T] += iou[:, :, 0].sum(0)
            blocks['iou'][T:2 * T] += iou[:, :, 1].sum(0)
            blocks['iou'][2 * T] += len(ids)
    return reduce_stats(stats)


def test_point(cfg, model, n_samples, batch_size, rank=0, world=1, device='cuda', eval_disp=False, eval_lr=False,
               eval_points=False, eval_unc=False, eval_fscore_curves=False, cloud_dir=None, eval_cloud=False,
               eval_speckle=False, eval_wls=False):
    """[sum CD in 2^-40 units, n_samples] (+ the disparity counters with eval_disp, the LR-check counters with eval_lr, the
    speckle-filter counters with eval_speckle, the WLS-filter counters with eval_wls, the uncertainty counters with eval_unc, the stereo-cloud counters with
    eval_cloud (and the PLY files with cloud_dir), as for test_voxel, + the point-cloud counters with eval_points, + the distance histograms of the same call with
    eval_fscore_curves (needs eval_points): module docstring).
    The vector's blocks: stats_layout(cfg, 'Stereo2Point', ...)."""
    from ..extensions.chamfer_dist import chamfer_per_sample
    layout = stats_layout(cfg, 'Stereo2Point', eval_disp, eval_lr, eval_unc, eval_points=eval_points,
                          eval_fscore_curves=eval_fscore_curves, eval_cloud=eval_cloud, eval_speckle=eval_speckle,
                          eval_wls=eval_wls)
    _check_cloud(cfg, eval_cloud, eval_unc, cloud_dir)
    kw = {k: True for k, on in (('lr_check', eval_lr), ('speckle', eval_speckle), ('wls', eval_wls), ('uncertainty', eval_unc),
                                ('fscore_curves', eval_fscore_curves)) if on}
    names = Stereo2Point.output_names(gt=eval_points, disp_gt=eval_disp, camera=eval_cloud, **kw)
    stats = torch.zeros(sum(n for _, n in layout), dtype=torch.int64, device=device)
    blocks = split_stats(stats, layout)
    lo, hi = shard_range(n_samples, rank, world)
    H, W = cfg.CONST.IMG_H, cfg.CONST.IMG_W
    with torch.no_grad():
        for s in range(lo, hi, batch_size):
            ids = range(s, min(s + batch_size, hi))
            pairs = [synthetic.stereo_pair(1, H, W, 2 * cfg.NETWORK.MAX_DISP, seed=i) for i in ids]
            left = torch.cat([p[0] for p in pairs]).to(device)
            right = torch.cat([p[1] for p in pairs]).to(device)
            gt = torch.cat([synthetic.point_clouds(1, 1, cfg.CONST.N_GT_POINTS, seed=200000 + i)[1] for i in ids]).to(device)
            head = (gt,) if eval_points else ()
            dgt = _disp_gt(pairs, H, W, device) if eval_disp or cloud_dir is not None else None
            if eval_disp:
                kw['disp_gt'] = dgt
            if eval_cloud:
                kw['camera'] = _camera(cfg, len(ids), device)
            out = dict(zip(names, model(left, right, *head, **kw)))
            _add_disp_blocks(blocks, out)
            if cloud_dir is not None:
                save_clouds(cloud_dir, ids, (out['cloud_xyz'], out['cloud_rgb'], out['cloud_counts']), left, right,
                            kw['camera'], dgt, cloud_min_disp(cfg))
            pts = out['points']
            if eval_points:
                blocks['points'] += point_block(out['point_stats'], pts.shape[1], gt.shape[1])
            if eval_fscore_curves:
                blocks['point_curves'] += point_curves_block(out['dist_hist'], pts.shape[1], gt.shape[1])
            cd = chamfer_per_sample(pts.contiguous(), gt)
            blocks['chamfer'][0] += torch.round(cd.sum() * _FX).to(torch.int64)
            blocks['chamfer'][1] += len(ids)
    return reduce_stats(stats)


def chamfer_summary(stats):
    n = int(stats[1].item())
    return {'n_samples': n, 'chamfer_distance': (stats[0].item() / _FX) / max(n, 1)}
