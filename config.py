# -*- coding: utf-8 -*-
"""Global configuration, ``cfg.SECTION.KEY`` style.

Mirrors the reference's ``config.py`` convention: a module-level EasyDict-like
object ``__C`` exported as ``cfg`` (reference: README.md:68-78, the only lines of
``config.py`` that are quoted on disk; ``easydict`` is requirements.txt:2 and is
NOT installed in this image, so a ~10-line attribute dict stands in for it).

Only the five ``DATASETS.SHAPENET.*`` keys are attested by the reference.  Every
other knob below is a [SPEC] decision of this repo (SURVEY.md section 8): the
upstream Stereo2Voxel / Stereo2Point branches are not available offline, so the
network is a restatement of BASELINE.json's ``north_star`` and its layer table
is frozen in DESIGN.md.
"""


class AttrDict(dict):
    """Minimal EasyDict: nested dict with attribute access."""

    def __getattr__(self, k):
        try:
            return self[k]
        except KeyError as e:  # pragma: no cover
            raise AttributeError(k) from e

    def __setattr__(self, k, v):
        self[k] = v

    def clone(self):
        out = AttrDict()
        for k, v in self.items():
            out[k] = v.clone() if isinstance(v, AttrDict) else (list(v) if isinstance(v, list) else v)
        return out


__C = AttrDict()
cfg = __C

#
# Dataset config (reference: README.md:68-78).  The data itself is unavailable
# offline; the paths are kept so that a user's edited config.py still loads.
#
__C.DATASETS = AttrDict()
__C.DATASETS.SHAPENET = AttrDict()
__C.DATASETS.SHAPENET.LEFT_RENDERING_PATH = '/path/to/ShapeNetStereoRendering/%s/%s/render_%02d_l.png'
__C.DATASETS.SHAPENET.RIGHT_RENDERING_PATH = '/path/to/ShapeNetStereoRendering/%s/%s/render_%02d_r.png'
__C.DATASETS.SHAPENET.LEFT_DISP_PATH = '/path/to/ShapeNetStereoRendering/%s/%s/disp_%02d_l.exr'
__C.DATASETS.SHAPENET.RIGHT_DISP_PATH = '/path/to/ShapeNetStereoRendering/%s/%s/disp_%02d_r.exr'
__C.DATASETS.SHAPENET.VOLUME_PATH = '/path/to/ShapeNetVox32/%s/%s.mat'

#
# Constants  [SPEC]
#
__C.CONST = AttrDict()
__C.CONST.IMG_H = 256            # declared default input size (SURVEY.md 8(d))
__C.CONST.IMG_W = 256
__C.CONST.N_VOX = 32             # 32^3 occupancy (README.md:77, ShapeNetVox32)
__C.CONST.N_POINTS = 2048        # Stereo2Point predicted points (BASELINE configs[3])
__C.CONST.N_GT_POINTS = 16384
__C.CONST.BATCH_SIZE = 64
__C.CONST.SEED = 0
__C.CONST.MICRO_BATCH = 64          # forward() splits larger batches into chunks of this many pairs

#
# Network  [SPEC]
#
__C.NETWORK = AttrDict()
__C.NETWORK.MAX_DISP = 32              # number of disparity planes D in the 1/4-res volume
__C.NETWORK.FEAT_CHANNELS = 32         # C, siamese feature channels
__C.NETWORK.ENC_CHANNELS = [32, 64]    # widths of the 1/2-res and 1/4-res encoder stages
__C.NETWORK.AGG_CHANNELS = 64          # A, width of the 3D aggregation stack
__C.NETWORK.COST_VOLUME = 'concat'     # 'concat' (-> 3D aggregation) | 'corr' (fused corr + soft-argmin)
__C.NETWORK.REC_CHANNELS = [32, 64, 128, 256, 256]   # RGB-D encoder, 5 stride-2 stages
__C.NETWORK.LATENT_HW = 8              # RGB-D encoder output is pooled to LATENT_HW^2
__C.NETWORK.DEC_CHANNELS = [2048, 512, 128, 32, 8]    # 2^3 -> 32^3 transposed-conv decoder
__C.NETWORK.MERGER_CHANNELS = [9, 16, 8, 4, 2, 1]     # context-aware fusion scorer
__C.NETWORK.LEAKY_VALUE = 0.2
__C.NETWORK.POINT_FC = 2048            # Stereo2Point hidden width
# 'bf16' | 'bf16x3' (bf16 hi/lo pairs, 3 MMAs per product: fp32 accuracy at a third of the bf16 rate) | 'tf32' (fp32
# storage, TF32 tensor cores) | 'tf32x3' (3 split TF32 passes through HBM, fp32 accuracy) | 'fp32' (SIMT, exact)
__C.NETWORK.PRECISION = 'bf16'

#
# Test  [SPEC]
#
__C.TEST = AttrDict()
__C.TEST.VOXEL_THRESH = [0.2, 0.3, 0.4, 0.5]
# bad-pixel thresholds of the disparity evaluation (forward(..., disp_gt=...)): |disp - gt| > t px at input resolution
__C.TEST.DISP_THRESH = [1.0, 3.0]
# left-right consistency check (forward(..., lr_check=True)): a pixel is kept when its disparity d and the other view's
# disparity at the pixel it points to (x -/+ round(d)) differ by at most this many px; finite, >= 0
__C.TEST.LR_THRESH = 1.0
# disparity uncertainty (forward(..., uncertainty=True)): a pixel counts as confident at t when the standard deviation of its
# soft-argmin distribution, in input px, is <= t; at most 4, each finite and >= 0
__C.TEST.UNC_THRESH = [1.0, 2.0, 4.0]
# F-score thresholds of the point-cloud evaluation (Stereo2Point forward(..., gt)): a point counts when its nearest neighbour
# in the other cloud is closer than t, a Euclidean distance in the points' units (0.01 = F-Score@1% on unit-scale shapes);
# at most 8, each finite and > 0
__C.TEST.FSCORE_THRESH = [0.01]
# iso-level of the exported mesh (forward(..., mesh=True), runner.py --test --save-meshes): marching cubes over the predicted
# occupancy, a voxel is inside when its value is >= this; finite and in (0, 1]
__C.TEST.MESH_THRESH = 0.5
# bins of the threshold-free occupancy evaluation (forward(..., curves=True), runner.py --test --curves): the IoU and precision-
# recall curves are exact at the thresholds k / CURVE_BINS, and the calibration merges them into min(CURVE_BINS, 16) bins;
# an int, a power of two in [2, 1024]
__C.TEST.CURVE_BINS = 256
