"""The constant-region skip of the aggregation layers (include/s3d.h dz_nref) changes no bit: every activation of the
chain dres0b -> dres1a -> dres1b and every model output equals the run with the skip switched off (knob no_dz_skip), on
the batched path, the z-split path (skip off there), a reduced network, ragged patches, D > w, the reference-once first layer
and single CTAs.  The kernel marches exactly the planes the schedule says, and exactly today's planes without a region."""
import pytest
import torch

from config import cfg as default_cfg
from stereo_3d_reconstruction_b200 import layers, models as M
from stereo_3d_reconstruction_b200.utils import synthetic
from tests.common import small_cfg

pytestmark = pytest.mark.gpu


def _model(cfg):
    return M.build_model('Stereo2Voxel', cfg, seed=0).cuda().pack()


def _inputs(cfg, B):
    left, right, _ = synthetic.stereo_pair(B, cfg.CONST.IMG_H, cfg.CONST.IMG_W, 2 * cfg.NETWORK.MAX_DISP, seed=5)
    return left.cuda(), right.cuda(), synthetic.gt_volume(B, seed=6).cuda()


def _run(model, inp):
    with torch.no_grad():
        out = [t.clone() for t in model(*inp)]
    acts = {k[0]: v.clone() for k, v in model._ws.items() if k[0] in ('a1', 'a2', 'a3')}
    return out, acts


CASES = {
    'default-B3': (lambda: default_cfg.clone(), 3, None),
    'default-B1-zsplit': (lambda: default_cfg.clone(), 1, None),
    # the reduced network (32-wide layers: the all-in-one kernel for the residual layer); B = 20 keeps whole columns
    'small': (lambda: small_cfg(), 20, None),
    'ragged': (lambda: small_cfg(CONST__IMG_H=200, CONST__IMG_W=212, NETWORK__MAX_DISP=24), 3, None),
    'D-above-w': (lambda: small_cfg(CONST__IMG_W=40, NETWORK__MAX_DISP=24), 20, None),
    'ref-once': (lambda: default_cfg.clone(), 3, 'no_sheared'),
    'no-pair': (lambda: default_cfg.clone(), 3, 'scatter_no_pair'),
}


@pytest.mark.parametrize('case', list(CASES))
def test_skip_is_bit_identical(knobs, case):
    make, B, knob = CASES[case]
    if knob:
        knobs(knob, 1)
    cfg = make()
    model = _model(cfg)
    inp = _inputs(cfg, B)
    knobs('no_dz_skip', 1)
    ref_out, ref_acts = _run(model, inp)
    knobs('no_dz_skip', 0)
    out, acts = _run(model, inp)
    assert set(acts) == {'a1', 'a2', 'a3'}
    for k in acts:
        assert torch.equal(acts[k], ref_acts[k]), k
    for a, b in zip(out, ref_out):
        assert torch.equal(a, b)


def _planes(model, inp, layer):
    counter = torch.zeros(1, dtype=torch.int64, device='cuda')
    conv = model._conv

    def one(name, x, **kw):
        layers.plane_counter = counter if name == layer else None
        try:
            return conv(name, x, **kw)
        finally:
            layers.plane_counter = None
    model._conv = one
    try:
        with torch.no_grad():
            model(*inp)
    finally:
        model._conv = conv
    return int(counter.item())


@pytest.mark.parametrize('layer,c,e', [('dres0b', 3, 1), ('dres1a', 5, 2), ('dres1b', 7, 3)])
def test_marched_planes(knobs, layer, c, e):
    cfg = default_cfg.clone()
    B, D = 3, cfg.NETWORK.MAX_DISP
    h, w = cfg.CONST.IMG_H // 4, cfg.CONST.IMG_W // 4
    model = _model(cfg)
    inp = _inputs(cfg, B)
    ncols = 2 * B * -(-h // 32) * -(-w // 8)
    knobs('no_dz_skip', 1)                        # region ignored: the round-robin march of today, one column per CTA here
    assert _planes(model, inp, layer) == ncols * D
    knobs('no_dz_skip', 0)
    npairs = min(torch.cuda.get_device_properties(0).multi_processor_count // 2, -(-ncols // 2))
    _, load = layers.dz_schedule(2 * B, B, h, w, D, c, e, npairs)
    got = _planes(model, inp, layer)
    assert got == 2 * sum(load) < ncols * D
