"""The constant region the aggregation layers declare to the plane-scatter kernel (include/s3d.h dz_nref), and the CTA-pair
schedule built for it (layers.py dz_schedule), on the CPU.

The concat volume is [ref(y, x) | tgt(y, x -/+ d)] with the target half zero outside the image, so along d it is the same
wherever the target pixel has left the image; each 3x3x3 layer shrinks that region by one plane at each end.  The layer
chain runs here in float64 on small integers, where every sum is exact: the test checks the region itself (which planes are
equal), independent of summation order.  That the kernel reproduces the skipped planes bit for bit is tests/test_gpu_dz_skip.py."""
import math

import pytest
import torch
import torch.nn.functional as F

from stereo_3d_reconstruction_b200.layers import dz_first, dz_jump, dz_march, dz_schedule

# (c, e) of each layer's output: plane d of pixel x equals plane xr + c for d in [xr + c, D - 1 - e]
REGIONS = {'dres0a': (3, 1), 'dres0b': (5, 2), 'dres1a': (7, 3), 'dres1b': (9, 4), 'cls_a': (11, 5)}


def _volume(fl, fr, D):
    """Concat cost volume of s3d_cost_volume_concat: [2, 2C, D, h, w], left-referenced first."""
    C, h, w = fl.shape
    vol = torch.zeros(2, 2 * C, D, h, w, dtype=fl.dtype)
    for d in range(D):
        vol[0, :C, d], vol[1, :C, d] = fl, fr
        if d < w:
            vol[0, C:, d, :, d:] = fr[:, :, :w - d]          # target at x - d
            vol[1, C:, d, :, :w - d] = fl[:, :, d:]          # target at x + d
    return vol


def _chain(D, h, w, C=4, A=4, seed=0):
    g = torch.Generator().manual_seed(seed)

    def ints(*shape, lo=-2, hi=3):
        return torch.randint(lo, hi, shape, generator=g).double()
    vol = _volume(ints(C, h, w), ints(C, h, w), D)
    Wt = {n: ints(A, 2 * C if n == 'dres0a' else A, 3, 3, 3, lo=-1, hi=2) for n in REGIONS}
    b = {n: ints(A) for n in REGIONS}

    def conv(n, x):
        return F.conv3d(x, Wt[n], b[n], padding=1)
    out = {'dres0a': F.relu(conv('dres0a', vol))}
    out['dres0b'] = F.relu(conv('dres0b', out['dres0a']))
    out['dres1a'] = F.relu(conv('dres1a', out['dres0b']))
    out['dres1b'] = conv('dres1b', out['dres1a']) + out['dres0b']
    out['cls_a'] = F.relu(conv('cls_a', out['dres1b']))
    return out


@pytest.mark.parametrize('D,h,w', [(4, 5, 8), (8, 6, 16), (13, 4, 24), (13, 5, 8), (8, 3, 16)])
def test_region_is_constant_along_d(D, h, w):
    out = _chain(D, h, w)
    for name, (c, e) in REGIONS.items():
        y = out[name]
        assert y.abs().max() < 2 ** 52                       # exact arithmetic
        for v in (0, 1):                                     # left-, right-referenced
            for x in range(w):
                xr = x if v == 0 else w - 1 - x
                lo, hi = xr + c, D - 1 - e
                for d in range(lo + 1, hi + 1):
                    assert torch.equal(y[v, :, d, :, x], y[v, :, lo, :, x]), (name, v, x, d)


def test_region_bounds_are_tight():
    """One plane further at either end is not the same any more (for some pixel of random data)."""
    D, h, w = 24, 4, 24
    out = _chain(D, h, w, seed=3)
    for name, (c, e) in REGIONS.items():
        y = out[name]
        for v in (0, 1):
            low = [x for x in range(w) if (x if v == 0 else w - 1 - x) + c + 1 <= D - 1 - e]
            xr = [x if v == 0 else w - 1 - x for x in low]
            assert low, name
            assert any(not torch.equal(y[v, :, r + c - 1, :, x], y[v, :, r + c, :, x]) for x, r in zip(low, xr) if r + c >= 1), name
            assert any(not torch.equal(y[v, :, D - e, :, x], y[v, :, D - 1 - e, :, x]) for x, r in zip(low, xr)), name


def _stored(zs, J, D):
    """Output planes the epilogue stores for a work item, in order: drained planes, and the copies of plane zs."""
    out, z = [], 0
    for p in dz_march(zs, J, D):
        for _ in range((p >= 1) + (p == D - 1)):
            out.append(z)
            if z == zs:
                out += list(range(z + 1, z + 1 + J))
                z += J
            z += 1
    return out


SHAPES = [(64, 64, 64, 32), (3, 64, 64, 32), (1, 50, 53, 24), (20, 16, 10, 24), (5, 40, 24, 8), (2, 8, 16, 13)]


@pytest.mark.parametrize('B,h,w,D', SHAPES)
@pytest.mark.parametrize('layer', ['dres0b', 'dres1a', 'dres1b'])
def test_schedule_pairs_and_copies(B, h, w, D, layer):
    c_in, e_in = {'dres0b': (3, 1), 'dres1a': (5, 2), 'dres1b': (7, 3)}[layer]
    N, ncols = 2 * B, 2 * B * math.ceil(h / 32) * math.ceil(w / 8)
    npairs = min(74, -(-ncols // 2))
    table, load = dz_schedule(N, B, h, w, D, c_in, e_in, npairs)
    offs, ent = table[:npairs + 1], table[npairs + 1:]
    assert offs[0] == 0 and offs == sorted(offs) and len(ent) == 2 * offs[-1]
    real = [k for k in ent if k < ncols]
    assert sorted(real) == list(range(ncols)) and all(k == ncols for k in ent if k >= ncols)
    ze = D - 2 - e_in
    for q in range(npairs):
        walked = 0
        for i in range(offs[q], offs[q + 1]):
            a, b = ent[2 * i], ent[2 * i + 1]
            first = [dz_first(k, N, B, h, w, c_in) for k in (a, b)]
            zs = max(first)                                  # both CTAs of the pair: the same run, so the same march
            J = dz_jump(zs, D, e_in)
            assert J % 3 == 0 and (J == 0 or zs + J <= ze)
            walked += len(dz_march(zs, J, D))
            stored = _stored(zs, J, D)
            assert sorted(stored) == list(range(D))          # every output plane exactly once
            for k, f in zip((a, b), first):
                if k < ncols and J:
                    assert f <= zs                           # copies only inside the column's own repeating run
        assert walked == load[q]
    mean = sum(load) / npairs
    assert max(load) <= mean + D
    if ncols >= 1024:
        assert max(load) <= 1.03 * mean
        assert max(load) < -(-ncols // (2 * npairs)) * D       # fewer planes than the round-robin march of today


def test_columns_repeat_on_their_run():
    """A column's run [zs, zs + J] (conv_scatter.cuh dz_first / dz_jump) lies inside every one of its pixels' regions."""
    D, h, w, B = 13, 6, 24, 1
    out = _chain(D, h, w, seed=5)
    for layer, src in (('dres0b', 'dres0a'), ('dres1a', 'dres0b'), ('dres1b', 'dres1a')):
        c_in, e_in = REGIONS[src]
        y = out[layer]
        for col in range(2 * B * math.ceil(w / 8)):
            n, x0 = col // math.ceil(w / 8), (col % math.ceil(w / 8)) * 8
            zs = dz_first(col, 2 * B, B, h, w, c_in)
            J = dz_jump(zs, D, e_in)
            for z in range(zs + 1, zs + J + 1):
                assert torch.equal(y[n, :, z, :, x0:x0 + 8], y[n, :, zs, :, x0:x0 + 8]), (layer, col, z)
