"""The marching-cubes rule of s3d_voxel_mesh on the CPU: the committed case table is the generator's output, and the meshes
of the reference statement (tests/mesh_oracle.py) are closed, oriented 2-manifolds of the right topology and volume."""
import os

import numpy as np
import pytest

from stereo_3d_reconstruction_b200 import mc_table
from tests import mesh_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_committed_header_is_generated():
    with open(os.path.join(ROOT, 'stereo_3d_reconstruction_b200', 'csrc', 'mc_table.cuh')) as fh:
        assert fh.read() == mc_table.header()


def test_case_table_loops_and_sizes():
    for case in range(256):
        inside = [(case >> c) & 1 for c in range(8)]
        crossing = sorted(e for e in range(12) if inside[mc_table.edge_corners(e)[0]] != inside[mc_table.edge_corners(e)[1]])
        loops = mc_table.case_loops(case)
        assert sorted(e for lp in loops for e in lp) == crossing, case          # each crossing edge in exactly one loop
        assert all(lp[0] == min(lp) for lp in loops)
        assert [lp[0] for lp in loops] == sorted(lp[0] for lp in loops)
        tris = mc_table.TABLE[case]
        assert len(tris) <= 5 and len(tris) == sum(len(lp) - 2 for lp in loops)
        assert set(e for t in tris for e in t) == set(crossing)
    assert mc_table.TABLE[0] == [] and mc_table.TABLE[255] == []


def _single(case):
    vol = np.zeros((2, 2, 2), np.float32)
    for c in range(8):
        if (case >> c) & 1:
            cx, cy, cz = mc_table.corner_xyz(c)
            vol[cz, cy, cx] = 1.0
    return vol


def _check_closed(v, f, degenerate=False):
    """degenerate: the field takes only the values 0 and t, so every vertex sits on an inside corner and the volume can be 0."""
    assert O.closed_manifold(v, f)
    vol = O.signed_volume(v, f)
    assert vol >= 0 if degenerate else vol > 0
    assert len(np.unique(f)) == len(v)                                          # every vertex is used


@pytest.mark.parametrize('t', [0.5, 1.0])
def test_every_single_cell_configuration_is_closed(t):
    for case in range(1, 256):
        v, f = O.mesh_one(_single(case), t)
        _check_closed(v, f, degenerate=t == 1.0)


def test_random_grids_are_closed():
    rng = np.random.default_rng(0)
    for r in range(120):
        n = (3, 4, 5, 6)[r % 4]
        vol = rng.random((n, n, n)).astype(np.float32)
        if r % 3 == 0:
            vol = np.where(vol < 0.5, 0.0, 0.5).astype(np.float32)              # binary, inside values equal to t
        v, f = O.mesh_one(vol, 0.5)
        if len(f):
            _check_closed(v, f, degenerate=r % 3 == 0)


def _grid(n):
    g = (np.arange(n) + 0.5) / n
    z, y, x = np.meshgrid(g, g, g, indexing='ij')
    return x - 0.5, y - 0.5, z - 0.5


def _field(sd, n):
    """Signed distance (positive inside, unit-cube units) -> occupancy with a one-voxel ramp around 0.5."""
    return np.clip(0.5 + sd * n, 0, 1).astype(np.float32)


def _shapes(n):
    x, y, z = _grid(n)
    d = np.sqrt(x * x + y * y + z * z)
    torus = 0.12 - np.sqrt((np.sqrt(x * x + y * y) - 0.28) ** 2 + z * z)
    two = np.maximum(0.15 - np.sqrt((x + 0.22) ** 2 + y * y + z * z), 0.15 - np.sqrt((x - 0.22) ** 2 + y * y + z * z))
    return {'ball': (_field(0.35 - d, n), 2), 'torus': (_field(torus, n), 0),
            'shell': (_field(np.minimum(0.4 - d, d - 0.2), n), 4), 'two_balls': (_field(two, n), 4)}


@pytest.mark.parametrize('name', ['ball', 'torus', 'shell', 'two_balls'])
def test_euler_characteristic(name):
    vol, chi = _shapes(32)[name]
    v, f = O.mesh_one(vol, 0.5)
    _check_closed(v, f)
    assert O.euler(v, f) == chi


def test_ball_volume():
    R = 0.35
    v, f = O.mesh_one(_shapes(24)['ball'][0], 0.5)
    assert abs(O.signed_volume(v, f) / (4 / 3 * np.pi * R ** 3) - 1) < 0.02


def test_vertices_interpolate_their_edges():
    """Independent scalar restatement: every crossing edge in (corner, axis) order and its fp32 vertex."""
    rng = np.random.default_rng(5)
    n = 4
    vol = rng.random((n, n, n)).astype(np.float32)
    vol[0, 1, 2], vol[1, 2, 3], vol[2, 2, 2], vol[3, 0, 1] = np.nan, np.inf, -3.0, 7.0
    for t in (0.3, 1.0):
        verts, _ = O.mesh_one(vol, t)
        t32 = np.float32(t)

        def val(k, j, i):
            if not (0 <= k < n and 0 <= j < n and 0 <= i < n):
                return np.float32(0)
            a = vol[k, j, i]
            return np.float32(0) if np.isnan(a) else np.float32(min(max(float(a), 0.0), 1.0))
        want = []
        for k in range(-1, n + 1):
            for j in range(-1, n + 1):
                for i in range(-1, n + 1):
                    p = (i, j, k)
                    for ax in range(3):
                        q = list(p)
                        q[ax] += 1
                        if q[ax] > n:
                            continue
                        a, b = val(k, j, i), val(q[2], q[1], q[0])
                        if (a >= t32) == (b >= t32):
                            continue
                        s = (t32 - a) / (b - a)
                        xyz = [(np.float32(c) + np.float32(0.5)) / np.float32(n) for c in p]
                        xyz[ax] = (np.float32(p[ax]) + np.float32(0.5) + s) / np.float32(n)
                        assert np.float32(0) <= s <= np.float32(1)
                        want.append(xyz)
        assert np.array_equal(verts.view(np.uint32), np.array(want, np.float32).view(np.uint32))


def test_obj_round_trip(tmp_path):
    from stereo_3d_reconstruction_b200.core import test as T
    rng = np.random.default_rng(2)
    v, f = O.mesh_one(rng.random((6, 6, 6)).astype(np.float32), 0.37)
    v = np.concatenate([v, np.array([[1e-38, 3.4e38, -0.1]], np.float32)])      # extremes of the format
    p = str(tmp_path / 'm.obj')
    T.write_obj(p, v, f)
    rv, rf = O.read_obj(p)
    assert np.array_equal(rv.view(np.uint32), v.view(np.uint32)) and np.array_equal(rf, f)
    with open(p) as fh:
        lines = fh.read().splitlines()
    assert lines[0].startswith('v ') and lines[-1].startswith('f ') and len(lines) == len(v) + len(f)
    assert min(int(x) for ln in lines if ln.startswith('f ') for x in ln.split()[1:]) == 1


def test_mesh_thresh_validation():
    from config import cfg as dcfg
    from stereo_3d_reconstruction_b200 import models as M
    c = dcfg.clone()
    assert M.mesh_thresh(c) == 0.5
    for good in (1.0, 1e-6, '0.25'):
        c.TEST.MESH_THRESH = good
        M.mesh_thresh(c)
    for bad in (0.0, -0.1, 1.0001, float('nan'), float('inf'), None, 'x', [0.5], 1e-46):
        c.TEST.MESH_THRESH = bad
        with pytest.raises(ValueError):
            M.mesh_thresh(c)
