"""Reference statement of s3d_voxel_mesh (include/s3d.h) in numpy: marching cubes over the zero-padded, clamped field with
the generated case table (stereo_3d_reconstruction_b200/mc_table.py), vertex ids by rank of their crossing edge, faces in
cell order, fp32 vertex arithmetic in the kernel's order.  Also the mesh checks the tests share and an OBJ reader."""
import numpy as np

from stereo_3d_reconstruction_b200 import mc_table

_TAB = np.zeros((256, mc_table.MAX_TRI, 3), np.int64)
_CNT = np.zeros(256, np.int64)
for _c, _tris in enumerate(mc_table.TABLE):
    _CNT[_c] = len(_tris)
    if _tris:
        _TAB[_c, :len(_tris)] = _tris
_EOFF = np.array([mc_table.edge_offset(e) for e in range(12)], np.int64)        # [12, (dx, dy, dz, axis)]


def bounds(n):
    return 3 * (n + 1) * (n + 2) ** 2, 5 * (n + 1) ** 3


def padded_field(vol):
    """One sample [n,n,n] -> the clamped field with one layer of 0 on every side, fp32 [n+2]^3 (index = grid index + 1)."""
    v = np.nan_to_num(np.asarray(vol, np.float32), nan=0.0, posinf=1.0, neginf=0.0)
    v = np.minimum(np.maximum(v, np.float32(0)), np.float32(1)).astype(np.float32)
    return np.pad(v, 1)


def mesh_one(vol, t):
    """One sample [n,n,n] at iso-level t -> (verts fp32 [V,3] xyz, faces int32 [F,3])."""
    n = vol.shape[0]
    t = np.float32(t)
    P = padded_field(vol)
    ins = P >= t
    m = n + 2
    keys, va, vb, lo = [], [], [], []
    for a in range(3):                               # axis a: x (last array dim), y, z
        ax = 2 - a
        sl0 = [slice(None)] * 3
        sl1 = [slice(None)] * 3
        sl0[ax], sl1[ax] = slice(0, m - 1), slice(1, m)
        cr = ins[tuple(sl0)] != ins[tuple(sl1)]
        k, j, i = np.nonzero(cr)
        keys.append(((k * m + j) * m + i) * 3 + a)
        va.append(P[tuple(sl0)][cr])
        vb.append(P[tuple(sl1)][cr])
        lo.append(np.stack([i, j, k], 1))
    keys = np.concatenate(keys)
    order = np.argsort(keys, kind='stable')
    keys = keys[order]
    va, vb = np.concatenate(va)[order], np.concatenate(vb)[order]
    lo = np.concatenate(lo)[order] - 1                 # grid coordinates of the lower corner, -1..n
    axis = keys % 3
    s = (t - va) / (vb - va)                           # fp32 throughout
    nf = np.float32(n)
    verts = (lo.astype(np.float32) + np.float32(0.5)) / nf
    along = (lo[np.arange(len(lo)), axis].astype(np.float32) + np.float32(0.5) + s) / nf
    verts[np.arange(len(lo)), axis] = along
    # cells: lower corner at padded index (k, j, i) in [0, n]^3, linear order
    case = np.zeros((n + 1,) * 3, np.int64)
    for c in range(8):
        cx, cy, cz = mc_table.corner_xyz(c)
        case |= ins[cz:cz + n + 1, cy:cy + n + 1, cx:cx + n + 1].astype(np.int64) << c
    case = case.reshape(-1)
    cells = np.nonzero(_CNT[case])[0]
    ck, cj, ci = np.unravel_index(cells, (n + 1,) * 3)
    tri = _TAB[case[cells]]                            # [C, 5, 3] edge ids
    valid = np.arange(mc_table.MAX_TRI)[None, :] < _CNT[case[cells]][:, None]
    off = _EOFF[tri]                                   # [C, 5, 3, 4]
    fk = ((ck[:, None, None] + off[..., 2]) * m + cj[:, None, None] + off[..., 1]) * m + ci[:, None, None] + off[..., 0]
    fkey = fk * 3 + off[..., 3]
    ids = np.searchsorted(keys, fkey)
    faces = ids[valid].reshape(-1, 3)
    assert np.array_equal(keys[faces.reshape(-1)], fkey[valid].reshape(-1))
    return verts.astype(np.float32), faces.astype(np.int32)


def mesh(vol, t):
    """[B,n,n,n] -> list of (verts, faces) per sample."""
    return [mesh_one(v, t) for v in np.asarray(vol)]


def closed_manifold(verts, faces):
    """Each directed edge exactly once and its reverse present, no repeated id in a face."""
    f = np.asarray(faces, np.int64)
    if len(f) == 0:
        return True
    if (f[:, 0] == f[:, 1]).any() or (f[:, 1] == f[:, 2]).any() or (f[:, 0] == f[:, 2]).any():
        return False
    e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    V = max(len(verts), int(f.max()) + 1)
    code = e[:, 0] * V + e[:, 1]
    u, cnt = np.unique(code, return_counts=True)
    if (cnt != 1).any():
        return False
    rev = e[:, 1] * V + e[:, 0]
    return bool(np.isin(rev, u).all())


def signed_volume(verts, faces):
    v = np.asarray(verts, np.float64)[np.asarray(faces, np.int64)]
    return float(np.einsum('ij,ij->i', v[:, 0], np.cross(v[:, 1], v[:, 2])).sum() / 6.0)


def euler(verts, faces):
    f = np.asarray(faces, np.int64)
    e = np.sort(np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]), 1)
    E = len(np.unique(e[:, 0] * (f.max() + 1) + e[:, 1]))
    return len(np.unique(f)) - E + len(f)


def read_obj(path):
    """-> (verts fp32 [V,3], faces int32 [F,3] 0-based) of a plain OBJ with `v x y z` and `f a b c` lines."""
    vs, fs = [], []
    with open(path) as fh:
        for line in fh:
            p = line.split()
            if not p:
                continue
            if p[0] == 'v':
                vs.append([np.float32(float(x)) for x in p[1:4]])
            elif p[0] == 'f':
                fs.append([int(x) - 1 for x in p[1:4]])
    return np.array(vs, np.float32).reshape(-1, 3), np.array(fs, np.int32).reshape(-1, 3)
