# -*- coding: utf-8 -*-
"""Marching-cubes case table of s3d_voxel_mesh, generated from its rule (pure Python, no dependencies).

One module states the rule; csrc/mc_table.cuh is its output (`python -m stereo_3d_reconstruction_b200.mc_table`), and the
test oracle (tests/mesh_oracle.py) builds its meshes from the same tables, so the two can never drift apart.

Numbering.  Corner c of a cell is (cx, cy, cz) = (c & 1, c >> 1 & 1, c >> 2 & 1).  Edge e runs along axis a = e >> 2 from
the corner with 0 on a to the one with 1; its bits on the other two axes o0 < o1 are e & 1 and e >> 1 & 1.  The case of a
cell is sum(inside(c) << c).

Rule.
  1. On each of the 6 cube faces, join the crossing edges with segments.  A face with 4 crossings (inside corners on a
     diagonal) gets one segment around each inside corner: inside corners are separated.  The choice depends on the four
     corners of that face alone, so the two cells that share the face always agree, and the mesh is closed.
  2. Every crossing edge lies on two faces, so the segments form disjoint closed loops.  Each loop starts at its lowest
     edge id and is oriented so that its Newell normal (over the edge midpoints) points from the inside corners of its
     edges to their outside corners.  Loops come in order of their first edge.
  3. Each loop is fan-triangulated from the first vertex, in loop order, whose fan diagonals never join two edges of one
     cube face (a diagonal on a face would be shared with the neighbouring cell's triangles and make the mesh
     non-manifold).  Triangles keep the loop's orientation: (v1 - v0) x (v2 - v0) points from inside to outside.
The result needs at most 5 triangles per case.
"""
import sys

MAX_TRI = 5


def corner_xyz(c):
    return (c & 1, (c >> 1) & 1, (c >> 2) & 1)


def edge_corners(e):
    """-> (lower corner, upper corner) of edge e."""
    a = e >> 2
    o0, o1 = [x for x in range(3) if x != a]
    p = [0, 0, 0]
    p[o0], p[o1] = e & 1, (e >> 1) & 1
    q = list(p)
    q[a] = 1
    return p[0] | p[1] << 1 | p[2] << 2, q[0] | q[1] << 1 | q[2] << 2


def edge_offset(e):
    """-> (dx, dy, dz, axis): the edge's lower corner relative to the cell's corner 0, and its axis."""
    c0, _ = edge_corners(e)
    x, y, z = corner_xyz(c0)
    return x, y, z, e >> 2


def _edge_between(c0, c1):
    for e in range(12):
        if set(edge_corners(e)) == {c0, c1}:
            return e
    raise AssertionError((c0, c1))


def _faces():
    """The 6 cube faces as 4 corners in cyclic order, each with the 4 edges between consecutive corners."""
    out = []
    for f in range(3):
        u, v = [x for x in range(3) if x != f]
        for s in (0, 1):
            cyc = []
            for bu, bv in ((0, 0), (1, 0), (1, 1), (0, 1)):
                p = [0, 0, 0]
                p[f], p[u], p[v] = s, bu, bv
                cyc.append(p[0] | p[1] << 1 | p[2] << 2)
            out.append((cyc, [_edge_between(cyc[i], cyc[(i + 1) % 4]) for i in range(4)]))
    return out


FACES = _faces()
_EDGE_FACES = [frozenset(i for i, (_, es) in enumerate(FACES) if e in es) for e in range(12)]


def _share_face(e0, e1):
    return bool(_EDGE_FACES[e0] & _EDGE_FACES[e1])


def _midpoint(e):
    c0, c1 = edge_corners(e)
    return tuple((a + b) / 2 for a, b in zip(corner_xyz(c0), corner_xyz(c1)))


def _loops(case):
    inside = [(case >> c) & 1 for c in range(8)]
    nbr = {}
    for cyc, es in FACES:
        cross = [e for e in es if inside[edge_corners(e)[0]] != inside[edge_corners(e)[1]]]
        if len(cross) == 2:
            segs = [tuple(cross)]
        elif len(cross) == 4:                               # inside corners on a diagonal: separate them
            segs = [(es[(i - 1) % 4], es[i]) for i in range(4) if inside[cyc[i]]]
        else:
            segs = []
        for a, b in segs:
            nbr.setdefault(a, []).append(b)
            nbr.setdefault(b, []).append(a)
    assert all(len(v) == 2 for v in nbr.values())
    loops, seen = [], set()
    for start in sorted(nbr):
        if start in seen:
            continue
        loop, prev, cur = [start], None, start
        seen.add(start)
        while True:
            a, b = nbr[cur]
            nxt = b if a == prev else a
            if nxt == start:
                break
            loop.append(nxt)
            seen.add(nxt)
            prev, cur = cur, nxt
        # orientation: Newell normal . (outside - inside corner, summed over the loop's edges) > 0
        pts = [_midpoint(e) for e in loop]
        nrm = [0.0, 0.0, 0.0]
        for i, p in enumerate(pts):
            q = pts[(i + 1) % len(pts)]
            nrm[0] += (p[1] - q[1]) * (p[2] + q[2])
            nrm[1] += (p[2] - q[2]) * (p[0] + q[0])
            nrm[2] += (p[0] - q[0]) * (p[1] + q[1])
        d = [0, 0, 0]
        for e in loop:
            c0, _ = edge_corners(e)
            d[e >> 2] += 1 if inside[c0] else -1                # inside at the lower corner: outside is +axis
        dot = sum(a * b for a, b in zip(nrm, d))
        assert dot != 0, (case, loop)
        if dot < 0:
            loop = [loop[0]] + loop[:0:-1]
        loops.append(loop)
    return loops


def _fan(loop):
    m = len(loop)
    for r in range(m):
        if all(not _share_face(loop[r], loop[(r + k) % m]) for k in range(2, m - 1)):
            return [(loop[r], loop[(r + k) % m], loop[(r + k + 1) % m]) for k in range(1, m - 1)]
    raise AssertionError('no fan root for loop %s' % (loop,))


def case_loops(case):
    """Loops of a case: lists of edge ids, oriented, each starting at its lowest edge."""
    return _loops(case)


def build_table():
    """-> list over the 256 cases of the triangles (edge-id triples), in table order."""
    table = []
    for case in range(256):
        tris = [t for loop in _loops(case) for t in _fan(loop)]
        assert len(tris) <= MAX_TRI, (case, tris)
        table.append(tris)
    return table


TABLE = build_table()


def header():
    """The text of csrc/mc_table.cuh."""
    cnt = [len(t) for t in TABLE]
    lines = [
        '// Marching-cubes case table of s3d_voxel_mesh.  GENERATED by stereo_3d_reconstruction_b200/mc_table.py, which',
        '// states the rule and the corner / edge numbering; do not edit (tests/test_voxel_mesh.py compares the two).',
        '#pragma once',
        '#include <stdint.h>',
        '',
        'namespace s3d {',
        '',
        'constexpr int kMcMaxTri = %d;' % MAX_TRI,
        '',
        '// triangles per case (bit c of the case set: corner c inside)',
        'static __device__ const uint8_t kMcTriCount[256] = {',
    ]
    for r in range(0, 256, 32):
        lines.append('  ' + ', '.join(str(c) for c in cnt[r:r + 32]) + ',')
    lines += ['};', '', '// their edge triples in table order, padded with 0',
              'static __device__ const uint8_t kMcTriEdges[256][3 * kMcMaxTri] = {']
    for case, tris in enumerate(TABLE):
        flat = [e for t in tris for e in t] + [0] * (3 * (MAX_TRI - len(tris)))
        lines.append('  {%s},  // %d' % (', '.join('%2d' % e for e in flat), case))
    lines += ['};', '', '}  // namespace s3d', '']
    return '\n'.join(lines)


if __name__ == '__main__':
    sys.stdout.write(header())
