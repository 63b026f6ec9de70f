"""numpy restatement of the geometry path of applications/extract_mesh.py (get_sigma_field_np :60-81, extract_geometry
:84-96) and the marching-cubes contract that pix2pix3d_b200/csrc/marching_cubes.cu implements.

The reference calls PyMCubes (`mcubes.marching_cubes(u, threshold)`), which is not available offline. This module defines
the mesh instead, and generates the triangle table the CUDA kernels use (`python -m p3d_oracle.mesh` from oracle/ writes
pix2pix3d_b200/csrc/mc_table.cuh).

Mesh definition:
- a grid value is inside when v > threshold (compared in float64); NaN is outside, v == threshold is outside;
- one vertex per grid edge whose endpoints differ in inside-ness. The edge p -> p + e_axis is owned by p; its vertex is
  p + t * e_axis with t = (thr - v_p) / (v_{p+e} - v_p) in float64. Vertices are ordered by owning point in C order, and
  by axis within a point. An edge with a NaN endpoint gets a NaN coordinate;
- faces: cubes in C order, inside a cube in table order, oriented outward (normals point toward lower values).

Triangle table (face walk): corners c = (c & 1, c >> 1 & 1, c >> 2 & 1) along axes (0, 1, 2); the 12 edges are the corner
pairs that differ in one bit, axis-major (edges 4a..4a+3 run along axis a, ordered by their lower corner). On each cube face
the crossing edges are joined by segments; a face with four crossings (diagonal corners inside) is resolved by cutting off
each inside corner, a rule that depends only on the face's own signs, so the two cubes sharing a face agree and the mesh
has no cracks. Segments are oriented so that, seen from outside the cube, the inside lies on a fixed side, chained into
loops and fan-triangulated from each loop's lowest edge id. Cutting off inside corners joins the outside regions across
an ambiguous face, and fan diagonals across such faces can make one vertex pair shared by four triangles; the mesh stays
closed in the directed-edge sense (every directed edge is matched by its reverse).

Unverified (cannot be checked offline): whether PyMCubes picks the same triangles in ambiguous cubes, its winding, and the
last float64 ulp of its interpolation. The vertex set is the one any marching cubes with these inside-ness rules produces.
"""
import os

import numpy as np

CORNER = np.array([(c & 1, c >> 1 & 1, c >> 2 & 1) for c in range(8)], np.int64)          # [8,3] offsets
EDGE_AXIS = np.array([e // 4 for e in range(12)], np.int64)
EDGE_CORNER = np.array([[b for b in range(8) if not b >> a & 1][e % 4] for a in range(3) for e in range(4 * a, 4 * a + 4)],
                       np.int64)                                                          # lower corner of each edge


def _midpoint(e):
    p = CORNER[EDGE_CORNER[e]].astype(np.float64)
    p[EDGE_AXIS[e]] += 0.5
    return p


# the six cube faces: (axis, side); corners of a face have bit `axis` == side
FACES = [(a, s) for a in range(3) for s in range(2)]


def _face_edges(a, s):
    return [e for e in range(12) if EDGE_AXIS[e] != a and (EDGE_CORNER[e] >> a & 1) == s]


def _face_segments(cfg, side):
    """Directed segments (face index, e_from, e_to) joining the crossing edges of each face. `side` = +1: the inside lies
    on the left of the segment seen from outside the cube; -1: on the right."""
    inside = [bool(cfg >> c & 1) for c in range(8)]
    segs = []
    for f, (a, s) in enumerate(FACES):
        n = np.zeros(3)
        n[a] = 2 * s - 1                                                                  # outward normal
        cross = [e for e in _face_edges(a, s) if inside[EDGE_CORNER[e]] != inside[EDGE_CORNER[e] + (1 << EDGE_AXIS[e])]]
        face_in = [c for c in range(8) if (c >> a & 1) == s and inside[c]]
        if len(cross) == 2:
            pairs = [(cross[0], cross[1], face_in[0])]
        elif len(cross) == 4:                                                             # ambiguous: cut off each inside corner
            pairs = []
            for c in face_in:
                inc = [e for e in cross if c in (EDGE_CORNER[e], EDGE_CORNER[e] + (1 << EDGE_AXIS[e]))]
                pairs.append((inc[0], inc[1], c))
        else:
            assert not cross
            pairs = []
        for e1, e2, c in pairs:
            p1, p2 = _midpoint(e1), _midpoint(e2)
            left = np.dot(np.cross(p2 - p1, CORNER[c] - p1), n) > 0
            segs.append((f, e1, e2) if left == (side > 0) else (f, e2, e1))
    return segs


def _loops(segs):
    nxt = {}
    for _, e1, e2 in segs:
        assert e1 not in nxt
        nxt[e1] = e2
    assert sorted(nxt) == sorted(nxt.values()), 'every crossing edge starts one segment and ends one'
    loops, seen = [], set()
    for e in sorted(nxt):
        if e in seen:
            continue
        loop = [e]
        seen.add(e)
        while nxt[loop[-1]] != e:
            loop.append(nxt[loop[-1]])
            seen.add(loop[-1])
        loops.append(loop)                                                                # starts at its lowest edge id
    return loops


def _fan(loops):
    return [(lp[0], lp[i], lp[i + 1]) for lp in loops for i in range(1, len(lp) - 1)]


def _outward_side():
    """Side that makes the triangles outward: with only corner 0 inside, the normal must point away from it."""
    for side in (1, -1):
        (t,) = _fan(_loops(_face_segments(1, side)))
        p = [_midpoint(e) for e in t]
        if np.dot(np.cross(p[1] - p[0], p[2] - p[0]), np.ones(3)) > 0:
            return side
    raise AssertionError('no orientation is outward')


SIDE = _outward_side()


def face_segments(cfg):
    """Directed boundary segments of configuration `cfg` (bit c = corner c inside), in the table's final orientation."""
    return _face_segments(cfg, SIDE)


def cube_loops(cfg):
    return _loops(face_segments(cfg))


def cube_triangles(cfg):
    return _fan(cube_loops(cfg))


def triangle_table():
    """(tri_count [256] int64, tri_edges [256,16] int8: 3 edge ids per triangle, -1 padded)."""
    count = np.zeros(256, np.int64)
    table = np.full((256, 16), -1, np.int8)
    for cfg in range(256):
        tris = cube_triangles(cfg)
        count[cfg] = len(tris)
        table[cfg, :3 * len(tris)] = np.array(tris, np.int8).reshape(-1)
    return count, table


TRI_COUNT, TRI_TABLE = triangle_table()
MAX_TRIANGLES = int(TRI_COUNT.max())


def table_header():
    """Text of pix2pix3d_b200/csrc/mc_table.cuh."""
    lines = ['// GENERATED by oracle/p3d_oracle/mesh.py (python -m p3d_oracle.mesh, run from oracle/) -- do not edit.',
             '// Marching-cubes triangle table built by a face walk; see that module for the definition.',
             '// Corner c = (c & 1, c >> 1 & 1, c >> 2 & 1) along axes (0, 1, 2). Edge e runs along axis e / 4 from corner',
             '// kMcEdgeCorner[e]. kMcTriEdges[cfg] holds 3 edge ids per triangle (-1 padded), cfg bit c = corner c inside.',
             '#pragma once', '',
             f'#define P3D_MC_MAX_TRIANGLES {MAX_TRIANGLES}', '',
             'static __constant__ signed char kMcEdgeCorner[12] = {' + ', '.join(str(int(b)) for b in EDGE_CORNER) + '};', '',
             'static __constant__ unsigned char kMcTriCount[256] = {']
    for r in range(0, 256, 32):
        lines.append('    ' + ', '.join(str(int(n)) for n in TRI_COUNT[r:r + 32]) + ',')
    lines += ['};', '', 'static __constant__ signed char kMcTriEdges[256][16] = {']
    for cfg in range(256):
        lines.append('    {' + ', '.join(str(int(e)) for e in TRI_TABLE[cfg]) + '},')
    lines += ['};', '']
    return '\n'.join(lines)


HEADER_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..', '..', 'pix2pix3d_b200', 'csrc', 'mc_table.cuh')


# ---------------------------------------------------------------------------------------------
# marching cubes on a dense grid
# ---------------------------------------------------------------------------------------------
def marching_cubes(volume, threshold):
    """(vertices float64 [V,3] in index coordinates, faces int64 [F,3]) of the mesh defined above."""
    v = np.ascontiguousarray(volume, np.float32)
    assert v.ndim == 3 and min(v.shape) >= 2
    nx, ny, nz = v.shape
    thr = np.float64(threshold)
    inside = v.astype(np.float64) > thr
    cross = np.zeros((nx, ny, nz, 3), bool)
    cross[:-1, :, :, 0] = inside[:-1] != inside[1:]
    cross[:, :-1, :, 1] = inside[:, :-1] != inside[:, 1:]
    cross[:, :, :-1, 2] = inside[:, :, :-1] != inside[:, :, 1:]
    owned = np.flatnonzero(cross.reshape(-1))                                           # point-major, then axis
    vid = np.full(cross.size, -1, np.int64)
    vid[owned] = np.arange(owned.size)
    p, a = owned // 3, owned % 3
    flat = v.reshape(-1)
    vp = flat[p].astype(np.float64)
    vq = flat[p + np.array([ny * nz, nz, 1])[a]].astype(np.float64)
    with np.errstate(invalid='ignore', divide='ignore'):
        t = (thr - vp) / (vq - vp)
    verts = np.stack(np.unravel_index(p, (nx, ny, nz)), 1).astype(np.float64)
    verts[np.arange(owned.size), a] += t

    cfg = np.zeros((nx - 1, ny - 1, nz - 1), np.int64)
    for c, (ox, oy, oz) in enumerate(CORNER):
        cfg |= inside[ox:ox + nx - 1, oy:oy + ny - 1, oz:oz + nz - 1].astype(np.int64) << c
    cfg = cfg.reshape(-1)
    cubes = np.flatnonzero(TRI_COUNT[cfg])                                               # C order over cubes
    ci, cj, ck = np.unravel_index(cubes, (nx - 1, ny - 1, nz - 1))
    edge_vid = np.empty((cubes.size, 12), np.int64)
    for e in range(12):
        ox, oy, oz = CORNER[EDGE_CORNER[e]]
        edge_vid[:, e] = vid[(((ci + ox) * ny + (cj + oy)) * nz + (ck + oz)) * 3 + EDGE_AXIS[e]]
    tri_edges = TRI_TABLE[cfg[cubes]][:, :3 * MAX_TRIANGLES].astype(np.int64)
    faces = np.take_along_axis(edge_vid, np.maximum(tri_edges, 0), 1).reshape(cubes.size, MAX_TRIANGLES, 3)
    faces = faces[np.arange(MAX_TRIANGLES)[None, :] < TRI_COUNT[cfg[cubes]][:, None]]
    assert (faces >= 0).all()
    return verts, faces.reshape(-1, 3)


# ---------------------------------------------------------------------------------------------
# extract_mesh.py: point layout and scaling
# ---------------------------------------------------------------------------------------------
def linspace_f32(start, end, steps):
    """torch.linspace(start, end, steps) on the CPU in float32 (the axis of get_sigma_field_np, extract_mesh.py:63):
    step = (end - start) / (steps - 1); the first half counts up from start, the second half down from end, each element
    rounded once (torch's CPU kernel uses a fused multiply-add; the float64 products and sums here are exact for
    float32 operands and steps < 2^20, so the cast is that one rounding)."""
    start, end = np.float32(start), np.float32(end)
    step = np.float64((end - start) / np.float32(steps - 1))
    i = np.arange(steps)
    lo = np.float64(start) + step * i
    hi = np.float64(end) - step * (steps - 1 - i)
    return np.where(i < steps // 2, lo, hi).astype(np.float32)


def sigma_grid_points(axis):
    """[R,R,R,3] float32 query points of get_sigma_field_np (extract_mesh.py:60-81): grid[i,j,k] is sigma at
    (X[i], X[j], X[k]), the meshgrid(..., indexing='ij') order of each 64^3 block placed at its offset."""
    axis = np.asarray(axis, np.float32)
    return np.stack(np.meshgrid(axis, axis, axis, indexing='ij'), -1)


def scale_vertices(vertices, resolution, bound):
    """extract_geometry (extract_mesh.py:92-95): index space -> [-bound, bound]^3 in float64, then one cast to float32."""
    b_min = np.array([-bound, -bound, -bound])
    b_max = np.array([bound, bound, bound])
    return (vertices / (resolution - 1.0) * (b_max - b_min)[None, :] + b_min[None, :]).astype('float32')


if __name__ == '__main__':
    with open(HEADER_PATH, 'w') as fh:
        fh.write(table_header())
    print(os.path.normpath(HEADER_PATH))
