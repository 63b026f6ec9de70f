"""numpy restatement of the mesh preview kernels (pix2pix3d_b200/csrc/mesh_raster.cu): orthographic projection, fixed-point
coverage with a top-left rule, packed depth keys resolved to the nearest fragment and the lowest face id, and the diffuse
spot-light shading. The contract is the comment above p3d_mesh_raster in include/p3d.h; every fp32 operation here is one
numpy float32 operation in the kernels' order, so the two agree bit for bit.

Inputs are the kernels' own: vertices float32 [V,3], faces int64 [F,3], views float32 [N,18] (p3d_mesh_view_t: world2cam
rows 0-2, eye, spot axis). The views are not rebuilt from poses here; both sides take the same float32 values.
"""
import numpy as np

f32 = np.float32
GUARD_PX = f32(2 ** 21)
GREY = f32(0.8)
COS_CONE = f32(np.cos(np.pi / 4))
PI = f32(np.pi)
EMPTY = np.uint64(0xFFFFFFFFFFFFFFFF)
ZNEAR, ZFAR = 0.05, 100.0
CHUNK = 1 << 22                  # candidate pixels expanded at once


def scales(H, W, xmag, ymag):
    """(kx, ky, hx, hy) = (W / (2 xmag), H / (2 ymag), W / 2, H / 2) in fp32."""
    return f32(W) / (f32(2) * f32(xmag)), f32(H) / (f32(2) * f32(ymag)), f32(0.5) * f32(W), f32(0.5) * f32(H)


def _sum3(a0, a1, a2):
    return (a0 + a1) + a2


def project(vertices, view, H, W, xmag, ymag):
    """Screen x, y (pixels, row 0 at the top) and depth -z_cam of every vertex, fp32 [V]."""
    v = np.asarray(vertices, f32).reshape(-1, 3)
    m = np.asarray(view, f32)[:12].reshape(3, 4)
    c = [_sum3(m[r, 0] * v[:, 0], m[r, 1] * v[:, 1], m[r, 2] * v[:, 2]) + m[r, 3] for r in range(3)]
    kx, ky, hx, hy = scales(H, W, xmag, ymag)
    return c[0] * kx + hx, hy - c[1] * ky, -c[2]


def _face_ok(vertices, faces):
    """Faces whose indices are in [0, V) and whose corners are finite (the rest are dropped silently)."""
    V = len(vertices)
    inb = ((faces >= 0) & (faces < V)).all(1)
    fin = np.isfinite(vertices).all(1)
    ok = inb.copy()
    ok[inb] = fin[faces[inb]].all(1)
    return ok


def setup(sx, sy, d, tri):
    """Triangle setup of faces `tri` (their vertex ids [T,3]) from the projected vertices: dict of fixed-point corners X, Y,
    depths, edge vectors after the winding flip, area A > 0 (0 where the triangle is skipped), clipped box, and `guard`
    (a corner outside the guard band). Entries of guarded triangles are meaningless."""
    with np.errstate(invalid='ignore'):
        gx, gy = sx[tri], sy[tri]
        guard = (~(np.abs(gx) <= GUARD_PX) | ~(np.abs(gy) <= GUARD_PX)).any(1)
        X = np.where(guard[:, None], 0, np.rint(gx * f32(256))).astype(np.int64)
        Y = np.where(guard[:, None], 0, np.rint(gy * f32(256))).astype(np.int64)
    A = (X[:, 1] - X[:, 0]) * (Y[:, 2] - Y[:, 0]) - (Y[:, 1] - Y[:, 0]) * (X[:, 2] - X[:, 0])
    s = np.where(A < 0, -1, 1)
    nxt, nxt2 = [1, 2, 0], [2, 0, 1]
    return dict(X=X, Y=Y, d=d[tri], guard=guard, A=s * A,
                dx=s[:, None] * (X[:, nxt2] - X[:, nxt]), dy=s[:, None] * (Y[:, nxt2] - Y[:, nxt]),
                j0=np.maximum(0, (X.min(1) + 127) >> 8), j1=(X.max(1) - 128) >> 8,
                i0=np.maximum(0, (Y.min(1) + 127) >> 8), i1=(Y.max(1) - 128) >> 8)


def cover(t, sel, i, j):
    """Coverage of pixel (i[p], j[p]) by triangle sel[p] of setup `t`: (covered bool [P], barycentrics fp32 [P,3])."""
    px, py = 256 * j.astype(np.int64) + 128, 256 * i.astype(np.int64) + 128
    X, Y, dx, dy = t['X'][sel], t['Y'][sel], t['dx'][sel], t['dy'][sel]
    nxt = [1, 2, 0]
    E = dx * (py[:, None] - Y[:, nxt]) - dy * (px[:, None] - X[:, nxt])
    top_left = (dy < 0) | ((dy == 0) & (dx > 0))
    covered = ((E > 0) | ((E == 0) & top_left)).all(1)
    b = E.astype(f32) / t['A'][sel].astype(f32)[:, None]         # int64 -> fp32 conversions round to nearest
    return covered, b


def _bary(b, a):
    """(b0 a0 + b1 a1) + b2 a2 for a [P,3] or [P,3,C]."""
    if a.ndim == 3:
        b = b[:, :, None]
    return _sum3(b[:, 0] * a[:, 0], b[:, 1] * a[:, 1], b[:, 2] * a[:, 2])


def raster(vertices, faces, views, H, W, xmag, ymag, znear=ZNEAR, zfar=ZFAR):
    """p3d_mesh_raster: (depth keys uint64 [N,H,W], number of (face, view) pairs dropped by the guard band)."""
    vertices = np.asarray(vertices, f32).reshape(-1, 3)
    faces = np.asarray(faces, np.int64).reshape(-1, 3)
    views = np.asarray(views, f32).reshape(-1, 18)
    znear, zfar = f32(znear), f32(zfar)
    keys = np.full((len(views), H, W), EMPTY, np.uint64)
    fid = np.flatnonzero(_face_ok(vertices, faces))
    tri = faces[fid]
    guards = 0
    for n, view in enumerate(views):
        sx, sy, d = project(vertices, view, H, W, xmag, ymag)
        t = setup(sx, sy, d, tri)
        guards += int(t['guard'].sum())
        j1, i1 = np.minimum(W - 1, t['j1']), np.minimum(H - 1, t['i1'])
        draw = np.flatnonzero(~t['guard'] & (t['A'] != 0) & (t['j0'] <= j1) & (t['i0'] <= i1))
        bw = (j1 - t['j0'] + 1)[draw]
        cnt = bw * (i1 - t['i0'] + 1)[draw]
        flat = keys[n].reshape(-1)
        ends = np.cumsum(cnt)
        lo = 0
        while lo < len(draw):
            hi = max(lo + 1, int(np.searchsorted(ends, (ends[lo - 1] if lo else 0) + CHUNK)))
            c = cnt[lo:hi]
            sel = np.repeat(draw[lo:hi], c)
            local = np.arange(int(c.sum())) - np.repeat(np.cumsum(c) - c, c)
            w = np.repeat(bw[lo:hi], c)
            i, j = t['i0'][sel] + local // w, t['j0'][sel] + local % w
            covered, b = cover(t, sel, i, j)
            dd = _bary(b, t['d'][sel])
            keep = covered & (dd >= znear) & (dd <= zfar)
            key = (dd[keep].view(np.uint32).astype(np.uint64) << np.uint64(32)) | fid[sel[keep]].astype(np.uint64)
            np.minimum.at(flat, i[keep] * W + j[keep], key)
            lo = hi
    return keys, guards


def shade(keys, vertices, faces, views, xmag, ymag, vertex_colors=None, light_intensity=3.0):
    """p3d_mesh_shade: uint8 [N,H,W,3] from the depth keys of `raster`."""
    keys = np.asarray(keys).view(np.uint64)
    N, H, W = keys.shape
    vertices = np.asarray(vertices, f32).reshape(-1, 3)
    faces = np.asarray(faces, np.int64).reshape(-1, 3)
    views = np.asarray(views, f32).reshape(-1, 18)
    intensity = f32(light_intensity)
    out = np.full((N, H, W, 3), 255, np.uint8)
    for n, view in enumerate(views):
        pix = np.flatnonzero(keys[n].reshape(-1) != EMPTY)
        if not len(pix):
            continue
        face = (keys[n].reshape(-1)[pix] & np.uint64(0xFFFFFFFF)).astype(np.int64)
        i, j = pix // W, pix % W
        sx, sy, d = project(vertices, view, H, W, xmag, ymag)
        tri = faces[face]
        t = setup(sx, sy, d, tri)
        covered, b = cover(t, np.arange(len(pix)), i, j)
        assert covered.all() and not t['guard'].any()
        w = vertices[tri]                                                   # [P,3 corners,3]
        if vertex_colors is None:
            colour = np.full((len(pix), 3), GREY, f32)
        else:
            colour = _bary(b, np.asarray(vertex_colors, np.uint8)[tri].astype(f32) / f32(255))
        e1, e2 = w[:, 1] - w[:, 0], w[:, 2] - w[:, 0]
        a, z = [1, 2, 0], [2, 0, 1]
        nrm = e1[:, a] * e2[:, z] - e1[:, z] * e2[:, a]
        q = view[12:15][None, :] - _bary(b, w)
        with np.errstate(all='ignore'):
            dot = lambda u, v: _sum3(u[:, 0] * v[:, 0], u[:, 1] * v[:, 1], u[:, 2] * v[:, 2])
            nlen = np.sqrt(dot(nrm, nrm))
            r2 = dot(q, q)
            nl, ll = nrm / nlen[:, None], q / np.sqrt(r2)[:, None]
            ndl = dot(nl, ll)
            cone = dot(ll, np.broadcast_to(view[15:18], ll.shape))
            s = (intensity * np.where(ndl > 0, ndl, f32(0))) / (PI * r2)
            s = np.where(cone > -COS_CONE, f32(0), s)
            x = ((f32(255) * colour) * s[:, None]) + f32(0.5)
            out[n].reshape(-1, 3)[pix] = np.where(x < 255, np.floor(x), f32(255)).astype(np.uint8)
    return out


def render(vertices, faces, views, H, W, xmag, ymag, vertex_colors=None, light_intensity=3.0, znear=ZNEAR, zfar=ZFAR):
    """raster + shade -> (frames uint8 [N,H,W,3], depth keys, guard drops)."""
    keys, guards = raster(vertices, faces, views, H, W, xmag, ymag, znear, zfar)
    return shade(keys, vertices, faces, views, xmag, ymag, vertex_colors, light_intensity), keys, guards
