"""Mesh preview without a GPU: the numpy restatement of the rasterizer and shader (coverage, projection, depth, shading),
the view setup, the turntable orbit and the GIF writer."""
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from conftest import ROOT
from p3d_oracle import mesh as M
from p3d_oracle import mesh_render as R
from test_mesh_cpu import sphere


def look_down_z(z=1.0, x=0.0, y=0.0):
    """OpenGL cam2world at (x, y, z) looking down -z, +y up."""
    c = np.eye(4)
    c[:3, 3] = (x, y, z)
    return c


def views_of(*poses):
    from pix2pix3d_b200 import native
    return native.mesh_views(np.stack(poses)).numpy()


def covered(keys):
    return keys != R.EMPTY


def test_int64_to_float32_conversion_rounds_to_nearest():
    """The oracle converts the integer edge functions with astype(float32); the kernels with __ll2float_rn. Both must be one
    round-to-nearest-even (no detour through float64, which rounds twice)."""
    x = np.array([2 ** 60 + 2 ** 36 + 1, -(2 ** 60 + 2 ** 36 + 1), 2 ** 61 - 1, 3 * 2 ** 40 + 2 ** 16], np.int64)
    want = [2 ** 60 + 2 ** 37, -(2 ** 60 + 2 ** 37), 2 ** 61, 3 * 2 ** 40]
    assert [int(v) for v in x.astype(np.float32)] == want


def test_view_struct_layout():
    from pix2pix3d_b200 import _lib
    prog = ('#include <stdio.h>\n#include <stddef.h>\n#include "p3d.h"\nint main(){printf("%zu %zu %zu\\n", sizeof(p3d_mesh_view_t),'
            ' offsetof(p3d_mesh_view_t, eye), offsetof(p3d_mesh_view_t, spot_axis));return 0;}\n')
    with tempfile.TemporaryDirectory() as td:
        c = os.path.join(td, 't.c')
        open(c, 'w').write(prog)
        subprocess.check_call(['gcc', '-I', os.path.join(ROOT, 'include'), c, '-o', os.path.join(td, 't')])
        size, eye, axis = (int(v) for v in subprocess.check_output([os.path.join(td, 't')]).split())
    assert (size, eye, axis) == (4 * _lib.MESH_VIEW_FLOATS, 48, 60)


def test_mesh_views_inverts_the_pose():
    from pix2pix3d_b200 import mesh
    poses = mesh.turntable_poses([0.0, 0.0, 0.2], 1.2, -3.14 / 2, np.pi, np.pi / 2, num_frames=7, device='cpu')
    v = views_of(*poses.double().numpy())
    for pose, view in zip(poses.double().numpy(), v):
        w2c = np.vstack([view[:12].reshape(3, 4), [0, 0, 0, 1]])
        assert np.abs(w2c @ pose - np.eye(4)).max() < 1e-6
        assert np.array_equal(view[12:15], pose[:3, 3].astype(np.float32))
        assert np.array_equal(view[15:18], (-pose[:3, 2]).astype(np.float32))


def test_projection_orientation_and_extents():
    """x right, row 0 at the top, depth = distance in front of the camera; xmag / ymag are the half-extents."""
    (view,) = views_of(look_down_z(2.0))
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [-0.5, -0.25, 1.5]], np.float32)
    sx, sy, d = R.project(v, view, 8, 16, 2.0, 1.0)
    assert np.array_equal(sx, np.float32([8, 12, 8, 6]))          # 16 px over 2 * xmag = 4 units
    assert np.array_equal(sy, np.float32([4, 4, 0, 5]))           # 8 px over 2 * ymag = 2 units, +y up
    assert np.array_equal(d, np.float32([2, 2, 2, 0.5]))


def small_triangle(x, y, z=0.0, r=0.01):
    return np.array([[x - r, y - r, z], [x + r, y - r, z], [x, y + r, z]], np.float32)


def test_small_triangle_lands_on_its_pixel():
    views = views_of(look_down_z())
    # pixel (i=1, j=6) of an 8x8 image with xmag = ymag = 1 has its centre at world (0.625, 0.625)
    keys, drops = R.raster(small_triangle(0.625, 0.625), [[0, 1, 2]], views, 8, 8, 1.0, 1.0)
    assert drops == 0
    assert list(zip(*np.nonzero(covered(keys[0])))) == [(1, 6)]
    # xmag = ymag = 2 halve the scale: twice the coordinates land on the same pixel, and (0.75, 0.75) on (i=2, j=5)
    keys, _ = R.raster(small_triangle(1.25, 1.25), [[0, 1, 2]], views, 8, 8, 2.0, 2.0)
    assert list(zip(*np.nonzero(covered(keys[0])))) == [(1, 6)]
    keys, _ = R.raster(small_triangle(0.75, 0.75), [[0, 1, 2]], views, 8, 8, 2.0, 2.0)
    assert list(zip(*np.nonzero(covered(keys[0])))) == [(2, 5)]


def screen_to_world(p, H, W, xmag, ymag):
    """Inverse of the projection of look_down_z(): screen (x, y) -> world (x, y, 0)."""
    return np.array([(p[0] - W / 2) * 2 * xmag / W, (H / 2 - p[1]) * 2 * ymag / H, 0.0])


def test_fan_covers_each_pixel_exactly_once():
    """A square cut into a fan of eight triangles whose shared edges run through rows, columns and diagonals of pixel
    centres: drawn one triangle at a time, no pixel is covered twice and every pixel inside the square once, for either
    winding of each triangle."""
    H = W = 16
    c = (8.5, 8.5)
    rim = [(2.5, 2.5), (8.5, 2.5), (14.5, 2.5), (14.5, 8.5), (14.5, 14.5), (8.5, 14.5), (2.5, 14.5), (2.5, 8.5)]
    verts = np.array([screen_to_world(p, H, W, 1.0, 1.0) for p in [c] + rim], np.float32)
    views = views_of(look_down_z())
    for flip in (0, 0b01010101, 0b11111111):
        count = np.zeros((H, W), np.int64)
        for k in range(8):
            f = [0, 1 + k, 1 + (k + 1) % 8]
            if flip >> k & 1:
                f = [f[0], f[2], f[1]]
            keys, _ = R.raster(verts, [f], views, H, W, 1.0, 1.0)
            count += covered(keys[0])
        assert count.max() == 1, flip
        assert (count[3:14, 3:14] == 1).all(), flip
        assert count[:2].sum() == count[15:].sum() == count[:, :2].sum() == count[:, 15:].sum() == 0


def sphere_mesh():
    centre = np.array([31.3, 30.8, 32.1])
    v, f = M.marching_cubes(sphere((64, 64, 64), centre, 25.0), 0.0)
    return M.scale_vertices(v, 64, 0.5), f, centre / 63 - 0.5, 25.0 / 63


def test_sphere_silhouette_has_no_holes():
    from pix2pix3d_b200 import mesh
    v, f, centre, radius = sphere_mesh()
    poses = mesh.turntable_poses([0.0, 0.0, 0.0], 1.0, 3.14 / 2, 0.35, 0.25, num_frames=4, device='cpu')
    views = views_of(*poses.double().numpy())
    H = W = 96
    keys, drops = R.raster(v, f, views, H, W, 0.6, 0.6)
    assert drops == 0
    for n, view in enumerate(views):
        sx, sy, _ = R.project(centre[None].astype(np.float32), view, H, W, 0.6, 0.6)
        jj, ii = np.meshgrid(np.arange(W) + 0.5, np.arange(H) + 0.5)
        rpx = np.hypot(jj - sx[0], ii - sy[0]) / (W / 1.2)            # distance from the centre in world units
        hit = covered(keys[n])
        assert hit[rpx < radius * 0.97].all(), n
        assert not hit[rpx > radius * 1.03].any(), n


def test_depth_order_and_ties():
    views = views_of(look_down_z())
    near = small_triangle(0.0, 0.0, z=0.2, r=0.5)                # depth 0.8
    far = small_triangle(0.0, 0.0, z=-0.3, r=0.5)                # depth 1.3
    v = np.concatenate([far, near, near])
    for faces, want in (([[0, 1, 2], [3, 4, 5]], 1), ([[3, 4, 5], [0, 1, 2]], 0),     # nearer wins in either order
                        ([[0, 1, 2], [6, 7, 8], [3, 4, 5]], 1), ([[0, 1, 2], [3, 4, 5], [6, 7, 8]], 1)):   # tie: lower id
        keys, _ = R.raster(v, faces, views, 8, 8, 1.0, 1.0)
        k = keys[0][covered(keys[0])]
        assert len(k) and (k & np.uint64(0xFFFFFFFF) == want).all(), faces
        assert (np.abs((k >> np.uint64(32)).astype(np.uint32).view(np.float32) - 0.8) < 1e-6).all()


def test_near_and_far_planes_cut_fragments():
    views = views_of(look_down_z(1.0))
    H = W = 32
    before = small_triangle(0.0, 0.0, z=0.96, r=0.5)             # depth 0.04 < znear
    beyond = small_triangle(0.0, 0.0, z=-99.5, r=0.5)            # depth 100.5 > zfar
    for tri in (before, beyond):
        keys, _ = R.raster(tri, [[0, 1, 2]], views, H, W, 1.0, 1.0)
        assert not covered(keys).any()
    # a triangle tilted through the near plane: depth goes from 0.5 at the bottom to -0.5 at the top of the image
    tilt = np.array([[-1, -1, 0.5], [1, -1, 0.5], [0, 1, 1.5]], np.float32)
    keys, _ = R.raster(tilt, [[0, 1, 2]], views, H, W, 1.0, 1.0)
    d = (keys[0] >> np.uint64(32)).astype(np.uint32).view(np.float32)
    hit = covered(keys[0])
    assert hit.any() and (d[hit] >= np.float32(R.ZNEAR)).all()
    rows = np.nonzero(hit.any(1))[0]
    assert rows.min() > 8 and rows.max() == H - 1                 # the top part of the triangle is cut away


def test_guard_band_and_nan_drops():
    views = views_of(look_down_z())
    v = np.concatenate([small_triangle(0, 0, r=0.5), [[1e7, 0, 0]], [[np.nan, 0, 0]]]).astype(np.float32)
    keys, drops = R.raster(v, [[0, 1, 2], [0, 1, 3], [0, 1, 4], [0, 1, 9]], views, 8, 8, 1.0, 1.0)
    assert drops == 1                                             # only the guard band counts; NaN and bad ids are silent
    assert (keys[0][covered(keys[0])] & np.uint64(0xFFFFFFFF) == 0).all()


def shade_one(tri, pose, xmag=1.0, colors=None, H=8, W=8):
    views = views_of(pose)
    frames, keys, _ = R.render(tri, [[0, 1, 2]], views, H, W, xmag, xmag, vertex_colors=colors)
    return frames[0], covered(keys[0])


def test_shading_facing_grazing_cone_and_background():
    pose = look_down_z(2.0)
    facing = small_triangle(0.0, 0.0, r=0.6)                      # normal +z, towards the eye
    img, hit = shade_one(facing, pose)
    assert (img[~hit] == 255).all()                               # white background
    centre = img[4, 4].astype(float)
    q = np.array([0, 0, 2.0]) - np.array([0.125, -0.125, 0])     # pixel (4, 4) shows world (0.125, -0.125, 0)
    want = np.floor(255 * 0.8 * 3.0 * q[2] / np.linalg.norm(q) / (np.pi * q @ q) + 0.5)   # I n.l / (pi r^2), grey 0.8
    assert np.abs(centre - want).max() <= 1 and (centre == centre[0]).all()
    back, _ = shade_one(facing[[0, 2, 1]], pose)                  # drawn, but lit from behind: black
    assert (back[4, 4] == 0).all()
    tilt = np.array([[-0.6, -0.6, -0.4], [0.6, -0.6, -0.4], [0.0, 0.6, 0.5]], np.float32)   # normal 37 degrees off the light
    oblique, _ = shade_one(tilt, pose)
    assert 0 < oblique[4, 4, 0] < centre[0]
    # a lit surface outside the pi/4 cone around the view axis is black: 1.3 to 2.3 to the side at distance 1 from the eye
    off = small_triangle(1.8, 0.0, z=1.0, r=0.5)
    img, hit = shade_one(off, pose, xmag=2.0, H=16, W=16)
    assert hit.any() and (img[hit] == 0).all()
    near_axis = small_triangle(0.3, 0.0, z=1.0, r=0.5)
    img, hit = shade_one(near_axis, pose, xmag=2.0, H=16, W=16)
    assert hit.any() and (img[hit] > 0).all()


def test_vertex_colours_are_interpolated():
    pose = look_down_z(2.0)
    tri = small_triangle(0.0, 0.0, r=0.9)
    img_red, hit = shade_one(tri, pose, colors=np.array([[255, 0, 0]] * 3, np.uint8))
    assert (img_red[hit][:, 1:] == 0).all() and (img_red[hit][:, 0] > 0).all()
    img, hit = shade_one(tri, pose, colors=np.array([[255, 0, 0], [0, 255, 0], [0, 0, 255]], np.uint8))
    px = img[hit].astype(int)
    assert (px.sum(1) > 0).all() and len(np.unique(px, axis=0)) > 3


@pytest.mark.parametrize('orbit', ['seg', 'car'])
def test_turntable_poses_equal_the_script_loop(orbit):
    """extract_mesh.py:244-254: one LookAtPoseSampler.sample per frame, columns 1 and 2 negated."""
    from pix2pix3d_b200 import mesh
    from pix2pix3d_b200.camera_utils import LookAtPoseSampler
    pivot = [0.0, 0.0, 0.2] if orbit == 'seg' else [0.0, 0.05, 0.0]
    if orbit == 'seg':
        yaw_c, yaw_range, pitch_range, radius = 3.14 / 2, 0.35, 0.25, 1
    else:
        yaw_c, yaw_range, pitch_range, radius = -3.14 / 2, np.pi, np.pi / 2, 1.2
    num_frames = 120
    want = []
    for frame_idx in range(num_frames):
        if orbit == 'seg':
            p = LookAtPoseSampler.sample(3.14/2 + yaw_range * np.sin(2 * 3.14 * frame_idx / num_frames),
                                         3.14/2 -0.05 + pitch_range * np.cos(2 * 3.14 * frame_idx / num_frames),
                                         torch.tensor(pivot, device='cpu'), radius=1, device='cpu')
        else:
            p = LookAtPoseSampler.sample(-3.14/2 + yaw_range * np.sin(2 * 3.14 * frame_idx / num_frames),
                                         3.14/2 -0.05 + pitch_range * np.cos(2 * 3.14 * frame_idx / num_frames),
                                         torch.tensor(pivot, device='cpu'), radius=1.2, device='cpu')
        p = p.reshape(4, 4).cpu().numpy().copy()
        p[:, 1] = -p[:, 1]
        p[:, 2] = -p[:, 2]
        want.append(p)
    got = mesh.turntable_poses(pivot, radius, yaw_c, yaw_range, pitch_range, num_frames, device='cpu')
    assert got.shape == (num_frames, 4, 4) and got.dtype == torch.float32
    assert np.array_equal(got.numpy().view(np.int32), np.stack(want).view(np.int32))


def test_write_gif_round_trip(tmp_path):
    import PIL.Image
    from pix2pix3d_b200 import mesh
    rng = np.random.RandomState(0)
    frames = np.zeros((5, 24, 40, 3), np.uint8)
    for n in range(5):
        frames[n, :, 8 * n:8 * n + 8] = rng.randint(0, 256, 3)
    p = str(tmp_path / 'turntable.gif')
    mesh.write_gif(p, torch.from_numpy(frames), fps=60)
    with PIL.Image.open(p) as im:
        assert im.n_frames == 5 and im.size == (40, 24)
        assert im.info.get('loop') == 0 and im.info.get('duration') == 20
    with pytest.raises(ValueError):
        mesh.write_gif(p, frames.astype(np.float32))
