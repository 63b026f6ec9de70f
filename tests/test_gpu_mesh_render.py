"""Mesh preview on the GPU (p3d_mesh_raster / p3d_mesh_shade, pix2pix3d_b200.mesh.render_mesh): the kernels against the numpy
oracle bit for bit (depth keys and frames), the guard band, the kernel names, the vertex labels against the reference's
G.sample_mixed procedure, and the extract_mesh.py pipeline end to end."""
import numpy as np
import pytest
import torch

from p3d_oracle import mesh as M
from p3d_oracle import mesh_render as R
from test_gpu_mesh import nan_field
from test_mesh_cpu import sphere, torus

pytestmark = pytest.mark.gpu

KERNELS = ('mesh_raster_kernel', 'mesh_shade_kernel')


def orbit_views(n):
    from pix2pix3d_b200 import mesh, native
    return native.mesh_views(mesh.turntable_poses([0.0, 0.0, 0.0], 1.0, 3.14 / 2, 0.35, 0.25, num_frames=n, device='cpu')).numpy()


def pose_views(*eyes):
    """Views looking at the origin from each eye position (OpenGL convention)."""
    from pix2pix3d_b200 import native
    poses = []
    for eye in eyes:
        eye = np.asarray(eye, np.float64)
        back = eye / np.linalg.norm(eye)                             # camera +z points away from the target
        right = np.cross([0.0, 1.0, 0.0], back)
        right /= np.linalg.norm(right)
        c = np.eye(4)
        c[:3, 0], c[:3, 1], c[:3, 2], c[:3, 3] = right, np.cross(back, right), back, eye
        poses.append(c)
    return native.mesh_views(np.stack(poses)).numpy()


def sphere_mesh():
    v, f = M.marching_cubes(sphere((64, 64, 64), np.array([31.3, 30.8, 32.1]), 25.0), 0.0)
    return M.scale_vertices(v, 64, 0.5), f


def torus_mesh():
    v, f = M.marching_cubes(torus((40, 57, 33), np.array([19.3, 27.6, 16.2]), 12.0, 6.0), 0.0)
    return (v / 56 - 0.5).astype(np.float32), f


def soup(seed, n=400):
    """Random overlapping triangles of all sizes and both windings, with degenerate ones (repeated and collinear corners)."""
    rng = np.random.RandomState(seed)
    centres = rng.uniform(-0.5, 0.5, (n, 1, 3))
    v = (centres + rng.randn(n, 3, 3) * rng.choice([0.002, 0.02, 0.2], (n, 1, 1))).astype(np.float32)
    v[::17, 2] = v[::17, 0]                                           # two equal corners
    v[5::17, 2] = (v[5::17, 0] + v[5::17, 1]) / 2                     # collinear
    return v.reshape(-1, 3), np.arange(3 * n, dtype=np.int64).reshape(n, 3)


def big_triangles():
    """Triangles covering most of the viewport (the warp-cooperative path), one larger than it, in both windings."""
    v = np.array([[-0.55, -0.55, 0.1], [0.55, -0.5, 0.0], [0.0, 0.58, -0.1],
                  [-0.6, 0.6, 0.2], [0.6, 0.55, 0.15], [-0.3, -0.6, -0.2],
                  [-3.0, -3.0, 0.0], [3.0, -3.0, 0.05], [0.0, 3.0, -0.05]], np.float32)
    return v, np.array([[0, 1, 2], [3, 5, 4], [6, 7, 8]], np.int64)


def border_and_near():
    """Triangles leaving the viewport on every side and crossing the near plane of views from distance 1."""
    v = np.array([[-0.8, -0.2, 0.0], [0.1, -0.1, 0.0], [-0.2, 0.3, 0.0],
                  [0.2, 0.25, 0.3], [0.9, 0.7, -0.2], [0.4, -0.9, 0.1],
                  [-0.3, -0.3, 1.2], [0.3, -0.2, 0.6], [0.0, 0.4, 0.98],
                  [-0.5, 0.2, 0.9], [0.5, 0.1, 0.99], [0.1, -0.5, 1.1]], np.float32)
    return v, np.arange(12, dtype=np.int64).reshape(4, 3)


def nan_mesh():
    v, f = M.marching_cubes(nan_field(), 0.0)
    assert np.isnan(v).any()
    return (v / 19 - 0.5).astype(np.float32), f


def colours(n, seed):
    return np.random.RandomState(seed).randint(0, 256, (n, 3)).astype(np.uint8)


CASES = {
    # name: (mesh, views, H, W, xmag, ymag, coloured)
    'sphere64-1view-512': (sphere_mesh, lambda: orbit_views(1), 512, 512, 0.6, 0.6, False),
    'sphere64-120views-128-colour': (sphere_mesh, lambda: orbit_views(120), 128, 128, 0.6, 0.6, True),
    'torus-1view-512-colour': (torus_mesh, lambda: orbit_views(1), 512, 512, 0.6, 0.6, True),
    'torus-120views-128': (torus_mesh, lambda: orbit_views(120), 128, 128, 0.6, 0.6, False),
    'soup-4views-colour': (lambda: soup(0), lambda: pose_views([0, 0, 1], [1, 0.3, 0.2], [-0.2, -1, 0.4], [0.5, 0.5, -0.7]),
                           96, 96, 0.6, 0.6, True),
    'soup-nonsquare-48x80': (lambda: soup(1), lambda: pose_views([0, 0.2, 1], [-1, 0.1, 0.1]), 48, 80, 0.7, 0.4, False),
    'big-512-colour': (big_triangles, lambda: pose_views([0, 0, 1], [0.1, 0.05, 1], [0, 0, -1]), 512, 512, 0.6, 0.6, True),
    'border-near-plane': (border_and_near, lambda: pose_views([0, 0, 1], [0.05, 0, 1], [1, 0, 0.1]), 64, 64, 0.5, 0.5, False),
    'nan-vertices': (nan_mesh, lambda: orbit_views(3), 96, 96, 0.6, 0.6, True),
    'empty': (lambda: (np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int64)), lambda: orbit_views(2), 32, 48, 0.3, 0.3, False),
}


def run_kernels(v, f, views, H, W, xmag, ymag, col):
    from pix2pix3d_b200 import native
    vt, ft, vw = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (v, f, views))
    keys = native.mesh_raster(vt, ft, vw, H, W, xmag, ymag, R.ZNEAR, R.ZFAR)
    img = native.mesh_shade(keys, vt, ft, vw, xmag, ymag, None if col is None else torch.from_numpy(col).cuda(), 3.0)
    return keys.cpu().numpy().view(np.uint64), img.cpu().numpy()


@pytest.mark.parametrize('case', sorted(CASES))
def test_kernels_match_oracle(case):
    make_mesh, make_views, H, W, xmag, ymag, coloured = CASES[case]
    v, f = make_mesh()
    views = make_views()
    col = colours(len(v), 3) if coloured else None
    keys, img = run_kernels(v, f, views, H, W, xmag, ymag, col)
    want_img, want_keys, drops = R.render(v, f, views, H, W, xmag, ymag, vertex_colors=col)
    assert drops == 0
    assert keys.shape == (len(views), H, W) and img.shape == (len(views), H, W, 3) and img.dtype == np.uint8
    bad = np.argwhere(keys != want_keys)
    assert not len(bad), f'{len(bad)} depth keys differ, first at {bad[0]}: {keys[tuple(bad[0])]:#x} vs {want_keys[tuple(bad[0])]:#x}'
    bad = np.argwhere(img != want_img)
    assert not len(bad), f'{len(bad)} colour bytes differ, first at {bad[0]}: {img[tuple(bad[0])]} vs {want_img[tuple(bad[0])]}'
    drawn = keys != R.EMPTY
    if case == 'empty':
        assert not drawn.any() and (img == 255).all()
    else:
        assert drawn.any(axis=(1, 2)).all()                           # every view shows something
    if case.startswith('big'):
        assert drawn[0].mean() > 0.5                                  # the warp path drew most of the viewport


def test_guard_band_raises():
    from pix2pix3d_b200 import mesh
    v = torch.tensor([[0.0, 0.0, 0.0], [0.1, 0.0, 0.0], [0.0, 0.1, 0.0], [1e7, 0.0, 0.0]], device='cuda')
    f = torch.tensor([[0, 1, 2], [0, 1, 3]], device='cuda')
    poses = mesh.turntable_poses([0.0, 0.0, 0.0], 1.0, 3.14 / 2, 0.35, 0.25, num_frames=2)
    assert mesh.render_mesh(v[:3], f[:1], poses, 0.3, 0.3).shape == (2, 512, 512, 3)
    with pytest.raises(ValueError, match='2\\^21'):
        mesh.render_mesh(v, f, poses, 0.3, 0.3)


def test_kernel_names_and_determinism():
    from torch.profiler import ProfilerActivity, profile
    from pix2pix3d_b200 import mesh
    v, f = (torch.from_numpy(a).cuda() for a in sphere_mesh())
    poses = mesh.turntable_poses([0.0, 0.0, 0.0], 1.0, 3.14 / 2, 0.35, 0.25, num_frames=16)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        a = mesh.render_mesh(v, f, poses, 0.6, 0.6)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    for k in KERNELS:
        assert any(k in n for n in names), f'{k} did not run; launched: {sorted(set(names))}'
    assert torch.equal(a, mesh.render_mesh(v, f, poses, 0.6, 0.6))


@pytest.fixture(scope='module')
def generator():
    from pix2pix3d_b200 import configs
    dev = torch.device('cuda')
    G = configs.build_generator('seg2cat_512', seed=0, device=dev, with_mapping=False)
    ws = configs.synthetic_ws(1, G.backbone.num_ws, 7).to(dev)
    return G, ws


@pytest.fixture(scope='module')
def mesh128(generator):
    from pix2pix3d_b200 import mesh
    G, ws = generator
    grid, _ = mesh.sigma_grid(G, ws, 128)
    thr = float(torch.quantile(grid.flatten(), 0.9))                 # random weights put sigma anywhere
    return mesh.extract_geometry(G, ws, 128, thr), thr


PALETTE = torch.tensor([[255, 255, 255], [200, 30, 30], [40, 160, 40], [210, 200, 20], [50, 60, 250], [190, 20, 190]],
                       dtype=torch.uint8)


def test_vertex_semantic_labels_match_reference_procedure(generator, mesh128):
    """extract_mesh.py:196-216: G.sample_mixed on the vertices (torch.manual_seed(0) before each chunk), argmax of rgb
    channels 32:38."""
    from pix2pix3d_b200 import mesh
    G, ws = generator
    (v, _), _ = mesh128
    with torch.no_grad():
        torch.manual_seed(0)
        out = G.sample_mixed(v.unsqueeze(0), None, ws, truncation_psi=1, noise_mode='const')
    want = torch.argmax(out['rgb'][0, :, 32:32 + 6], dim=-1)
    got = mesh.vertex_semantic_labels(G, ws, v)
    assert got.dtype == torch.int64 and got.shape == (v.shape[0],) and got.device == v.device
    assert torch.equal(got, want)
    assert torch.equal(mesh.vertex_semantic_labels(G, ws, v, max_batch=v.shape[0] // 3 + 1), want)   # chunked
    assert len(torch.unique(want)) > 1


def test_extract_mesh_pipeline_end_to_end(generator, mesh128, tmp_path):
    """extract_geometry -> vertex_semantic_labels -> render_mesh(turntable_poses(...)) -> write_gif, as extract_mesh.py does
    it for seg2cat; at 128^3 every tenth frame equals the oracle, at 512^3 every frame shows the mesh."""
    import PIL.Image
    from pix2pix3d_b200 import mesh, native
    G, ws = generator
    pivot = G.rendering_kwargs['avg_camera_pivot']
    poses = mesh.turntable_poses(pivot, 1, 3.14 / 2, 0.35, 0.25)
    (v, f), thr = mesh128
    col = PALETTE.cuda()[mesh.vertex_semantic_labels(G, ws, v)]
    frames = mesh.render_mesh(v, f, poses, 0.3, 0.3, vertex_colors=col, resolution=128)
    assert frames.shape == (120, 128, 128, 3) and frames.dtype == torch.uint8 and frames.is_cuda
    views = native.mesh_views(poses).numpy()[::10]
    want, _, drops = R.render(v.cpu().numpy(), f.cpu().numpy(), views, 128, 128, 0.3, 0.3, vertex_colors=col.cpu().numpy())
    assert drops == 0 and np.array_equal(frames[::10].cpu().numpy(), want)

    v, f = mesh.extract_geometry(G, ws, 512, thr)
    col = PALETTE.cuda()[mesh.vertex_semantic_labels(G, ws, v)]
    frames = mesh.render_mesh(v, f, poses, 0.3, 0.3, vertex_colors=col)
    assert frames.shape == (120, 512, 512, 3)
    assert ((frames != 255).any(-1).flatten(1).sum(1) > 1000).all()
    path = str(tmp_path / 'rendered_mesh.gif')
    mesh.write_gif(path, frames, fps=60)
    with PIL.Image.open(path) as im:
        assert im.n_frames == 120 and im.size == (512, 512)
