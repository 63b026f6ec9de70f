"""Mesh extraction on the GPU (pix2pix3d_b200.mesh): the marching-cubes kernels against the numpy oracle, bit for bit;
the dense sigma grid against G.sample_mixed run through the reference's block loop; extract_geometry end to end."""
import numpy as np
import pytest
import torch

from p3d_oracle import mesh as M
from test_mesh_cpu import index_grid, sphere, torus

pytestmark = pytest.mark.gpu

KERNELS = ('mc_count_kernel', 'mc_scan_kernel', 'mc_emit_verts_kernel', 'mc_emit_faces_kernel')


def assert_same_mesh(got, want):
    gv, gf = (t.cpu().numpy() for t in got)
    wv, wf = want
    assert gv.dtype == np.float64 and gf.dtype == np.int64
    assert gv.shape == wv.shape and gf.shape == wf.shape, (gv.shape, wv.shape, gf.shape, wf.shape)
    nan = np.isnan(wv)
    assert np.array_equal(np.isnan(gv), nan)
    assert np.array_equal(gv[~nan].view(np.int64), wv[~nan].view(np.int64)), 'vertices differ in their bits'
    assert np.array_equal(gf, wf)


def smooth_field(n):
    g = index_grid((n, n, n)) / n * 2 * np.pi
    return (np.sin(3 * g[..., 0]) * np.cos(2 * g[..., 1]) + np.sin(4 * g[..., 2] + g[..., 0])).astype(np.float32)


def noise_field(n, seed):
    return np.random.RandomState(seed).randn(n, n, n).astype(np.float32)


def at_threshold_field():
    rng = np.random.RandomState(4)
    return (rng.randint(-1, 2, (11, 13, 9)).astype(np.float32) + 0.5)   # a third of the values equal the threshold 0.5


def nan_field():
    v = noise_field(20, 5)
    v[np.random.RandomState(6).rand(*v.shape) < 0.05] = np.nan
    return v


CASES = {
    'sphere64': lambda: (sphere((64, 64, 64), np.array([31.3, 30.8, 32.1]), 25.0), 0.0),
    'torus40x57x33': lambda: (torus((40, 57, 33), np.array([19.3, 27.6, 16.2]), 12.0, 6.0), 0.0),
    'noise48': lambda: (noise_field(48, 1), 0.0),
    'smooth256': lambda: (smooth_field(256), 0.1),
    'all_outside': lambda: (np.zeros((17, 5, 9), np.float32), 1.0),
    'all_inside': lambda: (np.ones((17, 5, 9), np.float32), 0.0),
    'at_threshold': lambda: (at_threshold_field(), 0.5),
    'nan_corners': lambda: (nan_field(), 0.0),
    'cube2': lambda: (np.array([[[1, -1], [-1, 1]], [[-1, 1], [1, -2]]], np.float32), 0.0),
}


@pytest.mark.parametrize('case', sorted(CASES))
def test_marching_cubes_matches_oracle(case):
    from pix2pix3d_b200 import mesh
    vol, thr = CASES[case]()
    want = M.marching_cubes(vol, thr)
    got = mesh.marching_cubes(torch.from_numpy(vol).cuda(), thr)
    assert_same_mesh(got, want)
    assert got[0].device.type == 'cuda' and got[1].device.type == 'cuda'
    if case in ('all_outside', 'all_inside'):
        assert got[0].shape == (0, 3) and got[1].shape == (0, 3)
    if case in ('sphere64', 'noise48'):
        assert_same_mesh(mesh.marching_cubes(vol, thr), want)                      # numpy input: copied to the device


def test_marching_cubes_kernel_names_and_determinism():
    from torch.profiler import ProfilerActivity, profile
    from pix2pix3d_b200 import mesh
    vol = torch.from_numpy(noise_field(48, 2)).cuda()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        v1, f1 = mesh.marching_cubes(vol, 0.0)
        torch.cuda.synchronize()
    names = [e.name for e in prof.events()]
    for k in KERNELS:
        assert any(k in n for n in names), f'{k} did not run; launched: {sorted(set(names))}'
    v2, f2 = mesh.marching_cubes(vol, 0.0)
    assert torch.equal(v1.view(torch.int64), v2.view(torch.int64)) and torch.equal(f1, f2)


def test_marching_cubes_rejects_bad_input():
    from pix2pix3d_b200 import mesh
    with pytest.raises(TypeError):
        mesh.marching_cubes(torch.zeros(4, 4, 4, dtype=torch.float64, device='cuda'), 0.0)
    with pytest.raises(TypeError):
        mesh.marching_cubes(np.zeros((4, 4, 4)), 0.0)
    with pytest.raises(ValueError):
        mesh.marching_cubes(torch.zeros(4, 1, 4, device='cuda'), 0.0)


@pytest.fixture(scope='module')
def generator():
    from pix2pix3d_b200 import configs
    dev = torch.device('cuda')
    G = configs.build_generator('seg2cat_512', seed=0, device=dev, with_mapping=False)
    ws = configs.synthetic_ws(1, G.backbone.num_ws, 7).to(dev)
    return G, ws


def test_sigma_grid_matches_reference_block_loop(generator):
    """get_sigma_field_np (extract_mesh.py:60-81) calls G.sample_mixed once per 64^3 block; the dense grid must hold the
    same values bit for bit (first, a middle and the last block)."""
    from pix2pix3d_b200 import mesh
    G, ws = generator
    R, block = 512, 64
    grid, bound = mesh.sigma_grid(G, ws, R, block)
    assert grid.shape == (R, R, R) and grid.dtype == torch.float32 and bound == G.rendering_kwargs['box_warp'] * 0.5
    X = torch.linspace(-bound, bound, R).split(block)
    with torch.no_grad():
        for xi, yi, zi in ((0, 0, 0), (3, 5, 2), (7, 7, 7)):
            xx, yy, zz = torch.meshgrid(X[xi], X[yi], X[zi], indexing='ij')
            pts = torch.stack([xx, yy, zz], dim=-1).unsqueeze(0).to(ws.device)
            sigma = G.sample_mixed(pts.reshape(1, -1, 3), None, ws=ws, noise_mode='const')['sigma'].reshape(block, block, block)
            got = grid[xi * block:(xi + 1) * block, yi * block:(yi + 1) * block, zi * block:(zi + 1) * block]
            assert torch.equal(got, sigma), (xi, yi, zi)


def test_extract_geometry(generator):
    from pix2pix3d_b200 import mesh
    G, ws = generator
    # random weights put sigma anywhere: take the threshold from the field itself
    grid, bound = mesh.sigma_grid(G, ws, 128)
    thr = float(torch.quantile(grid.flatten(), 0.9))
    v, f = mesh.extract_geometry(G, ws, 128, thr)
    ov, of = M.marching_cubes(grid.cpu().numpy(), thr)
    assert len(of) > 1000
    assert v.dtype == torch.float32 and f.dtype == torch.int64
    assert np.array_equal(v.cpu().numpy(), M.scale_vertices(ov, 128, bound)) and np.array_equal(f.cpu().numpy(), of)

    v, f = mesh.extract_geometry(G, ws, 512, thr)
    n = v.shape[0]
    assert n > 0 and f.shape[0] > 0
    assert torch.isfinite(v).all() and (v.abs() <= bound).all()
    assert f.min() >= 0 and f.max() < n
    # closed in the directed-edge sense, except where the surface leaves the grid: edges with both ends on an outer face
    on_boundary = (v.abs() == bound).any(1)
    d = torch.cat([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]])
    keep = ~(on_boundary[d[:, 0]] & on_boundary[d[:, 1]])
    d = d[keep]
    fwd, _ = torch.sort(d[:, 0] * n + d[:, 1])
    rev, _ = torch.sort(d[:, 1] * n + d[:, 0])
    assert torch.equal(fwd, rev)
