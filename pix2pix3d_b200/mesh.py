"""Mesh extraction on the GPU: the geometry path of the reference's applications/extract_mesh.py without leaving the device.

    grid, bound = sigma_grid(G, ws)                    # get_sigma_field_np (extract_mesh.py:60-81), dense [R,R,R] on the GPU
    vertices, faces = marching_cubes(grid, 50.)        # mcubes.marching_cubes (:86), CUDA kernels
    vertices, faces = extract_geometry(G, ws)          # both plus the scaling to [-bound, bound]^3 (:84-96)
    write_ply('mesh.ply', vertices, faces)             # stands in for trimesh's PLY export

The mesh (inside-ness, vertex and face order, orientation, the triangle table) is defined in
oracle/p3d_oracle/mesh.py and summarised in include/p3d.h: a value is inside when it is > threshold (NaN is outside);
one vertex per crossing grid edge, ordered by owning grid point in C order and by axis; faces by cube in C order, oriented
outward (normals toward lower sigma). The mesh is closed wherever the surface does not leave the grid: every directed
edge is matched by its reverse. Ambiguous cube faces are resolved by cutting off their inside corners, and the fan
diagonals there can make one vertex pair shared by four triangles. Whether PyMCubes picks the same triangles in
ambiguous cubes, its winding and the last float64 ulp of its interpolation are unverified; the vertex set is the one any
marching cubes with these inside-ness rules produces.
"""
import numpy as np
import torch

from . import native
from .training import triplane


def _queries_backbone_planes(G):
    """True when G.sample_mixed is backbone + renderer.run_model on one plane set (training/triplane.py::query_points)."""
    return getattr(type(G).sample_mixed, '__qualname__', '') in ('TriPlaneGenerator.sample_mixed', '_CondGeneratorBase.sample_mixed')


def sigma_grid(G, ws, resolution=512, block_resolution=64):
    """Dense sigma grid of get_sigma_field_np (extract_mesh.py:60-81) -> (grid fp32 CUDA [R,R,R], bound).

    grid[i,j,k] is sigma at (X[i], X[j], X[k]), X = torch.linspace(-bound, bound, R) computed on the CPU as the reference
    does, bound = G.rendering_kwargs['box_warp'] * 0.5; the values equal those of G.sample_mixed(..., noise_mode='const')
    run through the reference's 64^3-block loop, bit for bit. The backbone runs once (through the same call as
    G.sample_mixed); the densities-only tensor-core query then fills x-slabs of `block_resolution` planes in place."""
    if not _queries_backbone_planes(G):
        raise NotImplementedError(f'sigma_grid needs a generator whose sample_mixed queries one plane set; got {type(G).__name__}')
    if G.rendering_kwargs.get('density_noise', 0) > 0:
        raise NotImplementedError('sigma_grid does not add density_noise')
    if ws.shape[0] != 1:
        raise ValueError(f'sigma_grid takes the latent of one sample, got a batch of {ws.shape[0]}')
    dev = ws.device
    if dev.type != 'cuda':
        raise ValueError('sigma_grid runs on a CUDA device')
    R, block = int(resolution), int(block_resolution)
    bound = G.rendering_kwargs['box_warp'] * 0.5
    with torch.no_grad():
        planes = triplane.query_planes(G, ws, False, {'noise_mode': 'const'})
        renderer = G.renderer
        renderer.plane_axes = renderer.plane_axes.to(dev)
        if not renderer._axes_ok() or native.describe_decoder(G.decoder) is None:
            raise NotImplementedError('no fused query kernel for these plane axes / this decoder')
        dec = native.pack_decoder(G.decoder)
        pcl = native.planes_to_channels_last(planes)
        axis = torch.linspace(-bound, bound, R).to(dev)
        yz = torch.stack(torch.meshgrid(axis, axis, indexing='ij'), -1)                 # [R,R,2]
        grid = torch.empty(R, R, R, device=dev, dtype=torch.float32)
        for x0 in range(0, R, block):
            xs = axis[x0:x0 + block]
            n = xs.shape[0]
            pts = torch.cat([xs.view(n, 1, 1, 1).expand(n, R, R, 1), yz.expand(n, R, R, 2)], -1).view(1, -1, 3)
            native.run_model(pcl, dec, pts, G.rendering_kwargs['box_warp'], sigma_only=True, out_sigma=grid[x0:x0 + n])
    return grid, bound


def marching_cubes(volume, threshold):
    """mcubes.marching_cubes(volume, threshold) on the device -> (vertices float64 [V,3] in index coordinates,
    faces int64 [F,3]), both on the volume's device.

    `volume`: float32 CUDA tensor [nx,ny,nz], each side >= 2; a float32 numpy array is copied to the current device; any
    other dtype raises. `threshold` is compared in float64. Reads the vertex and face counts back once (one
    synchronisation) before it allocates the outputs, which an output of unknown size needs."""
    if isinstance(volume, np.ndarray):
        if volume.dtype != np.float32:
            raise TypeError(f'volume must be float32, got {volume.dtype}')
        volume = torch.from_numpy(np.ascontiguousarray(volume)).to(torch.device('cuda', torch.cuda.current_device()))
    elif not isinstance(volume, torch.Tensor):
        raise TypeError(f'volume must be a torch tensor or numpy array, got {type(volume).__name__}')
    return native.marching_cubes(volume, float(threshold))


def extract_geometry(G, ws, resolution=512, threshold=50.):
    """extract_geometry of extract_mesh.py:84-96 -> (vertices float32 [V,3] in [-bound, bound]^3, faces int64 [F,3]) on the
    GPU: sigma_grid, marching_cubes, then v / (R - 1) * (2 bound) - bound in float64 and one cast to float32."""
    grid, bound = sigma_grid(G, ws, resolution)
    vertices, faces = marching_cubes(grid, threshold)
    f64 = dict(device=vertices.device, dtype=torch.float64)
    b_min, b_max = torch.full((3,), -bound, **f64), torch.full((3,), bound, **f64)
    vertices = vertices / torch.full((3,), resolution - 1.0, **f64) * (b_max - b_min)[None, :] + b_min[None, :]
    return vertices.float(), faces


def write_ply(path, vertices, faces, vertex_colors=None):
    """Binary little-endian PLY: float x, y, z [, uchar red, green, blue, alpha] per vertex, `list uchar int vertex_indices`
    per face. vertex_colors: uint8 [V,3] (alpha 255) or [V,4]. Tensors or arrays; written from the host."""
    def host(a):
        return a.detach().cpu().numpy() if isinstance(a, torch.Tensor) else np.asarray(a)
    v = host(vertices).astype('<f4').reshape(-1, 3)
    f = host(faces).astype('<i4').reshape(-1, 3)
    fields = [('x', '<f4'), ('y', '<f4'), ('z', '<f4')]
    header = ['ply', 'format binary_little_endian 1.0', f'element vertex {len(v)}'] + [f'property float {c}' for c in 'xyz']
    if vertex_colors is not None:
        c = host(vertex_colors).astype(np.uint8).reshape(len(v), -1)
        if c.shape[1] == 3:
            c = np.concatenate([c, np.full((len(v), 1), 255, np.uint8)], 1)
        if c.shape[1] != 4:
            raise ValueError(f'vertex_colors must be [V,3] or [V,4], got {c.shape}')
        fields += [(n, 'u1') for n in ('red', 'green', 'blue', 'alpha')]
        header += [f'property uchar {n}' for n in ('red', 'green', 'blue', 'alpha')]
    header += [f'element face {len(f)}', 'property list uchar int vertex_indices', 'end_header']
    vrec = np.empty(len(v), fields)
    vrec['x'], vrec['y'], vrec['z'] = v[:, 0], v[:, 1], v[:, 2]
    if vertex_colors is not None:
        for i, n in enumerate(('red', 'green', 'blue', 'alpha')):
            vrec[n] = c[:, i]
    frec = np.empty(len(f), [('n', 'u1'), ('i', '<i4', (3,))])
    frec['n'], frec['i'] = 3, f
    with open(path, 'wb') as fh:
        fh.write(('\n'.join(header) + '\n').encode('ascii'))
        fh.write(vrec.tobytes())
        fh.write(frec.tobytes())
