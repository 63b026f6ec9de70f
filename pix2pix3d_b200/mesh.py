"""Mesh extraction and preview on the GPU: the reference's applications/extract_mesh.py without leaving the device.

    grid, bound = sigma_grid(G, ws)                    # get_sigma_field_np (extract_mesh.py:60-81), dense [R,R,R] on the GPU
    vertices, faces = marching_cubes(grid, 50.)        # mcubes.marching_cubes (:86), CUDA kernels
    vertices, faces = extract_geometry(G, ws)          # both plus the scaling to [-bound, bound]^3 (:84-96)
    labels = vertex_semantic_labels(G, ws, vertices)   # the vertex query + argmax of :194-216, backbone once
    write_ply('mesh.ply', vertices, faces)             # stands in for trimesh's PLY export
    poses = turntable_poses(pivot, 1.0, 3.14 / 2, 0.35, 0.25)                  # the orbit of :244-254, OpenGL convention
    frames = render_mesh(vertices, faces, poses, 0.3, 0.3, vertex_colors=c)    # stands in for the pyrender loop (:226-258)
    write_gif('rendered_mesh.gif', frames, fps=60)                             # stands in for imageio.mimsave (:260)

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
from .camera_utils import LookAtPoseSampler
from .training import triplane

# near and far planes of the preview camera (pyrender's own defaults for an OrthographicCamera are unverified)
ZNEAR, ZFAR = 0.05, 100.0


def _queries_backbone_planes(G):
    """True when G.sample_mixed is backbone + renderer.run_model on one plane set (training/triplane.py::query_points)."""
    return getattr(type(G).sample_mixed, '__qualname__', '') in ('TriPlaneGenerator.sample_mixed', '_CondGeneratorBase.sample_mixed')


def _plane_query(G, ws, what):
    """(channels-last planes, packed decoder) of G.sample_mixed(..., ws, noise_mode='const'): the backbone runs once, as in
    that call. Refuses what the fused query cannot reproduce."""
    if not _queries_backbone_planes(G):
        raise NotImplementedError(f'{what} needs a generator whose sample_mixed queries one plane set; got {type(G).__name__}')
    if G.rendering_kwargs.get('density_noise', 0) > 0:
        raise NotImplementedError(f'{what} does not add density_noise')
    if ws.shape[0] != 1:
        raise ValueError(f'{what} takes the latent of one sample, got a batch of {ws.shape[0]}')
    dev = ws.device
    if dev.type != 'cuda':
        raise ValueError(f'{what} runs on a CUDA device')
    with torch.no_grad():
        planes = triplane.query_planes(G, ws, False, {'noise_mode': 'const'})
        renderer = G.renderer
        renderer.plane_axes = renderer.plane_axes.to(dev)
        if not renderer._axes_ok() or native.describe_decoder(G.decoder) is None:
            raise NotImplementedError('no fused query kernel for these plane axes / this decoder')
        return native.planes_to_channels_last(planes), native.pack_decoder(G.decoder)


def sigma_grid(G, ws, resolution=512, block_resolution=64):
    """Dense sigma grid of get_sigma_field_np (extract_mesh.py:60-81) -> (grid fp32 CUDA [R,R,R], bound).

    grid[i,j,k] is sigma at (X[i], X[j], X[k]), X = torch.linspace(-bound, bound, R) computed on the CPU as the reference
    does, bound = G.rendering_kwargs['box_warp'] * 0.5; the values equal those of G.sample_mixed(..., noise_mode='const')
    run through the reference's 64^3-block loop, bit for bit. The backbone runs once (through the same call as
    G.sample_mixed); the densities-only tensor-core query then fills x-slabs of `block_resolution` planes in place."""
    pcl, dec = _plane_query(G, ws, 'sigma_grid')
    dev = ws.device
    R, block = int(resolution), int(block_resolution)
    bound = G.rendering_kwargs['box_warp'] * 0.5
    with torch.no_grad():
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


def vertex_semantic_labels(G, ws, vertices, channels=(32, 38), max_batch=1 << 22):
    """Semantic class of each vertex (extract_mesh.py:196-216) -> int64 [V] on the vertices' device.

    The reference runs G.sample_mixed(vertices, None, ws, noise_mode='const') on chunks of vertices and takes
    torch.argmax(out['rgb'][0, :, 32:38], -1) (the first maximum); every chunk runs the backbone again. Here the backbone runs
    once (the planes of sigma_grid) and the colour query of G.sample_mixed (native.run_model, tensor cores) follows on chunks
    of `max_batch` vertices; the labels equal the reference's bit for bit. The palette is the caller's:
    torch.tensor(color_list)[labels] is the reference's own line 216."""
    pcl, dec = _plane_query(G, ws, 'vertex_semantic_labels')
    dev = ws.device
    pts = torch.as_tensor(vertices).to(device=dev, dtype=torch.float32).reshape(1, -1, 3)
    c0, c1 = channels
    labels = torch.empty(pts.shape[1], device=dev, dtype=torch.int64)
    with torch.no_grad():
        for head in range(0, pts.shape[1], max_batch):
            rgb, _ = native.run_model(pcl, dec, pts[:, head:head + max_batch], G.rendering_kwargs['box_warp'])
            labels[head:head + max_batch] = torch.argmax(rgb[0, :, c0:c1], dim=-1)
    return labels


def turntable_poses(pivot, radius, yaw_center, yaw_range, pitch_range, num_frames=120, device='cuda'):
    """The camera orbit of extract_mesh.py:244-254 as OpenGL-convention cam2world matrices [N,4,4] (columns 1 and 2
    negated, as the script does before handing them to pyrender).

    Frame i looks at `pivot` from `radius` at yaw = yaw_center + yaw_range * sin(2 * 3.14 * i / N) and pitch = 3.14/2 - 0.05
    + pitch_range * cos(2 * 3.14 * i / N), the angles in float64 on the host with the script's literal 3.14; each frame is one
    LookAtPoseSampler.sample call, as in the script, so the poses are the script's bit for bit. The script's orbits:
    seg / face: yaw_center = 3.14/2, yaw_range 0.35, pitch_range 0.25, radius 1; car: yaw_center = -3.14/2,
    yaw_range = pi, pitch_range = pi/2, radius 1.2; pivot = G.rendering_kwargs['avg_camera_pivot']."""
    pivot = pivot.to(device) if isinstance(pivot, torch.Tensor) else torch.tensor(pivot, device=device)
    poses = []
    for frame_idx in range(num_frames):
        pose = LookAtPoseSampler.sample(yaw_center + yaw_range * np.sin(2 * 3.14 * frame_idx / num_frames),
                                        3.14/2 - 0.05 + pitch_range * np.cos(2 * 3.14 * frame_idx / num_frames),
                                        pivot, radius=radius, device=device)
        poses.append(pose.reshape(4, 4))
    poses = torch.stack(poses)
    poses[:, :, 1] = -poses[:, :, 1]
    poses[:, :, 2] = -poses[:, :, 2]
    return poses


def render_mesh(vertices, faces, cam2world_gl, xmag, ymag, vertex_colors=None, resolution=512, light_intensity=3.0):
    """The preview frames of extract_mesh.py:226-258 -> uint8 CUDA [N,H,W,3], one per pose.

    An orthographic camera of half-extents xmag, ymag at each OpenGL-convention pose [N,4,4] (turntable_poses), a spot light
    of `light_intensity` and a pi/4 cone at the camera, diffuse shading of the vertex colours (uint8 [V,3] or [V,4], alpha
    ignored; grey when None) on a white background. `resolution`: an int or (H, W). The depth test, coverage and shading
    are this package's (include/p3d.h, above p3d_mesh_raster), not pyrender's: no specular or ambient term, no
    anti-aliasing. Raises ValueError when a triangle lies more than 2^21 pixels off screen."""
    H, W = (resolution, resolution) if isinstance(resolution, int) else (int(resolution[0]), int(resolution[1]))
    v = torch.as_tensor(vertices)
    dev = v.device if v.is_cuda else torch.device('cuda', torch.cuda.current_device())
    v = v.to(device=dev, dtype=torch.float32)
    f = torch.as_tensor(faces).to(device=dev, dtype=torch.int64)
    col = None
    if vertex_colors is not None:
        col = torch.as_tensor(vertex_colors).to(device=dev, dtype=torch.uint8)
        if col.dim() != 2 or col.shape[1] not in (3, 4):
            raise ValueError(f'vertex_colors must be [V,3] or [V,4], got {tuple(col.shape)}')
        col = col[:, :3]
    views = native.mesh_views(cam2world_gl).to(dev)
    keys = native.mesh_raster(v, f, views, H, W, xmag, ymag, ZNEAR, ZFAR)
    return native.mesh_shade(keys, v, f, views, xmag, ymag, col, light_intensity)


def write_gif(path, frames, fps=60):
    """Animated GIF of uint8 frames [N,H,W,3] (tensor or array), looping, through PIL (in place of imageio.mimsave).
    The frame time is 1/fps rounded to GIF's 10 ms unit; the palette quantisation is PIL's. PIL merges a frame identical to
    the one before it into that frame's duration."""
    import PIL.Image
    a = frames.detach().cpu().numpy() if isinstance(frames, torch.Tensor) else np.asarray(frames)
    if a.dtype != np.uint8 or a.ndim != 4 or a.shape[-1] != 3 or not len(a):
        raise ValueError(f'frames must be uint8 [N,H,W,3] with N >= 1, got {a.dtype} {a.shape}')
    images = [PIL.Image.fromarray(x) for x in a]
    images[0].save(path, save_all=True, append_images=images[1:], duration=10 * max(1, round(100 / fps)), loop=0)
