"""Time the mesh preview of applications/extract_mesh.py at its sizes on a seeded seg2cat_512 generator: the 512^3 mesh,
120 turntable frames of 512x512 and the vertex labels.

    python tools/time_mesh_render.py [--out profiles/r04_time_mesh_render.json] [--iters 5]

Reports CUDA-event times (after one warm-up call of each) of the depth pass (mesh_raster: key clear + mesh_raster_kernel),
of the shading pass (mesh_shade_kernel), of render_mesh end to end (view setup, both passes, the guard-band read-back) and
of vertex_semantic_labels; faces, vertices, the pixels written (frames x H x W) and the drawn ones; ms per frame and
(face, view) pairs per second of the depth pass; the GPU name and power limit. Random weights put sigma anywhere, so the
threshold is the 0.9 quantile of the grid (every 16th value).
"""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from time_mesh import event_ms, gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='profiles/r04_time_mesh_render.json')
    ap.add_argument('--iters', type=int, default=5)
    ap.add_argument('--resolution', type=int, default=512, help='sigma grid side')
    ap.add_argument('--image', type=int, default=512, help='frame side')
    ap.add_argument('--frames', type=int, default=120)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'time_mesh_render.py measures on a CUDA device'
    from pix2pix3d_b200 import configs, mesh, native
    dev = torch.device('cuda')
    G = configs.build_generator('seg2cat_512', seed=0, device=dev, with_mapping=False)
    ws = configs.synthetic_ws(1, G.backbone.num_ws, 7).to(dev)
    res = {'workload': 'seg2cat_512 (seeded random weights), one latent', 'grid': args.resolution, 'image': args.image,
           'frames': args.frames, **gpu_info()}

    grid, _ = mesh.sigma_grid(G, ws, args.resolution)
    thr = float(torch.quantile(grid.flatten()[::16], 0.9))
    del grid
    v, f = mesh.extract_geometry(G, ws, args.resolution, thr)
    res.update(threshold=thr, vertices=v.shape[0], faces=f.shape[0])

    labels = mesh.vertex_semantic_labels(G, ws, v)                                    # warm-up
    res['vertex_semantic_labels_ms'] = round(event_ms(lambda: mesh.vertex_semantic_labels(G, ws, v), args.iters), 3)
    palette = torch.randint(0, 256, (6, 3), generator=torch.Generator().manual_seed(0), dtype=torch.uint8).to(dev)
    col = palette[labels]

    H = W = args.image
    xmag = 0.3
    poses = mesh.turntable_poses(G.rendering_kwargs['avg_camera_pivot'], 1, 3.14 / 2, 0.35, 0.25, args.frames)
    views = native.mesh_views(poses).to(dev)
    keys = native.mesh_raster(v, f, views, H, W, xmag, xmag, mesh.ZNEAR, mesh.ZFAR)
    frames = native.mesh_shade(keys, v, f, views, xmag, xmag, col)
    raster_ms = event_ms(lambda: native.mesh_raster(v, f, views, H, W, xmag, xmag, mesh.ZNEAR, mesh.ZFAR), args.iters)
    shade_ms = event_ms(lambda: native.mesh_shade(keys, v, f, views, xmag, xmag, col), args.iters)
    mesh.render_mesh(v, f, poses, xmag, xmag, vertex_colors=col, resolution=H)
    total_ms = event_ms(lambda: mesh.render_mesh(v, f, poses, xmag, xmag, vertex_colors=col, resolution=H), args.iters)
    n = args.frames
    res.update(pixels_written=n * H * W, pixels_drawn=int((frames != 255).any(-1).sum()),
               raster_ms=round(raster_ms, 3), shade_ms=round(shade_ms, 3), render_mesh_ms=round(total_ms, 3),
               render_mesh_ms_per_frame=round(total_ms / n, 4),
               raster_face_views_per_s=round(f.shape[0] * n / (raster_ms * 1e-3), 1))
    res['note'] = ('raster_ms includes the cudaMemsetAsync of the [N,H,W] uint64 key buffer and the guard-count read-back; '
                   'render_mesh_ms adds the host view setup and its copy')
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(res, fh, indent=1)
        fh.write('\n')


if __name__ == '__main__':
    main()
