"""Time the GPU geometry path of applications/extract_mesh.py at 512^3 on a seeded seg2cat_512 generator.

    python tools/time_mesh.py [--out profiles/r03_time_mesh.json] [--iters 10]

Reports CUDA-event times of sigma_grid (backbone once + 8 densities-only slab queries), of the reference-style loop
(512 calls of G.sample_mixed on 64^3 blocks, each copied into a host numpy grid, as get_sigma_field_np does; host clock
around work that ends in a device-to-host copy), of the marching-cubes calls (count = mc_count_kernel + mc_scan_kernel,
emit = mc_emit_verts_kernel + mc_emit_faces_kernel) and of extract_geometry end to end; per-kernel times from
torch.profiler in a separate pass; V and F; the bytes the kernels must move (three reads of the grid plus the vertex and
face outputs, from shapes); the GPU name and power limit. Random weights put sigma anywhere, so the threshold is the 0.9
quantile of the grid (every 16th value).
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def gpu_info():
    try:
        out = subprocess.check_output(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                                      text=True).splitlines()[0]
        name, power, clock = (s.strip() for s in out.split(','))
        return {'gpu': name, 'power_limit': power, 'max_sm_clock': clock}
    except (OSError, subprocess.CalledProcessError, ValueError):
        return {'gpu': torch.cuda.get_device_name(), 'power_limit': 'unknown', 'max_sm_clock': 'unknown'}


def event_ms(fn, iters):
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    ev[0].record()
    for _ in range(iters):
        fn()
    ev[1].record()
    torch.cuda.synchronize()
    return ev[0].elapsed_time(ev[1]) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='profiles/r03_time_mesh.json')
    ap.add_argument('--iters', type=int, default=10)
    ap.add_argument('--resolution', type=int, default=512)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'time_mesh.py measures on a CUDA device'
    from pix2pix3d_b200 import _lib, configs, mesh, native
    dev = torch.device('cuda')
    R, block = args.resolution, 64
    G = configs.build_generator('seg2cat_512', seed=0, device=dev, with_mapping=False)
    ws = configs.synthetic_ws(1, G.backbone.num_ws, 7).to(dev)
    res = {'workload': 'seg2cat_512 (seeded random weights), one latent', 'resolution': R, **gpu_info()}

    grid, bound = mesh.sigma_grid(G, ws, R)                                            # warm-up
    thr = float(torch.quantile(grid.flatten()[::16], 0.9))
    res['threshold'] = thr
    res['sigma_grid_ms'] = round(event_ms(lambda: mesh.sigma_grid(G, ws, R), 3), 3)

    # the reference's loop through this package (extract_mesh.py:60-81)
    X = torch.linspace(-bound, bound, R).split(block)
    sigma_np = np.zeros([R, R, R], dtype=np.float32)

    def reference_loop():
        with torch.no_grad():
            for xi, xs in enumerate(X):
                for yi, ys in enumerate(X):
                    for zi, zs in enumerate(X):
                        xx, yy, zz = torch.meshgrid(xs, ys, zs, indexing='ij')
                        pts = torch.stack([xx, yy, zz], dim=-1).unsqueeze(0).to(dev)
                        out = G.sample_mixed(pts.reshape(1, -1, 3), None, ws=ws, noise_mode='const')
                        sigma_np[xi * block:xi * block + len(xs), yi * block:yi * block + len(ys), zi * block:zi * block + len(zs)] = \
                            out['sigma'].reshape(len(xs), len(ys), len(zs)).cpu().numpy()
    with torch.no_grad():
        G.sample_mixed(torch.zeros(1, block ** 3, 3, device=dev), None, ws=ws, noise_mode='const')
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    reference_loop()
    res['reference_loop_ms'] = round((time.perf_counter() - t0) * 1e3, 1)
    res['reference_loop_equals_sigma_grid'] = bool(np.array_equal(sigma_np, grid.cpu().numpy()))
    del sigma_np

    # marching cubes: the two C entry points, timed with events
    ws_bytes = _lib.lib().p3d_marching_cubes_workspace_bytes(R, R, R)
    work = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
    counts = torch.empty(2, device=dev, dtype=torch.int64)
    c_thr = ctypes.c_double(thr)
    count = lambda: _lib.call('p3d_marching_cubes_count', grid, R, R, R, c_thr, work, ws_bytes, counts, device=dev)
    count()
    V, F = counts.tolist()
    verts = torch.empty(V, 3, device=dev, dtype=torch.float64)
    faces = torch.empty(F, 3, device=dev, dtype=torch.int64)
    emit = lambda: _lib.call('p3d_marching_cubes_emit', grid, R, R, R, c_thr, work, ws_bytes, verts, faces, device=dev)
    emit()
    res['vertices'], res['faces'] = V, F
    res['count_ms'] = round(event_ms(count, args.iters), 4)
    res['emit_ms'] = round(event_ms(emit, args.iters), 4)
    res['marching_cubes_call_ms'] = round(event_ms(lambda: native.marching_cubes(grid, thr), args.iters), 4)
    moved = 3 * grid.numel() * 4 + V * 3 * 8 + F * 3 * 8
    res['kernel_bytes'] = moved
    res['kernel_bytes_note'] = 'three reads of the fp32 grid + float64 [V,3] vertices + int64 [F,3] faces'
    res['kernels_GB_per_s'] = round(moved / ((res['count_ms'] + res['emit_ms']) * 1e-3) / 1e9, 1)

    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.iters):
            count()
            emit()
        torch.cuda.synchronize()
    per_kernel = {}
    for e in prof.key_averages():
        for k in ('mc_count_kernel', 'mc_scan_kernel', 'mc_emit_verts_kernel', 'mc_emit_faces_kernel'):
            if k in e.key:
                total = getattr(e, 'device_time_total', None) or e.cuda_time_total
                per_kernel[k] = round(total / e.count / 1e3, 4)
    res['kernel_ms_profiler'] = per_kernel

    res['extract_geometry_ms'] = round(event_ms(lambda: mesh.extract_geometry(G, ws, R, thr), 3), 3)
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as fh:
        json.dump(res, fh, indent=1)
        fh.write('\n')


if __name__ == '__main__':
    main()
