"""Tensor-level wrappers over the C-ABI: allocate outputs with torch, pass raw device pointers.

These are the calls the reference-facing modules (training/..., torch_utils/ops/...) make; nothing here
has a CPU branch.
"""
import ctypes

import numpy as np
import torch

from . import _lib

PACKED_FLOATS = 2 * 4260
TC_PACKED_BYTES = 65536 + 324 * 4

# which fused renderer `render_fwd` uses: 'auto' (tensor-core decoder when the sample counts allow it), 'tc', 'simt',
# 'tc_pairs' (tensor-core decoder, ray-pair ownership: render_tc2.cu; sample counts <= 64)
render_impl = 'auto'

# when set to a list, timed_call records its launches here: ('render_fwd', start_event, end_event) from render_fwd and
# ('conv_gemm', start_event, end_event, flops, executed_flops) from the tcconv convolutions (bench.py)
kernel_events = None
# when set to a dict, every render_fwd call also writes the kernel's bookkeeping (importance indices, fine depths, sort
# permutation, interval weights) and leaves it there: lets tests score the bookkeeping of a whole G.synthesis call
render_debug_sink = None


def timed_call(event, name, *args, device, unsupported_ok=False):
    """_lib.call; with kernel_events set, a launch that ran is bracketed by CUDA events and recorded as
    (event[0], start, end, *event[1:])."""
    if kernel_events is None:
        return _lib.call(name, *args, device=device, unsupported_ok=unsupported_ok)
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    ran = _lib.call(name, *args, device=device, unsupported_ok=unsupported_ok)
    if ran:
        end.record()
        kernel_events.append((event[0], start, end, *event[1:]))
    return ran


def _f32c(t):
    assert t.is_cuda, 'native ops need CUDA tensors'
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def ray_sampler(cam2world, intrinsics, resolution):
    """RaySampler.forward -> (origins [B,M,3], dirs [B,M,3])."""
    c2w = _f32c(cam2world.reshape(-1, 16))
    K = _f32c(intrinsics.reshape(-1, 9))
    B = c2w.shape[0]
    M = resolution * resolution
    origins = torch.empty(B, M, 3, device=c2w.device, dtype=torch.float32)
    dirs = torch.empty_like(origins)
    _lib.call('p3d_ray_sampler', c2w, K, B, resolution, origins, dirs, device=c2w.device)
    return origins, dirs


def planes_to_channels_last(planes):
    """[B,3,C,H,W] (or [N,C,H,W]) fp32 -> [B,3,H,W,C]."""
    p = _f32c(planes)
    shp = p.shape
    C, H, W = shp[-3], shp[-2], shp[-1]
    N = p.numel() // (C * H * W)
    out = torch.empty(*shp[:-3], H, W, C, device=p.device, dtype=torch.float32)
    _lib.call('p3d_planes_to_channels_last', p, out, N, C, H, W, device=p.device)
    return out


class PackedDecoder:
    """Kernel-side weights of an OSG decoder plus its static description."""

    def __init__(self, packed, n_nets, sigma_net, masks, packed_tc=None):
        self.packed = packed
        self.packed_tc = packed_tc
        self.n_nets = n_nets
        self.sigma_net = sigma_net
        self.masks = masks
        self.out_channels = 32 * n_nets


def describe_decoder(decoder):
    """Map a decoder module onto (nets, sigma_net, sigmoid masks); None if the layout is not one of the
    OSG decoders the fused kernels implement (training/triplane.py:112, training/triplane_cond.py:859,926)."""
    name = type(decoder).__name__
    nets = []
    full = 0xFFFFFFFF
    if name == 'OSGDecoder':
        nets, sigma_net, masks = [decoder.net], 0, [full, 0]
    elif name == 'OSGDecoder_semantic':
        nets, sigma_net, masks = [decoder.net], 0, [full if decoder.final_sigmoid else 0, 0]
    elif name == 'OSGDecoder_semantic_lateSeparate':
        nets, sigma_net = [decoder.net, decoder.net_semantic], 1
        masks = [full, full if decoder.semantic_sigmoid else 0]
    elif name == 'OSGDecoder_semantic_entangle':
        if decoder.feature_sigmoid:
            m = full
        else:
            cs = int(decoder.semantic_channels)
            m = full & ~(((1 << cs) - 1) << 3)   # colour outputs 3..3+Cs-1 stay raw (triplane_cond.py:916-918)
        nets, sigma_net, masks = [decoder.net], 0, [m & full, 0]
    else:
        return None
    for net in nets:
        fc1, fc2 = net[0], net[2]
        if tuple(fc1.weight.shape) != (64, 32) or tuple(fc2.weight.shape) != (33, 64):
            return None
        if fc1.bias is None or fc2.bias is None:
            return None
    return nets, sigma_net, masks


def pack_decoder(decoder):
    desc = describe_decoder(decoder)
    if desc is None:
        raise NotImplementedError(f'no fused kernel for decoder type {type(decoder).__name__}')
    nets, sigma_net, masks = desc
    dev = nets[0][0].weight.device
    d = _lib.DecoderDesc()
    d.n_nets = len(nets)
    d.sigma_net = sigma_net
    keep = []
    for i, net in enumerate(nets):
        fc1, fc2 = net[0], net[2]
        w1, b1, w2, b2 = (_f32c(t.detach()) for t in (fc1.weight, fc1.bias, fc2.weight, fc2.bias))
        keep += [w1, b1, w2, b2]
        d.w1[i], d.b1[i], d.w2[i], d.b2[i] = w1.data_ptr(), b1.data_ptr(), w2.data_ptr(), b2.data_ptr()
        d.w1_gain[i], d.b1_gain[i] = float(fc1.weight_gain), float(fc1.bias_gain)
        d.w2_gain[i], d.b2_gain[i] = float(fc2.weight_gain), float(fc2.bias_gain)
        d.sigmoid_mask[i] = masks[i]
    packed = torch.empty(PACKED_FLOATS, device=dev, dtype=torch.float32)
    _lib.call('p3d_pack_decoder', ctypes.byref(d), packed, device=dev)
    packed_tc = torch.empty(TC_PACKED_BYTES, device=dev, dtype=torch.uint8)
    _lib.call('p3d_pack_decoder_tc', ctypes.byref(d), packed_tc, device=dev)
    del keep
    return PackedDecoder(packed, len(nets), sigma_net, masks, packed_tc)


def ray_limits_box(rays_o, rays_d, box_side_length):
    """math_utils.get_ray_limits_box on CUDA tensors: (t_near, t_far) of shape [..., 1]."""
    lead = rays_o.shape[:-1]
    o, d = _f32c(rays_o.detach().reshape(-1, 3)), _f32c(rays_d.detach().reshape(-1, 3))
    n = o.shape[0]
    tn = torch.empty(n, device=o.device, dtype=torch.float32)
    tf = torch.empty(n, device=o.device, dtype=torch.float32)
    _lib.call('p3d_ray_limits_box', o, d, n, float(box_side_length), tn, tf, device=o.device)
    return tn.reshape(*lead, 1), tf.reshape(*lead, 1)


def render_fwd(planes_nhwc, dec, ray_origins, ray_dirs, depths_coarse, u, box_warp, white_back=False, debug=False, impl=None,
               stratified=None, plane_index=None):
    """Fused ImportanceRenderer.forward. Returns (feat [B,R,C], depth [B,R,1], wsum [B,R,1][, debug dict]).
    `stratified` (instead of `depths_coarse`): the ingredients of sample_stratified, combined inside the kernel --
    dict(jitter=[B,R,Sc] U[0,1) draw, table=[Sc], delta=float) for scalar ray limits or dict(jitter, table, ray_start=[B,R],
    ray_end=[B,R]) for per-ray limits (p3d_render_args_t::depth_mode 1 / 2).
    `plane_index` ([B] int32): plane set of each image; lets B views share fewer plane sets (planes batch < B)."""
    Bp, _, H, W, C = planes_nhwc.shape
    B = ray_origins.shape[0]
    if plane_index is None and Bp != B:
        raise ValueError('planes batch and ray batch differ: pass plane_index')
    assert C == 32 and planes_nhwc.dtype == torch.float32
    impl = impl or render_impl
    # a strided view is read in place by the tensor-core kernel as long as channels are contiguous and rows are W pixels
    # apart (e.g. the backbone's NHWC [B,H,W,96] output viewed as [B,3,H,W,32]); everything else is made dense first
    st_img, st_plane, st_row, st_pix, st_ch = planes_nhwc.stride()
    strided = not planes_nhwc.is_contiguous()
    if strided and not (st_ch == 1 and st_row == W * st_pix and st_pix >= 32 and st_plane > 0 and st_img > 0 and impl != 'simt'):
        planes_nhwc = planes_nhwc.contiguous()
        strided = False
    R = ray_origins.shape[1]
    o, d = _f32c(ray_origins), _f32c(ray_dirs)
    keep = []
    if stratified is not None:
        jit = _f32c(stratified['jitter']).reshape(B, R, -1)
        Sc = jit.shape[-1]
        table = _f32c(stratified['table']).reshape(-1)
        assert table.numel() == Sc
        dc = None
    else:
        dc = _f32c(depths_coarse).reshape(B, R, -1)
        Sc = dc.shape[-1]
    Sf = 0 if u is None else int(u.shape[-1])
    uu = None if u is None else _f32c(u)
    dev = planes_nhwc.device
    feat = torch.empty(B, R, dec.out_channels, device=dev, dtype=torch.float32)
    depth = torch.empty(B, R, 1, device=dev, dtype=torch.float32)
    wsum = torch.empty(B, R, 1, device=dev, dtype=torch.float32)
    ws = torch.empty(4, device=dev, dtype=torch.int32)
    a = _lib.RenderArgs()
    a.planes_nhwc, a.ray_origins, a.ray_dirs = planes_nhwc.data_ptr(), o.data_ptr(), d.data_ptr()
    if dc is not None:
        a.depths_coarse = dc.data_ptr()
    else:
        a.jitter, a.depth_table = jit.data_ptr(), table.data_ptr()
        if 'ray_start' in stratified:
            rs, re_ = _f32c(stratified['ray_start']).reshape(B, R), _f32c(stratified['ray_end']).reshape(B, R)
            keep += [rs, re_]
            a.depth_mode, a.ray_start, a.ray_end = 2, rs.data_ptr(), re_.data_ptr()
            a.depth_delta = float(np.float32(1.0) / np.float32(Sc - 1))      # what `tensor / (Sc - 1)` multiplies by on CUDA
        else:
            a.depth_mode, a.depth_delta = 1, float(stratified['delta'])
    if plane_index is not None:
        pidx = plane_index.to(device=planes_nhwc.device, dtype=torch.int32).contiguous()
        assert pidx.numel() == B
        keep.append(pidx)
        a.plane_index = pidx.data_ptr()
    a.u_importance = None if uu is None else uu.data_ptr()
    a.decoder_packed = dec.packed.data_ptr()
    a.n_nets, a.sigma_net = dec.n_nets, dec.sigma_net
    a.sigmoid_mask[0], a.sigmoid_mask[1] = dec.masks[0], dec.masks[1]
    a.B, a.R, a.H, a.W, a.Sc, a.Sf = B, R, H, W, Sc, Sf         # B = images of rays; plane sets may be fewer (plane_index)
    a.coord_scale = 2.0 / float(box_warp)
    a.white_back = 1 if white_back else 0
    a.out_feat, a.out_depth, a.out_wsum = feat.data_ptr(), depth.data_ptr(), wsum.data_ptr()
    dbg = {}
    want_debug = debug or render_debug_sink is not None
    if want_debug:
        S = Sc + Sf
        dbg['weights_final'] = torch.empty(B, R, S - 1, device=dev, dtype=torch.float32)
        dbg['perm'] = torch.empty(B, R, S, device=dev, dtype=torch.int32)
        a.dbg_weights_final, a.dbg_perm = dbg['weights_final'].data_ptr(), dbg['perm'].data_ptr()
        if Sf > 0:
            dbg['weights_coarse'] = torch.empty(B, R, Sc - 1, device=dev, dtype=torch.float32)
            dbg['depths_fine'] = torch.empty(B, R, Sf, device=dev, dtype=torch.float32)
            dbg['inds'] = torch.empty(B, R, Sf, device=dev, dtype=torch.int32)
            a.dbg_weights_coarse = dbg['weights_coarse'].data_ptr()
            a.dbg_depths_fine, a.dbg_inds = dbg['depths_fine'].data_ptr(), dbg['inds'].data_ptr()
    a.workspace = ws.data_ptr()
    if strided:
        a.plane_strides[0], a.plane_strides[1], a.plane_strides[2] = st_img, st_plane, st_pix
    use_tc = impl in ('auto', 'tc', 'tc_pairs') and Sc % 8 == 0 and Sf % 8 == 0 and Sc <= 128 and Sf <= 128 and dec.packed_tc is not None
    if impl in ('tc', 'tc_pairs') and not use_tc:
        raise ValueError('tensor-core renderer needs sample counts that are multiples of 8')
    # ray-pair ownership fills its rows only at 64 samples per pass; there it is 6-8 % faster (1.58 vs 1.72 ms at the config-4
    # sampling), at 48 it is 21 % slower (profiles/r01_render_fwd_tc_ncu.md)
    a.tc_variant = 1 if (impl == 'tc_pairs' or (impl == 'auto' and Sc == 64 and Sf == 64)) else 0
    if use_tc:
        a.decoder_packed = dec.packed_tc.data_ptr()
    elif strided:   # the SIMT kernel reads dense planes only
        dense = planes_nhwc.contiguous()
        a.planes_nhwc = dense.data_ptr()
        a.plane_strides[0] = a.plane_strides[1] = a.plane_strides[2] = 0
    timed_call(('render_fwd',), 'p3d_render_fwd_tc' if use_tc else 'p3d_render_fwd', ctypes.byref(a), device=dev)
    if render_debug_sink is not None:
        render_debug_sink.update(dbg, feat=feat, depth=depth, wsum=wsum)
    if debug:
        return feat, depth, wsum, dbg
    return feat, depth, wsum


def run_model(planes_nhwc, dec, coords, box_warp, impl=None, sigma_only=False, out_sigma=None):
    """Fused sample_from_planes + decoder: coords [B,M,3] -> (rgb [B,M,C], sigma [B,M,1]).

    `impl`: 'auto' / 'tc' run the tensor-core query (p3d_run_model_tc), 'simt' the CUDA-core kernel.
    `sigma_only` (tensor-core query): skip the colours and return (None, sigma) -- the mesh-extraction query.
    `out_sigma`: optional contiguous fp32 tensor of B*M elements on the planes' device that receives the densities in
    place of a new [B,M,1] tensor (any shape, e.g. a slab of a dense grid); it is returned as `sigma`."""
    B, _, H, W, C = planes_nhwc.shape
    assert C == 32 and planes_nhwc.dtype == torch.float32
    impl = impl or render_impl
    use_tc = impl in ('auto', 'tc', 'tc_pairs') and dec.packed_tc is not None
    strides = None
    if not planes_nhwc.is_contiguous():
        st_img, st_plane, st_row, st_pix, st_ch = planes_nhwc.stride()
        if use_tc and st_ch == 1 and st_row == W * st_pix and st_pix >= 32 and st_plane > 0 and st_img > 0:
            strides = (ctypes.c_int64 * 3)(st_img, st_plane, st_pix)       # read in place (see render_fwd)
        else:
            planes_nhwc = planes_nhwc.contiguous()
    c = _f32c(coords)
    M = c.shape[1]
    dev = planes_nhwc.device
    sigma_only = bool(sigma_only) and use_tc
    rgb = None if sigma_only else torch.empty(B, M, dec.out_channels, device=dev, dtype=torch.float32)
    if out_sigma is None:
        sigma = torch.empty(B, M, 1, device=dev, dtype=torch.float32)
    else:
        if not (out_sigma.device == dev and out_sigma.dtype == torch.float32 and out_sigma.is_contiguous()
                and out_sigma.numel() == B * M):
            raise ValueError(f'out_sigma must be a contiguous float32 tensor of {B * M} elements on {dev}')
        sigma = out_sigma
    masks = (ctypes.c_uint32 * 2)(dec.masks[0], dec.masks[1])
    if use_tc:
        _lib.call('p3d_run_model_tc', planes_nhwc, strides, c, dec.packed_tc, dec.n_nets, dec.sigma_net, masks, B, M, H, W,
                  2.0 / float(box_warp), rgb, sigma, device=dev)
    else:
        _lib.call('p3d_run_model', planes_nhwc, c, dec.packed, dec.n_nets, dec.sigma_net, masks, B, M, H, W, 2.0 / float(box_warp),
                  rgb, sigma, device=dev)
    return rgb, sigma


def marching_cubes(volume, threshold):
    """Marching cubes (p3d_marching_cubes_*, the mesh of include/p3d.h) on a float32 CUDA grid [nx,ny,nz], each side >= 2:
    -> (vertices float64 [V,3] in index coordinates, faces int64 [F,3]) on the volume's device.

    The output size is known only after the count, so this reads the two counts back once (one synchronisation of the
    current stream) before it allocates the outputs; it cannot be captured in a CUDA graph. Refuses V >= 2^31."""
    if volume.dim() != 3 or min(volume.shape) < 2:
        raise ValueError(f'volume must be [nx,ny,nz] with every side >= 2, got {tuple(volume.shape)}')
    if volume.dtype != torch.float32 or not volume.is_cuda:
        raise TypeError(f'volume must be a float32 CUDA tensor, got {volume.dtype} on {volume.device}')
    v = volume.contiguous()
    nx, ny, nz = v.shape
    dev = v.device
    ws_bytes = _lib.lib().p3d_marching_cubes_workspace_bytes(nx, ny, nz)
    if ws_bytes < 0:
        raise ValueError(f'grid {tuple(v.shape)} is too large for p3d_marching_cubes')
    ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
    counts = torch.empty(2, device=dev, dtype=torch.int64)
    thr = ctypes.c_double(float(threshold))
    _lib.call('p3d_marching_cubes_count', v, nx, ny, nz, thr, ws, ws_bytes, counts, device=dev)
    n_verts, n_faces = counts.tolist()
    if n_verts >= 1 << 31:
        raise ValueError(f'{n_verts} vertices: p3d_marching_cubes supports fewer than 2^31')
    vertices = torch.empty(n_verts, 3, device=dev, dtype=torch.float64)
    faces = torch.empty(n_faces, 3, device=dev, dtype=torch.int64)
    if n_verts:
        _lib.call('p3d_marching_cubes_emit', v, nx, ny, nz, thr, ws, ws_bytes, vertices, faces, device=dev)
    return vertices, faces


def mesh_views(cam2world_gl):
    """p3d_mesh_view_t array of OpenGL-convention poses [N,4,4] (camera looks down -z, +y up): float32 CPU tensor
    [N,18] = world2cam rows 0-2, eye, spot axis (camera -z). The rigid inverse (R^T, -R^T t) is formed in float64 and cast
    to float32 once."""
    c = cam2world_gl.detach().cpu().double().numpy() if isinstance(cam2world_gl, torch.Tensor) else np.asarray(cam2world_gl, np.float64)
    c = c.reshape(-1, 4, 4)
    R, t = c[:, :3, :3], c[:, :3, 3]
    Rt = R.transpose(0, 2, 1)
    w2c = np.concatenate([Rt, -np.einsum('nij,nj->ni', Rt, t)[:, :, None]], 2)
    views = np.concatenate([w2c.reshape(-1, 12), t, -R[:, :, 2]], 1).astype(np.float32)
    return torch.from_numpy(np.ascontiguousarray(views))


def _mesh_inputs(vertices, faces, views):
    if not (vertices.is_cuda and vertices.dtype == torch.float32 and vertices.dim() == 2 and vertices.shape[1] == 3):
        raise TypeError(f'vertices must be a float32 CUDA tensor [V,3], got {vertices.dtype} {tuple(vertices.shape)} on {vertices.device}')
    if not (faces.dtype == torch.int64 and faces.dim() == 2 and faces.shape[1] == 3 and faces.device == vertices.device):
        raise TypeError(f'faces must be an int64 tensor [F,3] on {vertices.device}, got {faces.dtype} {tuple(faces.shape)} on {faces.device}')
    if not (views.dtype == torch.float32 and views.dim() == 2 and views.shape[1] == _lib.MESH_VIEW_FLOATS
            and views.device == vertices.device):
        raise TypeError(f'views must be float32 [N,{_lib.MESH_VIEW_FLOATS}] on {vertices.device} (mesh_views)')
    return vertices.contiguous(), faces.contiguous(), views.contiguous()


def mesh_raster(vertices, faces, views, height, width, xmag, ymag, znear, zfar):
    """Depth pass of the mesh preview (p3d_mesh_raster; contract in include/p3d.h): vertices float32 CUDA [V,3], faces int64
    [F,3], views float32 [N,18] (mesh_views) -> depth keys [N,H,W] (int64 tensor holding the uint64 keys; -1 = empty).
    Reads the guard-band drop count back (one synchronisation) and raises ValueError when a triangle left the guard band."""
    v, f, views = _mesh_inputs(vertices, faces, views)
    N, dev = views.shape[0], v.device
    keys = torch.empty(N, height, width, device=dev, dtype=torch.int64)
    drops = torch.empty(1, device=dev, dtype=torch.int64)
    _lib.call('p3d_mesh_raster', v, v.shape[0], f, f.shape[0], views, N, height, width, float(xmag), float(ymag), float(znear),
              float(zfar), keys, drops, device=dev)
    n_drop = int(drops.item())
    if n_drop:
        raise ValueError(f'{n_drop} (triangle, view) pairs have a vertex more than 2^21 pixels off screen; '
                         'move the camera or scale the mesh')
    return keys


def mesh_shade(keys, vertices, faces, views, xmag, ymag, vertex_colors=None, light_intensity=3.0):
    """Shading pass of the mesh preview (p3d_mesh_shade) over the keys of mesh_raster -> uint8 [N,H,W,3].
    vertex_colors: uint8 [V,3] on the vertices' device, or None (grey)."""
    v, f, views = _mesh_inputs(vertices, faces, views)
    N, H, W = keys.shape
    if keys.dtype != torch.int64 or keys.device != v.device or N != views.shape[0]:
        raise TypeError('keys must be the int64 [N,H,W] output of mesh_raster for these views')
    keys = keys.contiguous()
    col = None
    if vertex_colors is not None:
        if not (vertex_colors.dtype == torch.uint8 and tuple(vertex_colors.shape) == (v.shape[0], 3) and vertex_colors.device == v.device):
            raise TypeError(f'vertex_colors must be uint8 [{v.shape[0]},3] on {v.device}')
        col = vertex_colors.contiguous()
    out = torch.empty(N, H, W, 3, device=v.device, dtype=torch.uint8)
    _lib.call('p3d_mesh_shade', keys, v, v.shape[0], f, f.shape[0], views, N, H, W, float(xmag), float(ymag), col,
              float(light_intensity), out, device=v.device)
    return out


def sample_from_planes(planes_nhwc, coords, box_warp):
    """coords [B,M,3] -> features [B,3,M,32] (reference layout of sample_from_planes)."""
    B, _, H, W, _ = planes_nhwc.shape
    c = _f32c(coords)
    M = c.shape[1]
    out = torch.empty(B, 3, M, 32, device=planes_nhwc.device, dtype=torch.float32)
    _lib.call('p3d_sample_from_planes', planes_nhwc, c, B, M, H, W, 2.0 / float(box_warp), out, device=planes_nhwc.device)
    return out


def ray_march(colors, densities, depths, white_back=False):
    """MipRayMarcher2.run_forward on [B,R,S,C] / [B,R,S,1] / [B,R,S,1] tensors."""
    B, R, S, Cc = colors.shape
    col, den, dep = _f32c(colors), _f32c(densities), _f32c(depths)
    dev = col.device
    rgb = torch.empty(B, R, Cc, device=dev, dtype=torch.float32)
    depth = torch.empty(B, R, 1, device=dev, dtype=torch.float32)
    weights = torch.empty(B, R, S - 1, 1, device=dev, dtype=torch.float32)
    ws = torch.empty(4, device=dev, dtype=torch.int32)
    _lib.call('p3d_ray_march', col, den, dep, B * R, S, Cc, 1 if white_back else 0, rgb, depth, weights, ws, device=dev)
    return rgb, depth, weights


def sample_from_planes_bwd(grad_features, coords, box_warp, H, W):
    """grad_features [B,3,M,32] -> gradient w.r.t. channels-last planes [B,3,H,W,32]."""
    g = _f32c(grad_features)
    c = _f32c(coords)
    B, _, M, _ = g.shape
    out = torch.empty(B, 3, H, W, 32, device=g.device, dtype=torch.float32)
    _lib.call('p3d_sample_from_planes_bwd', g, c, B, M, H, W, 2.0 / float(box_warp), out, device=g.device)
    return out


def ray_march_bwd(colors, densities, depths, g_rgb, g_depth, g_weights, depth_range, white_back=False):
    """Gradients of MipRayMarcher2.run_forward w.r.t. colors [B,R,S,C] and densities [B,R,S,1]."""
    B, R, S, Cc = colors.shape
    col, den, dep = _f32c(colors), _f32c(densities), _f32c(depths)
    grgb = _f32c(g_rgb)
    gdep = None if g_depth is None else _f32c(g_depth)
    gw = None if g_weights is None else _f32c(g_weights)
    rng = None if depth_range is None else _f32c(depth_range)
    g_col = torch.empty_like(col)
    g_den = torch.empty_like(den)
    _lib.call('p3d_ray_march_bwd', col, den, dep, grgb, gdep, gw, rng, B * R, S, Cc, 1 if white_back else 0, g_col, g_den,
              device=col.device)
    return g_col, g_den


def sample_importance(z_vals, weights, u, return_inds=False):
    """z_vals [N,S], weights [N,S-1], u [N,Sf] -> samples [N,Sf] (and searchsorted indices)."""
    z, w, uu = _f32c(z_vals), _f32c(weights), _f32c(u)
    N, S = z.shape
    Sf = uu.shape[1]
    out = torch.empty(N, Sf, device=z.device, dtype=torch.float32)
    inds = torch.empty(N, Sf, device=z.device, dtype=torch.int32) if return_inds else None
    _lib.call('p3d_sample_importance', z, w, uu, N, S, Sf, out, inds, device=z.device)
    return (out, inds) if return_inds else out


# ----------------------------------------------------------------------------------------------
# OSG decoder MLP of the gradient-requiring passes (p3d_decoder_mlp_fwd / _bwd)
# ----------------------------------------------------------------------------------------------
DECODER_PARAM_FLOATS = 64 * 32 + 64 + 33 * 64 + 33


class _DecoderMLP(torch.autograd.Function):
    """feats [N,3,M,32] -> (rgb [N,M,32], sigma [N,M,1]) through mean(1) -> FC(32,64) -> softplus -> FC(64,33) [-> sigmoid], forward
    and first-order backward on libp3d. w1 / b1 / w2 / b2 are the EFFECTIVE parameters (runtime gains applied by the caller under
    autograd), so their gradients flow on to the module's parameters through ordinary torch ops."""

    @staticmethod
    def forward(ctx, feats, w1, b1, w2, b2, mask):
        f, w1c, b1c, w2c, b2c = (_f32c(t.detach()) for t in (feats, w1, b1, w2, b2))
        n, _, m, _ = f.shape
        rgb = torch.empty(n, m, 32, device=f.device, dtype=torch.float32)
        sigma = torch.empty(n, m, 1, device=f.device, dtype=torch.float32)
        # hidden pre-activations for the backward pass (256 bytes per point), only when a gradient can be asked for
        pre = torch.empty(n * m, 64, device=f.device, dtype=torch.float32) if any(ctx.needs_input_grad) else None
        _lib.call('p3d_decoder_mlp_fwd', f, n, m, w1c, b1c, w2c, b2c, int(mask), rgb, sigma, pre, device=f.device)
        if pre is not None:
            ctx.save_for_backward(f, w1c, b1c, w2c, b2c, pre, rgb)
        ctx.mask = int(mask)
        return rgb, sigma

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, g_rgb, g_sigma):
        f, w1, b1, w2, b2, pre, rgb = ctx.saved_tensors
        n, _, m, _ = f.shape
        gr = None if g_rgb is None else _f32c(g_rgb)
        gs = None if g_sigma is None else _f32c(g_sigma)
        g_feats = torch.empty_like(f)
        g_params = torch.empty(DECODER_PARAM_FLOATS, device=f.device, dtype=torch.float32)
        nws = _lib.lib().p3d_decoder_mlp_bwd_workspace_floats()
        ws = torch.empty(nws, device=f.device, dtype=torch.float32)
        _lib.call('p3d_decoder_mlp_bwd', f, pre, rgb, n, m, w1, b1, w2, b2, ctx.mask, gr, gs, g_feats, g_params, ws, nws,
                  device=f.device)
        gw1, gb1, gw2, gb2 = torch.split(g_params, [64 * 32, 64, 33 * 64, 33])
        return g_feats, gw1.view(64, 32), gb1, gw2.view(33, 64), gb2, None


def _effective_fc(fc):
    """weight * weight_gain, bias * bias_gain as FullyConnectedLayer.forward forms them (networks_stylegan2.py:111-119)."""
    w = fc.weight.to(torch.float32) * fc.weight_gain
    b = fc.bias.to(torch.float32)
    if fc.bias_gain != 1:
        b = b * fc.bias_gain
    return w, b


def decoder_mlp_supported(decoder, sampled_features):
    """True when `decoder(sampled_features, ...)` can run on p3d_decoder_mlp_*: a CUDA fp32 [N,3,M,32] feature tensor and one of the
    OSG decoder layouts the kernels implement."""
    f = sampled_features
    return (f.is_cuda and f.dtype == torch.float32 and f.ndim == 4 and f.shape[1] == 3 and f.shape[3] == 32 and f.numel() > 0
            and describe_decoder(decoder) is not None)


def decoder_mlp(decoder, sampled_features):
    """The OSG decoder modules' forward ({'rgb', 'sigma'}) on the fused kernels, differentiable to first order w.r.t. the features
    and the decoder parameters (training/triplane.py:122-135, triplane_cond.py:869-970)."""
    nets, sigma_net, masks = describe_decoder(decoder)
    outs = []
    for net, mask in zip(nets, masks):
        w1, b1 = _effective_fc(net[0])
        w2, b2 = _effective_fc(net[2])
        outs.append(_DecoderMLP.apply(sampled_features, w1, b1, w2, b2, mask))
    sigma = outs[sigma_net][1]
    rgb = outs[0][0] if len(outs) == 1 else torch.cat([o[0] for o in outs], dim=-1)
    return {'rgb': rgb, 'sigma': sigma}


def fc_bias_act(x, weight, bias, weight_gain, bias_gain, act, alpha, act_gain):
    """FullyConnectedLayer.forward on p3d_fc_bias_act: x [B,in] fp32 (no gradients), act = p3d_bias_act code."""
    xc, wc = _f32c(x.detach()), _f32c(weight.detach())
    bc = None if bias is None else _f32c(bias.detach())
    y = torch.empty(xc.shape[0], wc.shape[0], device=xc.device, dtype=torch.float32)
    _lib.call('p3d_fc_bias_act', xc, wc, bc, y, xc.shape[0], xc.shape[1], wc.shape[0], float(weight_gain), float(bias_gain),
              int(act), float(alpha), float(act_gain), device=xc.device)
    return y
