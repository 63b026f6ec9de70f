"""ctypes binding of libp3d.so (the C-ABI declared in include/p3d.h).

The library is built ahead of time by `pix2pix3d_b200.build`; there is no JIT and no fallback: a CUDA
tensor reaching an op without the library raises immediately.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'libp3d.so')
ABI_VERSION = 7

_lib = None

c_void_p, c_int, c_int8, c_int32, c_int64, c_float, c_uint32 = (
    ctypes.c_void_p, ctypes.c_int, ctypes.c_int8, ctypes.c_int32, ctypes.c_int64, ctypes.c_float, ctypes.c_uint32)

P3D_UNSUPPORTED = -1
P3D_F32, P3D_F16, P3D_F64 = 0, 1, 2
DTYPE_CODE = {torch.float32: P3D_F32, torch.float16: P3D_F16, torch.float64: P3D_F64}


class DecoderDesc(ctypes.Structure):  # p3d_decoder_t
    _fields_ = [
        ('n_nets', c_int32), ('sigma_net', c_int32), ('sigmoid_mask', c_uint32 * 2),
        ('w1', c_void_p * 2), ('b1', c_void_p * 2), ('w2', c_void_p * 2), ('b2', c_void_p * 2),
        ('w1_gain', c_float * 2), ('b1_gain', c_float * 2), ('w2_gain', c_float * 2), ('b2_gain', c_float * 2),
    ]


class RenderArgs(ctypes.Structure):  # p3d_render_args_t
    _fields_ = [
        ('planes_nhwc', c_void_p), ('ray_origins', c_void_p), ('ray_dirs', c_void_p), ('depths_coarse', c_void_p),
        ('u_importance', c_void_p), ('decoder_packed', c_void_p),
        ('n_nets', c_int32), ('sigma_net', c_int32), ('sigmoid_mask', c_uint32 * 2),
        ('B', c_int32), ('R', c_int32), ('H', c_int32), ('W', c_int32), ('Sc', c_int32), ('Sf', c_int32),
        ('coord_scale', c_float), ('white_back', c_int32),
        ('out_feat', c_void_p), ('out_depth', c_void_p), ('out_wsum', c_void_p),
        ('dbg_weights_coarse', c_void_p), ('dbg_depths_fine', c_void_p), ('dbg_inds', c_void_p),
        ('dbg_perm', c_void_p), ('dbg_weights_final', c_void_p),
        ('workspace', c_void_p),
        ('plane_strides', ctypes.c_int64 * 3),
        ('tc_variant', c_int32), ('depth_mode', c_int32),
        ('jitter', c_void_p), ('depth_table', c_void_p), ('ray_start', c_void_p), ('ray_end', c_void_p),
        ('depth_delta', c_float), ('reserved1', c_int32), ('plane_index', c_void_p),
    ]


class FilteredLReluArgs(ctypes.Structure):  # p3d_filtered_lrelu_args_t
    _fields_ = [
        ('x', c_void_p), ('y', c_void_p), ('b', c_void_p), ('s', c_void_p), ('fu', c_void_p), ('fd', c_void_p),
        ('dtype', c_int32), ('up', c_int32), ('down', c_int32),
        ('fu_w', c_int32), ('fu_h', c_int32), ('fd_w', c_int32), ('fd_h', c_int32),
        ('px0', c_int32), ('px1', c_int32), ('py0', c_int32), ('py1', c_int32),
        ('gain', c_float), ('slope', c_float), ('clamp', c_float), ('flip', c_int32),
        ('x_shape', c_int32 * 4), ('x_stride', c_int64 * 4), ('y_shape', c_int32 * 4), ('y_stride', c_int64 * 4),
        ('b_stride', c_int64), ('s_shape', c_int32 * 2), ('s_ofs', c_int32 * 2), ('sw_limit', c_int32), ('sign_mode', c_int32),
    ]


class ConvArgs(ctypes.Structure):  # p3d_conv_args_t
    _fields_ = [
        ('x', c_void_p), ('w', c_void_p),
        ('x_planes', c_int32), ('w_planes', c_int32), ('B', c_int32), ('Bw', c_int32),
        ('H', c_int32), ('W', c_int32), ('C', c_int32), ('Cout', c_int32),
        ('Cout_padded', c_int32), ('n_kblocks', c_int32), ('n_taps', c_int32),
        ('tap_dy', c_int8 * 9), ('tap_dx', c_int8 * 9), ('tap_k', c_int8 * 9),
        ('split', c_int32), ('gH', c_int32), ('gW', c_int32),
        ('oH', c_int32), ('oW', c_int32), ('sy', c_int32), ('oy', c_int32),
        ('sx', c_int32), ('ox', c_int32),
        ('y', c_void_p), ('y_lo', c_void_p),
        ('y_cstride', c_int32), ('y_coff', c_int32), ('out_mode', c_int32),
        ('bias', c_void_p), ('noise', c_void_p), ('dscale', c_void_p),
        ('act', c_int32), ('alpha', c_float), ('gain', c_float), ('clamp', c_float),
        ('acc_scale', c_float),
        ('up_prev', c_void_p), ('up_filter', c_void_p), ('round16', c_int32), ('out_nchw', c_int32),
        ('stride', c_int32), ('launch_flags', c_int32), ('residual', c_void_p),
        ('splitk_scratch', c_void_p), ('splitk_scratch_bytes', c_int64), ('noise_batch_stride', c_int64),
        ('rgb_w', c_void_p), ('rgb_bias', c_void_p), ('rgb_prev', c_void_p), ('rgb_filter', c_void_p),
        ('rgb_out', c_void_p), ('rgb_cout', c_int32), ('rgb_w_rows', c_int32), ('rgb_skip_x', c_int32),
        ('rgb_clamp', c_float), ('rgb_acc_scale', c_float),
    ]


class ModwDesc(ctypes.Structure):  # p3d_modw_desc_t
    _fields_ = [
        ('weight_t', c_void_p), ('wsq', c_void_p), ('styles_off', c_int64), ('out_off', c_int64),
        ('Cout', c_int32), ('Cin', c_int32), ('ktaps', c_int32), ('Cout_padded', c_int32),
        ('Cin_padded', c_int32), ('cin_offset', c_int32), ('demodulate', c_int32), ('planes', c_int32),
        ('pre_scale', c_float), ('out_scale', c_float), ('first_block', c_int32), ('reserved', c_int32),
    ]


# every struct of include/p3d.h except p3d_mesh_view_t, which crosses the ABI as MESH_VIEW_FLOATS floats
STRUCTS = {
    'p3d_decoder_t': DecoderDesc,
    'p3d_render_args_t': RenderArgs,
    'p3d_filtered_lrelu_args_t': FilteredLReluArgs,
    'p3d_conv_args_t': ConvArgs,
    'p3d_modw_desc_t': ModwDesc,
}

MESH_VIEW_FLOATS = 18    # p3d_mesh_view_t: world2cam rows 0-2 (12), eye (3), spot axis (3)

# entry -> (restype, argtypes, launches): argtypes is the header's full parameter list, the stream included; launches is what
# one successful call adds to launch_count, None for the query entries, which take no stream and return a value, not a status
_SIGNATURES = {
    'p3d_abi_version': (c_int, [], None),
    'p3d_build_info': (ctypes.c_char_p, [], None),
    'p3d_status_string': (ctypes.c_char_p, [c_int], None),
    'p3d_ray_sampler': (c_int, [c_void_p, c_void_p, c_int, c_int, c_void_p, c_void_p, c_void_p], 1),
    'p3d_ray_limits_box': (c_int, [c_void_p, c_void_p, c_int64, c_float, c_void_p, c_void_p, c_void_p], 1),
    'p3d_planes_to_channels_last': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p], 1),
    'p3d_pack_decoder': (c_int, [ctypes.POINTER(DecoderDesc), c_void_p, c_void_p], 1),
    'p3d_render_fwd': (c_int, [ctypes.POINTER(RenderArgs), c_void_p], 1),
    'p3d_pack_decoder_tc': (c_int, [ctypes.POINTER(DecoderDesc), c_void_p, c_void_p], 1),
    'p3d_render_fwd_tc': (c_int, [ctypes.POINTER(RenderArgs), c_void_p], 1),
    'p3d_run_model': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, ctypes.POINTER(c_uint32), c_int, c_int, c_int,
                              c_int, c_float, c_void_p, c_void_p, c_void_p], 1),
    'p3d_run_model_tc': (c_int, [c_void_p, ctypes.POINTER(ctypes.c_int64), c_void_p, c_void_p, c_int, c_int,
                                 ctypes.POINTER(c_uint32), c_int, ctypes.c_int64, c_int, c_int, c_float, c_void_p, c_void_p,
                                 c_void_p], 1),
    'p3d_resize_bilinear': (c_int, [c_void_p, c_void_p, c_int, ctypes.c_int64, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p], 1),
    'p3d_cross_entropy2d_fwd': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, ctypes.c_int64, ctypes.c_int64, c_void_p, c_void_p,
                                        c_void_p, c_void_p], 2),
    'p3d_cross_entropy2d_bwd': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, ctypes.c_int64,
                                        ctypes.c_int64, c_void_p, c_void_p], 1),
    'p3d_sample_from_planes_bwd': (c_int, [c_void_p, c_void_p, c_int, ctypes.c_int64, c_int, c_int, c_float, c_void_p, c_void_p], 1),
    'p3d_ray_march_bwd': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int,
                                  c_void_p, c_void_p, c_void_p], 1),
    'p3d_sample_from_planes': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p], 1),
    'p3d_ray_march': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
                              c_void_p, c_void_p], 1),
    'p3d_sample_importance': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p], 1),
    'p3d_bias_act': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float,
                             c_float, c_float, c_int64, c_int, c_int64, c_void_p], 1),
    'p3d_filtered_lrelu': (c_int, [ctypes.POINTER(FilteredLReluArgs), c_void_p], 1),
    'p3d_filtered_lrelu_act': (c_int, [c_void_p, c_void_p, c_int, ctypes.POINTER(c_int32), ctypes.POINTER(c_int64), ctypes.POINTER(c_int32),
                                       ctypes.POINTER(c_int32), c_float, c_float, c_float, c_int, c_void_p], 1),
    'p3d_upfirdn2d': (c_int, [c_void_p, c_void_p, c_void_p, c_int, ctypes.POINTER(c_int32), ctypes.POINTER(c_int64),
                              ctypes.POINTER(c_int32), ctypes.POINTER(c_int64), c_int, c_int, c_int, c_int, c_int, c_int,
                              c_int, c_int, c_int, c_float, c_void_p], 1),
    'p3d_fir_bias_act': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
                                 ctypes.POINTER(c_int32), ctypes.POINTER(c_int32), c_int, c_int, c_int, c_int, c_float,
                                 c_int, c_float, c_float, c_float, c_int64, c_void_p], 1),
    'p3d_decoder_mlp_fwd': (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_uint32, c_void_p, c_void_p,
                                    c_void_p, c_void_p], 1),
    'p3d_decoder_mlp_bwd_workspace_floats': (c_int, [], None),
    'p3d_decoder_mlp_bwd': (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_uint32, c_void_p, c_void_p,
                                    c_void_p, c_void_p, c_void_p, c_int64, c_void_p], 2),
    'p3d_fc_bias_act': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_float, c_float, c_int, c_float, c_float,
                                c_void_p], 1),
    'p3d_fma': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p], 1),
    'p3d_conv_gemm': (c_int, [c_void_p, c_void_p], 1),
    'p3d_conv_gemm_phases': (c_int, [c_void_p, c_int, c_void_p], 1),
    'p3d_prepare_weights': (c_int, [c_void_p, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p], 1),
    'p3d_modulate_weights_t': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float,
                                       c_float, c_int, c_void_p, c_void_p], 1),
    'p3d_modulate_weights_batch': (c_int, [c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_int, c_void_p], 1),
    'p3d_affine_batch': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p], 1),
    'p3d_modulate_weights': (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_float,
                                     c_int, c_void_p, c_void_p], 1),
    'p3d_nchw_to_nhwc_f16': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p], 1),
    'p3d_nhwc_to_nchw_f32': (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, c_void_p], 1),
    'p3d_fir_act_nhwc': (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int,
                                 c_int, c_int, c_int, c_int, c_float, c_int, c_float, c_float, c_float, c_int64, c_void_p], 1),
    'p3d_fir_act_nhwc_split': (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                       c_int, c_int, c_float, c_int, c_float, c_float, c_float, c_int64, c_void_p], 1),
    'p3d_fir_act_nhwc_sep': (c_int, [c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
                                     c_int, c_int, c_int, c_float, c_int, c_float, c_float, c_float, c_int64, c_void_p], 1),
    'p3d_upsample2x_nhwc': (c_int, [c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p], 1),
    'p3d_marching_cubes_workspace_bytes': (c_int64, [c_int64, c_int64, c_int64], None),
    'p3d_marching_cubes_count': (c_int, [c_void_p, c_int64, c_int64, c_int64, ctypes.c_double, c_void_p, c_int64, c_void_p,
                                         c_void_p], 2),
    'p3d_marching_cubes_emit': (c_int, [c_void_p, c_int64, c_int64, c_int64, ctypes.c_double, c_void_p, c_int64, c_void_p,
                                        c_void_p, c_void_p], 2),
    'p3d_mesh_raster': (c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int, c_int, c_int, c_float, c_float, c_float,
                                c_float, c_void_p, c_void_p, c_void_p], 1),
    'p3d_mesh_shade': (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int, c_int, c_int, c_float, c_float,
                               c_void_p, c_float, c_void_p, c_void_p], 1),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def available():
    return os.path.exists(LIB_PATH)


def lib():
    """Load (once) and return the ctypes handle; raises if the library has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f'{LIB_PATH} is missing: build it with `python -m pix2pix3d_b200.build` '
                '(there is no CPU or PyTorch fallback for CUDA tensors).')
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args, _) in _SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        got = handle.p3d_abi_version()
        if got != ABI_VERSION:
            raise RuntimeError(f'libp3d.so ABI {got} != expected {ABI_VERSION}; rebuild the library')
        _lib = handle
    return _lib


def check(status, what):
    if status != 0:
        msg = lib().p3d_status_string(status).decode()
        raise RuntimeError(f'{what} failed: {msg} (status {status})')


def stream_ptr(device=None):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


# count of native kernel launches issued through this module (bench.py reports it as gpu_launches)
launch_count = 0


def call(name, *args, device, unsupported_ok=False):
    """Run the launching entry `name` on the current stream of `device`. A torch.Tensor argument is passed as its data pointer,
    None as NULL and anything else (numbers, ctypes arrays, byref) as it is; the stream is appended. A nonzero status raises,
    except P3D_UNSUPPORTED under `unsupported_ok`, which returns False and counts nothing. Otherwise the entry's launches are
    added to launch_count and the result is True."""
    global launch_count
    launches = _SIGNATURES[name][2]
    if launches is None:
        raise ValueError(f'{name} is a query entry without a stream: call it on lib() directly')
    fn = getattr(lib(), name)
    args = [a.data_ptr() if isinstance(a, torch.Tensor) else a for a in args]
    with torch.cuda.device(device):
        st = fn(*args, stream_ptr())
    if st != 0:
        if unsupported_ok and st == P3D_UNSUPPORTED:
            return False
        check(st, name)
    launch_count += launches
    return True
