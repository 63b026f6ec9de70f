"""Filtered leaky ReLU: bias -> upsample FIR -> lrelu(gain, slope, clamp) -> downsample FIR.

Surface of the reference's torch_utils/ops/filtered_lrelu.py:58 `filtered_lrelu` (only caller: StyleGAN3's alias-free
synthesis layer, training/networks_stylegan3.py:357). CUDA tensors run the fused sm_100a kernel `p3d_filtered_lrelu`
(csrc/filtered_lrelu.cu: the up-sampled intermediate stays in shared memory); its gradient is the same kernel with the
filters swapped and flipped, steered by the 2-bit sign tensor the forward pass wrote (reference :155-274). Configurations
the kernel reports as unsupported (the reference's `rc = -1`) compose `upfirdn2d` + the in-place sign-aware activation
`p3d_filtered_lrelu_act` + `upfirdn2d`, as the reference's fallback does (:225-231). CPU tensors / `impl='ref'` evaluate
the four-op reference composition (:123-155), differentiable to any order.
"""
import ctypes
import warnings

import numpy as np
import torch

from ... import _lib
from .. import misc
from . import bias_act
from . import upfirdn2d


def _get_filter_size(f):
    if f is None:
        return 1, 1
    assert isinstance(f, torch.Tensor) and 1 <= f.ndim <= 2
    return f.shape[-1], f.shape[0]


def _parse_padding(padding):
    if isinstance(padding, int):
        padding = [padding, padding]
    assert isinstance(padding, (list, tuple))
    padding = [int(v) for v in padding]
    if len(padding) == 2:
        px, py = padding
        padding = [px, px, py, py]
    px0, px1, py0, py1 = padding
    return px0, px1, py0, py1


def filtered_lrelu(x, fu=None, fd=None, b=None, up=1, down=1, padding=0, gain=np.sqrt(2), slope=0.2, clamp=None,
                   flip_filter=False, impl='cuda'):
    assert isinstance(x, torch.Tensor) and x.ndim == 4
    assert impl in ('ref', 'cuda')
    if impl == 'cuda' and x.device.type == 'cuda':
        return _cuda_op(up, down, _parse_padding(padding), float(gain), float(slope),
                        float(clamp if clamp is not None else 'inf'), bool(flip_filter)).apply(x, fu, fd, b, None, 0, 0)
    return _filtered_lrelu_ref(x, fu=fu, fd=fd, b=b, up=up, down=down, padding=padding, gain=gain, slope=slope, clamp=clamp,
                               flip_filter=flip_filter)


def _filtered_lrelu_ref(x, fu=None, fd=None, b=None, up=1, down=1, padding=0, gain=np.sqrt(2), slope=0.2, clamp=None,
                        flip_filter=False):
    """The four-op composition (reference :123-155)."""
    fu_w, fu_h = _get_filter_size(fu)
    fd_w, fd_h = _get_filter_size(fd)
    if b is not None:
        assert isinstance(b, torch.Tensor) and b.dtype == x.dtype
        misc.assert_shape(b, [x.shape[1]])
    assert isinstance(up, int) and up >= 1 and isinstance(down, int) and down >= 1
    px0, px1, py0, py1 = _parse_padding(padding)
    assert gain == float(gain) and gain > 0
    assert slope == float(slope) and slope >= 0
    assert clamp is None or (clamp == float(clamp) and clamp >= 0)
    n, c, ih, iw = x.shape
    out_w = (iw * up + (px0 + px1) - (fu_w - 1) - (fd_w - 1) + (down - 1)) // down
    out_h = (ih * up + (py0 + py1) - (fu_h - 1) - (fd_h - 1) + (down - 1)) // down
    in_dtype = x.dtype
    x = bias_act.bias_act(x=x, b=b, impl='ref')
    x = upfirdn2d.upfirdn2d(x=x, f=fu, up=up, padding=[px0, px1, py0, py1], gain=up ** 2, flip_filter=flip_filter, impl='ref')
    x = bias_act.bias_act(x=x, act='lrelu', alpha=slope, gain=gain, clamp=clamp, impl='ref')
    x = upfirdn2d.upfirdn2d(x=x, f=fd, down=down, flip_filter=flip_filter, impl='ref')
    misc.assert_shape(x, [n, c, out_h, out_w])
    assert x.dtype == in_dtype
    return x


# ---------------------------------------------------------------------------------------------
# Plugin-level entry points: the call signatures of the reference's pybind module (filtered_lrelu.cpp:20, :217), served by
# libp3d.so; `torch_utils.custom_ops.get_plugin('filtered_lrelu_plugin')` hands these out.
# ---------------------------------------------------------------------------------------------
def _plugin_filtered_lrelu(x, fu, fd, b, si, up, down, px0, px1, py0, py1, sx, sy, gain, slope, clamp, flip_filter, write_signs):
    """-> (y, so, return_code); return_code -1 = no fused kernel for this configuration (y, so are then None)."""
    assert x.is_cuda and x.ndim == 4 and x.numel() > 0
    assert fu.dtype == torch.float32 and fd.dtype == torch.float32 and 1 <= fu.ndim <= 2 and 1 <= fd.ndim <= 2
    assert b.dtype == x.dtype and b.ndim == 1 and b.shape[0] == x.shape[1]
    assert up >= 1 and down >= 1
    if x.dtype not in (torch.float16, torch.float32):
        return None, None, -1
    fu, fd = fu.contiguous(), fd.contiguous()
    n, c, xh, xw = x.shape
    fut_w, fut_h = fu.shape[-1] - 1, fu.shape[0] - 1
    fdt_w, fdt_h = fd.shape[-1] - 1, fd.shape[0] - 1
    cw = xw * up + (px0 + px1) - fut_w
    ch = xh * up + (py0 + py1) - fut_h
    if not (cw > fdt_w and ch > fdt_h):
        raise ValueError('upsampled buffer must be at least the size of downsampling filter')
    yw = (cw - fdt_w + (down - 1)) // down
    yh = (ch - fdt_h + (down - 1)) // down
    assert yw > 0 and yh > 0, 'output must be at least 1x1'
    fmt = torch.channels_last if (x.stride(1) == 1 and c > 1) else torch.contiguous_format
    y = torch.empty([n, c, yh, yw], dtype=x.dtype, device=x.device, memory_format=fmt)
    read_signs = si is not None and si.numel() > 0
    so, s, sw_active = None, si, 0
    if write_signs:
        sw_active = yw * down - (down - 1) + fdt_w
        sh = yh * down - (down - 1) + fdt_h
        sw = (sw_active + 15) & ~15
        s = so = torch.empty([n, c, sh, sw >> 2], dtype=torch.uint8, device=x.device)
    elif read_signs:
        sw_active = s.shape[3] << 2
    if read_signs or write_signs:
        assert s.is_contiguous() and s.dtype == torch.uint8 and s.device == x.device and s.ndim == 4
        assert s.shape[0] == n and s.shape[1] == c
    a = _lib.FilteredLReluArgs()
    a.x, a.y, a.b = x.data_ptr(), y.data_ptr(), b.data_ptr()
    a.s = s.data_ptr() if (read_signs or write_signs) else None
    a.fu, a.fd = fu.data_ptr(), fd.data_ptr()
    a.dtype = _lib.DTYPE_CODE[x.dtype]
    a.up, a.down = up, down
    a.fu_w, a.fu_h = fu.shape[-1], (fu.shape[0] if fu.ndim == 2 else 0)
    a.fd_w, a.fd_h = fd.shape[-1], (fd.shape[0] if fd.ndim == 2 else 0)
    a.px0, a.px1, a.py0, a.py1 = px0, px1, py0, py1
    a.gain, a.slope, a.clamp, a.flip = gain, slope, clamp, 1 if flip_filter else 0
    for k, v in enumerate((xw, xh, c, n)):
        a.x_shape[k] = v
    for k, v in enumerate((x.stride(3), x.stride(2), x.stride(1), x.stride(0))):
        a.x_stride[k] = v
    for k, v in enumerate((yw, yh, c, n)):
        a.y_shape[k] = v
    for k, v in enumerate((y.stride(3), y.stride(2), y.stride(1), y.stride(0))):
        a.y_stride[k] = v
    a.b_stride = b.stride(0)
    if read_signs or write_signs:
        a.s_shape[0], a.s_shape[1] = s.shape[3], s.shape[2]
    a.s_ofs[0], a.s_ofs[1] = sx, sy
    a.sw_limit = (sw_active + 3) >> 2
    a.sign_mode = 1 if write_signs else (2 if read_signs else 0)
    if not _lib.call('p3d_filtered_lrelu', ctypes.byref(a), device=x.device, unsupported_ok=True):
        return None, None, -1                      # P3D_UNSUPPORTED: the reference's rc = -1
    return y, so, 0


def _plugin_filtered_lrelu_act_(x, si, sx, sy, gain, slope, clamp, write_signs):
    """In place on x; returns the sign tensor when write_signs (filtered_lrelu.cpp:217-270)."""
    assert x.is_cuda and x.ndim == 4 and x.numel() > 0
    if x.dtype not in _lib.DTYPE_CODE:
        raise TypeError('filtered_lrelu_act_: x must be float16, float32 or float64')
    n, c, h, w = x.shape
    read_signs = si is not None and si.numel() > 0
    so, s = None, si
    if write_signs:
        sw = (w + 15) & ~15
        s = so = torch.empty([n, c, h, sw >> 2], dtype=torch.uint8, device=x.device)
    mode = 1 if write_signs else (2 if read_signs else 0)
    xs = (_lib.c_int32 * 4)(w, h, c, n)
    xst = (_lib.c_int64 * 4)(x.stride(3), x.stride(2), x.stride(1), x.stride(0))
    ss = (_lib.c_int32 * 2)(s.shape[3] << 2, s.shape[2]) if mode else (_lib.c_int32 * 2)(0, 0)
    so_ = (_lib.c_int32 * 2)(sx, sy)
    _lib.call('p3d_filtered_lrelu_act', x, s if mode else None, _lib.DTYPE_CODE[x.dtype], xs, xst, ss, so_, gain, slope, clamp, mode,
              device=x.device)
    return so


# ---------------------------------------------------------------------------------------------
_op_cache = {}


def _cuda_op(up, down, pads, gain, slope, clamp, flip_filter):
    """Autograd node over the fused kernel. Forward writes the sign tensor when a gradient will be needed; backward is the
    same node type with (up, down) and (fu, fd) swapped, flipped filters, gain * up^2 / down^2, no clamp, reading the signs
    (reference :178-270)."""
    key = (up, down, pads, gain, slope, clamp, flip_filter)
    if key in _op_cache:
        return _op_cache[key]
    px0, px1, py0, py1 = pads

    class FilteredLRelu(torch.autograd.Function):
        @staticmethod
        def forward(ctx, x, fu, fd, b, si, sx, sy):
            dev = x.device
            fu = torch.ones([1, 1], dtype=torch.float32, device=dev) if fu is None else fu
            fd = torch.ones([1, 1], dtype=torch.float32, device=dev) if fd is None else fd
            if up == 1 and fu.ndim == 1 and fu.shape[0] == 1:
                fu = fu.square()[None]
            if down == 1 and fd.ndim == 1 and fd.shape[0] == 1:
                fd = fd.square()[None]
            si = torch.empty([0], device=dev) if si is None else si
            bb = torch.zeros([x.shape[1]], dtype=x.dtype, device=dev) if b is None else b
            write_signs = si.numel() == 0 and (x.requires_grad or (b is not None and b.requires_grad))
            rc, y, so = -1, None, None
            if x.dtype in (torch.float16, torch.float32):
                y, so, rc = _plugin_filtered_lrelu(x, fu, fd, bb, si, up, down, px0, px1, py0, py1, sx, sy, gain, slope, clamp,
                                                   flip_filter, write_signs)
            if rc < 0:
                warnings.warn('filtered_lrelu: no fused kernel for these parameters, composing upfirdn2d + activation', RuntimeWarning)
                y = x.add(bb.unsqueeze(-1).unsqueeze(-1))
                y = upfirdn2d.upfirdn2d(x=y, f=fu, up=up, padding=[px0, px1, py0, py1], gain=up ** 2, flip_filter=flip_filter)
                so = _plugin_filtered_lrelu_act_(y, si, sx, sy, gain, slope, clamp, write_signs)
                y = upfirdn2d.upfirdn2d(x=y, f=fd, down=down, flip_filter=flip_filter)
            ctx.save_for_backward(fu, fd, si if si.numel() else so)
            ctx.x_shape, ctx.y_shape, ctx.s_ofs = x.shape, y.shape, (sx, sy)
            return y

        @staticmethod
        def backward(ctx, dy):
            fu, fd, si = ctx.saved_tensors
            _, _, xh, xw = ctx.x_shape
            _, _, yh, yw = ctx.y_shape
            sx, sy = ctx.s_ofs
            dx = db = None
            if ctx.needs_input_grad[0] or ctx.needs_input_grad[3]:
                pp = (fu.shape[-1] - 1 + fd.shape[-1] - 1 - px0, xw * up - yw * down + px0 - (up - 1),
                      fu.shape[0] - 1 + fd.shape[0] - 1 - py0, xh * up - yh * down + py0 - (up - 1))
                dx = _cuda_op(down, up, pp, gain * (up ** 2) / (down ** 2), slope, float('inf'), not flip_filter).apply(
                    dy, fd, fu, None, si, sx - (fu.shape[-1] - 1) + px0, sy - (fu.shape[0] - 1) + py0)
            if ctx.needs_input_grad[3]:
                db = dx.sum([0, 2, 3])
            return dx, None, None, db, None, None, None

    _op_cache[key] = FilteredLRelu
    return FilteredLRelu
