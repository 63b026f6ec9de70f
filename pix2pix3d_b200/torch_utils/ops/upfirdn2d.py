"""Pad / upsample / FIR-filter / downsample of image batches.

Same surface as the reference's torch_utils/ops/upfirdn2d.py (`setup_filter` :72, `upfirdn2d` :120,
`filter2d` :279, `upsample2d` :315, `downsample2d` :354 and the private parsing helpers that
conv2d_resample imports). CUDA tensors go through `p3d_upfirdn2d` (include/p3d.h).
"""
import numpy as np
import torch

from ... import _lib
from .. import misc


def _parse_scaling(scaling):
    if isinstance(scaling, int):
        scaling = [scaling, scaling]
    assert isinstance(scaling, (list, tuple)) and len(scaling) == 2
    sx, sy = scaling
    assert isinstance(sx, int) and isinstance(sy, int) and sx >= 1 and sy >= 1
    return sx, sy


def _parse_padding(padding):
    if isinstance(padding, int):
        padding = [padding, padding]
    assert isinstance(padding, (list, tuple))
    assert all(isinstance(v, int) for v in padding)
    if len(padding) == 2:
        px, py = padding
        padding = [px, px, py, py]
    px0, px1, py0, py1 = padding
    return px0, px1, py0, py1


def _get_filter_size(f):
    if f is None:
        return 1, 1
    assert isinstance(f, torch.Tensor) and f.ndim in (1, 2)
    fw, fh = int(f.shape[-1]), int(f.shape[0])
    assert fw >= 1 and fh >= 1
    return fw, fh


def setup_filter(f, device=torch.device('cpu'), normalize=True, flip_filter=False, gain=1, separable=None):
    """Turn a tap list / matrix into the float32 filter tensor the ops expect (reference :72-115)."""
    if f is None:
        f = 1
    f = torch.as_tensor(f, dtype=torch.float32)
    assert f.ndim in (0, 1, 2) and f.numel() > 0
    if f.ndim == 0:
        f = f[np.newaxis]
    if separable is None:
        separable = (f.ndim == 1 and f.numel() >= 8)
    if f.ndim == 1 and not separable:
        f = f.ger(f)
    assert f.ndim == (1 if separable else 2)
    if normalize:
        f = f / f.sum()
    if flip_filter:
        f = f.flip(list(range(f.ndim)))
    f = f * (gain ** (f.ndim / 2))
    return f.to(device=device)


def upfirdn2d(x, f, up=1, down=1, padding=0, flip_filter=False, gain=1, impl='cuda'):
    """zero-insert upsample by `up`, pad, convolve with `f`, keep every `down`-th sample."""
    assert isinstance(x, torch.Tensor)
    assert impl in ('ref', 'cuda')
    if impl == 'cuda' and x.device.type == 'cuda':
        upx, upy = _parse_scaling(up)
        downx, downy = _parse_scaling(down)
        pads = _parse_padding(padding)
        return _Upfirdn2d.apply(x, f, (upx, upy), (downx, downy), pads, bool(flip_filter), float(gain))
    return _upfirdn2d_ref(x, f, up=up, down=down, padding=padding, flip_filter=flip_filter, gain=gain)


def _upfirdn2d_ref(x, f, up=1, down=1, padding=0, flip_filter=False, gain=1):
    """Composition of standard torch ops (reference :169-213)."""
    assert isinstance(x, torch.Tensor) and x.ndim == 4
    if f is None:
        f = torch.ones([1, 1], dtype=torch.float32, device=x.device)
    assert isinstance(f, torch.Tensor) and f.ndim in (1, 2) and f.dtype == torch.float32
    n, c, ih, iw = x.shape
    upx, upy = _parse_scaling(up)
    downx, downy = _parse_scaling(down)
    px0, px1, py0, py1 = _parse_padding(padding)
    assert iw * upx + px0 + px1 >= f.shape[-1] and ih * upy + py0 + py1 >= f.shape[0]

    # zero insertion
    z = x.new_zeros([n, c, ih, upy, iw, upx])
    z[:, :, :, 0, :, 0] = x
    x = z.reshape(n, c, ih * upy, iw * upx)
    # pad (positive) / crop (negative)
    x = torch.nn.functional.pad(x, [max(px0, 0), max(px1, 0), max(py0, 0), max(py1, 0)])
    x = x[:, :, max(-py0, 0): x.shape[2] - max(-py1, 0), max(-px0, 0): x.shape[3] - max(-px1, 0)]
    # filter
    k = f * (gain ** (f.ndim / 2))
    k = k.to(x.dtype)
    if not flip_filter:
        k = k.flip(list(range(k.ndim)))
    k = k[np.newaxis, np.newaxis].repeat([c, 1] + [1] * k.ndim)
    if k.ndim == 4:
        x = torch.nn.functional.conv2d(x, k, groups=c)
    else:
        x = torch.nn.functional.conv2d(x, k.unsqueeze(2), groups=c)
        x = torch.nn.functional.conv2d(x, k.unsqueeze(3), groups=c)
    return x[:, :, ::downy, ::downx]


def _launch(x, f2d, upx, upy, downx, downy, px0, px1, py0, py1, flip, gain):
    """Mirror of the plugin entry `upfirdn2d(x, f, upx, upy, downx, downy, padx0, padx1, pady0, pady1,
    flip, gain)` (reference upfirdn2d.cpp:20): f rank-2 fp32, output layout follows the input."""
    assert x.ndim == 4 and f2d.ndim == 2 and f2d.dtype == torch.float32
    if x.dtype not in _lib.DTYPE_CODE:
        raise TypeError(f'upfirdn2d: unsupported dtype {x.dtype}')
    n, c, ih, iw = x.shape
    fh, fw = f2d.shape
    ow = (iw * upx + px0 + px1 - fw + downx) // downx
    oh = (ih * upy + py0 + py1 - fh + downy) // downy
    if ow < 1 or oh < 1:
        raise ValueError('upfirdn2d: output must be at least 1x1')
    fmt = torch.channels_last if (x.stride(1) == 1 and c > 1) else torch.contiguous_format
    y = torch.empty([n, c, oh, ow], dtype=x.dtype, device=x.device, memory_format=fmt)
    f2d = f2d.contiguous()
    xs = (_lib.c_int32 * 4)(*x.shape)
    xst = (_lib.c_int64 * 4)(*x.stride())
    ys = (_lib.c_int32 * 4)(*y.shape)
    yst = (_lib.c_int64 * 4)(*y.stride())
    _lib.call('p3d_upfirdn2d', x, f2d, y, _lib.DTYPE_CODE[x.dtype], xs, xst, ys, yst, fw, fh, upx, upy, downx, downy, px0, py0,
              1 if flip else 0, gain, device=x.device)
    return y


class _Upfirdn2d(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, f, up, down, pads, flip_filter, gain):
        assert isinstance(x, torch.Tensor) and x.ndim == 4
        upx, upy = up
        downx, downy = down
        px0, px1, py0, py1 = pads
        if f is None:
            f = torch.ones([1, 1], dtype=torch.float32, device=x.device)
        if f.ndim == 1 and f.shape[0] == 1:
            f = f.square().unsqueeze(0)
        assert f.ndim in (1, 2)
        if f.device != x.device:
            f = f.to(x.device)
        if f.ndim == 2:
            y = _launch(x, f, upx, upy, downx, downy, px0, px1, py0, py1, flip_filter, gain)
        else:  # separable: a horizontal then a vertical pass
            y = _launch(x, f.unsqueeze(0), upx, 1, downx, 1, px0, px1, 0, 0, flip_filter, 1.0)
            y = _launch(y, f.unsqueeze(1), 1, upy, 1, downy, 0, 0, py0, py1, flip_filter, gain)
        ctx.save_for_backward(f)
        ctx.cfg = (up, down, pads, flip_filter, gain, tuple(x.shape))
        return y

    @staticmethod
    def backward(ctx, dy):
        f, = ctx.saved_tensors
        (upx, upy), (downx, downy), (px0, _px1, py0, _py1), flip_filter, gain, (_, _, ih, iw) = ctx.cfg
        _, _, oh, ow = dy.shape
        fw, fh = _get_filter_size(f)
        # adjoint = the same op with up/down swapped, mirrored filter and complementary padding
        pads = (fw - px0 - 1, iw * upx - ow * downx + px0 - upx + 1,
                fh - py0 - 1, ih * upy - oh * downy + py0 - upy + 1)
        dx = None
        if ctx.needs_input_grad[0]:
            dx = _Upfirdn2d.apply(dy, f, (downx, downy), (upx, upy), pads, not flip_filter, gain)
        return dx, None, None, None, None, None, None


def filter2d(x, f, padding=0, flip_filter=False, gain=1, impl='cuda'):
    """Same-size FIR filtering."""
    px0, px1, py0, py1 = _parse_padding(padding)
    fw, fh = _get_filter_size(f)
    p = [px0 + fw // 2, px1 + (fw - 1) // 2, py0 + fh // 2, py1 + (fh - 1) // 2]
    return upfirdn2d(x, f, padding=p, flip_filter=flip_filter, gain=gain, impl=impl)


def upsample2d(x, f, up=2, padding=0, flip_filter=False, gain=1, impl='cuda'):
    """Upsample by an integer factor; output is `up` times the input size."""
    upx, upy = _parse_scaling(up)
    px0, px1, py0, py1 = _parse_padding(padding)
    fw, fh = _get_filter_size(f)
    p = [px0 + (fw + upx - 1) // 2, px1 + (fw - upx) // 2, py0 + (fh + upy - 1) // 2, py1 + (fh - upy) // 2]
    return upfirdn2d(x, f, up=up, padding=p, flip_filter=flip_filter, gain=gain * upx * upy, impl=impl)


def downsample2d(x, f, down=2, padding=0, flip_filter=False, gain=1, impl='cuda'):
    """Downsample by an integer factor; output is 1/`down` of the input size."""
    downx, downy = _parse_scaling(down)
    px0, px1, py0, py1 = _parse_padding(padding)
    fw, fh = _get_filter_size(f)
    p = [px0 + (fw - downx + 1) // 2, px1 + (fw - downx) // 2, py0 + (fh - downy + 1) // 2, py1 + (fh - downy) // 2]
    return upfirdn2d(x, f, down=down, padding=p, flip_filter=flip_filter, gain=gain, impl=impl)
