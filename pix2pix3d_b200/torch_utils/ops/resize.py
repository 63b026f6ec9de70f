"""Bilinear resize with optional anti-aliasing, `F.interpolate(x, size, mode='bilinear', align_corners=False,
antialias=...)` as the reference calls it in training/superresolution.py:315-319 and in `filtered_resizing`
(training/dual_discriminator.py:86-102).

CUDA tensors go through `p3d_resize_bilinear` (include/p3d.h, csrc/resize.cu); the backward is the adjoint launch of the
same kernel and differentiates to any order by self-recursion (the R1 penalty differentiates through the resize of the
real raw image). CPU tensors evaluate `F.interpolate`, as every op of the reference does for CPU inputs.
"""
import torch

from ... import _lib


def interpolate_bilinear(x, size, antialias=True, impl='cuda'):
    """x [N,C,H,W] -> [N,C,size[0],size[1]]."""
    assert isinstance(x, torch.Tensor) and x.ndim == 4
    assert impl in ('ref', 'cuda')
    if isinstance(size, int):
        size = (size, size)
    size = (int(size[0]), int(size[1]))
    if impl == 'cuda' and x.device.type == 'cuda' and x.dtype in _lib.DTYPE_CODE:
        return _Resize.apply(x, x.shape[2], x.shape[3], size[0], size[1], bool(antialias), False)
    return torch.nn.functional.interpolate(x, size=size, mode='bilinear', align_corners=False, antialias=bool(antialias))


def _launch(x, in_hw, out_hw, antialias, transposed):
    x = x.contiguous()
    n, c = x.shape[:2]
    dst = in_hw if transposed else out_hw
    y = torch.empty(n, c, dst[0], dst[1], device=x.device, dtype=x.dtype)
    _lib.call('p3d_resize_bilinear', x, y, _lib.DTYPE_CODE[x.dtype], n * c, in_hw[0], in_hw[1], out_hw[0], out_hw[1], int(antialias),
              int(transposed), device=x.device)
    return y


class _Resize(torch.autograd.Function):
    """`transposed=False`: the resize [in] -> [out]; `transposed=True`: its adjoint [out] -> [in]. Each is the other's
    backward, so gradients of any order stay on the kernel."""

    @staticmethod
    def forward(ctx, x, in_h, in_w, out_h, out_w, antialias, transposed):
        ctx.cfg = (in_h, in_w, out_h, out_w, antialias, transposed)
        src = (out_h, out_w) if transposed else (in_h, in_w)
        assert tuple(x.shape[2:]) == src
        return _launch(x, (in_h, in_w), (out_h, out_w), antialias, transposed)

    @staticmethod
    def backward(ctx, dy):
        in_h, in_w, out_h, out_w, antialias, transposed = ctx.cfg
        dx = None
        if ctx.needs_input_grad[0]:
            dx = _Resize.apply(dy, in_h, in_w, out_h, out_w, antialias, not transposed)
        return dx, None, None, None, None, None, None
