"""Fused multiply-add `a * b + c` with broadcast-aware gradients (reference torch_utils/ops/fma.py:17-62).

CUDA tensors (fp16 / fp32 / fp64, up to four broadcast dimensions) run `p3d_fma` (csrc/fma.cu); the gradients are the same op with
other operands followed by sums over the broadcast dimensions, as the reference forms them -- so any order of differentiation
stays on the kernel. CPU tensors evaluate `torch.addcmul`, the reference's own forward.
"""
import ctypes

import torch


def fma(a, b, c):
    return _Fma.apply(a, b, c)


def _sum_to_shape(x, shape):
    """Reduce `x` over the dimensions that were broadcast from `shape`."""
    extra = x.ndim - len(shape)
    assert extra >= 0
    dims = [i for i in range(x.ndim) if i < extra or (x.shape[i] > 1 and shape[i - extra] == 1)]
    if dims:
        x = x.sum(dim=dims, keepdim=True)
    if extra:
        x = x.reshape(-1, *x.shape[extra + 1:])
    assert tuple(x.shape) == tuple(shape)
    return x


def _native_ok(a, b, c):
    if not (a.is_cuda and b.is_cuda and c.is_cuda):
        return False
    if not (a.dtype == b.dtype == c.dtype and a.dtype in (torch.float16, torch.float32, torch.float64)):
        return False
    return max(a.ndim, b.ndim, c.ndim) <= 4


def _addcmul(a, b, c):
    """out = a * b + c for broadcastable operands."""
    if not _native_ok(a, b, c):
        if a.is_cuda or b.is_cuda or c.is_cuda:
            if not (a.dtype == b.dtype == c.dtype):
                return torch.addcmul(c, a, b)          # mixed dtypes: type promotion is ATen's business (not on any pix2pix3D path)
            raise NotImplementedError('p3d_fma covers up to four dimensions')
        return torch.addcmul(c, a, b)
    from ... import _lib
    shape = torch.broadcast_shapes(a.shape, b.shape, c.shape)
    out = torch.empty(shape, device=a.device, dtype=a.dtype)
    if out.numel() == 0:
        return out
    pad = (1,) * (4 - len(shape))
    shape4 = pad + tuple(shape)

    def strides(t):
        e = t.expand(shape)
        return (0,) * len(pad) + tuple(0 if shape[i] == 1 else e.stride(i) for i in range(len(shape)))

    arr = ctypes.c_int64 * 4
    _lib.call('p3d_fma', a, b, c, out, _lib.DTYPE_CODE[a.dtype], arr(*shape4), arr(*strides(a)), arr(*strides(b)), arr(*strides(c)),
              device=a.device)
    return out


class _Fma(torch.autograd.Function):
    @staticmethod
    def forward(ctx, a, b, c):
        out = _addcmul(a, b, c)
        ctx.save_for_backward(a, b)
        ctx.c_shape = c.shape
        return out

    @staticmethod
    def backward(ctx, dout):
        a, b = ctx.saved_tensors
        da = db = dc = None
        if ctx.needs_input_grad[0]:
            da = _sum_to_shape(fma(dout, b, torch.zeros([], dtype=dout.dtype, device=dout.device)), a.shape)
        if ctx.needs_input_grad[1]:
            db = _sum_to_shape(fma(dout, a, torch.zeros([], dtype=dout.dtype, device=dout.device)), b.shape)
        if ctx.needs_input_grad[2]:
            dc = _sum_to_shape(dout, ctx.c_shape)
        return da, db, dc
