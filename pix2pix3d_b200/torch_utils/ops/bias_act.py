"""Fused bias + activation + gain + clamp.

Same surface as the reference's torch_utils/ops/bias_act.py (:54 `bias_act`, :23-33 `activation_funcs`).
CUDA tensors go through `p3d_bias_act` (include/p3d.h); CPU tensors, or `impl='ref'`, evaluate the op with
plain torch functions exactly as the reference does for those inputs (bias_act.py:86-88).
"""
import numpy as np
import torch

from ... import _lib
from ...dnnlib import EasyDict

_SQRT2 = float(np.sqrt(2))


def _spec(func, def_alpha, def_gain, cuda_idx, ref, has_2nd_grad):
    return EasyDict(func=func, def_alpha=def_alpha, def_gain=def_gain, cuda_idx=cuda_idx, ref=ref,
                    has_2nd_grad=has_2nd_grad)


activation_funcs = {
    'linear':   _spec(lambda x, **_: x,                                         0,   1,      1, '',  False),
    'relu':     _spec(lambda x, **_: torch.nn.functional.relu(x),               0,   _SQRT2, 2, 'y', False),
    'lrelu':    _spec(lambda x, alpha, **_: torch.nn.functional.leaky_relu(x, alpha), 0.2, _SQRT2, 3, 'y', False),
    'tanh':     _spec(lambda x, **_: torch.tanh(x),                             0,   1,      4, 'y', True),
    'sigmoid':  _spec(lambda x, **_: torch.sigmoid(x),                          0,   1,      5, 'y', True),
    'elu':      _spec(lambda x, **_: torch.nn.functional.elu(x),                0,   1,      6, 'y', True),
    'selu':     _spec(lambda x, **_: torch.nn.functional.selu(x),               0,   1,      7, 'y', True),
    'softplus': _spec(lambda x, **_: torch.nn.functional.softplus(x),           0,   1,      8, 'y', True),
    'swish':    _spec(lambda x, **_: torch.sigmoid(x) * x,                      0,   _SQRT2, 9, 'x', True),
}


def _resolve(act, alpha, gain, clamp):
    spec = activation_funcs[act]
    alpha = float(spec.def_alpha if alpha is None else alpha)
    gain = float(spec.def_gain if gain is None else gain)
    clamp = float(-1 if clamp is None else clamp)
    return spec, alpha, gain, clamp


def bias_act(x, b=None, dim=1, act='linear', alpha=None, gain=None, clamp=None, impl='cuda'):
    """y = clamp(act(x + b) * gain); differentiable to second order (needed by R1)."""
    assert isinstance(x, torch.Tensor)
    assert impl in ('ref', 'cuda')
    assert clamp is None or clamp >= 0
    if impl == 'cuda' and x.device.type == 'cuda':
        spec, alpha, gain, clamp = _resolve(act, alpha, gain, clamp)
        return _BiasAct.apply(x, b, int(dim), act, alpha, gain, clamp)
    return _bias_act_ref(x, b=b, dim=dim, act=act, alpha=alpha, gain=gain, clamp=clamp)


def _bias_act_ref(x, b=None, dim=1, act='linear', alpha=None, gain=None, clamp=None):
    """Composition of standard torch ops (reference bias_act.py:93-122)."""
    assert isinstance(x, torch.Tensor)
    spec, alpha, gain, clamp = _resolve(act, alpha, gain, clamp)
    if b is not None:
        assert isinstance(b, torch.Tensor) and b.ndim == 1
        assert 0 <= dim < x.ndim and b.shape[0] == x.shape[dim]
        shape = [1] * x.ndim
        shape[dim] = -1
        x = x + b.reshape(shape)
    x = spec.func(x, alpha=alpha)
    if gain != 1:
        x = x * gain
    if clamp >= 0:
        x = x.clamp(-clamp, clamp)
    return x


def _memory_format(t):
    return torch.channels_last if t.ndim > 2 and t.stride(1) == 1 else torch.contiguous_format


def _launch(x, b, xref, yref, dy, grad, dim, act_idx, alpha, gain, clamp):
    """Mirror of the plugin entry `bias_act(x, b, xref, yref, dy, grad, dim, act, alpha, gain, clamp)`
    (reference bias_act.cpp:36): all tensors dense and in the same memory format."""
    if x.dtype not in _lib.DTYPE_CODE:
        raise TypeError(f'bias_act: unsupported dtype {x.dtype}')
    if x.numel() > 0 and not (x.is_contiguous() or x.is_contiguous(memory_format=torch.channels_last)):
        raise ValueError('bias_act: x must be dense')
    for t in (xref, yref, dy):
        if t is not None:
            # same layout = equal strides on every dimension of size >= 2 (has_same_layout, reference bias_act.cpp:17-31)
            assert t.shape == x.shape and t.dtype == x.dtype
            assert all(ts == xs for ts, xs, n in zip(t.stride(), x.stride(), x.shape) if n >= 2)
    if b is not None:
        assert b.dtype == x.dtype and b.ndim == 1 and b.shape[0] == x.shape[dim] and b.is_contiguous()
    y = torch.empty_like(x)
    if x.numel() == 0:
        return y
    step_b = x.stride(dim) if b is not None else 1
    _lib.call('p3d_bias_act', x, b, xref, yref, dy, y, _lib.DTYPE_CODE[x.dtype], grad, act_idx, alpha, gain, clamp, x.numel(),
              0 if b is None else b.numel(), step_b, device=x.device)
    return y


class _BiasAct(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, b, dim, act, alpha, gain, clamp):
        spec = activation_funcs[act]
        fmt = _memory_format(x)
        x = x.contiguous(memory_format=fmt)
        b = b.contiguous() if b is not None else None
        y = x
        if act != 'linear' or gain != 1 or clamp >= 0 or b is not None:
            y = _launch(x, b, None, None, None, 0, dim, spec.cuda_idx, alpha, gain, clamp)
        need_x = ('x' in spec.ref) or spec.has_2nd_grad
        ctx.save_for_backward(x if need_x else None, b if need_x else None, y if 'y' in spec.ref else None)
        ctx.cfg = (dim, act, alpha, gain, clamp, fmt)
        ctx.has_b = b is not None
        return y

    @staticmethod
    def backward(ctx, dy):
        dim, act, alpha, gain, clamp, fmt = ctx.cfg
        x, b, y = ctx.saved_tensors
        dx = db = None
        if ctx.needs_input_grad[0] or ctx.needs_input_grad[1]:
            dy = dy.contiguous(memory_format=fmt)
            dx = dy
            if act != 'linear' or gain != 1 or clamp >= 0:
                dx = _BiasActGrad.apply(dy, x, b, y, dim, act, alpha, gain, clamp)
        if ctx.has_b and ctx.needs_input_grad[1]:
            db = dx.sum([i for i in range(dx.ndim) if i != dim])
        return dx, db, None, None, None, None, None


class _BiasActGrad(torch.autograd.Function):
    @staticmethod
    def forward(ctx, dy, x, b, y, dim, act, alpha, gain, clamp):
        spec = activation_funcs[act]
        fmt = _memory_format(dy)
        dx = _launch(dy, b, x, y, None, 1, dim, spec.cuda_idx, alpha, gain, clamp)
        ctx.save_for_backward(dy if spec.has_2nd_grad else None, x, b, y)
        ctx.cfg = (dim, act, alpha, gain, clamp, fmt)
        return dx

    @staticmethod
    def backward(ctx, d_dx):
        dim, act, alpha, gain, clamp, fmt = ctx.cfg
        spec = activation_funcs[act]
        dy, x, b, y = ctx.saved_tensors
        d_dx = d_dx.contiguous(memory_format=fmt)
        d_dy = d_x = d_b = None
        if ctx.needs_input_grad[0]:
            d_dy = _BiasActGrad.apply(d_dx, x, b, y, dim, act, alpha, gain, clamp)
        if spec.has_2nd_grad and (ctx.needs_input_grad[1] or ctx.needs_input_grad[2]):
            d_x = _launch(d_dx, b, x, y, dy, 2, dim, spec.cuda_idx, alpha, gain, clamp)
        if spec.has_2nd_grad and ctx.needs_input_grad[2]:
            d_b = d_x.sum([i for i in range(d_x.ndim) if i != dim])
        return d_dy, d_x, d_b, None, None, None, None, None, None
