"""Tensor-level wrappers of the tensor-core convolution path (include/p3d.h: p3d_conv_gemm and helpers).

Tensors on this path are NHWC fp16; a *split* tensor is `[2,B,H,W,C]` (hi, lo) with value hi + lo.
"""
import ctypes
import os

import torch

from . import _lib, native
from ._lib import ConvArgs

WEIGHT_SCALE = 128.0   # power of two folded into the fp16 weights so that the `lo` halves stay normal numbers


# A/B switches of the convolution launcher (p3d_conv_args_t::launch_flags; results do not depend on them): bit 0 = never the
# persistent kernel, bit 1 = never CTA pairs. The environment is read HERE, once, by the host binding -- the library has no
# process-global switches.
launch_flags = (1 if os.environ.get('P3D_CONV_PERSIST') == '0' else 0) | (2 if os.environ.get('P3D_CONV_PAIR') == '0' else 0)


def pad_to(n, m):
    return (n + m - 1) // m * m


def to_nhwc_f16(x, c_padded=None, planes=1):
    """NCHW fp32/fp16 -> [planes,N,H,W,Cp] fp16."""
    assert x.is_cuda and x.ndim == 4
    x = x.contiguous()
    n, c, h, w = x.shape
    cp = c_padded or c
    out = torch.empty(planes, n, h, w, cp, device=x.device, dtype=torch.float16)
    _lib.call('p3d_nchw_to_nhwc_f16', x, _lib.DTYPE_CODE[x.dtype], n, c, h, w, cp, planes, out, device=x.device)
    return out


def nhwc_to_nchw_f32(x, channels=None, c_offset=0):
    """[N,H,W,Cs] fp32 -> [N,channels,H,W] fp32 taking channels [c_offset, c_offset+channels)."""
    assert x.is_cuda and x.dtype == torch.float32 and x.ndim == 4 and x.is_contiguous()
    n, h, w, cs = x.shape
    c = channels or cs
    out = torch.empty(n, c, h, w, device=x.device, dtype=torch.float32)
    _lib.call('p3d_nhwc_to_nchw_f32', x, n, c, h, w, cs, c_offset, out, device=x.device)
    return out


def prepare_weights(weight):
    """weight [O,I,kh,kw] fp32 -> (weight_t [O,kh*kw,I], wsq [O,I]): the parameter-only part of modulate_weights."""
    w = weight.detach().float().contiguous()
    o, i, kh, kw = w.shape
    wt = torch.empty(o, kh * kw, i, device=w.device, dtype=torch.float32)
    wsq = torch.empty(o, i, device=w.device, dtype=torch.float32)
    _lib.call('p3d_prepare_weights', w, o, i, kh * kw, wt, wsq, device=w.device)
    return wt, wsq


def modulate_weights(weight, styles, demodulate=True, pre_scale=1.0, planes=1, cin_padded=None, out_scale=WEIGHT_SCALE,
                     cin_offset=0, prepared=None):
    """weight [O,I,kh,kw] fp32, styles [B,I] fp32 -> [planes,B,Op,kh*kw*Ip] fp16, K-major (tap-major, then channel).
    `prepared` = prepare_weights(weight) selects the streaming two-step kernel."""
    s = styles.detach().float().contiguous()
    o, i, kh, kw = weight.shape
    b = s.shape[0]
    op, ip = pad_to(o, 16), (cin_padded or pad_to(i, 64))
    out = torch.empty(planes, b, op, kh * kw * ip, device=s.device, dtype=torch.float16)
    nchunk = ip // 8
    if prepared is not None and ip % 8 == 0 and nchunk <= 256 and 256 % nchunk == 0:
        wt, wsq = prepared
        _lib.call('p3d_modulate_weights_t', wt, wsq, s, b, o, i, kh * kw, op, ip, cin_offset, 1 if demodulate else 0,
                  float(pre_scale), float(out_scale), planes, out, device=s.device)
        return out
    w = weight.detach().float().contiguous()
    _lib.call('p3d_modulate_weights', w, s, b, o, i, kh * kw, op, ip, cin_offset, 1 if demodulate else 0, float(pre_scale),
              float(out_scale), planes, out, device=w.device)
    return out


def modulate_weights_batch(descs_dev, block_layer_dev, n_blocks, styles_flat, out_flat, batch):
    """One launch for every layer described by `descs_dev` (device bytes of _lib.ModwDesc[]); see p3d_modulate_weights_batch."""
    _lib.call('p3d_modulate_weights_batch', descs_dev, block_layer_dev, n_blocks, styles_flat, out_flat, batch,
              device=styles_flat.device)


def affine_batch(ws, weight, bias, meta, out_numel):
    """ws [B,num_ws,w_dim] fp32; weight [rows,w_dim] (gains applied), bias [rows], meta int32 [rows,4] -> flat fp32 buffer."""
    ws = ws.detach().float().contiguous()
    b, num_ws, w_dim = ws.shape
    out = torch.empty(out_numel, device=ws.device, dtype=torch.float32)
    _lib.call('p3d_affine_batch', ws, weight, bias, meta, out, b, num_ws, w_dim, weight.shape[0], device=ws.device)
    return out


_SPLITK_SCRATCH = {}


def _splitk_scratch(device):
    """One fp32 scratch buffer per (device, stream) for split-K partial sums (launches on a stream are ordered, so consecutive
    convolutions can share it)."""
    key = (device, torch.cuda.current_stream(device).cuda_stream)
    buf = _SPLITK_SCRATCH.get(key)
    if buf is None:
        buf = torch.empty(8 << 20, device=device, dtype=torch.float32)      # 32 MB
        _SPLITK_SCRATCH[key] = buf
    return buf


def _conv_args(x, w, cout, taps, grid_hw, out, out_lo=None, out_mode=0, out_map=(1, 0, 1, 0), y_coff=0, split=False, bias=None,
               noise=None, dscale=None, act=1, alpha=0.2, gain=1.0, clamp=-1.0, acc_scale=1.0 / WEIGHT_SCALE, split_k=True,
               up_prev=None, up_filter=None, round16=False, out_nchw=False, stride=1, residual=None, rgb=None):
    """The p3d_conv_args_t of one convolution launch (see conv_gemm)."""
    xp, b, h, wd, c = x.shape
    wp, bw, op, kk = w.shape
    assert x.dtype == torch.float16 and w.dtype == torch.float16 and x.is_contiguous() and w.is_contiguous()
    assert kk % c == 0
    a = ConvArgs()
    a.x, a.w = x.data_ptr(), w.data_ptr()
    a.x_planes, a.w_planes, a.B, a.Bw, a.H, a.W, a.C = xp, wp, b, bw, h, wd, c
    a.Cout, a.Cout_padded, a.n_kblocks, a.n_taps = cout, op, kk // c, len(taps)
    for i, (dy, dx, kb) in enumerate(taps):
        a.tap_dy[i], a.tap_dx[i], a.tap_k[i] = dy, dx, kb
    a.split = 1 if split else 0
    a.gH, a.gW = grid_hw
    if out_nchw:
        ob, ocs, oh, ow = out.shape
    else:
        ob, oh, ow, ocs = out.shape
    assert ob == b and out.is_contiguous()
    a.oH, a.oW = oh, ow
    a.sy, a.oy, a.sx, a.ox = out_map
    a.y = out.data_ptr()
    a.y_lo = None if out_lo is None else out_lo.data_ptr()
    a.y_cstride, a.y_coff, a.out_mode = ocs, y_coff, out_mode
    if out_mode in (0, 1):
        assert out.dtype == torch.float16
    else:
        assert out.dtype == torch.float32
    a.bias = None if bias is None else bias.data_ptr()
    a.noise = None if noise is None else noise.data_ptr()
    # [oH,oW] shared by the batch (noise_mode='const') or [B,oH,oW] (noise_mode='random')
    a.noise_batch_stride = 0 if (noise is None or noise.ndim == 2) else noise.shape[-2] * noise.shape[-1]
    a.dscale = None if dscale is None else dscale.data_ptr()
    for t in (bias, noise, dscale):
        assert t is None or (t.dtype == torch.float32 and t.is_contiguous())
    a.act, a.alpha, a.gain, a.clamp, a.acc_scale = act, alpha, gain, clamp, acc_scale
    a.stride = stride
    a.launch_flags = launch_flags
    if residual is not None:
        assert residual.dtype == torch.float32 and residual.is_contiguous() and tuple(residual.shape) == (b, grid_hw[0], grid_hw[1], cout)
        a.residual = residual.data_ptr()
    if up_prev is not None:      # fused ToRGB tail: out = upsample2d(up_prev, up_filter) + result
        assert up_prev.dtype == torch.float32 and up_prev.is_contiguous() and up_filter.dtype == torch.float32 and up_filter.numel() == 16
        a.up_prev, a.up_filter = up_prev.data_ptr(), up_filter.contiguous().data_ptr()
        a.round16, a.out_nchw = int(round16), int(out_nchw)
    if split_k:
        scratch = _splitk_scratch(x.device)
        a.splitk_scratch, a.splitk_scratch_bytes = scratch.data_ptr(), scratch.numel() * 4
    if rgb is not None:          # fused ToRGB of the next layer (p3d_conv_args_t::rgb_*)
        rw, rprev, rout = rgb['w'], rgb['prev'], rgb['out']
        assert rw.dtype == torch.float16 and rw.is_contiguous() and rw.ndim == 3 and rw.shape[0] == b and rw.shape[2] == cout
        assert rprev.dtype == torch.float32 and rprev.is_contiguous() and rout.dtype == torch.float32 and rout.is_contiguous()
        a.rgb_w, a.rgb_prev, a.rgb_out = rw.data_ptr(), rprev.data_ptr(), rout.data_ptr()
        a.rgb_bias = None if rgb.get('bias') is None else rgb['bias'].data_ptr()
        a.rgb_filter = rgb['filter'].contiguous().data_ptr()
        a.rgb_cout, a.rgb_w_rows, a.rgb_skip_x = rout.shape[1], rw.shape[1], int(bool(rgb.get('skip_x', False)))
        a.rgb_clamp, a.rgb_acc_scale = float(rgb.get('clamp', -1.0)), float(rgb.get('acc_scale', 1.0 / WEIGHT_SCALE))
    return a


def _conv_event(flops, split):
    """The native.kernel_events record of a convolution launch: `flops` are the algorithmic FLOPs of the convolution it
    implements (one pass); the fp32 layers execute 3x that on the tensor pipe (hi*hi + hi*lo + lo*hi)."""
    return 'conv_gemm', flops, flops * (3 if split else 1)


def conv_gemm(x, w, cout, taps, grid_hw, out, split=False, **kw):
    """x [xp,B,H,W,C] fp16, w [wp,Bw,Op,nk*C] fp16; taps: list of (dy, dx, kblock); grid_hw: computed grid;
    out: NHWC tensor [B,oH,oW,Cs] (fp16 or fp32); out_map = (sy, oy, sx, ox)."""
    a = _conv_args(x, w, cout, taps, grid_hw, out, split=split, **kw)
    flops = 2.0 * x.shape[1] * grid_hw[0] * grid_hw[1] * cout * len(taps) * x.shape[4]
    native.timed_call(_conv_event(flops, split), 'p3d_conv_gemm', ctypes.byref(a), device=x.device)
    return out


def conv_gemm_try(x, w, cout, taps, grid_hw, out, split=False, **kw):
    """conv_gemm that reports P3D_UNSUPPORTED (-1) as False instead of raising: for optional fusions (`rgb=`) whose launch shape
    the library decides on; the caller then takes the unfused sequence."""
    a = _conv_args(x, w, cout, taps, grid_hw, out, split=split, **kw)
    flops = 2.0 * x.shape[1] * grid_hw[0] * grid_hw[1] * cout * (len(taps) * x.shape[4] + (a.rgb_cout if a.rgb_w else 0))
    return native.timed_call(_conv_event(flops, split), 'p3d_conv_gemm', ctypes.byref(a), device=x.device, unsupported_ok=True)


TAPS_3X3 = [(ky - 1, kx - 1, ky * 3 + kx) for ky in range(3) for kx in range(3)]
TAPS_1X1 = [(0, 0, 0)]


def tconv_phase_taps(py, px):
    """Taps of output phase (py, px) of conv_transpose2d(stride=2, k=3): out[2j+py] += x[j - (ky-py)/2] * w[ky]."""
    kys = (0, 2) if py == 0 else (1,)
    kxs = (0, 2) if px == 0 else (1,)
    return [(-(ky - py) // 2, -(kx - px) // 2, ky * 3 + kx) for ky in kys for kx in kxs]


# A/B switch (results do not depend on it): P3D_CONV_MERGE_PHASES=0 launches the four phases of a transposed convolution one by one
MERGE_PHASES = os.environ.get('P3D_CONV_MERGE_PHASES') != '0'


def conv_transpose3x3_s2(x, w, cout, out, split=False, acc_scale=1.0 / WEIGHT_SCALE):
    """Stride-2 transposed 3x3 convolution as four phase GEMMs: x [xp,B,h,w,C] -> out [B,2h+1,2w+1,Cs] (pre-FIR). The phases
    (4, 2, 2 and 1 taps: heaviest first) run as ONE launch whose tile schedule walks all four (p3d_conv_gemm_phases)."""
    _, b, h, wd, c = x.shape
    mode = 2 if out.dtype == torch.float32 else 0
    phases = [(py, px, (h + 1 if py == 0 else h, wd + 1 if px == 0 else wd)) for py in (0, 1) for px in (0, 1)]
    if not MERGE_PHASES:
        for py, px, ghw in phases:
            conv_gemm(x, w, cout, tconv_phase_taps(py, px), ghw, out, out_mode=mode, out_map=(2, py, 2, px), split=split,
                      acc_scale=acc_scale)
        return out
    arr = (ConvArgs * 4)()
    flops = 0.0
    for k, (py, px, ghw) in enumerate(phases):
        taps = tconv_phase_taps(py, px)
        arr[k] = _conv_args(x, w, cout, taps, ghw, out, out_mode=mode, out_map=(2, py, 2, px), split=split, acc_scale=acc_scale)
        flops += 2.0 * b * ghw[0] * ghw[1] * cout * len(taps) * c
    native.timed_call(_conv_event(flops, split), 'p3d_conv_gemm_phases', arr, 4, device=x.device)
    return out


# 3: separable filters (setup_filter builds them) take p3d_fir_act_nhwc_sep; 1: always the 16-tap kernel (A/B runs). Read once here.
FIR_VARIANT = int(os.environ.get('P3D_FIR_VARIANT', '3'))

def separable_factors(f):
    """(fx, fy) as ctypes float[4] arrays with f[j][i] == fy[j] * fx[i] exactly (in fp32), or None. Looked up once per filter
    tensor and version (a device -> host copy; the result is kept ON the tensor object, so a new tensor that happens to reuse the
    address never inherits it), hence it must first happen outside CUDA-graph capture; upfirdn2d.setup_filter([1,3,3,1]) qualifies."""
    hit = getattr(f, '_p3d_separable', None)
    if hit is None or hit[0] != f._version:
        res = None
        if tuple(f.shape) == (4, 4) and f.dtype == torch.float32:
            m = f.detach().cpu()
            if float(m[0, 0]) != 0.0:
                fx = m[0].clone()
                fy = (m[:, 0] / m[0, 0]).clone()
                if torch.equal(fy[:, None] * fx[None, :], m):
                    res = ((ctypes.c_float * 4)(*fx.tolist()), (ctypes.c_float * 4)(*fy.tolist()))
        hit = (f._version, res)
        f._p3d_separable = hit
    return hit[1]


def fir_act_nhwc(x, f, noise, bias, out_planes, out_hw, pad0=(1, 1), fir_gain=4.0, act=3, alpha=0.2, act_gain=1.0, clamp=-1.0):
    """x [B,inH,inW,C] fp32/fp16 NHWC, or a split fp16 pair [2,B,inH,inW,C] -> [out_planes,B,outH,outW,C] fp16."""
    split_in = x.ndim == 5
    if split_in:
        assert x.shape[0] == 2 and x.dtype == torch.float16 and x.is_contiguous()
        _, b, ih, iw, c = x.shape
    else:
        b, ih, iw, c = x.shape
    oh, ow = out_hw
    y = torch.empty(out_planes, b, oh, ow, c, device=x.device, dtype=torch.float16)
    nbs = 0 if (noise is None or noise.ndim == 2) else oh * ow          # per-sample noise images (noise_mode='random')
    if noise is not None:
        assert noise.is_contiguous() and noise.dtype == torch.float32 and noise.shape[-2:] == (oh, ow)
    sep = separable_factors(f) if (FIR_VARIANT == 3 and not split_in) else None
    tail = (out_planes, b, ih, iw, oh, ow, c, pad0[0], pad0[1], fir_gain, act, alpha, act_gain, clamp, nbs)
    if sep is not None:
        _lib.call('p3d_fir_act_nhwc_sep', x, _lib.DTYPE_CODE[x.dtype], sep[0], sep[1], noise, bias, y, *tail, device=x.device)
    elif split_in:
        _lib.call('p3d_fir_act_nhwc_split', x, f, noise, bias, y, *tail, device=x.device)
    else:
        _lib.call('p3d_fir_act_nhwc', x, _lib.DTYPE_CODE[x.dtype], f, noise, bias, y, *tail, device=x.device)
    return y


def upsample2x_nhwc(x, f):
    b, h, w, c = x.shape
    y = torch.empty(b, 2 * h, 2 * w, c, device=x.device, dtype=torch.float32)
    _lib.call('p3d_upsample2x_nhwc', x, f, y, b, h, w, c, device=x.device)
    return y
