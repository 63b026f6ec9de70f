"""Tensor-core convolution path (p3d_conv_gemm + helpers) against float64 torch references."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err

pytestmark = pytest.mark.gpu


def _h(x):   # value after fp16 rounding, as float64
    return x.half().double()


def _weights_kmajor(w, planes=1, scale=1.0):
    """[O,I,kh,kw] fp32 -> [planes,1,Op,kh*kw*Ip] fp16 K-major (tap-major) without modulation."""
    from pix2pix3d_b200 import tcconv
    o, i, kh, kw = w.shape
    ones = torch.ones(1, i, device=w.device)
    return tcconv.modulate_weights(w, ones, demodulate=False, planes=planes, out_scale=scale)


@pytest.mark.parametrize('shape', [(1, 64, 8, 16, 32), (2, 128, 5, 7, 48), (1, 64, 16, 16, 130), (3, 192, 4, 4, 16)])
def test_gemm_as_1x1_conv(shape):
    from pix2pix3d_b200 import tcconv
    b, c, h, w, cout = shape
    torch.manual_seed(0)
    x = torch.randn(b, c, h, w, device='cuda')
    wt = torch.randn(cout, c, 1, 1, device='cuda') / np.sqrt(c)
    xn = tcconv.to_nhwc_f16(x)
    wk = _weights_kmajor(wt)
    out = torch.zeros(b, h, w, cout, device='cuda', dtype=torch.float32)
    tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_1X1, (h, w), out, out_mode=2, acc_scale=1.0)
    ref = F.conv2d(_h(x).cpu(), _h(wt).cpu())
    assert rel_err(out.permute(0, 3, 1, 2).cpu().numpy(), ref.numpy()) < 2e-6


@pytest.mark.parametrize('shape', [(2, 64, 16, 16, 64), (1, 128, 9, 13, 32), (1, 64, 32, 32, 256), (2, 64, 4, 4, 16)])
def test_conv3x3_single_pass(shape):
    from pix2pix3d_b200 import tcconv
    b, c, h, w, cout = shape
    torch.manual_seed(1)
    x = torch.randn(b, c, h, w, device='cuda')
    wt = torch.randn(cout, c, 3, 3, device='cuda') / np.sqrt(9 * c)
    xn = tcconv.to_nhwc_f16(x)
    wk = _weights_kmajor(wt, scale=tcconv.WEIGHT_SCALE)
    out = torch.zeros(b, h, w, cout, device='cuda', dtype=torch.float32)
    tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_3X3, (h, w), out, out_mode=2)
    ref = F.conv2d(_h(x).cpu(), _h(wt * tcconv.WEIGHT_SCALE).cpu() / tcconv.WEIGHT_SCALE, padding=1)
    assert rel_err(out.permute(0, 3, 1, 2).cpu().numpy(), ref.numpy()) < 2e-6


def test_conv3x3_split_three_pass_is_fp32_accurate():
    from pix2pix3d_b200 import tcconv
    torch.manual_seed(2)
    b, c, h, w, cout = 2, 128, 16, 16, 96
    x = torch.randn(b, c, h, w, device='cuda') * 3
    wt = torch.randn(cout, c, 3, 3, device='cuda') / np.sqrt(9 * c)
    xn = tcconv.to_nhwc_f16(x, planes=2)
    assert rel_err((xn[0].float() + xn[1].float()).permute(0, 3, 1, 2).cpu().numpy(), x.cpu().numpy()) < 1e-6
    wk = _weights_kmajor(wt, planes=2, scale=tcconv.WEIGHT_SCALE)
    out = torch.zeros(b, h, w, cout, device='cuda', dtype=torch.float32)
    tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_3X3, (h, w), out, out_mode=2, split=True)
    ref = F.conv2d(x.double().cpu(), wt.double().cpu(), padding=1)
    # fp32-level, not fp16-level (5e-4); the tensor core's fp32 accumulator truncates, which leaves ~6e-6 over K = 3456
    assert rel_err(out.permute(0, 3, 1, 2).cpu().numpy(), ref.numpy()) < 2e-5
    single = torch.zeros_like(out)
    tcconv.conv_gemm(xn[:1].contiguous(), wk[:1].contiguous(), cout, tcconv.TAPS_3X3, (h, w), single, out_mode=2)
    assert rel_err(single.permute(0, 3, 1, 2).cpu().numpy(), ref.numpy()) > 1e-4    # the one-pass result is visibly coarser


@pytest.mark.parametrize('hw', [(4, 4), (8, 8), (7, 5), (16, 16), (33, 33)])
def test_transposed_conv_phases(hw):
    from pix2pix3d_b200 import tcconv
    torch.manual_seed(3)
    b, c, cout = 2, 64, 48
    h, w = hw
    x = torch.randn(b, c, h, w, device='cuda')
    wt = torch.randn(cout, c, 3, 3, device='cuda') / np.sqrt(9 * c)
    xn = tcconv.to_nhwc_f16(x)
    wk = _weights_kmajor(wt, scale=tcconv.WEIGHT_SCALE)
    out = torch.full((b, 2 * h + 1, 2 * w + 1, cout), float('nan'), device='cuda', dtype=torch.float32)
    tcconv.conv_transpose3x3_s2(xn, wk, cout, out)
    assert torch.isfinite(out).all(), 'every output pixel must be written by exactly one phase'
    ref = F.conv_transpose2d(_h(x).cpu(), (_h(wt * tcconv.WEIGHT_SCALE).cpu() / tcconv.WEIGHT_SCALE).transpose(0, 1), stride=2)
    assert rel_err(out.permute(0, 3, 1, 2).cpu().numpy(), ref.numpy()) < 2e-6


def test_epilogue_noise_bias_lrelu_clamp_and_output_modes():
    from pix2pix3d_b200 import tcconv
    torch.manual_seed(4)
    b, c, h, w, cout = 2, 64, 12, 12, 40
    x = torch.randn(b, c, h, w, device='cuda')
    wt = torch.randn(cout, c, 3, 3, device='cuda') / np.sqrt(9 * c)
    bias = torch.randn(cout, device='cuda')
    noise = torch.randn(h, w, device='cuda') * 0.5
    dscale = torch.rand(b, cout, device='cuda') + 0.5
    xn = tcconv.to_nhwc_f16(x)
    wk = _weights_kmajor(wt, scale=tcconv.WEIGHT_SCALE)
    ref = F.conv2d(_h(x).cpu(), _h(wt * tcconv.WEIGHT_SCALE).cpu() / tcconv.WEIGHT_SCALE, padding=1)
    ref = ref * dscale.double().cpu()[:, :, None, None] + noise.double().cpu() + bias.double().cpu()[None, :, None, None]
    ref = F.leaky_relu(ref, 0.2) * np.sqrt(2)
    ref = ref.clamp(-1.5, 1.5)
    kw = dict(bias=bias, noise=noise, dscale=dscale, act=3, alpha=0.2, gain=float(np.sqrt(2)), clamp=1.5)
    o32 = torch.zeros(b, h, w, cout, device='cuda')
    tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_3X3, (h, w), o32, out_mode=2, **kw)
    assert rel_err(o32.permute(0, 3, 1, 2).cpu().numpy(), ref.numpy()) < 3e-6
    # fp16 and split outputs, written at a channel offset inside a wider tensor
    wide = torch.zeros(b, h, w, 64, device='cuda', dtype=torch.float16)
    wide_lo = torch.zeros_like(wide)
    tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_3X3, (h, w), wide, out_lo=wide_lo, out_mode=1, y_coff=8, **kw)
    assert (wide[..., :8] == 0).all() and (wide[..., 48:] == 0).all()
    got = (wide.float() + wide_lo.float())[..., 8:48].permute(0, 3, 1, 2)
    assert rel_err(got.cpu().numpy(), ref.numpy()) < 3e-6
    assert rel_err(wide[..., 8:48].float().permute(0, 3, 1, 2).cpu().numpy(), ref.numpy()) < 1e-3
    # accumulate mode
    acc = torch.ones(b, h, w, cout, device='cuda')
    tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_3X3, (h, w), acc, out_mode=3, **kw)
    assert rel_err((acc - 1).permute(0, 3, 1, 2).cpu().numpy(), ref.numpy()) < 3e-6


def test_split_k_small_grids_match_single_pass_order():
    """4^2..16^2 backbone layers: the K range is split over up to 16 CTAs and reduced by a second kernel (deterministic)."""
    from pix2pix3d_b200 import tcconv
    torch.manual_seed(11)
    b, c, h, w, cout = 2, 512, 8, 8, 512
    x = torch.randn(b, c, h, w, device='cuda')
    wt = torch.randn(cout, c, 3, 3, device='cuda') / np.sqrt(9 * c)
    bias = torch.randn(cout, device='cuda')
    noise = torch.randn(h, w, device='cuda') * 0.5
    xn = tcconv.to_nhwc_f16(x, planes=2)
    wk = _weights_kmajor(wt, planes=2, scale=tcconv.WEIGHT_SCALE)
    kw = dict(split=True, bias=bias, noise=noise, act=3, alpha=0.2, gain=float(np.sqrt(2)))
    outs = []
    for split_k in (False, True, True):
        hi = torch.zeros(b, h, w, cout, device='cuda', dtype=torch.float16)
        lo = torch.zeros_like(hi)
        tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_3X3, (h, w), hi, out_lo=lo, out_mode=1, split_k=split_k, **kw)
        outs.append(hi.float() + lo.float())
    assert torch.equal(outs[1], outs[2])                                   # fixed reduction order
    ref = F.conv2d(x.double().cpu(), wt.double().cpu(), padding=1) + noise.double().cpu() + bias.double().cpu()[None, :, None, None]
    ref = F.leaky_relu(ref, 0.2) * np.sqrt(2)
    for o in outs:
        assert rel_err(o.permute(0, 3, 1, 2).cpu().numpy(), ref.numpy()) < 3e-5      # K = 4608: fp32 TMEM accumulation
    # the two orders differ by the tensor core's truncating fp32 accumulation over K = 4608 (split-K rounds partials properly)
    assert rel_err(outs[1].cpu().numpy(), outs[0].cpu().numpy()) < 4e-5


def test_modulate_weights_matches_modulated_conv2d_formula():
    from pix2pix3d_b200 import tcconv
    torch.manual_seed(5)
    b, o, i = 3, 40, 100
    wt = torch.randn(o, i, 3, 3, device='cuda')
    st = torch.randn(b, i, device='cuda') + 1
    prep = tcconv.prepare_weights(wt)
    for demod, prepared in ((True, None), (False, None), (True, prep), (False, prep)):
        wk = tcconv.modulate_weights(wt, st, demodulate=demod, pre_scale=0.7, planes=2, out_scale=4.0, prepared=prepared)
        assert wk.shape == (2, b, 48, 9 * 128)
        w = wt.double()[None] * (st.double() * 0.7)[:, None, :, None, None]
        if demod:
            w = w * (w.square().sum(dim=[2, 3, 4], keepdim=True) + 1e-8).rsqrt()
        ref = torch.zeros(b, 48, 9, 128, dtype=torch.float64, device='cuda')
        ref[:, :o, :, :i] = (w * 4.0).permute(0, 1, 3, 4, 2).reshape(b, o, 9, i)
        got = (wk[0].double() + wk[1].double()).reshape(b, 48, 9, 128)
        assert rel_err(got.cpu().numpy(), ref.cpu().numpy()) < 2e-6
    # channel-slice form (cin_offset) through both kernels
    for prepared in (None, prep):
        wk = tcconv.modulate_weights(wt, st, demodulate=True, planes=1, cin_padded=256, cin_offset=128, prepared=prepared)
        got = wk[0].double().reshape(b, 48, 9, 256)
        assert float(got[..., :128].abs().max()) == 0 and float(got[..., 228:].abs().max()) == 0
        w = wt.double()[None] * st.double()[:, None, :, None, None]
        w = w * (w.square().sum(dim=[2, 3, 4], keepdim=True) + 1e-8).rsqrt() * tcconv.WEIGHT_SCALE
        ref = w.permute(0, 1, 3, 4, 2).reshape(b, o, 9, i)
        assert rel_err(got[:, :o, :, 128:228].cpu().numpy(), ref.cpu().numpy()) < 2e-3     # single fp16 plane


def test_layout_converters_roundtrip():
    from pix2pix3d_b200 import tcconv
    torch.manual_seed(6)
    x = torch.randn(2, 37, 9, 11, device='cuda')
    n = tcconv.to_nhwc_f16(x, c_padded=64, planes=2)
    assert n.shape == (2, 2, 9, 11, 64) and (n[..., 37:] == 0).all()
    back = (n[0].float() + n[1].float())[..., :37].permute(0, 3, 1, 2)
    assert rel_err(back.cpu().numpy(), x.cpu().numpy()) < 1e-6
    img = torch.randn(2, 9, 11, 96, device='cuda')
    p = tcconv.nhwc_to_nchw_f32(img, channels=32, c_offset=32)
    assert torch.equal(p, img[..., 32:64].permute(0, 3, 1, 2).contiguous())


def test_fir_act_nhwc_and_upsample_match_reference_ops():
    from pix2pix3d_b200 import tcconv
    from pix2pix3d_b200.torch_utils.ops import bias_act, upfirdn2d
    torch.manual_seed(7)
    f = upfirdn2d.setup_filter([1, 3, 3, 1]).cuda()
    b, c, h = 2, 64, 9
    x = torch.randn(b, c, 2 * h + 1, 2 * h + 1, device='cuda')
    noise = torch.randn(2 * h, 2 * h, device='cuda') * 0.3
    bias = torch.randn(c, device='cuda')
    ref = upfirdn2d.upfirdn2d(x, f, padding=[1, 1, 1, 1], gain=4)
    ref = bias_act.bias_act(ref + noise, bias, act='lrelu', gain=1.3, clamp=2.0)
    y = tcconv.fir_act_nhwc(x.permute(0, 2, 3, 1).contiguous(), f, noise, bias, 2, (2 * h, 2 * h), act_gain=1.3 * float(np.sqrt(2)) / float(np.sqrt(2)) * float(np.sqrt(2)),
                            clamp=2.0)
    got = (y[0].float() + y[1].float()).permute(0, 3, 1, 2)
    ref2 = bias_act.bias_act(upfirdn2d.upfirdn2d(x, f, padding=[1, 1, 1, 1], gain=4) + noise, bias, act='lrelu', gain=1.3 * float(np.sqrt(2)), clamp=2.0)
    assert rel_err(got.cpu().numpy(), ref2.cpu().numpy()) < 2e-6
    xh = x.half()
    yh = tcconv.fir_act_nhwc(xh.permute(0, 2, 3, 1).contiguous(), f, noise, bias.float(), 1, (2 * h, 2 * h), act_gain=float(np.sqrt(2)), clamp=256.0)
    refh = bias_act.bias_act(upfirdn2d.upfirdn2d(xh, f, padding=[1, 1, 1, 1], gain=4).add_(noise), bias.half(), act='lrelu', clamp=256)
    assert rel_err(yh[0].float().permute(0, 3, 1, 2).cpu().numpy(), refh.float().cpu().numpy()) < 2e-3
    img = torch.randn(2, 6, 7, 5, device='cuda')
    up = tcconv.upsample2x_nhwc(img.permute(0, 2, 3, 1).contiguous(), f)
    assert rel_err(up.permute(0, 3, 1, 2).cpu().numpy(), upfirdn2d.upsample2d(img, f).cpu().numpy()) < 2e-6


def test_conv_large_tile_counts_and_fp16_output():
    """SR-sized layer slice: 128 channels at 128^2, many tiles per launch; fp16 NHWC output."""
    from pix2pix3d_b200 import tcconv
    torch.manual_seed(8)
    b, c, h, w, cout = 1, 128, 128, 128, 128
    x = torch.randn(b, c, h, w, device='cuda')
    wt = torch.randn(cout, c, 3, 3, device='cuda') / np.sqrt(9 * c)
    st = torch.randn(b, c, device='cuda') + 1
    xn = tcconv.to_nhwc_f16(x)
    wk = tcconv.modulate_weights(wt, st, demodulate=True)
    out = torch.zeros(b, h, w, cout, device='cuda', dtype=torch.float16)
    tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_3X3, (h, w), out, out_mode=0)
    wm = wt[None] * st[:, None, :, None, None]
    wm = wm * (wm.square().sum(dim=[2, 3, 4], keepdim=True) + 1e-8).rsqrt()
    torch.backends.cudnn.allow_tf32 = False
    ref = F.conv2d(x.half().float(), wm[0], padding=1)
    assert rel_err(out.float().permute(0, 3, 1, 2).cpu().numpy(), ref.cpu().numpy()) < 2e-3


@pytest.mark.parametrize('cout,hw,split,nchw', [(3, (32, 48), False, True), (6, (16, 16), False, False), (96, (32, 32), True, False),
                                                (19, (64, 64), False, True), (96, (256, 256), True, False),
                                                (3, (256, 256), False, True), (6, (256, 192), False, True)])
def test_fused_torgb_tail_matches_upsample_plus_conv(cout, hw, split, nchw):
    """out = upsample2d(prev, f) + ToRGB(x) in the convolution epilogue (networks_stylegan2.py:452-458), incl. the fp16
    rounding of y in fp16 blocks and the direct NCHW output of the last block."""
    from pix2pix3d_b200 import tcconv
    from pix2pix3d_b200.torch_utils.ops import upfirdn2d
    torch.manual_seed(12)
    b, c = 2, 128
    h, w = hw
    f = upfirdn2d.setup_filter([1, 3, 3, 1]).cuda()
    x = torch.randn(b, c, h, w, device='cuda')
    wt = torch.randn(cout, c, 1, 1, device='cuda') / np.sqrt(c)
    bias = torch.randn(cout, device='cuda')
    prev = torch.randn(b, h // 2, w // 2, cout, device='cuda')
    planes = 2 if split else 1
    xn = tcconv.to_nhwc_f16(x, planes=planes)
    wk = _weights_kmajor(wt, planes=planes, scale=tcconv.WEIGHT_SCALE)
    out = torch.empty((b, cout, h, w) if nchw else (b, h, w, cout), device='cuda')
    tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_1X1, (h, w), out, out_mode=2, split=split, bias=bias, act=1, gain=1.0, clamp=256.0,
                     up_prev=prev, up_filter=f, round16=not split, out_nchw=nchw)
    # composition of the separate kernels
    up = tcconv.upsample2x_nhwc(prev, f)
    if split:
        ref = up.clone()
        tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_1X1, (h, w), ref, out_mode=3, split=True, bias=bias, act=1, gain=1.0, clamp=256.0)
    else:
        y16 = torch.empty(b, h, w, cout, device='cuda', dtype=torch.float16)
        tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_1X1, (h, w), y16, out_mode=0, bias=bias, act=1, gain=1.0, clamp=256.0)
        ref = up + y16
    got = out.permute(0, 2, 3, 1) if nchw else out
    assert rel_err(got.cpu().numpy(), ref.cpu().numpy()) < 1e-6
    # and against the plain torch formulation
    y = F.conv2d(x if split else x.half().float(), wt if split else (wt * tcconv.WEIGHT_SCALE).half().float() / tcconv.WEIGHT_SCALE) + bias[None, :, None, None]
    y = y.clamp(-256, 256)
    if not split:
        y = y.half().float()
    tref = upfirdn2d.upsample2d(prev.permute(0, 3, 1, 2).contiguous(), f) + y
    assert rel_err(got.permute(0, 3, 1, 2).cpu().numpy(), tref.cpu().numpy()) < (3e-5 if split else 2e-3)


@pytest.mark.parametrize('split', [False, True])
def test_cta_pair_kernel_256_channel_tiles(split):
    """Layers with >= 256 output channels and >= 74 tile pairs run on CTA pairs (cta_group::2, one 256x256 tile per two
    SMs), here with weights shared by the batch, against float64 torch. tcconv.launch_flags is read on every call;
    test_gpu_kernel_instances.py runs per-sample-weight pair launches through the single-CTA kernels too and compares."""
    from pix2pix3d_b200 import tcconv
    torch.manual_seed(21)
    b, c, h, w, cout = 2, 128, 96, 80, 512           # 2 * ceil(96*80/256) * 2 = 120 tile pairs, odd tile edges
    x = torch.randn(b, c, h, w, device='cuda')
    wt = torch.randn(cout, c, 3, 3, device='cuda') / np.sqrt(9 * c)
    bias = torch.randn(cout, device='cuda')
    noise = torch.randn(h, w, device='cuda') * 0.3
    planes = 2 if split else 1
    xn = tcconv.to_nhwc_f16(x, planes=planes)
    wk = _weights_kmajor(wt, planes=planes, scale=tcconv.WEIGHT_SCALE)
    hi = torch.zeros(b, h, w, cout, device='cuda', dtype=torch.float16)
    lo = torch.zeros_like(hi)
    tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_3X3, (h, w), hi, out_lo=lo if split else None, out_mode=1 if split else 0, split=split,
                     bias=bias, noise=noise, act=3, alpha=0.2, gain=float(np.sqrt(2)), clamp=4.0)
    got = (hi.float() + lo.float()) if split else hi.float()
    torch.backends.cudnn.allow_tf32 = False
    xr = x.double() if split else _h(x)
    wr = wt.double() if split else (_h(wt * tcconv.WEIGHT_SCALE) / tcconv.WEIGHT_SCALE)
    ref = F.conv2d(xr.cpu(), wr.cpu(), padding=1) + noise.double().cpu() + bias.double().cpu()[None, :, None, None]
    ref = (F.leaky_relu(ref, 0.2) * np.sqrt(2)).clamp(-4, 4)
    assert rel_err(got.permute(0, 3, 1, 2).cpu().numpy(), ref.numpy()) < (2e-5 if split else 1e-3)


def test_strided_conv_and_residual_epilogue():
    """down=2 layers: out(y, x) = sum_d w[d] * in(2y + dy, 2x + dx) through TMA element strides, plus the resnet skip tensor
    added after the activation; small (split-K-sized) and large (persistent / pair kernel) shapes."""
    from pix2pix3d_b200 import tcconv
    torch.manual_seed(14)
    for b, c, hw, cout in ((2, 64, 17, 64), (2, 128, 129, 128), (1, 64, 257, 256)):
        x = torch.randn(b, c, hw, hw, device='cuda')
        wt = torch.randn(cout, c, 3, 3, device='cuda') / np.sqrt(9 * c)
        bias = torch.randn(cout, device='cuda')
        ho = (hw - 3) // 2 + 1
        res = torch.randn(b, ho, ho, cout, device='cuda')
        xn = tcconv.to_nhwc_f16(x, planes=2)
        wk = _weights_kmajor(wt, planes=2, scale=tcconv.WEIGHT_SCALE)
        hi = torch.zeros(b, ho, ho, cout, device='cuda', dtype=torch.float16)
        lo = torch.zeros_like(hi)
        taps = [(ky, kx, ky * 3 + kx) for ky in range(3) for kx in range(3)]
        tcconv.conv_gemm(xn, wk, cout, taps, (ho, ho), hi, out_lo=lo, out_mode=1, split=True, bias=bias, act=3, alpha=0.2,
                         gain=1.0, stride=2, residual=res)
        ref = F.leaky_relu(F.conv2d(x.double().cpu(), wt.double().cpu(), stride=2) + bias.double().cpu()[None, :, None, None], 0.2)
        ref = ref + res.double().cpu().permute(0, 3, 1, 2)
        got = (hi.float() + lo.float()).permute(0, 3, 1, 2)
        assert rel_err(got.cpu().numpy(), ref.numpy()) < 2e-5, (b, c, hw, cout)
        # 1x1 tap at the odd positions (the skip branch)
        w1 = torch.randn(cout, c, 1, 1, device='cuda') / np.sqrt(c)
        wk1 = _weights_kmajor(w1, planes=2, scale=tcconv.WEIGHT_SCALE)
        y = torch.empty(b, ho, ho, cout, device='cuda')
        tcconv.conv_gemm(xn, wk1, cout, [(1, 1, 0)], (ho, ho), y, out_mode=2, split=True, act=1, gain=0.5, stride=2)
        ref1 = F.conv2d(x.double().cpu()[:, :, 1::2, 1::2][:, :, :ho, :ho], w1.double().cpu()) * 0.5
        assert rel_err(y.permute(0, 3, 1, 2).cpu().numpy(), ref1.numpy()) < 2e-5
    # split (hi/lo) input FIR
    from pix2pix3d_b200.torch_utils.ops import upfirdn2d
    f = upfirdn2d.setup_filter([1, 3, 3, 1]).cuda()
    xs = torch.randn(2, 64, 33, 33, device='cuda')
    sp = tcconv.to_nhwc_f16(xs, planes=2)
    out = tcconv.fir_act_nhwc(sp, f, None, None, 2, (34, 34), pad0=(2, 2), fir_gain=1.0, act=1, act_gain=1.0)
    refd = upfirdn2d.upfirdn2d(xs, f, padding=[2, 2, 2, 2])
    assert rel_err((out[0].float() + out[1].float()).permute(0, 3, 1, 2).cpu().numpy(), refd.cpu().numpy()) < 2e-6


@pytest.mark.parametrize('b,c,cout,hw,split', [
    (2, 64, 48, (7, 5), False),          # grid kernel, no split-K (Cin 64: 4 k-steps in the heaviest phase)
    (4, 512, 512, (4, 4), True),         # grid kernel + split-K partials per phase + one finisher for all phases
    (4, 512, 512, (16, 16), True),       # the b32 up layer: grid kernel, split-K
    (2, 128, 128, (72, 64), False),      # persistent kernel (one tile schedule over the four phases)
    (1, 256, 256, (56, 72), True),       # CTA-pair kernel, three-pass split
])
def test_merged_transposed_conv_phases_equal_separate_launches(b, c, cout, hw, split, monkeypatch):
    """p3d_conv_gemm_phases: one launch over the four phases == four p3d_conv_gemm launches, bit for bit, and both match the
    float64 transposed convolution."""
    from pix2pix3d_b200 import tcconv
    torch.manual_seed(21)
    h, w = hw
    x = torch.randn(b, c, h, w, device='cuda')
    wt = torch.randn(cout, c, 3, 3, device='cuda') / np.sqrt(9 * c)
    planes = 2 if split else 1
    xn = tcconv.to_nhwc_f16(x, planes=planes)
    wk = _weights_kmajor(wt, planes=planes, scale=tcconv.WEIGHT_SCALE)
    dt = torch.float32 if split else torch.float16
    outs = []
    for merged in (True, False):
        monkeypatch.setattr(tcconv, 'MERGE_PHASES', merged)
        out = torch.full((b, 2 * h + 1, 2 * w + 1, cout), float('nan'), device='cuda', dtype=dt)
        tcconv.conv_transpose3x3_s2(xn, wk, cout, out, split=split)
        assert torch.isfinite(out).all(), 'every output pixel must be written by exactly one phase'
        outs.append(out)
    if split:
        # fp32 accumulators: the merged launch may pick another kernel shape (CTA pairs: M = 256 MMAs) or another split-K factor than
        # the separate launches do -> another summation grouping, equal to rounding
        assert torch.allclose(outs[0], outs[1], rtol=0, atol=1e-5 * float(outs[1].abs().max()))
    else:
        assert torch.equal(outs[0], outs[1])
    if split:
        ref = F.conv_transpose2d(x.double().cpu(), wt.double().cpu().transpose(0, 1), stride=2)
        tol = 2e-5
    else:
        ref = F.conv_transpose2d(_h(x).cpu(), (_h(wt * tcconv.WEIGHT_SCALE).cpu() / tcconv.WEIGHT_SCALE).transpose(0, 1), stride=2)
        tol = 2e-3
    assert rel_err(outs[0].float().permute(0, 3, 1, 2).cpu().numpy(), ref.numpy()) < tol


def test_conv_gemm_phases_rejects_mismatched_phases():
    import ctypes
    from pix2pix3d_b200 import tcconv, _lib
    x = tcconv.to_nhwc_f16(torch.randn(1, 64, 4, 4, device='cuda'))
    wk = _weights_kmajor(torch.randn(16, 64, 3, 3, device='cuda'))
    out = torch.zeros(1, 9, 9, 16, device='cuda', dtype=torch.float16)
    other = torch.zeros(1, 9, 9, 16, device='cuda', dtype=torch.float16)
    arr = (tcconv.ConvArgs * 2)()
    arr[0] = tcconv._conv_args(x, wk, 16, tcconv.tconv_phase_taps(0, 0), (5, 5), out, out_map=(2, 0, 2, 0))
    arr[1] = tcconv._conv_args(x, wk, 16, tcconv.tconv_phase_taps(0, 1), (5, 4), other, out_map=(2, 0, 2, 1))
    assert _lib.lib().p3d_conv_gemm_phases(arr, 2, _lib.stream_ptr()) == -2
    assert _lib.lib().p3d_conv_gemm_phases(arr, 5, _lib.stream_ptr()) == -2


@pytest.mark.parametrize('cout,ci,hw,b', [(128, 3, (256, 256), 2), (128, 6, (192, 256), 2), (64, 3, (256, 256), 3)])
def test_torgb_fused_into_the_producing_convolution(cout, ci, hw, b):
    """p3d_conv_args_t::rgb_*: the 3x3 convolution of the last super-resolution block also evaluates the block's ToRGB + skip
    (networks_stylegan2.py:452-458) on the outputs it holds -- against the two separate launches it replaces."""
    from pix2pix3d_b200 import tcconv
    from pix2pix3d_b200.torch_utils.ops import upfirdn2d
    torch.manual_seed(31)
    c = 128
    h, w = hw
    f = upfirdn2d.setup_filter([1, 3, 3, 1]).cuda()
    x = torch.randn(b, c, h, w, device='cuda')
    w3 = torch.randn(cout, c, 3, 3, device='cuda') / np.sqrt(9 * c)
    wrgb = torch.randn(ci, cout, 1, 1, device='cuda') / np.sqrt(cout)
    styles = torch.randn(b, cout, device='cuda') + 1
    bias3, brgb = torch.randn(cout, device='cuda') * 0.1, torch.randn(ci, device='cuda')
    prev = torch.randn(b, h // 2, w // 2, ci, device='cuda')
    xn = tcconv.to_nhwc_f16(x)
    wk = _weights_kmajor(w3, scale=tcconv.WEIGHT_SCALE)
    wk_rgb = tcconv.modulate_weights(wrgb, styles, demodulate=False, pre_scale=0.7)       # [1,B,16,cout]: per-sample ToRGB weights
    # separate launches: conv -> fp16 x, then the fused-tail ToRGB convolution on it
    y = torch.empty(1, b, h, w, cout, device='cuda', dtype=torch.float16)
    tcconv.conv_gemm(xn, wk, cout, tcconv.TAPS_3X3, (h, w), y[0], out_mode=0, bias=bias3, act=3, alpha=0.2, gain=float(np.sqrt(2)), clamp=256.0)
    ref = torch.empty(b, ci, h, w, device='cuda')
    tcconv.conv_gemm(y, wk_rgb, ci, tcconv.TAPS_1X1, (h, w), ref, out_mode=2, bias=brgb, act=1, gain=1.0, clamp=256.0, up_prev=prev,
                     up_filter=f, round16=True, out_nchw=True)
    for skip_x in (False, True):
        y2 = torch.full_like(y, float('nan'))
        out = torch.full((b, ci, h, w), float('nan'), device='cuda')
        ok = tcconv.conv_gemm_try(xn, wk, cout, tcconv.TAPS_3X3, (h, w), y2[0], out_mode=0, bias=bias3, act=3, alpha=0.2,
                                  gain=float(np.sqrt(2)), clamp=256.0,
                                  rgb=dict(w=wk_rgb[0], bias=brgb, prev=prev, filter=f, out=out, clamp=256.0, skip_x=skip_x))
        assert ok, 'this launch shape qualifies for the fused ToRGB'
        assert torch.isfinite(out).all()
        # same fp16 inputs and weights, fp32 dot products summed in another order, then one fp16 rounding: a rare 1-ulp flip
        assert rel_err(out.cpu().numpy(), ref.cpu().numpy()) < 2e-3
        assert (out - ref).abs().mean().item() < 1e-4 * ref.abs().mean().item()
        if skip_x:
            assert torch.isnan(y2).all(), 'rgb_skip_x: the convolution output itself must not be written'
        else:
            assert torch.equal(y2, y)


def test_torgb_fusion_is_refused_for_other_launch_shapes():
    from pix2pix3d_b200 import tcconv
    from pix2pix3d_b200.torch_utils.ops import upfirdn2d
    f = upfirdn2d.setup_filter([1, 3, 3, 1]).cuda()
    b, c, cout, ci, h = 1, 64, 64, 3, 16            # 1 tile: not the persistent kernel
    xn = tcconv.to_nhwc_f16(torch.randn(b, c, h, h, device='cuda'))
    wk = _weights_kmajor(torch.randn(cout, c, 3, 3, device='cuda'))
    wk_rgb = _weights_kmajor(torch.randn(ci, cout, 1, 1, device='cuda'))
    y = torch.empty(b, h, h, cout, device='cuda', dtype=torch.float16)
    out = torch.empty(b, ci, h, h, device='cuda')
    prev = torch.zeros(b, h // 2, h // 2, ci, device='cuda')
    ok = tcconv.conv_gemm_try(xn, wk, cout, tcconv.TAPS_3X3, (h, h), y, out_mode=0,
                              rgb=dict(w=wk_rgb[0].expand(b, -1, -1).contiguous(), prev=prev, filter=f, out=out))
    assert ok is False
