"""Host-side logic added around the kernels, checked without a GPU: filter factoring for the separable FIR entry, the tap tables of
the merged transposed-convolution phases, the broadcast bookkeeping of `fma`, the dispatch rules of the native training
convolutions and the decoder-op layout table."""
import ctypes

import numpy as np
import pytest
import torch


def test_separable_factors_are_exact_or_refused():
    from pix2pix3d_b200 import tcconv
    from pix2pix3d_b200.torch_utils.ops import upfirdn2d
    f = upfirdn2d.setup_filter([1, 3, 3, 1])
    fx, fy = tcconv.separable_factors(f)
    fx, fy = np.array(list(fx), np.float32), np.array(list(fy), np.float32)
    assert np.array_equal(np.outer(fy, fx).astype(np.float32), f.numpy())          # exact in fp32, as the kernel's contract requires
    assert tcconv.separable_factors(f) is tcconv.separable_factors(f)              # kept on the tensor object
    h = f.clone()
    assert tcconv.separable_factors(h) is not None
    h[1, 2] += 1e-3                                                                # in-place change bumps the version: re-examined
    assert tcconv.separable_factors(h) is None
    g = f.clone()
    g[1, 2] += 1e-3                                                                # not rank 1 any more
    assert tcconv.separable_factors(g) is None
    assert tcconv.separable_factors(torch.zeros(4, 4)) is None                     # f[0,0] == 0: no factoring
    assert tcconv.separable_factors(upfirdn2d.setup_filter([1, 2, 1])) is None     # only 4x4 filters take the separable entry
    f64 = upfirdn2d.setup_filter([1, 3, 3, 1]) * 4                                 # a gain folded into the buffer stays separable
    assert tcconv.separable_factors(f64) is not None


def test_transposed_conv_phase_taps_cover_the_3x3_kernel_once():
    """conv_transpose2d(stride 2, k 3): out[2j+py, 2i+px] += x[j - (ky-py)/2, i - (kx-px)/2] * w[ky, kx] for ky = py mod 2 ..."""
    from pix2pix3d_b200 import tcconv
    seen = []
    for py in (0, 1):
        for px in (0, 1):
            taps = tcconv.tconv_phase_taps(py, px)
            assert len(taps) == (2 if py == 0 else 1) * (2 if px == 0 else 1)
            for dy, dx, kb in taps:
                ky, kx = divmod(kb, 3)
                assert (ky - py) % 2 == 0 and (kx - px) % 2 == 0
                assert dy == -(ky - py) // 2 and dx == -(kx - px) // 2
                seen.append(kb)
    assert sorted(seen) == list(range(9))
    # a numpy transposed convolution assembled from the phase taps equals the scatter definition
    rng = np.random.default_rng(0)
    x, w = rng.standard_normal((5, 4)), rng.standard_normal((3, 3))
    ref = np.zeros((11, 9))
    for j in range(5):
        for i in range(4):
            ref[2 * j:2 * j + 3, 2 * i:2 * i + 3] += x[j, i] * w
    out = np.zeros_like(ref)
    xp = np.pad(x, 1)
    for py in (0, 1):
        for px in (0, 1):
            gh, gw = (6 if py == 0 else 5), (5 if px == 0 else 4)
            for dy, dx, kb in tcconv.tconv_phase_taps(py, px):
                for j in range(gh):
                    for i in range(gw):
                        out[2 * j + py, 2 * i + px] += xp[j + dy + 1, i + dx + 1] * w[kb // 3, kb % 3]
    assert np.allclose(out, ref)


def test_fma_cpu_path_and_unbroadcast():
    from pix2pix3d_b200.torch_utils.ops import fma
    torch.manual_seed(0)
    a = torch.randn(2, 3, 4, 5, dtype=torch.float64, requires_grad=True)
    b = torch.randn(2, 3, 1, 1, dtype=torch.float64, requires_grad=True)
    c = torch.randn(4, 5, dtype=torch.float64, requires_grad=True)
    y = fma.fma(a, b, c)
    assert torch.equal(y, torch.addcmul(c, a, b))
    assert torch.autograd.gradcheck(fma.fma, (a, b, c))
    assert torch.autograd.gradgradcheck(fma.fma, (a, b, c))
    assert tuple(fma._sum_to_shape(torch.ones(2, 3, 4, 5), (4, 5)).shape) == (4, 5)
    assert tuple(fma._sum_to_shape(torch.ones(2, 3, 4, 5), (2, 3, 1, 1)).shape) == (2, 3, 1, 1)


def test_native_conv_dispatch_rules_are_off_on_cpu_and_outside_first_order():
    from pix2pix3d_b200.torch_utils.ops import native_conv
    x = torch.randn(1, 64, 16, 16, requires_grad=True)
    w = torch.randn(64, 64, 3, 3)
    wt = torch.randn(64, 32, 3, 3)
    with native_conv.first_order():
        assert not native_conv.applies(x, w, None, (1, 1), (1, 1), (1, 1), 1)                      # CPU tensor
        assert not native_conv.applies_transposed(x, wt, None, (2, 2), (0, 0), (0, 0), (1, 1), 1)
    assert native_conv._depth == 0


def test_decoder_layout_table():
    from pix2pix3d_b200 import native
    from pix2pix3d_b200.training import triplane, triplane_cond as tc
    base = {'decoder_lr_mul': 1.0, 'decoder_output_dim': 32}
    full = 0xFFFFFFFF
    nets, sigma, masks = native.describe_decoder(triplane.OSGDecoder(32, dict(base)))
    assert (len(nets), sigma, masks[0]) == (1, 0, full)
    nets, sigma, masks = native.describe_decoder(tc.OSGDecoder_semantic_entangle(32, dict(base, sigmoid=False, semantic_channels=6)))
    assert (len(nets), sigma) == (1, 0) and masks[0] == full & ~(0x3F << 3)                        # outputs 3..8 stay raw logits
    nets, sigma, masks = native.describe_decoder(tc.OSGDecoder_semantic_lateSeparate(32, dict(base, sigmoid=False, semantic_channels=6)))
    assert (len(nets), sigma, masks) == (2, 1, [full, 0])
    assert native.describe_decoder(triplane.OSGDecoder(64, dict(base))) is None                    # 64 input features: not a fused layout
    feats = torch.randn(1, 3, 7, 32)
    assert not native.decoder_mlp_supported(triplane.OSGDecoder(32, dict(base)), feats)            # CPU tensors take the module's formula
