"""Inference engine for the StyleGAN2 synthesis / super-resolution blocks on the tensor-core path.

Executes `SynthesisBlock` / `SynthesisBlockNoUp` stacks (reference training/networks_stylegan2.py:419-463,
training/superresolution.py:244-289) with NHWC fp16 activations: per-sample modulated weights
(`p3d_modulate_weights`), tcgen05 implicit-GEMM convolutions (`p3d_conv_gemm`) with noise/bias/lrelu/clamp in the
epilogue, the four-phase stride-2 transposed convolution followed by one fused FIR+noise+bias+lrelu pass for up=2
layers, and ToRGB accumulated straight into the upsampled fp32 skip image.

fp32 blocks (the tri-plane backbone, or any block under force_fp32) run on hi/lo split fp16 tensors with three
tensor-core passes (fp32-level accuracy); fp16 blocks run single pass, rounding where the reference rounds.
The module classes call into this when the inputs are CUDA tensors and no gradient is required (any noise mode: 'random'
draws one noise image per sample and layer with the reference's own `torch.randn` calls, in its order); every other case
keeps the generic op-by-op formulation.
"""
import logging
import os
import weakref

import numpy as np
import torch

from . import _lib, tcconv

_SQRT2 = float(np.sqrt(2))

# set False to force the generic op-by-op formulation (A/B checks in tests)
enabled = True


_log = logging.getLogger('pix2pix3d_b200.engine')
_told = set()


def _refuse(reason):
    """A CUDA call leaves the tensor-core path: say so ONCE per reason (the op-by-op formulation is an order of magnitude
    slower; a silent drop would look like a performance bug). Needing gradients is the normal training case and stays quiet."""
    if reason not in _told:
        _told.add(reason)
        _log.warning('tensor-core fast path not taken: %s -- running the op-by-op formulation (libp3d ops + ATen convolutions)', reason)
    return False


def block_supported(block, ws, noise_mode, need_grad):
    if not enabled or ws.device.type != 'cuda' or need_grad:
        return False
    if noise_mode not in ('const', 'none', 'random'):
        return _refuse(f'noise_mode={noise_mode!r}')
    if block.architecture != 'skip':
        return _refuse(f"block architecture {block.architecture!r} (only 'skip' is built)")
    for name in ('conv0', 'conv1'):
        layer = getattr(block, name, None)
        if layer is not None and (layer.activation != 'lrelu' or layer.weight.shape[-1] != 3):
            return _refuse(f'{name}: activation {layer.activation!r} / kernel {layer.weight.shape[-1]} (lrelu 3x3 is built)')
    if not hasattr(block, 'torgb'):
        return _refuse('block without a ToRGB layer')
    return True


def grad_needed(*modules_and_tensors):
    if not torch.is_grad_enabled():
        return False
    for m in modules_and_tensors:
        if isinstance(m, torch.nn.Module):
            if any(p.requires_grad for p in m.parameters()):
                return True
        elif isinstance(m, torch.Tensor) and m.requires_grad:
            return True
    return False


# Tensors derived from parameters only (gain-scaled affine weights, padded biases, const noise x strength, the NHWC image
# of the learned constant) are computed once per parameter version instead of once per step.
_derived = weakref.WeakKeyDictionary()


def _cached(module, key, params, fn):
    ver = tuple((p.data_ptr(), p._version, p.device) for p in params)
    slot = _derived.setdefault(module, {})
    hit = slot.get(key)
    if hit is not None and hit[0] == ver:
        return hit[1]
    val = fn()
    slot[key] = (ver, val)
    return val


def _pad_vec(v, n):
    v = v.detach().float()
    if v.numel() == n:
        return v.contiguous()
    out = torch.zeros(n, device=v.device, dtype=torch.float32)
    out[:v.numel()] = v
    return out


def _bias(layer, n):
    return _cached(layer, ('bias', n), [layer.bias], lambda: _pad_vec(layer.bias, n))


def _prepared(layer):
    return _cached(layer, 'wprep', [layer.weight], lambda: tcconv.prepare_weights(layer.weight))


def _noise(layer, noise_mode, batch=None):
    if noise_mode == 'const' and layer.use_noise:
        return _cached(layer, 'noise', [layer.noise_const, layer.noise_strength],
                       lambda: (layer.noise_const * layer.noise_strength).detach().float().contiguous())
    if noise_mode == 'random' and layer.use_noise:
        # one image per sample, drawn exactly where the reference draws it (networks_stylegan2.py:320-321): same generator call,
        # same layer order, so the RNG stream is consumed identically
        res = layer.resolution
        nz = torch.randn([batch, 1, res, res], device=layer.noise_strength.device) * layer.noise_strength.detach()
        return nz.float().reshape(batch, res, res).contiguous()
    return None


class StylePlan:
    """All `layer.affine(w)` of a list of layers as one `p3d_affine_batch` launch.

    layers: [(layer, ws_index)] in execution order; `run(ws)` returns the styles in that order, each [B, in_channels]
    (contiguous slices of one buffer)."""

    def __init__(self, layers):
        affs = [l.affine for l, _ in layers]
        dev = affs[0].weight.device
        self.key = tuple((a.weight.data_ptr(), a.weight._version, a.bias.data_ptr(), a.bias._version) for a in affs) + \
            tuple(i for _, i in layers)
        with torch.no_grad():
            self.weight = torch.cat([a.weight.detach().float() * a.weight_gain for a in affs]).contiguous()
            self.bias = torch.cat([a.bias.detach().float() * a.bias_gain for a in affs]).contiguous()
        self.sizes = [a.out_features for a in affs]
        self.index = [i for _, i in layers]
        self.device = dev
        self._meta = {}

    def meta(self, b):
        m = self._meta.get(b)
        if m is None:
            rows, off = [], 0
            for n, wi in zip(self.sizes, self.index):
                j = np.arange(n, dtype=np.int64)
                rows.append(np.stack([np.full(n, wi, np.int64), off + j, np.full(n, n, np.int64), np.zeros(n, np.int64)], 1))
                off += b * n
            m = (torch.from_numpy(np.concatenate(rows).astype(np.int32)).to(self.device), off)
            self._meta[b] = m
        return m

    def run(self, ws):
        b = ws.shape[0]
        meta, total = self.meta(b)
        flat = tcconv.affine_batch(ws, self.weight, self.bias, meta, total)
        out, off = [], 0
        for n in self.sizes:
            out.append(flat[off:off + b * n].view(b, n))
            off += b * n
        return out


class ReadyWeights:
    """Modulated weights of one layer produced ahead of the layer loop (WeightPlan.run)."""
    __slots__ = ('wk', 'batch')

    def __init__(self, wk, batch):
        self.wk, self.batch = wk, batch


def _block_layers(block):
    names = (['conv1'] if block.in_channels == 0 else ['conv0', 'conv1']) + ['torgb']
    return [getattr(block, n) for n in names]


def _block_specs(block, force_fp32, first_cin_p=None, first_cin_off=0):
    """Per layer of `_block_layers(block)`: the arguments of its weight modulation (they depend on the modules only)."""
    split = not (block.use_fp16 and not force_fp32)
    planes = 2 if split else 1
    specs = []
    for k, layer in enumerate(_block_layers(block)):
        torgb = layer is block.torgb
        cin_p = tcconv.pad_to(layer.in_channels, 64)
        cin_off = 0
        if k == 0 and first_cin_p is not None and not torgb:
            cin_p, cin_off = first_cin_p, first_cin_off
        specs.append(dict(layer=layer, demodulate=not torgb, pre_scale=float(layer.weight_gain) if torgb else 1.0, planes=planes,
                          cin_padded=cin_p, cin_offset=cin_off))
    return specs


class WeightPlan(StylePlan):
    """StylePlan + every layer's weight modulation as one `p3d_modulate_weights_batch` launch: `run(ws)` returns the
    ReadyWeights of all layers (views into one fp16 buffer), i.e. two launches replace 2 x n_layers."""

    def __init__(self, layers, specs):
        super().__init__(layers)
        self.specs = specs
        self.key = self.key + tuple((sp['layer'].weight.data_ptr(), sp['layer'].weight._version, sp['planes'], sp['cin_padded'],
                                     sp['cin_offset']) for sp in specs)
        self.prepared = [_prepared(sp['layer']) for sp in specs]
        self._tables = {}

    def tables(self, b):
        t = self._tables.get(b)
        if t is None:
            descs = (_lib.ModwDesc * len(self.specs))()
            block_layer, out_off, styles_off, first = [], 0, 0, 0
            shapes = []
            for k, (sp, (wt, wsq), n_in) in enumerate(zip(self.specs, self.prepared, self.sizes)):
                layer = sp['layer']
                o, i, kh, kw = layer.weight.shape
                assert i == n_in
                op, ip = tcconv.pad_to(o, 16), sp['cin_padded']
                nchunk = ip // 8
                assert ip % 8 == 0 and nchunk <= 256 and 256 % nchunk == 0, 'unsupported channel padding for the batched kernel'
                d = descs[k]
                d.weight_t, d.wsq = wt.data_ptr(), wsq.data_ptr()
                d.styles_off, d.out_off = styles_off, out_off
                d.Cout, d.Cin, d.ktaps, d.Cout_padded, d.Cin_padded = o, i, kh * kw, op, ip
                d.cin_offset, d.demodulate, d.planes = sp['cin_offset'], 1 if sp['demodulate'] else 0, sp['planes']
                d.pre_scale, d.out_scale = sp['pre_scale'], tcconv.WEIGHT_SCALE
                d.first_block = first
                block_layer += [k] * op
                n_out = sp['planes'] * b * op * kh * kw * ip
                shapes.append((out_off, n_out, (sp['planes'], b, op, kh * kw * ip)))
                out_off += (n_out + 63) // 64 * 64            # keep every layer 128-byte aligned
                styles_off += b * i
                first += op
            raw = torch.frombuffer(bytearray(bytes(descs)), dtype=torch.uint8).to(self.device)
            bl = torch.tensor(block_layer, dtype=torch.int32, device=self.device)
            t = (raw, bl, first, out_off, shapes)
            self._tables[b] = t
        return t

    def run(self, ws):
        b = ws.shape[0]
        meta, total = self.meta(b)
        flat = tcconv.affine_batch(ws, self.weight, self.bias, meta, total)
        raw, bl, n_blocks, out_total, shapes = self.tables(b)
        out = torch.empty(out_total, device=self.device, dtype=torch.float16)
        tcconv.modulate_weights_batch(raw, bl, n_blocks, flat, out, b)
        return [ReadyWeights(out[off:off + n].view(shape), b) for off, n, shape in shapes]


def weight_plan(owner, tag, layers, specs):
    """Cached WeightPlan, stored against `owner`; rebuilt when any parameter it derives from changes."""
    slot = _derived.setdefault(owner, {})
    key = tuple((l.affine.weight.data_ptr(), l.affine.weight._version, l.affine.bias.data_ptr(), l.affine.bias._version)
                for l, _ in layers) + tuple(i for _, i in layers) + \
        tuple((sp['layer'].weight.data_ptr(), sp['layer'].weight._version, sp['planes'], sp['cin_padded'], sp['cin_offset'])
              for sp in specs)
    plan = slot.get(('weights', tag))
    if plan is None or plan.key != key:
        plan = WeightPlan(layers, specs)
        slot[('weights', tag)] = plan
    return plan


def style_plan(owner, tag, layers):
    """Cached StylePlan for `layers` ([(layer, ws_index)]), stored against `owner`."""
    slot = _derived.setdefault(owner, {})
    key = tuple((l.affine.weight.data_ptr(), l.affine.weight._version, l.affine.bias.data_ptr(), l.affine.bias._version)
                for l, _ in layers) + tuple(i for _, i in layers)
    plan = slot.get(('styles', tag))
    if plan is None or plan.key != key:
        plan = StylePlan(layers)
        slot[('styles', tag)] = plan
    return plan


def _alloc(planes, b, h, w, c, cp, device):
    shape = (planes, b, h, w, cp)
    return torch.zeros(shape, device=device, dtype=torch.float16) if cp != c else torch.empty(shape, device=device, dtype=torch.float16)


# A/B switch (same results to fp16 rounding): P3D_FUSE_RGB=0 keeps the last block's ToRGB a separate launch
FUSE_RGB = os.environ.get('P3D_FUSE_RGB') != '0'


def synthesis_layer(layer, x, styles, noise_mode, split, gain=1.0, cin_offset=0, rgb_tail=None):
    """SynthesisLayer.forward (networks_stylegan2.py:313-332) on NHWC tensors. x: [planes,B,h,w,Cp]; styles = layer.affine(w).

    rgb_tail = dict(torgb=ToRGBLayer, styles=ReadyWeights, prev=[B,h/2,w/2,Ci] fp32 skip image, filter=f): also evaluate the
    block's ToRGB + skip (:452-458) in this layer's epilogue and return (None, image [B,Ci,h,w]) -- the last super-resolution
    block, whose x nobody reads; returns None when the launch shape does not qualify (the caller then runs the two layers)."""
    planes = 2 if split else 1
    cin_p = x.shape[-1]
    cout = layer.out_channels
    cout_p = tcconv.pad_to(cout, 64)
    if isinstance(styles, ReadyWeights):
        wk, b = styles.wk, styles.batch
        assert wk.shape[0] == planes and wk.shape[-1] == layer.weight.shape[2] * layer.weight.shape[3] * cin_p
    else:
        b = styles.shape[0]
        wk = tcconv.modulate_weights(layer.weight, styles, demodulate=True, planes=planes, cin_padded=cin_p, cin_offset=cin_offset,
                                     prepared=_prepared(layer))
    noise = _noise(layer, noise_mode, b)
    bias = _bias(layer, cout_p)
    act_gain = layer.act_gain * gain
    clamp = float(layer.conv_clamp * gain) if layer.conv_clamp is not None else -1.0
    dev = x.device
    if layer.up == 1:
        h, w = x.shape[2], x.shape[3]
        if rgb_tail is not None:
            torgb, st = rgb_tail['torgb'], rgb_tail['styles']
            ci = torgb.out_channels
            if (split or cout_p != cout or not isinstance(st, ReadyWeights) or st.wk.shape[0] != 1 or st.wk.shape[-1] != cout
                    or ci > 8 or rgb_tail['prev'].shape[-1] != ci):
                return None
            y = torch.empty(1, b, h, w, cout, device=dev, dtype=torch.float16)       # never written (rgb_skip_x); the ABI wants a buffer
            image = torch.empty(b, ci, h, w, device=dev, dtype=torch.float32)
            rgb = dict(w=st.wk[0], bias=_bias(torgb, ci), prev=rgb_tail['prev'].contiguous(), filter=rgb_tail['filter'], out=image,
                       clamp=float(torgb.conv_clamp) if torgb.conv_clamp is not None else -1.0, skip_x=True)
            ok = tcconv.conv_gemm_try(x, wk, cout, tcconv.TAPS_3X3, (h, w), y[0], out_mode=0, split=False, bias=bias, noise=noise, act=3,
                                      alpha=0.2, gain=act_gain, clamp=clamp, rgb=rgb)
            return (None, image) if ok else None
        y = _alloc(planes, b, h, w, cout, cout_p, dev)
        tcconv.conv_gemm(x, wk, cout, tcconv.TAPS_3X3, (h, w), y[0], out_lo=(y[1] if split else None), out_mode=1 if split else 0,
                         split=split, bias=bias, noise=noise, act=3, alpha=0.2, gain=act_gain, clamp=clamp)
        return y
    assert layer.up == 2
    h, w = x.shape[2], x.shape[3]
    tmp_dtype = torch.float32 if split else torch.float16
    if cout_p != cout:
        tmp = torch.zeros(b, 2 * h + 1, 2 * w + 1, cout_p, device=dev, dtype=tmp_dtype)
    else:
        tmp = torch.empty(b, 2 * h + 1, 2 * w + 1, cout_p, device=dev, dtype=tmp_dtype)
    tcconv.conv_transpose3x3_s2(x, wk, cout, tmp, split=split)
    return tcconv.fir_act_nhwc(tmp, layer.resample_filter, noise, bias, planes, (2 * h, 2 * w), pad0=(1, 1), fir_gain=4.0, act=3,
                               alpha=0.2, act_gain=act_gain, clamp=clamp)


def torgb_layer(layer, x, styles, img, split, upsample_filter=None, final_nchw=False):
    """ToRGBLayer.forward (:354-359) plus the skip connection of SynthesisBlock.forward (:452-458).

    img: fp32 NHWC skip image at THIS resolution (the convolution accumulates into it), or, with `upsample_filter`, the
    skip image of the previous block at half resolution: `upsample2d(img, f) + y` is then formed in the convolution's
    epilogue (one launch instead of upsample + conv + add [+ layout change]). `final_nchw` makes that launch write the
    [B,C,H,W] tensor the caller returns."""
    planes = 2 if split else 1
    cout = layer.out_channels
    if isinstance(styles, ReadyWeights):
        wk, b = styles.wk, styles.batch
        assert wk.shape[0] == planes and wk.shape[-1] == x.shape[-1]
    else:
        b = styles.shape[0]
        wk = tcconv.modulate_weights(layer.weight, styles, demodulate=False, pre_scale=layer.weight_gain, planes=planes,
                                     cin_padded=x.shape[-1], prepared=_prepared(layer))
    h, w = x.shape[2], x.shape[3]
    bias = _bias(layer, cout)
    clamp = float(layer.conv_clamp) if layer.conv_clamp is not None else -1.0
    if upsample_filter is not None and img is not None:
        assert img.shape[1] * 2 == h and img.shape[2] * 2 == w and img.shape[3] == cout
        shape = (b, cout, h, w) if final_nchw else (b, h, w, cout)
        out = torch.empty(shape, device=x.device, dtype=torch.float32)
        # fp16 blocks: the reference rounds the ToRGB output to fp16 before the fp32 skip add (:455-457)
        tcconv.conv_gemm(x, wk, cout, tcconv.TAPS_1X1, (h, w), out, out_mode=2, split=split, bias=bias, act=1, gain=1.0, clamp=clamp,
                         up_prev=img.contiguous(), up_filter=upsample_filter, round16=not split, out_nchw=final_nchw)
        return out
    assert not final_nchw
    if img is None:
        img = torch.empty(b, h, w, cout, device=x.device, dtype=torch.float32)
        mode = 2
    else:
        mode = 3
    if not split:
        y16 = torch.empty(b, h, w, cout, device=x.device, dtype=torch.float16)
        tcconv.conv_gemm(x, wk, cout, tcconv.TAPS_1X1, (h, w), y16, out_mode=0, bias=bias, act=1, gain=1.0, clamp=clamp)
        if mode == 2:
            img.copy_(y16)
        else:
            img.add_(y16)
        return img
    tcconv.conv_gemm(x, wk, cout, tcconv.TAPS_1X1, (h, w), img, out_mode=mode, split=True, bias=bias, act=1, gain=1.0, clamp=clamp)
    return img


def _const_input(block, b, planes):
    def make():
        c = block.const.shape[0]
        return tcconv.to_nhwc_f16(block.const.detach().float().unsqueeze(0).expand(b, -1, -1, -1).contiguous(),
                                  c_padded=tcconv.pad_to(c, 64), planes=planes)
    return _cached(block, ('const', b, planes), [block.const], make)


def synthesis_block(block, x, img, styles, noise_mode='const', force_fp32=False, upsample=True, cin_offset=0, final_nchw=False):
    """One block on NHWC tensors. x: [planes,B,h,w,Cp] fp16 or None (first block); img: [B,h,w,Ci] fp32 or None;
    styles: the affine outputs of this block's layers in execution order (conv0, conv1, torgb).
    Returns (x, img) in the same representation. The precision of x switches at block boundaries as
    `x.to(dtype)` does in the reference (:438)."""
    split = not (block.use_fp16 and not force_fp32)
    planes = 2 if split else 1
    s_iter = iter(styles)
    if block.in_channels == 0:
        x = _const_input(block, styles[0].batch if isinstance(styles[0], ReadyWeights) else styles[0].shape[0], planes)
        x = synthesis_layer(block.conv1, x, next(s_iter), noise_mode, split)
    else:
        if x.shape[0] != planes:   # precision change between blocks
            x = x[:1].contiguous() if planes == 1 else torch.stack([x[0], torch.zeros_like(x[0])])
        x = synthesis_layer(block.conv0, x, next(s_iter), noise_mode, split, cin_offset=cin_offset)
        st1 = next(s_iter)
        if final_nchw and FUSE_RGB and upsample and img is not None and not split:
            # last block: ToRGB + skip in conv1's epilogue (its output x is read by nothing else)
            st_rgb = next(s_iter)
            fused = synthesis_layer(block.conv1, x, st1, noise_mode, split,
                                    rgb_tail=dict(torgb=block.torgb, styles=st_rgb, prev=img, filter=block.resample_filter))
            if fused is not None:
                return fused
            x = synthesis_layer(block.conv1, x, st1, noise_mode, split)
            return x, torgb_layer(block.torgb, x, st_rgb, img, split, upsample_filter=block.resample_filter, final_nchw=True)
        x = synthesis_layer(block.conv1, x, st1, noise_mode, split)
    if upsample and img is not None:
        img = torgb_layer(block.torgb, x, next(s_iter), img, split, upsample_filter=block.resample_filter, final_nchw=final_nchw)
    else:
        assert not final_nchw
        img = torgb_layer(block.torgb, x, next(s_iter), img, split)
    return x, img


def _network_layers(net):
    """[(layer, ws_index)] of a SynthesisNetwork in execution order (ws slicing of :505-516)."""
    out, w_idx = [], 0
    for res in net.block_resolutions:
        block = getattr(net, f'b{res}')
        for k, layer in enumerate(_block_layers(block)):
            out.append((layer, w_idx + k))
        w_idx += block.num_conv
    return out


def _run_network(net, styles, noise_mode, force_fp32):
    x = img = None
    pos = 0
    for res in net.block_resolutions:
        block = getattr(net, f'b{res}')
        n = len(_block_layers(block))
        x, img = synthesis_block(block, x, img, styles[pos:pos + n], noise_mode=noise_mode, force_fp32=force_fp32)
        pos += n
    return img


def synthesis_network(net, ws, noise_mode='const', force_fp32=False):
    """SynthesisNetwork.forward (:505-520) -> fp32 NHWC image [B,R,R,img_channels]."""
    specs = [sp for res in net.block_resolutions for sp in _block_specs(getattr(net, f'b{res}'), force_fp32)]
    styles = weight_plan(net, ('net', bool(force_fp32)), _network_layers(net), specs).run(ws.to(torch.float32))
    return _run_network(net, styles, noise_mode, force_fp32)


def _sr_layers(sr, ws_index):
    """Both SR blocks read the same latent three times (superresolution.py:49: ws[:, -1:].repeat(1, 3, 1))."""
    return [(layer, ws_index) for block in (sr.block0, sr.block1) for layer in _block_layers(block)]


def superresolution(sr, rgb_nhwc, feat_nchw, ws, noise_mode='none', force_fp32=False, return_block0_image=False):
    """Superresolution*.forward (superresolution.py:48-57) with the feature image as NCHW fp32 and the low-res image as
    fp32 NHWC; returns the fp32 NHWC output image (and block0's output image on request: a NoUp block0 adds its ToRGB
    term into the caller's tensor in the reference, superresolution.py:283)."""
    ws = ws.to(torch.float32)
    first_p = tcconv.pad_to(feat_nchw.shape[1], 64)
    specs = _block_specs(sr.block0, force_fp32, first_p, 0) + _block_specs(sr.block1, force_fp32)
    styles = weight_plan(sr, ('sr', bool(force_fp32), first_p), _sr_layers(sr, ws.shape[1] - 1), specs).run(ws)
    split0 = not (sr.block0.use_fp16 and not force_fp32)
    x = tcconv.to_nhwc_f16(feat_nchw, c_padded=tcconv.pad_to(feat_nchw.shape[1], 64), planes=2 if split0 else 1)
    up0 = sr.block0.conv0.up == 2
    n0 = len(_block_layers(sr.block0))
    x, img0 = synthesis_block(sr.block0, x, rgb_nhwc, styles[:n0], noise_mode=noise_mode, force_fp32=force_fp32, upsample=up0)
    x, img = synthesis_block(sr.block1, x, img0, styles[n0:], noise_mode=noise_mode, force_fp32=force_fp32, upsample=True)
    return (img, img0) if return_block0_image else img


# ----------------------------------------------------------------------------------------------
# label-map Encoder of the conditional mapping networks (SURVEY 8(f) rank 2; triplane_cond.py:66-196): a resnet pyramid
# of DiscriminatorBlocks (networks_stylegan2.py:559-643) with static weights, fp32 semantics -> three-pass split GEMMs
# ----------------------------------------------------------------------------------------------
_TAPS_3X3_VALID = [(ky, kx, ky * 3 + kx) for ky in range(3) for kx in range(3)]     # strided conv on the pre-padded FIR output


def _static_weights(layer, cin_p):
    """K-major fp16 hi/lo image of an unmodulated Conv2dLayer weight x weight_gain (computed once per weight version)."""
    def make():
        ones = torch.ones(1, layer.weight.shape[1], device=layer.weight.device)
        return tcconv.modulate_weights(layer.weight, ones, demodulate=False, pre_scale=float(layer.weight_gain), planes=2,
                                       cin_padded=cin_p)
    return _cached(layer, ('wstatic', cin_p), [layer.weight], make)


def encoder_supported(enc, img):
    if not enabled or img.device.type != 'cuda' or grad_needed(enc, img):
        return False
    if enc.architecture != 'resnet' or img.shape[-1] != enc.img_resolution or img.shape[-2] != enc.img_resolution:
        return False
    for res in enc.block_resolutions:
        blk = getattr(enc, f'b{res}')
        if blk.use_fp16 or blk.architecture != 'resnet' or blk.conv0.activation != 'lrelu' or blk.conv1.activation != 'lrelu':
            return False
        if blk.conv0.conv_clamp is not None or blk.conv0.out_channels % 64 or blk.conv1.out_channels % 64:
            return False
    return True


def _encoder_block(blk, x, xin, b, res):
    c, cout = blk.conv0.out_channels, blk.conv1.out_channels
    dev = (x if x is not None else xin).device
    if blk.in_channels == 0:                                   # fromrgb: 1x1 + bias + lrelu (:518-522)
        lay = blk.fromrgb
        x = _alloc(2, b, res, res, c, c, dev)
        tcconv.conv_gemm(xin, _static_weights(lay, xin.shape[-1]), c, tcconv.TAPS_1X1, (res, res), x[0], out_lo=x[1], out_mode=1,
                         split=True, bias=_bias(lay, c), act=3, alpha=0.2, gain=float(lay.act_gain))
    f = blk.resample_filter
    h2 = res // 2
    # skip = 1x1 conv of the FIR-downsampled input (conv2d_resample.py:96-99 with pad (1,1), down 2): the full-resolution FIR
    # output with pad (2,2), sampled at the odd positions -- i.e. tap (1,1) of the same stride-2 grid conv1 uses
    fx = tcconv.fir_act_nhwc(x, f, None, None, 2, (res + 1, res + 1), pad0=(2, 2), fir_gain=1.0, act=1, act_gain=1.0)
    y = torch.empty(b, h2, h2, cout, device=dev, dtype=torch.float32)
    tcconv.conv_gemm(fx, _static_weights(blk.skip, c), cout, [(1, 1, 0)], (h2, h2), y, out_mode=2, split=True, act=1,
                     gain=float(np.sqrt(0.5)), stride=2)
    # conv0: 3x3 + bias + lrelu, kept in fp32 for the FIR that precedes the strided conv1
    t = torch.empty(b, res, res, c, device=dev, dtype=torch.float32)
    tcconv.conv_gemm(x, _static_weights(blk.conv0, c), c, tcconv.TAPS_3X3, (res, res), t, out_mode=2, split=True,
                     bias=_bias(blk.conv0, c), act=3, alpha=0.2, gain=float(blk.conv0.act_gain))
    ft = tcconv.fir_act_nhwc(t, f, None, None, 2, (res + 1, res + 1), pad0=(2, 2), fir_gain=1.0, act=1, act_gain=1.0)
    # conv1: FIR (above) then 3x3 stride 2 (:108-111), bias + lrelu with gain sqrt(2) * sqrt(0.5), plus the skip branch (:524-528)
    xn = _alloc(2, b, h2, h2, cout, cout, dev)
    tcconv.conv_gemm(ft, _static_weights(blk.conv1, c), cout, _TAPS_3X3_VALID, (h2, h2), xn[0], out_lo=xn[1], out_mode=1, split=True,
                     bias=_bias(blk.conv1, cout), act=3, alpha=0.2, gain=float(blk.conv1.act_gain * np.sqrt(0.5)), stride=2, residual=y)
    return xn


def encoder_forward(enc, img):
    """Encoder.forward (triplane_cond.py:168-196) on the tensor-core path -> the projector's [B, out_dim] output."""
    b = img.shape[0]
    xin = tcconv.to_nhwc_f16(img.float(), c_padded=tcconv.pad_to(img.shape[1], 64), planes=2)
    x = None
    for res in enc.block_resolutions:
        x = _encoder_block(getattr(enc, f'b{res}'), x, xin, b, res)
    # projector: a 4x4 "valid" convolution of the 4x4 map = one GEMM over (y, x, c); cuDNN picks an FFT algorithm for this
    # shape (3.7 ms), a plain fp32 matmul against the NHWC-ordered weight streams the 117 MB of weights once
    proj = enc.projector
    wp = _cached(proj, 'proj_nhwc', [proj.weight],
                 lambda: (proj.weight.detach().float().permute(0, 2, 3, 1).reshape(proj.weight.shape[0], -1) * proj.scale).contiguous())
    feat = (x[0].float() + x[1].float()).reshape(b, -1)                          # [B, 4*4*512] in (y, x, c) order
    return feat @ wp.t()


# ----------------------------------------------------------------------------------------------
# whole-generator fast path
# ----------------------------------------------------------------------------------------------
def _sr_supported(sr, ws, noise_mode, feat_res):
    return (hasattr(sr, 'block0') and hasattr(sr, 'block1') and feat_res == sr.input_resolution
            and block_supported(sr.block0, ws, noise_mode, False) and block_supported(sr.block1, ws, noise_mode, False))


def generator_supported(gen, ws, c, synthesis_kwargs, use_cached_backbone):
    """Can `TriPlane*Generator.synthesis` run end to end on the tensor-core / fused-render path?"""
    if ws.device.type != 'cuda' or grad_needed(gen, ws, c):
        return False
    if not enabled:
        return False
    extra = set(synthesis_kwargs) - {'noise_mode', 'force_fp32', 'fused_modconv'}
    if extra:
        return _refuse(f'synthesis kwargs {sorted(extra)} are not understood by the engine')
    noise_mode = synthesis_kwargs.get('noise_mode', 'random')
    net = gen.backbone.synthesis
    if net.img_channels != 96:
        return _refuse(f'backbone emits {net.img_channels} channels (3 x 32 tri-plane channels expected)')
    if not all(block_supported(getattr(net, f'b{r}'), ws, noise_mode, False) for r in net.block_resolutions):
        return False
    gen.renderer.plane_axes = gen.renderer.plane_axes.to(ws.device)
    if not gen.renderer.fusable_options(gen.decoder, gen.rendering_kwargs):
        return _refuse('rendering options / decoder type outside the fused renderer (density_noise, clamp_mode, custom plane '
                       'axes, > 64 samples per pass or an unknown decoder class)')
    sr_noise = gen.rendering_kwargs['superresolution_noise_mode']
    nrr = gen.neural_rendering_resolution
    srs = [gen.superresolution] + ([gen.superresolution_semantic] if hasattr(gen, 'superresolution_semantic') else [])
    for sr in srs:
        if not (hasattr(sr, 'block0') and hasattr(sr, 'block1')):
            return _refuse(f'super-resolution class {type(sr).__name__} is not a two-block stack')
        if nrr != sr.input_resolution:
            return _refuse(f'neural_rendering_resolution {nrr} != super-resolution input {sr.input_resolution}: the resize runs on '
                           'the generic path (renderer, ops and SR stacks still use their own kernels)')
        if not _sr_supported(sr, ws, sr_noise, nrr):
            return False
    return True


def generator_synthesis(gen, ws, c, cache_backbone=False, use_cached_backbone=False, noise_mode='random', force_fp32=False):
    """TriPlaneGenerator / TriPlaneSemanticEntangleGenerator.synthesis (triplane_cond.py:661-697, 1020-1061) without
    leaving the NHWC representation between the backbone, the fused renderer and the super-resolution stacks."""
    from . import native
    nrr = gen.neural_rendering_resolution
    b = ws.shape[0]
    cam2world = c[:, :16].view(-1, 4, 4)
    intrinsics = c[:, 16:25].view(-1, 3, 3)
    ray_origins, ray_directions = gen.ray_sampler(cam2world, intrinsics, nrr)
    # every style affine of the step (backbone + both SR stacks) in one launch
    net = gen.backbone.synthesis
    semantic = hasattr(gen, 'superresolution_semantic')
    srs = [gen.superresolution] + ([gen.superresolution_semantic] if semantic else [])
    net_layers = _network_layers(net)
    n_net = len(net_layers)
    all_layers = net_layers + [lw for sr in srs for lw in _sr_layers(sr, ws.shape[1] - 1)]
    nch_feat = 64 if semantic else 32                      # feature channels the renderer returns (two decoder nets / one)
    specs = [sp for res in net.block_resolutions for sp in _block_specs(getattr(net, f'b{res}'), force_fp32)]
    for k, sr in enumerate(srs):
        specs += _block_specs(sr.block0, force_fp32, tcconv.pad_to(nch_feat, 64), nch_feat // 2 if k == 1 else 0)
        specs += _block_specs(sr.block1, force_fp32)
    styles = weight_plan(gen, ('gen', bool(force_fp32)), all_layers, specs).run(ws.to(torch.float32))
    plane_index = None
    if use_cached_backbone and gen._last_planes is not None:
        # multi-view rendering from one latent (generate_video.py:57-69): the planes cached by an earlier call, kept in the
        # gather layout next to the NCHW tensor the reference API exposes as `_last_planes`
        planes_nchw = gen._last_planes
        pb = planes_nchw.shape[0]
        if pb != b:
            # V camera views against ONE cached plane set: the renderer reads plane set 0 for every image (plane_index), the
            # planes are neither copied nor re-generated. Same results as V single-view calls.
            assert pb == 1, 'cached planes must hold one plane set or one per camera'
            plane_index = torch.zeros(b, dtype=torch.int32, device=ws.device)
        cached = _derived.get(gen, {}).get('planes_cl')
        if cached is not None and cached[0] is planes_nchw and cached[1] == planes_nchw._version:
            planes_cl = cached[2]
        else:
            planes_cl = native.planes_to_channels_last(planes_nchw.view(pb, 3, 32, planes_nchw.shape[-2], planes_nchw.shape[-1]))
            _derived.setdefault(gen, {})['planes_cl'] = (planes_nchw, planes_nchw._version, planes_cl)
    else:
        img = _run_network(net, styles[:n_net], noise_mode, force_fp32)                                      # [B,H,W,96]
        h, w = img.shape[1], img.shape[2]
        planes_cl = img.view(b, h, w, 3, 32).permute(0, 3, 1, 2, 4)     # strided view, read in place by the renderer
        if cache_backbone:
            gen._last_planes = tcconv.nhwc_to_nchw_f32(img)
            _derived.setdefault(gen, {})['planes_cl'] = (gen._last_planes, gen._last_planes._version, planes_cl)
    feats, depth, wsum = gen.renderer(None, gen.decoder, ray_origins, ray_directions, gen.rendering_kwargs,
                                      planes_channels_last=planes_cl, plane_index=plane_index)
    nch = feats.shape[-1]
    fimg = feats.view(b, nrr, nrr, nch)                     # [B,R,C] is already NHWC
    depth_image = depth.permute(0, 2, 1).reshape(b, 1, nrr, nrr)
    sr_noise = gen.rendering_kwargs['superresolution_noise_mode']
    half = nch // 2 if semantic else nch
    n_sr = len(_sr_layers(gen.superresolution, 0))

    def run_sr(sr, c_off, n_img, st):
        split0 = not (sr.block0.use_fp16 and not force_fp32)
        if split0:
            hi = fimg.half()
            x = torch.stack([hi, (fimg - hi.float()).half()])
        else:
            x = fimg.half().unsqueeze(0)
        if nch % 64:
            x = torch.nn.functional.pad(x, (0, tcconv.pad_to(nch, 64) - nch))
        x = x.contiguous()
        rgb = fimg[..., c_off:c_off + n_img].contiguous()
        up0 = sr.block0.conv0.up == 2
        n0 = len(_block_layers(sr.block0))
        # reference quirk kept: a NoUp block0 accumulates its ToRGB into the very tensor it was handed
        # (superresolution.py:283 `img.add_(y)` on the `feature_image[:, :3]` view), so the raw image returned by
        # synthesis includes that term whenever no resize happened; with an upsampling block0 it does not.
        raw = rgb if up0 else rgb.clone()
        x, im = synthesis_block(sr.block0, x, rgb, st[:n0], noise_mode=sr_noise, force_fp32=force_fp32, upsample=up0, cin_offset=c_off)
        if not up0:
            raw = im
        x, im = synthesis_block(sr.block1, x, im, st[n0:], noise_mode=sr_noise, force_fp32=force_fp32, upsample=True, final_nchw=True)
        return im, raw.permute(0, 3, 1, 2).contiguous()

    image, image_raw = run_sr(gen.superresolution, 0, 3, styles[n_net:n_net + n_sr])
    out = {'image': image, 'image_raw': image_raw, 'image_depth': depth_image}
    if semantic:
        cs = gen.semantic_channels
        out['semantic'], out['semantic_raw'] = run_sr(gen.superresolution_semantic, half, cs, styles[n_net + n_sr:])
    return out
