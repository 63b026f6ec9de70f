"""Every template instance of the convolution kernels (csrc/conv_gemm.cu) and of the FIR tail (csrc/synth_aux.cu) against
float64 references, with the instance that ran read back from the CUDA profiler.

The host code picks an instance at run time (launch shape from the grid size against the SM count, Cout_padded, the k-steps
and p3d_conv_args_t::launch_flags; activation form, clamp, noise and output planes from the arguments). Each case below
declares the instance it must reach, so a drift in those rules fails here by name instead of moving a case silently onto
another kernel. test_case_tables_cover_every_instance (no GPU) checks that the tables reach every instance there is.

Shapes are chosen for the 148 SMs of a B200. The float64 accumulator of each convolution shape is built once and reused by
every epilogue variant of that shape."""
import itertools
import re

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from conftest import rel_err

SQRT2 = float(np.sqrt(2))

# ------------------------------------------------------------------------------------------------------------------------
# Instances, written out as the product of the template parameters
# ------------------------------------------------------------------------------------------------------------------------
# conv: ('grid', kStages, kAct, kClamp), ('persist', kAct, kClamp), ('pair', kAct, kClamp); kAct 0 = linear,
# 1 = lrelu with 0 <= alpha <= 1 (max form), 2 = lrelu with any other alpha (select form).
# ('finish', act form): conv_splitk_finish_kernel, which takes the act form as a run-time argument.
# FIR: ('sep', TIn, kSplitOut, kNoise, kFast) and ('fir16', 'float' | 'half' | 'split') for the three fir_act_nhwc_kernel.
CONV_INSTANCES = ([('grid', st, a, c) for st in (3, 6) for a in (0, 1, 2) for c in (False, True)] +
                  [(kind, a, c) for kind in ('persist', 'pair') for a in (0, 1, 2) for c in (False, True)])
FINISH_INSTANCES = [('finish', a) for a in (0, 1, 2)]
FIR_INSTANCES = ([('sep', t, so, nz, fa) for t in ('float', 'half') for so, nz, fa in itertools.product((False, True), repeat=3)] +
                 [('fir16', t) for t in ('float', 'half', 'split')])


def _b(v):
    return '(?:true|1)' if v else '(?:false|0)'


def _instance_regex(inst):
    """Regex for the demangled kernel name of one instance, e.g. `void p3d::conv_gemm_persist_kernel<0, false>(...)`."""
    s = r'\s*,\s*'
    kind = inst[0]
    if kind == 'grid':
        return rf'(?<!\w)conv_gemm_kernel<\s*{inst[1]}{s}{inst[2]}{s}{_b(inst[3])}\s*>'
    if kind in ('persist', 'pair'):
        return rf'(?<!\w)conv_gemm_{kind}_kernel<\s*{inst[1]}{s}{_b(inst[2])}\s*>'
    if kind == 'finish':
        return r'(?<!\w)conv_splitk_finish_kernel\b'
    if kind == 'sep':
        t = 'float' if inst[1] == 'float' else '__half'
        return rf'(?<!\w)fir_act_nhwc_sep_kernel<\s*{t}{s}{_b(inst[2])}{s}{_b(inst[3])}{s}{_b(inst[4])}\s*>'
    if kind == 'fir16':
        t, vec, split_in = {'float': ('float', 4, False), 'half': ('__half', 8, False), 'split': ('__half', 8, True)}[inst[1]]
        return rf'(?<!\w)fir_act_nhwc_kernel<\s*{t}{s}{vec}{s}{_b(split_in)}\s*>'
    raise ValueError(inst)


# any instance of the two kernel families (to find launches a case did not declare)
_FAMILY = re.compile(r'(?<!\w)(?:conv_gemm_(?:persist_|pair_)?kernel<|conv_splitk_finish_kernel\b|fir_act_nhwc_(?:sep_)?kernel<)')


def launched_kernels(fn):
    """(fn(), names of the CUDA kernels it launched), read from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, [e.name for e in prof.events()]


def assert_instances(names, expected):
    """Every expected instance ran, and no other instance of the convolution / FIR families did."""
    ours = [n for n in names if _FAMILY.search(n)]
    assert ours, f'the profiler recorded no convolution / FIR kernel; it saw: {sorted(set(names))}'
    for inst in expected:
        assert any(re.search(_instance_regex(inst), n) for n in ours), f'{inst} did not run; launched: {sorted(set(ours))}'
    for n in ours:
        assert any(re.search(_instance_regex(inst), n) for inst in expected), f'unexpected launch {n!r} (expected {expected})'


def act_form(act, alpha):
    return 0 if act == 1 else (1 if 0.0 <= alpha <= 1.0 else 2)


def fir_fast(act, alpha, clamp, planes):
    """The host's choice of the kFast instance (p3d_fir_act_nhwc_sep)."""
    exact = clamp < 0 or planes == 2 or float(torch.tensor(clamp).half()) == clamp
    return act == 3 and 0.0 <= alpha <= 1.0 and exact


# ------------------------------------------------------------------------------------------------------------------------
# Convolution matrix
# ------------------------------------------------------------------------------------------------------------------------
# name: (B, Cin, H, W, Cout, kind, Bw). kind '3x3' (padding 1), '1x1', 's2' (3x3, stride 2, no padding: the down=2 layers).
# Launch shapes on 148 SMs (tcconv.launch_flags = 0):
#   small1x1  6 CTAs x 2 k-steps                       -> grid kernel, 3 stages (too few k-steps for 6 or for split-K)
#   deep      6 CTAs x 36 k-steps                      -> grid kernel, 6 stages (split_k=False); split-K 9 or 16 ways + finisher
#   persist   192 256-pixel tiles, Cout 128            -> persistent kernel; launch_flags=1: 384 CTAs, 3 stages; B=1: 6 stages
#   ragged    180 tiles, Cout 264 (Cout_padded 272)    -> persistent kernel (the last channel tile holds 8 valid channels)
#   strided   192 tiles at 128^2 out, residual          -> persistent kernel
#   pair      120 pair tiles, Cout 512                  -> CTA pairs; launch_flags=2: persistent; 3: grid, 3 stages
CONV_SHAPES = {
    'small1x1': (2, 128, 12, 20, 40, '1x1', 1),
    'deep': (2, 256, 8, 8, 264, '3x3', 2),
    'persist': (3, 128, 128, 128, 128, '3x3', 3),
    'ragged': (3, 64, 80, 64, 264, '3x3', 1),
    'strided': (3, 64, 257, 257, 128, 's2', 1),
    'pair': (2, 128, 96, 80, 512, '3x3', 2),
}


def _conv(name, shape, expect, act=1, alpha=0.2, gain=1.0, clamp=-1.0, mode=2, split=False, split_k=True, flags=0, bias=False,
          noise=None, dscale=False, residual=False, wide=False, alts=()):
    """One case. expect: instances that must run. alts: (label, launch_flags, split_k, batch 1 only, 'equal' | 'fp32' | 'splitk')
    -- the same inputs through another launch shape, compared with this one (see test_conv_instance)."""
    return pytest.param(shape, expect, dict(act=act, alpha=alpha, gain=gain, clamp=clamp, mode=mode, split=split, split_k=split_k,
                                            flags=flags, bias=bias, noise=noise, dscale=dscale, residual=residual, wide=wide),
                        alts, id=name)


GRID3, PERSIST, FIRST6 = ('grid3', 1, True, False, 'equal'), ('persist', 2, True, False, 'fp32'), ('b1-6stage', 0, True, True, 'equal')
PAIR_AS_GRID = ('grid3', 3, True, False, 'fp32')
CONV_CASES = [
    # grid kernel, 3 stages
    _conv('small-lin-acc', 'small1x1', [('grid', 3, 0, False)], act=1, mode=3, bias=True, noise='shared'),
    _conv('small-lrelu-clamp-hilo-wide', 'small1x1', [('grid', 3, 1, True)], act=3, gain=SQRT2, clamp=1.5, mode=1, wide=True,
          noise='sample', dscale=True),
    _conv('small-select-postgain-f16', 'small1x1', [('grid', 3, 2, False)], act=3, alpha=-0.3, gain=-0.7, mode=0, bias=True),
    _conv('small-lin-clamp', 'small1x1', [('grid', 3, 0, True)], act=1, gain=0.6, clamp=0.5, dscale=True),
    _conv('small-lrelu-f16-wide', 'small1x1', [('grid', 3, 1, False)], act=3, gain=SQRT2, mode=0, wide=True, bias=True,
          noise='sample'),
    _conv('small-select-clamp-split', 'small1x1', [('grid', 3, 2, True)], split=True, act=3, alpha=1.7, clamp=1.0, noise='sample'),
    # grid kernel, 6 stages (Cout 264: a ragged last channel tile; per-sample weights)
    _conv('deep-lin-split', 'deep', [('grid', 6, 0, False)], split=True, split_k=False, bias=True, noise='sample',
          alts=[('split-k', 0, True, False, 'splitk')]),
    _conv('deep-lin-clamp-postgain-f16-wide', 'deep', [('grid', 6, 0, True)], split_k=False, gain=-1.3, clamp=1.0, mode=0, wide=True,
          dscale=True),
    _conv('deep-lrelu-hilo', 'deep', [('grid', 6, 1, False)], split_k=False, act=3, gain=SQRT2, mode=1, bias=True, noise='sample',
          alts=[('split-k', 0, True, False, 'splitk')]),
    _conv('deep-lrelu-clamp-acc-split', 'deep', [('grid', 6, 1, True)], split=True, split_k=False, act=3, gain=SQRT2, clamp=2.0,
          mode=3, noise='shared', dscale=True),
    _conv('deep-select-f16', 'deep', [('grid', 6, 2, False)], split_k=False, act=3, alpha=1.7, gain=0.8, mode=0, bias=True),
    _conv('deep-select-clamp-split', 'deep', [('grid', 6, 2, True)], split=True, split_k=False, act=3, alpha=-0.3, gain=1.2,
          clamp=1.0, noise='sample'),
    # split-K: grid kernel partials + conv_splitk_finish_kernel, one case per act form
    _conv('splitk-lin-split-hilo', 'deep', [('grid', 3, 0, False), ('finish', 0)], split=True, mode=1, bias=True, noise='sample',
          alts=[('no-split-k', 0, False, False, 'splitk')]),
    _conv('splitk-lrelu-clamp', 'deep', [('grid', 3, 1, True), ('finish', 1)], act=3, gain=SQRT2, clamp=1.5, bias=True,
          noise='sample', dscale=True, alts=[('no-split-k', 0, False, False, 'splitk')]),
    _conv('splitk-select-f16', 'deep', [('grid', 3, 2, False), ('finish', 2)], act=3, alpha=1.7, gain=0.9, mode=0, noise='shared',
          alts=[('no-split-k', 0, False, False, 'splitk')]),
    # persistent kernel (per-sample weights and noise; launch_flags=1 gives the grid kernel, batch 1 alone its 6-stage ring)
    _conv('persist-lin-f16', 'persist', [('persist', 0, False)], mode=0, bias=True, noise='sample', alts=[GRID3, FIRST6]),
    _conv('persist-lin-clamp-hilo-wide-split', 'persist', [('persist', 0, True)], split=True, gain=0.7, clamp=0.5, mode=1,
          wide=True, noise='shared'),
    _conv('persist-lrelu', 'persist', [('persist', 1, False)], act=3, gain=SQRT2, bias=True, noise='sample', dscale=True,
          alts=[GRID3, FIRST6]),
    _conv('persist-lrelu-clamp-acc-split', 'persist', [('persist', 1, True)], split=True, act=3, gain=SQRT2, clamp=1.0, mode=3,
          noise='sample'),
    _conv('persist-select-clamp', 'persist', [('persist', 2, True)], act=3, alpha=1.7, gain=1.1, clamp=2.0, bias=True,
          noise='sample', alts=[GRID3]),
    _conv('persist-select-postgain-f16', 'persist', [('persist', 2, False)], act=3, alpha=-0.3, gain=-1.2, mode=0, noise='shared',
          dscale=True, alts=[GRID3, FIRST6]),
    _conv('ragged-lrelu-clamp-hilo-wide', 'ragged', [('persist', 1, True)], act=3, gain=SQRT2, clamp=256.0, mode=1, wide=True,
          bias=True, noise='sample', alts=[('grid3', 1, True, False, 'equal')]),
    _conv('ragged-lin-split', 'ragged', [('persist', 0, False)], split=True),
    _conv('strided-residual-split-hilo', 'strided', [('persist', 1, False)], split=True, act=3, mode=1, bias=True, residual=True,
          alts=[('grid3', 1, True, False, 'fp32')]),
    _conv('strided-residual-select-clamp', 'strided', [('persist', 2, True)], act=3, alpha=1.7, gain=0.9, clamp=1.0,
          residual=True, noise='sample', alts=[GRID3]),
    # CTA pairs (launch_flags=2: the single-CTA persistent kernel, 3: the grid kernel; other M=256 summation -> 'close')
    _conv('pair-lin-f16-wide', 'pair', [('pair', 0, False)], mode=0, wide=True, bias=True, noise='sample', alts=[PERSIST, PAIR_AS_GRID]),
    _conv('pair-lin-clamp-split-hilo', 'pair', [('pair', 0, True)], split=True, gain=0.8, clamp=1.0, mode=1, noise='shared',
          alts=[PERSIST]),
    _conv('pair-lrelu', 'pair', [('pair', 1, False)], act=3, gain=SQRT2, noise='sample', dscale=True, alts=[PERSIST, PAIR_AS_GRID]),
    _conv('pair-lrelu-clamp-f16', 'pair', [('pair', 1, True)], act=3, gain=SQRT2, clamp=4.0, mode=0, bias=True, noise='shared'),
    _conv('pair-lrelu-clamp-split-hilo', 'pair', [('pair', 1, True)], split=True, act=3, gain=SQRT2, clamp=4.0, mode=1, bias=True,
          noise='shared'),
    _conv('pair-select-acc', 'pair', [('pair', 2, False)], act=3, alpha=1.7, mode=3, noise='sample', alts=[PERSIST]),
    _conv('pair-select-clamp-postgain-split', 'pair', [('pair', 2, True)], split=True, act=3, alpha=-0.3, gain=-0.9, clamp=1.5,
          bias=True, dscale=True, alts=[PERSIST]),
]

# p3d_conv_gemm_phases (stride-2 transposed 3x3, four phases in one launch): (B, Cin, h, w, Cout, split, [(flags, instances)])
PHASE_CASES = [
    pytest.param(2, 64, 7, 5, 48, False, [(0, [('grid', 3, 0, False)])], id='grid'),
    pytest.param(2, 128, 72, 64, 128, False, [(0, [('persist', 0, False)]), (1, [('grid', 3, 0, False)])], id='persist'),
    pytest.param(1, 256, 56, 72, 256, True, [(0, [('pair', 0, False)]), (2, [('persist', 0, False)]), (3, [('grid', 3, 0, False)])],
                 id='pair-split'),
    pytest.param(4, 512, 4, 4, 512, True, [(0, [('grid', 3, 0, False), ('finish', 0)])], id='splitk-split'),
]

_PROBLEMS = {}


def _h(x):   # value after fp16 rounding, as float64
    return x.half().double()


def _problem(name):
    """Seeded operands of one convolution shape and their float64 accumulators, built once: 'acc16' from the fp16 operands the
    single-pass kernels read (x rounded to fp16, w * 128 rounded to fp16, / 128), 'acc32' from the unrounded fp32 operands
    that the 3-pass split reproduces."""
    if name in _PROBLEMS:
        return _PROBLEMS[name]
    from pix2pix3d_b200 import tcconv
    b, cin, h, w, cout, kind, bw = CONV_SHAPES[name]
    torch.manual_seed(sorted(CONV_SHAPES).index(name) + 100)
    ks = 1 if kind == '1x1' else 3
    kk = ks * ks
    x = torch.randn(b, cin, h, w, device='cuda')
    wt = torch.randn(cout, cin, ks, ks, device='cuda') / np.sqrt(kk * cin)
    if bw > 1:      # per-sample modulated weights, distinct styles
        styles = torch.rand(bw, cin, device='cuda') + 0.5
        wk = tcconv.modulate_weights(wt, styles, demodulate=True, planes=2)
        w64 = wt.double()[None] * styles.double()[:, None, :, None, None]
        w64 = w64 * (w64.square().sum(dim=[2, 3, 4], keepdim=True) + 1e-8).rsqrt()
    else:
        wk = tcconv.modulate_weights(wt, torch.ones(1, cin, device='cuda'), demodulate=False, planes=2)
        w64 = wt.double()[None]
    xn = tcconv.to_nhwc_f16(x, planes=2)
    if kind == 's2':
        taps, pad, stride = [(ky, kx, ky * 3 + kx) for ky in range(3) for kx in range(3)], 0, 2
    else:
        taps, pad, stride = (tcconv.TAPS_3X3 if ks == 3 else tcconv.TAPS_1X1), ks // 2, 1
    oh, ow = (h + 2 * pad - ks) // stride + 1, (w + 2 * pad - ks) // stride + 1
    op = wk.shape[2]
    w16 = wk[0].double().reshape(bw, op, kk, cin)[:, :cout].permute(0, 1, 3, 2) / tcconv.WEIGHT_SCALE     # [Bw,Cout,Cin,kk]

    def acc(xs, ws):      # float64 implicit GEMM on the GPU: unfold + matmul -> [B,oH,oW,Cout]
        cols = F.unfold(xs, ks, padding=pad, stride=stride)                                      # [B, Cin*kk, L]
        return torch.matmul(ws.reshape(bw, cout, cin * kk), cols).reshape(b, cout, oh, ow).permute(0, 2, 3, 1).contiguous()

    P = dict(b=b, cout=cout, oh=oh, ow=ow, taps=taps, stride=stride, xn=xn, wk=wk,
             acc16=acc(xn[0].double().permute(0, 3, 1, 2), w16), acc32=acc(x.double(), w64.reshape(bw, cout, cin, kk)),
             bias=torch.randn(cout, device='cuda') * 0.5,
             noise_shared=torch.randn(oh, ow, device='cuda') * 0.5,
             noise_sample=torch.randn(b, oh, ow, device='cuda') * 0.5,       # distinct image per sample
             dscale=torch.rand(b, cout, device='cuda') + 0.5,
             residual=torch.randn(b, oh, ow, cout, device='cuda'),
             acc_init=torch.randn(b, oh, ow, cout, device='cuda'))
    _PROBLEMS[name] = P
    return P


def _epilogue64(P, c, acc):
    """The kernel's epilogue in float64, in its order: act(acc * dscale + noise + bias) * gain, clamp, + residual. Also returns
    the scale the error bounds refer to: the largest magnitude before the clamp (the accumulation error follows the size of
    the sums, not of the clamped result)."""
    v = acc
    if c['dscale']:
        v = v * P['dscale'].double()[:, None, None, :]
    if c['noise'] == 'shared':
        v = v + P['noise_shared'].double()[None, :, :, None]
    elif c['noise'] == 'sample':
        v = v + P['noise_sample'].double()[..., None]
    if c['bias']:
        v = v + P['bias'].double()
    if c['act'] == 3:
        v = torch.where(v > 0, v, v * c['alpha'])
    v = v * c['gain']
    scale = float(v.abs().max())
    if c['clamp'] >= 0:
        v = v.clamp(-c['clamp'], c['clamp'])
    if c['residual']:
        v = v + P['residual'].double()
    return v, max(scale, float(v.abs().max()))


def _run_conv(P, c, flags, split_k, first_only, monkeypatch):
    """One p3d_conv_gemm launch of case c -> (channels the launch owns as float64 [B,oH,oW,Cout], hi plane or None, untouched
    channels of the output tensor)."""
    from pix2pix3d_b200 import tcconv
    monkeypatch.setattr(tcconv, 'launch_flags', flags)
    nb = 1 if first_only else P['b']
    planes = 2 if c['split'] else 1
    xn = P['xn'][:planes, :nb].contiguous()
    wk = P['wk'][:planes, :min(nb, P['wk'].shape[1])].contiguous()
    cout, oh, ow = P['cout'], P['oh'], P['ow']
    coff, cs = (8, cout + 24) if c['wide'] else (0, cout)
    mode = c['mode']
    if mode == 3:
        out = P['acc_init'][:nb].clone()
    else:
        out = torch.full((nb, oh, ow, cs), 7.0, device='cuda', dtype=torch.float16 if mode <= 1 else torch.float32)
    lo = torch.full_like(out, 7.0) if mode == 1 else None
    kw = dict(act=c['act'], alpha=c['alpha'], gain=c['gain'], clamp=c['clamp'], out_mode=mode, out_lo=lo, y_coff=coff,
              split=c['split'], split_k=split_k, stride=P['stride'])
    if c['bias']:
        kw['bias'] = P['bias']
    if c['noise']:
        kw['noise'] = P['noise_shared'] if c['noise'] == 'shared' else P['noise_sample'][:nb].contiguous()
    if c['dscale']:
        kw['dscale'] = P['dscale'][:nb].contiguous()
    if c['residual']:
        kw['residual'] = P['residual'][:nb].contiguous()
    tcconv.conv_gemm(xn, wk, cout, P['taps'], (oh, ow), out, **kw)
    own = out[..., coff:coff + cout]
    rest = torch.cat([out[..., :coff], out[..., coff + cout:]], dim=-1)
    if mode == 1:
        rest = torch.cat([rest, lo[..., :coff], lo[..., coff + cout:]], dim=-1)
        return own.double() + lo[..., coff:coff + cout].double(), own, rest
    if mode == 3:
        return own.double() - P['acc_init'][:nb].double(), None, rest
    return own.double(), (own if mode == 0 else None), rest


def _ulp16(r16):
    """Spacing of fp16 numbers at r16 (float64 holding fp16 values)."""
    return torch.exp2(torch.floor(torch.log2(r16.abs().clamp_min(2.0 ** -14))) - 10)


def _ulp_diff16(got16, ref, slack=0.0):
    """(|got - fp16(ref)| - slack) in units of the fp16 spacing at fp16(ref), elementwise. slack: the absolute error the fp32
    value before the rounding may carry (near zero it is larger than an fp16 ulp)."""
    r16 = ref.half().double()
    return ((got16.double() - r16).abs() - slack) / _ulp16(r16)


@pytest.mark.gpu
@pytest.mark.parametrize('shape,expect,c,alts', CONV_CASES)
def test_conv_instance(shape, expect, c, alts, monkeypatch):
    P = _problem(shape)
    (got, hi, rest), names = launched_kernels(lambda: _run_conv(P, c, c['flags'], c['split_k'], False, monkeypatch))
    assert_instances(names, expect)
    assert bool((rest == 7.0).all()), 'channels outside [y_coff, y_coff + Cout) must not be written'
    ref, scale = _epilogue64(P, c, P['acc32'] if c['split'] else P['acc16'])
    # fp32-level bounds relative to `scale`; the 3-pass split against the unrounded fp32 operands
    tol = 2e-5 if c['split'] else (3e-6 if c['mode'] == 1 else 2e-6)
    if c['mode'] != 0:
        err = float((got - ref).abs().max()) / scale
        assert err < tol
    if hi is not None:
        # the fp16 plane: within one fp16 ulp of the rounded float64 result, elementwise, once the fp32 error is allowed for
        d = float(_ulp_diff16(hi, ref, tol * scale).max())
        assert d <= 1.0, f'{d} ulp beyond the fp32 error'
    # the same inputs through other launch shapes
    for label, flags, split_k, first_only, how in alts:
        other, _, _ = _run_conv(P, c, flags, split_k, first_only, monkeypatch)
        mine = got[:other.shape[0]]
        if how == 'equal':
            # grid and persistent kernels, 3- and 6-stage rings: the same M=128 MMAs in the same k order, the same epilogue
            assert torch.equal(other, mine), label
            continue
        # CTA pairs (M=256 MMAs) group the k-sum differently: equal to fp32 rounding, and an fp16 output rarely rounds to the
        # neighbouring number. Split-K against one CTA per tile: the single CTA accumulates every k-step in the tensor core's
        # truncating fp32 adder, split-K adds its partials with round-to-nearest. Each is within 2e-5 of float64 over K = 6912
        # (3-pass), so they may be 4e-5 apart (as in test_split_k_small_grids_match_single_pass_order), and at that distance
        # fp16 outputs round differently in ~1 % of the elements (measured 0.8 %).
        bound = (1e-5 if how == 'fp32' else 4e-5) * scale
        if c['mode'] == 0:
            assert bool(((other - mine).abs() <= _ulp16(mine) + bound).all()), label
            if how == 'fp32':
                assert float((other != mine).double().mean()) < 1e-3, label
        else:
            assert float((other - mine).abs().max()) <= bound, label


@pytest.mark.gpu
@pytest.mark.parametrize('b,cin,h,w,cout,split,launches', PHASE_CASES)
def test_conv_phases_instance(b, cin, h, w, cout, split, launches, monkeypatch):
    """p3d_conv_gemm_phases (merged transposed convolution) under each launch shape, against float64 conv_transpose2d."""
    from pix2pix3d_b200 import tcconv
    monkeypatch.setattr(tcconv, 'MERGE_PHASES', True)
    torch.manual_seed(41)
    x = torch.randn(b, cin, h, w, device='cuda')
    wt = torch.randn(cout, cin, 3, 3, device='cuda') / np.sqrt(9 * cin)
    planes = 2 if split else 1
    xn = tcconv.to_nhwc_f16(x, planes=planes)
    wk = tcconv.modulate_weights(wt, torch.ones(1, cin, device='cuda'), demodulate=False, planes=planes)
    if split:
        xr, wr = x.double(), wt.double()
    else:
        xr = xn[0].double().permute(0, 3, 1, 2)
        wr = wk[0].double().reshape(cout, 9, cin).permute(0, 2, 1).reshape(cout, cin, 3, 3) / tcconv.WEIGHT_SCALE
    ref = F.conv_transpose2d(xr, wr.transpose(0, 1), stride=2).permute(0, 2, 3, 1)
    outs = []
    for flags, expect in launches:
        monkeypatch.setattr(tcconv, 'launch_flags', flags)
        out = torch.full((b, 2 * h + 1, 2 * w + 1, cout), float('nan'), device='cuda',
                         dtype=torch.float32 if split else torch.float16)
        _, names = launched_kernels(lambda: tcconv.conv_transpose3x3_s2(xn, wk, cout, out, split=split))
        assert_instances(names, expect)
        assert torch.isfinite(out).all(), 'every output pixel must be written by exactly one phase'
        if split:
            assert rel_err(out.cpu().numpy(), ref.cpu().numpy()) < 2e-5
        else:
            assert float(_ulp_diff16(out, ref, 2e-6 * float(ref.abs().max())).max()) <= 1.0
        outs.append(out.double())
    for o in outs[1:]:
        if split:
            assert torch.allclose(o, outs[0], rtol=0, atol=1e-5 * float(outs[0].abs().max()))
        else:
            assert torch.equal(o, outs[0])      # grid and persistent kernels, single pass


@pytest.mark.gpu
def test_fused_torgb_with_per_sample_noise(monkeypatch):
    """The fused ToRGB tail (rgb=) on a convolution with noise_mode='random' noise ([B,oH,oW]) and per-sample weights: the
    convolution output equals the unfused launch bit for bit, and the image equals the two separate launches it replaces."""
    from pix2pix3d_b200 import tcconv
    from pix2pix3d_b200.torch_utils.ops import upfirdn2d
    monkeypatch.setattr(tcconv, 'launch_flags', 0)
    P = _problem('persist')
    b, cout, oh, ow = P['b'], P['cout'], P['oh'], P['ow']
    torch.manual_seed(43)
    f = upfirdn2d.setup_filter([1, 3, 3, 1]).cuda()
    ci = 3
    wk_rgb = tcconv.modulate_weights(torch.randn(ci, cout, 1, 1, device='cuda') / np.sqrt(cout),
                                     torch.randn(b, cout, device='cuda') + 1, demodulate=False)
    brgb = torch.randn(ci, device='cuda')
    prev = torch.randn(b, oh // 2, ow // 2, ci, device='cuda')
    xn, wk = P['xn'][:1].contiguous(), P['wk'][:1].contiguous()
    kw = dict(out_mode=0, bias=P['bias'], noise=P['noise_sample'], act=3, alpha=0.2, gain=SQRT2, clamp=256.0)
    y = torch.empty(1, b, oh, ow, cout, device='cuda', dtype=torch.float16)
    tcconv.conv_gemm(xn, wk, cout, P['taps'], (oh, ow), y[0], **kw)
    ref = torch.empty(b, ci, oh, ow, device='cuda')
    tcconv.conv_gemm(y, wk_rgb, ci, tcconv.TAPS_1X1, (oh, ow), ref, out_mode=2, bias=brgb, act=1, gain=1.0, clamp=256.0,
                     up_prev=prev, up_filter=f, round16=True, out_nchw=True)
    y2 = torch.full_like(y, float('nan'))
    out = torch.full((b, ci, oh, ow), float('nan'), device='cuda')
    ok, names = launched_kernels(lambda: tcconv.conv_gemm_try(
        xn, wk, cout, P['taps'], (oh, ow), y2[0], rgb=dict(w=wk_rgb[0], bias=brgb, prev=prev, filter=f, out=out, clamp=256.0), **kw))
    assert ok, 'this launch shape qualifies for the fused ToRGB'
    assert_instances(names, [('persist', 1, True)])
    assert torch.equal(y2, y)
    c = dict(dscale=False, noise='sample', bias=True, act=3, alpha=0.2, gain=SQRT2, clamp=256.0, residual=False)
    ref_y, scale = _epilogue64(P, c, P['acc16'])
    assert float(_ulp_diff16(y2[0], ref_y, 2e-6 * scale).max()) <= 1.0
    assert torch.isfinite(out).all()
    # same fp16 inputs and weights, fp32 dot products summed in another order, then one fp16 rounding: a rare 1-ulp flip
    assert rel_err(out.cpu().numpy(), ref.cpu().numpy()) < 2e-3
    assert (out - ref).abs().mean().item() < 1e-4 * ref.abs().mean().item()


# ------------------------------------------------------------------------------------------------------------------------
# FIR matrix (tcconv.fir_act_nhwc)
# ------------------------------------------------------------------------------------------------------------------------
def _fir(name, expect, dtype, c, b, planes, noise=None, act=3, alpha=0.2, clamp=-1.0, bias=True, pad=1, filt='sym', variant=3,
         out_hw=(18, 34), vs_sep=False):
    """dtype: 'f32' | 'f16' input, or 'split' (hi/lo fp16 pair). pad 1: the up layers' pad0 (1,1) with gain 4 on a 2h+1 input;
    pad 2: the encoder's pad0 (2,2) with gain 1 on an h input. filt: 'sym' = setup_filter([1,3,3,1]), 'asym' = rank 1 with
    fx != fy, 'full' = not rank 1. vs_sep: also run the separable kernel on the same input and compare."""
    return pytest.param(expect, dict(dtype=dtype, c=c, b=b, planes=planes, noise=noise, act=act, alpha=alpha, clamp=clamp,
                                     bias=bias, pad=pad, filt=filt, variant=variant, out_hw=out_hw, vs_sep=vs_sep), id=name)


FIR_CASES = [
    _fir('f32-fast', [('sep', 'float', False, False, True)], 'f32', 32, 2, 1),
    _fir('f32-linear-nobias-enc', [('sep', 'float', False, False, False)], 'f32', 96, 1, 1, act=1, bias=False, pad=2),
    _fir('f32-noise-clamp256-asym', [('sep', 'float', False, True, True)], 'f32', 32, 2, 1, noise='shared', clamp=256.0, filt='asym'),
    _fir('f32-bnoise-select-clamp03', [('sep', 'float', False, True, False)], 'f32', 96, 3, 1, noise='sample', alpha=1.7, clamp=0.3),
    _fir('f32-hilo-clamp03', [('sep', 'float', True, False, True)], 'f32', 32, 2, 2, clamp=0.3),
    _fir('f32-hilo-select-clamp7e4-nobias-enc', [('sep', 'float', True, False, False)], 'f32', 32, 2, 2, alpha=-0.3, clamp=7e4,
         bias=False, pad=2),
    _fir('f32-hilo-bnoise-asym-enc', [('sep', 'float', True, True, True)], 'f32', 96, 3, 2, noise='sample', pad=2, filt='asym'),
    _fir('f32-hilo-noise-linear', [('sep', 'float', True, True, False)], 'f32', 32, 2, 2, noise='shared', act=1, clamp=256.0),
    _fir('f16-fast-clamp256', [('sep', 'half', False, False, True)], 'f16', 64, 2, 1, clamp=256.0),
    _fir('f16-clamp03', [('sep', 'half', False, False, False)], 'f16', 192, 1, 1, clamp=0.3),
    _fir('f16-bnoise-asym-130', [('sep', 'half', False, True, True)], 'f16', 64, 3, 1, noise='sample', filt='asym', out_hw=(130, 130)),
    _fir('f16-noise-linear-clamp7e4-nobias-enc', [('sep', 'half', False, True, False)], 'f16', 192, 2, 1, noise='shared', act=1,
         clamp=7e4, bias=False, pad=2),
    _fir('f16-hilo-clamp1-enc', [('sep', 'half', True, False, True)], 'f16', 64, 2, 2, clamp=1.0, pad=2),
    _fir('f16-hilo-select-asym', [('sep', 'half', True, False, False)], 'f16', 64, 2, 2, alpha=1.7, filt='asym'),
    _fir('f16-hilo-bnoise-clamp03', [('sep', 'half', True, True, True)], 'f16', 192, 3, 2, noise='sample', clamp=0.3),
    _fir('f16-hilo-noise-select-nobias', [('sep', 'half', True, True, False)], 'f16', 64, 2, 2, noise='shared', alpha=-0.3,
         clamp=256.0, bias=False),
    _fir('fir16-f32-hilo-bnoise-full', [('fir16', 'float')], 'f32', 32, 3, 2, noise='sample', filt='full'),
    _fir('fir16-f32-clamp03-nobias-enc-v1', [('fir16', 'float')], 'f32', 96, 2, 1, clamp=0.3, bias=False, pad=2, variant=1, vs_sep=True),
    _fir('fir16-f16-noise-v1', [('fir16', 'half')], 'f16', 64, 2, 1, noise='shared', clamp=256.0, variant=1, vs_sep=True),
    _fir('fir16-f16-hilo-bnoise-v1', [('fir16', 'half')], 'f16', 64, 2, 2, noise='sample', clamp=256.0, variant=1, vs_sep=True),
    _fir('fir16-f16-bnoise-select-full', [('fir16', 'half')], 'f16', 192, 3, 1, noise='sample', alpha=1.7, clamp=0.3, filt='full'),
    _fir('fir16-split-bnoise-linear-enc', [('fir16', 'split')], 'split', 64, 3, 2, noise='sample', act=1, bias=False, pad=2),
]


def _fir_filter(kind):
    from pix2pix3d_b200.torch_utils.ops import upfirdn2d
    if kind == 'sym':
        return upfirdn2d.setup_filter([1, 3, 3, 1]).cuda()
    if kind == 'asym':    # f[j][i] = fy[j] * fx[i], integer taps (exact in fp32): a swap of row and column taps changes it
        fy, fx = torch.tensor([1., 3., 3., 1.]), torch.tensor([1., 2., 3., 4.])
        return (torch.outer(fy, fx) / 64).cuda()
    return (torch.tensor([[1., 2., 0., 1.], [0., 3., 1., 2.], [2., 1., 4., 0.], [1., 0., 2., 3.]]) / 16).cuda()    # rank 4


def _fir_ref(x64, f, pad, out_hw, gain):
    """float64 upfirdn2d without up/down sampling: pad, true convolution with f (flip_filter=False), gain. [B,H,W,C] in and out."""
    b, h, w, c = x64.shape
    oh, ow = out_hw
    xc = F.pad(x64.permute(0, 3, 1, 2).reshape(b * c, 1, h, w), (pad, ow + 3 - w - pad, pad, oh + 3 - h - pad))
    y = F.conv2d(xc, (f.double() * gain).flip([0, 1])[None, None])
    return y.reshape(b, c, oh, ow).permute(0, 2, 3, 1)


@pytest.mark.gpu
@pytest.mark.parametrize('expect,c', FIR_CASES)
def test_fir_instance(expect, c, monkeypatch):
    from pix2pix3d_b200 import tcconv
    torch.manual_seed(51)
    b, ch, planes = c['b'], c['c'], c['planes']
    oh, ow = c['out_hw']
    pad, fir_gain = (1, 4.0) if c['pad'] == 1 else (2, 1.0)
    ih, iw = (oh + 1, ow + 1) if c['pad'] == 1 else (oh - 1, ow - 1)
    f = _fir_filter(c['filt'])
    sep = tcconv.separable_factors(f)
    assert (sep is None) == (c['filt'] == 'full')
    x32 = torch.randn(b, ih, iw, ch, device='cuda')
    if c['dtype'] == 'f16':
        x = x32.half()
        xv = x.double()
    elif c['dtype'] == 'split':
        hi = x32.half()
        x = torch.stack([hi, (x32 - hi.float()).half()])
        xv = x[0].double() + x[1].double()
    else:
        x = x32
        xv = x.double()
    noise = {None: None, 'shared': torch.randn(oh, ow, device='cuda') * 0.5,
             'sample': torch.randn(b, oh, ow, device='cuda') * 0.5}[c['noise']]
    bias = torch.randn(ch, device='cuda') * 0.5 if c['bias'] else None
    act, alpha, clamp = c['act'], c['alpha'], c['clamp']
    act_gain = SQRT2 if act == 3 else 1.0

    def run(variant):
        monkeypatch.setattr(tcconv, 'FIR_VARIANT', variant)
        return tcconv.fir_act_nhwc(x, f, noise, bias, planes, (oh, ow), pad0=(pad, pad), fir_gain=fir_gain, act=act, alpha=alpha,
                                   act_gain=act_gain, clamp=clamp)

    y, names = launched_kernels(lambda: run(c['variant']))
    assert_instances(names, expect)

    # reference: float64 FIR on the exact input values, then the kernel's rounding points
    v = _fir_ref(xv, f, pad, (oh, ow), fir_gain)
    nz = None if noise is None else (noise[None, :, :, None] if noise.ndim == 2 else noise[..., None])
    if c['dtype'] == 'f16':
        # fp16 path: FIR output rounded to fp16 (the fp32 sum of fp16 x tap products rounds exactly as float64 -> fp32 -> fp16
        # does); noise added in fp32 and rounded again; bias, act, gain, clamp in fp32
        v = v.float().half().float()
        if nz is not None:
            v = (v + nz).half().float()
        if bias is not None:
            v = v + bias
        if act == 3:
            v = torch.where(v > 0, v, v * alpha)
        v = v * act_gain
        scale = float(v.abs().max())
        if clamp >= 0:
            v = v.clamp(-clamp, clamp)
        v = v.double()
    else:
        if nz is not None:
            v = v + nz.double()
        if bias is not None:
            v = v + bias.double()
        if act == 3:
            v = torch.where(v > 0, v, v * alpha)
        v = v * act_gain
        scale = float(v.abs().max())
        if clamp >= 0:
            v = v.clamp(-clamp, clamp)
    # Where the fp32 FIR sum is not the float64 sum rounded to fp32 (fp32 input always; fp16 input where the tap products need
    # more than 24 bits), a value within that difference of an fp16 rounding midpoint rounds the other way: the final fp16
    # plane, or (fp16 input) the fp16 FIR output the epilogue starts from, moves by one fp16 ulp. Such elements are rare.
    d = float(_ulp_diff16(y[0], v, 0.0 if c['dtype'] == 'f16' else 1e-6 * scale).max())
    assert d <= 1.0, f'{d} ulp'
    if planes == 2:
        err = (y[0].double() + y[1].double() - v).abs() / scale
        if c['dtype'] == 'f16':
            # measured on a B200: 2.8e-6 of the elements beyond 2e-6 (max 1.8e-5) in f16-hilo-bnoise-clamp03, none elsewhere
            rate = float((err > 2e-6).double().mean())
            assert rate <= 1e-3, rate
            assert float(err.max()) < 2e-3
        else:
            assert float(err.max()) < 2e-6
    else:
        # measured on a B200: 2.6e-4 .. 6.1e-4 of the elements differ (by one ulp) for fp32 input, none for fp16 input
        rate = float((y[0].double() != v.half().double()).double().mean())
        assert rate <= 1e-3, rate
    if c['vs_sep']:
        # the separable kernel on the same input: another fp32 summation order -> at most 1 ulp apart
        y3 = run(3)
        assert float(_ulp_diff16(y3[0], y[0].double()).max()) <= 1.0     # measured: 2.9e-4 of the elements (fp32 in), none (fp16)


# ------------------------------------------------------------------------------------------------------------------------
# Table completeness (no GPU)
# ------------------------------------------------------------------------------------------------------------------------
def test_case_tables_cover_every_instance():
    """The GPU cases above declare instances that together are every instance the libraries compile: the 24 convolution
    kernels, the split-K finisher under each act form, the 16 separable FIR kernels and the three 16-tap FIR kernels. Each
    declaration also agrees with the arguments of its case."""
    assert len(CONV_INSTANCES) == 24 and len(FIR_INSTANCES) == 19
    seen = set()
    for p in CONV_CASES:
        shape, expect, c, alts = p.values
        form = act_form(c['act'], c['alpha'])
        for inst in expect:
            if inst[0] == 'finish':
                assert inst[1] == form, p.id
            else:
                assert inst[-2:] == (form, c['clamp'] >= 0), p.id
        assert shape in CONV_SHAPES
        seen.update(expect)
    for p in PHASE_CASES:
        for _, expect in p.values[-1]:
            assert all(inst[-2:] == (0, False) or inst == ('finish', 0) for inst in expect), p.id     # act=1, no clamp
            seen.update(expect)
    for p in FIR_CASES:
        expect, c = p.values
        (inst,) = expect
        if inst[0] == 'sep':
            assert c['variant'] == 3 and c['filt'] != 'full' and c['dtype'] != 'split', p.id
            assert inst[1:] == ('float' if c['dtype'] == 'f32' else 'half', c['planes'] == 2, c['noise'] is not None,
                                fir_fast(c['act'], c['alpha'], c['clamp'], c['planes'])), p.id
        else:
            assert c['variant'] == 1 or c['filt'] == 'full' or c['dtype'] == 'split', p.id
            assert inst[1] == {'f32': 'float', 'f16': 'half', 'split': 'split'}[c['dtype']], p.id
        seen.update(expect)
    assert seen == set(CONV_INSTANCES) | set(FINISH_INSTANCES) | set(FIR_INSTANCES), \
        (set(CONV_INSTANCES) | set(FINISH_INSTANCES) | set(FIR_INSTANCES)) ^ seen
    # every instance's name pattern is distinct from every other's
    demangled = {inst: _demangled(inst) for inst in seen}
    for inst, name in demangled.items():
        hits = {i for i in seen if re.search(_instance_regex(i), name)}
        assert hits == (set(FINISH_INSTANCES) if inst[0] == 'finish' else {inst}), name
    assert _FAMILY.search(demangled[('grid', 3, 0, False)])


def _demangled(inst):
    """A kernel name as torch.profiler shows it (profiles/r02b_train_step_kernels_ours.txt), for the regex self-check."""
    args = 'CUtensorMap_st, CUtensorMap_st, p3d::ConvKernelArgs'
    tf = lambda v: 'true' if v else 'false'
    if inst[0] == 'grid':
        return f'void p3d::conv_gemm_kernel<{inst[1]}, {inst[2]}, {tf(inst[3])}>({args})'
    if inst[0] in ('persist', 'pair'):
        return f'void p3d::conv_gemm_{inst[0]}_kernel<{inst[1]}, {tf(inst[2])}>({args}, int, int)'
    if inst[0] == 'finish':
        return 'p3d::conv_splitk_finish_kernel(p3d::ConvKernelArgs, int, int)'
    if inst[0] == 'sep':
        t = 'float' if inst[1] == 'float' else '__half'
        return f'void p3d::fir_act_nhwc_sep_kernel<{t}, {tf(inst[2])}, {tf(inst[3])}, {tf(inst[4])}>(CUtensorMap_st, p3d::FirSepTaps)'
    t, vec, s = {'float': ('float', 4, False), 'half': ('__half', 8, False), 'split': ('__half', 8, True)}[inst[1]]
    return f'void p3d::fir_act_nhwc_kernel<{t}, {vec}, {tf(s)}>(CUtensorMap_st, float const*)'
