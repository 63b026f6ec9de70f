"""Comparison with the reference's own PyTorch/CUDA path (the oracle of record, SURVEY 8c).

tests/golden/vs_reference_*.npz hold what the unmodified reference computed on a B200 through its JIT-built plugins and
cuDNN for the inputs below (oracle/make_golden_vs_reference.py): seeded generator weights, seeded ws / c, and the
renderer's two random draws fed in from seeded tensors. Inputs are regenerated from their seeds and checked against stored
digests; outputs are kept as a fixed sample of their elements, on which this package's results are compared."""
import os
import sys
import warnings

import numpy as np
import pytest
import torch

from conftest import ROOT, load_golden, rel_err

sys.path.insert(0, os.path.join(ROOT, 'baseline'))
import make_golden_vs_reference as M  # noqa: E402
import ref_harness as rh  # noqa: E402

pytestmark = pytest.mark.gpu


def _ours(name):
    """This package's G.synthesis on the golden's inputs; returns (outputs sampled as stored, golden)."""
    from pix2pix3d_b200 import configs
    workload, batch, force_fp32 = M.SYNTH_CASES[name]
    g = load_golden(name)
    dev = torch.device('cuda')
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    w = configs.WORKLOADS[workload]
    G = configs.build_generator(workload, seed=0, device=dev, with_mapping=False)
    keys, sumsq = M.state_dict_digest(G)
    assert list(keys) == list(g['sd_keys']) and np.array_equal(sumsq, g['sd_digest']), 'weights must be the reference\'s'
    rk = G.rendering_kwargs
    nrr = w['nrr']
    ws, c, jitter, u = M.synthesis_inputs(workload, batch, G.backbone.num_ws, nrr, rk['depth_resolution'],
                                          rk['depth_resolution_importance'])
    for k, t in (('ws', ws), ('c', c), ('jitter', jitter), ('u', u)):
        assert M.digest(t) == g[k + '_digest'], f'input {k} must be the reference\'s'
    kw = dict(noise_mode='const', neural_rendering_resolution=nrr, force_fp32=force_fp32)
    with torch.no_grad(), rh.replay_rand(jitter.to(dev), u.to(dev)):
        out = G.synthesis(ws.to(dev), c.to(dev), **kw)
    assert sorted(out) == list(g['out_keys'])
    for k, v in out.items():
        assert tuple(v.shape) == tuple(g['shape_' + k]), k
    return {k: M.sampled(v.float().cpu().numpy(), M.SYNTH_SAMPLE) for k, v in out.items()}, g


@pytest.mark.parametrize('workload,batch', [('seg2cat_512', 2), ('edge2car_128', 3)])
def test_synthesis_matches_reference_cuda_path_fp32(workload, batch):
    name = f'vs_reference_{workload}_fp32'
    assert M.SYNTH_CASES[name] == (workload, batch, True)
    out, g = _ours(name)
    errs = {k: rel_err(v, g['out_' + k]) for k, v in out.items()}
    print('VS-REFERENCE-CUDA fp32', workload, errs)
    for k, e in errs.items():
        assert e < 1e-3, (k, errs)


def test_synthesis_matches_reference_cuda_path_default_dtypes():
    """SR in fp16 on both sides (superresolution.py:304): the two fp16 paths round differently, so the bound is fp16-sized."""
    out, g = _ours('vs_reference_seg2cat_512_default')
    errs = {k: rel_err(v, g['out_' + k]) for k, v in out.items()}
    print('VS-REFERENCE-CUDA default dtypes', errs)
    for k in ('image_raw', 'image_depth', 'semantic_raw'):
        assert errs[k] < 1e-3, (k, errs)
    for k in ('image', 'semantic'):
        assert errs[k] < 2e-2, (k, errs)


def test_reference_op_wrappers_run_on_libp3d_plugins():
    """bias_act / upfirdn2d (forward, first- and second-order gradients) on libp3d against the reference's wrappers on its
    stock plugins (e.g. the stock CUDA path does not clamp the gradient of a clamped `linear` activation,
    bias_act.py:164-167 saves no `y` for it, and neither may this package). The forward also goes through the plugin
    objects `custom_ops.get_plugin` hands to the reference's wrappers, with the arguments those wrappers pass."""
    from pix2pix3d_b200.torch_utils import custom_ops as ours
    from pix2pix3d_b200.torch_utils.ops import bias_act as ba, upfirdn2d as up
    g = load_golden('vs_reference_bias_act_upfirdn2d')
    dev = torch.device('cuda')
    x, b = M.ops_inputs(dev)
    assert M.digest(x) == g['x_digest'] and M.digest(b) == g['b_digest'], 'inputs must be the reference\'s'
    f = torch.from_numpy(g['f']).to(dev)
    got = M.bias_act_upfirdn2d_cases(ba.bias_act, up.upfirdn2d, x, b, f)
    assert [n for n, _ in got] == list(g['names'])
    want = {}
    for i, (n, a) in enumerate(got):
        assert a.shape == tuple(g[f'shape{i:03d}']), n
        want[n] = g[f'res{i:03d}']
        assert rel_err(M.sampled(a, M.OPS_SAMPLE), want[n]) < 2e-6, n

    p_ba = ours.get_plugin('bias_act_plugin', sources=['bias_act.cpp', 'bias_act.cu'])
    p_up = ours.get_plugin('upfirdn2d_plugin', sources=['upfirdn2d.cpp', 'upfirdn2d.cu'])
    null = torch.empty([0], device=dev)
    with torch.no_grad():
        for act in ('lrelu', 'swish', 'linear', 'sigmoid', 'softplus'):
            spec, alpha, gain, clamp = ba._resolve(act, None, None, 1.5)
            y = p_ba.bias_act(x, b, null, null, null, 0, 1, spec.cuda_idx, alpha, gain, clamp)
            assert rel_err(M.sampled(y.cpu().numpy(), M.OPS_SAMPLE), want['bias_act ' + act]) < 2e-6, act
        for kw, (upxy, downxy, pads, gain) in (("{'up': 2, 'padding': [2, 1, 2, 1], 'gain': 4}", (2, 1, (2, 1, 2, 1), 4.0)),
                                                ("{'down': 2, 'padding': [1, 1, 1, 1]}", (1, 2, (1, 1, 1, 1), 1.0)),
                                                ("{'padding': [1, 1, 1, 1], 'gain': 4}", (1, 1, (1, 1, 1, 1), 4.0))):
            y = p_up.upfirdn2d(x, f, upxy, upxy, downxy, downxy, *pads, False, gain)
            assert rel_err(M.sampled(y.cpu().numpy(), M.OPS_SAMPLE), want['upfirdn2d ' + kw]) < 2e-6, kw


def test_reference_filtered_lrelu_wrapper_runs_on_libp3d_plugin():
    """filtered_lrelu (forward and gradients, fp32 and fp16) on libp3d against the reference's
    torch_utils/ops/filtered_lrelu.py on its stock JIT-built plugin."""
    from pix2pix3d_b200.torch_utils.ops import filtered_lrelu as fl
    g = load_golden('vs_reference_filtered_lrelu')
    dev = torch.device('cuda')
    x, b = M.filtered_lrelu_inputs(dev)
    assert M.digest(x) == g['x_digest'] and M.digest(b) == g['b_digest'], 'inputs must be the reference\'s'
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        got = M.filtered_lrelu_cases(fl.filtered_lrelu, x, b, M.filtered_lrelu_filters(dev))
    assert [d for d, _ in got] == list(g['dtypes'])
    for i, (d, a) in enumerate(got):
        assert a.shape == tuple(g[f'shape{i:03d}']), i
        a, w = M.sampled(a, M.OPS_SAMPLE), g[f'res{i:03d}']
        # fp16: both kernels hold fp32 inside but sum in different orders; an element within rounding of 0 / the clamp may
        # take the other branch, which moves single gradient entries
        tol = 2e-5 if d == str(torch.float32) else 2e-2
        assert rel_err(a, w) < tol, (i, d, rel_err(a, w))
