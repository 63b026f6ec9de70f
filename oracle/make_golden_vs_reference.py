"""Generate tests/golden/vs_reference_*.npz: what the reference's own CUDA path (its JIT-built plugins, cuDNN convolutions)
computes for the inputs of tests/test_gpu_vs_reference.py, so that the comparison runs without a reference checkout.

    python oracle/make_golden_vs_reference.py REFERENCE_ROOT [OUT_DIR]       # needs a CUDA device

REFERENCE_ROOT is a checkout of pix2pix3D; it is imported read-only under its own module names (`training`, `torch_utils`)
by baseline/ref_harness.py. Inputs come from the same seeds the tests use and are stored only as digests; outputs are
stored as a fixed sample of their elements (`sample_index`), which keeps all five files together near 200 KB.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

SYNTH_CASES = {                       # golden name -> (workload, batch, force_fp32)
    'vs_reference_seg2cat_512_fp32': ('seg2cat_512', 2, True),
    'vs_reference_edge2car_128_fp32': ('edge2car_128', 3, True),
    'vs_reference_seg2cat_512_default': ('seg2cat_512', 2, False),
}
SYNTH_SAMPLE = 2048                   # elements kept per synthesis output
OPS_SAMPLE = 512                      # elements kept per op output / gradient
SEED_IN = 7


def sample_index(n, k):
    """The flat indices kept of an n-element array: all of them when n <= k, else k distinct ones from a fixed seed."""
    if n <= k:
        return np.arange(n)
    return np.sort(np.random.RandomState(0).choice(n, k, replace=False))


def sampled(a, k):
    a = np.asarray(a, np.float32).reshape(-1)
    return a[sample_index(a.size, k)]


def digest(t):
    """float64 sum of squares of a tensor or array: equal digests mean the seeded inputs came out the same."""
    if hasattr(t, 'detach'):
        t = t.detach().cpu().double().numpy()
    return np.float64(np.square(np.asarray(t, np.float64)).sum())


def ops_inputs(dev):
    """x and b of the bias_act / upfirdn2d comparison."""
    import torch
    torch.manual_seed(0)
    x = torch.randn(3, 8, 33, 31, device=dev, requires_grad=True)
    b = torch.randn(8, device=dev, requires_grad=True)
    return x, b


def filtered_lrelu_inputs(dev):
    import torch
    x = torch.randn(2, 6, 25, 20, device=dev, generator=torch.Generator(dev).manual_seed(1))
    b = torch.randn(6, device=dev, generator=torch.Generator(dev).manual_seed(2))
    return x, b


def synthesis_inputs(workload, batch, num_ws, nrr, Sc, Sf):
    """ws, c and the renderer's two random draws (stratified jitter, importance-sampling u) for one comparison."""
    import torch
    from pix2pix3d_b200 import configs
    w = configs.WORKLOADS[workload]
    ws = configs.synthetic_ws(batch, num_ws, SEED_IN)
    c = configs.camera_labels(batch, SEED_IN + 1, w['preset'])
    g = torch.Generator().manual_seed(SEED_IN + 2)
    jitter = torch.rand(batch, nrr * nrr, Sc, 1, generator=g)
    u = torch.rand(batch * nrr * nrr, Sf, generator=g)
    return ws, c, jitter, u


def state_dict_digest(G):
    """Parameter / buffer names and the digest of each: equal digests mean equal seeded weights."""
    sd = G.state_dict()
    keys = sorted(sd)
    return np.array(keys), np.array([digest(sd[k]) for k in keys])


def bias_act_upfirdn2d_cases(bias_act, upfirdn2d, x, b, f):
    """Forward and gradients of bias_act / upfirdn2d through one wrapper implementation; returns [(name, array)]."""
    import torch
    res = []
    for act in ('lrelu', 'swish', 'linear', 'sigmoid', 'softplus'):
        y = bias_act(x, b, act=act, clamp=1.5, impl='cuda')
        gx, gb = torch.autograd.grad(y.square().sum(), [x, b], create_graph=True)
        (ggx,) = torch.autograd.grad(gx.square().sum() + gb.square().sum(), [x], allow_unused=True)
        res += [('bias_act ' + act, y), ('bias_act dx ' + act, gx), ('bias_act db ' + act, gb)]
        if ggx is not None:
            res.append(('bias_act d2 ' + act, ggx))
    for kw in (dict(up=2, padding=[2, 1, 2, 1], gain=4), dict(down=2, padding=[1, 1, 1, 1]), dict(padding=[1, 1, 1, 1], gain=4)):
        y = upfirdn2d(x, f, impl='cuda', **kw)
        (gx,) = torch.autograd.grad(y.square().sum(), [x])
        res += [(f'upfirdn2d {kw}', y), (f'upfirdn2d dx {kw}', gx)]
    return [(n, t.detach().float().cpu().numpy()) for n, t in res]


def filtered_lrelu_filters(dev):
    import scipy.signal
    import torch
    k12 = torch.as_tensor(scipy.signal.firwin(numtaps=12, cutoff=0.25, width=0.3, fs=2.0), dtype=torch.float32, device=dev)
    f4 = torch.tensor([1., 3., 3., 1.], device=dev)
    f4 = torch.outer(f4, f4) / 64
    return [dict(fu=k12, fd=k12, up=2, down=2, padding=[10, 9, 10, 9], gain=1.4, slope=0.2, clamp=256),
            dict(fu=f4, fd=f4, up=2, down=2, padding=[3, 2, 3, 2], gain=1.0, slope=0.2, clamp=0.8),
            dict(fu=k12, fd=None, up=2, down=1, padding=[5, 6, 5, 6], gain=2 ** 0.5, slope=0.2, clamp=None, flip_filter=True)]


def filtered_lrelu_cases(filtered_lrelu, x32, b32, cases):
    """Forward and gradients of filtered_lrelu; returns [(dtype name, array)]. The 2-D filter case runs in fp32 only: the
    reference's plugin has no fused kernel for 2-D filters at up = down = 2 and composes upfirdn2d + act + upfirdn2d, which
    in fp16 rounds the up-sampled tensor and so takes other lrelu / clamp branches than a kernel that keeps fp32 inside."""
    import torch
    res = []
    for kw in cases:
        for dtype in ((torch.float32, torch.float16) if kw['fu'].ndim == 1 else (torch.float32,)):
            x = x32.detach().to(dtype).requires_grad_(True)
            b = b32.detach().to(dtype).requires_grad_(True)
            y = filtered_lrelu(x, b=b, impl='cuda', **kw)
            gx, gb = torch.autograd.grad(y.float().square().sum(), [x, b])
            res += [(str(dtype), y), (str(dtype), gx), (str(dtype), gb)]
    return [(d, t.detach().float().cpu().numpy()) for d, t in res]


def main(ref_root, out_dir):
    import torch
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, 'baseline'))
    import ref_harness as rh
    from pix2pix3d_b200 import configs
    rh.REF_ROOT = os.path.abspath(ref_root)
    tc = rh.import_reference()
    assert torch.cuda.is_available(), 'the reference CUDA path needs a CUDA device'
    dev = torch.device('cuda')
    torch.backends.cudnn.allow_tf32 = False          # the reference's fp32 convolutions must be true fp32 for a 1e-3 comparison
    torch.backends.cuda.matmul.allow_tf32 = False
    os.makedirs(out_dir, exist_ok=True)
    print('reference:', os.path.dirname(os.path.dirname(tc.__file__)), '| device:', torch.cuda.get_device_name(0))

    for name, (workload, batch, force_fp32) in SYNTH_CASES.items():
        w = configs.WORKLOADS[workload]
        G = rh.build_generator(workload, seed=0, device=dev)
        rk = G.rendering_kwargs
        nrr = w['nrr']
        ws, c, jitter, u = synthesis_inputs(workload, batch, G.backbone.num_ws, nrr, rk['depth_resolution'],
                                            rk['depth_resolution_importance'])
        with torch.no_grad(), rh.replay_rand(jitter.to(dev), u.to(dev)):
            out = G.synthesis(ws.to(dev), c.to(dev), noise_mode='const', neural_rendering_resolution=nrr, force_fp32=force_fp32)
        keys, sumsq = state_dict_digest(G)
        d = dict(ws_digest=digest(ws), c_digest=digest(c), jitter_digest=digest(jitter), u_digest=digest(u), sd_keys=keys,
                 sd_digest=sumsq, out_keys=np.array(sorted(out)))
        for k, v in out.items():
            d['out_' + k] = sampled(v.float().cpu().numpy(), SYNTH_SAMPLE)
            d['shape_' + k] = np.array(v.shape)
        np.savez_compressed(os.path.join(out_dir, name + '.npz'), **d)
        print(name, {k: tuple(v.shape) for k, v in out.items()})
        del G, out
        torch.cuda.empty_cache()

    # the reference's op wrappers on its stock JIT-built plugins
    import torch_utils.ops.bias_act as r_ba
    import torch_utils.ops.filtered_lrelu as r_fl
    import torch_utils.ops.upfirdn2d as r_up
    assert r_ba._init() and r_up._init() and r_fl._init()
    x, b = ops_inputs(dev)
    f = r_up.setup_filter([1, 3, 3, 1], device=dev)
    res = bias_act_upfirdn2d_cases(r_ba.bias_act, r_up.upfirdn2d, x, b, f)
    d = dict(x_digest=digest(x), b_digest=digest(b), f=f.cpu().numpy(), names=np.array([n for n, _ in res]))
    for i, (n, a) in enumerate(res):
        d[f'res{i:03d}'] = sampled(a, OPS_SAMPLE)
        d[f'shape{i:03d}'] = np.array(a.shape)
    np.savez_compressed(os.path.join(out_dir, 'vs_reference_bias_act_upfirdn2d.npz'), **d)

    x32, b32 = filtered_lrelu_inputs(dev)
    import warnings
    with warnings.catch_warnings():
        warnings.simplefilter('ignore', RuntimeWarning)
        res = filtered_lrelu_cases(r_fl.filtered_lrelu, x32, b32, filtered_lrelu_filters(dev))
    d = dict(x_digest=digest(x32), b_digest=digest(b32), dtypes=np.array([n for n, _ in res]))
    for i, (_, a) in enumerate(res):
        d[f'res{i:03d}'] = sampled(a, OPS_SAMPLE)
        d[f'shape{i:03d}'] = np.array(a.shape)
    np.savez_compressed(os.path.join(out_dir, 'vs_reference_filtered_lrelu.npz'), **d)
    for fn in sorted(os.listdir(out_dir)):
        print(fn, os.path.getsize(os.path.join(out_dir, fn)))


if __name__ == '__main__':
    main(sys.argv[1], sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, 'tests', 'golden'))
