"""Tensor-core inference engine (pix2pix3d_b200/engine.py) against the generic op-by-op formulation and the fixtures."""
import numpy as np
import pytest
import torch

from conftest import load_golden, rel_err

pytestmark = pytest.mark.gpu


def _net(channel_base, channel_max, res, img_channels, num_fp16_res=0, conv_clamp=None):
    from pix2pix3d_b200.training.networks_stylegan2 import SynthesisNetwork
    torch.manual_seed(0)
    net = SynthesisNetwork(w_dim=64, img_resolution=res, img_channels=img_channels, channel_base=channel_base,
                           channel_max=channel_max, num_fp16_res=num_fp16_res, conv_clamp=conv_clamp).eval().requires_grad_(False)
    g = torch.Generator().manual_seed(1)
    for name, p in net.named_parameters():
        if name.endswith('noise_strength'):
            p.copy_(torch.randn([], generator=g) * 0.2)
        if name.endswith('.bias') and 'affine' not in name:
            p.copy_(torch.randn(p.shape, generator=g) * 0.2)
    return net.cuda()


@pytest.mark.parametrize('cfg', [dict(channel_base=2048, channel_max=64, res=32, img_channels=96),
                                 dict(channel_base=4096, channel_max=128, res=64, img_channels=3),
                                 dict(channel_base=1024, channel_max=16, res=16, img_channels=6)])
@pytest.mark.parametrize('noise_mode', ['const', 'none'])
def test_synthesis_network_engine_matches_generic_fp32(cfg, noise_mode):
    from pix2pix3d_b200 import _lib, engine
    net = _net(**cfg)
    ws = torch.randn(3, net.num_ws, 64, device='cuda')
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    with torch.no_grad():
        engine.enabled = False
        try:
            ref = net(ws, noise_mode=noise_mode)
        finally:
            engine.enabled = True
        n0 = _lib.launch_count
        out = net(ws, noise_mode=noise_mode)
    assert _lib.launch_count - n0 > 10
    assert out.shape == ref.shape and out.dtype == torch.float32
    assert rel_err(out.cpu().numpy(), ref.cpu().numpy()) < 2e-5      # three-pass split keeps fp32-level accuracy


@pytest.mark.parametrize('cfg', [dict(channel_base=2048, channel_max=64, res=32, img_channels=96),
                                 dict(channel_base=4096, channel_max=128, res=64, img_channels=3, num_fp16_res=2, conv_clamp=256)])
def test_synthesis_network_engine_random_noise_consumes_the_same_rng_stream(cfg):
    """noise_mode='random' (the API default, networks_stylegan2.py:320-321): the engine draws one noise image per sample and
    layer with the same torch.randn calls in the same order as the op-by-op formulation, so seeding the generator identically
    gives the same images -- and leaves the generator in the same state."""
    from pix2pix3d_b200 import _lib, engine
    net = _net(**cfg)
    ws = torch.randn(3, net.num_ws, 64, device='cuda')
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    with torch.no_grad():
        engine.enabled = False
        try:
            torch.manual_seed(123)
            ref = net(ws, noise_mode='random')
            after_ref = torch.rand(4, device='cuda')
        finally:
            engine.enabled = True
        n0 = _lib.launch_count
        torch.manual_seed(123)
        out = net(ws, noise_mode='random')
        after = torch.rand(4, device='cuda')
        torch.manual_seed(124)
        other = net(ws, noise_mode='random')
    assert _lib.launch_count - n0 > 10
    assert torch.equal(after, after_ref)
    tol = 2e-5 if not cfg.get('num_fp16_res') else 2e-2
    assert rel_err(out.cpu().numpy(), ref.cpu().numpy()) < tol
    assert rel_err(other.cpu().numpy(), ref.cpu().numpy()) > 10 * tol       # the noise is live


def test_synthesis_network_engine_fp16_blocks():
    """fp16 blocks with conv_clamp (the super-resolution configuration): engine vs the reference-style fp16 path."""
    from pix2pix3d_b200 import engine
    net = _net(channel_base=2048, channel_max=64, res=64, img_channels=3, num_fp16_res=2, conv_clamp=256)
    ws = torch.randn(2, net.num_ws, 64, device='cuda')
    with torch.no_grad():
        engine.enabled = False
        try:
            ref16 = net(ws, noise_mode='const')
            ref32 = net(ws, noise_mode='const', force_fp32=True)
        finally:
            engine.enabled = True
        out16 = net(ws, noise_mode='const')
        out32 = net(ws, noise_mode='const', force_fp32=True)
    assert rel_err(out32.cpu().numpy(), ref32.cpu().numpy()) < 2e-5
    e_ref = rel_err(ref16.cpu().numpy(), ref32.cpu().numpy())          # how far the fp16 reference path is from fp32
    e_out = rel_err(out16.cpu().numpy(), ref32.cpu().numpy())
    assert e_out < max(2 * e_ref, 5e-3)                               # the engine's fp16 path is no worse than that
    assert rel_err(out16.cpu().numpy(), ref16.cpu().numpy()) < max(3 * e_ref, 5e-3)


def test_superresolution_engine_matches_generic():
    from pix2pix3d_b200 import engine
    from pix2pix3d_b200.training.superresolution import SuperresolutionHybrid2X, SuperresolutionHybrid8XDC_semantic
    torch.manual_seed(3)
    for cls, res_in, kw in ((SuperresolutionHybrid2X, 64, {}), (SuperresolutionHybrid8XDC_semantic, 128, dict(semantic_channels=6))):
        sr = cls(channels=32, img_resolution=128 if res_in == 64 else 512, sr_num_fp16_res=4, sr_antialias=True, **kw).eval().requires_grad_(False).cuda()
        n_img = sr.block0.img_channels
        b = 1 if res_in == 128 else 2
        x = torch.randn(b, 32, res_in, res_in, device='cuda')
        rgb = torch.randn(b, n_img, res_in, res_in, device='cuda')
        ws = torch.randn(b, 14, 512, device='cuda')
        with torch.no_grad():
            engine.enabled = False
            try:
                # SynthesisBlockNoUp adds ToRGB into the image it was given (superresolution.py:283): pass clones
                ref = sr(rgb.clone(), x.clone(), ws, noise_mode='none', force_fp32=True)
            finally:
                engine.enabled = True
            out = sr(rgb.clone(), x.clone(), ws, noise_mode='none', force_fp32=True)
            out16 = sr(rgb.clone(), x.clone(), ws, noise_mode='none')
        assert rel_err(out.cpu().numpy(), ref.cpu().numpy()) < 2e-5
        assert rel_err(out16.cpu().numpy(), ref.cpu().numpy()) < 2e-2


def test_graphed_synthesis_replays_and_matches_eager():
    """CUDA-graph capture of G.synthesis: same result as the eager call for the same inputs and noise-free options."""
    import pix2pix3d_b200.training.triplane_cond as tc
    from make_golden import SYNTH_CASES, build_generator
    from pix2pix3d_b200.graphs import GraphedSynthesis
    case = dict(SYNTH_CASES['seg_nrr64'])
    G = build_generator(tc, case).cuda()
    g = load_golden('synthesis_seg_nrr64')
    ws, c = torch.from_numpy(g['ws']).cuda(), torch.from_numpy(g['c']).cuda()
    kw = dict(noise_mode='const', neural_rendering_resolution=case['nrr'])
    gs = GraphedSynthesis(G, ws, c, **kw)
    assert gs.native_launches > 40      # libp3d launches captured in the graph (an up layer is 2: merged phases + FIR)
    torch.manual_seed(123)
    a = {k: v.clone() for k, v in gs(ws, c).items()}
    torch.cuda.synchronize()
    assert all(torch.isfinite(v).all() for v in a.values())
    # a different camera gives a different image; the same inputs again reproduce statistics (fresh jitter each replay)
    c2 = c.clone(); c2[:, 3] += 0.05
    b = {k: v.clone() for k, v in gs(ws, c2).items()}
    assert (a['image'] - b['image']).abs().max() > 1e-4
    with torch.no_grad():
        e = G.synthesis(ws, c, **kw)
    # stratified jitter differs between calls, so compare loosely against the eager result
    assert rel_err(a['image'].cpu().numpy(), e['image'].cpu().numpy()) < 0.2
    assert a['image'].shape == e['image'].shape


@pytest.mark.parametrize('workload,batch,noise_mode', [
    pytest.param('seg2cat_512', 3, 'const', id='seg2cat_512-3'), pytest.param('seg2face_512', 2, 'const', id='seg2face_512-2'),
    pytest.param('edge2car_128', 5, 'const', id='edge2car_128-5'), pytest.param('seg2cat_512', 3, 'random', id='seg2cat_512-3-random')])
def test_full_size_workloads_engine_matches_generic_path(workload, batch, noise_mode):
    """BASELINE configs 2-4 at their real channel counts and resolutions (odd batch sizes on purpose): the whole-generator
    tensor-core path against the op-by-op formulation of the same modules (ATen convolutions + libp3d bias_act/upfirdn2d,
    staged or fused renderer), with identical renderer noise. noise_mode='random' (the default of G.synthesis) draws one
    noise image per sample and layer; both paths must draw them, and then the renderer's jitter and `u`, in the same order
    from the same seed, which the generator state after the call shows."""
    from pix2pix3d_b200 import _lib, configs, engine
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    w = configs.WORKLOADS[workload]
    G = configs.build_generator(workload, seed=3, device='cuda', with_mapping=False)
    ws = configs.synthetic_ws(batch, G.backbone.num_ws, seed=4).cuda()
    c = configs.camera_labels(batch, seed=5, preset=w['preset']).cuda()
    kw = dict(noise_mode=noise_mode, neural_rendering_resolution=w['nrr'])

    def run():
        torch.manual_seed(77)                     # same noise / jitter / u draws for both paths
        with torch.no_grad():
            out = {k: v.float().clone() for k, v in G.synthesis(ws, c, **kw).items()}
        return out, (torch.get_rng_state(), torch.cuda.get_rng_state())

    n0 = _lib.launch_count
    fast, rng_fast = run()
    n_fast = _lib.launch_count - n0
    engine.enabled = False
    try:
        n0 = _lib.launch_count
        ref, rng_ref = run()
        n_ref = _lib.launch_count - n0
    finally:
        engine.enabled = True
    assert n_fast > 60 and n_ref > 0
    assert all(torch.equal(a, b) for a, b in zip(rng_fast, rng_ref)), 'the two paths consumed the generators differently'
    # The two paths produce tri-planes that differ at fp32 rounding level (3-pass tensor-core split vs cuDNN); a handful of
    # rays then take a different searchsorted branch in the importance sampling, which moves single pixels by ~1e-3 of the
    # range. Bound the worst pixel loosely and the average tightly.
    for k in ('image_raw', 'image_depth', 'semantic_raw'):
        a, b = fast[k].cpu().numpy(), ref[k].cpu().numpy()
        assert rel_err(a, b) < 5e-3, k
        assert float(np.abs(a - b).mean()) < 1e-3 * float(np.abs(b).mean()) + 1e-7, k     # measured: 1e-5 (cat) .. 5e-4 (car)
    for k in ('image', 'semantic'):                # fp16 super-resolution stacks on both sides
        assert rel_err(fast[k].cpu().numpy(), ref[k].cpu().numpy()) < 2e-2, k
        assert fast[k].shape[-1] == w['img_resolution'] and torch.isfinite(fast[k]).all()


def test_cached_backbone_multi_view_rendering():
    """SURVEY 8(f) rank 1: one latent, several cameras (generate_video.py:57-69): `cache_backbone=True` then
    `use_cached_backbone=True` must reproduce what an uncached call renders for the same camera and noise."""
    import pix2pix3d_b200.training.triplane_cond as tc
    from make_golden import SYNTH_CASES, build_generator
    from pix2pix3d_b200 import _lib
    case = dict(SYNTH_CASES['seg_nrr64'])
    G = build_generator(tc, case).cuda()
    g = load_golden('synthesis_seg_nrr64')
    ws, c = torch.from_numpy(g['ws']).cuda(), torch.from_numpy(g['c']).cuda()
    kw = dict(noise_mode='const', neural_rendering_resolution=case['nrr'])
    with torch.no_grad():
        torch.manual_seed(3)
        first = G.synthesis(ws, c, cache_backbone=True, **kw)
        assert G._last_planes is not None and tuple(G._last_planes.shape[1:]) == (96, 256, 256)
        c2 = c.clone()
        c2[:, 3] += 0.04                                     # a second view
        n0 = _lib.launch_count
        torch.manual_seed(4)
        cached = G.synthesis(ws, c2, use_cached_backbone=True, **kw)
        n_cached = _lib.launch_count - n0
        n0 = _lib.launch_count
        torch.manual_seed(4)
        fresh = G.synthesis(ws, c2, **kw)
        n_fresh = _lib.launch_count - n0
    assert n_cached < n_fresh                                # the backbone was skipped
    for k in fresh:
        assert rel_err(cached[k].cpu().numpy(), fresh[k].cpu().numpy()) < 1e-6, k
    assert (first['image'] - cached['image']).abs().max() > 1e-4
    # the reference API contract: a caller may overwrite _last_planes with its own NCHW tensor
    with torch.no_grad():
        G._last_planes = G._last_planes.clone()
        torch.manual_seed(4)
        again = G.synthesis(ws, c2, use_cached_backbone=True, **kw)
    assert rel_err(again['image'].cpu().numpy(), fresh['image'].cpu().numpy()) < 1e-6


@pytest.mark.parametrize('fast', [True, False])
def test_batched_views_against_one_cached_plane_set(fast):
    """SURVEY 8(f) rank 1, second half: V cameras in ONE call against the plane set cached from one latent
    (`use_cached_backbone=True` with `_last_planes` of batch 1) == V single-camera calls fed the same renderer noise.
    fast=True: engine path (plane_index in the fused kernel, no plane copies); False: generic op-by-op path."""
    import pix2pix3d_b200.training.triplane_cond as tc
    from make_golden import SYNTH_CASES, build_generator
    from pix2pix3d_b200 import engine
    case = dict(SYNTH_CASES['seg_nrr64'])
    G = build_generator(tc, case).cuda()
    g = load_golden('synthesis_seg_nrr64')
    ws, c = torch.from_numpy(g['ws']).cuda(), torch.from_numpy(g['c']).cuda()
    V, nrr = 3, case['nrr']
    cv = c.repeat(V, 1)
    cv[:, 3] += torch.tensor([0.0, 0.05, -0.04], device='cuda')
    cv[:, 7] += torch.tensor([0.0, -0.03, 0.02], device='cuda')
    gen = torch.Generator().manual_seed(7)
    jit = torch.rand(V, nrr * nrr, case['Sc'], 1, generator=gen).cuda()
    u = torch.rand(V * nrr * nrr, case['Sf'], generator=gen).cuda()
    # fp32 super-resolution: split-K / algorithm choices depend on the batch size, which moves fp32 sums by an ulp and, in the
    # fp16 SR stacks, occasionally the fp16 rounding of an activation (1e-3 of the image range); fp32 isolates the geometry
    kw = dict(noise_mode='const', neural_rendering_resolution=nrr, force_fp32=True)

    def replay(fn, j, uu):
        it = iter([j, uu])
        o_like, o_rand = torch.rand_like, torch.rand
        torch.rand_like, torch.rand = (lambda x, *a, **k: next(it)), (lambda *a, **k: next(it))
        try:
            return fn()
        finally:
            torch.rand_like, torch.rand = o_like, o_rand

    engine.enabled = fast
    try:
        with torch.no_grad():
            replay(lambda: G.synthesis(ws, c, cache_backbone=True, **kw), jit[:1], u[:nrr * nrr])
            assert G._last_planes.shape[0] == 1
            batched = replay(lambda: G.synthesis(ws.expand(V, -1, -1), cv, use_cached_backbone=True, **kw), jit, u)
            singles = [replay(lambda v=v: G.synthesis(ws, cv[v:v + 1], use_cached_backbone=True, **kw), jit[v:v + 1],
                              u[v * nrr * nrr:(v + 1) * nrr * nrr]) for v in range(V)]
    finally:
        engine.enabled = True
    for k in batched:
        assert batched[k].shape[0] == V
        want = torch.cat([s[k] for s in singles]).float().cpu().numpy()
        # image_depth is clamped to the depth range of the CALL's batch (ray_marcher.py:50): compare where no clamp is active
        tol = 1e-3 if k == 'image_depth' else 2e-5
        assert rel_err(batched[k].float().cpu().numpy(), want) < tol, k
    assert (batched['image'][0] - batched['image'][1]).abs().max() > 1e-4


@pytest.mark.parametrize('res,in_ch', [(64, 6), (256, 1)])
def test_encoder_engine_matches_generic_path(res, in_ch):
    """Label-map Encoder (triplane_cond.py:66-196) on the tensor-core path -- static-weight 3x3 convs, FIR + stride-2 convs
    (TMA element strides), resnet skip added in the epilogue -- against the op-by-op fp32 formulation."""
    from pix2pix3d_b200 import _lib, engine
    from pix2pix3d_b200.training.triplane_cond import Encoder
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.manual_seed(31)
    enc = Encoder(img_resolution=res, img_channels=in_ch, model_kwargs={'num_ws': 7, 'w_dim': 512, 'output_mode': 'W+'}).cuda()
    enc.requires_grad_(False)
    with torch.no_grad():
        for n, p in enc.named_parameters():
            if n.endswith('.bias'):
                p.copy_(torch.randn_like(p) * 0.2)
    if in_ch > 1:
        lab = torch.randint(0, in_ch, (3, res, res), device='cuda')
        img = torch.nn.functional.one_hot(lab, in_ch).permute(0, 3, 1, 2).float()
    else:
        img = (torch.rand(3, 1, res, res, device='cuda') < 0.1).float() * 2 - 1
    n0 = _lib.launch_count
    with torch.no_grad():
        fast = enc(img)['ws']
    assert _lib.launch_count - n0 > 5 * len(enc.block_resolutions)
    engine.enabled = False
    try:
        with torch.no_grad():
            ref = enc(img)['ws']
    finally:
        engine.enabled = True
    assert fast.shape == ref.shape == (3, 7, 512)
    assert rel_err(fast.cpu().numpy(), ref.cpu().numpy()) < 2e-4
