"""Unconditional EG3D-style tri-plane generator pieces used by pix2pix3D.

Mirror of the reference's training/triplane.py: `OSGDecoder` (:112-135) is what `triplane_cond.TriPlaneGenerator`
decodes with; `TriPlaneGenerator` (:19-108) is the unconditional variant (mapping takes (z, c)).
"""
import torch

from .. import dnnlib, native
from ..torch_utils import persistence
from .networks_stylegan2 import FullyConnectedLayer
from .networks_stylegan2 import Generator as StyleGAN2Backbone
from .volumetric_rendering.ray_sampler import RaySampler
from .volumetric_rendering.renderer import ImportanceRenderer


def _mipnerf_sigmoid(x):
    return torch.sigmoid(x) * (1 + 2 * 0.001) - 0.001


def _decoder_mlp(n_features, hidden, out_dim, lr_mul):
    return torch.nn.Sequential(
        FullyConnectedLayer(n_features, hidden, lr_multiplier=lr_mul),
        torch.nn.Softplus(),
        FullyConnectedLayer(hidden, out_dim, lr_multiplier=lr_mul))


class OSGDecoder(torch.nn.Module):
    """mean over planes -> FC(32,64) -> softplus -> FC(64,1+C): sigma = ch 0, rgb = sigmoid(rest) (:112-135)."""

    def __init__(self, n_features, options):
        super().__init__()
        self.hidden_dim = 64
        self.net = _decoder_mlp(n_features, self.hidden_dim, 1 + options['decoder_output_dim'], options['decoder_lr_mul'])

    def forward(self, sampled_features, ray_directions):
        if native.decoder_mlp_supported(self, sampled_features):      # CUDA: fused forward / backward kernels
            return native.decoder_mlp(self, sampled_features)
        x = sampled_features.mean(1)
        n, m, c = x.shape
        x = self.net(x.view(n * m, c)).view(n, m, -1)
        return {'rgb': _mipnerf_sigmoid(x[..., 1:]), 'sigma': x[..., 0:1]}


def render_to_images(gen, ws, c, neural_rendering_resolution, update_emas, cache_backbone, use_cached_backbone, synthesis_kwargs):
    """Shared front half of every `synthesis`: rays -> backbone planes -> volume rendering -> raw feature image.
    Returns (feature_image [N,C,H,W], depth_image [N,1,H,W]). Reference: triplane_cond.py:1020-1050."""
    cam2world = c[:, :16].view(-1, 4, 4)
    intrinsics = c[:, 16:25].view(-1, 3, 3)
    if neural_rendering_resolution is None:
        neural_rendering_resolution = gen.neural_rendering_resolution
    else:
        gen.neural_rendering_resolution = neural_rendering_resolution
    ray_origins, ray_directions = gen.ray_sampler(cam2world, intrinsics, neural_rendering_resolution)
    n = ray_origins.shape[0]
    if use_cached_backbone and gen._last_planes is not None:
        planes = gen._last_planes
    else:
        planes = gen.backbone.synthesis(ws, update_emas=update_emas, **synthesis_kwargs)
    if cache_backbone:
        gen._last_planes = planes
    planes = planes.view(len(planes), 3, 32, planes.shape[-2], planes.shape[-1])
    if use_cached_backbone and planes.shape[0] == 1 and n > 1:
        # extension of the cached-backbone call pattern (generate_video.py:57-69 renders 120 views of one latent, one call per
        # view): a batch of cameras against ONE cached plane set; identical to n calls with one camera each
        planes = planes.expand(n, -1, -1, -1, -1)
    feats, depth, _ = gen.renderer(planes, gen.decoder, ray_origins, ray_directions, gen.rendering_kwargs)
    h = w = gen.neural_rendering_resolution
    feature_image = feats.permute(0, 2, 1).reshape(n, feats.shape[-1], h, w).contiguous()
    depth_image = depth.permute(0, 2, 1).reshape(n, 1, h, w)
    return feature_image, depth_image


def fast_synthesis(gen, ws, c, neural_rendering_resolution, cache_backbone, use_cached_backbone, synthesis_kwargs):
    """Whole-generator tensor-core / fused-render path (pix2pix3d_b200/engine.py); None when it does not apply."""
    if ws.device.type != 'cuda':
        return None
    from .. import engine
    if neural_rendering_resolution is not None:
        gen.neural_rendering_resolution = neural_rendering_resolution
    if not engine.generator_supported(gen, ws, c, synthesis_kwargs, use_cached_backbone):
        return None
    return engine.generator_synthesis(gen, ws, c, cache_backbone=cache_backbone, use_cached_backbone=use_cached_backbone,
                                      noise_mode=synthesis_kwargs.get('noise_mode', 'random'),
                                      force_fp32=bool(synthesis_kwargs.get('force_fp32', False)))


def _sr_kwargs(synthesis_kwargs):
    return {k: v for k, v in synthesis_kwargs.items() if k != 'noise_mode'}


def query_planes(gen, ws, update_emas, synthesis_kwargs):
    """The tri-planes [B,3,32,H,W] that `query_points` queries (also used by pix2pix3d_b200.mesh.sigma_grid)."""
    planes = gen.backbone.synthesis(ws, update_emas=update_emas, **synthesis_kwargs)
    return planes.view(len(planes), 3, 32, planes.shape[-2], planes.shape[-1])


def query_points(gen, coordinates, directions, ws, update_emas, synthesis_kwargs):
    """Backbone + `renderer.run_model` at arbitrary 3-D points (reference triplane_cond.py:1070-1074)."""
    planes = query_planes(gen, ws, update_emas, synthesis_kwargs)
    return gen.renderer.run_model(planes, gen.decoder, coordinates, directions, gen.rendering_kwargs)


@persistence.persistent_class
class TriPlaneGenerator(torch.nn.Module):
    def __init__(self, z_dim, c_dim, w_dim, img_resolution, img_channels, sr_num_fp16_res=0, mapping_kwargs={},
                 rendering_kwargs={}, sr_kwargs={}, **synthesis_kwargs):
        super().__init__()
        self.z_dim = z_dim
        self.c_dim = c_dim
        self.w_dim = w_dim
        self.img_resolution = img_resolution
        self.img_channels = img_channels
        self.renderer = ImportanceRenderer()
        self.ray_sampler = RaySampler()
        self.backbone = StyleGAN2Backbone(z_dim, c_dim, w_dim, img_resolution=256, img_channels=32 * 3,
                                          mapping_kwargs=mapping_kwargs, **synthesis_kwargs)
        self.superresolution = dnnlib.util.construct_class_by_name(
            class_name=rendering_kwargs['superresolution_module'], channels=32, img_resolution=img_resolution,
            sr_num_fp16_res=sr_num_fp16_res, sr_antialias=rendering_kwargs['sr_antialias'], **sr_kwargs)
        self.decoder = OSGDecoder(32, {'decoder_lr_mul': rendering_kwargs.get('decoder_lr_mul', 1), 'decoder_output_dim': 32})
        self.neural_rendering_resolution = 64
        self.rendering_kwargs = rendering_kwargs
        self._last_planes = None

    def mapping(self, z, c, truncation_psi=1, truncation_cutoff=None, update_emas=False):
        if self.rendering_kwargs['c_gen_conditioning_zero']:
            c = torch.zeros_like(c)
        return self.backbone.mapping(z, c * self.rendering_kwargs.get('c_scale', 0), truncation_psi=truncation_psi,
                                     truncation_cutoff=truncation_cutoff, update_emas=update_emas)

    def synthesis(self, ws, c, neural_rendering_resolution=None, update_emas=False, cache_backbone=False,
                  use_cached_backbone=False, **synthesis_kwargs):
        fast = fast_synthesis(self, ws, c, neural_rendering_resolution, cache_backbone, use_cached_backbone, synthesis_kwargs)
        if fast is not None:
            return fast
        feature_image, depth_image = render_to_images(self, ws, c, neural_rendering_resolution, update_emas,
                                                      cache_backbone, use_cached_backbone, synthesis_kwargs)
        rgb_image = feature_image[:, :3]
        sr_image = self.superresolution(rgb_image, feature_image, ws,
                                        noise_mode=self.rendering_kwargs['superresolution_noise_mode'],
                                        **_sr_kwargs(synthesis_kwargs))
        return {'image': sr_image, 'image_raw': rgb_image, 'image_depth': depth_image}

    def sample(self, coordinates, directions, z, c, truncation_psi=1, truncation_cutoff=None, update_emas=False, **synthesis_kwargs):
        ws = self.mapping(z, c, truncation_psi=truncation_psi, truncation_cutoff=truncation_cutoff, update_emas=update_emas)
        return query_points(self, coordinates, directions, ws, update_emas, synthesis_kwargs)

    def sample_mixed(self, coordinates, directions, ws, truncation_psi=1, truncation_cutoff=None, update_emas=False, **synthesis_kwargs):
        return query_points(self, coordinates, directions, ws, update_emas, synthesis_kwargs)

    def forward(self, z, c, truncation_psi=1, truncation_cutoff=None, neural_rendering_resolution=None, update_emas=False,
                cache_backbone=False, use_cached_backbone=False, **synthesis_kwargs):
        ws = self.mapping(z, c, truncation_psi=truncation_psi, truncation_cutoff=truncation_cutoff, update_emas=update_emas)
        return self.synthesis(ws, c, update_emas=update_emas, neural_rendering_resolution=neural_rendering_resolution,
                              cache_backbone=cache_backbone, use_cached_backbone=use_cached_backbone, **synthesis_kwargs)


def mark_first_order(*classes):
    """The generator is differentiated once per pass in every loss of the reference (training/loss.py: no path-length or other
    second-order term touches G): run its `mapping` / `synthesis` / `sample` / `sample_mixed` inside
    `native_conv.first_order()`, which lets the fp32 training convolutions use the tcgen05 implicit GEMM for forward and input
    gradient (torch_utils/ops/native_conv.py). The discriminators never enter such a region (R1 differentiates twice)."""
    import functools
    from ..torch_utils.ops import native_conv
    for cls in classes:
        for name in ('mapping', 'synthesis', 'sample', 'sample_mixed'):
            fn = cls.__dict__.get(name) or getattr(cls, name, None)
            if fn is None or getattr(fn, '_p3d_first_order', False):
                continue

            def wrapped(self, *args, __fn=fn, **kwargs):
                with native_conv.first_order():
                    return __fn(self, *args, **kwargs)
            functools.update_wrapper(wrapped, fn)
            wrapped._p3d_first_order = True
            setattr(cls, name, wrapped)


mark_first_order(TriPlaneGenerator)
