/*
 * p3d.h -- C-ABI of libp3d.so, the sm_100a replacement for pix2pix3D's render + StyleGAN2-op hot path.
 *
 * Every entry point takes plain device pointers, sizes and a CUDA stream; the caller owns all
 * memory (allocates outputs, keeps inputs alive until the stream reaches the call). Nothing is
 * retained past return and there is no global mutable state (no environment switches, no cached device properties: every decision follows from the arguments) (the reference's __constant__ filter
 * buffer, torch_utils/ops/filtered_lrelu.cu:81-82, is deliberately not reproduced).
 *
 * Return value: 0 = ok, <0 = p3d status (P3D_UNSUPPORTED: "no kernel for this configuration",
 * the analogue of rc=-1 in torch_utils/ops/filtered_lrelu.cpp:56-60), >0 = cudaError_t of the launch.
 *
 * Each declaration cites the reference interface it replaces (paths relative to the reference repo).
 */
#ifndef P3D_H_
#define P3D_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef void* p3d_stream_t; /* cudaStream_t */

enum {
    P3D_OK          = 0,
    P3D_UNSUPPORTED = -1,
    P3D_BAD_ARG     = -2,
};

enum { /* element types of activation tensors */
    P3D_F32 = 0,
    P3D_F16 = 1,
    P3D_F64 = 2,
};

/* Library ABI version (bumped on any signature change) and build info. */
int         p3d_abi_version(void);
const char* p3d_build_info(void);
const char* p3d_status_string(int status);

/* ---------------------------------------------------------------------------------------------
 * Renderer (training/volumetric_rendering/*)
 * ------------------------------------------------------------------------------------------- */

/* RaySampler.forward -- training/volumetric_rendering/ray_sampler.py:24-62.
 * cam2world [B,16] row-major 4x4, intrinsics [B,9] row-major 3x3 (normalised),
 * origins/dirs [B,res*res,3]; ray m = row*res + col. */
int p3d_ray_sampler(const float* cam2world, const float* intrinsics, int B, int res,
                    float* origins, float* dirs, p3d_stream_t stream);

/* Layout change for the tri-plane gather: [N,C,H,W] (backbone output viewed as N = B*3 planes,
 * training/triplane_cond.py:1042) -> [N,H,W,C] so that one bilinear tap of all C=32 channels is a
 * single 128-byte line. */
int p3d_planes_to_channels_last(const float* planes_nchw, float* planes_nhwc, int N, int C, int H, int W,
                                p3d_stream_t stream);

/* Decoder description: OSGDecoder (training/triplane.py:112-135), OSGDecoder_semantic
 * (training/triplane_cond.py:859-887), OSGDecoder_semantic_lateSeparate (:926-970).
 * Every net is FC(32->64) -> Softplus -> FC(64->33) (networks_stylegan2.py:96-127). */
typedef struct {
    int32_t n_nets;          /* 1 or 2 */
    int32_t sigma_net;       /* which net's output channel 0 is sigma */
    uint32_t sigmoid_mask[2];/* bit o set: colour output o (0..31) of that net gets sigmoid*1.002-0.001 */
    /* raw parameters as stored in the module (not yet multiplied by the equalised-lr gains) */
    const float* w1[2];      /* [64,32] */
    const float* b1[2];      /* [64] */
    const float* w2[2];      /* [33,64] */
    const float* b2[2];      /* [33] */
    float w1_gain[2], b1_gain[2], w2_gain[2], b2_gain[2]; /* FullyConnectedLayer.weight_gain / bias_gain */
} p3d_decoder_t;

#define P3D_DECODER_PACKED_FLOATS (2 * 4260)
/* Multiplies by the gains exactly as FullyConnectedLayer.forward does (networks_stylegan2.py:111-119)
 * and writes the kernel-side layout into packed[P3D_DECODER_PACKED_FLOATS]. */
int p3d_pack_decoder(const p3d_decoder_t* dec, float* packed, p3d_stream_t stream);

typedef struct {
    /* inputs */
    const float* planes_nhwc;    /* [B,3,H,W,32] fp32 (dense), or any layout with 32 contiguous channels described by plane_strides */
    const float* ray_origins;    /* [B,R,3] */
    const float* ray_dirs;       /* [B,R,3] */
    const float* depths_coarse;  /* [B,R,Sc]  (sample_stratified output, renderer.py:169-192) */
    const float* u_importance;   /* [B*R,Sf]  uniform draws of sample_pdf (renderer.py:237); unused if Sf==0 */
    const float* decoder_packed; /* from p3d_pack_decoder */
    int32_t n_nets, sigma_net;
    uint32_t sigmoid_mask[2];
    int32_t B, R, H, W, Sc, Sf;
    float   coord_scale;         /* 2/box_warp (renderer.py:61) */
    int32_t white_back;          /* rendering_options.get('white_back') (ray_marcher.py:52) */
    /* outputs */
    float* out_feat;             /* [B,R,32*n_nets]  composite_rgb*2-1 */
    float* out_depth;            /* [B,R]            clamped to the global [min,max] of all depths */
    float* out_wsum;             /* [B,R]            weights.sum(2) (renderer.py:140) */
    /* optional stage outputs for parity tests (NULL to skip) */
    float*   dbg_weights_coarse; /* [B,R,Sc-1]   MipRayMarcher2 weights of the coarse pass */
    float*   dbg_depths_fine;    /* [B,R,Sf] */
    int32_t* dbg_inds;           /* [B,R,Sf]     searchsorted(cdf,u,right=True) (renderer.py:240) */
    int32_t* dbg_perm;           /* [B,R,Sc+Sf]  sort permutation over cat(coarse,fine) (renderer.py:162) */
    float*   dbg_weights_final;  /* [B,R,Sc+Sf-1] */
    /* scratch: 4 x uint32, zeroed by the callee on the stream before launch */
    uint32_t* workspace;
    /* element strides {image, plane, pixel} of planes_nhwc; rows are W pixels apart. All zero = dense [B,3,H,W,32].
     * {H*W*96, 32, 96} reads the backbone's NHWC [B,H,W,96] output in place (p3d_render_fwd_tc only; p3d_render_fwd
     * returns P3D_UNSUPPORTED for non-dense planes). */
    int64_t plane_strides[3];
    /* p3d_render_fwd_tc only: 0 = one 8-ray tile per CTA shared by its three 128-row groups (render_tc.cu); 1 = ray-pair
     * ownership, groups never synchronise with each other (render_tc2.cu; Sc, Sf <= 64, else P3D_UNSUPPORTED). Same results. */
    int32_t tc_variant;
    /* How the coarse depths are obtained (ImportanceRenderer.sample_stratified, renderer.py:169-192):
     *   0  depths_coarse holds them (any sampling the caller computed);
     *   1  scalar ray limits (:187-190): d[k] = depth_table[k] + jitter * depth_delta, depth_table = torch.linspace(ray_start,
     *      ray_end, Sc), depth_delta = (ray_end - ray_start) / (Sc - 1), jitter = the torch.rand_like draw [B,R,Sc];
     *   2  per-ray limits (`ray_start == 'auto'`, :91-97, :181-186 with math_utils.linspace :101-118):
     *      d[k] = ray_start[r] + depth_table[k] * (ray_end[r] - ray_start[r]) + jitter * ((ray_end[r] - ray_start[r]) * depth_delta),
     *      depth_table = arange(Sc) / (Sc - 1), depth_delta = fp32(1) / fp32(Sc - 1) (torch's CUDA `tensor / scalar` multiplies
     *      by the reciprocal).
     * Products and sums are rounded separately, in the reference's order, so the depths equal the torch results bit for bit.
     * Neutral at zero: older callers that never set these keep mode 0. */
    int32_t depth_mode;
    const float* jitter;         /* [B,R,Sc]  modes 1, 2 */
    const float* depth_table;    /* [Sc]      modes 1, 2 */
    const float* ray_start;      /* [B,R]     mode 2 */
    const float* ray_end;        /* [B,R]     mode 2 */
    float   depth_delta;         /* modes 1, 2 */
    int32_t reserved1;
    /* Optional [B] plane-set index per image: rays of image b gather from plane set plane_index[b] (NULL: b). Lets V camera
     * views of one latent (applications/generate_video.py:57-69) share ONE resident plane set: planes batch 1, B = V. */
    const int32_t* plane_index;
} p3d_render_args_t;

/* math_utils.get_ray_limits_box (training/volumetric_rendering/math_utils.py:46-98): slab test of N rays against the cube of
 * side `box_side_length` centred at the origin. t_near / t_far [N]; (-1, -2) for rays that miss. */
int p3d_ray_limits_box(const float* rays_o, const float* rays_d, int64_t N, float box_side_length, float* t_near, float* t_far,
                       p3d_stream_t stream);

/* ImportanceRenderer.forward for scalar ray limits -- training/volumetric_rendering/renderer.py:88-140:
 * coarse sample+decode -> MipRayMarcher2 weights (ray_marcher.py:25-57) -> sample_importance (:194-253)
 * -> fine sample+decode -> unify_samples (:157-167) -> final ray march, as one persistent kernel. */
int p3d_render_fwd(const p3d_render_args_t* args, p3d_stream_t stream);

/* Tensor-core variant of the same pipeline (decoder MLP on tcgen05 with fp16 hi/lo split operands and fp32 TMEM
 * accumulation; pix2pix3d_b200/csrc/render_tc.cu). Takes the decoder image of p3d_pack_decoder_tc. Returns
 * P3D_UNSUPPORTED when Sc or Sf is not a multiple of 8 (callers then use p3d_render_fwd). */
#define P3D_DECODER_TC_PACKED_BYTES (65536 + 324 * 4)
int p3d_pack_decoder_tc(const p3d_decoder_t* dec, void* packed, p3d_stream_t stream);
int p3d_render_fwd_tc(const p3d_render_args_t* args, p3d_stream_t stream);

/* ImportanceRenderer.run_model -- renderer.py:142-148 (sample_from_planes :55-65 + decoder):
 * coords [B,M,3] -> rgb [B,M,32*n_nets], sigma [B,M]. density_noise is added by the host wrapper. */
int p3d_run_model(const float* planes_nhwc, const float* coords, const float* decoder_packed,
                  int n_nets, int sigma_net, const uint32_t sigmoid_mask[2],
                  int B, int M, int H, int W, float coord_scale,
                  float* out_rgb, float* out_sigma, p3d_stream_t stream);

/* The same query with the decoder MLP on tcgen05 (pix2pix3d_b200/csrc/query_tc.cu): the call behind
 * TriPlane*Generator.sample / sample_mixed (triplane_cond.py:1063-1074), e.g. the 512^3 sigma grid of
 * applications/extract_mesh.py:60-81. decoder_tc_packed is the image of p3d_pack_decoder_tc; plane_strides as in
 * p3d_render_args_t (NULL or all zero = dense [B,3,H,W,32]). out_rgb may be NULL: densities only (what extract_mesh
 * keeps), which skips layer 2 of the decoder and the colour writes. */
int p3d_run_model_tc(const float* planes_nhwc, const int64_t plane_strides[3], const float* coords,
                     const void* decoder_tc_packed, int n_nets, int sigma_net, const uint32_t sigmoid_mask[2],
                     int B, int64_t M, int H, int W, float coord_scale,
                     float* out_rgb, float* out_sigma, p3d_stream_t stream);

/* sample_from_planes alone -- renderer.py:55-65: features [B,3,M,32] (the reference's output layout). */
int p3d_sample_from_planes(const float* planes_nhwc, const float* coords, int B, int M, int H, int W,
                           float coord_scale, float* out_features, p3d_stream_t stream);

/* Gradient of sample_from_planes w.r.t. the planes (what autograd derives from F.grid_sample at renderer.py:64):
 * grad_features [B,3,M,32] -> grad_planes_nhwc [B,3,H,W,32] (zeroed here, then the bilinear taps are scattered with
 * vector atomics). Coordinates carry no gradient in the reference's pipeline. */
int p3d_sample_from_planes_bwd(const float* grad_features, const float* coords, int B, int64_t M, int H, int W,
                               float coord_scale, float* grad_planes_nhwc, p3d_stream_t stream);

/* OSG decoder MLP of the gradient-requiring passes (training/triplane.py:112-135, triplane_cond.py:859-924): for every point
 *   x = mean over the 3 planes of feats [N,3,M,32];  h = softplus(w1 x + b1);  o = w2 h + b2   (w1 [64,32], w2 [33,64], runtime
 *   gains of FullyConnectedLayer already applied by the caller, networks_stylegan2.py:111-119; Softplus(beta 1, threshold 20))
 *   out_sigma [N*M] = o[0];  out_rgb [N*M,32][k] = bit k of sigmoid_mask ? sigmoid(o[1+k]) * 1.002 - 0.001 : o[1+k].
 * out_pre (optional, [N*M,64]): the hidden pre-activations w1 x + b1, which p3d_decoder_mlp_bwd consumes (pass NULL when no
 * gradient will be taken). One launch instead of mean + addmm + softplus + addmm + slices + sigmoid + cat. */
int p3d_decoder_mlp_fwd(const float* feats, int64_t N, int64_t M, const float* w1, const float* b1, const float* w2,
                        const float* b2, uint32_t sigmoid_mask, float* out_rgb, float* out_sigma, float* out_pre,
                        p3d_stream_t stream);

/* First-order backward of p3d_decoder_mlp_fwd (what autograd derives from the module's forward): g_rgb [N*M,32] / g_sigma [N*M]
 * (either may be NULL = zeros) -> g_feats [N,3,M,32] and g_params [4257] = dL/dw1 [64,32] | dL/db1 [64] | dL/dw2 [33,64] |
 * dL/db2 [33]. pre / out_rgb: the forward's out_pre and out_rgb (nothing of the forward GEMMs is recomputed; the sigmoid
 * derivative follows from the output). Parameter gradients are accumulated per CTA and added in a fixed order (deterministic).
 * workspace: fp32 scratch of at least p3d_decoder_mlp_bwd_workspace_floats() elements. */
int p3d_decoder_mlp_bwd_workspace_floats(void);
int p3d_decoder_mlp_bwd(const float* feats, const float* pre, const float* out_rgb, int64_t N, int64_t M, const float* w1, const float* b1, const float* w2,
                        const float* b2, uint32_t sigmoid_mask, const float* g_rgb, const float* g_sigma, float* g_feats,
                        float* g_params, float* workspace, int64_t workspace_floats, p3d_stream_t stream);

/* MipRayMarcher2.run_forward on explicit tensors -- ray_marcher.py:25-57.
 * colors [N,S,Cc], densities [N,S], depths [N,S]; out_rgb [N,Cc], out_depth [N] (clamped),
 * out_weights [N,S-1]. N = B*R rays. */
int p3d_ray_march(const float* colors, const float* densities, const float* depths,
                  int N, int S, int Cc, int white_back,
                  float* out_rgb, float* out_depth, float* out_weights,
                  uint32_t* workspace, p3d_stream_t stream);

/* First-order backward of MipRayMarcher2.run_forward (ray_marcher.py:25-57) w.r.t. colours and densities.
 * grad_rgb [N,Cc]; grad_depth [N] or NULL; grad_weights [N,S-1] or NULL; depth_range[2] = {min, max} of all depths (device
 * pointer; needed with grad_depth: the clamp at :50 passes the gradient only inside the range, nan_to_num only where the
 * composite is finite). grad_colors [N,S,Cc], grad_densities [N,S]. Rays whose upstream depth gradient is exactly zero
 * skip the depth term (autograd would form 0/0 there when the weight sum is zero). */
int p3d_ray_march_bwd(const float* colors, const float* densities, const float* depths, const float* grad_rgb,
                      const float* grad_depth, const float* grad_weights, const float* depth_range, int N, int S,
                      int Cc, int white_back, float* grad_colors, float* grad_densities, p3d_stream_t stream);

/* sample_importance + sample_pdf -- renderer.py:194-253. z_vals [N,S], weights [N,S-1], u [N,Sf];
 * out_samples [N,Sf], out_inds [N,Sf] (may be NULL). */
int p3d_sample_importance(const float* z_vals, const float* weights, const float* u,
                          int N, int S, int Sf, float* out_samples, int32_t* out_inds, p3d_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * StyleGAN2 custom ops (torch_utils/ops/*)
 * ------------------------------------------------------------------------------------------- */

/* bias_act plugin -- torch_utils/ops/bias_act.cpp:36-94, kernel bias_act.cu:27-151.
 * y = clamp(act(x + b[(i/step_b) % size_b]) * gain). grad = 0/1/2 selects forward / first / second
 * order as in the reference; xref/yref/dy may be NULL when unused. act: 1..9 = linear, relu, lrelu,
 * tanh, sigmoid, elu, selu, softplus, swish (bias_act.py:23-33 cuda_idx). clamp < 0 disables. */
int p3d_bias_act(const void* x, const void* b, const void* xref, const void* yref, const void* dy, void* y,
                 int dtype, int grad, int act, float alpha, float gain, float clamp,
                 int64_t size_x, int size_b, int64_t step_b, p3d_stream_t stream);

/* upfirdn2d plugin -- torch_utils/ops/upfirdn2d.cpp:20-102, kernels upfirdn2d.cu:33-204.
 * x [N,C,inH,inW] with element strides x_stride[4] (n,c,h,w); f [fH,fW] fp32 contiguous (already
 * expanded to 2-D); y [N,C,outH,outW] with strides y_stride[4]. */
int p3d_upfirdn2d(const void* x, const float* f, void* y, int dtype,
                  const int32_t x_size[4], const int64_t x_stride[4],
                  const int32_t y_size[4], const int64_t y_stride[4],
                  int fw, int fh, int upx, int upy, int downx, int downy,
                  int padx0, int pady0, int flip, float gain, p3d_stream_t stream);

/* F.interpolate(x, size, mode='bilinear', align_corners=False, antialias=...) -- the resize of
 * Superresolution*.forward (training/superresolution.py:315-319) and `filtered_resizing`
 * (training/dual_discriminator.py:86-102): separable triangle filter of support max(in/out, 1) with per-output
 * renormalisation at the borders (antialias != 0), or the two clamped taps of plain bilinear interpolation.
 * x [planes, in_h, in_w] -> y [planes, out_h, out_w], dense, dtype P3D_F32 / P3D_F16 / P3D_F64.
 * transposed != 0 applies the adjoint (the op's backward): x is then [planes, out_h, out_w] (gradient w.r.t. the
 * output) and y [planes, in_h, in_w]; higher orders alternate between the two. */
int p3d_resize_bilinear(const void* x, void* y, int dtype, int64_t planes, int in_h, int in_w, int out_h, int out_w,
                        int antialias, int transposed, p3d_stream_t stream);

/* cross_entropy2d -- training/loss_utils.py:4-18 (after its optional label resize), called by training/loss.py:611-616:
 * logits [N,C,H,W] fp32 (read in place, no [N*H*W,C] copy), target [N,H,W] int64, class_weight [C] fp32 or NULL.
 * loss[0] = sum_i w[t_i] (logsumexp(x_i) - x_i[t_i]) / sum_i w[t_i] over the pixels with t_i != ignore_index
 * (F.cross_entropy, reduction='mean'); sum_w[0] = the denominator, kept for the backward. A target outside [0,C) makes
 * the loss NaN. workspace: P3D_CE_WORKSPACE_DOUBLES doubles; partial sums are combined in a fixed order (deterministic). */
#define P3D_CE_WORKSPACE_DOUBLES 2048
int p3d_cross_entropy2d_fwd(const float* logits, const int64_t* target, const float* class_weight, int N, int C,
                            int64_t HW, int64_t ignore_index, float* loss, float* sum_w, double* workspace,
                            p3d_stream_t stream);
/* grad_logits [N,C,H,W] = grad_loss[0] * w[t] * (softmax(x) - onehot(t)) / sum_w[0]; zero at ignored pixels. */
int p3d_cross_entropy2d_bwd(const float* logits, const int64_t* target, const float* class_weight,
                            const float* grad_loss, const float* sum_w, int N, int C, int64_t HW,
                            int64_t ignore_index, float* grad_logits, p3d_stream_t stream);

/* Fused epilogue of an up=2 modulated conv (networks_stylegan2.py:324-331 + conv2d_resample.py:128):
 * y = clamp(lrelu(upfirdn2d(x, f, pad, gain=up^2) [* dcoef[n,c]] + noise[h,w]*noise_strength + b[c]) * act_gain).
 * One read of x, one write of y instead of three passes. Any of dcoef/noise/b may be NULL. */
int p3d_fir_bias_act(const void* x, const float* f, const float* dcoef, const float* noise, const void* b, void* y,
                     int dtype, const int32_t x_size[4], const int32_t y_size[4],
                     int fw, int fh, int padx0, int pady0, float fir_gain,
                     int act, float alpha, float act_gain, float clamp,
                     int64_t noise_stride_n, p3d_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Tensor-core convolution path (training/networks_stylegan2.py:34-91 modulated_conv2d,
 * torch_utils/ops/conv2d_resample.py:48-143; the reference bottoms out in cuDNN through conv2d_gradfix.py:37-45)
 *
 * Activations of this path are NHWC fp16. A "split" tensor is a pair of fp16 planes (hi, lo) with x = hi + lo,
 * laid out [2][B][H][W][C]; fp32 layers of the reference (the tri-plane backbone) run on split tensors with three
 * tensor-core passes, fp16 layers (super-resolution) on single-plane tensors with one pass.
 * ------------------------------------------------------------------------------------------- */
typedef struct {
    const void* x;            /* [x_planes][B][H][W][C] fp16, C % 64 == 0 */
    const void* w;            /* [w_planes][Bw][Cout_padded][n_kblocks*C] fp16, K-major; Bw = B (modulated) or 1 */
    int32_t x_planes, w_planes, B, Bw, H, W, C, Cout, Cout_padded;
    int32_t n_kblocks;        /* number of C-sized K blocks stored in w (9 for a 3x3 kernel) */
    int32_t n_taps;           /* taps used by this launch (<= 9) */
    int8_t  tap_dy[9], tap_dx[9], tap_k[9];   /* input offset of each tap and its K block in w */
    int32_t split;            /* 0: one pass (plane 0 x plane 0); 1: hi*hi + hi*lo + lo*hi */
    int32_t gH, gW;           /* grid of output positions computed by this launch */
    int32_t oH, oW, sy, oy, sx, ox;   /* output tensor size and the affine map grid -> output (Y = y*sy + oy) */
    void* y; void* y_lo;      /* output NHWC; y_lo only for out_mode 1 */
    int32_t y_cstride, y_coff;/* channel stride of the output tensor and first channel written */
    int32_t out_mode;         /* 0 fp16, 1 fp16 split (hi, lo), 2 fp32, 3 fp32 accumulate (y += result) */
    const float* bias;        /* [Cout] or NULL */
    const float* noise;       /* [oH*oW] (already multiplied by noise_strength) or NULL */
    const float* dscale;      /* [B*Cout] per-sample output scale (demodulation) or NULL */
    int32_t act;              /* 1 linear, 3 lrelu */
    float alpha, gain, clamp; /* activation slope, output gain, clamp (<0: none) */
    float acc_scale;          /* multiplies the accumulator first (undoes the power-of-two weight scaling) */
    /* fused ToRGB tail (networks_stylegan2.py:452-458): when up_prev != NULL the launch writes
     *   y = upsample2d(up_prev, up_filter) + result     (result rounded to fp16 first when round16, as fp16 blocks do)
     * with up_prev [B, oH/2, oW/2, Cout] fp32 NHWC; out_mode must be 2; out_nchw writes y as [B, Cout, oH, oW]. */
    const float* up_prev; const float* up_filter;
    int32_t round16, out_nchw;
    /* strided convolutions (conv2d_resample.py:108-111, the down=2 layers of DiscriminatorBlock / the label-map Encoder):
     * output pixel (y, x) reads input pixels (stride*y + dy, stride*x + dx); stride 0/1 = dense, 2 supported. */
    int32_t stride;
    int32_t launch_flags;     /* A/B switches, results unchanged: bit 0 = never the persistent kernel, bit 1 = never CTA pairs */
    /* resnet skip connection (networks_stylegan2.py:524-528): fp32 [B, oH, oW, Cout] (32-byte aligned, Cout % 8 == 0 for the
     * vector path) added after activation / gain / clamp; out_mode 0-2 with the identity output map. NULL = none. */
    const float* residual;
    void* splitk_scratch;     /* optional fp32 scratch (32-byte aligned): lets launches much smaller than the machine split */
    int64_t splitk_scratch_bytes; /* their K range over up to 16 CTAs each (deterministic two-kernel reduction); NULL/0 = never */
    /* noise_mode='random' (networks_stylegan2.py:320-321): noise is [B, oH*oW], one image per sample; elements between
     * consecutive samples. 0 = the single [oH*oW] image of noise_mode='const' shared by the batch. */
    int64_t noise_batch_stride;
    /* Fused 1x1 ToRGB of the NEXT layer (ABI 5; all zero = off): a launch whose single channel tile holds every output channel
     * (Cout == Cout_padded <= 128, a multiple of 32; out_mode 0; 1:1 output map; persistent kernel) also evaluates, per pixel,
     *   rgb[c] = round16(clamp(dot(x_out[:], rgb_w[b][c][:]) * rgb_acc_scale + rgb_bias[c]))       c < rgb_cout <= 8
     * on the fp16-rounded outputs it has in registers, and writes rgb_out [B, rgb_cout, oH, oW] (fp32 NCHW) =
     * upsample2d(rgb_prev [B, oH/2, oW/2, rgb_cout] fp32 NHWC, rgb_filter) + rgb -- SynthesisBlock.forward's ToRGB + skip
     * (networks_stylegan2.py:452-458) of the last super-resolution block without re-reading its input. rgb_w: fp16
     * [B][rgb_w_rows][Cout] (the modulated ToRGB weights). rgb_skip_x != 0: y itself is not written (nothing reads it).
     * P3D_UNSUPPORTED when the launch shape does not qualify (callers then run the ToRGB convolution separately). */
    const void* rgb_w;
    const float* rgb_bias;
    const float* rgb_prev;
    const float* rgb_filter;
    float* rgb_out;
    int32_t rgb_cout, rgb_w_rows, rgb_skip_x;
    float rgb_clamp, rgb_acc_scale;
} p3d_conv_args_t;

/* One implicit-GEMM convolution launch (tcgen05 + TMA): 3x3 / 1x1 convolutions and the four phases of a stride-2
 * transposed 3x3 convolution are all expressed through the tap list and the output map. */
int p3d_conv_gemm(const p3d_conv_args_t* args, p3d_stream_t stream);

/* Up to four launches that differ ONLY in their tap list, computed grid (gH, gW) and output offset (oy, ox) -- the four
 * phases of a stride-2 transposed 3x3 convolution (conv2d_resample.py:114-131) -- as ONE launch whose tile schedule walks all
 * phases, heaviest first (the 1- and 2-tap phases alone are prologue-bound and leave most of the machine idle at their tails).
 * Every other field must be equal across phases[0..n_phases); up_prev / residual are not accepted. P3D_BAD_ARG otherwise.
 * Results are identical to n_phases separate p3d_conv_gemm calls. */
int p3d_conv_gemm_phases(const p3d_conv_args_t* phases, int n_phases, p3d_stream_t stream);

/* Per-sample modulated (and optionally demodulated) weights, modulated_conv2d lines :58-67:
 *   w'[b,o,i,k] = weight[o,i,k] * styles[b,i];  d[b,o] = rsqrt(sum_{i,k} w'^2 + 1e-8);  out = w' * d * scale
 * written K-major [planes][B][Cout_padded][kh*kw][Cin_padded] as fp16 (planes = 2: hi/lo split). Rows >= Cout and
 * channels outside [cin_offset, cin_offset+Cin) are zero (cin_offset lets a layer read a channel slice of a wider
 * activation tensor). pre_scale multiplies styles first (ToRGB's 1/sqrt(fan_in), :355). */
int p3d_modulate_weights(const float* weight, const float* styles, int B, int Cout, int Cin, int ktaps,
                         int Cout_padded, int Cin_padded, int cin_offset, int demodulate, float pre_scale,
                         float out_scale, int planes, void* out, p3d_stream_t stream);

/* Two-step form of p3d_modulate_weights for weights that change rarely (inference): p3d_prepare_weights runs once
 * per parameter version and writes weight_t [Cout][ktaps][Cin] (K-major copy) and wsq [Cout][Cin] = sum_k w^2;
 * p3d_modulate_weights_t then streams weight_t * styles * d with d[b,o] = rsqrt(sum_i styles[b,i]^2 wsq[o,i] + 1e-8)
 * (the same sum as :62 factored over taps). Same output layout and arguments as p3d_modulate_weights; needs
 * Cin_padded % 8 == 0 and 256 % (Cin_padded / 8) == 0, else P3D_UNSUPPORTED. */
int p3d_prepare_weights(const float* weight, int Cout, int Cin, int ktaps, float* weight_t, float* wsq, p3d_stream_t stream);
int p3d_modulate_weights_t(const float* weight_t, const float* wsq, const float* styles, int B, int Cout, int Cin, int ktaps,
                           int Cout_padded, int Cin_padded, int cin_offset, int demodulate, float pre_scale,
                           float out_scale, int planes, void* out, p3d_stream_t stream);

/* p3d_modulate_weights_t for every layer of a synthesis stack in one launch. descs_dev: device array, one entry per
 * layer (same meaning as the arguments of p3d_modulate_weights_t; styles_off / out_off are element offsets into
 * styles_base (fp32) / out_base (fp16)); block_layer_dev: int32 [n_blocks], the layer each CTA belongs to, CTAs of a layer
 * being consecutive and starting at first_block (n_blocks = sum of Cout_padded). Constraints on Cin_padded as above. */
typedef struct {
    const float* weight_t;
    const float* wsq;
    int64_t styles_off, out_off;
    int32_t Cout, Cin, ktaps, Cout_padded, Cin_padded, cin_offset, demodulate, planes;
    float pre_scale, out_scale;
    int32_t first_block, reserved;
} p3d_modw_desc_t;
int p3d_modulate_weights_batch(const p3d_modw_desc_t* descs_dev, const int32_t* block_layer_dev, int n_blocks,
                               const float* styles_base, void* out_base, int B, p3d_stream_t stream);

/* Every style affine of a synthesis stack in one launch (layer.affine(w) of SynthesisLayer.forward / ToRGBLayer.forward,
 * networks_stylegan2.py:313-315, 354-355; FullyConnectedLayer.forward :111-123 with the weight and bias gains already
 * applied by the caller): for each row r of weight [rows, w_dim],
 *   out[meta[r].out_off + b * meta[r].out_stride] = bias[r] + dot(ws[b, meta[r].ws_index, :], weight[r, :]).
 * meta: int32 [rows][4] = {ws_index, out_off, out_stride, 0}; ws: [B, num_ws, w_dim] fp32. */
int p3d_affine_batch(const float* ws, const float* weight, const float* bias, const int32_t* meta, float* out,
                     int B, int num_ws, int w_dim, int rows, p3d_stream_t stream);

/* FullyConnectedLayer.forward (networks_stylegan2.py:111-123) for small batches (mapping networks):
 *   y[b, o] = act( dot(x[b, :], weight[o, :] * weight_gain) + bias[o] * bias_gain ) * act_gain
 * x [B, in] fp32, weight [out, in], bias [out] or NULL, y [B, out]; act: 1 linear, 2 relu, 3 lrelu(alpha) (codes of p3d_bias_act).
 * One launch instead of the weight scaling + addmm / matmul + bias_act; P3D_UNSUPPORTED for other activations. */
int p3d_fc_bias_act(const float* x, const float* weight, const float* bias, float* y, int B, int in_features, int out_features,
                    float weight_gain, float bias_gain, int act, float alpha, float act_gain, p3d_stream_t stream);

/* Layout / precision converters between the reference's NCHW tensors and the NHWC fp16 tensors of this path. */
int p3d_nchw_to_nhwc_f16(const void* x, int src_dtype, int N, int C, int H, int W, int C_padded, int planes,
                         void* out, p3d_stream_t stream);
int p3d_nhwc_to_nchw_f32(const float* x, int N, int C, int H, int W, int c_stride, int c_offset, float* out,
                         p3d_stream_t stream);

/* Fused filtered leaky ReLU -- the plugin entry `filtered_lrelu(x, fu, fd, b, si, up, down, px0, px1, py0, py1, sx, sy, gain,
 * slope, clamp, flip_filter, writeSigns)` of the reference (torch_utils/ops/filtered_lrelu.cpp:20-213; kernel parameters
 * filtered_lrelu.h:18-57):  y = downsample_fd( lrelu_clamp( upsample_fu(x + b) * up^2 * gain ) ), everything between x and y
 * in shared memory. Shapes are {width, height, channels, batch}; strides are in ELEMENTS in the same order.
 * Filters: fp32, dense; fu_h == 0 / fd_h == 0 marks a separable 1-D filter of fu_w / fd_w taps (applied along x and y).
 * Sign tensor `s` (uint8, contiguous [N, C, s_shape[1], s_shape[0]], four 2-bit records per byte: 1 = was negative,
 * 2 = was clamped): sign_mode 0 ignores it, 1 writes it (forward pass that needs gradients), 2 reads it (the gradient pass:
 * same op with fu / fd swapped, flip inverted; records are looked up at up-sampled coordinate + s_ofs). sw_limit = active
 * width in bytes. Returns P3D_UNSUPPORTED when no tile of this configuration fits shared memory (filters > 32 taps, ...):
 * the reference's `rc = -1`, upon which callers compose upfirdn2d + p3d_filtered_lrelu_act + upfirdn2d (filtered_lrelu.py:225-231). */
typedef struct {
    const void* x; void* y; const void* b;      /* b: [C] in x's dtype or NULL */
    unsigned char* s;
    const float* fu; const float* fd;
    int32_t dtype;                               /* P3D_F32 or P3D_F16 */
    int32_t up, down;
    int32_t fu_w, fu_h, fd_w, fd_h;
    int32_t px0, px1, py0, py1;                  /* padding with respect to the up-sampled image */
    float   gain, slope, clamp;                  /* clamp = +inf for none */
    int32_t flip;                                /* flip_filter: 0 = convolution (filters are mirrored), 1 = correlation */
    int32_t x_shape[4]; int64_t x_stride[4];
    int32_t y_shape[4]; int64_t y_stride[4];
    int64_t b_stride;
    int32_t s_shape[2];                          /* {width in BYTES, height} */
    int32_t s_ofs[2];
    int32_t sw_limit;
    int32_t sign_mode;
} p3d_filtered_lrelu_args_t;
int p3d_filtered_lrelu(const p3d_filtered_lrelu_args_t* args, p3d_stream_t stream);

/* In-place `x = lrelu_clamp(x * gain)` with the same sign contract -- `filtered_lrelu_act_` of the reference
 * (filtered_lrelu.cpp:217-270, kernel filtered_lrelu.cu:1110-1215), the activation of the generic fallback path.
 * s_shape = {width in ELEMENTS (multiple of 4), height}. */
int p3d_filtered_lrelu_act(void* x, unsigned char* s, int dtype, const int32_t x_shape[4], const int64_t x_stride[4],
                           const int32_t s_shape[2], const int32_t s_ofs[2], float gain, float slope, float clamp,
                           int sign_mode, p3d_stream_t stream);

/* Broadcasting fused multiply-add y = a * b + c -- `fma(a, b, c)` of the reference (torch_utils/ops/fma.py:17-34, forward =
 * torch.addcmul(c, a, b)): the demodulation + noise step of the non-fused modulated convolution (networks_stylegan2.py:79-82).
 * y: dense [shape[0..3]] (row-major); a / b / c: element strides over the same four dimensions, 0 on broadcast dimensions.
 * dtype: P3D_F16 (fp32 arithmetic, one rounding) / P3D_F32 / P3D_F64. */
int p3d_fma(const void* a, const void* b, const void* c, void* y, int dtype, const int64_t shape[4], const int64_t a_stride[4],
            const int64_t b_stride[4], const int64_t c_stride[4], p3d_stream_t stream);

/* 4x4 FIR (upfirdn2d up=down=1) + noise + bias + lrelu + gain + clamp on NHWC tensors: the tail of an up=2
 * SynthesisLayer (networks_stylegan2.py:324-331 after conv2d_resample.py:128). in_dtype: P3D_F32 or P3D_F16;
 * out_planes 1 (fp16) or 2 (fp16 hi/lo). x [B,inH,inW,C] -> y [out_planes][B,outH,outW,C]. noise: [outH*outW] shared by the
 * batch (noise_batch_stride 0, noise_mode='const') or one image per sample (noise_batch_stride = outH*outW, 'random'). */
int p3d_fir_act_nhwc(const void* x, int in_dtype, const float* f, const float* noise, const float* bias, void* y,
                     int out_planes, int B, int inH, int inW, int outH, int outW, int C, int padx0, int pady0,
                     float fir_gain, int act, float alpha, float act_gain, float clamp, int64_t noise_batch_stride,
                     p3d_stream_t stream);

/* The same operation on a split (hi/lo) fp16 input [2][B][inH][inW][C] whose value is hi + lo (fp32 semantics, no fp16
 * rounding of the filtered value): the FIR in front of the strided convolutions of the down=2 layers
 * (conv2d_resample.py:108-111) when the producer wrote a split tensor. */
int p3d_fir_act_nhwc_split(const void* x_hi_lo, const float* f, const float* noise, const float* bias, void* y,
                           int out_planes, int B, int inH, int inW, int outH, int outW, int C, int padx0, int pady0,
                           float fir_gain, int act, float alpha, float act_gain, float clamp, int64_t noise_batch_stride,
                           p3d_stream_t stream);

/* The same operation for a SEPARABLE 4x4 filter f[j][i] = fy[j] * fx[i] (what upfirdn2d.setup_filter builds from a 1-D tap list,
 * upfirdn2d.py:60-63): fx / fy are HOST arrays (the caller factors the filter once per buffer); the kernel runs the row pass and
 * the column pass on a 4x2 output block per thread, 11 instead of 16 multiply-adds per output element. Same rounding points as
 * p3d_fir_act_nhwc (fp32 accumulation, one rounding of the filtered value in the fp16 case); sums are formed in another order, so
 * results agree with it to fp32 rounding, not bit for bit. */
int p3d_fir_act_nhwc_sep(const void* x, int in_dtype, const float fx[4], const float fy[4], const float* noise, const float* bias,
                         void* y, int out_planes, int B, int inH, int inW, int outH, int outW, int C, int padx0, int pady0,
                         float fir_gain, int act, float alpha, float act_gain, float clamp, int64_t noise_batch_stride,
                         p3d_stream_t stream);



/* ---------------------------------------------------------------------------------------------
 * Mesh extraction (applications/extract_mesh.py:84-96: mcubes.marching_cubes on the dense sigma grid)
 * ------------------------------------------------------------------------------------------- */

/* Marching cubes on a dense fp32 grid volume [nx][ny][nz] (C order), each side >= 2 (pix2pix3d_b200/csrc/marching_cubes.cu;
 * the mesh is defined in oracle/p3d_oracle/mesh.py). A point is inside when (double)v > threshold (NaN is outside). One
 * vertex per grid edge p -> p + e_axis whose endpoints differ in inside-ness, at p + t e_axis, t = (threshold - v_p) /
 * (v_{p+e} - v_p) in float64, ordered by owning point p in C order and by axis within a point; faces are listed by cube in
 * C order and in table order inside a cube, oriented outward (normals toward lower values). No atomics: the output depends
 * only on the input.
 * Two calls on one workspace of p3d_marching_cubes_workspace_bytes() bytes (P3D_BAD_ARG there for a side < 2 or a grid of
 * 2^40 points or more): p3d_marching_cubes_count writes counts[2] = {V, F} (device int64); the caller allocates
 * vertices [V,3] float64 (index coordinates) and faces [F,3] int64 and calls p3d_marching_cubes_emit with the same volume,
 * threshold and workspace. Vertex ids are int32 in the workspace: V must be < 2^31. */
int64_t p3d_marching_cubes_workspace_bytes(int64_t nx, int64_t ny, int64_t nz);
int p3d_marching_cubes_count(const float* volume, int64_t nx, int64_t ny, int64_t nz, double threshold,
                             void* workspace, int64_t workspace_bytes, int64_t* counts, p3d_stream_t stream);
int p3d_marching_cubes_emit(const float* volume, int64_t nx, int64_t ny, int64_t nz, double threshold,
                            void* workspace, int64_t workspace_bytes, double* vertices, int64_t* faces, p3d_stream_t stream);

/* ---------------------------------------------------------------------------------------------
 * Mesh preview (applications/extract_mesh.py:226-262: the pyrender turntable of the extracted mesh)
 *
 * A triangle rasterizer with a depth buffer and a diffuse shader (pix2pix3d_b200/csrc/mesh_raster.cu; the numpy
 * restatement is oracle/p3d_oracle/mesh_render.py). It is not pyrender and does not reproduce its pixels.
 * From the script: the orthographic camera and its extents (xmag = ymag = 0.3 for seg, 0.6 for car), the 512x512 frames,
 * the orbit of OpenGL-convention poses and a spot light of intensity 3 with a pi/4 cone placed at the camera.
 * This package's choices: diffuse shading only (no ambient, no specular), a hard cone edge, grey 0.8 when the mesh has
 * no vertex colours, a white background, and znear = 0.05 / zfar = 100 (pyrender's own defaults for the planes, the
 * outer cone and the background are unverified).
 *
 * Views: per view, world2cam rows 0-2 of the inverse of an OpenGL cam2world (camera looks down -z, +y is up), the eye
 * (camera position) and the spot axis (the camera's -z in world space), all fp32.
 * Every product and sum below is one fp32 operation rounded to nearest, in the order written (no FMA contraction):
 *   c = ((m[r][0] x + m[r][1] y) + m[r][2] z) + m[r][3]       camera coordinates, r = 0, 1, 2
 *   sx = c0 (W / (2 xmag)) + W / 2,  sy = H / 2 - c1 (H / (2 ymag)),  d = -c2      (row 0 is the top)
 * Coverage: X = rint(256 sx), Y = rint(256 sy) (int64, 8 sub-pixel bits). Pixel (i, j) has its centre at
 * (256 j + 128, 256 i + 128). Edge functions E_k (edge opposite vertex k, from vertex k+1 to k+2) are exact integers and
 * sum to the area A. A triangle with A < 0 has every E_k and A negated (either winding is drawn); A == 0 is skipped.
 * A pixel is covered when every E_k > 0, or E_k == 0 on a top-left edge (edge vector (dx, dy) after the negation:
 * dy < 0, or dy == 0 and dx > 0), so two triangles sharing an edge cover each pixel on it exactly once.
 * Dropped triangles: a non-finite vertex coordinate or a face index outside [0, V) (silently: marching cubes emits NaN
 * vertices next to NaN grid values), and a vertex with |sx| or |sy| not <= 2^21 (counted into guard_drops[0]).
 * Depth: b_k = fp32(E_k) / fp32(A) (correctly rounded conversions), d = (b0 d0 + b1 d1) + b2 d2; a fragment is kept when
 * znear <= d <= zfar. depth_keys [N,H,W] = min over fragments of (float_bits(d) << 32 | face id): the nearest fragment
 * wins, the lower face id on equal depth, whatever the launch order; ~0 = empty.
 * Shading, per covered pixel, with the same b_k, world vertices v_k and colours c_k (uint8 / 255 or grey 0.8):
 *   colour = (b0 c0 + b1 c1) + b2 c2 per channel;  n = cross(v1 - v0, v2 - v0) / |.|  (outward for marching_cubes faces);
 *   p = (b0 v0 + b1 v1) + b2 v2;  q = eye - p;  r2 = (qx qx + qy qy) + qz qz;  l = q / sqrt(r2);
 *   shade = (I max(0, n . l)) / (pi r2), or 0 when (axis . l) > -cos(pi/4) (outside the cone);
 *   out = x < 255 ? floor(x) : 255 with x = ((255 colour) shade) + 0.5; empty pixels are white (255, 255, 255).
 * Vector lengths are sqrt of (x x + y y) + z z and divisions are correctly rounded (no reciprocal square roots). */
typedef struct {
    float world2cam[12];     /* rows 0-2 of the 4x4 world-to-camera matrix, row-major */
    float eye[3];            /* camera position in world space (where the light sits) */
    float spot_axis[3];      /* camera -z in world space */
} p3d_mesh_view_t;

/* Depth pass: vertices [V,3] fp32, faces [F,3] int64 (what p3d_marching_cubes_emit writes), views [N] (device array),
 * depth_keys uint64 [N,H,W] (cleared to ~0 here), guard_drops: one device int64 (zeroed here, then the number of
 * (face, view) pairs dropped by the guard band). One launch covers every face and view. P3D_BAD_ARG on bad sizes
 * (N, H or W < 1, F >= 2^32, xmag / ymag not > 0, not 0 < znear < zfar). */
int p3d_mesh_raster(const float* vertices, int64_t V, const int64_t* faces, int64_t F, const p3d_mesh_view_t* views, int N,
                    int H, int W, float xmag, float ymag, float znear, float zfar, uint64_t* depth_keys, int64_t* guard_drops,
                    p3d_stream_t stream);
/* Shading pass over the keys of p3d_mesh_raster (same vertices, faces, views and extents): out uint8 [N,H,W,3].
 * vertex_colors: uint8 [V,3] or NULL (grey). light_intensity: I above. */
int p3d_mesh_shade(const uint64_t* depth_keys, const float* vertices, int64_t V, const int64_t* faces, int64_t F,
                   const p3d_mesh_view_t* views, int N, int H, int W, float xmag, float ymag,
                   const unsigned char* vertex_colors, float light_intensity, unsigned char* out, p3d_stream_t stream);

/* upsample2d(img, f) with up=2 (upfirdn2d.py:315-350) on an fp32 NHWC image: [B,H,W,C] -> [B,2H,2W,C]. */
int p3d_upsample2x_nhwc(const float* x, const float* f, float* y, int B, int H, int W, int C, p3d_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* P3D_H_ */
