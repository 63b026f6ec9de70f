// Fused volumetric renderer for sm_100a: tri-plane gather + OSG decoder MLP + ray marching +
// importance resampling + merge, replacing the ~60 ATen launches of
// training/volumetric_rendering/renderer.py:88-253 and ray_marcher.py:25-57 (reference repo).
//
// Data layout: planes are channels-last [B,3,H,W,32] fp32, so a bilinear tap of all 32 channels is
// one 128-byte line and a warp (lane = channel) fetches it with a single coalesced request.
// Work decomposition: one CTA owns a tile of RT rays; thread <-> one coarse and one fine sample.
//   P1 gather coarse features (lane = channel) into shared memory, transposed to lane = sample
//   P2 sigma-only MLP                         P3 coarse ray march (warp per ray, shuffle scans)
//   P3b importance sampling (exact fp32 order) P4 gather + sigma for fine samples
//   P5 rank-merge of coarse+fine, final march  P6 colour MLP, coefficient-weighted shuffle reduce
// Features stay in shared memory between P1/P4 and P6, so every plane texel is gathered once.
#include "render_common.cuh"

namespace p3d {

// packed decoder layout per net (floats); see p3d_pack_decoder
constexpr int kW1T = 0;                    // [32][64]  W1^T * gain
constexpr int kB1 = kW1T + kC * kHid;      // [64]
constexpr int kW2S = kB1 + kHid;           // [64]      row 0 of W2 (sigma)
constexpr int kW2T = kW2S + kHid;          // [64][32]  rows 1..32 of W2, transposed
constexpr int kB2S = kW2T + kHid * kOut;   // [4]       b2[0] (+pad)
constexpr int kB2C = kB2S + 4;             // [32]      b2[1..32]
constexpr int kNetFloats = kB2C + kOut;    // 4260
static_assert(2 * kNetFloats == P3D_DECODER_PACKED_FLOATS, "packed decoder size");

// ---------------------------------------------------------------------------------------------
// p3d_pack_decoder
// ---------------------------------------------------------------------------------------------
struct PackArgs {
    const float* w1[2]; const float* b1[2]; const float* w2[2]; const float* b2[2];
    float w1g[2], b1g[2], w2g[2], b2g[2];
    int n_nets;
};

__global__ void pack_decoder_kernel(PackArgs a, float* __restrict__ out) {
    int net = blockIdx.y;
    float* o = out + net * kNetFloats;
    if (net >= a.n_nets) {
        for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < kNetFloats; i += gridDim.x * blockDim.x) o[i] = 0.f;
        return;
    }
    const float* w1 = a.w1[net]; const float* b1 = a.b1[net];
    const float* w2 = a.w2[net]; const float* b2 = a.b2[net];
    // products rounded once in fp32, exactly like `self.weight * self.weight_gain`
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < kNetFloats; i += gridDim.x * blockDim.x) {
        float v = 0.f;
        if (i < kB1) { int k = i / kHid, j = i % kHid; v = __fmul_rn(w1[j * kC + k], a.w1g[net]); }
        else if (i < kW2S) { int j = i - kB1; v = (a.b1g[net] != 1.f) ? __fmul_rn(b1[j], a.b1g[net]) : b1[j]; }
        else if (i < kW2T) { int j = i - kW2S; v = __fmul_rn(w2[j], a.w2g[net]); }
        else if (i < kB2S) { int t = i - kW2T; int j = t / kOut, o2 = t % kOut; v = __fmul_rn(w2[(o2 + 1) * kHid + j], a.w2g[net]); }
        else if (i < kB2C) { int t = i - kB2S; v = (t == 0) ? ((a.b2g[net] != 1.f) ? __fmul_rn(b2[0], a.b2g[net]) : b2[0]) : 0.f; }
        else { int o2 = i - kB2C; v = (a.b2g[net] != 1.f) ? __fmul_rn(b2[o2 + 1], a.b2g[net]) : b2[o2 + 1]; }
        o[i] = v;
    }
}

// ---------------------------------------------------------------------------------------------
// Ray / box slab test (math_utils.py:46-98): thread per ray, the reference's operation order (inverse direction first, then
// (bound - origin) * inverse), comparisons before the min / max update, misses marked (-1, -2)
// ---------------------------------------------------------------------------------------------
__global__ void ray_limits_box_kernel(const float* __restrict__ ro, const float* __restrict__ rd, int64_t n, float half,
                                      float* __restrict__ t_near, float* __restrict__ t_far) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    float tin[3], tout[3];
#pragma unroll
    for (int ax = 0; ax < 3; ++ax) {
        const float o = ro[i * 3 + ax], inv = __fdiv_rn(1.f, rd[i * 3 + ax]);
        const bool neg = inv < 0.f;
        tin[ax] = __fmul_rn(__fsub_rn(neg ? half : -half, o), inv);
        tout[ax] = __fmul_rn(__fsub_rn(neg ? -half : half, o), inv);
    }
    bool valid = true;
    float tmin = tin[0], tmax = tout[0];
#pragma unroll
    for (int ax = 1; ax < 3; ++ax) {
        if ((tmin > tout[ax]) || (tin[ax] > tmax)) valid = false;
        // torch.max / torch.min propagate NaN (a zero direction component against an origin on the slab plane gives 0 * inf)
        tmin = (tmin != tmin || tin[ax] != tin[ax]) ? __int_as_float(0x7fc00000) : fmaxf(tmin, tin[ax]);
        tmax = (tmax != tmax || tout[ax] != tout[ax]) ? __int_as_float(0x7fc00000) : fminf(tmax, tout[ax]);
    }
    t_near[i] = valid ? tmin : -1.f;
    t_far[i] = valid ? tmax : -2.f;
}

// ---------------------------------------------------------------------------------------------
// Ray sampler (ray_sampler.py:24-62)
// ---------------------------------------------------------------------------------------------
__global__ void ray_sampler_kernel(const float* __restrict__ c2w, const float* __restrict__ K, int B, int res,
                                   float* __restrict__ origins, float* __restrict__ dirs) {
    int M = res * res;
    int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (int64_t)B * M) return;
    int b = (int)(idx / M), m = (int)(idx % M);
    int row = m / res, col = m % res;
    const float* Mx = c2w + b * 16;
    const float* Kb = K + b * 9;
    float fx = Kb[0], sk = Kb[1], cx = Kb[2], fy = Kb[4], cy = Kb[5];
    float inv = 1.f / (float)res, half = 0.5f / (float)res;
    float x_cam = __fadd_rn(__fmul_rn((float)col, inv), half);
    float y_cam = __fadd_rn(__fmul_rn((float)row, inv), half);
    // (x_cam - cx + cy*sk/fy - sk*y_cam/fy) / fx * z_cam, evaluated left to right (ray_sampler.py:51)
    float t = __fsub_rn(x_cam, cx);
    t = __fadd_rn(t, __fdiv_rn(__fmul_rn(cy, sk), fy));
    t = __fsub_rn(t, __fdiv_rn(__fmul_rn(sk, y_cam), fy));
    float xl = __fdiv_rn(t, fx);
    float yl = __fdiv_rn(__fsub_rn(y_cam, cy), fy);
    float w[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        // cam2world @ [xl, yl, 1, 1]
        float acc = __fmul_rn(Mx[i * 4 + 0], xl);
        acc = __fadd_rn(acc, __fmul_rn(Mx[i * 4 + 1], yl));
        acc = __fadd_rn(acc, Mx[i * 4 + 2]);
        acc = __fadd_rn(acc, Mx[i * 4 + 3]);
        w[i] = __fsub_rn(acc, Mx[i * 4 + 3]);
    }
    float n2 = __fadd_rn(__fadd_rn(__fmul_rn(w[0], w[0]), __fmul_rn(w[1], w[1])), __fmul_rn(w[2], w[2]));
    float n = fmaxf(__fsqrt_rn(n2), 1e-12f);
    float* o = origins + idx * 3;
    float* d = dirs + idx * 3;
#pragma unroll
    for (int i = 0; i < 3; ++i) { o[i] = Mx[i * 4 + 3]; d[i] = __fdiv_rn(w[i], n); }
}

// ---------------------------------------------------------------------------------------------
// NCHW -> NHWC transpose for the plane stack (C = 32)
// ---------------------------------------------------------------------------------------------
__global__ void planes_to_cl_kernel(const float* __restrict__ in, float* __restrict__ out, int C, int HW) {
    __shared__ float tile[32][33];
    int n = blockIdx.z;
    int p0 = blockIdx.x * 32;
    int c0 = blockIdx.y * 32;
    const float* src = in + (int64_t)n * C * HW;
    float* dst = out + (int64_t)n * HW * C;
    int tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
    for (int j = ty; j < 32; j += 8) {
        int c = c0 + j, p = p0 + tx;
        tile[j][tx] = (c < C && p < HW) ? src[(int64_t)c * HW + p] : 0.f;
    }
    __syncthreads();
    for (int j = ty; j < 32; j += 8) {
        int p = p0 + j, c = c0 + tx;
        if (c < C && p < HW) dst[(int64_t)p * C + c] = tile[tx][j];
    }
}

// swizzled feature tile: row r holds 32 floats; 16-byte chunk q is stored at chunk (q ^ (r & 7)) so
// that both the lane = channel stores and the lane = sample float4 loads are bank-conflict free.
__device__ __forceinline__ int feat_index(int row, int c) {
    return row * kC + ((((c >> 2) ^ (row & 7)) << 2) | (c & 3));
}

// Warp-cooperative gather: every lane brings (row, b, px, py, pz) of its own sample (row < 0: none);
// the warp then walks the 32 samples with lane = channel and stores features into `feat`.
__device__ __forceinline__ void warp_gather(const float* __restrict__ planes, int H, int W,
                                            float* __restrict__ feat, int row, int b,
                                            float px, float py, float pz, int lane) {
    unsigned active = __ballot_sync(0xffffffffu, row >= 0);
    size_t isz = (size_t)3 * H * W * kC;
    while (active) {
        int s = __ffs(active) - 1;
        active &= active - 1;
        int rs = __shfl_sync(0xffffffffu, row, s);
        int bs = __shfl_sync(0xffffffffu, b, s);
        float x = __shfl_sync(0xffffffffu, px, s);
        float y = __shfl_sync(0xffffffffu, py, s);
        float z = __shfl_sync(0xffffffffu, pz, s);
        float f0, f1, f2;
        plane_values(planes + (size_t)bs * isz, H, W, x, y, z, lane, f0, f1, f2);
        feat[feat_index(rs, lane)] = plane_mean(f0, f1, f2);
    }
    __syncwarp();
}

// ---------------------------------------------------------------------------------------------
// Decoder MLP, lane = sample, weights broadcast from shared memory
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void mlp_hidden(const float* __restrict__ net, const float* __restrict__ feat,
                                           int row, float (&h)[kHid]) {
    const float4* b1v = reinterpret_cast<const float4*>(net + kB1);
#pragma unroll
    for (int j = 0; j < kHid / 4; ++j) {
        float4 b = b1v[j];
        h[4 * j + 0] = b.x; h[4 * j + 1] = b.y; h[4 * j + 2] = b.z; h[4 * j + 3] = b.w;
    }
    const float4* frow = reinterpret_cast<const float4*>(feat + row * kC);
    const int sw = row & 7;
    const float4* w1v = reinterpret_cast<const float4*>(net + kW1T);
#pragma unroll 1
    for (int q = 0; q < kC / 4; ++q) {
        float4 xv = frow[q ^ sw];
        const float4* wq = w1v + q * 4 * (kHid / 4);
#pragma unroll
        for (int kk = 0; kk < 4; ++kk) {
            float x = (kk == 0) ? xv.x : (kk == 1) ? xv.y : (kk == 2) ? xv.z : xv.w;
#pragma unroll
            for (int j = 0; j < kHid / 4; ++j) {
                float4 w = wq[kk * (kHid / 4) + j];
                h[4 * j + 0] = fmaf(w.x, x, h[4 * j + 0]);
                h[4 * j + 1] = fmaf(w.y, x, h[4 * j + 1]);
                h[4 * j + 2] = fmaf(w.z, x, h[4 * j + 2]);
                h[4 * j + 3] = fmaf(w.w, x, h[4 * j + 3]);
            }
        }
    }
#pragma unroll
    for (int j = 0; j < kHid; ++j) h[j] = softplus_f(h[j]);
}

__device__ __forceinline__ float mlp_sigma(const float* __restrict__ net, const float (&h)[kHid]) {
    const float4* wv = reinterpret_cast<const float4*>(net + kW2S);
    float a0 = net[kB2S], a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
    for (int j = 0; j < kHid / 4; ++j) {
        float4 w = wv[j];
        a0 = fmaf(w.x, h[4 * j + 0], a0);
        a1 = fmaf(w.y, h[4 * j + 1], a1);
        a2 = fmaf(w.z, h[4 * j + 2], a2);
        a3 = fmaf(w.w, h[4 * j + 3], a3);
    }
    return (a0 + a1) + (a2 + a3);
}

// eight colour outputs [8*oc, 8*oc+8) (pre-activation)
__device__ __forceinline__ void mlp_colors8(const float* __restrict__ net, const float (&h)[kHid], int oc,
                                            float (&acc)[8]) {
    const float4* bv = reinterpret_cast<const float4*>(net + kB2C + oc * 8);
    float4 b0 = bv[0], b1 = bv[1];
    acc[0] = b0.x; acc[1] = b0.y; acc[2] = b0.z; acc[3] = b0.w;
    acc[4] = b1.x; acc[5] = b1.y; acc[6] = b1.z; acc[7] = b1.w;
    const float4* wv = reinterpret_cast<const float4*>(net + kW2T + oc * 8);
#pragma unroll
    for (int j = 0; j < kHid; ++j) {
        float4 w0 = wv[j * (kOut / 4)], w1 = wv[j * (kOut / 4) + 1];
        float x = h[j];
        acc[0] = fmaf(w0.x, x, acc[0]); acc[1] = fmaf(w0.y, x, acc[1]);
        acc[2] = fmaf(w0.z, x, acc[2]); acc[3] = fmaf(w0.w, x, acc[3]);
        acc[4] = fmaf(w1.x, x, acc[4]); acc[5] = fmaf(w1.y, x, acc[5]);
        acc[6] = fmaf(w1.z, x, acc[6]); acc[7] = fmaf(w1.w, x, acc[7]);
    }
}

// ---------------------------------------------------------------------------------------------
// Fused forward kernel
// ---------------------------------------------------------------------------------------------
struct RenderLayout {   // shared-memory carve-up (float offsets), identical on host and device
    int RT, Sc, Sf, S, Scp, Sfp, gc, gf, NGc, NGf, NT;
    int off_dec, off_feat, off_ray, ray_stride, off_part, off_scal, total_floats;
    int o_dC, o_sC, o_dF, o_sF, o_sd, o_ss, o_w, o_cdf, o_om;  // inside a ray block
};


__host__ __device__ inline RenderLayout make_layout(int RT, int Sc, int Sf, int n_nets) {
    RenderLayout L;
    L.RT = RT; L.Sc = Sc; L.Sf = Sf; L.S = Sc + Sf;
    L.Scp = round_up(Sc, 8); L.Sfp = Sf > 0 ? round_up(Sf, 8) : 0;
    L.gc = pow2_group(L.Scp); L.gf = Sf > 0 ? pow2_group(L.Sfp) : 1;
    L.NGc = L.Scp / L.gc; L.NGf = Sf > 0 ? L.Sfp / L.gf : 0;
    int mx = L.Scp > L.Sfp ? L.Scp : L.Sfp;
    L.NT = round_up(RT * mx, 32);
    int o = 0;
    L.off_dec = o; o += n_nets * kNetFloats;
    o = round_up(o, 32);
    L.off_feat = o; o += RT * L.S * kC;
    int r = 0;
    L.o_dC = r; r += round_up(Sc, 4);
    L.o_sC = r; r += round_up(Sc, 4);
    L.o_dF = r; r += round_up(Sf, 4);
    L.o_sF = r; r += round_up(Sf, 4);
    L.o_sd = r; r += round_up(L.S, 4);
    L.o_ss = r; r += round_up(L.S, 4);
    L.o_w = r; r += round_up(L.S, 4);
    L.o_cdf = r; r += round_up(Sc, 4);
    L.o_om = r; r += round_up(Sc, 4);
    L.ray_stride = r;
    L.off_ray = o; o += RT * r;
    L.off_part = o; o += RT * (L.NGc + L.NGf) * (kOut * n_nets);
    L.off_scal = o; o += 4 * RT + 4;
    L.total_floats = o;
    return L;
}

struct RenderParams {
    p3d_render_args_t a;
    RenderLayout L;
    int total_rays, n_tiles, cout;
};

__global__ void __launch_bounds__(256, 2) render_fwd_kernel(const RenderParams P) {
    extern __shared__ __align__(16) float smem[];
    const p3d_render_args_t& a = P.a;
    const RenderLayout& L = P.L;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = blockDim.x >> 5;
    const int RT = L.RT, Sc = L.Sc, Sf = L.Sf, S = L.S;
    const int n_nets = a.n_nets;

    float* dec = smem + L.off_dec;
    float* feat = smem + L.off_feat;
    float* rayb = smem + L.off_ray;
    float* part = smem + L.off_part;
    float* scal = smem + L.off_scal;  // per ray: [0]=sum_w, [1]=depth ; tail: CTA min/max keys
    uint32_t* cta_keys = reinterpret_cast<uint32_t*>(scal + 4 * RT);

    // decoder weights -> shared memory (once per CTA)
    {
        const float4* src = reinterpret_cast<const float4*>(a.decoder_packed);
        float4* dst = reinterpret_cast<float4*>(dec);
        for (int i = tid; i < n_nets * kNetFloats / 4; i += blockDim.x) dst[i] = __ldg(src + i);
    }
    if (tid < 2) cta_keys[tid] = 0u;
    __syncthreads();
    const float* net_sigma = dec + a.sigma_net * kNetFloats;

    // thread <-> sample slots
    const int rC = tid / L.Scp, sC = tid % L.Scp;
    const int rF = (Sf > 0) ? tid / L.Sfp : RT, sF = (Sf > 0) ? tid % L.Sfp : 0;

    for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
        const int ray0 = tile * RT;
        const bool vC = (rC < RT) && (sC < Sc) && (ray0 + rC < P.total_rays);
        const bool vF = (rF < RT) && (sF < Sf) && (ray0 + rF < P.total_rays);
        const int gC = ray0 + rC, gF = ray0 + rF;     // global ray ids
        // image of the ray -> plane set it gathers from (p3d_render_args_t::plane_index: V views of one resident plane set)
        const int bC = vC ? plane_set(a, gC / a.R) : 0, bF = vF ? plane_set(a, gF / a.R) : 0;
        const int rowC = rC * Sc + sC, rowF = RT * Sc + rF * Sf + sF;
        float* rbC = rayb + (rC < RT ? rC : 0) * L.ray_stride;
        float* rbF = rayb + (rF < RT ? rF : 0) * L.ray_stride;

        // ---- P1: coarse gather ------------------------------------------------------------
        float dC = 0.f;
        {
            float px = 0.f, py = 0.f, pz = 0.f;
            if (vC) {
                dC = coarse_depth(a, gC, sC, Sc);
                const float* o = a.ray_origins + (size_t)gC * 3;
                const float* d = a.ray_dirs + (size_t)gC * 3;
                px = __fmul_rn(a.coord_scale, __fadd_rn(__ldg(o + 0), __fmul_rn(dC, __ldg(d + 0))));
                py = __fmul_rn(a.coord_scale, __fadd_rn(__ldg(o + 1), __fmul_rn(dC, __ldg(d + 1))));
                pz = __fmul_rn(a.coord_scale, __fadd_rn(__ldg(o + 2), __fmul_rn(dC, __ldg(d + 2))));
            }
            warp_gather(a.planes_nhwc, a.H, a.W, feat, vC ? rowC : -1, bC, px, py, pz, lane);
        }
        // ---- P2: coarse sigma --------------------------------------------------------------
        if (vC) {
            float h[kHid];
            mlp_hidden(net_sigma, feat, rowC, h);
            float sg = mlp_sigma(net_sigma, h);
            rbC[L.o_dC + sC] = dC;
            rbC[L.o_sC + sC] = sg;
        }
        __syncthreads();

        // ---- P3: coarse march + importance cdf (warp per ray) --------------------------------
        if (Sf > 0) {
            for (int r = warp; r < RT; r += nwarps) {
                if (ray0 + r >= P.total_rays) continue;
                float* rb = rayb + r * L.ray_stride;
                float sw, swd;
                warp_march(rb + L.o_dC, rb + L.o_sC, Sc, rb + L.o_w, lane, sw, swd);
                __syncwarp();
                if (a.dbg_weights_coarse) {
                    float* o = a.dbg_weights_coarse + (size_t)(ray0 + r) * (Sc - 1);
                    for (int i = lane; i < Sc - 1; i += 32) o[i] = rb[L.o_w + i];
                }
                warp_importance_cdf(rb + L.o_w, Sc, rb + L.o_om, rb + L.o_cdf, lane);
            }
            __syncthreads();

            // ---- P3b + P4: fine depths, gather, sigma ---------------------------------------
            float dF = 0.f;
            {
                float px = 0.f, py = 0.f, pz = 0.f;
                if (vF) {
                    float u = __ldg(a.u_importance + (size_t)gF * Sf + sF);
                    int inds;
                    dF = importance_sample(rbF + L.o_cdf, rbF + L.o_dC, Sc, u, inds);
                    if (a.dbg_inds) a.dbg_inds[(size_t)gF * Sf + sF] = inds;
                    if (a.dbg_depths_fine) a.dbg_depths_fine[(size_t)gF * Sf + sF] = dF;
                    const float* o = a.ray_origins + (size_t)gF * 3;
                    const float* d = a.ray_dirs + (size_t)gF * 3;
                    px = __fmul_rn(a.coord_scale, __fadd_rn(__ldg(o + 0), __fmul_rn(dF, __ldg(d + 0))));
                    py = __fmul_rn(a.coord_scale, __fadd_rn(__ldg(o + 1), __fmul_rn(dF, __ldg(d + 1))));
                    pz = __fmul_rn(a.coord_scale, __fadd_rn(__ldg(o + 2), __fmul_rn(dF, __ldg(d + 2))));
                }
                warp_gather(a.planes_nhwc, a.H, a.W, feat, vF ? rowF : -1, bF, px, py, pz, lane);
            }
            if (vF) {
                float h[kHid];
                mlp_hidden(net_sigma, feat, rowF, h);
                float sg = mlp_sigma(net_sigma, h);
                rbF[L.o_dF + sF] = dF;
                rbF[L.o_sF + sF] = sg;
            }
            __syncthreads();
        }

        // ---- P5: stable rank merge (torch.sort over cat(coarse, fine), renderer.py:157-167) ----
        int rankC = sC, rankF = 0;
        if (vC) {
            const float* dc = rbC + L.o_dC;
            const float* df = rbC + L.o_dF;
            int cnt = 0;
            for (int i = 0; i < Sc; ++i) { float v = dc[i]; cnt += (v < dC) || (v == dC && i < sC); }
            for (int k = 0; k < Sf; ++k) cnt += (df[k] < dC);
            rankC = cnt;
            rbC[L.o_sd + cnt] = dC;
            rbC[L.o_ss + cnt] = rbC[L.o_sC + sC];
            if (a.dbg_perm) a.dbg_perm[(size_t)gC * S + cnt] = sC;
        }
        if (vF) {
            const float* dc = rbF + L.o_dC;
            const float* df = rbF + L.o_dF;
            float dFv = df[sF];
            int cnt = 0;
            for (int i = 0; i < Sc; ++i) cnt += (dc[i] <= dFv);
            for (int k = 0; k < Sf; ++k) { float v = df[k]; cnt += (v < dFv) || (v == dFv && k < sF); }
            rankF = cnt;
            rbF[L.o_sd + cnt] = dFv;
            rbF[L.o_ss + cnt] = rbF[L.o_sF + sF];
            if (a.dbg_perm) a.dbg_perm[(size_t)gF * S + cnt] = Sc + sF;
        }
        __syncthreads();

        // ---- P5b: final march (warp per ray) -----------------------------------------------
        for (int r = warp; r < RT; r += nwarps) {
            if (ray0 + r >= P.total_rays) continue;
            float* rb = rayb + r * L.ray_stride;
            float sw, swd;
            warp_march(rb + L.o_sd, rb + L.o_ss, S, rb + L.o_w, lane, sw, swd);
            if (lane == 0) {
                rb[L.o_w + S - 1] = 0.f;
                scal[4 * r + 0] = sw;
                float depth = __fdiv_rn(swd, sw);          // NaN when sw == 0; resolved by the clamp pass
                a.out_depth[ray0 + r] = depth;
                a.out_wsum[ray0 + r] = sw;
                atomicMax(&cta_keys[0], float_to_key(rb[L.o_sd + S - 1]));   // max depth
                atomicMax(&cta_keys[1], ~float_to_key(rb[L.o_sd]));          // min depth (complemented)
            }
            __syncwarp();
            if (a.dbg_weights_final) {
                float* o = a.dbg_weights_final + (size_t)(ray0 + r) * (S - 1);
                for (int i = lane; i < S - 1; i += 32) o[i] = rb[L.o_w + i];
            }
        }
        __syncthreads();

        // ---- P6: colour MLP + coefficient-weighted reduction ----------------------------------
        // rgb = sum_i w_i (c_i + c_{i+1})/2 = sum_j c_j (w_{j-1} + w_j)/2  (ray_marcher.py:28,45)
#pragma unroll 1
        for (int pass = 0; pass < 2; ++pass) {
            if (pass == 1 && Sf == 0) break;
            const bool v = pass == 0 ? vC : vF;
            const int row = pass == 0 ? rowC : rowF;
            const int rank = pass == 0 ? rankC : rankF;
            const float* rb = pass == 0 ? rbC : rbF;
            const int g = pass == 0 ? L.gc : L.gf;
            const int rr = pass == 0 ? rC : rF;
            const int grp = pass == 0 ? sC / L.gc : L.NGc + sF / L.gf;
            float coef = 0.f;
            if (v) {
                float wl = rank > 0 ? rb[L.o_w + rank - 1] : 0.f;
                float wr = rb[L.o_w + rank];  // w[S-1] was zeroed
                coef = 0.5f * (wl + wr);
            }
#pragma unroll 1
            for (int net = 0; net < n_nets; ++net) {
                const float* nw = dec + net * kNetFloats;
                float h[kHid];
                if (v) mlp_hidden(nw, feat, row, h);
                const uint32_t smask = a.sigmoid_mask[net];
#pragma unroll 1
                for (int oc = 0; oc < kOut / 8; ++oc) {
                    float acc[8];
                    if (v) {
                        mlp_colors8(nw, h, oc, acc);
#pragma unroll
                        for (int i = 0; i < 8; ++i) {
                            float c = ((smask >> (oc * 8 + i)) & 1u) ? sigmoid_clamp_f(acc[i]) : acc[i];
                            acc[i] = c * coef;
                        }
                    } else {
#pragma unroll
                        for (int i = 0; i < 8; ++i) acc[i] = 0.f;
                    }
                    for (int o = g >> 1; o > 0; o >>= 1) {
#pragma unroll
                        for (int i = 0; i < 8; ++i) acc[i] += __shfl_xor_sync(0xffffffffu, acc[i], o);
                    }
                    if ((lane & (g - 1)) == 0 && rr < RT) {
                        float* dst = part + ((size_t)rr * (L.NGc + L.NGf) + grp) * P.cout + net * kOut + oc * 8;
                        *reinterpret_cast<float4*>(dst) = make_float4(acc[0], acc[1], acc[2], acc[3]);
                        *reinterpret_cast<float4*>(dst + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
                    }
                }
            }
        }
        __syncthreads();
        {
            const int NG = L.NGc + L.NGf;
            for (int i = tid; i < RT * P.cout; i += blockDim.x) {
                int r = i / P.cout, c = i % P.cout;
                if (ray0 + r >= P.total_rays) continue;
                const float* src = part + (size_t)r * NG * P.cout + c;
                float acc = 0.f;
                for (int gi = 0; gi < NG; ++gi) acc += src[gi * P.cout];
                if (a.white_back) acc = acc + 1.f - scal[4 * r + 0];
                a.out_feat[(size_t)(ray0 + r) * P.cout + c] = acc * 2.f - 1.f;
            }
        }
        __syncthreads();
    }

    // ---- global depth clamp: torch.clamp(depth, min(depths), max(depths)) (ray_marcher.py:49-50) ----
    __shared__ bool is_last;
    __threadfence();          // every thread publishes its out_depth stores before the CTA signs off
    __syncthreads();
    if (tid == 0) {
        atomicMax(a.workspace + 0, cta_keys[0]);
        atomicMax(a.workspace + 1, cta_keys[1]);
        __threadfence();
        unsigned done = atomicAdd(a.workspace + 2, 1u);
        is_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        float dmax = key_to_float(atomicMax(a.workspace + 0, 0u));
        float dmin = key_to_float(~atomicMax(a.workspace + 1, 0u));
        for (int i = tid; i < P.total_rays; i += blockDim.x) {
            float v = __ldcg(a.out_depth + i);
            if (v != v) v = __int_as_float(0x7f800000);   // nan_to_num(nan=inf)
            v = fminf(fmaxf(v, dmin), dmax);
            a.out_depth[i] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------
// run_model / sample_from_planes: warp handles 32 points
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) run_model_kernel(const float* __restrict__ planes, const float* __restrict__ coords,
                                                        const float* __restrict__ decoder_packed, int n_nets, int sigma_net,
                                                        uint32_t mask0, uint32_t mask1, int B, int M, int H, int W,
                                                        float coord_scale, float* __restrict__ out_rgb,
                                                        float* __restrict__ out_sigma) {
    extern __shared__ __align__(16) float smem[];
    float* dec = smem;
    float* feat = smem + round_up(n_nets * kNetFloats, 32);
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    {
        const float4* src = reinterpret_cast<const float4*>(decoder_packed);
        float4* dst = reinterpret_cast<float4*>(dec);
        for (int i = tid; i < n_nets * kNetFloats / 4; i += blockDim.x) dst[i] = __ldg(src + i);
    }
    __syncthreads();
    const int64_t total = (int64_t)B * M;
    const int cout = n_nets * kOut;
    float* wfeat = feat + warp * 32 * kC;
    for (int64_t base = ((int64_t)blockIdx.x * (blockDim.x >> 5) + warp) * 32; base < total;
         base += (int64_t)gridDim.x * (blockDim.x >> 5) * 32) {
        int64_t p = base + lane;
        bool v = p < total;
        float px = 0.f, py = 0.f, pz = 0.f;
        int b = 0;
        if (v) {
            b = (int)(p / M);
            px = __fmul_rn(coord_scale, __ldg(coords + p * 3 + 0));
            py = __fmul_rn(coord_scale, __ldg(coords + p * 3 + 1));
            pz = __fmul_rn(coord_scale, __ldg(coords + p * 3 + 2));
        }
        __syncwarp();
        warp_gather(planes, H, W, wfeat, v ? lane : -1, b, px, py, pz, lane);
        if (v) {
#pragma unroll 1
            for (int net = 0; net < n_nets; ++net) {
                const float* nw = dec + net * kNetFloats;
                float h[kHid];
                mlp_hidden(nw, wfeat, lane, h);
                if (net == sigma_net) out_sigma[p] = mlp_sigma(nw, h);
                const uint32_t smask = net == 0 ? mask0 : mask1;
#pragma unroll 1
                for (int oc = 0; oc < kOut / 8; ++oc) {
                    float acc[8];
                    mlp_colors8(nw, h, oc, acc);
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        if ((smask >> (oc * 8 + i)) & 1u) acc[i] = sigmoid_clamp_f(acc[i]);
                    float* dst = out_rgb + p * cout + net * kOut + oc * 8;
                    *reinterpret_cast<float4*>(dst) = make_float4(acc[0], acc[1], acc[2], acc[3]);
                    *reinterpret_cast<float4*>(dst + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
                }
            }
        }
        __syncwarp();
    }
}

// features [B,3,M,32] exactly as sample_from_planes returns them (renderer.py:64)
__global__ void __launch_bounds__(256) sample_planes_kernel(const float* __restrict__ planes, const float* __restrict__ coords,
                                                            int B, int M, int H, int W, float coord_scale,
                                                            float* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const int64_t total = (int64_t)B * M;
    const int64_t wid = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int64_t nw = ((int64_t)gridDim.x * blockDim.x) >> 5;
    const size_t isz = (size_t)3 * H * W * kC;
    for (int64_t p = wid; p < total; p += nw) {
        int b = (int)(p / M);
        int64_t m = p % M;
        float px = __fmul_rn(coord_scale, __ldg(coords + p * 3 + 0));
        float py = __fmul_rn(coord_scale, __ldg(coords + p * 3 + 1));
        float pz = __fmul_rn(coord_scale, __ldg(coords + p * 3 + 2));
        float f0, f1, f2;
        plane_values(planes + (size_t)b * isz, H, W, px, py, pz, lane, f0, f1, f2);
        float* o = out + ((size_t)b * 3 * M + m) * kC + lane;
        o[0] = f0;
        o[(size_t)M * kC] = f1;
        o[(size_t)2 * M * kC] = f2;
    }
}

// ---------------------------------------------------------------------------------------------
// Stand-alone MipRayMarcher2 and sample_importance (stage-level drop-ins)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) ray_march_kernel(const float* __restrict__ colors, const float* __restrict__ dens,
                                                        const float* __restrict__ depths, int N, int S, int Cc,
                                                        int white_back, float* __restrict__ out_rgb,
                                                        float* __restrict__ out_depth, float* __restrict__ out_w,
                                                        uint32_t* __restrict__ workspace) {
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int Sp = round_up(S, 4);
    float* d = smem + warp * 3 * Sp;
    float* s = d + Sp;
    float* w = s + Sp;
    __shared__ uint32_t keys[2];
    if (threadIdx.x < 2) keys[threadIdx.x] = 0u;
    __syncthreads();
    uint32_t kmax = 0u, kmin = 0u;
    for (int ray = blockIdx.x * nwarps + warp; ray < N; ray += gridDim.x * nwarps) {
        for (int i = lane; i < S; i += 32) {
            float dv = __ldg(depths + (size_t)ray * S + i);
            d[i] = dv;
            s[i] = __ldg(dens + (size_t)ray * S + i);
            kmax = max(kmax, float_to_key(dv));
            kmin = max(kmin, ~float_to_key(dv));
        }
        __syncwarp();
        float sw, swd;
        warp_march(d, s, S, w, lane, sw, swd);
        __syncwarp();
        for (int i = lane; i < S - 1; i += 32) out_w[(size_t)ray * (S - 1) + i] = w[i];
        if (lane == 0) out_depth[ray] = __fdiv_rn(swd, sw);
        const float* col = colors + (size_t)ray * S * Cc;
        for (int c = lane; c < Cc; c += 32) {
            float acc = 0.f;
            float prev = __ldg(col + c);
            for (int i = 0; i < S - 1; ++i) {
                float nxt = __ldg(col + (size_t)(i + 1) * Cc + c);
                acc = fmaf(w[i], __fmul_rn(__fadd_rn(prev, nxt), 0.5f), acc);
                prev = nxt;
            }
            if (white_back) acc = acc + 1.f - sw;
            out_rgb[(size_t)ray * Cc + c] = acc * 2.f - 1.f;
        }
        __syncwarp();
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
        kmin = max(kmin, __shfl_xor_sync(0xffffffffu, kmin, o));
    }
    if (lane == 0) { atomicMax(&keys[0], kmax); atomicMax(&keys[1], kmin); }
    __threadfence();
    __syncthreads();
    __shared__ bool is_last;
    if (threadIdx.x == 0) {
        atomicMax(workspace + 0, keys[0]);
        atomicMax(workspace + 1, keys[1]);
        __threadfence();
        unsigned done = atomicAdd(workspace + 2, 1u);
        is_last = (done == gridDim.x - 1);
    }
    __syncthreads();
    if (is_last) {
        __threadfence();
        float dmax = key_to_float(atomicMax(workspace + 0, 0u));
        float dmin = key_to_float(~atomicMax(workspace + 1, 0u));
        for (int i = threadIdx.x; i < N; i += blockDim.x) {
            float v = __ldcg(out_depth + i);
            if (v != v) v = __int_as_float(0x7f800000);
            out_depth[i] = fminf(fmaxf(v, dmin), dmax);
        }
    }
}

__global__ void __launch_bounds__(128) sample_importance_kernel(const float* __restrict__ z_vals, const float* __restrict__ weights,
                                                                const float* __restrict__ u, int N, int S, int Sf,
                                                                float* __restrict__ out, int32_t* __restrict__ out_inds) {
    extern __shared__ __align__(16) float smem[];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarps = blockDim.x >> 5;
    const int Sp = round_up(S, 4);
    float* z = smem + warp * 4 * Sp;
    float* w = z + Sp;
    float* om = w + Sp;
    float* cdf = om + Sp;
    for (int ray = blockIdx.x * nwarps + warp; ray < N; ray += gridDim.x * nwarps) {
        for (int i = lane; i < S; i += 32) z[i] = __ldg(z_vals + (size_t)ray * S + i);
        for (int i = lane; i < S - 1; i += 32) w[i] = __ldg(weights + (size_t)ray * (S - 1) + i);
        __syncwarp();
        warp_importance_cdf(w, S, om, cdf, lane);
        for (int k = lane; k < Sf; k += 32) {
            int inds;
            float v = importance_sample(cdf, z, S, __ldg(u + (size_t)ray * Sf + k), inds);
            out[(size_t)ray * Sf + k] = v;
            if (out_inds) out_inds[(size_t)ray * Sf + k] = inds;
        }
        __syncwarp();
    }
}

// SMs of the CURRENT device, queried on every call (an attribute read, no cache: the library keeps no state and a process
// may drive several devices)
int sm_count() {
    int dev = 0, n = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) return 148;
    return n;
}

}  // namespace p3d

using namespace p3d;

extern "C" {

int p3d_abi_version(void) { return 7; }
const char* p3d_build_info(void) { return "libp3d sm_100a " __DATE__ " " __TIME__; }
const char* p3d_status_string(int status) {
    if (status == P3D_OK) return "ok";
    if (status == P3D_UNSUPPORTED) return "unsupported configuration";
    if (status == P3D_BAD_ARG) return "bad argument";
    if (status > 0) return cudaGetErrorString((cudaError_t)status);
    return "unknown";
}

int p3d_ray_limits_box(const float* rays_o, const float* rays_d, int64_t N, float box_side_length, float* t_near, float* t_far,
                       p3d_stream_t stream) {
    if (!rays_o || !rays_d || !t_near || !t_far || N < 0) return P3D_BAD_ARG;
    if (N == 0) return P3D_OK;
    const int threads = 256;
    const int64_t blocks = (N + threads - 1) / threads;
    if (blocks > INT32_MAX) return P3D_UNSUPPORTED;
    ray_limits_box_kernel<<<(unsigned)blocks, threads, 0, (cudaStream_t)stream>>>(rays_o, rays_d, N, box_side_length / 2, t_near, t_far);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

int p3d_ray_sampler(const float* cam2world, const float* intrinsics, int B, int res, float* origins, float* dirs,
                    p3d_stream_t stream) {
    if (!cam2world || !intrinsics || !origins || !dirs || B <= 0 || res <= 0) return P3D_BAD_ARG;
    int64_t n = (int64_t)B * res * res;
    int block = 256;
    ray_sampler_kernel<<<(unsigned)ceil_div64(n, block), block, 0, (cudaStream_t)stream>>>(cam2world, intrinsics, B, res,
                                                                                           origins, dirs);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

int p3d_planes_to_channels_last(const float* in, float* out, int N, int C, int H, int W, p3d_stream_t stream) {
    if (!in || !out || N <= 0 || C <= 0 || H <= 0 || W <= 0) return P3D_BAD_ARG;
    if (N > 65535) return P3D_UNSUPPORTED;
    dim3 grid(ceil_div(H * W, 32), ceil_div(C, 32), N), block(32, 8);
    planes_to_cl_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(in, out, C, H * W);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

int p3d_pack_decoder(const p3d_decoder_t* dec, float* packed, p3d_stream_t stream) {
    if (!dec || !packed || dec->n_nets < 1 || dec->n_nets > 2) return P3D_BAD_ARG;
    PackArgs a;
    a.n_nets = dec->n_nets;
    for (int i = 0; i < 2; ++i) {
        a.w1[i] = dec->w1[i]; a.b1[i] = dec->b1[i]; a.w2[i] = dec->w2[i]; a.b2[i] = dec->b2[i];
        a.w1g[i] = dec->w1_gain[i]; a.b1g[i] = dec->b1_gain[i]; a.w2g[i] = dec->w2_gain[i]; a.b2g[i] = dec->b2_gain[i];
        if (i < dec->n_nets && (!a.w1[i] || !a.b1[i] || !a.w2[i] || !a.b2[i])) return P3D_BAD_ARG;
    }
    pack_decoder_kernel<<<dim3(8, 2), 256, 0, (cudaStream_t)stream>>>(a, packed);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

int p3d_render_fwd(const p3d_render_args_t* args, p3d_stream_t stream) {
    if (!args) return P3D_BAD_ARG;
    const p3d_render_args_t& a = *args;
    if (!a.planes_nhwc || !a.ray_origins || !a.ray_dirs || !depth_args_ok(a) || !a.decoder_packed || !a.out_feat ||
        !a.out_depth || !a.out_wsum || !a.workspace)
        return P3D_BAD_ARG;
    if (a.plane_strides[0] || a.plane_strides[1] || a.plane_strides[2]) {
        const int64_t psz = (int64_t)a.H * a.W * kC;
        if (a.plane_strides[0] != 3 * psz || a.plane_strides[1] != psz || a.plane_strides[2] != kC) return P3D_UNSUPPORTED;
    }
    if (a.B <= 0 || a.R <= 0 || a.H <= 0 || a.W <= 0 || a.Sc < 2 || a.Sf < 0) return P3D_BAD_ARG;
    if (a.Sf > 0 && (!a.u_importance || a.Sc < 4)) return P3D_BAD_ARG;
    if (a.n_nets < 1 || a.n_nets > 2 || a.sigma_net < 0 || a.sigma_net >= a.n_nets) return P3D_BAD_ARG;
    if (a.Sc + a.Sf > 32 * kMaxIvPerLane) return P3D_UNSUPPORTED;
    if ((int64_t)a.B * a.R > INT32_MAX / (a.Sc + a.Sf + 1)) return P3D_UNSUPPORTED;

    int dev = 0, max_smem = 0;
    P3D_CUDA_TRY(cudaGetDevice(&dev));
    P3D_CUDA_TRY(cudaDeviceGetAttribute(&max_smem, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    const int nsm = sm_count();

    // rays per CTA: as many as fit two CTAs per SM within 256 threads
    const int mx = round_up(a.Sc > a.Sf ? a.Sc : a.Sf, 8);
    int RT = 256 / mx;
    if (RT < 1) return P3D_UNSUPPORTED;
    if (RT > 8) RT = 8;
    RenderLayout L = make_layout(RT, a.Sc, a.Sf, a.n_nets);
    const int budget2 = (max_smem - 2048) / 2;
    while (RT > 1 && (int)(L.total_floats * sizeof(float)) > budget2) { --RT; L = make_layout(RT, a.Sc, a.Sf, a.n_nets); }
    size_t smem = (size_t)L.total_floats * sizeof(float);
    if ((int)smem > max_smem) return P3D_UNSUPPORTED;

    RenderParams P;
    P.a = a; P.L = L;
    P.total_rays = a.B * a.R;
    P.n_tiles = ceil_div(P.total_rays, RT);
    P.cout = kOut * a.n_nets;
    P3D_CUDA_TRY(cudaMemsetAsync(a.workspace, 0, 4 * sizeof(uint32_t), (cudaStream_t)stream));
    P3D_CUDA_TRY(cudaFuncSetAttribute(render_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    P3D_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, render_fwd_kernel, L.NT, smem));
    if (per_sm < 1) per_sm = 1;
    int grid = nsm * per_sm;
    if (grid > P.n_tiles) grid = P.n_tiles;
    render_fwd_kernel<<<grid, L.NT, smem, (cudaStream_t)stream>>>(P);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

int p3d_run_model(const float* planes_nhwc, const float* coords, const float* decoder_packed, int n_nets, int sigma_net,
                  const uint32_t sigmoid_mask[2], int B, int M, int H, int W, float coord_scale, float* out_rgb,
                  float* out_sigma, p3d_stream_t stream) {
    if (!planes_nhwc || !coords || !decoder_packed || !out_rgb || !out_sigma || !sigmoid_mask) return P3D_BAD_ARG;
    if (B <= 0 || M <= 0 || n_nets < 1 || n_nets > 2 || sigma_net < 0 || sigma_net >= n_nets) return P3D_BAD_ARG;
    const int block = 128;
    size_t smem = (size_t)(round_up(n_nets * kNetFloats, 32) + (block / 32) * 32 * kC) * sizeof(float);
    P3D_CUDA_TRY(cudaFuncSetAttribute(run_model_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 1;
    P3D_CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, run_model_kernel, block, smem));
    if (per_sm < 1) per_sm = 1;
    int64_t need = ceil_div64((int64_t)B * M, block);
    int grid = (int)(need < (int64_t)sm_count() * per_sm ? need : (int64_t)sm_count() * per_sm);
    run_model_kernel<<<grid, block, smem, (cudaStream_t)stream>>>(planes_nhwc, coords, decoder_packed, n_nets, sigma_net,
                                                                  sigmoid_mask[0], sigmoid_mask[1], B, M, H, W,
                                                                  coord_scale, out_rgb, out_sigma);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

int p3d_sample_from_planes(const float* planes_nhwc, const float* coords, int B, int M, int H, int W, float coord_scale,
                           float* out_features, p3d_stream_t stream) {
    if (!planes_nhwc || !coords || !out_features || B <= 0 || M <= 0) return P3D_BAD_ARG;
    const int block = 256;
    int64_t need = ceil_div64((int64_t)B * M * 32, block);
    int64_t cap = (int64_t)sm_count() * 16;
    int grid = (int)(need < cap ? need : cap);
    sample_planes_kernel<<<grid, block, 0, (cudaStream_t)stream>>>(planes_nhwc, coords, B, M, H, W, coord_scale,
                                                                   out_features);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

int p3d_ray_march(const float* colors, const float* densities, const float* depths, int N, int S, int Cc, int white_back,
                  float* out_rgb, float* out_depth, float* out_weights, uint32_t* workspace, p3d_stream_t stream) {
    if (!colors || !densities || !depths || !out_rgb || !out_depth || !out_weights || !workspace) return P3D_BAD_ARG;
    if (N <= 0 || S < 2 || Cc <= 0) return P3D_BAD_ARG;
    if (S > 32 * kMaxIvPerLane) return P3D_UNSUPPORTED;
    const int block = 128;
    size_t smem = (size_t)(block / 32) * 3 * round_up(S, 4) * sizeof(float);
    P3D_CUDA_TRY(cudaMemsetAsync(workspace, 0, 4 * sizeof(uint32_t), (cudaStream_t)stream));
    int64_t need = ceil_div64(N, block / 32);
    int64_t cap = (int64_t)sm_count() * 8;
    int grid = (int)(need < cap ? need : cap);
    ray_march_kernel<<<grid, block, smem, (cudaStream_t)stream>>>(colors, densities, depths, N, S, Cc, white_back, out_rgb,
                                                                  out_depth, out_weights, workspace);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

int p3d_sample_importance(const float* z_vals, const float* weights, const float* u, int N, int S, int Sf,
                          float* out_samples, int32_t* out_inds, p3d_stream_t stream) {
    if (!z_vals || !weights || !u || !out_samples) return P3D_BAD_ARG;
    if (N <= 0 || S < 4 || Sf <= 0) return P3D_BAD_ARG;
    const int block = 128;
    size_t smem = (size_t)(block / 32) * 4 * round_up(S, 4) * sizeof(float);
    if (smem > 48 * 1024) return P3D_UNSUPPORTED;
    int64_t need = ceil_div64(N, block / 32);
    int64_t cap = (int64_t)sm_count() * 8;
    int grid = (int)(need < cap ? need : cap);
    sample_importance_kernel<<<grid, block, smem, (cudaStream_t)stream>>>(z_vals, weights, u, N, S, Sf, out_samples,
                                                                          out_inds);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

}  // extern "C"
