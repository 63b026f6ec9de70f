// Implicit-GEMM convolution on the 5th-generation tensor cores (tcgen05, sm_100a) for the modulated 3x3 / 1x1
// convolutions of the synthesis and super-resolution blocks (reference: training/networks_stylegan2.py:34-91,
// torch_utils/ops/conv2d_resample.py:48-143, which bottom out in cuDNN).
//
//   D[128 pixels x BN channels] (TMEM, fp32) += A[128 x 64] (smem) * B[BN x 64]^T (smem), fp16 operands
//
// * Activations are NHWC fp16, so the im2col operand of one filter tap is a plain 4-D TMA box
//   {64 channels, BW, BH, 1 image} shifted by the tap offset; out-of-bounds coordinates are zero-filled by the
//   TMA unit, which implements the convolution padding (and the borders of the transposed-conv phases) for free.
// * Weights are pre-modulated per sample (w * style * demod, fused_modconv semantics) and stored K-major
//   [B][Cout][taps*Cin] fp16.
// * fp32 layers (the tri-plane backbone) run as three fp16 passes over split operands, x = hi + lo,
//   hi*hi + hi*lo + lo*hi, accumulated in the same fp32 TMEM tile (error ~2^-22, products are exact in fp32).
// * Warp roles: warp 0 = TMA producer, warp 1 = TMEM owner + single-thread MMA issuer, warps 2-5 = epilogue
//   (tcgen05.ld -> scale/noise/bias/activation/clamp -> NHWC store). mbarrier ring of kStages smem stages.
// * A launch may carry up to four PHASES (ConvPhase: tap subset, grid, output offset): the four parities of a stride-2
//   transposed 3x3 convolution run as one launch whose tile order walks them heaviest first (p3d_conv_gemm_phases).
// * The persistent kernel can also evaluate the NEXT layer's 1x1 ToRGB + skip on the outputs it holds (rgb_* arguments): the last
//   super-resolution block then needs no ToRGB launch and never writes its activation tensor.
#include <stdlib.h>
#include <string.h>
#include "p3d_common.cuh"
#include "tc05.cuh"
#include "tmap.cuh"

namespace p3d {

constexpr int kBM = 128;        // pixels per tile (= TMEM lanes)
constexpr int kBK = 64;         // fp16 elements per k-step (128-byte swizzle span)
constexpr int kMaxGroups = 27;  // 9 taps x 3 precision passes

// One output phase of a launch. An ordinary convolution has one; a stride-2 transposed convolution run as ONE launch has four
// (tap subsets of the same weight tensor over the same input, each writing its own parity of the (2H+1) x (2W+1) grid).
struct ConvPhase {
    int g0, ng;                       // groups [g0, g0 + ng) of the k-loop tables below
    int gH, gW, oy, ox;               // computed grid and output offset (Y = y*sy + oy)
    int tiles_x, tiles_y;             // tiles of this phase's grid
    int t0;                           // first tile of the phase in the launch's tile order
    int pad;
    long long p0;                     // split-K: offset (floats) of the phase's partials [splits][B][gH][gW][Cout_pad]
};

struct ConvKernelArgs {
    // k-loop: groups of (tap, A plane, B plane); each group covers Cin channels in kc steps
    int n_phases, kc_steps;
    ConvPhase ph[4];
    int8_t dy[kMaxGroups], dx[kMaxGroups], a_plane[kMaxGroups], b_plane[kMaxGroups], tap[kMaxGroups];
    int Cin;
    // tiling
    int BW, BH, BN, w_per_sample;
    uint32_t idesc, tmem_cols;
    // epilogue
    int oH, oW, sy, sx;               // output tensor size and the stride of the output map (Y = y*sy + phase.oy)
    int Cout, y_cstride, y_coff;      // valid channels, channel stride of the output tensor, channel offset
    void* y; void* y_lo;
    int out_mode;                     // 0: f16, 1: f16 hi/lo split, 2: f32, 3: f32 accumulate (+=)
    const float* bias; const float* noise; const float* dscale;
    int64_t noise_bstride;            // elements between the noise images of consecutive samples (0: one image for the batch)
    float alpha, clamp, acc_scale;
    int base_aligned;                 // y / y_lo are 32-byte aligned (256-bit stores allowed)
    int splits;                       // split-K: blockIdx.z = b * splits + s; s covers k-steps [s*total/splits, (s+1)*total/splits)
    float* partial;                   // split-K: raw fp32 accumulators, per phase [splits][B][gH][gW][Cout_pad] (finished by a second kernel)
    int Cout_pad;
    // fused ToRGB tail (SynthesisBlock.forward, networks_stylegan2.py:452-458): out = upsample2d(prev, f) + [fp16-rounded] y
    const float* up_prev;             // [B, oH/2, oW/2, Cout] fp32 NHWC skip image of the previous block, or NULL
    const float* up_f;                // 4x4 FIR
    int stride;                       // input pixels per output pixel (1, or 2 for the down=2 layers)
    const float* residual;            // fp32 [B, oH, oW, Cout]: added after the activation (resnet skip), or NULL
    int round16, out_nchw;            // round y to fp16 first (fp16 blocks); write [B, Cout, oH, oW] instead of NHWC
    float pre_gain, post_gain;        // gain folded into scale/bias/noise (lrelu is positively homogeneous) or applied last
    // fused ToRGB of the next layer (persistent kernel only; p3d_conv_args_t::rgb_*)
    const __half* rgb_w; const float* rgb_bias; const float* rgb_prev; const float* rgb_f; float* rgb_out;
    int rgb_cout, rgb_w_rows, rgb_skip_x;
    float rgb_clamp, rgb_acc_scale;
};

// phase that owns tile `t` of the launch's tile order (phases are consecutive ranges starting at ph[q].t0)
__device__ __forceinline__ ConvPhase conv_phase_of(const ConvKernelArgs& a, int t) {
    ConvPhase P = a.ph[0];
#pragma unroll
    for (int q = 1; q < 4; ++q)
        if (q < a.n_phases && t >= a.ph[q].t0) P = a.ph[q];
    return P;
}

// 256-bit global accesses (sm_100): one full 32-byte sector per lane
__device__ __forceinline__ void st_global_256(void* p, const uint32_t (&v)[8]) {
    asm volatile("st.global.v8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};" ::"l"(p), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]),
                 "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7])
                 : "memory");
}
__device__ __forceinline__ void ld_global_256(const void* p, uint32_t (&v)[8]) {
    asm volatile("ld.global.v8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "l"(p)
                 : "memory");
}

// kAct: 0 linear, 1 leaky-relu with 0 <= alpha <= 1 (max form), 2 leaky-relu, any alpha (select form)
template <int kAct, bool kClamp>
__device__ __forceinline__ float conv_epilogue_act(float x, float alpha, float post_gain, float clamp) {
    if (kAct == 1) x = fmaxf(x, x * alpha);
    if (kAct == 2) x = x > 0.f ? x : x * alpha;
    x *= post_gain;                                   // 1.0 when the gain was folded (always, for gain > 0)
    if (kClamp) x = fminf(fmaxf(x, -clamp), clamp);
    return x;
}

// Epilogue of one 32-channel chunk held by a thread (= one pixel): per-channel constants from shared memory, noise,
// activation, clamp, and the store in the requested output mode.
template <int kAct, bool kClamp>
__device__ __forceinline__ void conv_store_chunk(const ConvKernelArgs& a, uint32_t (&v)[32], const float* s_scale,
                                                 const float* s_bias, int c0, int ch0, size_t off, float nz, bool vec_ok,
                                                 int b, int Y, int X, float* xq = nullptr, bool do_store = true) {
    const float alpha = a.alpha, post_gain = a.post_gain, clampv = a.clamp;
    const int out_mode = a.out_mode;
    if (a.up_prev) {
        // out = upsample2d(prev)[b, Y, X, :] + y. Polyphase form of the zero-insert x2 + 4x4 FIR + gain 4 (upfirdn2d.py:344-350):
        // output row Y = 2*iy + py reads prev rows iy - 1 + py + {0, 1} with filter taps of parity py (same in x).
        const int ph = a.oH >> 1, pw = a.oW >> 1, C = a.Cout;
        const int iy = Y >> 1, py = Y & 1, ix = X >> 1, px = X & 1;
        float w4[2][2];
        const float* pp[2][2];
#pragma unroll
        for (int aa = 0; aa < 2; ++aa)
#pragma unroll
            for (int cc = 0; cc < 2; ++cc) {
                const int ry = iy - 1 + py + aa, rx = ix - 1 + px + cc;
                const bool ok = ry >= 0 && ry < ph && rx >= 0 && rx < pw;
                w4[aa][cc] = ok ? __ldg(a.up_f + (3 - (py + 2 * aa)) * 4 + (3 - (px + 2 * cc))) * 4.f : 0.f;
                pp[aa][cc] = a.up_prev + (((size_t)b * ph + (ok ? ry : 0)) * pw + (ok ? rx : 0)) * C;
            }
        const int nvalid = min(32, C - ch0);
        float* yo = reinterpret_cast<float*>(a.y);
        if (!a.out_nchw && (C & 7) == 0 && nvalid == 32 && a.base_aligned && ((reinterpret_cast<uintptr_t>(a.up_prev) & 31) == 0)) {
            // one full 32-byte sector per lane and access: the lanes of a warp are different pixels (C * 4 bytes apart), so the
            // number of sectors an access touches is what its cost follows
#pragma unroll
            for (int g8 = 0; g8 < 4; ++g8) {
                const int ch = ch0 + 8 * g8;
                float u[8];
#pragma unroll
                for (int t = 0; t < 8; ++t) u[t] = 0.f;
#pragma unroll
                for (int aa = 0; aa < 2; ++aa)
#pragma unroll
                    for (int cc = 0; cc < 2; ++cc) {
                        uint32_t tq[8];
                        ld_global_256(pp[aa][cc] + ch, tq);
                        const float w = w4[aa][cc];
#pragma unroll
                        for (int t = 0; t < 8; ++t) u[t] = fmaf(w, __uint_as_float(tq[t]), u[t]);
                    }
                uint32_t o[8];
#pragma unroll
                for (int t = 0; t < 8; ++t) {
                    float x = conv_epilogue_act<kAct, kClamp>(fmaf(__uint_as_float(v[8 * g8 + t]), s_scale[c0 + 8 * g8 + t], s_bias[c0 + 8 * g8 + t]) + nz,
                                                              alpha, post_gain, clampv);
                    if (a.round16) x = __half2float(__float2half_rn(x));
                    o[t] = __float_as_uint(u[t] + x);
                }
                st_global_256(yo + off + 8 * g8, o);
            }
        } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                if (i >= nvalid) break;
                const int ch = ch0 + i;
                float u = 0.f;
#pragma unroll
                for (int aa = 0; aa < 2; ++aa)
#pragma unroll
                    for (int cc = 0; cc < 2; ++cc) u = fmaf(w4[aa][cc], __ldg(pp[aa][cc] + ch), u);
                float x = conv_epilogue_act<kAct, kClamp>(fmaf(__uint_as_float(v[i]), s_scale[c0 + i], s_bias[c0 + i]) + nz, alpha,
                                                          post_gain, clampv);
                if (a.round16) x = __half2float(__float2half_rn(x));
                const size_t o = a.out_nchw ? (((size_t)b * C + ch) * a.oH + Y) * a.oW + X : off + i;
                yo[o] = u + x;
            }
        }
        return;
    }
                if (vec_ok) {
    #pragma unroll
                    for (int j = 0; j < 2; ++j) {           // 16 channels per step
                        float r[16];
    #pragma unroll
                        for (int t4 = 0; t4 < 4; ++t4) {
                            const float4 sc = *reinterpret_cast<const float4*>(s_scale + c0 + 16 * j + 4 * t4);
                            const float4 bi = *reinterpret_cast<const float4*>(s_bias + c0 + 16 * j + 4 * t4);
                            const uint32_t* vv = v + 16 * j + 4 * t4;
                            r[4 * t4 + 0] = fmaf(__uint_as_float(vv[0]), sc.x, bi.x) + nz;
                            r[4 * t4 + 1] = fmaf(__uint_as_float(vv[1]), sc.y, bi.y) + nz;
                            r[4 * t4 + 2] = fmaf(__uint_as_float(vv[2]), sc.z, bi.z) + nz;
                            r[4 * t4 + 3] = fmaf(__uint_as_float(vv[3]), sc.w, bi.w) + nz;
                        }
    #pragma unroll
                        for (int t = 0; t < 16; ++t) r[t] = conv_epilogue_act<kAct, kClamp>(r[t], alpha, post_gain, clampv);
                        if (a.residual) {       // resnet skip (networks_stylegan2.py:524-528): added after the activation
                            const float* rp = a.residual + (((size_t)b * a.oH + Y) * a.oW + X) * a.Cout + ch0 + 16 * j;
    #pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                uint32_t o[8];
                                ld_global_256(rp + 8 * h, o);
    #pragma unroll
                                for (int t = 0; t < 8; ++t) r[8 * h + t] += __uint_as_float(o[t]);
                            }
                        }
                        if (out_mode >= 2) {
                            float* yp = reinterpret_cast<float*>(a.y) + off + 16 * j;
    #pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                uint32_t o[8];
                                if (out_mode == 3) {
                                    ld_global_256(yp + 8 * h, o);
    #pragma unroll
                                    for (int t = 0; t < 8; ++t) o[t] = __float_as_uint(__uint_as_float(o[t]) + r[8 * h + t]);
                                } else {
    #pragma unroll
                                    for (int t = 0; t < 8; ++t) o[t] = __float_as_uint(r[8 * h + t]);
                                }
                                st_global_256(yp + 8 * h, o);
                            }
                        } else {
                            uint32_t oh[8], ol[8];
    #pragma unroll
                            for (int t = 0; t < 8; ++t) {
                                const __half2 hv = __floats2half2_rn(r[2 * t], r[2 * t + 1]);
                                oh[t] = *reinterpret_cast<const uint32_t*>(&hv);
                                if (xq) {           // the fp16-rounded outputs, for the fused ToRGB of the next layer
                                    const float2 back = __half22float2(hv);
                                    xq[16 * j + 2 * t] = back.x; xq[16 * j + 2 * t + 1] = back.y;
                                }
                                if (out_mode == 1) {
                                    const float2 back = __half22float2(hv);
                                    const __half2 lv = __floats2half2_rn(r[2 * t] - back.x, r[2 * t + 1] - back.y);
                                    ol[t] = *reinterpret_cast<const uint32_t*>(&lv);
                                }
                            }
                            if (do_store) st_global_256(reinterpret_cast<__half*>(a.y) + off + 16 * j, oh);
                            if (out_mode == 1) st_global_256(reinterpret_cast<__half*>(a.y_lo) + off + 16 * j, ol);
                        }
                    }
                } else {
                    // ragged chunk (ToRGB's 3 channels, channel tails, unaligned concat offsets): scalar stores
                    const int nvalid = min(32, a.Cout - ch0);
    #pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        if (i < nvalid) {
                            float x = conv_epilogue_act<kAct, kClamp>(
                                fmaf(__uint_as_float(v[i]), s_scale[c0 + i], s_bias[c0 + i]) + nz, alpha, post_gain, clampv);
                            if (a.residual) x += __ldg(a.residual + (((size_t)b * a.oH + Y) * a.oW + X) * a.Cout + ch0 + i);
                            if (out_mode <= 1) {
                                const __half h = __float2half_rn(x);
                                reinterpret_cast<__half*>(a.y)[off + i] = h;
                                if (out_mode == 1) reinterpret_cast<__half*>(a.y_lo)[off + i] = __float2half_rn(x - __half2float(h));
                            } else {
                                float* yf = reinterpret_cast<float*>(a.y) + off + i;
                                *yf = (out_mode == 3 ? *yf : 0.f) + x;
                            }
                        }
                    }
                }
}

template <int kStages, int kAct, bool kClamp>
__global__ void __launch_bounds__(192, 2) conv_gemm_kernel(const __grid_constant__ CUtensorMap tmA,
                                                           const __grid_constant__ CUtensorMap tmB,
                                                           const ConvKernelArgs a) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    // carve: [stages][A 16 KB][B BN*128 B] | barriers | tmem ptr | per-channel scale, bias
    // round up inside the shared window (pointer arithmetic on smem_raw keeps the address space known to the compiler)
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t a_bytes = (uint32_t)kBM * 128, b_bytes = (uint32_t)a.BN * 128;
    const uint32_t stage_bytes = a_bytes + b_bytes;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kStages * stage_bytes);
    uint64_t* empty_bar = full_bar + kStages;
    uint64_t* tmem_full_bar = empty_bar + kStages;
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_full_bar + 1);
    float* s_scale = reinterpret_cast<float*>(smem + kStages * stage_bytes + (((2 * kStages + 1) * 8 + 4 + 15) & ~15));
    float* s_bias = s_scale + 128;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int tile_n = blockIdx.y;
    const ConvPhase P = conv_phase_of(a, (int)blockIdx.x);      // t0 counts spatial tiles here (blockIdx.x)
    const int tile_m = (int)blockIdx.x - P.t0;
    const int b = blockIdx.z / a.splits, ksplit = blockIdx.z - b * a.splits;
    const int ty = tile_m / P.tiles_x, tx = tile_m % P.tiles_x;
    const int n0 = tile_n * a.BN;
    const int all_k = P.ng * a.kc_steps;
    const int k_begin = (int)((long long)all_k * ksplit / a.splits), k_end = (int)((long long)all_k * (ksplit + 1) / a.splits);
    const int total_k = k_end - k_begin;

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmA);
        tc::tma_prefetch_desc(&tmB);
        for (int s = 0; s < kStages; ++s) { tc::mbar_init(&full_bar[s], 1); tc::mbar_init(&empty_bar[s], 1); }
        tc::mbar_init(tmem_full_bar, 1);
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_ptr_smem, a.tmem_cols);
    if (warp >= 2) {
        // per-channel epilogue constants: accumulator scale (1/weight scale x demodulation x gain) and bias x gain; channels
        // beyond Cout get zeros so the hot loop needs no channel predicate
        const int i = threadIdx.x - 64;
        if (i < a.BN) {
            const int ch = n0 + i;
            float sc = 0.f, bi = 0.f;
            if (ch < a.Cout) {
                sc = a.acc_scale * a.pre_gain;
                if (a.dscale) sc *= __ldg(a.dscale + (size_t)b * a.Cout + ch);
                if (a.bias) bi = __ldg(a.bias + ch) * a.pre_gain;
            }
            s_scale[i] = sc;
            s_bias[i] = bi;
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int g = k_begin / a.kc_steps, kc = k_begin - g * a.kc_steps;
            g += P.g0;
            for (int k = 0; k < total_k; ++k) {
                const int x0 = tx * a.BW * a.stride + a.dx[g], y0 = ty * a.BH * a.stride + a.dy[g];
                const int kb = a.tap[g] * a.Cin;
                tc::mbar_wait(&empty_bar[stage], phase ^ 1);
                uint8_t* sa = smem + stage * stage_bytes;
                uint8_t* sb = sa + a_bytes;
                tc::mbar_expect_tx(&full_bar[stage], stage_bytes);
                tc::tma_load_5d(sa, &tmA, &full_bar[stage], kc * kBK, x0, y0, b, a.a_plane[g]);
                tc::tma_load_4d(sb, &tmB, &full_bar[stage], kb + kc * kBK, n0, a.w_per_sample ? b : 0, a.b_plane[g]);
                if (++stage == kStages) { stage = 0; phase ^= 1; }
                if (++kc == a.kc_steps) { kc = 0; ++g; }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one thread) =====
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int k = 0; k < total_k; ++k) {
                tc::mbar_wait(&full_bar[stage], phase);
                tc::tc_fence_after();
                const uint32_t sa = tc::smem_u32(smem + stage * stage_bytes);
                const uint64_t da = tc::umma_desc_k128(sa), db = tc::umma_desc_k128(sa + a_bytes);
#pragma unroll
                for (int j = 0; j < kBK / 16; ++j)   // 4 MMAs of K=16: advance 32 bytes inside the swizzle span
                    tc::umma_f16(tmem_base, da + (uint64_t)(j * 2), db + (uint64_t)(j * 2), a.idesc, (k | j) != 0);
                tc::umma_commit(&empty_bar[stage]);                 // frees the smem stage when these MMAs retire
                if (k == total_k - 1) tc::umma_commit(tmem_full_bar);
                if (++stage == kStages) { stage = 0; phase ^= 1; }
            }
        }
    } else {
        // ===== epilogue: warps 2..5 own TMEM lane quarters (warp % 4); thread = pixel, 32 channels per TMEM load =====
        const int q = warp & 3;
        const int m = q * 32 + lane;                    // tile row = TMEM lane
        const int gy = ty * a.BH + m / a.BW, gx = tx * a.BW + m % a.BW;
        const bool pix_ok = (gy < P.gH) && (gx < P.gW);
        const int Y = gy * a.sy + P.oy, X = gx * a.sx + P.ox;
        const size_t pix = ((size_t)b * a.oH + Y) * a.oW + X;
        const float nz = (a.noise && pix_ok) ? __ldg(a.noise + (size_t)b * a.noise_bstride + (size_t)Y * a.oW + X) * a.pre_gain : 0.f;
        const int out_mode = a.out_mode;
        // vector path: every 32-channel chunk of this CTA is full and its stores are 32-byte aligned
        const bool vec_ok = a.base_aligned && ((n0 + a.BN) <= a.Cout) && (a.BN % 32 == 0) &&
                            (out_mode <= 1 ? ((a.y_cstride % 16) == 0 && ((a.y_coff + n0) % 16) == 0)
                                           : ((a.y_cstride % 8) == 0 && ((a.y_coff + n0) % 8) == 0));
        tc::mbar_wait(tmem_full_bar, 0);
        tc::tc_fence_after();
        for (int c0 = 0; c0 < a.BN; c0 += 32) {
            uint32_t v[32];
            tc::tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
            tc::tmem_ld_wait();
            if (!pix_ok) continue;
            const int ch0 = n0 + c0;
            if (a.partial) {
                // split-K: raw accumulators of this k-range; conv_splitk_finish_kernel sums the ranges and applies the epilogue.
                // Partial rows are Cout_pad wide: when Cout_pad > BN is not a multiple of BN, the last channel tile reaches past
                // the row, and those columns would land in the next pixel's row.
                if (ch0 >= a.Cout_pad) continue;
                float* pp = a.partial + P.p0 + ((((size_t)ksplit * (gridDim.z / a.splits) + b) * P.gH + gy) * P.gW + gx) * a.Cout_pad + ch0;
                const int ncols = min(min(32, a.BN - c0), a.Cout_pad - ch0);
#pragma unroll
                for (int j = 0; j < 4; ++j)
                    if (8 * j < ncols) {
                        const uint32_t o[8] = {v[8 * j], v[8 * j + 1], v[8 * j + 2], v[8 * j + 3], v[8 * j + 4], v[8 * j + 5], v[8 * j + 6], v[8 * j + 7]};
                        st_global_256(pp + 8 * j, o);
                    }
                continue;
            }
            if (ch0 >= a.Cout) continue;
            const size_t off = pix * a.y_cstride + a.y_coff + ch0;
            conv_store_chunk<kAct, kClamp>(a, v, s_scale, s_bias, c0, ch0, off, nz, vec_ok, b, Y, X);
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_base, a.tmem_cols);
    }
}

// ---------------------------------------------------------------------------------------------
// Persistent variant for launches with many tiles: one CTA per SM walks a static tile schedule. A tile is 256 pixels
// (two stacked 128-row sub-tiles that share every B stage) x BN channels, so a k-step moves 32 KB + BN*128 B for twice the
// FLOPs of the kernel above (the mainloop is bound by the per-SM L2 -> shared-memory ingest rate, ~50 B/clk). The four
// 128-column accumulators are double-buffered in TMEM (2 tiles x 2 sub-tiles = 512 columns), so the epilogue of tile i
// (warps 2-9, one warp per sub-tile and lane quarter) runs under the MMAs of tile i+1.
// ---------------------------------------------------------------------------------------------
constexpr int kPStages = 4;

template <int kAct, bool kClamp>
__global__ void __launch_bounds__(320, 1) conv_gemm_persist_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                    const __grid_constant__ CUtensorMap tmB,
                                                                    const ConvKernelArgs a, int n_tiles, int tiles_n) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    const uint32_t a_bytes = 2u * kBM * 128, b_bytes = (uint32_t)a.BN * 128;
    const uint32_t stage_bytes = a_bytes + b_bytes;
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kPStages * stage_bytes);
    uint64_t* empty_bar = full_bar + kPStages;
    uint64_t* tmem_full_bar = empty_bar + kPStages;      // [2]
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;        // [2]
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
    float* s_const = reinterpret_cast<float*>(smem + kPStages * stage_bytes + 128);     // [2 parities][scale 128 | bias 128]
    float* s_rgbw = s_const + 512;                                                      // [2 parities][8][128] (fused ToRGB only)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmA);
        tc::tma_prefetch_desc(&tmB);
        for (int s = 0; s < kPStages; ++s) { tc::mbar_init(&full_bar[s], 1); tc::mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { tc::mbar_init(&tmem_full_bar[s], 1); tc::mbar_init(&tmem_empty_bar[s], 8); }
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc(tmem_ptr_smem, 512);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp == 0) {
        // ===== TMA producer =====
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const ConvPhase P = conv_phase_of(a, tile);
                const int lt = tile - P.t0, tiles_m = P.tiles_x * P.tiles_y;
                const int tm = lt % tiles_m, tn = (lt / tiles_m) % tiles_n, b = lt / (tiles_m * tiles_n);
                const int ty = tm / P.tiles_x, tx = tm % P.tiles_x;
                const int n0 = tn * a.BN;
                const int total_k = P.ng * a.kc_steps;
                int g = P.g0, kc = 0;
                for (int k = 0; k < total_k; ++k) {
                    const int x0 = tx * a.BW * a.stride + a.dx[g], y0 = ty * 2 * a.BH * a.stride + a.dy[g];
                    const int kb = a.tap[g] * a.Cin;
                    tc::mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* sa = smem + stage * stage_bytes;
                    tc::mbar_expect_tx(&full_bar[stage], stage_bytes);
                    tc::tma_load_5d(sa, &tmA, &full_bar[stage], kc * kBK, x0, y0, b, a.a_plane[g]);
                    tc::tma_load_4d(sa + a_bytes, &tmB, &full_bar[stage], kb + kc * kBK, n0, a.w_per_sample ? b : 0, a.b_plane[g]);
                    if (++stage == kPStages) { stage = 0; phase ^= 1; }
                    if (++kc == a.kc_steps) { kc = 0; ++g; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer (one thread) =====
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int as = 0; uint32_t aphase = 0;
            for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
                const int total_k = conv_phase_of(a, tile).ng * a.kc_steps;
                tc::mbar_wait(&tmem_empty_bar[as], aphase ^ 1);        // the epilogue drained this accumulator pair
                tc::tc_fence_after();
                const uint32_t acc0 = tmem_base + (uint32_t)(as * 256);
                for (int k = 0; k < total_k; ++k) {
                    tc::mbar_wait(&full_bar[stage], phase);
                    tc::tc_fence_after();
                    const uint32_t sa = tc::smem_u32(smem + stage * stage_bytes);
                    const uint64_t da = tc::umma_desc_k128(sa), db = tc::umma_desc_k128(sa + a_bytes);
#pragma unroll
                    for (int mt = 0; mt < 2; ++mt) {
                        const uint64_t dam = da + (uint64_t)(mt * (kBM * 128 >> 4));
#pragma unroll
                        for (int j = 0; j < kBK / 16; ++j)
                            tc::umma_f16(acc0 + (uint32_t)(mt * 128), dam + (uint64_t)(j * 2), db + (uint64_t)(j * 2), a.idesc, (k | j) != 0);
                    }
                    tc::umma_commit(&empty_bar[stage]);
                    if (k == total_k - 1) tc::umma_commit(&tmem_full_bar[as]);
                    if (++stage == kPStages) { stage = 0; phase ^= 1; }
                }
                if (++as == 2) { as = 0; aphase ^= 1; }
            }
        }
    } else {
        // ===== epilogue: warps 2..9; sub-tile = (warp - 2) / 4, TMEM lane quarter = warp % 4 =====
        const int e = warp - 2, mt = e >> 2, q = warp & 3;
        const int m = q * 32 + lane;                    // row inside the 128-row sub-tile = TMEM lane
        const int et = threadIdx.x - 64;                // 0..255 among the epilogue threads
        int as = 0; uint32_t aphase = 0;
        int parity = 0;
        for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
            const ConvPhase P = conv_phase_of(a, tile);
            const int lt = tile - P.t0, tiles_m = P.tiles_x * P.tiles_y;
            const int tm = lt % tiles_m, tn = (lt / tiles_m) % tiles_n, b = lt / (tiles_m * tiles_n);
            const int ty = tm / P.tiles_x, tx = tm % P.tiles_x;
            const int n0 = tn * a.BN;
            float* s_scale = s_const + parity * 256;
            float* s_bias = s_scale + 128;
            if (et < a.BN) {
                const int ch = n0 + et;
                float sc = 0.f, bi = 0.f;
                if (ch < a.Cout) {
                    sc = a.acc_scale * a.pre_gain;
                    if (a.dscale) sc *= __ldg(a.dscale + (size_t)b * a.Cout + ch);
                    if (a.bias) bi = __ldg(a.bias + ch) * a.pre_gain;
                }
                s_scale[et] = sc;
                s_bias[et] = bi;
            }
            float* s_rw = s_rgbw + parity * 1024;
            if (a.rgb_w) {
                // modulated ToRGB weights of this tile's sample as fp32 [8][128] (rows beyond rgb_cout are zero)
                for (int i = et; i < 8 * 128; i += 256) {
                    const int c = i >> 7, k = i & 127;
                    s_rw[i] = (c < a.rgb_cout && k < a.Cout)
                                  ? __half2float(__ldg(a.rgb_w + ((size_t)b * a.rgb_w_rows + c) * a.Cout + k)) : 0.f;
                }
            }
            tc::named_bar_sync(1, 256);                 // constants of this tile visible to all epilogue warps
            const int gy = (ty * 2 + mt) * a.BH + m / a.BW, gx = tx * a.BW + m % a.BW;
            const bool pix_ok = (gy < P.gH) && (gx < P.gW);
            const int Y = gy * a.sy + P.oy, X = gx * a.sx + P.ox;
            const size_t pix = ((size_t)b * a.oH + Y) * a.oW + X;
            const float nz = (a.noise && pix_ok) ? __ldg(a.noise + (size_t)b * a.noise_bstride + (size_t)Y * a.oW + X) * a.pre_gain : 0.f;
            const bool vec_ok = a.base_aligned && ((n0 + a.BN) <= a.Cout) && (a.BN % 32 == 0) &&
                                (a.out_mode <= 1 ? ((a.y_cstride % 16) == 0 && ((a.y_coff + n0) % 16) == 0)
                                                 : ((a.y_cstride % 8) == 0 && ((a.y_coff + n0) % 8) == 0));
            tc::mbar_wait(&tmem_full_bar[as], aphase);
            tc::tc_fence_after();
            const uint32_t acc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * 256 + mt * 128);
            float dot[8];
#pragma unroll
            for (int c = 0; c < 8; ++c) dot[c] = 0.f;
            for (int c0 = 0; c0 < a.BN; c0 += 32) {
                uint32_t v[32];
                tc::tmem_ld_32x32(acc + (uint32_t)c0, v);
                tc::tmem_ld_wait();
                const int ch0 = n0 + c0;
                if (!pix_ok || ch0 >= a.Cout) continue;
                if (a.rgb_w) {
                    // fused ToRGB of the next layer: dot products of this pixel's fp16-rounded outputs with the 1x1 weights
                    float xq[32];
                    conv_store_chunk<kAct, kClamp>(a, v, s_scale, s_bias, c0, ch0, pix * a.y_cstride + a.y_coff + ch0, nz, vec_ok, b, Y, X,
                                                   xq, a.rgb_skip_x == 0);
#pragma unroll
                    for (int c = 0; c < 8; ++c) {
                        if (c < a.rgb_cout) {
                            const float4* wr = reinterpret_cast<const float4*>(s_rw + c * 128 + c0);
                            float acc_c = dot[c];
#pragma unroll
                            for (int qd = 0; qd < 8; ++qd) {
                                const float4 w4 = wr[qd];
                                acc_c = fmaf(xq[4 * qd], w4.x, acc_c); acc_c = fmaf(xq[4 * qd + 1], w4.y, acc_c);
                                acc_c = fmaf(xq[4 * qd + 2], w4.z, acc_c); acc_c = fmaf(xq[4 * qd + 3], w4.w, acc_c);
                            }
                            dot[c] = acc_c;
                        }
                    }
                } else {
                    conv_store_chunk<kAct, kClamp>(a, v, s_scale, s_bias, c0, ch0, pix * a.y_cstride + a.y_coff + ch0, nz, vec_ok, b, Y, X);
                }
            }
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive(&tmem_empty_bar[as]);      // 8 warps -> accumulator pair free for the MMA warp
            if (a.rgb_w && pix_ok) {
                // out = upsample2d(prev)[b, Y, X, :] + round16(clamp(dot * scale + bias)), written NCHW (lanes = consecutive X)
                const int ph = a.oH >> 1, pw = a.oW >> 1, C = a.rgb_cout;
                const int iy = Y >> 1, py = Y & 1, ix = X >> 1, px = X & 1;
                float w4[2][2];
                const float* pp[2][2];
#pragma unroll
                for (int aa = 0; aa < 2; ++aa)
#pragma unroll
                    for (int cc = 0; cc < 2; ++cc) {
                        const int ry = iy - 1 + py + aa, rx = ix - 1 + px + cc;
                        const bool ok = ry >= 0 && ry < ph && rx >= 0 && rx < pw;
                        w4[aa][cc] = ok ? __ldg(a.rgb_f + (3 - (py + 2 * aa)) * 4 + (3 - (px + 2 * cc))) * 4.f : 0.f;
                        pp[aa][cc] = a.rgb_prev + (((size_t)b * ph + (ok ? ry : 0)) * pw + (ok ? rx : 0)) * C;
                    }
#pragma unroll
                for (int c = 0; c < 8; ++c) {
                    if (c < C) {
                        float u = 0.f;
#pragma unroll
                        for (int aa = 0; aa < 2; ++aa)
#pragma unroll
                            for (int cc = 0; cc < 2; ++cc) u = fmaf(w4[aa][cc], __ldg(pp[aa][cc] + c), u);
                        float x = fmaf(dot[c], a.rgb_acc_scale, a.rgb_bias ? __ldg(a.rgb_bias + c) : 0.f);
                        if (a.rgb_clamp >= 0.f) x = fminf(fmaxf(x, -a.rgb_clamp), a.rgb_clamp);
                        x = __half2float(__float2half_rn(x));
                        a.rgb_out[(((size_t)b * C + c) * a.oH + Y) * a.oW + X] = u + x;
                    }
                }
            }
            if (++as == 2) { as = 0; aphase ^= 1; }
            parity ^= 1;
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc(tmem_base, 512);
    }
}

// ---------------------------------------------------------------------------------------------
// CTA-pair variant (cta_group::2) for layers with >= 256 output channels: the two CTAs of a cluster sit on the two SMs of a
// TPC and issue ONE M=256 x N=256 MMA per k-step. Each CTA stages its own 128 pixel rows of A and HALF of the weight
// tile (128 of the 256 channel rows), so a k-step costs 32 KB per SM for 4.2 MFLOP per SM (131 FLOP/B, against 87 for
// the single-CTA persistent kernel) -- the quantity that bounds these kernels is bytes into each SM per FLOP.
// Persistent over a static schedule of (256-pixel, 256-channel) tiles; accumulators double-buffered (2 x 256 TMEM columns
// per CTA). Leader (cluster rank 0): counts both CTAs' TMA bytes on its `full` barriers and issues the MMAs; completion is
// multicast to both CTAs' `empty` / `tmem_full` barriers; both CTAs' epilogue warps arrive on the leader's `tmem_empty`.
// ---------------------------------------------------------------------------------------------
constexpr int kQStages = 6;

template <int kAct, bool kClamp>
__global__ void __launch_bounds__(320, 1) conv_gemm_pair_kernel(const __grid_constant__ CUtensorMap tmA,
                                                                 const __grid_constant__ CUtensorMap tmB,
                                                                 const ConvKernelArgs a, int n_tiles, int tiles_n) {
    extern __shared__ __align__(1024) uint8_t smem_raw[];
    uint8_t* smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    constexpr uint32_t a_bytes = kBM * 128, b_bytes = 128 * 128, stage_bytes = a_bytes + b_bytes;   // per CTA
    uint64_t* full_bar = reinterpret_cast<uint64_t*>(smem + kQStages * stage_bytes);
    uint64_t* empty_bar = full_bar + kQStages;
    uint64_t* tmem_full_bar = empty_bar + kQStages;      // [2]
    uint64_t* tmem_empty_bar = tmem_full_bar + 2;        // [2] (the leader's are used)
    uint32_t* tmem_ptr_smem = reinterpret_cast<uint32_t*>(tmem_empty_bar + 2);
    float* s_const = reinterpret_cast<float*>(smem + kQStages * stage_bytes + 256);     // [2 parities][scale 256 | bias 256]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = tc::cluster_ctarank();
    const int pair = blockIdx.x >> 1, n_pairs = gridDim.x >> 1;

    if (warp == 0 && lane == 0) {
        tc::tma_prefetch_desc(&tmA);
        tc::tma_prefetch_desc(&tmB);
        for (int s = 0; s < kQStages; ++s) { tc::mbar_init(&full_bar[s], 1); tc::mbar_init(&empty_bar[s], 1); }
        for (int s = 0; s < 2; ++s) { tc::mbar_init(&tmem_full_bar[s], 1); tc::mbar_init(&tmem_empty_bar[s], 16); }
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc_pair(tmem_ptr_smem, 512);
    tc::tc_fence_before();
    __syncthreads();
    tc::cluster_sync_all();                               // both CTAs' barriers exist before any remote arrive / complete_tx
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_ptr_smem;

    if (warp == 0) {
        // ===== TMA producer (both CTAs): own A rows, own half of B; bytes counted on the leader's barrier =====
        if (lane == 0) {
            int stage = 0; uint32_t phase = 0;
            for (int tile = pair; tile < n_tiles; tile += n_pairs) {
                const ConvPhase P = conv_phase_of(a, tile);
                const int lt = tile - P.t0, tiles_m = P.tiles_x * P.tiles_y;
                const int tm = lt % tiles_m, tn = (lt / tiles_m) % tiles_n, b = lt / (tiles_m * tiles_n);
                const int ty = tm / P.tiles_x, tx = tm % P.tiles_x;
                const int n0 = tn * 256 + (int)rank * 128;
                const int total_k = P.ng * a.kc_steps;
                int g = P.g0, kc = 0;
                for (int k = 0; k < total_k; ++k) {
                    const int x0 = tx * a.BW * a.stride + a.dx[g], y0 = (ty * 2 + (int)rank) * a.BH * a.stride + a.dy[g];
                    const int kb = a.tap[g] * a.Cin;
                    tc::mbar_wait(&empty_bar[stage], phase ^ 1);
                    uint8_t* sa = smem + stage * stage_bytes;
                    const uint32_t lead_full = tc::mapa_u32(tc::smem_u32(&full_bar[stage]), 0);
                    if (rank == 0) tc::mbar_expect_tx(&full_bar[stage], 2 * stage_bytes);
                    tc::tma_load_5d_pair(sa, &tmA, lead_full, kc * kBK, x0, y0, b, a.a_plane[g]);
                    tc::tma_load_4d_pair(sa + a_bytes, &tmB, lead_full, kb + kc * kBK, n0, a.w_per_sample ? b : 0, a.b_plane[g]);
                    if (++stage == kQStages) { stage = 0; phase ^= 1; }
                    if (++kc == a.kc_steps) { kc = 0; ++g; }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: one thread of the leader CTA =====
        if (rank == 0 && lane == 0) {
            int stage = 0; uint32_t phase = 0;
            int as = 0; uint32_t aphase = 0;
            for (int tile = pair; tile < n_tiles; tile += n_pairs) {
                const int total_k = conv_phase_of(a, tile).ng * a.kc_steps;
                tc::mbar_wait(&tmem_empty_bar[as], aphase ^ 1);        // both CTAs' epilogues drained this accumulator
                tc::tc_fence_after();
                const uint32_t acc = tmem_base + (uint32_t)(as * 256);
                for (int k = 0; k < total_k; ++k) {
                    tc::mbar_wait(&full_bar[stage], phase);
                    tc::tc_fence_after();
                    const uint32_t sa = tc::smem_u32(smem + stage * stage_bytes);
                    const uint64_t da = tc::umma_desc_k128(sa), db = tc::umma_desc_k128(sa + a_bytes);
#pragma unroll
                    for (int j = 0; j < kBK / 16; ++j)
                        tc::umma_f16_pair(acc, da + (uint64_t)(j * 2), db + (uint64_t)(j * 2), a.idesc, (k | j) != 0);
                    tc::umma_commit_pair(&empty_bar[stage], 3);        // stage free in both CTAs
                    if (k == total_k - 1) tc::umma_commit_pair(&tmem_full_bar[as], 3);
                    if (++stage == kQStages) { stage = 0; phase ^= 1; }
                }
                if (++as == 2) { as = 0; aphase ^= 1; }
            }
        }
    } else {
        // ===== epilogue (both CTAs): warps 2..9; column half = (warp - 2) / 4, TMEM lane quarter = warp % 4 =====
        const int e = warp - 2, hsel = e >> 2, q = warp & 3;
        const int m = q * 32 + lane;
        const int et = threadIdx.x - 64;                // 0..255
        const uint32_t lead_empty0 = tc::mapa_u32(tc::smem_u32(&tmem_empty_bar[0]), 0);
        const uint32_t lead_empty1 = tc::mapa_u32(tc::smem_u32(&tmem_empty_bar[1]), 0);
        int as = 0; uint32_t aphase = 0;
        int parity = 0;
        for (int tile = pair; tile < n_tiles; tile += n_pairs) {
            const ConvPhase P = conv_phase_of(a, tile);
            const int lt = tile - P.t0, tiles_m = P.tiles_x * P.tiles_y;
            const int tm = lt % tiles_m, tn = (lt / tiles_m) % tiles_n, b = lt / (tiles_m * tiles_n);
            const int ty = tm / P.tiles_x, tx = tm % P.tiles_x;
            const int n0 = tn * 256;
            float* s_scale = s_const + parity * 512;
            float* s_bias = s_scale + 256;
            {
                const int ch = n0 + et;
                float sc = 0.f, bi = 0.f;
                if (ch < a.Cout) {
                    sc = a.acc_scale * a.pre_gain;
                    if (a.dscale) sc *= __ldg(a.dscale + (size_t)b * a.Cout + ch);
                    if (a.bias) bi = __ldg(a.bias + ch) * a.pre_gain;
                }
                s_scale[et] = sc;
                s_bias[et] = bi;
            }
            tc::named_bar_sync(1, 256);
            const int gy = (ty * 2 + (int)rank) * a.BH + m / a.BW, gx = tx * a.BW + m % a.BW;
            const bool pix_ok = (gy < P.gH) && (gx < P.gW);
            const int Y = gy * a.sy + P.oy, X = gx * a.sx + P.ox;
            const size_t pix = ((size_t)b * a.oH + Y) * a.oW + X;
            const float nz = (a.noise && pix_ok) ? __ldg(a.noise + (size_t)b * a.noise_bstride + (size_t)Y * a.oW + X) * a.pre_gain : 0.f;
            const bool vec_ok = a.base_aligned && ((n0 + 256) <= a.Cout) &&
                                (a.out_mode <= 1 ? ((a.y_cstride % 16) == 0 && ((a.y_coff + n0) % 16) == 0)
                                                 : ((a.y_cstride % 8) == 0 && ((a.y_coff + n0) % 8) == 0));
            tc::mbar_wait(&tmem_full_bar[as], aphase);
            tc::tc_fence_after();
            const uint32_t acc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * 256 + hsel * 128);
            for (int c0 = 0; c0 < 128; c0 += 32) {
                uint32_t v[32];
                tc::tmem_ld_32x32(acc + (uint32_t)c0, v);
                tc::tmem_ld_wait();
                const int cc = hsel * 128 + c0, ch0 = n0 + cc;
                if (!pix_ok || ch0 >= a.Cout) continue;
                conv_store_chunk<kAct, kClamp>(a, v, s_scale, s_bias, cc, ch0, pix * a.y_cstride + a.y_coff + ch0, nz, vec_ok, b, Y, X);
            }
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive_cluster(as == 0 ? lead_empty0 : lead_empty1);
            if (++as == 2) { as = 0; aphase ^= 1; }
            parity ^= 1;
        }
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::cluster_sync_all();                               // the peer may still be reading this CTA's smem / signalling its barriers
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc_pair(tmem_base, 512);
    }
}

// Second half of a split-K convolution: sums the k-range partials in a fixed order (deterministic) and applies the same
// epilogue as the fused path. One thread per (pixel, 4 channels).
__global__ void __launch_bounds__(256) conv_splitk_finish_kernel(const ConvKernelArgs a, int B, int act) {
    const int cq = a.Cout_pad >> 2;
    {
        ConvPhase P = a.ph[0];                        // blockIdx.y = phase
#pragma unroll
        for (int q = 1; q < 4; ++q)
            if ((int)blockIdx.y == q) P = a.ph[q];
        const size_t total = (size_t)B * P.gH * P.gW * cq;
        const size_t split_stride = (size_t)B * P.gH * P.gW * a.Cout_pad;
        for (size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
            const int c4 = (int)(idx % cq) * 4;
            size_t t = idx / cq;
            const int gx = (int)(t % P.gW); t /= P.gW;
            const int gy = (int)(t % P.gH);
            const int b = (int)(t / P.gH);
            if (c4 >= a.Cout) continue;
            const float* pp = a.partial + P.p0 + (((size_t)b * P.gH + gy) * P.gW + gx) * a.Cout_pad + c4;
            float4 acc = *reinterpret_cast<const float4*>(pp);
            for (int s = 1; s < a.splits; ++s) {
                const float4 q = *reinterpret_cast<const float4*>(pp + s * split_stride);
                acc.x += q.x; acc.y += q.y; acc.z += q.z; acc.w += q.w;
            }
            const int Y = gy * a.sy + P.oy, X = gx * a.sx + P.ox;
            const size_t pix = ((size_t)b * a.oH + Y) * a.oW + X;
            const float nz = a.noise ? __ldg(a.noise + (size_t)b * a.noise_bstride + (size_t)Y * a.oW + X) * a.pre_gain : 0.f;
            const float accv[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
            for (int k = 0; k < 4; ++k) {
                const int ch = c4 + k;
                if (ch >= a.Cout) break;
                float sc = a.acc_scale * a.pre_gain;
                if (a.dscale) sc *= __ldg(a.dscale + (size_t)b * a.Cout + ch);
                const float bi = a.bias ? __ldg(a.bias + ch) * a.pre_gain : 0.f;
                float x = fmaf(accv[k], sc, bi) + nz;
                if (act == 1) x = fmaxf(x, x * a.alpha);
                if (act == 2) x = x > 0.f ? x : x * a.alpha;
                x *= a.post_gain;
                if (a.clamp >= 0.f) x = fminf(fmaxf(x, -a.clamp), a.clamp);
                const size_t off = pix * a.y_cstride + a.y_coff + ch;
                if (a.out_mode <= 1) {
                    const __half h = __float2half_rn(x);
                    reinterpret_cast<__half*>(a.y)[off] = h;
                    if (a.out_mode == 1) reinterpret_cast<__half*>(a.y_lo)[off] = __float2half_rn(x - __half2float(h));
                } else {
                    float* yf = reinterpret_cast<float*>(a.y) + off;
                    *yf = (a.out_mode == 3 ? *yf : 0.f) + x;
                }
            }
        }
    }
}

// ---------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------
static int make_tmap_f16_sw128(CUtensorMap* tm, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                               const uint32_t* box, const uint32_t* elem_strides = nullptr) {
    return make_tmap(tm, base, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, CU_TENSOR_MAP_SWIZZLE_128B, rank, dims, strides_bytes, box, elem_strides);
}

}  // namespace p3d

using namespace p3d;

// phases[0..n_phases): launches that differ only in their tap list, computed grid (gH, gW) and output offset (oy, ox)
static int conv_launch(const p3d_conv_args_t* phases, int n_phases, p3d_stream_t stream) {
    if (!phases || n_phases < 1 || n_phases > 4) return P3D_BAD_ARG;
    const p3d_conv_args_t* p = phases;
    if (!p->x || !p->w || !p->y) return P3D_BAD_ARG;
    if (p->C % kBK != 0 || p->C <= 0) return P3D_UNSUPPORTED;
    if (p->x_planes < 1 || p->x_planes > 2 || p->w_planes < 1 || p->w_planes > 2) return P3D_BAD_ARG;
    if (p->split && (p->x_planes != 2 || p->w_planes != 2)) return P3D_BAD_ARG;
    if (p->out_mode < 0 || p->out_mode > 3 || (p->out_mode == 1 && !p->y_lo)) return P3D_BAD_ARG;
    if (p->Cout_padded % 16 != 0 || p->Cout_padded < p->Cout) return P3D_BAD_ARG;
    if (p->B <= 0) return P3D_BAD_ARG;
    const int passes = p->split ? 3 : 1;
    int taps_total = 0, taps_max = 0, gH_max = 0, gW_max = 0;
    for (int q = 0; q < n_phases; ++q) {
        const p3d_conv_args_t* r = phases + q;
        if (r->n_taps < 1 || r->n_taps > 9 || r->gH <= 0 || r->gW <= 0) return q == 0 ? P3D_UNSUPPORTED : P3D_BAD_ARG;
        if (q > 0 && (r->x != p->x || r->w != p->w || r->y != p->y || r->y_lo != p->y_lo || r->x_planes != p->x_planes ||
                      r->w_planes != p->w_planes || r->B != p->B || r->Bw != p->Bw || r->H != p->H || r->W != p->W || r->C != p->C ||
                      r->Cout != p->Cout || r->Cout_padded != p->Cout_padded || r->n_kblocks != p->n_kblocks || r->split != p->split ||
                      r->oH != p->oH || r->oW != p->oW || r->sy != p->sy || r->sx != p->sx || r->y_cstride != p->y_cstride ||
                      r->y_coff != p->y_coff || r->out_mode != p->out_mode || r->bias != p->bias || r->noise != p->noise ||
                      r->dscale != p->dscale || r->act != p->act || r->alpha != p->alpha || r->gain != p->gain || r->clamp != p->clamp ||
                      r->acc_scale != p->acc_scale || r->up_prev || p->up_prev || r->residual || p->residual || r->stride != p->stride ||
                      r->noise_batch_stride != p->noise_batch_stride || r->rgb_w || p->rgb_w))
            return P3D_BAD_ARG;
        taps_total += r->n_taps;
        if (r->n_taps > taps_max) taps_max = r->n_taps;
        if (r->gH > gH_max) gH_max = r->gH;
        if (r->gW > gW_max) gW_max = r->gW;
    }
    if (taps_total * passes > kMaxGroups) return P3D_UNSUPPORTED;

    const int BN = p->Cout_padded > 128 ? 128 : p->Cout_padded;
    // spatial tile BW x BH = 128 pixels: the power-of-two split with the least padded area (ties -> wider rows), summed over
    // the phases (they share the TMA box); `rows` = sub-tiles stacked in y per CTA tile (2 for the persistent kernels)
    const int stride = p->stride > 1 ? p->stride : 1;
    if (stride > 2) return P3D_UNSUPPORTED;
    auto pick_bw = [&](int rows, long* area_out) {
        int bw_best = 1;
        long best = -1;
        for (int bw = 1; bw <= 64; bw *= 2) {
            int bh = kBM / bw * rows;
            if (bw * stride > 256 || bh * stride > 256) continue;      // TMA box extent (in input pixels) <= 256
            long area = 0;
            for (int q = 0; q < n_phases; ++q) area += (long)ceil_div(phases[q].gW, bw) * bw * ceil_div(phases[q].gH, bh) * bh;
            if (best < 0 || area <= best) { best = area; bw_best = bw; }
        }
        if (area_out) *area_out = best;
        return bw_best;
    };
    // persistent 256-pixel tiles when there is at least one tile per SM (launch_flags bit 0 disables, for A/B runs)
    bool persist = false, pair = false;
    int BW = pick_bw(1, nullptr);
    {
        const int env = (p->launch_flags & 1) ? 0 : 1;
        long area2 = 0;
        const int bw2 = pick_bw(2, &area2);
        const long tiles2 = area2 / 256 * ceil_div(p->Cout_padded, BN) * p->B;
        if (env && tiles2 >= sm_count()) { persist = true; BW = bw2; }
        // CTA pairs (cta_group::2) for >= 256 output channels: one 256-pixel x 256-channel tile per pair
        // (launch_flags bit 1 keeps the single-CTA persistent kernel, for A/B runs)
        const int env_pair = (p->launch_flags & 2) ? 0 : 1;
        const long tiles_pair = area2 / 256 * (p->Cout_padded / 256) * p->B;
        // (launches with a handful of k-steps per tile -- the 1- and 2-tap phases of a narrow transposed convolution -- are
        //  prologue/epilogue-bound and measured slightly slower on pairs; a merged launch is judged by its heaviest phase)
        const int k_steps = passes * taps_max * (p->C / kBK);
        if (persist && env_pair && p->Cout_padded % 256 == 0 && tiles_pair * 2 >= sm_count() && k_steps >= 8) pair = true;
    }
    const int BH = kBM / BW;
    const int K = p->n_kblocks * p->C;
    if (p->n_kblocks < 1) return P3D_BAD_ARG;

    CUtensorMap tmA, tmB;
    {
        uint64_t dims[5] = {(uint64_t)p->C, (uint64_t)p->W, (uint64_t)p->H, (uint64_t)p->B, (uint64_t)p->x_planes};
        uint64_t str[4] = {(uint64_t)p->C * 2, (uint64_t)p->W * p->C * 2, (uint64_t)p->H * p->W * p->C * 2,
                           (uint64_t)p->B * p->H * p->W * p->C * 2};
        // a strided convolution samples every `stride`-th input pixel: the TMA walks the box with that element stride
        // (box extents are then given in input pixels: N loaded pixels need an extent of N * stride)
        uint32_t box[5] = {(uint32_t)kBK, (uint32_t)(BW * stride), (uint32_t)(((persist && !pair) ? 2 * BH : BH) * stride), 1, 1};
        uint32_t es[5] = {1, (uint32_t)stride, (uint32_t)stride, 1, 1};
        int rc = make_tmap_f16_sw128(&tmA, p->x, 5, dims, str, box, es);
        if (rc != P3D_OK) return rc;
    }
    {
        uint64_t dims[4] = {(uint64_t)K, (uint64_t)p->Cout_padded, (uint64_t)p->Bw, (uint64_t)p->w_planes};
        uint64_t str[3] = {(uint64_t)K * 2, (uint64_t)p->Cout_padded * K * 2, (uint64_t)p->Bw * p->Cout_padded * K * 2};
        uint32_t box[4] = {(uint32_t)kBK, (uint32_t)(pair ? 128 : BN), 1, 1};     // a pair CTA stages half of a 256-channel tile
        int rc = make_tmap_f16_sw128(&tmB, p->w, 4, dims, str, box);
        if (rc != P3D_OK) return rc;
    }

    ConvKernelArgs a;
    memset(&a, 0, sizeof(a));
    static const int pa[3] = {0, 0, 1}, pb[3] = {0, 1, 0};     // hi*hi, hi*lo, lo*hi
    const int tiles_n = pair ? p->Cout_padded / 256 : ceil_div(p->Cout_padded, BN);
    int g = 0, tiles_m_total = 0, max_total_k = 0, min_total_k = 1 << 30;
    a.n_phases = n_phases;
    a.kc_steps = p->C / kBK;
    for (int q = 0; q < n_phases; ++q) {
        const p3d_conv_args_t* r = phases + q;
        ConvPhase& P = a.ph[q];
        P.g0 = g;
        for (int pass = 0; pass < passes; ++pass)
            for (int t = 0; t < r->n_taps; ++t) {
                a.dy[g] = r->tap_dy[t]; a.dx[g] = r->tap_dx[t]; a.tap[g] = r->tap_k[t];
                a.a_plane[g] = (int8_t)pa[pass]; a.b_plane[g] = (int8_t)pb[pass];
                ++g;
            }
        P.ng = g - P.g0;
        P.gH = r->gH; P.gW = r->gW; P.oy = r->oy; P.ox = r->ox;
        P.tiles_x = ceil_div(r->gW, BW); P.tiles_y = ceil_div(r->gH, persist ? 2 * BH : BH);
        // tile order: spatial tiles for the grid kernel (blockIdx.x), whole (spatial, channel, sample) tiles for the persistent ones
        P.t0 = persist ? tiles_m_total * tiles_n * p->B : tiles_m_total;
        tiles_m_total += P.tiles_x * P.tiles_y;
        const int tk = P.ng * a.kc_steps;
        if (tk > max_total_k) max_total_k = tk;
        if (tk < min_total_k) min_total_k = tk;
    }
    a.Cin = p->C;
    a.BW = BW; a.BH = BH;
    a.BN = BN; a.w_per_sample = p->Bw > 1 ? 1 : 0;
    a.idesc = tc::umma_idesc_f16(kBM, BN, 0);
    a.tmem_cols = BN <= 32 ? 32u : BN <= 64 ? 64u : 128u;
    a.oH = p->oH; a.oW = p->oW; a.sy = p->sy; a.sx = p->sx;
    a.Cout = p->Cout; a.y_cstride = p->y_cstride; a.y_coff = p->y_coff;
    a.y = p->y; a.y_lo = p->y_lo; a.out_mode = p->out_mode;
    a.bias = p->bias; a.noise = p->noise; a.dscale = p->dscale;
    a.noise_bstride = p->noise_batch_stride;
    a.alpha = p->alpha; a.clamp = p->clamp; a.acc_scale = p->acc_scale;
    a.base_aligned = ((((uintptr_t)p->y) | ((uintptr_t)p->y_lo)) & 31) == 0;
    a.up_prev = p->up_prev; a.up_f = p->up_filter; a.round16 = p->round16; a.out_nchw = p->out_nchw;
    a.stride = stride; a.residual = p->residual;
    if (p->rgb_w) {
        // fused ToRGB of the next layer: one channel tile holding every output channel, fp16 output, 1:1 output map, persistent
        // single-CTA kernel (its epilogue thread sees all channels of its pixel)
        if (n_phases != 1 || !persist || pair || p->up_prev || p->residual || p->out_mode != 0 || p->Cout != p->Cout_padded ||
            p->Cout > 128 || p->Cout % 32 != 0 || p->sy != 1 || p->sx != 1 || p->oy != 0 || p->ox != 0 || p->gH != p->oH ||
            p->gW != p->oW || (p->oH & 1) || (p->oW & 1) || stride != 1 || p->y_coff != 0 || p->y_cstride != p->Cout)
            return P3D_UNSUPPORTED;
        if (!p->rgb_prev || !p->rgb_filter || !p->rgb_out || p->rgb_cout < 1 || p->rgb_cout > 8 || p->rgb_w_rows < p->rgb_cout ||
            !a.base_aligned)
            return P3D_BAD_ARG;
        a.rgb_w = reinterpret_cast<const __half*>(p->rgb_w); a.rgb_bias = p->rgb_bias; a.rgb_prev = p->rgb_prev; a.rgb_f = p->rgb_filter;
        a.rgb_out = p->rgb_out; a.rgb_cout = p->rgb_cout; a.rgb_w_rows = p->rgb_w_rows; a.rgb_skip_x = p->rgb_skip_x;
        a.rgb_clamp = p->rgb_clamp; a.rgb_acc_scale = p->rgb_acc_scale;
    }
    if (p->residual && (p->up_prev || p->out_mode > 2 || p->sy != 1 || p->sx != 1 || p->oy != 0 || p->ox != 0 ||
                        (((uintptr_t)p->residual) & 31) != 0))
        return P3D_BAD_ARG;
    if (p->up_prev) {
        // fused ToRGB tail: full-resolution 1:1 output map, fp32 output, even size, prev / y 16-byte aligned
        if (!p->up_filter || p->out_mode != 2 || p->sy != 1 || p->sx != 1 || p->oy != 0 || p->ox != 0 || (p->oH & 1) || (p->oW & 1) ||
            p->gH != p->oH || p->gW != p->oW || p->y_coff != 0 || (!p->out_nchw && p->y_cstride != p->Cout) ||
            ((((uintptr_t)p->up_prev) | ((uintptr_t)p->y)) & 15) != 0)
            return P3D_BAD_ARG;
    } else if (p->out_nchw || p->round16) {
        return P3D_BAD_ARG;
    }
    // act(x) * gain == act(x * gain) for gain > 0 (linear and leaky-relu are positively homogeneous): fold the gain into the
    // per-channel scale / bias / noise so the per-element epilogue is fma + add + max (+ clamp)
    const bool fold = p->gain > 0.f;
    a.pre_gain = fold ? p->gain : 1.f;
    a.post_gain = fold ? 1.f : p->gain;
    if (p->act != 1 && p->act != 3) return P3D_UNSUPPORTED;
    const int act = p->act == 1 ? 0 : (p->alpha >= 0.f && p->alpha <= 1.f ? 1 : 2);
    const bool clamp = p->clamp >= 0.f;

    // 3 stages (96 KB at BN = 128): two CTAs per SM, so one tile's epilogue / TMA latency hides behind the other's MMAs.
    // Grids that leave at most one CTA per SM anyway (the 4^2..32^2 backbone layers: 16-128 CTAs with 200+ k-steps each)
    // are bound by TMA latency x bytes in flight instead; they get a 6-stage ring (192 KB).
    dim3 grid(tiles_m_total, ceil_div(p->Cout_padded, BN), p->B);
    const long base_ctas = (long)grid.x * grid.y * grid.z;
    if (pair) {
        a.splits = 1; a.partial = nullptr; a.Cout_pad = p->Cout_padded;
        a.BN = 256;
        a.idesc = tc::umma_idesc_f16(256, 256, 0);
        const int n_tiles = tiles_m_total * tiles_n * p->B;
        const size_t smem_q = kQStages * (size_t)(kBM * 128 + 128 * 128) + 256 + 2 * 512 * sizeof(float) + 1024;
        int pairs = sm_count() / 2;
        if (pairs > n_tiles) pairs = n_tiles;
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(2 * pairs, 1, 1);
        cfg.blockDim = dim3(320, 1, 1);
        cfg.dynamicSmemBytes = smem_q;
        cfg.stream = (cudaStream_t)stream;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
#define P3D_LAUNCH_PAIR(ACT, CL)                                                                                              \
    do {                                                                                                                      \
        P3D_CUDA_TRY(cudaFuncSetAttribute(conv_gemm_pair_kernel<ACT, CL>, cudaFuncAttributeMaxDynamicSharedMemorySize,        \
                                          (int)smem_q));                                                                      \
        P3D_CUDA_TRY(cudaLaunchKernelEx(&cfg, conv_gemm_pair_kernel<ACT, CL>, tmA, tmB, a, n_tiles, tiles_n));                \
    } while (0)
        if (act == 0) { if (clamp) P3D_LAUNCH_PAIR(0, true); else P3D_LAUNCH_PAIR(0, false); }
        else if (act == 1) { if (clamp) P3D_LAUNCH_PAIR(1, true); else P3D_LAUNCH_PAIR(1, false); }
        else { if (clamp) P3D_LAUNCH_PAIR(2, true); else P3D_LAUNCH_PAIR(2, false); }
#undef P3D_LAUNCH_PAIR
        P3D_LAUNCH_CHECK();
        return P3D_OK;
    }
    if (persist) {
        a.splits = 1; a.partial = nullptr; a.Cout_pad = p->Cout_padded;
        const int n_tiles = (int)base_ctas;
        const size_t stage_bytes_p = 2 * (size_t)kBM * 128 + (size_t)BN * 128;
        const size_t smem_p = kPStages * stage_bytes_p + 128 + 2 * 256 * sizeof(float) + 2 * 1024 * sizeof(float) + 1024;
        const int ctas = n_tiles < sm_count() ? n_tiles : sm_count();
#define P3D_LAUNCH_PERSIST(ACT, CL)                                                                                           \
    do {                                                                                                                      \
        P3D_CUDA_TRY(cudaFuncSetAttribute(conv_gemm_persist_kernel<ACT, CL>, cudaFuncAttributeMaxDynamicSharedMemorySize,     \
                                          (int)smem_p));                                                                      \
        conv_gemm_persist_kernel<ACT, CL><<<ctas, 320, smem_p, (cudaStream_t)stream>>>(tmA, tmB, a, n_tiles, tiles_n);        \
    } while (0)
        if (act == 0) { if (clamp) P3D_LAUNCH_PERSIST(0, true); else P3D_LAUNCH_PERSIST(0, false); }
        else if (act == 1) { if (clamp) P3D_LAUNCH_PERSIST(1, true); else P3D_LAUNCH_PERSIST(1, false); }
        else { if (clamp) P3D_LAUNCH_PERSIST(2, true); else P3D_LAUNCH_PERSIST(2, false); }
#undef P3D_LAUNCH_PERSIST
        P3D_LAUNCH_CHECK();
        return P3D_OK;
    }
    // split-K for grids far smaller than the machine (4^2..16^2 layers: 16-32 CTAs each streaming 100-200 k-steps at
    // the per-SM L2 ingest rate): every k-range becomes its own CTA writing raw fp32 partials into the caller's scratch
    // buffer; conv_splitk_finish_kernel adds them in a fixed order and applies the epilogue. Two CTAs fit an SM, so the
    // split count aims at two waves' worth of CTAs; every phase of a merged launch is split the same number of ways.
    a.splits = 1; a.partial = nullptr; a.Cout_pad = p->Cout_padded;
    if (p->splitk_scratch && !p->up_prev && !p->residual && base_ctas * 2 <= sm_count() && min_total_k >= 8) {
        int splits = (int)((n_phases > 1 ? 2 * sm_count() : sm_count()) / base_ctas);
        if (splits > min_total_k / 4) splits = min_total_k / 4;
        if (splits > 16) splits = 16;
        size_t per_split = 0;
        for (int q = 0; q < n_phases; ++q) per_split += (size_t)p->B * phases[q].gH * phases[q].gW * p->Cout_padded * sizeof(float);
        while (splits > 1 && per_split * splits > (size_t)p->splitk_scratch_bytes) --splits;
        if (splits > 1 && (((uintptr_t)p->splitk_scratch) & 31) == 0) {
            a.splits = splits;
            a.partial = reinterpret_cast<float*>(p->splitk_scratch);
            grid.z = p->B * splits;
            long long off = 0;
            for (int q = 0; q < n_phases; ++q) {
                a.ph[q].p0 = off;
                off += (long long)splits * p->B * phases[q].gH * phases[q].gW * p->Cout_padded;
            }
        }
    }
    const bool deep = (long)grid.x * grid.y * grid.z <= sm_count() && max_total_k / a.splits > 6;
    const size_t stage_bytes = (size_t)kBM * 128 + (size_t)BN * 128;
    const size_t smem = (deep ? 6 : 3) * stage_bytes + 64 + 2 * 128 * sizeof(float) + 1024 + (deep ? 64 : 0);
#define P3D_LAUNCH_CONV_S(ST, ACT, CL)                                                                                        \
    do {                                                                                                                      \
        P3D_CUDA_TRY(cudaFuncSetAttribute(conv_gemm_kernel<ST, ACT, CL>, cudaFuncAttributeMaxDynamicSharedMemorySize,         \
                                          (int)smem));                                                                        \
        conv_gemm_kernel<ST, ACT, CL><<<grid, 192, smem, (cudaStream_t)stream>>>(tmA, tmB, a);                                \
    } while (0)
#define P3D_LAUNCH_CONV(ACT, CL)                                                                                              \
    do { if (deep) P3D_LAUNCH_CONV_S(6, ACT, CL); else P3D_LAUNCH_CONV_S(3, ACT, CL); } while (0)
    if (act == 0) { if (clamp) P3D_LAUNCH_CONV(0, true); else P3D_LAUNCH_CONV(0, false); }
    else if (act == 1) { if (clamp) P3D_LAUNCH_CONV(1, true); else P3D_LAUNCH_CONV(1, false); }
    else { if (clamp) P3D_LAUNCH_CONV(2, true); else P3D_LAUNCH_CONV(2, false); }
#undef P3D_LAUNCH_CONV_S
#undef P3D_LAUNCH_CONV
    P3D_LAUNCH_CHECK();
    if (a.splits > 1) {
        size_t items = 0;
        for (int q = 0; q < n_phases; ++q) {
            const size_t it = (size_t)p->B * phases[q].gH * phases[q].gW * (p->Cout_padded / 4);
            if (it > items) items = it;
        }
        size_t blocks = (items + 255) / 256;
        const size_t cap = (size_t)sm_count() * 16;
        if (blocks > cap) blocks = cap;
        conv_splitk_finish_kernel<<<dim3((unsigned)blocks, (unsigned)n_phases), 256, 0, (cudaStream_t)stream>>>(a, p->B, act);
        P3D_LAUNCH_CHECK();
    }
    return P3D_OK;
}

extern "C" int p3d_conv_gemm(const p3d_conv_args_t* p, p3d_stream_t stream) { return conv_launch(p, 1, stream); }

extern "C" int p3d_conv_gemm_phases(const p3d_conv_args_t* phases, int n_phases, p3d_stream_t stream) {
    return conv_launch(phases, n_phases, stream);
}
