// Triangle rasterizer with a depth buffer and a diffuse shader: the turntable preview of the reference's
// applications/extract_mesh.py:226-262 (pyrender there) on the device. The contract (projection, coverage, depth keys,
// shading) is the comment above p3d_mesh_raster in include/p3d.h; oracle/p3d_oracle/mesh_render.py restates it in numpy
// and the tests compare bit for bit, so every fp32 operation here is an explicitly rounded intrinsic (no contraction).
//
// Two launches:
//   mesh_raster_kernel  one thread per face and kRasterViews views (the face's vertices are loaded once for them); per
//                       view the thread projects the triangle and, when its clipped bounding box has at most
//                       kSmallBoxPixels pixels, tests them itself. Larger triangles go to the warp: the lanes holding one
//                       are taken one at a time and all 32 lanes sweep its box. Fragments resolve with a 64-bit atomicMin
//                       on (depth bits << 32 | face id), so the result does not depend on the path or the launch order.
//   mesh_shade_kernel   one thread per pixel: reads the key, recomputes the face's projection and barycentrics with the
//                       same code, and writes the shaded uint8 RGB (white where no face was drawn).
#include "p3d_common.cuh"

namespace p3d {

constexpr int kRasterThreads = 256;
constexpr int kRasterViews = 8;
constexpr int kSmallBoxPixels = 16;
constexpr int kShadeThreads = 256;
constexpr float kGuardPx = 2097152.f;                    // 2^21
constexpr float kGrey = 0.8f;
constexpr float kCosCone = 0.70710678118654752f;         // cos(pi/4)
constexpr float kPi = 3.14159265358979323846f;
constexpr uint64_t kEmpty = ~0ull;

struct MeshGeom {
    const float* v;
    const int64_t* f;
    int64_t V, F;
    int H, W;
    float kx, ky, hx, hy;      // W / (2 xmag), H / (2 ymag), W / 2, H / 2
};

// the face's world-space corners; false when an index is outside [0, V) or a coordinate is not finite
__device__ __forceinline__ bool load_face(const MeshGeom& g, int64_t face, float (&w)[3][3]) {
    bool ok = true;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int64_t idx = __ldg(g.f + 3 * face + k);
        if (idx < 0 || idx >= g.V) return false;
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            w[k][c] = __ldg(g.v + 3 * idx + c);
            ok = ok && isfinite(w[k][c]);
        }
    }
    return ok;
}

// a triangle on the screen: fixed-point corners, depths, edge vectors after the winding flip, area > 0, clipped box
struct Tri {
    int64_t X[3], Y[3];
    float d[3];
    int64_t dx[3], dy[3], A;
    int i0, i1, j0, j1;
};

enum { kTriNone = 0, kTriDraw = 1, kTriGuard = 2 };

__device__ __forceinline__ float cam_row(const float* m, const float (&p)[3]) {
    return __fadd_rn(__fadd_rn(__fadd_rn(__fmul_rn(m[0], p[0]), __fmul_rn(m[1], p[1])), __fmul_rn(m[2], p[2])), m[3]);
}

// corners in fixed point -> edges, area, box; kTriNone for a zero area or an empty box
__device__ __forceinline__ int tri_finish(const MeshGeom& g, Tri& t) {
    const int64_t A = (t.X[1] - t.X[0]) * (t.Y[2] - t.Y[0]) - (t.Y[1] - t.Y[0]) * (t.X[2] - t.X[0]);
    if (A == 0) return kTriNone;
    const int64_t s = A < 0 ? -1 : 1;
    t.A = s * A;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int a = (k + 1) % 3, b = (k + 2) % 3;
        t.dx[k] = s * (t.X[b] - t.X[a]);
        t.dy[k] = s * (t.Y[b] - t.Y[a]);
    }
    const int64_t xmin = min(t.X[0], min(t.X[1], t.X[2])), xmax = max(t.X[0], max(t.X[1], t.X[2]));
    const int64_t ymin = min(t.Y[0], min(t.Y[1], t.Y[2])), ymax = max(t.Y[0], max(t.Y[1], t.Y[2]));
    // centres 256 j + 128 inside [xmin, xmax]; arithmetic shifts are floor divisions
    t.j0 = (int)max((int64_t)0, (xmin + 127) >> 8);
    t.j1 = (int)min((int64_t)g.W - 1, (xmax - 128) >> 8);
    t.i0 = (int)max((int64_t)0, (ymin + 127) >> 8);
    t.i1 = (int)min((int64_t)g.H - 1, (ymax - 128) >> 8);
    return (t.j0 <= t.j1 && t.i0 <= t.i1) ? kTriDraw : kTriNone;
}

__device__ __forceinline__ int tri_setup(const MeshGeom& g, const p3d_mesh_view_t& vw, const float (&w)[3][3], Tri& t) {
    bool guard = false;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const float cx = cam_row(vw.world2cam, w[k]), cy = cam_row(vw.world2cam + 4, w[k]), cz = cam_row(vw.world2cam + 8, w[k]);
        const float sx = __fadd_rn(__fmul_rn(cx, g.kx), g.hx);
        const float sy = __fsub_rn(g.hy, __fmul_rn(cy, g.ky));
        guard = guard || !(fabsf(sx) <= kGuardPx) || !(fabsf(sy) <= kGuardPx);
        t.X[k] = __float2ll_rn(__fmul_rn(sx, 256.f));
        t.Y[k] = __float2ll_rn(__fmul_rn(sy, 256.f));
        t.d[k] = -cz;
    }
    if (guard) return kTriGuard;
    return tri_finish(g, t);
}

// barycentrics at pixel (i, j); false when the pixel centre is not covered
__device__ __forceinline__ bool tri_cover(const Tri& t, int i, int j, float (&b)[3]) {
    const int64_t px = 256 * (int64_t)j + 128, py = 256 * (int64_t)i + 128;
    int64_t E[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int a = (k + 1) % 3;
        E[k] = t.dx[k] * (py - t.Y[a]) - t.dy[k] * (px - t.X[a]);
        const bool top_left = t.dy[k] < 0 || (t.dy[k] == 0 && t.dx[k] > 0);
        if (!(E[k] > 0 || (E[k] == 0 && top_left))) return false;
    }
    const float A = __ll2float_rn(t.A);
#pragma unroll
    for (int k = 0; k < 3; ++k) b[k] = __fdiv_rn(__ll2float_rn(E[k]), A);
    return true;
}

__device__ __forceinline__ float bary_sum(const float (&b)[3], float a0, float a1, float a2) {
    return __fadd_rn(__fadd_rn(__fmul_rn(b[0], a0), __fmul_rn(b[1], a1)), __fmul_rn(b[2], a2));
}

__device__ __forceinline__ float dot3(const float (&a)[3], const float (&b)[3]) {
    return bary_sum(a, b[0], b[1], b[2]);
}

__device__ __forceinline__ void fragment(const Tri& t, int i, int j, uint32_t face, float znear, float zfar,
                                         unsigned long long* keys_view, int W) {
    float b[3];
    if (!tri_cover(t, i, j, b)) return;
    const float d = bary_sum(b, t.d[0], t.d[1], t.d[2]);
    if (!(d >= znear && d <= zfar)) return;
    const unsigned long long key = (unsigned long long)__float_as_uint(d) << 32 | face;
    unsigned long long* dst = keys_view + (int64_t)i * W + j;
    if (*(volatile unsigned long long*)dst > key) atomicMin(dst, key);    // a stale read only costs an atomic
}

__global__ void __launch_bounds__(kRasterThreads) mesh_raster_kernel(const MeshGeom g, const p3d_mesh_view_t* __restrict__ views,
                                                                     int N, float znear, float zfar,
                                                                     unsigned long long* __restrict__ keys,
                                                                     unsigned long long* __restrict__ guard_drops) {
    __shared__ p3d_mesh_view_t s_views[kRasterViews];
    const int n0 = blockIdx.y * kRasterViews, nv = min(kRasterViews, N - n0);
    for (int x = threadIdx.x; x < nv * (int)(sizeof(p3d_mesh_view_t) / 4); x += kRasterThreads)
        reinterpret_cast<float*>(s_views)[x] = __ldg(reinterpret_cast<const float*>(views + n0) + x);
    __syncthreads();
    const int lane = threadIdx.x & 31;
    const int64_t face = (int64_t)blockIdx.x * kRasterThreads + threadIdx.x;
    float w[3][3];
    const bool valid = face < g.F && load_face(g, face, w);
    unsigned long long guards = 0;
    for (int v = 0; v < nv; ++v) {
        unsigned long long* kv = keys + (int64_t)(n0 + v) * g.H * g.W;
        Tri t;
        int st = kTriNone;
        if (valid) st = tri_setup(g, s_views[v], w, t);
        guards += st == kTriGuard;
        int bw = 0, pixels = 0;
        if (st == kTriDraw) {
            bw = t.j1 - t.j0 + 1;
            pixels = bw * (t.i1 - t.i0 + 1);
        }
        if (st == kTriDraw && pixels <= kSmallBoxPixels) {
            for (int i = t.i0; i <= t.i1; ++i)
                for (int j = t.j0; j <= t.j1; ++j) fragment(t, i, j, (uint32_t)face, znear, zfar, kv, g.W);
        }
        unsigned big = __ballot_sync(0xffffffffu, st == kTriDraw && pixels > kSmallBoxPixels);
        while (big) {
            const int src = __ffs(big) - 1;
            big &= big - 1;
            Tri u;
#pragma unroll
            for (int k = 0; k < 3; ++k) {
                u.X[k] = __shfl_sync(0xffffffffu, t.X[k], src);
                u.Y[k] = __shfl_sync(0xffffffffu, t.Y[k], src);
                u.d[k] = __shfl_sync(0xffffffffu, t.d[k], src);
            }
            const uint32_t uf = (uint32_t)__shfl_sync(0xffffffffu, (long long)face, src);
            tri_finish(g, u);
            const int ubw = u.j1 - u.j0 + 1, upix = ubw * (u.i1 - u.i0 + 1);
            for (int p = lane; p < upix; p += 32) fragment(u, u.i0 + p / ubw, u.j0 + p % ubw, uf, znear, zfar, kv, g.W);
        }
    }
    if (guards) atomicAdd(guard_drops, guards);
}

__global__ void __launch_bounds__(kShadeThreads) mesh_shade_kernel(const MeshGeom g, const p3d_mesh_view_t* __restrict__ views,
                                                                   const unsigned long long* __restrict__ keys,
                                                                   const unsigned char* __restrict__ colors, float intensity,
                                                                   int64_t pixels, unsigned char* __restrict__ out) {
    const int64_t idx = (int64_t)blockIdx.x * kShadeThreads + threadIdx.x;
    if (idx >= pixels) return;
    const unsigned long long key = __ldg(keys + idx);
    unsigned char* o = out + 3 * idx;
    if (key == kEmpty) {
        o[0] = o[1] = o[2] = 255;
        return;
    }
    const int64_t hw = (int64_t)g.H * g.W;
    const int n = (int)(idx / hw);
    const int i = (int)((idx - n * hw) / g.W), j = (int)(idx - n * hw - (int64_t)i * g.W);
    const int64_t face = (int64_t)(key & 0xffffffffu);
    const p3d_mesh_view_t vw = views[n];
    float w[3][3], b[3];
    Tri t;
    load_face(g, face, w);                         // the face was drawn: its corners and its coverage of (i, j) hold
    tri_setup(g, vw, w, t);
    tri_cover(t, i, j, b);

    float colour[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        if (colors) {
            float ck[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) ck[k] = __fdiv_rn((float)__ldg(colors + 3 * __ldg(g.f + 3 * face + k) + c), 255.f);
            colour[c] = bary_sum(b, ck[0], ck[1], ck[2]);
        } else {
            colour[c] = kGrey;
        }
    }
    float e1[3], e2[3], nrm[3], q[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        e1[c] = __fsub_rn(w[1][c], w[0][c]);
        e2[c] = __fsub_rn(w[2][c], w[0][c]);
        q[c] = __fsub_rn(vw.eye[c], bary_sum(b, w[0][c], w[1][c], w[2][c]));
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const int a = (c + 1) % 3, z = (c + 2) % 3;
        nrm[c] = __fsub_rn(__fmul_rn(e1[a], e2[z]), __fmul_rn(e1[z], e2[a]));
    }
    const float nlen = __fsqrt_rn(dot3(nrm, nrm));
    const float r2 = dot3(q, q);
    const float r = __fsqrt_rn(r2);
    float nl[3], ll[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        nl[c] = __fdiv_rn(nrm[c], nlen);
        ll[c] = __fdiv_rn(q[c], r);
    }
    const float ndl = dot3(nl, ll);
    const float cone = dot3(ll, vw.spot_axis);
    float shade = __fdiv_rn(__fmul_rn(intensity, ndl > 0.f ? ndl : 0.f), __fmul_rn(kPi, r2));
    if (cone > -kCosCone) shade = 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float x = __fadd_rn(__fmul_rn(__fmul_rn(255.f, colour[c]), shade), 0.5f);
        o[c] = (unsigned char)(x < 255.f ? floorf(x) : 255.f);
    }
}

static bool mesh_geom(const float* vertices, int64_t V, const int64_t* faces, int64_t F, const p3d_mesh_view_t* views, int N,
                      int H, int W, float xmag, float ymag, MeshGeom& g) {
    if (V < 0 || F < 0 || F >= ((int64_t)1 << 32) || N < 1 || H < 1 || W < 1 || H > 32768 || W > 32768 || !views) return false;
    if (!(xmag > 0.f) || !(ymag > 0.f) || (F > 0 && (!vertices || !faces))) return false;
    if ((int64_t)N * H * W > ((int64_t)1 << 40)) return false;
    // host fp32 arithmetic is IEEE round-to-nearest, as the kernels' intrinsics
    g = MeshGeom{vertices, faces, V, F, H, W, (float)W / (2.f * xmag), (float)H / (2.f * ymag), 0.5f * (float)W, 0.5f * (float)H};
    return true;
}

}  // namespace p3d

using namespace p3d;

extern "C" {

int p3d_mesh_raster(const float* vertices, int64_t V, const int64_t* faces, int64_t F, const p3d_mesh_view_t* views, int N,
                    int H, int W, float xmag, float ymag, float znear, float zfar, uint64_t* depth_keys, int64_t* guard_drops,
                    p3d_stream_t stream) {
    MeshGeom g;
    if (!depth_keys || !guard_drops || !mesh_geom(vertices, V, faces, F, views, N, H, W, xmag, ymag, g)) return P3D_BAD_ARG;
    if (!(znear > 0.f) || !(znear < zfar)) return P3D_BAD_ARG;
    cudaStream_t s = (cudaStream_t)stream;
    P3D_CUDA_TRY(cudaMemsetAsync(depth_keys, 0xff, (size_t)N * H * W * sizeof(uint64_t), s));
    P3D_CUDA_TRY(cudaMemsetAsync(guard_drops, 0, sizeof(int64_t), s));
    if (F == 0) return P3D_OK;
    const dim3 grid((unsigned)ceil_div64(F, kRasterThreads), (unsigned)ceil_div(N, kRasterViews));
    mesh_raster_kernel<<<grid, kRasterThreads, 0, s>>>(g, views, N, znear, zfar, reinterpret_cast<unsigned long long*>(depth_keys),
                                                       reinterpret_cast<unsigned long long*>(guard_drops));
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

int p3d_mesh_shade(const uint64_t* depth_keys, const float* vertices, int64_t V, const int64_t* faces, int64_t F,
                   const p3d_mesh_view_t* views, int N, int H, int W, float xmag, float ymag,
                   const unsigned char* vertex_colors, float light_intensity, unsigned char* out, p3d_stream_t stream) {
    MeshGeom g;
    if (!depth_keys || !out || !mesh_geom(vertices, V, faces, F, views, N, H, W, xmag, ymag, g)) return P3D_BAD_ARG;
    const int64_t pixels = (int64_t)N * H * W;
    mesh_shade_kernel<<<(unsigned)ceil_div64(pixels, kShadeThreads), kShadeThreads, 0, (cudaStream_t)stream>>>(
        g, views, reinterpret_cast<const unsigned long long*>(depth_keys), vertex_colors, light_intensity, pixels, out);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

}  // extern "C"
