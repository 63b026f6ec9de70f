// Marching cubes on a dense fp32 grid: the mcubes.marching_cubes(u, threshold) call of the reference's
// applications/extract_mesh.py:84-96, on the device. The mesh (inside-ness, vertex and face order, orientation) is defined
// in oracle/p3d_oracle/mesh.py, which also generates the triangle table in mc_table.cuh.
//
// Four launches, no atomics (the output depends only on the input):
//   mc_count_kernel       one thread per grid point and item: the point's owned-edge mask (3 bits: which of the edges
//                         p -> p + e_axis cross the threshold) and, at a cube origin, the cube's triangle count; one
//                         (vertices, triangles) partial per CTA;
//   mc_scan_kernel        one CTA: exclusive scan of the CTA partials in place, and the totals (V, F);
//   mc_emit_verts_kernel  recomputes the masks, adds the in-CTA prefix to the CTA offset, writes each point's first vertex
//                         id and its mask into the workspace, and the vertices;
//   mc_emit_faces_kernel  recomputes the cube configurations and writes the faces (they need ids owned by neighbouring
//                         points, hence the second pass).
// A CTA covers kMcPoints consecutive points in C order, thread t taking points base + t + r * kMcThreads, so both the
// vertex order (owning point, then axis) and the face order (cube, then table order) follow from the scans.
// HBM traffic: each pass reads the grid once (neighbour reads hit L1/L2); the emit passes add the outputs and the
// workspace entries of surface points.
#include "p3d_common.cuh"
#include "mc_table.cuh"

namespace p3d {

constexpr int kMcThreads = 256;
constexpr int kMcItems = 8;
constexpr int kMcPoints = kMcThreads * kMcItems;
constexpr int kMcScanThreads = 1024;

struct McGrid {
    const float* v;
    int64_t N, sx;          // points, stride of axis 0 (ny * nz)
    int32_t nx, ny, nz;
    double thr;
};

__device__ __forceinline__ bool mc_inside(const McGrid& g, int64_t idx) { return (double)__ldg(g.v + idx) > g.thr; }

// owned-edge mask of point (i, j, k) and, when it is a cube origin, the cube configuration (bit c = corner c inside,
// corner c = (c & 1, c >> 1 & 1, c >> 2 & 1) along axes 0, 1, 2); loads a kernel does not use are dropped by the compiler
__device__ __forceinline__ void mc_point(const McGrid& g, int64_t idx, int i, int j, int k, int& mask, int& cfg) {
    const bool xi = i < g.nx - 1, yj = j < g.ny - 1, zk = k < g.nz - 1;
    const int b0 = mc_inside(g, idx);
    const int b1 = xi && mc_inside(g, idx + g.sx);
    const int b2 = yj && mc_inside(g, idx + g.nz);
    const int b4 = zk && mc_inside(g, idx + 1);
    mask = (xi && b1 != b0) | (yj && b2 != b0) << 1 | (zk && b4 != b0) << 2;
    cfg = 0;
    if (xi && yj && zk) {
        const int b3 = mc_inside(g, idx + g.sx + g.nz), b5 = mc_inside(g, idx + g.sx + 1), b6 = mc_inside(g, idx + g.nz + 1);
        const int b7 = mc_inside(g, idx + g.sx + g.nz + 1);
        cfg = b0 | b1 << 1 | b2 << 2 | b3 << 3 | b4 << 4 | b5 << 5 | b6 << 6 | b7 << 7;
    }
}

// coordinates of the CTA's first point (one division per CTA), then per thread and item by stepping
struct McCursor {
    int64_t idx;
    int i, j, k;
    __device__ __forceinline__ void step(const McGrid& g, int n) {
        idx += n;
        k += n;
        while (k >= g.nz) {
            k -= g.nz;
            if (++j == g.ny) { j = 0; ++i; }
        }
    }
};

__device__ __forceinline__ McCursor mc_start(const McGrid& g, int* s_coord) {
    const int64_t base = (int64_t)blockIdx.x * kMcPoints;
    if (threadIdx.x == 0) {
        const int64_t row = base / g.nz;
        s_coord[0] = (int)(row / g.ny);
        s_coord[1] = (int)(row - (int64_t)s_coord[0] * g.ny);
        s_coord[2] = (int)(base - row * g.nz);
    }
    __syncthreads();
    McCursor c{base, s_coord[0], s_coord[1], s_coord[2]};
    c.step(g, threadIdx.x);
    return c;
}

// exclusive scan over the CTA in thread order; `total` = sum over the CTA. s_warp: one T per warp.
template <int kThreads, typename T>
__device__ __forceinline__ T mc_block_scan(T v, T* s_warp, T& total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    T x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const T y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
    }
    if (lane == 31) s_warp[warp] = x;
    __syncthreads();
    T before = 0, sum = 0;
#pragma unroll
    for (int w = 0; w < kThreads / 32; ++w) {
        const T s = s_warp[w];
        if (w < warp) before += s;
        sum += s;
    }
    __syncthreads();
    total = sum;
    return before + x - v;
}

__global__ void __launch_bounds__(kMcThreads) mc_count_kernel(const McGrid g, int64_t* __restrict__ partial, int nblocks) {
    __shared__ int s_coord[3];
    __shared__ int s_warp[kMcThreads / 32];
    __shared__ unsigned char s_count[256];
    s_count[threadIdx.x] = kMcTriCount[threadIdx.x];
    McCursor c = mc_start(g, s_coord);
    int nv = 0, nt = 0;
#pragma unroll 1
    for (int r = 0; r < kMcItems && c.idx < g.N; ++r, c.step(g, kMcThreads)) {
        int mask, cfg;
        mc_point(g, c.idx, c.i, c.j, c.k, mask, cfg);
        nv += __popc(mask);
        nt += s_count[cfg];
    }
    int tv, tt;
    mc_block_scan<kMcThreads>(nv, s_warp, tv);
    mc_block_scan<kMcThreads>(nt, s_warp, tt);
    if (threadIdx.x == 0) {
        partial[blockIdx.x] = tv;
        partial[nblocks + blockIdx.x] = tt;
    }
}

// partial [2][nblocks] -> exclusive offsets in place; counts = {V, F}
__global__ void __launch_bounds__(kMcScanThreads) mc_scan_kernel(int64_t* __restrict__ partial, int nblocks,
                                                                 int64_t* __restrict__ counts) {
    __shared__ long long s_warp[kMcScanThreads / 32];
    const int per = (nblocks + kMcScanThreads - 1) / kMcScanThreads;
    const int lo = min(nblocks, (int)threadIdx.x * per), hi = min(nblocks, lo + per);
    for (int a = 0; a < 2; ++a) {
        int64_t* p = partial + (int64_t)a * nblocks;
        long long s = 0;
        for (int x = lo; x < hi; ++x) s += p[x];
        long long total;
        long long run = mc_block_scan<kMcScanThreads>(s, s_warp, total);
        for (int x = lo; x < hi; ++x) {
            const long long n = p[x];
            p[x] = run;
            run += n;
        }
        if (threadIdx.x == 0) counts[a] = total;
    }
}

__global__ void __launch_bounds__(kMcThreads) mc_emit_verts_kernel(const McGrid g, const int64_t* __restrict__ offsets,
                                                                   int32_t* __restrict__ ids, unsigned char* __restrict__ masks,
                                                                   double* __restrict__ vertices) {
    __shared__ int s_coord[3];
    __shared__ int s_warp[kMcThreads / 32];
    McCursor c = mc_start(g, s_coord);
    int64_t next = offsets[blockIdx.x];
    const int64_t stride[3] = {g.sx, g.nz, 1};
#pragma unroll 1
    for (int r = 0; r < kMcItems; ++r, c.step(g, kMcThreads)) {
        int mask = 0, cfg;
        if (c.idx < g.N) mc_point(g, c.idx, c.i, c.j, c.k, mask, cfg);
        int total;
        int64_t id = next + mc_block_scan<kMcThreads>(__popc(mask), s_warp, total);
        next += total;
        if (!mask) continue;
        ids[c.idx] = (int32_t)id;
        masks[c.idx] = (unsigned char)mask;
        const double vp = (double)__ldg(g.v + c.idx);
        const int pc[3] = {c.i, c.j, c.k};
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (!(mask >> a & 1)) continue;
            const double vq = (double)__ldg(g.v + c.idx + stride[a]);
            // t = (thr - v_p) / (v_q - v_p), rounded operation by operation (no contraction), then p_a + t
            const double t = __ddiv_rn(__dsub_rn(g.thr, vp), __dsub_rn(vq, vp));
            double* o = vertices + 3 * id;
#pragma unroll
            for (int d = 0; d < 3; ++d) o[d] = d == a ? __dadd_rn((double)pc[d], t) : (double)pc[d];
            ++id;
        }
    }
}

__global__ void __launch_bounds__(kMcThreads) mc_emit_faces_kernel(const McGrid g, const int64_t* __restrict__ offsets,
                                                                   const int32_t* __restrict__ ids,
                                                                   const unsigned char* __restrict__ masks,
                                                                   int64_t* __restrict__ faces) {
    __shared__ int s_coord[3];
    __shared__ int s_warp[kMcThreads / 32];
    __shared__ signed char s_edges[256][16];
    __shared__ unsigned char s_count[256];
    __shared__ int64_t s_edge_off[12];
    for (int x = threadIdx.x; x < 256 * 16; x += kMcThreads) (&s_edges[0][0])[x] = (&kMcTriEdges[0][0])[x];
    s_count[threadIdx.x] = kMcTriCount[threadIdx.x];
    if (threadIdx.x < 12) {
        const int b = kMcEdgeCorner[threadIdx.x];
        s_edge_off[threadIdx.x] = (b & 1) * g.sx + (b >> 1 & 1) * g.nz + (b >> 2 & 1);
    }
    McCursor c = mc_start(g, s_coord);        // its __syncthreads() also publishes the tables
    int64_t next = offsets[blockIdx.x];
#pragma unroll 1
    for (int r = 0; r < kMcItems; ++r, c.step(g, kMcThreads)) {
        int mask, cfg = 0;
        if (c.idx < g.N) mc_point(g, c.idx, c.i, c.j, c.k, mask, cfg);
        const int nt = s_count[cfg];
        int total;
        int64_t f = next + mc_block_scan<kMcThreads>(nt, s_warp, total);
        next += total;
        for (int e = 0; e < 3 * nt; ++e) {
            const int edge = s_edges[cfg][e], axis = edge >> 2;
            const int64_t q = c.idx + s_edge_off[edge];
            faces[3 * f + e] = (int64_t)__ldg(ids + q) + __popc(__ldg(masks + q) & ((1 << axis) - 1));
        }
    }
}

struct McLayout {
    int nblocks;
    int64_t partial_off, ids_off, masks_off, bytes;
};

static bool mc_layout(int64_t nx, int64_t ny, int64_t nz, McLayout& L) {
    if (nx < 2 || ny < 2 || nz < 2 || nx > INT32_MAX || ny > INT32_MAX || nz > INT32_MAX) return false;
    if (nx > ((int64_t)1 << 40) / ny / nz) return false;
    const int64_t N = nx * ny * nz;
    const int64_t nb = ceil_div64(N, kMcPoints);
    if (nb > INT32_MAX) return false;
    auto align = [](int64_t b) { return (b + 255) & ~(int64_t)255; };
    L.nblocks = (int)nb;
    L.partial_off = 0;
    L.ids_off = align(16 * nb);
    L.masks_off = L.ids_off + align(4 * N);
    L.bytes = L.masks_off + align(N);
    return true;
}

static McGrid mc_grid(const float* volume, int64_t nx, int64_t ny, int64_t nz, double threshold) {
    return McGrid{volume, nx * ny * nz, ny * nz, (int32_t)nx, (int32_t)ny, (int32_t)nz, threshold};
}

}  // namespace p3d

using namespace p3d;

extern "C" {

int64_t p3d_marching_cubes_workspace_bytes(int64_t nx, int64_t ny, int64_t nz) {
    McLayout L;
    return mc_layout(nx, ny, nz, L) ? L.bytes : P3D_BAD_ARG;
}

int p3d_marching_cubes_count(const float* volume, int64_t nx, int64_t ny, int64_t nz, double threshold, void* workspace,
                             int64_t workspace_bytes, int64_t* counts, p3d_stream_t stream) {
    McLayout L;
    if (!volume || !workspace || !counts || !mc_layout(nx, ny, nz, L) || workspace_bytes < L.bytes) return P3D_BAD_ARG;
    const McGrid g = mc_grid(volume, nx, ny, nz, threshold);
    int64_t* partial = reinterpret_cast<int64_t*>(static_cast<char*>(workspace) + L.partial_off);
    mc_count_kernel<<<L.nblocks, kMcThreads, 0, (cudaStream_t)stream>>>(g, partial, L.nblocks);
    P3D_LAUNCH_CHECK();
    mc_scan_kernel<<<1, kMcScanThreads, 0, (cudaStream_t)stream>>>(partial, L.nblocks, counts);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

int p3d_marching_cubes_emit(const float* volume, int64_t nx, int64_t ny, int64_t nz, double threshold, void* workspace,
                            int64_t workspace_bytes, double* vertices, int64_t* faces, p3d_stream_t stream) {
    McLayout L;
    if (!volume || !workspace || !mc_layout(nx, ny, nz, L) || workspace_bytes < L.bytes) return P3D_BAD_ARG;
    const McGrid g = mc_grid(volume, nx, ny, nz, threshold);
    char* ws = static_cast<char*>(workspace);
    const int64_t* partial = reinterpret_cast<const int64_t*>(ws + L.partial_off);
    int32_t* ids = reinterpret_cast<int32_t*>(ws + L.ids_off);
    unsigned char* masks = reinterpret_cast<unsigned char*>(ws + L.masks_off);
    mc_emit_verts_kernel<<<L.nblocks, kMcThreads, 0, (cudaStream_t)stream>>>(g, partial, ids, masks, vertices);
    P3D_LAUNCH_CHECK();
    mc_emit_faces_kernel<<<L.nblocks, kMcThreads, 0, (cudaStream_t)stream>>>(g, partial + L.nblocks, ids, masks, faces);
    P3D_LAUNCH_CHECK();
    return P3D_OK;
}

}  // extern "C"
