// Marching cubes on the device: the mesh half of create_mesh (pi_GAN/utils.py:99-180, skimage marching cubes at level -20).
// The triangle table, its numbering and the rule that generates it are in mc_tables.cuh / oracle/marching_cubes.py.
//
// Three streaming passes over the lattice, one thread per point along the fastest axis (coalesced), tiles of kTile
// consecutive linear indices per CTA:
//   mc_count_kernel     reads the field; writes one 32-bit word per point (crossing bits of the point's 3 owned edges,
//                       the configuration of the cell it is the minimum corner of, the point's first vertex index within
//                       its tile) and the tile's vertex / triangle counts
//   mc_scan_kernel      exclusive scan of the tile counts (one CTA) + the totals (V, F)
//   mc_vertices_kernel  reads the words, and the field at crossing points only; writes the vertices
//   mc_faces_kernel     reads the words of the cell corners; writes the triangles
//   mc_normals_kernel   (optional, b2r_mc_normals) like mc_vertices_kernel; reads the field around both ends of every crossing
//                       edge and writes the unit vertex normals in vertex order
// HBM traffic: 4 B (field) + 4 B (word) written, 4 B read twice, plus the field at the crossing points and the output.
// Every vertex component is formed with separately rounded operations (no FMA), so numpy float32 reproduces it bit for bit.
#include "common.cuh"
#include "mc_tables.cuh"

namespace b2r {
namespace mc {

constexpr int kThreads = 256;
constexpr int kPer = 8;                         // points per thread: q * kThreads + threadIdx.x within the tile
constexpr int kTile = kThreads * kPer;
constexpr int kWarps = kThreads / kWarp;
constexpr int kScanThreads = 1024;
static_assert(kPer * kWarps == 2 * kWarp, "tile_scan: warp 0 scans two warp totals per lane");
static_assert(kTile * 3 < 65536 && kTile * kMaxTriangles < 65536, "tile counts are packed as two 16-bit fields");

// word per point: bits 0..2 = crossing edge owned along axis 0..2, bits 8..15 = cell configuration (0 when the point is not
// a cell's minimum corner), bits 16..31 = index of the point's first vertex within its tile
constexpr unsigned kCfgShift = 8, kVertShift = 16;

struct Layout {
    size_t words, counts, offsets, total;
};

inline size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

inline Layout layout(long long n) {
    const long long tiles = (n + kTile - 1) / kTile;
    Layout l;
    l.words = 0;
    l.counts = l.words + align256((size_t)n * 4);
    l.offsets = l.counts + align256((size_t)tiles * 4);
    l.total = l.offsets + align256((size_t)tiles * sizeof(longlong2));
    return l;
}

// Exclusive prefix of v[q] over the tile in linear order (q-major, then thread); returns the tile total.
__device__ __forceinline__ unsigned tile_scan(unsigned (&v)[kPer], unsigned* s /* [kPer * kWarps + 1] */) {
    const int lane = threadIdx.x & (kWarp - 1), warp = threadIdx.x >> 5;
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        unsigned x = v[q];
#pragma unroll
        for (int o = 1; o < kWarp; o <<= 1) {
            const unsigned y = __shfl_up_sync(kFull, x, o);
            if (lane >= o) x += y;
        }
        if (lane == kWarp - 1) s[q * kWarps + warp] = x;
        v[q] = x - v[q];
    }
    __syncthreads();
    if (warp == 0) {
        const unsigned a = s[2 * lane], b = s[2 * lane + 1];
        unsigned x = a + b;
#pragma unroll
        for (int o = 1; o < kWarp; o <<= 1) {
            const unsigned y = __shfl_up_sync(kFull, x, o);
            if (lane >= o) x += y;
        }
        s[2 * lane] = x - a - b;
        s[2 * lane + 1] = x - b;
        if (lane == kWarp - 1) s[kPer * kWarps] = x;
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < kPer; ++q) v[q] += s[q * kWarps + warp];
    return s[kPer * kWarps];
}

__global__ void __launch_bounds__(kThreads) mc_count_kernel(const float* __restrict__ f, int n0, int n1, int n2, float level,
                                                            unsigned* __restrict__ words, unsigned* __restrict__ tile_counts) {
    __shared__ unsigned s_ntri[256];
    __shared__ unsigned s_scan[kPer * kWarps + 1];
    static_assert(kThreads == 256, "one configuration per thread");
    s_ntri[threadIdx.x] = (unsigned)(kTriangles[threadIdx.x] >> 60);
    __syncthreads();
    const unsigned n = (unsigned)n0 * n1 * n2, s1 = (unsigned)n2, s0 = (unsigned)n1 * n2;
    const unsigned base = blockIdx.x * (unsigned)kTile;
    unsigned word[kPer], cnt[kPer];
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        const unsigned idx = base + q * kThreads + threadIdx.x;
        word[q] = 0;
        cnt[q] = 0;
        if (idx >= n) continue;
        const unsigned k = idx % s1, r = idx / s1, j = r % (unsigned)n1, i = r / (unsigned)n1;
        const bool ci = i + 1 < (unsigned)n0, cj = j + 1 < (unsigned)n1, ck = k + 1 < (unsigned)n2;
        auto below = [&](unsigned at) -> unsigned { return f[at] < level ? 1u : 0u; };   // NaN is not below
        unsigned b = below(idx);                                   // bit c = corner c (offset (c>>2, c>>1 & 1, c & 1))
        if (ck) b |= below(idx + 1) << 1;
        if (cj) b |= below(idx + s1) << 2;
        if (ci) b |= below(idx + s0) << 4;
        const bool cell = ci && cj && ck;
        if (cell) {
            b |= below(idx + s1 + 1) << 3;
            b |= below(idx + s0 + 1) << 5;
            b |= below(idx + s0 + s1) << 6;
            b |= below(idx + s0 + s1 + 1) << 7;
        }
        const unsigned bits = (ci ? ((b ^ (b >> 4)) & 1) : 0) | (cj ? ((b ^ (b >> 2)) & 1) << 1 : 0) |
                              (ck ? ((b ^ (b >> 1)) & 1) << 2 : 0);
        const unsigned cfg = cell ? b : 0;
        word[q] = bits | cfg << kCfgShift;
        cnt[q] = __popc(bits) | s_ntri[cfg] << 16;
    }
    const unsigned total = tile_scan(cnt, s_scan);
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        const unsigned idx = base + q * kThreads + threadIdx.x;
        if (idx < n) words[idx] = word[q] | (cnt[q] & 0xffffu) << kVertShift;
    }
    if (threadIdx.x == 0) tile_counts[blockIdx.x] = total;
}

// One CTA: thread t owns a contiguous run of tiles.  offsets[b] = (first vertex, first triangle) of tile b.
__global__ void __launch_bounds__(kScanThreads) mc_scan_kernel(const unsigned* __restrict__ tile_counts, int tiles,
                                                               longlong2* __restrict__ offsets, long long* __restrict__ totals) {
    __shared__ long long s_v[kScanThreads / kWarp], s_t[kScanThreads / kWarp];
    const int lane = threadIdx.x & (kWarp - 1), warp = threadIdx.x >> 5;
    const int per = (tiles + kScanThreads - 1) / kScanThreads;
    const int beg = min(tiles, (int)threadIdx.x * per), end = min(tiles, beg + per);
    long long sv = 0, st = 0;
    for (int b = beg; b < end; ++b) {
        const unsigned c = tile_counts[b];
        sv += c & 0xffffu;
        st += c >> 16;
    }
    long long xv = sv, xt = st;
#pragma unroll
    for (int o = 1; o < kWarp; o <<= 1) {
        const long long yv = __shfl_up_sync(kFull, xv, o), yt = __shfl_up_sync(kFull, xt, o);
        if (lane >= o) { xv += yv; xt += yt; }
    }
    if (lane == kWarp - 1) { s_v[warp] = xv; s_t[warp] = xt; }
    __syncthreads();
    if (warp == 0) {
        long long av = s_v[lane], at = s_t[lane], yv = av, yt = at;
#pragma unroll
        for (int o = 1; o < kWarp; o <<= 1) {
            const long long pv = __shfl_up_sync(kFull, yv, o), pt = __shfl_up_sync(kFull, yt, o);
            if (lane >= o) { yv += pv; yt += pt; }
        }
        s_v[lane] = yv - av;
        s_t[lane] = yt - at;
        if (lane == kWarp - 1) { totals[0] = yv; totals[1] = yt; }
    }
    __syncthreads();
    long long pv = s_v[warp] + xv - sv, pt = s_t[warp] + xt - st;
    for (int b = beg; b < end; ++b) {
        const unsigned c = tile_counts[b];
        offsets[b] = make_longlong2(pv, pt);
        pv += c & 0xffffu;
        pt += c >> 16;
    }
}

__global__ void __launch_bounds__(kThreads) mc_vertices_kernel(const float* __restrict__ f, int n0, int n1, int n2, float level,
                                                               float spacing, float ox, float oy, float oz,
                                                               const unsigned* __restrict__ words,
                                                               const longlong2* __restrict__ offsets, float* __restrict__ verts) {
    const unsigned n = (unsigned)n0 * n1 * n2, s1 = (unsigned)n2, s0 = (unsigned)n1 * n2;
    const unsigned base = blockIdx.x * (unsigned)kTile;
    const long long tile_v = offsets[blockIdx.x].x;
#pragma unroll 2
    for (int q = 0; q < kPer; ++q) {
        const unsigned idx = base + q * kThreads + threadIdx.x;
        if (idx >= n) break;
        const unsigned w = words[idx];
        if (!(w & 7u)) continue;
        const unsigned k = idx % s1, r = idx / s1, j = r % (unsigned)n1, i = r / (unsigned)n1;
        const float f0 = f[idx];
        const float p[3] = {(float)i, (float)j, (float)k}, o[3] = {ox, oy, oz};
        const unsigned step[3] = {s0, s1, 1u};
        float* out = verts + 3 * (tile_v + (w >> kVertShift));
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (!(w >> a & 1u)) continue;
            const float t = __fdiv_rn(__fsub_rn(level, f0), __fsub_rn(f[idx + step[a]], f0));
#pragma unroll
            for (int c = 0; c < 3; ++c) out[c] = __fadd_rn(o[c], __fmul_rn(c == a ? __fadd_rn(p[c], t) : p[c], spacing));
            out += 3;
        }
    }
}

// Component of the field's gradient along one axis at lattice coordinate c of n (np.gradient's scheme with the isotropic spacing
// dropped): central difference inside, one-sided on the faces.  step = the axis' linear-index stride.
__device__ __forceinline__ float grad_axis(const float* __restrict__ f, unsigned idx, unsigned c, unsigned n, unsigned step) {
    if (c == 0) return __fsub_rn(f[idx + step], f[idx]);
    if (c + 1 == n) return __fsub_rn(f[idx], f[idx - step]);
    return __fmul_rn(0.5f, __fsub_rn(f[idx + step], f[idx - step]));
}

// The normal of the vertex on the edge p -> p + e_a is g(p) + t (g(p + e_a) - g(p)) with the vertex's own t, divided by its length;
// it points toward increasing field (the side the triangle normals face).  Zero length gives (0, 0, 0).
__global__ void __launch_bounds__(kThreads) mc_normals_kernel(const float* __restrict__ f, int n0, int n1, int n2, float level,
                                                              const unsigned* __restrict__ words,
                                                              const longlong2* __restrict__ offsets, float* __restrict__ normals) {
    const unsigned n = (unsigned)n0 * n1 * n2, s1 = (unsigned)n2, s0 = (unsigned)n1 * n2;
    const unsigned base = blockIdx.x * (unsigned)kTile;
    const long long tile_v = offsets[blockIdx.x].x;
#pragma unroll 1
    for (int q = 0; q < kPer; ++q) {
        const unsigned idx = base + q * kThreads + threadIdx.x;
        if (idx >= n) break;
        const unsigned w = words[idx];
        if (!(w & 7u)) continue;
        const unsigned k = idx % s1, r = idx / s1, j = r % (unsigned)n1, i = r / (unsigned)n1;
        const float f0 = f[idx];
        const unsigned p[3] = {i, j, k}, dims[3] = {(unsigned)n0, (unsigned)n1, (unsigned)n2}, step[3] = {s0, s1, 1u};
        float g0[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) g0[c] = grad_axis(f, idx, p[c], dims[c], step[c]);
        float* out = normals + 3 * (tile_v + (w >> kVertShift));
#pragma unroll
        for (int a = 0; a < 3; ++a) {
            if (!(w >> a & 1u)) continue;
            const unsigned at = idx + step[a];
            const float t = __fdiv_rn(__fsub_rn(level, f0), __fsub_rn(f[at], f0));
            float g[3];
#pragma unroll
            for (int c = 0; c < 3; ++c) {
                const float g1 = grad_axis(f, at, c == a ? p[c] + 1 : p[c], dims[c], step[c]);
                g[c] = __fadd_rn(g0[c], __fmul_rn(t, __fsub_rn(g1, g0[c])));
            }
            const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(g[0], g[0]), __fmul_rn(g[1], g[1])), __fmul_rn(g[2], g[2])));
#pragma unroll
            for (int c = 0; c < 3; ++c) out[c] = len > 0.f ? __fdiv_rn(g[c], len) : 0.f;
            out += 3;
        }
    }
}

__global__ void __launch_bounds__(kThreads) mc_faces_kernel(int n0, int n1, int n2, const unsigned* __restrict__ words,
                                                            const longlong2* __restrict__ offsets, int* __restrict__ faces) {
    __shared__ uint64_t s_tri[256];
    __shared__ unsigned s_scan[kPer * kWarps + 1];
    s_tri[threadIdx.x] = kTriangles[threadIdx.x];
    __syncthreads();
    const unsigned n = (unsigned)n0 * n1 * n2, s1 = (unsigned)n2, s0 = (unsigned)n1 * n2;
    const unsigned base = blockIdx.x * (unsigned)kTile;
    unsigned cnt[kPer], cfg[kPer];
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        const unsigned idx = base + q * kThreads + threadIdx.x;
        cfg[q] = idx < n ? (words[idx] >> kCfgShift) & 0xffu : 0u;
        cnt[q] = (unsigned)(s_tri[cfg[q]] >> 60);
    }
    tile_scan(cnt, s_scan);
    const long long tile_f = offsets[blockIdx.x].y;
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        const uint64_t tri = s_tri[cfg[q]];
        const int m3 = 3 * (int)(tri >> 60);
        if (!m3) continue;
        const unsigned idx = base + q * kThreads + threadIdx.x;
        int* out = faces + 3 * (tile_f + cnt[q]);
        for (int m = 0; m < m3; ++m) {
            const unsigned e = (unsigned)(tri >> (4 * m)) & 15u;
            const unsigned code = (unsigned)(kEdgeCode >> (5 * e)) & 31u, owner = code & 7u, axis = code >> 3;
            const unsigned at = idx + (owner >> 2) * s0 + ((owner >> 1) & 1u) * s1 + (owner & 1u);
            const unsigned w = words[at];
            out[m] = (int)(offsets[at / kTile].x + (w >> kVertShift) + __popc(w & ((1u << axis) - 1u)));
        }
    }
}

int check_grid(const char* what, int n0, int n1, int n2) {
    B2R_CHECK_ARG(n0 >= 2 && n1 >= 2 && n2 >= 2, "%s: every axis needs n >= 2 (got %d x %d x %d)", what, n0, n1, n2);
    B2R_CHECK_ARG((long long)n0 * n1 * n2 <= INT32_MAX, "%s: n0*n1*n2 = %lld exceeds INT32_MAX", what, (long long)n0 * n1 * n2);
    return 0;
}

}  // namespace mc
}  // namespace b2r

extern "C" size_t b2r_mc_scratch_bytes(int n0, int n1, int n2) {
    if (n0 < 2 || n1 < 2 || n2 < 2 || (long long)n0 * n1 * n2 > INT32_MAX) return 0;
    return b2r::mc::layout((long long)n0 * n1 * n2).total;
}

extern "C" int b2r_mc_count(const float* field, int n0, int n1, int n2, float level, void* scratch, long long* totals_dev,
                            void* stream) {
    using namespace b2r::mc;
    if (int rc = check_grid("b2r_mc_count", n0, n1, n2)) return rc;
    B2R_CHECK_ARG(field && scratch && totals_dev, "b2r_mc_count: NULL pointer");
    B2R_CHECK_ARG(((uintptr_t)scratch & 15) == 0, "b2r_mc_count: scratch must be 16-byte aligned");
    const long long n = (long long)n0 * n1 * n2;
    const Layout l = layout(n);
    const int tiles = (int)((n + kTile - 1) / kTile);
    char* s = static_cast<char*>(scratch);
    cudaStream_t st = (cudaStream_t)stream;
    mc_count_kernel<<<tiles, kThreads, 0, st>>>(field, n0, n1, n2, level, (unsigned*)(s + l.words), (unsigned*)(s + l.counts));
    mc_scan_kernel<<<1, kScanThreads, 0, st>>>((const unsigned*)(s + l.counts), tiles, (longlong2*)(s + l.offsets), totals_dev);
    B2R_LAUNCH_CHECK("b2r_mc_count");
    return 0;
}

extern "C" int b2r_mc_emit(const float* field, int n0, int n1, int n2, float level, float spacing, float ox, float oy, float oz,
                           const void* scratch, float* verts, int* faces, void* stream) {
    using namespace b2r::mc;
    if (int rc = check_grid("b2r_mc_emit", n0, n1, n2)) return rc;
    B2R_CHECK_ARG(field && scratch && verts && faces, "b2r_mc_emit: NULL pointer");
    B2R_CHECK_ARG(((uintptr_t)scratch & 15) == 0, "b2r_mc_emit: scratch must be 16-byte aligned");
    const long long n = (long long)n0 * n1 * n2;
    const Layout l = layout(n);
    const int tiles = (int)((n + kTile - 1) / kTile);
    const char* s = static_cast<const char*>(scratch);
    const unsigned* words = (const unsigned*)(s + l.words);
    const longlong2* offsets = (const longlong2*)(s + l.offsets);
    cudaStream_t st = (cudaStream_t)stream;
    mc_vertices_kernel<<<tiles, kThreads, 0, st>>>(field, n0, n1, n2, level, spacing, ox, oy, oz, words, offsets, verts);
    mc_faces_kernel<<<tiles, kThreads, 0, st>>>(n0, n1, n2, words, offsets, faces);
    B2R_LAUNCH_CHECK("b2r_mc_emit");
    return 0;
}

extern "C" int b2r_mc_normals(const float* field, int n0, int n1, int n2, float level, const void* scratch, float* normals,
                              void* stream) {
    using namespace b2r::mc;
    if (int rc = check_grid("b2r_mc_normals", n0, n1, n2)) return rc;
    B2R_CHECK_ARG(field && scratch && normals, "b2r_mc_normals: NULL pointer");
    B2R_CHECK_ARG(((uintptr_t)scratch & 15) == 0, "b2r_mc_normals: scratch must be 16-byte aligned");
    const long long n = (long long)n0 * n1 * n2;
    const Layout l = layout(n);
    const int tiles = (int)((n + kTile - 1) / kTile);
    const char* s = static_cast<const char*>(scratch);
    mc_normals_kernel<<<tiles, kThreads, 0, (cudaStream_t)stream>>>(field, n0, n1, n2, level, (const unsigned*)(s + l.words),
                                                                    (const longlong2*)(s + l.offsets), normals);
    B2R_LAUNCH_CHECK("b2r_mc_normals");
    return 0;
}
