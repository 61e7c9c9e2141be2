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
#include <cmath>

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

// ---- connected components of a triangle mesh (b2r_mesh_cc_*) ----------------------------------------------------------------
// Vertices are joined by the edges (v0,v1), (v1,v2) of every face.  Labelling is union-find over the faces, ECL-CC style: a
// union hooks the larger root under the smaller with atomicCAS, so parent[v] <= v always, the minimum vertex of a component is
// its only root once every union is done, and the labels (root of each vertex) are the minimum-index labels whatever the
// schedule.  Selection counts the faces per label (warp-aggregated: faces arrive in lattice order, so one dominant component
// would otherwise serialise nearly every atomic on one address), takes their integer maximum and marks what is kept.
// Compaction (mark_kernel, compact_kernel, shared with the edge collapse) writes the kept vertices and faces in their relative
// order, no sort and no atomics.
//
// Scratch: a[V] (the parent array while labelling, triangle counts per label while selecting), then the compaction tail, whose
// last 256 bytes hold the maximum.

// The end of every compaction scratch, from byte `at`: vword[V], tile counts and offsets as in marching cubes, and 256 bytes
// that the caller uses for its own device scalars.
struct CompactTail {
    size_t vword, counts, offsets, last, total;
};

inline long long compact_tiles(long long n_verts, long long n_faces) {
    return ((n_verts > n_faces ? n_verts : n_faces) + kTile - 1) / kTile;
}

inline CompactTail compact_tail(size_t at, long long n_verts, long long n_faces) {
    const long long tiles = compact_tiles(n_verts, n_faces);
    CompactTail t;
    t.vword = at;
    t.counts = t.vword + align256((size_t)n_verts * 4);
    t.offsets = t.counts + align256((size_t)tiles * 4);
    t.last = t.offsets + align256((size_t)tiles * sizeof(longlong2));
    t.total = t.last + 256;
    return t;
}

struct CcLayout {
    size_t a;
    CompactTail tail;
};

inline CcLayout cc_layout(long long n_verts, long long n_faces) {
    CcLayout l;
    l.a = 0;
    l.tail = compact_tail(l.a + align256((size_t)n_verts * 4), n_verts, n_faces);
    return l;
}

// vword per vertex: bit 31 = kept, bits 0..15 = rank of the vertex among the kept ones of its tile.  Tile b covers vertices AND
// faces [b*kTile, +kTile): its kept-vertex and kept-face counts are the two 16-bit fields mc_scan_kernel expects, so the scan
// writes (V', F') and every tile's (first vertex, first face).
constexpr unsigned kKept = 1u << 31;

// Keep: __device__ bool vert(unsigned v) const and bool face(unsigned f) const, whether vertex v / face f survives.
// Keep and Emit carry their pointers as struct members, where __restrict__ has no effect, so their read-only loads use __ldg: that
// keeps them on the read-only path and lets them be issued ahead of the stores of compact_kernel.
template <class Keep>
__global__ void __launch_bounds__(kThreads) mark_kernel(Keep keep, unsigned n_faces, unsigned n_verts, unsigned* __restrict__ vword,
                                                        unsigned* __restrict__ tile_counts) {
    __shared__ unsigned s_scan[kPer * kWarps + 1];
    const unsigned base = blockIdx.x * (unsigned)kTile;
    unsigned cnt[kPer], kept = 0;
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        const unsigned idx = base + q * kThreads + threadIdx.x;
        const unsigned kv = idx < n_verts && keep.vert(idx) ? 1u : 0u;
        const unsigned kf = idx < n_faces && keep.face(idx) ? 1u : 0u;
        kept |= kv << q;
        cnt[q] = kv | kf << 16;
    }
    const unsigned total = tile_scan(cnt, s_scan);
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        const unsigned idx = base + q * kThreads + threadIdx.x;
        if (idx < n_verts) vword[idx] = (kept >> q & 1u ? kKept : 0u) | (cnt[q] & 0xffffu);
    }
    if (threadIdx.x == 0) tile_counts[blockIdx.x] = total;
}

// Kept vertex v goes to offsets[v / kTile].x + its rank; a kept face goes to its tile's first face + its rank among the tile's
// kept faces, each index u replaced by the kept vertex it maps to.  Emit: __device__ void vert(unsigned v, size_t to) const writes
// kept vertex v's payload as output vertex `to`; bool face(unsigned f, const unsigned (&t)[3]) const, whether face f with indices t
// survives; unsigned target(unsigned u) const, the kept vertex index u maps to.
template <class Emit>
__global__ void __launch_bounds__(kThreads) compact_kernel(Emit emit, const int* __restrict__ faces, unsigned n_faces, unsigned n_verts,
                                                           const unsigned* __restrict__ vword, const longlong2* __restrict__ offsets,
                                                           int* __restrict__ faces_out) {
    __shared__ unsigned s_scan[kPer * kWarps + 1];
    const unsigned base = blockIdx.x * (unsigned)kTile;
    const longlong2 off = offsets[blockIdx.x];
#pragma unroll 2
    for (int q = 0; q < kPer; ++q) {
        const unsigned v = base + q * kThreads + threadIdx.x;
        if (v >= n_verts) break;
        const unsigned w = vword[v];
        if (w & kKept) emit.vert(v, (size_t)(off.x + (w & 0xffffu)));
    }
    // The face indices are read again for the remap rather than held across tile_scan: holding all kPer * 3 of them takes
    // both instantiations to 64 registers (48 for DecEmit this way), one resident CTA per SM fewer.
    unsigned cnt[kPer];
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        const unsigned f = base + q * kThreads + threadIdx.x;
        cnt[q] = 0;
        if (f >= n_faces) continue;
        unsigned t[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) t[c] = (unsigned)faces[3 * (size_t)f + c];
        cnt[q] = emit.face(f, t) ? 1u : 0u;
    }
    unsigned kept = 0;
#pragma unroll
    for (int q = 0; q < kPer; ++q) kept |= cnt[q] << q;
    tile_scan(cnt, s_scan);
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        if (!(kept >> q & 1u)) continue;
        const unsigned f = base + q * kThreads + threadIdx.x;
        int* out = faces_out + 3 * (off.y + cnt[q]);
#pragma unroll
        for (int c = 0; c < 3; ++c) {
            const unsigned u = emit.target((unsigned)faces[3 * (size_t)f + c]);
            out[c] = (int)(offsets[u / kTile].x + (vword[u] & 0xffffu));
        }
    }
}

__global__ void cc_init_kernel(unsigned* __restrict__ parent, unsigned n_verts) {
    const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n_verts) parent[v] = v;
}

// Root of v with path halving.  Other threads hook roots and halve paths at the same time; every store replaces a parent by one
// of its ancestors, so any value read is an ancestor and the walk ends at the current root.
__device__ __forceinline__ unsigned cc_find(unsigned* parent, unsigned v) {
    volatile unsigned* p = parent;
    unsigned u = p[v];
    while (u != v) {
        const unsigned w = p[u];
        if (w == u) return u;
        p[v] = w;
        v = w;
        u = p[v];
    }
    return v;
}

__device__ __forceinline__ void cc_union(unsigned* parent, unsigned a, unsigned b) {
    a = cc_find(parent, a);
    b = cc_find(parent, b);
    while (a != b) {
        const unsigned lo = min(a, b), hi = max(a, b);
        const unsigned old = atomicCAS(parent + hi, hi, lo);
        if (old == hi) return;
        a = cc_find(parent, old);      // hi was hooked meanwhile: retry from its new root
        b = lo;
    }
}

__global__ void cc_hook_kernel(const int* __restrict__ faces, unsigned n_faces, unsigned* __restrict__ parent) {
    const unsigned f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= n_faces) return;
    const unsigned v0 = (unsigned)faces[3 * (size_t)f], v1 = (unsigned)faces[3 * (size_t)f + 1], v2 = (unsigned)faces[3 * (size_t)f + 2];
    cc_union(parent, v0, v1);
    cc_union(parent, v1, v2);
}

__global__ void cc_labels_kernel(unsigned* __restrict__ parent, unsigned n_verts, int* __restrict__ labels) {
    const unsigned v = blockIdx.x * blockDim.x + threadIdx.x;
    if (v < n_verts) labels[v] = (int)cc_find(parent, v);
}

// tri[label of v0] += 1 per face, one atomic per distinct label per warp.
__global__ void cc_count_kernel(const int* __restrict__ faces, unsigned n_faces, const int* __restrict__ labels,
                                unsigned* __restrict__ tri) {
    const unsigned f = blockIdx.x * blockDim.x + threadIdx.x;
    const unsigned l = f < n_faces ? (unsigned)labels[faces[3 * (size_t)f]] : ~0u;
    const unsigned same = __match_any_sync(kFull, l);
    if (l != ~0u && (threadIdx.x & (kWarp - 1)) == (unsigned)(__ffs(same) - 1)) atomicAdd(tri + l, (unsigned)__popc(same));
}

__global__ void __launch_bounds__(kThreads) cc_max_kernel(const unsigned* __restrict__ tri, unsigned n_verts, unsigned* __restrict__ out) {
    __shared__ unsigned s[kWarps];
    unsigned m = 0;
    for (unsigned v = blockIdx.x * kThreads + threadIdx.x; v < n_verts; v += gridDim.x * kThreads) m = max(m, tri[v]);
    m = __reduce_max_sync(kFull, m);
    if ((threadIdx.x & (kWarp - 1)) == 0) s[threadIdx.x >> 5] = m;
    __syncthreads();
    if (threadIdx.x < kWarp) {
        m = __reduce_max_sync(kFull, threadIdx.x < kWarps ? s[threadIdx.x] : 0u);
        if (threadIdx.x == 0) atomicMax(out, m);
    }
}

// A component with t triangles is kept iff t > 0 and t >= ratio * t_max in float64 (ratio 0 keeps everything).
__device__ __forceinline__ unsigned cc_keep(unsigned t, float ratio, unsigned t_max) {
    return ratio == 0.f || (t > 0 && (double)t >= __dmul_rn((double)ratio, (double)t_max)) ? 1u : 0u;
}

// A vertex is kept iff its component is; a face iff its first vertex is (its three vertices share one component).
struct CcKeep {
    const int* faces;
    const int* labels;
    const unsigned* tri;
    const unsigned* t_max;
    float ratio;
    __device__ bool vert(unsigned v) const { return cc_keep(__ldg(tri + __ldg(labels + v)), ratio, __ldg(t_max)); }
    __device__ bool face(unsigned f) const { return vert((unsigned)__ldg(faces + 3 * (size_t)f)); }
};

// Kept vertices keep their position (and normal, when normals is given) and index; a face is kept iff its first vertex is.
struct CcEmit {
    const float* verts;
    const float* normals;
    const unsigned* vword;
    float* verts_out;
    float* normals_out;
    __device__ void vert(unsigned v, size_t to) const {
#pragma unroll
        for (int c = 0; c < 3; ++c) verts_out[3 * to + c] = __ldg(verts + 3 * (size_t)v + c);
        if (normals) {
#pragma unroll
            for (int c = 0; c < 3; ++c) normals_out[3 * to + c] = __ldg(normals + 3 * (size_t)v + c);
        }
    }
    __device__ bool face(unsigned, const unsigned (&t)[3]) const { return __ldg(vword + t[0]) >> 31; }
    __device__ unsigned target(unsigned u) const { return u; }
};

// ---- vertex-face adjacency, Taubin smoothing and mesh normals (b2r_mesh_adjacency / _smooth / _normals) -------------------------
// A corner is (f, c) with faces[f][c] == v; each vertex's corners are stored contiguously in ascending (f, c), so every sum over
// them runs in one fixed order and the float path needs no atomics.  Build: count the corners of each vertex (64-bit atomics into
// ends[]), exclusive 64-bit scan of the counts (tile sums, one-CTA scan of the tile sums, tile scans), fill the corner keys
// 3f + c with an atomic cursor (ends[v] then holds the END of v's list: begin(v) = ends[v-1], begin(0) = 0), and sort each
// vertex's keys (insertion sort up to kAdjInsertion keys, heapsort above, so any degree is exact in O(d log d)), replacing each key
// by its record in place.  The record is the int2 (a, b) = (faces[f][(c+1)%3], faces[f][(c+2)%3]) with c in the two spare high
// bits (bit 31 of a = c & 1, bit 31 of b = c >> 1): a half-step only gathers positions, and the normals kernel rebuilds the face's
// own corner order from (v, a, b, c).
// Scratch: ends[V] (u64), tile sums (u64 per kTile vertices), the records [3F] (int2), and a [V,3] position buffer that the
// half-steps ping-pong through.
struct AdjLayout {
    size_t ends, tile_sums, adj, pos, total;
};

inline AdjLayout adj_layout(long long n_verts, long long n_faces) {
    const long long tiles = (n_verts + kTile - 1) / kTile;
    AdjLayout l;
    l.ends = 0;
    l.tile_sums = l.ends + align256((size_t)n_verts * 8);
    l.adj = l.tile_sums + align256((size_t)tiles * 8);
    l.pos = l.adj + align256((size_t)n_faces * 24);
    l.total = l.pos + align256((size_t)n_verts * 12);
    return l;
}

constexpr int kAdjInsertion = 16;
constexpr unsigned kIndexMask = 0x7fffffffu;
constexpr float kTaubinLambda = 0.5f, kTaubinMu = -0.53f;

__device__ __forceinline__ unsigned rec_a(int2 r) { return (unsigned)r.x & kIndexMask; }
__device__ __forceinline__ unsigned rec_b(int2 r) { return (unsigned)r.y & kIndexMask; }

// The face of record r of vertex v in its own corner order: the cyclic order (v, a, b) starts at corner c of the face.
__device__ __forceinline__ void rec_face(int2 r, unsigned v, unsigned (&f)[3]) {
    const unsigned a = rec_a(r), b = rec_b(r);
    const unsigned c = (unsigned)r.x >> 31 | ((unsigned)r.y >> 31) << 1;
    f[0] = c == 0 ? v : c == 1 ? b : a;
    f[1] = c == 0 ? a : c == 1 ? v : b;
    f[2] = c == 0 ? b : c == 1 ? a : v;
}

__global__ void __launch_bounds__(kThreads) adj_count_kernel(const int* __restrict__ faces, unsigned n_faces,
                                                             unsigned long long* __restrict__ ends) {
    const unsigned f = blockIdx.x * kThreads + threadIdx.x;
    if (f >= n_faces) return;
#pragma unroll
    for (int c = 0; c < 3; ++c) atomicAdd(ends + faces[3 * (size_t)f + c], 1ull);
}

__device__ __forceinline__ unsigned long long warp_inclusive_scan64(unsigned long long x, int lane) {
#pragma unroll
    for (int o = 1; o < kWarp; o <<= 1) {
        const unsigned long long y = __shfl_up_sync(kFull, x, o);
        if (lane >= o) x += y;
    }
    return x;
}

// Thread t of tile b owns the kPer consecutive counts from b * kTile + t * kPer.
__global__ void __launch_bounds__(kThreads) adj_tile_sum_kernel(const unsigned long long* __restrict__ cnt, unsigned n,
                                                                unsigned long long* __restrict__ tile_sums) {
    __shared__ unsigned long long s_w[kWarps];
    const unsigned base = blockIdx.x * (unsigned)kTile + threadIdx.x * kPer;
    unsigned long long t = 0;
#pragma unroll
    for (int q = 0; q < kPer; ++q)
        if (base + q < n) t += cnt[base + q];
#pragma unroll
    for (int o = kWarp / 2; o; o >>= 1) t += __shfl_down_sync(kFull, t, o);
    if ((threadIdx.x & (kWarp - 1)) == 0) s_w[threadIdx.x >> 5] = t;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long s = 0;
#pragma unroll
        for (int w = 0; w < kWarps; ++w) s += s_w[w];
        tile_sums[blockIdx.x] = s;
    }
}

// One CTA, in place: tile_sums[b] becomes the sum of the tiles before b.  Thread t owns a contiguous run of tiles.
__global__ void __launch_bounds__(kScanThreads) adj_scan_tiles_kernel(unsigned long long* __restrict__ tile_sums, int tiles) {
    __shared__ unsigned long long s_w[kScanThreads / kWarp];
    const int lane = threadIdx.x & (kWarp - 1), warp = threadIdx.x >> 5;
    const int per = (tiles + kScanThreads - 1) / kScanThreads;
    const int beg = min(tiles, (int)threadIdx.x * per), end = min(tiles, beg + per);
    unsigned long long t = 0;
    for (int b = beg; b < end; ++b) t += tile_sums[b];
    const unsigned long long incl = warp_inclusive_scan64(t, lane);
    if (lane == kWarp - 1) s_w[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const unsigned long long x = s_w[lane];
        s_w[lane] = warp_inclusive_scan64(x, lane) - x;
    }
    __syncthreads();
    unsigned long long run = s_w[warp] + incl - t;
    for (int b = beg; b < end; ++b) {
        const unsigned long long x = tile_sums[b];
        tile_sums[b] = run;
        run += x;
    }
}

// In place: cnt[v] becomes the exclusive prefix sum of the counts (the first slot of v's corners).
__global__ void __launch_bounds__(kThreads) adj_tile_scan_kernel(unsigned long long* __restrict__ cnt, unsigned n,
                                                                 const unsigned long long* __restrict__ tile_offsets) {
    __shared__ unsigned long long s_w[kWarps];
    const int lane = threadIdx.x & (kWarp - 1), warp = threadIdx.x >> 5;
    const unsigned base = blockIdx.x * (unsigned)kTile + threadIdx.x * kPer;
    unsigned long long v[kPer], t = 0;
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        v[q] = base + q < n ? cnt[base + q] : 0ull;
        t += v[q];
    }
    const unsigned long long incl = warp_inclusive_scan64(t, lane);
    if (lane == kWarp - 1) s_w[warp] = incl;
    __syncthreads();
    if (warp == 0) {
        const unsigned long long x = lane < kWarps ? s_w[lane] : 0ull;
        const unsigned long long y = warp_inclusive_scan64(x, lane);
        __syncwarp();
        if (lane < kWarps) s_w[lane] = y - x;
    }
    __syncthreads();
    unsigned long long run = tile_offsets[blockIdx.x] + s_w[warp] + incl - t;
#pragma unroll
    for (int q = 0; q < kPer; ++q) {
        if (base + q < n) cnt[base + q] = run;
        run += v[q];
    }
}

// Corner (f, c) takes the next free slot of its vertex; ends[v] moves from v's first slot to one past its last.
__global__ void __launch_bounds__(kThreads) adj_fill_kernel(const int* __restrict__ faces, unsigned n_faces,
                                                            unsigned long long* __restrict__ ends, unsigned long long* __restrict__ keys) {
    const unsigned f = blockIdx.x * kThreads + threadIdx.x;
    if (f >= n_faces) return;
#pragma unroll
    for (int c = 0; c < 3; ++c) keys[atomicAdd(ends + faces[3 * (size_t)f + c], 1ull)] = 3ull * f + c;
}

__device__ __forceinline__ unsigned long long adj_begin(const unsigned long long* __restrict__ ends, unsigned v) {
    return v ? ends[v - 1] : 0ull;
}

// Sorts the keys of one vertex ascending and replaces each by its record (a, b, c), stored as the int2's little-endian u64.
__global__ void __launch_bounds__(kThreads) adj_sort_kernel(const int* __restrict__ faces, unsigned n_verts,
                                                            const unsigned long long* __restrict__ ends, unsigned long long* __restrict__ keys) {
    const unsigned v = blockIdx.x * kThreads + threadIdx.x;
    if (v >= n_verts) return;
    const unsigned long long beg = adj_begin(ends, v);
    const long long d = (long long)(ends[v] - beg);
    unsigned long long* a = keys + beg;
    if (d <= kAdjInsertion) {
        for (long long i = 1; i < d; ++i) {
            const unsigned long long k = a[i];
            long long j = i;
            for (; j > 0 && a[j - 1] > k; --j) a[j] = a[j - 1];
            a[j] = k;
        }
    } else {
        auto sift = [a](long long root, long long n) {
            const unsigned long long k = a[root];
            for (long long child = 2 * root + 1; child < n; child = 2 * root + 1) {
                if (child + 1 < n && a[child + 1] > a[child]) ++child;
                if (a[child] <= k) break;
                a[root] = a[child];
                root = child;
            }
            a[root] = k;
        };
        for (long long i = d / 2 - 1; i >= 0; --i) sift(i, d);
        for (long long i = d - 1; i > 0; --i) {
            const unsigned long long top = a[0];
            a[0] = a[i];
            a[i] = top;
            sift(0, i);
        }
    }
    for (long long i = 0; i < d; ++i) {
        const unsigned long long k = a[i], f = k / 3;
        const unsigned c = (unsigned)(k - 3 * f);
        const unsigned ra = (unsigned)faces[3 * f + (c + 1) % 3] | (c & 1u) << 31;
        const unsigned rb = (unsigned)faces[3 * f + (c + 2) % 3] | (c >> 1) << 31;
        a[i] = (unsigned long long)ra | (unsigned long long)rb << 32;
    }
}

// One umbrella half-step, Jacobi: out[v] = p[v] + w (m - p[v]), m = (sum over v's corners of p[a] + p[b]) / (2k), every
// operation rounded separately (no FMA).  A vertex without corners keeps its position.
__global__ void __launch_bounds__(kThreads) smooth_kernel(const float* __restrict__ p, unsigned n_verts,
                                                          const unsigned long long* __restrict__ ends, const int2* __restrict__ adj,
                                                          float w, float* __restrict__ out) {
    const unsigned v = blockIdx.x * kThreads + threadIdx.x;
    if (v >= n_verts) return;
    const unsigned long long beg = adj_begin(ends, v), end = ends[v];
    const float* pv = p + 3 * (size_t)v;
    float* o = out + 3 * (size_t)v;
    if (beg == end) {
#pragma unroll
        for (int c = 0; c < 3; ++c) o[c] = pv[c];
        return;
    }
    float s[3] = {0.f, 0.f, 0.f};
    for (unsigned long long i = beg; i < end; ++i) {
        const int2 r = adj[i];
        const float* pa = p + 3 * (size_t)rec_a(r);
        const float* pb = p + 3 * (size_t)rec_b(r);
#pragma unroll
        for (int c = 0; c < 3; ++c) s[c] = __fadd_rn(__fadd_rn(s[c], pa[c]), pb[c]);
    }
    const float k2 = __ull2float_rn(2 * (end - beg));
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const float x = pv[c];
        o[c] = __fadd_rn(x, __fmul_rn(w, __fsub_rn(__fdiv_rn(s[c], k2), x)));
    }
}

// Area-weighted vertex normals: the sum over v's corners of the face normal (p[f1] - p[f0]) x (p[f2] - p[f0]) in the face's
// own corner order, divided by its length like mc_normals_kernel; (0, 0, 0) when the length is 0.
__global__ void __launch_bounds__(kThreads) mesh_normals_kernel(const float* __restrict__ p, unsigned n_verts,
                                                                const unsigned long long* __restrict__ ends,
                                                                const int2* __restrict__ adj, float* __restrict__ normals) {
    const unsigned v = blockIdx.x * kThreads + threadIdx.x;
    if (v >= n_verts) return;
    const unsigned long long end = ends[v];
    float n[3] = {0.f, 0.f, 0.f};
    for (unsigned long long i = adj_begin(ends, v); i < end; ++i) {
        unsigned f[3];
        rec_face(adj[i], v, f);
        const float* p0 = p + 3 * (size_t)f[0];
        const float* p1 = p + 3 * (size_t)f[1];
        const float* p2 = p + 3 * (size_t)f[2];
        float e1[3], e2[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            e1[k] = __fsub_rn(p1[k], p0[k]);
            e2[k] = __fsub_rn(p2[k], p0[k]);
        }
#pragma unroll
        for (int k = 0; k < 3; ++k) {
            const int k1 = (k + 1) % 3, k2 = (k + 2) % 3;
            n[k] = __fadd_rn(n[k], __fsub_rn(__fmul_rn(e1[k1], e2[k2]), __fmul_rn(e1[k2], e2[k1])));
        }
    }
    const float len = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(n[0], n[0]), __fmul_rn(n[1], n[1])), __fmul_rn(n[2], n[2])));
    float* o = normals + 3 * (size_t)v;
#pragma unroll
    for (int k = 0; k < 3; ++k) o[k] = len > 0.f ? __fdiv_rn(n[k], len) : 0.f;
}

// ---- quadric edge collapse (b2r_mesh_quadrics / _decimate_round / _decimate_compact) ------------------------------------------
// The rules are oracle/mesh_decimation.py's.  One round over the adjacency of the current faces: dec_flags_kernel marks frozen
// vertices and counts distinct neighbours; dec_key_kernel gives every vertex the smallest key (cost, a, b) of its valid edges and
// that edge's placement; dec_min_kernel takes the smallest key over each closed neighbourhood; dec_select_kernel keeps an edge
// iff both ends agree with its key and with both minima.  Compaction (mark_kernel, compact_kernel with DecKeep / DecEmit) writes
// the surviving vertices and faces in order.  One thread per vertex and plain loads of the neighbours' keys: the result does not
// depend on the schedule, and the float64 / float32 values are formed with separately rounded intrinsics.  An edge's key is the
// ulonglong2 (float64 bits of the cost, a << 32 | b); the cost is >= 0, so comparing (x, y) as unsigned integers is the
// lexicographic order.
// Scratch: info[V] (bit 31 frozen, low bits the valence), key[V], m[V] (ulonglong2), part[V] (the partner of a selected vertex or
// -1), place[V,3] (the placement of the vertex's key edge), then the compaction tail, whose last 256 bytes hold the totals.
struct DecLayout {
    size_t info, key, m, part, place;
    CompactTail tail;
};

inline DecLayout dec_layout(long long n_verts, long long n_faces) {
    DecLayout l;
    l.info = 0;
    l.key = l.info + align256((size_t)n_verts * 4);
    l.m = l.key + align256((size_t)n_verts * 16);
    l.part = l.m + align256((size_t)n_verts * 16);
    l.place = l.part + align256((size_t)n_verts * 4);
    l.tail = compact_tail(l.place + align256((size_t)n_verts * 12), n_verts, n_faces);
    return l;
}

constexpr unsigned kFrozen = 1u << 31;
constexpr unsigned long long kNoKey = ~0ull;
constexpr long long kNotSelected = 0x7fffffffffffffffll;

__device__ __forceinline__ bool key_less(ulonglong2 x, ulonglong2 y) { return x.x < y.x || (x.x == y.x && x.y < y.y); }
__device__ __forceinline__ bool key_eq(ulonglong2 x, ulonglong2 y) { return x.x == y.x && x.y == y.y; }

// Slot s of v's neighbour list: the a (even s) or b (odd s) of record s / 2.
__device__ __forceinline__ unsigned nb_slot(const int2* __restrict__ adj, unsigned long long beg, unsigned long long s) {
    const int2 r = adj[beg + s / 2];
    return s & 1 ? rec_b(r) : rec_a(r);
}

// Whether slot s holds the first occurrence of its vertex in the list.
__device__ __forceinline__ bool nb_first(const int2* __restrict__ adj, unsigned long long beg, unsigned long long s, unsigned u) {
    for (unsigned long long t = 0; t < s; ++t)
        if (nb_slot(adj, beg, t) == u) return false;
    return true;
}

__device__ __forceinline__ bool nb_has(const int2* __restrict__ adj, unsigned long long beg, unsigned long long end, unsigned u) {
    for (unsigned long long i = beg; i < end; ++i) {
        const int2 r = adj[i];
        if (rec_a(r) == u || rec_b(r) == u) return true;
    }
    return false;
}

__device__ __forceinline__ void cross64(const double (&e1)[3], const double (&e2)[3], double (&n)[3]) {
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        const int k1 = (k + 1) % 3, k2 = (k + 2) % 3;
        n[k] = __dsub_rn(__dmul_rn(e1[k1], e2[k2]), __dmul_rn(e1[k2], e2[k1]));
    }
}

__device__ __forceinline__ double dot64(const double (&n)[3], const double (&m)[3]) {
    return __dadd_rn(__dadd_rn(__dmul_rn(n[0], m[0]), __dmul_rn(n[1], m[1])), __dmul_rn(n[2], m[2]));
}

// (p1 - p0) x (p2 - p0) in float64 of three float32 points.
__device__ __forceinline__ void face_normal64(const float* p0, const float* p1, const float* p2, double (&n)[3]) {
    double e1[3], e2[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
        e1[k] = __dsub_rn((double)p1[k], (double)p0[k]);
        e2[k] = __dsub_rn((double)p2[k], (double)p0[k]);
    }
    cross64(e1, e2, n);
}

// Sum over v's corners in order of their faces' area-weighted plane quadrics.
__global__ void __launch_bounds__(kThreads) dec_quadric_kernel(const float* __restrict__ p, unsigned n_verts,
                                                               const unsigned long long* __restrict__ ends,
                                                               const int2* __restrict__ adj, double* __restrict__ q) {
    const unsigned v = blockIdx.x * kThreads + threadIdx.x;
    if (v >= n_verts) return;
    const unsigned long long end = ends[v];
    double s[10];
#pragma unroll
    for (int i = 0; i < 10; ++i) s[i] = 0.0;
    for (unsigned long long i = adj_begin(ends, v); i < end; ++i) {
        unsigned f[3];
        rec_face(adj[i], v, f);
        const float* p0 = p + 3 * (size_t)f[0];
        double n[3];
        face_normal64(p0, p + 3 * (size_t)f[1], p + 3 * (size_t)f[2], n);
        const double len = __dsqrt_rn(dot64(n, n));
        if (!(len > 0.0)) continue;                                // adds zeros
        double e[4];
#pragma unroll
        for (int k = 0; k < 3; ++k) e[k] = __ddiv_rn(n[k], len);
        e[3] = -__dadd_rn(__dadd_rn(__dmul_rn(e[0], (double)p0[0]), __dmul_rn(e[1], (double)p0[1])), __dmul_rn(e[2], (double)p0[2]));
        const double w = __dmul_rn(len, 0.5);
        int k = 0;
#pragma unroll
        for (int r = 0; r < 4; ++r)
#pragma unroll
            for (int c = r; c < 4; ++c, ++k) s[k] = __dadd_rn(s[k], __dmul_rn(w, __dmul_rn(e[r], e[c])));
    }
    double* o = q + 10 * (size_t)v;
#pragma unroll
    for (int i = 0; i < 10; ++i) o[i] = s[i];
}

// Frozen (listed twice by a face, or an edge on other than two faces) and the number of distinct neighbours.
__global__ void __launch_bounds__(kThreads) dec_flags_kernel(unsigned n_verts, const unsigned long long* __restrict__ ends,
                                                             const int2* __restrict__ adj, unsigned* __restrict__ info) {
    const unsigned v = blockIdx.x * kThreads + threadIdx.x;
    if (v >= n_verts) return;
    const unsigned long long beg = adj_begin(ends, v), end = ends[v];
    unsigned frozen = 0, valence = 0;
    for (unsigned long long i = beg; i < end; ++i) {
        const int2 r = adj[i];
        if (rec_a(r) == v || rec_b(r) == v) frozen = kFrozen;
    }
    for (unsigned long long s = 0; s < 2 * (end - beg); ++s) {
        const unsigned u = nb_slot(adj, beg, s);
        if (u == v || !nb_first(adj, beg, s, u)) continue;
        ++valence;
        unsigned faces = 0;
        for (unsigned long long i = beg; i < end; ++i) {
            const int2 r = adj[i];
            faces += rec_a(r) == u || rec_b(r) == u;
        }
        if (faces != 2) frozen = kFrozen;
    }
    info[v] = frozen | valence;
}

// c(p) = p^T Q p over homogeneous p, as the oracle's fixed expression, clamped to 0 when not > 0.
__device__ __forceinline__ double quadric_cost(const double (&q)[10], const float* x) {
    const double X = x[0], Y = x[1], Z = x[2];
    constexpr int idx[4][4] = {{0, 1, 2, 3}, {1, 4, 5, 6}, {2, 5, 7, 8}, {3, 6, 8, 9}};
    double r[4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
        r[i] = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(q[idx[i][0]], X), __dmul_rn(q[idx[i][1]], Y)), __dmul_rn(q[idx[i][2]], Z)),
                         q[idx[i][3]]);
    const double c = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(r[0], X), __dmul_rn(r[1], Y)), __dmul_rn(r[2], Z)), r[3]);
    return c > 0.0 ? c : 0.0;
}

// Whether every face around x that does not hold y keeps dot(n_before, n_after) > 0 with x moved to pos.
__device__ bool dec_no_flip(const float* __restrict__ p, const unsigned long long* __restrict__ ends, const int2* __restrict__ adj,
                            unsigned x, unsigned y, const float (&pos)[3]) {
    const unsigned long long end = ends[x];
    for (unsigned long long i = adj_begin(ends, x); i < end; ++i) {
        const int2 r = adj[i];
        if (rec_a(r) == y || rec_b(r) == y) continue;
        unsigned f[3];
        rec_face(r, x, f);
        const float* q0 = p + 3 * (size_t)f[0];
        const float* q1 = p + 3 * (size_t)f[1];
        const float* q2 = p + 3 * (size_t)f[2];
        double nb[3], na[3];
        face_normal64(q0, q1, q2, nb);
        face_normal64(f[0] == x ? pos : q0, f[1] == x ? pos : q1, f[2] == x ? pos : q2, na);
        if (!(dot64(nb, na) > 0.0)) return false;
    }
    return true;
}

__global__ void __launch_bounds__(kThreads) dec_key_kernel(const float* __restrict__ p, const double* __restrict__ q, unsigned n_verts,
                                                           const unsigned long long* __restrict__ ends, const int2* __restrict__ adj,
                                                           const unsigned* __restrict__ info, ulonglong2* __restrict__ key,
                                                           float* __restrict__ place) {
    const unsigned v = blockIdx.x * kThreads + threadIdx.x;
    if (v >= n_verts) return;
    const unsigned iv = info[v];
    ulonglong2 best = make_ulonglong2(kNoKey, kNoKey);
    float best_p[3] = {0.f, 0.f, 0.f};
    const unsigned long long beg = adj_begin(ends, v), end = ends[v];
    if (!(iv & kFrozen)) {
        for (unsigned long long s = 0; s < 2 * (end - beg); ++s) {
            const unsigned u = nb_slot(adj, beg, s);
            if (!nb_first(adj, beg, s, u)) continue;
            const unsigned iu = info[u];
            if ((iu & kFrozen) || (iv & ~kFrozen) + (iu & ~kFrozen) < 7) continue;
            const unsigned a = min(u, v), b = max(u, v);
            double qs[10];
#pragma unroll
            for (int i = 0; i < 10; ++i) qs[i] = __dadd_rn(q[10 * (size_t)a + i], q[10 * (size_t)b + i]);
            const float* pa = p + 3 * (size_t)a;
            const float* pb = p + 3 * (size_t)b;
            float mid[3], pos[3];
#pragma unroll
            for (int k = 0; k < 3; ++k) mid[k] = __fmul_rn(__fadd_rn(pa[k], pb[k]), 0.5f);
            double c = quadric_cost(qs, pa);
            const float* pick = pa;
            const double cb = quadric_cost(qs, pb);
            if (cb < c) { c = cb; pick = pb; }
            const double cm = quadric_cost(qs, mid);
            if (cm < c) { c = cm; pick = mid; }
            const ulonglong2 k = make_ulonglong2((unsigned long long)__double_as_longlong(c), (unsigned long long)a << 32 | b);
            if (!key_less(k, best)) continue;                      // cannot lower key(v): its validity does not matter
            // link condition: the opposite vertices of the edge's two faces differ, and they are the only common neighbours
            unsigned o[2] = {~0u, ~0u}, no = 0;
            for (unsigned long long i = beg; i < end; ++i) {
                const int2 r = adj[i];
                if (rec_a(r) == u) o[no++ & 1] = rec_b(r);
                else if (rec_b(r) == u) o[no++ & 1] = rec_a(r);
            }
            if (o[0] == o[1]) continue;
            const unsigned long long ub = adj_begin(ends, u), ue = ends[u];
            unsigned common = 0;
            for (unsigned long long t = 0; t < 2 * (end - beg) && common <= 2; ++t) {
                const unsigned w = nb_slot(adj, beg, t);
                if (w != u && nb_first(adj, beg, t, w) && nb_has(adj, ub, ue, w)) ++common;
            }
            if (common != 2) continue;
#pragma unroll
            for (int i = 0; i < 3; ++i) pos[i] = pick[i];
            if (!dec_no_flip(p, ends, adj, a, b, pos) || !dec_no_flip(p, ends, adj, b, a, pos)) continue;
            best = k;
#pragma unroll
            for (int i = 0; i < 3; ++i) best_p[i] = pos[i];
        }
    }
    key[v] = best;
#pragma unroll
    for (int i = 0; i < 3; ++i) place[3 * (size_t)v + i] = best_p[i];
}

__global__ void __launch_bounds__(kThreads) dec_min_kernel(unsigned n_verts, const unsigned long long* __restrict__ ends,
                                                           const int2* __restrict__ adj, const ulonglong2* __restrict__ key,
                                                           ulonglong2* __restrict__ m) {
    const unsigned v = blockIdx.x * kThreads + threadIdx.x;
    if (v >= n_verts) return;
    ulonglong2 best = key[v];
    const unsigned long long end = ends[v];
    for (unsigned long long i = adj_begin(ends, v); i < end; ++i) {
        const int2 r = adj[i];
        const ulonglong2 ka = key[rec_a(r)], kb = key[rec_b(r)];
        if (key_less(ka, best)) best = ka;
        if (key_less(kb, best)) best = kb;
    }
    m[v] = best;
}

// part[v] = the other end of v's selected edge, or -1; sel_keys[a] = the cost bits of a selected edge at its survivor a, kNotSelected
// everywhere else; *count += the selected edges (warp-aggregated).
__global__ void __launch_bounds__(kThreads) dec_select_kernel(unsigned n_verts, const ulonglong2* __restrict__ key,
                                                              const ulonglong2* __restrict__ m, int* __restrict__ part,
                                                              long long* __restrict__ sel_keys, long long* __restrict__ count) {
    const unsigned v = blockIdx.x * kThreads + threadIdx.x;
    bool survivor = false;
    if (v < n_verts) {
        const ulonglong2 k = key[v];
        int partner = -1;
        if (k.x != kNoKey && key_eq(m[v], k)) {
            const unsigned a = (unsigned)(k.y >> 32), b = (unsigned)k.y;
            const unsigned u = v == a ? b : a;
            if (key_eq(key[u], k) && key_eq(m[u], k)) partner = (int)u;
        }
        part[v] = partner;
        survivor = partner > (int)v;
        sel_keys[v] = survivor ? (long long)k.x : kNotSelected;
    }
    const unsigned votes = __ballot_sync(kFull, survivor);
    if ((threadIdx.x & (kWarp - 1)) == 0 && votes) atomicAdd((unsigned long long*)count, (unsigned long long)__popc(votes));
}

__global__ void dec_count_kernel(long long n_faces, long long* __restrict__ counts) { counts[1] = n_faces - 2 * counts[0]; }

// Whether the selected edge at survivor a collapses: every selected edge, or with a cut (cost bits, a) the ones up to it.
__device__ __forceinline__ bool dec_kept(const int* __restrict__ part, const long long* __restrict__ sel_keys,
                                         const long long* __restrict__ cut, unsigned a) {
    if (__ldg(part + a) <= (int)a) return false;
    if (!cut) return true;
    const long long k = __ldg(sel_keys + a), c0 = __ldg(cut);
    return k < c0 || (k == c0 && (long long)a <= __ldg(cut + 1));
}

// The survivor vertex u collapses into, or u itself.
__device__ __forceinline__ unsigned dec_target(const int* __restrict__ part, const long long* __restrict__ sel_keys,
                                               const long long* __restrict__ cut, unsigned u) {
    const int t = __ldg(part + u);
    return t >= 0 && t < (int)u && dec_kept(part, sel_keys, cut, (unsigned)t) ? (unsigned)t : u;
}

// A face with indices t is deleted iff it holds both ends of a collapsing edge.
__device__ __forceinline__ bool dec_face_dies(const unsigned (&t)[3], const int* __restrict__ part, const long long* __restrict__ sel_keys,
                                              const long long* __restrict__ cut) {
    bool dies = false;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const unsigned g = dec_target(part, sel_keys, cut, t[c]);
        dies |= g != t[c] && (g == t[(c + 1) % 3] || g == t[(c + 2) % 3]);
    }
    return dies;
}

// A vertex survives iff it does not collapse into another; a face iff it does not hold both ends of a collapsing edge.
struct DecKeep {
    const int* faces;
    const int* part;
    const long long* sel_keys;
    const long long* cut;
    __device__ bool vert(unsigned v) const { return dec_target(part, sel_keys, cut, v) == v; }
    __device__ bool face(unsigned f) const {
        unsigned t[3];
#pragma unroll
        for (int c = 0; c < 3; ++c) t[c] = (unsigned)__ldg(faces + 3 * (size_t)f + c);
        return !dec_face_dies(t, part, sel_keys, cut);
    }
};

// A collapsing survivor moves to its placement with Q_a + Q_b, any other survivor keeps its position and Q; face indices map
// through the collapses.
struct DecEmit {
    const float* verts;
    const double* q;
    const int* part;
    const long long* sel_keys;
    const long long* cut;
    const float* place;
    float* verts_out;
    double* q_out;
    __device__ void vert(unsigned v, size_t to) const {
        const bool moves = dec_kept(part, sel_keys, cut, v);
        const float* from = (moves ? place : verts) + 3 * (size_t)v;
#pragma unroll
        for (int c = 0; c < 3; ++c) verts_out[3 * to + c] = __ldg(from + c);
        const double* qa = q + 10 * (size_t)v;
        const double* qb = q + 10 * (size_t)(moves ? __ldg(part + v) : 0);
#pragma unroll
        for (int i = 0; i < 10; ++i) q_out[10 * to + i] = moves ? __dadd_rn(__ldg(qa + i), __ldg(qb + i)) : __ldg(qa + i);
    }
    __device__ bool face(unsigned, const unsigned (&t)[3]) const { return !dec_face_dies(t, part, sel_keys, cut); }
    __device__ unsigned target(unsigned u) const { return dec_target(part, sel_keys, cut, u); }
};

int check_grid(const char* what, int n0, int n1, int n2) {
    B2R_CHECK_ARG(n0 >= 2 && n1 >= 2 && n2 >= 2, "%s: every axis needs n >= 2 (got %d x %d x %d)", what, n0, n1, n2);
    B2R_CHECK_ARG((long long)n0 * n1 * n2 <= INT32_MAX, "%s: n0*n1*n2 = %lld exceeds INT32_MAX", what, (long long)n0 * n1 * n2);
    return 0;
}

// mark_kernel, then mc_scan_kernel over its tile counts: vword, every tile's (first vertex, first face) and the totals (V', F').
template <class Keep>
static void mark_and_scan(Keep keep, long long n_faces, long long n_verts, char* s, const CompactTail& t, long long* totals,
                          cudaStream_t st) {
    const int tiles = (int)compact_tiles(n_verts, n_faces);
    if (tiles)
        mark_kernel<<<tiles, kThreads, 0, st>>>(keep, (unsigned)n_faces, (unsigned)n_verts, (unsigned*)(s + t.vword),
                                                (unsigned*)(s + t.counts));
    mc_scan_kernel<<<1, kScanThreads, 0, st>>>((const unsigned*)(s + t.counts), tiles, (longlong2*)(s + t.offsets), totals);
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

namespace {

int check_counts(const char* what, long long n_faces, long long n_verts) {
    B2R_CHECK_ARG(n_faces >= 0 && n_faces <= INT32_MAX, "%s: n_faces = %lld must be in [0, INT32_MAX]", what, n_faces);
    B2R_CHECK_ARG(n_verts >= 0 && n_verts <= INT32_MAX, "%s: n_verts = %lld must be in [0, INT32_MAX]", what, n_verts);
    return 0;
}

int check_scratch(const char* what, const void* scratch) {
    B2R_CHECK_ARG(scratch, "%s: NULL scratch", what);
    B2R_CHECK_ARG(((uintptr_t)scratch & 15) == 0, "%s: scratch must be 16-byte aligned", what);
    return 0;
}

unsigned blocks_of(long long n, int threads) { return (unsigned)((n + threads - 1) / threads); }

constexpr unsigned kMaxBlocks = 8 * 148;      // cc_max_kernel: grid-stride, a few CTAs per SM, one atomic per CTA

}  // namespace

extern "C" size_t b2r_mesh_cc_scratch_bytes(long long n_verts, long long n_faces) {
    if (n_verts < 0 || n_verts > INT32_MAX || n_faces < 0 || n_faces > INT32_MAX) return 0;
    return b2r::mc::cc_layout(n_verts, n_faces).tail.total;
}

extern "C" int b2r_mesh_cc_label(const int* faces, long long n_faces, long long n_verts, int* labels, void* scratch, void* stream) {
    using namespace b2r::mc;
    const char* what = "b2r_mesh_cc_label";
    if (int rc = check_counts(what, n_faces, n_verts)) return rc;
    B2R_CHECK_ARG((faces || !n_faces) && (labels || !n_verts), "%s: NULL pointer (faces and labels may be NULL only when their count is 0)",
                  what);
    if (int rc = check_scratch(what, scratch)) return rc;
    if (!n_verts) return 0;
    unsigned* parent = (unsigned*)((char*)scratch + cc_layout(n_verts, n_faces).a);
    cudaStream_t st = (cudaStream_t)stream;
    cc_init_kernel<<<blocks_of(n_verts, kThreads), kThreads, 0, st>>>(parent, (unsigned)n_verts);
    if (n_faces) cc_hook_kernel<<<blocks_of(n_faces, kThreads), kThreads, 0, st>>>(faces, (unsigned)n_faces, parent);
    cc_labels_kernel<<<blocks_of(n_verts, kThreads), kThreads, 0, st>>>(parent, (unsigned)n_verts, labels);
    B2R_LAUNCH_CHECK(what);
    return 0;
}

extern "C" int b2r_mesh_cc_select(const int* faces, long long n_faces, long long n_verts, const int* labels, float ratio, void* scratch,
                                  long long* totals_dev, void* stream) {
    using namespace b2r::mc;
    const char* what = "b2r_mesh_cc_select";
    if (int rc = check_counts(what, n_faces, n_verts)) return rc;
    B2R_CHECK_ARG((faces || !n_faces) && (labels || !n_verts) && totals_dev,
                  "%s: NULL pointer (faces and labels may be NULL only when their count is 0)", what);
    B2R_CHECK_ARG(std::isfinite(ratio) && ratio >= 0.f && ratio <= 1.f, "%s: ratio = %g must be finite and in [0, 1]", what, (double)ratio);
    if (int rc = check_scratch(what, scratch)) return rc;
    const CcLayout l = cc_layout(n_verts, n_faces);
    char* s = static_cast<char*>(scratch);
    unsigned* tri = (unsigned*)(s + l.a);
    unsigned* t_max = (unsigned*)(s + l.tail.last);
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = b2r::cuda_result(cudaMemsetAsync(tri, 0, (size_t)n_verts * 4, st), what)) return rc;
    if (int rc = b2r::cuda_result(cudaMemsetAsync(t_max, 0, 4, st), what)) return rc;
    if (n_faces) cc_count_kernel<<<blocks_of(n_faces, kThreads), kThreads, 0, st>>>(faces, (unsigned)n_faces, labels, tri);
    if (n_verts) {
        const unsigned blocks = blocks_of(n_verts, kThreads);
        cc_max_kernel<<<blocks < kMaxBlocks ? blocks : kMaxBlocks, kThreads, 0, st>>>(tri, (unsigned)n_verts, t_max);
    }
    mark_and_scan(CcKeep{faces, labels, tri, t_max, ratio}, n_faces, n_verts, s, l.tail, totals_dev, st);
    B2R_LAUNCH_CHECK(what);
    return 0;
}

extern "C" int b2r_mesh_cc_compact(const float* verts, const float* normals_or_null, const int* faces, long long n_faces, long long n_verts,
                                   const void* scratch, float* verts_out, float* normals_out, int* faces_out, void* stream) {
    using namespace b2r::mc;
    const char* what = "b2r_mesh_cc_compact";
    if (int rc = check_counts(what, n_faces, n_verts)) return rc;
    B2R_CHECK_ARG((faces && faces_out) || !n_faces, "%s: NULL faces / faces_out with n_faces > 0", what);
    B2R_CHECK_ARG((verts && verts_out && (!normals_or_null || normals_out)) || !n_verts,
                  "%s: NULL verts / verts_out, or normals given and NULL normals_out, with n_verts > 0", what);
    if (int rc = check_scratch(what, scratch)) return rc;
    const CompactTail t = cc_layout(n_verts, n_faces).tail;
    const int tiles = (int)compact_tiles(n_verts, n_faces);
    if (!tiles) return 0;
    const char* s = static_cast<const char*>(scratch);
    const unsigned* vword = (const unsigned*)(s + t.vword);
    compact_kernel<<<tiles, kThreads, 0, (cudaStream_t)stream>>>(CcEmit{verts, normals_or_null, vword, verts_out, normals_out}, faces,
                                                                 (unsigned)n_faces, (unsigned)n_verts, vword,
                                                                 (const longlong2*)(s + t.offsets), faces_out);
    B2R_LAUNCH_CHECK(what);
    return 0;
}

extern "C" size_t b2r_mesh_adj_scratch_bytes(long long n_verts, long long n_faces) {
    if (n_verts < 0 || n_verts > INT32_MAX || n_faces < 0 || n_faces > INT32_MAX) return 0;
    return b2r::mc::adj_layout(n_verts, n_faces).total;
}

extern "C" int b2r_mesh_adjacency(const int* faces, long long n_faces, long long n_verts, void* scratch, void* stream) {
    using namespace b2r::mc;
    const char* what = "b2r_mesh_adjacency";
    if (int rc = check_counts(what, n_faces, n_verts)) return rc;
    B2R_CHECK_ARG(faces || !n_faces, "%s: NULL faces with n_faces > 0", what);
    if (!n_verts) return 0;                  // an empty mesh has a 0-byte scratch, which may be NULL
    if (int rc = check_scratch(what, scratch)) return rc;
    const AdjLayout l = adj_layout(n_verts, n_faces);
    const int tiles = (int)((n_verts + kTile - 1) / kTile);
    char* s = static_cast<char*>(scratch);
    unsigned long long* ends = (unsigned long long*)(s + l.ends);
    unsigned long long* tile_sums = (unsigned long long*)(s + l.tile_sums);
    unsigned long long* keys = (unsigned long long*)(s + l.adj);
    const unsigned nv = (unsigned)n_verts, nf = (unsigned)n_faces;
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = b2r::cuda_result(cudaMemsetAsync(ends, 0, (size_t)n_verts * 8, st), what)) return rc;
    if (nf) adj_count_kernel<<<blocks_of(nf, kThreads), kThreads, 0, st>>>(faces, nf, ends);
    adj_tile_sum_kernel<<<tiles, kThreads, 0, st>>>(ends, nv, tile_sums);
    adj_scan_tiles_kernel<<<1, kScanThreads, 0, st>>>(tile_sums, tiles);
    adj_tile_scan_kernel<<<tiles, kThreads, 0, st>>>(ends, nv, tile_sums);
    if (nf) {
        adj_fill_kernel<<<blocks_of(nf, kThreads), kThreads, 0, st>>>(faces, nf, ends, keys);
        adj_sort_kernel<<<blocks_of(nv, kThreads), kThreads, 0, st>>>(faces, nv, ends, keys);
    }
    B2R_LAUNCH_CHECK(what);
    return 0;
}

extern "C" int b2r_mesh_smooth(const float* verts, long long n_faces, long long n_verts, int iterations, void* scratch, float* verts_out,
                               void* stream) {
    using namespace b2r::mc;
    const char* what = "b2r_mesh_smooth";
    if (int rc = check_counts(what, n_faces, n_verts)) return rc;
    B2R_CHECK_ARG((verts && verts_out) || !n_verts, "%s: NULL verts / verts_out with n_verts > 0", what);
    B2R_CHECK_ARG(iterations >= 0, "%s: iterations = %d must be >= 0", what, iterations);
    if (!n_verts) return 0;                  // an empty mesh has a 0-byte scratch, which may be NULL
    if (int rc = check_scratch(what, scratch)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    if (!iterations) {
        if (verts == verts_out) return 0;
        return b2r::cuda_result(cudaMemcpyAsync(verts_out, verts, (size_t)n_verts * 12, cudaMemcpyDeviceToDevice, st), what);
    }
    const AdjLayout l = adj_layout(n_verts, n_faces);
    char* s = static_cast<char*>(scratch);
    const unsigned long long* ends = (const unsigned long long*)(s + l.ends);
    const int2* adj = (const int2*)(s + l.adj);
    float* tmp = (float*)(s + l.pos);
    const unsigned nv = (unsigned)n_verts, blocks = blocks_of(nv, kThreads);
    for (int it = 0; it < iterations; ++it) {
        smooth_kernel<<<blocks, kThreads, 0, st>>>(it ? verts_out : verts, nv, ends, adj, kTaubinLambda, tmp);
        smooth_kernel<<<blocks, kThreads, 0, st>>>(tmp, nv, ends, adj, kTaubinMu, verts_out);
    }
    B2R_LAUNCH_CHECK(what);
    return 0;
}

extern "C" int b2r_mesh_normals(const float* verts, long long n_faces, long long n_verts, const void* scratch, float* normals,
                                void* stream) {
    using namespace b2r::mc;
    const char* what = "b2r_mesh_normals";
    if (int rc = check_counts(what, n_faces, n_verts)) return rc;
    B2R_CHECK_ARG((verts && normals) || !n_verts, "%s: NULL verts / normals with n_verts > 0", what);
    if (!n_verts) return 0;                  // an empty mesh has a 0-byte scratch, which may be NULL
    if (int rc = check_scratch(what, scratch)) return rc;
    const AdjLayout l = adj_layout(n_verts, n_faces);
    const char* s = static_cast<const char*>(scratch);
    mesh_normals_kernel<<<blocks_of(n_verts, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
        verts, (unsigned)n_verts, (const unsigned long long*)(s + l.ends), (const int2*)(s + l.adj), normals);
    B2R_LAUNCH_CHECK(what);
    return 0;
}

extern "C" size_t b2r_mesh_decimate_scratch_bytes(long long n_verts, long long n_faces) {
    if (n_verts < 0 || n_verts > INT32_MAX || n_faces < 0 || n_faces > INT32_MAX) return 0;
    return b2r::mc::dec_layout(n_verts, n_faces).tail.total;
}

extern "C" int b2r_mesh_quadrics(const float* verts, long long n_faces, long long n_verts, const void* adj_scratch, double* quadrics,
                                 void* stream) {
    using namespace b2r::mc;
    const char* what = "b2r_mesh_quadrics";
    if (int rc = check_counts(what, n_faces, n_verts)) return rc;
    B2R_CHECK_ARG((verts && quadrics) || !n_verts, "%s: NULL verts / quadrics with n_verts > 0", what);
    if (!n_verts) return 0;
    if (int rc = check_scratch(what, adj_scratch)) return rc;
    const AdjLayout l = adj_layout(n_verts, n_faces);
    const char* s = static_cast<const char*>(adj_scratch);
    dec_quadric_kernel<<<blocks_of(n_verts, kThreads), kThreads, 0, (cudaStream_t)stream>>>(
        verts, (unsigned)n_verts, (const unsigned long long*)(s + l.ends), (const int2*)(s + l.adj), quadrics);
    B2R_LAUNCH_CHECK(what);
    return 0;
}

extern "C" int b2r_mesh_decimate_round(const float* verts, const double* quadrics, long long n_faces, long long n_verts,
                                       const void* adj_scratch, void* scratch, long long* sel_keys, long long* counts_dev,
                                       void* stream) {
    using namespace b2r::mc;
    const char* what = "b2r_mesh_decimate_round";
    if (int rc = check_counts(what, n_faces, n_verts)) return rc;
    B2R_CHECK_ARG(counts_dev, "%s: NULL counts_dev", what);
    B2R_CHECK_ARG((verts && quadrics && sel_keys) || !n_verts, "%s: NULL verts / quadrics / sel_keys with n_verts > 0", what);
    cudaStream_t st = (cudaStream_t)stream;
    if (int rc = b2r::cuda_result(cudaMemsetAsync(counts_dev, 0, 8, st), what)) return rc;
    if (n_verts) {
        if (int rc = check_scratch(what, adj_scratch)) return rc;
        if (int rc = check_scratch(what, scratch)) return rc;
        const AdjLayout al = adj_layout(n_verts, n_faces);
        const DecLayout l = dec_layout(n_verts, n_faces);
        const char* a = static_cast<const char*>(adj_scratch);
        char* s = static_cast<char*>(scratch);
        const unsigned long long* ends = (const unsigned long long*)(a + al.ends);
        const int2* adj = (const int2*)(a + al.adj);
        unsigned* info = (unsigned*)(s + l.info);
        ulonglong2* key = (ulonglong2*)(s + l.key);
        ulonglong2* m = (ulonglong2*)(s + l.m);
        const unsigned nv = (unsigned)n_verts, blocks = blocks_of(nv, kThreads);
        dec_flags_kernel<<<blocks, kThreads, 0, st>>>(nv, ends, adj, info);
        dec_key_kernel<<<blocks, kThreads, 0, st>>>(verts, quadrics, nv, ends, adj, info, key, (float*)(s + l.place));
        dec_min_kernel<<<blocks, kThreads, 0, st>>>(nv, ends, adj, key, m);
        dec_select_kernel<<<blocks, kThreads, 0, st>>>(nv, key, m, (int*)(s + l.part), sel_keys, counts_dev);
    }
    dec_count_kernel<<<1, 1, 0, st>>>(n_faces, counts_dev);
    B2R_LAUNCH_CHECK(what);
    return 0;
}

extern "C" int b2r_mesh_decimate_compact(const float* verts, const double* quadrics, const int* faces, long long n_faces,
                                         long long n_verts, const long long* sel_keys, const long long* cut_or_null, void* scratch,
                                         float* verts_out, double* quadrics_out, int* faces_out, void* stream) {
    using namespace b2r::mc;
    const char* what = "b2r_mesh_decimate_compact";
    if (int rc = check_counts(what, n_faces, n_verts)) return rc;
    B2R_CHECK_ARG((faces && faces_out) || !n_faces, "%s: NULL faces / faces_out with n_faces > 0", what);
    B2R_CHECK_ARG((verts && quadrics && sel_keys && verts_out && quadrics_out) || !n_verts,
                  "%s: NULL verts / quadrics / sel_keys / verts_out / quadrics_out with n_verts > 0", what);
    if (!n_verts) return 0;
    if (int rc = check_scratch(what, scratch)) return rc;
    const DecLayout l = dec_layout(n_verts, n_faces);
    const int tiles = (int)compact_tiles(n_verts, n_faces);
    char* s = static_cast<char*>(scratch);
    const int* part = (const int*)(s + l.part);
    cudaStream_t st = (cudaStream_t)stream;
    mark_and_scan(DecKeep{faces, part, sel_keys, cut_or_null}, n_faces, n_verts, s, l.tail, (long long*)(s + l.tail.last), st);
    compact_kernel<<<tiles, kThreads, 0, st>>>(
        DecEmit{verts, quadrics, part, sel_keys, cut_or_null, (const float*)(s + l.place), verts_out, quadrics_out}, faces,
        (unsigned)n_faces, (unsigned)n_verts, (const unsigned*)(s + l.tail.vword), (const longlong2*)(s + l.tail.offsets), faces_out);
    B2R_LAUNCH_CHECK(what);
    return 0;
}
