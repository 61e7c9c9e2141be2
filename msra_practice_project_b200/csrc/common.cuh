// Shared helpers for libb2r (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include "../../include/b2r.h"

namespace b2r {

// thread-local last-error text (b2r_last_error)
char* err_buf();
int fail(int code, const char* fmt, ...);

inline int cuda_result(cudaError_t e, const char* what) {
    if (e == cudaSuccess) return 0;
    return fail((int)e, "%s: %s", what, cudaGetErrorString(e));
}

#define B2R_CHECK_ARG(cond, ...)                         \
    do {                                                 \
        if (!(cond)) return ::b2r::fail(-1, __VA_ARGS__); \
    } while (0)

#define B2R_LAUNCH_CHECK(what)                                         \
    do {                                                               \
        int rc__ = ::b2r::cuda_result(cudaGetLastError(), what);       \
        if (rc__) return rc__;                                         \
    } while (0)

constexpr int kWarp = 32;
constexpr unsigned kFull = 0xffffffffu;

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// ---- flat parameter layout (state-dict order, weight then bias) -----------------------------
struct LayerDesc {
    int out, in;
    long long w_off, b_off;
};

// NeRF (nerf/nerf.py:56-73): layers_pos.0..7, layers_dir.0, layers_dir.1, sigma, rgb
constexpr int kNerfLayers = 12;
__host__ __device__ constexpr LayerDesc nerf_layer(int i) {
    constexpr int outs[kNerfLayers] = {256, 256, 256, 256, 256, 256, 256, 256, 256, 128, 1, 3};
    constexpr int ins[kNerfLayers] = {60, 256, 256, 256, 256, 316, 256, 256, 256, 280, 256, 128};
    long long off = 0;
    for (int k = 0; k < i; ++k) off += (long long)outs[k] * ins[k] + outs[k];
    return LayerDesc{outs[i], ins[i], off, off + (long long)outs[i] * ins[i]};
}
// FiLM-SIREN (pi_GAN/modules.py:73-94): input, hidden 0..6, sigma, hidden_rgb, rgb
constexpr int kFilmLayers = 11;
__host__ __device__ constexpr LayerDesc film_layer(int i, bool use_dir) {
    const int outs[kFilmLayers] = {256, 256, 256, 256, 256, 256, 256, 256, 1, 256, 3};
    const int ins[kFilmLayers] = {3, 256, 256, 256, 256, 256, 256, 256, 256, use_dir ? 259 : 256, 256};
    long long off = 0;
    for (int k = 0; k < i; ++k) off += (long long)outs[k] * ins[k] + outs[k];
    return LayerDesc{outs[i], ins[i], off, off + (long long)outs[i] * ins[i]};
}
// SirenNeRF (nerf/nerf.py:120-150): same topology as NeRF on raw 3-d inputs: layers_pos.0..7 (sin), layers_dir.0 (linear),
// layers_dir.1 (sin), sigma, rgb
constexpr int kSirenLayers = 12;
__host__ __device__ constexpr LayerDesc siren_layer(int i) {
    constexpr int outs[kSirenLayers] = {256, 256, 256, 256, 256, 256, 256, 256, 256, 128, 1, 3};
    constexpr int ins[kSirenLayers] = {3, 256, 256, 256, 256, 259, 256, 256, 256, 259, 256, 128};
    long long off = 0;
    for (int k = 0; k < i; ++k) off += (long long)outs[k] * ins[k] + outs[k];
    return LayerDesc{outs[i], ins[i], off, off + (long long)outs[i] * ins[i]};
}
static_assert(siren_layer(11).b_off + 3 == B2R_SIREN_NUMEL, "SirenNeRF flat layout");
static_assert(nerf_layer(11).b_off + 3 == B2R_NERF_NUMEL, "NeRF flat layout");
static_assert(film_layer(10, true).b_off + 3 == B2R_FILM_NUMEL, "FiLM flat layout");
static_assert(film_layer(10, false).b_off + 3 == B2R_FILM_NODIR_NUMEL, "FiLM (no dir) flat layout");

// ---- MLP input row -> (position, direction) --------------------------------------------------
struct RowSource {
    const float* rays;
    const float* z;
    const float* x;
    long long n_rays;
    int n_samples;
    // lattice rows: row r is lattice index lat_begin + r (axis 0 slowest) of the N^3 pi-GAN cube (grid_n > 0: origin -0.1) or of
    // the n0 x n1 x n2 box lattice at lat_origin
    long long lat_begin;
    int grid_n, lat_n1, lat_n2;
    float lat_origin[3];
    float voxel;
    // gather mode (b2r_mlp_f32_last_sigma): row i of the launch is the LAST sample of ray pick[i], i.e. source row
    // pick[i] * pick_s + pick_s - 1 of the rays / x description above
    const int* pick;
    int pick_s;
};

inline RowSource make_row_source(const b2r_mlp_input* in) {
    RowSource s = {};
    s.rays = in->rays; s.z = in->z; s.x = in->x; s.n_rays = in->n_rays; s.n_samples = in->n_samples;
    s.lat_begin = in->grid_begin;
    s.grid_n = in->grid_n;
    if (in->grid_n > 0) {
        s.voxel = in->grid_n > 1 ? (float)(0.2 / (double)(in->grid_n - 1)) : 0.f;   // 0.2/(N-1) rounded to float (pi_GAN/utils.py:57)
    } else {
        s.lat_n1 = in->lattice_dims[1]; s.lat_n2 = in->lattice_dims[2];
        for (int c = 0; c < 3; ++c) s.lat_origin[c] = in->lattice_origin[c];
        s.voxel = in->lattice_voxel;
    }
    s.pick = nullptr; s.pick_s = 0;
    return s;
}
inline bool lattice_mode(const b2r_mlp_input* in) {
    return in->lattice_dims[0] != 0 || in->lattice_dims[1] != 0 || in->lattice_dims[2] != 0;
}
inline long long row_count(const b2r_mlp_input* in) {
    return in->rays ? in->n_rays * (long long)in->n_samples : in->n_rays;
}
int check_mlp_input(const b2r_mlp_input* in);

// position = o + d*z as two rounded ops (torch: mul then add, nerf/render.py:134), unit view
// direction = d/|d| (render.py:122), lattice point = origin + index * voxel as two rounded ops (pi_GAN/utils.py:64-72).
// ray_out (optional): the ray the row belongs to (rays mode; the row itself otherwise).
// The pi-GAN cube keeps its own branch: its N^3 may pass 2^32 and needs 64-bit index arithmetic, while the box lattice has at most
// INT32_MAX points and uses 32-bit; one 64-bit path with per-axis divisors and origins costs the register-capped tensor-core
// kernels spills.  kBoxLattice = false compiles the box branch out: the tensor-core kernels have an instantiation for box-lattice
// rows and one for every other mode, so the other modes run the code they ran before the box lattice existed.
template <bool kBoxLattice = true>
__device__ __forceinline__ void load_row(const RowSource& s, long long row, float p[3], float v[3], long long* ray_out = nullptr) {
    if (s.pick) row = (long long)s.pick[row] * s.pick_s + (s.pick_s - 1);
    if (ray_out) *ray_out = row;
    if (s.rays) {
        long long r = row / s.n_samples;
        if (ray_out) *ray_out = r;
        const float* ray = s.rays + r * 6;
        float zz = s.z[row];
        float d0 = ray[3], d1 = ray[4], d2 = ray[5];
        p[0] = __fadd_rn(ray[0], __fmul_rn(d0, zz));
        p[1] = __fadd_rn(ray[1], __fmul_rn(d1, zz));
        p[2] = __fadd_rn(ray[2], __fmul_rn(d2, zz));
        float n = sqrtf(__fadd_rn(__fadd_rn(__fmul_rn(d0, d0), __fmul_rn(d1, d1)), __fmul_rn(d2, d2)));
        v[0] = d0 / n; v[1] = d1 / n; v[2] = d2 / n;
    } else if (s.x) {
        const float* x = s.x + row * 6;
        p[0] = x[0]; p[1] = x[1]; p[2] = x[2]; v[0] = x[3]; v[1] = x[4]; v[2] = x[5];
    } else {
        if (!kBoxLattice || s.grid_n) {
            const long long idx = s.lat_begin + row, n = s.grid_n;
            float iz = (float)(idx % n), iy = (float)((idx / n) % n), ix = (float)((idx / n / n) % n);
            p[0] = __fadd_rn(__fmul_rn(ix, s.voxel), -0.1f);
            p[1] = __fadd_rn(__fmul_rn(iy, s.voxel), -0.1f);
            p[2] = __fadd_rn(__fmul_rn(iz, s.voxel), -0.1f);
        } else {
            const unsigned idx = (unsigned)(s.lat_begin + row), n1 = (unsigned)s.lat_n1, n2 = (unsigned)s.lat_n2, r = idx / n2;
            float iz = (float)(idx % n2), iy = (float)(r % n1), ix = (float)(r / n1);
            p[0] = __fadd_rn(s.lat_origin[0], __fmul_rn(ix, s.voxel));
            p[1] = __fadd_rn(s.lat_origin[1], __fmul_rn(iy, s.voxel));
            p[2] = __fadd_rn(s.lat_origin[2], __fmul_rn(iz, s.voxel));
        }
        v[0] = v[1] = v[2] = 0.f;
    }
}

}  // namespace b2r
