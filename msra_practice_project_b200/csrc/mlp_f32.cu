// K3 (fp32 path): the radiance-field MLPs evaluated layer by layer in fp32 on CUDA cores, with
// every layer output kept so that the reverse mode (K8) can run.  This is the exact path: it is
// what the fp32 parity configuration (C1) and training (C3) use; the bf16 tensor-core path in
// mlp_tc.cu is the throughput path for rendering.
//   run_network            nerf/render.py:59-75
//   PositionalEncoding     nerf/nerf.py:44-49
//   NeRF.forward           nerf/nerf.py:75-94
//   FilmSiren / FilmSirenNeRF.forward   pi_GAN/modules.py:22-25, 101-118
//   backward               autograd in the reference (nerf/train_nerf.py:167, pi_GAN/train.py:134,
//                          pi_GAN/synthesis.py:107); formulas SURVEY.md A.5 / A.6
#include "sgemm.cuh"
#include "tgemm.cuh"

namespace b2r {

// ---- activation workspace layouts (floats per row) -------------------------------------------
// NeRF:  B5[316] = pe(60) || h4(256) | H0..H3[256] | H5,H6,H7[256] | B9[280] = g(256) || de(24) | HD[128]
struct NerfWs {
    static constexpr int kB5 = 316, kB9 = 280, kHD = 128, kH = 256;
    static constexpr int per_row = kB5 + 4 * kH + 3 * kH + kB9 + kHD;   // 2516
    float *B5, *H[8], *B9, *HD;   // H[4] aliases B5+60 (ld 316)
    long long ldH[8];
    NerfWs(float* base, long long rows) {
        float* p = base;
        B5 = p; p += rows * kB5;
        for (int l = 0; l < 4; ++l) { H[l] = p; ldH[l] = kH; p += rows * kH; }
        H[4] = B5 + 60; ldH[4] = kB5;
        for (int l = 5; l < 8; ++l) { H[l] = p; ldH[l] = kH; p += rows * kH; }
        B9 = p; p += rows * kB9;
        HD = p;
    }
};
// FiLM: X0[4] (pos) | A0..A7[256] (pre-FiLM linear outputs) | H0..H6[256] | B8[260] = h7(256) || dir(3) |
//       A8[256] | HC[256]
struct FilmWs {
    static constexpr int kX0 = 4, kB8 = 260, kH = 256;
    static constexpr int per_row = kX0 + 8 * kH + 7 * kH + kB8 + 2 * kH;   // 4616
    float *X0, *A[9], *H[8], *B8, *HC;
    long long ldH[8];
    FilmWs(float* base, long long rows) {
        float* p = base;
        X0 = p; p += rows * kX0;
        for (int l = 0; l < 8; ++l) { A[l] = p; p += rows * kH; }
        for (int l = 0; l < 7; ++l) { H[l] = p; ldH[l] = kH; p += rows * kH; }
        B8 = p; p += rows * kB8;
        H[7] = B8; ldH[7] = kB8;
        A[8] = p; p += rows * kH;
        HC = p;
    }
};

// SirenNeRF: X0[4] (pos) | A0..A7[256] (pre-sine linear outputs) | H0..H3[256] | B5[260] = pos(3) || h4(256) | H5, H6, H7[256] |
//            B9[260] = g(256) || dir(3) | A9[128] | HD[128]
struct SirenWs {
    static constexpr int kX0 = 4, kB = 260, kH = 256;
    static constexpr int per_row = kX0 + 8 * kH + 4 * kH + kB + 3 * kH + kB + 128 + 128;   // 4620
    float *X0, *A[8], *H[8], *B5, *B9, *A9, *HD;
    long long ldH[8];
    SirenWs(float* base, long long rows) {
        float* p = base;
        X0 = p; p += rows * kX0;
        for (int l = 0; l < 8; ++l) { A[l] = p; p += rows * kH; }
        for (int l = 0; l < 4; ++l) { H[l] = p; ldH[l] = kH; p += rows * kH; }
        B5 = p; p += rows * kB;
        H[4] = B5 + 3; ldH[4] = kB;
        for (int l = 5; l < 8; ++l) { H[l] = p; ldH[l] = kH; p += rows * kH; }
        B9 = p; p += rows * kB;
        A9 = p; p += rows * 128;
        HD = p;
    }
};

constexpr long long kInferChunk = 65536;   // rows per pass when activations are not kept

// ---- input encoders ---------------------------------------------------------------------------
// one thread per (row, octave): octaves 0..9 position (B5 columns 6i..6i+5), 10..13 direction
// (B9 columns 256+6i..).  sin/cos are the accurate libdevice versions: |2^9 x| reaches ~3000 rad.
__global__ void nerf_encode_kernel(RowSource src, long long row0, long long rows, float* __restrict__ B5,
                                   float* __restrict__ B9) {
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t >= rows * 14) return;
    long long row = t / 14;
    int o = (int)(t % 14);
    float p[3], v[3];
    load_row(src, row0 + row, p, v);
    if (o < 10) {
        float f = (float)(1 << o);
        float* out = B5 + row * NerfWs::kB5 + 6 * o;
#pragma unroll
        for (int c = 0; c < 3; ++c) { float a = __fmul_rn(f, p[c]); out[c] = sinf(a); out[3 + c] = cosf(a); }
    } else {
        int i = o - 10;
        float f = (float)(1 << i);
        float* out = B9 + row * NerfWs::kB9 + 256 + 6 * i;
#pragma unroll
        for (int c = 0; c < 3; ++c) { float a = __fmul_rn(f, v[c]); out[c] = sinf(a); out[3 + c] = cosf(a); }
    }
}

__global__ void film_encode_kernel(RowSource src, long long row0, long long rows, float* __restrict__ X0,
                                   float* __restrict__ B8) {
    long long row = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (row >= rows) return;
    float p[3], v[3];
    load_row(src, row0 + row, p, v);
    float* x = X0 + row * FilmWs::kX0;
    x[0] = p[0]; x[1] = p[1]; x[2] = p[2]; x[3] = 0.f;
    float* d = B8 + row * FilmWs::kB8 + 256;
    d[0] = v[0]; d[1] = v[1]; d[2] = v[2]; d[3] = 0.f;
}

// SirenNeRF takes raw inputs: pos -> X0 (layer 0) and B5[:, 0:3] (skip), dir -> B9[:, 256:259]
__global__ void siren_encode_kernel(RowSource src, long long row0, long long rows, float* __restrict__ X0, float* __restrict__ B5,
                                    float* __restrict__ B9) {
    long long row = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (row >= rows) return;
    float p[3], v[3];
    load_row(src, row0 + row, p, v);
    float* x = X0 + row * SirenWs::kX0;
    x[0] = p[0]; x[1] = p[1]; x[2] = p[2]; x[3] = 0.f;
    float* b5 = B5 + row * SirenWs::kB;
    b5[0] = p[0]; b5[1] = p[1]; b5[2] = p[2]; b5[259] = 0.f;
    float* d = B9 + row * SirenWs::kB + 256;
    d[0] = v[0]; d[1] = v[1]; d[2] = v[2]; d[3] = 0.f;
}

// ---- narrow heads (N <= 3 outputs): one warp per row ---------------------------------------------
// out[row*4 + col0 + n] = act(x[row,:] . W[n,:] + b[n]);  act: 1 relu, 2 sigmoid
// pick != NULL (b2r_mlp_f32_last_sigma): row i is the last sample of ray pick[i] and its result goes to that row of raw.
template <int N>
__global__ void __launch_bounds__(256) head_fwd_kernel(const float* __restrict__ X, long long ldx, int K,
                                                       const float* __restrict__ W, const float* __restrict__ b,
                                                       long long rows, int act, float* __restrict__ raw, int col0,
                                                       const int* __restrict__ pick = nullptr, int pick_s = 0) {
    const int lane = threadIdx.x & 31;
    long long row = (blockIdx.x * (long long)blockDim.x + threadIdx.x) >> 5;
    if (row >= rows) return;
    const long long out_row = pick ? (long long)pick[row] * pick_s + (pick_s - 1) : row;
    float acc[N];
#pragma unroll
    for (int n = 0; n < N; ++n) acc[n] = 0.f;
    for (int k = lane; k < K; k += 32) {
        float x = X[row * ldx + k];
#pragma unroll
        for (int n = 0; n < N; ++n) acc[n] = fmaf(x, W[n * K + k], acc[n]);
    }
#pragma unroll
    for (int n = 0; n < N; ++n) acc[n] = warp_sum(acc[n]);
    if (lane == 0) {
#pragma unroll
        for (int n = 0; n < N; ++n) {
            float v = __fadd_rn(acc[n], b[n]);
            v = act == 1 ? fmaxf(v, 0.f) : 1.0f / (1.0f + expf(-v));
            raw[out_row * 4 + col0 + n] = v;
        }
    }
}

// reverse of a narrow head.  g[row, n] = d_raw[row*4+col0+n] * act'(raw):  relu' = (raw>0),
// sigmoid' = raw (1-raw).  One CTA walks a slab of rows; thread k owns input column k:
//   dW[n,k] += sum_rows g x[row,k] ;  db[n] += sum_rows g ;  dX[row,k] (+)= sum_n g W[n,k]
template <int N>
__global__ void __launch_bounds__(256) head_bwd_kernel(const float* __restrict__ X, long long ldx, int K,
                                                       const float* __restrict__ W, long long rows, int rows_per_cta,
                                                       int act, const float* __restrict__ raw,
                                                       const float* __restrict__ d_raw, int col0,
                                                       float* __restrict__ dW, float* __restrict__ db,
                                                       float* __restrict__ dX, long long lddx) {
    const int k = threadIdx.x;
    long long r0 = (long long)blockIdx.x * rows_per_cta;
    long long r1 = min(rows, r0 + rows_per_cta);
    float w[N], aw[N], ab[N];
#pragma unroll
    for (int n = 0; n < N; ++n) { w[n] = k < K ? W[n * K + k] : 0.f; aw[n] = 0.f; ab[n] = 0.f; }
    for (long long row = r0; row < r1; ++row) {
        float x = k < K ? X[row * ldx + k] : 0.f;
        float dx = 0.f;
#pragma unroll
        for (int n = 0; n < N; ++n) {
            float y = raw[row * 4 + col0 + n];
            float g = d_raw[row * 4 + col0 + n] * (act == 1 ? (y > 0.f ? 1.0f : 0.f) : y * (1.0f - y));
            aw[n] = fmaf(g, x, aw[n]);
            ab[n] += g;
            dx = fmaf(g, w[n], dx);
        }
        if (dX && k < K) dX[row * lddx + k] = dx;
    }
    if (k < K) {
#pragma unroll
        for (int n = 0; n < N; ++n) atomicAdd(dW + n * K + k, aw[n]);
    }
    if (k == 0) {
#pragma unroll
        for (int n = 0; n < N; ++n) atomicAdd(db + n, ab[n]);
    }
}

// dX[row,k] = sum_n g[row,n] W[n,k] only (weights frozen: pi_GAN/synthesis.py:51-52)
__global__ void __launch_bounds__(256) head_dx_kernel(const float* __restrict__ W, long long rows, int K, int N, int act,
                                                      const float* __restrict__ raw, const float* __restrict__ d_raw,
                                                      int col0, float* __restrict__ dX, long long lddx) {
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t >= rows * K) return;
    long long row = t / K;
    int k = (int)(t % K);
    float dx = 0.f;
    for (int n = 0; n < N; ++n) {
        float y = raw[row * 4 + col0 + n];
        float g = d_raw[row * 4 + col0 + n] * (act == 1 ? (y > 0.f ? 1.0f : 0.f) : y * (1.0f - y));
        dx = fmaf(g, W[n * K + k], dx);
    }
    dX[row * lddx + k] = dx;
}

// G[e] = Y[e] > 0 ? G[e] : 0
__global__ void __launch_bounds__(256) relu_mask_kernel(float* __restrict__ G, const float* __restrict__ Y, long long n) {
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t < n && !(Y[t] > 0.f)) G[t] = 0.f;
}

// db[j] += sum_rows G[row, j]   (J <= 256 columns; one CTA per slab of rows, thread = column)
__global__ void __launch_bounds__(256) colsum_kernel(const float* __restrict__ G, long long ldg, int J, long long rows,
                                                     int rows_per_cta, float* __restrict__ db) {
    const int j = threadIdx.x;
    if (j >= J) return;
    long long r0 = (long long)blockIdx.x * rows_per_cta;
    long long r1 = min(rows, r0 + rows_per_cta);
    float s = 0.f;
    for (long long row = r0; row < r1; ++row) s += G[row * ldg + j];
    atomicAdd(db + j, s);
}

// FiLM-SIREN activation reverse (SURVEY A.6), in place on the incoming gradient:
//   t = 30 (gamma a + beta); g_t = dH cos t; dgamma += 30 sum g_t a; dbeta += 30 sum g_t; G = 30 gamma g_t
// gamma == NULL: plain SIREN layer (gamma 1, beta 0; nerf/nerf.py:111-112).  J = columns (<= 256), A has leading dimension J.
__global__ void __launch_bounds__(256) film_act_bwd_kernel(float* __restrict__ dH, long long ldd,
                                                           const float* __restrict__ A, long long rows, int rows_per_cta,
                                                           const float* __restrict__ gamma, const float* __restrict__ beta,
                                                           float* __restrict__ d_gamma, float* __restrict__ d_beta, int J = 256) {
    const int j = threadIdx.x;
    if (j >= J) return;
    long long r0 = (long long)blockIdx.x * rows_per_cta;
    long long r1 = min(rows, r0 + rows_per_cta);
    const float gm = gamma ? gamma[j] : 1.0f, bt = gamma ? beta[j] : 0.0f;
    float sg = 0.f, sb = 0.f;
    long long row = r0;
    for (; row + 4 <= r1; row += 4) {                       // 4 rows in flight per thread (the loop is load-latency bound)
        float a[4], d[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) { a[u] = A[(row + u) * J + j]; d[u] = dH[(row + u) * ldd + j]; }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            float t = __fmul_rn(30.0f, __fadd_rn(__fmul_rn(gm, a[u]), bt));
            float gt = d[u] * cosf(t);
            sg = fmaf(gt, a[u], sg);
            sb += gt;
            dH[(row + u) * ldd + j] = 30.0f * gm * gt;
        }
    }
    for (; row < r1; ++row) {
        float a = A[row * J + j];
        float t = __fmul_rn(30.0f, __fadd_rn(__fmul_rn(gm, a), bt));
        float gt = dH[row * ldd + j] * cosf(t);
        sg = fmaf(gt, a, sg);
        sb += gt;
        dH[row * ldd + j] = 30.0f * gm * gt;
    }
    if (d_gamma) { atomicAdd(d_gamma + j, 30.0f * sg); atomicAdd(d_beta + j, 30.0f * sb); }
}

// First layer of the SIREN networks (K = 3 inputs): y = sin(30 (gamma (W x + b) + beta)), pre = W x + b.  No GEMM: one thread per
// (row, 4 output columns), exact fp32 with the same individually rounded operations as the sgemm epilogue; coalesced float4 stores.
__global__ void __launch_bounds__(256) siren_first_layer_kernel(const float* __restrict__ X, long long ldx, const float* __restrict__ W,
                                                                const float* __restrict__ b, const float* __restrict__ gamma,
                                                                const float* __restrict__ beta, long long rows, float* __restrict__ Y,
                                                                long long ldy, float* __restrict__ pre) {
    const long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const long long row = t >> 6;                     // 64 column groups of 4 = 256 outputs
    const int n0 = (int)(t & 63) * 4;
    if (row >= rows) return;
    const float x0 = X[row * ldx], x1 = X[row * ldx + 1], x2 = X[row * ldx + 2];
    float y[4], a[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const float* w = W + (n0 + q) * 3;
        float acc = fmaf(x2, w[2], fmaf(x1, w[1], x0 * w[0]));          // same k order as the sgemm inner loop
        a[q] = __fadd_rn(acc, b[n0 + q]);
        y[q] = gamma ? sinf(__fmul_rn(30.0f, __fadd_rn(__fmul_rn(gamma[n0 + q], a[q]), beta[n0 + q]))) : sinf(__fmul_rn(30.0f, a[q]));
    }
    *reinterpret_cast<float4*>(Y + row * ldy + n0) = make_float4(y[0], y[1], y[2], y[3]);
    if (pre) *reinterpret_cast<float4*>(pre + row * 256 + n0) = make_float4(a[0], a[1], a[2], a[3]);
}

// GEMM engine of the current call on this host thread: 0 = fp32 CUDA cores (exact), 1 = tf32 tensor cores (tgemm.cuh).
// thread_local, set at every API entry: the library stays re-entrant (nn.DataParallel calls it from one thread per GPU).
static thread_local int t_gemm_mode = 0;
// b2r_mlp_f32_last_sigma on a latent batch: latent of every gathered row (FiLM scale / shift row of the sine epilogue)
static thread_local const int* t_row_lat = nullptr;

template <bool kPT, bool kQT>
static int launch_gemm(GemmArgs g, cudaStream_t st, const char* what) {
    // tiny reductions (K = 3 input layer) stay on the CUDA cores
    if (t_gemm_mode == 1 && g.R >= 16) return tg::launch_tgemm<kPT, kQT>(g, st, what);
    return launch_sgemm<kPT, kQT>(g, st, what);
}

// ---- helpers ------------------------------------------------------------------------------------
struct Lin { const float* W; const float* b; int out, in; };
static inline Lin lin(const float* params, LayerDesc d) { return Lin{params + d.w_off, params + d.b_off, d.out, d.in}; }

static int fwd_layer(const float* X, long long ldx, Lin L, int k_off, int K, float* Y, long long ldy, long long rows,
                     int epi, cudaStream_t st, const float* gamma = nullptr, const float* beta = nullptr,
                     float* pre = nullptr) {
    if (t_gemm_mode == 1 && K == 3 && L.in == 3 && L.out == 256 && epi == EPI_FILM_SIN && ldy % 4 == 0 && aligned16(Y) && (!pre || aligned16(pre))) {
        // tf32 mode: the K = 3 first layer is no GEMM (the exact fp32 mode keeps the sgemm path its parity fixtures were made with)
        const long long threads = rows * 64;
        siren_first_layer_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(X, ldx, L.W, L.b, gamma, beta, rows, Y, ldy, pre);
        return cuda_result(cudaGetLastError(), "siren first layer");
    }
    GemmArgs g{};
    g.P = X; g.ldp = ldx; g.Q = L.W + k_off; g.ldq = L.in; g.C = Y; g.ldc = ldy;
    g.I = rows; g.J = L.out; g.R = K; g.r_chunk = K; g.epi = epi; g.bias = L.b;
    g.gamma = gamma; g.beta = beta; g.pre = pre; g.ldpre = 256;
    if (gamma && t_row_lat) { g.row_lat = t_row_lat; g.lat_stride = B2R_FILM_PARAMS; }
    return launch_gemm<false, false>(g, st, "mlp_f32 forward gemm");
}
// dX = G W[:, k_off:k_off+K]  (optionally += existing, optionally relu-masked by `mask`)
static int dgrad_layer(const float* G, long long ldg, Lin L, int k_off, int K, float* dX, long long lddx, long long rows,
                       const float* mask, long long ldmask, int accumulate, cudaStream_t st) {
    GemmArgs g{};
    g.P = G; g.ldp = ldg; g.Q = L.W + k_off; g.ldq = L.in; g.C = dX; g.ldc = lddx;
    g.I = rows; g.J = K; g.R = L.out; g.r_chunk = L.out; g.epi = EPI_DGRAD;
    g.mask = mask; g.ldmask = ldmask; g.accumulate = accumulate;
    return launch_gemm<false, true>(g, st, "mlp_f32 dgrad gemm");
}
// dW += G^T X ; db += colsum(G)
static int wgrad_layer(const float* G, long long ldg, const float* X, long long ldx, LayerDesc d, float* d_params,
                       long long rows, cudaStream_t st) {
    GemmArgs g{};
    g.P = G; g.ldp = ldg; g.Q = X; g.ldq = ldx; g.C = d_params + d.w_off; g.ldc = d.in;
    g.I = d.out; g.J = d.in; g.R = rows; g.r_chunk = t_gemm_mode == 1 ? 8192 : 2048; g.epi = EPI_ATOMIC;
    int rc = launch_gemm<true, true>(g, st, "mlp_f32 wgrad gemm");
    if (rc) return rc;
    int rpc = 512;
    unsigned grid = (unsigned)((rows + rpc - 1) / rpc);
    colsum_kernel<<<grid, 256, 0, st>>>(G, ldg, d.out, rows, rpc, d_params + d.b_off);
    return cuda_result(cudaGetLastError(), "mlp_f32 colsum");
}

#define B2R_TRY(expr) do { int rc__ = (expr); if (rc__) return rc__; } while (0)

// ---- NeRF forward on rows [row0, row0+rows) into workspace ws (indexed from 0) -----------------------
// last_only: the rows are the gathered last samples of src.pick's rays; stop after the sigma head and scatter its output
static int nerf_forward_rows(const float* params, const RowSource& src, long long row0, long long rows, NerfWs& ws,
                             float* raw, cudaStream_t st, bool last_only = false) {
    {
        long long threads = rows * 14;
        nerf_encode_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(src, row0, rows, ws.B5, ws.B9);
        B2R_TRY(cuda_result(cudaGetLastError(), "nerf_encode"));
    }
    B2R_TRY(fwd_layer(ws.B5, NerfWs::kB5, lin(params, nerf_layer(0)), 0, 60, ws.H[0], ws.ldH[0], rows, EPI_RELU, st));
    for (int l = 1; l <= 4; ++l)
        B2R_TRY(fwd_layer(ws.H[l - 1], ws.ldH[l - 1], lin(params, nerf_layer(l)), 0, 256, ws.H[l], ws.ldH[l], rows, EPI_RELU, st));
    B2R_TRY(fwd_layer(ws.B5, NerfWs::kB5, lin(params, nerf_layer(5)), 0, 316, ws.H[5], ws.ldH[5], rows, EPI_RELU, st));
    B2R_TRY(fwd_layer(ws.H[5], 256, lin(params, nerf_layer(6)), 0, 256, ws.H[6], 256, rows, EPI_RELU, st));
    B2R_TRY(fwd_layer(ws.H[6], 256, lin(params, nerf_layer(7)), 0, 256, ws.H[7], 256, rows, EPI_RELU, st));
    unsigned hgrid = (unsigned)((rows * 32 + 255) / 256);
    {
        Lin s = lin(params, nerf_layer(10));
        if (last_only) head_fwd_kernel<1><<<hgrid, 256, 0, st>>>(ws.H[7], 256, 256, s.W, s.b, rows, 1, raw, 3, src.pick + row0, src.pick_s);
        else head_fwd_kernel<1><<<hgrid, 256, 0, st>>>(ws.H[7], 256, 256, s.W, s.b, rows, 1, raw + row0 * 4, 3);
        B2R_TRY(cuda_result(cudaGetLastError(), "nerf sigma head"));
        if (last_only) return 0;
    }
    B2R_TRY(fwd_layer(ws.H[7], 256, lin(params, nerf_layer(8)), 0, 256, ws.B9, NerfWs::kB9, rows, EPI_STORE, st));
    B2R_TRY(fwd_layer(ws.B9, NerfWs::kB9, lin(params, nerf_layer(9)), 0, 280, ws.HD, 128, rows, EPI_RELU, st));
    {
        Lin c = lin(params, nerf_layer(11));
        head_fwd_kernel<3><<<hgrid, 256, 0, st>>>(ws.HD, 128, 128, c.W, c.b, rows, 2, raw + row0 * 4, 0);
        B2R_TRY(cuda_result(cudaGetLastError(), "nerf rgb head"));
    }
    return 0;
}

static int film_forward_rows(const float* params, const float* film, bool use_dir, const RowSource& src, long long row0,
                             long long rows, FilmWs& ws, float* raw, bool save, cudaStream_t st, bool last_only = false) {
    film_encode_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(src, row0, rows, ws.X0, ws.B8);
    B2R_TRY(cuda_result(cudaGetLastError(), "film_encode"));
    B2R_TRY(fwd_layer(ws.X0, FilmWs::kX0, lin(params, film_layer(0, use_dir)), 0, 3, ws.H[0], ws.ldH[0], rows, EPI_FILM_SIN, st,
                      film, film + 256, save ? ws.A[0] : nullptr));
    for (int l = 1; l <= 7; ++l)
        B2R_TRY(fwd_layer(ws.H[l - 1], ws.ldH[l - 1], lin(params, film_layer(l, use_dir)), 0, 256, ws.H[l], ws.ldH[l], rows,
                          EPI_FILM_SIN, st, film + l * 512, film + l * 512 + 256, save ? ws.A[l] : nullptr));
    unsigned hgrid = (unsigned)((rows * 32 + 255) / 256);
    {
        Lin s = lin(params, film_layer(8, use_dir));
        if (last_only) head_fwd_kernel<1><<<hgrid, 256, 0, st>>>(ws.B8, FilmWs::kB8, 256, s.W, s.b, rows, 1, raw, 3, src.pick + row0, src.pick_s);
        else head_fwd_kernel<1><<<hgrid, 256, 0, st>>>(ws.B8, FilmWs::kB8, 256, s.W, s.b, rows, 1, raw + row0 * 4, 3);
        B2R_TRY(cuda_result(cudaGetLastError(), "film sigma head"));
        if (last_only) return 0;
    }
    int kc = use_dir ? 259 : 256;
    B2R_TRY(fwd_layer(ws.B8, FilmWs::kB8, lin(params, film_layer(9, use_dir)), 0, kc, ws.HC, 256, rows, EPI_FILM_SIN, st,
                      film + 8 * 512, film + 8 * 512 + 256, save ? ws.A[8] : nullptr));
    {
        Lin c = lin(params, film_layer(10, use_dir));
        head_fwd_kernel<3><<<hgrid, 256, 0, st>>>(ws.HC, 256, 256, c.W, c.b, rows, 2, raw + row0 * 4, 0);
        B2R_TRY(cuda_result(cudaGetLastError(), "film rgb head"));
    }
    return 0;
}

static int siren_forward_rows(const float* params, const RowSource& src, long long row0, long long rows, SirenWs& ws, float* raw, bool save,
                              cudaStream_t st, bool last_only = false) {
    siren_encode_kernel<<<(unsigned)((rows + 255) / 256), 256, 0, st>>>(src, row0, rows, ws.X0, ws.B5, ws.B9);
    B2R_TRY(cuda_result(cudaGetLastError(), "siren_encode"));
    auto L = [&](int i) { return lin(params, siren_layer(i)); };
    B2R_TRY(fwd_layer(ws.X0, SirenWs::kX0, L(0), 0, 3, ws.H[0], ws.ldH[0], rows, EPI_FILM_SIN, st, nullptr, nullptr, save ? ws.A[0] : nullptr));
    for (int l = 1; l <= 4; ++l)
        B2R_TRY(fwd_layer(ws.H[l - 1], ws.ldH[l - 1], L(l), 0, 256, ws.H[l], ws.ldH[l], rows, EPI_FILM_SIN, st, nullptr, nullptr,
                          save ? ws.A[l] : nullptr));
    B2R_TRY(fwd_layer(ws.B5, SirenWs::kB, L(5), 0, 259, ws.H[5], 256, rows, EPI_FILM_SIN, st, nullptr, nullptr, save ? ws.A[5] : nullptr));   // [pos | h4]
    B2R_TRY(fwd_layer(ws.H[5], 256, L(6), 0, 256, ws.H[6], 256, rows, EPI_FILM_SIN, st, nullptr, nullptr, save ? ws.A[6] : nullptr));
    B2R_TRY(fwd_layer(ws.H[6], 256, L(7), 0, 256, ws.H[7], 256, rows, EPI_FILM_SIN, st, nullptr, nullptr, save ? ws.A[7] : nullptr));
    unsigned hgrid = (unsigned)((rows * 32 + 255) / 256);
    {
        Lin s = L(10);
        if (last_only) head_fwd_kernel<1><<<hgrid, 256, 0, st>>>(ws.H[7], 256, 256, s.W, s.b, rows, 1, raw, 3, src.pick + row0, src.pick_s);
        else head_fwd_kernel<1><<<hgrid, 256, 0, st>>>(ws.H[7], 256, 256, s.W, s.b, rows, 1, raw + row0 * 4, 3);
        B2R_TRY(cuda_result(cudaGetLastError(), "siren sigma head"));
        if (last_only) return 0;
    }
    B2R_TRY(fwd_layer(ws.H[7], 256, L(8), 0, 256, ws.B9, SirenWs::kB, rows, EPI_STORE, st));                                                  // linear
    {
        GemmArgs g{};                                                                                                                      // [g | dir] -> 128, sin
        Lin l9 = L(9);
        g.P = ws.B9; g.ldp = SirenWs::kB; g.Q = l9.W; g.ldq = l9.in; g.C = ws.HD; g.ldc = 128;
        g.I = rows; g.J = 128; g.R = 259; g.r_chunk = 259; g.epi = EPI_FILM_SIN; g.bias = l9.b;
        g.pre = save ? ws.A9 : nullptr; g.ldpre = 128;
        B2R_TRY((launch_gemm<false, false>(g, st, "siren layers_dir.1")));
    }
    {
        Lin c = L(11);
        head_fwd_kernel<3><<<hgrid, 256, 0, st>>>(ws.HD, 128, 128, c.W, c.b, rows, 2, raw + row0 * 4, 0);
        B2R_TRY(cuda_result(cudaGetLastError(), "siren rgb head"));
    }
    return 0;
}

static inline bool known_kind(int kind) { return kind == B2R_MODEL_NERF || kind == B2R_MODEL_FILM || kind == B2R_MODEL_SIREN; }
static inline int per_row(int kind) {
    return kind == B2R_MODEL_NERF ? NerfWs::per_row : (kind == B2R_MODEL_FILM ? FilmWs::per_row : SirenWs::per_row);
}

}  // namespace b2r

extern "C" size_t b2r_mlp_f32_workspace_bytes(int model_kind, long long rows, int save_activations) {
    using namespace b2r;
    if (rows < 0 || !known_kind(model_kind)) return 0;
    long long r = save_activations ? rows : (rows < kInferChunk ? rows : kInferChunk);
    return (size_t)r * per_row(model_kind) * sizeof(float);
}

extern "C" int b2r_mlp_f32_fwd(int model_kind, const float* params, const float* film, int use_dir,
                               const b2r_mlp_input* in, float* raw_out, void* workspace, size_t workspace_bytes,
                               int save_activations, int gemm_mode, void* stream) {
    using namespace b2r;
    B2R_CHECK_ARG(gemm_mode == 0 || gemm_mode == 1, "b2r_mlp_f32_fwd: gemm_mode must be 0 (fp32) or 1 (tf32)");
    t_gemm_mode = gemm_mode;
    B2R_CHECK_ARG(known_kind(model_kind), "b2r_mlp_f32_fwd: unknown model kind %d", model_kind);
    B2R_CHECK_ARG(params && raw_out && workspace, "b2r_mlp_f32_fwd: NULL pointer");
    B2R_CHECK_ARG(model_kind != B2R_MODEL_FILM || film, "b2r_mlp_f32_fwd: FiLM model needs film params");
    B2R_TRY(check_mlp_input(in));
    long long rows = row_count(in);
    B2R_CHECK_ARG(workspace_bytes >= b2r_mlp_f32_workspace_bytes(model_kind, rows, save_activations),
                  "b2r_mlp_f32_fwd: workspace too small (%zu B)", workspace_bytes);
    B2R_CHECK_ARG(aligned16(workspace) && aligned16(params), "b2r_mlp_f32_fwd: params / workspace must be 16-byte aligned");
    if (rows == 0) return 0;
    RowSource src = make_row_source(in);
    cudaStream_t st = (cudaStream_t)stream;
    long long step = save_activations ? rows : kInferChunk;
    for (long long r0 = 0; r0 < rows; r0 += step) {
        long long n = rows - r0 < step ? rows - r0 : step;
        if (model_kind == B2R_MODEL_NERF) {
            NerfWs ws((float*)workspace, n);
            B2R_TRY(nerf_forward_rows(params, src, r0, n, ws, raw_out, st));
        } else if (model_kind == B2R_MODEL_SIREN) {
            SirenWs ws((float*)workspace, n);
            B2R_TRY(siren_forward_rows(params, src, r0, n, ws, raw_out, save_activations != 0, st));
        } else {
            FilmWs ws((float*)workspace, n);
            B2R_TRY(film_forward_rows(params, film, use_dir != 0, src, r0, n, ws, raw_out, save_activations != 0, st));
        }
    }
    return 0;
}

namespace b2r {
// latent of every gathered row: source row = pick[i] * s + s - 1
__global__ void row_latent_kernel(const int* __restrict__ pick, int n, int s, long long rows_per_latent, int n_latents, int* __restrict__ row_lat) {
    int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    long long lat = ((long long)pick[i] * s + (s - 1)) / rows_per_latent;
    row_lat[i] = (int)(lat < n_latents ? lat : n_latents - 1);
}
}  // namespace b2r

// The last interval of a ray is 1e10 (nerf/render.py:92): sign(sigma_pre) of the last sample decides the ray (include/b2r.h,
// b2r_last_sample).  Re-evaluates the listed rays' last samples with the exact fp32 engine -- the same kernels, operand order
// and rounding as b2r_mlp_f32_fwd, so the result equals what the fp32 path computes for that row bit for bit.
extern "C" int b2r_mlp_f32_last_sigma(int model_kind, const float* params, const float* film, int use_dir, int n_latents,
                                      long long rows_per_latent, const b2r_mlp_input* in, int samples_per_ray, const int* ray_ids,
                                      int n_ids, float* raw_io, void* workspace, size_t workspace_bytes, void* stream) {
    using namespace b2r;
    t_gemm_mode = 0;
    B2R_CHECK_ARG(known_kind(model_kind), "b2r_mlp_f32_last_sigma: unknown model kind %d", model_kind);
    B2R_CHECK_ARG(params && raw_io && workspace && ray_ids, "b2r_mlp_f32_last_sigma: NULL pointer");
    B2R_CHECK_ARG(model_kind != B2R_MODEL_FILM || film, "b2r_mlp_f32_last_sigma: FiLM model needs film params");
    B2R_TRY(check_mlp_input(in));
    B2R_CHECK_ARG(in->grid_n == 0 && !lattice_mode(in), "b2r_mlp_f32_last_sigma: rays / x rows only");
    B2R_CHECK_ARG(samples_per_ray >= 1 && (!in->rays || samples_per_ray == in->n_samples), "b2r_mlp_f32_last_sigma: samples_per_ray (%d) must equal n_samples in rays mode", samples_per_ray);
    B2R_CHECK_ARG(n_ids >= 0 && n_latents >= 1 && (n_latents == 1 || rows_per_latent > 0), "b2r_mlp_f32_last_sigma: bad n_ids / n_latents / rows_per_latent");
    const size_t lat_bytes = ((size_t)n_ids * 4 + 15) & ~(size_t)15;
    B2R_CHECK_ARG(workspace_bytes >= b2r_mlp_f32_workspace_bytes(model_kind, n_ids, 0) + lat_bytes, "b2r_mlp_f32_last_sigma: workspace too small (%zu B)", workspace_bytes);
    B2R_CHECK_ARG(aligned16(workspace) && aligned16(params), "b2r_mlp_f32_last_sigma: params / workspace must be 16-byte aligned");
    if (n_ids == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    RowSource src = make_row_source(in);
    src.pick = ray_ids; src.pick_s = samples_per_ray;
    int* row_lat = (int*)workspace;
    float* act = (float*)((char*)workspace + lat_bytes);
    const bool batched = model_kind == B2R_MODEL_FILM && n_latents > 1;
    if (batched) {
        row_latent_kernel<<<(unsigned)((n_ids + 255) / 256), 256, 0, st>>>(ray_ids, n_ids, samples_per_ray, rows_per_latent, n_latents, row_lat);
        B2R_TRY(cuda_result(cudaGetLastError(), "row_latent"));
    }
    int rc = 0;
    for (long long r0 = 0; r0 < n_ids && rc == 0; r0 += kInferChunk) {
        long long n = n_ids - r0 < kInferChunk ? n_ids - r0 : kInferChunk;
        if (model_kind == B2R_MODEL_NERF) {
            NerfWs ws(act, n);
            rc = nerf_forward_rows(params, src, r0, n, ws, raw_io, st, true);
        } else if (model_kind == B2R_MODEL_SIREN) {
            SirenWs ws(act, n);
            rc = siren_forward_rows(params, src, r0, n, ws, raw_io, false, st, true);
        } else {
            FilmWs ws(act, n);
            t_row_lat = batched ? row_lat + r0 : nullptr;
            rc = film_forward_rows(params, film, use_dir != 0, src, r0, n, ws, raw_io, false, st, true);
            t_row_lat = nullptr;
        }
    }
    return rc;
}

extern "C" size_t b2r_mlp_f32_bwd_scratch_bytes(int model_kind, long long rows) {
    if (rows < 0 || !b2r::known_kind(model_kind)) return 0;
    return (size_t)rows * (2 * 256) * sizeof(float);   // two ping-pong gradient buffers [rows,256]
}

extern "C" int b2r_mlp_f32_bwd(int model_kind, const float* params, const float* film, int use_dir,
                               const b2r_mlp_input* in, const float* raw, const float* d_raw, const void* saved,
                               void* scratch, size_t scratch_bytes, float* d_params, float* d_film, int gemm_mode, void* stream) {
    using namespace b2r;
    B2R_CHECK_ARG(gemm_mode == 0 || gemm_mode == 1, "b2r_mlp_f32_bwd: gemm_mode must be 0 (fp32) or 1 (tf32)");
    t_gemm_mode = gemm_mode;
    B2R_CHECK_ARG(known_kind(model_kind), "b2r_mlp_f32_bwd: unknown model kind %d", model_kind);
    B2R_CHECK_ARG(params && raw && d_raw && saved && scratch, "b2r_mlp_f32_bwd: NULL pointer");
    B2R_CHECK_ARG(d_params || d_film, "b2r_mlp_f32_bwd: nothing to differentiate (d_params and d_film are NULL)");
    B2R_TRY(check_mlp_input(in));
    long long rows = row_count(in);
    B2R_CHECK_ARG(scratch_bytes >= b2r_mlp_f32_bwd_scratch_bytes(model_kind, rows), "b2r_mlp_f32_bwd: scratch too small");
    B2R_CHECK_ARG(aligned16(scratch) && aligned16(saved), "b2r_mlp_f32_bwd: buffers must be 16-byte aligned");
    if (rows == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    float* G0 = (float*)scratch;
    float* G1 = G0 + rows * 256;
    const int rpc = 512;
    const unsigned slab_grid = (unsigned)((rows + rpc - 1) / rpc);

    if (model_kind == B2R_MODEL_NERF) {
        B2R_CHECK_ARG(d_params, "b2r_mlp_f32_bwd: NeRF needs d_params");
        NerfWs ws((float*)const_cast<void*>(saved), rows);
        // rgb head (sigmoid) -> dHD
        {
            LayerDesc d = nerf_layer(11);
            head_bwd_kernel<3><<<slab_grid, 256, 0, st>>>(ws.HD, 128, 128, params + d.w_off, rows, rpc, 2, raw, d_raw, 0,
                                                         d_params + d.w_off, d_params + d.b_off, G0, 128);
            B2R_TRY(cuda_result(cudaGetLastError(), "nerf rgb head bwd"));
        }
        // relu'(layers_dir.1 output), in place
        relu_mask_kernel<<<(unsigned)((rows * 128 + 255) / 256), 256, 0, st>>>(G0, ws.HD, rows * 128);
        B2R_TRY(cuda_result(cudaGetLastError(), "relu mask"));
        // layers_dir.1: [g || de] (280) -> 128
        B2R_TRY(wgrad_layer(G0, 128, ws.B9, NerfWs::kB9, nerf_layer(9), d_params, rows, st));
        B2R_TRY(dgrad_layer(G0, 128, lin(params, nerf_layer(9)), 0, 256, G1, 256, rows, nullptr, 0, 0, st));   // dg (linear layer: no mask)
        // layers_dir.0: h7 -> g
        B2R_TRY(wgrad_layer(G1, 256, ws.H[7], 256, nerf_layer(8), d_params, rows, st));
        // sigma head writes its contribution to dH7 first, dgrad accumulates on top and applies relu'(h7)
        {
            LayerDesc d = nerf_layer(10);
            head_bwd_kernel<1><<<slab_grid, 256, 0, st>>>(ws.H[7], 256, 256, params + d.w_off, rows, rpc, 1, raw, d_raw, 3,
                                                         d_params + d.w_off, d_params + d.b_off, G0, 256);
            B2R_TRY(cuda_result(cudaGetLastError(), "nerf sigma head bwd"));
        }
        B2R_TRY(dgrad_layer(G1, 256, lin(params, nerf_layer(8)), 0, 256, G0, 256, rows, ws.H[7], 256, 1, st));
        // trunk layers 7, 6, 5
        float* Gc = G0; float* Gn = G1;
        for (int l = 7; l >= 6; --l) {
            B2R_TRY(wgrad_layer(Gc, 256, ws.H[l - 1], ws.ldH[l - 1], nerf_layer(l), d_params, rows, st));
            B2R_TRY(dgrad_layer(Gc, 256, lin(params, nerf_layer(l)), 0, 256, Gn, 256, rows, ws.H[l - 1], ws.ldH[l - 1], 0, st));
            float* t = Gc; Gc = Gn; Gn = t;
        }
        B2R_TRY(wgrad_layer(Gc, 256, ws.B5, NerfWs::kB5, nerf_layer(5), d_params, rows, st));
        B2R_TRY(dgrad_layer(Gc, 256, lin(params, nerf_layer(5)), 60, 256, Gn, 256, rows, ws.H[4], ws.ldH[4], 0, st));
        { float* t = Gc; Gc = Gn; Gn = t; }
        for (int l = 4; l >= 1; --l) {
            B2R_TRY(wgrad_layer(Gc, 256, ws.H[l - 1], ws.ldH[l - 1], nerf_layer(l), d_params, rows, st));
            B2R_TRY(dgrad_layer(Gc, 256, lin(params, nerf_layer(l)), 0, 256, Gn, 256, rows, ws.H[l - 1], ws.ldH[l - 1], 0, st));
            float* t = Gc; Gc = Gn; Gn = t;
        }
        B2R_TRY(wgrad_layer(Gc, 256, ws.B5, NerfWs::kB5, nerf_layer(0), d_params, rows, st));
        return 0;
    }

    if (model_kind == B2R_MODEL_SIREN) {
        // SirenNeRF (nerf/nerf.py:152-170): y = sin(30 a), a = W x + b  ->  dA = 30 cos(30 a) dY (film_act_bwd with gamma 1, beta 0)
        B2R_CHECK_ARG(d_params, "b2r_mlp_f32_bwd: SirenNeRF needs d_params");
        SirenWs ws((float*)const_cast<void*>(saved), rows);
        auto act_bwd = [&](float* G, long long ldg, const float* A, int J) -> int {
            film_act_bwd_kernel<<<slab_grid, 256, 0, st>>>(G, ldg, A, rows, rpc, nullptr, nullptr, nullptr, nullptr, J);
            return cuda_result(cudaGetLastError(), "siren act bwd");
        };
        {
            LayerDesc d = siren_layer(11);
            head_bwd_kernel<3><<<slab_grid, 256, 0, st>>>(ws.HD, 128, 128, params + d.w_off, rows, rpc, 2, raw, d_raw, 0,
                                                         d_params + d.w_off, d_params + d.b_off, G0, 128);
            B2R_TRY(cuda_result(cudaGetLastError(), "siren rgb head bwd"));
        }
        B2R_TRY(act_bwd(G0, 128, ws.A9, 128));
        B2R_TRY(wgrad_layer(G0, 128, ws.B9, SirenWs::kB, siren_layer(9), d_params, rows, st));
        B2R_TRY(dgrad_layer(G0, 128, lin(params, siren_layer(9)), 0, 256, G1, 256, rows, nullptr, 0, 0, st));          // d g
        B2R_TRY(wgrad_layer(G1, 256, ws.H[7], 256, siren_layer(8), d_params, rows, st));
        {
            LayerDesc d = siren_layer(10);
            head_bwd_kernel<1><<<slab_grid, 256, 0, st>>>(ws.H[7], 256, 256, params + d.w_off, rows, rpc, 1, raw, d_raw, 3,
                                                         d_params + d.w_off, d_params + d.b_off, G0, 256);
            B2R_TRY(cuda_result(cudaGetLastError(), "siren sigma head bwd"));
        }
        B2R_TRY(dgrad_layer(G1, 256, lin(params, siren_layer(8)), 0, 256, G0, 256, rows, nullptr, 0, 1, st));          // d h7 (+ sigma term)
        float* Gc = G0; float* Gn = G1;
        for (int l = 7; l >= 0; --l) {
            B2R_TRY(act_bwd(Gc, 256, ws.A[l], 256));
            if (l == 0) { B2R_TRY(wgrad_layer(Gc, 256, ws.X0, SirenWs::kX0, siren_layer(0), d_params, rows, st)); break; }
            if (l == 5) {
                B2R_TRY(wgrad_layer(Gc, 256, ws.B5, SirenWs::kB, siren_layer(5), d_params, rows, st));
                B2R_TRY(dgrad_layer(Gc, 256, lin(params, siren_layer(5)), 3, 256, Gn, 256, rows, nullptr, 0, 0, st));
            } else {
                B2R_TRY(wgrad_layer(Gc, 256, ws.H[l - 1], ws.ldH[l - 1], siren_layer(l), d_params, rows, st));
                B2R_TRY(dgrad_layer(Gc, 256, lin(params, siren_layer(l)), 0, 256, Gn, 256, rows, nullptr, 0, 0, st));
            }
            float* t = Gc; Gc = Gn; Gn = t;
        }
        return 0;
    }

    // ---- FiLM-SIREN
    B2R_CHECK_ARG(film, "b2r_mlp_f32_bwd: FiLM model needs film params");
    const bool ud = use_dir != 0;
    FilmWs ws((float*)const_cast<void*>(saved), rows);
    auto dgam = [&](int l) { return d_film ? d_film + l * 512 : nullptr; };
    auto dbet = [&](int l) { return d_film ? d_film + l * 512 + 256 : nullptr; };
    // weight gradients are skipped when d_params is NULL (inversion: only d_film is wanted)
    {
        LayerDesc d = film_layer(10, ud);
        if (d_params)
            head_bwd_kernel<3><<<slab_grid, 256, 0, st>>>(ws.HC, 256, 256, params + d.w_off, rows, rpc, 2, raw, d_raw, 0,
                                                         d_params + d.w_off, d_params + d.b_off, G0, 256);
        else
            head_dx_kernel<<<(unsigned)((rows * 256 + 255) / 256), 256, 0, st>>>(params + d.w_off, rows, 256, 3, 2, raw, d_raw, 0, G0, 256);
        B2R_TRY(cuda_result(cudaGetLastError(), "film rgb head bwd"));
    }
    // hidden_layer_rgb (film index 8): input B8 = [h7 || dir]
    film_act_bwd_kernel<<<slab_grid, 256, 0, st>>>(G0, 256, ws.A[8], rows, rpc, film + 8 * 512, film + 8 * 512 + 256, dgam(8), dbet(8));
    B2R_TRY(cuda_result(cudaGetLastError(), "film act bwd"));
    if (d_params) B2R_TRY(wgrad_layer(G0, 256, ws.B8, FilmWs::kB8, film_layer(9, ud), d_params, rows, st));
    // sigma head contribution to dH7 first, then dgrad accumulates
    {
        LayerDesc d = film_layer(8, ud);
        if (d_params) {
            head_bwd_kernel<1><<<slab_grid, 256, 0, st>>>(ws.B8, FilmWs::kB8, 256, params + d.w_off, rows, rpc, 1, raw, d_raw, 3,
                                                         d_params + d.w_off, d_params + d.b_off, G1, 256);
        } else {
            head_dx_kernel<<<(unsigned)((rows * 256 + 255) / 256), 256, 0, st>>>(params + d.w_off, rows, 256, 1, 1, raw, d_raw, 3, G1, 256);
        }
        B2R_TRY(cuda_result(cudaGetLastError(), "film sigma head bwd"));
    }
    B2R_TRY(dgrad_layer(G0, 256, lin(params, film_layer(9, ud)), 0, 256, G1, 256, rows, nullptr, 0, 1, st));
    float* Gc = G1; float* Gn = G0;
    for (int l = 7; l >= 0; --l) {
        film_act_bwd_kernel<<<slab_grid, 256, 0, st>>>(Gc, 256, ws.A[l], rows, rpc, film + l * 512, film + l * 512 + 256, dgam(l), dbet(l));
        B2R_TRY(cuda_result(cudaGetLastError(), "film act bwd"));
        if (l == 0) {
            if (d_params) B2R_TRY(wgrad_layer(Gc, 256, ws.X0, FilmWs::kX0, film_layer(0, ud), d_params, rows, st));
            break;
        }
        if (d_params) B2R_TRY(wgrad_layer(Gc, 256, ws.H[l - 1], ws.ldH[l - 1], film_layer(l, ud), d_params, rows, st));
        B2R_TRY(dgrad_layer(Gc, 256, lin(params, film_layer(l, ud)), 0, 256, Gn, 256, rows, nullptr, 0, 0, st));
        float* t = Gc; Gc = Gn; Gn = t;
    }
    return 0;
}
