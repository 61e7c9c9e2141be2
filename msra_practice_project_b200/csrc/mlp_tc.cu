// K3 (tensor-core path): the whole radiance-field MLP of a tile of samples evaluated inside ONE
// persistent kernel on the Blackwell 5th-generation tensor cores.
//   run_network + NeRF.forward            nerf/render.py:59-75, nerf/nerf.py:44-49, 75-94
//   FilmSirenNeRF.forward / create_mesh   pi_GAN/modules.py:22-25, 101-118, pi_GAN/utils.py:59-91
//
// Design: CTA PAIRS (cluster of 2, tcgen05 cta_group::2), one CTA per SM, 640 threads, persistent.
// Each CTA owns a 256-row tile = two 128-row sub-tiles; one MMA instruction covers sub-tile g of BOTH
// CTAs (M = 256) and every CTA stages only ITS HALF of the weight rows (N/2), so the L2 -> shared-memory
// weight stream and the shared-memory -> tensor-core B traffic per SM are half of a single-CTA design.
//   warp 0        weight producer (one thread per CTA): streams this CTA's half of each pre-swizzled bf16
//                 weight chunk (N/2 x 64 K, SWIZZLE_128B image, packed once by b2r_mlp_tc_pack) L2 ->
//                 shared memory with cp.async.bulk (TMA engine) through a 3-stage mbarrier ring;
//   warp 1        leader CTA: tcgen05.mma issuer (one thread): M=256, N=256|128, K=16 bf16 MMAs, A = the
//                 sub-tile's activations in each CTA's shared memory (K-major, SWIZZLE_128B), D = fp32
//                 accumulators in each CTA's tensor memory (2 x 256 columns = the two sub-tiles, ping-pong);
//                 tcgen05.commit multicast frees the ring stage / publishes the accumulator in both CTAs.
//                 peer CTA: relay thread forwarding "my half landed" to the leader's ring barrier;
//   warps 4-11    epilogue of sub-tile 0, warps 12-19 epilogue of sub-tile 1 (thread = row = TMEM lane,
//                 two warps per lane quadrant, each converting half of the columns):
//                 tcgen05.ld the accumulator, + bias, ReLU (or sin(s*acc+t) for FiLM-SIREN), round to
//                 bf16 and write the next layer's A operand back into shared memory IN PLACE -- the
//                 activations never touch HBM.  The first stage of the same threads generates the
//                 sample (o + d z), its positional encoding and the view-direction encoding; the last
//                 stage computes the narrow heads (sigma: 256 -> 1, rgb: 128|256 -> 3) on CUDA cores
//                 in fp32 and writes raw[row] = (sigmoid rgb, relu sigma) as one float4.
//   The MMA issuer alternates the two sub-tiles layer by layer, so the epilogue of one overlaps the
//   MMAs of the other.  Skip connections are extra K-chunks ([pe | h] for layers_pos.5,
//   [h | dir-enc] for layers_dir.1), zero-padded to the MMA K granularity in the packed weights.
//
// Algorithmic work: 1,182,976 FLOP per NeRF row (SURVEY 8d); issued (padded): 1,191,936 (+0.8 %).

#include "tc_core.cuh"

namespace b2r {
namespace tc {

// ---- pack kernels: fp32 state-dict parameters -> swizzled bf16 half-chunk images + fp32 tables ---------------
__global__ void nerf_pack_kernel(const float* __restrict__ params, uint8_t* __restrict__ packed) {
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t < kNerfChunkBytes / 16) {
        int s, c, hf, row, grp;
        locate<NerfSched>(t * 16, s, c, hf, row, grp);
        LayerDesc L = nerf_layer(s);                              // 0..7 trunk, 8 layers_dir.0, 9 layers_dir.1
        const int n = hf * (NerfSched::n(s) / 2) + row;           // output feature (weight row)
        __nv_bfloat16 v[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
            int kk = grp * 8 + e;                                 // 0..63 inside the chunk
            int col = -1;
            if (s == 0) col = kk < 60 ? kk : -1;
            else if (s == 5) col = c == 0 ? (kk < 60 ? kk : -1) : 60 + (c - 1) * 64 + kk;
            else if (s == 9) col = c < 4 ? c * 64 + kk : (kk < 24 ? 256 + kk : -1);
            else col = c * 64 + kk;
            v[e] = __float2bfloat16_rn(col >= 0 ? params[L.w_off + (long long)n * L.in + col] : 0.f);
        }
        uint8_t* dst = packed + step_base<NerfSched>(s) + (long long)(c * 2 + hf) * half_bytes<NerfSched>(s) +
                       sw128_offset((uint32_t)row, (uint32_t)grp);
        *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(v);
    }
    if (t < kNerfTabFloats) {
        float* tab = reinterpret_cast<float*>(packed + kNerfChunkBytes);
        int i = (int)t;
        float val = 0.f;
        if (i < kNerfTabWSigma) {
            int s = i / 256, n = i % 256;
            LayerDesc L = nerf_layer(s);
            val = n < L.out ? params[L.b_off + n] : 0.f;
        } else if (i < kNerfTabWRgb) val = params[nerf_layer(10).w_off + (i - kNerfTabWSigma)];
        else if (i < kNerfTabBHead) val = params[nerf_layer(11).w_off + (i - kNerfTabWRgb)];
        else if (i == kNerfTabBHead) val = params[nerf_layer(10).b_off];
        else val = params[nerf_layer(11).b_off + (i - kNerfTabBHead - 1)];
        tab[i] = val;
    }
}

// FiLM scale / shift of tensor-core step s (film row s + 1: 1..7 hidden, 8 rgb layer), column n:
//   sin(30 (gamma (W x + b) + beta)) = sin((30 gamma) W x + 30 (gamma b + beta))      (pi_GAN/modules.py:22-25)
__device__ __forceinline__ void film_scale_shift(const float* __restrict__ params, const float* __restrict__ film, bool ud, int s, int n,
                                                 float& scale, float& shift) {
    const int fl = s + 1;
    LayerDesc L = film_layer(s < 7 ? s + 1 : 9, ud);
    const float gm = film[fl * 512 + n], bt = film[fl * 512 + 256 + n], b = params[L.b_off + n];
    scale = 30.0f * gm;
    shift = 30.0f * (gm * b + bt);
}

// fp32 table entry i of a (weights, film) pair (layout kFW0 .. kFBH, tc_core.cuh)
__device__ __forceinline__ float film_table_value(const float* __restrict__ params, const float* __restrict__ film, bool ud, int i) {
    float val;
    if (i < kFS0) {
        // input_layer weights with the FiLM scale folded in: t_n = sum_k (30 gamma_n W_nk) p_k + shift_n (three fma per output)
        int k = (i - kFW0) / 256, n = (i - kFW0) % 256;
        val = (30.0f * film[n]) * params[film_layer(0, ud).w_off + n * 3 + k];
    } else if (i < kFT0) val = 30.0f * film[i - kFS0];
    else if (i < kFWS) { int n = i - kFT0; val = 30.0f * (film[n] * params[film_layer(0, ud).b_off + n] + film[256 + n]); }
    else if (i < kFWR) val = params[film_layer(8, ud).w_off + (i - kFWS)];
    else if (i < kFBH) val = params[film_layer(10, ud).w_off + (i - kFWR)];
    else if (i == kFBH) val = params[film_layer(8, ud).b_off];
    else val = params[film_layer(10, ud).b_off + (i - kFBH - 1)];
    return val;
}

// the 8 bf16 of 16-byte group `grp` of weight row n in chunk c (0..3: h columns c*64 + grp*8 ..; 4: the post chunk) of step s
__device__ __forceinline__ void film_pack_group(const float* __restrict__ params, const float* __restrict__ film, bool ud, int s, int c, int n, int grp,
                                                __nv_bfloat16 (&v)[8]) {
    LayerDesc L = film_layer(s < 7 ? s + 1 : 9, ud);           // hidden_layers.s | hidden_layer_rgb
    float scale, shift;
    film_scale_shift(params, film, ud, s, n, scale, shift);
    const __nv_bfloat16 sh_hi = __float2bfloat16_rn(shift);
    const __nv_bfloat16 sh_lo = __float2bfloat16_rn(shift - __bfloat162float(sh_hi));
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        int kk = grp * 8 + e;
        if (c < 4) v[e] = __float2bfloat16_rn(scale * params[L.w_off + (long long)n * L.in + c * 64 + kk]);
        else if (kk < 3) v[e] = __float2bfloat16_rn((s == 7 && ud) ? scale * params[L.w_off + (long long)n * L.in + 256 + kk] : 0.f);
        else if (kk == 3) v[e] = sh_hi;
        else if (kk == 4) v[e] = sh_lo;
        else v[e] = __float2bfloat16_rn(0.f);
    }
}

// blockIdx.y = latent: packed[latent] = chunks (bf16, rows pre-multiplied by the FiLM scale; post chunk = [W_dir(3) | shift hi | shift lo])
// + fp32 tables + the inference kernel's blobs.  film: [n_latents][9][512]
__global__ void film_pack_kernel(const float* __restrict__ params, const float* __restrict__ film_all, int use_dir,
                                 uint8_t* __restrict__ packed_all) {
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    const bool ud = use_dir != 0;
    const float* __restrict__ film = film_all + (size_t)blockIdx.y * B2R_FILM_PARAMS;
    uint8_t* __restrict__ packed = packed_all + (size_t)blockIdx.y * kFilmPackedBytes;
    if (t < kFilmChunkBytes / 16) {
        int s, c, hf, row, grp;
        locate<FilmSched>(t * 16, s, c, hf, row, grp);
        __nv_bfloat16 v[8];
        film_pack_group(params, film, ud, s, c, hf * 128 + row, grp, v);
        uint8_t* dst = packed + step_base<FilmSched>(s) + (long long)(c * 2 + hf) * half_bytes<FilmSched>(s) +
                       sw128_offset((uint32_t)row, (uint32_t)grp);
        *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(v);
    }
    if (t < (kFilmPackedBytes - kFilmExtraOff) / 16) {          // blobs [h chunk 3 | compact post chunk] of the inference kernel (tc_core.cuh)
        int s, c, hf, row, grp;
        locate_extra<FilmSched>(t * 16, s, c, hf, row, grp);
        __nv_bfloat16 v[8];
        film_pack_group(params, film, ud, s, c, hf * 128 + row, grp, v);
        *reinterpret_cast<uint4*>(packed + kFilmExtraOff + extra_dst<FilmSched>(s, c, hf, row, grp)) = *reinterpret_cast<const uint4*>(v);
    }
    if (t < kFilmTabFloats) {
        float* tab = reinterpret_cast<float*>(packed + kFilmChunkBytes);
        tab[t] = film_table_value(params, film, ud, (int)t);
    }
}

// One NeRF layer's epilogue for this warp's half of the columns, fully unrolled (no per-step branches in the hot loop).
//   MODE 0: + bias, ReLU -> bf16 h                       (layers_pos.0..6)
//   MODE 1: same + partial sigma head on the fp32 values  (layers_pos.7; output_layer_sigma, nerf/nerf.py:72,88)
//   MODE 2: + bias, linear -> bf16 h                      (layers_dir.0)
//   MODE 3: + bias, ReLU -> partial rgb head, no store    (layers_dir.1, N = 128; output_layer_rgb, nerf/nerf.py:73,93)
// t_half / bias_half / h_half already include this warp's column-half offset; xoff[c] = ((c ^ (row & 7)) << 4).
// kSave (training forward): the relu bits of every activation are gathered into mk[jj] (tc_core.cuh: mask_put) and MODE 3
// also writes relu(h_d) as bf16 into shared memory (block = this half at h_half), so that the spill thread can copy the
// tile to global memory with the bulk-copy engine.
// want_abs (MODE 1; warp-uniform: some row of this warp is the last sample of a ray and the sign check is on): asum += sum |w_sigma h|
// of this half (the scale of the bf16 error band, tc_core.cuh LastFlag); only warps that hold a ray's last sample pay for it.
template <int MODE, bool kSave>
__device__ __forceinline__ void nerf_epi(uint32_t t_half, uint32_t bias_half, uint32_t head_half, uint32_t h_half,
                                         const uint32_t (&xoff)[8], float& sigma, float& rgb0, float& rgb1, float& rgb2,
                                         uint32_t (&mk)[4], bool want_abs = false, float* asum = nullptr) {
    constexpr int NJH = MODE == 3 ? 2 : 4;
#pragma unroll
    for (int jj = 0; jj < NJH; ++jj) {
        uint32_t v[32];
        tmem_ld32(t_half + (uint32_t)jj * 32u, v);
        float4 b[8];
#pragma unroll
        for (int q = 0; q < 8; ++q) b[q] = lds128(bias_half + (uint32_t)(jj * 32 + q * 4) * 4u);     // overlaps the TMEM load
        tmem_ld_wait();
        float f[32];
#pragma unroll
        for (int q = 0; q < 8; ++q) {
            f[4 * q + 0] = __uint_as_float(v[4 * q + 0]); f[4 * q + 1] = __uint_as_float(v[4 * q + 1]);
            f[4 * q + 2] = __uint_as_float(v[4 * q + 2]); f[4 * q + 3] = __uint_as_float(v[4 * q + 3]);
            add2(f[4 * q + 0], f[4 * q + 1], b[q].x, b[q].y);
            add2(f[4 * q + 2], f[4 * q + 3], b[q].z, b[q].w);
        }
        if (MODE == 1) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                float4 w = lds128(head_half + (uint32_t)(jj * 32 + q * 4) * 4u);
                sigma = fmaf(fmaxf(f[4 * q + 0], 0.f), w.x, sigma);
                sigma = fmaf(fmaxf(f[4 * q + 1], 0.f), w.y, sigma);
                sigma = fmaf(fmaxf(f[4 * q + 2], 0.f), w.z, sigma);
                sigma = fmaf(fmaxf(f[4 * q + 3], 0.f), w.w, sigma);
            }
            if (want_abs) {                                         // separate pass: keeps the hot loop's register allocation
                float a = *asum;
#pragma unroll
                for (int q = 0; q < 8; ++q) {
                    float4 w = lds128(head_half + (uint32_t)(jj * 32 + q * 4) * 4u);
                    a = fmaf(fmaxf(f[4 * q + 0], 0.f), fabsf(w.x), a);
                    a = fmaf(fmaxf(f[4 * q + 1], 0.f), fabsf(w.y), a);
                    a = fmaf(fmaxf(f[4 * q + 2], 0.f), fabsf(w.z), a);
                    a = fmaf(fmaxf(f[4 * q + 3], 0.f), fabsf(w.w), a);
                }
                *asum = a;
            }
        }
        if (MODE == 3) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const uint32_t wa = head_half + (uint32_t)(jj * 32 + q * 4) * 4u;
                float4 w0 = lds128(wa), w1 = lds128(wa + 512u), w2 = lds128(wa + 1024u);
                float h0 = fmaxf(f[4 * q + 0], 0.f), h1 = fmaxf(f[4 * q + 1], 0.f);
                float h2 = fmaxf(f[4 * q + 2], 0.f), h3 = fmaxf(f[4 * q + 3], 0.f);
                rgb0 = fmaf(h0, w0.x, fmaf(h1, w0.y, fmaf(h2, w0.z, fmaf(h3, w0.w, rgb0))));
                rgb1 = fmaf(h0, w1.x, fmaf(h1, w1.y, fmaf(h2, w1.z, fmaf(h3, w1.w, rgb1))));
                rgb2 = fmaf(h0, w2.x, fmaf(h1, w2.y, fmaf(h2, w2.z, fmaf(h3, w2.w, rgb2))));
            }
            if (kSave) {                                            // HD tile: block = this half, chunks jj * 4 .. + 3
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const uint32_t w0 = pack_bf16_relu(f[8 * q + 0], f[8 * q + 1]), w1 = pack_bf16_relu(f[8 * q + 2], f[8 * q + 3]);
                    const uint32_t w2 = pack_bf16_relu(f[8 * q + 4], f[8 * q + 5]), w3 = pack_bf16_relu(f[8 * q + 6], f[8 * q + 7]);
                    mask_put(mk[jj], w0, 4 * q + 0); mask_put(mk[jj], w1, 4 * q + 1); mask_put(mk[jj], w2, 4 * q + 2); mask_put(mk[jj], w3, 4 * q + 3);
                    st_shared_v4(h_half + xoff[jj * 4 + q], w0, w1, w2, w3);
                }
            }
        } else {
            // columns of this 32-group = K of the next layer: K-block (jj >> 1) of this half, chunks (jj & 1) * 4 .. + 3
            const uint32_t blk = h_half + (uint32_t)(jj >> 1) * 16384u;
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                uint32_t w0, w1, w2, w3;
                if (MODE == 2) {
                    w0 = pack_bf16(f[8 * q + 0], f[8 * q + 1]); w1 = pack_bf16(f[8 * q + 2], f[8 * q + 3]);
                    w2 = pack_bf16(f[8 * q + 4], f[8 * q + 5]); w3 = pack_bf16(f[8 * q + 6], f[8 * q + 7]);
                } else {
                    w0 = pack_bf16_relu(f[8 * q + 0], f[8 * q + 1]); w1 = pack_bf16_relu(f[8 * q + 2], f[8 * q + 3]);
                    w2 = pack_bf16_relu(f[8 * q + 4], f[8 * q + 5]); w3 = pack_bf16_relu(f[8 * q + 6], f[8 * q + 7]);
                }
                st_shared_v4(blk + xoff[(jj & 1) * 4 + q], w0, w1, w2, w3);
                if (kSave && MODE != 2) {
                    mask_put(mk[jj], w0, 4 * q + 0); mask_put(mk[jj], w1, 4 * q + 1); mask_put(mk[jj], w2, 4 * q + 2); mask_put(mk[jj], w3, 4 * q + 3);
                }
            }
        }
    }
}

// ======================================================================================================
// NeRF (nerf/nerf.py:52-94)
// ======================================================================================================
// kSave = training forward: additionally keeps every layer input the reverse mode needs (pos-enc, h0..h7, layers_dir.0
// output, dir-enc, h_d) as tiled bf16 tensors in `saved` (5,120 B per row) plus one relu bit per activation (272 B per row).
// The tiles are already in shared memory as the next layer's A operand: warps 2 / 3 (one thread each, sub-tile 0 / 1) copy them
// out with the bulk-copy engine (64 KB per layer and sub-tile, full-line writes) while the next layer's MMAs run; the epilogue
// warps wait for "tile has been read" (spill_done) before they overwrite it in place.
// kSigmaOnly (inference): the walk stops after layers_pos.7 + the sigma head (steps 0..7); raw = (0, 0, 0, relu sigma).  For passes
// whose colour nobody reads -- the coarse pass of render_image, which returns the fine maps only (nerf/render.py:150-167) and needs
// the coarse weights, a function of sigma alone, for sample_pdf: sigma is bit-identical to the full walk's (same MMAs, same epilogue).
template <bool kSave, bool kSigmaOnly = false, bool kBox = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
nerf_tc_kernel(const uint8_t* __restrict__ packed, RowSource src, long long rows, float4* __restrict__ raw_out, uint8_t* __restrict__ saved,
               LastFlag lf) {
    static_assert(!(kSave && kSigmaOnly), "the training forward evaluates the whole network");
    constexpr int kWalk = kSigmaOnly ? 8 : NerfSched::kSteps;
    extern __shared__ uint8_t smem_raw[];
    const Ctx cx = make_ctx(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const PairLoop pl(rows);

    {   // bias / head-weight tables -> shared memory
        const float4* tab_g = reinterpret_cast<const float4*>(packed + kNerfChunkBytes);
        for (int i = threadIdx.x; i < kNerfTabFloats / 4; i += kThreads) {
            float4 v = __ldg(tab_g + i);
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(cx.smem + kTabOff + 16u * i), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
        }
    }
    const uint32_t tmem_base = tc_prologue(cx, warp);

    if (warp == 0) {
        if (lane == 0) producer_loop<NerfSched>(cx, packed, pl, kWalk, 0);
    } else if (warp == 1) {
        if (cx.rank == 0) mma_loop<NerfSched>(cx, tmem_base, pl, kWalk, 0);
        else if (lane == 0) relay_loop<NerfSched>(cx, pl, kWalk, 0);
    } else if (warp < kCtrlWarps) {
        if (kSave && lane == 0) {
            // ===== spill thread of sub-tile g: shared-memory tiles -> tiled tensors in global memory =====
            const int g = warp - 2;
            const uint32_t aux = cx.smem + (uint32_t)g * kSubBytes, hreg = aux + kPeBytes;
            const uint32_t ready = cx.spill_ready + 8 * g, done = cx.spill_done + 8 * g;
            const size_t n_sub = (size_t)pl.n_pairs * 4;
            uint32_t ph = 0;
            for (long long p = pl.first; p < pl.n_pairs; p += pl.stride) {
                const size_t T = (size_t)((2 * p + cx.rank) * 2 + g);
                auto tile = [&](int off, int nb) -> uint8_t* { return saved + ((size_t)off * n_sub + T * (size_t)nb) * kBlk; };
                auto finish = [&]() { bulk_commit(); bulk_wait_read(); mbar_arrive(done); ph ^= 1u; };
                mbar_wait(ready, ph); bulk_s2g(tile(kSavPE, 1), aux, kBlk); finish();                       // positional encoding
                for (int l = 0; l < 8; ++l) { mbar_wait(ready, ph); spill_tile(tile(sav_h(l), 4), hreg, 4); finish(); }   // h0 .. h7
                mbar_wait(ready, ph); spill_tile(tile(kSavGL, 4), hreg, 4); bulk_s2g(tile(kSavDE, 1), aux, kBlk); finish();   // g, dir-enc
                mbar_wait(ready, ph); spill_tile(tile(kSavHD, 2), hreg, 2); finish();                  // h_d
            }
            bulk_wait_all();
        }
    } else {
        // ===== input generation + epilogue =====
        // warp = 4 + g*8 + half*4 + quad;  thread = row (quad*32 + lane) of sub-tile g = TMEM lane;
        // `half` selects which half of the columns of every layer this warp converts.
        const int ew = warp - kCtrlWarps;
        const int g = ew >> 3, half = (ew >> 2) & 1, quad = ew & 3;
        const int r = (quad << 5) | lane;
        const uint32_t sub = cx.smem + (uint32_t)g * kSubBytes;
        const uint32_t pe_base = sub, h_base = sub + kPeBytes;
        const uint32_t t_addr = tmem_base + ((uint32_t)quad << 21) + (uint32_t)g * 256u;
        const uint32_t row_off = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u;   // SW128 row offset
        const uint32_t xr = (uint32_t)(r & 7);
        const uint32_t tab = cx.smem + kTabOff;
        const uint32_t part = cx.smem + kPartOff + (uint32_t)(g * kRowsSub + r) * 16u;
        const uint32_t part2 = cx.smem + kPart2Off + (uint32_t)(g * kRowsSub + r) * 4u;
        const uint32_t bar_id = 1 + g;                      // named barrier of this sub-tile's 8 warps
        const uint32_t act_local = cx.act_ready + 8 * g, act_leader = mapa(act_local, 0);
        const uint32_t acc_bar = cx.acc_full + 8 * g;
        // this warp's column half (N = 256 layers): TMEM columns, bias slice, destination K-blocks
        const uint32_t t_half = t_addr + (uint32_t)half * 128u;
        const uint32_t bias_half = tab + (uint32_t)(kNerfTabBias + half * 128) * 4u;
        const uint32_t h_half = h_base + row_off + (uint32_t)half * 2u * 16384u;
        uint32_t xoff[8];
#pragma unroll
        for (uint32_t c = 0; c < 8; ++c) xoff[c] = (c ^ xr) << 4;
        uint32_t acc_phase = 0, sp_phase = 0;
        bool first_tile = true;
        const size_t n_sub = (size_t)pl.n_pairs * 4;               // 128-row sub-tiles in the saved tensors
        for (long long p = pl.first; p < pl.n_pairs; p += pl.stride) {
            const long long row = (2 * p + cx.rank) * kRowsTile + g * kRowsSub + r;
            const bool valid = row < rows;
            const size_t T = (size_t)((2 * p + cx.rank) * 2 + g);
            // kSave: tile written (and fenced) -> spill thread; wait until the previous tile copy has read shared memory
            auto spill_sig = [&]() { if (kSave && lane == 0) mbar_arrive(cx.spill_ready + 8 * g); };
            auto spill_wait = [&]() { if (kSave) { mbar_wait(cx.spill_done + 8 * g, sp_phase); sp_phase ^= 1u; } };
            auto put_mask = [&](int l, const uint32_t (&mk)[4]) {
                if (kSave) *reinterpret_cast<uint4*>(saved + mask_off(n_sub, l, T, half, r)) = make_uint4(mk[0], mk[1], mk[2], mk[3]);
            };
            float pnt[3], vdir[3];
            long long ray = 0;
            load_row<kBox>(src, valid ? row : rows - 1, pnt, vdir, &ray);
            const bool check_last = valid && last_of_ray(lf, src, row, ray);      // this row decides its ray's last interval
            const bool warp_checks = __any_sync(0xffffffffu, check_last);
            float asum = 0.f;
            if (!first_tile) spill_wait();                          // previous tile's h_d copy
            first_tile = false;
            {
                // positional encoding: 60 values + 4 zero pads = 32 words = 8 chunks; this half writes 4 of them
                uint32_t pw[32];
                posenc_words<10>(pnt, pw);
                pw[30] = 0u; pw[31] = 0u;
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const uint32_t cidx = (uint32_t)(half * 4 + q);
                    uint32_t a0 = half ? pw[16 + 4 * q + 0] : pw[4 * q + 0];
                    uint32_t a1 = half ? pw[16 + 4 * q + 1] : pw[4 * q + 1];
                    uint32_t a2 = half ? pw[16 + 4 * q + 2] : pw[4 * q + 2];
                    uint32_t a3 = half ? pw[16 + 4 * q + 3] : pw[4 * q + 3];
                    st_shared_v4(pe_base + row_off + ((cidx ^ xr) << 4), a0, a1, a2, a3);
                }
            }
            arrive_act(act_local, act_leader, cx.rank, lane);
            spill_sig();

            float sigma = 0.f, rgb0 = 0.f, rgb1 = 0.f, rgb2 = 0.f;
            auto wait_acc = [&]() {
                mbar_wait_cluster(acc_bar, acc_phase);
                acc_phase ^= 1u;
                tc_fence_after();
            };
            for (int s = 0; s < 7; ++s) {                               // layers_pos.0 .. layers_pos.6
                wait_acc();
                spill_wait();
                uint32_t mk[4] = {0u, 0u, 0u, 0u};
                nerf_epi<0, kSave>(t_half, bias_half + (uint32_t)s * 1024u, 0u, h_half, xoff, sigma, rgb0, rgb1, rgb2, mk);
                arrive_act(act_local, act_leader, cx.rank, lane);
                spill_sig();
                put_mask(s, mk);
            }
            {
                wait_acc();                                             // layers_pos.7 (+ sigma head)
                spill_wait();
                uint32_t mk[4] = {0u, 0u, 0u, 0u};
                nerf_epi<1, kSave>(t_half, bias_half + 7u * 1024u, tab + (uint32_t)(kNerfTabWSigma + half * 128) * 4u, h_half, xoff, sigma, rgb0, rgb1, rgb2, mk,
                                   warp_checks, &asum);
                if (!kSigmaOnly) arrive_act(act_local, act_leader, cx.rank, lane);   // (sigma only: no MMA reads h7)
                spill_sig();
                put_mask(7, mk);
            }
            uint32_t mk[4] = {0u, 0u, 0u, 0u};
            if (!kSigmaOnly) {
            wait_acc();                                                 // layers_dir.0 (linear) + view-direction encoding
            spill_wait();
            nerf_epi<2, kSave>(t_half, bias_half + 8u * 1024u, 0u, h_half, xoff, sigma, rgb0, rgb1, rgb2, mk);
            {
                // layers_dir.1's extra K: 24 values + 8 zero pads = 16 words = chunks 0..3 of the aux block; each half writes two
                uint32_t dw[16];
                posenc_words<4>(vdir, dw);
                dw[12] = dw[13] = dw[14] = dw[15] = 0u;
#pragma unroll
                for (int q = 0; q < 2; ++q) {
                    uint32_t a0 = half ? dw[8 + 4 * q + 0] : dw[4 * q + 0];
                    uint32_t a1 = half ? dw[8 + 4 * q + 1] : dw[4 * q + 1];
                    uint32_t a2 = half ? dw[8 + 4 * q + 2] : dw[4 * q + 2];
                    uint32_t a3 = half ? dw[8 + 4 * q + 3] : dw[4 * q + 3];
                    st_shared_v4(pe_base + row_off + ((((uint32_t)(half * 2 + q)) ^ xr) << 4), a0, a1, a2, a3);
                    // DE tile kept for wgrad: chunks 0..3 = the encoding, 4..7 = zero
                    if (kSave) st_shared_v4(pe_base + row_off + ((((uint32_t)(4 + half * 2 + q)) ^ xr) << 4), 0u, 0u, 0u, 0u);
                }
            }
            arrive_act(act_local, act_leader, cx.rank, lane);
            spill_sig();
            wait_acc();                                                 // layers_dir.1 (N = 128) + rgb head
            spill_wait();
            nerf_epi<3, kSave>(tmem_base + ((uint32_t)quad << 21) + (uint32_t)g * 256u + (uint32_t)half * 64u,
                               tab + (uint32_t)(kNerfTabBias + 9 * 256 + half * 64) * 4u, tab + (uint32_t)(kNerfTabWRgb + half * 64) * 4u,
                               h_base + row_off + (uint32_t)half * kBlk, xoff, sigma, rgb0, rgb1, rgb2, mk);
            }
            if (kSave) {
                fence_proxy_async_smem();
                __syncwarp();
                spill_sig();
                *reinterpret_cast<uint2*>(saved + hdmask_off(n_sub, T, half, r)) = make_uint2(mk[0], mk[1]);
            }
            tc_fence_before();
            // combine the two halves' head partial sums and write raw[row] = (sigmoid rgb, relu sigma)
            if (half == 1) {
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(part), "f"(rgb0), "f"(rgb1), "f"(rgb2), "f"(sigma) : "memory");
                if (check_last) asm volatile("st.shared.f32 [%0], %1;" ::"r"(part2), "f"(asum) : "memory");
            }
            asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");
            if (half == 0) {
                float4 o2 = lds128(part);
                if (valid) {
                    float4 bh = lds128(tab + (uint32_t)kNerfTabBHead * 4u);      // (b_sigma, b_rgb[3])
                    float4 o;
                    o.x = 1.0f / (1.0f + __expf(-(rgb0 + o2.x + bh.y)));
                    o.y = 1.0f / (1.0f + __expf(-(rgb1 + o2.y + bh.z)));
                    o.z = 1.0f / (1.0f + __expf(-(rgb2 + o2.z + bh.w)));
                    if (kSigmaOnly) { o.x = 0.f; o.y = 0.f; o.z = 0.f; }
                    const float pre = sigma + o2.w + bh.x;
                    o.w = fmaxf(pre, 0.f);
                    raw_out[row] = o;
                    if (check_last) {
                        // sign(pre) is a step function of the ray's colour (nerf/render.py:92): inside the bf16 error band
                        // the fp32 path decides (b2r_mlp_f32_last_sigma)
                        float a2;
                        asm volatile("ld.shared.f32 %0, [%1];" : "=f"(a2) : "r"(part2));
                        if (fabsf(pre) <= fmaf(lf.rel, asum + a2, lf.abs)) flag_ray(lf, ray);
                    }
                }
            }
            asm volatile("bar.sync %0, 256;" ::"r"(bar_id) : "memory");         // partial slot reusable
        }
    }
    tc_teardown(tmem_base, warp);
}

// One FiLM-SIREN layer's epilogue for this warp's QUARTER of the columns (64 = one K-block of the next layer).  The FiLM
// scale is folded into the weight rows and the shift rides on the aux chunk, so the accumulator is the sine's argument:
//   MODE 0: sin(acc) -> bf16 h (hidden_layers.0..5);  MODE 1: -> bf16 h + partial sigma head (hidden_layers.6, modules.py:112);
//   MODE 2: -> partial rgb head, no store (hidden_layer_rgb, modules.py:114-116)
// t_q: TMEM address of the quarter; head: shared-memory address of the quarter's fp32 head weights; h_blk: this thread's row in
// the destination K-block.  No table loads in MODE 0: per element FMUL (1/2pi) + MUFU.SIN + half a bf16x2 pack.
// kSave (training forward): cos(acc) is stored as one byte per element, one uint4 per 16-column unit, thread-major at
// cosp + u * 2048 (tc_core.cuh: cos_q4, film_cos_off), and MODE 2 also writes its bf16 output into shared memory (h_blk) for the spill.
template <int MODE, bool kSave>
__device__ __forceinline__ void film_epi(uint32_t t_q, uint32_t head, uint32_t h_blk, const uint32_t (&xoff)[8], float& sigma, float& rgb0,
                                         float& rgb1, float& rgb2, uint8_t* __restrict__ cosp, bool write_h = true) {
    // 4 units of 16 columns, the TMEM load of unit u+1 in flight while unit u is evaluated
    uint32_t va[16], vb[16];
    tmem_ld16(t_q, va);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
        uint32_t (&v)[16] = (u & 1) ? vb : va;
        tmem_ld_wait();
        if (u < 3) tmem_ld16(t_q + (uint32_t)(u + 1) * 16u, (u & 1) ? va : vb);
        float f[16];
        sin16(v, f);
        if (kSave) {
            uint32_t cw[4];
#pragma unroll
            for (int e = 0; e < 4; ++e)
                cw[e] = cos_q4(__uint_as_float(v[4 * e]), __uint_as_float(v[4 * e + 1]), __uint_as_float(v[4 * e + 2]), __uint_as_float(v[4 * e + 3]));
            stg128(cosp + (size_t)u * 2048, cw[0], cw[1], cw[2], cw[3]);
        }
        if (MODE == 1) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                float4 w = lds128(head + (uint32_t)(u * 16 + q * 4) * 4u);
                sigma = fmaf(f[4 * q + 0], w.x, fmaf(f[4 * q + 1], w.y, fmaf(f[4 * q + 2], w.z, fmaf(f[4 * q + 3], w.w, sigma))));
            }
        }
        if (MODE == 2) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t wa = head + (uint32_t)(u * 16 + q * 4) * 4u;
                float4 w0 = lds128(wa), w1 = lds128(wa + 1024u), w2 = lds128(wa + 2048u);
                rgb0 = fmaf(f[4 * q + 0], w0.x, fmaf(f[4 * q + 1], w0.y, fmaf(f[4 * q + 2], w0.z, fmaf(f[4 * q + 3], w0.w, rgb0))));
                rgb1 = fmaf(f[4 * q + 0], w1.x, fmaf(f[4 * q + 1], w1.y, fmaf(f[4 * q + 2], w1.z, fmaf(f[4 * q + 3], w1.w, rgb1))));
                rgb2 = fmaf(f[4 * q + 0], w2.x, fmaf(f[4 * q + 1], w2.y, fmaf(f[4 * q + 2], w2.z, fmaf(f[4 * q + 3], w2.w, rgb2))));
            }
        }
        if ((MODE != 2 || kSave) && write_h) {               // (write_h = false: sigma_only's last step, nobody reads its h)
#pragma unroll
            for (int q = 0; q < 2; ++q)
                st_shared_v4(h_blk + xoff[u * 2 + q], pack_bf16(f[8 * q + 0], f[8 * q + 1]), pack_bf16(f[8 * q + 2], f[8 * q + 3]),
                             pack_bf16(f[8 * q + 4], f[8 * q + 5]), pack_bf16(f[8 * q + 6], f[8 * q + 7]));
        }
    }
}

// =====================================================================================================
// FiLM-SIREN (pi_GAN/modules.py:22-25, 70-118): sin(30 (gamma (W x + b) + beta)) layers.
//   input_layer (3 -> 256) runs on CUDA cores in fp32 inside the input stage (K = 3 is no GEMM and its 30x-amplified
//   argument must not see bf16 inputs; tables in shared memory); hidden_layers.0..6 and hidden_layer_rgb are tcgen05 steps
//   whose accumulator already is the sine's argument: the pack kernel folds scale = 30 gamma into the bf16 weight rows and
//   puts shift = 30 (gamma b + beta), split into two bf16 terms, on two extra K columns that meet constant ones in the aux
//   block [dir(3), 1, 1] (one 16-K MMA per step).  The sigma head (256 -> 1) rides on the epilogue of hidden_layers.6 and
//   the rgb head (256 -> 3) on the epilogue of hidden_layer_rgb, both fp32.
//   sigma_only (create_mesh, pi_GAN/utils.py:82-90) stops after hidden_layers.6: 919,552 FLOP per row.
// Per row the epilogue issues 2304 MUFU.SIN: the sine epilogue of a sub-tile is longer than its MMAs, so the 16 epilogue
// warps are NOT split between the two sub-tiles (as in nerf_tc_kernel, where a sub-tile's warps idle while its own MMAs
// run): every warp owns one 64-column quarter (= one K-block of the next layer) of BOTH sub-tiles and alternates between
// them, so that the epilogue of one sub-tile always overlaps the MMAs of the other and no warp waits for "its" MMA.
//
// Batched mode (Generator.forward's latent loop in one launch, pi_GAN/modules.py:176-184): n_latents > 1 packed images one
// after the other (b2r_mlp_tc_pack_film_batched); rows [b * rows_per_latent, (b+1) * rows_per_latent) belong to latent b
// (rows_per_latent is a multiple of the 512 rows of a CTA pair, which shares one set of weights); the producer streams the tile's latent's weights and the epilogue
// warps reload the small fp32 tables when their next tile is another latent's.
// kSave = training forward (one latent): tiles + cosine checkpoints for the reverse mode, as in siren_tc_kernel<true>.
template <bool kSave, bool kBox = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
film_tc_kernel(const uint8_t* __restrict__ packed, RowSource src, long long rows, int sigma_only, float4* __restrict__ raw_out,
               int n_latents, long long rows_per_latent, uint8_t* __restrict__ saved, LastFlag lf) {
    // inference (kSave = false): compact map -- 4 KB no-swizzle aux operand, 4-stage ring, 4 copies per step (tc_core.cuh MapC)
    constexpr bool kC = !kSave;
    constexpr uint32_t kSub = kC ? MapC::kSub : kSubBytes, kAux = kC ? MapC::kAux : kPeBytes;
    extern __shared__ uint8_t smem_raw[];
    const Ctx cx = kC ? make_ctx_c(smem_raw) : make_ctx(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const PairLoop pl(rows);
    const bool batched = n_latents > 1;
    auto latent_of = [&](long long p) -> long long { return batched ? ((2 * p + cx.rank) * kRowsTile) / rows_per_latent : 0; };
    auto packed_of = [&](long long p) -> const uint8_t* { return packed + (size_t)latent_of(p) * kFilmPackedBytes; };
    long long cur_lat = latent_of(pl.first < pl.n_pairs ? pl.first : 0);
    const int n_steps = sigma_only ? 7 : FilmSched::kSteps;
    static_assert(kFilmTabFloats * 4 <= (int)(kTabBytes + kPartBytes), "FiLM table region");
    const uint32_t tab = cx.smem + (kC ? MapC::kTab : kTabOff);   // fp32 tables of the current latent (9.2 KB)
    {
        const float4* tab_g = reinterpret_cast<const float4*>(packed + (size_t)cur_lat * kFilmPackedBytes + kFilmChunkBytes);
        for (int i = threadIdx.x; i < kFilmTabFloats / 4; i += kThreads) {
            float4 v = __ldg(tab_g + i);
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(tab + 16u * i), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
        }
    }
    if (kSave) {   // the aux blocks are copied out whole: their never-written chunks must not hold stale bits
        for (int i = threadIdx.x; i < 2 * (int)(kPeBytes / 16); i += kThreads) {
            const uint32_t gg = (uint32_t)i / (kPeBytes / 16), o = (uint32_t)i % (kPeBytes / 16);
            st_shared_v4(cx.smem + gg * kSubBytes + o * 16u, 0u, 0u, 0u, 0u);
        }
    }
    const uint32_t tmem_base = tc_prologue(cx, warp, 32, 16, kC ? MapC::kStagesC : kStages);  // act_ready: 16 warps x 2 CTAs arrive per sub-tile and step

    if (warp == 0) {
        if (lane == 0) {
            if (kC) producer_loop_c<FilmSched>(cx, packed_of, kFilmExtraOff, pl, n_steps);
            else producer_loop_fn<FilmSched>(cx, packed_of, pl, n_steps, 1);
        }
    } else if (warp == 1) {
        if (kC) {
            if (cx.rank == 0) mma_loop_c<FilmSched>(cx, tmem_base, pl, n_steps);
            else if (lane == 0) relay_loop_c(cx, pl, n_steps);
        } else {
            if (cx.rank == 0) mma_loop<FilmSched>(cx, tmem_base, pl, n_steps, 1);
            else if (lane == 0) relay_loop<FilmSched>(cx, pl, n_steps, 1);
        }
    } else if (warp < kCtrlWarps) {
        if (kSave && lane == 0) {
            // ===== spill thread of sub-tile g =====
            const int g = warp - 2;
            const uint32_t aux = cx.smem + (uint32_t)g * kSubBytes, hreg = aux + kPeBytes;
            const uint32_t ready = cx.spill_ready + 8 * g, done = cx.spill_done + 8 * g;
            const size_t n_sub = (size_t)pl.n_pairs * 4;
            uint32_t ph = 0;
            for (long long p = pl.first; p < pl.n_pairs; p += pl.stride) {
                const size_t T = (size_t)((2 * p + cx.rank) * 2 + g);
                auto tile = [&](int off, int nb) -> uint8_t* { return saved + ((size_t)off * n_sub + T * (size_t)nb) * kBlk; };
                auto finish = [&]() { bulk_commit(); bulk_wait_read(); mbar_arrive(done); ph ^= 1u; };
                mbar_wait(ready, ph); bulk_s2g(tile(kFsAUX, 1), aux, kBlk); spill_tile(tile(fs_h(0), 4), hreg, 4); finish();    // aux, h0
                for (int l = 1; l < 8; ++l) { mbar_wait(ready, ph); spill_tile(tile(fs_h(l), 4), hreg, 4); finish(); }             // h1 .. h7
                mbar_wait(ready, ph); spill_tile(tile(kFsHC, 4), hreg, 4); finish();                                                // hidden_layer_rgb output
            }
            bulk_wait_all();
        }
    } else {
        // warp = 4 + cq*4 + quad: column quarter cq (64 columns = K-block cq), TMEM lane quadrant quad; thread = row r of BOTH sub-tiles
        const int ew = warp - kCtrlWarps;
        const int cq = ew >> 2, quad = ew & 3;
        const int r = (quad << 5) | lane;
        const uint32_t row_off = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u;
        const uint32_t xr = (uint32_t)(r & 7);
        const uint32_t act_leader0 = mapa(cx.act_ready, 0);
        uint32_t xoff[8];
#pragma unroll
        for (uint32_t c = 0; c < 8; ++c) xoff[c] = (c ^ xr) << 4;
        uint32_t acc_phase[2] = {0u, 0u}, sp_phase[2] = {0u, 0u};
        bool first_tile = true;
        const size_t n_sub = (size_t)pl.n_pairs * 4;
        // last-sample sign check (tc_core.cuh LastFlag): sine outputs are bounded by 1, so the error band of sigma_pre scales with
        // |w_sigma|_1 (the same for every latent: FiLM only modulates the hidden layers)
        float wl1 = 0.f;
        if (lf.count && cq < 2) {
            for (int i = 0; i < 64; ++i) {
                const float4 w = lds128(tab + (uint32_t)(kFWS + 4 * i) * 4u);
                wl1 += (fabsf(w.x) + fabsf(w.y)) + (fabsf(w.z) + fabsf(w.w));
            }
        }
        auto spill_sig = [&](int g) { if (kSave && lane == 0) mbar_arrive(cx.spill_ready + 8 * g); };
        auto spill_wait = [&](int g) { if (kSave) { mbar_wait(cx.spill_done + 8 * g, sp_phase[g]); sp_phase[g] ^= 1u; } };
        auto sub_base = [&](int g) -> uint32_t { return cx.smem + (uint32_t)g * kSub; };
        auto t_q = [&](int g) -> uint32_t { return tmem_base + ((uint32_t)quad << 21) + (uint32_t)g * 256u + (uint32_t)cq * 64u; };
        auto h_blk = [&](int g) -> uint32_t { return sub_base(g) + kAux + (uint32_t)cq * 16384u + row_off; };
        // head partials part[g][r][cq] (float4): upper half of the 16 KB aux block / first K-block of h on the compact map -- both free
        // once the sub-tile's last MMA is done
        auto part_of = [&](int g) -> uint32_t { return sub_base(g) + (kC ? kAux : 8192u); };
        auto arrive = [&](int g) { arrive_act(cx.act_ready + 8 * g, act_leader0 + 8 * g, cx.rank, lane); };
        auto wait_acc = [&](int g) {
            mbar_wait_cluster(cx.acc_full + 8 * g, acc_phase[g]);
            acc_phase[g] ^= 1u;
            tc_fence_after();
        };
        for (long long p = pl.first; p < pl.n_pairs; p += pl.stride) {
            if (batched) {
                const long long lat = latent_of(p);
                if (lat != cur_lat) {
                    // another latent: all 16 epilogue warps are done with the old tables, then reload them (9.2 KB)
                    cur_lat = lat;
                    asm volatile("bar.sync 3, 512;" ::: "memory");
                    const float4* tab_g = reinterpret_cast<const float4*>(packed + (size_t)lat * kFilmPackedBytes + kFilmChunkBytes);
                    for (int i = threadIdx.x - kCtrlWarps * 32; i < kFilmTabFloats / 4; i += kEpiWarps * 32) {
                        float4 v = __ldg(tab_g + i);
                        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(tab + 16u * i), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
                    }
                    asm volatile("bar.sync 3, 512;" ::: "memory");
                }
            }
            bool valid[2], chk[2];
            long long row[2];
            int ray[2];
#pragma unroll
            for (int g = 0; g < 2; ++g) {
                row[g] = (2 * p + cx.rank) * kRowsTile + g * kRowsSub + r;
                valid[g] = row[g] < rows;
                float pnt[3], vdir[3];
                long long ray_ll = 0;
                load_row<kBox>(src, valid[g] ? row[g] : rows - 1, pnt, vdir, &ray_ll);
                chk[g] = valid[g] && last_of_ray(lf, src, row[g], ray_ll);
                ray[g] = (int)ray_ll;
                if (!first_tile) spill_wait(g);                      // previous tile's last copy
                const size_t T = (size_t)((2 * p + cx.rank) * 2 + g);
                // ---- input_layer on CUDA cores: this warp produces columns cq*64 .. +63 of h0 (K-block cq)
if constexpr (kC) {
                    // column-owned form (tc_core.cuh sine_input_layer): the table stays in registers, positions come by shuffle
                    sine_input_layer(tab + kFW0 * 4u, tab + kFT0 * 4u, sub_base(g) + kAux + (uint32_t)cq * 16384u, cq, quad, lane, pnt);
                } else {
    #pragma unroll
                    for (int jj = 0; jj < 2; ++jj) {
                        uint32_t pk[16], ck[8];
    #pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const uint32_t n0 = (uint32_t)(cq * 64 + jj * 32 + q * 4) * 4u;
                            const float4 wx = lds128(tab + kFW0 * 4u + n0), wy = lds128(tab + (kFW0 + 256) * 4u + n0), wz = lds128(tab + (kFW0 + 512) * 4u + n0);
                            const float4 sh = lds128(tab + kFT0 * 4u + n0);
                            // scale folded into the table's weights: 3 packed fma per pair of outputs (the input stage is issue-bound)
                            float t0, t1, t2, t3;
                            ffma2(t0, t1, wx.x, wx.y, pnt[0], sh.x, sh.y);
                            ffma2(t2, t3, wx.z, wx.w, pnt[0], sh.z, sh.w);
                            ffma2(t0, t1, wy.x, wy.y, pnt[1], t0, t1);
                            ffma2(t2, t3, wy.z, wy.w, pnt[1], t2, t3);
                            ffma2(t0, t1, wz.x, wz.y, pnt[2], t0, t1);
                            ffma2(t2, t3, wz.z, wz.w, pnt[2], t2, t3);
                            pk[2 * q + 0] = pack_bf16(__sinf(t0), __sinf(t1));
                            pk[2 * q + 1] = pack_bf16(__sinf(t2), __sinf(t3));
                            if (kSave) ck[q] = cos_q4(t0, t1, t2, t3);
                        }
    #pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            st_shared_v4(h_blk(g) + xoff[jj * 4 + q], pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
                            if (kSave && q < 2) stg128(saved + film_cos_off(n_sub, 0, T, cq, jj * 2 + q, r), ck[4 * q], ck[4 * q + 1], ck[4 * q + 2], ck[4 * q + 3]);
                        }
                    }
                }
                if (cq == 0) {
                    // aux block = [view direction (3), 1, 1, position (3), 0 ...] (16 K): the direction columns of hidden_layer_rgb and the
                    // two constant ones that pick up every layer's FiLM shift (hi + lo); the position columns meet zero weights in the
                    // forward and are the input-layer operand of the training wgrad
                    // (compact map: 16-byte K chunk c of row r at c * 2 KB + r * 16, no swizzle)
                    st_shared_v4(sub_base(g) + (kC ? (uint32_t)r * 16u : row_off + ((0u ^ xr) << 4)), pack_bf16(vdir[0], vdir[1]), pack_bf16(vdir[2], 1.0f),
                                 pack_bf16(1.0f, pnt[0]), pack_bf16(pnt[1], pnt[2]));
                    st_shared_v4(sub_base(g) + (kC ? 2048u + (uint32_t)r * 16u : row_off + ((1u ^ xr) << 4)), 0u, 0u, 0u, 0u);
                }
                arrive(g);
                spill_sig(g);
            }
            first_tile = false;
            auto cosp = [&](int layer, int g) -> uint8_t* {
                return kSave ? saved + film_cos_off(n_sub, layer, (size_t)((2 * p + cx.rank) * 2 + g), cq, 0, r) : nullptr;
            };

            float sigma[2] = {0.f, 0.f}, rgb0[2] = {0.f, 0.f}, rgb1[2] = {0.f, 0.f}, rgb2[2] = {0.f, 0.f};
            for (int s = 0; s < 6; ++s) {                               // hidden_layers.0 .. 5
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    wait_acc(g);
                    spill_wait(g);
                    film_epi<0, kSave>(t_q(g), 0u, h_blk(g), xoff, sigma[g], rgb0[g], rgb1[g], rgb2[g], cosp(s + 1, g));
                    arrive(g);
                    spill_sig(g);
                }
            }
#pragma unroll
            for (int g = 0; g < 2; ++g) {                               // hidden_layers.6 (+ sigma head)
                wait_acc(g);
                spill_wait(g);
                film_epi<1, kSave>(t_q(g), tab + (uint32_t)(kFWS + cq * 64) * 4u, h_blk(g), xoff, sigma[g], rgb0[g], rgb1[g], rgb2[g], cosp(7, g),
                                   kSave || !sigma_only);
                if (!sigma_only) { arrive(g); spill_sig(g); }
            }
            if (!sigma_only) {
#pragma unroll
                for (int g = 0; g < 2; ++g) {                           // hidden_layer_rgb (+ rgb head)
                    wait_acc(g);
                    spill_wait(g);
                    film_epi<2, kSave>(t_q(g), tab + (uint32_t)(kFWR + cq * 64) * 4u, h_blk(g), xoff, sigma[g], rgb0[g], rgb1[g], rgb2[g], cosp(8, g));
                    if (kSave) {
                        fence_proxy_async_smem();
                        __syncwarp();
                        spill_sig(g);
                    }
                }
            }
            tc_fence_before();
            // head partials of the four column quarters (part_of):
            // (compact map: the slots overlay h, which sigma_only's last epilogue still writes -- every warp must be past it)
            if (kC) asm volatile("bar.sync 3, 512;" ::: "memory");
            // part[g][r][cq] as float4; the quarter-0 / quarter-1 warps finish sub-tile 0 / 1
#pragma unroll
            for (int g = 0; g < 2; ++g)
                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(part_of(g) + (uint32_t)(r * 4 + cq) * 16u), "f"(rgb0[g]),
                             "f"(rgb1[g]), "f"(rgb2[g]), "f"(sigma[g]) : "memory");
            asm volatile("bar.sync 3, 512;" ::: "memory");
            if (cq < 2) {
                const int g = cq;
                const bool ok = cq == 0 ? valid[0] : valid[1];
                const long long out_row = cq == 0 ? row[0] : row[1];
                const uint32_t pa = part_of(g) + (uint32_t)(r * 4) * 16u;
                const float4 p0 = lds128(pa), p1 = lds128(pa + 16u), p2 = lds128(pa + 32u), p3 = lds128(pa + 48u);
                if (ok) {
                    const float4 bh = lds128(tab + kFBH * 4u);          // (b_sigma, b_rgb[3])
                    float4 o;
                    if (sigma_only) { o.x = o.y = o.z = 0.f; }
                    else {
                        o.x = 1.0f / (1.0f + __expf(-((p0.x + p1.x) + (p2.x + p3.x) + bh.y)));
                        o.y = 1.0f / (1.0f + __expf(-((p0.y + p1.y) + (p2.y + p3.y) + bh.z)));
                        o.z = 1.0f / (1.0f + __expf(-((p0.z + p1.z) + (p2.z + p3.z) + bh.w)));
                    }
                    const float pre = (p0.w + p1.w) + (p2.w + p3.w) + bh.x;
                    o.w = fmaxf(pre, 0.f);
                    raw_out[out_row] = o;
                    if ((cq == 0 ? chk[0] : chk[1]) && fabsf(pre) <= fmaf(lf.rel, wl1, lf.abs)) flag_ray(lf, cq == 0 ? ray[0] : ray[1]);
                }
            }
            asm volatile("bar.sync 3, 512;" ::: "memory");         // partial slots (and the aux rows they overlay) reusable
        }
    }
    tc_teardown(tmem_base, warp);
}

}  // namespace tc
}  // namespace b2r

namespace b2r {
namespace tc {
// SirenNeRF (mlp_tc_siren.cu)
size_t siren_packed_bytes();
int siren_pack(const float* params, void* packed_out, cudaStream_t st);
int siren_fwd(const void* packed, const b2r_mlp_input* in, long long rows, float* raw_out, const b2r_last_sample* last, cudaStream_t st);
size_t siren_saved_bytes(long long rows);
int siren_train_fwd(const void* packed, const b2r_mlp_input* in, long long rows, float* raw_out, void* saved, const b2r_last_sample* last, cudaStream_t st);
}  // namespace tc
}  // namespace b2r

extern "C" size_t b2r_mlp_tc_packed_bytes(int model_kind) {
    if (model_kind == B2R_MODEL_SIREN) return b2r::tc::siren_packed_bytes();
    if (model_kind == B2R_MODEL_NERF) return (size_t)b2r::tc::kNerfPackedBytes;
    if (model_kind == B2R_MODEL_FILM) return (size_t)b2r::tc::kFilmPackedBytes;
    return 0;
}

extern "C" int b2r_mlp_tc_pack(int model_kind, const float* params, const float* film, int use_dir,
                               void* packed_out, void* stream) {
    using namespace b2r;
    B2R_CHECK_ARG(params && packed_out, "b2r_mlp_tc_pack: NULL pointer");
    B2R_CHECK_ARG(((uintptr_t)packed_out & 15) == 0, "b2r_mlp_tc_pack: packed_out must be 16-byte aligned");
    if (model_kind == B2R_MODEL_NERF) {
        long long threads = tc::kNerfChunkBytes / 16;
        tc::nerf_pack_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, (cudaStream_t)stream>>>(params, (uint8_t*)packed_out);
        B2R_LAUNCH_CHECK("b2r_mlp_tc_pack");
        return 0;
    }
    if (model_kind == B2R_MODEL_FILM) {
        B2R_CHECK_ARG(film, "b2r_mlp_tc_pack: FiLM model needs film params");
        long long threads = tc::kFilmChunkBytes / 16;
        tc::film_pack_kernel<<<dim3((unsigned)((threads + 255) / 256), 1), 256, 0, (cudaStream_t)stream>>>(params, film, use_dir, (uint8_t*)packed_out);
        B2R_LAUNCH_CHECK("b2r_mlp_tc_pack");
        return 0;
    }
    if (model_kind == B2R_MODEL_SIREN) return tc::siren_pack(params, packed_out, (cudaStream_t)stream);
    return fail(-2, "b2r_mlp_tc_pack: unknown model kind %d", model_kind);
}

namespace b2r {
namespace tc {
// grid of a fused-MLP launch: one CTA pair per two SMs; a pair walks tile pairs (2 x 256 rows)
int pair_grid(long long rows, unsigned* grid) {
    int dev = 0, sms = 0;
    int rc = cuda_result(cudaGetDevice(&dev), "cudaGetDevice");
    if (rc) return rc;
    rc = cuda_result(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev), "SM count");
    if (rc) return rc;
    long long n_tiles = (rows + kRowsTile - 1) / kRowsTile;
    long long n_pairs = (n_tiles + 1) / 2;
    long long clusters = sms / 2 < n_pairs ? sms / 2 : n_pairs;
    *grid = (unsigned)(2 * clusters);
    return 0;
}
}  // namespace tc
}  // namespace b2r

namespace b2r {
namespace tc {
int check_last_sample(const b2r_last_sample* last, const b2r_mlp_input* in, const char* who) {
    if (!last) return 0;
    B2R_CHECK_ARG(last->count && last->ray_ids && last->capacity >= 0, "%s: last-sample check needs count / ray_ids", who);
    B2R_CHECK_ARG(in->grid_n == 0 && !lattice_mode(in), "%s: the last-sample check is for rays / x rows, not grid queries", who);
    B2R_CHECK_ARG(last->samples_per_ray >= 1 && (!in->rays || last->samples_per_ray == in->n_samples),
                  "%s: samples_per_ray (%d) must equal n_samples in rays mode", who, last->samples_per_ray);
    B2R_CHECK_ARG(last->rel >= 0.f && last->abs >= 0.f, "%s: negative last-sample thresholds", who);
    return 0;
}
}  // namespace tc
}  // namespace b2r

extern "C" int b2r_mlp_tc_fwd(int model_kind, const void* packed, int use_dir, const b2r_mlp_input* in, float* raw_out,
                              int sigma_only, const b2r_last_sample* last, void* stream) {
    using namespace b2r;
    B2R_CHECK_ARG(packed && raw_out, "b2r_mlp_tc_fwd: NULL pointer");
    B2R_CHECK_ARG((((uintptr_t)packed | (uintptr_t)raw_out) & 15) == 0, "b2r_mlp_tc_fwd: packed / raw_out must be 16-byte aligned");
    int rc = check_mlp_input(in);
    if (rc) return rc;
    long long rows = row_count(in);
    if (rows == 0) return 0;
    B2R_CHECK_ARG(model_kind == B2R_MODEL_NERF || model_kind == B2R_MODEL_FILM || model_kind == B2R_MODEL_SIREN, "b2r_mlp_tc_fwd: unknown model kind %d", model_kind);
    B2R_CHECK_ARG(!(sigma_only && model_kind == B2R_MODEL_SIREN), "b2r_mlp_tc_fwd: sigma_only is a NeRF / FiLM-SIREN mode");
    rc = tc::check_last_sample(last, in, "b2r_mlp_tc_fwd");
    if (rc) return rc;
    if (model_kind == B2R_MODEL_SIREN) return tc::siren_fwd(packed, in, rows, raw_out, last, (cudaStream_t)stream);
    unsigned grid = 0;
    rc = tc::pair_grid(rows, &grid);
    if (rc) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    // box-lattice rows run their own instantiations, so the index arithmetic they need costs the other modes nothing
    const bool box = lattice_mode(in);
    if (model_kind == B2R_MODEL_FILM) {
        auto kern = box ? tc::film_tc_kernel<false, true> : tc::film_tc_kernel<false>;
        rc = cuda_result(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::MapC::kSmem), "tc smem attribute");
        if (rc) return rc;
        kern<<<grid, tc::kThreads, tc::MapC::kSmem, st>>>((const uint8_t*)packed, make_row_source(in), rows, sigma_only, (float4*)raw_out, 1, 0, nullptr,
                                                          tc::make_last_flag(last));
    } else {
        auto kern = box ? (sigma_only ? tc::nerf_tc_kernel<false, true, true> : tc::nerf_tc_kernel<false, false, true>)
                        : (sigma_only ? tc::nerf_tc_kernel<false, true> : tc::nerf_tc_kernel<false, false>);
        rc = cuda_result(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::kSmemBytes), "tc smem attribute");
        if (rc) return rc;
        kern<<<grid, tc::kThreads, tc::kSmemBytes, st>>>((const uint8_t*)packed, make_row_source(in), rows, (float4*)raw_out, nullptr, tc::make_last_flag(last));
    }
    B2R_LAUNCH_CHECK("b2r_mlp_tc_fwd");
    return 0;
}

extern "C" int b2r_mlp_tc_pack_film_batched(const float* params, const float* film, int use_dir, int n_latents, void* packed_out, void* stream) {
    using namespace b2r;
    B2R_CHECK_ARG(params && film && packed_out, "b2r_mlp_tc_pack_film_batched: NULL pointer");
    B2R_CHECK_ARG(((uintptr_t)packed_out & 15) == 0, "b2r_mlp_tc_pack_film_batched: packed_out must be 16-byte aligned");
    B2R_CHECK_ARG(n_latents >= 0 && n_latents <= 65535, "b2r_mlp_tc_pack_film_batched: n_latents out of range");
    if (n_latents == 0) return 0;
    long long threads = tc::kFilmChunkBytes / 16;
    tc::film_pack_kernel<<<dim3((unsigned)((threads + 255) / 256), (unsigned)n_latents), 256, 0, (cudaStream_t)stream>>>(params, film, use_dir,
                                                                                                                  (uint8_t*)packed_out);
    B2R_LAUNCH_CHECK("b2r_mlp_tc_pack_film_batched");
    return 0;
}

extern "C" int b2r_mlp_tc_fwd_film_batched(const void* packed, int n_latents, long long rows_per_latent, const b2r_mlp_input* in, float* raw_out,
                                           int sigma_only, const b2r_last_sample* last, void* stream) {
    using namespace b2r;
    B2R_CHECK_ARG(packed && raw_out, "b2r_mlp_tc_fwd_film_batched: NULL pointer");
    B2R_CHECK_ARG((((uintptr_t)packed | (uintptr_t)raw_out) & 15) == 0, "b2r_mlp_tc_fwd_film_batched: buffers must be 16-byte aligned");
    int rc = check_mlp_input(in);
    if (rc) return rc;
    long long rows = row_count(in);
    B2R_CHECK_ARG(!lattice_mode(in), "b2r_mlp_tc_fwd_film_batched: box-lattice rows go to b2r_mlp_tc_fwd");
    // a CTA pair (2 x 256 rows) shares one set of weights: both of its tiles must belong to the same latent
    B2R_CHECK_ARG(rows_per_latent > 0 && rows_per_latent % (2 * tc::kRowsTile) == 0,
                  "b2r_mlp_tc_fwd_film_batched: rows_per_latent (%lld) must be a positive multiple of %d", rows_per_latent, 2 * tc::kRowsTile);
    B2R_CHECK_ARG(n_latents >= 1 && rows <= rows_per_latent * (long long)n_latents, "b2r_mlp_tc_fwd_film_batched: %lld rows need more than %d latents", rows, n_latents);
    if (rows == 0) return 0;
    rc = tc::check_last_sample(last, in, "b2r_mlp_tc_fwd_film_batched");
    if (rc) return rc;
    unsigned grid = 0;
    rc = tc::pair_grid(rows, &grid);
    if (rc) return rc;
    rc = cuda_result(cudaFuncSetAttribute(tc::film_tc_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::MapC::kSmem), "tc smem attribute");
    if (rc) return rc;
    // n_latents == 1 still goes through the batched indexing (latent 0 for every row) when rows_per_latent covers all rows
    tc::film_tc_kernel<false><<<grid, tc::kThreads, tc::MapC::kSmem, (cudaStream_t)stream>>>((const uint8_t*)packed, make_row_source(in), rows, sigma_only,
                                                                                            (float4*)raw_out, n_latents, rows_per_latent, nullptr,
                                                                                            tc::make_last_flag(last));
    B2R_LAUNCH_CHECK("b2r_mlp_tc_fwd_film_batched");
    return 0;
}

extern "C" int b2r_mlp_tc_train_fwd_film_batched(const void* packed, int n_latents, long long rows_per_latent, const b2r_mlp_input* in,
                                                 float* raw_out, void* saved, size_t saved_bytes, const b2r_last_sample* last, void* stream) {
    using namespace b2r;
    B2R_CHECK_ARG(packed && raw_out && saved, "b2r_mlp_tc_train_fwd_film_batched: NULL pointer");
    B2R_CHECK_ARG((((uintptr_t)packed | (uintptr_t)raw_out | (uintptr_t)saved) & 15) == 0, "b2r_mlp_tc_train_fwd_film_batched: buffers must be 16-byte aligned");
    int rc = check_mlp_input(in);
    if (rc) return rc;
    long long rows = row_count(in);
    B2R_CHECK_ARG(!lattice_mode(in), "b2r_mlp_tc_train_fwd_film_batched: box-lattice rows are for inference");
    B2R_CHECK_ARG(rows_per_latent > 0 && rows_per_latent % (2 * tc::kRowsTile) == 0,
                  "b2r_mlp_tc_train_fwd_film_batched: rows_per_latent (%lld) must be a positive multiple of %d", rows_per_latent, 2 * tc::kRowsTile);
    B2R_CHECK_ARG(n_latents >= 1 && rows <= rows_per_latent * (long long)n_latents, "b2r_mlp_tc_train_fwd_film_batched: %lld rows need more than %d latents", rows, n_latents);
    B2R_CHECK_ARG(saved_bytes >= b2r_mlp_tc_train_saved_bytes(B2R_MODEL_FILM, rows), "b2r_mlp_tc_train_fwd_film_batched: saved buffer too small (%zu B)", saved_bytes);
    if (rows == 0) return 0;
    rc = tc::check_last_sample(last, in, "b2r_mlp_tc_train_fwd_film_batched");
    if (rc) return rc;
    unsigned grid = 0;
    rc = tc::pair_grid(rows, &grid);
    if (rc) return rc;
    rc = cuda_result(cudaFuncSetAttribute(tc::film_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::kSmemBytes), "tc smem attribute");
    if (rc) return rc;
    tc::film_tc_kernel<true><<<grid, tc::kThreads, tc::kSmemBytes, (cudaStream_t)stream>>>((const uint8_t*)packed, make_row_source(in), rows, 0,
                                                                                           (float4*)raw_out, n_latents, rows_per_latent, (uint8_t*)saved,
                                                                                           tc::make_last_flag(last));
    B2R_LAUNCH_CHECK("b2r_mlp_tc_train_fwd_film_batched");
    return 0;
}

extern "C" size_t b2r_mlp_tc_train_saved_bytes(int model_kind, long long rows) {
    if (model_kind == B2R_MODEL_SIREN && rows >= 0) return b2r::tc::siren_saved_bytes(rows);
    if (model_kind == B2R_MODEL_FILM && rows >= 0) return (size_t)b2r::tc::n_sub_tiles(rows) * b2r::tc::film_saved_bytes_per_sub();
    if (model_kind != B2R_MODEL_NERF || rows < 0) return 0;
    return (size_t)b2r::tc::n_sub_tiles(rows) * b2r::tc::saved_bytes_per_sub();
}

extern "C" int b2r_mlp_tc_train_fwd(int model_kind, const void* packed, const b2r_mlp_input* in, float* raw_out, void* saved,
                                    size_t saved_bytes, const b2r_last_sample* last, void* stream) {
    using namespace b2r;
    B2R_CHECK_ARG(model_kind == B2R_MODEL_NERF || model_kind == B2R_MODEL_SIREN || model_kind == B2R_MODEL_FILM,
                  "b2r_mlp_tc_train_fwd: unknown model kind %d", model_kind);
    B2R_CHECK_ARG(packed && raw_out && saved, "b2r_mlp_tc_train_fwd: NULL pointer");
    B2R_CHECK_ARG((((uintptr_t)packed | (uintptr_t)raw_out | (uintptr_t)saved) & 15) == 0, "b2r_mlp_tc_train_fwd: buffers must be 16-byte aligned");
    int rc = check_mlp_input(in);
    if (rc) return rc;
    long long rows = row_count(in);
    B2R_CHECK_ARG(!lattice_mode(in), "b2r_mlp_tc_train_fwd: box-lattice rows are for inference");
    B2R_CHECK_ARG(saved_bytes >= b2r_mlp_tc_train_saved_bytes(model_kind, rows), "b2r_mlp_tc_train_fwd: saved buffer too small (%zu B)", saved_bytes);
    if (rows == 0) return 0;
    rc = tc::check_last_sample(last, in, "b2r_mlp_tc_train_fwd");
    if (rc) return rc;
    if (model_kind == B2R_MODEL_SIREN) return tc::siren_train_fwd(packed, in, rows, raw_out, saved, last, (cudaStream_t)stream);
    if (model_kind == B2R_MODEL_FILM) {                 // packed = one latent's image (use_dir = 1 layout)
        unsigned fgrid = 0;
        rc = tc::pair_grid(rows, &fgrid);
        if (rc) return rc;
        rc = cuda_result(cudaFuncSetAttribute(tc::film_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::kSmemBytes), "tc smem attribute");
        if (rc) return rc;
        tc::film_tc_kernel<true><<<fgrid, tc::kThreads, tc::kSmemBytes, (cudaStream_t)stream>>>((const uint8_t*)packed, make_row_source(in), rows, 0,
                                                                                               (float4*)raw_out, 1, 0, (uint8_t*)saved, tc::make_last_flag(last));
        B2R_LAUNCH_CHECK("b2r_mlp_tc_train_fwd (FiLM-SIREN)");
        return 0;
    }
    unsigned grid = 0;
    rc = tc::pair_grid(rows, &grid);
    if (rc) return rc;
    rc = cuda_result(cudaFuncSetAttribute(tc::nerf_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)tc::kSmemBytes), "tc smem attribute");
    if (rc) return rc;
    tc::nerf_tc_kernel<true><<<grid, tc::kThreads, tc::kSmemBytes, (cudaStream_t)stream>>>((const uint8_t*)packed, make_row_source(in), rows,
                                                                                           (float4*)raw_out, (uint8_t*)saved, tc::make_last_flag(last));
    B2R_LAUNCH_CHECK("b2r_mlp_tc_train_fwd");
    return 0;
}
