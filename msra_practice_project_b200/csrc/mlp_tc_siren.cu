// K3 for SirenNeRF (nerf/nerf.py:97-170; `use_siren`, nerf/train_nerf.py:89-91) on the tensor cores: the same CTA-pair
// machinery as nerf_tc_kernel / film_tc_kernel (tc_core.cuh) with SirenNeRF's layer program
//   layers_pos.0 (3 -> 256)          CUDA cores, fp32, in the input stage (K = 3 is no GEMM; its 30x-amplified argument must
//                                    not see bf16 inputs)
//   layers_pos.1..4                  tcgen05 steps 0..3, epilogue sin(acc): the weight rows carry the factor 30 and the bias rides
//                                    on two constant-one K columns of the aux chunk (hi + lo bf16 terms)
//   layers_pos.5 on [pos | h4]       step 4: 4 h chunks + the aux chunk [pos(3), 1, 1, dir(3)] (raw position columns)
//   layers_pos.6, 7                  steps 5, 6; output_layer_sigma (256 -> 1) rides on step 6's epilogue in fp32
//   layers_dir.0 (linear)            step 7, epilogue = the accumulator itself
//   layers_dir.1 on [g | dir]        step 8: N = 128, 4 h chunks + the aux chunk (view-direction columns), epilogue sin;
//                                    output_layer_rgb (128 -> 3) on its epilogue in fp32
// Algorithmic work: 2 * (3*256 + 4*65536 + 259*256 + 2*65536 + 256 + 65536 + 259*128 + 384) = 1,123,840 FLOP per row.
#include "tc_core.cuh"

namespace b2r {
namespace tc {

// Every step has a 16-K "post" chunk read from the aux block [pos(3), 1, 1, dir(3), 0...]: its weights carry the raw-input
// columns of the two skip layers and the layer's shift (30 b, or b for the linear layer) as two bf16 terms against the two
// constant ones; the weight rows of the sine layers are pre-multiplied by 30, so the accumulator is the sine's argument.
struct SirenSched {
    static constexpr int kSteps = 9;
    __host__ __device__ static constexpr int n_pre(int, int) { return 0; }
    __host__ __device__ static constexpr int n_h(int, int) { return 4; }
    __host__ __device__ static constexpr int n_post(int, int) { return 1; }
    __host__ __device__ static constexpr int n(int s) { return s == 8 ? 128 : 256; }
    static constexpr int kPostMmas = 1;
};
constexpr long long kSirenChunkBytes = step_base<SirenSched>(SirenSched::kSteps);
static_assert(kSirenChunkBytes == 8 * 5 * 32768LL + 5 * 16384LL, "siren packed chunk bytes");
// fp32 tables (staged in shared memory): w0[3][256] (layers_pos.0, column-major) | shift0[256] | w_sigma[256] | w_rgb[3][128] |
//                                        b_sigma, b_rgb[3]
constexpr int kSW0 = 0, kST0 = 768, kSWS = 1024, kSWR = 1280, kSBH = 1664, kSirenTabFloats = 1668;
constexpr long long kSirenExtraOff = kSirenChunkBytes + kSirenTabFloats * 4;             // blobs of the inference kernel (tc_core.cuh: extra_base)
constexpr long long kSirenPackedBytes = kSirenExtraOff + extra_base<SirenSched>(SirenSched::kSteps);
static_assert(kSirenExtraOff % 16 == 0 && kSirenPackedBytes % 16 == 0, "bulk copies need 16-byte alignment");
static_assert(kSirenTabFloats * 4 <= (int)(kTabBytes + kPartBytes), "siren tables fit the table region");

__host__ __device__ constexpr int siren_step_layer(int s) { return s + 1; }      // steps 0..8 = siren_layer 1..9

// the 8 bf16 of 16-byte group `grp` of weight row n in chunk c (0..3: h columns; 4: the post chunk) of step s
__device__ __forceinline__ void siren_pack_group(const float* __restrict__ params, int s, int c, int n, int grp, __nv_bfloat16 (&v)[8]) {
    LayerDesc L = siren_layer(siren_step_layer(s));
    const float scale = s == 7 ? 1.0f : 30.0f;                                          // layers_dir.0 is linear
    const float shift = scale * params[L.b_off + n];
    const __nv_bfloat16 sh_hi = __float2bfloat16_rn(shift);
    const __nv_bfloat16 sh_lo = __float2bfloat16_rn(shift - __bfloat162float(sh_hi));
    const int h_off = s == 4 ? 3 : 0;                                                   // [pos | h4] (nerf/nerf.py:158)
#pragma unroll
    for (int e = 0; e < 8; ++e) {
        int kk = grp * 8 + e;
        float w = 0.f;
        if (c < 4) w = scale * params[L.w_off + (long long)n * L.in + h_off + c * 64 + kk];
        else if (kk < 3) w = s == 4 ? scale * params[L.w_off + (long long)n * L.in + kk] : 0.f;          // raw position
        else if (kk >= 5 && kk < 8) w = s == 8 ? scale * params[L.w_off + (long long)n * L.in + 256 + (kk - 5)] : 0.f;   // [g | dir] (:166)
        v[e] = (c == 4 && kk == 3) ? sh_hi : ((c == 4 && kk == 4) ? sh_lo : __float2bfloat16_rn(w));
    }
}

__global__ void siren_pack_kernel(const float* __restrict__ params, uint8_t* __restrict__ packed) {
    long long t = blockIdx.x * (long long)blockDim.x + threadIdx.x;
    if (t < kSirenChunkBytes / 16) {
        int s, c, hf, row, grp;
        locate<SirenSched>(t * 16, s, c, hf, row, grp);
        __nv_bfloat16 v[8];
        siren_pack_group(params, s, c, hf * (SirenSched::n(s) / 2) + row, grp, v);
        uint8_t* dst = packed + step_base<SirenSched>(s) + (long long)(c * 2 + hf) * half_bytes<SirenSched>(s) +
                       sw128_offset((uint32_t)row, (uint32_t)grp);
        *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(v);
    }
    if (t < (kSirenPackedBytes - kSirenExtraOff) / 16) {        // blobs [h chunk 3 | compact post chunk] of the inference kernel
        int s, c, hf, row, grp;
        locate_extra<SirenSched>(t * 16, s, c, hf, row, grp);
        __nv_bfloat16 v[8];
        siren_pack_group(params, s, c, hf * (SirenSched::n(s) / 2) + row, grp, v);
        *reinterpret_cast<uint4*>(packed + kSirenExtraOff + extra_dst<SirenSched>(s, c, hf, row, grp)) = *reinterpret_cast<const uint4*>(v);
    }
    if (t < kSirenTabFloats) {
        float* tab = reinterpret_cast<float*>(packed + kSirenChunkBytes);
        int i = (int)t;
        float val;
        if (i < kST0) {
            int k = (i - kSW0) / 256, n = (i - kSW0) % 256;
            val = 30.0f * params[siren_layer(0).w_off + n * 3 + k];       // t_n = sum_k (30 W_nk) p_k + 30 b_n
        } else if (i < kSWS) val = 30.0f * params[siren_layer(0).b_off + (i - kST0)];
        else if (i < kSWR) val = params[siren_layer(10).w_off + (i - kSWS)];
        else if (i < kSBH) val = params[siren_layer(11).w_off + (i - kSWR)];
        else if (i == kSBH) val = params[siren_layer(10).b_off];
        else val = params[siren_layer(11).b_off + (i - kSBH - 1)];
        tab[i] = val;
    }
}

// One SirenNeRF step's epilogue for this warp's quarter of the columns (64, or 32 of the 128 of the last layer).
//   MODE 0: sin(acc) -> bf16 h;   MODE 1: same + partial sigma head;   MODE 2: acc -> bf16 h (linear layers_dir.0);
//   MODE 3: N = 128 (32 columns per quarter): sin(acc) -> partial rgb head (kSave: also bf16 h_d into shared memory at h_blk)
// head: shared-memory address of this quarter's fp32 head weights.  kSave (training forward): cos(acc) of the sine layers is
// stored as one byte per element, one uint4 per 16-column unit, thread-major at cosp + u * 2048 (tc_core.cuh: cos_q4, siren_cos_off).
template <int MODE, bool kSave>
__device__ __forceinline__ void siren_epi(uint32_t t_q, uint32_t head, uint32_t h_blk, const uint32_t (&xoff)[8], float& sigma, float& rgb0,
                                          float& rgb1, float& rgb2, uint8_t* __restrict__ cosp) {
    constexpr int NU = MODE == 3 ? 2 : 4;                       // units of 16 columns
    uint32_t va[16], vb[16];
    tmem_ld16(t_q, va);
#pragma unroll
    for (int u = 0; u < NU; ++u) {
        uint32_t (&v)[16] = (u & 1) ? vb : va;
        tmem_ld_wait();
        if (u < NU - 1) tmem_ld16(t_q + (uint32_t)(u + 1) * 16u, (u & 1) ? va : vb);
        float f[16];
#pragma unroll
        for (int e = 0; e < 16; ++e) f[e] = __uint_as_float(v[e]);
        if (MODE != 2) sin16(v, f);
        if (kSave && MODE != 2) {
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
        if (MODE == 3) {
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                const uint32_t wa = head + (uint32_t)(u * 16 + q * 4) * 4u;
                float4 w0 = lds128(wa), w1 = lds128(wa + 512u), w2 = lds128(wa + 1024u);
                rgb0 = fmaf(f[4 * q + 0], w0.x, fmaf(f[4 * q + 1], w0.y, fmaf(f[4 * q + 2], w0.z, fmaf(f[4 * q + 3], w0.w, rgb0))));
                rgb1 = fmaf(f[4 * q + 0], w1.x, fmaf(f[4 * q + 1], w1.y, fmaf(f[4 * q + 2], w1.z, fmaf(f[4 * q + 3], w1.w, rgb1))));
                rgb2 = fmaf(f[4 * q + 0], w2.x, fmaf(f[4 * q + 1], w2.y, fmaf(f[4 * q + 2], w2.z, fmaf(f[4 * q + 3], w2.w, rgb2))));
            }
        }
        if (MODE != 3 || kSave) {
#pragma unroll
            for (int q = 0; q < 2; ++q)
                st_shared_v4(h_blk + xoff[u * 2 + q], pack_bf16(f[8 * q + 0], f[8 * q + 1]), pack_bf16(f[8 * q + 2], f[8 * q + 3]),
                             pack_bf16(f[8 * q + 4], f[8 * q + 5]), pack_bf16(f[8 * q + 6], f[8 * q + 7]));
        }
    }
}

// Like film_tc_kernel, the 16 epilogue warps are shared by the two sub-tiles: a warp owns one 64-column quarter (= one
// K-block of the next layer) of BOTH and alternates between them.
// kSave = training forward: the layer inputs (aux, h0..h7, layers_dir.0 output, h_d) leave shared memory as tiled bf16 tensors
// through the bulk-copy engine (warps 2 / 3: one spill thread per sub-tile, as in nerf_tc_kernel<true>) and cos(t) of every
// sine layer is stored thread-major for the reverse mode (mlp_tc_train.cu).
template <bool kSave, bool kBox = false>
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(kThreads, 1)
siren_tc_kernel(const uint8_t* __restrict__ packed, RowSource src, long long rows, float4* __restrict__ raw_out, uint8_t* __restrict__ saved,
                LastFlag lf) {
    // inference (kSave = false): compact map -- 4 KB no-swizzle aux operand, 4-stage ring, 4 copies per step (tc_core.cuh MapC)
    constexpr bool kC = !kSave;
    constexpr uint32_t kSub = kC ? MapC::kSub : kSubBytes, kAux = kC ? MapC::kAux : kPeBytes;
    extern __shared__ uint8_t smem_raw[];
    const Ctx cx = kC ? make_ctx_c(smem_raw) : make_ctx(smem_raw);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const PairLoop pl(rows);
    const uint32_t tab = cx.smem + (kC ? MapC::kTab : kTabOff);
    {   // fp32 tables (6.7 KB) -> shared memory
        const float4* tab_g = reinterpret_cast<const float4*>(packed + kSirenChunkBytes);
        for (int i = threadIdx.x; i < kSirenTabFloats / 4; i += kThreads) {
            float4 v = __ldg(tab_g + i);
            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(tab + 16u * i), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w));
        }
    }
    if (kSave) {   // the aux blocks are copied out whole: their never-written chunks must not hold stale bits
        for (int i = threadIdx.x; i < 2 * (int)(kPeBytes / 16); i += kThreads) {
            const uint32_t g = (uint32_t)i / (kPeBytes / 16), o = (uint32_t)i % (kPeBytes / 16);
            st_shared_v4(cx.smem + g * kSubBytes + o * 16u, 0u, 0u, 0u, 0u);
        }
    }
    const uint32_t tmem_base = tc_prologue(cx, warp, 32, 16, kC ? MapC::kStagesC : kStages);

    if (warp == 0) {
        if (lane == 0) {
            if (kC) producer_loop_c<SirenSched>(cx, [packed](long long) { return packed; }, kSirenExtraOff, pl, SirenSched::kSteps);
            else producer_loop<SirenSched>(cx, packed, pl, SirenSched::kSteps, 0);
        }
    } else if (warp == 1) {
        if (kC) {
            if (cx.rank == 0) mma_loop_c<SirenSched>(cx, tmem_base, pl, SirenSched::kSteps);
            else if (lane == 0) relay_loop_c(cx, pl, SirenSched::kSteps);
        } else {
            if (cx.rank == 0) mma_loop<SirenSched>(cx, tmem_base, pl, SirenSched::kSteps, 0);
            else if (lane == 0) relay_loop<SirenSched>(cx, pl, SirenSched::kSteps, 0);
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
                mbar_wait(ready, ph); bulk_s2g(tile(kSsAUX, 1), aux, kBlk); spill_tile(tile(ss_h(0), 4), hreg, 4); finish();    // aux, h0
                for (int l = 1; l < 8; ++l) { mbar_wait(ready, ph); spill_tile(tile(ss_h(l), 4), hreg, 4); finish(); }             // h1 .. h7
                mbar_wait(ready, ph); spill_tile(tile(kSsGL, 4), hreg, 4); finish();                                                // layers_dir.0 output
                mbar_wait(ready, ph); spill_tile(tile(kSsHD, 2), hreg, 2); finish();                                                // h_d
            }
            bulk_wait_all();
        }
    } else {
        const int ew = warp - kCtrlWarps;
        const int cq = ew >> 2, quad = ew & 3;
        const int r = (quad << 5) | lane;
        const uint32_t row_off = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u;
        const uint32_t xr = (uint32_t)(r & 7);
        const uint32_t act_leader0 = mapa(cx.act_ready, 0);
        uint32_t xoff[8];
#pragma unroll
        for (uint32_t c = 0; c < 8; ++c) xoff[c] = (c ^ xr) << 4;
        uint32_t xoff_hd[8];                                      // h_d: this quarter's 32 columns = chunks (cq & 1) * 4 .. + 3 of a K-block
#pragma unroll
        for (uint32_t c = 0; c < 8; ++c) xoff_hd[c] = ((((uint32_t)(cq & 1) * 4u + (c & 3u)) ^ xr) << 4);
        uint32_t acc_phase[2] = {0u, 0u}, sp_phase[2] = {0u, 0u};
        bool first_tile = true;
        const size_t n_sub = (size_t)pl.n_pairs * 4;
        // last-sample sign check (tc_core.cuh LastFlag): |h| <= 1, so the error band of sigma_pre scales with |w_sigma|_1
        float wl1 = 0.f;
        if (lf.count && cq < 2) {
            for (int i = 0; i < 64; ++i) {
                const float4 w = lds128(tab + (uint32_t)(kSWS + 4 * i) * 4u);
                wl1 += (fabsf(w.x) + fabsf(w.y)) + (fabsf(w.z) + fabsf(w.w));
            }
        }
        // kSave: tile written (and fenced by arrive_act) -> spill thread; wait until the previous copy has read shared memory
        auto spill_sig = [&](int g) { if (kSave && lane == 0) mbar_arrive(cx.spill_ready + 8 * g); };
        auto spill_wait = [&](int g) { if (kSave) { mbar_wait(cx.spill_done + 8 * g, sp_phase[g]); sp_phase[g] ^= 1u; } };
        auto sub_base = [&](int g) -> uint32_t { return cx.smem + (uint32_t)g * kSub; };
        auto part_of = [&](int g) -> uint32_t { return sub_base(g) + (kC ? kAux : 8192u); };      // head partials (see film_tc_kernel)
        auto t_row = [&](int g) -> uint32_t { return tmem_base + ((uint32_t)quad << 21) + (uint32_t)g * 256u; };
        auto h_blk = [&](int g) -> uint32_t { return sub_base(g) + kAux + (uint32_t)cq * 16384u + row_off; };
        auto arrive = [&](int g) { arrive_act(cx.act_ready + 8 * g, act_leader0 + 8 * g, cx.rank, lane); };
        auto wait_acc = [&](int g) {
            mbar_wait_cluster(cx.acc_full + 8 * g, acc_phase[g]);
            acc_phase[g] ^= 1u;
            tc_fence_after();
        };
        for (long long p = pl.first; p < pl.n_pairs; p += pl.stride) {
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
                if (!first_tile) spill_wait(g);                      // previous tile's h_d copy
                const size_t T = (size_t)((2 * p + cx.rank) * 2 + g);
                // ---- layers_pos.0 on CUDA cores: this warp produces columns cq*64 .. +63 of h0 (K-block cq)
if constexpr (kC) {
                    // column-owned form (tc_core.cuh sine_input_layer): the table stays in registers, positions come by shuffle
                    sine_input_layer(tab + kSW0 * 4u, tab + kST0 * 4u, sub_base(g) + kAux + (uint32_t)cq * 16384u, cq, quad, lane, pnt);
                } else {
    #pragma unroll
                    for (int jj = 0; jj < 2; ++jj) {
                        uint32_t pk[16], ck[8];
    #pragma unroll
                        for (int q = 0; q < 8; ++q) {
                            const uint32_t n0 = (uint32_t)(cq * 64 + jj * 32 + q * 4) * 4u;
                            const float4 wx = lds128(tab + kSW0 * 4u + n0), wy = lds128(tab + (kSW0 + 256) * 4u + n0), wz = lds128(tab + (kSW0 + 512) * 4u + n0);
                            const float4 sh = lds128(tab + kST0 * 4u + n0);
                            // the factor 30 is folded into the table's weights: 3 fma per output (the packed fp32x2 form cost 132 B of spills here)
                            const float t0 = fmaf(wz.x, pnt[2], fmaf(wy.x, pnt[1], fmaf(wx.x, pnt[0], sh.x)));
                            const float t1 = fmaf(wz.y, pnt[2], fmaf(wy.y, pnt[1], fmaf(wx.y, pnt[0], sh.y)));
                            const float t2 = fmaf(wz.z, pnt[2], fmaf(wy.z, pnt[1], fmaf(wx.z, pnt[0], sh.z)));
                            const float t3 = fmaf(wz.w, pnt[2], fmaf(wy.w, pnt[1], fmaf(wx.w, pnt[0], sh.w)));
                            pk[2 * q + 0] = pack_bf16(__sinf(t0), __sinf(t1));
                            pk[2 * q + 1] = pack_bf16(__sinf(t2), __sinf(t3));
                            if (kSave) ck[q] = cos_q4(t0, t1, t2, t3);
                        }
    #pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            st_shared_v4(h_blk(g) + xoff[jj * 4 + q], pk[4 * q], pk[4 * q + 1], pk[4 * q + 2], pk[4 * q + 3]);
                            if (kSave && q < 2) stg128(saved + siren_cos_off(n_sub, 0, T, cq, jj * 2 + q, r), ck[4 * q], ck[4 * q + 1], ck[4 * q + 2], ck[4 * q + 3]);
                        }
                    }
                }
                if (cq == 0) {
                    // aux block = [pos(3), 1, 1, dir(3), 0 ...] (16 K): raw inputs of the two skip layers + the constant ones of the shifts
                    // (compact map: 16-byte K chunk c of row r at c * 2 KB + r * 16, no swizzle)
                    st_shared_v4(sub_base(g) + (kC ? (uint32_t)r * 16u : row_off + ((0u ^ xr) << 4)), pack_bf16(pnt[0], pnt[1]), pack_bf16(pnt[2], 1.0f),
                                 pack_bf16(1.0f, vdir[0]), pack_bf16(vdir[1], vdir[2]));
                    st_shared_v4(sub_base(g) + (kC ? 2048u + (uint32_t)r * 16u : row_off + ((1u ^ xr) << 4)), 0u, 0u, 0u, 0u);
                }
                arrive(g);
                spill_sig(g);
            }
            first_tile = false;
            auto cosp = [&](int layer, int g) -> uint8_t* {
                return kSave ? saved + siren_cos_off(n_sub, layer, (size_t)((2 * p + cx.rank) * 2 + g), cq, 0, r) : nullptr;
            };

            float sigma[2] = {0.f, 0.f}, rgb0[2] = {0.f, 0.f}, rgb1[2] = {0.f, 0.f}, rgb2[2] = {0.f, 0.f};
            for (int s = 0; s < 6; ++s) {                               // layers_pos.1 .. layers_pos.6
#pragma unroll
                for (int g = 0; g < 2; ++g) {
                    wait_acc(g);
                    spill_wait(g);
                    siren_epi<0, kSave>(t_row(g) + (uint32_t)cq * 64u, 0u, h_blk(g), xoff, sigma[g], rgb0[g], rgb1[g], rgb2[g], cosp(s + 1, g));
                    arrive(g);
                    spill_sig(g);
                }
            }
#pragma unroll
            for (int g = 0; g < 2; ++g) {                               // layers_pos.7 (+ sigma head)
                wait_acc(g);
                spill_wait(g);
                siren_epi<1, kSave>(t_row(g) + (uint32_t)cq * 64u, tab + (uint32_t)(kSWS + cq * 64) * 4u, h_blk(g), xoff, sigma[g], rgb0[g], rgb1[g], rgb2[g],
                                    cosp(7, g));
                arrive(g);
                spill_sig(g);
            }
#pragma unroll
            for (int g = 0; g < 2; ++g) {                               // layers_dir.0 (linear)
                wait_acc(g);
                spill_wait(g);
                siren_epi<2, kSave>(t_row(g) + (uint32_t)cq * 64u, 0u, h_blk(g), xoff, sigma[g], rgb0[g], rgb1[g], rgb2[g], nullptr);
                arrive(g);
                spill_sig(g);
            }
#pragma unroll
            for (int g = 0; g < 2; ++g) {                               // layers_dir.1 (N = 128: 32 columns per quarter) + rgb head
                wait_acc(g);
                spill_wait(g);
                // kSave: bf16 h_d goes to K-block cq / 2 of the (now free) h region, chunks (cq & 1) * 4 ..; its cosine to the 4-word layout
                siren_epi<3, kSave>(t_row(g) + (uint32_t)cq * 32u, tab + (uint32_t)(kSWR + cq * 32) * 4u,
                                    sub_base(g) + kAux + (uint32_t)(cq >> 1) * 16384u + row_off + (uint32_t)0, xoff_hd, sigma[g], rgb0[g], rgb1[g], rgb2[g],
                                    kSave ? saved + siren_cos9_off(n_sub, (size_t)((2 * p + cx.rank) * 2 + g), cq, 0, r) : nullptr);
                if (kSave) {
                    fence_proxy_async_smem();
                    __syncwarp();
                    spill_sig(g);
                }
            }
            tc_fence_before();
            // head partials of the four column quarters (part_of)
            if (kC) asm volatile("bar.sync 3, 512;" ::: "memory");      // the slots overlay h: every warp is past its last epilogue
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
                    const float4 bh = lds128(tab + kSBH * 4u);          // (b_sigma, b_rgb[3])
                    float4 o;
                    o.x = 1.0f / (1.0f + __expf(-((p0.x + p1.x) + (p2.x + p3.x) + bh.y)));
                    o.y = 1.0f / (1.0f + __expf(-((p0.y + p1.y) + (p2.y + p3.y) + bh.z)));
                    o.z = 1.0f / (1.0f + __expf(-((p0.z + p1.z) + (p2.z + p3.z) + bh.w)));
                    const float pre = (p0.w + p1.w) + (p2.w + p3.w) + bh.x;
                    o.w = fmaxf(pre, 0.f);
                    raw_out[out_row] = o;
                    if ((cq == 0 ? chk[0] : chk[1]) && fabsf(pre) <= fmaf(lf.rel, wl1, lf.abs)) flag_ray(lf, cq == 0 ? ray[0] : ray[1]);
                }
            }
            asm volatile("bar.sync 3, 512;" ::: "memory");
        }
    }
    tc_teardown(tmem_base, warp);
}

int pair_grid(long long rows, unsigned* grid);   // mlp_tc.cu

size_t siren_packed_bytes() { return (size_t)kSirenPackedBytes; }

int siren_pack(const float* params, void* packed_out, cudaStream_t st) {
    long long threads = kSirenChunkBytes / 16;
    siren_pack_kernel<<<(unsigned)((threads + 255) / 256), 256, 0, st>>>(params, (uint8_t*)packed_out);
    B2R_LAUNCH_CHECK("b2r_mlp_tc_pack (SirenNeRF)");
    return 0;
}

int siren_fwd(const void* packed, const b2r_mlp_input* in, long long rows, float* raw_out, const b2r_last_sample* last, cudaStream_t st) {
    unsigned grid = 0;
    int rc = pair_grid(rows, &grid);
    if (rc) return rc;
    auto kern = lattice_mode(in) ? siren_tc_kernel<false, true> : siren_tc_kernel<false>;      // box-lattice rows: own instantiation
    rc = cuda_result(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)MapC::kSmem), "tc smem attribute");
    if (rc) return rc;
    kern<<<grid, kThreads, MapC::kSmem, st>>>((const uint8_t*)packed, make_row_source(in), rows, (float4*)raw_out, nullptr, make_last_flag(last));
    B2R_LAUNCH_CHECK("b2r_mlp_tc_fwd (SirenNeRF)");
    return 0;
}

size_t siren_saved_bytes(long long rows) { return (size_t)n_sub_tiles(rows) * siren_saved_bytes_per_sub(); }

int siren_train_fwd(const void* packed, const b2r_mlp_input* in, long long rows, float* raw_out, void* saved, const b2r_last_sample* last, cudaStream_t st) {
    unsigned grid = 0;
    int rc = pair_grid(rows, &grid);
    if (rc) return rc;
    rc = cuda_result(cudaFuncSetAttribute(siren_tc_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes), "tc smem attribute");
    if (rc) return rc;
    siren_tc_kernel<true><<<grid, kThreads, kSmemBytes, st>>>((const uint8_t*)packed, make_row_source(in), rows, (float4*)raw_out, (uint8_t*)saved,
                                                              make_last_flag(last));
    B2R_LAUNCH_CHECK("b2r_mlp_tc_train_fwd (SirenNeRF)");
    return 0;
}

}  // namespace tc
}  // namespace b2r
