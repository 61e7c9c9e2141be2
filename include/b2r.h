/*
 * b2r.h -- C ABI of libb2r.so, the B200 (sm_100a) implementation of the volumetric
 * ray-march render path of JeffreyXiang/MSRA-practice-project.
 *
 * The reference has no FFI: its boundary for this path is the Python module surface of
 * nerf/render.py and pi_GAN/render.py (SURVEY.md 8b).  Each entry point below names the
 * reference function (file:line, relative to the reference root) whose arithmetic it
 * replaces; the Python mirrors of those functions (msra_practice_project_b200/nerf_render.py,
 * pigan_render.py) call these through ctypes (INTEGRATION.md shows the binding).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to caller-owned memory unless marked "host";
 *   - tensors are dense row-major float32 unless stated;
 *   - the last argument is the CUDA stream (cudaStream_t, passed as void*); no function
 *     allocates, synchronises or throws;
 *   - return 0 = OK, <0 = bad argument, >0 = cudaError_t; b2r_last_error() gives the message
 *     (thread-local);
 *   - the library is re-entrant: no mutable global state (nn.DataParallel calls it from one
 *     thread per GPU, pi_GAN/train.py:50).
 */
#ifndef B2R_H_
#define B2R_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B2R_VERSION 100

/* model kinds */
#define B2R_MODEL_NERF 0      /* nerf/nerf.py:52-94            */
#define B2R_MODEL_FILM 1      /* pi_GAN/modules.py:70-118      */
#define B2R_MODEL_SIREN 2     /* nerf/nerf.py:120-170 (SirenNeRF)       */

/* flat fp32 parameter counts (state-dict order: weight,bias per layer) */
#define B2R_NERF_NUMEL 593924
#define B2R_FILM_NUMEL 529156
#define B2R_SIREN_NUMEL 562052
#define B2R_FILM_NODIR_NUMEL 528388
#define B2R_FILM_PARAMS 4608   /* film_params [9,512] = gamma(256)||beta(256) per layer */

const char* b2r_last_error(void);
int b2r_version(void);
/* 1 when the library was compiled for sm_100a and the current device is compute capability 10.x */
int b2r_device_ok(void);

/* ---- K1: ray generation -------------------------------- get_rays  nerf/render.py:7-23 ----
 * rays_out[ray_count,2,3] = (origin, direction) for flattened pixel indices
 * [ray_begin, ray_begin+ray_count) of a W x H image (row-major, column fastest), i.e. rows of
 * the [H*W,2,3] table render_image builds (nerf/render.py:151-154).
 * c2w: host pointer to the 3x4 camera-to-world matrix (row-major, 12 doubles; a float32 pose
 * converts exactly).
 * compute_f64 reproduces numpy's float64 promotion: bit 0 = the caller's focal is an np.float64
 * (pi_GAN/modules.py:127: the division is done in double), bit 1 = the pose is a float64 array.
 * When non-zero the rotation is computed in double and rounded to float32 at the end
 * (render_image casts, nerf/render.py:159). */
int b2r_raygen(const double* c2w_host, int width, int height, double focal, int compute_f64,
               long long ray_begin, long long ray_count, float* rays_out, void* stream);

/* The same ray table for n_poses FULL images whose poses live in DEVICE memory: poses_dev[n_poses,12] doubles (row-major 3x4),
 * rays_out[n_poses * H * W, 2, 3].  Replaces the per-latent get_rays calls of Generator.forward's loop
 * (pi_GAN/modules.py:176-184 -> Renderer.__call__ :153-161 -> render_image pi_GAN/render.py:197-200); nothing that changes from
 * step to step is a kernel argument, so a captured CUDA graph replays with new poses.  Bit-identical to b2r_raygen per pose. */
int b2r_raygen_poses(const double* poses_dev, int n_poses, int width, int height, double focal, int compute_f64,
                     float* rays_out, void* stream);

/* ---- K2: stratified coarse samples ------------------- render_rays nerf/render.py:123-132 --
 * z_lin[Sc] = torch.linspace(near, far, Sc) made by the caller (its rounding is a contract);
 * t_rand[N,Sc] = the jitter (torch.rand in the reference, :131);
 * z_out[N,Sc] = lower + (upper-lower)*t_rand;  mids_out[Sc-1] (nullable) = 0.5*(z_lin[1:]+z_lin[:-1]). */
int b2r_stratified_z(const float* z_lin, const float* t_rand, long long n_rays, int n_coarse,
                     float* z_out, float* mids_out, void* stream);

/* ---- K4: alpha compositing ------------------------ raw_to_outputs nerf/render.py:78-103 ---
 * raw[N,S,4] (rgb, sigma), z[N,S], rays_d: N direction vectors d_stride floats apart (3 for a
 * dense [N,3], 6 for rays[:,1] of an [N,2,3] table).  weights_out[N,S] is nullable. */
int b2r_composite_fwd(const float* raw, const float* z, const float* rays_d, int d_stride,
                      long long n_rays, int n_samples, float* rgb_out, float* depth_out,
                      float* acc_out, float* weights_out, void* stream);

/* the same with strided outputs: ray r's colour at rgb_out[r * rgb_stride .. + 2], depth at depth_out[r * depth_stride], acc at
 * acc_out[r * acc_stride] -- e.g. (base, 5), (base + 3, 5), (base + 4, 5) writes rows of the packed [N,5] frame buffer that the
 * multi-GPU image gather exchanges (nerf/render.py:161-166 concatenates the three maps on the host). */
int b2r_composite_fwd_strided(const float* raw, const float* z, const float* rays_d, int d_stride,
                              long long n_rays, int n_samples, float* rgb_out, int rgb_stride, float* depth_out,
                              int depth_stride, float* acc_out, int acc_stride, float* weights_out, void* stream);

/* reverse mode of the above wrt raw (autograd in the reference, nerf/train_nerf.py:167).
 * g_depth / g_acc nullable (treated as zero).  d_raw[N,S,4]. */
int b2r_composite_bwd(const float* raw, const float* z, const float* rays_d, int d_stride,
                      long long n_rays, int n_samples, const float* g_rgb, const float* g_depth,
                      const float* g_acc, float* d_raw, void* stream);

/* training: the loss of nerf/train_nerf.py:157-166 and the reverse mode of the composite in one launch.
 *   loss = mean((rgb - target_rgb)^2) [+ alpha_weight * mean((acc - target_acc)^2)] over the GLOBAL batch of 1 / *inv_count rays
 * (inv_count: device float, so that a CUDA graph replays with the count of a short last batch); the kernel recomputes the ray's
 * forward, forms g_rgb = 2 (rgb - target) inv_count / 3 and g_acc = 2 alpha_weight (acc - target_acc) inv_count itself (g_depth = 0:
 * the reference's loss never uses depth) and writes d_raw[N,S,4].  ray_weight[N] (nullable) scales a ray's loss term (0 for padding).
 * sums[0] += sum w (rgb - target)^2 over rays and channels, sums[1] += sum w (acc - target_acc)^2 (caller zeroes). */
int b2r_composite_loss_bwd(const float* raw, const float* z, const float* rays_d, int d_stride, long long n_rays, int n_samples,
                           const float* target_rgb, const float* target_acc, const float* ray_weight, const float* inv_count,
                           float alpha_weight, float* d_raw, float* sums, void* stream);

/* loss and PSNR of a training step from the four sums of two b2r_composite_loss_bwd calls (sums[0..1] fine pass, [2..3] coarse):
 * loss = (s0 + s2) inv_count / 3 + alpha_weight (s1 + s3) inv_count; psnr = -10 log10(s0 inv_local / 3)  (train_nerf.py:158-166). */
int b2r_train_loss_finish(const float* sums, const float* inv_count, float alpha_weight, const float* inv_local, float* loss,
                          float* psnr, void* stream);

/* ---- K5/K6: hierarchical resampling --- sample_pdf nerf/render.py:27-56, sort-merge :142 ---
 * bins: nb values per ray, bins_stride floats apart (0 = one shared row, as in render_rays);
 * weights: nb-1 values per ray, w_stride floats apart (render_rays passes weights[:,1:-1]:
 * pointer +1, stride Sc); u[Sf] = torch.linspace(0,1,Sf) from the caller.
 * samples_out[N,Sf] nullable; if z_coarse != NULL, sorted_out[N,Sc+Sf] = sort(cat(z_coarse,
 * samples)) (both are monotone, so a merge).  cdf_out[N,nb] nullable (parity harness:
 * "indices bit-exact given identical CDFs"). */
int b2r_sample_pdf(const float* bins, long long bins_stride, const float* weights, long long w_stride,
                   const float* u, long long n_rays, int nb, int n_fine,
                   const float* z_coarse, int n_coarse,
                   float* samples_out, float* sorted_out, float* cdf_out, void* stream);
/* b2r_sample_pdf runs instantiations with compile-time sizes for the shapes of BASELINE.json's configs (64+128, 64+64,
 * 24+24) and the run-time-size kernel otherwise; b2r_sample_pdf_generic forces the latter (same arguments, bit-identical
 * results: the parity tests compare the two). */
int b2r_sample_pdf_generic(const float* bins, long long bins_stride, const float* weights, long long w_stride,
                        const float* u, long long n_rays, int nb, int n_fine,
                        const float* z_coarse, int n_coarse,
                        float* samples_out, float* sorted_out, float* cdf_out, void* stream);

/* ---- K3: radiance-field MLP --- run_network nerf/render.py:59-75 + NeRF.forward nerf/nerf.py:75-94
 *                                 + FilmSirenNeRF.forward pi_GAN/modules.py:101-118 ------------
 * Input rows are described in one of four ways (exactly one must be given):
 *   rays != NULL : rows = n_rays*n_samples, point = o + d*z[r,s], dir = d/|d|   (render_rays)
 *   x    != NULL : rows = n_rays (n_samples must be 1), x[rows,6] = (pos, dir)  (network(x))
 *   grid_n  > 0  : rows = n_rays = count of grid indices starting at grid_begin of an
 *                  N^3 lattice in [-0.1,0.1]^3, dir = 0            (create_mesh, pi_GAN/utils.py:59-91)
 *   lattice_dims != 0 : box lattice, rows = n_rays = count of lattice indices starting at grid_begin of an
 *                  n0 x n1 x n2 lattice (axis 0 slowest); index (i,j,k) is the point
 *                  origin + (i,j,k) * voxel (each component a rounded fp32 multiply, then a rounded add), dir = 0.
 *                  Needs every n >= 2, n0*n1*n2 <= INT32_MAX and a finite voxel > 0.  grid_n = N is the box lattice
 *                  (N, N, N), origin -0.1, voxel (float)(0.2/(N-1)), row for row.
 * Grid and lattice rows are for inference and mesh extraction: the last-sample check rejects them, and box-lattice rows go to
 * b2r_mlp_tc_fwd / b2r_mlp_f32_fwd (the batched FiLM and tensor-core training entry points reject them).
 * raw_out[rows,4] = (sigmoid rgb, relu sigma).
 * The struct grew by the three lattice_* fields after grid_begin (B2R_VERSION unchanged): a caller that zero-initialises
 * it and sets only the older fields gets the older behaviour.
 */
typedef struct b2r_mlp_input {
    const float* rays;      /* [n_rays,2,3] or NULL */
    const float* z;         /* [n_rays,n_samples] (with rays) */
    const float* x;         /* [rows,6] or NULL */
    long long n_rays;
    int n_samples;
    int grid_n;             /* >0: lattice mode */
    long long grid_begin;   /* first lattice index (grid_n or box-lattice mode) */
    int lattice_dims[3];    /* any non-zero: box-lattice mode, points per axis (n0, n1, n2) */
    float lattice_origin[3];
    float lattice_voxel;
} b2r_mlp_input;

/* ---- the last interval of every ray ------------------------------------ raw_to_outputs nerf/render.py:91-93 ----
 * dists[-1] = 1e10 makes alpha_last = 1 - exp(-sigma_last * 1e10 * |d|) a STEP FUNCTION of sign(sigma_last): the sign
 * of the LAST sample's pre-relu density decides whether the ray's remaining transmittance lands on that sample or on
 * the white background, so a bf16-rounded sigma that crosses zero changes a ray's colour by up to T_last (SURVEY.md 0).
 * The bf16 tensor-core kernels therefore report, for rows r with (r + 1) % samples_per_ray == 0, every ray whose
 * |sigma_pre| is inside the error band of the bf16 arithmetic:
 *     |sigma_pre| <= rel * scale + abs,   scale = sum_k |w_sigma[k] * h[k]| of that row   (ReLU trunk: NeRF)
 *                                         scale = sum_k |w_sigma[k]|                      (sine trunks, |h| <= 1)
 * and b2r_mlp_f32_last_sigma re-evaluates exactly those rows with the fp32 CUDA-core path (bit-identical to
 * b2r_mlp_f32_fwd on the same rows) and overwrites raw[row, 3].
 * count: one device int the CALLER ZEROES; ray_ids[capacity]: flagged ray indices (row / samples_per_ray) in
 * arbitrary order; count may exceed capacity (entries beyond it are dropped: size capacity = number of rays). */
typedef struct b2r_last_sample {
    int samples_per_ray;
    int capacity;
    int* count;
    int* ray_ids;
    float rel, abs;
} b2r_last_sample;

/* fp32 path (CUDA cores).  params: flat fp32 parameters (B2R_*_NUMEL floats, state-dict order);
 * film: [9,512] (FiLM model only).  workspace: b2r_mlp_f32_workspace_bytes(kind, rows, save)
 * bytes; with save_activations != 0 the workspace holds every layer's output afterwards and is
 * the `saved` argument of b2r_mlp_f32_bwd.  use_dir: FilmSirenNeRF(use_dir=...) flag. */
size_t b2r_mlp_f32_workspace_bytes(int model_kind, long long rows, int save_activations);
/* gemm_mode: 0 = fp32 FMAs on the CUDA cores (exact: the fp32 parity path), 1 = the same layer-wise algorithm with the
 * GEMMs on the tensor cores in TF32 (tcgen05 kind::tf32, fp32 accumulate; ~1e-3 relative).  Any other value is rejected. */
int b2r_mlp_f32_fwd(int model_kind, const float* params, const float* film, int use_dir,
                    const b2r_mlp_input* in, float* raw_out, void* workspace, size_t workspace_bytes,
                    int save_activations, int gemm_mode, void* stream);
/* backward of the fp32 path: d_raw[rows,4] -> d_params (flat, ACCUMULATED into: caller zeroes),
 * d_film[9,512] (FiLM only, accumulated, nullable).  saved = workspace of the forward call made with
 * save_activations=1 on the same inputs; scratch = b2r_mlp_f32_bwd_scratch_bytes(kind, rows). */
size_t b2r_mlp_f32_bwd_scratch_bytes(int model_kind, long long rows);
int b2r_mlp_f32_bwd(int model_kind, const float* params, const float* film, int use_dir,
                    const b2r_mlp_input* in, const float* raw, const float* d_raw, const void* saved,
                    void* scratch, size_t scratch_bytes, float* d_params, float* d_film, int gemm_mode, void* stream);

/* bf16 tensor-core path (tcgen05 / TMEM, weights streamed by the TMA bulk-copy engine).
 * packed: b2r_mlp_tc_packed_bytes(kind) bytes produced by b2r_mlp_tc_pack from the flat fp32
 * parameters (+ film for the FiLM model: gamma/beta/bias are folded into per-column scale/shift).  The image is opaque to the
 * caller: bf16 weight chunks in the kernels' shared-memory layouts, fp32 tables and, for the sine models, a second copy of every
 * step's last chunks in the layout of the inference kernels' 4-stage ring (csrc/tc_core.cuh). */
size_t b2r_mlp_tc_packed_bytes(int model_kind);
int b2r_mlp_tc_pack(int model_kind, const float* params, const float* film, int use_dir,
                    void* packed_out, void* stream);
/* use_dir: the FilmSirenNeRF(use_dir=...) flag the weights were packed with (ignored for NeRF).
 * sigma_only != 0 (NeRF, FiLM-SIREN): stop after the sigma head, raw_out[:, :3] = 0 (create_mesh density query; coarse passes whose
 * colour nobody reads); sigma is bit-identical to the full evaluation's. */
/* last: nullable; when given (rays or x mode), the kernel also lists the rays whose last sample needs the fp32 sign check. */
int b2r_mlp_tc_fwd(int model_kind, const void* packed, int use_dir, const b2r_mlp_input* in, float* raw_out,
                   int sigma_only, const b2r_last_sample* last, void* stream);
/* fp32 re-evaluation of sigma for the last sample of the n_ids listed rays (trunk + sigma head only): raw_io[(ray *
 * samples_per_ray + samples_per_ray - 1) * 4 + 3] = relu(sigma_pre) with the arithmetic of b2r_mlp_f32_fwd (gemm_mode 0).
 * film: [n_latents,9,512] for the FiLM model (n_latents = 1: one [9,512] tensor); with n_latents > 1 source row r belongs
 * to latent r / rows_per_latent (the batched entry points below).  workspace: b2r_mlp_f32_workspace_bytes(kind, n_ids, 0)
 * + 4 * n_ids bytes. */
int b2r_mlp_f32_last_sigma(int model_kind, const float* params, const float* film, int use_dir, int n_latents,
                           long long rows_per_latent, const b2r_mlp_input* in, int samples_per_ray, const int* ray_ids,
                           int n_ids, float* raw_io, void* workspace, size_t workspace_bytes, void* stream);

/* ---- K8 on the tensor cores: training forward + reverse mode of the NeRF MLP (bf16 operands, fp32 accumulate) --------
 * Replaces autograd through NeRF.forward (nerf/nerf.py:75-94) as used by nerf/train_nerf.py:151-168.
 * b2r_mlp_tc_train_fwd = b2r_mlp_tc_fwd that also keeps every layer input as tiled bf16 tensors in `saved`
 * (b2r_mlp_tc_train_saved_bytes(kind, rows) bytes, 5,120 B per row, rows padded to 512).
 * b2r_mlp_tc_train_bwd: d_raw[rows,4] -> d_params (flat fp32, ACCUMULATED into: caller zeroes).  packed_bwd: transposed
 * weights from b2r_mlp_tc_pack_bwd (b2r_mlp_tc_bwd_packed_bytes bytes); raw = the forward's output; scratch:
 * b2r_mlp_tc_train_scratch_bytes(kind, rows) bytes (per-layer d(pre-activation) tiles for the weight-gradient GEMMs).
 * B2R_MODEL_NERF and B2R_MODEL_SIREN (nerf/nerf.py:97-170) use these entry points as they are.  B2R_MODEL_FILM
 * (FilmSirenNeRF; autograd through pi_GAN/modules.py:101-118 as used by pi_GAN/train.py:134 and
 * synthesis.py:107): b2r_mlp_tc_train_fwd takes ONE latent's packed image (b2r_mlp_tc_pack with that latent's film);
 * the reverse mode is b2r_mlp_tc_pack_bwd_film + b2r_mlp_tc_train_bwd_film, which also returns d film[9,512]
 * (d gamma | d beta per layer).  d_folded: B2R_FILM_NUMEL floats of workspace (zeroed by the call: gradients of the
 * FiLM-folded weights W' = 30 gamma W, s' = 30 (gamma b + beta)); d_params / d_film are ACCUMULATED into and either may
 * be NULL (synthesis.py only needs d film). */
size_t b2r_mlp_tc_train_saved_bytes(int model_kind, long long rows);
/* last (nullable): the last-sample sign check of b2r_mlp_tc_fwd, so that the training forward reports the same raw values
 * as the render (the caller then runs b2r_mlp_f32_last_sigma on raw_out before it composites). */
int b2r_mlp_tc_train_fwd(int model_kind, const void* packed, const b2r_mlp_input* in, float* raw_out, void* saved,
                         size_t saved_bytes, const b2r_last_sample* last, void* stream);
size_t b2r_mlp_tc_bwd_packed_bytes(int model_kind);
int b2r_mlp_tc_pack_bwd(int model_kind, const float* params, void* packed_out, void* stream);
size_t b2r_mlp_tc_train_scratch_bytes(int model_kind, long long rows);
int b2r_mlp_tc_train_bwd(int model_kind, const void* packed_bwd, long long rows, const float* raw, const float* d_raw,
                         const void* saved, void* scratch, size_t scratch_bytes, float* d_params, void* stream);
/* FiLM-SIREN, B latents in one launch sequence (Generator.forward's loop WITH gradients, pi_GAN/modules.py:176-184 +
 * pi_GAN/train.py:134): packed = B images from b2r_mlp_tc_pack_film_batched, rows [b*rows_per_latent, (b+1)*rows_per_latent)
 * belong to latent b (rows_per_latent a multiple of 512); film [B,9,512]; packed_bwd = B images from b2r_mlp_tc_pack_bwd_film;
 * d_folded: B * B2R_FILM_NUMEL floats; d_film [B,9,512]; d_params sums over the latents.  n_latents = 1: rows_per_latent ignored.
 * use_dir: the FilmSirenNeRF(use_dir=...) flag (0: hidden_layer_rgb has 256 inputs, flat layout B2R_FILM_NODIR_NUMEL). */
int b2r_mlp_tc_train_fwd_film_batched(const void* packed, int n_latents, long long rows_per_latent, const b2r_mlp_input* in,
                                      float* raw_out, void* saved, size_t saved_bytes, const b2r_last_sample* last, void* stream);
int b2r_mlp_tc_pack_bwd_film(const float* params, const float* film, int use_dir, int n_latents, void* packed_out, void* stream);
int b2r_mlp_tc_train_bwd_film(const void* packed_bwd, const float* params, const float* film, int use_dir, int n_latents, long long rows_per_latent,
                              long long rows, const float* raw, const float* d_raw, const void* saved, void* scratch,
                              size_t scratch_bytes, float* d_folded, float* d_params, float* d_film, void* stream);

/* ---- fused Adam on a flat fp32 bucket ----------- optimizer.step() + LR decay, nerf/train_nerf.py:168-175 ----------
 * torch.optim.Adam semantics (no weight decay / amsgrad) on n contiguous floats; grads are multiplied by grad_scale first
 * (1/world for an averaged all-reduce).  state: 4 device floats, zero-initialised by the caller before the first step,
 * owned by the optimiser afterwards ([0] = step count as int32 bits, [1] = current lr, [2], [3] = bias corrections): the
 * step count and the decayed learning rate lr0 * decay_rate^((t-1)/decay_steps) (decay_steps <= 0: constant lr0) advance
 * ON THE DEVICE, so the two launches replay unchanged inside a CUDA graph. */
int b2r_adam_step(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, float* state,
                  float lr0, float decay_rate, float decay_steps, float beta1, float beta2, float eps, float grad_scale,
                  void* stream);

/* The same step with the schedule of pi_GAN/train.py:140-145: lr_t = lr_end + (lr0 - lr_end) * decay_rate^((t-1)/decay_steps)
 * (the generator's Adam, pi_GAN/train.py:53: betas (0, 0.9)); lr_end = 0 is b2r_adam_step. */
int b2r_adam_step_floor(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long long n, float* state,
                        float lr0, float lr_end, float decay_rate, float decay_steps, float beta1, float beta2, float eps,
                        float grad_scale, void* stream);

/* ---- batched FiLM-SIREN evaluation --------- Generator.forward's per-latent loop, pi_GAN/modules.py:176-184 --------
 * One launch for B latents.  packed: B images of b2r_mlp_tc_packed_bytes(B2R_MODEL_FILM) bytes one after the other, made by
 * b2r_mlp_tc_pack_film_batched from film[B,9,512] (the FiLM scale / shift are folded into each latent's bf16 weights).
 * Rows [b*rows_per_latent, (b+1)*rows_per_latent) of the input are evaluated with latent b; rows_per_latent must be a
 * multiple of 512 (the two 256-row tiles of a CTA pair share one set of weights). */
int b2r_mlp_tc_pack_film_batched(const float* params, const float* film, int use_dir, int n_latents, void* packed_out, void* stream);
int b2r_mlp_tc_fwd_film_batched(const void* packed, int n_latents, long long rows_per_latent, const b2r_mlp_input* in, float* raw_out,
                                int sigma_only, const b2r_last_sample* last, void* stream);

/* ---- image-space output ---------------------------------------------------- to8b  nerf/render.py:5 ---------------
 * out[i] = (uint8)(255 * clip(x[i], 0, 1)) with numpy's float32 product and truncation (show_nerf.py:60-66,
 * train_nerf.py:199 quantise every frame on the host); lets frames leave the device as 1 byte per channel. */
int b2r_to8b(const float* x, long long n, unsigned char* out, void* stream);

/* ---- marching cubes ------------------------------------------- create_mesh  pi_GAN/utils.py:99-180 ----------------
 * The level set of field[n0,n1,n2] (fp32, axis 0 slowest) as a triangle mesh; the table, the numbering and the rule that
 * generates it: oracle/marching_cubes.py.  Two calls, because the output size is data-dependent:
 *   b2r_mc_count: writes the per-point codes into scratch (b2r_mc_scratch_bytes(n0, n1, n2) bytes, 16-byte aligned) and
 *                 totals_dev[2] = (V, F), the vertex and triangle counts, as two long long in DEVICE memory;
 *   b2r_mc_emit:  given the scratch b2r_mc_count wrote for the same field and level, writes verts[V,3] (fp32) and
 *                 faces[F,3] (int32 vertex indices).  The caller reads (V, F) first and must not call it when V or F
 *                 exceeds INT32_MAX.
 * Vertices are ordered by owner lattice point (linear index), then edge axis; the vertex on the edge from point p along
 * axis a is origin + (p + t e_a) * spacing, t = (level - f(p)) / (f(p + e_a) - f(p)), every operation rounded separately.
 * Triangles are ordered by cell (linear index of its minimum corner), then table order; their normals
 * (v1-v0) x (v2-v0) point from below (f < level) to above.  Both calls need n >= 2 on every axis and n0*n1*n2 <= INT32_MAX;
 * b2r_mc_scratch_bytes returns 0 for any other shape. */
size_t b2r_mc_scratch_bytes(int n0, int n1, int n2);
int b2r_mc_count(const float* field, int n0, int n1, int n2, float level, void* scratch, long long* totals_dev, void* stream);
int b2r_mc_emit(const float* field, int n0, int n1, int n2, float level, float spacing, float ox, float oy, float oz,
                const void* scratch, float* verts, int* faces, void* stream);
/* Vertex normals of the same mesh: given the scratch b2r_mc_count wrote for the same field and level, writes normals[V,3] (fp32)
 * in the vertex order of b2r_mc_emit.  g(p) is the field's gradient at lattice point p by differences along each axis,
 * 0.5 (f[i+1] - f[i-1]) inside and f[i+1] - f[i] / f[i] - f[i-1] on the faces (np.gradient's scheme; the spacing is isotropic
 * and dropped).  The vertex on the edge p -> p + e_a with parameter t gets n = g(p) + t (g(p + e_a) - g(p)) divided by |n|,
 * every operation rounded separately (sqrt and division correctly rounded), so it points toward increasing field, the side
 * the triangle normals face.  A zero-length n (a flat field there) gives (0, 0, 0). */
int b2r_mc_normals(const float* field, int n0, int n1, int n2, float level, const void* scratch, float* normals, void* stream);

/* ---- narrow-band marching cubes (no reference counterpart: the density query of create_mesh limited to the surface's bricks) --
 * Bricks of `stride` (>= 2) cells per axis: an axis of n points has nb = ceil((n - 1) / stride) bricks; brick b covers the cells
 * [b stride, min((b + 1) stride, n - 1)) and its coarse corners are the points min(b stride, n - 1), min((b + 1) stride, n - 1).
 * Flags are one byte per brick, [nb0, nb1, nb2], axis 0 slowest.  "Below" is field < level, NaN not below (b2r_mc_count).
 *   b2r_band_select:   given a field whose values are valid at every coarse corner (+inf elsewhere keeps the rest above the
 *                      level), flags[b] = 1 for every brick within one brick (26-neighbourhood, clamped at the box) of a brick
 *                      whose 8 coarse corners are not all on the same side of the level, 0 otherwise; index[] = the linear indices,
 *                      ascending, of the needed points: every point of the closure of a flagged brick and every point one step
 *                      along one axis from such a point (the differences of b2r_mc_normals read them); count_dev[0] = their number
 *                      M, one long long in DEVICE memory.  index must hold n0*n1*n2 ints.  scratch: b2r_band_scratch_bytes(n0, n1,
 *                      n2, stride) bytes, 16-byte aligned (0 for a shape b2r_mc_scratch_bytes rejects or stride < 2).
 *   b2r_lattice_rows:  x[r] = (point, direction) of row index[r] of the grid_n or lattice_dims description `in`, for r < m, with
 *                      the point formula of those rows (so an MLP on x equals the MLP on the description at those rows).
 *                      PRECONDITION: every index[r] lies in [0, in->n_rays) (not checked: the indices are in device memory).
 *   b2r_mc_count_band: b2r_mc_count limited to the flagged bricks: a cell outside a flagged brick gets configuration 0, and a
 *                      crossing edge is counted only when it is an edge of a cell in a flagged brick.  b2r_mc_emit and
 *                      b2r_mc_normals then give the mesh of b2r_mc_count with the faces of the other cells and the vertices on
 *                      no counted edge removed, in the same relative order.  scratch as for b2r_mc_count. */
size_t b2r_band_scratch_bytes(int n0, int n1, int n2, int stride);
int b2r_band_select(const float* field, int n0, int n1, int n2, float level, int stride, void* scratch, unsigned char* flags,
                    int* index, long long* count_dev, void* stream);
int b2r_lattice_rows(const b2r_mlp_input* in, const int* index, long long m, float* x, void* stream);
int b2r_mc_count_band(const float* field, int n0, int n1, int n2, float level, const unsigned char* flags, int stride,
                      void* scratch, long long* totals_dev, void* stream);

/* ---- connected components of a triangle mesh (no reference counterpart: clean-up of exported meshes) ----------------------
 * faces[F,3] (int32) index verts[V,3]; two vertices are connected when a face has them as (v0,v1) or (v1,v2).  PRECONDITION:
 * every face index lies in [0, n_verts) (not checked: the indices are in device memory; ops.py checks them first).  Counts are
 * in [0, INT32_MAX]; faces / labels / verts may be NULL only when their count is 0.  scratch: b2r_mesh_cc_scratch_bytes(V, F)
 * bytes, 16-byte aligned (0 for counts outside [0, INT32_MAX]).
 *   b2r_mesh_cc_label:   labels[V] (int32) = the smallest vertex index of each vertex's component (a vertex no face uses is its
 *                        own component), the same whatever the schedule of the union-find that computes it.
 *   b2r_mesh_cc_select:  given those labels, marks the vertices and faces of every component with t triangles where t >= 1 and
 *                        t >= ratio * t_max in float64 (t_max = the largest component's count; ratio finite, in [0, 1]; ratio 0
 *                        keeps everything) and writes totals_dev[2] = (V', F'), two long long in DEVICE memory.
 *   b2r_mesh_cc_compact: given the scratch b2r_mesh_cc_select wrote for the same mesh, writes the kept vertices (and normals,
 *                        when normals_or_null is not NULL) to verts_out[V',3] / normals_out[V',3] and the kept faces, indices
 *                        remapped to the new vertex order, to faces_out[F',3]; both in their original relative order.  Its
 *                        output pointers must be valid whenever n_verts / n_faces is not 0, so the caller reads (V', F') first
 *                        and skips the call when V' = 0 (nothing is kept). */
size_t b2r_mesh_cc_scratch_bytes(long long n_verts, long long n_faces);
int b2r_mesh_cc_label(const int* faces, long long n_faces, long long n_verts, int* labels, void* scratch, void* stream);
int b2r_mesh_cc_select(const int* faces, long long n_faces, long long n_verts, const int* labels, float ratio, void* scratch,
                       long long* totals_dev, void* stream);
int b2r_mesh_cc_compact(const float* verts, const float* normals_or_null, const int* faces, long long n_faces, long long n_verts,
                        const void* scratch, float* verts_out, float* normals_out, int* faces_out, void* stream);

/* ---- Taubin smoothing and normals of a triangle mesh (no reference counterpart: clean-up of exported meshes) ---------------
 * Same mesh conventions and PRECONDITION as the connected components above (faces[F,3] int32 index verts[V,3] fp32, every index
 * in [0, n_verts), counts in [0, INT32_MAX], NULL allowed only for a count of 0).  A corner of vertex v is (f, c) with
 * faces[f][c] == v; v's corners are taken in ascending (f, c), a face listing v twice gives two.  scratch:
 * b2r_mesh_adj_scratch_bytes(V, F) bytes, 16-byte aligned (0 for counts outside [0, INT32_MAX]; with V = 0 the calls do
 * nothing and scratch may be NULL).
 *   b2r_mesh_adjacency: builds each vertex's corner list into scratch, exactly ordered whatever the schedule.
 *   b2r_mesh_smooth:    given that scratch, writes verts_out[V,3] = verts after `iterations` (>= 0) Taubin iterations, each a
 *                       half-step with w = 0.5f then one with w = -0.53f.  A half-step is Jacobi: for v with k > 0 corners,
 *                       s = 0, then s += p[faces[f][(c+1)%3]], s += p[faces[f][(c+2)%3]] per corner in order; m = s / (float)(2k);
 *                       p'[v] = p[v] + w (m - p[v]); a vertex with k = 0 keeps p.  verts_out may equal verts.
 *   b2r_mesh_normals:   given that scratch, writes normals[V,3], the sum over v's corners in order of the face normal
 *                       (p[f1]-p[f0]) x (p[f2]-p[f0]) in the face's own corner order, divided by sqrt((x x + y y) + z z), or
 *                       (0, 0, 0) when that is 0.
 * Every float operation is rounded separately (no FMA; division and sqrt correctly rounded), so the result is reproducible bit for
 * bit.  The scratch stays valid for any number of _smooth / _normals calls on the same faces. */
size_t b2r_mesh_adj_scratch_bytes(long long n_verts, long long n_faces);
int b2r_mesh_adjacency(const int* faces, long long n_faces, long long n_verts, void* scratch, void* stream);
int b2r_mesh_smooth(const float* verts, long long n_faces, long long n_verts, int iterations, void* scratch, float* verts_out,
                    void* stream);
int b2r_mesh_normals(const float* verts, long long n_faces, long long n_verts, const void* scratch, float* normals, void* stream);

/* ---- quadric edge collapse of a triangle mesh (no reference counterpart: size budget of exported meshes) ------------------
 * Same mesh conventions and PRECONDITION as above.  The rules (frozen vertices, valid edges, placement, cost, selection) are
 * those of oracle/mesh_decimation.py; every float64 / float32 operation is rounded separately, so the result is reproducible bit
 * for bit.  quadrics are [V,10] float64 (the upper triangle of the symmetric 4x4, row by row).  adj_scratch is the scratch of
 * b2r_mesh_adjacency built on the same (faces, n_faces, n_verts); scratch is b2r_mesh_decimate_scratch_bytes(V, F) bytes,
 * 16-byte aligned (0 for counts outside [0, INT32_MAX]).  Scratch sized for larger counts serves smaller ones.
 *   b2r_mesh_quadrics:        quadrics[v] = the sum over v's corners in ascending (f, c) of the area-weighted plane quadric of
 *                             the corner's face.
 *   b2r_mesh_decimate_round:  selects a set of independent valid edges.  Writes sel_keys[V] (int64): at the smaller end a of a
 *                             selected edge the float64 bits of its cost (>= 0, so they order like the cost), INT64_MAX
 *                             everywhere else; counts_dev[0] = the selected edges S, counts_dev[1] = n_faces - 2 S.
 *   b2r_mesh_decimate_compact: after _round on the same mesh and scratch, collapses the selected edges, or with cut_or_null
 *                             (int64 [2] on the device: cost bits, a) only those with (sel_keys[a], a) <= cut, and writes the
 *                             surviving vertices (collapsed survivors at their placement), their quadrics (Q_a + Q_b on
 *                             collapse) and the surviving faces, remapped, each in its original order.  verts_out / quadrics_out
 *                             hold V - k rows and faces_out F - 2k, k the number of collapses. */
size_t b2r_mesh_decimate_scratch_bytes(long long n_verts, long long n_faces);
int b2r_mesh_quadrics(const float* verts, long long n_faces, long long n_verts, const void* adj_scratch, double* quadrics, void* stream);
int b2r_mesh_decimate_round(const float* verts, const double* quadrics, long long n_faces, long long n_verts, const void* adj_scratch,
                            void* scratch, long long* sel_keys, long long* counts_dev, void* stream);
int b2r_mesh_decimate_compact(const float* verts, const double* quadrics, const int* faces, long long n_faces, long long n_verts,
                              const long long* sel_keys, const long long* cut_or_null, void* scratch, float* verts_out,
                              double* quadrics_out, int* faces_out, void* stream);

/* ---- texture atlas of a triangle mesh (no reference counterpart: colour detail of exported meshes beyond the vertices) -----
 * Same mesh conventions and PRECONDITION as above; the layout, a pure function of (n_faces F, size R), is that of
 * oracle/mesh_texture.py.  R is in [16, 16384].  Faces 2k and 2k+1 share cell k; the P = ceil(F / 2) cells sit C per row, C the
 * smallest integer with C C >= P, each s = R / C texels square, with top-left texel (X, Y) = ((k % C) s, (k / C) s), row 0 at
 * the top.  F must be at most 2 (R / 4)^2, so that s >= 4.  With L = s - 3, face 2k's corners 0, 1, 2 sit at the local texel
 * centres (0, 0), (L, 0), (0, L) and face 2k+1's at (s-1, s-1), (2, s-1), (s-1, 2).  A local texel (x, y) is baked for face
 * 2k+1 when x + y >= s and that face exists, for face 2k otherwise, so a bilinear lookup inside a face's UV triangle reads only
 * texels baked for that face.  Texel weights: (a, b) = (x, y) for face 2k, (s-1-x, s-1-y) for 2k+1; (w0, w1, w2) =
 * ((L-a-b) / L, a / L, b / L) when a + b <= L, (0, a / (a+b), b / (a+b)) otherwise.  Row r = k s^2 + y s + x, for the
 * P s^2 rows of the used cells; [row_begin, +row_count) must lie within them.  Every float operation is rounded separately (no
 * FMA; division and sqrt correctly rounded), so the results are reproducible bit for bit.
 *   b2r_mesh_atlas_uvs:     uvs[F,3,2] (fp32): corner (x, y) of cell (X, Y) gets u = ((X+x) + 0.5) / R, v = 1 - ((Y+y) + 0.5) / R.
 *   b2r_mesh_atlas_rows:    x[row_count,6] (fp32): row row_begin + i gets [p, -n^], p = (w0 v0 + w1 v1) + w2 v2 of its face's
 *                           vertices per component, n^ the same sum of the vertex normals divided by sqrt((x x + y y) + z z), or
 *                           (0, 0, 0) when that is 0 (the MLP query of b2r_mlp_tc_fwd on x then sees the surface point along -n^).
 *   b2r_mesh_atlas_texture: raw[row_count,4] (fp32, 16-byte aligned; the MLP output on those rows): writes the b2r_to8b quantisation
 *                           of raw[i][0..2] into the texel of row row_begin + i of texture[R,R,3] (uint8); other texels are left
 *                           as they are (the caller zeroes the texture first). */
int b2r_mesh_atlas_uvs(long long n_faces, int size, float* uvs, void* stream);
int b2r_mesh_atlas_rows(const float* verts, const float* normals, const int* faces, long long n_faces, int size, long long row_begin,
                        long long row_count, float* x, void* stream);
int b2r_mesh_atlas_texture(const float* raw, long long n_faces, int size, long long row_begin, long long row_count,
                           unsigned char* texture, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B2R_H_ */
