"""Host-side operators over the C ABI of libb2r.so (include/b2r.h).

Each function mirrors one stage of the reference's render path and calls exactly one CUDA entry
point; the autograd-aware ones (``composite``, ``mlp``) own their saved-for-backward buffers, as
torch autograd does for the reference (nerf/train_nerf.py:167).  Everything here requires CUDA
tensors and raises otherwise -- there is no CPU or PyTorch-op fallback.
"""
from __future__ import annotations

import ctypes as C
import math
import threading
import weakref

import numpy as np
import torch

from . import _lib, models
from ._lib import LastSample, MlpInput, check, lib, ptr

# MLP arithmetic used when no gradient is required: "bf16" = fused tcgen05 kernel (mlp_tc.cu),
# "fp32" = layer-wise path on CUDA-core FMAs (mlp_f32.cu, sgemm.cuh), "tf32" = the same layer-wise path with its GEMMs on
# tcgen05 kind::tf32 (tgemm.cuh).  The arithmetic of the gradient path is _GRAD_PRECISION below.
_MLP_PRECISION = "bf16"


def set_mlp_precision(p: str) -> str:
    global _MLP_PRECISION
    if p not in ("bf16", "fp32", "tf32"):
        raise ValueError("precision must be 'bf16', 'fp32' or 'tf32'")
    old, _MLP_PRECISION = _MLP_PRECISION, p
    return old


def get_mlp_precision() -> str:
    return _MLP_PRECISION


# Arithmetic of the path used whenever gradients are required, one engine each: "fp32" = layer-wise, CUDA-core FMAs (sgemm.cuh;
# exact: the path the gradient parity fixtures are checked on), "tf32" = the same layer-wise algorithm with every GEMM on the
# tensor cores (tgemm.cuh, tcgen05 kind::tf32, fp32 accumulate), "bf16" (default) = the fused tensor-core training path of all
# three model kinds (mlp_tc.cu / mlp_tc_siren.cu forward with kept bf16 activations + mlp_tc_train.cu reverse mode, fp32 master
# weights / gradients): the same arithmetic class the no-grad render path uses by default.
_GRAD_PRECISION = "bf16"


def set_grad_precision(p: str) -> str:
    global _GRAD_PRECISION
    if p not in ("fp32", "tf32", "bf16"):
        raise ValueError("grad precision must be 'fp32', 'tf32' or 'bf16'")
    old, _GRAD_PRECISION = _GRAD_PRECISION, p
    return old


def get_grad_precision() -> str:
    return _GRAD_PRECISION


# ---- the last interval of every ray (nerf/render.py:92: dists[-1] = 1e10) ------------------------------------------------------
# alpha_last is a step function of sign(sigma_last), so a bf16-rounded density that crosses zero at the LAST sample flips a whole
# ray (SURVEY.md 0).  The bf16 kernels list the rays whose last pre-relu sigma is inside the bf16 error band
#     |sigma_pre| <= rel * scale + abs      (include/b2r.h: b2r_last_sample; scale = sum |w_sigma h| for the ReLU trunk,
#                                            |w_sigma|_1 for the sine trunks)
# and those rows (a few % of the rays) are re-evaluated by the exact fp32 engine.  On by default for every no-grad bf16 render;
# `exact_last_sample=False` / set_exact_last_sample(False) gives the raw bf16 result.  rel: >= 8 standard deviations of the measured
# bf16 error of sigma_pre relative to the scale (DESIGN.md 3.2).
_EXACT_LAST = True
# Passes that carry gradients (ops.mlp under autograd, NerfTrainStep) evaluate the RAW bf16 forward by default: the mixed-precision
# training recipe (DESIGN.md 3.3).  d sigma_last is zero on both sides of the step, so only the forward value of ~0.2 % of the rays
# differs, and the two host syncs + fp32 launches per pass would cost ~8 % of a training step.  set_exact_last_sample(train=True)
# makes the autograd forward apply the same check as the render (its reverse mode is unaffected).
_EXACT_LAST_TRAIN = False
_LAST_REL = {models.KIND_NERF: 2.0 ** -7, models.KIND_FILM: 2.0 ** -9, models.KIND_SIREN: 2.0 ** -9}
_LAST_ABS = 1e-6
last_sample_stats = {"calls": 0, "rays": 0, "flagged": 0}      # running totals (bench / tests report the flagged fraction)


def set_exact_last_sample(flag: bool | None = None, train: bool | None = None) -> bool:
    """Switch the last-sample sign check of no-grad bf16 passes (``flag``) and / or of the autograd training forward (``train``).
    Returns the previous value of ``flag``'s switch."""
    global _EXACT_LAST, _EXACT_LAST_TRAIN
    old = _EXACT_LAST
    if flag is not None:
        _EXACT_LAST = bool(flag)
    if train is not None:
        _EXACT_LAST_TRAIN = bool(train)
    return old


def get_exact_last_sample() -> bool:
    return _EXACT_LAST


def set_last_sample_band(kind: int, rel: float, abs_: float | None = None) -> None:
    """Override the flagging band of one model kind (calibration runs)."""
    global _LAST_ABS
    _LAST_REL[kind] = float(rel)
    if abs_ is not None:
        _LAST_ABS = float(abs_)


def _last_sample_begin(kind: int, rows: int, spr: int, dev):
    """(LastSample struct, tensors to keep alive) for a launch of `rows` rows with `spr` samples per ray."""
    n_rays = rows // spr
    count = torch.zeros((1,), dtype=torch.int32, device=dev)
    ids = torch.empty((max(n_rays, 1),), dtype=torch.int32, device=dev)
    ls = LastSample(int(spr), int(n_rays), count.data_ptr(), ids.data_ptr(), float(_LAST_REL[kind]), float(_LAST_ABS))
    return ls, (count, ids)


def _with_last_sample(want: bool, launch, kind: int, inp, spr: int, raw, weights, n_latents: int = 1,
                      rows_per_latent: int = 0) -> None:
    """``launch(ls)`` of a bf16 forward into ``raw`` (ls: a LastSample pointer, or None).  With ``want`` the forward lists the
    rays whose last sample is in the bf16 error band; their count is read (the one host sync of the pass) and those last
    samples are re-evaluated in fp32 with ``weights = (flat, film | None, use_dir)``."""
    if not want:
        launch(None)
        return
    flat, film, use_dir = weights
    ls, (count, ids) = _last_sample_begin(kind, raw.shape[0], spr, raw.device)
    launch(C.byref(ls))
    n_rays = ids.shape[0]
    n = min(int(count.item()), n_rays)
    last_sample_stats["calls"] += 1
    last_sample_stats["rays"] += int(n_rays)
    last_sample_stats["flagged"] += n
    if n == 0:
        return
    ws_bytes = lib().b2r_mlp_f32_workspace_bytes(kind, n, 0) + ((n * 4 + 15) & ~15)
    ws = torch.empty((ws_bytes // 4,), dtype=torch.float32, device=raw.device)
    check(lib().b2r_mlp_f32_last_sigma(kind, ptr(flat), ptr(film), int(use_dir), int(n_latents), int(rows_per_latent), C.byref(inp), int(spr),
                                       ids.data_ptr(), n, ptr(raw), ptr(ws), ws_bytes, _stream(raw)), "b2r_mlp_f32_last_sigma")


def _cuda_f32(t: torch.Tensor, name: str) -> torch.Tensor:
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError(f"{name} must be a CUDA tensor: the B200 render path has no CPU fallback")
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _stream(t: torch.Tensor) -> int:
    return torch.cuda.current_stream(t.device).cuda_stream


def _model_args(model):
    """``(net, kind, use_dir, params, device)`` of a radiance-field model: ``net`` unwrapped from DataParallel, ``params`` in
    flat order (models.param_list); TypeError for an unknown model, RuntimeError unless its parameters are on a CUDA device."""
    kind = models.model_kind(model)
    net = model.module if isinstance(model, torch.nn.DataParallel) else model
    ps = models.param_list(net, kind)
    if ps[0].device.type != "cuda":
        raise RuntimeError("model parameters must live on a CUDA device: the B200 render path has no CPU fallback")
    return net, kind, bool(getattr(net, "use_dir", True)), ps, ps[0].device


# ---- K1 / K2 ---------------------------------------------------------------------------------------
def raygen(width: int, height: int, focal, c2w, begin: int = 0, count: int | None = None,
           device=None) -> torch.Tensor:
    """rows [begin, begin+count) of the [H*W,2,3] ray table (get_rays + render_image reshaping,
    nerf/render.py:7-23,151-154)."""
    device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
    c2w_np = c2w.detach().cpu().numpy() if isinstance(c2w, torch.Tensor) else np.asarray(c2w)
    f64 = (1 if isinstance(focal, np.float64) else 0) | (2 if c2w_np.dtype == np.float64 else 0)
    m = np.ascontiguousarray(c2w_np[:3, :4], dtype=np.float64)
    count = width * height - begin if count is None else count
    out = torch.empty((count, 2, 3), dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        check(lib().b2r_raygen(m.ctypes.data_as(C.POINTER(C.c_double)), int(width), int(height), float(focal), f64,
                               int(begin), int(count), ptr(out), _stream(out)), "b2r_raygen")
    return out


def raygen_poses(width: int, height: int, focal, poses: torch.Tensor, pose_f64: bool = False) -> torch.Tensor:
    """The [B*H*W,2,3] ray table of B full images whose poses are a DEVICE tensor [B,3|4,4] (b2r_raygen_poses): per pose bit-identical
    to raygen(), but nothing step-dependent is a kernel argument, so it can sit inside a captured CUDA graph (train_step.GeneratorStep).
    ``pose_f64``: the poses came from float64 numpy matrices (numpy's promotion, see b2r_raygen); float32 poses convert exactly."""
    if not isinstance(poses, torch.Tensor) or not poses.is_cuda or poses.dim() != 3 or poses.shape[1] < 3 or poses.shape[2] != 4:
        raise RuntimeError("poses must be a CUDA tensor [B,3,4] or [B,4,4]")
    p = poses[:, :3, :].to(torch.float64).contiguous()
    b = p.shape[0]
    f64 = (1 if isinstance(focal, np.float64) else 0) | (2 if pose_f64 else 0)
    out = torch.empty((b * int(width) * int(height), 2, 3), dtype=torch.float32, device=p.device)
    with torch.cuda.device(p.device):
        check(lib().b2r_raygen_poses(ptr(p), b, int(width), int(height), float(focal), f64, ptr(out), _stream(out)), "b2r_raygen_poses")
    return out


_linspace_cache: dict = {}


def host_linspace(a: float, b: float, n: int, device) -> torch.Tensor:
    """torch.linspace(a, b, n) made on the HOST (its last-bit rounding is a contract, SURVEY A.2) and kept on the device, cached per
    (a, b, n, device): callers inside a captured CUDA graph must not issue a host-to-device copy."""
    key = (float(a), float(b), int(n), str(device))
    t = _linspace_cache.get(key)
    if t is None:
        if len(_linspace_cache) >= 64:
            _linspace_cache.clear()
        t = torch.linspace(float(a), float(b), steps=int(n), device="cpu").to(device)
        _linspace_cache[key] = t
    return t


def stratified_z(z_lin: torch.Tensor, t_rand: torch.Tensor):
    """z_vals[N,Sc], mids[Sc-1] from linspace(near,far,Sc) and the jitter (nerf/render.py:123-132)."""
    z_lin = _cuda_f32(z_lin, "z_lin")
    t_rand = _cuda_f32(t_rand, "t_rand")
    n, sc = t_rand.shape
    z = torch.empty_like(t_rand)
    mids = torch.empty((sc - 1,), dtype=torch.float32, device=t_rand.device)
    with torch.cuda.device(t_rand.device):
        check(lib().b2r_stratified_z(ptr(z_lin), ptr(t_rand), n, sc, ptr(z), ptr(mids), _stream(z)), "b2r_stratified_z")
    return z, mids


# ---- K4 ----------------------------------------------------------------------------------------------
def _dirs_view(rays_d: torch.Tensor):
    """(tensor to keep alive, pointer, stride in floats) for N direction vectors."""
    if rays_d.dim() != 2 or rays_d.shape[1] != 3:
        raise RuntimeError("rays_d must be [N,3]")
    if rays_d.dtype == torch.float32 and rays_d.is_cuda and rays_d.stride(1) == 1 and rays_d.stride(0) >= 3:
        return rays_d, rays_d.data_ptr(), rays_d.stride(0)          # e.g. rays[:,1] of an [N,2,3] table: stride 6
    d = _cuda_f32(rays_d, "rays_d")
    return d, d.data_ptr(), 3


def _aligned16(t: torch.Tensor) -> torch.Tensor:
    """float4 accesses need 16-byte aligned rows: a contiguous-but-offset view such as raw[1:] is copied (the reference accepts it)."""
    return t if t.data_ptr() % 16 == 0 else t.clone()


def composite_forward(raw, z, rays_d, want_weights: bool = True, packed_out: torch.Tensor | None = None):
    """b2r_composite_fwd without autograd: (rgb, depth, acc, weights | None, (raw, z, dirs tensor, dirs stride)).
    packed_out [N,5] (optional): the kernel writes (rgb, depth, acc) straight into its rows and the returned maps are views of it
    (the rank's slice of the gathered frame buffer, dist.py)."""
    raw = _aligned16(_cuda_f32(raw, "raw"))
    z = _cuda_f32(z, "z_vals")
    keep, dptr, dstride = _dirs_view(rays_d.detach())
    n, s = z.shape
    dev = z.device
    if packed_out is not None:
        if tuple(packed_out.shape) != (n, 5) or packed_out.dtype != torch.float32 or not packed_out.is_cuda or not packed_out.is_contiguous():
            raise RuntimeError(f"packed_out must be a contiguous fp32 CUDA tensor [{n},5]")
        rgb, depth, acc = packed_out[:, :3], packed_out[:, 3], packed_out[:, 4]
        strides = (5, 5, 5)
    else:
        rgb = torch.empty((n, 3), dtype=torch.float32, device=dev)
        depth = torch.empty((n,), dtype=torch.float32, device=dev)
        acc = torch.empty((n,), dtype=torch.float32, device=dev)
        strides = (3, 1, 1)
    w = torch.empty((n, s), dtype=torch.float32, device=dev) if want_weights else None
    if n > 0:
        with torch.cuda.device(dev):
            check(lib().b2r_composite_fwd_strided(ptr(raw), ptr(z), dptr, dstride, n, s, rgb.data_ptr(), strides[0], depth.data_ptr(), strides[1],
                                                  acc.data_ptr(), strides[2], ptr(w), _stream(z)), "b2r_composite_fwd")
    return rgb, depth, acc, w, (raw, z, keep, dstride)


def composite_backward(ctx4, g_rgb, g_depth=None, g_acc=None) -> torch.Tensor:
    """b2r_composite_bwd: d_raw[N,S,4] from the upstream gradients of (rgb, depth, acc); ctx4 = composite_forward's last item."""
    raw, z, keep, dstride = ctx4
    n, s = z.shape
    d_raw = torch.empty(raw.shape, dtype=torch.float32, device=raw.device)
    if n == 0:
        return d_raw
    g_rgb = _cuda_f32(g_rgb, "g_rgb")
    g_depth = None if g_depth is None else _cuda_f32(g_depth, "g_depth")
    g_acc = None if g_acc is None else _cuda_f32(g_acc, "g_acc")
    with torch.cuda.device(z.device):
        check(lib().b2r_composite_bwd(ptr(raw), ptr(z), keep.data_ptr(), dstride, n, s, ptr(g_rgb), ptr(g_depth), ptr(g_acc),
                                      ptr(d_raw), _stream(z)), "b2r_composite_bwd")
    return d_raw


def composite_loss_backward(raw, z, rays_d, target_rgb, target_acc, ray_weight, inv_count, alpha_weight: float, sums: torch.Tensor) -> torch.Tensor:
    """b2r_composite_loss_bwd: the train_nerf.py:157-166 loss and the composite's reverse mode in one launch -> d_raw[N,S,4];
    sums[0] += sum w (rgb - target)^2, sums[1] += sum w (acc - target_acc)^2 (2 floats, caller zeroes)."""
    raw = _aligned16(_cuda_f32(raw, "raw"))
    z = _cuda_f32(z, "z_vals")
    keep, dptr, dstride = _dirs_view(rays_d.detach())
    n, s = z.shape
    d_raw = torch.empty(raw.shape, dtype=torch.float32, device=raw.device)
    if n > 0:
        with torch.cuda.device(z.device):
            check(lib().b2r_composite_loss_bwd(ptr(raw), ptr(z), dptr, dstride, n, s, ptr(target_rgb), ptr(target_acc), ptr(ray_weight), ptr(inv_count),
                                               float(alpha_weight), ptr(d_raw), ptr(sums), _stream(z)), "b2r_composite_loss_bwd")
    del keep
    return d_raw


class _Composite(torch.autograd.Function):
    @staticmethod
    def forward(ctx, raw, z, rays_d, want_weights):
        rgb, depth, acc, w, (raw, z, keep, dstride) = composite_forward(raw, z, rays_d, want_weights)
        dev = z.device
        ctx.save_for_backward(raw, z, keep)
        ctx.dstride = dstride
        if w is None:
            w = torch.empty((0,), device=dev)
        ctx.mark_non_differentiable(w)
        return rgb, depth, acc, w

    @staticmethod
    def backward(ctx, g_rgb, g_depth, g_acc, _g_w):
        raw, z, keep = ctx.saved_tensors
        if g_rgb is None:
            g_rgb = torch.zeros((z.shape[0], 3), device=z.device)
        return composite_backward((raw, z, keep, ctx.dstride), g_rgb, g_depth, g_acc), None, None, None


def composite(raw, z_vals, rays_d, want_weights: bool = True, packed_out: torch.Tensor | None = None):
    """raw_to_outputs (nerf/render.py:78-103): (rgb[N,3], depth[N], acc[N], weights[N,S] or None).
    Differentiable wrt ``raw``; the weights are returned detached (the reference only uses them
    through sample_pdf, whose result is detached, nerf/render.py:141).  ``packed_out`` [N,5] (no-grad passes only): the three
    maps are written into its rows and returned as views (composite_forward)."""
    if packed_out is not None:
        if torch.is_grad_enabled() and isinstance(raw, torch.Tensor) and raw.requires_grad:
            raise RuntimeError("packed_out is for passes without gradients")
        rgb, depth, acc, w, _ = composite_forward(raw.detach(), z_vals, rays_d, want_weights, packed_out)
        return rgb, depth, acc, w
    rgb, depth, acc, w = _Composite.apply(raw, z_vals, rays_d, bool(want_weights))
    return rgb, depth, acc, (w if want_weights else None)


# ---- K5 / K6 -------------------------------------------------------------------------------------------
def sample_pdf(bins: torch.Tensor, weights: torch.Tensor, n_samples: int, u: torch.Tensor | None = None,
               z_coarse: torch.Tensor | None = None, want_samples: bool = True, want_cdf: bool = False):
    """sample_pdf (nerf/render.py:27-56) and, when ``z_coarse`` is given, the sort-merge of :142.

    ``weights`` may be a strided view such as ``w[:, 1:-1]`` (no copy).  Returns a dict with the
    requested tensors: samples[N,Sf], sorted[N,Sc+Sf], cdf[N,nb]."""
    if not weights.is_cuda:
        raise RuntimeError("weights must be a CUDA tensor")
    weights = weights.detach()
    if weights.dtype != torch.float32 or weights.stride(1) != 1:
        weights = weights.float().contiguous()
    n, nw = weights.shape
    nb = nw + 1
    dev = weights.device
    bins = bins.detach()
    if bins.dim() == 1 or bins.stride(0) == 0:
        b = _cuda_f32(bins if bins.dim() == 1 else bins[0], "bins")
        b_stride = 0
    else:
        b = _cuda_f32(bins, "bins")
        b_stride = nb
    if b.shape[-1] != nb:
        raise RuntimeError(f"bins has {b.shape[-1]} entries, expected len(weights)+1 = {nb}")
    if u is None:
        u = torch.linspace(0.0, 1.0, steps=int(n_samples), device="cpu").to(dev)   # host-made: its rounding is a contract
    u = _cuda_f32(u, "u")
    sf = int(n_samples)
    if u.dim() != 1 or u.numel() != sf:
        # the kernel reads exactly n_samples entries and merges them as a SORTED list (non-decreasing, like torch.linspace(0, 1, n))
        raise RuntimeError(f"u must be a 1-D tensor of n_samples = {sf} non-decreasing values, got shape {tuple(u.shape)}")
    samples = torch.empty((n, sf), dtype=torch.float32, device=dev) if want_samples else None
    cdf = torch.empty((n, nb), dtype=torch.float32, device=dev) if want_cdf else None
    merged, zc, sc = None, None, 0
    if z_coarse is not None:
        zc = _cuda_f32(z_coarse.detach(), "z_coarse")
        sc = zc.shape[1]
        merged = torch.empty((n, sc + sf), dtype=torch.float32, device=dev)
    if n == 0:
        return {"samples": samples, "sorted": merged, "cdf": cdf}
    with torch.cuda.device(dev):
        check(lib().b2r_sample_pdf(ptr(b), b_stride, weights.data_ptr(), weights.stride(0), ptr(u), n, nb, sf, ptr(zc), sc,
                                   ptr(samples), ptr(merged), ptr(cdf), _stream(weights)), "b2r_sample_pdf")
    return {"samples": samples, "sorted": merged, "cdf": cdf}


# ---- K3 / K7 / K8 ------------------------------------------------------------------------------------------
_pack_cache: "weakref.WeakKeyDictionary" = weakref.WeakKeyDictionary()
_pack_bwd_cache: "weakref.WeakKeyDictionary" = weakref.WeakKeyDictionary()
_pack_lock = threading.Lock()       # nn.DataParallel renders from one thread per GPU (pi_GAN/train.py:50): guard the shared dicts


def invalidate_packed(model) -> None:
    """Forget the cached bf16 weight images of `model` (call after changing its parameters in a way torch cannot see,
    e.g. a kernel writing the flat master buffer: train_step.NerfTrainStep does this after every step)."""
    with _pack_lock:
        _pack_cache.pop(model, None)
        _pack_bwd_cache.pop(model, None)


def _packed_weights(model, kind: int, flat: torch.Tensor, film: torch.Tensor | None, use_dir: bool) -> torch.Tensor:
    """bf16 / swizzled copy of the weights for the tensor-core kernel, cached per model and
    invalidated when any parameter (or the FiLM tensor) changes in place or is replaced."""
    ps = models.param_list(model, kind)
    key = tuple((p.data_ptr(), p._version) for p in ps)
    # FiLM tensors are rebuilt per latent (set_film_params) and may reuse a freed address, so a pointer /
    # version key cannot prove they are unchanged: FiLM models are re-packed on every call (~10 us).
    with _pack_lock:
        hit = _pack_cache.get(model) if film is None else None
    if hit is not None and hit[0] == key:
        return hit[1]
    packed = pack_tc(flat, kind, film, use_dir)
    if film is None:
        with _pack_lock:
            _pack_cache[model] = (key, packed)
    return packed


def _make_input(rays, z, x, grid, lattice=None):
    """(MlpInput, rows, tensors to keep alive)"""
    inp = MlpInput()
    if lattice is not None:
        dims, origin, voxel, begin, count = lattice
        inp.lattice_dims[:] = [int(d) for d in dims]
        inp.lattice_origin[:] = [float(o) for o in origin]
        inp.lattice_voxel, inp.grid_begin, inp.n_rays, inp.n_samples = float(voxel), int(begin), int(count), 1
        return inp, int(count), ()
    if rays is not None:
        rays = _cuda_f32(rays, "rays")
        z = _cuda_f32(z, "z_vals")
        if rays.dim() != 3 or tuple(rays.shape[1:]) != (2, 3) or z.shape[0] != rays.shape[0]:
            raise RuntimeError("rays must be [N,2,3] and z [N,S]")
        inp.rays, inp.z, inp.n_rays, inp.n_samples = rays.data_ptr(), z.data_ptr(), rays.shape[0], z.shape[1]
        return inp, rays.shape[0] * z.shape[1], (rays, z)
    if x is not None:
        x = _cuda_f32(x, "x")
        if x.dim() != 2 or x.shape[1] != 6:
            raise RuntimeError("x must be [M,6] = (position, direction)")
        inp.x, inp.n_rays, inp.n_samples = x.data_ptr(), x.shape[0], 1
        return inp, x.shape[0], (x,)
    n, begin, count = grid
    inp.grid_n, inp.grid_begin, inp.n_rays, inp.n_samples = int(n), int(begin), int(count), 1
    return inp, int(count), ()


def _mlp_f32_forward(kind: int, flat, film, use_dir, inp, raw, keep: int, gemm_mode: int) -> torch.Tensor:
    """b2r_mlp_f32_fwd of the rows ``inp`` describes into ``raw``; returns the workspace, which with ``keep`` = 1 holds every
    layer's output for b2r_mlp_f32_bwd.  ``gemm_mode`` 1 runs the GEMMs in tf32, 0 in fp32."""
    dev = raw.device
    ws_bytes = lib().b2r_mlp_f32_workspace_bytes(kind, raw.shape[0], keep)
    ws = torch.empty((max(ws_bytes, 16) // 4,), dtype=torch.float32, device=dev)
    with torch.cuda.device(dev):
        check(lib().b2r_mlp_f32_fwd(kind, ptr(flat), ptr(film), int(use_dir), C.byref(inp), ptr(raw), ptr(ws), ws_bytes, keep,
                                    gemm_mode, _stream(flat)), "b2r_mlp_f32_fwd")
    return ws


class _MlpF32(torch.autograd.Function):
    """fp32 forward that keeps every layer's output, and its reverse mode (K8)."""

    @staticmethod
    def forward(ctx, flat, film, kind, use_dir, rays, z, x, gemm_mode):
        inp, rows, keep = _make_input(rays, z, x, None)
        raw = torch.empty((rows, 4), dtype=torch.float32, device=flat.device)
        ws = _mlp_f32_forward(kind, flat, film, use_dir, inp, raw, 1, gemm_mode)
        ctx.kind, ctx.use_dir, ctx.gemm_mode = kind, use_dir, gemm_mode
        ctx.inp, ctx.keep = inp, keep          # the rows' description and the tensors it points into
        ctx.has_film = film is not None
        ctx.save_for_backward(flat, film if film is not None else flat.new_empty(0), raw, ws)
        return raw

    @staticmethod
    def backward(ctx, d_raw):
        flat, film, raw, ws = ctx.saved_tensors
        film = film if ctx.has_film else None
        rows = raw.shape[0]
        dev = flat.device
        d_raw = _cuda_f32(d_raw, "d_raw")
        need_w = ctx.needs_input_grad[0]
        need_f = ctx.has_film and ctx.needs_input_grad[1]
        d_flat = torch.zeros_like(flat) if need_w else None
        d_film = torch.zeros_like(film) if need_f else None
        if d_flat is None and d_film is None:
            return (None,) * 8
        sc_bytes = lib().b2r_mlp_f32_bwd_scratch_bytes(ctx.kind, rows)
        scratch = torch.empty((max(sc_bytes, 16) // 4,), dtype=torch.float32, device=dev)
        with torch.cuda.device(dev):
            check(lib().b2r_mlp_f32_bwd(ctx.kind, ptr(flat), ptr(film), int(ctx.use_dir), C.byref(ctx.inp), ptr(raw), ptr(d_raw),
                                        ptr(ws), ptr(scratch), sc_bytes, ptr(d_flat), ptr(d_film), ctx.gemm_mode, _stream(flat)),
                  "b2r_mlp_f32_bwd")
        return d_flat, d_film, None, None, None, None, None, None


def _packed_bwd_weights(model, kind: int, flat: torch.Tensor) -> torch.Tensor:
    """transposed bf16 weight images for the dgrad kernel, cached per model like the forward pack."""
    ps = models.param_list(model, kind)
    key = tuple((p.data_ptr(), p._version) for p in ps)
    with _pack_lock:
        hit = _pack_bwd_cache.get(model)
    if hit is not None and hit[0] == key:
        return hit[1]
    packed = pack_tc_bwd(flat, kind)
    with _pack_lock:
        _pack_bwd_cache[model] = (key, packed)
    return packed


def pack_tc(flat: torch.Tensor, kind: int, film=None, use_dir: bool = True) -> torch.Tensor:
    """b2r_mlp_tc_pack of a flat fp32 parameter tensor (no cache)."""
    nbytes = lib().b2r_mlp_tc_packed_bytes(kind)
    if nbytes == 0:
        raise RuntimeError(f"model kind {kind} has no tensor-core path in this build")
    packed = torch.empty((nbytes,), dtype=torch.uint8, device=flat.device)
    with torch.cuda.device(flat.device):
        check(lib().b2r_mlp_tc_pack(kind, ptr(flat), ptr(film), int(use_dir), ptr(packed), _stream(flat)), "b2r_mlp_tc_pack")
    return packed


def pack_tc_bwd(flat: torch.Tensor, kind: int) -> torch.Tensor:
    """b2r_mlp_tc_pack_bwd (transposed weights for the dgrad kernel; no cache)."""
    packed = torch.empty((lib().b2r_mlp_tc_bwd_packed_bytes(kind),), dtype=torch.uint8, device=flat.device)
    with torch.cuda.device(flat.device):
        check(lib().b2r_mlp_tc_pack_bwd(kind, ptr(flat), ptr(packed), _stream(flat)), "b2r_mlp_tc_pack_bwd")
    return packed


def _pack_film_batched(flat: torch.Tensor, film: torch.Tensor, use_dir, n_latents: int) -> torch.Tensor:
    """b2r_mlp_tc_pack_film_batched: the FiLM-SIREN weights folded with each of the ``n_latents`` latents of ``film``,
    [n_latents, packed bytes] (no cache)."""
    packed = torch.empty((n_latents, lib().b2r_mlp_tc_packed_bytes(models.KIND_FILM)), dtype=torch.uint8, device=flat.device)
    with torch.cuda.device(flat.device):
        check(lib().b2r_mlp_tc_pack_film_batched(ptr(flat), ptr(film), int(use_dir), n_latents, ptr(packed), _stream(flat)),
              "b2r_mlp_tc_pack_film_batched")
    return packed


def tc_train_forward(packed: torch.Tensor, kind: int, rays: torch.Tensor | None = None, z: torch.Tensor | None = None, *,
                     x: torch.Tensor | None = None, n_latents: int = 1, rows_per_latent: int = 0, last_sample: tuple | None = None):
    """Fused bf16 training forward on the rows of (rays, z) or x: (raw[rows,4], saved activation buffer).  One latent:
    b2r_mlp_tc_train_fwd; FiLM-SIREN with ``n_latents`` > 1 (``packed`` [n_latents, bytes] from _pack_film_batched):
    b2r_mlp_tc_train_fwd_film_batched, rows [b * rows_per_latent, (b+1) * rows_per_latent) on latent b.
    ``last_sample = (flat, film | None, use_dir)``: on (rays, z) rows, the render's last-sample sign check, whose flagged rays
    are re-evaluated in fp32 with those weights (_with_last_sample); None gives the raw bf16 forward."""
    inp, rows, keep = _make_input(rays, z, x, None)
    dev = packed.device
    raw = torch.empty((rows, 4), dtype=torch.float32, device=dev)
    nbytes = lib().b2r_mlp_tc_train_saved_bytes(kind, rows)
    saved = torch.empty((max(nbytes, 16),), dtype=torch.uint8, device=dev)
    if rows == 0:
        return raw, saved

    def launch(ls):
        if n_latents == 1:
            check(lib().b2r_mlp_tc_train_fwd(kind, ptr(packed), C.byref(inp), ptr(raw), ptr(saved), nbytes, ls, _stream(packed)),
                  "b2r_mlp_tc_train_fwd")
        else:
            check(lib().b2r_mlp_tc_train_fwd_film_batched(ptr(packed), n_latents, int(rows_per_latent), C.byref(inp), ptr(raw),
                                                          ptr(saved), nbytes, ls, _stream(packed)), "b2r_mlp_tc_train_fwd_film_batched")
    spr = z.shape[1] if rays is not None else 0
    with torch.cuda.device(dev):
        _with_last_sample(last_sample is not None and spr > 0, launch, kind, inp, spr, raw, last_sample, n_latents, rows_per_latent)
    del keep
    return raw, saved


def tc_train_backward(packed_bwd: torch.Tensor, kind: int, raw: torch.Tensor, d_raw: torch.Tensor, saved: torch.Tensor,
                      d_flat: torch.Tensor) -> None:
    """b2r_mlp_tc_train_bwd: ACCUMULATES the parameter gradients into d_flat (flat fp32, state-dict order)."""
    rows = raw.shape[0]
    if rows == 0:
        return
    dev = raw.device
    d_raw = _cuda_f32(d_raw, "d_raw")
    sbytes = lib().b2r_mlp_tc_train_scratch_bytes(kind, rows)
    scratch = torch.empty((sbytes,), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        check(lib().b2r_mlp_tc_train_bwd(kind, ptr(packed_bwd), rows, ptr(raw), ptr(d_raw), ptr(saved), ptr(scratch), sbytes,
                                         ptr(d_flat), _stream(raw)), "b2r_mlp_tc_train_bwd")


def adam_step(params: torch.Tensor, grads: torch.Tensor, exp_avg: torch.Tensor, exp_avg_sq: torch.Tensor, state: torch.Tensor,
              lr0: float, decay_rate: float = 1.0, decay_steps: float = 0.0, betas=(0.9, 0.999), eps: float = 1e-8,
              grad_scale: float = 1.0, lr_end: float = 0.0) -> None:
    """b2r_adam_step_floor: torch.optim.Adam on a flat fp32 bucket with the learning-rate decay of train_nerf.py:170-175 (lr_end = 0)
    or pi_GAN/train.py:140-145 (floor lr_end); the step counter lives in `state` (4 floats on the device, zero before the first step)."""
    for t in (params, grads, exp_avg, exp_avg_sq, state):
        if not t.is_cuda or t.dtype != torch.float32 or not t.is_contiguous():
            raise RuntimeError("adam_step needs contiguous fp32 CUDA tensors")
    with torch.cuda.device(params.device):
        check(lib().b2r_adam_step_floor(ptr(params), ptr(grads), ptr(exp_avg), ptr(exp_avg_sq), params.numel(), ptr(state), float(lr0),
                                        float(lr_end), float(decay_rate), float(decay_steps), float(betas[0]), float(betas[1]), float(eps),
                                        float(grad_scale), _stream(params)), "b2r_adam_step_floor")


def train_loss_finish(sums, inv_count, alpha_weight: float, inv_local, loss, psnr) -> None:
    """b2r_train_loss_finish: loss / PSNR of a training step from the four sums of the two composite_loss_backward calls."""
    with torch.cuda.device(sums.device):
        check(lib().b2r_train_loss_finish(ptr(sums), ptr(inv_count), float(alpha_weight), ptr(inv_local), ptr(loss), ptr(psnr), _stream(sums)),
              "b2r_train_loss_finish")


class _MlpTcTrain(torch.autograd.Function):
    """Fused bf16 tensor-core forward that keeps the layer inputs as tiled bf16 tensors, and its reverse mode
    (dgrad + wgrad + heads, mlp_tc_train.cu).  NeRF and SirenNeRF models."""

    @staticmethod
    def forward(ctx, flat, model, kind, rays, z, x):
        fd = flat.detach()
        packed = _packed_weights(model, kind, fd, None, True)
        # opt-in (_EXACT_LAST_TRAIN): the same last-sample sign check as the render, so that autograd callers see the render's raw
        # values; d sigma_last is zero on either side of the step, so the reverse mode is unaffected
        raw, saved = tc_train_forward(packed, kind, rays, z, x=x, last_sample=(fd, None, True) if _EXACT_LAST_TRAIN else None)
        ctx.model, ctx.kind = model, kind
        ctx.save_for_backward(flat, raw, saved)
        return raw

    @staticmethod
    def backward(ctx, d_raw):
        flat, raw, saved = ctx.saved_tensors
        if not ctx.needs_input_grad[0]:
            return (None,) * 6
        d_flat = torch.zeros_like(flat)
        if raw.shape[0]:
            tc_train_backward(_packed_bwd_weights(ctx.model, ctx.kind, flat.detach()), ctx.kind, raw, d_raw, saved, d_flat)
        return d_flat, None, None, None, None, None


class _MlpTcTrainFilm(torch.autograd.Function):
    """FiLM-SIREN (use_dir) on the fused tensor-core training path: forward with the latents' folded weights that keeps the
    sine layers' inputs as bf16 tiles and cos(t) as thread-major bf16x2 words; reverse mode = dgrad + wgrad on the folded
    weights + the kernel that unfolds them into d weights and d film (mlp_tc_train.cu).  Replaces autograd through
    FilmSirenNeRF.forward (pi_GAN/modules.py:101-118) for pi_GAN/train.py:134 and synthesis.py:107.
    film [9,512] (one latent) or [B,9,512] with rows [b * rows_per_latent, (b+1) * rows_per_latent) evaluated with latent b
    (Generator.forward's loop, pi_GAN/modules.py:176-184, in one launch sequence)."""

    @staticmethod
    def forward(ctx, flat, film, rays, z, x, rows_per_latent, use_dir=True):
        fd, fl = flat.detach(), film.detach().contiguous()
        n_lat = 1 if film.dim() == 2 else film.shape[0]
        raw, saved = tc_train_forward(_pack_film_batched(fd, fl, use_dir, n_lat), models.KIND_FILM, rays, z, x=x, n_latents=n_lat,
                                      rows_per_latent=int(rows_per_latent),
                                      last_sample=(fd, fl, use_dir) if _EXACT_LAST_TRAIN else None)
        ctx.rows, ctx.n_lat, ctx.rows_per_latent, ctx.use_dir = raw.shape[0], n_lat, int(rows_per_latent), int(bool(use_dir))
        ctx.save_for_backward(flat, film, raw, saved)
        return raw

    @staticmethod
    def backward(ctx, d_raw):
        flat, film, raw, saved = ctx.saved_tensors
        need_w, need_f = ctx.needs_input_grad[0], ctx.needs_input_grad[1]
        if not (need_w or need_f):
            return (None,) * 7
        dev = flat.device
        d_flat = torch.zeros_like(flat) if need_w else None
        d_film = torch.zeros(film.shape, dtype=torch.float32, device=dev) if need_f else None
        if ctx.rows > 0:
            kind = models.KIND_FILM
            d_raw = _cuda_f32(d_raw, "d_raw")
            fd, fl = flat.detach(), film.detach().contiguous()
            packed_bwd = torch.empty((ctx.n_lat, lib().b2r_mlp_tc_bwd_packed_bytes(kind)), dtype=torch.uint8, device=dev)
            sbytes = lib().b2r_mlp_tc_train_scratch_bytes(kind, ctx.rows)
            scratch = torch.empty((sbytes,), dtype=torch.uint8, device=dev)
            d_folded = torch.empty((ctx.n_lat, fd.numel()), dtype=torch.float32, device=dev)
            with torch.cuda.device(dev):
                check(lib().b2r_mlp_tc_pack_bwd_film(ptr(fd), ptr(fl), ctx.use_dir, ctx.n_lat, ptr(packed_bwd), _stream(flat)), "b2r_mlp_tc_pack_bwd_film")
                check(lib().b2r_mlp_tc_train_bwd_film(ptr(packed_bwd), ptr(fd), ptr(fl), ctx.use_dir, ctx.n_lat, ctx.rows_per_latent, ctx.rows, ptr(raw),
                                                      ptr(d_raw), ptr(saved), ptr(scratch), sbytes, ptr(d_folded), ptr(d_flat), ptr(d_film),
                                                      _stream(flat)), "b2r_mlp_tc_train_bwd_film")
        return d_flat, d_film, None, None, None, None, None


def mlp_film_batched_train(model, film: torch.Tensor, rays: torch.Tensor, z: torch.Tensor, rows_per_latent: int) -> torch.Tensor:
    """Differentiable counterpart of mlp_film_batched: FiLM-SIREN on (rays, z) rows for B latents in one launch sequence with the
    autograd graph to the model's parameters and to film[B,9,512] (fused tensor-core training path, bf16 arithmetic)."""
    if models.model_kind(model) != models.KIND_FILM:
        raise TypeError("mlp_film_batched_train needs a FilmSirenNeRF model")
    if rows_per_latent <= 0 or rows_per_latent % 512 != 0:
        raise RuntimeError("rows_per_latent must be a positive multiple of 512")
    net, kind, use_dir, _, _ = _model_args(model)
    if film.dim() != 3 or tuple(film.shape[1:]) != (9, 512) or not film.is_cuda:
        raise RuntimeError(f"film must be a CUDA tensor [B,9,512], got {tuple(film.shape)}")
    return _MlpTcTrainFilm.apply(models.flat_params(net, kind), film.float(), rays, z, None, int(rows_per_latent), use_dir)


def mlp(model, rays: torch.Tensor | None = None, z: torch.Tensor | None = None, x: torch.Tensor | None = None,
        grid: tuple | None = None, precision: str | None = None, sigma_only: bool = False,
        exact_last_sample: bool | None = None, samples_per_ray: int | None = None, lattice: tuple | None = None) -> torch.Tensor:
    """Evaluate the radiance field on rows described by (rays, z) | x | grid | lattice -> raw[rows,4]
    (run_network + network.forward, nerf/render.py:59-75).  Differentiable wrt the model's
    parameters (and FiLM parameters) when any of them requires grad and grad mode is on.
    ``grid = (N, begin, count)``: indices [begin, begin+count) of the N^3 lattice of [-0.1,0.1]^3 (pi-GAN's create_mesh);
    ``lattice = ((n0, n1, n2), (ox, oy, oz), voxel, begin, count)``: indices of a box lattice, point origin + index * voxel in
    fp32 (axis 0 slowest).  Both have zero view direction and are inference-only.

    bf16 inference on ray samples -- (rays, z), or x with ``samples_per_ray`` given -- also runs the last-sample sign check
    (see _EXACT_LAST above) unless ``exact_last_sample`` is False."""
    net, kind, use_dir, ps, dev = _model_args(model)
    if kind == models.KIND_SIREN:
        sigma_only = False                       # no such kernel for SirenNeRF: the full evaluation is a superset
    film = None
    if kind == models.KIND_FILM:
        film = models.film_tensor(net)
        film = film.to(dev).float()
        if tuple(film.shape) != (9, 512):
            raise RuntimeError(f"film_params must be [9,512], got {tuple(film.shape)}")
        film = film.contiguous()
    needs_grad = torch.is_grad_enabled() and (any(p.requires_grad for p in ps) or (film is not None and film.requires_grad))
    flat = models.flat_params(net, kind) if needs_grad else torch.cat([p.detach().reshape(-1) for p in ps]).float()
    precision = precision or _MLP_PRECISION
    if needs_grad:
        if grid is not None or lattice is not None:
            raise RuntimeError("grid / lattice queries are inference-only")
        if _GRAD_PRECISION == "bf16":
            if kind == models.KIND_FILM:
                return _MlpTcTrainFilm.apply(flat, film, rays, z, x, 0, use_dir)
            return _MlpTcTrain.apply(flat, net, kind, rays, z, x)
        return _MlpF32.apply(flat, film, kind, use_dir, rays, z, x, 1 if _GRAD_PRECISION == "tf32" else 0)
    inp, rows, keep = _make_input(rays, z, x, grid, lattice)
    raw = torch.empty((rows, 4), dtype=torch.float32, device=dev)
    if rows == 0:
        return raw
    if precision != "bf16":
        _mlp_f32_forward(kind, flat, film, use_dir, inp, raw, 0, 1 if precision == "tf32" else 0)
        return raw
    packed = _packed_weights(net, kind, flat, film, use_dir)

    def launch(ls):
        check(lib().b2r_mlp_tc_fwd(kind, ptr(packed), int(use_dir), C.byref(inp), ptr(raw), int(sigma_only), ls, _stream(flat)),
              "b2r_mlp_tc_fwd")
    spr = z.shape[1] if rays is not None else (int(samples_per_ray) if (x is not None and samples_per_ray) else 0)
    want_last = (_EXACT_LAST if exact_last_sample is None else bool(exact_last_sample)) and spr > 0 and not sigma_only \
        and rows % spr == 0
    with torch.cuda.device(dev):
        _with_last_sample(want_last, launch, kind, inp, spr, raw, (flat, film, use_dir))
    del keep
    return raw


def mlp_film_batched(model, film: torch.Tensor, rays: torch.Tensor, z: torch.Tensor, rows_per_latent: int,
                     sigma_only: bool = False, exact_last_sample: bool | None = None) -> torch.Tensor:
    """FiLM-SIREN on (rays, z) rows for B latents in ONE launch (Generator.forward's per-latent loop, pi_GAN/modules.py:176-184):
    film[B,9,512]; rows [b * rows_per_latent, (b+1) * rows_per_latent) use latent b.  Inference only (bf16 tensor-core kernel)."""
    if models.model_kind(model) != models.KIND_FILM:
        raise TypeError("mlp_film_batched needs a FilmSirenNeRF model")
    net, kind, use_dir, ps, dev = _model_args(model)
    film = _cuda_f32(film.detach(), "film")
    if film.dim() != 3 or tuple(film.shape[1:]) != (9, 512):
        raise RuntimeError(f"film must be [B,9,512], got {tuple(film.shape)}")
    flat = torch.cat([p.detach().reshape(-1) for p in ps]).float()
    inp, rows, keep = _make_input(rays, z, None, None)
    raw = torch.empty((rows, 4), dtype=torch.float32, device=dev)
    if rows == 0:
        return raw
    n_lat = film.shape[0]
    packed = _pack_film_batched(flat, film, use_dir, n_lat)

    def launch(ls):
        check(lib().b2r_mlp_tc_fwd_film_batched(ptr(packed), n_lat, int(rows_per_latent), C.byref(inp), ptr(raw), int(sigma_only), ls,
                                                _stream(flat)), "b2r_mlp_tc_fwd_film_batched")
    want_last = (_EXACT_LAST if exact_last_sample is None else bool(exact_last_sample)) and not sigma_only
    with torch.cuda.device(dev):
        _with_last_sample(want_last, launch, kind, inp, z.shape[1], raw, (flat, film, use_dir), n_lat, int(rows_per_latent))
    del keep
    return raw


def to8b(x: torch.Tensor) -> torch.Tensor:
    """to8b (nerf/render.py:5) on the device: uint8 tensor of the same shape, (255 * clip(x, 0, 1)) truncated like numpy."""
    x = _cuda_f32(x, "x")
    out = torch.empty(x.shape, dtype=torch.uint8, device=x.device)
    with torch.cuda.device(x.device):
        check(lib().b2r_to8b(ptr(x), x.numel(), ptr(out), _stream(x)), "b2r_to8b")
    return out


_INT32_MAX = 2 ** 31 - 1


def _mc_field(field: torch.Tensor) -> torch.Tensor:
    """``field`` as a contiguous [n0,n1,n2] float32 CUDA tensor with every n >= 2 and at most 2^31 - 1 points; RuntimeError
    otherwise."""
    field = _cuda_f32(field, "field")
    if field.dim() != 3 or min(field.shape) < 2:
        raise RuntimeError(f"field must be [n0,n1,n2] with every n >= 2, got {list(field.shape)}")
    if field.numel() > _INT32_MAX:
        raise RuntimeError(f"field has {field.numel()} points; marching_cubes takes at most 2^31 - 1")
    return field


def brick_dims(shape, stride: int) -> tuple:
    """Bricks per axis of a lattice of ``shape`` points for bricks of ``stride`` cells: ``ceil((n - 1) / stride)`` each."""
    return tuple((int(n) - 2) // stride + 1 for n in shape)


def band_select(field: torch.Tensor, level: float, stride: int):
    """Flagged bricks and needed points of a narrow-band query (b2r_band_select) on ``field`` [n0,n1,n2], whose values must be
    valid at every coarse corner (the points ``min(b * stride, n - 1)`` on every axis) and may be +inf elsewhere.  Returns
    ``(flags uint8 [nb0,nb1,nb2], index int32 [M])`` on the field's device: a brick is flagged when its 8 coarse corners are
    not all on the same side of ``level`` (``field < level``, NaN not below), dilated by one brick over the 26-neighbourhood;
    ``index`` lists, ascending, every point of the closure of a flagged brick and every point one step along one axis from
    one.  Synchronises once with the host to read M.  The list is allocated for every lattice point (4 B each) before M is known;
    ``index`` is a view of that allocation."""
    field = _mc_field(field)
    stride = _check_int("stride", stride, 2, _INT32_MAX)
    n0, n1, n2 = (int(s) for s in field.shape)
    dev = field.device
    flags = torch.empty(brick_dims(field.shape, stride), dtype=torch.uint8, device=dev)
    index = torch.empty((field.numel(),), dtype=torch.int32, device=dev)
    count = torch.empty((1,), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        scratch = torch.empty((lib().b2r_band_scratch_bytes(n0, n1, n2, stride),), dtype=torch.uint8, device=dev)
        check(lib().b2r_band_select(ptr(field), n0, n1, n2, float(level), stride, ptr(scratch), ptr(flags), ptr(index), ptr(count),
                                    _stream(field)), "b2r_band_select")
        return flags, index[:int(count.item())]


def _lattice_rows(index: torch.Tensor, grid=None, lattice=None) -> torch.Tensor:
    """lattice_rows for an index already known to lie in range."""
    inp, _, _ = _make_input(None, None, None, grid, lattice)
    x = torch.empty((index.shape[0], 6), dtype=torch.float32, device=index.device)
    with torch.cuda.device(index.device):
        check(lib().b2r_lattice_rows(C.byref(inp), ptr(index), index.shape[0], ptr(x), _stream(index)), "b2r_lattice_rows")
    return x


def lattice_rows(index: torch.Tensor, grid: tuple | None = None, lattice: tuple | None = None) -> torch.Tensor:
    """x rows [M,6] = (point, zero direction) of rows ``index`` (int32 [M], on the device) of one ``grid`` or ``lattice``
    description as ``mlp`` takes it (b2r_lattice_rows), so ``mlp(model, x=lattice_rows(index, ...))`` evaluates those rows'
    points.  Checks that every index lies in [0, count) first (RuntimeError otherwise; one host synchronisation)."""
    if (grid is None) == (lattice is None):
        raise ValueError("give exactly one of grid / lattice")
    if not isinstance(index, torch.Tensor) or not index.is_cuda or index.dtype != torch.int32 or index.dim() != 1:
        raise RuntimeError("index must be a 1-d int32 CUDA tensor")
    count = int((grid or lattice)[-1])
    if index.numel():
        lo, hi = (int(v) for v in torch.aminmax(index))
        if lo < 0 or hi >= count:
            raise RuntimeError(f"row indices span [{lo}, {hi}], outside [0, {count})")
    return _lattice_rows(index.contiguous(), grid, lattice)


def marching_cubes(field: torch.Tensor, level: float, spacing: float = 1.0, origin=(0.0, 0.0, 0.0), *, normals: bool = False,
                   bricks: tuple | None = None):
    """Marching cubes of ``field`` [n0,n1,n2] (axis 0 slowest) at ``level`` on the device (b2r_mc_count / b2r_mc_emit; the
    table and its rule: oracle/marching_cubes.py).  Returns ``(verts [V,3] float32, faces [F,3] int32)`` on the field's
    device; vertex ``origin + (p + t e_a) * spacing`` lies on the lattice edge from point ``p`` along axis ``a``, and the
    triangle normals point from ``field < level`` to ``field >= level``.  Synchronises once with the host to read the
    mesh size (V, F), as ``torch.nonzero`` does.  Empty meshes are ``[0,3]`` tensors.
    ``normals=True`` also returns the unit vertex normals [V,3] (b2r_mc_normals: the field's central-difference gradient
    interpolated along the vertex's edge, pointing toward increasing field; (0, 0, 0) where it vanishes).
    ``bricks=(stride, flags)`` (flags uint8 [nb0,nb1,nb2] on the field's device, as ``band_select`` returns them) limits the
    mesh to the flagged bricks (b2r_mc_count_band): the faces of cells in other bricks and the vertices on no edge of a cell
    in a flagged brick are removed, and the rest keeps its order."""
    field = _mc_field(field)
    if bricks is not None:
        if not isinstance(bricks, tuple) or len(bricks) != 2:
            raise ValueError("bricks must be a tuple (stride, flags)")
        stride = _check_int("stride", bricks[0], 2, _INT32_MAX)
        flags = bricks[1]
        if not isinstance(flags, torch.Tensor) or flags.dtype != torch.uint8 or not flags.is_cuda:
            raise RuntimeError("brick flags must be a uint8 CUDA tensor")
        if tuple(flags.shape) != brick_dims(field.shape, stride):
            raise RuntimeError(f"brick flags must be {list(brick_dims(field.shape, stride))} for stride {stride}, "
                               f"got {list(flags.shape)}")
        if flags.device != field.device:
            raise RuntimeError("field and brick flags must be on the same device")
        flags = flags.contiguous()
    n0, n1, n2 = (int(s) for s in field.shape)
    level, spacing = float(level), float(spacing)
    ox, oy, oz = (float(o) for o in origin)
    dev = field.device
    scratch = torch.empty((lib().b2r_mc_scratch_bytes(n0, n1, n2),), dtype=torch.uint8, device=dev)
    totals = torch.empty((2,), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        if bricks is None:
            check(lib().b2r_mc_count(ptr(field), n0, n1, n2, level, ptr(scratch), ptr(totals), _stream(field)), "b2r_mc_count")
        else:
            check(lib().b2r_mc_count_band(ptr(field), n0, n1, n2, level, ptr(flags), stride, ptr(scratch), ptr(totals),
                                          _stream(field)), "b2r_mc_count_band")
        n_verts, n_faces = (int(v) for v in totals.tolist())
        if n_verts > _INT32_MAX or n_faces > _INT32_MAX:
            raise RuntimeError(f"mesh of {n_verts} vertices / {n_faces} triangles: int32 vertex indices hold at most 2^31 - 1")
        verts = torch.empty((n_verts, 3), dtype=torch.float32, device=dev)
        faces = torch.empty((n_faces, 3), dtype=torch.int32, device=dev)
        if n_verts and n_faces:
            check(lib().b2r_mc_emit(ptr(field), n0, n1, n2, level, spacing, ox, oy, oz, ptr(scratch), ptr(verts), ptr(faces),
                                    _stream(field)), "b2r_mc_emit")
        if not normals:
            return verts, faces
        nrm = torch.empty((n_verts, 3), dtype=torch.float32, device=dev)
        if n_verts and n_faces:
            check(lib().b2r_mc_normals(ptr(field), n0, n1, n2, level, ptr(scratch), ptr(nrm), _stream(field)), "b2r_mc_normals")
    return verts, faces, nrm


def _mesh_faces(faces: torch.Tensor, n_verts: int) -> torch.Tensor:
    """``faces`` as a contiguous [F,3] int32 CUDA tensor whose every index lies in [0, n_verts); raises RuntimeError otherwise,
    before anything is launched on the mesh (reads the indices' min / max: one host synchronisation when F > 0)."""
    if not isinstance(faces, torch.Tensor) or not faces.is_cuda or faces.dtype != torch.int32 or faces.dim() != 2 or faces.shape[1] != 3:
        raise RuntimeError("faces must be an [F,3] int32 CUDA tensor")
    if not 0 <= n_verts <= _INT32_MAX or faces.shape[0] > _INT32_MAX:
        raise RuntimeError(f"{n_verts} vertices / {faces.shape[0]} faces: the mesh kernels take at most 2^31 - 1 of each")
    if faces.numel():
        lo, hi = (int(v) for v in torch.aminmax(faces))
        if lo < 0 or hi >= n_verts:
            raise RuntimeError(f"face indices span [{lo}, {hi}], outside [0, {n_verts}) for {n_verts} vertices")
    return faces.contiguous()


def _mesh_args(verts: torch.Tensor, faces: torch.Tensor, normals: torch.Tensor | None = None):
    """The checked ``(verts, faces, normals)`` of a mesh op: ``verts`` and ``normals`` (when given) contiguous [V,3] float32
    CUDA tensors, ``faces`` as ``_mesh_faces`` leaves it, all on one device; raises RuntimeError otherwise, before any launch."""
    verts = _cuda_f32(verts, "verts")
    if verts.dim() != 2 or verts.shape[1] != 3:
        raise RuntimeError(f"verts must be [V,3], got {list(verts.shape)}")
    if normals is not None:
        normals = _cuda_f32(normals, "normals")
        if normals.shape != verts.shape:
            raise RuntimeError(f"normals must have the shape of verts {list(verts.shape)}, got {list(normals.shape)}")
    faces = _mesh_faces(faces, verts.shape[0])
    if faces.device != verts.device or (normals is not None and normals.device != verts.device):
        names = "verts and faces" if normals is None else "verts, faces and normals"
        raise RuntimeError(f"{names} must be on the same device")
    return verts, faces, normals


def _check_int(name: str, value, lo: int, hi: int | None = None) -> int:
    """``value`` as an int in [lo, hi] (no upper bound when ``hi`` is None); ValueError for anything else, bools included."""
    if isinstance(value, bool) or not isinstance(value, (int, np.integer)) or value < lo or (hi is not None and value > hi):
        bound = f">= {lo}" if hi is None else f"in [{lo}, {'2^31 - 1' if hi == _INT32_MAX else hi}]"
        raise ValueError(f"{name} must be an int {bound}, got {value!r}")
    return int(value)


def _cc_label(faces: torch.Tensor, n_verts: int, scratch: torch.Tensor) -> torch.Tensor:
    labels = torch.empty((n_verts,), dtype=torch.int32, device=faces.device)
    check(lib().b2r_mesh_cc_label(ptr(faces), faces.shape[0], n_verts, ptr(labels), ptr(scratch), _stream(faces)), "b2r_mesh_cc_label")
    return labels


def mesh_components(faces: torch.Tensor, n_verts: int) -> torch.Tensor:
    """Connected components of the mesh ``faces`` [F,3] (int32, on the device) over ``n_verts`` vertices, joined by the edges
    of its triangles (b2r_mesh_cc_label): int32 labels [V], the smallest vertex index of each vertex's component (a vertex no
    face uses is its own component), equal to ``oracle.mesh_components.component_labels``.  Checks that every index lies in
    [0, n_verts) first (RuntimeError otherwise; one host synchronisation)."""
    n_verts = int(n_verts)
    faces = _mesh_faces(faces, n_verts)
    with torch.cuda.device(faces.device):
        scratch = torch.empty((lib().b2r_mesh_cc_scratch_bytes(n_verts, faces.shape[0]),), dtype=torch.uint8, device=faces.device)
        return _cc_label(faces, n_verts, scratch)


def _check_ratio(ratio) -> float:
    r = float(ratio)
    if not (math.isfinite(r) and 0.0 <= r <= 1.0):
        raise ValueError(f"ratio must be finite and in [0, 1], got {ratio}")
    return float(np.float32(r))


def _filter_components(verts: torch.Tensor, faces: torch.Tensor, ratio: float, normals: torch.Tensor | None):
    """filter_components for faces already known to index [0, V) (label, select, one host read of (V', F'), compact)."""
    dev, n_verts, n_faces = verts.device, verts.shape[0], faces.shape[0]
    with torch.cuda.device(dev):
        st = _stream(verts)
        scratch = torch.empty((lib().b2r_mesh_cc_scratch_bytes(n_verts, n_faces),), dtype=torch.uint8, device=dev)
        labels = _cc_label(faces, n_verts, scratch)
        totals = torch.empty((2,), dtype=torch.int64, device=dev)
        check(lib().b2r_mesh_cc_select(ptr(faces), n_faces, n_verts, ptr(labels), ratio, ptr(scratch), ptr(totals), st),
              "b2r_mesh_cc_select")
        kv, kf = (int(v) for v in totals.tolist())
        v_out = torch.empty((kv, 3), dtype=torch.float32, device=dev)
        f_out = torch.empty((kf, 3), dtype=torch.int32, device=dev)
        n_out = None if normals is None else torch.empty((kv, 3), dtype=torch.float32, device=dev)
        if kv:
            check(lib().b2r_mesh_cc_compact(ptr(verts), ptr(normals), ptr(faces), n_faces, n_verts, ptr(scratch), ptr(v_out), ptr(n_out),
                                            ptr(f_out), st), "b2r_mesh_cc_compact")
    return v_out, f_out, n_out


def filter_components(verts: torch.Tensor, faces: torch.Tensor, ratio: float, normals: torch.Tensor | None = None):
    """Removes the small connected components of a mesh on the device (b2r_mesh_cc_label / _select / _compact).  A component
    (vertices joined by the edges of its triangles) with t triangles is kept iff t >= 1 and t >= ratio * t_max, compared in
    float64 with ``ratio`` rounded to float32, where t_max is the largest component's count: ratio 1 keeps the largest component
    and any tied with it, and a vertex no face uses is dropped.  Kept vertices (and their ``normals``) and faces keep their
    relative order; face indices are remapped.  Returns ``(verts [V',3], faces [F',3] int32, normals [V',3] | None)``, equal to
    ``oracle.mesh_components.filter_components``.  ``ratio`` must be finite and in [0, 1] (ValueError); 0 returns the inputs
    unchanged without a launch.  Otherwise checks that ``faces`` is [F,3] int32 on the device with every index in [0, V)
    (RuntimeError otherwise, before any launch; one host synchronisation), then synchronises once more to read (V', F')."""
    r = _check_ratio(ratio)
    if r == 0.0:
        return verts, faces, normals
    verts, faces, normals = _mesh_args(verts, faces, normals)
    return _filter_components(verts, faces, r, normals)


def _mesh_adjacency(faces: torch.Tensor, n_verts: int, scratch: torch.Tensor | None = None) -> torch.Tensor:
    """b2r_mesh_adjacency of ``faces`` over ``n_verts`` vertices into ``scratch`` (allocated for this mesh when None; one sized
    for a larger mesh also serves, the layout starts at its beginning); returns the scratch."""
    if scratch is None:
        scratch = torch.empty((lib().b2r_mesh_adj_scratch_bytes(n_verts, faces.shape[0]),), dtype=torch.uint8, device=faces.device)
    check(lib().b2r_mesh_adjacency(ptr(faces), faces.shape[0], n_verts, ptr(scratch), _stream(faces)), "b2r_mesh_adjacency")
    return scratch


def _smooth_mesh(verts: torch.Tensor, faces: torch.Tensor, iterations: int, normals: bool):
    """smooth_mesh for faces already known to index [0, V): (verts', normals' | None), no host synchronisation."""
    dev, n_verts, n_faces = verts.device, verts.shape[0], faces.shape[0]
    with torch.cuda.device(dev):
        st = _stream(verts)
        scratch = _mesh_adjacency(faces, n_verts)
        out = verts
        if iterations:
            out = torch.empty_like(verts)
            check(lib().b2r_mesh_smooth(ptr(verts), n_faces, n_verts, iterations, ptr(scratch), ptr(out), st), "b2r_mesh_smooth")
        nrm = None
        if normals:
            nrm = torch.empty_like(verts)
            check(lib().b2r_mesh_normals(ptr(out), n_faces, n_verts, ptr(scratch), ptr(nrm), st), "b2r_mesh_normals")
    return out, nrm


def smooth_mesh(verts: torch.Tensor, faces: torch.Tensor, iterations: int, *, normals: bool = False):
    """Taubin lambda|mu smoothing of a triangle mesh on the device (b2r_mesh_adjacency / _smooth / _normals).  Each iteration
    is two umbrella half-steps, p' = p + w (m - p) with w = 0.5 then w = -0.53, where m is the mean over the vertex's corners
    of the other two vertices of the corner's face (on a closed manifold mesh: the mean of its neighbours); a vertex no face
    uses stays where it is.  Topology, vertex order and faces are unchanged.  Returns ``verts' [V,3]``, or
    ``(verts', normals' [V,3])`` with ``normals``: the unit area-weighted vertex normals of the smoothed mesh ((0, 0, 0) where
    the fan has no area), which point the way the faces are wound.  Equal to ``oracle.mesh_smoothing.smooth`` /
    ``mesh_normals``.  ``iterations`` must be an int >= 0 (ValueError); 0 without ``normals`` returns ``verts`` without a
    launch.  Otherwise checks that ``faces`` is [F,3] int32 on the device with every index in [0, V) (RuntimeError otherwise,
    before any launch; one host synchronisation)."""
    iterations = _check_int("iterations", iterations, 0, _INT32_MAX)
    if not iterations and not normals:
        return verts
    verts, faces, _ = _mesh_args(verts, faces)
    out, nrm = _smooth_mesh(verts, faces, iterations, normals)
    return (out, nrm) if normals else out


def _decimate_mesh(verts: torch.Tensor, faces: torch.Tensor, max_faces: int, stats: dict | None = None):
    """decimate_mesh for faces already known to index [0, V): one host read of the round's counts per round."""
    dev, n_verts, n_faces = verts.device, verts.shape[0], faces.shape[0]
    if max_faces >= n_faces:
        return verts, faces
    rounds = []
    with torch.cuda.device(dev):
        st = _stream(verts)
        # sized for the input mesh: every round's mesh is smaller and lays its scratch out from the start
        adj = torch.empty((lib().b2r_mesh_adj_scratch_bytes(n_verts, n_faces),), dtype=torch.uint8, device=dev)
        scratch = torch.empty((lib().b2r_mesh_decimate_scratch_bytes(n_verts, n_faces),), dtype=torch.uint8, device=dev)
        sel_keys = torch.empty((n_verts,), dtype=torch.int64, device=dev)
        counts = torch.empty((2,), dtype=torch.int64, device=dev)
        _mesh_adjacency(faces, n_verts, adj)
        quadrics = torch.empty((n_verts, 10), dtype=torch.float64, device=dev)
        check(lib().b2r_mesh_quadrics(ptr(verts), n_faces, n_verts, ptr(adj), ptr(quadrics), st), "b2r_mesh_quadrics")
        while n_faces > max_faces:
            if rounds:
                _mesh_adjacency(faces, n_verts, adj)
            check(lib().b2r_mesh_decimate_round(ptr(verts), ptr(quadrics), n_faces, n_verts, ptr(adj), ptr(scratch), ptr(sel_keys),
                                                ptr(counts), st), "b2r_mesh_decimate_round")
            selected = int(counts[0])
            if not selected:
                break
            cut = None
            budget = (n_faces - max_faces + 1) // 2
            if selected > budget:
                # the budget's cheapest selected edges: (cost bits, a) of the last one, read on the device by the compaction
                keys = sel_keys[:n_verts]
                last = torch.sort(keys, stable=True).indices[budget - 1]
                cut = torch.stack([keys[last], last])
                selected = budget
            v_out = torch.empty((n_verts - selected, 3), dtype=torch.float32, device=dev)
            q_out = torch.empty((n_verts - selected, 10), dtype=torch.float64, device=dev)
            f_out = torch.empty((n_faces - 2 * selected, 3), dtype=torch.int32, device=dev)
            check(lib().b2r_mesh_decimate_compact(ptr(verts), ptr(quadrics), ptr(faces), n_faces, n_verts, ptr(sel_keys), ptr(cut),
                                                  ptr(scratch), ptr(v_out), ptr(q_out), ptr(f_out), st), "b2r_mesh_decimate_compact")
            verts, quadrics, faces = v_out, q_out, f_out
            n_verts, n_faces = n_verts - selected, n_faces - 2 * selected
            rounds.append(selected)
    if stats is not None:
        stats["rounds"] = len(rounds)
        stats["collapses"] = rounds
    return verts, faces


def decimate_mesh(verts: torch.Tensor, faces: torch.Tensor, max_faces: int):
    """Quadric edge collapse of a triangle mesh on the device down to ``max_faces`` triangles (b2r_mesh_adjacency / _quadrics /
    _decimate_round / _decimate_compact).  Rounds of independent collapses preserve the topology: closed stays closed, genus
    and components do not change, no non-manifold edge appears and no face flips.  Vertices on an open boundary (an edge on one
    face) or on non-manifold input never move.  Each round collapses the edges that are the cheapest (area-weighted plane
    quadrics, placement at either end or the midpoint) within both ends' neighbourhoods; the round that would pass the budget
    collapses only its cheapest ones, so the result has ``max_faces`` or ``max_faces - 1`` triangles unless no edge can
    collapse first.  Surviving vertices and faces keep their order.  Returns ``(verts' [V',3] float32, faces' [F',3] int32)``,
    equal to ``oracle.mesh_decimation.decimate``.  ``max_faces`` must be an int >= 1 (ValueError).  Checks that ``faces`` is
    [F,3] int32 on the device with every index in [0, V) (RuntimeError otherwise, before any launch; one host
    synchronisation); ``max_faces >= F`` then returns the inputs without a launch.  Every round synchronises once more to read
    its collapse count."""
    max_faces = _check_int("max_faces", max_faces, 1)
    verts, faces, _ = _mesh_args(verts, faces)
    return _decimate_mesh(verts, faces, max_faces)


ATLAS_SIZES = (16, 16384)


def atlas_layout(n_faces: int, size: int):
    """``(cells, per_row, s)`` of the per-face texture atlas of ``n_faces`` triangles in a ``size`` x ``size`` texture
    (include/b2r.h, oracle/mesh_texture.py): faces 2k and 2k+1 share cell k, ``cells = ceil(n_faces / 2)`` cells sit ``per_row``
    to a row (the smallest C with C * C >= cells) and each is ``s = size // per_row`` texels square; the atlas has
    ``cells * s * s`` texel rows.  ``size`` must be an int in [16, 16384] and ``n_faces`` at most ``2 * (size // 4) ** 2``, so
    that every cell has at least 4 x 4 texels (ValueError otherwise).  Host arithmetic only."""
    size = _check_int("texture size", size, *ATLAS_SIZES)
    n_faces = _check_int("n_faces", n_faces, 0, _INT32_MAX)
    limit = 2 * (size // 4) ** 2
    if n_faces > limit:
        raise ValueError(f"{n_faces} faces do not fit a {size} x {size} texture atlas: it holds at most {limit} "
                         f"(2 * (size // 4)^2, cells of 4 x 4 texels); use a larger texture or fewer faces (max_faces)")
    cells = (n_faces + 1) // 2
    per_row = math.isqrt(cells - 1) + 1 if cells else 0
    return cells, per_row, size // per_row if per_row else 0


def _atlas_uvs(n_faces: int, size: int, device) -> torch.Tensor:
    """float32 [F,3,2] UVs of the atlas of ``n_faces`` faces (b2r_mesh_atlas_uvs); the layout is known to fit."""
    uvs = torch.empty((n_faces, 3, 2), dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        check(lib().b2r_mesh_atlas_uvs(n_faces, size, ptr(uvs), torch.cuda.current_stream(device).cuda_stream), "b2r_mesh_atlas_uvs")
    return uvs


def _atlas_rows(verts: torch.Tensor, faces: torch.Tensor, normals: torch.Tensor, size: int, begin: int, count: int) -> torch.Tensor:
    """x rows [count,6] = [surface point, -unit normal] of atlas texel rows [begin, +count) (b2r_mesh_atlas_rows), for a mesh
    already checked by _mesh_args and a layout known to fit."""
    x = torch.empty((count, 6), dtype=torch.float32, device=verts.device)
    check(lib().b2r_mesh_atlas_rows(ptr(verts), ptr(normals), ptr(faces), faces.shape[0], size, begin, count, ptr(x), _stream(verts)),
          "b2r_mesh_atlas_rows")
    return x


def _atlas_texture(raw: torch.Tensor, n_faces: int, size: int, begin: int, texture: torch.Tensor) -> None:
    """Quantises raw[:, :3] (the MLP output of atlas rows [begin, +len(raw))) into ``texture`` [R,R,3] uint8
    (b2r_mesh_atlas_texture)."""
    check(lib().b2r_mesh_atlas_texture(ptr(raw), n_faces, size, begin, raw.shape[0], ptr(texture), _stream(raw)),
          "b2r_mesh_atlas_texture")
