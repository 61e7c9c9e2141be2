"""Drop-in replacement for the reference's ``nerf/render.py`` backed by libb2r.so (sm_100a CUDA).

Same names, argument order and return conventions as the reference module (file:line cited per
function), so ``from render import *`` callers (nerf/train_nerf.py:8, test_nerf.py:8,
show_nerf.py:5, demo_view.py:8, demo_param.py:8) keep working; ``np``, ``torch`` and ``tqdm`` are
re-exported because those callers rely on the star-import leaking them (train_nerf.py:69,78-83).

Backwards-compatible keyword-only additions: ``t_rand`` (inject the jitter the reference draws
with torch.rand, for parity runs), ``z_lin`` / ``u`` (inject the two torch.linspace vectors),
``precision`` ("bf16" tensor-core MLP or "fp32"), ``stages`` (dict that receives intermediates),
``exact_last_sample`` (None = the module default ops.get_exact_last_sample(), which is True: the bf16 path
re-evaluates in fp32 the last sample of every ray whose sigma is inside the bf16 error band of zero, because the
1e10 last interval of nerf/render.py:92 turns the SIGN of that sigma into a whole-ray decision).

There is no CPU path: tensors and models must live on a CUDA device.
"""
from __future__ import annotations

import math

import numpy as np
import torch
from tqdm import tqdm

from . import mesh, ops

__all__ = ["np", "torch", "tqdm", "to8b", "get_rays", "sample_pdf", "run_network", "raw_to_outputs", "render_rays",
           "render_image", "render_video", "render_video_u8"]

to8b = lambda x: (255 * np.clip(x, 0, 1)).astype(np.uint8)       # nerf/render.py:5

REFERENCE_RAY_CHUNK = 1024 * 16                                  # nerf/render.py:150


def _model_device(model) -> torch.device:
    return next(model.parameters()).device


def get_rays(width, height, focal, c2w):
    """nerf/render.py:7-23 -- (rays_o, rays_d) numpy arrays [H,W,3], generated on the GPU (K1)."""
    rays = ops.raygen(int(width), int(height), focal, c2w).cpu().numpy()
    rays = rays.reshape(int(height), int(width), 2, 3)
    return rays[:, :, 0], rays[:, :, 1]


def sample_pdf(bins, weights, N_samples, *, u=None):
    """nerf/render.py:27-56 -- hierarchical inverse-CDF samples [N, N_samples] (K5)."""
    return ops.sample_pdf(bins, weights, int(N_samples), u=u)["samples"]


def run_network(ray_samples, view_dirs, network, chunk=1024 * 64, *, precision=None, exact_last_sample=None):
    """nerf/render.py:59-75 -- evaluate ``network`` on every sample point -> [N,S,4].

    ``chunk`` is accepted for signature compatibility; the fused kernel has O(tile) memory so the
    points are evaluated in one launch.  The rows keep their [N,S] structure, so the bf16 path can apply
    the last-sample sign check exactly as render_rays does."""
    n, s = ray_samples.shape[0], ray_samples.shape[1]
    pts = ray_samples.reshape(-1, 3)
    vd = view_dirs[:, None, :].expand(n, s, 3).reshape(-1, 3)
    x = torch.cat([pts, vd], -1)
    return ops.mlp(network, x=x, precision=precision, exact_last_sample=exact_last_sample, samples_per_ray=s).reshape(n, s, 4)


def raw_to_outputs(raw, z_vals, rays_d):
    """nerf/render.py:78-103 -- (rgb_map[N,3], depth_map[N], acc_map[N], weights[N,S]) (K4)."""
    return ops.composite(raw, z_vals, rays_d, want_weights=True)


def render_rays(rays, near, far, coarse_model, fine_model, coarse_sample_num, fine_sample_num, *,
                t_rand=None, z_lin=None, u=None, precision=None, stages=None, coarse_no_grad=False,
                exact_last_sample=None, fine_out=None, coarse_outputs_unused=False, coarse_sigma_only=False):
    """nerf/render.py:106-147 -- coarse pass, sample_pdf on the un-jittered mids with
    weights[:,1:-1], sort-merge, fine pass on all Sc+Sf samples.  Returns the reference's 6-tuple
    (rgb_c, depth_c, acc_c, rgb_f, depth_f, acc_f).  ``coarse_no_grad`` runs the coarse pass in
    inference mode (used by the pi-GAN wrappers, whose loss never touches the coarse outputs).
    ``exact_last_sample`` (default on): the bf16 tensor-core path lists the rays whose LAST sample's
    pre-relu sigma lies inside the bf16 error band and re-evaluates those rows with the fp32 engine:
    that sample's interval is 1e10 (nerf/render.py:92), so alpha_last is a step function of
    sign(sigma_last) and a bf16 rounding would flip ~0.2 % of rays by up to 0.6 (SURVEY.md 0).
    ``fine_out`` [N,5] (no-grad renders): the fine pass writes (rgb, depth, acc) into its rows -- a rank's slice
    of the gathered frame buffer -- and the returned fine maps are views of it.
    ``coarse_outputs_unused`` (render_image / render_video and the pi-GAN wrappers, which return only the fine maps): the COARSE pass
    evaluates the whole network as always but skips the check --
    its last sample only reaches the coarse rgb / depth / acc maps (sample_pdf reads weights[:, 1:-1], nerf/render.py:140),
    so nothing the caller sees changes, and a training step keeps running without a host synchronisation.
    ``coarse_sigma_only`` (opt-in, off by default; bf16 inference of NeRF / FiLM-SIREN models): the coarse pass stops after the sigma
    head -- dead-code elimination for callers that return only the fine maps (render_image): the coarse weights, and with them every
    fine output, are bit-identical (tested); the returned coarse rgb map carries no colour (background term only).  Needs a gradient-free coarse pass.
    Applies to passes that run without gradients (renders; the pi-GAN coarse pass).  Passes that carry
    gradients run the raw bf16 forward (mixed-precision training; d sigma_last is zero either way) unless
    ops.set_exact_last_sample(train=True) is set -- an explicit switch, not a silent skip."""
    if not isinstance(rays, torch.Tensor):
        rays = torch.as_tensor(np.asarray(rays), dtype=torch.float32)
    if not rays.is_cuda:
        rays = rays.to(_model_device(coarse_model))
    rays = rays.float().reshape(-1, 2, 3).contiguous()          # no .squeeze(): N == 1 works (SURVEY app. D)
    dev = rays.device
    sc, sf = int(coarse_sample_num), int(fine_sample_num)       # callers pass floats (test_nerf.py:34-35)
    n = rays.shape[0]
    if z_lin is None:
        # made on the host: torch.linspace's last-bit rounding is part of the contract (SURVEY A.2)
        z_lin = torch.linspace(float(near), float(far), steps=sc, device="cpu")
    z_lin = torch.as_tensor(z_lin, dtype=torch.float32).to(dev)
    if t_rand is None:
        t_rand = torch.rand((n, sc), device=dev)                # nerf/render.py:131 (jitter is always on)
    t_rand = torch.as_tensor(t_rand, dtype=torch.float32).to(dev)
    rays_d = rays[:, 1]

    z_vals, mids = ops.stratified_z(z_lin, t_rand)
    with torch.set_grad_enabled(torch.is_grad_enabled() and not coarse_no_grad):
        if coarse_sigma_only and torch.is_grad_enabled() and any(p.requires_grad for p in coarse_model.parameters()):
            raise RuntimeError("coarse_sigma_only needs a gradient-free coarse pass (torch.no_grad() or coarse_no_grad=True)")
        raw = _mlp_rays(coarse_model, rays, z_vals, precision, False if (coarse_outputs_unused or coarse_sigma_only) else exact_last_sample,
                        sigma_only=bool(coarse_sigma_only))
        rgb_c, depth_c, acc_c, weights = ops.composite(raw, z_vals, rays_d, want_weights=True)

    if u is None:
        u = torch.linspace(0.0, 1.0, steps=sf, device="cpu")
    res = ops.sample_pdf(mids, weights[:, 1:-1], sf, u=torch.as_tensor(u, dtype=torch.float32).to(dev), z_coarse=z_vals,
                         want_samples=stages is not None)
    z_fine = res["sorted"]
    raw_f = _mlp_rays(fine_model, rays, z_fine, precision, exact_last_sample)
    rgb_f, depth_f, acc_f, w_f = ops.composite(raw_f, z_fine, rays_d, want_weights=stages is not None, packed_out=fine_out)
    if stages is not None:
        stages.update(z_coarse=z_vals, mids=mids, raw_coarse=raw, weights_coarse=weights, z_samples=res["samples"],
                      z_fine=z_fine, raw_fine=raw_f, weights_fine=w_f)
    return rgb_c, depth_c, acc_c, rgb_f, depth_f, acc_f


def _mlp_rays(model, rays, z, precision, exact_last_sample, sigma_only=False):
    """run_network on (rays, z) -> raw[N,S,4] (bf16 inference: with the last-sample sign check, ops.mlp)."""
    n, s = z.shape
    return ops.mlp(model, rays=rays, z=z, precision=precision, exact_last_sample=exact_last_sample, sigma_only=sigma_only).view(n, s, 4)


def _draw_t_rand(n: int, sc: int, chunk: int, device) -> torch.Tensor:
    """The jitter of a whole image, drawn exactly as the reference does: one torch.rand([chunk,Sc])
    per ray chunk (nerf/render.py:158-160,131), so a seeded render reproduces the reference."""
    parts = [torch.rand((min(chunk, n - i), sc), device=device) for i in range(0, n, chunk)]
    return parts[0] if len(parts) == 1 else torch.cat(parts)


def render_image_device(width, height, focal, pose, near, far, coarse_model, fine_model, coarse_sample_num,
                        fine_sample_num, chunk=REFERENCE_RAY_CHUNK, *, ray_begin=0, ray_count=None, t_rand=None,
                        precision=None, launch_rays=1 << 20, coarse_no_grad=False, exact_last_sample=None, fine_out=None,
                        coarse_outputs_unused=False, coarse_sigma_only=False):
    """Device-resident core of render_image: renders flattened pixel rows [ray_begin, +ray_count)
    and returns the six per-ray outputs of the fine AND coarse pass as CUDA tensors.  Rays are
    generated on the device (K1); ``launch_rays`` bounds the rays per kernel launch sequence.
    ``fine_out`` [ray_count,5]: destination rows of the fine (rgb, depth, acc) -- see render_rays."""
    dev = _model_device(coarse_model)
    width, height = int(width), int(height)
    total = width * height
    ray_count = total - ray_begin if ray_count is None else ray_count
    sc = int(coarse_sample_num)
    if t_rand is None:
        t_full = _draw_t_rand(total, sc, int(chunk), dev)
        t_rand = t_full[ray_begin:ray_begin + ray_count]
    outs = []
    for b in range(0, ray_count, launch_rays):
        cnt = min(launch_rays, ray_count - b)
        rays = ops.raygen(width, height, focal, pose, ray_begin + b, cnt, device=dev)
        outs.append(render_rays(rays, near, far, coarse_model, fine_model, coarse_sample_num, fine_sample_num,
                                t_rand=t_rand[b:b + cnt], precision=precision, coarse_no_grad=coarse_no_grad,
                                exact_last_sample=exact_last_sample, fine_out=None if fine_out is None else fine_out[b:b + cnt],
                                coarse_outputs_unused=coarse_outputs_unused, coarse_sigma_only=coarse_sigma_only))
    if len(outs) == 1:
        return outs[0]
    if fine_out is not None:                   # the fine maps already sit in fine_out's rows
        return tuple(torch.cat([o[i] for o in outs]) for i in range(3)) + (fine_out[:, :3], fine_out[:, 3], fine_out[:, 4])
    return tuple(torch.cat([o[i] for o in outs]) for i in range(6))


_host_stage: dict = {}      # (device index, rays) -> [(pinned [rays*5] staging buffer, its idle storage use count), ...]
_STAGE_POOL = 4             # staging buffers per frame size: frames the caller may hold at once without a host copy


def _storage_uses(buf: torch.Tensor):
    """Owners of the buffer's storage (the pool's tensor + every live numpy view chain made from it), or None if this torch
    build cannot tell."""
    f = getattr(torch._C, "_storage_Use_Count", None)
    return None if f is None else int(f(buf.untyped_storage()._cdata))


def maps_to_numpy(packed: torch.Tensor, h: int, w: int):
    """The frame's fine (rgb, depth, acc) rows [H*W,5] on the device -> the three numpy images the reference returns
    (nerf/render.py:161-166).  The rows are de-interleaved on the device and cross PCIe as ONE copy into a page-locked buffer
    (12.8 MB for an 800x800 frame); the three images are VIEWS of that buffer -- no host-side copy (three fresh 2.5-7.7 MB
    arrays cost 1.3-4.6 ms per frame in page faults, and far more on a busy host).  The caller owns them like any array: a
    buffer goes back to the pool only when the last view of it is gone (storage use count), up to _STAGE_POOL frames of a size can
    be held at once, and beyond that -- or when the use count is not available -- the images are fresh pageable arrays."""
    n = int(packed.shape[0])
    key = (packed.device.index, n)
    flat = torch.cat([packed[:, :3].reshape(-1), packed[:, 3], packed[:, 4]])
    pool = _host_stage.get(key)
    if pool is None:
        if len(_host_stage) >= 8:
            _host_stage.clear()
        pool = _host_stage[key] = []
    stage = None
    for buf, idle in pool:
        if idle is not None and _storage_uses(buf) == idle:
            stage = buf
            break
    if stage is None and len(pool) < _STAGE_POOL:
        stage = torch.empty((n * 5,), dtype=torch.float32, device="cpu", pin_memory=True)
        pool.append((stage, _storage_uses(stage)))
        if pool[-1][1] is None:                # cannot track the views: hand out copies of this one buffer
            stage = None
    if stage is None:
        idle0 = pool[0][1]
        if idle0 is None:                      # untracked single buffer: pinned copy + host copies
            buf = pool[0][0]
            buf.copy_(flat, non_blocking=True)
            torch.cuda.current_stream(packed.device).synchronize()
            a = buf.numpy().copy()
        else:                                  # every pooled buffer is still held by the caller
            a = flat.cpu().numpy()
    else:
        stage.copy_(flat, non_blocking=True)
        torch.cuda.current_stream(packed.device).synchronize()
        a = stage.numpy()
    return a[:3 * n].reshape(h, w, 3), a[3 * n:4 * n].reshape(h, w, 1), a[4 * n:].reshape(h, w, 1)


def render_image(width, height, focal, pose, near, far, coarse_model, fine_model, coarse_sample_num, fine_sample_num,
                 chunk=1024 * 16, *, t_rand=None, precision=None, exact_last_sample=None, coarse_sigma_only=False):
    """nerf/render.py:150-167 -- numpy (H,W,3), (H,W,1), (H,W,1) = fine rgb / depth / acc.
    ``coarse_sigma_only=True`` (opt-in): the coarse pass, whose colour this function never returns, stops after the sigma head
    (render_rays); the three images are bit-identical either way."""
    h, w = int(height), int(width)
    with torch.no_grad():
        packed = torch.empty((h * w, 5), dtype=torch.float32, device=_model_device(coarse_model))
        render_image_device(width, height, focal, pose, near, far, coarse_model, fine_model, coarse_sample_num,
                            fine_sample_num, chunk, t_rand=t_rand, precision=precision,
                            exact_last_sample=exact_last_sample, fine_out=packed, coarse_sigma_only=coarse_sigma_only,
                            coarse_outputs_unused=True)      # only the fine maps leave this function: no sign check on coarse rays
    return maps_to_numpy(packed, h, w)


def render_video(width, height, focal, poses, near, far, coarse_model, fine_model, coarse_sample_num, fine_sample_num,
                 chunk=1024 * 16, *, precision=None, exact_last_sample=None):
    """nerf/render.py:170-182 -- stacked per-pose render_image outputs."""
    poses = list(poses)
    h, w = int(height), int(width)
    # every frame is copied into the stacked result as it arrives (np.stack's copy, done early): the frame's staging buffer is free
    # again for the next pose
    rgb_video = np.empty((len(poses), h, w, 3), np.float32)
    depth_video, acc_video = np.empty((len(poses), h, w, 1), np.float32), np.empty((len(poses), h, w, 1), np.float32)
    for i, p in enumerate(tqdm(poses)):
        rgb, depth, acc = render_image(width, height, focal, p, near, far, coarse_model, fine_model, coarse_sample_num,
                                       fine_sample_num, chunk, precision=precision, exact_last_sample=exact_last_sample)
        rgb_video[i], depth_video[i], acc_video[i] = rgb, depth, acc
        del rgb, depth, acc
    return rgb_video, depth_video, acc_video


def render_video_u8(width, height, focal, poses, near, far, coarse_model, fine_model, coarse_sample_num, fine_sample_num,
                    chunk=1024 * 16, *, precision=None, exact_last_sample=None):
    """render_video + to8b (what show_nerf.py:55-66 does per frame on the host) with the quantisation on the device and the
    frames streamed out through two pinned buffers: frame k's 1.9 MB uint8 copy overlaps frame k+1's render, and the host
    waits only once per frame on an event.  Returns rgb uint8 [P,H,W,3]."""
    dev = _model_device(coarse_model)
    h, w = int(height), int(width)
    poses = list(poses)
    out = np.empty((len(poses), h, w, 3), dtype=np.uint8)
    # device="cpu": the reference's scripts set a CUDA default tensor type (demo_view.py, test_nerf.py)
    pinned = [torch.empty((h, w, 3), dtype=torch.uint8, device="cpu", pin_memory=True) for _ in range(2)]
    events = [torch.cuda.Event() for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    pending = [None, None]
    with torch.no_grad():
        for k, p in enumerate(tqdm(poses)):
            o = render_image_device(width, height, focal, p, near, far, coarse_model, fine_model, coarse_sample_num,
                                    fine_sample_num, chunk, precision=precision, exact_last_sample=exact_last_sample,
                                    coarse_outputs_unused=True)
            frame = ops.to8b(o[3]).reshape(h, w, 3)
            slot = k & 1
            if pending[slot] is not None:                       # the buffer's previous frame must have landed
                events[slot].synchronize()
                out[pending[slot]] = pinned[slot].numpy()
            copy_stream.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(copy_stream):
                pinned[slot].copy_(frame, non_blocking=True)
                frame.record_stream(copy_stream)
                events[slot].record(copy_stream)
            pending[slot] = k
    for slot in range(2):
        if pending[slot] is not None:
            events[slot].synchronize()
            out[pending[slot]] = pinned[slot].numpy()
    return out


def density_lattice(model, box_min=(-1.5, -1.5, -1.5), box_max=(1.5, 1.5, 1.5), N=256, *, max_batch=256 ** 3, precision=None):
    """Density of ``model`` (NeRF or SirenNeRF) on the box lattice of [box_min, box_max] with ``N`` points along the longest
    edge (mesh.box_lattice): ``(sigma [n0,n1,n2] on the device, origin, voxel)``, axis 0 slowest.  The points are made on the
    device from the lattice index with zero view direction; the bf16 NeRF path stops after the sigma head.  ``max_batch``
    bounds the points per launch."""
    dev = ops._model_args(model)[4]
    dims, origin, voxel = mesh.box_lattice(box_min, box_max, N)
    total = dims[0] * dims[1] * dims[2]
    sigma = torch.empty((total,), dtype=torch.float32, device=dev)
    with torch.no_grad():
        for b in range(0, total, int(max_batch)):
            c = min(int(max_batch), total - b)
            sigma[b:b + c] = ops.mlp(model, lattice=(dims, origin, voxel, b, c), precision=precision, sigma_only=True)[:, 3]
    return sigma.reshape(dims), origin, voxel


def create_mesh(model, ply_filename=None, N=256, *, box_min=(-1.5, -1.5, -1.5), box_max=(1.5, 1.5, 1.5), threshold=50.0,
                normals=True, colors=True, precision=None, max_batch=256 ** 3, min_component_ratio=0.0, smooth_iterations=0,
                max_faces=None, narrow_band=None, texture=None):
    """Mesh of a trained NeRF / SirenNeRF field on the device: the level set ``sigma = threshold`` of ``density_lattice``
    (marching cubes on -sigma at -threshold, so triangle and vertex normals point out of the object, toward lower density),
    the unit vertex normals, and the uint8 colour the model's rgb head gives each vertex seen by a camera looking along the
    inward normal (rows x = [vertex, -normal]).  Returns ``(verts [V,3] float32, faces [F,3] int32, normals [V,3] | None,
    colors [V,3] uint8 | None)`` on the device; with ``ply_filename`` also writes them as a binary PLY.  Synchronises with the
    host once to size the mesh.  The default box and threshold fit the Blender scenes (camera radius 4, near 2, far 6).
    ``min_component_ratio`` (finite, in [0, 1]) above 0 removes the floaters: every connected component with fewer triangles
    than that share of the largest component's (ops.filter_components; 1 keeps the largest and any tied with it), before the
    colour query; the call then synchronises with the host twice, once for the marching-cubes size and once for the filtered
    size.  0 (the default) keeps every triangle.
    ``smooth_iterations`` (an int >= 0) above 0 runs that many Taubin lambda|mu iterations on the mesh after the component
    filter and before the colour query (ops.smooth_mesh): the terraces marching cubes leaves where the density rises steeply
    through ``threshold`` are smoothed out without shrinking the surface, and the topology is unchanged.  The normals are then
    the smoothed mesh's own area-weighted vertex normals (still out of the object) and the colours are sampled at the smoothed
    vertices along them; no host synchronisation is added.  0 (the default) leaves the mesh as extracted.
    ``max_faces`` (an int >= 1) decimates the mesh to that many triangles (or one fewer) after the component filter and the
    smoothing and before the colour query (ops.decimate_mesh: rounds of quadric edge collapses that keep the topology, leave
    the open boundary where the surface meets the lattice box in place and never flip a face), so removed vertices cost no MLP
    rows.  The normals are then the decimated mesh's own area-weighted vertex normals (still out of the object) and the
    colours are sampled at the decimated vertices along them; the field normals are not computed.  Each round synchronises
    with the host once, to read its collapse count.  None (the default) leaves the mesh at its extracted size.
    ``narrow_band`` (an int B >= 2) queries the density only near the surface (mesh.band_field): at the corners of bricks of B
    cells, then in the bricks whose corners are not all on one side of ``threshold`` and their 26 neighbours, and marching cubes
    runs on those bricks only.  The mesh, normals and colours are the dense ones less the triangles outside those bricks, bit
    for bit, so a surface the brick corners cannot see -- a piece that lies within a brick and its neighbours without changing
    which side of the threshold any brick corner is on, such as a blob smaller than a brick -- is missed.  It adds one host
    synchronisation, to size the band.  The lattice may hold at most 2^31 - 1 points (RuntimeError before any launch
    otherwise), and the band's index list takes 4 B per lattice point beside the field.  None (the default) queries every
    lattice point.
    ``texture`` (an int R in [16, 16384]) bakes the colour of the final mesh -- after the component filter, the smoothing and
    the decimation -- into an R x R texture (mesh.bake_texture: one chart per face, every texel queried on the surface along
    the inward normal that the vertex colours use, ``max_batch`` rows per launch), so the colour detail no longer depends on
    the vertex count.  The mesh may have at most 2 * (R // 4)^2 faces (ValueError otherwise; ``max_faces`` bounds it).  The
    result gains ``(uvs [F,3,2] float32, texture [R,R,3] uint8)``; with ``ply_filename`` the PLY's faces carry
    ``texcoord`` lists, its header names the texture, and the texture is written as ``<stem>.png`` beside it.  None (the
    default) bakes nothing."""
    texture = None if texture is None else ops._check_int("texture", texture, *ops.ATLAS_SIZES)
    stride = None if narrow_band is None else ops._check_int("narrow_band", narrow_band, 2, ops._INT32_MAX)
    if stride is None:
        sigma, origin, voxel = density_lattice(model, box_min, box_max, N, max_batch=max_batch, precision=precision)
        field, bricks = sigma.neg_(), None
    else:
        dims, origin, voxel = mesh.box_lattice(box_min, box_max, N)
        mesh.check_band_lattice(dims)
        field, flags = mesh.band_field(model, dims, -float(threshold), stride, lattice=(dims, origin, voxel, 0, math.prod(dims)),
                                       max_batch=int(max_batch), precision=precision)
        bricks = (stride, flags)
    return mesh.export(model, field, -float(threshold), voxel, origin, ply_filename, normals, colors, precision,
                       min_component_ratio, smooth_iterations, max_faces, bricks, texture, int(max_batch))
