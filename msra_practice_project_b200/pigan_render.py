"""Drop-in replacement for the reference's ``pi_GAN/render.py`` backed by libb2r.so (sm_100a CUDA).

Lines 52-192 of the reference file are byte-identical to ``nerf/render.py:7-147`` (SURVEY.md 0), so
the shared functions are re-exported from :mod:`nerf_render`; this module adds the radian camera
helpers (pi_GAN/render.py:6-49) and the pi-GAN image wrappers (:195-241).  Callers:
pi_GAN/modules.py:3,160, train.py:8, synthesis.py:9, extract_mesh.py:8, utils.py.
"""
from __future__ import annotations

import numpy as np
import torch
from tqdm import tqdm

from . import ops
from .mesh import band_field, check_band_lattice, export as _export_mesh, write_ply  # noqa: F401  (pigan_render.write_ply is public)
from .nerf_render import (REFERENCE_RAY_CHUNK, _draw_t_rand, get_rays, maps_to_numpy, raw_to_outputs, render_image_device, render_rays,
                          run_network, sample_pdf, to8b)

__all__ = ["np", "torch", "tqdm", "to8b", "trans_t", "rot_phi", "rot_theta", "blender_coord",
           "camera_pos_to_transform_matrix", "get_rays", "sample_pdf", "run_network", "raw_to_outputs", "render_rays",
           "render_image", "render_image_np", "render_video_np", "render_batch", "density_grid"]

# pi_GAN/render.py:6-35 (angles in radians)
trans_t = lambda t: np.array([[1, 0, 0, 0], [0, 1, 0, 0], [0, 0, 1, t], [0, 0, 0, 1]], dtype=np.float32)
rot_phi = lambda phi: np.array([[1, 0, 0, 0], [0, np.cos(phi), -np.sin(phi), 0], [0, np.sin(phi), np.cos(phi), 0],
                                [0, 0, 0, 1]], dtype=np.float32)
rot_theta = lambda th: np.array([[np.cos(th), 0, -np.sin(th), 0], [0, 1, 0, 0], [np.sin(th), 0, np.cos(th), 0],
                                 [0, 0, 0, 1]], dtype=np.float32)
blender_coord = np.array([[-1, 0, 0, 0], [0, 0, 1, 0], [0, 1, 0, 0], [0, 0, 0, 1]], dtype=np.float32)


def camera_pos_to_transform_matrix(radius, theta, phi):
    """pi_GAN/render.py:38-49 -- camera-to-world matrix of a camera on a sphere."""
    c2w = trans_t(radius)
    c2w = rot_phi(phi) @ c2w
    c2w = rot_theta(theta) @ c2w
    return c2w


def render_image(width, height, focal, pose, near, far, coarse_model, fine_model, coarse_sample_num, fine_sample_num,
                 chunk=1024 * 16, *, t_rand=None, precision=None, exact_last_sample=None, coarse_sigma_only=False):
    """pi_GAN/render.py:195-206 -- fine rgb as a torch tensor [H,W,3] on the device, carrying the
    autograd graph to the model parameters and the FiLM parameters (pi_GAN/train.py:134,
    synthesis.py:107).  In pi-GAN coarse_model is fine_model and only the fine rgb is consumed, so
    the coarse pass carries no gradient (SURVEY A.6) and runs in inference mode."""
    out = _render(width, height, focal, pose, near, far, coarse_model, fine_model, coarse_sample_num, fine_sample_num,
                  chunk, t_rand, precision, coarse_no_grad=True, exact_last_sample=exact_last_sample, coarse_outputs_unused=True,
                  coarse_sigma_only=coarse_sigma_only)
    return out[3].reshape(int(height), int(width), 3)


def _render(width, height, focal, pose, near, far, coarse_model, fine_model, sc, sf, chunk, t_rand, precision,
            coarse_no_grad=False, exact_last_sample=None, coarse_outputs_unused=False, coarse_sigma_only=False):
    return render_image_device(width, height, focal, pose, near, far, coarse_model, fine_model, sc, sf, chunk,
                               t_rand=t_rand, precision=precision, coarse_no_grad=coarse_no_grad,
                               exact_last_sample=exact_last_sample, coarse_outputs_unused=coarse_outputs_unused,
                               coarse_sigma_only=coarse_sigma_only)


def render_image_np(width, height, focal, pose, near, far, coarse_model, fine_model, coarse_sample_num,
                    fine_sample_num, chunk=1024 * 16, *, t_rand=None, precision=None, exact_last_sample=None):
    """pi_GAN/render.py:209-226 -- numpy (H,W,3), (H,W,1), (H,W,1)."""
    h, w = int(height), int(width)
    with torch.no_grad():
        packed = torch.empty((h * w, 5), dtype=torch.float32, device=next(coarse_model.parameters()).device)
        render_image_device(width, height, focal, pose, near, far, coarse_model, fine_model, coarse_sample_num, fine_sample_num,
                            chunk, t_rand=t_rand, precision=precision, exact_last_sample=exact_last_sample, fine_out=packed,
                            coarse_outputs_unused=True)
    return maps_to_numpy(packed, h, w)


def render_video_np(width, height, focal, poses, near, far, coarse_model, fine_model, coarse_sample_num,
                    fine_sample_num, chunk=1024 * 16, *, precision=None, exact_last_sample=None):
    """pi_GAN/render.py:229-241.  The reference unpacks three values from render_image (which returns
    one tensor) and so raises as shipped (SURVEY app. D); this calls render_image_np as evidently meant."""
    poses = list(poses)
    h, w = int(height), int(width)
    rgb_video = np.empty((len(poses), h, w, 3), np.float32)       # frames copied in as they arrive: their staging buffers are reused
    depth_video, acc_video = np.empty((len(poses), h, w, 1), np.float32), np.empty((len(poses), h, w, 1), np.float32)
    for i, p in enumerate(tqdm(poses)):
        rgb, depth, acc = render_image_np(width, height, focal, p, near, far, coarse_model, fine_model, coarse_sample_num,
                                          fine_sample_num, chunk, precision=precision, exact_last_sample=exact_last_sample)
        rgb_video[i], depth_video[i], acc_video[i] = rgb, depth, acc
        del rgb, depth, acc
    return rgb_video, depth_video, acc_video


def render_batch(model, film_params, poses, width, height, focal, near, far, coarse_sample_num, fine_sample_num, *,
                 t_rand=None, precision=None, exact_last_sample=None, coarse_sigma_only=False):
    """Batched counterpart of Generator.forward's per-latent loop (pi_GAN/modules.py:176-184):
    film_params[B,9,512], poses[B,4,4] -> images [B,3,H,W].  This is the latent-sharding unit for
    multi-GPU runs (each rank renders its slice of B).

    With the bf16 tensor-core MLP the B latents are rendered by ONE launch sequence (rays of all poses, one batched MLP launch
    per pass with per-latent FiLM tables) -- also WITH gradients (pi_GAN/train.py:134: the fine pass runs on the fused
    training path for all latents at once, the coarse pass carries no gradient as in render_image); otherwise latent by
    latent through render_image.  ``coarse_sigma_only=True`` (opt-in): the coarse pass, whose colour never reaches the image, stops
    after the sigma head; the images are bit-identical either way."""
    b = film_params.shape[0]
    w, h, sc, sf = int(width), int(height), int(coarse_sample_num), int(fine_sample_num)
    dev = ops._model_args(model)[4]
    used = precision or ops.get_mlp_precision()
    grad = torch.is_grad_enabled() and _needs_grad(model, film_params)
    grad_ok = ops.get_grad_precision() == "bf16" and isinstance(film_params, torch.Tensor)
    batched = (not grad or grad_ok) and used == "bf16" and b > 0 and (w * h * sc) % 512 == 0 and (w * h * (sc + sf)) % 512 == 0
    if not batched:
        imgs = []
        for i in range(b):
            model.set_film_params(film_params[i])
            tr = None if t_rand is None else t_rand[i]
            imgs.append(render_image(width, height, focal, poses[i], near, far, model, model, coarse_sample_num,
                                     fine_sample_num, t_rand=tr, precision=precision, exact_last_sample=exact_last_sample,
                                     coarse_sigma_only=coarse_sigma_only))
        return torch.stack(imgs).permute(0, 3, 1, 2).contiguous()
    n = w * h
    with torch.no_grad():
        if isinstance(poses, torch.Tensor) and poses.is_cuda:
            rays = ops.raygen_poses(w, h, focal, poses)         # poses on the device: one launch, replayable inside a CUDA graph
        else:
            rays = torch.cat([ops.raygen(w, h, focal, poses[i], device=dev) for i in range(b)])        # [B*HW,2,3]
        if t_rand is None:
            t_all = torch.cat([_draw_t_rand(n, sc, REFERENCE_RAY_CHUNK, dev) for _ in range(b)])         # the reference's draw order
        else:
            t_all = torch.as_tensor(t_rand, dtype=torch.float32).to(dev).reshape(b * n, sc)
        z_lin = ops.host_linspace(near, far, sc, dev)
        u = ops.host_linspace(0.0, 1.0, sf, dev)
        film = torch.as_tensor(film_params, dtype=torch.float32).to(dev).reshape(b, 9, 512)
        z, mids = ops.stratified_z(z_lin, t_all)
        # coarse pass: only weights[:, 1:-1] are used (the image is the fine colour), so its last sample needs no sign check
        raw = ops.mlp_film_batched(model, film, rays, z, n * sc, exact_last_sample=False, sigma_only=bool(coarse_sigma_only))
        _, _, _, wts, _ = ops.composite_forward(raw, z, rays[:, 1], True)
        z_f = ops.sample_pdf(mids, wts[:, 1:-1], sf, u=u, z_coarse=z, want_samples=False)["sorted"]
        if not grad:
            raw_f = ops.mlp_film_batched(model, film, rays, z_f, n * (sc + sf), exact_last_sample=exact_last_sample)
            rgb, _, _, _, _ = ops.composite_forward(raw_f, z_f, rays[:, 1], False)
    if grad:
        film_g = film_params.to(dev).reshape(b, 9, 512)
        raw_f = ops.mlp_film_batched_train(model, film_g, rays, z_f, n * (sc + sf))
        rgb = ops.composite(raw_f, z_f, rays[:, 1], False)[0]
    return rgb.reshape(b, h, w, 3).permute(0, 3, 1, 2).contiguous()


def _needs_grad(model, film_params) -> bool:
    return any(p.requires_grad for p in model.parameters()) or (isinstance(film_params, torch.Tensor) and film_params.requires_grad)


def density_grid(model, N=256, max_batch=64 ** 3, *, begin=0, count=None, precision=None):
    """The sampling loop of create_mesh (pi_GAN/utils.py:59-91): -sigma at the N^3 lattice points of
    [-0.1,0.1]^3 with zero view direction, as a CUDA tensor [count].  Coordinates are generated on
    the device from the linear index; ``max_batch`` bounds the points per launch like the reference."""
    n3 = N ** 3
    count = n3 - begin if count is None else count
    out = []
    with torch.no_grad():
        for b in range(begin, begin + count, max_batch):
            c = min(max_batch, begin + count - b)
            raw = ops.mlp(model, grid=(N, b, c), precision=precision, sigma_only=True)
            out.append(-raw[:, 3])
    return out[0] if len(out) == 1 else torch.cat(out)


def _sdf_device(generator, N, max_batch, z, precision, band=None):
    """-sigma of the generator conditioned on z (drawn when None) on the N^3 lattice, as a CUDA tensor [N,N,N] (x slowest).
    With ``band = (level, stride)`` the narrow-band query of mesh.band_field instead: ``(sdf, flags)``."""
    dev = next(generator.parameters()).device
    if dev.type != "cuda":
        raise RuntimeError("generator parameters must live on a CUDA device: the B200 render path has no CPU fallback")
    if z is None:
        z = torch.randn(1, generator.input_dim, device=dev)               # pi_GAN/utils.py:48
    with torch.no_grad():
        film_params = generator.get_mapping(z.to(dev))
        generator.set_film_params(film_params[0])
        if band is not None:
            return band_field(generator.film_siren_nerf, (N, N, N), band[0], band[1], grid=(N, 0, N ** 3), max_batch=max_batch,
                              precision=precision)
        sdf = density_grid(generator.film_siren_nerf, N=N, max_batch=max_batch, precision=precision)
    return sdf.reshape(N, N, N)


def create_mesh_sdf(generator, N=256, max_batch=64 ** 3, *, z=None, precision=None):
    """The sampling half of ``create_mesh`` (pi_GAN/utils.py:42-97; called by extract_mesh.py:49): draw z ~ N(0,1) on the
    device, map it to FiLM parameters, condition the field and query -sigma on the N^3 lattice of [-0.1, 0.1]^3 with zero view
    direction.  Returns what the reference hands to ``convert_sdf_samples_to_ply`` -- ``sdf_values`` as a CPU tensor
    [N,N,N] (x slowest) -- plus ``voxel_origin`` and ``voxel_size``; ``create_mesh`` below keeps the sdf on the device and
    extracts the mesh there.  ``generator``: models.Generator or the reference's Generator (same attributes)."""
    return _sdf_device(generator, N, max_batch, z, precision).cpu(), [-0.1, -0.1, -0.1], 0.2 / (N - 1)


def create_mesh(generator, ply_filename=None, N=256, max_batch=64 ** 3, *, level=-20.0, z=None, precision=None, normals=False,
                colors=False, min_component_ratio=0.0, smooth_iterations=0, max_faces=None, narrow_band=None, texture=None):
    """``create_mesh`` (pi_GAN/utils.py:42-180) on the device: the sdf of ``create_mesh_sdf`` never leaves the GPU,
    ``ops.marching_cubes`` extracts its level set (the reference's skimage call at level -20: below = sigma > 20, so the
    triangle normals point out of the object), and only the mesh crosses to the host.  Returns ``(verts [V,3] float32,
    faces [F,3] int32)`` on the device, in world coordinates (voxel origin -0.1, voxel size 0.2/(N-1)).  With
    ``ply_filename`` the mesh is also written as the binary PLY the reference writes with plyfile (``vertex`` x/y/z f4,
    ``face`` vertex_indices as a uchar-counted list of i4).  Synchronises with the host once to size the mesh.
    ``normals`` / ``colors``: also compute the unit vertex normals (out of the object) and the uint8 colours the conditioned
    generator's rgb head gives each vertex seen along the inward normal; the PLY then carries nx/ny/nz and red/green/blue,
    and the return value is ``(verts, faces, normals | None, colors | None)``.
    ``min_component_ratio`` (finite, in [0, 1]) above 0 removes every connected component with fewer triangles than that share
    of the largest component's (ops.filter_components; 1 keeps the largest and any tied with it), before the colour query; the
    call then synchronises with the host twice, once for the marching-cubes size and once for the filtered size.  0 (the
    default) keeps every triangle.
    ``smooth_iterations`` (an int >= 0) above 0 runs that many Taubin lambda|mu iterations on the mesh after the component
    filter and before the colour query (ops.smooth_mesh): the terraces marching cubes leaves along the lattice are smoothed
    out without moving the surface inward, and the topology is unchanged.  The normals are then the smoothed mesh's own
    area-weighted vertex normals and the colours are sampled at the smoothed vertices; no host synchronisation is added.
    0 (the default) leaves the mesh as extracted.
    ``max_faces`` (an int >= 1) decimates the mesh to that many triangles (or one fewer) after the component filter and the
    smoothing and before the colour query (ops.decimate_mesh: rounds of quadric edge collapses that keep the topology, leave
    the open boundary where the surface meets the lattice box in place and never flip a face), so removed vertices cost no MLP
    rows.  The normals are then the decimated mesh's own area-weighted vertex normals (still out of the object) and the
    colours are sampled at the decimated vertices along them; the field normals are not computed.  Each round synchronises
    with the host once, to read its collapse count.  None (the default) leaves the mesh at its extracted size.
    ``narrow_band`` (an int B >= 2) queries the density only near the surface (mesh.band_field): at the corners of bricks of B
    cells, then in the bricks whose corners are not all on one side of ``level`` and their 26 neighbours, and marching cubes
    runs on those bricks only.  The mesh, normals and colours are the dense ones less the triangles outside those bricks, bit
    for bit, so a surface the brick corners cannot see -- a piece that lies within a brick and its neighbours without changing
    which side of the level any brick corner is on, such as a blob smaller than a brick -- is missed.  It adds one host
    synchronisation, to size the band.  The lattice may hold at most 2^31 - 1 points (RuntimeError before any launch
    otherwise), and the band's index list takes 4 B per lattice point beside the field.  None (the default) queries every
    lattice point; ``create_mesh_sdf`` and ``density_grid`` always do.
    ``texture`` (an int R in [16, 16384]) bakes the conditioned generator's colour on the final mesh -- after the component
    filter, the smoothing and the decimation -- into an R x R texture (mesh.bake_texture: one chart per face, every texel
    queried on the surface along the inward normal, ``max_batch`` rows per launch).  The mesh may have at most 2 * (R // 4)^2
    faces (ValueError otherwise; ``max_faces`` bounds it).  The return value is then ``(verts, faces, normals | None,
    colors | None, uvs [F,3,2] float32, texture [R,R,3] uint8)``; with ``ply_filename`` the PLY's faces carry ``texcoord``
    lists, its header names the texture, and the texture is written as ``<stem>.png`` beside it.  None (the default) bakes
    nothing."""
    texture = None if texture is None else ops._check_int("texture", texture, *ops.ATLAS_SIZES)
    stride = None if narrow_band is None else ops._check_int("narrow_band", narrow_band, 2, ops._INT32_MAX)
    if stride is None:
        sdf, bricks = _sdf_device(generator, N, max_batch, z, precision), None
    else:
        check_band_lattice((N, N, N))
        sdf, flags = _sdf_device(generator, N, max_batch, z, precision, (float(level), stride))
        bricks = (stride, flags)
    out = _export_mesh(generator.film_siren_nerf, sdf, level, 0.2 / (N - 1), (-0.1, -0.1, -0.1), ply_filename, normals, colors,
                       precision, min_component_ratio, smooth_iterations, max_faces, bricks, texture, int(max_batch))
    return out if (normals or colors or texture is not None) else out[:2]
