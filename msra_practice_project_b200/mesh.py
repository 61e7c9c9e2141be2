"""Mesh export shared by ``nerf_render.create_mesh`` and ``pigan_render.create_mesh``: level-set extraction with vertex
normals, per-vertex colour from the model's rgb head, texture baking into a per-face atlas, and the binary PLY and PNG writers.
Everything up to the file writes stays on the device."""
from __future__ import annotations

import math
import os
import struct
import zlib

import numpy as np
import torch

from . import ops


def box_lattice(box_min, box_max, n):
    """(dims, origin, voxel) of the lattice spanning [box_min, box_max]: ``n`` points along the longest edge
    (voxel = longest / (n - 1)) and ``ceil(extent / voxel) + 1`` points along every axis, starting at ``box_min``; origin and
    voxel are rounded to float32, the precision the kernels use."""
    lo = [float(v) for v in box_min]
    hi = [float(v) for v in box_max]
    ext = [b - a for a, b in zip(lo, hi)]
    if len(lo) != 3 or len(hi) != 3 or min(ext) <= 0 or int(n) < 2:
        raise ValueError("box_min / box_max must be 3-vectors with box_min < box_max on every axis, and N >= 2")
    step = max(ext) / (int(n) - 1)
    dims = tuple(int(math.ceil(round(e / step, 9))) + 1 for e in ext)      # the longest axis gets exactly n points
    return dims, tuple(float(np.float32(v)) for v in lo), float(np.float32(step))


def check_band_lattice(dims) -> None:
    """RuntimeError unless a lattice of ``dims`` points fits the narrow-band export: its int32 point indices and marching cubes
    take at most 2^31 - 1 points.  Runs on the host, so create_mesh raises it before any launch."""
    points = math.prod(int(d) for d in dims)
    if points > ops._INT32_MAX:
        raise RuntimeError(f"lattice of {points} points; the narrow-band export and marching_cubes take at most 2^31 - 1")


def coarse_index(dims, stride, device) -> torch.Tensor:
    """int32 linear indices (ascending) of the coarse corners of bricks of ``stride`` cells: the points ``min(b * stride, n - 1)``
    on every axis."""
    axes = [torch.clamp(torch.arange(nb + 1, device=device) * stride, max=n - 1) for n, nb in zip(dims, ops.brick_dims(dims, stride))]
    return ((axes[0][:, None, None] * dims[1] + axes[1][None, :, None]) * dims[2] + axes[2][None, None, :]).reshape(-1).to(torch.int32)


def query_rows(model, field, index, *, grid=None, lattice=None, max_batch, precision=None) -> None:
    """field.view(-1)[index] = -sigma of ``model`` at rows ``index`` of the ``grid`` or ``lattice`` description (the sigma-only MLP
    on ``ops.lattice_rows`` x rows, ``max_batch`` rows per launch), so each value is the dense query's."""
    flat = field.view(-1)
    for b in range(0, index.shape[0], max_batch):
        rows = index[b:b + max_batch]
        raw = ops.mlp(model, x=ops._lattice_rows(rows, grid, lattice), precision=precision, sigma_only=True)
        flat.index_copy_(0, rows.long(), -raw[:, 3])


def band_field(model, dims, level, stride, *, grid=None, lattice=None, max_batch, precision=None):
    """-sigma of ``model`` on the lattice of ``dims`` points queried only near the level set: at the coarse corners of bricks of
    ``stride`` cells, then at the points ``ops.band_select`` lists for them; every other point holds +inf.  The lattice is one
    ``grid = (N, 0, N^3)`` or ``lattice = (dims, origin, voxel, 0, count)`` description as ``ops.mlp`` takes it (query_rows).
    Returns ``(field [n0,n1,n2], flags)``; synchronises with the host once, in ``ops.band_select``.  Besides the field, the
    index list of ``ops.band_select`` (4 B per lattice point) is held until the band query ends."""
    check_band_lattice(dims)
    dev = ops._model_args(model)[4]
    field = torch.full(tuple(dims), math.inf, dtype=torch.float32, device=dev)
    with torch.no_grad():
        query_rows(model, field, coarse_index(dims, stride, dev), grid=grid, lattice=lattice, max_batch=max_batch,
                   precision=precision)
        flags, index = ops.band_select(field, level, stride)
        query_rows(model, field, index, grid=grid, lattice=lattice, max_batch=max_batch, precision=precision)
    return field, flags


def vertex_colors(model, verts, normals, precision=None):
    """uint8 [V,3] colours of the model's rgb head at each vertex, seen by a camera looking along ``-normals``
    (rows x = [vertex, -normal]), quantised on the device by ops.to8b."""
    if verts.shape[0] == 0:
        return torch.empty((0, 3), dtype=torch.uint8, device=verts.device)
    with torch.no_grad():
        raw = ops.mlp(model, x=torch.cat([verts, -normals], 1), precision=precision)
        return ops.to8b(raw[:, :3])


def _bake_texture(model, verts, faces, normals, size, precision, max_batch):
    """bake_texture for a mesh already checked by ops._mesh_args."""
    cells, _, s = ops.atlas_layout(faces.shape[0], size)
    dev = verts.device
    uvs = ops._atlas_uvs(faces.shape[0], size, dev)
    texture = torch.zeros((size, size, 3), dtype=torch.uint8, device=dev)
    rows = cells * s * s
    with torch.no_grad(), torch.cuda.device(dev):
        for b in range(0, rows, max_batch):
            c = min(max_batch, rows - b)
            raw = ops.mlp(model, x=ops._atlas_rows(verts, faces, normals, size, b, c), precision=precision)
            ops._atlas_texture(raw, faces.shape[0], size, b, texture)
    return uvs, texture


def bake_texture(model, verts, faces, normals, size, *, precision=None, max_batch=256 ** 3):
    """Bakes the colour of ``model``'s rgb head on the surface of a triangle mesh into a ``size`` x ``size`` texture on the
    device.  Each face gets its own chart in a per-face atlas (ops.atlas_layout; include/b2r.h): faces 2k and 2k+1 share a square
    cell, and a bilinear lookup inside a face's UV triangle reads only texels baked for that face, so charts do not bleed into
    each other (mipmap levels do).  Every texel is queried at its barycentric point on its face, seen by a camera looking along
    the inward interpolated normal (rows x = [point, -normal], as ``vertex_colors`` queries the vertices), and quantised like
    ops.to8b; texels of no face are 0.  The rows are made and queried ``max_batch`` at a time (b2r_mesh_atlas_rows, the MLP,
    b2r_mesh_atlas_texture).  Returns ``(uvs [F,3,2] float32, texture [size,size,3] uint8)`` on the device; row 0 of the texture
    is the top of the image (v = 1).  Works for NeRF, SirenNeRF and FilmSirenNeRF (with its FiLM parameters set).
    ``verts`` / ``normals`` [V,3] float32 and ``faces`` [F,3] int32 are checked like every mesh op (RuntimeError, one host
    synchronisation); ``size`` must be an int in [16, 16384] and F at most 2 * (size // 4)^2 (ValueError), both before any
    launch."""
    size = ops._check_int("texture size", size, *ops.ATLAS_SIZES)
    max_batch = ops._check_int("max_batch", max_batch, 1)
    verts, faces, normals = ops._mesh_args(verts, faces, normals)
    if normals is None:
        raise RuntimeError("bake_texture needs the vertex normals [V,3]")
    ops.atlas_layout(faces.shape[0], size)
    return _bake_texture(model, verts, faces, normals, size, precision, max_batch)


def write_png(filename, rgb):
    """8-bit RGB PNG of a uint8 [H,W,3] image, row 0 at the top: zlib-compressed rows, each with filter 0 (none)."""
    rgb = np.ascontiguousarray(rgb, dtype=np.uint8)
    if rgb.ndim != 3 or rgb.shape[2] != 3 or not rgb.shape[0] or not rgb.shape[1]:
        raise ValueError(f"write_png takes a non-empty [H,W,3] uint8 image, got shape {list(rgb.shape)}")
    h, w = rgb.shape[:2]
    raw = np.concatenate([np.zeros((h, 1), np.uint8), rgb.reshape(h, 3 * w)], 1).tobytes()

    def chunk(tag, data):
        return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data))
    with open(filename, "wb") as fh:
        fh.write(b"\x89PNG\r\n\x1a\n" + chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 2, 0, 0, 0))
                 + chunk(b"IDAT", zlib.compress(raw)) + chunk(b"IEND", b""))


def write_ply(filename, verts, faces, normals=None, colors=None, uvs=None, texture_file=None):
    """Binary little-endian PLY of a triangle mesh: ``vertex`` with float x/y/z, then float nx/ny/nz when ``normals`` is given
    and uchar red/green/blue when ``colors`` is given; ``face`` with ``property list uchar int vertex_indices``.  Without
    normals and colours it is byte for byte what plyfile writes for the reference's elements (pi_GAN/utils.py:158-180).
    ``uvs`` [F,3,2] adds ``property list uchar float texcoord`` (u0 v0 u1 v1 u2 v2 per face) and ``texture_file`` the header
    line ``comment TextureFile <texture_file>``, the convention MeshLab reads."""
    verts = np.asarray(verts, dtype="<f4").reshape(-1, 3)
    faces = np.asarray(faces).reshape(-1, 3)
    fields = [("x", "<f4"), ("y", "<f4"), ("z", "<f4")]
    props = "property float x\nproperty float y\nproperty float z\n"
    if normals is not None:
        fields += [("nx", "<f4"), ("ny", "<f4"), ("nz", "<f4")]
        props += "property float nx\nproperty float ny\nproperty float nz\n"
    if colors is not None:
        fields += [("red", "u1"), ("green", "u1"), ("blue", "u1")]
        props += "property uchar red\nproperty uchar green\nproperty uchar blue\n"
    vbody = np.empty(len(verts), dtype=fields)
    for c, name in enumerate("xyz"):
        vbody[name] = verts[:, c]
    if normals is not None:
        normals = np.asarray(normals, dtype="<f4").reshape(-1, 3)
        for c, name in enumerate(("nx", "ny", "nz")):
            vbody[name] = normals[:, c]
    if colors is not None:
        colors = np.asarray(colors, dtype=np.uint8).reshape(-1, 3)
        for c, name in enumerate(("red", "green", "blue")):
            vbody[name] = colors[:, c]
    ffields = [("n", "u1"), ("vertex_indices", "<i4", (3,))]
    fprops = "property list uchar int vertex_indices\n"
    if uvs is not None:
        ffields += [("nt", "u1"), ("texcoord", "<f4", (6,))]
        fprops += "property list uchar float texcoord\n"
    fbody = np.empty(len(faces), dtype=ffields)
    fbody["n"] = 3
    fbody["vertex_indices"] = faces
    if uvs is not None:
        fbody["nt"] = 6
        fbody["texcoord"] = np.asarray(uvs, dtype="<f4").reshape(-1, 6)
    comment = "" if texture_file is None else f"comment TextureFile {texture_file}\n"
    header = (f"ply\nformat binary_little_endian 1.0\n{comment}"
              f"element vertex {len(verts)}\n{props}"
              f"element face {len(faces)}\n{fprops}end_header\n")
    with open(filename, "wb") as fh:
        fh.write(header.encode("ascii"))
        vbody.tofile(fh)
        fbody.tofile(fh)


def export(model, field, level, spacing, origin, ply_filename, normals, colors, precision, min_component_ratio=0.0,
           smooth_iterations=0, max_faces=None, bricks=None, texture=None, max_batch=256 ** 3):
    """Extract the level set of ``field`` (vertex normals toward increasing field), colour it with ``model`` and write the PLY.
    Returns (verts, faces, normals | None, colors | None) on the device.  A ``min_component_ratio`` above 0 removes the
    components with fewer triangles than that share of the largest one (ops.filter_components) before the colour query, so
    dropped vertices cost no MLP rows; it synchronises with the host once more, to size the filtered mesh.
    ``smooth_iterations`` above 0 then runs that many Taubin iterations (ops.smooth_mesh) before the colour query, and the
    normals become the smoothed mesh's own, so colours are sampled on the smoothed surface; the field normals are not computed.
    ``max_faces`` (an int >= 1) then decimates the mesh to that many triangles (ops.decimate_mesh; one host synchronisation per
    round) before the colour query, so removed vertices cost no MLP rows, and the normals are the decimated mesh's own.
    ``bricks = (stride, flags)`` limits the extraction to the flagged bricks (``ops.marching_cubes(bricks=...)``; the field of
    ``band_field``).
    ``texture`` (an int R in [16, 16384]) bakes the final mesh's colour into an R x R texture last (``bake_texture`` along the
    normals the colour query uses, ``max_batch`` rows per launch) and appends ``(uvs, texture)`` to the result; with
    ``ply_filename`` the PLY gets the face texcoords and a TextureFile comment, and the texture is written as ``<stem>.png``
    beside it."""
    iterations = ops._check_int("iterations", smooth_iterations, 0, ops._INT32_MAX)
    budget = None if max_faces is None else ops._check_int("max_faces", max_faces, 1)
    size = None if texture is None else ops._check_int("texture", texture, *ops.ATLAS_SIZES)
    want_normals = normals or colors or size is not None
    own_normals = want_normals and (iterations or budget is not None)
    if want_normals and not own_normals:
        verts, faces, nrm = ops.marching_cubes(field, level, spacing, origin, normals=True, bricks=bricks)
    else:
        (verts, faces), nrm = ops.marching_cubes(field, level, spacing, origin, bricks=bricks), None
    if min_component_ratio:
        # marching-cubes faces index their own vertices, so the index checks of ops.filter_components / ops.smooth_mesh are not needed
        verts, faces, nrm = ops._filter_components(verts, faces, ops._check_ratio(min_component_ratio), nrm)
    if iterations:
        verts, nrm = ops._smooth_mesh(verts, faces, iterations, want_normals and budget is None)
    if budget is not None:
        verts, faces = ops._decimate_mesh(verts, faces, budget)
        if want_normals:
            verts, nrm = ops._smooth_mesh(verts, faces, 0, True)
    rgb = vertex_colors(model, verts, nrm, precision) if colors else None
    baked = None if size is None else _bake_texture(model, verts, faces, nrm, size, precision, max_batch)
    if not normals:
        nrm = None
    if ply_filename is not None:
        png = None if baked is None else os.path.splitext(ply_filename)[0] + ".png"
        write_ply(ply_filename, verts.cpu().numpy(), faces.cpu().numpy(), None if nrm is None else nrm.cpu().numpy(),
                  None if rgb is None else rgb.cpu().numpy(), None if baked is None else baked[0].cpu().numpy(),
                  None if png is None else os.path.basename(png))
        if png is not None:
            write_png(png, baked[1].cpu().numpy())
    return (verts, faces, nrm, rgb) + (() if baked is None else baked)
