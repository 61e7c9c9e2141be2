"""Mesh export shared by ``nerf_render.create_mesh`` and ``pigan_render.create_mesh``: level-set extraction with vertex
normals, per-vertex colour from the model's rgb head, and the binary PLY writer.  Everything up to the PLY write stays on the
device."""
from __future__ import annotations

import math

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


def write_ply(filename, verts, faces, normals=None, colors=None):
    """Binary little-endian PLY of a triangle mesh: ``vertex`` with float x/y/z, then float nx/ny/nz when ``normals`` is given
    and uchar red/green/blue when ``colors`` is given; ``face`` with ``property list uchar int vertex_indices``.  Without
    normals and colours it is byte for byte what plyfile writes for the reference's elements (pi_GAN/utils.py:158-180)."""
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
    fbody = np.empty(len(faces), dtype=[("n", "u1"), ("vertex_indices", "<i4", (3,))])
    fbody["n"] = 3
    fbody["vertex_indices"] = faces
    header = ("ply\nformat binary_little_endian 1.0\n"
              f"element vertex {len(verts)}\n{props}"
              f"element face {len(faces)}\nproperty list uchar int vertex_indices\nend_header\n")
    with open(filename, "wb") as fh:
        fh.write(header.encode("ascii"))
        vbody.tofile(fh)
        fbody.tofile(fh)


def export(model, field, level, spacing, origin, ply_filename, normals, colors, precision, min_component_ratio=0.0,
           smooth_iterations=0, max_faces=None, bricks=None):
    """Extract the level set of ``field`` (vertex normals toward increasing field), colour it with ``model`` and write the PLY.
    Returns (verts, faces, normals | None, colors | None) on the device.  A ``min_component_ratio`` above 0 removes the
    components with fewer triangles than that share of the largest one (ops.filter_components) before the colour query, so
    dropped vertices cost no MLP rows; it synchronises with the host once more, to size the filtered mesh.
    ``smooth_iterations`` above 0 then runs that many Taubin iterations (ops.smooth_mesh) before the colour query, and the
    normals become the smoothed mesh's own, so colours are sampled on the smoothed surface; the field normals are not computed.
    ``max_faces`` (an int >= 1) then decimates the mesh to that many triangles (ops.decimate_mesh; one host synchronisation per
    round) before the colour query, so removed vertices cost no MLP rows, and the normals are the decimated mesh's own.
    ``bricks = (stride, flags)`` limits the extraction to the flagged bricks (``ops.marching_cubes(bricks=...)``; the field of
    ``band_field``)."""
    iterations = ops._check_int("iterations", smooth_iterations, 0, ops._INT32_MAX)
    budget = None if max_faces is None else ops._check_int("max_faces", max_faces, 1)
    want_normals = normals or colors
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
    if not normals:
        nrm = None
    if ply_filename is not None:
        write_ply(ply_filename, verts.cpu().numpy(), faces.cpu().numpy(), None if nrm is None else nrm.cpu().numpy(),
                  None if rgb is None else rgb.cpu().numpy())
    return verts, faces, nrm, rgb
