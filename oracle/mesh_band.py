"""Numpy definition of the narrow-band mesh export (TEST INFRASTRUCTURE ONLY): the brick flags and needed points of
``b2r_band_select`` and the mesh of ``b2r_mc_count_band`` (``csrc/mesh.cu``), so the GPU tests compare the kernels with them
exactly.

Bricks of ``stride`` cells per axis: an axis of n points has ``ceil((n - 1) / stride)`` bricks; brick b covers the cells
``[b stride, min((b + 1) stride, n - 1))``, its closure the points ``[b stride, min((b + 1) stride, n - 1)]`` and its coarse
corners are the points ``min(b stride, n - 1)`` and ``min((b + 1) stride, n - 1)``.  As in ``oracle.marching_cubes``, a point is
below when ``field < level`` (NaN is not below)."""
from __future__ import annotations

import itertools

import numpy as np

from oracle import marching_cubes as mc
from oracle import mesh_attributes as ma

F32 = np.float32


def brick_dims(shape, stride):
    return tuple((int(n) - 2) // int(stride) + 1 for n in shape)


def coarse_axes(shape, stride):
    """Per axis, the coordinates of the coarse corners: ``min(b stride, n - 1)`` for b = 0 .. nb."""
    return [np.minimum(np.arange(nb + 1) * int(stride), int(n) - 1) for n, nb in zip(shape, brick_dims(shape, stride))]


def coarse_points(shape, stride):
    """Linear indices (int64, ascending) of every coarse corner."""
    a0, a1, a2 = coarse_axes(shape, stride)
    return ((a0[:, None, None] * shape[1] + a1[None, :, None]) * shape[2] + a2[None, None, :]).ravel()


def raw_flags(field, level, stride):
    """bool [nb0,nb1,nb2]: the brick's 8 coarse corners are not all on the same side of the level."""
    f = np.asarray(field, dtype=F32)
    below = (f[np.ix_(*coarse_axes(f.shape, stride))] < F32(level)).astype(np.int64)
    count = sum(below[o0:below.shape[0] - 1 + o0, o1:below.shape[1] - 1 + o1, o2:below.shape[2] - 1 + o2]
                for o0, o1, o2 in itertools.product((0, 1), repeat=3))
    return (count > 0) & (count < 8)


def dilate(raw):
    """uint8 flags: any raw flag in the 26-neighbourhood (the brick itself included), clamped at the box."""
    p = np.pad(np.asarray(raw, bool), 1)
    n0, n1, n2 = raw.shape
    out = np.zeros(raw.shape, bool)
    for o0, o1, o2 in itertools.product((0, 1, 2), repeat=3):
        out |= p[o0:o0 + n0, o1:o1 + n1, o2:o2 + n2]
    return out.astype(np.uint8)


def brick_flags(field, level, stride):
    """The flags of ``b2r_band_select``: the raw flags of the coarse corners, dilated by one brick."""
    return dilate(raw_flags(field, level, stride))


def band_points(flags, shape, stride):
    """int32 linear indices, ascending, of every point of the closure of a flagged brick and every point one step along one
    axis from such a point."""
    closure = np.zeros(tuple(shape), bool)
    for b in zip(*np.nonzero(flags)):
        lo = [bb * stride for bb in b]
        hi = [min((bb + 1) * stride, n - 1) for bb, n in zip(b, shape)]
        closure[lo[0]:hi[0] + 1, lo[1]:hi[1] + 1, lo[2]:hi[2] + 1] = True
    need = closure.copy()
    for a in range(3):
        c = np.moveaxis(closure, a, 0)
        nd = np.moveaxis(need, a, 0)
        nd[1:] |= c[:-1]
        nd[:-1] |= c[1:]
    return np.flatnonzero(need).astype(np.int32)


def band_field(field, level, stride):
    """Steps 2-5 of the narrow-band query on a known field: +inf everywhere, the field at the coarse corners, the flags, then
    the field at the band points.  Returns (band field, flags)."""
    f = np.asarray(field, dtype=F32)
    out = np.full(f.shape, np.inf, F32)
    c = coarse_points(f.shape, stride)
    out.flat[c] = f.flat[c]
    flags = brick_flags(out, level, stride)
    idx = band_points(flags, f.shape, stride)
    out.flat[idx] = f.flat[idx]
    return out, flags


def _cell_flags(shape, flags, stride):
    """bool [n0-1,n1-1,n2-1]: the cell lies in a flagged brick."""
    i, j, k = (np.arange(n - 1) // stride for n in shape)
    return np.asarray(flags, bool)[np.ix_(i, j, k)]


def masked_marching_cubes(field, level, stride, flags, spacing=1.0, origin=(0.0, 0.0, 0.0), normals=False):
    """``oracle.marching_cubes.marching_cubes`` less the faces of cells outside flagged bricks and the vertices on no crossing
    edge of a cell in a flagged brick, both in their dense order, faces remapped (with ``normals``: the vertex normals of
    ``oracle.mesh_attributes.vertex_normals``, filtered alike, as a third array)."""
    f = np.ascontiguousarray(field, dtype=F32)
    verts, faces = mc.marching_cubes(f, level, spacing, origin)
    nrm = ma.vertex_normals(f, level) if normals else None
    n0, n1, n2 = f.shape
    cells = _cell_flags(f.shape, flags, stride)
    # the cell of every dense face: cells in linear order, each repeated by its triangle count (the oracle's face order)
    below = (f < F32(level)).astype(np.int64)
    config = np.zeros(cells.shape, np.int64)
    for c in range(8):
        o0, o1, o2 = mc.corner_offset(c)
        config |= below[o0:n0 - 1 + o0, o1:n1 - 1 + o1, o2:n2 - 1 + o2] << c
    ntri = np.array([len(t) for t in mc.TRIANGLES])[config].ravel()
    keep_face = np.repeat(cells.ravel(), ntri)
    # a vertex (p, a) is kept when a cell holding the edge p -> p + e_a lies in a flagged brick: that cell's axis-a
    # coordinate is p_a, and on the other axes it is p_b - 1 or p_b
    pad = np.zeros((n0 + 1, n1 + 1, n2 + 1), bool)
    pad[1:n0, 1:n1, 1:n2] = cells
    edge = np.zeros(f.shape + (3,), bool)
    for a in range(3):
        for d in itertools.product((0, 1), repeat=2):
            s = list(d)
            s.insert(a, 1)
            edge[..., a] |= pad[s[0]:s[0] + n0, s[1]:s[1] + n1, s[2]:s[2] + n2]
    with np.errstate(invalid="ignore"):
        lv = F32(level)
        bl = f < lv
    bits = np.zeros(f.shape + (3,), bool)
    bits[:-1, :, :, 0] = bl[:-1] != bl[1:]
    bits[:, :-1, :, 1] = bl[:, :-1] != bl[:, 1:]
    bits[:, :, :-1, 2] = bl[:, :, :-1] != bl[:, :, 1:]
    keep_vert = edge[bits]                                 # dense vertex order: (point, axis) of every crossing edge
    assert len(keep_vert) == len(verts) and len(keep_face) == len(faces)
    remap = np.cumsum(keep_vert) - 1
    kept_faces = faces[keep_face]
    assert keep_vert[kept_faces].all(), "a kept face uses a removed vertex"
    out = (verts[keep_vert], remap[kept_faces].astype(np.int32))
    return out + (nrm[keep_vert],) if normals else out
