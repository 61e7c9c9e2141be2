"""Per-face texture atlas of a triangle mesh in numpy (TEST INFRASTRUCTURE ONLY): the layout, texel ownership, UVs and MLP rows
that ``b2r_mesh_atlas_uvs`` / ``_rows`` / ``_texture`` (``csrc/mesh.cu``) compute on the device, with every float32 operation
rounded separately and in the same order, so the GPU tests compare them bit for bit.

Layout, a pure function of the face count F and the texture size R: faces 2k ("A") and 2k+1 ("B") share cell k.  The
P = ceil(F / 2) cells sit C per row, C the smallest integer with C * C >= P, each s = R // C texels square, with top-left texel
(X, Y) = ((k % C) s, (k // C) s) (column, row; row 0 is the top of the image).  With L = s - 3, A's corners 0, 1, 2 sit at the
local texel centres (0, 0), (L, 0), (0, L) and B's, A reflected through the cell centre, at (s-1, s-1), (2, s-1), (s-1, 2).  A
local texel (x, y) is baked for B when x + y >= s and B exists, for A otherwise.  A's hypotenuse x + y = L = s - 3 makes a
bilinear lookup read texel sums up to s - 2, and B's, x + y = s + 1, sums from s up, so a lookup inside a face's UV triangle reads
only texels baked for that face and no dilation is needed."""
from __future__ import annotations

import math

import numpy as np

F32 = np.float32


def layout(n_faces, size):
    """``(cells, per_row, s)``; ValueError unless 16 <= size <= 16384 and n_faces <= 2 * (size // 4)^2 (s >= 4)."""
    n_faces, size = int(n_faces), int(size)
    if not 16 <= size <= 16384:
        raise ValueError(f"size must be in [16, 16384], got {size}")
    if not 0 <= n_faces <= 2 * (size // 4) ** 2:
        raise ValueError(f"{n_faces} faces do not fit a {size}^2 atlas (at most {2 * (size // 4) ** 2})")
    cells = (n_faces + 1) // 2
    per_row = math.isqrt(cells - 1) + 1 if cells else 0
    return cells, per_row, size // per_row if per_row else 0


def texels(n_faces, size):
    """Per atlas row r = k s^2 + y s + x (k < cells): ``(col, row, face, w [rows,3] float32)``, the texel's image column and row,
    the face it is baked for and its barycentric weights on that face's corners 0, 1, 2."""
    cells, per_row, s = layout(n_faces, size)
    if not cells:
        e = np.zeros(0, np.int64)
        return e, e, e, np.zeros((0, 3), F32)
    r = np.arange(cells * s * s, dtype=np.int64)
    k, t = r // (s * s), r % (s * s)
    x, y = t % s, t // s
    b_face = (x + y >= s) & (2 * k + 1 < n_faces)
    a = np.where(b_face, s - 1 - x, x)
    b = np.where(b_face, s - 1 - y, y)
    inside = a + b <= s - 3
    l_f = F32(s - 3)
    ab = np.maximum(a + b, 1).astype(F32)                       # a + b >= 1 wherever it is used
    w = np.empty((len(r), 3), F32)
    w[:, 0] = np.where(inside, (s - 3 - a - b).astype(F32) / l_f, F32(0))
    w[:, 1] = np.where(inside, a.astype(F32) / l_f, a.astype(F32) / ab)
    w[:, 2] = np.where(inside, b.astype(F32) / l_f, b.astype(F32) / ab)
    return (k % per_row) * s + x, (k // per_row) * s + y, 2 * k + b_face, w


def uvs(n_faces, size):
    """float32 [F,3,2]: corner (x, y) of cell (X, Y) at u = ((X+x) + 0.5) / R, v = 1 - ((Y+y) + 0.5) / R."""
    cells, per_row, s = layout(n_faces, size)
    f = np.arange(n_faces, dtype=np.int64)
    k, odd = f // 2, (f & 1).astype(bool)
    lx, ly = np.array([0, s - 3, 0]), np.array([0, 0, s - 3])
    x = np.where(odd[:, None], s - 1 - lx, lx)
    y = np.where(odd[:, None], s - 1 - ly, ly)
    per_row = max(per_row, 1)                                   # F = 0: no faces to place
    cx, cy = ((k % per_row) * s)[:, None], ((k // per_row) * s)[:, None]
    r = F32(size)
    out = np.empty((n_faces, 3, 2), F32)
    out[..., 0] = ((cx + x).astype(F32) + F32(0.5)) / r
    out[..., 1] = F32(1) - ((cy + y).astype(F32) + F32(0.5)) / r
    return out


def rows(verts, faces, normals, size):
    """x rows [cells s^2, 6] = [p, -n^]: p = (w0 v0 + w1 v1) + w2 v2 per component of the texel's face, n^ the same sum of the
    vertex normals divided by sqrt((x x + y y) + z z), or (0, 0, 0) where that is 0."""
    v = np.asarray(verts, F32).reshape(-1, 3)
    n = np.asarray(normals, F32).reshape(-1, 3)
    f = np.asarray(faces, np.int64).reshape(-1, 3)
    _, _, face, w = texels(len(f), size)
    idx = f[face]
    p = (w[:, 0:1] * v[idx[:, 0]] + w[:, 1:2] * v[idx[:, 1]]) + w[:, 2:3] * v[idx[:, 2]]
    m = (w[:, 0:1] * n[idx[:, 0]] + w[:, 1:2] * n[idx[:, 1]]) + w[:, 2:3] * n[idx[:, 2]]
    length = np.sqrt((m[:, 0] * m[:, 0] + m[:, 1] * m[:, 1]) + m[:, 2] * m[:, 2])
    safe = np.where(length > 0, length, F32(1))[:, None]
    nh = np.where((length > 0)[:, None], m / safe, F32(0))
    return np.concatenate([p, -nh], 1).astype(F32)


def texture(rgb8, n_faces, size):
    """uint8 [R,R,3]: row r's colour ``rgb8[r]`` in its texel, 0 elsewhere."""
    col, row, _, _ = texels(n_faces, size)
    out = np.zeros((int(size), int(size), 3), np.uint8)
    out[row, col] = np.asarray(rgb8, np.uint8).reshape(-1, 3)
    return out


def to8b(x):
    """b2r_to8b: (uint8)(255 * clip(x, 0, 1)), float32 product, truncation."""
    return (F32(255) * np.clip(np.asarray(x, F32), F32(0), F32(1))).astype(np.uint8)
