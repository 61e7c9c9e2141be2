"""Taubin lambda|mu smoothing and area-weighted mesh normals in numpy float32 (TEST INFRASTRUCTURE ONLY): what
``b2r_mesh_adjacency`` / ``_smooth`` / ``_normals`` (``csrc/mesh.cu``) compute on the device, with every operation rounded
separately and in the same order, so the GPU tests compare them bit for bit.

A corner of vertex v is a pair (f, c) with ``faces[f][c] == v``; v's corners are taken in ascending (f, c), and a face that lists
v twice gives it two corners.  Sums over corners accumulate slot by slot over the corner lists padded to the largest degree:
``np.sum`` would add them pairwise, in another order."""
from __future__ import annotations

import numpy as np

F32 = np.float32
LAMBDA = F32(0.5)
MU = F32(-0.53)


def _faces(faces, n_verts):
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    if f.size and (f.min() < 0 or f.max() >= n_verts):
        raise ValueError(f"face indices must lie in [0, {n_verts})")
    return f


def corners(faces, n_verts):
    """``(face, corner, valid)``, each [V, K] with K the largest corner count: slot j of row v is v's j-th corner in ascending
    (f, c) order where ``valid`` is set."""
    f = _faces(faces, n_verts)
    vert = f.reshape(-1)
    order = np.argsort(vert, kind="stable")                    # by vertex, then by corner id 3f + c: ascending (f, c)
    k = np.bincount(vert, minlength=n_verts)
    start = np.cumsum(k) - k
    width = int(k.max()) if len(k) and len(vert) else 0
    face = np.zeros((n_verts, width), np.int64)
    corner = np.zeros((n_verts, width), np.int64)
    valid = np.zeros((n_verts, width), bool)
    rows = vert[order]
    slots = np.arange(len(order)) - start[rows]
    face[rows, slots] = order // 3
    corner[rows, slots] = order % 3
    valid[rows, slots] = True
    return face, corner, valid


def _slots(faces, n_verts):
    """The corner lists as slots: vertices reordered by descending corner count (``order``), so the vertices that have a j-th
    corner are the first ``rows[j]`` of that order; ``a[j]`` / ``b[j]`` are the other two vertices of their j-th corner's face
    (faces[f][(c+1)%3], faces[f][(c+2)%3]) and ``face[j]`` its face.  ``k`` is the corner count per vertex."""
    f = _faces(faces, n_verts)
    face, corner, valid = corners(f, n_verts)
    k = valid.sum(1)
    order = np.argsort(-k, kind="stable")
    ks = k[order]
    rows = [int(np.count_nonzero(ks > j)) for j in range(face.shape[1])]
    fj = [face[order[:r], j] for j, r in enumerate(rows)]
    cj = [corner[order[:r], j] for j, r in enumerate(rows)]
    a = [f[x, (c + 1) % 3] for x, c in zip(fj, cj)]
    b = [f[x, (c + 2) % 3] for x, c in zip(fj, cj)]
    return order, rows, a, b, fj, k


def half_step(verts, faces, w, slots=None):
    """One umbrella half-step with weight ``w`` (Jacobi): for a vertex with k > 0 corners, s = 0, then for each corner (f, c)
    s = s + p[faces[f][(c+1)%3]] and s = s + p[faces[f][(c+2)%3]]; m = s / float32(2k); p' = p + w (m - p).  A vertex with no
    corners keeps its position."""
    p = np.asarray(verts, dtype=F32).reshape(-1, 3)
    order, rows, a, b, _, k = _slots(faces, len(p)) if slots is None else slots
    s = np.zeros_like(p)                                       # in ``order``
    for r, aj, bj in zip(rows, a, b):
        s[:r] = (s[:r] + p[aj]) + p[bj]
    out = p.copy()
    has = order[k[order] > 0]
    n = len(has)
    m = s[:n] / (2 * k[has]).astype(F32)[:, None]
    out[has] = p[has] + F32(w) * (m - p[has])
    return out


def smooth(verts, faces, iterations):
    """``iterations`` Taubin iterations: a half-step with lambda = float32(0.5), then one with mu = float32(-0.53)."""
    if int(iterations) < 0:
        raise ValueError("iterations must be >= 0")
    p = np.asarray(verts, dtype=F32).reshape(-1, 3)
    slots = _slots(faces, len(p))
    for _ in range(int(iterations)):
        p = half_step(half_step(p, faces, LAMBDA, slots), faces, MU, slots)
    return p


def mesh_normals(verts, faces):
    """Unit area-weighted vertex normals [V,3]: the sum over the vertex's corners, in order, of its face's e1 x e2 with
    e1 = p[f1] - p[f0], e2 = p[f2] - p[f0] in the face's own corner order (x = e1y e2z - e1z e2y, and cyclically), divided
    by sqrt((x x + y y) + z z); (0, 0, 0) when that length is 0."""
    p = np.asarray(verts, dtype=F32).reshape(-1, 3)
    f = _faces(faces, len(p))
    e1 = p[f[:, 1]] - p[f[:, 0]]
    e2 = p[f[:, 2]] - p[f[:, 0]]
    fn = np.stack([e1[:, (c + 1) % 3] * e2[:, (c + 2) % 3] - e1[:, (c + 2) % 3] * e2[:, (c + 1) % 3] for c in range(3)], 1)
    order, rows, _, _, fj, _ = _slots(f, len(p))
    acc = np.zeros_like(p)                                     # in ``order``
    for r, x in zip(rows, fj):
        acc[:r] = acc[:r] + fn[x]
    n = np.empty_like(p)
    n[order] = acc
    with np.errstate(divide="ignore", invalid="ignore", over="ignore", under="ignore"):
        length = np.sqrt((n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2]).astype(F32)
        out = np.where(length[:, None] > 0, n / length[:, None], F32(0)).astype(F32)
    return out
