"""Connected components of a triangle mesh in numpy + scipy (TEST INFRASTRUCTURE ONLY): the labels, triangle counts and
small-component removal that ``b2r_mesh_cc_label`` / ``_select`` / ``_compact`` (``csrc/mesh.cu``) compute on the device, so the
GPU tests compare them bit for bit.

Two vertices are connected when a face has them as (v0, v1) or (v1, v2).  The label of a vertex is the smallest vertex index of
its component, which does not depend on how the device schedules its union-find; a vertex no face uses is a component of its
own with 0 triangles."""
from __future__ import annotations

import math

import numpy as np
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components


def _faces(faces, n_verts):
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    if f.size and (f.min() < 0 or f.max() >= n_verts):
        raise ValueError(f"face indices must lie in [0, {n_verts})")
    return f


def component_labels(faces, n_verts):
    """int32 [V]: the smallest vertex index of each vertex's connected component."""
    n = int(n_verts)
    f = _faces(faces, n)
    if n == 0:
        return np.zeros(0, np.int32)
    rows = np.concatenate([f[:, 0], f[:, 1]])
    cols = np.concatenate([f[:, 1], f[:, 2]])
    graph = coo_matrix((np.ones(len(rows), np.int8), (rows, cols)), shape=(n, n)).tocsr()
    _, comp = connected_components(graph, directed=False)
    _, first = np.unique(comp, return_index=True)        # component ids 0..k-1 -> their first (smallest) vertex
    return first[comp].astype(np.int32)


def component_triangles(faces, labels):
    """int64 [V]: the number of triangles of each component at its label's index; 0 everywhere else."""
    labels = np.asarray(labels, dtype=np.int64)
    f = _faces(faces, len(labels))
    return np.bincount(labels[f[:, 0]], minlength=len(labels)).astype(np.int64)


def filter_components(verts, faces, ratio, normals=None):
    """``(verts, faces, normals | None)`` without the small components.  ``ratio`` must be finite and in [0, 1]; it is taken
    as float32, the precision of the C ABI.  0 returns the inputs unchanged.  Otherwise a component with t triangles is kept
    iff t >= 1 and t >= ratio * t_max in float64 (t_max: the largest component's count).  Kept vertices (with their normals)
    and kept faces keep their relative order; face indices are remapped through the exclusive prefix count of the kept
    vertices."""
    r = float(ratio)
    if not (math.isfinite(r) and 0.0 <= r <= 1.0):
        raise ValueError(f"ratio must be finite and in [0, 1], got {ratio}")
    r32 = np.float32(r)
    if r32 == 0:
        return verts, faces, normals
    v = np.asarray(verts, dtype=np.float32).reshape(-1, 3)
    f = _faces(faces, len(v))
    labels = component_labels(f, len(v))
    tri = component_triangles(f, labels)
    t = tri[labels]
    t_max = np.float64(tri.max()) if len(tri) else np.float64(0)
    keep = (t > 0) & (t.astype(np.float64) >= np.float64(r32) * t_max)
    new_index = np.cumsum(keep) - keep
    kept_faces = f[keep[f[:, 0]]] if len(f) else f
    out_f = new_index[kept_faces].astype(np.int32).reshape(-1, 3)
    out_n = None if normals is None else np.asarray(normals, dtype=np.float32).reshape(-1, 3)[keep]
    return v[keep], out_f, out_n
