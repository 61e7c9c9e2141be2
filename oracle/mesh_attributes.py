"""Numpy restatements of the mesh-export kernels (TEST INFRASTRUCTURE ONLY): the box-lattice MLP input rows (``load_row`` in
``csrc/common.cuh``) and the vertex normals of ``b2r_mc_normals`` (``csrc/mesh.cu``), both in float32 with every operation
rounded separately, so the GPU tests compare the kernels with them bit for bit.  The vertex order is that of
``oracle.marching_cubes.marching_cubes``."""
from __future__ import annotations

import numpy as np

F32 = np.float32


def lattice_points(dims, origin, voxel, begin=0, count=None):
    """Points [count,3] (float32) of lattice indices [begin, begin+count) of an n0 x n1 x n2 box lattice, axis 0 slowest:
    ``p_c = origin_c + idx_c * voxel``, a rounded float32 multiply, then a rounded add."""
    n0, n1, n2 = (int(d) for d in dims)
    count = n0 * n1 * n2 - begin if count is None else count
    idx = np.arange(begin, begin + count, dtype=np.int64)
    ijk = np.stack([idx // (n1 * n2), (idx // n2) % n1, idx % n2], 1).astype(F32)
    v = F32(voxel)
    return np.stack([F32(origin[c]) + ijk[:, c] * v for c in range(3)], 1).astype(F32)


def gradient(field):
    """[n0,n1,n2,3] float32 gradient at the lattice points: 0.5 (f[i+1] - f[i-1]) inside, f[1] - f[0] and f[-1] - f[-2] on the
    faces (np.gradient's scheme; the isotropic spacing is dropped)."""
    f = np.ascontiguousarray(field, dtype=F32)
    g = np.empty(f.shape + (3,), F32)
    for a in range(3):
        fa = np.moveaxis(f, a, 0)
        ga = np.moveaxis(g[..., a], a, 0)
        ga[1:-1] = F32(0.5) * (fa[2:] - fa[:-2])
        ga[0] = fa[1] - fa[0]
        ga[-1] = fa[-1] - fa[-2]
    return g


def vertex_normals(field, level):
    """Unit normals [V,3] (float32) of the vertices of ``marching_cubes(field, level)``, in its order.  The vertex on the edge
    p -> p + e_a with parameter t = (level - f(p)) / (f(p + e_a) - f(p)) gets n = g(p) + t (g(p + e_a) - g(p)), divided by
    sqrt((n_x^2 + n_y^2) + n_z^2); it points toward increasing field.  A zero length gives (0, 0, 0)."""
    f = np.ascontiguousarray(field, dtype=F32)
    assert f.ndim == 3 and min(f.shape) >= 2
    lv = F32(level)
    below = f < lv
    bits = np.zeros(f.shape, np.int64)
    bits[:-1, :, :] |= (below[:-1] != below[1:]).astype(np.int64)
    bits[:, :-1, :] |= (below[:, :-1] != below[:, 1:]).astype(np.int64) << 1
    bits[:, :, :-1] |= (below[:, :, :-1] != below[:, :, 1:]).astype(np.int64) << 2
    pi, pj, pk, ax = np.nonzero((bits[..., None] >> np.arange(3)) & 1)
    q = np.stack([pi, pj, pk], 1) + np.eye(3, dtype=np.int64)[ax]
    f0 = f[pi, pj, pk]
    f1 = f[q[:, 0], q[:, 1], q[:, 2]]
    g = gradient(f)
    g0 = g[pi, pj, pk]
    g1 = g[q[:, 0], q[:, 1], q[:, 2]]
    with np.errstate(divide="ignore", invalid="ignore", over="ignore", under="ignore"):
        t = ((lv - f0) / (f1 - f0)).astype(F32)
        n = (g0 + t[:, None] * (g1 - g0)).astype(F32)
        length = np.sqrt((n[:, 0] * n[:, 0] + n[:, 1] * n[:, 1]) + n[:, 2] * n[:, 2]).astype(F32)
        out = np.where(length[:, None] > 0, n / length[:, None], F32(0)).astype(F32)
    return out.reshape(-1, 3)
