"""Marching cubes without a GPU: the checked-in triangle table against its generator, the table's per-configuration
properties, the numpy oracle's meshes of analytic fields (closed, consistently oriented, right topology and volume), and the
argument checks / scratch sizes of the C ABI."""
import ctypes as C

import numpy as np
import pytest

from msra_practice_project_b200 import _lib
from oracle import marching_cubes as mc


def test_checked_in_table_is_the_generators_output():
    with open(mc.HEADER) as fh:
        assert fh.read() == mc.header_text(), "run `python -m oracle.marching_cubes`"


def test_table_uses_exactly_the_crossing_edges():
    for config, tris in enumerate(mc.TRIANGLES):
        below = [(config >> c) & 1 for c in range(8)]
        crossing = {e for e, (a, b) in enumerate(mc.EDGES) if below[a] != below[b]}
        assert {e for t in tris for e in t} == crossing, config
        assert len(tris) <= 5
    assert mc.TRIANGLES[0] == [] and mc.TRIANGLES[255] == []
    assert np.bincount([len(t) for t in mc.TRIANGLES]).tolist() == [2, 16, 50, 80, 76, 32]


def test_packed_table_round_trips():
    for config, w in enumerate(mc.packed_table()):
        n = w >> 60
        edges = [(w >> (4 * m)) & 15 for m in range(3 * n)]
        assert [tuple(edges[3 * i:3 * i + 3]) for i in range(n)] == mc.TRIANGLES[config]


def _mesh_stats(verts, faces):
    """(closed, oriented, Euler characteristic, signed volume)."""
    e = np.concatenate([faces[:, [0, 1]], faces[:, [1, 2]], faces[:, [2, 0]]]).astype(np.int64)
    _, undirected = np.unique(np.sort(e, 1), axis=0, return_counts=True)
    _, directed = np.unique(e, axis=0, return_counts=True)
    v = verts.astype(np.float64)
    vol = np.einsum("ij,ij->i", v[faces[:, 0]], np.cross(v[faces[:, 1]], v[faces[:, 2]])).sum() / 6
    euler = len(np.unique(faces)) - len(undirected) + len(faces)
    return bool((undirected == 2).all()), bool((directed == 1).all()), euler, vol


def _grid(n):
    x = np.linspace(-1, 1, n, dtype=np.float32)
    return np.meshgrid(x, x, x, indexing="ij"), np.float32(2 / (n - 1))


def test_oracle_sphere():
    (x, y, z), sp = _grid(40)
    r = 0.7
    verts, faces = mc.marching_cubes(np.sqrt(x * x + y * y + z * z) - r, 0.0, sp, (-1, -1, -1))
    closed, oriented, euler, vol = _mesh_stats(verts, faces)
    assert closed and oriented and euler == 2
    exact = 4 / 3 * np.pi * r ** 3
    assert 0 < vol and abs(vol - exact) < 0.02 * exact
    assert np.abs(np.linalg.norm(verts, axis=1) - r).max() < 1e-3
    assert verts.dtype == np.float32 and faces.dtype == np.int32


def test_oracle_torus():
    (x, y, z), sp = _grid(40)
    big, small = 0.6, 0.25
    verts, faces = mc.marching_cubes(np.sqrt((np.sqrt(x * x + y * y) - big) ** 2 + z * z) - small, 0.0, sp, (-1, -1, -1))
    closed, oriented, euler, vol = _mesh_stats(verts, faces)
    assert closed and oriented and euler == 0
    exact = 2 * np.pi ** 2 * big * small ** 2
    assert 0 < vol and abs(vol - exact) < 0.02 * exact


def test_oracle_two_spheres():
    (x, y, z), sp = _grid(40)
    f = np.minimum(np.sqrt((x - 0.5) ** 2 + y * y + z * z), np.sqrt((x + 0.5) ** 2 + y * y + z * z)) - 0.3
    closed, oriented, euler, vol = _mesh_stats(*mc.marching_cubes(f, 0.0, sp, (-1, -1, -1)))
    assert closed and oriented and euler == 4 and vol > 0


def test_oracle_padded_random_field_closed_and_oriented():
    """Ambiguous faces everywhere: the neighbours' choices must agree for the mesh to close."""
    f = np.full((14, 15, 13), 5.0, np.float32)
    f[1:-1, 1:-1, 1:-1] = np.random.default_rng(0).standard_normal((12, 13, 11))
    verts, faces = mc.marching_cubes(f, 0.0)
    closed, oriented, _, vol = _mesh_stats(verts, faces)
    assert len(faces) > 1000 and closed and oriented and vol > 0


def test_oracle_output_order_and_vertex_formula():
    """Vertices by owner point then axis, each on its lattice edge at t = (level - f(p)) / (f(p+e_a) - f(p))."""
    f = np.array([[[0.0, 1.0], [0.0, 0.0]], [[0.0, 0.0], [0.0, 0.0]]], np.float32)
    verts, faces = mc.marching_cubes(f, 0.25, 2.0, (1.0, 2.0, 3.0))
    # only point (0,0,1) is above: its three edges are owned by (0,0,0) (axis 2, t = 0.25) and by (0,0,1) itself (axis 0, then
    # axis 1, t = 0.75)
    np.testing.assert_array_equal(verts, np.array([[1, 2, 3 + 2 * 0.25], [1 + 2 * 0.75, 2, 5], [1, 2 + 2 * 0.75, 5]], np.float32))
    assert faces.shape == (1, 3) and sorted(faces[0].tolist()) == [0, 1, 2]


def test_abi_scratch_bytes_and_argument_checks():
    lib = _lib.lib()
    assert lib.b2r_mc_scratch_bytes(2, 2, 2) == 3 * 256
    assert lib.b2r_mc_scratch_bytes(512, 512, 512) == 2 ** 29 + 65536 * 4 + 65536 * 16
    assert lib.b2r_mc_scratch_bytes(1, 4, 4) == 0 and lib.b2r_mc_scratch_bytes(4, 4, 0) == 0
    assert lib.b2r_mc_scratch_bytes(2048, 1024, 1024) == 0
    totals = (C.c_longlong * 2)()
    fake = 256      # never dereferenced: every call below is rejected before any launch
    for call in (lambda *dims: lib.b2r_mc_count(fake, *dims, 0.0, fake, C.addressof(totals), None),
                 lambda *dims: lib.b2r_mc_emit(fake, *dims, 0.0, 1.0, 0.0, 0.0, 0.0, fake, fake, fake, None)):
        assert call(1, 4, 4) < 0 and b"n >= 2" in lib.b2r_last_error()
        assert call(4, 4, 1) < 0 and b"n >= 2" in lib.b2r_last_error()
        assert call(2048, 1024, 1024) < 0 and b"INT32_MAX" in lib.b2r_last_error()
    assert lib.b2r_mc_count(None, 4, 4, 4, 0.0, fake, C.addressof(totals), None) < 0 and b"NULL" in lib.b2r_last_error()
    assert lib.b2r_mc_count(fake, 4, 4, 4, 0.0, None, C.addressof(totals), None) < 0 and b"NULL" in lib.b2r_last_error()
    assert lib.b2r_mc_count(fake, 4, 4, 4, 0.0, fake, None, None) < 0 and b"NULL" in lib.b2r_last_error()
    assert lib.b2r_mc_count(fake, 4, 4, 4, 0.0, fake + 4, C.addressof(totals), None) < 0 and b"aligned" in lib.b2r_last_error()
    for i in range(4):
        args = [fake, fake, fake, fake]
        args[i] = None
        assert lib.b2r_mc_emit(args[0], 4, 4, 4, 0.0, 1.0, 0.0, 0.0, 0.0, args[1], args[2], args[3], None) < 0
        assert b"NULL" in lib.b2r_last_error()
    with pytest.raises(RuntimeError):
        _lib.check(lib.b2r_mc_count(None, 4, 4, 4, 0.0, None, None, None), "b2r_mc_count")


def test_ops_marching_cubes_rejects_host_tensors():
    import torch
    from msra_practice_project_b200 import ops
    with pytest.raises(RuntimeError):
        ops.marching_cubes(torch.zeros(4, 4, 4), 0.0)
