"""Taubin smoothing without a GPU: the numpy oracle (oracle/mesh_smoothing.py) on hand-made meshes for its rules, on a planar
triangulation, on the marching-cubes mesh of a blurred ball (terracing against the true radius, shrinkage against plain
Laplacian smoothing) and on a sphere (mesh normals against analytic and field normals); the argument checks of the
b2r_mesh_adjacency / _smooth / _normals entry points and of ops.smooth_mesh, and the scratch size formula."""
import numpy as np
import pytest
import torch
from scipy.ndimage import gaussian_filter

from msra_practice_project_b200 import _lib, ops
from oracle import marching_cubes as mc
from oracle import mesh_attributes as ma
from oracle import mesh_smoothing as sm

F32 = np.float32


def test_zero_iterations_is_the_identity_and_isolated_vertices_stay():
    verts = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0.3, 0.3, 1], [5, 5, 5]], F32)
    faces = np.array([[0, 1, 3], [1, 2, 3], [2, 0, 3]], np.int32)
    assert np.array_equal(sm.smooth(verts, faces, 0), verts)
    for it in (1, 3):
        out = sm.smooth(verts, faces, it)
        assert np.array_equal(out[4], verts[4]) and not np.array_equal(out[:4], verts[:4])
    assert np.array_equal(sm.mesh_normals(verts, faces)[4], [0, 0, 0])
    with pytest.raises(ValueError):
        sm.smooth(verts, faces, -1)


def test_degenerate_faces_follow_the_corner_rule():
    # face 1 lists vertex 0 twice: vertex 0 has corners (0,0), (1,0), (1,2) -> a/b pairs (1,2), (0,3), (3,0)
    verts = np.array([[0, 0, 0], [4, 0, 0], [0, 8, 0], [2, 2, 6]], F32)
    faces = np.array([[0, 1, 2], [0, 0, 3]], np.int32)
    face, corner, valid = sm.corners(faces, 4)
    assert valid.sum(1).tolist() == [3, 1, 1, 1]
    assert face[0, :3].tolist() == [0, 1, 1] and corner[0, :3].tolist() == [0, 0, 1]
    p = verts
    s = ((((((F32(0) + p[1]) + p[2]) + p[0]) + p[3]) + p[3]) + p[0]).astype(F32)
    m = s / F32(6)
    want0 = p[0] + F32(0.5) * (m - p[0])
    out = sm.half_step(verts, faces, F32(0.5))
    assert np.array_equal(out[0], want0.astype(F32))
    # vertex 3 has one corner, (1, 2): a = faces[1][0] = 0, b = faces[1][1] = 0
    assert np.array_equal(out[3], (p[3] + F32(0.5) * (((p[0] + p[0]) / F32(2)) - p[3])).astype(F32))
    # the degenerate face has zero area: vertex 3's fan has none, vertex 0's normal is face 0's
    n = sm.mesh_normals(verts, faces)
    assert np.array_equal(n[3], [0, 0, 0]) and np.array_equal(n[0], [0, 0, 1])


def test_the_corner_order_is_pinned():
    # a closed fan of nine triangles whose corner sum in order differs from numpy's pairwise sum in float32
    rng = np.random.default_rng(0)
    for _ in range(200):
        vals = (rng.standard_normal(9) * 10.0 ** rng.integers(-4, 5, 9)).astype(F32)
        centre = np.zeros((1, 3), F32)
        ring = np.zeros((9, 3), F32)
        ring[:, 0] = vals
        verts = np.concatenate([centre, ring])
        faces = np.array([[0, 1 + i, 1 + (i + 1) % 9] for i in range(9)], np.int32)     # a closed fan: each ring vertex twice
        got = sm.half_step(verts, faces, F32(1.0))[0, 0]
        s = F32(0)
        for i in range(9):
            s = (s + vals[i]) + vals[(i + 1) % 9]
        assert got == s / F32(18)
        naive = np.sum(np.stack([vals, np.roll(vals, -1)], 1).reshape(-1)) / F32(18)
        if naive != got:
            return
    pytest.fail("no input separated the ordered sum from np.sum")


def test_planar_triangulation_stays_in_its_plane():
    n = 12
    i, j = np.meshgrid(np.arange(n), np.arange(n), indexing="ij")
    x, y = i.astype(F32) * F32(0.25), j.astype(F32) * F32(0.25)
    verts = np.stack([x, y, F32(0.5) * x + F32(0.25) * y + F32(1)], -1).reshape(-1, 3).astype(F32)
    idx = (i * n + j)[:-1, :-1].reshape(-1)
    faces = np.concatenate([np.stack([idx, idx + n, idx + 1], 1), np.stack([idx + 1, idx + n, idx + n + 1], 1)]).astype(np.int32)
    out = sm.smooth(verts, faces, 10)
    plane = out[:, 2] - (out[:, 0] * 0.5 + out[:, 1] * 0.25 + 1.0)
    assert np.abs(plane).max() < 1e-5
    # six symmetric neighbours: the mean is the vertex itself.  The open boundary is not pinned and its motion spreads one ring
    # per half-step, so after one iteration the vertices three rings in or deeper have not moved
    one = sm.smooth(verts, faces, 1)
    deep = ((i > 2) & (i < n - 3) & (j > 2) & (j < n - 3)).reshape(-1)
    assert np.abs(one[deep] - verts[deep]).max() < 1e-5
    assert np.abs(one[~deep] - verts[~deep]).max() > 1e-3
    normals = sm.mesh_normals(out, faces)
    want = np.array([-0.5, -0.25, 1.0]) / np.linalg.norm([-0.5, -0.25, 1.0])
    assert np.abs(normals - want).max() < 1e-4


def _ball(n=64, r=20.0, blur=0.4):
    c = (n - 1) / 2
    g = np.stack(np.meshgrid(*[np.arange(n, dtype=np.float64)] * 3, indexing="ij"), -1)
    inside = (np.linalg.norm(g - c, axis=-1) <= r).astype(np.float32)
    return gaussian_filter(inside, blur).astype(np.float32), c, r


def test_smoothing_reduces_terracing_without_shrinking():
    field, c, r = _ball()
    verts, faces = mc.marching_cubes(-field, -0.5)
    radius = lambda v: np.linalg.norm(v.astype(np.float64) - c, axis=1)          # noqa: E731
    rms = lambda v: float(np.sqrt(np.mean((radius(v) - r) ** 2)))                 # noqa: E731
    taubin = sm.smooth(verts, faces, 10)
    laplace = verts
    for _ in range(20):
        laplace = sm.half_step(laplace, faces, sm.LAMBDA)
    before, after = rms(verts), rms(taubin)
    shift_taubin = abs(radius(taubin).mean() - radius(verts).mean())
    shift_laplace = abs(radius(laplace).mean() - radius(verts).mean())
    print(f"ball r={r}: V {len(verts)}, rms {before:.4f} -> {after:.4f}; mean radius shift taubin {shift_taubin:.4f}, "
          f"laplace {shift_laplace:.4f}")
    assert after < 0.65 * before
    assert shift_taubin < 0.1 * shift_laplace


def test_sphere_mesh_normals():
    n, r = 48, 17.0
    c = (n - 1) / 2
    g = np.stack(np.meshgrid(*[np.arange(n, dtype=np.float64)] * 3, indexing="ij"), -1)
    field = (np.linalg.norm(g - c, axis=-1) - r).astype(np.float32)
    verts, faces = mc.marching_cubes(field, 0.0)
    mesh_n = sm.mesh_normals(verts, faces)
    field_n = ma.vertex_normals(field, 0.0)
    analytic = (verts - c) / np.linalg.norm(verts - c, axis=1, keepdims=True)
    lengths = np.linalg.norm(mesh_n, axis=1)
    has_area = lengths > 0
    assert has_area.mean() > 0.99 and np.allclose(lengths[has_area], 1.0, atol=1e-6)
    assert np.all(np.sum(mesh_n * field_n, 1)[has_area] > 0)
    assert np.percentile(np.sum(mesh_n * analytic, 1)[has_area], 1) > 0.98
    # smoothing keeps them pointing out
    sv = sm.smooth(verts, faces, 10)
    sn = sm.mesh_normals(sv, faces)
    assert np.all(np.sum(sn * field_n, 1)[np.linalg.norm(sn, axis=1) > 0] > 0)


def _align256(b):
    return (b + 255) & ~255


@pytest.mark.parametrize("nv,nf", [(0, 0), (1, 0), (0, 5), (2048, 2049), (75_000_000, 151_000_000), (2 ** 31 - 1, 2 ** 31 - 1)])
def test_scratch_bytes_formula(nv, nf):
    tiles = -(-nv // 2048)
    want = _align256(8 * nv) + _align256(8 * tiles) + _align256(24 * nf) + _align256(12 * nv)
    assert _lib.lib().b2r_mesh_adj_scratch_bytes(nv, nf) == want


def test_scratch_bytes_out_of_range_is_zero():
    lib = _lib.lib()
    for nv, nf in ((-1, 0), (0, -1), (2 ** 31, 0), (0, 2 ** 31)):
        assert lib.b2r_mesh_adj_scratch_bytes(nv, nf) == 0


def test_abi_argument_checks():
    lib = _lib.lib()
    F, S, T = 256, 512, 768          # stand-in device addresses; every call below fails its checks before touching them

    def fails(rc, text):
        return rc < 0 and text.encode() in lib.b2r_last_error()

    # adjacency(faces, n_faces, n_verts, scratch, stream)
    assert fails(lib.b2r_mesh_adjacency(F, -1, 4, S, None), "n_faces")
    assert fails(lib.b2r_mesh_adjacency(F, 1, 2 ** 31, S, None), "n_verts")
    assert fails(lib.b2r_mesh_adjacency(None, 1, 4, S, None), "NULL faces")
    assert fails(lib.b2r_mesh_adjacency(F, 1, 4, None, None), "NULL scratch")
    assert fails(lib.b2r_mesh_adjacency(F, 1, 4, S + 8, None), "16-byte aligned")
    assert lib.b2r_mesh_adjacency(None, 0, 0, S, None) == 0            # nothing to build: no launch
    assert lib.b2r_mesh_adjacency(None, 0, 0, None, None) == 0         # an empty mesh's scratch has 0 bytes
    # smooth(verts, n_faces, n_verts, iterations, scratch, verts_out, stream)
    assert fails(lib.b2r_mesh_smooth(T, 2 ** 31, 4, 1, S, T, None), "n_faces")
    assert fails(lib.b2r_mesh_smooth(T, 1, -4, 1, S, T, None), "n_verts")
    assert fails(lib.b2r_mesh_smooth(None, 1, 4, 1, S, T, None), "NULL verts")
    assert fails(lib.b2r_mesh_smooth(T, 1, 4, 1, S, None, None), "NULL verts")
    assert fails(lib.b2r_mesh_smooth(T, 1, 4, -1, S, T, None), "iterations")
    assert fails(lib.b2r_mesh_smooth(T, 1, 4, 1, None, T, None), "NULL scratch")
    assert fails(lib.b2r_mesh_smooth(T, 1, 4, 1, S + 4, T, None), "16-byte aligned")
    assert lib.b2r_mesh_smooth(None, 0, 0, 3, None, None, None) == 0
    assert lib.b2r_mesh_normals(None, 5, 0, None, None, None) == 0
    # normals(verts, n_faces, n_verts, scratch, normals, stream)
    assert fails(lib.b2r_mesh_normals(T, -1, 4, S, T, None), "n_faces")
    assert fails(lib.b2r_mesh_normals(T, 1, 4, S, None, None), "NULL verts")
    assert fails(lib.b2r_mesh_normals(None, 1, 4, S, T, None), "NULL verts")
    assert fails(lib.b2r_mesh_normals(T, 1, 4, None, T, None), "NULL scratch")
    assert fails(lib.b2r_mesh_normals(T, 1, 4, S + 12, T, None), "16-byte aligned")
    with pytest.raises(RuntimeError, match="iterations"):
        _lib.check(lib.b2r_mesh_smooth(T, 1, 4, -2, S, T, None), "b2r_mesh_smooth")


@pytest.mark.parametrize("bad", [-1, 1.0, 2.5, "3", None, True, 2 ** 31])
def test_ops_rejects_bad_iterations(bad):
    verts, faces = torch.zeros(3, 3), torch.tensor([[0, 1, 2]], dtype=torch.int32)
    with pytest.raises(ValueError):
        ops.smooth_mesh(verts, faces, bad)


def test_ops_zero_iterations_and_host_tensors():
    verts, faces = torch.zeros(3, 3), torch.tensor([[0, 1, 2]], dtype=torch.int32)
    assert ops.smooth_mesh(verts, faces, 0) is verts
    assert ops.smooth_mesh(verts, faces, np.int64(0)) is verts
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.smooth_mesh(verts, faces, 0, normals=True)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.smooth_mesh(verts, faces, 2)
