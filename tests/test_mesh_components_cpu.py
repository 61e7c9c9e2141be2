"""Connected components of meshes without a GPU: the numpy/scipy oracle (oracle/mesh_components.py) on analytic fields -- spheres
and a torus whose level sets are separate pieces -- and on hand-made meshes for its rules, the argument checks of the
b2r_mesh_cc_* entry points and of ops.mesh_components / ops.filter_components, and the scratch size formula."""
import ctypes as C

import numpy as np
import pytest
import torch

from msra_practice_project_b200 import _lib, ops
from oracle import marching_cubes as mc
from oracle import mesh_attributes as ma
from oracle import mesh_components as cc

N = 64
_P = np.stack(np.meshgrid(*[np.arange(N, dtype=np.float64)] * 3, indexing="ij"), -1)


def _sphere(c, r):
    return (np.linalg.norm(_P - np.array(c, np.float64), axis=-1) - r).astype(np.float32)


def _torus(c, big, small):
    d = _P - np.array(c, np.float64)
    return (np.sqrt((np.hypot(d[..., 0], d[..., 1]) - big) ** 2 + d[..., 2] ** 2) - small).astype(np.float32)


# signed distances in voxels, level 0; every two surfaces at least 7 voxels apart, so the union min(...) equals each shape's own
# field within 2 voxels of its surface: the crossing edges and the gradient stencils of its normals see only that shape
BIG = _sphere((20, 32, 32), 14.0)
TORUS = _torus((48, 20, 32), 7.0, 2.5)
SMALL = [_sphere((50, 48, 20), 3.0), _sphere((50, 48, 44), 2.0), _sphere((10, 56, 56), 2.5)]


def _union(*fields):
    out = fields[0]
    for f in fields[1:]:
        out = np.minimum(out, f)
    return out


def _mesh(field):
    v, f = mc.marching_cubes(field, 0.0)
    return v, f, ma.vertex_normals(field, 0.0)


def test_components_of_separate_shapes():
    v, f, _ = _mesh(_union(BIG, TORUS, *SMALL))
    labels = cc.component_labels(f, len(v))
    tri = cc.component_triangles(f, labels)
    assert labels.dtype == np.int32 and tri.dtype == np.int64 and len(labels) == len(tri) == len(v)
    roots = np.flatnonzero(tri)
    assert len(np.unique(labels)) == len(roots) == 5
    assert np.array_equal(labels[roots], roots) and np.all(labels <= np.arange(len(v)))      # a label is its component's minimum
    expected = sorted(len(_mesh(s)[1]) for s in (BIG, TORUS, *SMALL))
    assert sorted(tri[roots].tolist()) == expected and tri.sum() == len(f)
    # every face lies in one component
    assert np.all(labels[f[:, 0]] == labels[f[:, 1]]) and np.all(labels[f[:, 1]] == labels[f[:, 2]])


@pytest.mark.parametrize("with_normals", [False, True])
def test_filter_equals_the_kept_shapes_alone(with_normals):
    v, f, n = _mesh(_union(BIG, TORUS, *SMALL))
    t_big, t_torus = len(_mesh(BIG)[1]), len(_mesh(TORUS)[1])
    assert t_torus < 0.5 * t_big and all(len(_mesh(s)[1]) < 0.5 * t_torus for s in SMALL)
    for ratio, kept in ((0.5, (BIG,)), (0.5 * t_torus / t_big, (BIG, TORUS)), (1.0, (BIG,))):
        rv, rf, rn = _mesh(_union(*kept))
        gv, gf, gn = cc.filter_components(v, f, ratio, n if with_normals else None)
        assert np.array_equal(gv, rv) and np.array_equal(gf, rf) and gf.dtype == np.int32
        assert (gn is None) if not with_normals else np.array_equal(gn, rn)


def test_ratio_zero_is_the_identity():
    v, f, n = _mesh(_union(BIG, *SMALL))
    out = cc.filter_components(v, f, 0.0, n)
    assert out[0] is v and out[1] is f and out[2] is n
    assert cc.filter_components(v, f, 1e-50)[0] is v          # rounds to float32 0


def test_ratio_one_keeps_ties():
    # two spheres that differ by an integer translation have identical meshes; the smaller one goes
    a, b = _sphere((16, 16, 16), 9.0), _sphere((44, 44, 44), 9.0)
    v, f, _ = _mesh(_union(a, b, _sphere((16, 48, 48), 4.0)))
    gv, gf, _ = cc.filter_components(v, f, 1.0)
    rv, rf, _ = _mesh(_union(a, b))
    assert np.array_equal(gv, rv) and np.array_equal(gf, rf)
    # by hand: two components of 2 triangles, one of 1
    verts = np.arange(33, dtype=np.float32).reshape(11, 3)
    faces = np.array([[0, 1, 2], [2, 1, 3], [4, 5, 6], [7, 8, 9], [9, 8, 10]], np.int32)
    gv, gf, _ = cc.filter_components(verts, faces, 1.0)
    assert np.array_equal(gv, verts[[0, 1, 2, 3, 7, 8, 9, 10]])
    assert np.array_equal(gf, [[0, 1, 2], [2, 1, 3], [4, 5, 6], [6, 5, 7]])
    gv, gf, _ = cc.filter_components(verts, faces, 0.5)
    assert np.array_equal(gv, verts) and np.array_equal(gf, faces)


def test_labels_by_hand_and_unused_vertices():
    faces = np.array([[3, 1, 2], [6, 4, 5], [2, 7, 3]], np.int32)
    assert cc.component_labels(faces, 9).tolist() == [0, 1, 1, 1, 4, 4, 4, 1, 8]
    tri = cc.component_triangles(faces, cc.component_labels(faces, 9))
    assert tri.tolist() == [0, 2, 0, 0, 1, 0, 0, 0, 0]
    verts = np.arange(27, dtype=np.float32).reshape(9, 3)
    normals = -verts
    gv, gf, gn = cc.filter_components(verts, faces, 1e-6, normals)        # any ratio > 0 drops the unused vertices 0 and 8
    assert np.array_equal(gv, verts[1:8]) and np.array_equal(gn, normals[1:8])
    assert np.array_equal(gf, faces - 1)
    gv, gf, _ = cc.filter_components(verts, faces, 1.0)
    assert np.array_equal(gv, verts[[1, 2, 3, 7]]) and np.array_equal(gf, [[2, 0, 1], [1, 3, 2]])


def test_empty_meshes():
    v0, f0 = np.zeros((0, 3), np.float32), np.zeros((0, 3), np.int32)
    assert cc.component_labels(f0, 0).shape == (0,)
    gv, gf, gn = cc.filter_components(v0, f0, 0.3, v0)
    assert gv.shape == (0, 3) and gf.shape == (0, 3) and gn.shape == (0, 3)
    v = np.ones((4, 3), np.float32)
    assert cc.component_labels(f0, 4).tolist() == [0, 1, 2, 3]
    gv, gf, _ = cc.filter_components(v, f0, 0.3)           # no component has a triangle
    assert gv.shape == (0, 3) and gf.shape == (0, 3)


@pytest.mark.parametrize("ratio", [float("nan"), float("inf"), -0.1, 1.0001])
def test_bad_ratios_raise(ratio):
    v, f = np.zeros((3, 3), np.float32), np.array([[0, 1, 2]], np.int32)
    with pytest.raises(ValueError):
        cc.filter_components(v, f, ratio)
    with pytest.raises(ValueError):
        ops.filter_components(torch.zeros(3, 3), torch.tensor([[0, 1, 2]], dtype=torch.int32), ratio)


def test_ops_rejects_host_tensors_before_any_launch():
    faces = torch.tensor([[0, 1, 2]], dtype=torch.int32)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.mesh_components(faces, 3)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.filter_components(torch.zeros(3, 3), faces, 0.5)


def _align256(b):
    return (b + 255) & ~255


@pytest.mark.parametrize("nv,nf", [(0, 0), (1, 0), (0, 5), (2048, 2049), (75_000_000, 151_000_000), (2 ** 31 - 1, 2 ** 31 - 1)])
def test_scratch_bytes_formula(nv, nf):
    tiles = -(-max(nv, nf) // 2048)
    want = 2 * _align256(4 * nv) + _align256(4 * tiles) + _align256(16 * tiles) + 256
    assert _lib.lib().b2r_mesh_cc_scratch_bytes(nv, nf) == want


def test_scratch_bytes_out_of_range_is_zero():
    lib = _lib.lib()
    for nv, nf in ((-1, 0), (0, -1), (2 ** 31, 0), (0, 2 ** 31)):
        assert lib.b2r_mesh_cc_scratch_bytes(nv, nf) == 0


def test_abi_argument_checks():
    lib = _lib.lib()
    F, S, T = 256, 512, 768          # stand-in device addresses; every call below fails its checks before touching them

    def fails(rc, text):
        return rc < 0 and text.encode() in lib.b2r_last_error()

    # label(faces, n_faces, n_verts, labels, scratch, stream)
    assert fails(lib.b2r_mesh_cc_label(F, -1, 4, T, S, None), "n_faces")
    assert fails(lib.b2r_mesh_cc_label(F, 1, 2 ** 31, T, S, None), "n_verts")
    assert fails(lib.b2r_mesh_cc_label(None, 1, 4, T, S, None), "NULL")
    assert fails(lib.b2r_mesh_cc_label(F, 1, 4, None, S, None), "NULL")
    assert fails(lib.b2r_mesh_cc_label(F, 1, 4, T, None, None), "NULL scratch")
    assert fails(lib.b2r_mesh_cc_label(F, 1, 4, T, S + 8, None), "16-byte aligned")
    assert lib.b2r_mesh_cc_label(None, 0, 0, None, S, None) == 0           # nothing to label: no launch
    # select(faces, n_faces, n_verts, labels, ratio, scratch, totals, stream)
    assert fails(lib.b2r_mesh_cc_select(F, 2 ** 31, 4, T, 0.5, S, T, None), "n_faces")
    assert fails(lib.b2r_mesh_cc_select(F, 1, -3, T, 0.5, S, T, None), "n_verts")
    assert fails(lib.b2r_mesh_cc_select(F, 1, 4, None, 0.5, S, T, None), "NULL")
    assert fails(lib.b2r_mesh_cc_select(F, 1, 4, T, 0.5, S, None, None), "NULL")
    for bad in (float("nan"), float("inf"), -0.25, 1.5):
        assert fails(lib.b2r_mesh_cc_select(F, 1, 4, T, bad, S, T, None), "ratio")
    assert fails(lib.b2r_mesh_cc_select(F, 1, 4, T, 0.5, S + 4, T, None), "16-byte aligned")
    # compact(verts, normals, faces, n_faces, n_verts, scratch, verts_out, normals_out, faces_out, stream)
    assert fails(lib.b2r_mesh_cc_compact(T, None, F, -2, 4, S, T, None, T, None), "n_faces")
    assert fails(lib.b2r_mesh_cc_compact(None, None, F, 1, 4, S, T, None, T, None), "NULL verts")
    assert fails(lib.b2r_mesh_cc_compact(T, None, F, 1, 4, S, T, None, None, None), "NULL faces")
    assert fails(lib.b2r_mesh_cc_compact(T, T, F, 1, 4, S, T, None, T, None), "normals_out")
    assert fails(lib.b2r_mesh_cc_compact(T, None, F, 1, 4, None, T, None, T, None), "NULL scratch")
    assert fails(lib.b2r_mesh_cc_compact(T, None, F, 1, 4, S + 12, T, None, T, None), "16-byte aligned")
    with pytest.raises(RuntimeError, match="ratio"):
        _lib.check(lib.b2r_mesh_cc_select(F, 1, 4, T, -1.0, S, T, None), "b2r_mesh_cc_select")
