"""Quadric edge collapse without a GPU: the numpy oracle (oracle/mesh_decimation.py) on marching-cubes meshes of a sphere, a torus,
two spheres and a surface clipped by the lattice box (topology, orientation, shape and the fixed boundary), on hand-made meshes
where the cheapest edge fails the link condition, the valence rule or the flip test, on a tetrahedron, and for the budget
arithmetic; the argument checks of the b2r_mesh_quadrics / _decimate_round / _decimate_compact entry points and of
ops.decimate_mesh, and the scratch size formula."""
import numpy as np
import pytest
import torch

from msra_practice_project_b200 import _lib, ops
from oracle import marching_cubes as mc
from oracle import mesh_components as mcc
from oracle import mesh_decimation as md

from test_mesh_cpu import _grid, _mesh_stats

F32 = np.float32


def _sphere_mesh(n=128, r=0.7):
    (x, y, z), sp = _grid(n)
    return mc.marching_cubes(np.sqrt(x * x + y * y + z * z) - r, 0.0, sp, (-1, -1, -1))


def test_sphere_to_2000_faces():
    r = 0.7
    verts, faces = _sphere_mesh(128, r)
    v, f = md.decimate(verts, faces, 2000)
    assert len(f) in (1999, 2000) and v.dtype == np.float32 and f.dtype == np.int32
    closed, oriented, euler, vol = _mesh_stats(v, f)
    assert closed and oriented and euler == 2
    assert len(np.unique(f)) == len(v)                                     # no vertex left without a face
    p = v.astype(np.float64)
    n = np.cross(p[f[:, 1]] - p[f[:, 0]], p[f[:, 2]] - p[f[:, 0]])
    centroid = (p[f[:, 0]] + p[f[:, 1]] + p[f[:, 2]]) / 3
    assert np.all(np.einsum("ij,ij->i", n, centroid) > 0)                  # no face turned against the radial direction
    exact = 4 / 3 * np.pi * r ** 3
    radial = np.abs(np.linalg.norm(p, axis=1) - r)
    print(f"sphere: F {len(faces)} -> {len(f)}, volume error {abs(vol - exact) / exact:.5f}, radial deviation max {radial.max():.5f}")
    # measured: volume error 0.00968 of the exact ball, radial deviation max 0.00168 (the lattice spacing is 0.0157)
    assert abs(vol - exact) < 0.015 * exact
    assert radial.max() < 0.004


def test_torus_keeps_genus_one():
    (x, y, z), sp = _grid(64)
    field = np.sqrt((np.hypot(x, y) - 0.55) ** 2 + z * z) - 0.25
    verts, faces = mc.marching_cubes(field, 0.0, sp, (-1, -1, -1))
    v, f = md.decimate(verts, faces, 800)
    closed, oriented, euler, _ = _mesh_stats(v, f)
    assert len(f) in (799, 800) and closed and oriented and euler == 0


def test_two_spheres_stay_two_components():
    (x, y, z), sp = _grid(64)
    field = np.minimum(np.sqrt((x - 0.45) ** 2 + y * y + z * z) - 0.35, np.sqrt((x + 0.5) ** 2 + y * y + z * z) - 0.3)
    verts, faces = mc.marching_cubes(field, 0.0, sp, (-1, -1, -1))
    v, f = md.decimate(verts, faces, 600)
    closed, oriented, euler, _ = _mesh_stats(v, f)
    assert closed and oriented and euler == 4
    assert len(np.unique(mcc.component_labels(f, len(v)))) == 2


def _boundary_loops(v, f):
    """The boundary edges (on one face) as a set of coordinate pairs, direction kept."""
    e = np.concatenate([f[:, [0, 1]], f[:, [1, 2]], f[:, [2, 0]]]).astype(np.int64)
    key, count = np.unique(np.sort(e, 1), axis=0, return_counts=True)
    once = {tuple(k) for k in key[count == 1]}
    return {(tuple(v[a]), tuple(v[b])) for a, b in e if (min(a, b), max(a, b)) in once}


def test_box_clipped_surface_keeps_its_boundary():
    (x, y, z), sp = _grid(48)
    verts, faces = mc.marching_cubes(np.sqrt(x * x + y * y + (z + 1.2) ** 2) - 1.6, 0.0, sp, (-1, -1, -1))
    e = np.concatenate([faces[:, [0, 1]], faces[:, [1, 2]], faces[:, [2, 0]]]).astype(np.int64)
    key, count = np.unique(np.sort(e, 1), axis=0, return_counts=True)
    boundary = np.unique(key[count == 1])
    assert len(boundary) > 100
    v, f = md.decimate(verts, faces, len(faces) // 8)
    assert len(f) <= len(faces) // 8
    # surviving vertices keep their order: the boundary vertices are the first len(boundary) of their positions, bit for bit
    kept_pos = {tuple(p) for p in v}
    assert all(tuple(verts[b]) in kept_pos for b in boundary)
    order = [i for i, p in enumerate(map(tuple, v)) if p in {tuple(verts[b]) for b in boundary}]
    assert np.array_equal(v[order], verts[boundary])
    assert _boundary_loops(v, f) == _boundary_loops(verts, faces)
    _, oriented, _, _ = _mesh_stats(v, f)
    assert oriented


def test_tetrahedron_is_left_as_it_is():
    # every edge passes the link condition (its two common neighbours are the opposite vertices) and fails only the valence
    # rule: 3 + 3 - 4 = 2 < 3
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], F32)
    f = np.array([[0, 2, 1], [0, 1, 3], [0, 3, 2], [1, 2, 3]], np.int32)
    out_v, out_f = md.decimate(v, f, 1)
    assert np.array_equal(out_v, v) and np.array_equal(out_f, f)


def test_octahedron_stops_at_a_tetrahedron():
    v = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], F32)
    f = np.array([[0, 2, 4], [2, 1, 4], [1, 3, 4], [3, 0, 4], [2, 0, 5], [1, 2, 5], [3, 1, 5], [0, 3, 5]], np.int32)
    stats = {}
    out_v, out_f = md.decimate(v, f, 1, stats)
    closed, oriented, euler, _ = _mesh_stats(out_v, out_f)
    assert len(out_f) == 4 and closed and oriented and euler == 2
    assert stats["collapses"] == [1, 1]                     # every vertex is within two edges of any other: one per round


def _bipyramid(k, h=1.0, ring_z=None):
    """A closed k-gon bipyramid: ring 0..k-1, apexes k (top) and k+1 (bottom)."""
    ang = np.arange(k) * 2 * np.pi / k
    ring = np.stack([np.cos(ang), np.sin(ang), np.zeros(k) if ring_z is None else ring_z], 1)
    v = np.concatenate([ring, [[0, 0, h], [0, 0, -h]]]).astype(F32)
    f = [[i, (i + 1) % k, k] for i in range(k)] + [[(i + 1) % k, i, k + 1] for i in range(k)]
    return v, np.array(f, np.int32)


def _edge_table(v, f):
    """(cost, a, b, link, valence, no_flip) of every edge in key order, each rule restated edge by edge."""
    q = md.vertex_quadrics(v, f)
    nb = [set() for _ in v]
    for t in f:
        for x in t:
            nb[x] |= {int(y) for y in t if y != x}
    rows = []
    for a, b in md._edges(f.astype(np.int64), len(v))[0]:
        cand = [v[a], v[b], (v[a] + v[b]) * F32(0.5)]
        costs = [md.cost((q[a] + q[b])[None], c[None])[0] for c in cand]
        p = cand[int(np.argmin(costs))]
        opp = {int(x) for t in f if a in t and b in t for x in t if x != a and x != b}
        link = len(nb[a] & nb[b]) == 2 and len(opp) == 2
        valence = len(nb[a]) + len(nb[b]) - 4 >= 3
        no_flip = True
        for x, y in ((a, b), (b, a)):
            for t in f:
                if x in t and y not in t:
                    before = v[t].astype(np.float64)
                    after = before.copy()
                    after[list(t).index(x)] = p
                    no_flip &= bool(np.cross(before[1] - before[0], before[2] - before[0])
                                    @ np.cross(after[1] - after[0], after[2] - after[0]) > 0)
        rows.append((min(costs), int(a), int(b), link, valence, no_flip))
    return sorted(rows)


def test_edges_failing_the_link_condition_never_collapse():
    # a triangular bipyramid: a ring edge has three common neighbours (the third ring vertex and both apexes)
    v, f = _bipyramid(3)
    table = _edge_table(v, f)
    ring = [r for r in table if r[1] < 3 and r[2] < 3]
    assert len(ring) == 3 and not any(r[3] for r in ring)
    best = next(r for r in table if r[3] and r[4] and r[5])
    out_v, out_f = md.decimate(v, f, 1)
    assert len(out_f) == 4                                  # one apex edge collapsed, then the tetrahedron stays
    # the survivor a = best[1] keeps its index, b = best[2] is gone, every other vertex is untouched
    assert np.array_equal(np.delete(out_v, best[1], 0), np.delete(v, [best[1], best[2]], 0))


def test_the_cheapest_edge_is_skipped_when_it_would_flip_a_face():
    # a hexagonal bipyramid with a perturbed ring (found by search): its cheapest edge that passes the link condition and the
    # valence rule, (1, 6), folds a face over; the round takes the next one, (0, 6)
    v = np.array([[3.5844663e-01, 0.0, 5.1783717e-01], [2.7172786e-01, 4.7064644e-01, -4.7161523e-01],
                  [-2.6098698e-01, 4.5204270e-01, 5.2688694e-01], [-8.8267004e-01, 1.0809591e-16, 4.4374861e-02],
                  [-4.4014138e-01, -7.6234722e-01, 2.6857990e-01], [5.1949871e-01, -8.9979815e-01, -1.7862834e-01],
                  [0.0, 0.0, 3.0000001e-01], [0.0, 0.0, -3.0000001e-01]], F32)
    f = _bipyramid(6)[1]
    table = [r for r in _edge_table(v, f) if r[3] and r[4]]
    assert table[0][1:3] == (1, 6) and not table[0][5]
    nxt = next(r for r in table if r[5])
    assert nxt[1:3] == (0, 6)
    out_v, out_f = md.decimate(v, f, len(f) - 2)
    assert len(out_f) == len(f) - 2
    assert np.array_equal(out_v[1:], np.delete(v, [0, 6], 0))
    assert any(np.array_equal(out_v[0], c) for c in (v[0], v[6], (v[0] + v[6]) * F32(0.5)))
    _, oriented, euler, _ = _mesh_stats(out_v, out_f)
    assert oriented and euler == 2


def test_the_valence_rule_is_what_stops_a_tetrahedron():
    v = np.array([[0, 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], F32)
    f = np.array([[0, 2, 1], [0, 1, 3], [0, 3, 2], [1, 2, 3]], np.int32)
    table = _edge_table(v, f)
    assert all(r[3] and not r[4] for r in table)


@pytest.mark.parametrize("max_faces", [1999, 2000, 2001, 5000, 12345])
def test_budget_arithmetic(max_faces):
    verts, faces = _sphere_mesh(64)
    _, f = md.decimate(verts, faces, max_faces)
    assert len(f) in (max_faces - 1, max_faces)


def test_max_faces_at_least_f_is_the_identity_and_bad_budgets_raise():
    verts, faces = _sphere_mesh(24)
    for budget in (len(faces), len(faces) + 1, 10 ** 9):
        out = md.decimate(verts, faces, budget)
        assert out[0] is verts and out[1] is faces
    for bad in (0, -1, 2.0, None, True, "5"):
        with pytest.raises(ValueError):
            md.decimate(verts, faces, bad)


def test_quadric_cost_vanishes_on_the_face_planes():
    v = np.array([[1, 0, 0], [-1, 0, 0], [0, 1, 0], [0, -1, 0], [0, 0, 1], [0, 0, -1]], F32)
    f = np.array([[0, 2, 4], [2, 1, 4], [1, 3, 4], [3, 0, 4], [2, 0, 5], [1, 2, 5], [3, 1, 5], [0, 3, 5]], np.int32)
    q = md.vertex_quadrics(v, f)
    assert np.array_equal(md.cost(q, v), np.zeros(len(v)))
    assert np.all(md.cost(q, v * F32(1.5)) > 0)
    # a face's quadric is its area times the squared plane distance
    fq = md.face_quadrics(v, f)
    area = np.sqrt(3) / 2 * 2 / 2
    assert np.isclose(md.cost(fq[:1], np.array([[0, 0, 0]], F32))[0], area * (1 / np.sqrt(3)) ** 2)


def _align256(b):
    return (b + 255) & ~255


@pytest.mark.parametrize("nv,nf", [(0, 0), (1, 0), (0, 5), (2048, 2049), (75_000_000, 151_000_000), (2 ** 31 - 1, 2 ** 31 - 1)])
def test_scratch_bytes_formula(nv, nf):
    tiles = -(-max(nv, nf) // 2048)
    want = (_align256(4 * nv) + 2 * _align256(16 * nv) + _align256(4 * nv) + _align256(12 * nv) + _align256(4 * nv)
            + _align256(4 * tiles) + _align256(16 * tiles) + 256)
    assert _lib.lib().b2r_mesh_decimate_scratch_bytes(nv, nf) == want


def test_scratch_bytes_out_of_range_is_zero():
    lib = _lib.lib()
    for nv, nf in ((-1, 0), (0, -1), (2 ** 31, 0), (0, 2 ** 31)):
        assert lib.b2r_mesh_decimate_scratch_bytes(nv, nf) == 0


def test_abi_argument_checks():
    lib = _lib.lib()
    V, Q, S, T, K = 256, 512, 768, 1024, 1280          # stand-in device addresses; every call below fails before touching them

    def fails(rc, text):
        return rc < 0 and text.encode() in lib.b2r_last_error()

    # quadrics(verts, n_faces, n_verts, adj_scratch, quadrics, stream)
    assert fails(lib.b2r_mesh_quadrics(V, -1, 4, S, Q, None), "n_faces")
    assert fails(lib.b2r_mesh_quadrics(V, 1, 2 ** 31, S, Q, None), "n_verts")
    assert fails(lib.b2r_mesh_quadrics(None, 1, 4, S, Q, None), "NULL verts")
    assert fails(lib.b2r_mesh_quadrics(V, 1, 4, S, None, None), "NULL verts")
    assert fails(lib.b2r_mesh_quadrics(V, 1, 4, None, Q, None), "NULL scratch")
    assert fails(lib.b2r_mesh_quadrics(V, 1, 4, S + 8, Q, None), "16-byte aligned")
    assert lib.b2r_mesh_quadrics(None, 0, 0, None, None, None) == 0
    # round(verts, quadrics, n_faces, n_verts, adj_scratch, scratch, sel_keys, counts_dev, stream)
    assert fails(lib.b2r_mesh_decimate_round(V, Q, 2 ** 31, 4, S, T, K, K, None), "n_faces")
    assert fails(lib.b2r_mesh_decimate_round(V, Q, 1, -4, S, T, K, K, None), "n_verts")
    assert fails(lib.b2r_mesh_decimate_round(V, Q, 1, 4, S, T, K, None, None), "NULL counts_dev")
    assert fails(lib.b2r_mesh_decimate_round(V, None, 1, 4, S, T, K, K, None), "NULL verts")
    assert fails(lib.b2r_mesh_decimate_round(V, Q, 1, 4, S, T, None, K, None), "NULL verts")
    # compact(verts, quadrics, faces, n_faces, n_verts, sel_keys, cut, scratch, verts_out, quadrics_out, faces_out, stream)
    assert fails(lib.b2r_mesh_decimate_compact(V, Q, K, -1, 4, K, None, T, V, Q, K, None), "n_faces")
    assert fails(lib.b2r_mesh_decimate_compact(V, Q, None, 1, 4, K, None, T, V, Q, K, None), "NULL faces")
    assert fails(lib.b2r_mesh_decimate_compact(V, Q, K, 1, 4, K, None, T, V, Q, None, None), "NULL faces")
    assert fails(lib.b2r_mesh_decimate_compact(V, Q, K, 1, 4, None, None, T, V, Q, K, None), "NULL verts")
    assert fails(lib.b2r_mesh_decimate_compact(V, Q, K, 1, 4, K, None, T, V, None, K, None), "NULL verts")
    assert fails(lib.b2r_mesh_decimate_compact(V, Q, K, 1, 4, K, None, None, V, Q, K, None), "NULL scratch")
    assert fails(lib.b2r_mesh_decimate_compact(V, Q, K, 1, 4, K, None, T + 4, V, Q, K, None), "16-byte aligned")
    assert lib.b2r_mesh_decimate_compact(None, None, None, 0, 0, None, None, None, None, None, None, None) == 0
    with pytest.raises(RuntimeError, match="n_faces"):
        _lib.check(lib.b2r_mesh_decimate_round(V, Q, -2, 4, S, T, K, K, None), "b2r_mesh_decimate_round")


@pytest.mark.parametrize("bad", [0, -1, 1.0, 2.5, "3", None, True])
def test_ops_rejects_bad_max_faces(bad):
    verts, faces = torch.zeros(3, 3), torch.tensor([[0, 1, 2]], dtype=torch.int32)
    with pytest.raises(ValueError):
        ops.decimate_mesh(verts, faces, bad)


def test_ops_host_tensors_raise():
    verts, faces = torch.zeros(3, 3), torch.tensor([[0, 1, 2]], dtype=torch.int32)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.decimate_mesh(verts, faces, 1)
