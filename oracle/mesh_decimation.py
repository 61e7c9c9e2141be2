"""Topology-preserving quadric edge collapse to a face budget in numpy (TEST INFRASTRUCTURE ONLY): what
``b2r_mesh_quadrics`` / ``_decimate_round`` / ``_decimate_compact`` (``csrc/mesh.cu``) compute on the device, with every
float operation rounded separately and in the same order, so the GPU tests compare them bit for bit.

The mesh shrinks in rounds of independent edge collapses:

* Quadrics (float64, computed once from the input).  Face f with corners p0, p1, p2 in its own order: n = (p1 - p0) x (p2 - p0)
  (x = e1y e2z - e1z e2y, and cyclically), l = sqrt((nx nx + ny ny) + nz nz), u = n / l, d = -((ux p0x + uy p0y) + uz p0z),
  w = l * 0.5; its 10 coefficients are w (e_i e_j) for i <= j over e = (ux, uy, uz, d), row by row.  l == 0 gives zeros.  A
  vertex sums the quadrics of its corners in ascending (f, c) order; a collapse of b into a sets Q_a = Q_a + Q_b.
* Frozen vertex: it appears twice in one face, or one of its edges lies on a number of faces other than two (an open boundary
  or non-manifold input).  Frozen vertices never move and are never removed.
* Valid edge (a, b), a < b: neither end frozen; the ends have exactly two common neighbours and the two faces on the edge have
  different opposite vertices (the link condition); valence(a) + valence(b) - 4 >= 3 (valence: distinct neighbours); and
  every face around a or b that does not hold both keeps dot(n_before, n_after) > 0 in float64, its end moved to p.
* Placement: the first of p_a, p_b, (p_a + p_b) * 0.5 (float32) with the strictly smallest cost c(p) = p^T (Q_a + Q_b) p over
  homogeneous p, evaluated as r_i = ((q_i0 x + q_i1 y) + q_i2 z) + q_i3, c = ((r_0 x + r_1 y) + r_2 z) + r_3, and clamped to
  0 when not > 0 (so the float64 bits of a cost sort like the cost).
* Selection: key(e) = (cost, a, b) lexicographically; key(v) = the smallest key of v's valid edges; m(v) = the smallest key(w)
  over v and its neighbours.  Edge e is selected iff key(a) == key(b) == m(a) == m(b) == key(e).  Selected edges are at least
  two edges apart, so their collapses commute, and the cheapest valid edge is always selected.
* Collapse: a moves to the placement and keeps its index, b is removed, the two faces on the edge are deleted and b becomes a
  in the other faces.  Surviving vertices and faces keep their relative order and face indices are remapped.
* Budget: rounds run while F > max_faces and an edge is valid.  A round that would end below max_faces collapses only its
  ceil((F - max_faces) / 2) cheapest selected edges (key order), so it ends at max_faces or max_faces - 1."""
from __future__ import annotations

import numpy as np
from scipy.sparse import coo_matrix

from oracle.mesh_smoothing import corners

F32 = np.float32
F64 = np.float64


def _cross(e1, e2):
    return np.stack([e1[..., (k + 1) % 3] * e2[..., (k + 2) % 3] - e1[..., (k + 2) % 3] * e2[..., (k + 1) % 3] for k in range(3)], -1)


def _dot(n, m):
    return (n[..., 0] * m[..., 0] + n[..., 1] * m[..., 1]) + n[..., 2] * m[..., 2]


def face_quadrics(verts, faces):
    """float64 [F,10]: the area-weighted plane quadric of every face."""
    p = np.asarray(verts, dtype=F32).reshape(-1, 3).astype(F64)
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    p0 = p[f[:, 0]]
    n = _cross(p[f[:, 1]] - p0, p[f[:, 2]] - p0)
    length = np.sqrt(_dot(n, n))
    ok = length > 0
    with np.errstate(divide="ignore", invalid="ignore"):
        u = n / length[:, None]
    d = -((u[:, 0] * p0[:, 0] + u[:, 1] * p0[:, 1]) + u[:, 2] * p0[:, 2])
    w = length * F64(0.5)
    e = np.concatenate([u, d[:, None]], 1)
    q = np.stack([w * (e[:, i] * e[:, j]) for i in range(4) for j in range(i, 4)], 1)
    return np.where(ok[:, None], q, F64(0))


def vertex_quadrics(verts, faces):
    """float64 [V,10]: the sum of each vertex's corner quadrics in ascending (f, c) order, slot by slot."""
    p = np.asarray(verts, dtype=F32).reshape(-1, 3)
    fq = face_quadrics(p, faces)
    face, _, valid = corners(faces, len(p))
    q = np.zeros((len(p), 10), F64)
    for j in range(face.shape[1]):
        rows = valid[:, j]
        q[rows] = q[rows] + fq[face[rows, j]]
    return q


def cost(q, x):
    """c(p) of the quadrics q [...,10] at the float32 points x [...,3], clamped to 0 when not > 0."""
    x = np.asarray(x, dtype=F32).astype(F64)
    X, Y, Z = x[..., 0], x[..., 1], x[..., 2]
    # symmetric 4x4 from the 10 row-major upper-triangle coefficients
    idx = [[0, 1, 2, 3], [1, 4, 5, 6], [2, 5, 7, 8], [3, 6, 8, 9]]
    r = [((q[..., i[0]] * X + q[..., i[1]] * Y) + q[..., i[2]] * Z) + q[..., i[3]] for i in idx]
    c = ((r[0] * X + r[1] * Y) + r[2] * Z) + r[3]
    return np.where(c > 0, c, F64(0))


def _edges(f, n):
    """Unique undirected edges (lo, hi) of the faces, each face counted once per edge, with the number of faces on it."""
    lo = np.stack([np.minimum(f[:, i], f[:, (i + 1) % 3]) for i in range(3)], 1)
    hi = np.stack([np.maximum(f[:, i], f[:, (i + 1) % 3]) for i in range(3)], 1)
    k = lo * n + hi
    keep = lo != hi
    keep[:, 1] &= k[:, 1] != k[:, 0]                                # a face listing a vertex twice gives its edge once
    keep[:, 2] &= (k[:, 2] != k[:, 0]) & (k[:, 2] != k[:, 1])
    e, count = np.unique(k[keep], return_counts=True)
    return np.stack([e // n, e % n], 1), count


def _round(p, q, f, budget):
    """One round: (p', q', f', collapses) with at most ``budget`` collapses (None: no limit)."""
    n = len(p)
    e, count = _edges(f, n)
    ea, eb = e[:, 0], e[:, 1]
    frozen = np.zeros(n, bool)
    frozen[f[:, 0][(f[:, 0] == f[:, 1]) | (f[:, 0] == f[:, 2])]] = True
    frozen[f[:, 1][f[:, 1] == f[:, 2]]] = True
    bad = count != 2
    frozen[ea[bad]] = True
    frozen[eb[bad]] = True
    valence = np.bincount(ea, minlength=n) + np.bincount(eb, minlength=n)
    adj = coo_matrix((np.ones(2 * len(e), np.int8), (np.concatenate([ea, eb]), np.concatenate([eb, ea]))), shape=(n, n)).tocsr()

    cand = np.flatnonzero(~frozen[ea] & ~frozen[eb] & (valence[ea] + valence[eb] - 4 >= 3))
    a, b = ea[cand], eb[cand]
    common = np.asarray(adj[a].multiply(adj[b]).sum(1)).reshape(-1)
    # opposite vertices of the two faces on each edge
    ok = common == 2
    a, b, cand = a[ok], b[ok], cand[ok]
    fo = np.concatenate([f[:, [0, 1, 2]], f[:, [1, 2, 0]], f[:, [2, 0, 1]]])       # (x, y, opposite) per face edge
    lo, hi, opp = fo[:, :2].min(1), fo[:, :2].max(1), fo[:, 2]
    order = np.lexsort((hi, lo))
    keys_sorted = lo[order] * n + hi[order]
    want = a * n + b
    first = np.searchsorted(keys_sorted, want)
    o1, o2 = opp[order[first]], opp[order[first + 1]]
    ok = o1 != o2
    a, b = a[ok], b[ok]

    qs = q[a] + q[b]
    pa, pb = p[a], p[b]
    mid = (pa + pb) * F32(0.5)
    c0, c1, c2 = cost(qs, pa), cost(qs, pb), cost(qs, mid)
    place, best = pa.copy(), c0.copy()
    better = c1 < best
    place[better], best[better] = pb[better], c1[better]
    better = c2 < best
    place[better], best[better] = mid[better], c2[better]

    # no flip: the faces around a (b) without b (a), with a (b) moved to the placement
    face, _, valid = corners(f, n)
    pd = p.astype(F64)
    keep = np.ones(len(a), bool)
    for x, y in ((a, b), (b, a)):
        for j in range(face.shape[1]):
            has = valid[x, j]
            tri = f[face[x, j]]
            use = has & ~np.any(tri == y[:, None], 1)
            pts = pd[tri]
            moved = np.where((tri == x[:, None])[..., None], place.astype(F64)[:, None, :], pts)
            nb = _cross(pts[:, 1] - pts[:, 0], pts[:, 2] - pts[:, 0])
            na = _cross(moved[:, 1] - moved[:, 0], moved[:, 2] - moved[:, 0])
            keep &= ~use | (_dot(nb, na) > 0)
    a, b, place, best = a[keep], b[keep], place[keep], best[keep]
    if not len(a):
        return p, q, f, 0

    # selection: rank of every valid edge in (cost, a, b) order; key(v), m(v) as ranks
    rank = np.empty(len(a), np.int64)
    rank[np.lexsort((b, a, best))] = np.arange(len(a))
    none = np.iinfo(np.int64).max
    key = np.full(n, none, np.int64)
    np.minimum.at(key, a, rank)
    np.minimum.at(key, b, rank)
    m = key.copy()
    np.minimum.at(m, ea, key[eb])
    np.minimum.at(m, eb, key[ea])
    sel = (key[a] == rank) & (key[b] == rank) & (m[a] == rank) & (m[b] == rank)
    sel_idx = np.flatnonzero(sel)
    if budget is not None and len(sel_idx) > budget:
        sel_idx = sel_idx[np.argsort(rank[sel_idx], kind="stable")[:budget]]
    a, b, place = a[sel_idx], b[sel_idx], place[sel_idx]

    p = p.copy()
    q = q.copy()
    p[a] = place
    q[a] = q[a] + q[b]
    target = np.arange(n)
    target[b] = a
    removed = np.zeros(n, bool)
    removed[b] = True
    dead = np.zeros(len(f), bool)                                 # the faces holding both ends of a collapsed edge
    for i in range(3):
        u = f[:, i]
        dead |= removed[u] & ((target[u] == f[:, (i + 1) % 3]) | (target[u] == f[:, (i + 2) % 3]))
    g = target[f]
    keepv = ~removed
    new_index = np.cumsum(keepv) - keepv
    return p[keepv], q[keepv], new_index[g[~dead]], len(a)


def decimate(verts, faces, max_faces, stats=None):
    """``(verts' [V',3] float32, faces' [F',3] int32)`` after edge-collapse rounds down to ``max_faces`` (an int >= 1).
    ``max_faces >= F`` returns the inputs.  ``stats``, a dict when given, receives the number of rounds and the collapses of
    each round."""
    if isinstance(max_faces, bool) or not isinstance(max_faces, (int, np.integer)) or max_faces < 1:
        raise ValueError(f"max_faces must be an int >= 1, got {max_faces!r}")
    p = np.asarray(verts, dtype=F32).reshape(-1, 3)
    f = np.asarray(faces, dtype=np.int64).reshape(-1, 3)
    if f.size and (f.min() < 0 or f.max() >= len(p)):
        raise ValueError(f"face indices must lie in [0, {len(p)})")
    if int(max_faces) >= len(f):
        return verts, faces
    q = vertex_quadrics(p, f)
    per_round = []
    while len(f) > max_faces:
        budget = (len(f) - int(max_faces) + 1) // 2
        p, q, f, k = _round(p, q, f, budget)
        if not k:
            break
        per_round.append(k)
    if stats is not None:
        stats["rounds"] = len(per_round)
        stats["collapses"] = per_round
    return p, f.astype(np.int32)
