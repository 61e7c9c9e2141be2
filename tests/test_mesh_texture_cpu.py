"""CPU checks of the per-face texture atlas (oracle/mesh_texture.py, ops.atlas_layout): the ownership invariant in exact
arithmetic, disjoint cells, UVs, the odd last cell, corner rows, the face bound, the PNG and textured PLY writers, and the
argument checks of the b2r_mesh_atlas_* entry points and of create_mesh(texture=...), which need no device."""
import struct
import zlib

import numpy as np
import pytest

from msra_practice_project_b200 import _lib, mesh, models, nerf_render, ops, pigan_render
from oracle import mesh_texture as mt

from test_mesh_export_cpu import read_ply


def _corners(f, size, n_faces):
    """Integer local-to-image texel corners of face f: [(col, row)] * 3."""
    _, per_row, s = mt.layout(n_faces, size)
    k = f // 2
    cx, cy, l = (k % per_row) * s, (k // per_row) * s, s - 3
    loc = [(0, 0), (l, 0), (0, l)]
    if f & 1:
        loc = [(s - 1 - x, s - 1 - y) for x, y in loc]
    return [(cx + x, cy + y) for x, y in loc]


@pytest.mark.parametrize("s", range(4, 13))
@pytest.mark.parametrize("odd", [False, True])
def test_bilinear_lookups_read_only_the_faces_own_texels(s, odd):
    """Every point of every face's UV triangle, corners and edges included, on a grid of 1/8 texel (exact integers in units of
    1/8 texel centre): each texel with a non-zero bilinear weight is baked for that face."""
    size, n_faces = 4 * s, 32 - int(odd)            # 16 cells, 4 per row, s texels each; with odd F the last cell has no B
    assert mt.layout(n_faces, size) == (16, 4, s)
    col, row, face, _ = mt.texels(n_faces, size)
    owner = np.full((size, size), -1, np.int64)
    owner[row, col] = face
    l8 = 8 * (s - 3)
    i, j = np.meshgrid(np.arange(l8 + 1), np.arange(l8 + 1), indexing="ij")
    keep = i + j <= l8
    i, j = i[keep], j[keep]
    for f in range(n_faces):
        (x0, y0), _, _ = _corners(f, size, n_faces)
        px, py = (8 * x0 - i, 8 * y0 - j) if f & 1 else (8 * x0 + i, 8 * y0 + j)
        for dx in (0, 1):
            for dy in (0, 1):
                used = ((px % 8 > 0) | (dx == 0)) & ((py % 8 > 0) | (dy == 0))
                assert np.all(owner[py[used] // 8 + dy, px[used] // 8 + dx] == f), (s, f, dx, dy)


@pytest.mark.parametrize("n_faces,size", [(1, 16), (2, 16), (3, 16), (7, 64), (32, 16), (31, 16), (1000, 256), (999, 100),
                                          (2 * 25 ** 2, 101), (5, 1024)])
def test_cells_are_disjoint_and_margins_stay_zero(n_faces, size):
    cells, per_row, s = mt.layout(n_faces, size)
    assert per_row * per_row >= cells > (per_row - 1) ** 2 and s == size // per_row >= 4
    col, row, face, w = mt.texels(n_faces, size)
    assert len(col) == cells * s * s
    assert len(np.unique(row * size + col)) == len(col)                  # one row per texel
    assert col.max() < per_row * s and row.max() < -(-cells // per_row) * s
    assert np.array_equal(np.unique(face), np.arange(n_faces))            # every face owns texels
    assert np.all(w >= 0) and np.all(np.abs(w.sum(1, dtype=np.float64) - 1) < 1e-6)
    tex = mt.texture(np.full((len(col), 3), 7, np.uint8), n_faces, size)
    assert int(np.count_nonzero(tex[..., 0])) == len(col)
    assert not tex[per_row * s:].any() and not tex[:, per_row * s:].any()


@pytest.mark.parametrize("n_faces,size", [(1, 16), (5, 16), (31, 16), (999, 100), (12345, 512), (2 * 4 ** 2, 17)])
def test_uvs_are_the_corner_texel_centres_inside_the_unit_square(n_faces, size):
    uv = mt.uvs(n_faces, size)
    assert uv.dtype == np.float32 and uv.shape == (n_faces, 3, 2)
    assert np.all(uv > 0) and np.all(uv < 1)
    for f in (0, n_faces // 2, n_faces - 1):
        for c, (x, y) in enumerate(_corners(f, size, n_faces)):
            assert uv[f, c, 0] == np.float32(np.float32(x) + np.float32(0.5)) / np.float32(size)
            assert uv[f, c, 1] == np.float32(1) - np.float32(np.float32(y) + np.float32(0.5)) / np.float32(size)
            assert abs(float(uv[f, c, 0]) * size - 0.5 - x) < 1e-3 and abs((1 - float(uv[f, c, 1])) * size - 0.5 - y) < 1e-3
    # A and B wind the same way in UV space (B is A turned by 180 degrees; v runs up the image, so the turn is clockwise)
    e1, e2 = uv[:, 1] - uv[:, 0], uv[:, 2] - uv[:, 0]
    assert np.all(e1[:, 0] * e2[:, 1] - e1[:, 1] * e2[:, 0] < 0)


def test_odd_face_count_gives_the_last_cell_to_its_a_face():
    n_faces, size = 9, 64
    cells, per_row, s = mt.layout(n_faces, size)
    col, row, face, w = mt.texels(n_faces, size)
    last = np.arange(len(col)) >= (cells - 1) * s * s
    assert np.all(face[last] == n_faces - 1)
    t = np.arange(s * s)
    x, y = t % s, t // s
    on_or_beyond = x + y >= s - 3                             # on A's hypotenuse, or projected onto it
    wl = w[last]
    assert np.all(wl[on_or_beyond, 0] == 0) and np.all(wl[~on_or_beyond, 0] > 0)
    # a full cell splits at x + y = s
    first = np.arange(len(col)) < s * s
    assert np.array_equal(face[first], np.where(x + y >= s, 1, 0))


@pytest.mark.parametrize("n_faces,size", [(1, 16), (6, 32), (9, 16)])
def test_corner_texels_query_their_vertices_bit_for_bit(n_faces, size):
    rng = np.random.default_rng(n_faces)
    verts = rng.uniform(0.25, 2.0, (3 * n_faces, 3)).astype(np.float32) * rng.choice([-1, 1], (3 * n_faces, 3)).astype(np.float32)
    normals = rng.normal(size=(3 * n_faces, 3)).astype(np.float32)
    faces = rng.permutation(3 * n_faces).reshape(n_faces, 3).astype(np.int32)
    x = mt.rows(verts, faces, normals, size)
    cells, per_row, s = mt.layout(n_faces, size)
    for f in range(n_faces):
        k = f // 2
        for c, (cx, cy) in enumerate(_corners(f, size, n_faces)):
            lx, ly = cx - (k % per_row) * s, cy - (k // per_row) * s
            r = k * s * s + ly * s + lx
            assert np.array_equal(x[r, :3], verts[faces[f, c]]), (f, c)
            n = normals[faces[f, c]]
            assert np.allclose(x[r, 3:], -n / np.linalg.norm(n), atol=1e-6)
    # a zero normal sum gives a zero direction
    x0 = mt.rows(verts, faces, np.zeros_like(normals), size)
    assert np.all(x0[:, 3:] == 0)


@pytest.mark.parametrize("size", [16, 17, 19, 100, 2048, 4096, 16384])
def test_face_bound_and_layout_match_the_oracle(size):
    limit = 2 * (size // 4) ** 2
    for n_faces in (0, 1, 2, 3, limit // 3, limit - 1, limit):
        assert ops.atlas_layout(n_faces, size) == mt.layout(n_faces, size)
        assert n_faces == 0 or ops.atlas_layout(n_faces, size)[2] >= 4
    with pytest.raises(ValueError, match=f"at most {limit}"):
        ops.atlas_layout(limit + 1, size)


@pytest.mark.parametrize("size", [15, 16385, 0, -16, 64.0, True, None, "64"])
def test_bad_texture_sizes_raise(size):
    with pytest.raises(ValueError):
        ops.atlas_layout(4, size)


def _decode_png(path):
    data = open(path, "rb").read()
    assert data[:8] == b"\x89PNG\r\n\x1a\n"
    pos, chunks = 8, []
    while pos < len(data):
        n, tag = struct.unpack(">I4s", data[pos:pos + 8])
        body = data[pos + 8:pos + 8 + n]
        assert struct.unpack(">I", data[pos + 8 + n:pos + 12 + n])[0] == zlib.crc32(tag + body)
        chunks.append((tag, body))
        pos += 12 + n
    assert [t for t, _ in chunks] == [b"IHDR", b"IDAT", b"IEND"]
    w, h, depth, ctype, comp, filt, inter = struct.unpack(">IIBBBBB", chunks[0][1])
    assert (depth, ctype, comp, filt, inter) == (8, 2, 0, 0, 0)
    raw = np.frombuffer(zlib.decompress(chunks[1][1]), np.uint8).reshape(h, 1 + 3 * w)
    assert np.all(raw[:, 0] == 0)
    return raw[:, 1:].reshape(h, w, 3)


@pytest.mark.parametrize("h,w", [(16, 16), (3, 17), (1, 1)])
def test_png_round_trip(tmp_path, h, w):
    img = np.random.default_rng(h * w).integers(0, 256, (h, w, 3), dtype=np.uint8)
    path = str(tmp_path / "t.png")
    mesh.write_png(path, img)
    assert np.array_equal(_decode_png(path), img)
    with pytest.raises(ValueError):
        mesh.write_png(path, img[..., :2])


def test_textured_ply_round_trip(tmp_path):
    rng = np.random.default_rng(1)
    verts = rng.normal(size=(10, 3)).astype(np.float32)
    normals = rng.normal(size=(10, 3)).astype(np.float32)
    colors = rng.integers(0, 256, (10, 3), dtype=np.uint8)
    faces = rng.integers(0, 10, (7, 3)).astype(np.int32)
    uvs = mt.uvs(7, 64)
    path = str(tmp_path / "m.ply")
    mesh.write_ply(path, verts, faces, normals, colors, uvs, "m.png")
    data = open(path, "rb").read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    lines = data[:end].decode("ascii").splitlines()
    assert lines[:3] == ["ply", "format binary_little_endian 1.0", "comment TextureFile m.png"]
    assert lines[-3:] == ["property list uchar int vertex_indices", "property list uchar float texcoord", "end_header"]
    fields = [(ln.split()[2], {"float": "<f4", "uchar": "u1"}[ln.split()[1]]) for ln in lines if ln.startswith("property ")
              and "list" not in ln]
    vrec = np.frombuffer(data, dtype=fields, count=10, offset=end)
    assert np.array_equal(np.stack([vrec[c] for c in "xyz"], 1), verts)
    assert np.array_equal(np.stack([vrec[c] for c in ("red", "green", "blue")], 1), colors)
    frec = np.frombuffer(data, dtype=[("n", "u1"), ("vi", "<i4", (3,)), ("nt", "u1"), ("uv", "<f4", (6,))], count=7,
                         offset=end + vrec.nbytes)
    assert end + vrec.nbytes + frec.nbytes == len(data)
    assert np.all(frec["n"] == 3) and np.all(frec["nt"] == 6)
    assert np.array_equal(frec["vi"], faces) and np.array_equal(frec["uv"], uvs.reshape(7, 6))
    # without uvs the writer is what it was: read_ply (which knows no texcoords) takes the file whole
    plain = str(tmp_path / "p.ply")
    mesh.write_ply(plain, verts, faces, normals, colors)
    _, _, pf = read_ply(plain)
    assert np.array_equal(pf, faces) and open(plain, "rb").read().count(b"texcoord") == 0


def test_abi_argument_checks():
    lib = _lib.lib()

    def fails(rc, text):
        return rc < 0 and text.encode() in lib.b2r_last_error()

    P = 256                                          # a fake, 16-byte aligned pointer: every call below fails before using it
    assert fails(lib.b2r_mesh_atlas_uvs(4, 15, P, None), "size")
    assert fails(lib.b2r_mesh_atlas_uvs(4, 16385, P, None), "size")
    assert fails(lib.b2r_mesh_atlas_uvs(-1, 64, P, None), "n_faces")
    assert fails(lib.b2r_mesh_atlas_uvs(2 ** 31, 64, P, None), "n_faces")
    assert fails(lib.b2r_mesh_atlas_uvs(33, 16, P, None), "at most 32")
    assert fails(lib.b2r_mesh_atlas_uvs(2 * 4096 ** 2 + 1, 16384, P, None), "do not fit")
    assert fails(lib.b2r_mesh_atlas_uvs(4, 16, None, None), "NULL uvs")
    assert lib.b2r_mesh_atlas_uvs(0, 16, None, None) == 0
    rows = 2 * 8 * 8                                  # 4 faces in 16^2: 2 cells of 8 x 8
    assert fails(lib.b2r_mesh_atlas_rows(P, P, P, 4, 16, 0, rows + 1, P, None), "outside")
    assert fails(lib.b2r_mesh_atlas_rows(P, P, P, 4, 16, -1, 1, P, None), "outside")
    assert fails(lib.b2r_mesh_atlas_rows(P, P, P, 4, 16, rows, 1, P, None), "outside")
    assert fails(lib.b2r_mesh_atlas_rows(P, P, P, 4, 16, 0, -1, P, None), "outside")
    assert fails(lib.b2r_mesh_atlas_rows(P, P, P, 33, 16, 0, 1, P, None), "do not fit")
    assert fails(lib.b2r_mesh_atlas_rows(P, None, P, 4, 16, 0, 1, P, None), "NULL")
    assert fails(lib.b2r_mesh_atlas_rows(P, P, None, 4, 16, 0, 1, P, None), "NULL")
    assert fails(lib.b2r_mesh_atlas_rows(P, P, P, 4, 16, 0, 1, None, None), "NULL")
    assert lib.b2r_mesh_atlas_rows(None, None, None, 4, 16, rows, 0, None, None) == 0
    assert lib.b2r_mesh_atlas_rows(None, None, None, 0, 16, 0, 0, None, None) == 0
    assert fails(lib.b2r_mesh_atlas_texture(P, 4, 16, 0, rows + 1, P, None), "outside")
    assert fails(lib.b2r_mesh_atlas_texture(P, 4, 8, 0, 1, P, None), "size")
    assert fails(lib.b2r_mesh_atlas_texture(None, 4, 16, 0, 1, P, None), "NULL")
    assert fails(lib.b2r_mesh_atlas_texture(P, 4, 16, 0, 1, None, None), "NULL")
    assert fails(lib.b2r_mesh_atlas_texture(P + 4, 4, 16, 0, 1, P, None), "16-byte aligned")
    assert lib.b2r_mesh_atlas_texture(None, 4, 16, 0, 0, None, None) == 0


@pytest.mark.parametrize("texture", [15, 16385, 0, 64.0, True, "64"])
def test_create_mesh_rejects_bad_textures_before_any_launch(texture):
    """The texture size is checked before the density query (which would raise a RuntimeError for these CPU models)."""
    with pytest.raises(ValueError, match="texture"):
        nerf_render.create_mesh(models.NeRF(), N=8, texture=texture)
    with pytest.raises(ValueError, match="texture"):
        pigan_render.create_mesh(models.Generator(256, 16), N=8, texture=texture)
    with pytest.raises(ValueError, match="texture"):
        mesh.bake_texture(models.NeRF(), None, None, None, texture)
