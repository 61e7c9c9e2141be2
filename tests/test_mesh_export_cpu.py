"""Mesh export without a GPU: the numpy oracle's vertex normals on analytic fields (unit length, close to the analytic normal,
oriented like the triangles), the one-sided gradient on the lattice faces, the PLY writer with and without vertex attributes,
the box-lattice arithmetic, and the argument checks of b2r_mc_normals and of box-lattice MLP input."""
import ctypes as C

import numpy as np
import pytest

from msra_practice_project_b200 import _lib, mesh, pigan_render
from oracle import marching_cubes as mc
from oracle import mesh_attributes as ma


def _grid(n, lo, hi):
    a = np.linspace(lo, hi, n)
    return np.stack(np.meshgrid(a, a, a, indexing="ij"), -1), (hi - lo) / (n - 1)


def _check_against(field, level, lo, h, analytic, tol):
    verts, faces = mc.marching_cubes(field, level, h, (lo, lo, lo))
    nrm = ma.vertex_normals(field, level)
    assert nrm.shape == verts.shape and nrm.dtype == np.float32 and len(verts) > 100
    np.testing.assert_allclose(np.linalg.norm(nrm.astype(np.float64), axis=1), 1.0, atol=1e-6)
    assert np.abs(nrm - analytic(verts.astype(np.float64))).max() < tol
    v = verts.astype(np.float64)
    fn = np.cross(v[faces[:, 1]] - v[faces[:, 0]], v[faces[:, 2]] - v[faces[:, 0]])
    for c in range(3):                      # every vertex normal agrees in orientation with every face it belongs to
        assert np.all(np.einsum("ij,ij->i", fn, nrm[faces[:, c]]) > 0)
    return verts, nrm


def test_sphere_normals():
    # f = |x|^2: central differences are exact for a quadratic and the interpolation is linear, so the normal is x/|x|
    x, h = _grid(64, -1.0, 1.0)
    f = (x ** 2).sum(-1).astype(np.float32)
    _check_against(f, 0.5, -1.0, h, lambda v: v / np.linalg.norm(v, axis=1, keepdims=True), 1e-3)


def test_torus_normals():
    x, h = _grid(128, -1.0, 1.0)
    big, small = 0.6, 0.25
    q = np.sqrt(x[..., 0] ** 2 + x[..., 1] ** 2)
    f = ((q - big) ** 2 + x[..., 2] ** 2).astype(np.float32)

    def analytic(v):
        qv = np.sqrt(v[:, 0] ** 2 + v[:, 1] ** 2)
        g = np.stack([2 * (qv - big) * v[:, 0] / qv, 2 * (qv - big) * v[:, 1] / qv, 2 * v[:, 2]], 1)
        return g / np.linalg.norm(g, axis=1, keepdims=True)

    _check_against(f, small ** 2, -1.0, h, analytic, 1e-3)


def test_gradient_is_numpys_scheme():
    rng = np.random.default_rng(3)
    f = rng.standard_normal((5, 7, 3)).astype(np.float32)
    g = ma.gradient(f)
    for a, ga in enumerate(np.gradient(f)):
        np.testing.assert_array_equal(g[..., a], ga)


def test_surface_through_the_lattice_faces_uses_one_sided_differences():
    # a sphere of radius 1 on [-0.8, 0.8]^3 leaves through every face; f = |x|^2 again, where the one-sided difference
    # on a face is off by the curvature term h^2 only
    x, h = _grid(48, -0.8, 0.8)
    f = (x ** 2).sum(-1).astype(np.float32)
    verts, nrm = _check_against(f, 1.0, -0.8, h, lambda v: v / np.linalg.norm(v, axis=1, keepdims=True), 0.1)
    on_face = np.any(np.abs(np.abs(verts) - 0.8) < 1e-6, axis=1)
    assert on_face.sum() > 50
    g = ma.gradient(f)
    assert g[0, 10, 10, 0] == f[1, 10, 10] - f[0, 10, 10] and g[-1, 10, 10, 0] == f[-1, 10, 10] - f[-2, 10, 10]


def test_flat_field_gives_zero_normals():
    f = np.zeros((3, 3, 3), np.float32)
    f[:, :, 1:] = 1.0                          # a step: the gradient is 0.5 or 1 along axis 2 and 0 elsewhere
    nrm = ma.vertex_normals(f, 0.5)
    np.testing.assert_array_equal(nrm, np.tile(np.array([0, 0, 1], np.float32), (9, 1)))
    f = np.full((3, 3, 3), 2.0, np.float32)
    f[1, 1, 1] = 0.0                           # one below point: gradients of the symmetric field vanish at the centre only
    assert np.isfinite(ma.vertex_normals(f, 1.0)).all()


def _old_write_ply(filename, verts, faces):
    verts = np.ascontiguousarray(verts, dtype="<f4").reshape(-1, 3)
    faces = np.asarray(faces).reshape(-1, 3)
    body = np.empty(len(faces), dtype=[("n", "u1"), ("vertex_indices", "<i4", (3,))])
    body["n"] = 3
    body["vertex_indices"] = faces
    header = ("ply\nformat binary_little_endian 1.0\n"
              f"element vertex {len(verts)}\nproperty float x\nproperty float y\nproperty float z\n"
              f"element face {len(faces)}\nproperty list uchar int vertex_indices\nend_header\n")
    with open(filename, "wb") as fh:
        fh.write(header.encode("ascii"))
        verts.view([("x", "<f4"), ("y", "<f4"), ("z", "<f4")]).reshape(-1).tofile(fh)
        body.tofile(fh)


def read_ply(path):
    """(header lines, vertex record array, faces [F,3]) of a binary PLY written by mesh.write_ply."""
    data = open(path, "rb").read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    lines = data[:end].decode("ascii").splitlines()
    nv = int(next(ln for ln in lines if ln.startswith("element vertex")).split()[-1])
    nf = int(next(ln for ln in lines if ln.startswith("element face")).split()[-1])
    types = {"float": "<f4", "uchar": "u1"}
    fields = [(ln.split()[2], types[ln.split()[1]]) for ln in lines if ln.startswith("property ") and "list" not in ln]
    vrec = np.frombuffer(data, dtype=fields, count=nv, offset=end)
    frec = np.frombuffer(data, dtype=[("n", "u1"), ("vi", "<i4", (3,))], count=nf, offset=end + vrec.nbytes)
    assert np.all(frec["n"] == 3) and end + vrec.nbytes + frec.nbytes == len(data)
    return lines, vrec, frec["vi"]


@pytest.mark.parametrize("with_normals,with_colors", [(False, False), (True, False), (False, True), (True, True)])
def test_ply_header_and_round_trip(tmp_path, with_normals, with_colors):
    rng = np.random.default_rng(1)
    verts = rng.standard_normal((7, 3)).astype(np.float32)
    faces = rng.integers(0, 7, (5, 3)).astype(np.int32)
    nrm = rng.standard_normal((7, 3)).astype(np.float32) if with_normals else None
    rgb = rng.integers(0, 256, (7, 3)).astype(np.uint8) if with_colors else None
    path = tmp_path / "m.ply"
    mesh.write_ply(path, verts, faces, nrm, rgb)
    lines, vrec, got_faces = read_ply(path)
    props = ["property float x", "property float y", "property float z"]
    props += ["property float nx", "property float ny", "property float nz"] if with_normals else []
    props += ["property uchar red", "property uchar green", "property uchar blue"] if with_colors else []
    assert lines == ["ply", "format binary_little_endian 1.0", "element vertex 7", *props, "element face 5",
                     "property list uchar int vertex_indices", "end_header"]
    np.testing.assert_array_equal(np.stack([vrec[c] for c in "xyz"], 1), verts)
    if with_normals:
        np.testing.assert_array_equal(np.stack([vrec[c] for c in ("nx", "ny", "nz")], 1), nrm)
    if with_colors:
        np.testing.assert_array_equal(np.stack([vrec[c] for c in ("red", "green", "blue")], 1), rgb)
    np.testing.assert_array_equal(got_faces, faces)


@pytest.mark.parametrize("nv,nf", [(7, 5), (0, 0)])
def test_ply_without_attributes_is_byte_identical_to_the_plain_writer(tmp_path, nv, nf):
    rng = np.random.default_rng(2)
    verts = rng.standard_normal((nv, 3)).astype(np.float32)
    faces = rng.integers(0, max(nv, 1), (nf, 3)).astype(np.int32)
    _old_write_ply(tmp_path / "a.ply", verts, faces)
    pigan_render.write_ply(tmp_path / "b.ply", verts, faces)
    assert (tmp_path / "a.ply").read_bytes() == (tmp_path / "b.ply").read_bytes()


def test_box_lattice():
    assert mesh.box_lattice((-1.5,) * 3, (1.5,) * 3, 256) == ((256, 256, 256), (-1.5, -1.5, -1.5), float(np.float32(3.0 / 255)))
    assert mesh.box_lattice((-1, -2, 0), (1, 2, 0.5), 9) == ((5, 9, 2), (-1.0, -2.0, 0.0), 0.5)
    dims, _, _ = mesh.box_lattice((0, 0, 0), (1.0, 0.3, 0.999), 11)       # ceil(3) + 1 and ceil(9.99) + 1
    assert dims == (11, 4, 11)
    with pytest.raises(ValueError):
        mesh.box_lattice((0, 0, 0), (1, 0, 1), 8)
    p = ma.lattice_points((3, 4, 5), (-1.0, 0.5, 2.0), 0.25, begin=23, count=3)
    np.testing.assert_array_equal(p, np.array([[-0.75, 0.5, 2.75], [-0.75, 0.5, 3.0], [-0.75, 0.75, 2.0]], np.float32))


def test_abi_normals_entry_point_and_lattice_input_checks():
    lib = _lib.lib()
    assert hasattr(lib, "b2r_mc_normals") and "b2r_mc_normals" in _lib.SIGNATURES
    fake = 256      # never dereferenced: every call below is rejected before any launch
    assert lib.b2r_mc_normals(fake, 1, 4, 4, 0.0, fake, fake, None) < 0 and b"n >= 2" in lib.b2r_last_error()
    assert lib.b2r_mc_normals(fake, 2048, 1024, 1024, 0.0, fake, fake, None) < 0 and b"INT32_MAX" in lib.b2r_last_error()
    for i in range(3):
        args = [fake, fake, fake]
        args[i] = None
        assert lib.b2r_mc_normals(args[0], 4, 4, 4, 0.0, args[1], args[2], None) < 0 and b"NULL" in lib.b2r_last_error()
    assert lib.b2r_mc_normals(fake, 4, 4, 4, 0.0, fake + 4, fake, None) < 0 and b"aligned" in lib.b2r_last_error()

    def lattice(dims=(4, 5, 6), voxel=0.1, begin=0, count=8):
        inp = _lib.MlpInput()
        inp.lattice_dims[:] = list(dims)
        inp.lattice_origin[:] = [-1.0, -1.0, -1.0]
        inp.lattice_voxel, inp.grid_begin, inp.n_rays, inp.n_samples = voxel, begin, count, 1
        return inp

    def tc(inp, last=None):
        return lib.b2r_mlp_tc_fwd(0, fake, 1, C.byref(inp), fake, 0, last, None)

    assert C.sizeof(_lib.MlpInput) == 80
    for bad, msg in ((lattice(dims=(1, 5, 6)), b"n >= 2"), (lattice(dims=(4, 0, 6)), b"n >= 2"),
                     (lattice(dims=(2048, 1024, 1024)), b"INT32_MAX"), (lattice(voxel=0.0), b"voxel"),
                     (lattice(voxel=-1.0), b"voxel"), (lattice(voxel=float("inf")), b"voxel"), (lattice(voxel=float("nan")), b"voxel"),
                     (lattice(begin=-1), b"range"), (lattice(begin=115, count=6), b"range")):
        assert tc(bad) < 0 and msg in lib.b2r_last_error(), msg
    both = lattice()
    both.grid_n = 4
    assert tc(both) < 0 and b"exactly one" in lib.b2r_last_error()
    both = lattice()
    both.x = fake
    assert tc(both) < 0 and b"exactly one" in lib.b2r_last_error()
    ls = _lib.LastSample(1, 8, fake, fake, 0.01, 0.0)
    assert tc(lattice(), C.byref(ls)) < 0 and b"grid" in lib.b2r_last_error()
    assert lib.b2r_mlp_f32_last_sigma(0, fake, None, 1, 1, 0, C.byref(lattice()), 1, fake, 1, fake, fake, 1 << 30, None) < 0 \
        and b"rays / x rows only" in lib.b2r_last_error()
    assert lib.b2r_mlp_tc_train_fwd(0, fake, C.byref(lattice()), fake, fake, 1 << 30, None, None) < 0 \
        and b"inference" in lib.b2r_last_error()
    assert lib.b2r_mlp_tc_train_fwd_film_batched(fake, 1, 512, C.byref(lattice()), fake, fake, 1 << 30, None, None) < 0 \
        and b"inference" in lib.b2r_last_error()
    assert lib.b2r_mlp_tc_fwd_film_batched(fake, 1, 512, C.byref(lattice()), fake, 0, None, None) < 0 \
        and b"box-lattice" in lib.b2r_last_error()
    assert lib.b2r_mlp_f32_fwd(0, fake, None, 1, C.byref(lattice(dims=(1, 2, 2))), fake, fake, 1 << 30, 0, 0, None) < 0 \
        and b"n >= 2" in lib.b2r_last_error()

