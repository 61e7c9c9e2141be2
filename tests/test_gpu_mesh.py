"""Marching cubes on the device (csrc/mesh.cu via ops.marching_cubes and pigan_render.create_mesh) against the numpy oracle
(oracle/marching_cubes.py): vertices and triangles must be EQUAL, bit for bit and in the same order."""
import numpy as np
import pytest
import torch

from msra_practice_project_b200 import models, ops, pigan_render
from oracle import marching_cubes as mc

pytestmark = pytest.mark.gpu


def _check(field, level, spacing=1.0, origin=(0.0, 0.0, 0.0)):
    f = np.ascontiguousarray(field, dtype=np.float32)
    verts, faces = ops.marching_cubes(torch.from_numpy(f).cuda(), level, spacing, origin)
    assert verts.dtype == torch.float32 and faces.dtype == torch.int32 and verts.is_cuda and faces.is_cuda
    rv, rf = mc.marching_cubes(f, level, spacing, origin)
    v, fa = verts.cpu().numpy(), faces.cpu().numpy()
    assert v.shape == rv.shape and fa.shape == rf.shape
    assert np.array_equal(v, rv) and np.array_equal(fa, rf)
    return v, fa


def _sphere(n, r, noise=0.0, seed=0):
    x = np.linspace(-1, 1, n, dtype=np.float32)
    g = np.meshgrid(x, x, x, indexing="ij")
    f = np.sqrt(g[0] * g[0] + g[1] * g[1] + g[2] * g[2]) - np.float32(r)
    if noise:
        f = f + np.float32(noise) * np.random.default_rng(seed).standard_normal(f.shape, dtype=np.float32)
    return f.astype(np.float32), np.float32(2 / (n - 1))


def test_all_256_single_cell_configurations():
    for config in range(256):
        f = np.array([1.0 if (config >> c) & 1 else -1.0 for c in range(8)], np.float32)
        # corner c sits at (c>>2 & 1, c>>1 & 1, c & 1) = its row-major position in a 2x2x2 array, and is below when f < 0
        f = -f.reshape(2, 2, 2)
        _, faces = _check(f, 0.0, 0.5, (0.25, -1.0, 3.0))
        assert len(faces) == len(mc.TRIANGLES[config]), config


def test_sphere_64():
    f, sp = _sphere(64, 0.6)
    v, fa = _check(f, 0.0, sp, (-1.0, -1.0, -1.0))
    assert len(fa) > 10000


def test_random_field_with_values_at_the_level():
    rng = np.random.default_rng(1)
    f = rng.standard_normal((37, 41, 29)).astype(np.float32)
    f[rng.random(f.shape) < 0.1] = np.float32(0.3)
    _check(f, 0.3, 0.1, (0.5, 0.25, -2.0))


@pytest.mark.parametrize("shape", [(3, 300, 257), (130, 2, 2)])
def test_shapes_off_the_tile(shape):
    f = np.random.default_rng(2).standard_normal(shape).astype(np.float32)
    _check(f, 0.1, 0.7)


def test_constant_fields_give_empty_meshes():
    for value, level in ((0.0, 0.0), (0.0, 1.0), (-3.0, -20.0)):
        f = torch.full((17, 5, 9), value, device="cuda")
        verts, faces = ops.marching_cubes(f, level)
        assert tuple(verts.shape) == (0, 3) and tuple(faces.shape) == (0, 3)
        assert verts.dtype == torch.float32 and faces.dtype == torch.int32


def test_sphere_plus_noise_256_and_deterministic():
    f, sp = _sphere(256, 0.6, noise=0.02)
    v, fa = _check(f, 0.0, sp, (-1.0, -1.0, -1.0))
    assert len(fa) > 10 ** 6
    v2, f2 = ops.marching_cubes(torch.from_numpy(f).cuda(), 0.0, sp, (-1.0, -1.0, -1.0))
    assert torch.equal(v2.cpu(), torch.from_numpy(v)) and torch.equal(f2.cpu(), torch.from_numpy(fa))


def test_rejects_bad_fields():
    with pytest.raises(RuntimeError):
        ops.marching_cubes(torch.zeros(1, 4, 4, device="cuda"), 0.0)
    with pytest.raises(RuntimeError):
        ops.marching_cubes(torch.zeros(4, 4, device="cuda"), 0.0)


def _generator():
    """A seeded Generator whose field has structure: untrained, sigma is 0 on the whole [-0.1, 0.1]^3 box, so the input
    layer's frequencies are raised, the sigma head is centred and scaled until sigma crosses the reference's level 20."""
    torch.manual_seed(0)
    gen = models.Generator(256, 16).cuda()
    with torch.no_grad():
        net = gen.film_siren_nerf
        net.input_layer.weight.mul_(20.0)
        net.output_layer_sigma[0].weight.mul_(100.0)
        net.output_layer_sigma[0].bias.zero_()
    z = torch.randn(1, 256, generator=torch.Generator().manual_seed(3)).cuda()
    return gen, z


def _read_ply(path):
    with open(path, "rb") as fh:
        data = fh.read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    header = data[:end].decode("ascii").splitlines()
    nv, nf = int(header[2].split()[-1]), int(header[6].split()[-1])
    assert header == ["ply", "format binary_little_endian 1.0", f"element vertex {nv}", "property float x", "property float y",
                      "property float z", f"element face {nf}", "property list uchar int vertex_indices", "end_header"]
    verts = np.frombuffer(data, dtype="<f4", count=3 * nv, offset=end).reshape(nv, 3)
    body = np.frombuffer(data, dtype=[("n", "u1"), ("vertex_indices", "<i4", (3,))], count=nf, offset=end + 12 * nv)
    assert len(data) == end + 12 * nv + 13 * nf and (body["n"] == 3).all()
    return verts, body["vertex_indices"]


def test_generator_sdf_128():
    """The sdf of a generator at N = 128, at the middle of its range and at the reference's level -20."""
    gen, z = _generator()
    n = 128
    sdf, origin, voxel = pigan_render.create_mesh_sdf(gen, N=n, z=z)
    s = sdf.numpy()
    assert s.min() < s.max()
    level = float((s.min() + s.max()) / 2)
    v, fa = _check(s, level, voxel, origin)
    assert len(fa) > 0
    assert s.min() < -20.0
    _, f20 = _check(s, -20.0, voxel, origin)
    assert len(f20) > 0


def test_create_mesh_writes_the_ply_and_matches_the_oracle(tmp_path):
    gen, z = _generator()
    n = 96
    sdf, origin, voxel = pigan_render.create_mesh_sdf(gen, N=n, z=z)
    level = float((sdf.min() + sdf.max()) / 2)
    path = str(tmp_path / "mesh.ply")
    verts, faces = pigan_render.create_mesh(gen, path, N=n, level=level, z=z)
    assert verts.is_cuda and faces.is_cuda and len(faces) > 0
    rv, rf = mc.marching_cubes(sdf.numpy(), level, voxel, origin)
    assert np.array_equal(verts.cpu().numpy(), rv) and np.array_equal(faces.cpu().numpy(), rf)
    pv, pf = _read_ply(path)
    assert np.array_equal(pv, rv) and np.array_equal(pf, rf)
    # the reference's level -20, and an empty mesh (sigma never reaches 1e9)
    v20, f20 = pigan_render.create_mesh(gen, path, N=n, z=z)
    pv, pf = _read_ply(path)
    assert np.array_equal(pv, v20.cpu().numpy()) and np.array_equal(pf, f20.cpu().numpy()) and len(pf) > 0
    v20, f20 = pigan_render.create_mesh(gen, path, N=n, z=z, level=-1e9)
    assert len(v20) == 0 and len(f20) == 0
    pv, pf = _read_ply(path)
    assert np.array_equal(pv, v20.cpu().numpy()) and np.array_equal(pf, f20.cpu().numpy())
    assert "create_mesh" not in pigan_render.__all__
