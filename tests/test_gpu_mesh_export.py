"""Mesh export on the device against the numpy oracles (oracle/marching_cubes.py, oracle/mesh_attributes.py): box-lattice MLP rows
equal x rows built from the oracle's point formula, b2r_mc_normals equals oracle.vertex_normals, and nerf_render.create_mesh /
pigan_render.create_mesh(normals=True, colors=True) give the oracle's mesh, normals and colours -- all bit for bit."""
import numpy as np
import pytest
import torch

from msra_practice_project_b200 import mesh, models, nerf_render, ops, pigan_render
from oracle import marching_cubes as mc
from oracle import mesh_attributes as ma

from test_mesh_export_cpu import read_ply

pytestmark = pytest.mark.gpu


def _film_net():
    torch.manual_seed(4)
    net = models.FilmSirenNeRF().cuda()
    g = torch.Generator().manual_seed(1)
    net.set_film_params(torch.cat([1.0 + 0.2 * torch.randn(9, 256, generator=g), 0.1 * torch.randn(9, 256, generator=g)], -1).cuda())
    return net


def _nets():
    torch.manual_seed(0)
    return {"nerf": models.NeRF().cuda(), "siren": models.SirenNeRF().cuda(), "film": _film_net()}


@pytest.mark.parametrize("kind", ["nerf", "siren", "film"])
@pytest.mark.parametrize("precision,sigma_only", [("bf16", False), ("bf16", True), ("fp32", False)])
def test_lattice_rows_equal_x_rows(kind, precision, sigma_only):
    net = _nets()[kind]
    for dims, origin, voxel, begin, count in (((5, 7, 9), (-0.3, 0.2, -1.1), 0.0731, 13, 250),
                                              ((11, 13, 17), (0.5, -0.25, 0.125), 0.0123, 777, 1100),
                                              ((2, 2, 2), (0.0, 0.0, 0.0), 1.0, 0, 8)):
        pts = ma.lattice_points(dims, origin, voxel, begin, count)
        x = torch.from_numpy(np.concatenate([pts, np.zeros_like(pts)], 1)).cuda()
        with torch.no_grad():
            got = ops.mlp(net, lattice=(dims, origin, voxel, begin, count), precision=precision, sigma_only=sigma_only)
            ref = ops.mlp(net, x=x, precision=precision, sigma_only=sigma_only)
        assert got.shape == (count, 4)
        assert torch.equal(got, ref), (dims, begin, count)
        assert got.abs().max() > 0 or sigma_only


@pytest.mark.parametrize("precision", ["bf16", "fp32"])
def test_pigan_cube_as_box_lattice_equals_grid(precision):
    net = _film_net()
    n, begin, count = 37, 1234, 20000
    with torch.no_grad():
        grid = ops.mlp(net, grid=(n, begin, count), precision=precision, sigma_only=True)
        box = ops.mlp(net, lattice=((n, n, n), (-0.1, -0.1, -0.1), float(np.float32(0.2 / (n - 1))), begin, count), precision=precision,
                      sigma_only=True)
    assert torch.equal(grid, box)


def _check_normals(field, level):
    f = np.ascontiguousarray(field, dtype=np.float32)
    verts, faces, nrm = ops.marching_cubes(torch.from_numpy(f).cuda(), level, normals=True)
    rv, rf = mc.marching_cubes(f, level)
    rn = ma.vertex_normals(f, level)
    assert np.array_equal(verts.cpu().numpy(), rv) and np.array_equal(faces.cpu().numpy(), rf)
    assert nrm.shape == verts.shape and np.array_equal(nrm.cpu().numpy(), rn)
    return nrm


def _sphere(n, r, noise=0.0, seed=0):
    x = np.linspace(-1, 1, n, dtype=np.float32)
    g = np.meshgrid(x, x, x, indexing="ij")
    f = np.sqrt(g[0] * g[0] + g[1] * g[1] + g[2] * g[2]) - np.float32(r)
    if noise:
        f = f + np.float32(noise) * np.random.default_rng(seed).standard_normal(f.shape, dtype=np.float32)
    return f.astype(np.float32)


def test_normals_all_256_single_cell_configurations():
    rng = np.random.default_rng(5)
    for config in range(256):
        f = np.array([-1.0 if (config >> c) & 1 else 1.0 for c in range(8)], np.float32) * rng.uniform(0.5, 2.0, 8).astype(np.float32)
        _check_normals(f.reshape(2, 2, 2), 0.0)


@pytest.mark.parametrize("n,noise", [(64, 0.0), (256, 0.02)])
def test_normals_spheres(n, noise):
    nrm = _check_normals(_sphere(n, 0.6, noise), 0.0)
    assert len(nrm) > 1000


def test_normals_values_at_the_level_and_off_tile_shapes():
    rng = np.random.default_rng(1)
    f = rng.standard_normal((37, 41, 29)).astype(np.float32)
    f[rng.random(f.shape) < 0.1] = np.float32(0.3)
    _check_normals(f, 0.3)
    for shape in ((3, 300, 257), (130, 2, 2)):
        _check_normals(np.random.default_rng(2).standard_normal(shape).astype(np.float32), 0.1)


def test_normals_generator_sdf():
    torch.manual_seed(0)
    gen = models.Generator(256, 16).cuda()
    with torch.no_grad():
        net = gen.film_siren_nerf
        net.input_layer.weight.mul_(20.0)
        net.output_layer_sigma[0].weight.mul_(100.0)
        net.output_layer_sigma[0].bias.zero_()
    z = torch.randn(1, 256, generator=torch.Generator().manual_seed(3)).cuda()
    sdf, _, _ = pigan_render.create_mesh_sdf(gen, N=96, z=z)
    s = sdf.numpy()
    _check_normals(s, float((s.min() + s.max()) / 2))
    _check_normals(s, -20.0)


def _seeded(kind):
    """A seeded model whose density has structure in the default box: the sigma head is scaled up and its bias zeroed."""
    torch.manual_seed(0)
    net = models.NeRF().cuda() if kind == "nerf" else models.SirenNeRF().cuda()
    with torch.no_grad():
        if kind == "siren":
            net.layers_pos[0].weight.mul_(3.0)
        net.output_layer_sigma.weight.mul_(100.0)
        net.output_layer_sigma.bias.zero_()
    return net


def _expected(model, sigma, level, origin, voxel, precision):
    field = -sigma
    rv, rf = mc.marching_cubes(field, level, voxel, origin)
    rn = ma.vertex_normals(field, level)
    with torch.no_grad():
        x = torch.from_numpy(np.concatenate([rv, -rn], 1)).cuda()
        rc = ops.to8b(ops.mlp(model, x=x, precision=precision)[:, :3]).cpu().numpy() if len(rv) else np.zeros((0, 3), np.uint8)
    return rv, rf, rn, rc


def _check_export(out, expected, path):
    verts, faces, nrm, rgb = out
    rv, rf, rn, rc = expected
    assert verts.is_cuda and faces.is_cuda and nrm.is_cuda and rgb.is_cuda and rgb.dtype == torch.uint8
    assert np.array_equal(verts.cpu().numpy(), rv) and np.array_equal(faces.cpu().numpy(), rf)
    assert np.array_equal(nrm.cpu().numpy(), rn) and np.array_equal(rgb.cpu().numpy(), rc)
    lines, vrec, pf = read_ply(path)
    assert lines[3:9] == ["property float x", "property float y", "property float z", "property float nx", "property float ny",
                          "property float nz"] and lines[9:12] == ["property uchar red", "property uchar green", "property uchar blue"]
    assert np.array_equal(np.stack([vrec[c] for c in "xyz"], 1), rv) and np.array_equal(pf, rf)
    assert np.array_equal(np.stack([vrec[c] for c in ("nx", "ny", "nz")], 1), rn)
    assert np.array_equal(np.stack([vrec[c] for c in ("red", "green", "blue")], 1), rc)


@pytest.mark.parametrize("kind,precision", [("nerf", "bf16"), ("nerf", "fp32"), ("siren", "bf16")])
def test_nerf_create_mesh_end_to_end(tmp_path, kind, precision):
    net = _seeded(kind)
    n, lo, hi = 80, (-1.5, -1.2, -1.0), (1.5, 1.3, 1.1)
    sigma, origin, voxel = nerf_render.density_lattice(net, lo, hi, n, max_batch=100000, precision=precision)
    assert (origin, voxel) == mesh.box_lattice(lo, hi, n)[1:] and tuple(sigma.shape) == mesh.box_lattice(lo, hi, n)[0]
    s = sigma.cpu().numpy()
    thr = float(np.percentile(s, 70))
    assert s.min() < thr < s.max()
    path = str(tmp_path / "nerf.ply")
    out = nerf_render.create_mesh(net, path, n, box_min=lo, box_max=hi, threshold=thr, precision=precision)
    expected = _expected(net, s, -thr, origin, voxel, precision)
    assert len(expected[1]) > 1000
    _check_export(out, expected, path)
    out2 = nerf_render.create_mesh(net, None, n, box_min=lo, box_max=hi, threshold=thr, precision=precision)
    assert all(torch.equal(a, b) for a, b in zip(out, out2))
    # a threshold above every sigma: an empty mesh and a valid PLY
    empty = nerf_render.create_mesh(net, path, n, box_min=lo, box_max=hi, threshold=float(s.max()) + 1.0, precision=precision)
    assert all(t.shape == (0, 3) for t in empty)
    lines, vrec, pf = read_ply(path)
    assert "element vertex 0" in lines and "element face 0" in lines and len(vrec) == 0 and len(pf) == 0
    assert "create_mesh" not in nerf_render.__all__ and "density_lattice" not in nerf_render.__all__


def test_nerf_create_mesh_without_attributes(tmp_path):
    net = _seeded("nerf")
    path = str(tmp_path / "plain.ply")
    verts, faces, nrm, rgb = nerf_render.create_mesh(net, path, 48, threshold=30.0, normals=False, colors=False)
    assert nrm is None and rgb is None
    lines, vrec, pf = read_ply(path)
    assert lines[3:6] == ["property float x", "property float y", "property float z"] and lines[6].startswith("element face")
    assert np.array_equal(np.stack([vrec[c] for c in "xyz"], 1), verts.cpu().numpy()) and np.array_equal(pf, faces.cpu().numpy())


def test_pigan_create_mesh_with_normals_and_colors(tmp_path):
    torch.manual_seed(0)
    gen = models.Generator(256, 16).cuda()
    with torch.no_grad():
        net = gen.film_siren_nerf
        net.input_layer.weight.mul_(20.0)
        net.output_layer_sigma[0].weight.mul_(100.0)
        net.output_layer_sigma[0].bias.zero_()
    z = torch.randn(1, 256, generator=torch.Generator().manual_seed(3)).cuda()
    n = 96
    sdf, origin, voxel = pigan_render.create_mesh_sdf(gen, N=n, z=z)
    path = str(tmp_path / "pigan.ply")
    out = pigan_render.create_mesh(gen, path, N=n, z=z, normals=True, colors=True)
    s = sdf.numpy()
    expected = _expected(gen.film_siren_nerf, -s, -20.0, origin, voxel, None)
    assert len(expected[1]) > 0
    _check_export(out, expected, path)
    plain = pigan_render.create_mesh(gen, None, N=n, z=z)
    assert len(plain) == 2 and torch.equal(plain[0], out[0]) and torch.equal(plain[1], out[1])
