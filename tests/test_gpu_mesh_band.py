"""Narrow-band mesh export on the device against oracle/mesh_band.py, bit for bit: ops.band_select, ops.marching_cubes(bricks=...),
lattice rows as x rows, and create_mesh(narrow_band=...) against the dense create_mesh filtered to the flagged bricks."""
import numpy as np
import pytest
import torch

from msra_practice_project_b200 import mesh, models, nerf_render, ops, pigan_render
from oracle import mesh_attributes as ma
from oracle import mesh_band as mb

pytestmark = pytest.mark.gpu


def _sphere(shape, r, noise=0.0, seed=0):
    g = np.meshgrid(*[np.linspace(-1, 1, n, dtype=np.float32) for n in shape], indexing="ij")
    f = np.sqrt(g[0] * g[0] + g[1] * g[1] + g[2] * g[2]) - np.float32(r)
    if noise:
        f = f + np.float32(noise) * np.random.default_rng(seed).standard_normal(f.shape, dtype=np.float32)
    return f.astype(np.float32)


def _torus(shape, big, small):
    g = np.meshgrid(*[np.linspace(-1, 1, n, dtype=np.float32) for n in shape], indexing="ij")
    q = np.sqrt(g[0] * g[0] + g[1] * g[1]) - np.float32(big)
    return (np.sqrt(q * q + g[2] * g[2]) - np.float32(small)).astype(np.float32)


FIELDS = {"sphere": lambda s: _sphere(s, 0.6), "torus": lambda s: _torus(s, 0.5, 0.2), "noisy": lambda s: _sphere(s, 0.6, 0.02, 1)}


@pytest.mark.parametrize("name", sorted(FIELDS))
@pytest.mark.parametrize("shape,stride", [((64, 64, 64), 4), ((130, 41, 77), 8), ((33, 20, 47), 5)])
def test_band_select_equals_the_oracle(name, shape, stride):
    f = FIELDS[name](shape)
    band = np.full(f.shape, np.inf, np.float32)
    c = mb.coarse_points(f.shape, stride)
    band.flat[c] = f.flat[c]
    flags, index = ops.band_select(torch.from_numpy(band).cuda(), 0.0, stride)
    rf = mb.brick_flags(band, 0.0, stride)
    assert flags.dtype == torch.uint8 and index.dtype == torch.int32
    assert np.array_equal(flags.cpu().numpy(), rf)
    assert np.array_equal(index.cpu().numpy(), mb.band_points(rf, f.shape, stride))


@pytest.mark.parametrize("name", sorted(FIELDS))
@pytest.mark.parametrize("shape,stride", [((64, 64, 64), 4), ((130, 41, 77), 8), ((33, 20, 47), 5)])
def test_masked_marching_cubes_equals_the_oracle(name, shape, stride):
    f = FIELDS[name](shape)
    dims = mb.brick_dims(shape, stride)
    ft = torch.from_numpy(f).cuda()
    rng = np.random.default_rng(7)
    for flags in (np.ones(dims, np.uint8), np.zeros(dims, np.uint8), (rng.random(dims) < 0.3).astype(np.uint8),
                  (rng.random(dims) < 0.7).astype(np.uint8)):
        got = ops.marching_cubes(ft, 0.0, 0.5, (0.1, -0.2, 0.3), normals=True, bricks=(stride, torch.from_numpy(flags).cuda()))
        ref = mb.masked_marching_cubes(f, 0.0, stride, flags, 0.5, (0.1, -0.2, 0.3), normals=True)
        for g, r in zip(got, ref):
            assert np.array_equal(g.cpu().numpy(), r)
    # the band field of a surface the coarse lattice cannot miss gives the dense mesh
    band, flags = mb.band_field(f, 0.0, stride)
    if name != "noisy":
        dense = ops.marching_cubes(ft, 0.0, normals=True)
        got = ops.marching_cubes(torch.from_numpy(band).cuda(), 0.0, normals=True, bricks=(stride, torch.from_numpy(flags).cuda()))
        assert all(torch.equal(a, b) for a, b in zip(got, dense))


def _film_net():
    torch.manual_seed(4)
    net = models.FilmSirenNeRF().cuda()
    g = torch.Generator().manual_seed(1)
    net.set_film_params(torch.cat([1.0 + 0.2 * torch.randn(9, 256, generator=g), 0.1 * torch.randn(9, 256, generator=g)], -1).cuda())
    return net


@pytest.mark.parametrize("kind", ["nerf", "siren", "film"])
@pytest.mark.parametrize("precision,sigma_only", [("bf16", True), ("bf16", False), ("fp32", False)])
def test_lattice_rows_equal_lattice_and_grid_queries(kind, precision, sigma_only):
    torch.manual_seed(0)
    net = {"nerf": models.NeRF, "siren": models.SirenNeRF}[kind]().cuda() if kind != "film" else _film_net()
    rng = np.random.default_rng(3)
    dims, origin, voxel = (37, 29, 53), (-0.3, 0.2, -1.1), 0.0731
    total = int(np.prod(dims))
    idx = torch.from_numpy(np.sort(rng.choice(total, 3000, replace=False)).astype(np.int32)).cuda()
    desc = (dims, origin, voxel, 0, total)
    x = ops.lattice_rows(idx, lattice=desc)
    assert np.array_equal(x[:, :3].cpu().numpy(), ma.lattice_points(dims, origin, voxel)[idx.cpu().numpy()])
    assert not x[:, 3:].any()
    with torch.no_grad():
        got = ops.mlp(net, x=x, precision=precision, sigma_only=sigma_only)
        ref = ops.mlp(net, lattice=desc, precision=precision, sigma_only=sigma_only)[idx.long()]
        assert torch.equal(got, ref)
        n = 40
        gi = torch.from_numpy(np.sort(rng.choice(n ** 3, 3000, replace=False)).astype(np.int32)).cuda()
        got = ops.mlp(net, x=ops.lattice_rows(gi, grid=(n, 0, n ** 3)), precision=precision, sigma_only=sigma_only)
        ref = ops.mlp(net, grid=(n, 0, n ** 3), precision=precision, sigma_only=sigma_only)[gi.long()]
        assert torch.equal(got, ref)


def _generator():
    torch.manual_seed(0)
    gen = models.Generator(256, 16).cuda()
    with torch.no_grad():
        net = gen.film_siren_nerf
        net.input_layer.weight.mul_(20.0)
        net.output_layer_sigma[0].weight.mul_(100.0)
        net.output_layer_sigma[0].bias.zero_()
    return gen, torch.randn(1, 256, generator=torch.Generator().manual_seed(3)).cuda()


def _seeded(kind):
    torch.manual_seed(0)
    net = models.NeRF().cuda() if kind == "nerf" else models.SirenNeRF().cuda()
    with torch.no_grad():
        if kind == "siren":
            net.layers_pos[0].weight.mul_(3.0)
        net.output_layer_sigma.weight.mul_(100.0)
        net.output_layer_sigma.bias.zero_()
    return net


OPTIONS = [{}, {"min_component_ratio": 0.05}, {"smooth_iterations": 3}, {"max_faces": 2000}]


def _same(a, b):
    return len(a) == len(b) and all((x is None and y is None) or torch.equal(x, y) for x, y in zip(a, b))


def _expected(model, field, level, stride, voxel, origin, opts, precision, normals, colors):
    """The dense create_mesh filtered to the flagged bricks: the dense field, the flags of its coarse corners, the masked mesh."""
    f = field.cpu().numpy()
    band = np.full(f.shape, np.inf, np.float32)
    c = mb.coarse_points(f.shape, stride)
    band.flat[c] = f.flat[c]
    flags = torch.from_numpy(mb.brick_flags(band, level, stride)).cuda()
    out = mesh.export(model, field, level, voxel, origin, None, normals, colors, precision, bricks=(stride, flags), **opts)
    if not opts:
        v, fa, n = mb.masked_marching_cubes(f, level, stride, flags.cpu().numpy(), voxel, origin, normals=True)
        assert np.array_equal(out[0].cpu().numpy(), v) and np.array_equal(out[1].cpu().numpy(), fa)
        if normals:
            assert np.array_equal(out[2].cpu().numpy(), n)
    return out


@pytest.mark.parametrize("n", [128, 256])
@pytest.mark.parametrize("stride", [4, 8])
def test_pigan_create_mesh_narrow_band(n, stride):
    gen, z = _generator()
    sdf, origin, voxel = pigan_render.create_mesh_sdf(gen, N=n, z=z)
    for opts in OPTIONS if n == 128 else OPTIONS[:1]:
        got = pigan_render.create_mesh(gen, None, N=n, z=z, normals=True, colors=True, narrow_band=stride, **opts)
        exp = _expected(gen.film_siren_nerf, sdf.cuda(), -20.0, stride, 0.2 / (n - 1), (-0.1, -0.1, -0.1), opts, None, True, True)
        assert len(got[1]) > 0 and _same(got, exp), opts
        if not opts:
            plain = pigan_render.create_mesh(gen, None, N=n, z=z, narrow_band=stride)
            assert _same(plain, got[:2])


@pytest.mark.parametrize("kind,precision", [("nerf", "bf16"), ("nerf", "fp32"), ("siren", "bf16")])
@pytest.mark.parametrize("stride", [4, 8])
def test_nerf_create_mesh_narrow_band(kind, precision, stride):
    net = _seeded(kind)
    n, lo, hi = 96, (-1.5, -1.2, -1.0), (1.5, 1.3, 1.1)
    sigma, origin, voxel = nerf_render.density_lattice(net, lo, hi, n, max_batch=100000, precision=precision)
    thr = float(np.percentile(sigma.cpu().numpy(), 70))
    for opts in OPTIONS:
        got = nerf_render.create_mesh(net, None, n, box_min=lo, box_max=hi, threshold=thr, precision=precision, max_batch=30000,
                                      narrow_band=stride, **opts)
        exp = _expected(net, -sigma, -thr, stride, voxel, origin, opts, precision, True, True)
        assert len(got[1]) > 0 and _same(got, exp), opts


def test_bad_arguments_raise_before_any_launch():
    gen, z = _generator()
    net = _seeded("nerf")
    for bad in (0, 1, True, 4.0):
        with pytest.raises(ValueError, match="narrow_band"):
            pigan_render.create_mesh(gen, None, N=32, z=z, narrow_band=bad)
        with pytest.raises(ValueError, match="narrow_band"):
            nerf_render.create_mesh(net, None, 32, narrow_band=bad)
        with pytest.raises(ValueError, match="stride"):
            ops.band_select(torch.zeros(9, 9, 9, device="cuda"), 0.0, bad)
    f = torch.zeros(17, 9, 5, device="cuda")
    good = torch.zeros(mb.brick_dims(f.shape, 4), dtype=torch.uint8, device="cuda")
    assert tuple(good.shape) == (4, 2, 1)
    for flags, err in ((good.float(), RuntimeError), (torch.zeros(4, 2, 2, dtype=torch.uint8, device="cuda"), RuntimeError),
                       (good.cpu(), RuntimeError), (good[None], RuntimeError)):
        with pytest.raises(err):
            ops.marching_cubes(f, 0.0, bricks=(4, flags))
    for bricks in ((1, good), (4.0, good), [4, good], (4,)):
        with pytest.raises(ValueError):
            ops.marching_cubes(f, 0.0, bricks=bricks)
    # a lattice past 2^31 - 1 points is refused before the mapping network or any query runs
    torch.cuda.synchronize()
    before = torch.cuda.memory_allocated()
    with pytest.raises(RuntimeError, match="2\\^31 - 1"):
        pigan_render.create_mesh(gen, None, N=1291, z=z, narrow_band=4)
    with pytest.raises(RuntimeError, match="2\\^31 - 1"):
        nerf_render.create_mesh(net, None, 1291, narrow_band=4)
    torch.cuda.synchronize()
    assert torch.cuda.memory_allocated() == before
    with pytest.raises(RuntimeError, match="outside"):
        ops.lattice_rows(torch.tensor([0, 8], dtype=torch.int32, device="cuda"), grid=(2, 0, 8))
    with pytest.raises(ValueError):
        ops.lattice_rows(torch.tensor([0], dtype=torch.int32, device="cuda"))
