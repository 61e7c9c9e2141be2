"""Quadric edge collapse on the device against the numpy oracle (oracle/mesh_decimation.py), bit for bit: ops.decimate_mesh on
marching-cubes meshes of sphere / torus fields, a surface clipped by the lattice box, smoothed and raw noise meshes, and the same
meshes renumbered and shuffled, with a repeat run; and create_mesh(max_faces=...) of NeRF, SirenNeRF and pi-GAN, alone and with
min_component_ratio and smooth_iterations, against its stages (oracle decimation, mesh normals, colour query) and its PLY."""
import numpy as np
import pytest
import torch

from msra_practice_project_b200 import mesh, models, nerf_render, ops, pigan_render
from oracle import marching_cubes as mc
from oracle import mesh_decimation as md
from oracle import mesh_smoothing as sm

from test_gpu_mesh_components import _gpu_mesh, _noise, _permuted
from test_gpu_mesh_export import _seeded
from test_mesh_components_cpu import BIG, SMALL, TORUS, _union
from test_mesh_export_cpu import read_ply

pytestmark = pytest.mark.gpu


def _check(verts, faces, budgets):
    """ops.decimate_mesh equals the oracle at each budget, and a second run is identical."""
    v = np.ascontiguousarray(verts, np.float32)
    f = np.ascontiguousarray(faces, np.int32)
    vd, fd = torch.from_numpy(v).cuda(), torch.from_numpy(f).cuda()
    for budget in budgets:
        got_v, got_f = ops.decimate_mesh(vd, fd, budget)
        ref_v, ref_f = md.decimate(v, f, budget)
        assert got_v.dtype == torch.float32 and got_f.dtype == torch.int32
        assert np.array_equal(got_v.cpu().numpy(), ref_v), budget
        assert np.array_equal(got_f.cpu().numpy(), ref_f), budget
        again = ops.decimate_mesh(vd, fd, budget)
        assert torch.equal(again[0], got_v) and torch.equal(again[1], got_f)
    assert np.array_equal(vd.cpu().numpy(), v) and np.array_equal(fd.cpu().numpy(), f)          # the inputs are not touched
    same = ops.decimate_mesh(vd, fd, len(f))
    assert same[0] is vd and same[1] is fd


@pytest.mark.parametrize("name", ["shapes", "torus"])
def test_decimate_sphere_and_torus_fields(name):
    field = _union(BIG, TORUS, *SMALL) if name == "shapes" else TORUS
    v, f = mc.marching_cubes(field, 0.0)
    _check(v, f, (len(f) // 2, len(f) // 10, 1))
    for seed in (1, 2):
        _check(*_permuted(v, f, seed), (len(f) // 5,))


def test_decimate_box_clipped_surface():
    # a sphere larger than the lattice: the surface leaves through the box faces and has open boundaries there
    g = np.stack(np.meshgrid(*[np.arange(48, dtype=np.float64)] * 3, indexing="ij"), -1)
    field = (np.linalg.norm(g - np.array([24.0, 24.0, -6.0]), axis=-1) - 30.0).astype(np.float32)
    v, f = mc.marching_cubes(field, 0.0)
    _check(v, f, (len(f) // 3, 100))


@pytest.mark.parametrize("n,sigma,frac", [(64, 1.5, 0.3), (128, 1.5, 0.5), (64, 0.0, 0.5)])
def test_decimate_noise_fields(n, sigma, frac):
    verts, faces = _gpu_mesh(_noise(n, sigma))
    v, f = verts.cpu().numpy(), faces.cpu().numpy()
    print(f"noise {n}^3 sigma {sigma}: V {len(v)} F {len(f)}")
    _check(v, f, (int(len(f) * frac),))
    if n <= 64:
        _check(*_permuted(v, f, 3), (int(len(f) * frac),))


def test_decimate_smoothed_mesh():
    verts, faces = _gpu_mesh(_noise(96, 2.0))
    sv = ops.smooth_mesh(verts, faces, 10)
    _check(sv.cpu().numpy(), faces.cpu().numpy(), (len(faces) // 4,))


def test_empty_faceless_and_bad_inputs():
    v = torch.randn(10, 3, device="cuda")
    f0 = torch.zeros((0, 3), dtype=torch.int32, device="cuda")
    got = ops.decimate_mesh(v, f0, 1)
    assert got[0] is v and got[1] is f0
    for bad in ([[0, 1, 10]], [[0, -1, 2]]):
        with pytest.raises(RuntimeError, match="outside"):
            ops.decimate_mesh(v, torch.tensor(bad, dtype=torch.int32, device="cuda"), 1)
    for bad in (0, -3, 2.0, None, True):
        with pytest.raises(ValueError):
            ops.decimate_mesh(v, torch.tensor([[0, 1, 2]], dtype=torch.int32, device="cuda"), bad)
    torch.cuda.synchronize()


def _expected(full, max_faces, model, precision):
    """The oracle decimation of an undecimated call's (verts, faces), its mesh normals and the colours mesh.vertex_colors gives
    the decimated mesh."""
    v, f = md.decimate(full[0].cpu().numpy(), full[1].cpu().numpy(), max_faces)
    n = sm.mesh_normals(v, f)
    rgb = mesh.vertex_colors(model, torch.from_numpy(v).cuda(), torch.from_numpy(n).cuda(), precision).cpu().numpy()
    return v, f, n, rgb


def _check_export(out, expected, path):
    assert all(t.is_cuda for t in out)
    for got, ref in zip(out, expected):
        assert np.array_equal(got.cpu().numpy(), ref)
    lines, vrec, pf = read_ply(path)
    assert f"element vertex {len(expected[0])}" in lines and f"element face {len(expected[1])}" in lines
    assert np.array_equal(np.stack([vrec[c] for c in "xyz"], 1), expected[0]) and np.array_equal(pf, expected[1])
    assert np.array_equal(np.stack([vrec[c] for c in ("nx", "ny", "nz")], 1), expected[2])
    assert np.array_equal(np.stack([vrec[c] for c in ("red", "green", "blue")], 1), expected[3])


@pytest.mark.parametrize("kind,precision", [("nerf", "bf16"), ("nerf", "fp32"), ("siren", "bf16")])
def test_nerf_create_mesh_max_faces(tmp_path, kind, precision):
    net = _seeded(kind)
    n, lo, hi = 80, (-1.5, -1.2, -1.0), (1.5, 1.3, 1.1)
    sigma, _, _ = nerf_render.density_lattice(net, lo, hi, n, max_batch=100000, precision=precision)
    thr = float(np.percentile(sigma.cpu().numpy(), 70))
    kw = dict(box_min=lo, box_max=hi, threshold=thr, precision=precision)
    path = str(tmp_path / "decimated.ply")
    for ratio, iterations in ((0.0, 0), (0.01, 0), (0.0, 5), (0.01, 5)):
        full = nerf_render.create_mesh(net, None, n, min_component_ratio=ratio, smooth_iterations=iterations, **kw)
        budget = len(full[1]) // 3
        assert budget > 1000
        out = nerf_render.create_mesh(net, path, n, min_component_ratio=ratio, smooth_iterations=iterations, max_faces=budget, **kw)
        _check_export(out, _expected(full, budget, net, precision), path)
    same = nerf_render.create_mesh(net, None, n, max_faces=None, **kw)
    assert all(torch.equal(a, b) for a, b in zip(same, nerf_render.create_mesh(net, None, n, **kw)))
    for bad in (0, 1.5):
        with pytest.raises(ValueError):
            nerf_render.create_mesh(net, None, n, max_faces=bad, **kw)


def test_pigan_create_mesh_max_faces(tmp_path):
    torch.manual_seed(0)
    gen = models.Generator(256, 16).cuda()
    with torch.no_grad():
        net = gen.film_siren_nerf
        net.input_layer.weight.mul_(20.0)
        net.output_layer_sigma[0].weight.mul_(100.0)
        net.output_layer_sigma[0].bias.zero_()
    z = torch.randn(1, 256, generator=torch.Generator().manual_seed(3)).cuda()
    path = str(tmp_path / "pigan.ply")
    for ratio, iterations in ((0.0, 0), (0.05, 10)):
        full = pigan_render.create_mesh(gen, None, N=96, z=z, min_component_ratio=ratio, smooth_iterations=iterations)
        budget = max(1, len(full[1]) // 4)
        out = pigan_render.create_mesh(gen, path, N=96, z=z, normals=True, colors=True, min_component_ratio=ratio,
                                       smooth_iterations=iterations, max_faces=budget)
        _check_export(out, _expected(full, budget, gen.film_siren_nerf, None), path)
        plain = pigan_render.create_mesh(gen, path, N=96, z=z, min_component_ratio=ratio, smooth_iterations=iterations, max_faces=budget)
        assert len(plain) == 2 and torch.equal(plain[0], out[0]) and torch.equal(plain[1], out[1])
        lines, vrec, pf = read_ply(path)
        assert lines[3:6] == ["property float x", "property float y", "property float z"]
        assert np.array_equal(np.stack([vrec[c] for c in "xyz"], 1), out[0].cpu().numpy()) and np.array_equal(pf, out[1].cpu().numpy())
