"""Taubin smoothing and mesh normals on the device against the numpy oracle (oracle/mesh_smoothing.py), bit for bit:
ops.smooth_mesh on marching-cubes meshes of sphere / torus fields and of smoothed and raw noise, the same meshes renumbered and
shuffled, a fan vertex of high degree and a mesh with degenerate faces; and create_mesh(smooth_iterations=...) of NeRF, SirenNeRF
and pi-GAN, with and without min_component_ratio, against the oracle smoothing of the unsmoothed call's mesh."""
import numpy as np
import pytest
import torch

from msra_practice_project_b200 import mesh, models, nerf_render, ops, pigan_render
from oracle import marching_cubes as mc
from oracle import mesh_smoothing as sm

from test_gpu_mesh_components import _gpu_mesh, _noise, _permuted
from test_gpu_mesh_export import _seeded
from test_mesh_components_cpu import BIG, SMALL, TORUS, _union
from test_mesh_export_cpu import read_ply

pytestmark = pytest.mark.gpu


def _check(verts, faces, iterations=(1, 10)):
    """ops.smooth_mesh (positions and normals) equals the oracle at each iteration count, and a second run is identical."""
    v = np.ascontiguousarray(verts, np.float32)
    f = np.ascontiguousarray(faces, np.int32)
    vd, fd = torch.from_numpy(v).cuda(), torch.from_numpy(f).cuda()
    for it in iterations:
        got_v, got_n = ops.smooth_mesh(vd, fd, it, normals=True)
        ref_v = sm.smooth(v, f, it)
        assert got_v.shape == vd.shape and got_v.dtype == torch.float32
        assert np.array_equal(got_v.cpu().numpy(), ref_v), it
        assert np.array_equal(got_n.cpu().numpy(), sm.mesh_normals(ref_v, f)), it
        again = ops.smooth_mesh(vd, fd, it)
        assert torch.equal(again, got_v)
    assert np.array_equal(vd.cpu().numpy(), v)                    # the input is not touched
    got_v, got_n = ops.smooth_mesh(vd, fd, 0, normals=True)
    assert got_v is vd and np.array_equal(got_n.cpu().numpy(), sm.mesh_normals(v, f))


@pytest.mark.parametrize("name", ["shapes", "torus"])
def test_smooth_sphere_and_torus_fields(name):
    field = _union(BIG, TORUS, *SMALL) if name == "shapes" else TORUS
    v, f = mc.marching_cubes(field, 0.0)
    _check(v, f)
    for seed in (1, 2):
        _check(*_permuted(v, f, seed), iterations=(10,))


@pytest.mark.parametrize("n,sigma", [(64, 1.5), (256, 1.5), (64, 0.0)])
def test_smooth_noise_fields(n, sigma):
    verts, faces = _gpu_mesh(_noise(n, sigma))
    v, f = verts.cpu().numpy(), faces.cpu().numpy()
    print(f"noise {n}^3 sigma {sigma}: V {len(v)} F {len(f)}")
    _check(v, f)
    if n <= 64:
        _check(*_permuted(v, f, 3), iterations=(10,))


def test_fan_vertex_of_high_degree_and_degenerate_faces():
    rng = np.random.default_rng(11)
    k = 2500
    ang = np.linspace(0, 2 * np.pi, k, endpoint=False)
    ring = np.stack([np.cos(ang), np.sin(ang), 0.1 * rng.standard_normal(k)], 1).astype(np.float32)
    verts = np.concatenate([np.array([[0, 0, 0.5]], np.float32), ring])
    i = np.arange(k)
    faces = np.stack([np.zeros(k, np.int64), 1 + i, 1 + (i + 1) % k], 1)
    faces = faces[rng.permutation(k)]                               # the fan vertex's corners arrive out of order
    faces[::7] = np.roll(faces[::7], 1, axis=1)
    # degenerate faces: a vertex listed twice and three times, and an unused vertex at the end
    faces = np.concatenate([faces, [[0, 0, 5], [7, 9, 7], [3, 3, 3]]]).astype(np.int32)
    verts = np.concatenate([verts, [[2.0, 2.0, 2.0]]]).astype(np.float32)
    assert np.bincount(faces.reshape(-1))[0] >= 2000
    _check(verts, faces)
    out = ops.smooth_mesh(torch.from_numpy(verts).cuda(), torch.from_numpy(faces).cuda(), 4)
    assert np.array_equal(out[-1].cpu().numpy(), verts[-1])


def test_empty_and_faceless_meshes():
    v0 = torch.zeros((0, 3), device="cuda")
    f0 = torch.zeros((0, 3), dtype=torch.int32, device="cuda")
    got_v, got_n = ops.smooth_mesh(v0, f0, 3, normals=True)
    assert got_v.shape == (0, 3) and got_n.shape == (0, 3)
    v = torch.randn(10, 3, device="cuda")
    got_v, got_n = ops.smooth_mesh(v, f0, 3, normals=True)
    assert torch.equal(got_v, v) and torch.equal(got_n, torch.zeros_like(v))


def test_bad_face_indices_raise_before_any_launch():
    verts = torch.randn(6, 3, device="cuda")
    for bad in ([[0, 1, 6]], [[0, -1, 2]]):
        with pytest.raises(RuntimeError, match="outside"):
            ops.smooth_mesh(verts, torch.tensor(bad, dtype=torch.int32, device="cuda"), 2)
    with pytest.raises(RuntimeError, match="int32"):
        ops.smooth_mesh(verts, torch.tensor([[0, 1, 2]], device="cuda"), 2)
    torch.cuda.synchronize()


def _expected_smoothed(full, iterations, model, precision):
    """The oracle smoothing of an unsmoothed call's (verts, faces), its mesh normals and the colours mesh.vertex_colors gives
    the smoothed mesh."""
    v, f = full[0].cpu().numpy(), full[1].cpu().numpy()
    sv = sm.smooth(v, f, iterations)
    sn = sm.mesh_normals(sv, f)
    rgb = mesh.vertex_colors(model, torch.from_numpy(sv).cuda(), torch.from_numpy(sn).cuda(), precision).cpu().numpy()
    return sv, f, sn, rgb


def _check_smoothed_export(out, expected, path):
    assert all(t.is_cuda for t in out)
    for got, ref in zip(out, expected):
        assert np.array_equal(got.cpu().numpy(), ref)
    lines, vrec, pf = read_ply(path)
    assert f"element vertex {len(expected[0])}" in lines and f"element face {len(expected[1])}" in lines
    assert np.array_equal(np.stack([vrec[c] for c in "xyz"], 1), expected[0]) and np.array_equal(pf, expected[1])
    assert np.array_equal(np.stack([vrec[c] for c in ("nx", "ny", "nz")], 1), expected[2])
    assert np.array_equal(np.stack([vrec[c] for c in ("red", "green", "blue")], 1), expected[3])


@pytest.mark.parametrize("kind,precision", [("nerf", "bf16"), ("nerf", "fp32"), ("siren", "bf16")])
def test_nerf_create_mesh_smooth_iterations(tmp_path, kind, precision):
    net = _seeded(kind)
    n, lo, hi = 80, (-1.5, -1.2, -1.0), (1.5, 1.3, 1.1)
    sigma, _, _ = nerf_render.density_lattice(net, lo, hi, n, max_batch=100000, precision=precision)
    thr = float(np.percentile(sigma.cpu().numpy(), 70))
    kw = dict(box_min=lo, box_max=hi, threshold=thr, precision=precision)
    path = str(tmp_path / "smoothed.ply")
    for ratio in (0.0, 0.01):
        full = nerf_render.create_mesh(net, None, n, min_component_ratio=ratio, **kw)
        assert len(full[1]) > 1000
        for it in (1, 10):
            out = nerf_render.create_mesh(net, path, n, min_component_ratio=ratio, smooth_iterations=it, **kw)
            _check_smoothed_export(out, _expected_smoothed(full, it, net, precision), path)
    same = nerf_render.create_mesh(net, None, n, smooth_iterations=0, **kw)
    assert all(torch.equal(a, b) for a, b in zip(same, nerf_render.create_mesh(net, None, n, **kw)))
    for bad in (-1, 1.5):
        with pytest.raises(ValueError):
            nerf_render.create_mesh(net, None, n, smooth_iterations=bad, **kw)


def test_pigan_create_mesh_smooth_iterations(tmp_path):
    torch.manual_seed(0)
    gen = models.Generator(256, 16).cuda()
    with torch.no_grad():
        net = gen.film_siren_nerf
        net.input_layer.weight.mul_(20.0)
        net.output_layer_sigma[0].weight.mul_(100.0)
        net.output_layer_sigma[0].bias.zero_()
    z = torch.randn(1, 256, generator=torch.Generator().manual_seed(3)).cuda()
    path = str(tmp_path / "pigan.ply")
    for ratio in (0.0, 0.05):
        full = pigan_render.create_mesh(gen, None, N=96, z=z, min_component_ratio=ratio)
        assert len(full[1]) > 0
        out = pigan_render.create_mesh(gen, path, N=96, z=z, normals=True, colors=True, min_component_ratio=ratio, smooth_iterations=10)
        _check_smoothed_export(out, _expected_smoothed(full, 10, gen.film_siren_nerf, None), path)
        plain = pigan_render.create_mesh(gen, path, N=96, z=z, min_component_ratio=ratio, smooth_iterations=10)
        assert len(plain) == 2 and torch.equal(plain[0], out[0]) and torch.equal(plain[1], out[1])
        lines, vrec, pf = read_ply(path)
        assert lines[3:6] == ["property float x", "property float y", "property float z"]
        assert np.array_equal(np.stack([vrec[c] for c in "xyz"], 1), out[0].cpu().numpy()) and np.array_equal(pf, out[1].cpu().numpy())
