"""Connected components of meshes on the device against the numpy/scipy oracle (oracle/mesh_components.py), bit for bit:
ops.mesh_components on marching-cubes meshes of sphere / torus fields and of smoothed and raw noise, the same meshes with their
vertex numbering and face order permuted, and a long strip numbered against the hook direction; ops.filter_components with and
without normals; and create_mesh(min_component_ratio=...) of NeRF, SirenNeRF and pi-GAN against the oracle filter of the
unfiltered call."""
import numpy as np
import pytest
import torch
from scipy.ndimage import gaussian_filter

from msra_practice_project_b200 import models, nerf_render, ops, pigan_render
from oracle import mesh_components as cc

from test_gpu_mesh_export import _seeded
from test_mesh_components_cpu import BIG, SMALL, TORUS, _sphere, _union
from test_mesh_export_cpu import read_ply

pytestmark = pytest.mark.gpu


def _noise(n, sigma, seed=0):
    f = np.random.default_rng(seed).standard_normal((n, n, n), dtype=np.float32)
    if sigma:
        f = gaussian_filter(f, sigma).astype(np.float32)
    return f


def _gpu_mesh(field, level=None, normals=False):
    level = float(np.quantile(field, 0.7)) if level is None else level
    return ops.marching_cubes(torch.from_numpy(np.ascontiguousarray(field)).cuda(), level, normals=normals)


def _permuted(verts, faces, seed):
    """The same mesh with its vertices renumbered and its faces shuffled (and each face's corners rotated)."""
    rng = np.random.default_rng(seed)
    nv = len(verts)
    perm = rng.permutation(nv)                    # new vertex i is old vertex perm[i]
    inv = np.empty(nv, np.int64)
    inv[perm] = np.arange(nv)
    f = inv[faces][rng.permutation(len(faces))]
    f = np.roll(f, 1, axis=1) if seed % 2 else f
    return verts[perm], f.astype(np.int32)


def _check_labels(faces, n_verts):
    faces = np.ascontiguousarray(faces, np.int32)
    got = ops.mesh_components(torch.from_numpy(faces).cuda(), n_verts)
    ref = cc.component_labels(faces, n_verts)
    assert got.dtype == torch.int32 and got.shape == (n_verts,)
    assert np.array_equal(got.cpu().numpy(), ref)
    return ref


def _fields():
    rng = np.random.default_rng(7)
    spheres = [_union(*[_sphere(rng.uniform(8, 56, 3), rng.uniform(1.5, 6.0)) for _ in range(k)]) for k in (1, 12, 40)]
    return {"shapes": _union(BIG, TORUS, *SMALL), "spheres1": spheres[0], "spheres12": spheres[1], "spheres40": spheres[2]}


@pytest.mark.parametrize("name", ["shapes", "spheres1", "spheres12", "spheres40"])
def test_labels_of_sphere_fields(name):
    from oracle import marching_cubes as mc
    v, f = mc.marching_cubes(_fields()[name], 0.0)
    ref = _check_labels(f, len(v))
    assert len(np.unique(ref)) >= (5 if name == "shapes" else 1)
    for seed in (1, 2):
        pv, pf = _permuted(v, f, seed)
        _check_labels(pf, len(pv))


@pytest.mark.parametrize("n,sigma", [(64, 1.5), (256, 1.5), (64, 0.0)])
def test_labels_of_noise_fields(n, sigma):
    verts, faces = _gpu_mesh(_noise(n, sigma))
    f = faces.cpu().numpy()
    ref = _check_labels(f, len(verts))
    n_comp = len(np.unique(ref))
    assert n_comp > (20 if sigma else 200)
    print(f"noise {n}^3 sigma {sigma}: V {len(verts)} F {len(f)} components {n_comp}")
    pv, pf = _permuted(verts.cpu().numpy(), f, 3)
    _check_labels(pf, len(pv))


@pytest.mark.parametrize("reverse", [True, False])
def test_labels_of_a_long_strip(reverse):
    # one component whose faces (i, i+1, i+2) are numbered so that every union hooks toward the far end of the strip
    n = 3_000_001
    i = np.arange(n - 2, dtype=np.int64)
    f = np.stack([i, i + 1, i + 2], 1)
    f = (n - 1 - f) if reverse else f
    ref = _check_labels(f, n)
    assert np.all(ref == 0)
    _check_labels(f[::-1], n)
    _check_labels(f[np.random.default_rng(0).permutation(len(f))], n)


def _check_filter(verts, faces, normals, ratio):
    got = ops.filter_components(verts, faces, ratio, normals)
    again = ops.filter_components(verts, faces, ratio, normals)
    ref = cc.filter_components(verts.cpu().numpy(), faces.cpu().numpy(), ratio, None if normals is None else normals.cpu().numpy())
    assert got[0].is_cuda and got[1].dtype == torch.int32
    assert np.array_equal(got[0].cpu().numpy(), ref[0]) and np.array_equal(got[1].cpu().numpy(), ref[1])
    assert (got[2] is None and ref[2] is None) or np.array_equal(got[2].cpu().numpy(), ref[2])
    assert all((a is None and b is None) or torch.equal(a, b) for a, b in zip(got, again))
    return got


@pytest.mark.parametrize("with_normals", [False, True])
@pytest.mark.parametrize("field", ["noise128", "shapes"])
def test_filter_components(field, with_normals):
    f = _noise(128, 1.5, 1) if field == "noise128" else _fields()["shapes"]
    verts, faces, nrm = _gpu_mesh(f, None if field == "noise128" else 0.0, normals=True)
    nrm = nrm if with_normals else None
    out = ops.filter_components(verts, faces, 0.0, nrm)
    assert out[0] is verts and out[1] is faces and out[2] is nrm
    sizes = []
    for ratio in (0.0, 1e-4, 0.01, 0.3, 1.0):
        got = _check_filter(verts, faces, nrm, ratio)
        sizes.append(len(got[1]))
    assert sizes[0] == len(faces) and sizes[-1] > 0 and sizes == sorted(sizes, reverse=True) and sizes[-1] < sizes[1]
    # a vertex no face uses is dropped
    extra = torch.cat([verts, verts[:5]])
    got = _check_filter(extra, faces, None if nrm is None else torch.cat([nrm, nrm[:5]]), 1e-6)
    assert len(got[0]) <= len(verts)


def test_filter_empty_and_faceless_meshes():
    v0 = torch.zeros((0, 3), device="cuda")
    f0 = torch.zeros((0, 3), dtype=torch.int32, device="cuda")
    for v in (v0, torch.randn(10, 3, device="cuda")):
        got = ops.filter_components(v, f0, 0.5, v)
        assert all(t.shape == (0, 3) for t in got)
    assert ops.mesh_components(f0, 0).shape == (0,)
    assert ops.mesh_components(f0, 4).tolist() == [0, 1, 2, 3]


def test_bad_face_indices_raise_before_any_launch():
    verts = torch.randn(6, 3, device="cuda")
    for bad in ([[0, 1, 6]], [[0, -1, 2]], [[0, 1, 2], [3, 4, 2 ** 31 - 1]]):
        faces = torch.tensor(bad, dtype=torch.int32, device="cuda")
        with pytest.raises(RuntimeError, match="outside"):
            ops.mesh_components(faces, 6)
        with pytest.raises(RuntimeError, match="outside"):
            ops.filter_components(verts, faces, 0.5)
    with pytest.raises(RuntimeError, match="int32"):
        ops.mesh_components(torch.tensor([[0, 1, 2]], device="cuda"), 6)
    with pytest.raises(RuntimeError, match="int32"):
        ops.filter_components(verts, torch.tensor([0, 1, 2], dtype=torch.int32, device="cuda"), 0.5)
    torch.cuda.synchronize()


def _expected_filtered(full, ratio):
    """The oracle filter of the unfiltered call's (verts, faces, normals); the colours of the kept vertices ride along in the
    normals slot (uint8 -> float32 -> uint8 is exact)."""
    v, f, n, rgb = (t.cpu().numpy() for t in full)
    kv, kf, kn = cc.filter_components(v, f, ratio, n)
    _, _, krgb = cc.filter_components(v, f, ratio, rgb.astype(np.float32))
    return kv, kf, kn, krgb.astype(np.uint8)


def _check_filtered_export(out, expected, path):
    assert all(t.is_cuda for t in out)
    for got, ref in zip(out, expected):
        assert np.array_equal(got.cpu().numpy(), ref)
    lines, vrec, pf = read_ply(path)
    assert f"element vertex {len(expected[0])}" in lines and f"element face {len(expected[1])}" in lines
    assert np.array_equal(np.stack([vrec[c] for c in "xyz"], 1), expected[0]) and np.array_equal(pf, expected[1])
    assert np.array_equal(np.stack([vrec[c] for c in ("nx", "ny", "nz")], 1), expected[2])
    assert np.array_equal(np.stack([vrec[c] for c in ("red", "green", "blue")], 1), expected[3])


@pytest.mark.parametrize("kind,precision", [("nerf", "bf16"), ("nerf", "fp32"), ("siren", "bf16")])
def test_nerf_create_mesh_min_component_ratio(tmp_path, kind, precision):
    net = _seeded(kind)
    n, lo, hi = 80, (-1.5, -1.2, -1.0), (1.5, 1.3, 1.1)
    sigma, _, _ = nerf_render.density_lattice(net, lo, hi, n, max_batch=100000, precision=precision)
    thr = float(np.percentile(sigma.cpu().numpy(), 70))
    kw = dict(box_min=lo, box_max=hi, threshold=thr, precision=precision)
    full = nerf_render.create_mesh(net, None, n, **kw)
    labels = cc.component_labels(full[1].cpu().numpy(), len(full[0]))
    assert len(np.unique(labels)) > 2
    path = str(tmp_path / "filtered.ply")
    for ratio in (0.01, 1.0):
        out = nerf_render.create_mesh(net, path, n, min_component_ratio=ratio, **kw)
        expected = _expected_filtered(full, ratio)
        assert 0 < len(expected[1]) <= len(full[1]) and (ratio < 1 or len(expected[1]) < len(full[1]))
        _check_filtered_export(out, expected, path)
    with pytest.raises(ValueError):
        nerf_render.create_mesh(net, None, n, min_component_ratio=-0.5, **kw)


def test_pigan_create_mesh_min_component_ratio(tmp_path):
    torch.manual_seed(0)
    gen = models.Generator(256, 16).cuda()
    with torch.no_grad():
        net = gen.film_siren_nerf
        net.input_layer.weight.mul_(20.0)
        net.output_layer_sigma[0].weight.mul_(100.0)
        net.output_layer_sigma[0].bias.zero_()
    z = torch.randn(1, 256, generator=torch.Generator().manual_seed(3)).cuda()
    full = pigan_render.create_mesh(gen, None, N=96, z=z, normals=True, colors=True)
    path = str(tmp_path / "pigan.ply")
    for ratio in (0.05, 1.0):
        out = pigan_render.create_mesh(gen, path, N=96, z=z, normals=True, colors=True, min_component_ratio=ratio)
        expected = _expected_filtered(full, ratio)
        assert len(expected[1]) > 0
        _check_filtered_export(out, expected, path)
    plain = pigan_render.create_mesh(gen, None, N=96, z=z, min_component_ratio=1.0)
    kv, kf, _ = cc.filter_components(full[0].cpu().numpy(), full[1].cpu().numpy(), 1.0)
    assert len(plain) == 2 and np.array_equal(plain[0].cpu().numpy(), kv) and np.array_equal(plain[1].cpu().numpy(), kf)
