"""Texture baking on the device against the numpy oracle (oracle/mesh_texture.py), bit for bit: the atlas rows and UVs of
marching-cubes meshes of sphere / torus fields, a decimated mesh, one face, an odd face count and the smallest cells (s = 4);
the baked texture against to8b of the MLP on the oracle's rows placed by the oracle's layout; and create_mesh(texture=...) of
NeRF, SirenNeRF and pi-GAN, alone and with min_component_ratio, smooth_iterations and max_faces: the mesh, normals and colours
are those of the call without it, and the PLY and PNG round-trip."""
import functools
import os

import numpy as np
import pytest
import torch

from msra_practice_project_b200 import mesh, nerf_render, ops, pigan_render
from oracle import marching_cubes as mc
from oracle import mesh_decimation as md
from oracle import mesh_smoothing as sm
from oracle import mesh_texture as mt

from test_gpu_mesh import _generator
from test_gpu_mesh_export import _seeded
from test_mesh_components_cpu import BIG, SMALL, TORUS, _union
from test_mesh_texture_cpu import _decode_png

pytestmark = pytest.mark.gpu


@functools.lru_cache(maxsize=None)
def _meshes():
    shapes = _union(BIG, TORUS, *SMALL)
    v, f = mc.marching_cubes(shapes, 0.0)
    tv, tf = mc.marching_cubes(TORUS, 0.0)
    dv, df = md.decimate(v, f, len(f) // 7)
    return {"shapes": (v, f), "torus": (tv, tf), "decimated": (dv, df), "one_face": (v, f[:1]), "odd": (tv, tf[:len(tf) // 2 * 2 - 1])}


def _rows_device(v, f, n, size, batches=1):
    vd, fd, nd = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (v, f, n))
    cells, _, s = ops.atlas_layout(len(f), size)
    total = cells * s * s
    cuts = np.linspace(0, total, batches + 1).astype(int)
    return torch.cat([ops._atlas_rows(vd, fd, nd, size, int(a), int(b - a)) for a, b in zip(cuts[:-1], cuts[1:])])


@pytest.mark.parametrize("name", ["shapes", "torus", "decimated", "one_face", "odd"])
@pytest.mark.parametrize("size", [16, 512, 2048])
def test_rows_and_uvs_equal_the_oracle(name, size):
    v, f = _meshes()[name]
    f = np.ascontiguousarray(f, np.int32)
    if len(f) > 2 * (size // 4) ** 2:
        f = f[:2 * (size // 4) ** 2]                                  # s = 4: the smallest cells
        assert ops.atlas_layout(len(f), size)[2] == 4
    n = sm.mesh_normals(v, f)
    ref = mt.rows(v, f, n, size)
    for batches in (1, 3):
        got = _rows_device(v, f, n, size, batches).cpu().numpy()
        assert got.shape == ref.shape and np.array_equal(got.view(np.uint32), ref.view(np.uint32)), (name, size, batches)
    uv = ops._atlas_uvs(len(f), size, torch.device("cuda")).cpu().numpy()
    assert np.array_equal(uv.view(np.uint32), mt.uvs(len(f), size).view(np.uint32))


@pytest.mark.parametrize("kind", ["nerf", "siren", "pigan"])
@pytest.mark.parametrize("size,max_batch", [(256, 256 ** 3), (256, 4099), (64, 1000)])
def test_texture_is_the_mlp_on_the_oracle_rows(kind, size, max_batch):
    if kind == "pigan":
        gen, z = _generator()
        model = gen.film_siren_nerf
        with torch.no_grad():
            gen.set_film_params(gen.get_mapping(z)[0])
    else:
        model = _seeded(kind)
    v, f = _meshes()["torus"]
    scale = 0.2 / 64 if kind == "pigan" else 3.0 / 64
    v = ((v - 32.0) * np.float32(scale)).astype(np.float32)
    f = np.ascontiguousarray(f[:2 * (size // 4) ** 2], np.int32)
    n = sm.mesh_normals(v, f)
    uvs, tex = mesh.bake_texture(model, torch.from_numpy(v).cuda(), torch.from_numpy(f).cuda(), torch.from_numpy(n).cuda(), size,
                                 max_batch=max_batch)
    assert uvs.is_cuda and tex.is_cuda and tex.dtype == torch.uint8 and tuple(tex.shape) == (size, size, 3)
    with torch.no_grad():
        raw = ops.mlp(model, x=torch.from_numpy(mt.rows(v, f, n, size)).cuda())
    rgb = ops.to8b(raw[:, :3]).cpu().numpy()
    assert np.array_equal(rgb, mt.to8b(raw[:, :3].cpu().numpy()))
    assert np.array_equal(tex.cpu().numpy(), mt.texture(rgb, len(f), size))
    assert np.array_equal(uvs.cpu().numpy(), mt.uvs(len(f), size))
    assert tex.cpu().numpy().any()


def test_bake_texture_argument_checks():
    net = _seeded("nerf")
    v = torch.rand(10, 3, device="cuda")
    f = torch.tensor([[0, 1, 2], [2, 3, 4]], dtype=torch.int32, device="cuda")
    with pytest.raises(RuntimeError, match="outside"):
        mesh.bake_texture(net, v, torch.tensor([[0, 1, 10]], dtype=torch.int32, device="cuda"), v, 16)
    with pytest.raises(RuntimeError, match="normals"):
        mesh.bake_texture(net, v, f, None, 16)
    with pytest.raises(RuntimeError):
        mesh.bake_texture(net, v.cpu(), f, v, 16)
    for bad in (15, 16385, 16.0, None):
        with pytest.raises(ValueError):
            mesh.bake_texture(net, v, f, v, bad)
    many = torch.zeros((33, 3), dtype=torch.int32, device="cuda")
    with pytest.raises(ValueError, match="at most 32"):
        mesh.bake_texture(net, v, many, v, 16)
    uvs, tex = mesh.bake_texture(net, v, f[:0], v, 16)                          # no faces: an empty atlas
    assert uvs.shape == (0, 3, 2) and not tex.any()


def _check_textured(out, plain, model, size, used_normals, path=None):
    """``out`` = plain + (uvs, texture), the texture baked on the final mesh along ``used_normals``; the files round-trip."""
    assert len(out) == len(plain) + 2
    for a, b in zip(out, plain):
        assert (a is None and b is None) or torch.equal(a, b)
    uvs, tex = mesh.bake_texture(model, out[0], out[1], used_normals, size)
    assert torch.equal(out[-2], uvs) and torch.equal(out[-1], tex)
    if path is None:
        return
    png = os.path.splitext(path)[0] + ".png"
    assert np.array_equal(_decode_png(png), tex.cpu().numpy())
    data = open(path, "rb").read()
    end = data.index(b"end_header\n") + len(b"end_header\n")
    lines = data[:end].decode("ascii").splitlines()
    assert lines[2] == f"comment TextureFile {os.path.basename(png)}" and "property list uchar float texcoord" in lines
    nf = out[1].shape[0]
    frec = np.frombuffer(data[len(data) - nf * 38:], dtype=[("n", "u1"), ("vi", "<i4", (3,)), ("nt", "u1"), ("uv", "<f4", (6,))])
    assert np.array_equal(frec["vi"], out[1].cpu().numpy()) and np.array_equal(frec["uv"], out[-2].cpu().numpy().reshape(-1, 6))


@pytest.mark.parametrize("kind", ["nerf", "siren"])
def test_nerf_create_mesh_texture(tmp_path, kind):
    net = _seeded(kind)
    n, lo, hi = 64, (-1.5, -1.2, -1.0), (1.5, 1.3, 1.1)
    sigma, _, _ = nerf_render.density_lattice(net, lo, hi, n, max_batch=100000)
    thr = float(np.percentile(sigma.cpu().numpy(), 70))
    kw = dict(box_min=lo, box_max=hi, threshold=thr, max_batch=300000)
    path = str(tmp_path / "m.ply")
    for extra in ({}, {"min_component_ratio": 0.01}, {"smooth_iterations": 3}, {"max_faces": 4000},
                  {"min_component_ratio": 0.01, "smooth_iterations": 3, "max_faces": 4000}):
        plain = nerf_render.create_mesh(net, None, n, **kw, **extra)
        size = 2048 if len(plain[1]) > 2 * 256 ** 2 else 1024
        out = nerf_render.create_mesh(net, path, n, texture=size, **kw, **extra)
        _check_textured(out, plain, net, size, plain[2], path)
    # without normals and colours the texture still uses the normals the colour query would use
    plain = nerf_render.create_mesh(net, None, n, max_faces=4000, **kw)
    out = nerf_render.create_mesh(net, None, n, normals=False, colors=False, max_faces=4000, texture=512, **kw)
    assert out[2] is None and out[3] is None
    _check_textured(out, (plain[0], plain[1], None, None), net, 512, plain[2])
    with pytest.raises(ValueError, match="at most 32"):
        nerf_render.create_mesh(net, None, n, texture=16, **kw)


def test_pigan_create_mesh_texture(tmp_path):
    gen, z = _generator()
    path = str(tmp_path / "pigan.ply")
    for extra in ({}, {"min_component_ratio": 0.05, "smooth_iterations": 5, "max_faces": 3000}):
        plain = pigan_render.create_mesh(gen, None, N=96, z=z, normals=True, colors=True, **extra)
        out = pigan_render.create_mesh(gen, path, N=96, z=z, normals=True, colors=True, texture=2048, **extra)
        _check_textured(out, plain, gen.film_siren_nerf, 2048, plain[2], path)
        only = pigan_render.create_mesh(gen, None, N=96, z=z, texture=2048, **extra)
        assert len(only) == 6 and only[2] is None and only[3] is None
        assert all(torch.equal(a, b) for a, b in zip(only[:2] + only[4:], out[:2] + out[4:]))
    assert len(pigan_render.create_mesh(gen, None, N=96, z=z)) == 2
