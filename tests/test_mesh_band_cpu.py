"""The narrow-band export's oracle (oracle/mesh_band.py) on hand cases, the band query's central property (the band field gives
the same masked mesh and normals as the full field), and the argument checks that run before any launch."""
import numpy as np
import pytest

from oracle import marching_cubes as mc
from oracle import mesh_attributes as ma
from oracle import mesh_band as mb


def _sphere(shape, r, centre=None, noise=0.0, seed=0):
    centre = [(n - 1) / 2 for n in shape] if centre is None else centre
    g = np.meshgrid(*[np.arange(n, dtype=np.float32) - np.float32(c) for n, c in zip(shape, centre)], indexing="ij")
    f = np.sqrt(g[0] * g[0] + g[1] * g[1] + g[2] * g[2]) - np.float32(r)
    if noise:
        f = f + np.float32(noise) * np.random.default_rng(seed).standard_normal(f.shape, dtype=np.float32)
    return f.astype(np.float32)


def _torus(shape, big, small):
    c = [(n - 1) / 2 for n in shape]
    g = np.meshgrid(*[np.arange(n, dtype=np.float32) - np.float32(cc) for n, cc in zip(shape, c)], indexing="ij")
    q = np.sqrt(g[0] * g[0] + g[1] * g[1]) - np.float32(big)
    return (np.sqrt(q * q + g[2] * g[2]) - np.float32(small)).astype(np.float32)


def _dense(field, level):
    v, f = mc.marching_cubes(field, level)
    return v, f, ma.vertex_normals(field, level)


def _equal(a, b):
    return len(a) == len(b) and all(np.array_equal(x, y) for x, y in zip(a, b))


def test_brick_geometry_with_a_partial_last_brick():
    assert mb.brick_dims((130, 130, 130), 8) == (17, 17, 17)            # 129 cells: 16 full bricks and one of 1 cell
    assert mb.brick_dims((129, 9, 2), 8) == (16, 1, 1)
    ax = mb.coarse_axes((130, 17, 5), 8)
    assert list(ax[0][-3:]) == [120, 128, 129] and list(ax[1]) == [0, 8, 16] and list(ax[2]) == [0, 4]


def test_single_sign_change_at_a_coarse_corner():
    f = np.ones((17, 17, 17), np.float32)
    f[8, 8, 8] = -1.0                                           # a coarse corner of the 8 bricks around it (stride 4)
    raw = mb.raw_flags(f, 0.0, 4)
    assert raw.shape == (4, 4, 4) and np.array_equal(np.argwhere(raw), np.argwhere(np.ones((2, 2, 2))) + 1)
    flags = mb.brick_flags(f, 0.0, 4)
    assert flags.sum() == 64                                    # dilated to every brick of the 4^3 box
    assert _equal(mb.masked_marching_cubes(f, 0.0, 4, flags, normals=True), _dense(f, 0.0))
    # the sign change seen by one cell only (not at a coarse corner): the coarse lattice misses it
    g = np.ones((17, 17, 17), np.float32)
    g[9, 9, 9] = -1.0
    assert not mb.brick_flags(g, 0.0, 4).any() and len(mc.marching_cubes(g, 0.0)[1]) > 0


def test_dilation_is_clamped_at_the_box():
    raw = np.zeros((5, 4, 6), bool)
    raw[0, 0, 0] = True
    assert np.array_equal(np.argwhere(mb.dilate(raw)), np.argwhere(np.ones((2, 2, 2))))
    raw[:] = False
    raw[4, 3, 5] = True
    assert np.array_equal(np.argwhere(mb.dilate(raw)), np.argwhere(np.ones((2, 2, 2))) + [3, 2, 4])


def test_band_points_closure_and_apron():
    flags = np.zeros((3, 3, 3), np.uint8)
    flags[1, 1, 1] = 1
    shape, stride = (13, 13, 13), 4
    idx = mb.band_points(flags, shape, stride)
    pts = np.stack(np.unravel_index(idx, shape), 1)
    inside = np.all((pts >= 4) & (pts <= 8), 1)                 # the brick's closure: points 4..8 on every axis
    steps = np.sum((pts < 4) | (pts > 8), 1)
    assert inside.sum() == 5 ** 3 and np.all(steps <= 1)
    assert np.all((pts >= 3) & (pts <= 9)) and len(idx) == 5 ** 3 + 6 * 5 ** 2
    assert np.all(np.diff(idx) > 0) and idx.dtype == np.int32


@pytest.mark.parametrize("shape,stride", [((130, 130, 130), 8), ((33, 20, 47), 4), ((40, 40, 40), 5)])
def test_band_field_gives_the_masked_mesh_of_the_full_field(shape, stride):
    r = min(shape) * 0.35
    for f in (_sphere(shape, r), _sphere(shape, r, noise=0.3, seed=2), _torus(shape, min(shape) * 0.3, min(shape) * 0.12)):
        band, flags = mb.band_field(f, 0.0, stride)
        assert np.array_equal(flags, mb.brick_flags(band, 0.0, stride))
        got = mb.masked_marching_cubes(band, 0.0, stride, flags, normals=True)
        assert _equal(got, mb.masked_marching_cubes(f, 0.0, stride, flags, normals=True))
        assert len(got[1]) > 100


@pytest.mark.parametrize("shape,stride", [((130, 130, 130), 8), ((33, 20, 47), 4)])
def test_smooth_surfaces_are_caught_whole(shape, stride):
    """A sphere and a torus that cross the coarse lattice everywhere: every dense triangle lies in a flagged brick."""
    for f in (_sphere(shape, min(shape) * 0.35), _torus(shape, min(shape) * 0.3, min(shape) * 0.12)):
        band, flags = mb.band_field(f, 0.0, stride)
        assert 0 < flags.sum() < flags.size
        assert _equal(mb.masked_marching_cubes(band, 0.0, stride, flags, normals=True), _dense(f, 0.0))


def test_all_flagged_is_dense_and_none_flagged_is_empty():
    f = _sphere((33, 20, 47), 7.0, noise=0.5, seed=1)
    dims = mb.brick_dims(f.shape, 4)
    assert _equal(mb.masked_marching_cubes(f, 0.0, 4, np.ones(dims, np.uint8), normals=True), _dense(f, 0.0))
    v, fa, n = mb.masked_marching_cubes(f, 0.0, 4, np.zeros(dims, np.uint8), normals=True)
    assert v.shape == (0, 3) and fa.shape == (0, 3) and n.shape == (0, 3)


def test_arbitrary_flags_keep_the_dense_order():
    f = _sphere((40, 40, 40), 14.0, noise=0.2, seed=3)
    flags = (np.random.default_rng(0).random(mb.brick_dims(f.shape, 4)) < 0.4).astype(np.uint8)
    v, fa = mb.masked_marching_cubes(f, 0.0, 4, flags)
    dv, df = mc.marching_cubes(f, 0.0)
    assert 0 < len(fa) < len(df)
    rows = {tuple(r): i for i, r in enumerate(dv)}               # sphere vertices are distinct: find each kept one
    at = np.array([rows[tuple(r)] for r in v])
    assert np.all(np.diff(at) > 0)
    assert {tuple(t) for t in at[fa]} <= {tuple(t) for t in df}


def test_a_small_sphere_inside_one_brick_is_missed():
    shape = (33, 33, 33)
    f = _sphere(shape, 2.0, centre=(12.0, 12.0, 12.0))          # inside brick (1, 1, 1) of stride 8, clear of its corners
    band, flags = mb.band_field(f, 0.0, 8)
    assert not flags.any() and len(mc.marching_cubes(f, 0.0)[1]) > 0
    assert len(mb.masked_marching_cubes(band, 0.0, 8, flags)[1]) == 0


def test_python_argument_checks_raise_before_any_launch():
    """The checks of ops, mesh and create_mesh that need no device: bad strides and narrow_band values are rejected first."""
    torch = pytest.importorskip("torch")
    from msra_practice_project_b200 import models, nerf_render, ops, pigan_render
    assert ops.brick_dims((130, 20, 2), 8) == (17, 3, 1) == mb.brick_dims((130, 20, 2), 8)
    net = models.NeRF()
    for bad in (0, 1, True, 2.0, 8.0, "8", -4):
        with pytest.raises(ValueError, match="narrow_band"):
            nerf_render.create_mesh(net, None, 16, narrow_band=bad)
        with pytest.raises(ValueError, match="narrow_band"):
            pigan_render.create_mesh(models.Generator(256, 16), None, N=16, narrow_band=bad)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.band_select(torch.zeros(4, 4, 4), 0.0, 2)
    with pytest.raises(RuntimeError, match="CUDA"):
        ops.marching_cubes(torch.zeros(4, 4, 4), 0.0, bricks=(2, torch.zeros(2, 2, 2, dtype=torch.uint8)))


def test_lattices_past_int32_are_rejected_on_the_host():
    """N^3 > 2^31 - 1 (N >= 1291) cannot take int32 point indices: both create_mesh raise before anything reaches a device."""
    from msra_practice_project_b200 import mesh, models, nerf_render, pigan_render
    mesh.check_band_lattice((1290, 1290, 1290))
    for dims in ((1291, 1291, 1291), (2 ** 16, 2 ** 16, 2)):
        with pytest.raises(RuntimeError, match="2\\^31 - 1"):
            mesh.check_band_lattice(dims)
    with pytest.raises(RuntimeError, match="2\\^31 - 1"):
        pigan_render.create_mesh(models.Generator(256, 16), None, N=1291, narrow_band=4)
    with pytest.raises(RuntimeError, match="2\\^31 - 1"):
        nerf_render.create_mesh(models.NeRF(), None, 1291, narrow_band=4)
