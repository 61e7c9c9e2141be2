"""GPU parity tests: every CUDA stage of the render path, called through the C ABI (ctypes ->
libb2r.so), against the golden outputs of the unmodified reference (tests/golden/*.npz) and the
numpy oracle on the same seeded inputs.  Tolerances are the ones BASELINE.json's north_star states:
bit-exact sample_pdf given identical CDFs, <= 1e-4 max-abs for fp32 stages, <= 2e-2 for the bf16 MLP.
"""
import os
import subprocess

import numpy as np
import pytest
import torch

from oracle import render_oracle as orc
from msra_practice_project_b200 import models, nerf_render, ops, pigan_render

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def cu(a):
    return torch.as_tensor(np.ascontiguousarray(a)).cuda()


def seeded_nerf():
    torch.manual_seed(0)
    return models.NeRF().cuda(), models.NeRF().cuda()


@pytest.fixture
def exact_grads():
    """gradient fixtures hold the reference's fp32 autograd results: check them on the exact (fp32 CUDA-core) reverse mode"""
    old = ops.set_grad_precision("fp32")
    yield
    ops.set_grad_precision(old)


def seeded_film(use_dir=True):
    torch.manual_seed(0)
    return models.FilmSirenNeRF(use_dir=use_dir).cuda()


def test_library_loaded_and_device_ok():
    from msra_practice_project_b200 import _lib
    assert _lib.lib().b2r_version() == 100
    assert _lib.lib().b2r_device_ok() == 1, "not a compute-capability 10.x device"


def test_umma_probe():
    """Hardware probe of the tcgen05 / swizzle / bulk-copy primitives (tests/native/umma_probe.cu)."""
    exe = os.path.join(ROOT, "tests", "native", "umma_probe")
    if not os.path.exists(exe):
        pytest.skip("probe binary not built")
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    print(out.stdout)
    assert "PROBE OK" in out.stdout, out.stdout + out.stderr
    # the encoding the product uses (first two cases) must be the one that matches
    lines = [l for l in out.stdout.splitlines() if l.startswith("PROBE A=")]
    assert "mismatches 0 " in lines[0] and "mismatches 0 " in lines[1], out.stdout


def test_umma_kmajor_noswizzle_probe():
    """The no-swizzle K-major operand layout of the sine models' compact aux / post chunks (tc_core.cuh MapC): LBO = pitch of the two
    16-byte K chunks, SBO = pitch of the 8-row groups, and the mix with a SWIZZLE_128B A operand."""
    exe = os.path.join(ROOT, "tests", "native", "umma_kmajor_noswizzle_probe")
    if not os.path.exists(exe):
        pytest.skip("probe binary not built")
    out = subprocess.run([exe], capture_output=True, text=True, timeout=120)
    print(out.stdout)
    assert "PROBE OK" in out.stdout, out.stdout + out.stderr
    ok = [l for l in out.stdout.splitlines() if "<-- OK" in l]
    assert len(ok) == 2 and all("LBO=2048 SBO=128" in l for l in ok), out.stdout        # the assignment the kernels use


# ---- K1 / K2 -------------------------------------------------------------------------------------------
def test_raygen(golden):
    k = golden.kernels
    rays = ops.raygen(20, 12, 20 * 1.3875, k["rays_c2w"]).cpu().numpy().reshape(12, 20, 2, 3)
    assert np.array_equal(rays[:, :, 0], k["rays_o_20x12"])
    np.testing.assert_allclose(rays[:, :, 1], k["rays_d_20x12"], rtol=0, atol=1.2e-7)
    assert np.mean(rays[:, :, 1] == k["rays_d_20x12"]) > 0.99
    f64 = np.float64(9 / 2 / np.tan(6 * np.pi / 180))
    r2 = ops.raygen(9, 7, f64, k["rays_c2w"]).cpu().numpy().reshape(7, 9, 2, 3)
    assert np.array_equal(r2[:, :, 1], k["rays_d_9x7_f64focal"].astype(np.float32))
    # a sub-range equals the slice of the full table
    part = ops.raygen(20, 12, 20 * 1.3875, k["rays_c2w"], begin=33, count=50).cpu().numpy()
    assert np.array_equal(part, rays.reshape(-1, 2, 3)[33:83])
    # get_rays drop-in
    o, d = nerf_render.get_rays(20, 12, 20 * 1.3875, k["rays_c2w"])
    assert o.shape == (12, 20, 3) and np.array_equal(d, rays[:, :, 1])


def test_stratified_z_bit_exact(golden):
    s = golden.nerf_stages
    z, mids = ops.stratified_z(cu(s["z_lin"]), cu(s["t_rand"]))
    assert np.array_equal(z.cpu().numpy(), s["z_coarse"])
    assert np.array_equal(mids.cpu().numpy(), s["mids"])


# ---- K4 -----------------------------------------------------------------------------------------------------
def test_composite_forward(golden):
    k = golden.kernels
    rgb, depth, acc, w = ops.composite(cu(k["c_raw"]), cu(k["c_z"]), cu(k["c_dirs"]))
    np.testing.assert_allclose(w.cpu().numpy(), k["c_w"], atol=1e-5, rtol=0)
    np.testing.assert_allclose(rgb.cpu().numpy(), k["c_rgb"], atol=1e-5, rtol=0)
    np.testing.assert_allclose(depth.cpu().numpy(), k["c_depth"], atol=1e-4, rtol=0)
    np.testing.assert_allclose(acc.cpu().numpy(), k["c_acc"], atol=1e-5, rtol=0)
    # without weights, strided directions (rays[:,1] of an [N,2,3] table)
    rays = torch.zeros(37, 2, 3, device="cuda"); rays[:, 1] = cu(k["c_dirs"])
    rgb2, depth2, acc2, w2 = ops.composite(cu(k["c_raw"]), cu(k["c_z"]), rays[:, 1], want_weights=False)
    assert w2 is None and torch.equal(rgb2, rgb) and torch.equal(depth2, depth) and torch.equal(acc2, acc)


def test_composite_kats():
    n, s = 5, 192
    z = torch.linspace(2, 6, s).expand(n, s).contiguous().cuda()
    d = torch.tensor([[0., 0., -1.]]).expand(n, 3).contiguous().cuda()
    raw = torch.rand(n, s, 4, device="cuda"); raw[..., 3] = 0
    rgb, depth, acc, w = ops.composite(raw, z, d)                  # sigma == 0 -> white, empty
    assert torch.all(w == 0) and torch.all(acc == 0) and torch.all(depth == 0) and torch.all(rgb == 1)
    c = 0.7
    raw[..., 3] = c                                                  # constant sigma -> closed form
    rgb, depth, acc, w = ops.composite(raw, z, d)
    delta = float(z[0, 1] - z[0, 0])
    k = np.arange(s)
    w_ref = (1 - np.exp(-c * delta)) * np.exp(-c * delta * k)
    w_ref[-1] = np.exp(-c * delta * (s - 1))
    np.testing.assert_allclose(w[0].cpu().numpy(), w_ref, atol=2e-6)
    np.testing.assert_allclose(acc.cpu().numpy(), 1.0, atol=1e-5)


def test_composite_backward(golden):
    k = golden.kernels
    raw = cu(k["c_raw"]).requires_grad_(True)
    rgb, depth, acc, _ = ops.composite(raw, cu(k["c_z"]), cu(k["c_dirs"]))
    loss = (rgb * cu(k["c_g_rgb"])).sum() + (depth * cu(k["c_g_depth"])).sum() + (acc * cu(k["c_g_acc"])).sum()
    (d_raw,) = torch.autograd.grad(loss, raw)
    ref = k["c_d_raw"].astype(np.float64)
    got = d_raw.cpu().numpy().astype(np.float64)
    scale = np.maximum(1.0, np.abs(ref))        # last-sample d sigma is O(1e10) when sigma == 0: relative there
    assert np.max(np.abs(got - ref) / scale) < 1e-4
    want = orc.raw_to_outputs_backward(k["c_raw"], k["c_z"], k["c_dirs"], k["c_g_rgb"], k["c_g_depth"], k["c_g_acc"])
    assert np.max(np.abs(got - want) / np.maximum(1.0, np.abs(want))) < 1e-4


@pytest.mark.parametrize("s", [1, 31, 64, 100, 192, 384])
def test_composite_ragged_sizes_vs_oracle(s):
    g = torch.Generator().manual_seed(s)
    n = 33
    raw = torch.rand(n, s, 4, generator=g); raw[..., 3] = torch.relu(torch.randn(n, s, generator=g)) * 4
    z = torch.sort(torch.rand(n, s, generator=g) * 4 + 2, -1).values
    d = torch.randn(n, 3, generator=g)
    rgb, depth, acc, w = ops.composite(raw.cuda(), z.cuda(), d.cuda())
    r_rgb, r_depth, r_acc, r_w = orc.raw_to_outputs(raw.numpy(), z.numpy(), d.numpy())
    np.testing.assert_allclose(w.cpu().numpy(), r_w, atol=1e-5)
    np.testing.assert_allclose(rgb.cpu().numpy(), r_rgb, atol=1e-5)
    np.testing.assert_allclose(depth.cpu().numpy(), r_depth, atol=1e-4)
    gr, gd, ga = torch.randn(n, 3, generator=g), torch.randn(n, generator=g), torch.randn(n, generator=g)
    rawg = raw.cuda().requires_grad_(True)
    o = ops.composite(rawg, z.cuda(), d.cuda())
    ((o[0] * gr.cuda()).sum() + (o[1] * gd.cuda()).sum() + (o[2] * ga.cuda()).sum()).backward()
    want = orc.raw_to_outputs_backward(raw.numpy(), z.numpy(), d.numpy(), gr.numpy(), gd.numpy(), ga.numpy())
    got = rawg.grad.cpu().numpy().astype(np.float64)
    assert np.max(np.abs(got - want) / np.maximum(1.0, np.abs(want))) < 2e-4


# ---- K5 / K6 -------------------------------------------------------------------------------------------------
def _check_pdf(bins, w, u, ref_out, atol):
    res = ops.sample_pdf(cu(bins), cu(w), len(u), u=cu(u), want_cdf=True)
    got, cdf = res["samples"].cpu().numpy(), res["cdf"].cpu().numpy()
    # (1) bit-exact GIVEN the CDF: rerun the reference's post-CDF arithmetic on the kernel's CDF
    want, inds = orc.sample_pdf_from_cdf(bins, cdf, u)
    assert np.array_equal(got, want), "samples differ from the reference arithmetic on the same CDF"
    # (2) the CDF itself agrees with the reference CDF to float rounding, and so do the samples
    _, cdf_ref, _ = orc.sample_pdf(bins, w, len(u), u=u, return_cdf=True)
    np.testing.assert_allclose(cdf, cdf_ref, atol=2.5e-7, rtol=0)
    tol = orc.sample_pdf_tolerance(bins, w, u)
    err = np.abs(got.astype(np.float64) - ref_out)
    assert np.all(err <= np.maximum(tol, atol)), float(np.max(err))
    return got


def test_sample_pdf_golden(golden):
    k = golden.kernels
    _check_pdf(k["sp_bins"], k["sp_w"], k["sp_u"], k["sp_out"], 1e-6)
    _check_pdf(k["sp2_bins"], k["sp2_w"], k["sp2_u"], k["sp2_out"], 4e-6)      # per-ray bins
    s = golden.nerf_stages
    _check_pdf(s["mids"], s["weights_coarse"][:, 1:-1], s["u"], s["z_samples"], 2e-6)


def test_sample_pdf_kats_and_merge(golden):
    bins = np.linspace(2, 6, 33, dtype=np.float32)
    u = orc.linspace_f32(0, 1, 17)
    z = ops.sample_pdf(cu(bins), torch.ones(3, 32).cuda(), 17, u=cu(u))["samples"].cpu().numpy()
    np.testing.assert_allclose(z[0], bins[0] + u * (bins[-1] - bins[0]), atol=2e-6)
    assert np.all(z[:, 0] == bins[0])                                     # u = 0 -> bins[0] exactly
    s = golden.nerf_stages
    w = cu(s["weights_coarse"])
    res = ops.sample_pdf(cu(s["mids"]), w[:, 1:-1], int(s["Sf"]), u=cu(s["u"]), z_coarse=cu(s["z_coarse"]))
    zs, merged = res["samples"].cpu().numpy(), res["sorted"].cpu().numpy()
    assert np.array_equal(merged, np.sort(np.concatenate([s["z_coarse"], zs], -1), -1))
    assert np.all(np.diff(merged, axis=-1) >= 0)
    # strided weights view == contiguous copy
    res2 = ops.sample_pdf(cu(s["mids"]), w[:, 1:-1].contiguous(), int(s["Sf"]), u=cu(s["u"]))
    assert np.array_equal(res2["samples"].cpu().numpy(), zs)


# ---- K3 fp32 --------------------------------------------------------------------------------------------------
def test_mlp_fp32_nerf(golden):
    k = golden.kernels
    c, f = seeded_nerf()
    with torch.no_grad():
        out_c = ops.mlp(c, x=cu(k["mlp_x"]), precision="fp32").cpu().numpy()
        out_f = f(cu(k["mlp_x"]))          # module call -> ops.mlp_points (default precision applies)
        out_f32 = ops.mlp(f, x=cu(k["mlp_x"]), precision="fp32").cpu().numpy()
    np.testing.assert_allclose(out_c, k["nerf_seed0_coarse_out"], atol=1e-4, rtol=0)
    np.testing.assert_allclose(out_f32, k["nerf_seed0_fine_out"], atol=1e-4, rtol=0)
    assert out_f.shape == (96, 4)


def test_mlp_fp32_film_and_grid(golden):
    k = golden.kernels
    m = seeded_film()
    m.set_film_params(cu(k["film_params"]))
    with torch.no_grad():
        out = ops.mlp(m, x=cu(k["film_x"]), precision="fp32").cpu().numpy()
    np.testing.assert_allclose(out, k["film_seed0_out"], atol=1e-4, rtol=0)
    p = golden.pigan
    m.set_film_params(cu(p["film"]))
    neg = pigan_render.density_grid(m, int(p["grid_N"]), max_batch=100, precision="fp32").cpu().numpy()
    np.testing.assert_allclose(neg, p["grid_neg_sigma"], atol=1e-4, rtol=0)
    with pytest.raises(ValueError):
        models.FilmSirenNeRF().cuda()(cu(k["film_x"]))           # film params unset (pi_GAN/modules.py:107)


def test_mlp_rays_mode_matches_points_mode(golden):
    s = golden.nerf_stages
    c, _ = seeded_nerf()
    with torch.no_grad():
        raw = ops.mlp(c, rays=cu(s["rays"]), z=cu(s["z_coarse"]), precision="fp32").view(144, 64, 4).cpu().numpy()
    np.testing.assert_allclose(raw, s["raw_coarse"], atol=1e-4, rtol=0)


def test_render_rays_fp32_staged(golden):
    """Teacher-forced per stage (the end-to-end map is chaotic on Xavier weights, SURVEY 7.3-2)."""
    s = golden.nerf_stages
    c, f = seeded_nerf()
    st = {}
    with torch.no_grad():
        out = nerf_render.render_rays(cu(s["rays"]), 2.0, 6.0, c, f, 64, 64, t_rand=cu(s["t_rand"]), z_lin=s["z_lin"],
                                      u=s["u"], precision="fp32", stages=st)
    assert np.array_equal(st["z_coarse"].cpu().numpy(), s["z_coarse"])
    np.testing.assert_allclose(st["raw_coarse"].cpu().numpy(), s["raw_coarse"], atol=1e-4, rtol=0)
    np.testing.assert_allclose(st["weights_coarse"].cpu().numpy(), s["weights_coarse"], atol=1e-4, rtol=0)
    np.testing.assert_allclose(out[0].cpu().numpy(), s["rgb_c"], atol=1e-4, rtol=0)
    np.testing.assert_allclose(out[2].cpu().numpy(), s["acc_c"], atol=1e-4, rtol=0)
    # fine pass, teacher-forced with the reference's z_fine
    with torch.no_grad():
        raw_f = ops.mlp(f, rays=cu(s["rays"]), z=cu(s["z_fine"]), precision="fp32").view(144, 128, 4)
        rgb_f, depth_f, acc_f, w_f = ops.composite(raw_f, cu(s["z_fine"]), cu(s["rays"])[:, 1])
    np.testing.assert_allclose(raw_f.cpu().numpy(), s["raw_fine"], atol=1e-4, rtol=0)
    np.testing.assert_allclose(rgb_f.cpu().numpy(), s["rgb_f"], atol=1e-4, rtol=0)
    np.testing.assert_allclose(depth_f.cpu().numpy(), s["depth_f"], atol=1e-4, rtol=0)
    np.testing.assert_allclose(w_f.cpu().numpy(), s["weights_fine"], atol=1e-4, rtol=0)


# ---- K3 bf16 tensor-core --------------------------------------------------------------------------------------
def test_mlp_tc_nerf_vs_reference(golden):
    k, s = golden.kernels, golden.nerf_stages
    c, f = seeded_nerf()
    with torch.no_grad():
        out = ops.mlp(c, x=cu(k["mlp_x"]), precision="bf16").cpu().numpy()
    ref = k["nerf_seed0_coarse_out"]
    err = np.abs(out - ref)
    print("bf16 MLP max-abs rgb %.4g sigma %.4g" % (err[:, :3].max(), err[:, 3].max()))
    # rgb is bounded (sigmoid): absolute 2e-2.  sigma is an unbounded relu output that only acts through
    # alpha = 1 - exp(-sigma * dist) with dist ~ 0.03..0.06: 4e-2 relative to max(1, sigma) moves alpha by < 3e-3
    assert err[:, :3].max() < 2e-2 and np.all(err[:, 3] < 4e-2 * np.maximum(1.0, ref[:, 3]))
    with torch.no_grad():
        raw = ops.mlp(f, rays=cu(s["rays"]), z=cu(s["z_fine"]), precision="bf16").view(144, 128, 4).cpu().numpy()
    err = np.abs(raw - s["raw_fine"])
    print("bf16 MLP (rays mode, 18432 rows) max-abs rgb %.4g sigma %.4g" % (err[..., :3].max(), err[..., 3].max()))
    assert err[..., :3].max() < 2e-2 and np.all(err[..., 3] < 4e-2 * np.maximum(1.0, s["raw_fine"][..., 3]))
    # and the composited outputs (what north_star bounds: rgb / depth / weights), teacher-forced on z_fine
    with torch.no_grad():
        rgb, depth, acc, w = ops.composite(cu(raw), cu(s["z_fine"]), cu(s["rays"])[:, 1])
    e_rgb = np.abs(rgb.cpu().numpy() - s["rgb_f"]).max(axis=-1)
    e_w = np.abs(w.cpu().numpy() - s["weights_fine"]).max(axis=-1)
    print("  composited: rays with rgb err > 2e-2: %d / 144 (max %.3g), weights err max %.3g" % ((e_rgb > 2e-2).sum(), e_rgb.max(), e_w.max()))
    # rays mode runs the last-sample sign check (ops._EXACT_LAST): EVERY ray -- including the last interval, whose alpha is a step
    # function of sign(sigma_last) (SURVEY 0) -- is within the north_star bound of the reference's golden
    assert np.abs(w.cpu().numpy() - s["weights_fine"]).max() < 2e-2
    assert (e_rgb > 2e-2).sum() == 0
    with torch.no_grad():
        raw0 = ops.mlp(f, rays=cu(s["rays"]), z=cu(s["z_fine"]), precision="bf16", exact_last_sample=False).view(144, 128, 4)
        rgb0 = ops.composite(raw0, cu(s["z_fine"]), cu(s["rays"])[:, 1])[0]
    print("  without the check: rays with rgb err > 2e-2: %d / 144" % int((np.abs(rgb0.cpu().numpy() - s["rgb_f"]).max(axis=-1) > 2e-2).sum()))


@pytest.mark.parametrize("rows", [1, 127, 128, 129, 255, 256, 257, 1000, 40000])
def test_mlp_tc_ragged_rows_vs_fp32(rows):
    c, _ = seeded_nerf()
    g = torch.Generator().manual_seed(rows)
    x = torch.cat([torch.rand(rows, 3, generator=g) * 8 - 4,
                   torch.nn.functional.normalize(torch.randn(rows, 3, generator=g), dim=-1)], -1).cuda()
    with torch.no_grad():
        a = ops.mlp(c, x=x, precision="bf16")
        b = ops.mlp(c, x=x, precision="fp32")
    assert torch.isfinite(a).all()
    err = (a - b).abs()
    assert err[:, :3].max().item() < 2e-2
    assert bool(torch.all(err[:, 3] < 4e-2 * torch.clamp(b[:, 3], min=1.0)))


def test_packed_blob_area_matches_chunk_area():
    """The sine models' packed images carry every step's LAST h chunk and post chunk twice: in the chunk area (SWIZZLE_128B images, read by
    the training kernels) and as one blob per step and N-half behind the fp32 tables ([h chunk 3 | post chunk in the no-swizzle layout
    [16-byte K chunk][weight row][16 B]], read by the inference kernels with one bulk copy: tc_core.cuh extra_base / MapC).  Both must hold
    the same bf16 values."""
    import numpy as np
    torch.manual_seed(3)
    film_net = models.FilmSirenNeRF().cuda()
    g = torch.Generator().manual_seed(1)
    film_net.set_film_params(torch.cat([1.0 + 0.2 * torch.randn(9, 256, generator=g), 0.1 * torch.randn(9, 256, generator=g)], -1).cuda())
    siren_net = models.SirenNeRF().cuda()
    cases = [(models.KIND_FILM, film_net, models.film_tensor(film_net).contiguous(), [256] * 8, 2308),
             (models.KIND_SIREN, siren_net, None, [256] * 8 + [128], 1668)]

    def sw128(row, chunk16):
        return (row >> 3) * 1024 + (row & 7) * 128 + ((chunk16 ^ (row & 7)) << 4)

    for kind, net, film, n_of, tab_floats in cases:
        packed = ops.pack_tc(models.flat_params(net, kind), kind, film=film).cpu().numpy()
        hb = [n // 2 * 128 for n in n_of]                          # half-chunk image: n/2 weight rows x 64 K bf16
        pb = [n // 2 * 32 for n in n_of]                           # compact post chunk: n/2 rows x 16 K bf16
        step_base = np.concatenate([[0], np.cumsum([2 * 5 * h for h in hb])])
        extra_off = int(step_base[-1]) + tab_floats * 4
        extra_base = np.concatenate([[0], np.cumsum([2 * (h + q) for h, q in zip(hb, pb)])])
        assert packed.size == extra_off + int(extra_base[-1])
        for s in range(len(n_of)):
            rows = n_of[s] // 2
            for hf in range(2):
                blob = packed[extra_off + int(extra_base[s]) + hf * (hb[s] + pb[s]):][:hb[s] + pb[s]]
                chunk3 = packed[int(step_base[s]) + (3 * 2 + hf) * hb[s]:][:hb[s]]
                post = packed[int(step_base[s]) + (4 * 2 + hf) * hb[s]:][:hb[s]]
                assert np.array_equal(blob[:hb[s]], chunk3), (kind, s, hf)
                for c2 in range(2):
                    for row in range(rows):
                        a = blob[hb[s] + c2 * (pb[s] // 2) + row * 16:][:16]
                        b = post[sw128(row, c2):][:16]
                        assert np.array_equal(a, b), (kind, s, hf, c2, row)
                # the post chunk uses only its first 16 K columns: the rest of the SWIZZLE_128B image is zero
                used = np.zeros(hb[s], dtype=bool)
                for row in range(rows):
                    for c2 in range(2):
                        used[sw128(row, c2):sw128(row, c2) + 16] = True
                assert not post[~used].any(), (kind, s, hf)


def test_mlp_tc_film_vs_reference(golden):
    """FiLM-SIREN on the tensor-core path: points mode, sigma-only grid mode, use_dir=False, film update."""
    k, p = golden.kernels, golden.pigan
    m = seeded_film()
    m.set_film_params(cu(k["film_params"]))
    with torch.no_grad():
        out = ops.mlp(m, x=cu(k["film_x"]), precision="bf16").cpu().numpy()
    ref = k["film_seed0_out"]
    err = np.abs(out - ref)
    print("bf16 FiLM-SIREN max-abs rgb %.4g sigma %.4g (sigma max %.3g)" % (err[:, :3].max(), err[:, 3].max(), ref[:, 3].max()))
    assert err[:, :3].max() < 2e-2 and np.all(err[:, 3] < 4e-2 * np.maximum(1.0, ref[:, 3]))
    m.set_film_params(cu(p["film"]))                      # new FiLM tensor -> packed tables must be rebuilt
    n = int(p["grid_N"])
    neg = pigan_render.density_grid(m, n, max_batch=100, precision="bf16").cpu().numpy()
    assert np.all(np.abs(neg - p["grid_neg_sigma"]) < 4e-2 * np.maximum(1.0, -p["grid_neg_sigma"]))
    m2 = seeded_film(use_dir=False)
    m2.set_film_params(cu(k["film_params"]))
    g = torch.Generator().manual_seed(3)
    x = torch.cat([torch.rand(700, 3, generator=g) * 0.6 - 0.3, torch.nn.functional.normalize(torch.randn(700, 3, generator=g), dim=-1)], -1).cuda()
    with torch.no_grad():
        a = ops.mlp(m2, x=x, precision="bf16")
        b = ops.mlp(m2, x=x, precision="fp32")
    e = (a - b).abs()
    assert e[:, :3].max().item() < 2e-2 and bool(torch.all(e[:, 3] < 4e-2 * torch.clamp(b[:, 3], min=1.0)))


def test_pigan_render_bf16_vs_fp32(golden):
    p = golden.pigan
    m = seeded_film()
    m.set_film_params(cu(p["film"]))
    w = 32
    focal = np.float64(w / 2 / np.tan(6 * np.pi / 180))
    torch.manual_seed(3)
    t = torch.rand(w * w, 24, device="cuda")
    a = pigan_render.render_image_np(w, w, focal, p["pose"], 0.5, 1.5, m, m, 24, 24, t_rand=t, precision="fp32")
    b = pigan_render.render_image_np(w, w, focal, p["pose"], 0.5, 1.5, m, m, 24, 24, t_rand=t, precision="bf16")
    err = np.abs(a[0] - b[0]).max(axis=-1)
    print("pi-GAN 32x32 24+24 bf16 vs fp32: max-abs rgb %.4g, rays > 2e-2: %d / %d, PSNR %.1f dB"
          % (err.max(), (err > 2e-2).sum(), w * w, orc.psnr(a[0], b[0])))
    assert (err > 2e-2).sum() == 0 and orc.psnr(a[0], b[0]) >= 60


# ---- the last interval: sign(sigma_last) decides the ray (nerf/render.py:92) ------------------------------------------------
def _last_sample_case(model, rays, z, fp32_last, **kw):
    """default bf16 launch vs raw bf16 vs the fp32 path's sigma at the last sample of every ray"""
    n, s_ = z.shape
    before = dict(ops.last_sample_stats)
    with torch.no_grad():
        a = kw["run"](True).view(n, s_, 4)
        flagged = ops.last_sample_stats["flagged"] - before["flagged"]
        a0 = kw["run"](False).view(n, s_, 4)
    la, l0, lb = a[:, -1, 3], a0[:, -1, 3], fp32_last
    raw_flips = int(((l0 > 0) != (lb > 0)).sum())
    print("  last-sample check: %d / %d rays flagged (%.2f %%), raw bf16 sign flips %d, after the check %d"
          % (flagged, n, 100.0 * flagged / n, raw_flips, int(((la > 0) != (lb > 0)).sum())))
    assert bool(((la > 0) == (lb > 0)).all()), "sign(sigma_last) differs from the fp32 path"
    changed = la != l0
    assert torch.equal(la[changed], lb[changed]), "re-evaluated rows must be bit-identical to the fp32 path"
    assert int(changed.sum()) <= flagged <= 0.25 * n
    assert torch.equal(a[:, :-1], a0[:, :-1]) and torch.equal(a[:, -1, :3], a0[:, -1, :3]), "only sigma of the last sample may change"
    return flagged, raw_flips


def test_last_sample_sign_check_nerf_and_run_network():
    c, _ = seeded_nerf()
    pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)
    rays = ops.raygen(256, 200, 256 * 1.3875, pose)                        # 51,200 rays
    torch.manual_seed(11)
    z, _ = ops.stratified_z(torch.linspace(2.0, 6.0, 64).cuda(), torch.rand(rays.shape[0], 64, device="cuda"))
    with torch.no_grad():
        lb = ops.mlp(c, rays=rays, z=z[:, -1:].contiguous(), precision="fp32")[:, 3]
    flagged, raw_flips = _last_sample_case(c, rays, z, lb, run=lambda on: ops.mlp(c, rays=rays, z=z, precision="bf16", exact_last_sample=on))
    assert flagged > 0 and raw_flips > 0, "this seeded case is known to contain bf16 sign flips: the check must have had work to do"
    # the drop-in run_network (points [N,S,3]) keeps the [N,S] structure and applies the same check
    pts = rays[:, None, 0] + rays[:, None, 1] * z[..., None]
    vd = rays[:, 1] / rays[:, 1].norm(dim=-1, keepdim=True)
    _last_sample_case(c, rays, z, lb, run=lambda on: nerf_render.run_network(pts, vd, c, precision="bf16", exact_last_sample=on))
    # ragged: ray count not a multiple of the 512-row tile pair, 1 sample per ray (every row is a last sample)
    z1 = z[:777, -1:].contiguous()
    _last_sample_case(c, rays[:777], z1, lb[:777], run=lambda on: ops.mlp(c, rays=rays[:777], z=z1, precision="bf16", exact_last_sample=on))


def test_last_sample_sign_check_sine_models():
    """FiLM-SIREN (one latent and the batched launch with per-latent FiLM rows) and SirenNeRF."""
    p_ = pigan_render.camera_pos_to_transform_matrix(1.0, 0.2, 0.1)
    focal = np.float64(64 / 2 / np.tan(6 * np.pi / 180))
    rays1 = ops.raygen(64, 64, focal, p_)
    n = rays1.shape[0]
    torch.manual_seed(12)
    g = torch.Generator().manual_seed(0)
    films = torch.cat([1.0 + 0.2 * torch.randn(3, 9, 256, generator=g), 0.1 * torch.randn(3, 9, 256, generator=g)], -1).cuda()
    m = seeded_film()
    rays = torch.cat([rays1, rays1, rays1])
    z, _ = ops.stratified_z(torch.linspace(0.5, 1.5, 24).cuda(), torch.rand(3 * n, 24, device="cuda"))
    lbs = []
    with torch.no_grad():
        for b in range(3):
            m.set_film_params(films[b])
            lbs.append(ops.mlp(m, rays=rays1, z=z[b * n:(b + 1) * n, -1:].contiguous(), precision="fp32")[:, 3])
    m.set_film_params(films[1])
    z_b = z[n:2 * n].contiguous()
    _last_sample_case(m, rays1, z_b, lbs[1], run=lambda on: ops.mlp(m, rays=rays1, z=z_b, precision="bf16", exact_last_sample=on))
    flagged, _ = _last_sample_case(m, rays, z, torch.cat(lbs),
                                   run=lambda on: ops.mlp_film_batched(m, films, rays, z, n * 24, exact_last_sample=on))
    assert flagged > 0
    torch.manual_seed(0)
    sn = models.SirenNeRF().cuda()
    pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)
    rays_s = ops.raygen(128, 100, 128 * 1.3875, pose)
    zs, _ = ops.stratified_z(torch.linspace(2.0, 6.0, 64).cuda(), torch.rand(rays_s.shape[0], 64, device="cuda"))
    with torch.no_grad():
        lb = ops.mlp(sn, rays=rays_s, z=zs[:, -1:].contiguous(), precision="fp32")[:, 3]
    _last_sample_case(sn, rays_s, zs, lb, run=lambda on: ops.mlp(sn, rays=rays_s, z=zs, precision="bf16", exact_last_sample=on))


def test_last_sample_check_in_the_autograd_forward_is_an_explicit_switch():
    """ops.set_exact_last_sample(train=True): the training forward reports the render's raw values (default: raw bf16)."""
    c, _ = seeded_nerf()
    pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)
    rays = ops.raygen(128, 100, 128 * 1.3875, pose)
    torch.manual_seed(11)
    z, _ = ops.stratified_z(torch.linspace(2.0, 6.0, 64).cuda(), torch.rand(rays.shape[0], 64, device="cuda"))
    with torch.no_grad():
        on = ops.mlp(c, rays=rays, z=z, precision="bf16")
        off = ops.mlp(c, rays=rays, z=z, precision="bf16", exact_last_sample=False)
    assert not torch.equal(on, off)
    old = ops.set_grad_precision("bf16")
    try:
        assert torch.equal(ops.mlp(c, rays=rays, z=z).detach(), off)
        ops.set_exact_last_sample(train=True)
        raw = ops.mlp(c, rays=rays, z=z)
        assert torch.equal(raw.detach(), on)
        raw.sum().backward()
        assert all(torch.isfinite(p.grad).all() for p in c.parameters())
    finally:
        ops.set_exact_last_sample(train=False)
        ops.set_grad_precision(old)


def test_tc_pack_cache_invalidation():
    c, _ = seeded_nerf()
    x = torch.rand(300, 6, device="cuda")
    with torch.no_grad():
        a = ops.mlp(c, x=x, precision="bf16")
        c.output_layer_rgb.bias.add_(1.0)          # in-place update, as an optimiser step does
        b = ops.mlp(c, x=x, precision="bf16")
    assert (a[:, :3] - b[:, :3]).abs().max().item() > 0.05


def test_end_to_end_damped_field_bf16_vs_fp32():
    """End-to-end bf16 vs fp32 on the spectrally damped synthetic field (SURVEY 7.3-2 / 8d)."""
    torch.manual_seed(0)
    c, f = models.damp_nerf_(models.NeRF()).cuda(), models.damp_nerf_(models.NeRF()).cuda()
    pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)
    torch.manual_seed(5)
    t = torch.rand(64 * 64, 64, device="cuda")
    a = nerf_render.render_image(64, 64, 64 * 1.3875, pose, 2.0, 6.0, c, f, 64, 64, t_rand=t, precision="fp32")
    b = nerf_render.render_image(64, 64, 64 * 1.3875, pose, 2.0, 6.0, c, f, 64, 64, t_rand=t, precision="bf16",
                                 exact_last_sample=False)
    err = np.abs(a[0] - b[0]).max(axis=-1)
    flipped = int((err > 2e-2).sum())
    print("damped field, raw bf16 (sign check off) vs fp32: max-abs rgb %.4g, rays > 2e-2: %d / 4096, PSNR %.1f dB"
          % (err.max(), flipped, orc.psnr(a[0], b[0])))
    # the last interval (dists = 1e10) makes alpha_last a step function of sign(sigma_last): WITHOUT the sign check a
    # reduced-precision MLP flips a few rays by up to ~0.6 (SURVEY 0, landmine 1); everything else is well inside 2e-2
    assert flipped <= 0.005 * 4096
    assert np.median(err) < 2e-3 and np.percentile(err, 99) < 2e-2
    # the DEFAULT bf16 render (sign check on): north_star's bound holds for every ray
    c_ = nerf_render.render_image(64, 64, 64 * 1.3875, pose, 2.0, 6.0, c, f, 64, 64, t_rand=t, precision="bf16")
    err2 = np.abs(a[0] - c_[0]).max(axis=-1)
    print("  default bf16 render: max-abs rgb %.4g, rays > 2e-2: %d, PSNR %.1f dB" % (err2.max(), (err2 > 2e-2).sum(), orc.psnr(a[0], c_[0])))
    assert (err2 > 2e-2).sum() == 0 and orc.psnr(a[0], c_[0]) >= 60


# ---- K8 backward ---------------------------------------------------------------------------------------------
def _grad_check(model, tag, tr, rel=2e-3):
    for name, p in model.named_parameters():
        g = p.grad.detach().reshape(-1).double().cpu()
        ref_l2 = float(tr[f"g_{tag}.{name}.l2"]) if tag else float(tr[f"g.{name}.l2"])
        key = f"g_{tag}.{name}.sample" if tag else f"g.{name}.sample"
        ref = tr[key].astype(np.float64)
        got = g[::97].numpy()
        assert abs(float(g.norm()) - ref_l2) <= rel * max(ref_l2, 1e-8) + 1e-9, (name, float(g.norm()), ref_l2)
        np.testing.assert_allclose(got, ref, rtol=0, atol=rel * max(np.abs(ref).max(), ref_l2 / np.sqrt(g.numel())) + 1e-9,
                                   err_msg=name)


def test_nerf_train_step_gradients(golden):
    """render_rays + the train_nerf.py loss (nerf/train_nerf.py:151-167) -> gradients of both MLPs."""
    tr = golden.nerf_train
    torch.manual_seed(0)
    c, f = models.damp_nerf_(models.NeRF()).cuda(), models.damp_nerf_(models.NeRF()).cuda()
    sc, sf = int(tr["Sc"]), int(tr["Sf"])
    old = ops.set_grad_precision("fp32")            # the exact path: the fixture holds the reference's fp32 autograd gradients
    try:
        rc, _, ac, rf, _, af = nerf_render.render_rays(cu(tr["rays"]), 2.0, 6.0, c, f, sc, sf, t_rand=cu(tr["t_rand"]),
                                                       z_lin=tr["z_lin"], u=tr["u"])
        target, target_a = cu(tr["target"]), cu(tr["target_a"])
        loss = ((rf - target) ** 2).mean() + ((rc - target) ** 2).mean() + 0.1 * ((ac - target_a) ** 2).mean() \
            + 0.1 * ((af - target_a) ** 2).mean()
        loss.backward()
    finally:
        ops.set_grad_precision(old)
    np.testing.assert_allclose(rc.detach().cpu().numpy(), tr["rgb_c"], atol=1e-4)
    np.testing.assert_allclose(rf.detach().cpu().numpy(), tr["rgb_f"], atol=1e-3)
    assert abs(float(loss.detach()) - float(tr["loss"])) < 1e-4
    _grad_check(c, "coarse", tr, rel=5e-3)
    _grad_check(f, "fine", tr, rel=2e-2)     # fine samples move with the coarse weights (ill-conditioned bins)


def test_pigan_render_image_and_film_gradients(golden, exact_grads):
    """pi_GAN render_image -> image, d/d film_params and d/d weights (pi_GAN/train.py:134, synthesis.py:107)."""
    p = golden.pigan
    m = seeded_film()
    film = cu(p["film"]).requires_grad_(True)
    m.set_film_params(film)
    w = int(p["W"])
    img = pigan_render.render_image(w, w, np.float64(p["focal"]), p["pose"], 0.5, 1.5, m, m, 12, 12, t_rand=cu(p["t_rand"]),
                                    precision="fp32")
    assert img.shape == (w, w, 3) and img.requires_grad
    np.testing.assert_allclose(img.detach().cpu().numpy(), p["image"], atol=1e-4)
    (img * cu(p["g_image"])).sum().backward()
    gf, ref = film.grad.cpu().numpy(), p["g_film"]
    assert np.max(np.abs(gf - ref)) <= 2e-3 * np.abs(ref).max() + 1e-6
    _grad_check(m, "", p, rel=5e-3)
    # inversion mode: weights frozen, only film wanted
    m2 = seeded_film()
    for q in m2.parameters():
        q.requires_grad_(False)
    film2 = cu(p["film"]).requires_grad_(True)
    m2.set_film_params(film2)
    img2 = pigan_render.render_image(w, w, np.float64(p["focal"]), p["pose"], 0.5, 1.5, m2, m2, 12, 12,
                                     t_rand=cu(p["t_rand"]), precision="fp32")
    (img2 * cu(p["g_image"])).sum().backward()
    np.testing.assert_allclose(film2.grad.cpu().numpy(), gf, atol=1e-5 * np.abs(gf).max() + 1e-7)
    assert all(q.grad is None for q in m2.parameters())


def test_non_cuda_inputs_fail_loudly():
    with pytest.raises(RuntimeError):
        ops.composite(torch.zeros(2, 4, 4), torch.zeros(2, 4), torch.zeros(2, 3))
    with pytest.raises(TypeError):
        ops.mlp(torch.nn.Linear(6, 4).cuda(), x=torch.zeros(4, 6).cuda())


# ---- full-size property tests (BASELINE.json configs[1]: 800x800, 64+128) ---------------------------------------
def test_full_size_render_properties():
    """Size-independent properties at the headline size: sortedness / sub-sequence of the merged samples, weights sum to
    acc, ranges, determinism, sharded == slice of the full frame, white-background linearity of the composite."""
    torch.manual_seed(0)
    c, f = models.NeRF().cuda(), models.NeRF().cuda()
    pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)
    W = H = 800
    n = W * H
    torch.manual_seed(5)
    t = torch.rand(n, 64, device="cuda")
    rays = ops.raygen(W, H, W * 1.3875, pose)
    st = {}
    with torch.no_grad():
        out = nerf_render.render_rays(rays, 2.0, 6.0, c, f, 64, 128, t_rand=t, stages=st)
        out2 = nerf_render.render_rays(rays, 2.0, 6.0, c, f, 64, 128, t_rand=t)
    assert all(torch.equal(a, b) for a, b in zip(out, out2)), "render is not deterministic"
    zc, zf, zs = st["z_coarse"], st["z_fine"], st["z_samples"]
    assert zf.shape == (n, 192) and bool((zf[:, 1:] >= zf[:, :-1]).all())                  # sorted
    assert bool((zc[:, 1:] >= zc[:, :-1]).all()) and bool((zs[:, 1:] >= zs[:, :-1]).all())
    assert torch.equal(torch.sort(torch.cat([zc, zs], -1), -1).values, zf)                  # exactly the merged multiset
    mids = st["mids"]
    assert float(zs.min()) >= float(mids[0]) - 1e-6 and float(zs.max()) <= float(mids[-1]) + 1e-6
    wc = st["weights_coarse"]
    assert torch.allclose(wc.sum(-1), out[2], atol=1e-5) and float(out[2].max()) <= 1.0 + 1e-4 and float(wc.min()) >= 0.0
    for rgb in (out[0], out[3]):
        assert float(rgb.min()) >= -1e-4 and float(rgb.max()) <= 1.0 + 1e-4 and bool(torch.isfinite(rgb).all())
    assert bool((out[4] >= 0).all()) and float(out[4].max()) <= 6.0 * 1.3                    # depth <= far * |d|max
    # a pixel-row shard renders exactly the slice of the full frame (what multi-GPU sharding relies on)
    b0, cnt = 800 * 300, 800 * 100
    with torch.no_grad():
        part = nerf_render.render_image_device(W, H, W * 1.3875, pose, 2.0, 6.0, c, f, 64, 128, ray_begin=b0, ray_count=cnt,
                                               t_rand=t[b0:b0 + cnt])
    assert all(torch.equal(p, o[b0:b0 + cnt]) for p, o in zip(part, out))
    # composite: rgb_map - (1 - acc) is linear in the sample colours
    raw = st["raw_fine"][:50000].clone()
    z, d = zf[:50000], rays[:50000, 1]
    r1 = ops.composite(raw, z, d, want_weights=False)
    raw2 = raw.clone(); raw2[..., :3] *= 0.5
    r2 = ops.composite(raw2, z, d, want_weights=False)
    lin1 = r1[0] - (1 - r1[2])[:, None]; lin2 = r2[0] - (1 - r2[2])[:, None]
    assert torch.allclose(lin2, 0.5 * lin1, atol=2e-6) and torch.equal(r1[1], r2[1]) and torch.equal(r1[2], r2[2])


def test_edge_shapes():
    """N == 1 (crashes the reference, SURVEY app. D), float sample counts, tiny sample counts, empty input."""
    c, f = seeded_nerf()
    rays = torch.tensor([[[0.0, 0.0, 4.0], [0.05, -0.02, -1.0]]], device="cuda")
    with torch.no_grad():
        out = nerf_render.render_rays(rays, 2.0, 6.0, c, f, 64.0, 128.0)             # float counts (test_nerf.py:34-35)
        assert out[3].shape == (1, 3) and bool(torch.isfinite(out[3]).all())
        out = nerf_render.render_rays(rays.expand(5, 2, 3).contiguous(), 2.0, 6.0, c, f, 4, 3)
        assert out[0].shape == (5, 3)
        empty = ops.mlp(c, x=torch.zeros(0, 6, device="cuda"))
        assert empty.shape == (0, 4)
    r = ops.composite(torch.zeros(0, 7, 4, device="cuda"), torch.zeros(0, 7, device="cuda"), torch.zeros(0, 3, device="cuda"))
    assert r[0].shape == (0, 3)


def test_drop_in_usage_like_the_reference_scripts():
    """The way nerf/train_nerf.py and show_nerf.py use the module: CUDA default tensor type, star import, render_image to
    numpy, then a training step (render_rays + MSE + backward + Adam, train_nerf.py:151-168) on the same models."""
    torch.set_default_tensor_type('torch.cuda.FloatTensor')                       # nerf/train_nerf.py:11
    try:
        ns = {}
        exec("from msra_practice_project_b200.nerf_render import *", ns)          # `from render import *`
        for name in ("np", "torch", "tqdm", "to8b", "get_rays", "sample_pdf", "run_network", "raw_to_outputs", "render_rays",
                     "render_image", "render_video"):
            assert name in ns, name
        torch.manual_seed(0)
        coarse, fine = models.NeRF(), models.NeRF()                                # created on the default (CUDA) device
        pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.1, -0.5)
        with torch.no_grad():
            rgb, depth, acc = ns["render_image"](40, 30, 40 * 1.3875, pose, 2.0, 6.0, coarse, fine, 64, 128)
        assert rgb.shape == (30, 40, 3) and depth.shape == (30, 40, 1) and acc.shape == (30, 40, 1) and rgb.dtype == np.float32
        img8 = ns["to8b"](rgb)
        assert img8.dtype == np.uint8
        vid = ns["render_video"](8, 6, 8 * 1.3875, [pose, pose], 2.0, 6.0, coarse, fine, 8, 8)
        assert vid[0].shape == (2, 6, 8, 3)
        opt = torch.optim.Adam(list(coarse.parameters()) + list(fine.parameters()), lr=5e-4)
        rays = torch.tensor(np.stack(ns["get_rays"](16, 16, 16 * 1.3875, pose), 0).transpose(1, 2, 0, 3).reshape(-1, 2, 3))
        target = torch.rand(256, 3)
        losses = []
        for _ in range(3):
            rc, _, _, rf, _, _ = ns["render_rays"](rays, 2.0, 6.0, coarse, fine, 16, 16)
            loss = torch.mean((rf - target) ** 2) + torch.mean((rc - target) ** 2)
            opt.zero_grad(); loss.backward(); opt.step()
            losses.append(float(loss.detach()))
        assert all(np.isfinite(losses)) and all(p.grad is not None for p in coarse.parameters())
    finally:
        torch.set_default_tensor_type(torch.FloatTensor)
        torch.set_default_device("cpu")


def test_coarse_sigma_only_is_dead_code_elimination():
    """render_image(coarse_sigma_only=True) stops the COARSE pass after the sigma head (its colour is never returned,
    nerf/render.py:150-167 / pi_GAN/render.py:195-206): sigma of the shortened walk, the coarse weights and every fine output must be
    bit-identical to the full evaluation's, for NeRF and for the FiLM-SIREN batch render; a coarse pass that carries gradients refuses."""
    from msra_practice_project_b200 import nerf_render
    torch.manual_seed(1)
    coarse, fine = models.NeRF().cuda(), models.NeRF().cuda()
    pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.2, -0.4)
    rays = ops.raygen(48, 40, 48 * 1.3875, pose, 0, 48 * 40, device=torch.device("cuda"))
    z = torch.sort(torch.rand(48 * 40, 64, device="cuda") * 4 + 2, -1).values
    with torch.no_grad():
        raw_full = ops.mlp(coarse, rays=rays, z=z, precision="bf16", exact_last_sample=False)
        raw_sig = ops.mlp(coarse, rays=rays, z=z, precision="bf16", sigma_only=True)
        assert torch.equal(raw_full[:, 3], raw_sig[:, 3]) and float(raw_sig[:, :3].abs().max()) == 0.0
        t_rand = torch.rand(48 * 40, 64, device="cuda")
        a = nerf_render.render_image_device(48, 40, 48 * 1.3875, pose, 2.0, 6.0, coarse, fine, 64, 128, t_rand=t_rand)
        b = nerf_render.render_image_device(48, 40, 48 * 1.3875, pose, 2.0, 6.0, coarse, fine, 64, 128, t_rand=t_rand, coarse_sigma_only=True)
        for i in (3, 4, 5):
            assert torch.equal(a[i], b[i]), i
        assert torch.equal(b[0][:, 0], b[0][:, 1]) and torch.equal(b[0][:, 0], b[0][:, 2])     # coarse colour map: the white background term only
        ia = nerf_render.render_image(48, 40, 48 * 1.3875, pose, 2.0, 6.0, coarse, fine, 64, 128, t_rand=t_rand)
        ib = nerf_render.render_image(48, 40, 48 * 1.3875, pose, 2.0, 6.0, coarse, fine, 64, 128, t_rand=t_rand, coarse_sigma_only=True)
        assert all(np.array_equal(x, y) for x, y in zip(ia, ib))
        # SirenNeRF has no shortened walk: the switch is accepted and changes nothing
        sa, sb = models.SirenNeRF().cuda(), models.SirenNeRF().cuda()
        c = nerf_render.render_image_device(16, 16, 22.0, pose, 2.0, 6.0, sa, sb, 16, 16, t_rand=t_rand[:256, :16])
        d = nerf_render.render_image_device(16, 16, 22.0, pose, 2.0, 6.0, sa, sb, 16, 16, t_rand=t_rand[:256, :16], coarse_sigma_only=True)
        assert all(torch.equal(c[i], d[i]) for i in range(6))
        # FiLM-SIREN batch render (4 latents x 32x32, 24+24: rows per latent a multiple of 512)
        net = models.FilmSirenNeRF().cuda()
        g = torch.Generator().manual_seed(0)
        film = torch.cat([1.0 + 0.2 * torch.randn(4, 9, 256, generator=g), 0.1 * torch.randn(4, 9, 256, generator=g)], -1).cuda()
        poses = [pigan_render.camera_pos_to_transform_matrix(1, 0.3 * np.sin(i), 0.15 * np.cos(i)) for i in range(4)]
        tr = torch.rand(4 * 32 * 32, 24, device="cuda")
        focal = 32 / 2 / np.tan(6 * np.pi / 180)
        p1 = pigan_render.render_batch(net, film, poses, 32, 32, focal, 0.5, 1.5, 24, 24, t_rand=tr)
        p2 = pigan_render.render_batch(net, film, poses, 32, 32, focal, 0.5, 1.5, 24, 24, t_rand=tr, coarse_sigma_only=True)
        assert torch.equal(p1, p2)
    with pytest.raises(RuntimeError):
        nerf_render.render_rays(rays.reshape(-1, 2, 3)[:64], 2.0, 6.0, coarse, fine, 16, 16, coarse_sigma_only=True)


def test_render_image_frames_are_owned_by_the_caller():
    """render_image hands out views of pooled page-locked buffers (no host copy).  A frame the caller still holds must never be
    overwritten by later renders -- also beyond the pool size, where the images become fresh pageable arrays -- and a buffer must go
    back to the pool once its frame is dropped."""
    from msra_practice_project_b200 import nerf_render
    torch.manual_seed(0)
    coarse, fine = models.NeRF().cuda(), models.NeRF().cuda()
    poses = [pigan_render.camera_pos_to_transform_matrix(4.0, 0.1 * i, -0.5) for i in range(7)]
    t_rand = torch.rand(24 * 20, 16, device="cuda")
    held, copies = [], []
    for p in poses:                                                            # 7 frames held at once (pool: 4)
        f = nerf_render.render_image(24, 20, 24 * 1.3875, p, 2.0, 6.0, coarse, fine, 16, 16, t_rand=t_rand)
        assert f[0].shape == (20, 24, 3) and f[1].shape == (20, 24, 1) and f[0].dtype == np.float32
        held.append(f)
        copies.append(tuple(a.copy() for a in f))
    for f, c in zip(held, copies):
        for a, b in zip(f, c):
            assert np.array_equal(a, b)
    assert not np.array_equal(copies[0][0], copies[1][0])                      # the poses do differ
    pool = nerf_render._host_stage[(torch.cuda.current_device(), 24 * 20)]
    assert len(pool) == nerf_render._STAGE_POOL
    if pool[0][1] is not None:                                                 # use counts available: zero-copy hand-out and reuse
        assert all(nerf_render._storage_uses(b) > idle for b, idle in pool)
        first = held[0][0]
        held.clear(); del f, a
        assert sum(nerf_render._storage_uses(b) == idle for b, idle in pool) == nerf_render._STAGE_POOL - 1     # `first` keeps one
        again = nerf_render.render_image(24, 20, 24 * 1.3875, poses[3], 2.0, 6.0, coarse, fine, 16, 16, t_rand=t_rand)
        assert np.array_equal(first, copies[0][0]) and np.array_equal(again[0], copies[3][0])
        assert len(pool) == nerf_render._STAGE_POOL
        again[0][0, 0, 0] = 7.0                                                # writable like any array
    vid = nerf_render.render_video(24, 20, 24 * 1.3875, poses[:3], 2.0, 6.0, coarse, fine, 16, 16)
    assert vid[0].shape == (3, 20, 24, 3) and vid[1].shape == (3, 20, 24, 1)


def test_tf32_layerwise_path_matches_fp32(golden):
    """The tensor-core (tcgen05 kind::tf32) layer-wise path: forward and every gradient against the fp32 CUDA-core path."""
    tr = golden.nerf_train
    sc, sf = int(tr["Sc"]), int(tr["Sf"])
    grads = {}
    outs = {}
    for mode in ("fp32", "tf32"):
        torch.manual_seed(0)
        c, f = models.damp_nerf_(models.NeRF()).cuda(), models.damp_nerf_(models.NeRF()).cuda()
        old = ops.set_grad_precision(mode)
        try:
            g = torch.Generator().manual_seed(9)
            rays = torch.cat([cu(tr["rays"])] * 40)[:900]                      # 900 rays x 32 samples: ragged 128-row tiles
            t = torch.rand(900, sc, generator=g).cuda()
            target = torch.rand(900, 3, generator=g).cuda()
            rc, _, ac, rf, _, af = nerf_render.render_rays(rays, 2.0, 6.0, c, f, sc, sf, t_rand=t, z_lin=tr["z_lin"], u=tr["u"])
            loss = ((rf - target) ** 2).mean() + ((rc - target) ** 2).mean() + 0.1 * (ac ** 2).mean() + 0.1 * (af ** 2).mean()
            loss.backward()
        finally:
            ops.set_grad_precision(old)
        outs[mode] = (rc.detach(), rf.detach())
        grads[mode] = {n: p.grad.detach().clone() for m_, tag in ((c, "c"), (f, "f")) for n, p in ((tag + "." + k, v) for k, v in m_.named_parameters())}
    assert (outs["tf32"][0] - outs["fp32"][0]).abs().max().item() < 5e-3
    worst = 0.0
    for n in grads["fp32"]:
        a, b = grads["fp32"][n], grads["tf32"][n]
        if n.startswith("f."):
            continue            # fine-pass gradients inherit moved sample positions (ill-conditioned bins): checked through the coarse net
        rel = (a - b).norm().item() / max(a.norm().item(), 1e-12)
        worst = max(worst, rel)
        assert rel < 5e-2, (n, rel)
    print("tf32 vs fp32 layer-wise path: max-abs rgb %.3g, worst relative gradient error %.3g"
          % ((outs["tf32"][0] - outs["fp32"][0]).abs().max().item(), worst))
    # FiLM-SIREN through the tf32 engine (forward values and d/dfilm)
    p = golden.pigan
    res = {}
    for mode in ("fp32", "tf32"):
        m = seeded_film()
        film = cu(p["film"]).requires_grad_(True)
        m.set_film_params(film)
        old = ops.set_grad_precision(mode)
        try:
            img = pigan_render.render_image(8, 8, np.float64(p["focal"]), p["pose"], 0.5, 1.5, m, m, 12, 12, t_rand=cu(p["t_rand"]), precision="fp32")
            (img * cu(p["g_image"])).sum().backward()
        finally:
            ops.set_grad_precision(old)
        res[mode] = (img.detach(), film.grad.clone())
    assert (res["tf32"][0] - res["fp32"][0]).abs().max().item() < 2e-2
    assert (res["tf32"][1] - res["fp32"][1]).norm().item() < 5e-2 * res["fp32"][1].norm().item()


def _emulate_bf16_nerf(net, rays, z, up):
    """The training kernels' arithmetic restated in torch (test oracle for mlp_tc_train.cu): bf16-rounded operands, fp32
    accumulation, bf16-rounded saved activations / gradients, relu' from the rounded activation, heads in fp32 on the
    un-rounded activation (nerf/nerf.py:75-94 forward, its autograd reverse mode)."""
    bf = lambda t: t.to(torch.bfloat16).float()
    P = {k: v.detach() for k, v in net.named_parameters()}
    W = lambda k: bf(P[k + ".weight"])
    B = lambda k: P[k + ".bias"]
    pts = (rays[:, None, 0] + rays[:, None, 1] * z[..., None]).reshape(-1, 3)
    vd = torch.nn.functional.normalize(rays[:, 1], dim=-1)[:, None].expand(-1, z.shape[1], -1).reshape(-1, 3)
    enc = lambda x, L: torch.cat([f(x * 2.0 ** i) for i in range(L) for f in (torch.sin, torch.cos)], -1)
    pe, de = bf(enc(pts, 10)), bf(enc(vd, 4))
    h, hs = pe, []
    for l in range(8):
        x = torch.cat([pe, h], -1) if l == 5 else h
        hs.append(x)
        h32 = torch.relu(x @ W(f"layers_pos.{l}").T + B(f"layers_pos.{l}"))
        h = bf(h32)
    sig_pre = h32 @ P["output_layer_sigma.weight"].T + P["output_layer_sigma.bias"]
    gl = bf(h @ W("layers_dir.0").T + B("layers_dir.0"))
    xd = torch.cat([gl, de], -1)
    hd32 = torch.relu(xd @ W("layers_dir.1").T + B("layers_dir.1"))
    hd = bf(hd32)
    rgb = torch.sigmoid(hd32 @ P["output_layer_rgb.weight"].T + P["output_layer_rgb.bias"])
    raw = torch.cat([rgb, torch.relu(sig_pre)], -1)
    G = {}
    gc = up[:, :3] * rgb * (1 - rgb)
    gs = up[:, 3:] * (sig_pre > 0)
    G["output_layer_rgb.weight"], G["output_layer_rgb.bias"] = gc.T @ hd, gc.sum(0)
    G["output_layer_sigma.weight"], G["output_layer_sigma.bias"] = gs.T @ h, gs.sum(0)
    gd1 = bf((gc @ P["output_layer_rgb.weight"]) * (hd > 0))
    G["layers_dir.1.weight"], G["layers_dir.1.bias"] = gd1.T @ xd, gd1.sum(0)
    gg = bf(gd1 @ W("layers_dir.1")[:, :256])
    G["layers_dir.0.weight"], G["layers_dir.0.bias"] = gg.T @ h, gg.sum(0)
    gh = bf((gg @ W("layers_dir.0") + gs * P["output_layer_sigma.weight"]) * (h > 0))
    for l in range(7, -1, -1):
        G[f"layers_pos.{l}.weight"], G[f"layers_pos.{l}.bias"] = gh.T @ hs[l], gh.sum(0)
        if l == 0:
            break
        w = W(f"layers_pos.{l}")[:, 60:] if l == 5 else W(f"layers_pos.{l}")
        prev = hs[l][:, 60:] if l == 5 else hs[l]
        gh = bf((gh @ w) * (prev > 0))
    return raw, G


@pytest.mark.parametrize("rows_shape", [(37, 24), (700, 64), (4096, 3), (1, 1)])
def test_bf16_tensor_core_training_path(rows_shape):
    """Fused tcgen05 training path (mlp_tc.cu forward with kept activations + mlp_tc_train.cu dgrad / wgrad / heads): raw
    outputs and EVERY parameter gradient on identical inputs and an adversarial (zero-mean random) upstream gradient
      (a) against the torch restatement of the same bf16 pipeline: <= 4e-2 relative L2 per tensor (what remains are relu-bit
          flips of activations that round across 0 differently: the kernel's posenc uses the double-angle recurrence);
      (b) against the exact fp32 layer-wise path: raw <= 2e-2 max-abs on rgb (north_star), gradient direction (cosine) >= 0.95
          and norm within 6 % per tensor -- the bf16-vs-fp32 gap itself (<= 0.2 relative on this cancelling upstream) is the
          arithmetic's, the restatement shows the same gap."""
    n, s = rows_shape
    g = torch.Generator().manual_seed(n)
    torch.manual_seed(0)
    net = models.damp_nerf_(models.NeRF()).cuda()
    o = torch.tensor([0.0, 0.0, 4.0]).expand(n, 3)
    d = torch.nn.functional.normalize(torch.randn(n, 3, generator=g) * 0.25 + torch.tensor([0.0, 0.0, -1.0]), dim=-1) * 1.1
    rays = torch.stack([o, d], 1).cuda()
    z = (torch.sort(torch.rand(n, s, generator=g), -1).values * 4 + 2).cuda()
    up = torch.randn(n * s, 4, generator=g).cuda()
    res = {}
    for mode in ("fp32", "bf16"):
        old = ops.set_grad_precision(mode)
        try:
            net.zero_grad(set_to_none=True)
            raw = ops.mlp(net, rays=rays, z=z)
            (raw * up).sum().backward()
        finally:
            ops.set_grad_precision(old)
        res[mode] = (raw.detach().clone(), {k: p.grad.detach().clone() for k, p in net.named_parameters()})
    old_tf32 = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        raw_e, g_e = _emulate_bf16_nerf(net, rays, z, up)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old_tf32
    a, b = res["fp32"][0], res["bf16"][0]
    assert (a[:, :3] - b[:, :3]).abs().max().item() < 2e-2
    # sigma is an unbounded relu output (x8 head gain on the damped field): bound what compositing sees, alpha at the mean
    # sample spacing (far - near) / 64, by the north_star's 2e-2 and the value itself relatively
    alpha = lambda sg: 1 - torch.exp(-sg * (4.0 / 64))
    assert (alpha(a[:, 3]) - alpha(b[:, 3])).abs().max().item() < 2e-2
    assert ((a[:, 3] - b[:, 3]).abs() / (1 + a[:, 3].abs())).max().item() < 8e-2
    assert (raw_e[:, :3] - b[:, :3]).abs().max().item() < 1e-2
    worst_e = worst_f = 0.0
    big = n * s >= 2048
    for k in res["fp32"][1]:
        gf, gb, ge = res["fp32"][1][k].reshape(-1), res["bf16"][1][k].reshape(-1), g_e[k].reshape(-1)
        rel_e = (ge - gb).norm().item() / max(ge.norm().item(), 1e-20)
        rel_f = (gf - gb).norm().item() / max(gf.norm().item(), 1e-20)
        worst_e, worst_f = max(worst_e, rel_e), max(worst_f, rel_f)
        if big:
            assert rel_e < 4e-2, (k, rel_e)
            cos = torch.dot(gf, gb).item() / max(gf.norm().item() * gb.norm().item(), 1e-30)
            assert cos > 0.95 and abs(gb.norm().item() / max(gf.norm().item(), 1e-30) - 1) < 0.06, (k, cos, gf.norm().item(), gb.norm().item())
        else:   # a handful of rows: single relu-bit flips dominate; only bound the error
            assert rel_e < 0.5 and rel_f < 0.6, (k, rel_e, rel_f)
    print("bf16 training path (%d x %d rows): worst relative gradient error %.3g vs bf16 restatement, %.3g vs fp32"
          % (n, s, worst_e, worst_f))


def test_bf16_training_step_like_train_nerf(golden):
    """nerf/train_nerf.py:151-168 with the tensor-core training path: loss and its decrease over Adam steps match the fp32
    path (coherent gradients: the regime training runs in)."""
    tr = golden.nerf_train
    sc, sf = int(tr["Sc"]), int(tr["Sf"])
    g = torch.Generator().manual_seed(4)
    rays = torch.cat([cu(tr["rays"])] * 50)[:1024]
    t = torch.rand(1024, sc, generator=g).cuda()
    target = torch.rand(1024, 3, generator=g).cuda() * 0.5 + 0.25
    hist = {}
    for mode in ("fp32", "bf16"):
        torch.manual_seed(0)
        c, f = models.damp_nerf_(models.NeRF()).cuda(), models.damp_nerf_(models.NeRF()).cuda()
        opt = torch.optim.Adam(list(c.parameters()) + list(f.parameters()), lr=5e-4)
        old = ops.set_grad_precision(mode)
        losses = []
        try:
            for _ in range(8):
                opt.zero_grad(set_to_none=True)
                rc, _, _, rf, _, _ = nerf_render.render_rays(rays, 2.0, 6.0, c, f, sc, sf, t_rand=t, z_lin=tr["z_lin"], u=tr["u"])
                loss = ((rf - target) ** 2).mean() + ((rc - target) ** 2).mean()
                loss.backward()
                opt.step()
                losses.append(float(loss.detach()))
        finally:
            ops.set_grad_precision(old)
        hist[mode] = losses
    print("losses fp32", ["%.5f" % x for x in hist["fp32"]], "bf16", ["%.5f" % x for x in hist["bf16"]])
    assert abs(hist["bf16"][0] - hist["fp32"][0]) < 2e-3
    assert hist["bf16"][-1] < hist["bf16"][0] and hist["fp32"][-1] < hist["fp32"][0]
    assert abs(hist["bf16"][-1] - hist["fp32"][-1]) < 0.05 * hist["fp32"][0]


def test_adam_kernel_matches_torch_adam():
    """b2r_adam_step (optim.cu) against torch.optim.Adam + the train_nerf.py:170-175 learning-rate decay, 6 steps."""
    g = torch.Generator().manual_seed(3)
    n = 100003                                       # not a multiple of 4: exercises the tail
    p0 = torch.randn(n + 1, generator=g).cuda()[:n + 1]
    p_ref = torch.nn.Parameter(p0[:n].clone())
    opt = torch.optim.Adam([p_ref], lr=5e-4)
    buf = torch.zeros(4 * ((n + 3) // 4), device="cuda")
    p = buf[:n]; p.copy_(p0[:n])
    m, v, state = torch.zeros_like(p), torch.zeros_like(p), torch.zeros(4, device="cuda")
    for t in range(1, 7):
        grad = torch.randn(n, generator=g).cuda() * (10.0 ** (t - 4))
        for group in opt.param_groups:
            group["lr"] = 5e-4 * 0.1 ** ((t - 1) / 3.0)
        p_ref.grad = grad.clone()
        opt.step()
        ops.adam_step(p, grad, m, v, state, 5e-4, 0.1, 3.0)
        assert int(state[:1].view(torch.int32).item()) == t
        np.testing.assert_allclose(p.cpu().numpy(), p_ref.detach().cpu().numpy(), rtol=2e-6, atol=2e-7)


@pytest.mark.parametrize("graph", [False, True])
def test_fused_train_step_matches_autograd_path(golden, graph):
    """train_step.NerfTrainStep (explicit kernel sequence, fused Adam, CUDA graphs) against the drop-in route the
    reference script takes -- render_rays + autograd + torch.optim.Adam + LR decay (nerf/train_nerf.py:151-176) -- with the
    same bf16 tensor-core arithmetic, same rays / targets / jitter, 6 steps."""
    from msra_practice_project_b200.train_step import NerfTrainStep
    tr = golden.nerf_train
    sc, sf, nb = 32, 48, 640
    gen = torch.Generator().manual_seed(8)
    rays = torch.cat([cu(tr["rays"])] * 40)[:nb].contiguous()
    target = (torch.rand(nb, 3, generator=gen) * 0.5 + 0.25).cuda()
    alpha = torch.rand(nb, generator=gen).cuda()
    ts = [torch.rand(nb, sc, generator=gen).cuda() for _ in range(6)]
    # reference-style loop
    torch.manual_seed(0)
    c, f = models.damp_nerf_(models.NeRF()).cuda(), models.damp_nerf_(models.NeRF()).cuda()
    opt = torch.optim.Adam(list(c.parameters()) + list(f.parameters()), lr=5e-4)
    old = ops.set_grad_precision("bf16")
    ref_losses = []
    try:
        for k in range(6):
            rc, _, ac, rf, _, af = nerf_render.render_rays(rays, 2.0, 6.0, c, f, sc, sf, t_rand=ts[k])
            opt.zero_grad()
            loss = ((rf - target) ** 2).mean() + 0.1 * ((af - alpha) ** 2).mean() + ((rc - target) ** 2).mean() + 0.1 * ((ac - alpha) ** 2).mean()
            loss.backward()
            opt.step()
            for group in opt.param_groups:
                group["lr"] = 5e-4 * 0.1 ** ((k + 1) / 2000.0)
            ref_losses.append(float(loss.detach()))
    finally:
        ops.set_grad_precision(old)
    # fused step
    torch.manual_seed(0)
    c2, f2 = models.damp_nerf_(models.NeRF()).cuda(), models.damp_nerf_(models.NeRF()).cuda()
    step = NerfTrainStep(c2, f2, 2.0, 6.0, sc, sf, nb, learning_rate=5e-4, learning_rate_decay=2, use_alpha=True, graph=graph)
    losses = [float(step(rays, target, alpha, t_rand=ts[k])[0]) for k in range(6)]
    print("fused step losses", ["%.6f" % x for x in losses], "reference-style", ["%.6f" % x for x in ref_losses])
    assert step.global_step == 6
    np.testing.assert_allclose(losses, ref_losses, rtol=2e-3, atol=1e-5)
    # the nn.Modules alias the flat master weights: state_dict / render keep working, and the weights moved the same way
    worst, mean = 0.0, 0.0
    for (k1, a), (k2, b) in zip(c.state_dict().items(), c2.state_dict().items()):
        assert k1 == k2
        worst = max(worst, (a - b).abs().max().item())
        mean = max(mean, (a - b).abs().mean().item())
    # Adam moves every weight by ~lr per step whatever the gradient's size: a weight whose gradient is summation-order noise
    # (float atomics in wgrad) may walk the other way -> bounded by 2 * 6 * lr; on average the updates agree
    assert worst <= 2 * 6 * 5e-4 + 1e-6 and mean < 2e-4, (worst, mean)
    # a render through the drop-in module in the middle of training must see the CURRENT weights (the fused step updates the
    # flat master buffer behind torch's version counters): compare with fresh models loaded from the state dicts
    c3, f3 = models.NeRF().cuda(), models.NeRF().cuda()
    c3.load_state_dict(c2.state_dict()); f3.load_state_dict(f2.state_dict())
    with torch.no_grad():
        img = nerf_render.render_rays(rays[:64], 2.0, 6.0, c2, f2, sc, sf, t_rand=ts[0][:64])[3]
        step(rays, target, alpha, t_rand=ts[0])
        img_after = nerf_render.render_rays(rays[:64], 2.0, 6.0, c2, f2, sc, sf, t_rand=ts[0][:64])[3]
        img_ref = nerf_render.render_rays(rays[:64], 2.0, 6.0, c3, f3, sc, sf, t_rand=ts[0][:64])[3]
    assert torch.isfinite(img).all() and torch.equal(img, img_ref)
    assert not torch.equal(img_after, img), "render after another training step used stale packed weights"


def test_siren_nerf_forward_and_training_gradients(golden, exact_grads):
    """SirenNeRF (nerf/nerf.py:97-170; `use_siren`, nerf/train_nerf.py:89-91) through the layer-wise fp32 path: network(x)
    against the reference's forward, then render_rays + MSE loss + backward against the reference's autograd gradients of
    all 24 tensors of both models (fixture tests/golden/siren.npz)."""
    g = golden.siren
    torch.manual_seed(0)
    m = models.SirenNeRF().cuda()
    with torch.no_grad():
        out = ops.mlp(m, x=cu(g["x"]), precision="fp32").cpu().numpy()
        out_bf16 = ops.mlp(m, x=cu(g["x"])).cpu().numpy()              # default precision -> fused bf16 tensor-core kernel
    np.testing.assert_allclose(out[:, :3], g["out"][:, :3], atol=2e-4, rtol=0)
    np.testing.assert_allclose(out[:, 3], g["out"][:, 3], atol=2e-4, rtol=1e-3)
    assert np.abs(out_bf16[:, :3] - g["out"][:, :3]).max() < 2e-2
    torch.manual_seed(0)
    c, f = models.SirenNeRF().cuda(), models.SirenNeRF().cuda()
    rc, _, _, rf, _, _ = nerf_render.render_rays(cu(g["rays"]), 2.0, 6.0, c, f, 16, 16, t_rand=cu(g["t_rand"]), z_lin=g["z_lin"], u=g["u"],
                                                 precision="fp32")
    target = cu(g["target"])
    loss = ((rf - target) ** 2).mean() + ((rc - target) ** 2).mean()
    loss.backward()
    np.testing.assert_allclose(rc.detach().cpu().numpy(), g["rgb_c"], atol=2e-4)
    np.testing.assert_allclose(rf.detach().cpu().numpy(), g["rgb_f"], atol=2e-3)
    assert abs(float(loss.detach()) - float(g["loss"])) < 2e-4
    _grad_check(c, "coarse", g, rel=2e-2)
    _grad_check(f, "fine", g, rel=5e-2)


@pytest.mark.parametrize("rows", [96, 1000, 70000])
def test_siren_nerf_tensor_core_kernel(golden, rows):
    """Fused tcgen05 SirenNeRF kernel (mlp_tc_siren.cu) against the fp32 layer-wise path and, for the fixture rows, the
    reference's own forward: <= 2e-2 max-abs on rgb (north_star bf16 tolerance), sigma relative to max(1, sigma)."""
    g = golden.siren
    torch.manual_seed(0)
    m = models.SirenNeRF().cuda()
    if rows == 96:
        x, ref = cu(g["x"]), g["out"]
    else:
        gen = torch.Generator().manual_seed(rows)
        x = torch.cat([torch.rand(rows, 3, generator=gen) * 4 - 2,
                       torch.nn.functional.normalize(torch.randn(rows, 3, generator=gen), dim=-1)], -1).cuda()
        with torch.no_grad():
            ref = ops.mlp(m, x=x, precision="fp32").cpu().numpy()
    with torch.no_grad():
        out = ops.mlp(m, x=x, precision="bf16").cpu().numpy()
    err_rgb = np.abs(out[:, :3] - ref[:, :3]).max()
    err_sig = (np.abs(out[:, 3] - ref[:, 3]) / np.maximum(1.0, ref[:, 3])).max()
    print("SirenNeRF bf16 kernel, %d rows: max-abs rgb %.4g, sigma (rel. to max(1, sigma)) %.4g" % (rows, err_rgb, err_sig))
    # sigma is an unbounded relu output of a 256-wide sum of bf16-evaluated sines (30x argument gain per layer): bound it
    # relatively, and by what compositing sees (alpha at the mean sample spacing 4/64) with the north_star's 2e-2
    alpha = lambda sg: 1 - np.exp(-sg * (4.0 / 64))
    assert err_rgb < 2e-2 and err_sig < 8e-2 and np.abs(alpha(out[:, 3]) - alpha(ref[:, 3])).max() < 2e-2
    # rays mode = points mode
    if rows == 1000:
        o = torch.tensor([0.0, 0.0, 1.5]).expand(50, 3)
        d = torch.nn.functional.normalize(torch.randn(50, 3, generator=gen) * 0.3 + torch.tensor([0.0, 0.0, -1.0]), dim=-1)
        rays = torch.stack([o, d], 1).cuda()
        z = torch.linspace(0.5, 2.5, 20).expand(50, 20).contiguous().cuda()
        with torch.no_grad():
            a = ops.mlp(m, rays=rays, z=z, precision="bf16", exact_last_sample=False)      # the raw kernel output in both modes
            pts = (rays[:, None, 0] + rays[:, None, 1] * z[..., None]).reshape(-1, 3)
            vd = d.cuda()[:, None].expand(50, 20, 3).reshape(-1, 3)
            b = ops.mlp(m, x=torch.cat([pts, vd], -1), precision="bf16")
        assert (a - b).abs().max().item() < 2e-2


def test_pigan_render_batch_one_launch_matches_per_latent_loop():
    """render_batch's batched path (one MLP launch per pass for all latents, per-latent FiLM tables reloaded at latent
    boundaries; Generator.forward's loop pi_GAN/modules.py:176-184) against the per-latent loop, same jitter: identical
    kernels and arithmetic -> bit-identical images."""
    torch.manual_seed(0)
    net = models.FilmSirenNeRF().cuda()
    g = torch.Generator().manual_seed(2)
    b, res, s_ = 5, 32, 8                                     # 32*32*8 = 8192 rows per latent: several latents per CTA
    film = torch.cat([1.0 + 0.2 * torch.randn(b, 9, 256, generator=g), 0.1 * torch.randn(b, 9, 256, generator=g)], -1).cuda()
    poses = [pigan_render.camera_pos_to_transform_matrix(1, 0.3 * np.sin(i), 0.15 * np.cos(i)) for i in range(b)]
    focal = np.float64(res / 2 / np.tan(6 * np.pi / 180))
    t = torch.rand(b, res * res, s_, generator=g).cuda()
    with torch.no_grad():
        batched = pigan_render.render_batch(net, film, poses, res, res, focal, 0.5, 1.5, s_, s_, t_rand=t)
        loop = []
        for i in range(b):
            net.set_film_params(film[i])
            loop.append(pigan_render.render_image(res, res, focal, poses[i], 0.5, 1.5, net, net, s_, s_, t_rand=t[i]))
        loop = torch.stack(loop).permute(0, 3, 1, 2)
    assert batched.shape == (b, 3, res, res)
    assert torch.equal(batched, loop), (batched - loop).abs().max().item()
    # (the per-latent path's own parity against the reference is test_pigan_render_bf16_vs_fp32 / test_mlp_tc_film_vs_reference)


def test_to8b_device_and_streamed_video():
    """b2r_to8b against the reference's numpy to8b (nerf/render.py:5) bit for bit, and render_video_u8 (device quantise +
    double-buffered pinned copies) against to8b(render_video(...)) with the same seeds."""
    g = torch.Generator().manual_seed(0)
    x = torch.cat([torch.rand(100003, generator=g) * 1.4 - 0.2, torch.tensor([0.0, 1.0, -0.0, 0.5, 1.0 / 255, 254.999 / 255, 2.0, -3.0])])
    got = ops.to8b(x.cuda()).cpu().numpy()
    assert np.array_equal(got, nerf_render.to8b(x.numpy()))
    c, f = seeded_nerf()
    poses = [pigan_render.camera_pos_to_transform_matrix(4.0, 0.2 * i, -0.5) for i in range(3)]
    torch.manual_seed(11)
    vid = nerf_render.render_video_u8(24, 16, 24 * 1.3875, poses, 2.0, 6.0, c, f, 8, 8)
    torch.manual_seed(11)
    ref, _, _ = nerf_render.render_video(24, 16, 24 * 1.3875, poses, 2.0, 6.0, c, f, 8, 8)
    assert vid.shape == (3, 16, 24, 3) and vid.dtype == np.uint8
    assert np.array_equal(vid, nerf_render.to8b(ref))


def test_fused_train_step_draws_its_own_jitter_inside_the_graph(golden):
    """NerfTrainStep with t_rand=None: the jitter of nerf/render.py:131 is drawn by torch.rand INSIDE the captured graph
    (philox state advanced on every replay): steps see different jitter, the loss goes down, state_dict round-trips."""
    from msra_practice_project_b200.train_step import NerfTrainStep
    tr = golden.nerf_train
    nb, sc, sf = 256, 16, 16
    gen = torch.Generator().manual_seed(1)
    rays = torch.cat([cu(tr["rays"])] * 20)[:nb].contiguous()
    target = (torch.rand(nb, 3, generator=gen) * 0.5 + 0.25).cuda()
    torch.manual_seed(0)
    c, f = models.damp_nerf_(models.NeRF()).cuda(), models.damp_nerf_(models.NeRF()).cuda()
    step = NerfTrainStep(c, f, 2.0, 6.0, sc, sf, nb, learning_rate=5e-4, learning_rate_decay=1)
    jit, losses = [], []
    for _ in range(6):
        loss, psnr = step(rays, target)
        losses.append(float(loss)); jit.append(step.in_t.clone())
    assert all(np.isfinite(losses)) and losses[-1] < losses[0]
    assert not torch.equal(jit[0], jit[1]) and not torch.equal(jit[1], jit[2])
    assert 0.0 <= float(jit[3].min()) and float(jit[3].max()) < 1.0
    assert step.global_step == 6 and abs(step.learning_rate - 5e-4 * 0.1 ** (6 / 1000.0)) < 1e-9
    sd = step.state_dict()
    c2, f2 = models.NeRF().cuda(), models.NeRF().cuda()
    c2.load_state_dict(c.state_dict()); f2.load_state_dict(f.state_dict())
    step2 = NerfTrainStep(c2, f2, 2.0, 6.0, sc, sf, nb, learning_rate=5e-4, learning_rate_decay=1, graph=False)
    step2.load_state_dict(sd)
    t = torch.rand(nb, sc, generator=gen).cuda()
    l1 = float(step(rays, target, t_rand=t)[0]); l2 = float(step2(rays, target, t_rand=t)[0])
    assert abs(l1 - l2) < 1e-5 * max(1.0, abs(l1)) and step2.global_step == 7
    assert (step.params - step2.params).abs().max().item() <= 2 * 5e-4 + 1e-6


@pytest.mark.parametrize("rows_shape", [(37, 24), (700, 32), (1, 1)])
def test_siren_nerf_fused_training_path(rows_shape):
    """SirenNeRF on the fused tensor-core training path (siren_tc_kernel<true> with bf16 activation + cosine checkpoints,
    nerf_tc_bwd_kernel<true>, MN-major wgrad with the aux tile): the training forward is bit-identical to the inference
    kernel; every parameter gradient against the exact fp32 layer-wise path (direction cosine >= 0.98, <= 0.12 relative L2
    with >= 4096 rows)."""
    n, s = rows_shape
    g = torch.Generator().manual_seed(n + 5)
    torch.manual_seed(0)
    net = models.SirenNeRF().cuda()
    o = torch.tensor([0.0, 0.0, 1.2]).expand(n, 3)
    d = torch.nn.functional.normalize(torch.randn(n, 3, generator=g) * 0.25 + torch.tensor([0.0, 0.0, -1.0]), dim=-1)
    rays = torch.stack([o, d], 1).cuda()
    z = (torch.sort(torch.rand(n, s, generator=g), -1).values * 1.0 + 0.5).cuda()
    up = torch.randn(n * s, 4, generator=g).cuda()
    with torch.no_grad():
        raw_inf = ops.mlp(net, rays=rays, z=z, precision="bf16", exact_last_sample=False)   # gradient passes run the raw bf16 forward
    res = {}
    for mode in ("fp32", "bf16"):
        old = ops.set_grad_precision(mode)
        try:
            net.zero_grad(set_to_none=True)
            raw = ops.mlp(net, rays=rays, z=z)
            (raw * up).sum().backward()
        finally:
            ops.set_grad_precision(old)
        res[mode] = (raw.detach().clone(), {k: p.grad.detach().clone() for k, p in net.named_parameters()})
    assert torch.equal(res["bf16"][0], raw_inf), "training forward differs from the inference kernel"
    assert (res["bf16"][0][:, :3] - res["fp32"][0][:, :3]).abs().max().item() < 2e-2
    worst = 0.0
    for k in res["fp32"][1]:
        gf, gb = res["fp32"][1][k].reshape(-1), res["bf16"][1][k].reshape(-1)
        rel = (gf - gb).norm().item() / max(gf.norm().item(), 1e-20)
        cos = torch.dot(gf, gb).item() / max(gf.norm().item() * gb.norm().item(), 1e-30)
        worst = max(worst, rel)
        assert torch.isfinite(gb).all()
        if n * s >= 4096:
            assert cos > 0.98 and rel < 0.12, (k, rel, cos)
        else:           # a few hundred rows: the bf16 rounding of the raw position (first-layer wgrad operand) is not averaged out
            assert rel < 0.5, (k, rel)
    print("SirenNeRF fused training path (%d x %d rows): worst relative gradient error %.3g vs fp32" % (n, s, worst))


def test_siren_fused_train_step_trains(golden):
    """NerfTrainStep on two SirenNeRF models (train_nerf.py with use_siren): the loss follows the autograd + torch Adam route."""
    from msra_practice_project_b200.train_step import NerfTrainStep
    tr = golden.nerf_train
    nb, sc, sf = 512, 16, 16
    gen = torch.Generator().manual_seed(2)
    rays = torch.cat([cu(tr["rays"])] * 30)[:nb].contiguous()
    target = (torch.rand(nb, 3, generator=gen) * 0.5 + 0.25).cuda()
    ts = [torch.rand(nb, sc, generator=gen).cuda() for _ in range(5)]
    torch.manual_seed(0)
    c, f = models.SirenNeRF().cuda(), models.SirenNeRF().cuda()
    lr = 2e-5               # SIREN's default init reacts violently to Adam steps of 5e-4 on this toy problem: keep the comparison well-posed
    opt = torch.optim.Adam(list(c.parameters()) + list(f.parameters()), lr=lr)
    ref = []
    for t in ts:
        rc, _, _, rf, _, _ = nerf_render.render_rays(rays, 2.0, 6.0, c, f, sc, sf, t_rand=t)
        opt.zero_grad()
        loss = ((rf - target) ** 2).mean() + ((rc - target) ** 2).mean()
        loss.backward(); opt.step(); ref.append(float(loss.detach()))
    torch.manual_seed(0)
    c2, f2 = models.SirenNeRF().cuda(), models.SirenNeRF().cuda()
    step = NerfTrainStep(c2, f2, 2.0, 6.0, sc, sf, nb, learning_rate=lr)
    got = [float(step(rays, target, t_rand=t)[0]) for t in ts]
    print("SirenNeRF fused step losses", ["%.5f" % x for x in got], "autograd route", ["%.5f" % x for x in ref])
    np.testing.assert_allclose(got, ref, rtol=5e-3, atol=1e-5)
    assert step.global_step == 5 and torch.isfinite(step.params).all()


@pytest.mark.parametrize("rows_shape", [(37, 24), (700, 32), (1, 1), (300, 16, False)])
def test_film_siren_fused_training_path(rows_shape):
    """FiLM-SIREN on the fused tensor-core training path (film_tc_kernel<true> with bf16 tiles + cosine checkpoints,
    film_tc_bwd_kernel, MN-major wgrad on the FOLDED weights, film_grad_finish_kernel unfolding them into d W, d b, d gamma,
    d beta): the training forward is bit-identical to the inference kernel; every parameter gradient and d film[9,512] against
    the exact fp32 layer-wise path; the d-film-only call (synthesis.py:92-107: weights frozen) returns the same d film."""
    n, s = rows_shape[:2]
    g = torch.Generator().manual_seed(n + 11)
    net = seeded_film(use_dir=len(rows_shape) < 3)            # (.., False): FilmSirenNeRF(use_dir=False), 256-input hidden_layer_rgb
    film = torch.cat([1.0 + 0.1 * torch.randn(9, 256, generator=g), 0.1 * torch.randn(9, 256, generator=g)], -1).cuda().requires_grad_(True)
    o = torch.tensor([0.0, 0.0, 1.0]).expand(n, 3)
    d = torch.nn.functional.normalize(torch.randn(n, 3, generator=g) * 0.25 + torch.tensor([0.0, 0.0, -1.0]), dim=-1)
    rays = torch.stack([o, d], 1).cuda()
    z = (torch.sort(torch.rand(n, s, generator=g), -1).values * 1.0 + 0.5).cuda()
    up = torch.randn(n * s, 4, generator=g).cuda()
    net.set_film_params(film)
    with torch.no_grad():
        raw_inf = ops.mlp(net, rays=rays, z=z, precision="bf16", exact_last_sample=False)   # gradient passes run the raw bf16 forward
        raw_f32 = ops.mlp(net, rays=rays, z=z, precision="fp32")
    # relu(sigma) is a step function of the pre-activation's sign: on the few rows where bf16 rounds it across zero the
    # two paths differentiate different functions, so those rows get no upstream sigma gradient (teacher-forced parity)
    flips = (raw_inf[:, 3] > 0) != (raw_f32[:, 3] > 0)
    assert int(flips.sum()) <= max(2, n * s // 50)
    up[flips, 3] = 0.0
    res = {}
    for mode in ("fp32", "bf16"):
        old = ops.set_grad_precision(mode)
        try:
            net.zero_grad(set_to_none=True)
            film.grad = None
            net.set_film_params(film)
            raw = ops.mlp(net, rays=rays, z=z)
            (raw * up).sum().backward()
        finally:
            ops.set_grad_precision(old)
        grads = {k: p.grad.detach().clone() for k, p in net.named_parameters()}
        grads["film"] = film.grad.detach().clone()
        res[mode] = (raw.detach().clone(), grads)
    assert torch.equal(res["bf16"][0], raw_inf), "training forward differs from the inference kernel"
    assert (res["bf16"][0][:, :3] - res["fp32"][0][:, :3]).abs().max().item() < 2e-2
    worst = 0.0
    for k in res["fp32"][1]:
        gf, gb = res["fp32"][1][k].reshape(-1), res["bf16"][1][k].reshape(-1)
        rel = (gf - gb).norm().item() / max(gf.norm().item(), 1e-20)
        cos = torch.dot(gf, gb).item() / max(gf.norm().item() * gb.norm().item(), 1e-30)
        worst = max(worst, rel)
        assert torch.isfinite(gb).all()
        if n * s >= 4096:
            assert cos > 0.98 and rel < 0.12, (k, rel, cos)
        else:
            assert rel < 0.5, (k, rel)
    # weights frozen: only d film (no d_params buffer, no head wgrad)
    for p in net.parameters():
        p.requires_grad_(False)
    film.grad = None
    net.set_film_params(film)
    raw = ops.mlp(net, rays=rays, z=z)
    (raw * up).sum().backward()
    rel = (film.grad - res["bf16"][1]["film"]).norm().item() / max(res["bf16"][1]["film"].norm().item(), 1e-20)
    assert rel < 1e-3, rel                  # float atomics: the summation order differs between runs
    print("FiLM-SIREN fused training path (%d x %d rows): worst relative gradient error %.3g vs fp32" % (n, s, worst))


def test_pigan_render_batch_with_gradients_matches_per_latent_loop():
    """render_batch with autograd on (pi_GAN/train.py:134: Generator.forward's latent loop + loss.backward()): all latents go
    through ONE fused training forward / dgrad launch with per-latent folded weights, one wgrad launch per latent and the
    unfold kernel -- images bit-identical to the per-latent loop, d film[B,9,512] and the weight gradients equal up to the
    summation order of the float atomics."""
    torch.manual_seed(0)
    net = models.FilmSirenNeRF().cuda()
    g = torch.Generator().manual_seed(4)
    b, res, s_ = 3, 32, 8                                     # 32*32*16 = 16384 fine rows per latent
    film = torch.cat([1.0 + 0.2 * torch.randn(b, 9, 256, generator=g), 0.1 * torch.randn(b, 9, 256, generator=g)], -1).cuda().requires_grad_(True)
    poses = [pigan_render.camera_pos_to_transform_matrix(1, 0.3 * np.sin(i), 0.15 * np.cos(i)) for i in range(b)]
    focal = np.float64(res / 2 / np.tan(6 * np.pi / 180))
    t = torch.rand(b, res * res, s_, generator=g).cuda()
    target = torch.rand(b, 3, res, res, generator=g).cuda()
    imgs = pigan_render.render_batch(net, film, poses, res, res, focal, 0.5, 1.5, s_, s_, t_rand=t)
    ((imgs - target) ** 2).mean().backward()
    got = {k: p.grad.detach().clone() for k, p in net.named_parameters()}
    got["film"] = film.grad.detach().clone()
    net.zero_grad(set_to_none=True)
    film.grad = None
    loop = []
    for i in range(b):
        net.set_film_params(film[i])
        loop.append(pigan_render.render_image(res, res, focal, poses[i], 0.5, 1.5, net, net, s_, s_, t_rand=t[i]))
    loop = torch.stack(loop).permute(0, 3, 1, 2)
    ((loop - target) ** 2).mean().backward()
    assert torch.equal(imgs.detach(), loop.detach()), (imgs - loop).abs().max().item()
    ref = {k: p.grad.detach().clone() for k, p in net.named_parameters()}
    ref["film"] = film.grad.detach().clone()
    for k in ref:
        rel = (ref[k] - got[k]).norm().item() / max(ref[k].norm().item(), 1e-20)
        assert rel < 1e-3, (k, rel)
    assert got["film"].abs().sum(dim=(1, 2)).min().item() > 0          # every latent received its own d film


@pytest.mark.parametrize("shape", [(40000, 63, 128, 64, False), (33000, 23, 24, 24, True), (5000, 63, 64, 64, False), (3000, 31, 37, 18, False),
                                   (2000, 2, 5, 3, True)])
def test_sample_pdf_specialised_kernels_bit_identical_to_generic(shape):
    """b2r_sample_pdf runs instantiations with compile-time sizes for the BASELINE shapes (64+128, 64+64, 24+24): samples,
    merged rows and CDF must be bit-identical to the run-time-size kernel (b2r_sample_pdf_generic) on the same inputs --
    peaked / flat / zero weights, shared and per-ray bins, odd row lengths (both entries run the generic kernel there) -- and,
    given the kernel's CDF, to the oracle's searchsorted + lerp (north_star: indices bit-exact given identical CDFs)."""
    from msra_practice_project_b200._lib import lib, check
    n, nb, sf, sc, per_ray_bins = shape
    g = torch.Generator().manual_seed(nb * 1000 + sf)
    w_full = torch.rand(n, nb + 1, generator=g) ** 8                      # peaked, like compositing weights
    w_full[::7] = 0.0                                                    # all-zero rows: uniform pdf, denom clamp
    w_full[1::11, : nb // 2] = 0.0
    w_full = w_full.cuda()
    w = w_full[:, 1:-1] if nb > 2 else w_full[:, 1:2]                    # strided view, pointer + 1 (render_rays' weights[:, 1:-1])
    if per_ray_bins:
        bins = (torch.sort(torch.rand(n, nb, generator=g), -1).values * 4 + 2).cuda()
        b_stride = nb
    else:
        bins = torch.linspace(2.1, 5.9, nb).cuda()
        b_stride = 0
    u = torch.linspace(0.0, 1.0, sf, device="cpu").cuda()
    zc = (torch.sort(torch.rand(n, sc, generator=g), -1).values * 4 + 2).cuda()
    if not per_ray_bins:
        zc = zc.clamp(min=2.1)                                           # ties between coarse and fine entries (u = 0 -> bins[0] = 2.1)
    outs = {}
    for name in ("b2r_sample_pdf", "b2r_sample_pdf_generic"):
        samples = torch.full((n, sf), -1.0, device="cuda")
        merged = torch.full((n, sc + sf), -1.0, device="cuda")
        cdf = torch.full((n, nb), -1.0, device="cuda")
        fn = getattr(lib(), name)
        check(fn(bins.data_ptr(), b_stride, w.data_ptr(), w.stride(0), u.data_ptr(), n, nb, sf, zc.data_ptr(), sc, samples.data_ptr(),
                 merged.data_ptr(), cdf.data_ptr(), torch.cuda.current_stream().cuda_stream), name)
        # merge only (the render path's call: no samples / cdf output)
        merged2 = torch.full((n, sc + sf), -1.0, device="cuda")
        check(fn(bins.data_ptr(), b_stride, w.data_ptr(), w.stride(0), u.data_ptr(), n, nb, sf, zc.data_ptr(), sc, None, merged2.data_ptr(), None,
                 torch.cuda.current_stream().cuda_stream), name)
        torch.cuda.synchronize()
        assert torch.equal(merged, merged2)
        outs[name] = (samples, merged, cdf)
    a, b = outs["b2r_sample_pdf"], outs["b2r_sample_pdf_generic"]
    assert torch.equal(a[2], b[2]), "cdf"
    assert torch.equal(a[0], b[0]), "samples"
    assert torch.equal(a[1], b[1]), "merged"
    assert torch.equal(a[1], torch.sort(torch.cat([zc, a[0]], -1), -1).values)
    sub = slice(0, 512)
    ref, _ = orc.sample_pdf_from_cdf(bins[sub].cpu().numpy() if per_ray_bins else bins.cpu().numpy(), a[2][sub].cpu().numpy(), u.cpu().numpy())
    assert np.array_equal(a[0][sub].cpu().numpy(), ref)


@pytest.mark.parametrize("shape", [(70001, 63, 128, 64), (9000, 63, 64, 64), (20011, 23, 24, 24)])
@pytest.mark.parametrize("u_kind", ["linspace", "random", "negative"])
def test_sample_pdf_rank_kernel_on_render_rays_inputs(shape, u_kind):
    """The inputs render_rays really passes (nerf/render.py:126-142): bins = mid-points of the coarse strata, shared by all rays,
    z_coarse = jittered stratified samples (a few jitters exactly 0 or 1-ulp-below-1: coarse samples ON a stratum boundary, where
    the rank kernel's b + 1 / b + 2 guess is wrong and the ray is redone exactly), weights peaked / zero / flat.  b2r_sample_pdf
    (rank kernel: guess + verification, exact redo otherwise) must be bit-identical to b2r_sample_pdf_generic in samples, merged
    rows and CDF, for the reference's linspace u, for a sorted random u (perturbed sampling) and for a u that starts below zero
    (searchsorted index 0: the whole launch takes the exact path)."""
    from msra_practice_project_b200._lib import lib, check
    n, nb, sf, sc = shape
    g = torch.Generator().manual_seed(nb * 77 + sf)
    z_lin = torch.linspace(2.0, 6.0, sc)
    mids = 0.5 * (z_lin[1:] + z_lin[:-1])
    upper, lower = torch.cat([mids, z_lin[-1:]]), torch.cat([z_lin[:1], mids])
    t = torch.rand(n, sc, generator=g)
    t[::5, ::3] = 0.0                                                     # coarse sample exactly on the lower stratum boundary
    t[3::7, 1::4] = 1.0                                                   # ... on the upper one (ties with the next bin edge)
    zc = (lower + (upper - lower) * t).cuda().contiguous()
    w_full = torch.rand(n, sc, generator=g) ** 8
    w_full[::7] = 0.0
    w_full[1::11, : sc // 2] = 0.0
    w_full[2::13] = 1.0
    w_full[4::17, 5] = 50.0                                               # one dominant bin: most samples in one stratum
    w_full = w_full.cuda()
    w = w_full[:, 1:-1]
    bins = mids.cuda()
    if u_kind == "linspace":
        u = torch.linspace(0.0, 1.0, sf)
    elif u_kind == "random":
        u = torch.sort(torch.rand(sf, generator=g)).values
    else:
        u = torch.linspace(-0.05, 0.9, sf)
    u = u.cuda()
    outs = {}
    for name in ("b2r_sample_pdf", "b2r_sample_pdf_generic"):
        samples = torch.full((n, sf), -1.0, device="cuda")
        merged = torch.full((n, sc + sf), -1.0, device="cuda")
        cdf = torch.full((n, nb), -1.0, device="cuda")
        fn = getattr(lib(), name)
        check(fn(bins.data_ptr(), 0, w.data_ptr(), w.stride(0), u.data_ptr(), n, nb, sf, zc.data_ptr(), sc, samples.data_ptr(),
                 merged.data_ptr(), cdf.data_ptr(), torch.cuda.current_stream().cuda_stream), name)
        merged2 = torch.full((n, sc + sf), -1.0, device="cuda")
        check(fn(bins.data_ptr(), 0, w.data_ptr(), w.stride(0), u.data_ptr(), n, nb, sf, zc.data_ptr(), sc, None, merged2.data_ptr(), None,
                 torch.cuda.current_stream().cuda_stream), name)
        torch.cuda.synchronize()
        assert torch.equal(merged, merged2), name
        outs[name] = (samples, merged, cdf)
    a, b = outs["b2r_sample_pdf"], outs["b2r_sample_pdf_generic"]
    assert torch.equal(a[2], b[2]), "cdf"
    assert torch.equal(a[0], b[0]), "samples"
    assert torch.equal(a[1], b[1]), "merged"
    assert torch.equal(a[1], torch.sort(torch.cat([zc, a[0]], -1), -1).values)
    sub = slice(0, 512)
    ref, _ = orc.sample_pdf_from_cdf(bins.cpu().numpy(), a[2][sub].cpu().numpy(), u.cpu().numpy())
    assert np.array_equal(a[0][sub].cpu().numpy(), ref)


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_generator_forward_backward_vs_reference(golden, mode):
    """models.Generator.forward (pi_GAN/modules.py:176-184 + train.py:134) against the unmodified reference's Generator on the
    same z, poses (np.random.seed(3)) and jitter: image and the gradient of an image loss with respect to EVERY parameter of
    the FiLM-SIREN field and of the mapping network (which receives d film[B,9,512] from the renderer).  fp32: the exact
    per-latent path (1e-4 on the image); bf16: all latents in one fused launch sequence (2e-2 on the image)."""
    gg = golden.generator
    torch.manual_seed(0)
    gen = models.Generator(256, 8, near=0.5, far=1.5, fov=12, coarse_samples=8, fine_samples=8).cuda()
    z, target, t_rand = cu(gg["z"]), cu(gg["target"]), cu(gg["t_rand"])
    old_g = ops.set_grad_precision(mode)
    try:
        np.random.seed(3)
        img = gen(z, t_rand=t_rand, precision=mode)
        loss = ((img - target) ** 2).mean()
        loss.backward()
    finally:
        ops.set_grad_precision(old_g)
    err = (img.detach().cpu().numpy() - gg["img"])
    tol = 1e-4 if mode == "fp32" else 2e-2
    assert np.abs(err).max() < tol, np.abs(err).max()
    assert abs(float(loss.detach()) - float(gg["loss"])) < (1e-5 if mode == "fp32" else 2e-3)
    worst = 0.0
    for name, p in gen.named_parameters():
        assert p.grad is not None, name
        g = p.grad.detach().reshape(-1).double().cpu()
        ref_l2, ref_s = float(gg[f"g.{name}.l2"]), gg[f"g.{name}.sample"].astype(np.float64)
        got_s = g[::53].numpy()
        rel = np.linalg.norm(got_s - ref_s) / max(np.linalg.norm(ref_s), 1e-20)
        worst = max(worst, rel)
        if mode == "fp32":
            assert abs(float(g.norm()) - ref_l2) <= 2e-2 * ref_l2 + 1e-9 and rel < 2e-2, (name, rel, float(g.norm()), ref_l2)
        else:       # 128 rays: bf16 rounding is not averaged out (cf. test_film_siren_fused_training_path)
            assert abs(float(g.norm()) - ref_l2) <= 0.3 * ref_l2 + 1e-9 and rel < 0.5, (name, rel, float(g.norm()), ref_l2)
    print("Generator %s: image max-abs %.3g, worst relative gradient-sample error %.3g" % (mode, np.abs(err).max(), worst))


def test_ray_batcher_matches_train_nerf_batching():
    """train_step.RayBatcher against a numpy restatement of nerf/train_nerf.py:78-84 (shuffled [N*H*W,10] buffer), :125-137
    (start-up centre-crop sampler) and :139-145 (batch slices; the epoch 'reshuffle' that never takes effect) under the same
    np.random seed: identical pixel order (rgba bit-exact, ray origins bit-exact, directions to 1 ulp)."""
    from msra_practice_project_b200.train_step import RayBatcher
    rs = np.random.RandomState(1)
    n, h, w, bs = 3, 8, 12, 40
    images = rs.rand(n, h, w, 4).astype(np.float32)
    poses = np.stack([pigan_render.camera_pos_to_transform_matrix(4.0, 0.4 * i, -0.5 + 0.1 * i) for i in range(n)]).astype(np.float32)
    focal = w * 1.3875
    # reference arithmetic (numpy on the host)
    np.random.seed(7)
    rays = np.stack([np.stack(orc.get_rays(w, h, focal, p[:3, :4]), 0) for p in poses], 0)          # [N, ro+rd, H, W, 3]
    rays = np.reshape(np.transpose(rays, [0, 2, 3, 1, 4]), [-1, 6])
    ref = np.concatenate([rays, np.reshape(images, [-1, 4])], 1).astype(np.float32)
    np.random.shuffle(ref)
    si = np.random.choice(range(n))
    s_rays = np.reshape(np.transpose(np.stack(orc.get_rays(int(w / 2), int(h / 2), focal, poses[si][:3, :4]), 0), [1, 2, 0, 3]), [-1, 6])
    s_rgba = np.reshape(images[si][int(h / 4):int(h / 4) + int(h / 2), int(w / 4):int(w / 4) + int(w / 2)], [-1, 4])
    s_ref = np.concatenate([s_rays, s_rgba], 1).astype(np.float32)[np.random.choice(range(s_rays.shape[0]), size=bs // 2, replace=False)]
    # device batcher, same numpy stream
    np.random.seed(7)
    rb = RayBatcher(images, poses, focal, bs)
    got = rb.rays_rgba.cpu().numpy()
    assert got.shape == ref.shape == (n * h * w, 10)
    assert np.array_equal(got[:, 6:], ref[:, 6:]) and np.array_equal(got[:, :3], ref[:, :3])
    np.testing.assert_allclose(got[:, 3:6], ref[:, 3:6], rtol=3e-7, atol=1e-7)
    rb.batch = bs // 2
    r0, c0, a0 = rb.startup_batch()
    assert np.array_equal(torch.cat([c0, a0[:, None]], 1).cpu().numpy(), s_ref[:, 6:])
    np.testing.assert_allclose(r0.reshape(-1, 6).cpu().numpy(), s_ref[:, :6], rtol=3e-7, atol=1e-7)
    rb.batch = bs
    seen = []
    for _ in range(rb.batch_num + 1):                        # one epoch + the first batch of the next
        r, c, a = rb.next_batch()
        seen.append(torch.cat([r.reshape(-1, 6), c, a[:, None]], 1).cpu().numpy())
    assert np.array_equal(np.concatenate(seen[:-1])[:, 6:], ref[:, 6:])
    assert np.array_equal(seen[-1], seen[0])                 # as shipped, the reference never reorders the buffer
    rb2 = RayBatcher(images, poses, focal, bs, rank=1, world=2)
    assert rb2.next_batch()[0].shape == (bs // 2, 2, 3)


@pytest.mark.parametrize("graph", [False, True])
def test_train_step_takes_the_short_last_batch_of_an_epoch(graph):
    """nerf/train_nerf.py:139-150 trains on whatever the last slice of an epoch holds.  NerfTrainStep(batch_size=B) takes n < B rays:
    padded with zero-weight rays, loss normalised by n -- the same loss / PSNR / weights as a step built for exactly n rays."""
    from msra_practice_project_b200.train_step import NerfTrainStep, RayBatcher
    pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -0.5)
    sc, sf, big, small = 16, 24, 96, 40
    rays = ops.raygen(32, 24, 32 * 1.3875, pose, 100, big)
    g = torch.Generator().manual_seed(4)
    target, alpha = torch.rand(big, 3, generator=g).cuda(), torch.rand(big, generator=g).cuda()
    ts = [torch.rand(big, sc, generator=g).cuda() for _ in range(3)]
    def fresh(b):
        torch.manual_seed(0)
        c, f = models.damp_nerf_(models.NeRF()).cuda(), models.damp_nerf_(models.NeRF()).cuda()
        return NerfTrainStep(c, f, 2.0, 6.0, sc, sf, b, learning_rate=5e-4, use_alpha=True, graph=graph)
    small_step = fresh(small)
    ls, ps = small_step(rays[:small], target[:small], alpha[:small], t_rand=ts[1][:small])
    step = fresh(big)
    l, p_ = step(rays[:small], target[:small], alpha[:small], t_rand=ts[1][:small])           # the big trainer's first step is SHORT
    assert abs(float(l) - float(ls)) < 1e-5 * max(1.0, float(ls)) and abs(float(p_) - float(ps)) < 1e-3, (float(l), float(ls))
    dp = (step.params - small_step.params).abs()          # Adam's first step is +-lr: a near-zero gradient may flip sign with the atomics' order
    assert dp.max().item() <= 2 * 5e-4 + 1e-6 and dp.mean().item() < 2e-5, (dp.max().item(), dp.mean().item())
    for n_, t in ((big, ts[0]), (small, ts[2]), (big, ts[1])):                                 # full, short, full again
        l, p_ = step(rays[:n_], target[:n_], alpha[:n_], t_rand=t[:n_])
        assert np.isfinite(float(l)) and np.isfinite(float(p_))
    assert step.global_step == 4
    # the batcher + trainer run a whole epoch incl. its short last batch
    rs = np.random.RandomState(1)
    images = rs.rand(2, 6, 10, 4).astype(np.float32)                                   # 120 rays, batches of 32: 32, 32, 32, 24
    poses = np.stack([pigan_render.camera_pos_to_transform_matrix(4.0, 0.4 * i, -0.5) for i in range(2)]).astype(np.float32)
    rb = RayBatcher(images, poses, 10 * 1.3875, 32)
    torch.manual_seed(0)
    c, f = models.damp_nerf_(models.NeRF()).cuda(), models.damp_nerf_(models.NeRF()).cuda()
    tr = NerfTrainStep(c, f, 2.0, 6.0, sc, sf, 32, use_alpha=True, graph=graph)
    sizes = []
    for _ in range(rb.batch_num):
        r, cc, a = rb.next_batch()
        sizes.append(r.shape[0])
        l, _ = tr(r, cc, a, global_count=rb.global_count)
        assert np.isfinite(float(l))
    assert sizes == [32, 32, 32, 24] and tr.global_step == 4
    with pytest.raises(ValueError):
        RayBatcher(images, poses, 10 * 1.3875, 33, world=2)


def test_create_mesh_sdf_matches_density_query(golden):
    """pigan_render.create_mesh_sdf (the sampling half of create_mesh, pi_GAN/utils.py:42-97, as extract_mesh.py:49 calls it on a
    Generator): -sigma on the lattice equals the per-point MLP evaluation of the conditioned field (fp32 path 1e-4; the
    lattice coordinates themselves are pinned against the reference by test_mlp_fp32_film_and_grid's 6^3 golden)."""
    torch.manual_seed(0)
    gen = models.Generator(256, 16, near=0.5, far=1.5).cuda()
    z = torch.randn(1, 256, generator=torch.Generator().manual_seed(5)).cuda()
    n = 12
    sdf, origin, voxel = pigan_render.create_mesh_sdf(gen, N=n, max_batch=500, z=z, precision="fp32")
    assert tuple(sdf.shape) == (n, n, n) and origin == [-0.1, -0.1, -0.1] and abs(voxel - 0.2 / (n - 1)) < 1e-12
    idx = torch.arange(n ** 3)
    pts = torch.stack([(idx // n // n) % n, (idx // n) % n, idx % n], -1).float() * np.float32(voxel) + (-0.1)
    x = torch.cat([pts, torch.zeros_like(pts)], -1).cuda()
    with torch.no_grad():
        ref = -ops.mlp(gen.film_siren_nerf, x=x, precision="fp32")[:, 3]
    np.testing.assert_allclose(sdf.reshape(-1).numpy(), ref.cpu().numpy(), atol=1e-4, rtol=0)
    sdf_bf, _, _ = pigan_render.create_mesh_sdf(gen, N=n, z=z)
    assert np.abs(sdf_bf.numpy() - sdf.numpy()).max() < 2e-2


def test_bench_contract_one_json_line_with_all_keys():
    """bench.py's contract on a reduced frame: stdout carries exactly ONE JSON line with the driver's keys (metric, value, unit,
    n_gpus, steps, warmup, ms_per_step, higher_is_better, scaling, vs_baseline, dtype, data, config.workload, e2e with byte
    counts, gpu_launches, clocks, roofline with bound / achieved / peak / frac / traffic); everything else goes to stderr."""
    import json
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--width", "128", "--height", "128", "--steps", "2", "--warmup", "3",
                        "--no-cpu-baseline", "--no-secondary"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, r.stdout[:2000]
    d = json.loads(lines[0])
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data",
              "config", "e2e", "gpu_launches", "clocks", "roofline"):
        assert k in d, k
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["warmup"] >= 3 and d["unit"] == "rays/s" and d["value"] > 0
    assert "workload" in d["config"] and d["e2e"]["value"] > 0 and d["e2e"]["d2h_bytes_per_step"] == 128 * 128 * 5 * 4
    assert d["gpu_launches"] > 0 and d["roofline"]["bound"] == "tensor" and 0 < d["roofline"]["frac"] < 1.2
    for k in ("achieved", "peak", "unit", "traffic"):
        assert k in d["roofline"]


def test_bench_dump_outputs_are_the_seeded_render(tmp_path):
    """bench.py --dump-outputs writes the six per-ray maps of the last timed step as float32 .npy files, and they are the maps
    render_image_device returns for the bench's seeded inputs (weights seed 0, jitter seed 5, its camera)."""
    import sys
    w = h = 96
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--width", str(w), "--height", str(h), "--steps", "2", "--warmup", "3",
                        "--no-cpu-baseline", "--no-secondary", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    names = ("rgb_c", "depth_c", "acc_c", "rgb_f", "depth_f", "acc_f")
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(n + ".npy" for n in names)
    torch.manual_seed(0)
    coarse, fine = models.NeRF().cuda(), models.NeRF().cuda()
    pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)
    torch.manual_seed(5)
    t_rand = torch.rand((w * h, 64), device="cuda")
    with torch.no_grad():
        want = nerf_render.render_image_device(w, h, w * 1.3875, pose, 2.0, 6.0, coarse, fine, 64, 128, t_rand=t_rand, precision="bf16",
                                               exact_last_sample=True, coarse_outputs_unused=True)
    for name, ref in zip(names, want):
        got = np.load(tmp_path / (name + ".npy"))
        assert got.dtype == np.float32 and np.isfinite(got).all(), name
        assert np.array_equal(got, ref.cpu().numpy()), name


def test_film_batched_training_random_shapes():
    """tools/stress_film_train.py (random latent counts, rows per latent, samples per ray: odd tile counts, latents that
    start in the middle of a CTA's tile walk): the batched fused training call reproduces latent 0's rows bit-exactly and its
    d film to the summation order; no barrier-protocol hang (run under a timeout)."""
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "stress_film_train.py")], capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert r.returncode == 0 and "stress ok" in r.stdout, (r.stdout[-1500:], r.stderr[-1500:])


@pytest.mark.parametrize("kind", ["nerf", "siren", "film"])
def test_fused_training_full_size_properties(kind):
    """The fused tensor-core training path at BASELINE's full training shape (4096 rays x 256 MLP rows = 1,048,576 rows: too
    many for the fp32 comparison to be cheap) through size-independent properties:
      * head bias gradients are plain column sums of the head gradients: d b_sigma = sum_rows [sigma > 0] d_raw_sigma and
        d b_rgb = sum_rows d_raw_rgb * y (1 - y), recomputed here from (raw, d_raw) alone;
      * the reverse mode is linear in d_raw and scaling by 2 is exact in binary floating point (bf16 rounding included), so
        doubling the upstream gradient must double every gradient up to the summation order of the fp32 atomics;
      * everything is finite and no gradient tensor is identically zero."""
    g = torch.Generator().manual_seed(17)
    n, s = 4096, 256
    torch.manual_seed(0)
    film = None
    if kind == "nerf":
        net = models.damp_nerf_(models.NeRF()).cuda()
        sig_b, rgb_b = "output_layer_sigma.bias", "output_layer_rgb.bias"
    elif kind == "siren":
        net = models.SirenNeRF().cuda()
        sig_b, rgb_b = "output_layer_sigma.bias", "output_layer_rgb.bias"
    else:
        net = models.FilmSirenNeRF().cuda()
        film = torch.cat([1.0 + 0.1 * torch.randn(9, 256, generator=g), 0.1 * torch.randn(9, 256, generator=g)], -1).cuda().requires_grad_(True)
        sig_b, rgb_b = "output_layer_sigma.0.bias", "output_layer_rgb.0.bias"
    o = torch.tensor([0.0, 0.0, 1.2]).expand(n, 3)
    d = torch.nn.functional.normalize(torch.randn(n, 3, generator=g) * 0.25 + torch.tensor([0.0, 0.0, -1.0]), dim=-1)
    rays = torch.stack([o, d], 1).cuda()
    z = (torch.sort(torch.rand(n, s, generator=g), -1).values * 1.0 + 0.5).cuda()
    up = torch.randn(n * s, 4, generator=g).cuda()
    res = []
    for scale in (1.0, 2.0):
        net.zero_grad(set_to_none=True)
        if film is not None:
            film.grad = None
            net.set_film_params(film)
        raw = ops.mlp(net, rays=rays, z=z)
        assert raw.shape == (n * s, 4)
        (raw * (up * scale)).sum().backward()
        grads = {k: p.grad.detach().clone() for k, p in net.named_parameters()}
        if film is not None:
            grads["film"] = film.grad.detach().clone()
        res.append((raw.detach(), grads))
    raw, g1 = res[0]
    g2 = res[1][1]
    y = raw[:, :3].double()
    want_rgb = (up[:, :3].double() * y * (1 - y)).sum(0)
    want_sig = (up[:, 3].double() * (raw[:, 3] > 0)).sum()
    assert torch.allclose(g1[rgb_b].double(), want_rgb, rtol=2e-4, atol=2e-3), (g1[rgb_b], want_rgb)
    assert abs(g1[sig_b].double().item() - want_sig.item()) <= 2e-4 * abs(want_sig.item()) + 2e-2, (g1[sig_b], want_sig)
    for k in g1:
        a, b = g1[k].reshape(-1).double(), g2[k].reshape(-1).double()
        assert torch.isfinite(a).all() and a.abs().max() > 0, k
        rel = (2 * a - b).norm().item() / max(b.norm().item(), 1e-30)
        assert rel < 1e-4, (k, rel)


@pytest.mark.parametrize("kind", ["nerf", "film", "siren"])
def test_training_kernels_stay_inside_their_buffers(kind):
    """The training forward / reverse mode write exactly the bytes their size queries declare: `saved`, `scratch`, `d_folded`
    and the gradient buffers are carved out of larger allocations filled with a canary byte; after forward + backward through
    the C ABI every byte past the declared sizes is untouched and the declared regions were actually written."""
    import ctypes as C
    from msra_practice_project_b200._lib import lib, check, MlpInput
    L = lib()
    kid = {"nerf": models.KIND_NERF, "film": models.KIND_FILM, "siren": models.KIND_SIREN}[kind]
    torch.manual_seed(0)
    net = {"nerf": models.NeRF, "film": models.FilmSirenNeRF, "siren": models.SirenNeRF}[kind]().cuda()
    flat = models.flat_params(net).detach().contiguous()
    g = torch.Generator().manual_seed(5)
    n_lat, rows = (3, 3 * 1536) if kind == "film" else (1, 1000)          # FiLM: 3 latents x 1536 rows; others: a ragged count
    x = torch.cat([torch.rand(rows, 3, generator=g) - 0.5, torch.nn.functional.normalize(torch.randn(rows, 3, generator=g), dim=-1)], -1).cuda()
    d_raw = torch.randn(rows, 4, generator=g).cuda()
    inp = MlpInput()
    inp.x, inp.n_rays, inp.n_samples = x.data_ptr(), rows, 1
    st = torch.cuda.current_stream().cuda_stream
    pad, canary = 1 << 20, 0xCD

    def guarded(nbytes):
        buf = torch.full((nbytes + pad,), canary, dtype=torch.uint8, device="cuda")
        return buf

    def intact(buf, nbytes, name):
        assert bool((buf[nbytes:] == canary).all()), f"{name}: wrote past its {nbytes} declared bytes"
        assert not bool((buf[:nbytes] == canary).all()), f"{name}: never written"

    sv_bytes = L.b2r_mlp_tc_train_saved_bytes(kid, rows)
    sc_bytes = L.b2r_mlp_tc_train_scratch_bytes(kid, rows)
    saved, scratch = guarded(sv_bytes), guarded(sc_bytes)
    raw = guarded(rows * 16)
    n_par = flat.numel()
    d_params = guarded(n_par * 4)
    d_params[:n_par * 4] = 0
    if kind == "film":
        film = torch.cat([1.0 + 0.1 * torch.randn(n_lat, 9, 256, generator=g), 0.1 * torch.randn(n_lat, 9, 256, generator=g)], -1).cuda().contiguous()
        pk_bytes, pb_bytes = L.b2r_mlp_tc_packed_bytes(kid), L.b2r_mlp_tc_bwd_packed_bytes(kid)
        packed, packed_bwd = guarded(n_lat * pk_bytes), guarded(n_lat * pb_bytes)
        d_folded, d_film = guarded(n_lat * n_par * 4), guarded(n_lat * 4608 * 4)
        d_film[:n_lat * 4608 * 4] = 0
        check(L.b2r_mlp_tc_pack_film_batched(flat.data_ptr(), film.data_ptr(), 1, n_lat, packed.data_ptr(), st), "pack")
        check(L.b2r_mlp_tc_train_fwd_film_batched(packed.data_ptr(), n_lat, 1536, C.byref(inp), raw.data_ptr(), saved.data_ptr(), sv_bytes, None, st), "fwd")
        check(L.b2r_mlp_tc_pack_bwd_film(flat.data_ptr(), film.data_ptr(), 1, n_lat, packed_bwd.data_ptr(), st), "pack_bwd")
        check(L.b2r_mlp_tc_train_bwd_film(packed_bwd.data_ptr(), flat.data_ptr(), film.data_ptr(), 1, n_lat, 1536, rows, raw.data_ptr(), d_raw.data_ptr(),
                                          saved.data_ptr(), scratch.data_ptr(), sc_bytes, d_folded.data_ptr(), d_params.data_ptr(), d_film.data_ptr(),
                                          st), "bwd")
        torch.cuda.synchronize()
        for buf, nb, name in ((packed, n_lat * pk_bytes, "packed"), (packed_bwd, n_lat * pb_bytes, "packed_bwd"), (d_folded, n_lat * n_par * 4, "d_folded"),
                              (d_film, n_lat * 4608 * 4, "d_film")):
            intact(buf, nb, name)
    else:
        pk_bytes, pb_bytes = L.b2r_mlp_tc_packed_bytes(kid), L.b2r_mlp_tc_bwd_packed_bytes(kid)
        packed, packed_bwd = guarded(pk_bytes), guarded(pb_bytes)
        check(L.b2r_mlp_tc_pack(kid, flat.data_ptr(), None, 1, packed.data_ptr(), st), "pack")
        check(L.b2r_mlp_tc_train_fwd(kid, packed.data_ptr(), C.byref(inp), raw.data_ptr(), saved.data_ptr(), sv_bytes, None, st), "fwd")
        check(L.b2r_mlp_tc_pack_bwd(kid, flat.data_ptr(), packed_bwd.data_ptr(), st), "pack_bwd")
        check(L.b2r_mlp_tc_train_bwd(kid, packed_bwd.data_ptr(), rows, raw.data_ptr(), d_raw.data_ptr(), saved.data_ptr(), scratch.data_ptr(), sc_bytes,
                                     d_params.data_ptr(), st), "bwd")
        torch.cuda.synchronize()
        intact(packed, pk_bytes, "packed"); intact(packed_bwd, pb_bytes, "packed_bwd")
    intact(saved, sv_bytes, "saved"); intact(scratch, sc_bytes, "scratch"); intact(raw, rows * 16, "raw"); intact(d_params, n_par * 4, "d_params")
    gp = d_params[:n_par * 4].view(torch.float32)
    assert torch.isfinite(gp).all() and gp.abs().max() > 0
