"""create_mesh on the device, stage by stage, at N = 256 and 512 (pi_GAN/extract_mesh.py runs N = 512): the density query,
marching cubes (b2r_mc_count + b2r_mc_emit, device events, median of 20 after warm-up; the host read of (V, F) between the two
calls timed on its own), the mesh's size and bytes moved, and the mesh D2H + PLY write.  Prints the card and its power limit
and one JSON line.  The field is the sdf of a seeded models.Generator(256, 16) at the reference's level -20; untrained, its
sigma is 0 on the whole box, so (as in tests/test_gpu_mesh.py) the input layer's frequencies are raised and the sigma head is
centred and scaled.  The 256^3 field (67 MB) fits in the 126 MB L2, the 512^3 one (537 MB) does not.  Also times the numpy oracle at 128^3 on the host, for scale."""
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from msra_practice_project_b200 import models, ops, pigan_render  # noqa: E402
from msra_practice_project_b200._lib import check, lib, ptr  # noqa: E402
from oracle import marching_cubes as mc  # noqa: E402

COPY_PEAK_GBS = 6554.0      # measured HBM copy peak of the B200 (DESIGN.md §3)
REPS = 20


def _events():
    return torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)


def density_ms(gen, n, reps=3):
    ts = []
    for i in range(reps + 1):
        a, b = _events()
        a.record()
        sdf = pigan_render.density_grid(gen.film_siren_nerf, N=n)
        b.record()
        torch.cuda.synchronize()
        if i:
            ts.append(a.elapsed_time(b))
    return statistics.median(ts), sdf.reshape(n, n, n)


def mc_times(field, level, spacing, origin):
    n0, n1, n2 = field.shape
    scratch = torch.empty((lib().b2r_mc_scratch_bytes(n0, n1, n2),), dtype=torch.uint8, device=field.device)
    totals = torch.empty((2,), dtype=torch.int64, device=field.device)
    st = torch.cuda.current_stream().cuda_stream
    dev_ms, host_ms = [], []
    verts = faces = None
    for i in range(REPS + 3):
        e0, e1 = _events()
        e2, e3 = _events()
        e0.record()
        check(lib().b2r_mc_count(ptr(field), n0, n1, n2, level, ptr(scratch), ptr(totals), st), "b2r_mc_count")
        e1.record()
        t0 = time.perf_counter()
        nv, nf = (int(v) for v in totals.tolist())
        t1 = time.perf_counter()
        if verts is None:
            verts = torch.empty((nv, 3), dtype=torch.float32, device=field.device)
            faces = torch.empty((nf, 3), dtype=torch.int32, device=field.device)
        e2.record()
        check(lib().b2r_mc_emit(ptr(field), n0, n1, n2, level, spacing, *origin, ptr(scratch), ptr(verts), ptr(faces), st),
              "b2r_mc_emit")
        e3.record()
        torch.cuda.synchronize()
        if i >= 3:
            dev_ms.append(e0.elapsed_time(e1) + e2.elapsed_time(e3))
            host_ms.append((t1 - t0) * 1e3)
    return statistics.median(dev_ms), statistics.median(host_ms), verts, faces


def mc_bytes(n0, n1, n2, nv, nf):
    """Bytes the four passes move, from shapes: count reads the field and writes a word per point, vertices and faces read
    the words, vertices reads f(p) and f(p + e_a) per vertex; 12 B per vertex and per triangle written; tile counts and
    offsets (4 + 16 B per 2,048-point tile) written once and read twice."""
    n = n0 * n1 * n2
    tiles = -(-n // 2048)
    return 16 * n + 8 * nv + 12 * nv + 12 * nf + tiles * (4 + 4 + 16 + 16 + 16)


def main():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    print("gpu:", smi.stdout.strip().splitlines()[0] if smi.returncode == 0 and smi.stdout.strip() else "unknown")
    assert torch.cuda.is_available(), "bench_mesh needs a CUDA device"
    torch.manual_seed(0)
    gen = models.Generator(256, 16).cuda()
    z = torch.randn(1, 256, generator=torch.Generator().manual_seed(3)).cuda()
    with torch.no_grad():
        net = gen.film_siren_nerf
        net.input_layer.weight.mul_(20.0)
        net.output_layer_sigma[0].weight.mul_(100.0)
        net.output_layer_sigma[0].bias.zero_()
        gen.set_film_params(gen.get_mapping(z)[0])
    out = {"metric": "create_mesh on the device: density query, marching cubes, mesh D2H + PLY", "gpu": smi.stdout.strip(),
           "copy_peak_GBs": COPY_PEAK_GBS, "sizes": {}}
    for n in (256, 512):
        q_ms, sdf = density_ms(gen, n)
        lo, hi = float(sdf.min()), float(sdf.max())
        level = -20.0
        spacing, origin = 0.2 / (n - 1), (-0.1, -0.1, -0.1)
        dev_ms, host_ms, verts, faces = mc_times(sdf, level, spacing, origin)
        ref_v, ref_f = ops.marching_cubes(sdf, level, spacing, origin)
        same = bool(torch.equal(ref_v, verts) and torch.equal(ref_f, faces))
        nb = mc_bytes(n, n, n, verts.shape[0], faces.shape[0])
        with tempfile.TemporaryDirectory() as tmp:
            ts = []
            for _ in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                pigan_render.write_ply(os.path.join(tmp, "mesh.ply"), verts.cpu().numpy(), faces.cpu().numpy())
                ts.append((time.perf_counter() - t0) * 1e3)
            ply_bytes = os.path.getsize(os.path.join(tmp, "mesh.ply"))
        out["sizes"][str(n)] = {
            "density_query_ms": round(q_ms, 3), "sdf_range": [lo, hi], "level": level, "marching_cubes_device_ms": round(dev_ms, 4),
            "host_read_VF_ms": round(host_ms, 4), "V": int(verts.shape[0]), "F": int(faces.shape[0]), "bytes": int(nb),
            "GBs": round(nb / (dev_ms * 1e-3) / 1e9, 1), "frac_of_copy_peak": round(nb / (dev_ms * 1e-3) / 1e9 / COPY_PEAK_GBS, 3),
            "mc_over_query": round(dev_ms / q_ms, 4), "d2h_plus_ply_ms": round(statistics.median(ts), 2), "ply_bytes": ply_bytes,
            "repeat_run_identical": same, "field_fits_l2": n ** 3 * 4 < 126e6}
        del sdf, verts, faces, ref_v, ref_f
        torch.cuda.empty_cache()
    # the numpy oracle at 128^3, host only, for scale
    sdf = pigan_render.density_grid(gen.film_siren_nerf, N=128).reshape(128, 128, 128).cpu().numpy()
    t0 = time.perf_counter()
    v, f = mc.marching_cubes(sdf, -20.0, 0.2 / 127, (-0.1, -0.1, -0.1))
    out["numpy_oracle_128_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
    out["numpy_oracle_128_VF"] = [int(len(v)), int(len(f))]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
