"""Narrow-band mesh export (create_mesh(narrow_band=B)) against the dense density query, stage by stage, at 256^3, 512^3 and
1024^3.  Prints the card and its power limit and one JSON line.

Workloads:
  pigan  the sdf of a seeded models.Generator(256, 16) at level -20, input frequencies raised and the sigma head scaled as in
         tools/bench_mesh.py: one large piece and many blobs a few cells across, which bricks of B cells can miss;
  damp   models.damp_nerf_(models.NeRF()) (seed 0) on the default box [-1.5, 1.5]^3, threshold = 70th percentile of sigma;
  noise  the seeded NeRF of tools/bench_mesh.py (sigma head x100, zero bias), threshold = its 70th percentile: noise-like, the
         worst case, where nearly every brick is flagged (256^3 and 512^3 only: its dense 1024^3 mesh would not be useful).
Per size and brick edge B: the dense density query (density_grid / density_lattice), then the band stages with device events,
median of REPS after a warm-up: the coarse query (index list, lattice rows, sigma-only MLP, scatter into the +inf field), the
select (ops.band_select, including its one host read of M), the band query, and the masked marching cubes (count, host read of
(V, F), emit).  band_total_ms is the sum of the four, steps 2-6 of the extraction; queried_share = (coarse points + M) / points.
It also reports whether the band mesh equals the dense mesh and how many dense triangles it dropped."""
import json
import math
import os
import statistics
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from msra_practice_project_b200 import mesh, models, nerf_render, ops, pigan_render  # noqa: E402

REPS = 3


def _ev():
    e = torch.cuda.Event(enable_timing=True)
    e.record()
    return e


def _median_ms(fn, reps=REPS):
    ts, out = [], None
    for i in range(reps + 1):
        a = _ev()
        out = fn()
        b = _ev()
        torch.cuda.synchronize()
        if i:
            ts.append(a.elapsed_time(b))
    return statistics.median(ts), out


def band_stages(model, dims, level, stride, grid, lattice, max_batch):
    """mesh.band_field's steps (mesh.coarse_index, mesh.query_rows, ops.band_select) and the masked marching cubes, with an event
    between the stages: (times ms, field, flags, M, n coarse, verts, faces)."""
    dev = next(model.parameters()).device
    e = [_ev()]
    field = torch.full(tuple(dims), math.inf, dtype=torch.float32, device=dev)
    with torch.no_grad():
        coarse = mesh.coarse_index(dims, stride, dev)
        mesh.query_rows(model, field, coarse, grid=grid, lattice=lattice, max_batch=max_batch)
        e.append(_ev())
        flags, index = ops.band_select(field, level, stride)
        e.append(_ev())
        mesh.query_rows(model, field, index, grid=grid, lattice=lattice, max_batch=max_batch)
        e.append(_ev())
        verts, faces = ops.marching_cubes(field, level, bricks=(stride, flags))
        e.append(_ev())
    torch.cuda.synchronize()
    ms = [e[i].elapsed_time(e[i + 1]) for i in range(4)]
    return ms, field, flags, int(index.shape[0]), int(coarse.numel()), verts, faces


def run(name, model, dims, level, grid, lattice, dense_fn, strides, max_batch):
    q_ms, field = _median_ms(dense_fn)
    dv, df = ops.marching_cubes(field, level)
    pts = math.prod(dims)
    res = {"dims": list(dims), "level": level, "dense_query_ms": round(q_ms, 3), "dense_F": int(df.shape[0]), "bands": {}}
    for stride in strides:
        runs = [band_stages(model, dims, level, stride, grid, lattice, max_batch) for _ in range(REPS + 1)][1:]
        ms = [statistics.median(r[0][i] for r in runs) for i in range(4)]
        _, bfield, flags, m, nc, bv, bf = runs[-1]
        total = sum(ms)
        res["bands"][str(stride)] = {
            "coarse_query_ms": round(ms[0], 3), "select_ms": round(ms[1], 3), "band_query_ms": round(ms[2], 3),
            "masked_mc_ms": round(ms[3], 3), "band_total_ms": round(total, 3), "band_over_dense_query": round(total / q_ms, 3),
            "coarse_points": nc, "band_points": m, "queried_share": round((nc + m) / pts, 4),
            "flagged_bricks": int(flags.sum()), "bricks": int(flags.numel()), "band_F": int(bf.shape[0]),
            "equals_dense_mesh": bool(torch.equal(bv, dv) and torch.equal(bf, df)),
            "dropped_dense_triangles": int(df.shape[0] - bf.shape[0])}
        del bfield
    print(name, json.dumps(res), flush=True)
    return res


def main():
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                         text=True)
    gpu = smi.stdout.strip().splitlines()[0] if smi.returncode == 0 and smi.stdout.strip() else "unknown"
    print("gpu:", gpu)
    assert torch.cuda.is_available(), "bench_mesh_band needs a CUDA device"
    sizes = [int(s) for s in sys.argv[1:]] or [256, 512, 1024]
    out = {"metric": "narrow-band create_mesh: coarse query, select, band query, masked marching cubes vs the dense query", "gpu": gpu,
           "pigan": {}, "damp": {}, "noise": {}}
    torch.manual_seed(0)
    gen = models.Generator(256, 16).cuda()
    z = torch.randn(1, 256, generator=torch.Generator().manual_seed(3)).cuda()
    with torch.no_grad():
        net = gen.film_siren_nerf
        net.input_layer.weight.mul_(20.0)
        net.output_layer_sigma[0].weight.mul_(100.0)
        net.output_layer_sigma[0].bias.zero_()
        gen.set_film_params(gen.get_mapping(z)[0])
    for n in sizes:
        out["pigan"][n] = run("pigan", net, (n, n, n), -20.0, (n, 0, n ** 3), None,
                              lambda: pigan_render.density_grid(net, N=n).reshape(n, n, n), (4, 8), 64 ** 3)
    torch.manual_seed(0)
    damp = models.damp_nerf_(models.NeRF()).cuda()
    torch.manual_seed(0)
    noise = models.NeRF().cuda()
    with torch.no_grad():
        noise.output_layer_sigma.weight.mul_(100.0)
        noise.output_layer_sigma.bias.zero_()
    for key, model, top in (("damp", damp, 1024), ("noise", noise, 512)):
        for n in [s for s in sizes if s <= top]:
            dims, origin, voxel = mesh.box_lattice((-1.5,) * 3, (1.5,) * 3, n)
            sigma = nerf_render.density_lattice(model, N=n)[0]
            thr = float(torch.quantile(sigma.flatten()[::97].float(), 0.7))
            del sigma
            out[key][n] = run(key, model, dims, -thr, None, (dims, origin, voxel, 0, math.prod(dims)),
                              lambda: nerf_render.density_lattice(model, N=n)[0].neg_(), (4, 8), 256 ** 3)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
