"""create_mesh on the device, stage by stage, at N = 256 and 512 (pi_GAN/extract_mesh.py runs N = 512): the density query,
marching cubes (b2r_mc_count + b2r_mc_emit, device events, median of 20 after warm-up; the host read of (V, F) between the two
calls timed on its own), the mesh's size and bytes moved, and the mesh D2H + PLY write.  Prints the card and its power limit
and one JSON line.  The field is the sdf of a seeded models.Generator(256, 16) at the reference's level -20; untrained, its
sigma is 0 on the whole box, so (as in tests/test_gpu_mesh.py) the input layer's frequencies are raised and the sigma head is
centred and scaled.  The 256^3 field (67 MB) fits in the 126 MB L2, the 512^3 one (537 MB) does not.  Also times the numpy oracle at 128^3 on the host, for scale.

The NeRF lines time nerf_render.create_mesh stage by stage on the default box [-1.5, 1.5]^3 of a seeded models.NeRF whose sigma
head is scaled by 100 with a zeroed bias (the threshold is the 70th percentile of its sigma): the box-lattice density query
(bf16 sigma-only kernel) in ms and points/s, marching cubes, the vertex normals (b2r_mc_normals), the colour query at
x = [vertex, -normal] with to8b, the D2H copy + PLY write with normals and colours, and one whole create_mesh call that writes the
coloured PLY.

The "components" entries time the connected-component stages of both meshes (b2r_mesh_cc_label, _select at ratio 0.01 without
the host read of (V', F'), _compact; device events, median of 20 after warm-up; the pi-GAN mesh without normals, the NeRF one
with them): ms and triangles/s per stage, the least bytes each stage moves against the copy peak, the number of components,
(V', F'), and their share of the density query.  For the NeRF mesh also the colour query, the D2H + PLY write and one whole
create_mesh(min_component_ratio=0.01) call on the filtered mesh, against the unfiltered numbers above.

The "smoothing" entries time Taubin smoothing on the pi-GAN 512^3 mesh and both NeRF meshes (b2r_mesh_adjacency, one
b2r_mesh_smooth call of SMOOTH_ITERS iterations divided by SMOOTH_ITERS, b2r_mesh_normals; device events, median of 20 after a
warm-up): ms per stage, the least bytes each stage moves (smooth_bytes) against the copy peak, the scratch bytes and the peak of
torch's allocator over one ops.smooth_mesh(normals=True) call above what was allocated before it, and a check against that call.
For the NeRF meshes also one whole create_mesh(smooth_iterations=SMOOTH_ITERS) call against the unsmoothed one above, and whether
it equals its stages (ops.smooth_mesh, then the colour query).

The "decimation" entries (``--decimation`` runs only these) time ops.decimate_mesh on the pi-GAN 512^3 mesh down to 25,000 faces
and on the NeRF 512^3 mesh down to 1,000,000: the number of rounds and the collapses of each, the wall time of the whole call
(host clock around a call that ends in a device synchronise; it includes the one host read per round) and its mean per round,
and the peak of torch's allocator over the call above what was allocated before it.  For the NeRF mesh also one whole
create_mesh(max_faces=1_000_000) call against create_mesh() on the same field, each split into the call without a PLY (device
work and the host reads) and the D2H copy + PLY write of its outputs, and whether the decimated call equals its stages
(ops.decimate_mesh, the mesh normals, the colour query)."""
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

from msra_practice_project_b200 import mesh, models, nerf_render, ops, pigan_render  # noqa: E402
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


def _timed(fn, reps):
    """(median device ms over reps after one warm-up, last result) of fn() between two events."""
    ts, res = [], None
    for i in range(reps + 1):
        a, b = _events()
        a.record()
        res = fn()
        b.record()
        torch.cuda.synchronize()
        if i:
            ts.append(a.elapsed_time(b))
    return statistics.median(ts), res


CC_RATIO = 0.01


def cc_bytes(nv, nf, kv, kf, normals):
    """Bytes the component stages move at the least, from the mesh's sizes: label writes parent[V], reads the faces (12 B each)
    and finds every face's three roots, then reads parent[V] and writes labels[V] (16 B/vertex + 12 B/face before any parent
    traffic of the finds); select clears the counts, reads a label per face for the counts and again for the marks, the counts
    and labels per vertex, and writes a word per vertex (16 B/vertex + 32 B/face); compact reads the words, the vertices (and
    normals) and the faces, and writes what is kept."""
    w = 24 if normals else 12
    return {"label": 16 * nv + 12 * nf, "select": 16 * nv + 32 * nf, "compact": (4 + w) * nv + w * kv + 12 * nf + 12 * kf}


def cc_times(verts, faces, normals, ratio=CC_RATIO):
    """Device ms (median of REPS after 3 warm-ups) of b2r_mesh_cc_label, b2r_mesh_cc_select and b2r_mesh_cc_compact, plus the
    number of components (vertices that are their own label), (V', F') and a check against ops.filter_components."""
    nv, nf = verts.shape[0], faces.shape[0]
    dev = verts.device
    st = torch.cuda.current_stream().cuda_stream
    scratch = torch.empty((lib().b2r_mesh_cc_scratch_bytes(nv, nf),), dtype=torch.uint8, device=dev)
    labels = torch.empty((nv,), dtype=torch.int32, device=dev)
    totals = torch.empty((2,), dtype=torch.int64, device=dev)
    label = lambda: check(lib().b2r_mesh_cc_label(ptr(faces), nf, nv, ptr(labels), ptr(scratch), st), "b2r_mesh_cc_label")  # noqa: E731
    select = lambda: check(lib().b2r_mesh_cc_select(ptr(faces), nf, nv, ptr(labels), ratio, ptr(scratch), ptr(totals), st),  # noqa: E731
                           "b2r_mesh_cc_select")
    ms = {}
    ms["label"], _ = _timed(label, REPS)
    ms["select"], _ = _timed(select, REPS)
    kv, kf = (int(v) for v in totals.tolist())
    v_out = torch.empty((kv, 3), dtype=torch.float32, device=dev)
    n_out = None if normals is None else torch.empty((kv, 3), dtype=torch.float32, device=dev)
    f_out = torch.empty((kf, 3), dtype=torch.int32, device=dev)
    compact = lambda: check(lib().b2r_mesh_cc_compact(ptr(verts), ptr(normals), ptr(faces), nf, nv, ptr(scratch), ptr(v_out), ptr(n_out),  # noqa: E731
                                                      ptr(f_out), st), "b2r_mesh_cc_compact")
    ms["compact"], _ = _timed(compact, REPS)
    n_comp = int((labels == torch.arange(nv, dtype=torch.int32, device=dev)).sum())
    ref = ops.filter_components(verts, faces, ratio, normals)
    same = bool(torch.equal(ref[0], v_out) and torch.equal(ref[1], f_out) and (normals is None or torch.equal(ref[2], n_out)))
    nb = cc_bytes(nv, nf, kv, kf, normals is not None)
    out = {"components": n_comp, "ratio": ratio, "V_kept": kv, "F_kept": kf, "equals_ops_filter_components": same}
    for k in ("label", "select", "compact"):
        out[f"{k}_ms"] = round(ms[k], 4)
        out[f"{k}_Gtri_per_s"] = round(nf / (ms[k] * 1e-3) / 1e9, 3)
        out[f"{k}_min_bytes"] = nb[k]
        out[f"{k}_frac_of_copy_peak"] = round(nb[k] / (ms[k] * 1e-3) / 1e9 / COPY_PEAK_GBS, 3)
    out["total_ms"] = round(sum(ms.values()), 4)
    out["parent_bytes"] = 4 * nv
    out["parent_fits_l2"] = 4 * nv < 126e6
    del scratch, labels, v_out, n_out, f_out, ref
    return out


SMOOTH_ITERS = 10


def smooth_bytes(nv, nf):
    """Bytes the smoothing stages move at the least, from the mesh's sizes (neighbour positions gathered through the corner
    records are not counted): the adjacency build reads the faces three times (count, fill, the sort's record lookup; 36 B/face),
    writes the 8-byte corner keys, then reads and rewrites them as records (72 B/face), and touches ends[] five times (40 B/vertex);
    a half-step reads ends[], the records and its own position and writes one (32 B/vertex + 24 B/face), an iteration is two;
    the normals read ends[], the records and a position and write a normal (32 B/vertex + 24 B/face)."""
    return {"adjacency": 40 * nv + 108 * nf, "iteration": 2 * (32 * nv + 24 * nf), "normals": 32 * nv + 24 * nf}


def smooth_times(verts, faces):
    """Device ms of b2r_mesh_adjacency, of one Taubin iteration and of b2r_mesh_normals, their least bytes against the copy
    peak, the adjacency's memory, and a check against ops.smooth_mesh."""
    nv, nf = verts.shape[0], faces.shape[0]
    dev = verts.device
    st = torch.cuda.current_stream().cuda_stream
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    ref_v, ref_n = ops.smooth_mesh(verts, faces, SMOOTH_ITERS, normals=True)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated(dev) - base
    nbytes = lib().b2r_mesh_adj_scratch_bytes(nv, nf)
    scratch = torch.empty((nbytes,), dtype=torch.uint8, device=dev)
    out_v, out_n = torch.empty_like(verts), torch.empty_like(verts)
    adj = lambda: check(lib().b2r_mesh_adjacency(ptr(faces), nf, nv, ptr(scratch), st), "b2r_mesh_adjacency")  # noqa: E731
    ms = {}
    ms["adjacency"], _ = _timed(adj, REPS)
    ms["iteration"], _ = _timed(lambda: check(lib().b2r_mesh_smooth(ptr(verts), nf, nv, SMOOTH_ITERS, ptr(scratch), ptr(out_v), st),
                                              "b2r_mesh_smooth"), REPS)
    ms["iteration"] /= SMOOTH_ITERS
    ms["normals"], _ = _timed(lambda: check(lib().b2r_mesh_normals(ptr(out_v), nf, nv, ptr(scratch), ptr(out_n), st), "b2r_mesh_normals"),
                              REPS)
    nb = smooth_bytes(nv, nf)
    out = {"iterations": SMOOTH_ITERS, "equals_ops_smooth_mesh": bool(torch.equal(ref_v, out_v) and torch.equal(ref_n, out_n)),
           "scratch_bytes": int(nbytes), "peak_alloc_bytes_smooth_mesh_call": int(peak)}
    for k in ("adjacency", "iteration", "normals"):
        out[f"{k}_ms"] = round(ms[k], 4)
        out[f"{k}_min_bytes"] = nb[k]
        out[f"{k}_frac_of_copy_peak"] = round(nb[k] / (ms[k] * 1e-3) / 1e9 / COPY_PEAK_GBS, 3)
    out["total_ms"] = round(ms["adjacency"] + SMOOTH_ITERS * ms["iteration"] + ms["normals"], 4)
    del scratch, out_v, out_n
    return out, ref_v, ref_n


NERF_TRUNK_FLOP = 2 * (60 * 256 + 4 * 256 * 256 + 316 * 256 + 2 * 256 * 256 + 256)    # 8-layer trunk + sigma head, per point


def nerf_lines():
    torch.manual_seed(0)
    net = models.NeRF().cuda()
    with torch.no_grad():
        net.output_layer_sigma.weight.mul_(100.0)
        net.output_layer_sigma.bias.zero_()
    res = {}
    for n in (256, 512):
        q_ms, (sigma, origin, voxel) = _timed(lambda: nerf_render.density_lattice(net, N=n), 3)
        pts = sigma.numel()
        thr = float(torch.quantile(sigma.flatten()[::97].float(), 0.7))
        field = -sigma
        dev_ms, host_ms, verts, faces = mc_times(field, -thr, voxel, origin)
        n0, n1, n2 = field.shape
        scratch = torch.empty((lib().b2r_mc_scratch_bytes(n0, n1, n2),), dtype=torch.uint8, device=field.device)
        totals = torch.empty((2,), dtype=torch.int64, device=field.device)
        st = torch.cuda.current_stream().cuda_stream
        check(lib().b2r_mc_count(ptr(field), n0, n1, n2, -thr, ptr(scratch), ptr(totals), st), "b2r_mc_count")
        nrm = torch.empty_like(verts)
        nrm_ms, _ = _timed(lambda: check(lib().b2r_mc_normals(ptr(field), n0, n1, n2, -thr, ptr(scratch), ptr(nrm), st), "b2r_mc_normals"),
                           REPS)
        col_ms, rgb = _timed(lambda: mesh.vertex_colors(net, verts, nrm), 5)
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "mesh.ply")
            ts = []
            for _ in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                mesh.write_ply(path, verts.cpu().numpy(), faces.cpu().numpy(), nrm.cpu().numpy(), rgb.cpu().numpy())
                ts.append((time.perf_counter() - t0) * 1e3)
            ply_bytes = os.path.getsize(path)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            whole = nerf_render.create_mesh(net, path, n, threshold=thr)
            torch.cuda.synchronize()
            whole_ms = (time.perf_counter() - t0) * 1e3
        same = bool(torch.equal(whole[0], verts) and torch.equal(whole[1], faces) and torch.equal(whole[2], nrm) and torch.equal(whole[3], rgb))
        del whole
        cc = cc_times(verts, faces, nrm)
        cc["over_density_query"] = round(cc["total_ms"] / q_ms, 4)
        fv, ff, fn = ops.filter_components(verts, faces, CC_RATIO, nrm)
        cc["color_query_filtered_ms"], frgb = _timed(lambda: mesh.vertex_colors(net, fv, fn), 5)
        cc["color_query_filtered_ms"] = round(cc["color_query_filtered_ms"], 3)
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "mesh.ply")
            fts = []
            for _ in range(2):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                mesh.write_ply(path, fv.cpu().numpy(), ff.cpu().numpy(), fn.cpu().numpy(), frgb.cpu().numpy())
                fts.append((time.perf_counter() - t0) * 1e3)
            cc["d2h_plus_ply_filtered_ms"] = round(statistics.median(fts), 2)
            cc["ply_bytes_filtered"] = os.path.getsize(path)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            whole = nerf_render.create_mesh(net, path, n, threshold=thr, min_component_ratio=CC_RATIO)
            torch.cuda.synchronize()
            cc["create_mesh_call_filtered_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
        cc["create_mesh_filtered_equals_stages"] = bool(torch.equal(whole[0], fv) and torch.equal(whole[1], ff) and torch.equal(whole[2], fn)
                                                        and torch.equal(whole[3], frgb))
        del fv, ff, fn, frgb
        sm, sv, sn = smooth_times(verts, faces)
        sm["over_density_query"] = round(sm["total_ms"] / q_ms, 4)
        srgb = mesh.vertex_colors(net, sv, sn)
        with tempfile.TemporaryDirectory() as tmp:
            path = os.path.join(tmp, "mesh.ply")
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            whole = nerf_render.create_mesh(net, path, n, threshold=thr, smooth_iterations=SMOOTH_ITERS)
            torch.cuda.synchronize()
            sm["create_mesh_call_smoothed_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
        sm["create_mesh_smoothed_equals_stages"] = bool(torch.equal(whole[0], sv) and torch.equal(whole[1], faces)
                                                        and torch.equal(whole[2], sn) and torch.equal(whole[3], srgb))
        del sv, sn, srgb
        res[str(n)] = {
            "dims": list(field.shape), "points": pts, "density_query_ms": round(q_ms, 3), "points_per_s": round(pts / (q_ms * 1e-3) / 1e9, 3),
            "points_per_s_unit": "G/s", "trunk_TFLOPs": round(pts * NERF_TRUNK_FLOP / (q_ms * 1e-3) / 1e12, 1), "threshold": thr,
            "marching_cubes_device_ms": round(dev_ms, 4), "host_read_VF_ms": round(host_ms, 4), "normals_ms": round(nrm_ms, 4),
            "color_query_ms": round(col_ms, 3), "V": int(verts.shape[0]), "F": int(faces.shape[0]),
            "d2h_plus_ply_ms": round(statistics.median(ts), 2), "ply_bytes": ply_bytes, "create_mesh_call_ms": round(whole_ms, 1),
            "create_mesh_equals_stages": same, "components": cc, "smoothing": sm}
        del sigma, field, verts, faces, nrm, rgb, whole, scratch
        torch.cuda.empty_cache()
    return res


DEC_PIGAN, DEC_NERF = 25_000, 1_000_000


def decimate_times(verts, faces, max_faces):
    """Rounds, wall ms of one ops.decimate_mesh call (and per round), allocator peak above the inputs, (V', F')."""
    dev = verts.device
    ops._decimate_mesh(verts, faces, max_faces)                  # warm-up
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    stats = {}
    t0 = time.perf_counter()
    dv, df = ops._decimate_mesh(verts, faces, max_faces, stats)
    torch.cuda.synchronize()
    ms = (time.perf_counter() - t0) * 1e3
    peak = torch.cuda.max_memory_allocated(dev) - base
    again = ops._decimate_mesh(verts, faces, max_faces)
    return {"V": int(verts.shape[0]), "F": int(faces.shape[0]), "max_faces": max_faces, "V_out": int(dv.shape[0]), "F_out": int(df.shape[0]),
            "rounds": stats["rounds"], "collapses_per_round": stats["collapses"], "call_ms": round(ms, 2),
            "mean_ms_per_round": round(ms / max(1, stats["rounds"]), 3), "peak_alloc_bytes": int(peak),
            "repeat_run_identical": bool(torch.equal(again[0], dv) and torch.equal(again[1], df))}, dv, df


def _call_split(fn, path):
    """(ms of fn(None) ended by a device synchronise, ms of the D2H copy + PLY write of its outputs, the outputs)."""
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn(None)
    torch.cuda.synchronize()
    dev_ms = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    mesh.write_ply(path, *(t.cpu().numpy() for t in out))
    return dev_ms, (time.perf_counter() - t0) * 1e3, out


def decimation_lines(gen):
    res = {}
    sdf = pigan_render.density_grid(gen.film_siren_nerf, N=512).reshape(512, 512, 512)
    verts, faces = ops.marching_cubes(sdf, -20.0, 0.2 / 511, (-0.1, -0.1, -0.1))
    res["pigan_512"] = decimate_times(verts, faces, DEC_PIGAN)[0]
    del sdf, verts, faces
    torch.manual_seed(0)
    net = models.NeRF().cuda()
    with torch.no_grad():
        net.output_layer_sigma.weight.mul_(100.0)
        net.output_layer_sigma.bias.zero_()
    sigma, origin, voxel = nerf_render.density_lattice(net, N=512)
    thr = float(torch.quantile(sigma.flatten()[::97].float(), 0.7))
    verts, faces = ops.marching_cubes(-sigma, -thr, voxel, origin)
    del sigma
    torch.cuda.empty_cache()
    d, dv, df = decimate_times(verts, faces, DEC_NERF)
    del verts, faces
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "mesh.ply")
        for name, kw in (("none", {}), ("max_faces", {"max_faces": DEC_NERF})):
            dev_ms, ply_ms, out = _call_split(lambda p: nerf_render.create_mesh(net, p, 512, threshold=thr, **kw), path)
            d[f"create_mesh_{name}_no_ply_ms"] = round(dev_ms, 1)
            d[f"create_mesh_{name}_d2h_plus_ply_ms"] = round(ply_ms, 1)
            d[f"create_mesh_{name}_ply_bytes"] = os.path.getsize(path)
            if name == "max_faces":
                _, dn = ops.smooth_mesh(dv, df, 0, normals=True)
                rgb = mesh.vertex_colors(net, dv, dn)
                d["create_mesh_max_faces_equals_stages"] = bool(all(torch.equal(a, b) for a, b in zip(out, (dv, df, dn, rgb))))
            del out
            torch.cuda.empty_cache()
    res["nerf_512"] = d
    return res


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
    if "--decimation" in sys.argv[1:]:
        print(json.dumps({"metric": "mesh decimation on the device", "gpu": smi.stdout.strip(), "decimation": decimation_lines(gen)}))
        return
    out = {"metric": "create_mesh on the device: density query, marching cubes, connected components, smoothing, mesh D2H + PLY", "gpu": smi.stdout.strip(),
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
        cc = cc_times(verts, faces, None)
        cc["over_density_query"] = round(cc["total_ms"] / q_ms, 4)
        out["sizes"][str(n)]["components"] = cc
        if n == 512:
            out["sizes"][str(n)]["smoothing"] = smooth_times(verts, faces)[0]
        del sdf, verts, faces, ref_v, ref_f
        torch.cuda.empty_cache()
    out["nerf_sizes"] = nerf_lines()
    out["decimation"] = decimation_lines(gen)
    # the numpy oracle at 128^3, host only, for scale
    sdf = pigan_render.density_grid(gen.film_siren_nerf, N=128).reshape(128, 128, 128).cpu().numpy()
    t0 = time.perf_counter()
    v, f = mc.marching_cubes(sdf, -20.0, 0.2 / 127, (-0.1, -0.1, -0.1))
    out["numpy_oracle_128_ms"] = round((time.perf_counter() - t0) * 1e3, 1)
    out["numpy_oracle_128_VF"] = [int(len(v)), int(len(f))]
    print(json.dumps(out))


if __name__ == "__main__":
    main()
