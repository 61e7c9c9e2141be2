#!/usr/bin/env python
"""Headline benchmark: rays/s of the NeRF 800x800, 64 coarse + 128 fine render (BASELINE.json
configs[1]) through the B200 render path, one process per GPU.

    python bench.py --gpus 1 --steps 5 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
    python bench.py --impl reference ...      # CPU arm: the oracle port on the host cores
    python bench.py --dump-outputs DIR ...    # also write what the last timed step returned, DIR/<name>.npy

A step renders ONE full frame: the 640,000 rays are sharded over the ranks by contiguous pixel rows
(no data-path collective; the final image gather is the only exchange), so scaling is "strong".
`value` times the device-resident path (rays generated on the device, outputs left in HBM);
`e2e` times the public API call `nerf_render.render_image` whose pose comes from host memory and
whose images are returned as numpy arrays (D2H inside the timed region).
"""
from __future__ import annotations

import argparse
import gc
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

NERF_FLOP_PER_ROW = 1182976          # SURVEY.md 8(d): unpadded algorithmic FLOP per MLP evaluation


def tc_dram_traffic(rows: int):
    """(bytes, source) of one fused-MLP launch of `rows` rows: dram__bytes_read.sum + dram__bytes_write.sum of the ncu --set full capture of
    the HEADLINE launches (profiles/r2_headline_nerf_tc_ncu.json: the 122.88 M-row fine pass of the 800x800 frame); the launch this bench
    times has exactly that shape at N = 1, other row counts are scaled per row."""
    try:
        d = json.load(open(os.path.join(ROOT, "profiles", "r2_headline_nerf_tc_ncu.json")))["fine"]
    except Exception:
        return None, "profiles/r2_headline_nerf_tc_ncu.json missing"
    exact = rows == d["rows"]
    return int(d["dram_bytes_read"] + d["dram_bytes_write"]) if exact else int(d["bytes_per_row"] * rows), \
        ("dram__bytes_read.sum + dram__bytes_write.sum of this very launch shape (122.88 M rows), " if exact else
         f"{d['bytes_per_row']:.2f} B/row measured on the 122.88 M-row launch, scaled to this launch's rows, ") + \
        "ncu --set full, profiles/r2_headline_nerf_tc_ncu.txt; algorithmic = 16 B/row written + 4 B/row (z) + 24 B/ray read"
METRIC = "rays/s, NeRF 800x800 render, 64 coarse + 128 fine samples/ray"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--width", type=int, default=800)
    ap.add_argument("--height", type=int, default=800)
    ap.add_argument("--coarse", type=int, default=64)
    ap.add_argument("--fine", type=int, default=128)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--grad-precision", default="bf16", choices=["fp32", "tf32", "bf16"],
                    help="training config: bf16 = fused tensor-core forward + reverse mode, tf32 / fp32 = layer-wise GEMMs")
    ap.add_argument("--cpu-rays", type=int, default=32768, help="rays in the bounded CPU-baseline sample")
    ap.add_argument("--ref-rays", type=int, default=16384, help="--impl reference: rays per step (the reference's own chunk, nerf/render.py:150)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="headline run: skip the other BASELINE.json configs")
    ap.add_argument("--train-batch", type=int, default=4096, help="training configs: rays of the GLOBAL batch (4096 = BASELINE.json configs[2]; "
                    "512 on one GPU reproduces one rank's share of the 8-GPU step for profiling)")
    ap.add_argument("--no-graph", action="store_true", help="training config: launch the step's kernels directly (for ncu)")
    ap.add_argument("--config", default="render", choices=["render", "train", "pigan", "grid", "siren", "siren_train", "pigan_grad"],
                    help="render = the headline NeRF 800x800 frame (default; BASELINE.json configs[1]); the others are the "
                         "secondary BASELINE configs: train = 4096-ray NeRF training step (configs[2]), pigan = pi-GAN 128x128 "
                         "24+24 x 64 latents (configs[3]), grid = 256^3 density query (configs[4])")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="headline render on one GPU: after the timed steps, write the six per-ray maps the last timed step returned "
                         "(rgb_c, depth_c, acc_c, rgb_f, depth_f, acc_f) as DIR/<name>.npy in float32, so that two builds can be "
                         "compared output for output; inputs are seeded, so the same arguments give the same inputs")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and (args.impl != "b200" or args.config != "render"):
        ap.error("--dump-outputs applies to the headline render (--impl b200 --config render)")
    return args


DUMP_LIMIT_BYTES = 64_000_000


def dump_outputs(out_dir: str, maps: dict) -> None:
    """Writes each per-ray map (first dimension = rays) as out_dir/<name>.npy in float32.  When the maps together exceed
    DUMP_LIMIT_BYTES, every map is cut to the same fixed, seeded sample of rays, whose indices go to ray_index.npy (float64)."""
    os.makedirs(out_dir, exist_ok=True)
    maps = {k: v.detach().float().cpu().numpy() for k, v in maps.items()}
    n = len(next(iter(maps.values())))
    ray_bytes = sum(a[:1].nbytes for a in maps.values())
    if n * ray_bytes > DUMP_LIMIT_BYTES:
        keep = (DUMP_LIMIT_BYTES - 4096) // (ray_bytes + 8)         # 4096: room for the .npy headers
        idx = np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
        maps = {k: a[idx] for k, a in maps.items()}
        maps["ray_index"] = idx.astype(np.float64)
    for k, a in maps.items():
        np.save(os.path.join(out_dir, k + ".npy"), a)


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], bf16=d["bf16_tflops"], bf16_sustained=d.get("bf16_tflops_sustained"), src="measured")
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src="fallback")


# ---- CPU arm: the reference's own render path on the host cores ---------------------------------------------------
def cpu_baseline(args, n_rays: int, repeats: int = 1):
    """Times the reference's CPU implementation of the path on a bounded sample of the same workload (same weights -- seed 0
    reproduces the reference's init bit for bit --, sample counts, camera, a contiguous block of the frame's rays); rays are
    independent, so rays/s extrapolates linearly to the frame (BASELINE.md 4).

    kind "reference": the UNMODIFIED nerf/render.py + nerf/nerf.py (oracle/_ref, a git-ignored verbatim copy made by
    tools/install_ref.sh; oracle/ref_loader.py) -- render_rays called exactly as nerf/render.py:160 calls it, torch CPU ops on
    every host thread.  kind "port": oracle/torch_port.py (the same ATen calls restated) when no copy of the reference is
    reachable."""
    import torch
    from oracle import ref_loader, render_oracle as orc, torch_port as tp
    from msra_practice_project_b200 import models, pigan_render
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    ref = ref_loader.load_reference()
    torch.manual_seed(0)
    if ref is not None:
        c, f = ref["nerf_nerf"].NeRF(), ref["nerf_nerf"].NeRF()
    else:
        c, f = models.NeRF(), models.NeRF()
        sc_, sf_ = dict(c.state_dict()), dict(f.state_dict())
    pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)
    rays = orc.image_rays(args.width, args.height, args.width * 1.3875, pose)
    mid = (args.height // 2) * args.width
    rays = torch.from_numpy(np.ascontiguousarray(rays[mid:mid + n_rays]))
    best = None
    torch.manual_seed(5)
    with torch.no_grad():
        for _ in range(repeats):
            t0 = time.perf_counter()
            if ref is not None:
                ref["nerf_render"].render_rays(rays, 2.0, 6.0, c, f, args.coarse, args.fine)       # draws its own jitter (:131)
            else:
                t_rand = torch.rand(rays.shape[0], args.coarse)
                tp.render_rays(rays, 2.0, 6.0, lambda x: tp.nerf_mlp(sc_, x), lambda x: tp.nerf_mlp(sf_, x), args.coarse, args.fine, t_rand)
            dt = time.perf_counter() - t0
            best = dt if best is None else min(best, dt)
    what = ("the unmodified reference nerf/render.py:render_rays + nerf/nerf.py:NeRF (oracle/_ref)" if ref is not None
            else "ATen port of the reference path (oracle/torch_port.py)")
    return dict(value=rays.shape[0] / best, unit="rays/s", cores=int(torch.get_num_threads()), kind="reference" if ref is not None else "port",
                sample=f"{rays.shape[0]} rays of the {args.width}x{args.height} frame, {args.coarse}+{args.fine} samples, fp32, "
                       f"{what}, {best:.2f} s; host has {os.cpu_count()} logical cores"), best


def cpu_baseline_secondary(args, config: str):
    """cpu_baseline of a secondary BASELINE.json config (BASELINE.md 4): the unmodified reference on the host cores, on a bounded
    sample of that config's workload (units are independent: rays / latents / grid points extrapolate linearly).  None when
    no copy of the reference is reachable."""
    import torch
    from oracle import ref_loader, render_oracle as orc
    from msra_practice_project_b200 import pigan_render
    ref = ref_loader.load_reference()
    if ref is None:
        return None
    torch.set_num_threads(os.cpu_count() or 1)
    cores = int(torch.get_num_threads())
    pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)

    def frame_rays(n):
        r = orc.image_rays(800, 800, 800 * 1.3875, pose)
        return torch.from_numpy(np.ascontiguousarray(r[320000:320000 + n]))
    if config in ("train", "siren_train"):
        # nerf/train_nerf.py:151-167: render_rays + MSE(coarse) + MSE(fine) + backward on a 1024-ray sample (the reference's own batch
        # size, nerf/configs/lego.json:16); anomaly mode as shipped (nerf/nerf.py:2 switches it on) and off
        n = 1024
        torch.manual_seed(0)
        cls = ref["nerf_nerf"].NeRF if config == "train" else ref["nerf_nerf"].SirenNeRF
        c, f = cls(), cls()
        rays = frame_rays(n)
        torch.manual_seed(1)
        target = torch.rand(n, 3)
        out = {}
        for anomaly in (True, False):
            torch.autograd.set_detect_anomaly(anomaly)
            t0 = time.perf_counter()
            rc, _, _, rf, _, _ = ref["nerf_render"].render_rays(rays, 2.0, 6.0, c, f, args.coarse, args.fine)
            loss = torch.mean((rc - target) ** 2) + torch.mean((rf - target) ** 2)
            loss.backward()
            out[anomaly] = time.perf_counter() - t0
        torch.autograd.set_detect_anomaly(True)
        return dict(value=n / out[False], unit="rays/s", cores=cores, kind="reference", value_anomaly_mode_as_shipped=n / out[True],
                    sample=f"{n}-ray batch: unmodified render_rays + MSE losses + backward (no optimiser), {out[False]:.2f} s with anomaly mode off, "
                           f"{out[True]:.2f} s as shipped (nerf/nerf.py:2)")
    if config == "siren":
        n = 4096
        torch.manual_seed(0)
        c, f = ref["nerf_nerf"].SirenNeRF(), ref["nerf_nerf"].SirenNeRF()
        rays = frame_rays(n)
        with torch.no_grad():
            t0 = time.perf_counter()
            ref["nerf_render"].render_rays(rays, 2.0, 6.0, c, f, args.coarse, args.fine)
            dt = time.perf_counter() - t0
        return dict(value=n / dt, unit="rays/s", cores=cores, kind="reference", sample=f"{n} rays of the frame through the unmodified render_rays + SirenNeRF, {dt:.2f} s")
    torch.manual_seed(0)
    net = ref["pigan_modules"].FilmSirenNeRF()
    g = torch.Generator().manual_seed(0)
    film = torch.cat([1.0 + 0.2 * torch.randn(9, 256, generator=g), 0.1 * torch.randn(9, 256, generator=g)], -1)
    net.set_film_params(film)
    if config in ("pigan", "pigan_grad"):
        res = 64 if config == "pigan_grad" else 128
        focal = np.float64(res / 2 / np.tan(6 * np.pi / 180))
        p = pigan_render.camera_pos_to_transform_matrix(1, 0.0, 0.15)
        if config == "pigan":
            with torch.no_grad():
                t0 = time.perf_counter()
                ref["pigan_render"].render_image(res, res, focal, p, 0.5, 1.5, net, net, 24, 24)
                dt = time.perf_counter() - t0
            what = "one latent (1 of 64): unmodified pi_GAN/render.py:render_image + FilmSirenNeRF"
        else:
            film_g = film.clone().requires_grad_(True)
            net.set_film_params(film_g)
            t0 = time.perf_counter()
            img = ref["pigan_render"].render_image(res, res, focal, p, 0.5, 1.5, net, net, 24, 24)
            (img ** 2).mean().backward()
            dt = time.perf_counter() - t0
            what = "one latent (1 of 4): unmodified render_image + backward to the FiLM parameters and weights (anomaly mode as shipped)"
        return dict(value=res * res / dt, unit="rays/s", cores=cores, kind="reference", sample=f"{what}, {res}x{res}, 24+24 samples, {dt:.2f} s")
    # grid: the create_mesh query loop (pi_GAN/utils.py:80-91) on 1/64 of the 256^3 lattice, 65,536-point batches, zero directions
    n = 256 ** 3 // 64
    idx = torch.arange(n)
    xyz = torch.stack([(idx // 256 // 256 % 256).float(), (idx // 256 % 256).float(), (idx % 256).float()], -1) * (0.2 / 255) - 0.1
    with torch.no_grad():
        t0 = time.perf_counter()
        for h in range(0, n, 65536):
            x = torch.cat([xyz[h:h + 65536], torch.zeros(min(65536, n - h), 3)], -1)
            _ = -net(x)[:, 3]
        dt = time.perf_counter() - t0
    return dict(value=n / dt, unit="points/s", cores=cores, kind="reference", sample=f"{n} lattice points (1/64 of 256^3) through the unmodified FilmSirenNeRF.forward in 65,536-point batches, {dt:.2f} s")


def gpu_eager_incumbent(args, n_rays: int = 16384, repeats: int = 3):
    """The same ATen port run with every tensor on the B200 (stock eager PyTorch, fp32 matmuls, the reference's own 16,384-ray
    chunk, nerf/render.py:150): the honest GPU incumbent SURVEY 8(d) asks to be timed beside the CPU path -- what the
    reference itself would reach on this GPU.  A baseline like cpu_baseline, never part of the measured product path."""
    import torch
    from oracle import render_oracle as orc, torch_port as tp
    from msra_practice_project_b200 import models, pigan_render
    torch.manual_seed(0)
    c, f = models.NeRF(), models.NeRF()
    dev = torch.device("cuda", torch.cuda.current_device())
    sc_ = {k: v.to(dev) for k, v in c.state_dict().items()}
    sf_ = {k: v.to(dev) for k, v in f.state_dict().items()}
    pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)
    rays = orc.image_rays(args.width, args.height, args.width * 1.3875, pose)
    mid = (args.height // 2) * args.width
    rays = torch.from_numpy(np.ascontiguousarray(rays[mid:mid + n_rays])).to(dev)
    best = None
    with torch.no_grad(), torch.device(dev):
        for _ in range(repeats + 1):                       # first pass = warm-up, not counted
            t_rand = torch.rand(rays.shape[0], args.coarse)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            tp.render_rays(rays, 2.0, 6.0, lambda x: tp.nerf_mlp(sc_, x), lambda x: tp.nerf_mlp(sf_, x), args.coarse, args.fine, t_rand)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if _ > 0:
                best = dt if best is None else min(best, dt)
    return dict(value=rays.shape[0] / best, unit="rays/s", kind="port", device="this B200, stock eager PyTorch fp32",
                sample=f"{rays.shape[0]}-ray chunk of the frame (the reference's own chunk size), {args.coarse}+{args.fine} samples, best of {repeats}: {best * 1e3:.1f} ms")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    times = []
    base = None
    for i in range(args.warmup + args.steps):
        base, dt = cpu_baseline(args, args.ref_rays)
        if i >= args.warmup:
            times.append(dt)
    t = float(np.mean(times)) if times else float("nan")
    v = args.ref_rays / t
    base["value"] = v
    line = dict(impl="reference", metric=METRIC, value=v, unit="rays/s", n_gpus=args.gpus, steps=args.steps, warmup=args.warmup,
                ms_per_step=t * 1e3, higher_is_better=True, scaling="strong", vs_baseline=None, dtype="f32", data="synthetic",
                config=dict(workload=f"NeRF {args.width}x{args.height} render, {args.coarse}+{args.fine} samples/ray, random-init 8x256 ReLU MLP + posenc; "
                                     f"each step = a {args.ref_rays}-ray sample of the frame on the host CPU"),
                cpu_baseline=base, e2e=dict(value=v, unit="rays/s", h2d_bytes_per_step=0, d2h_bytes_per_step=0),
                samples_per_s=v * (2 * args.coarse + args.fine), gpu_launches=0)
    emit(line)


# ---- clocks sampler ---------------------------------------------------------------------------------------
class Clocks(threading.Thread):
    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
            "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.rows:
            return dict(sm_mhz=None, sm_max_mhz=None, reasons=["unsampled"])
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows if len(r) > 2 + i)]
        return dict(sm_mhz=float(np.median(sm)) if sm else None, sm_max_mhz=float(self.rows[0][1]), reasons=reasons,
                    samples=len(self.rows))


def run_b200(args):
    import torch
    import torch.distributed as dist
    from msra_practice_project_b200 import _lib, dist as shard, models, nerf_render, ops, pigan_render

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (the product has no CPU path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert _lib.lib().b2r_device_ok() == 1
    if args.dump_outputs is not None and world > 1:
        raise SystemExit("--dump-outputs writes the maps of one process's render: run it on one GPU")

    W, H, sc, sf = args.width, args.height, args.coarse, args.fine
    n_rays = W * H
    begin, count = shard.shard_range(n_rays, rank, world)
    torch.manual_seed(0)
    coarse, fine = models.NeRF().to(dev), models.NeRF().to(dev)
    pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)
    focal = W * 1.3875
    torch.manual_seed(5)
    t_rand = torch.rand((n_rays, sc), device=dev)[begin:begin + count].contiguous()
    gathered = torch.empty((n_rays, 5), dtype=torch.float32, device=dev) if world > 1 else None

    my_rows = shard.frame_slice(gathered, n_rays, rank, world) if world > 1 else None

    def step_device():
        with torch.no_grad():
            # N > 1: the fine composite writes (rgb, depth, acc) straight into this rank's rows of the frame buffer and the
            # all-gather runs in place on it (no pack / staging copy)
            # what render_image runs: the whole network on every coarse and fine sample, fine maps conformant (last-sample sign check);
            # the coarse maps are not part of the frame (nerf/render.py:161-166 returns the fine ones), so the coarse pass's last
            # samples -- which reach nothing but those maps -- get no sign check (coarse_outputs_unused)
            out = nerf_render.render_image_device(W, H, focal, pose, 2.0, 6.0, coarse, fine, sc, sf, ray_begin=begin,
                                                  ray_count=count, t_rand=t_rand, precision=args.precision, fine_out=my_rows,
                                                  coarse_outputs_unused=True)
            if world > 1:
                shard.gather_image(out[3], out[4], out[5], gathered, n_rays, rank, world)
        return out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """(total ms of `steps` calls of fn, what the last call returned)"""
        barrier()
        gc.collect(); gc.disable()              # no cyclic-GC pause of the interpreter inside a timed region
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps - 1):
            fn()
        last = fn()                             # kept: the earlier steps free their outputs before the next step allocates
        e1.record()
        barrier()
        gc.enable()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), last

    for _ in range(max(args.warmup, 3)):
        step_device()
    clocks = Clocks(local)
    if rank == 0:
        clocks.start()
    stats0 = dict(ops.last_sample_stats)
    total_ms, last = timed(step_device, args.steps)
    if rank == 0:                       # clocks are sampled during the headline's timed region only: every nvidia-smi query takes a driver
        clocks.stop_flag = True         # lock, which the host-synchronous end-to-end loop below would feel as stalls of several ms
        clocks.join(timeout=6)
    if args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, dict(zip(("rgb_c", "depth_c", "acc_c", "rgb_f", "depth_f", "acc_f"), last)))
    del last
    ms_per_step = total_ms / args.steps
    value = n_rays / (ms_per_step * 1e-3)
    # the headline runs with the last-sample sign check ON (the tolerance-conformant default, DESIGN.md 3.2); the same frame with the
    # check off (raw bf16: ~0.25 % of rays flip by up to 0.6) is timed beside it so that the cost of conformance is on record
    stats1 = dict(ops.last_sample_stats)
    last_sample = None
    if args.precision == "bf16":
        passes = max(stats1["calls"] - stats0["calls"], 1)
        ops.set_exact_last_sample(False)
        step_device()
        off_ms = timed(step_device, args.steps)[0] / args.steps
        ops.set_exact_last_sample(True)
        last_sample = dict(check="on (default)", rays_checked_per_step=(stats1["rays"] - stats0["rays"]) // args.steps,
                           rays_reevaluated_fp32_per_step=(stats1["flagged"] - stats0["flagged"]) // args.steps,
                           reevaluated_fraction=(stats1["flagged"] - stats0["flagged"]) / max(stats1["rays"] - stats0["rays"], 1),
                           passes_per_step=passes // args.steps, ms_per_step_check_off=off_ms, rays_per_s_check_off=n_rays / (off_ms * 1e-3),
                           cost_fraction=ms_per_step / off_ms - 1.0)

    # ---- the same frame with the coarse pass stopped after the sigma head (opt-in `coarse_sigma_only`: render_image never returns the
    # coarse colour, nerf/render.py:150-167).  NOT the headline -- the headline evaluates the whole network on every coarse sample as
    # the reference does; this is reported as an additional secondary line, with the fine maps compared bit for bit.
    dce = None
    if args.precision == "bf16":
        def step_dce():
            with torch.no_grad():
                return nerf_render.render_image_device(W, H, focal, pose, 2.0, 6.0, coarse, fine, sc, sf, ray_begin=begin, ray_count=count,
                                                       t_rand=t_rand, precision=args.precision, coarse_sigma_only=True)
        full = step_device()
        alt = step_dce()
        same = all(bool(torch.equal(full[i], alt[i])) for i in (3, 4, 5))
        del full, alt
        step_dce()
        dce_ms = timed(step_dce, args.steps)[0] / args.steps
        dce = dict(metric=METRIC + " (coarse pass sigma-only)", value=n_rays / (dce_ms * 1e-3), unit="rays/s", ms_per_step=dce_ms, dtype="bf16",
                   scaling="strong", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3), higher_is_better=True, vs_baseline=None,
                   data="synthetic", fine_maps_bit_identical_to_headline=same,
                   config=dict(workload="the headline frame with render_image(coarse_sigma_only=True): the coarse pass stops after layers_pos.7 + "
                                        "the sigma head (its colour is never returned; weights and every fine output are unchanged), "
                                        "no gather; dead-code elimination, not the headline"))
        assert same, "coarse_sigma_only changed the fine maps"

    # ---- N > 1: the gathered frame must equal what ONE GPU renders.  Rank 0 re-renders, alone, the two pixel rows either side of
    # every shard boundary (and the frame's first / last row) from the same global jitter and compares them bit for bit with the
    # rows the other ranks sent (the driver's GPU test box has one GPU, so the 2-GPU pytest never runs there).
    sharded_equals_single = None
    if world > 1:
        step_device()
        torch.cuda.synchronize()
        if rank == 0:
            torch.manual_seed(5)
            t_full = torch.rand((n_rays, sc), device=dev)
            ok, checked = True, 0
            spans = [(0, W), (n_rays - W, W)] + [(shard.shard_range(n_rays, r, world)[0] - W, 2 * W) for r in range(1, world)]
            with torch.no_grad():
                for b0, cnt in spans:
                    o = nerf_render.render_image_device(W, H, focal, pose, 2.0, 6.0, coarse, fine, sc, sf, ray_begin=b0, ray_count=cnt,
                                                        t_rand=t_full[b0:b0 + cnt], precision=args.precision, coarse_outputs_unused=True)
                    alone = torch.cat([o[3], o[4][:, None], o[5][:, None]], -1)
                    ok = ok and bool(torch.equal(alone, gathered[b0:b0 + cnt]))
                    checked += cnt
            sharded_equals_single = dict(equal=ok, rays_checked=checked, what="rank 0 alone vs the gathered frame: first / last pixel row and "
                                         "the two rows either side of every shard boundary, bit for bit")
            assert ok, "the gathered frame differs from the single-GPU render"
            del t_full
        barrier()

    # ---- end to end through the public API: host pose in, numpy images out
    pinned_pose = torch.from_numpy(np.ascontiguousarray(pose)).pin_memory()

    def step_e2e():
        with torch.no_grad():
            p = pinned_pose.numpy()              # host pose -> kernel arguments of the ray generator (the step's H2D)
            if world == 1:                       # the call a user of nerf/render.py makes: numpy images out (one pinned D2H of [rays,5])
                return nerf_render.render_image(W, H, focal, p, 2.0, 6.0, coarse, fine, sc, sf, precision=args.precision)
            out = nerf_render.render_image_device(W, H, focal, p, 2.0, 6.0, coarse, fine, sc, sf, ray_begin=begin,
                                                  ray_count=count, t_rand=None if world == 1 else t_rand, precision=args.precision,
                                                  fine_out=my_rows, coarse_outputs_unused=True)
            if world > 1:
                shard.gather_image(out[3], out[4], out[5], gathered, n_rays, rank, world)
                if rank == 0:
                    return nerf_render.maps_to_numpy(gathered, H, W)
            return None

    for _ in range(3):                                  # warm-up like the device loop (first call: pinned staging buffer, lazy inits)
        step_e2e()
    barrier()
    per_frame = []                                      # wall clock of every timed frame (diagnostic: shows stalls of single frames)

    def step_e2e_clocked():
        t1 = time.perf_counter(); step_e2e(); per_frame.append(round((time.perf_counter() - t1) * 1e3, 2))
    e2e_event_ms = timed(step_e2e_clocked, args.steps)[0]
    wall_ms = float(sum(per_frame))                     # every frame ends with its own synchronisation: the frames' wall clocks add up
    stage_pool = [(_u, _i) for _b, _i in nerf_render._host_stage.get((dev.index, n_rays), []) for _u in [nerf_render._storage_uses(_b)]]
    e2e_ms = max(e2e_event_ms, wall_ms) / args.steps    # the D2H copies block the host: take the larger clock
    # the frame's read-back alone (one pinned 12.8 MB copy at 800x800): PCIe speed differs between boxes and is part of e2e
    d2h_src, d2h_dst = torch.empty((n_rays * 5,), device=dev), torch.empty((n_rays * 5,), pin_memory=True)
    d2h_dst.copy_(d2h_src); torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(3):
        d2h_dst.copy_(d2h_src, non_blocking=True)
        torch.cuda.synchronize()
    d2h_ms = (time.perf_counter() - t0) * 1e3 / 3
    del d2h_src, d2h_dst
    e2e_value = n_rays / (e2e_ms * 1e-3)

    # ---- roofline of the dominant kernel (fused MLP, fine pass) timed alone with CUDA events
    roof = None
    if args.precision == "bf16":
        import ctypes as C
        with torch.no_grad():
            rays = ops.raygen(W, H, focal, pose, begin, count, device=dev)
            z = torch.sort(torch.rand((count, sc + sf), device=dev) * 4 + 2, -1).values.contiguous()
            flat = models.flat_params(fine).detach()
            packed = ops._packed_weights(fine, 0, flat, None, True)
            inp, rows, keep = ops._make_input(rays, z, None, None)
            raw = torch.empty((rows, 4), dtype=torch.float32, device=dev)
            lib = _lib.lib()
            st = torch.cuda.current_stream(dev).cuda_stream
            for _ in range(2):
                _lib.check(lib.b2r_mlp_tc_fwd(0, packed.data_ptr(), 1, C.byref(inp), raw.data_ptr(), 0, None, st), "tc")
            torch.cuda.synchronize()
            reps = 5
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                _lib.check(lib.b2r_mlp_tc_fwd(0, packed.data_ptr(), 1, C.byref(inp), raw.data_ptr(), 0, None, st), "tc")
            e1.record()
            torch.cuda.synchronize()
            k_ms = e0.elapsed_time(e1) / reps
        pk = peaks()
        achieved = rows * NERF_FLOP_PER_ROW / (k_ms * 1e-3) / 1e12
        roof = dict(bound="tensor", kernel="nerf_tc_kernel (fine pass)", achieved=achieved, peak=pk["bf16"], unit="TFLOP/s",
                    frac=achieved / pk["bf16"], frac_of_sustained=achieved / pk["bf16_sustained"] if pk["bf16_sustained"] else None,
                    peak_source=pk["src"], rows_per_launch=rows, ms_per_launch=k_ms, flop_per_row=NERF_FLOP_PER_ROW,
                    traffic=tc_dram_traffic(rows)[0], traffic_source=tc_dram_traffic(rows)[1])
    # ---- the HBM-bound stages, each timed alone with CUDA events on the launching stream
    hbm_kernels = []
    with torch.no_grad():
        pk = peaks()
        rays = ops.raygen(W, H, focal, pose, begin, count, device=dev)
        zc, mids = ops.stratified_z(torch.linspace(2.0, 6.0, sc).to(dev), t_rand)
        raw_c = torch.rand((count, sc, 4), device=dev)
        raw_f = torch.rand((count, sc + sf, 4), device=dev)
        zf = torch.sort(torch.rand((count, sc + sf), device=dev) * 4 + 2, -1).values.contiguous()
        w_c = torch.rand((count, sc), device=dev)
        u = torch.linspace(0.0, 1.0, sf).to(dev)

        def time_it(fn, reps=20):
            fn(); fn(); torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(reps):
                fn()
            e1.record(); torch.cuda.synchronize()
            return e0.elapsed_time(e1) / reps

        # kernel-only timings: the C ABI is called directly on preallocated buffers (no autograd wrapper, no allocation, no
        # host-side linspace inside the timed loop), back to back on the current stream
        import ctypes as C
        L, P_, st = _lib.lib(), _lib.ptr, torch.cuda.current_stream(dev).cuda_stream
        S2 = sc + sf
        o_rgb, o_d, o_a = torch.empty((count, 3), device=dev), torch.empty((count,), device=dev), torch.empty((count,), device=dev)
        o_w, o_sorted, o_z = torch.empty((count, sc), device=dev), torch.empty((count, S2), device=dev), torch.empty((count, sc), device=dev)
        o_mids, o_rays = torch.empty((sc - 1,), device=dev), torch.empty((count, 2, 3), device=dev)
        z_lin_d = torch.linspace(2.0, 6.0, sc).to(dev)
        dptr = rays.data_ptr() + 12
        c2w = np.ascontiguousarray(np.asarray(pose)[:3, :4], dtype=np.float64)

        def chk(rc):
            assert rc == 0, L.b2r_last_error()
        cases = [
            ("composite_fwd coarse (weights written)",
             lambda: chk(L.b2r_composite_fwd(P_(raw_c), P_(zc), dptr, 6, count, sc, P_(o_rgb), P_(o_d), P_(o_a), P_(o_w), st)), count * (sc * 24 + 32)),
            ("composite_fwd fine (weights skipped)",
             lambda: chk(L.b2r_composite_fwd(P_(raw_f), P_(zf), dptr, 6, count, S2, P_(o_rgb), P_(o_d), P_(o_a), None, st)), count * (S2 * 20 + 32)),
            ("sample_pdf + merge",
             lambda: chk(L.b2r_sample_pdf(P_(mids), 0, w_c.data_ptr() + 4, sc, P_(u), count, sc - 1, sf, P_(zc), sc, None, P_(o_sorted), None, st)),
             count * ((sc - 2) * 4 + sc * 4 + S2 * 4)),
            ("stratified_z", lambda: chk(L.b2r_stratified_z(P_(z_lin_d), P_(t_rand), count, sc, P_(o_z), P_(o_mids), st)), count * sc * 8),
            ("raygen", lambda: chk(L.b2r_raygen(c2w.ctypes.data_as(C.POINTER(C.c_double)), W, H, float(focal), 0, begin, count, P_(o_rays), st)),
             count * 24),
        ]
        for name, fn, nbytes in cases:
            ms = time_it(fn)
            gbs = nbytes / (ms * 1e-3) / 1e9
            hbm_kernels.append(dict(kernel=name, bound="hbm", algorithmic_bytes=int(nbytes), ms=ms, achieved=gbs, unit="GB/s",
                                    peak=pk["hbm"], frac=gbs / pk["hbm"]))
        del raw_c, raw_f, zf, w_c
    base = None
    if rank == 0 and not args.no_cpu_baseline and world == 1:
        base, _ = cpu_baseline(args, args.cpu_rays)
        try:
            base["gpu_eager_incumbent"] = gpu_eager_incumbent(args)
        except Exception as e:
            base["gpu_eager_incumbent"] = {"error": repr(e)[:200]}

    # the other BASELINE.json configs (training step, pi-GAN batch, density grid, SirenNeRF frame), measured in the same job
    secondary = [dce] if dce is not None else []
    if not args.no_secondary:
        for cfg in ("train", "pigan", "grid", "siren", "siren_train", "pigan_grad"):
            try:
                res = run_secondary(args, cfg, embedded=True)
            except Exception as e:          # a secondary config must never take the headline line down
                res = {"config": {"workload": cfg}, "error": repr(e)[:300]}
            secondary.append(res)

    if rank == 0:
        line = dict(metric=METRIC, value=value, unit="rays/s", n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3),
                    ms_per_step=ms_per_step, higher_is_better=True, scaling="strong", vs_baseline=None,
                    dtype="bf16" if args.precision == "bf16" else "f32", data="synthetic",
                    config=dict(workload=f"NeRF {W}x{H} Blender-shape render, {sc} coarse + {sf} fine samples/ray, random-init 8x256 ReLU MLP "
                                         f"+ posenc (L=10/4), {args.precision} MLP; rays sharded by pixel rows over {world} GPU(s); "
                                         "per-step working set (2 GB of raw samples) exceeds the 126 MB L2",
                                rays=n_rays, mlp_rows_per_ray=2 * sc + sf),
                    samples_per_s=value * (2 * sc + sf),
                    e2e=dict(value=e2e_value, unit="rays/s", h2d_bytes_per_step=96,
                             d2h_bytes_per_step=int(n_rays * 5 * 4), ms_per_step=e2e_ms,
                             cuda_event_ms_per_step=e2e_event_ms / args.steps, wall_ms_per_step=wall_ms / args.steps,
                             d2h_copy_alone_ms=d2h_ms, frames_ms=per_frame, stage_pool=stage_pool),
                    # raygen, stratified_z, 2 x (fused MLP, composite), sample_pdf + per pass with flagged rays the fp32 re-evaluation
                    # (encode, 8 layer GEMMs, sigma head)
                    gpu_launches=int((7 + (10 * last_sample["passes_per_step"] if last_sample and last_sample["rays_reevaluated_fp32_per_step"] else 0)) * args.steps * world),
                    last_sample=last_sample, sharded_equals_single=sharded_equals_single, clocks=clocks.summary(), roofline=roof,
                    hbm_kernels=hbm_kernels,
                    cpu_baseline=base, secondary=secondary)
        emit(line)
    if world > 1:
        dist.destroy_process_group()



# ---- secondary BASELINE.json configs (not the headline line; printed with the same keys) ----------------------
def run_secondary(args, config=None, embedded=False):
    """One of the other BASELINE.json configs.  embedded=True: called from the headline run (process group already up);
    returns the result dict on rank 0 instead of printing it."""
    import torch
    import torch.distributed as dist
    from msra_practice_project_b200 import _lib, dist as shard, models, nerf_render, pigan_render

    config = config or args.config
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1 and not embedded:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    assert _lib.lib().b2r_device_ok() == 1

    def timed(fn, steps, warmup):
        for _ in range(max(warmup, 3)):
            fn()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        gc.collect(); gc.disable()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        gc.enable()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()) / steps

    if config == "train":
        # nerf/train_nerf.py:151-168: render_rays on a 4096-ray batch, MSE(coarse)+MSE(fine), backward, Adam; the batch is
        # sharded over ranks and the flat fp32 gradient bucket is all-reduced once per step
        n_batch, sc, sf = args.train_batch, args.coarse, args.fine
        b, c = shard.shard_range(n_batch, rank, world)
        torch.manual_seed(0)
        coarse, fine = models.NeRF().to(dev), models.NeRF().to(dev)
        opt = torch.optim.Adam(list(coarse.parameters()) + list(fine.parameters()), lr=5e-4)
        pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)
        from msra_practice_project_b200 import ops
        ops.set_grad_precision(args.grad_precision)
        rays = ops.raygen(800, 800, 800 * 1.3875, pose, 320000 + b, c, device=dev)
        torch.manual_seed(1)
        target = torch.rand((n_batch, 3), device=dev)[b:b + c]
        torch.manual_seed(5)
        t_rand = torch.rand((n_batch, sc), device=dev)[b:b + c].contiguous()

        if args.grad_precision == "bf16":
            # fused step (train_step.py): explicit kernel sequence on flat buffers, CUDA-graph replay, fused Adam
            from msra_practice_project_b200.train_step import NerfTrainStep
            trainer = NerfTrainStep(coarse, fine, 2.0, 6.0, sc, sf, c, learning_rate=5e-4, learning_rate_decay=500, graph=not args.no_graph)

            def step():
                trainer(rays, target, t_rand=t_rand)
        else:
            def step():
                opt.zero_grad(set_to_none=True)
                rc, _, _, rf, _, _ = nerf_render.render_rays(rays, 2.0, 6.0, coarse, fine, sc, sf, t_rand=t_rand)
                loss = ((rf - target) ** 2).sum() / (n_batch * 3) + ((rc - target) ** 2).sum() / (n_batch * 3)
                loss.backward()
                shard.allreduce_gradients([coarse, fine], average=False)
                opt.step()
        ms = timed(step, args.steps, args.warmup)
        rows = n_batch * (2 * sc + sf)
        line = dict(metric=f"rays/s, NeRF training step ({n_batch}-ray batch, fwd+bwd, 64+128 samples, Adam)", value=n_batch / (ms * 1e-3),
                    unit="rays/s", ms_per_step=ms, dtype={"tf32": "tf32", "fp32": "f32", "bf16": "bf16"}[args.grad_precision], scaling="strong",
                    config=dict(workload=f"NeRF train step, {n_batch} rays sharded over ranks, " + (
                        "fused tcgen05 MLP forward with bf16 activations kept in HBM + fused dgrad / MN-major wgrad reverse mode (bf16 operands, fp32 "
                        "accumulate), fused Adam, whole step replayed as CUDA graphs, " if args.grad_precision == "bf16" else
                        f"layer-wise MLP forward with saved fp32 activations + CUDA reverse mode, GEMMs in {args.grad_precision}, ") +
                        "one NCCL all-reduce of the 4.75 MB gradient bucket" + ("" if args.grad_precision == "bf16" else ", torch Adam")),
                    tflops=rows * 1182976 * 3 / (ms * 1e-3) / 1e12)
        if args.grad_precision == "bf16":
            # the fused training kernels are HBM-bound (DESIGN.md 3.3): algorithmic bytes per MLP row = checkpoints + relu bits written by
            # the forward (5,392), d(pre-activation) tiles written + bits read by dgrad (5,152 incl. head gradients), tiles read by wgrad +
            # heads (10,624 + 784), raw / d_raw (48)
            bytes_row = 5392 + 5152 + 10624 + 784 + 48
            pk = peaks()
            line["roofline"] = dict(bound="hbm", kernel="whole training step (nerf_tc_kernel<true> + nerf_tc_bwd_kernel + nerf_tc_wgrad_kernel + heads)",
                                    achieved=rows / world * bytes_row / (ms * 1e-3) / 1e9, peak=pk["hbm"], unit="GB/s",
                                    frac=rows / world * bytes_row / (ms * 1e-3) / 1e9 / pk["hbm"], peak_source=pk["src"],
                                    bytes_per_row=bytes_row, traffic=None,
                                    note="per-kernel DRAM traffic and times: profiles/r2_train_{fwd,bwd,wgrad}_ncu.txt (wgrad reads 8.35 GB in 1.21 ms = "
                                         "at the copy peak; forward / dgrad write 4.3 / 3.8 GB at 4.2 / 3.9 TB/s: bound by the SM-side copy engine "
                                         "shared between the weight ring and the tile copies, profiles/r2_role_timers.txt, not by HBM)")
    elif config == "siren":
        # SirenNeRF (use_siren, nerf/train_nerf.py:89-91): the 800x800, 64+128 render with the fused SIREN kernel
        w = h = 800
        n = w * h
        b, c = shard.shard_range(n, rank, world)
        torch.manual_seed(0)
        coarse, fine = models.SirenNeRF().to(dev), models.SirenNeRF().to(dev)
        pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)
        torch.manual_seed(5)
        t_rand = torch.rand((n, args.coarse), device=dev)[b:b + c].contiguous()

        def step():
            with torch.no_grad():
                nerf_render.render_image_device(w, h, w * 1.3875, pose, 2.0, 6.0, coarse, fine, args.coarse, args.fine, ray_begin=b, ray_count=c,
                                                t_rand=t_rand, precision=args.precision, coarse_outputs_unused=True)
        ms = timed(step, args.steps, args.warmup)
        rows = n * (2 * args.coarse + args.fine)
        line = dict(metric="rays/s, SirenNeRF 800x800 render, 64 coarse + 128 fine samples/ray", value=n / (ms * 1e-3), unit="rays/s",
                    ms_per_step=ms, dtype="bf16" if args.precision == "bf16" else "f32", scaling="strong",
                    config=dict(workload="SirenNeRF 800x800 render, 64+128 samples, rays sharded by pixel rows, fused tcgen05 SIREN kernel"),
                    tflops=rows * 1123840 / (ms * 1e-3) / 1e12)
    elif config == "siren_train":
        # train_nerf.py with use_siren (nerf/train_nerf.py:89-91,151-168): the fused training step on two SirenNeRF models
        n_batch, sc, sf = 4096, args.coarse, args.fine
        b, c = shard.shard_range(n_batch, rank, world)
        torch.manual_seed(0)
        coarse, fine = models.SirenNeRF().to(dev), models.SirenNeRF().to(dev)
        opt = torch.optim.Adam(list(coarse.parameters()) + list(fine.parameters()), lr=5e-4)
        pose = pigan_render.camera_pos_to_transform_matrix(4.0, 0.3, -30 * np.pi / 180)
        from msra_practice_project_b200 import ops
        rays = ops.raygen(800, 800, 800 * 1.3875, pose, 320000 + b, c, device=dev)
        torch.manual_seed(1)
        target = torch.rand((n_batch, 3), device=dev)[b:b + c]
        torch.manual_seed(5)
        t_rand = torch.rand((n_batch, sc), device=dev)[b:b + c].contiguous()

        from msra_practice_project_b200.train_step import NerfTrainStep
        trainer = NerfTrainStep(coarse, fine, 2.0, 6.0, sc, sf, c, learning_rate=5e-4, learning_rate_decay=500, graph=not args.no_graph)

        def step():
            trainer(rays, target, t_rand=t_rand)
        ms = timed(step, args.steps, args.warmup)
        rows = n_batch * (2 * sc + sf)
        line = dict(metric="rays/s, SirenNeRF training step (4096-ray batch, fwd+bwd, 64+128 samples, Adam)", value=n_batch / (ms * 1e-3),
                    unit="rays/s", ms_per_step=ms, dtype="bf16", scaling="strong",
                    config=dict(workload="SirenNeRF train step, 4096 rays sharded over ranks, fused tcgen05 forward with bf16 activation + cosine "
                                         "checkpoints, fused dgrad / MN-major wgrad reverse mode, fused Adam, CUDA-graph replay"),
                    tflops=rows * 1123840 * 3 / (ms * 1e-3) / 1e12)
    elif config == "pigan_grad":
        # pi-GAN generator update (pi_GAN/train.py:121-145 without the discriminator, which is out of scope): 4 latents x 64x64, 24+24
        # samples; z -> mapping network -> FiLM -> all latents rendered in one launch sequence (coarse pass without gradient, SURVEY A.6;
        # fine pass on the fused tensor-core training path) -> image loss -> gradients of every generator parameter (FiLM-SIREN weights
        # and, through d film, the mapping network) -> Adam(betas (0, 0.9)) with the train.py:140-145 schedule.  train_step.GeneratorStep:
        # captured once, replayed as three CUDA graphs (forward | backward | optimiser) with the gradient all-reduce between the last two.
        from msra_practice_project_b200.train_step import GeneratorStep
        n_lat, res, s_ = 4, 64, 24
        b, c = shard.shard_range(n_lat, rank, world)
        torch.manual_seed(0)
        gen = models.Generator(256, res, near=0.5, far=1.5, fov=12, coarse_samples=s_, fine_samples=s_).to(dev)
        gstep = GeneratorStep(gen, max(c, 1), graph=not args.no_graph)
        g = torch.Generator().manual_seed(0)
        zs = torch.randn((n_lat, 256), generator=g).to(dev)
        poses = np.stack([pigan_render.camera_pos_to_transform_matrix(1, 0.3 * np.sin(i), 0.15 * np.cos(i)) for i in range(n_lat)])
        target = torch.rand((n_lat, 3, res, res), generator=g).to(dev)

        def step():
            if c > 0:
                imgs = gstep.forward(zs[b:b + c], poses[b:b + c])
                gstep.backward(2.0 * (imgs - target[b:b + c]) / float(n_lat * 3 * res * res))      # d/d imgs of the global-batch MSE
            else:                                    # more ranks than latents: this rank only joins the all-reduce and applies the update
                dist.all_reduce(gstep.grads.zero_())
                gstep._opt()
        ms = timed(step, args.steps, args.warmup)
        rows = n_lat * res * res * 2 * s_
        line = dict(metric="rays/s, pi-GAN gradient step through the renderer (4 latents x 64x64, 24+24 samples; d/dfilm + d/dweights)",
                    value=n_lat * res * res / (ms * 1e-3), unit="rays/s", ms_per_step=ms, dtype="bf16", scaling="strong",
                    config=dict(workload="pi-GAN generator update (train.py:121-145 minus the discriminator), latents sharded over ranks: mapping network, "
                                         "coarse pass bf16 inference (no gradient), fine pass on the fused tcgen05 training path for all latents in one "
                                         "launch sequence (bf16 tile + cosine checkpoints, fused dgrad, MN-major wgrad on the FiLM-folded weights, unfold "
                                         "into d gamma / d beta / d weights), mapping-network backward, fused Adam; the whole step replayed as CUDA graphs "
                                         "(train_step.GeneratorStep)" + ("" if not args.no_graph else " [--no-graph: launched eagerly]")),
                    tflops=rows * 1053696 * 3 / (ms * 1e-3) / 1e12)
    elif config == "pigan":
        n_lat, res, s_ = 64, 128, 24
        b, c = shard.shard_range(n_lat, rank, world)
        torch.manual_seed(0)
        net = models.FilmSirenNeRF().to(dev)
        g = torch.Generator().manual_seed(0)
        film = torch.cat([1.0 + 0.2 * torch.randn(n_lat, 9, 256, generator=g), 0.1 * torch.randn(n_lat, 9, 256, generator=g)], -1).to(dev)
        focal = np.float64(res / 2 / np.tan(6 * np.pi / 180))
        poses = [pigan_render.camera_pos_to_transform_matrix(1, 0.3 * np.sin(i), 0.15 * np.cos(i)) for i in range(n_lat)]
        out_all = torch.empty((n_lat, 3, res, res), device=dev) if world > 1 else None

        def step():
            with torch.no_grad():
                imgs = pigan_render.render_batch(net, film[b:b + c], poses[b:b + c], res, res, focal, 0.5, 1.5, s_, s_, precision=args.precision)
                if world > 1:
                    dist.all_gather_into_tensor(out_all, imgs.contiguous())
        ms = timed(step, args.steps, args.warmup)
        rays = n_lat * res * res
        line = dict(metric="rays/s, pi-GAN FiLM-SIREN render 128x128, 24+24 samples, 64 latents", value=rays / (ms * 1e-3), unit="rays/s",
                    ms_per_step=ms, dtype="bf16" if args.precision == "bf16" else "f32", scaling="strong",
                    config=dict(workload="pi-GAN generator render, 64 latents sharded over ranks, all latents of a rank in one launch sequence (per-latent FiLM tables)"),
                    images_per_s=n_lat / (ms * 1e-3), tflops=rays * 72 * 1053696 / (ms * 1e-3) / 1e12)
        if args.precision == "bf16":
            # opt-in variant (not the number above): coarse pass stopped after the sigma head -- pi_GAN/render.py:195-206 returns the fine colour only
            t_fix = torch.rand((c * res * res, s_), device=dev)
            with torch.no_grad():
                a = pigan_render.render_batch(net, film[b:b + c], poses[b:b + c], res, res, focal, 0.5, 1.5, s_, s_, t_rand=t_fix, precision=args.precision)
                a2 = pigan_render.render_batch(net, film[b:b + c], poses[b:b + c], res, res, focal, 0.5, 1.5, s_, s_, t_rand=t_fix, precision=args.precision,
                                               coarse_sigma_only=True)
            same = bool(torch.equal(a, a2))
            del a, a2, t_fix

            def step_dce():
                with torch.no_grad():
                    imgs = pigan_render.render_batch(net, film[b:b + c], poses[b:b + c], res, res, focal, 0.5, 1.5, s_, s_, precision=args.precision,
                                                     coarse_sigma_only=True)
                    if world > 1:
                        dist.all_gather_into_tensor(out_all, imgs.contiguous())
            ms2 = timed(step_dce, args.steps, args.warmup)
            line["coarse_sigma_only"] = dict(ms_per_step=ms2, value=rays / (ms2 * 1e-3), unit="rays/s", images_bit_identical=same,
                                             note="opt-in dead-code elimination of the coarse pass's colour layer; not the number above")
    else:
        n = 256
        n3 = n ** 3
        b, c = shard.shard_range(n3, rank, world)
        torch.manual_seed(0)
        net = models.FilmSirenNeRF().to(dev)
        g = torch.Generator().manual_seed(0)
        net.set_film_params(torch.cat([1.0 + 0.2 * torch.randn(9, 256, generator=g), 0.1 * torch.randn(9, 256, generator=g)], -1).to(dev))
        out_all = torch.empty((n3,), device=dev) if world > 1 else None

        def step():
            sig = pigan_render.density_grid(net, n, max_batch=n3, begin=b, count=c, precision=args.precision)
            if world > 1:
                dist.all_gather_into_tensor(out_all, sig.contiguous())
        ms = timed(step, args.steps, args.warmup)
        line = dict(metric="points/s, pi-GAN create_mesh density query on a 256^3 grid (sigma only)", value=n3 / (ms * 1e-3), unit="points/s",
                    ms_per_step=ms, dtype="bf16" if args.precision == "bf16" else "f32", scaling="strong",
                    config=dict(workload="256^3 lattice in [-0.1,0.1]^3, coordinates generated on the device, sigma-only FiLM-SIREN kernel"),
                    tflops=n3 * 919552 / (ms * 1e-3) / 1e12)
    # sine models: the fused kernel has TWO rooflines, the tensor pipe and the MUFU unit (one MUFU.SIN per hidden activation, 16 results
    # per clock and SM); both fractions are reported, the MUFU one at the 1,965 MHz the part can reach without the power cap
    sines = {"pigan": 72 * 2304, "grid": 2048, "siren": 256 * 2176 / 1.0}.get(config)
    if sines is not None and world == 1 and args.precision == "bf16":
        pk = peaks()
        units = {"pigan": rays if config == "pigan" else 0, "grid": n3 if config == "grid" else 0, "siren": n if config == "siren" else 0}[config]
        mufu_peak = 16 * 148 * 1.965e9
        line["roofline"] = dict(bound="tensor", kernel="film_tc_kernel<false>" if config != "siren" else "siren_tc_kernel<false>",
                                achieved=line["tflops"], peak=pk["bf16"], unit="TFLOP/s", frac=line["tflops"] / pk["bf16"],
                                frac_of_sustained=(line["tflops"] / pk["bf16_sustained"]) if pk.get("bf16_sustained") else None, peak_source=pk["src"],
                                traffic=None,
                                mufu=dict(sines_per_unit=sines, achieved_gsin_s=units * sines / (ms * 1e-3) / 1e9, peak_gsin_s=mufu_peak / 1e9,
                                          frac=units * sines / (ms * 1e-3) / mufu_peak),
                                note="whole-pass time (the fused MLP kernel is 95 % of it: profiles/r2_film_grid_ncu.txt, r2_film_role_timers.txt); "
                                     "the kernel is MUFU-bound (XU pipe 71 % busy under the power cap, 78 % of the epilogue warps' samples on MUFU.SIN)")
    line.update(n_gpus=world, steps=args.steps, warmup=max(args.warmup, 3), higher_is_better=True, vs_baseline=None, data="synthetic")
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            line["cpu_baseline"] = cpu_baseline_secondary(args, config)
        except Exception as e:
            line["cpu_baseline"] = {"error": repr(e)[:200]}
    if embedded:
        torch.cuda.empty_cache()
        return line
    if rank == 0:
        emit(line)
    if world > 1:
        dist.destroy_process_group()


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The ONE JSON line of the contract, written to the process's original stdout."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    # Libraries print to fd 1 behind Python's back (NCCL's "NCCL version ..." banner under NCCL_DEBUG=VERSION): keep stdout for the
    # JSON line alone by pointing fd 1 at stderr for everything else.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.config != "render":
        run_secondary(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
