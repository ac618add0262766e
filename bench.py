#!/usr/bin/env python
"""Benchmark of the hot path: rasterizer fwd+bwd frames/s @ 1 M Gaussians, 1200x680 (BASELINE.json).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One JSON line on stdout (rank 0). See DESIGN.md "Measurement" for what every field means.
* value      : frames/s with the Gaussian map, camera and upstream gradients resident in HBM (device events).
* e2e        : frames/s through the public API (Renderer.render -> loss -> backward) with the RGB-D frame and the
               camera matrices copied from pinned host memory and the loss read back every step.
* roofline   : algorithmic bytes (SURVEY.md section 8(d)) / measured duration of the dominant kernel.
* cpu_baseline / --impl reference: the CPU oracle port of the reference algorithm on the host cores (the
               reference ships no CPU render path; its rasterizer is CUDA-only).
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time
import types

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "rasterizer fwd+bwd frames/sec @1M Gaussians 1200x680"
UNIT = "frames/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--gaussians", type=int, default=1_000_000)
    ap.add_argument("--camera", default="replica")
    ap.add_argument("--no-extras", action="store_true", help="skip cpu_baseline / reference-CUDA / ICP / Adam side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def workload_name(P, cam):
    return f"surfel-room seed2024 P={P} {cam.width}x{cam.height} all tiles, sh_degree 3 (BASELINE configs[1] shape at the metric's 1M Gaussians)"


def shared_config(args, cam):
    """The `config` object: identical in the repo arm and in the reference arm (the driver compares them); everything that
    only one arm can know (kernel statistics, parallelism, copies) goes into `workload_stats` / other keys."""
    return {"workload": workload_name(args.gaussians, cam), "gaussians": args.gaussians, "width": cam.width, "height": cam.height,
            "sh_degree": 3, "tile_mask": "all tiles", "seed": 2024}


# --------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


# --------------------------------------------------------------------------- reference arm (CPU oracle port)
def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle.splat_oracle import OracleRender
    from rtg_slam_b200 import scene
    cam = scene.make_camera(args.camera)
    g = scene.surfel_room(args.gaussians, seed=2024)
    gc, gd = scene.upstream_grads(cam, seed=5)
    cores = os.cpu_count() or 1
    th, tw = cam.tile_grid

    def one(mask):
        t0 = time.perf_counter()
        o = OracleRender(cam, g, tile_mask=mask, precision="f32", nthreads=cores)
        o.backward(gc, gd, nthreads=cores)
        o.close()
        return time.perf_counter() - t0

    # bounded sample: a fraction of the tiles if a full frame would blow the time budget
    frac = 1.0
    t_full = one(None)
    budget = 150.0
    n = args.steps + args.warmup
    if t_full * n > budget:
        frac = max(0.02, min(1.0, budget / (t_full * n)))
    mask = None
    if frac < 1.0:
        rng = np.random.default_rng(0)
        mask = (rng.uniform(size=(th, tw)) < frac).astype(np.int32)
        frac = float(mask.mean())
    for _ in range(max(0, args.warmup - 1)):
        one(mask)
    ts = [one(mask) for _ in range(args.steps)]
    t = float(np.mean(ts))
    # per-tile work dominates: a frame costs t/frac (preprocess is amortised inside t and counted in full)
    value = frac / t
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * t, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(args, cam),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{'full frame' if frac >= 1.0 else f'{frac:.3f} of the tiles of one frame (random tile mask), scaled'}; "
                                   "oracle/splat_oracle.c (C restatement of the reference CUDA rasterizer, OpenMP over Gaussians and tiles); "
                                   "the reference has no CPU render path"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------- outputs of the timed path
DUMP_MAPS = ("color", "depth", "hit_color", "hit_depth", "hit_color_weight", "hit_depth_weight", "T_map")
DUMP_GRADS = (("means3D", "xyz"), ("shs", "shs"), ("opacities", "opacity"), ("scales", "scales"), ("rotations", "rotations"))
DUMP_PIXELS = 1_000_000     # frames above this (1920x1080) keep a seeded pixel sample
DUMP_ROWS = 1 << 15         # per-Gaussian outputs keep a seeded sample of the Gaussians
DUMP_BYTES = 64_000_000


def dump_outputs(path, out, grads):
    """Writes the rasterizer outputs `out` and the per-Gaussian gradients `grads` of one step as DIR/<name>.npy: floats
    as float32, index maps and radii as float64 (exact). Pixel maps keep shape (C, H, W), or (C, n) at the pixels of
    pixel_index.npy when the frame has more than DUMP_PIXELS pixels; radii.npy and grad_<name>.npy hold the Gaussians
    of gaussian_index.npy. Both samples are seeded, so the same arguments give the same files in any build."""
    import torch

    def pick(n, k, seed):
        if n <= k:
            return None
        return np.sort(np.random.default_rng(seed).choice(n, k, replace=False))

    H, W = out[0].shape[-2:]
    P = out[7].shape[0]
    px, rows = pick(H * W, DUMP_PIXELS, 1), pick(P, DUMP_ROWS, 2)
    rows = np.arange(P) if rows is None else rows
    dev_rows = torch.from_numpy(rows).to(out[7].device)
    arrays = {}
    for name, t in zip(DUMP_MAPS, out):
        t = t.detach()
        arrays[name] = t if px is None else t.reshape(t.shape[0], -1)[:, torch.from_numpy(px).to(t.device)]
    arrays["radii"] = out[7].detach()[dev_rows]
    for name, g in grads.items():
        arrays["grad_" + name] = g.detach()[dev_rows]
    if px is not None:
        arrays["pixel_index"] = torch.from_numpy(px)
    arrays["gaussian_index"] = torch.from_numpy(rows)
    host = {k: v.cpu().numpy() for k, v in arrays.items()}
    host = {k: v.astype(np.float64 if v.dtype.kind in "iub" else np.float32, copy=False) for k, v in host.items()}
    total = sum(v.nbytes for v in host.values())
    if total > DUMP_BYTES:
        raise SystemExit(f"--dump-outputs: {total} bytes exceed {DUMP_BYTES}")
    os.makedirs(path, exist_ok=True)
    for k, v in host.items():
        np.save(os.path.join(path, k + ".npy"), v)


# --------------------------------------------------------------------------- our arm
def main():
    args = parse()
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import torch.distributed as dist

    from rtg_slam_b200 import _lib, scene
    from rtg_slam_b200.rasterizer import GaussianRasterizer, GaussianRasterizationSettings
    from rtg_slam_b200.render import Renderer
    from rtg_slam_b200.loss import l1_color_depth_loss

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs CUDA devices: the product path has no CPU fallback (use --impl reference for the CPU port)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    _lib.lib()

    P = args.gaussians
    # every rank renders its own frame of the same map: rank r looks from a slightly different pose
    poses = [np.eye(4)] + [scene.small_pose((0.8 * r, -0.6 * r, 0.3 * r), (0.02 * r, -0.01 * r, 0.015 * r)) for r in range(1, 8)]
    cam = scene.make_camera(args.camera, c2w=poses[rank % 8])
    H, W = cam.height, cam.width

    # the shared Gaussian map: generated on rank 0, broadcast over NCCL (north_star: "NCCL only to broadcast the shared map")
    keys = ("xyz", "opacity", "scales", "rotations", "shs", "normal")
    shapes = {"xyz": (P, 3), "opacity": (P, 1), "scales": (P, 3), "rotations": (P, 4), "shs": (P, 16, 3), "normal": (P, 3)}
    if rank == 0:
        g = scene.surfel_room(P, seed=2024)
        t = {k: torch.from_numpy(g[k]).to(dev) for k in keys}
    else:
        t = {k: torch.empty(shapes[k], dtype=torch.float32, device=dev) for k in keys}
    if world > 1:
        for k in keys:
            dist.broadcast(t[k], src=0)
    leaves = {k: t[k].clone().requires_grad_(True) for k in ("xyz", "shs", "opacity", "scales", "rotations")}

    def settings():
        return GaussianRasterizationSettings(
            image_height=H, image_width=W, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=torch.zeros(3, device=dev), scale_modifier=1.0,
            viewmatrix=torch.from_numpy(cam.viewmatrix).to(dev), projmatrix=torch.from_numpy(cam.projmatrix).to(dev), sh_degree=3,
            campos=torch.from_numpy(cam.campos).to(dev), opaque_threshold=0.6, normal_threshold=float(np.cos(np.deg2rad(60.0))),
            depth_threshold=1.0, prefiltered=False, debug=False, cx=cam.cx, cy=cam.cy, color_sigma=3.0, T_threshold=1e-4)

    rast = GaussianRasterizer(settings())
    gc_np, gd_np = scene.upstream_grads(cam, seed=5)
    gc, gd = torch.from_numpy(gc_np).to(dev), torch.from_numpy(gd_np).to(dev)

    # N > 1: the per-rank gradients are gathered inside the timed region (north_star: "gather per-rank gradients"). The
    # backward writes straight into one of two flat buffers (no packing copy) and ONE NCCL all-reduce per step sums it over
    # the ranks, asynchronously: it overlaps the next frame's forward + backward and is waited for when its buffer is
    # needed again, two steps later (a pipelined optimiser consumes the summed gradient one step behind).
    from rtg_slam_b200 import rasterizer as rz
    from rtg_slam_b200.parallel import FlatGrads
    flats = [FlatGrads(P, dev), FlatGrads(P, dev)] if world > 1 else None
    works = [None, None]
    tick = {"k": 0}

    def step(tile_mask=None, gather=True):
        for v in leaves.values():
            v.grad = None
        out = rast(means3D=leaves["xyz"], opacities=leaves["opacity"], shs=leaves["shs"], scales=leaves["scales"],
                   rotations=leaves["rotations"], tile_mask=tile_mask)
        if flats is None or not gather:
            torch.autograd.backward([out[0], out[1]], [gc, gd])
            return out
        b = tick["k"] & 1
        tick["k"] += 1
        if works[b] is not None:
            works[b].wait()  # stream-side wait: the all-reduce issued two steps ago has released this buffer
        with rz.grad_buffers(flats[b].views):
            torch.autograd.backward([out[0], out[1]], [gc, gd])
        works[b] = flats[b].allreduce(async_op=True)
        return out

    def drain():
        for b in range(2):
            if works[b] is not None:
                works[b].wait()
                works[b] = None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    parity = parity_section(dev, cam, t) if (rank == 0 and world == 1 and not args.no_extras) else None
    # ------------------------------------------------------------------ device-resident throughput
    clocks = ClockSampler(local)
    if rank == 0:
        clocks.start()
    for _ in range(max(3, args.warmup)):
        out = step()
    torch.cuda.synchronize()
    counters = rast_counters(dev)
    vis = int((out[7] > 0).sum())
    _lib.profile_read(reset=True)
    _lib.profile_enable(True)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    marks = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]  # per-step spread (SURVEY 8(d): median, p10/p90)
    e0.record()
    for k in range(args.steps):
        if k == args.steps - 1:
            out = step()  # only the last step's outputs are held on to (--dump-outputs)
        else:
            step()
        marks[k].record()
    drain()  # the last two all-reduces end inside the timed region
    e1.record()
    barrier()
    _lib.profile_enable(False)
    prof = _lib.profile_read(reset=True)
    if args.dump_outputs and rank == 0:  # before anything else renders or steps the map
        grads = flats[(tick["k"] - 1) & 1].views if flats else {n: leaves[k].grad for n, k in DUMP_GRADS}
        dump_outputs(args.dump_outputs, out, grads)
    ms_total = e0.elapsed_time(e1)
    tm = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms_step = float(tm.item()) / args.steps
    value = world * 1e3 / ms_step  # every rank processed one frame per step
    per_step = np.array([(e0 if k == 0 else marks[k - 1]).elapsed_time(marks[k]) for k in range(args.steps)])
    step_ms = {"p10": float(np.percentile(per_step, 10)), "p50": float(np.percentile(per_step, 50)),
               "p90": float(np.percentile(per_step, 90)), "note": "rank 0, same timed region as ms_per_step"}

    # ------------------------------------------------------------------ end to end through the public API
    rargs = types.SimpleNamespace(renderer_opaque_threshold=0.6, renderer_normal_threshold=60, renderer_depth_threshold=1.0,
                                  max_sh_degree=3, color_sigma=3.0, active_sh_degree=3)
    renderer = Renderer(rargs)
    # "measured" RGB-D frame of this step lives in pinned host memory, like a frame coming from the camera driver
    with torch.no_grad():
        ref_out = rast(means3D=t["xyz"], opacities=t["opacity"], shs=t["shs"], scales=t["scales"], rotations=t["rotations"])
        frame_host = torch.cat([ref_out[0], ref_out[1]], 0).add_(0.01).cpu().pin_memory()  # (4,H,W)
    view_host = torch.from_numpy(np.stack([cam.viewmatrix, cam.projmatrix])).pin_memory()
    campos_host = torch.from_numpy(cam.campos).pin_memory()
    # double-buffered upload on a side stream: frame k+1 is copied while frame k is rendered (what a SLAM loop does with
    # the next camera frame); every step still pays for its own host->device copy inside the timed region
    copy_stream = torch.cuda.Stream(device=dev)
    frame_dev = [torch.empty_like(frame_host, device=dev) for _ in range(2)]
    view_dev = [torch.empty((2, 4, 4), device=dev) for _ in range(2)]
    campos_dev = [torch.empty(3, device=dev) for _ in range(2)]
    uploaded = [torch.cuda.Event() for _ in range(2)]
    consumed = [torch.cuda.Event() for _ in range(2)]
    loss_host = [torch.zeros(1).pin_memory() for _ in range(2)]
    loss_ready = [torch.cuda.Event() for _ in range(2)]
    losses = []
    vcs = [types.SimpleNamespace(FoVx=2 * math.atan(cam.tanfovx), FoVy=2 * math.atan(cam.tanfovy), image_height=H, image_width=W,
                                 world_view_transform=view_dev[k][0], full_proj_transform=view_dev[k][1], camera_center=campos_dev[k],
                                 cx=cam.cx, cy=cam.cy) for k in range(2)]
    data = dict(xyz=leaves["xyz"], opacity=leaves["opacity"], scales=leaves["scales"], rotations=leaves["rotations"], shs=leaves["shs"],
                normal=t["normal"])
    state = {"k": 0}

    def upload(k):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[k])
            frame_dev[k].copy_(frame_host, non_blocking=True)
            view_dev[k].copy_(view_host, non_blocking=True)
            campos_dev[k].copy_(campos_host, non_blocking=True)
            uploaded[k].record(copy_stream)

    for k in range(2):
        consumed[k].record()
    upload(0)

    def e2e_step():
        k = state["k"]
        state["k"] = 1 - k
        for v in leaves.values():
            v.grad = None
        cur = torch.cuda.current_stream(dev)
        upload(1 - k)                # next frame, overlapped with this frame's compute
        cur.wait_event(uploaded[k])
        fd = frame_dev[k]
        out = renderer.render(vcs[k], data)
        # colour L1 + depth L1 of Mapping.loss_update (mapper.py:402-431), weights of configs/base.yaml:76-77
        loss, _parts = l1_color_depth_loss(out, fd[:3], fd[3], color_weight=0.8, depth_weight=1.0, depth_error_max=0.1)
        if flats is None:
            loss.backward()
        else:  # same pipelined gradient gather as in the device-resident loop
            b = tick["k"] & 1
            tick["k"] += 1
            if works[b] is not None:
                works[b].wait()
            with rz.grad_buffers(flats[b].views):
                loss.backward()
            works[b] = flats[b].allreduce(async_op=True)
        consumed[k].record(cur)
        # the step's loss goes to pinned host memory (the loss.item() of mapper.py:459); it is *consumed* one step later,
        # after the next step has been queued, so the device never idles while the host waits for a scalar
        loss_host[k].copy_(loss.detach().reshape(1), non_blocking=True)
        loss_ready[k].record(cur)
        if state.get("pending") is not None:
            j = state["pending"]
            loss_ready[j].synchronize()
            losses.append(float(loss_host[j][0]))
        state["pending"] = k

    def e2e_drain():
        if state.get("pending") is not None:
            j = state["pending"]
            loss_ready[j].synchronize()
            losses.append(float(loss_host[j][0]))
            state["pending"] = None

    for _ in range(3):
        e2e_step()
    e2e_drain()
    barrier()
    n_before = len(losses)
    t0 = time.perf_counter()
    e0.record()
    for _ in range(args.steps):
        e2e_step()
    e2e_drain()  # the last step's loss is read inside the timed region too
    drain()
    e1.record()
    barrier()
    assert len(losses) - n_before == args.steps and all(math.isfinite(x) for x in losses), "every step's loss must reach the host"
    wall = (time.perf_counter() - t0) * 1e3
    tm = torch.tensor([max(e0.elapsed_time(e1), wall)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    e2e_value = world * 1e3 / (float(tm.item()) / args.steps)
    if rank == 0 and len(clocks.rows) < 3:  # very short runs: keep the GPU busy until nvidia-smi has reported a few times
        t_end = time.perf_counter() + 0.6
        while time.perf_counter() < t_end:
            step()
        torch.cuda.synchronize()
    clk = clocks.stop() if rank == 0 else None
    h2d = frame_host.numel() * 4 + view_host.numel() * 4 + campos_host.numel() * 4  # per step, double-buffered
    d2h = 4 + _lib.RTG_CNT_WORDS * 4  # loss + the mapped counters written by the scan kernel

    # ------------------------------------------------------------------ roofline of the dominant kernel
    R = int(counters[0]); n_tiles = int(counters[1])
    N_a = H * W  # all tiles active, image is tile-aligned except the last half row
    A = {  # algorithmic bytes per launch, SURVEY.md section 8(d)
        "preprocess_fwd": 236 * P + 52 * vis,
        "tile_scan": 0, "scatter": 12 * R, "tile_sort": 12 * R,
        "render_fwd": 40 * R + 72 * N_a,
        "render_bwd": 40 * R + 52 * N_a + 64 * vis,
        "preprocess_bwd": (236 + 64 + 8) * vis + 236 * P,
    }
    kern = {k: (ms / max(c, 1), c) for k, (ms, c) in prof.items() if c > 0}
    dom = max((k for k in kern if k in A), key=lambda k: kern[k][0] * kern[k][1])
    peaks = {}
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    if os.path.exists(pk_path):
        peaks = json.load(open(pk_path))
        peak, peak_src = float(peaks["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    ach = A[dom] / (kern[dom][0] * 1e-3) / 1e9
    traffic = None
    tr_path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tr_path):
        traffic = json.load(open(tr_path)).get(dom)
    roofline = {"bound": "hbm", "kernel": dom, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                "peak_source": peak_src, "algorithmic_bytes": A[dom], "ms_per_launch": kern[dom][0],
                "per_kernel": {k: {"ms": kern[k][0], "launches": kern[k][1], "algorithmic_GBps": (A.get(k, 0) / (kern[k][0] * 1e-3) / 1e9) if kern[k][0] > 0 else None}
                               for k in kern}}
    launches = sum(c for _, c in prof.values())

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": shared_config(args, cam),
        "workload_stats": {
            "e2e": "per step: RGB-D frame (4xHxW fp32) + camera matrices copied from pinned host memory (double-buffered on a side stream), Renderer.render, fused L1 colour+depth loss, backward, loss copied to pinned host memory and read one step later; the Gaussian map stays resident, as in the SLAM loop",
            "parallelism": (f"dp{world}: one frame per GPU per step on a replicated map; every step's per-Gaussian gradients (236 B x P, written by "
                            "the backward straight into a flat buffer) are summed over the ranks with ONE ncclAllReduce inside the timed "
                            "region, asynchronously (it overlaps the next frame's forward + backward, waited for two steps later)") if world > 1 else "single GPU",
            "collective_bytes_per_step": int(flats[0].flat.numel() * 4) if flats else 0,
            "l2": "inputs larger than L2: 236 MB of Gaussian parameters + 84 MB of splat records + 236 MB of gradients are streamed every step (L2 = 126 MB)",
            "visible_gaussians": vis, "num_rendered": R, "active_tiles": n_tiles, "mean_tile_list": R / max(n_tiles, 1), "max_tile_list": int(counters[3])},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
        "gpu_launches": launches, "clocks": clk, "roofline": roofline, "step_ms": step_ms,
    }
    if parity is not None:
        line["parity"] = parity

    if world > 1 and not args.no_extras:
        # side measurements of the multi-GPU modes with an exchange step (every rank takes the same path, so a
        # failure is symmetric and cannot strand the other ranks in a collective)
        ex = {}
        drain()
        for name, kw in (("dp_sync_optimize", {}), ("tile_sharded_records_optimize", {"tile_shard": (H, W), "records": True})):
            try:
                ex[name] = dp_optimize(args, dev, world, leaves, step, barrier, **kw)
            except Exception as e:  # the headline line must still be printed
                ex[name] = {"error": repr(e)}
        try:
            del flats[:]
            torch.cuda.empty_cache()
            ex["gaussian_sharded_4M"] = gaussian_sharded(args, dev, world, rank, barrier)
        except Exception as e:
            ex["gaussian_sharded_4M"] = {"error": repr(e)}
        if rank == 0:
            line["extras"] = ex
    if rank == 0 and world == 1 and not args.no_extras:
        line["cpu_baseline"] = cpu_baseline(args, cam)
        line["extras"] = extras(dev, cam, t, leaves, step)
        line["optimize_step"] = line["extras"].pop("optimize_step", None)
        line["map_optimize_step"] = line["extras"].pop("map_optimize_step", None)
        line["icp"] = icp_section(dev, cam)
        try:
            torch.cuda.empty_cache()
            line["extras"]["gaussian_sharded_4M"] = gaussian_sharded(args, dev, 1, 0, barrier)
        except Exception as e:
            line["extras"]["gaussian_sharded_4M"] = {"error": repr(e)}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def dp_optimize(args, dev, world, leaves, step, barrier, tile_shard=None, records=False):
    """Complete mapping iterations with a blocking exchange (reported next to the headline): every rank renders +
    back-propagates its own keyframe straight into the flat gradient buffer, ONE NCCL all-reduce sums it, every rank applies
    the same fused Adam step -- no staleness. With `tile_shard=(H, W)` the ranks instead share ONE frame: each renders +
    back-propagates only its tiles (parallel.TileShard, SURVEY 8(e)); `records=True` exchanges the 64-byte gradient records
    inside the backward instead of the dense gradient."""
    import torch
    import torch.distributed as dist
    from rtg_slam_b200 import rasterizer as rz
    from rtg_slam_b200.optim import FusedAdam
    from rtg_slam_b200.parallel import FlatGrads, TileShard
    shard = None if tile_shard is None else TileShard(tile_shard[0], tile_shard[1], device=dev)
    mask = None if shard is None else shard.mask
    P = leaves["xyz"].shape[0]
    flat = FlatGrads(P, dev)
    names = {"means3D": "xyz", "shs": "shs", "opacities": "opacity", "scales": "scales", "rotations": "rotations"}
    lrs = {"xyz": 1e-6, "shs": 1e-6, "opacity": 0.0, "scales": 1e-6, "rotations": 1e-6}  # tiny steps: keep the scene (and R) stable
    opt = FusedAdam([{"params": [leaves[v]], "lr": lrs[v]} for v in names.values()], lr=0.0, eps=1e-15)

    def it():
        if records:  # exchange the 64-byte gradient records inside the backward: complete gradients on every rank
            with shard.exchange_records():
                step(mask, gather=False)
            opt.step()
            return
        with rz.grad_buffers(flat.views):  # the backward writes into the all-reduce buffer
            step(mask, gather=False)
        flat.allreduce()
        opt.step()

    for _ in range(3):
        it()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    n = max(10, min(args.steps, 50))
    for _ in range(n):
        it()
    e1.record()
    barrier()
    tm = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms = float(tm.item()) / n
    if records:
        return {"frames_per_s": 1e3 / ms, "ms_per_step": ms, "allreduce_bytes": int(P * 64), "scaling": "strong",
                "note": "ONE frame for the whole job: the rank's tiles, all-reduce of the 64-byte gradient records between "
                        "render_bwd and preprocess_bwd (NCCL), fused Adam on every rank"}
    if tile_shard is not None:
        return {"frames_per_s": 1e3 / ms, "ms_per_step": ms, "allreduce_bytes": int(flat.flat.numel() * 4), "scaling": "strong",
                "note": "ONE frame for the whole job: fwd+bwd of the rank's tiles + flat gradient all-reduce (NCCL) + fused "
                        "Adam on every rank"}
    return {"frames_per_s": world * 1e3 / ms, "ms_per_step": ms, "allreduce_bytes": int(flat.flat.numel() * 4),
            "note": "fwd+bwd of one frame per rank (gradients written into the flat buffer) + blocking flat gradient all-reduce "
                    "(NCCL) + fused Adam on every rank"}


def gaussian_sharded(args, dev, world, rank, barrier, P=4_000_000, camera="replica"):
    """BASELINE configs[4]: 4 M Gaussians, 1200x680, ONE frame per step for the whole job, Gaussians AND tiles sharded
    (parallel.GaussianShard): all-gather of the per-Gaussian records, reduce-scatter of the gradient records, owner-side
    per-Gaussian backward + fused Adam on the owned shard. Strong scaling: compare frames_per_s across N."""
    import torch
    import torch.distributed as dist
    from rtg_slam_b200 import scene
    from rtg_slam_b200.optim import FusedAdam
    from rtg_slam_b200.parallel import GaussianShard
    from rtg_slam_b200.rasterizer import GaussianRasterizationSettings
    cam = scene.make_camera(camera)
    H, W = cam.height, cam.width
    sh = GaussianShard(P, H, W, dev, world_size=world, r=rank)
    a, b = sh.p_begin, sh.p_end
    # every rank generates the same map and keeps only its slice (no rank ever holds the other slices' parameters again)
    g = scene.surfel_room(P, seed=2024)
    own = {k: torch.from_numpy(g[k][a:b]).to(dev).requires_grad_(False) for k in ("xyz", "opacity", "shs", "scales", "rotations")}
    del g
    rs = GaussianRasterizationSettings(
        image_height=H, image_width=W, tanfovx=cam.tanfovx, tanfovy=cam.tanfovy, bg=torch.zeros(3, device=dev), scale_modifier=1.0,
        viewmatrix=torch.from_numpy(cam.viewmatrix).to(dev), projmatrix=torch.from_numpy(cam.projmatrix).to(dev), sh_degree=3,
        campos=torch.from_numpy(cam.campos).to(dev), opaque_threshold=0.6, normal_threshold=float(np.cos(np.deg2rad(60.0))),
        depth_threshold=1.0, prefiltered=False, debug=False, cx=cam.cx, cy=cam.cy, color_sigma=3.0, T_threshold=1e-4)
    gc_np, gd_np = scene.upstream_grads(cam, seed=5)
    gc, gd = torch.from_numpy(gc_np).to(dev), torch.from_numpy(gd_np).to(dev)
    params = [own["xyz"], own["shs"], own["opacity"], own["scales"], own["rotations"]]
    for p_ in params:
        p_.requires_grad_(True)
    opt = FusedAdam([{"params": [p_], "lr": lr} for p_, lr in zip(params, (1e-6, 1e-6, 0.0, 1e-6, 1e-6))], lr=0.0, eps=1e-15)

    def it():
        sh.forward(rs, own["xyz"], own["opacity"], own["shs"], own["scales"], own["rotations"])
        gr = sh.backward(gc, gd)
        for p_, k in zip(params, ("means3D", "shs", "opacities", "scales", "rotations")):
            p_.grad = gr[k].view_as(p_)
        opt.step()

    for _ in range(3):
        it()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    n = max(5, min(args.steps, 20))
    e0.record()
    for _ in range(n):
        it()
    e1.record()
    barrier()
    tm = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tm, op=dist.ReduceOp.MAX)
    ms = float(tm.item()) / n
    ex = sh.exchange_bytes()
    # where the step goes (rank 0, a few extra steps outside the timed region): library kernels by their own event
    # profiler, the two exchanges by CUDA events around the collectives
    from rtg_slam_b200 import _lib
    _lib.profile_read(reset=True)
    _lib.profile_enable(True)
    coll_ms = {"all_gather": 0.0, "reduce_scatter": 0.0}
    orig_ag, orig_rs = sh.exchange_records_forward, sh.coll.reduce_scatter_rows

    def timed(name, fn):
        def wrapped(*a, **k):
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            r = fn(*a, **k)
            a1.record()
            torch.cuda.synchronize()
            coll_ms[name] += a0.elapsed_time(a1)
            return r
        return wrapped
    sh.exchange_records_forward = timed("all_gather", orig_ag)
    sh.coll.reduce_scatter_rows = timed("reduce_scatter", orig_rs)
    m = 3
    for _ in range(m):
        it()
    torch.cuda.synchronize()
    _lib.profile_enable(False)
    prof = _lib.profile_read(reset=True)
    sh.exchange_records_forward, sh.coll.reduce_scatter_rows = orig_ag, orig_rs
    breakdown = {k: round(v[0] / m, 4) for k, v in prof.items() if v[1] > 0}
    breakdown.update({k: round(v / m, 4) for k, v in coll_ms.items()})
    barrier()
    return {"frames_per_s": 1e3 / ms, "ms_per_step": ms, "gaussians": P, "scaling": "strong", "num_rendered_own_tiles": int(sh.num_rendered),
            "breakdown_ms_rank0": breakdown, "longest_tile_list_rank0": int(sh.pinned[3]),
            "all_gather_bytes_received": ex["all_gather"], "reduce_scatter_bytes_received": ex["reduce_scatter"],
            "note": "BASELINE configs[4]: ONE frame per step for the whole job; each rank owns P/N Gaussians (parameters, Adam state) and "
                    "1/N of the tiles: forward preprocess of the owned Gaussians, ncclAllGather of the 84-byte records, binning + "
                    "compositing of the owned tiles, compositing backward, ncclReduceScatter of the 64-byte gradient records, "
                    "per-Gaussian backward + fused Adam on the owned shard"}


def rast_counters(dev):
    """num_rendered / active tiles of the last forward (pinned copy written by the scan kernel)."""
    from rtg_slam_b200 import rasterizer
    return [int(x) for x in rasterizer.last_counters(dev)]


def cpu_baseline(args, cam):
    """The reference algorithm on the host cores (oracle port): one full frame of the same workload, fwd+bwd."""
    from oracle.splat_oracle import OracleRender
    from rtg_slam_b200 import scene
    cores = os.cpu_count() or 1
    g = scene.surfel_room(args.gaussians, seed=2024)
    gc, gd = scene.upstream_grads(cam, seed=5)
    best = None
    for _ in range(2):  # first pass warms the page cache / OpenMP pool
        t0 = time.perf_counter()
        o = OracleRender(cam, g, precision="f32", nthreads=cores)
        o.backward(gc, gd, nthreads=cores)
        o.close()
        dt = time.perf_counter() - t0
        best = dt if best is None else min(best, dt)
    return {"value": 1.0 / best, "unit": UNIT, "cores": cores, "kind": "port",
            "sample": "one full frame (all tiles), fwd+bwd, best of 2; oracle/splat_oracle.c with OpenMP (the reference has no CPU render path)"}


def extras(dev, cam, t, leaves, step):
    import math
    """Side measurements reported next to the headline: reference CUDA rasterizer on this GPU, Adam step, ICP."""
    import torch
    from rtg_slam_b200 import scene
    ex = {}
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    try:
        import helpers
        mod = helpers.ref_cuda_module()
        if mod is not None:
            g = {k: v.detach().cpu().numpy() for k, v in t.items()}
            grads = scene.upstream_grads(cam, seed=5)
            for _ in range(2):
                helpers.run_ref_cuda(cam, g, dev, grads=grads)
            ex["reference_cuda"] = time_ref_cuda(mod, cam, t, dev, grads)
    except Exception as e:  # the comparator is optional
        ex["reference_cuda"] = {"error": repr(e)}
    # Adam over the six parameter groups (59 floats per Gaussian)
    from rtg_slam_b200.optim import FusedAdam
    P = t["xyz"].shape[0]
    params = [torch.zeros(s, device=dev).requires_grad_(True) for s in ((P, 3), (P, 1, 3), (P, 15, 3), (P, 1), (P, 3), (P, 4))]
    lrs = [1e-3, 5e-4, 2.5e-5, 0.0, 4e-3, 1e-3]
    for name, cls in (("fused", FusedAdam), ("torch", torch.optim.Adam)):
        opt = cls([{"params": [p], "lr": lr} for p, lr in zip(params, lrs)], lr=0.0, eps=1e-15)
        for p in params:
            p.grad = torch.randn_like(p)
        for _ in range(3):
            opt.step()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(10):
            opt.step()
        b.record()
        torch.cuda.synchronize()
        ms = a.elapsed_time(b) / 10
        ex[f"adam_{name}_ms"] = ms
        ex[f"adam_{name}_GBps"] = 1652 * P / (ms * 1e-3) / 1e9
    # SURVEY 8(d): second run with a random 50 % tile mask (the masked path of the mapper)
    try:
        tm = torch.from_numpy(scene.random_tile_mask(cam, 0.5, seed=7)).to(dev)
        for _ in range(3):
            step(tm)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(30):
            step(tm)
        b.record()
        torch.cuda.synchronize()
        ex["masked_50pct_ms_per_step"] = a.elapsed_time(b) / 30
    except Exception as e:
        ex["masked_50pct_ms_per_step"] = {"error": repr(e)}
    # map statistics (SURVEY 8(f) #2) on the rasterizer's outputs of this frame
    try:
        from rtg_slam_b200 import mapstats
        out = step()
        H, W = out[0].shape[-2:]
        err = mapstats.color_error_map(out[0].detach(), torch.rand_like(out[0]))
        z = torch.zeros_like(err)

        def ms_of(fn, n=20):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n
        P_ = t["xyz"].shape[0]
        ex["accumulate_gaussian_error_ms"] = ms_of(lambda: mapstats.accumulate_gaussian_error(
            H, W, P_, err, z, z, out[2], out[3], 0.1, 0.1, 0.1, True))
        ex["transmission_masks_ms"] = ms_of(lambda: mapstats.transmission_masks(out[6], 0.5))
        ex["colorerror2tilemask_ms"] = ms_of(lambda: mapstats.colorerror2tilemask(err, 16, 0.4))
    except Exception as e:
        ex["mapstats"] = {"error": repr(e)}
    # BASELINE configs[2]: full optimisation iteration at 1920x1080 (render + loss + backward + Adam), same map
    try:
        from rtg_slam_b200.render import Renderer
        from rtg_slam_b200.loss import l1_color_depth_loss
        camh = scene.make_camera("hd")
        rargs = types.SimpleNamespace(renderer_opaque_threshold=0.6, renderer_normal_threshold=60, renderer_depth_threshold=1.0,
                                      max_sh_degree=3, color_sigma=3.0, active_sh_degree=3)
        rend = Renderer(rargs)
        vc = types.SimpleNamespace(FoVx=2 * math.atan(camh.tanfovx), FoVy=2 * math.atan(camh.tanfovy), image_height=camh.height,
                                   image_width=camh.width, world_view_transform=torch.from_numpy(camh.viewmatrix).to(dev),
                                   full_proj_transform=torch.from_numpy(camh.projmatrix).to(dev),
                                   camera_center=torch.from_numpy(camh.campos).to(dev), cx=camh.cx, cy=camh.cy)
        data = dict(xyz=leaves["xyz"], opacity=leaves["opacity"], scales=leaves["scales"], rotations=leaves["rotations"],
                    shs=leaves["shs"], normal=t["normal"])
        with torch.no_grad():
            o0 = rend.render(vc, data)
            gt_c, gt_d = (o0["render"] + 0.01).clone(), (o0["depth"][0] + 0.01).clone()
        opt = FusedAdam([{"params": [leaves[k]], "lr": lr} for k, lr in (("xyz", 1e-6), ("shs", 1e-6), ("opacity", 0.0), ("scales", 1e-6), ("rotations", 1e-6))],
                        lr=0.0, eps=1e-15)

        def opt_step():
            opt.zero_grad(set_to_none=True)
            loss, _ = l1_color_depth_loss(rend.render(vc, data), gt_c, gt_d)
            loss.backward()
            opt.step()
        for _ in range(3):
            opt_step()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(20):
            opt_step()
        b.record()
        torch.cuda.synchronize()
        ms_opt = a.elapsed_time(b) / 20
        ex["optimize_step"] = {"ms_per_step": ms_opt, "steps_per_s": 1e3 / ms_opt, "workload": "BASELINE configs[2]: 1 M Gaussians, "
                               "1920x1080, Renderer.render + fused L1 colour+depth loss + backward + FusedAdam (59 floats per Gaussian)",
                               "algorithmic_bytes_adam": 1652 * P, "note": "the Adam step alone is reported under extras.adam_fused_*"}
    except Exception as e:
        ex["optimize_step"] = {"error": repr(e)}
    # the same iteration from RAW parameters, as Mapping.loss_update runs it (mapper.py:376-468): activations, attach
    # regulariser, Adam over the six groups, confidence update -- fused (mapoptim.MapOptimizer) vs the reference's eager
    # torch expressions around the same rasterizer
    try:
        import torch.nn.functional as F
        from rtg_slam_b200 import _lib
        from rtg_slam_b200.mapoptim import MapOptimizer
        from rtg_slam_b200.rasterizer import visible_rows_only
        with torch.no_grad():
            op = leaves["opacity"].detach().clamp(1e-4, 1 - 1e-4)
            raw = dict(xyz=leaves["xyz"].detach().clone(), features_dc=leaves["shs"].detach()[:, :1].clone(),
                       features_rest=leaves["shs"].detach()[:, 1:].clone(), opacity=torch.log(op / (1 - op)),
                       scaling=torch.log(leaves["scales"].detach()), rotation=leaves["rotations"].detach().clone())
            init_stat = {"opacity": raw["opacity"].clone(), "scaling": raw["scaling"].clone(), "xyz": raw["xyz"].clone(),
                         "rotation_raw": raw["rotation"].clone()}
            init_stat["opacity"][::2] = 0.0  # half of the rows carry the attach term
        lrs = dict(xyz=1e-6, f_dc=1e-6, f_rest=1e-6, opacity=0.0, scaling=1e-6, rotation=1e-6)
        conf = torch.zeros(P, device=dev)
        mo = MapOptimizer(raw["xyz"], raw["features_dc"], raw["features_rest"], raw["opacity"], raw["scaling"], raw["rotation"], lrs,
                          confidence=conf)
        mo.set_attach(init_stat)

        def fused_step():
            o = rend.render(vc, mo.gaussian_data())
            loss, _ = l1_color_depth_loss(o, gt_c, gt_d)
            with visible_rows_only():
                loss.backward()
            mo.step(radii=o["radii"])

        pr = {k: torch.nn.Parameter(v.clone()) for k, v in raw.items()}
        topt = torch.optim.Adam([{"params": [pr["xyz"]], "lr": lrs["xyz"]}, {"params": [pr["features_dc"]], "lr": lrs["f_dc"]},
                                 {"params": [pr["features_rest"]], "lr": lrs["f_rest"]}, {"params": [pr["opacity"]], "lr": 0.0},
                                 {"params": [pr["scaling"]], "lr": lrs["scaling"]}, {"params": [pr["rotation"]], "lr": lrs["rotation"]}],
                                lr=0.0, eps=1e-15)
        conf2 = torch.zeros(P, device=dev)
        amask = (torch.sigmoid(init_stat["opacity"]) < 0.9).squeeze()
        l2 = lambda a_, b_: ((a_ - b_) ** 2).mean()

        def eager_step():  # mapper.py:384-401,444-468 + the get_* properties of gaussian_pointcloud.py around our rasterizer
            d = dict(xyz=pr["xyz"], opacity=torch.sigmoid(pr["opacity"]), scales=torch.exp(pr["scaling"]),
                     rotations=F.normalize(pr["rotation"]), shs=torch.cat((pr["features_dc"], pr["features_rest"]), dim=1), normal=t["normal"])
            attach = 1000 * (l2(pr["scaling"][amask], init_stat["scaling"][amask]) + l2(pr["xyz"][amask], init_stat["xyz"][amask])
                             + l2(pr["rotation"][amask], init_stat["rotation_raw"][amask]))
            loss, _ = l1_color_depth_loss(rend.render(vc, d), gt_c, gt_d)
            (loss + attach).backward()
            topt.step()
            conf2[(pr["features_dc"].grad.abs() != 0).any(dim=-1).squeeze(-1)] += 1
            topt.zero_grad(set_to_none=True)

        def timed(fn, n=20):
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            a_, b_ = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a_.record()
            for _ in range(n):
                fn()
            b_.record()
            torch.cuda.synchronize()
            return a_.elapsed_time(b_) / n
        ms_fused = timed(fused_step)
        ms_eager = timed(eager_step)
        # the fused step kernel alone
        o = rend.render(vc, mo.gaussian_data())
        l1_color_depth_loss(o, gt_c, gt_d)[0].backward()
        keep = {k: getattr(mo, k).grad for k in ("xyz", "shs", "opacity", "scales", "rotations")}

        def step_only():
            for k, g_ in keep.items():
                getattr(mo, k).grad = g_
            mo.step(radii=o["radii"], zero_grad=False)
        timed(step_only, 5)
        _lib.profile_enable(True)
        _lib.profile_read(reset=True)
        for _ in range(30):
            step_only()
        prof = _lib.profile_read(reset=True)
        _lib.profile_enable(False)
        ms_step = prof["adam"][0] / max(1, prof["adam"][1])  # CUDA events around the kernel on its stream
        vis_frac = float((o["radii"] > 0).float().mean())
        step_bytes = P * (59 * 24 + 59 * 4 * vis_frac + 32 + 12 + 4 + 41)
        ex["map_optimize_step"] = {
            "workload": "BASELINE configs[2] from RAW parameters: 1 M Gaussians, 1920x1080, render + fused L1 loss + backward + "
                        "activation backward + attach regulariser + Adam (6 groups) + confidence update",
            "fused_ms_per_step": ms_fused, "fused_steps_per_s": 1e3 / ms_fused,
            "eager_reference_flow_ms_per_step": ms_eager,
            "eager_note": "the reference's torch expressions (exp / sigmoid / normalize / cat, masked l2 attach loss, "
                          "torch.optim.Adam, confidence update) around THIS library's rasterizer and loss",
            "map_adam_step_kernel_ms": ms_step, "map_adam_step_GBps": step_bytes / ms_step / 1e6,
            "map_adam_step_algorithmic_bytes": int(step_bytes), "visible_fraction": vis_frac}
    except Exception as e:
        ex["map_optimize_step"] = {"error": repr(e)}
    return ex


def icp_section(dev, cam):
    """Second half of BASELINE.json's metric: ICP iterations/s. One `IcpTracker.predict_pose` at 1200x680 = pyramid of the
    model depth (icp_use_model_depth, the setting of every shipped dataset config) + 3 levels x 5 Gauss-Newton iterations
    + point-to-plane loss + the 72-byte result read-back. Baselines: the UNMODIFIED reference SLAM/icp.py (baseline/_ref,
    oracle/ref_python.py) on CUDA tensors on this GPU (BASELINE.md B3) and on CPU tensors on the host cores (B5)."""
    import torch
    from rtg_slam_b200 import icp as ricp
    from rtg_slam_b200 import scene
    H, W = cam.height, cam.width
    cam0 = scene.make_camera("replica")
    cam1 = scene.make_camera("replica", c2w=scene.small_pose())
    d0n = scene.raycast_room_depth(cam0, noise_sigma=0.002, seed=3)
    d1n = scene.raycast_room_depth(cam1, noise_sigma=0.002, seed=4)
    d0, d1 = torch.from_numpy(d0n).to(dev), torch.from_numpy(d1n).to(dev)
    targs = dict(icp_downscales=[0.25, 0.5, 1.0], icp_warmup_frames=0, icp_use_model_depth=True, icp_downscale_iters=[5, 5, 5],
                 icp_distance_threshold=0.1, icp_normal_threshold=20, icp_damping=1e-4, verbose=False,
                 icp_sample_distance_threshold=0.01, icp_sample_normal_threshold=0.01, icp_fail_threshold=0.02)
    Kt = torch.from_numpy(cam.K)
    out = {"unit": "iterations/s", "iterations_per_predict_pose": 15,
           "workload": f"IcpTracker.predict_pose, {W}x{H}, levels 0.25/0.5/1.0 x 5 iterations, icp_use_model_depth=True (pyramid of the model "
                       "depth rebuilt inside the call), ray-cast box-room depth 2 cm / 1 deg apart + 2 mm noise"}

    def drive(trk, depth0, depth1):
        trk.update_curr_status(depth0, Kt)
        trk.move_last_status()
        trk.update_curr_status(depth1, Kt)

    trk = ricp.IcpTracker(types.SimpleNamespace(**targs))
    drive(trk, d0, d1)
    frame = {"K": Kt, "frame_id": 1}
    for _ in range(5):
        pose_ours, _ = trk.predict_pose(frame)
    torch.cuda.synchronize()
    n = 50
    t0 = time.perf_counter()
    for _ in range(n):
        trk.predict_pose(frame)
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / n
    out["value"] = 15 / dt
    out["ms_per_predict_pose"] = dt * 1e3
    # device time of the solve alone (one cooperative kernel), CUDA events on the launching stream
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(n):
        trk.predict_pose(frame)
    b.record()
    torch.cuda.synchronize()
    out["device_ms_per_predict_pose"] = a.elapsed_time(b) / n
    from rtg_slam_b200 import _lib
    _lib.profile_read(reset=True)
    _lib.profile_enable(True)
    for _ in range(20):
        trk.predict_pose(frame)
    _lib.profile_enable(False)
    prof = _lib.profile_read(reset=True)
    out["kernel_ms"] = {"pyramid (model depth)": prof["icp_build_level"][0] / 20, "solve + loss (one cooperative kernel)": prof["icp_iter"][0] / 20}
    # roofline: 48 B per pixel and iteration (SURVEY 8(d)), 5 iterations on each of the three levels
    bytes_solve = 48 * 5 * (H * W + (H // 2) * (W // 2) + (H // 4) * (W // 4))
    peak = 6650.0
    pk_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(pk_path):
        peak = float(json.load(open(pk_path))["hbm_gbs"])
    ach = bytes_solve / (out["device_ms_per_predict_pose"] * 1e-3) / 1e9
    out["roofline"] = {"bound": "hbm (nominal; the solve is latency-bound: 15 dependent iterations with a grid barrier each)",
                       "algorithmic_bytes": bytes_solve, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak}
    # ---- the reference's own file
    try:
        from oracle import ref_python
        mods = ref_python.load()
    except Exception as e:
        mods = None
        out["reference_error"] = repr(e)
    if mods is None:
        out["reference_cuda"] = out["reference_cpu"] = {"unavailable": "baseline/_ref not installed (oracle/ref_python.py install())"}
        return out
    rmod, rutils = mods
    try:  # B3: unmodified SLAM/icp.py IcpTracker on CUDA tensors, same frames, same GPU
        rtrk = rmod.IcpTracker(types.SimpleNamespace(**targs))
        Kc = Kt.to(dev).float()
        rtrk.update_curr_status(d0, Kc); rtrk.move_last_status(); rtrk.update_curr_status(d1, Kc)
        rframe = {"K": Kc, "frame_id": 1}
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):  # predict_pose prints the loss
            for _ in range(2):
                pose_ref, _ = rtrk.predict_pose(rframe)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            m = 5
            for _ in range(m):
                rtrk.predict_pose(rframe)
            torch.cuda.synchronize()
            dtr = (time.perf_counter() - t0) / m
        out["reference_cuda"] = {"value": 15 / dtr, "ms_per_predict_pose": dtr * 1e3, "kind": "reference",
                                 "note": "unmodified SLAM/icp.py IcpTracker.predict_pose (eager PyTorch) on CUDA tensors on this GPU"}
        out["vs_reference_cuda"] = out["value"] / out["reference_cuda"]["value"]
        out["pose_diff_vs_reference"] = float(np.linalg.norm(np.asarray(pose_ours, np.float64) - np.asarray(pose_ref, np.float64)))
    except Exception as e:
        out["reference_cuda"] = {"error": repr(e)}
    try:  # B5: the same file on CPU tensors (the level loop of predict_pose; its .cuda() line is the only GPU-specific one)
        builder = rmod.ImagePyramids([2, 1, 0], "max")
        v0 = rutils.build_vertex_pyramid(torch.from_numpy(d0n), builder, Kt.float())
        v1 = rutils.build_vertex_pyramid(torch.from_numpy(d1n), builder, Kt.float())
        n0, n1 = rutils.build_normal_pyramid(v0), rutils.build_normal_pyramid(v1)
        t0 = time.perf_counter()
        pose = torch.eye(4)
        for lvl, sc in enumerate([0.25, 0.5, 1.0]):
            Kl = Kt.float() * sc
            Kl[2, 2] = 1.0
            tr = rmod.ICP(5, damping=1e-4, distance_threshold=0.1, normal_threshold=20)
            pose, _ = tr.icp(pose, v1[lvl], v0[lvl], n1[lvl], n0[lvl], Kl)
        dtc = time.perf_counter() - t0
        out["reference_cpu"] = {"value": 15 / dtc, "s_per_solve": dtc, "cores": torch.get_num_threads(), "kind": "reference",
                                "note": "unmodified SLAM/icp.py ICP.icp level loop on CPU tensors (one solve; pyramids excluded)"}
        out["vs_reference_cpu"] = out["value"] / out["reference_cpu"]["value"]
    except Exception as e:
        out["reference_cpu"] = {"error": repr(e)}
    return out


def parity_section(dev, cam, t):
    """Index-map equality against the reference's own CUDA rasterizer (oracle/_ref) on the benchmark tensors, once, before
    anything is timed. The alpha of a pair is evaluated with one ex2 here (exact recheck only at the 1/255 cut), so a handful
    of pixels whose deciding alpha or T sits within ~1e-6 of a threshold may resolve differently (the oracle's tie band)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    try:
        import helpers
        if helpers.ref_cuda_module() is None:
            return {"unavailable": "oracle/_ref not built"}
        g = {k: v.detach().cpu().numpy() for k, v in t.items()}
        ours = helpers.run_ours(cam, g, dev)
        ref = helpers.run_ref_cuda(cam, g, dev)
        px = cam.height * cam.width
        res = {"pixels": px, "reference": "unmodified reference CUDA rasterizer (oracle/_ref), same tensors, same GPU"}
        for k in ("hit_color", "hit_depth"):
            res[k + "_mismatches"] = int((ours[k] != ref[k]).sum())
        same = (ours["hit_color"] == ref["hit_color"]) & (ours["hit_depth"] == ref["hit_depth"])
        over = np.zeros(same.shape[1:], bool)
        for k in ("color", "depth", "T_map", "hit_color_weight", "hit_depth_weight"):
            d = np.abs(ours[k].astype(np.float64) - ref[k].astype(np.float64)).max(axis=0)
            over |= d >= 1e-4
            srt = np.sort(d[same[0]].ravel())
            res[k + "_linf"] = float(srt[-1])
            res[k + "_linf_without_worst_8_pixels"] = float(srt[-9])
        res["pixels_beyond_1e-4"] = int(over.sum())
        res["radii_mismatches"] = int((ours["radii"] != ref["radii"]).sum())
        res["num_rendered_reference"] = int(ref["num_rendered"])
        res["note"] = ("a pixel whose transmittance lands within ~1e-6 (relative) of T_threshold may add or drop its last splat "
                       "(the oracle's tie class); the bound is at most 8 such pixels per frame")
        bad = res["hit_color_mismatches"] + res["hit_depth_mismatches"] + res["pixels_beyond_1e-4"]
        assert bad <= 8 and res["color_linf_without_worst_8_pixels"] < 1e-4 and res["radii_mismatches"] == 0, \
            f"parity with the reference lost: {res}"
        return res
    except AssertionError:
        raise
    except Exception as e:
        return {"error": repr(e)}


def time_ref_cuda(mod, cam, t, dev, grads):
    """The reference's own CUDA rasterizer (oracle/_ref) on the same tensors, fwd+bwd, CUDA events."""
    import torch
    H, W = cam.height, cam.width
    th, tw = cam.tile_grid
    tm = torch.ones((th, tw), dtype=torch.int32, device=dev)
    bg = torch.zeros(3, device=dev)
    vm = torch.from_numpy(cam.viewmatrix).to(dev); pm = torch.from_numpy(cam.projmatrix).to(dev); cp = torch.from_numpy(cam.campos).to(dev)
    e = torch.Tensor([])
    gc, gd = torch.from_numpy(grads[0]).to(dev), torch.from_numpy(grads[1]).to(dev)
    nt = float(np.cos(np.deg2rad(60.0)))

    def one():
        r = mod.rasterize_gaussians(bg, t["xyz"], e, t["opacity"], t["scales"], t["rotations"], 1.0, e, vm, pm, tm, cam.tanfovx, cam.tanfovy,
                                    H, W, cam.cx, cam.cy, t["shs"], 3, 3.0, cp, 0.6, 1.0, nt, 1e-4, False, False)
        mod.rasterize_gaussians_backward(r[13], r[1], bg, t["xyz"], r[9], e, t["scales"], t["rotations"], 1.0, e, vm, pm, cam.tanfovx,
                                         cam.tanfovy, cam.cx, cam.cy, 1.0, nt, gc, gd, t["shs"], 3, cp, r[10], r[0], r[11], r[12], r[5], False)
        return r[0]
    for _ in range(3):
        one()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    n = 10
    for _ in range(n):
        R = one()
    b.record()
    torch.cuda.synchronize()
    ms = a.elapsed_time(b) / n
    return {"ms_per_step": ms, "frames_per_s": 1e3 / ms, "num_rendered": int(R),
            "note": "unmodified reference rasterizer (sm_100 build) called as its python shim does, same tensors, same GPU"}


if __name__ == "__main__":
    main()
