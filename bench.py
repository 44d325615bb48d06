#!/usr/bin/env python
"""bench.py -- train frames/s (forward + backward render) of the B200-native 3DGUT path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload c2|c3|c1|c4] [--exchange compact|allreduce]

One "step" = one view rendered forward + backward (trace + trace_bwd with dL/d(RGBA, dist) given) over the
synthetic scene of BASELINE.json `configs[1]` (lego-like: 800x800, 300k Gaussians, 3DGUT) at N=1 (c3 = 6M Gaussians at
1237x822, c4 = the c2 scene through the 3DGRT path).  With N>1 every rank renders a different camera of the same replicated
scene and the per-Gaussian gradients are summed once per step (view-parallel training, SURVEY.md section 8e; scaling is weak):
`compact` = all-reduce [N,12] + all-gather [N,4] + local rebuild of the [N,48] SH gradient, `allreduce` = one NCCL all-reduce of
[N,12]+[N,48] (DESIGN.md section 8).

Prints ONE JSON line (rank 0).  `value` = device-timed frames/s with inputs resident in HBM; `e2e` = the same
metric through the public API (threedgut_tracer.Tracer.render + loss.backward) with every step's camera batch copied from
pinned host memory (one step ahead, on a copy stream) and every step's loss read back; `roofline` is for the dominant kernel
of the step; `cpu_baseline` is the CPU oracle (oracle/gut_oracle.c) on a bounded sample; `optimizer_step` (N=1) times the fused
Adam step of SURVEY 8f row 2 on the workload's N -- reported beside the metric, never inside it.

--impl reference: the reference has no CPU implementation and its CUDA build cannot be produced in this image
(needs slangc, see DESIGN.md); per the tier rules this arm times the CPU port (oracle/) of the reference algorithm
on the host cores, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "3dgrut_b200")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

import numpy as np  # noqa: E402

METRIC = "train frames/sec (fwd+bwd render)"
UNIT = "frames/s"


DUMP_BYTES = 64 * 1024 * 1024


def dump_outputs(path, arrays):
    """--dump-outputs: write each device tensor of `arrays` ({name: tensor}) to path/<name>.npy as float32.  The files total at most
    DUMP_BYTES: an array over its equal share keeps a fixed sample of its rows (np.random.default_rng(0), sorted), the same rows in
    every run of the same workload, so that two builds can be compared file for file."""
    os.makedirs(path, exist_ok=True)
    share = DUMP_BYTES // max(1, len(arrays))
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        a = a.reshape(a.shape[0], -1) if a.ndim > 1 else a.reshape(-1, 1)
        row_bytes = a.shape[1] * 4
        if a.nbytes > share:
            a = a[np.sort(np.random.default_rng(0).choice(a.shape[0], share // row_bytes, replace=False))]
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(a, np.float32))


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def make_scene(workload: str):
    import scenes

    if workload == "c4":  # C2's scene through the 3DGRT path
        return scenes.scene_c2()
    if workload.startswith("c4:"):
        return scenes.scene_c2(n=int(workload.split(":")[1]))
    if workload == "c1":
        return scenes.scene_c1()
    if workload == "c3":
        return scenes.scene_c3()
    if workload.startswith("c2:"):  # c2:<n> -- reduced particle count, debugging only
        return scenes.scene_c2(n=int(workload.split(":")[1]))
    return scenes.scene_c2()


class ClockSampler:
    """nvidia-smi clock / throttle sampling during the timed region (B200_PROFILING.md)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for name, val in zip(names, parts[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons),
                "samples": len(sm)}


def cpu_port_frames_per_s(sc, tile_stride: int, frames: int = 1, warm: int = 0):
    """Frames/s of the CPU port (oracle) on a bounded sample: projection + binning in full, compositing
    forward/backward on every `tile_stride`-th tile, extrapolated to the whole frame."""
    from oracle import gut_oracle as go
    import scenes

    cfg = go.default_config()
    ro, rd = sc.rays()
    rng = np.random.default_rng(0)
    go.set_tile_stride(tile_stride)
    times = []
    try:
        for f in range(warm + frames):
            pose = scenes.pose7_from_c2w(sc.camera(f, 100))
            cam = go.make_camera(sc.width, sc.height, sc.fx, sc.fy, sc.cx, sc.cy, pose)
            t0 = time.perf_counter()
            pr = go.project(cfg, cam, sc.particles, sc.sph, sc.sph_degree)
            bn = go.bin_tiles(cfg, cam, pr)
            t1 = time.perf_counter()
            rgba, dist, hits = go.render_forward(cfg, cam, ro, rd, sc.particles, pr, bn)
            d_rgba = rng.normal(size=rgba.shape).astype(np.float32)
            d_dist = np.zeros_like(dist)
            t2 = time.perf_counter()
            go.render_backward(cfg, cam, ro, rd, sc.particles, sc.sph, sc.sph_degree, pr, bn, rgba, dist, d_rgba, d_dist)
            t3 = time.perf_counter()
            if f >= warm:
                times.append((t1 - t0) + ((t2 - t1) + (t3 - t2)) * tile_stride)
    finally:
        go.set_tile_stride(1)
    return 1.0 / float(np.mean(times)), times


def grt_cpu_port_frames_per_s(sc, ray_stride: int, frames: int = 1, warm: int = 0):
    """3DGRT CPU port (brute-force oracle) on a bounded sample: every `ray_stride`-th ray of one view, extrapolated."""
    from oracle import gut_oracle as go

    cfg = go.grt_config()
    ro, rd = sc.rays()
    ro, rd = ro.reshape(-1, 3)[::ray_stride], rd.reshape(-1, 3)[::ray_stride]
    rng = np.random.default_rng(0)
    times = []
    for f in range(warm + frames):
        c2w = np.asarray(sc.camera(f, 100), np.float32)
        t0 = time.perf_counter()
        rgb, alpha, dist, hits, vis = go.grt_trace(cfg, sc.particles, sc.sph, sc.sph_degree, ro, rd, c2w)
        d_rgb = rng.normal(size=rgb.shape).astype(np.float32)
        go.grt_trace_bwd(cfg, sc.particles, sc.sph, sc.sph_degree, ro, rd, c2w, rgb, alpha, dist, d_rgb, np.zeros_like(alpha), np.zeros_like(alpha))
        if f >= warm:
            times.append((time.perf_counter() - t0) * ray_stride)
    return 1.0 / float(np.mean(times)), times


def run_reference_arm(args, rank, world):
    """CPU port of the reference algorithm on the host cores (rank 0 only)."""
    if rank != 0:
        return
    sc = make_scene(args.workload)
    if args.workload.startswith("c4"):
        stride = args.cpu_ray_stride
        cores = os.cpu_count() or 1
        fps, _ = grt_cpu_port_frames_per_s(sc, stride, frames=args.steps, warm=args.warmup)
        sample = f"per step: every {stride}th ray of one {sc.width}x{sc.height} view, brute force over all {sc.n} particles (no BVH), fwd+bwd, extrapolated x{stride}"
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1000.0 / fps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": sc.name, "gaussians": sc.n, "resolution": [sc.width, sc.height], "path": "3dgrt",
                       "note": "CPU port of the reference algorithm (oracle/); the reference needs OptiX + slangc"},
            "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))
        return
    cores = os.cpu_count() or 1
    # every step = ONE WHOLE VIEW through the CPU port (all tiles, no extrapolation: the every-16th-tile sample of round 1 mis-estimated the
    # frame by up to 5x because the heavy tiles dominate a strided subset); the number of timed views is bounded by a time budget
    _, t_first = cpu_port_frames_per_s(sc, 1, frames=1, warm=0)
    budget_s = 90.0
    timed = int(max(1, min(args.steps, budget_s / max(t_first[0], 1e-3))))
    warm = 1 if (args.warmup > 0 and t_first[0] * (timed + 1) < budget_s * 1.5) else 0
    fps, times = cpu_port_frames_per_s(sc, 1, frames=timed, warm=warm)
    sample = (f"whole views (every tile) through the CPU port: {timed} timed view(s) of {sc.width}x{sc.height} (requested steps {args.steps}, bounded by a "
              f"{budget_s:.0f} s budget), OpenMP over tiles on {cores} host threads")
    line = {
        "impl": "reference", "metric": METRIC, "value": fps, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1000.0 / fps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": sc.name, "gaussians": sc.n, "resolution": [sc.width, sc.height], "path": "3dgut", "timed_views": timed,
                   "note": "CPU port of the reference algorithm (oracle/); the reference ships no CPU path and its CUDA build needs slangc"},
        "cpu_baseline": {"value": fps, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": fps, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    # second, clearly labelled block: the reference's OWN CUDA kernels on this box's GPU (when one is present and the prebuilt library
    # travelled) -- the same-box GPU denominator; the tier's reference arm stays the CPU port above
    try:
        import torch

        if torch.cuda.is_available() and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libgut_ref_cuda.so")):
            import scenes

            dev = torch.device("cuda", 0)
            ro_np, rd_np = sc.rays()
            t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)  # noqa: E731
            gen = torch.Generator(device=dev).manual_seed(1234)
            d_rgba = torch.randn((sc.height, sc.width, 4), device=dev, generator=gen)
            d_dist = 0.05 * torch.randn((sc.height, sc.width, 1), device=dev, generator=gen)
            flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
            poses = [scenes.pose7_from_c2w(sc.camera(i, 100)) for i in range(100)]
            rg = time_reference_gpu(torch, dev, sc, poses, t(sc.particles), t(sc.sph), t(ro_np), t(rd_np), d_rgba, d_dist, flush, lambda s_: s_ % 100,
                                    steps=min(max(args.steps, 10), 30))
            if rg is not None:
                line["reference_gpu"] = rg
    except Exception as e:  # noqa: BLE001
        line["reference_gpu"] = {"unavailable": repr(e)}
    print(json.dumps(line))



def time_optimizer_step(torch, dev, n, flush, peak, peak_src, iters=20):
    """Next-row measurement (SURVEY.md 8f row 2), reported beside the render metric, never inside it: the fused activation-chain +
    Adam step of all six parameter tensors (gut_optim.cu) on this workload's N, CUDA events, L2 flushed between launches.
    Algorithmic bytes = 1660 B per Gaussian (59 floats x (param r/w + two moments r/w) + 240 B gradients + 4 B visibility)."""
    import optimizers

    g = torch.Generator(device=dev).manual_seed(5)
    widths = dict(zip(optimizers.GROUPS, optimizers.WIDTHS))
    leaves = {k: torch.randn((n, w), device=dev, generator=g) for k, w in widths.items()}
    lrs = dict(positions=1.6e-4, density=0.05, rotation=1e-3, scale=5e-3, features_albedo=2.5e-3, features_specular=1.25e-4)
    opt = optimizers.FusedGaussianAdam(leaves, lrs, eps=1e-15)
    dp = torch.randn((n, 12), device=dev, generator=g)
    ds = torch.randn((n, 48), device=dev, generator=g)
    for _ in range(3):
        opt.step(dp, ds)
    ms = []
    for i in range(iters):
        flush.fill_(float(i))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        opt.step(dp, ds)
        b.record()
        torch.cuda.synchronize(dev)
        ms.append(a.elapsed_time(b))
    t = float(np.median(ms))
    nbytes = 1660 * n
    ach = nbytes / (t * 1e-3) / 1e9
    return {"kernel": "gaussian_adam_kernel", "ms": t, "algorithmic_bytes": nbytes, "achieved": ach, "peak": peak, "unit": "GB/s",
            "frac": ach / peak if peak else None, "peak_source": peak_src, "bound": "hbm"}


def time_image_loss(torch, dev, H, W, flush, peak, peak_src, iters=20):
    """Next-row measurement (SURVEY.md 8f row 3), beside the metric: lambda_l1 L1 + lambda_ssim (1 - SSIM) and its image gradient
    (gut_loss.cu, two launches) at the workload's resolution.  Algorithmic bytes per pixel: 16 prediction + 12 target read twice, 36
    derivative maps written and read, 16 gradient written = 116 B."""
    import losses

    g = torch.Generator(device=dev).manual_seed(3)
    pred = torch.rand((H, W, 4), device=dev, generator=g)
    tgt = torch.rand((H, W, 3), device=dev, generator=g)
    out = torch.empty((H, W, 4), device=dev)
    for _ in range(3):
        losses.image_loss(pred, tgt, 0.8, 0.2, d_rgba=out)
    ms = []
    for i in range(iters):
        flush.fill_(float(i))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        losses.image_loss(pred, tgt, 0.8, 0.2, d_rgba=out)
        b.record()
        torch.cuda.synchronize(dev)
        ms.append(a.elapsed_time(b))
    t = float(np.median(ms))
    nbytes = 116 * H * W
    ach = nbytes / (t * 1e-3) / 1e9
    return {"kernel": "ssim_stats_kernel + loss_grad_kernel", "ms": t, "algorithmic_bytes": nbytes, "achieved": ach, "peak": peak, "unit": "GB/s",
            "frac": ach / peak if peak else None, "peak_source": peak_src, "bound": "hbm (the 11x11 window makes it FP32-bound at this size)"}


def time_reference_gpu(torch, dev, sc, poses, particles, sph, rays_o, rays_d, d_rgba, d_dist, flush, view_of, steps, warmup=5):
    """Same-box GPU denominator: the REFERENCE's own 3DGUT renderer (threedgut_tracer/src/gutRenderer.cu and the headers it includes,
    compiled unmodified for sm_100a in the build container with the reference's flags; only the slangc output is a hand translation --
    oracle/ref_cuda/) on the same tensors, same cameras, same CUDA-event / L2-flush protocol as our timed region.  Baseline only: nothing
    on the product path touches it.  Returns None when the prebuilt library did not travel."""
    try:
        from oracle import gut_ref_cuda as grc

        if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "libgut_ref_cuda.so")):
            return None
        rr = grc.ReferenceRaster()
    except Exception as e:  # noqa: BLE001
        return {"unavailable": repr(e)}
    H, W, n = sc.height, sc.width, sc.n
    s = torch.cuda.current_stream(dev).cuda_stream
    dp, ds = torch.empty((n, 12), device=dev), torch.empty((n, 48), device=dev)

    def step(i):
        pose = poses[view_of(i)]
        rgba, dist, hits, vis = rr.trace(torch, s, i, sc.sph_degree, particles, sph, W, H, sc.fx, sc.fy, sc.cx, sc.cy, pose, rays_o, rays_d)
        rr.trace_bwd(torch, s, i, sc.sph_degree, particles, sph, W, H, sc.fx, sc.fy, sc.cx, sc.cy, pose, rays_o, rays_d, rgba, d_rgba, dist, d_dist,
                     out=(dp, ds))

    for i in range(warmup):
        step(i)
    torch.cuda.synchronize(dev)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for i in range(steps):
        flush.fill_(float(i))
        ev[i][0].record()
        step(warmup + i)
        ev[i][1].record()
    torch.cuda.synchronize(dev)
    ms = float(np.mean([a.elapsed_time(b) for a, b in ev]))
    rr.set_timing(True)
    rr.stage_times()
    for i in range(min(steps, 10)):
        flush.fill_(float(i))
        step(warmup + i)
    torch.cuda.synchronize(dev)
    stage = rr.stage_times()
    rr.set_timing(False)
    rr.close()
    return {"value": 1000.0 / ms, "unit": UNIT, "ms_per_step": ms, "steps": steps, "stage_ms": stage,
            "what": "reference threedgut_tracer/src/gutRenderer.cu (projectOnTiles, CUB scan, expand, 44-bit CUB sort, ranges, render, renderBackward, "
                    "projectBackward + its host orchestration incl. the per-frame host sync and output zero-fills) compiled unmodified with "
                    "-O3 -use_fast_math for sm_100a; slangc output replaced by the hand translation oracle/ref_cuda/threedgutSlang.cuh",
            "timing": "CUDA events around trace+trace_bwd per step, L2 flushed between steps, same cameras and tensors as our arm"}


class HostFeed:
    """End-to-end input feed: every step's rays and target image are copied from pinned host memory on a copy stream
    while the previous step computes (what a DataLoader with pinned memory does), and every step's loss is read back
    to the host through a pinned slot one step later.  All copies stay inside the timed region: K steps issue K
    host->device input copies and K device->host loss reads."""

    def __init__(self, torch, dev, pinned):
        self.torch, self.dev, self.pinned = torch, dev, pinned
        self.layout = [(tuple(t.shape), t.numel()) for t in pinned]
        self.slab = torch.cat([t.reshape(-1) for t in pinned]).pin_memory()  # what a collating DataLoader hands over: one pinned buffer
        self.stream = torch.cuda.Stream(device=dev)
        self.next = None
        self.loss_slots = [torch.zeros(1, dtype=torch.float32).pin_memory() for _ in range(2)]
        self.loss_events = [None, None]
        self.count = 0
        self.last_loss = float("nan")

    def _issue(self):
        torch = self.torch
        self.stream.wait_stream(torch.cuda.current_stream(self.dev))  # buffers freed by older steps are safe to reuse
        with torch.cuda.stream(self.stream):
            slab = self.slab.to(self.dev, non_blocking=True)  # ONE copy per step: the collated batch (rays + target image)
            ev = torch.cuda.Event()
            ev.record(self.stream)
        tensors, at = [], 0
        for shape, numel in self.layout:
            tensors.append(slab[at:at + numel].view(shape))
            at += numel
        return tensors, ev, slab

    def take(self):
        """This step's device tensors (copy already in flight) + issue the next step's copy."""
        torch = self.torch
        if self.next is None:
            self.next = self._issue()
        tensors, ev, slab = self.next
        cur = torch.cuda.current_stream(self.dev)
        cur.wait_event(ev)
        slab.record_stream(cur)
        self.next = self._issue()
        return tensors

    def give_loss(self, loss):
        """Queue the device->host read of this step's loss; return the previous step's value."""
        torch = self.torch
        k = self.count & 1
        if self.loss_events[k ^ 1] is not None:
            self.loss_events[k ^ 1].synchronize()
            self.last_loss = float(self.loss_slots[k ^ 1][0])
        self.loss_slots[k].copy_(loss.detach().reshape(1), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record(torch.cuda.current_stream(self.dev))
        self.loss_events[k] = ev
        self.count += 1
        return self.last_loss

    def drain(self):
        for ev in self.loss_events:
            if ev is not None:
                ev.synchronize()
        self.torch.cuda.synchronize(self.dev)


def run_grt(args, rank, local_rank, world, dev, dist, sub=False):
    """C4: the C2 scene through the 3DGRT path.  A step = build_bvh (the reference's default config rebuilds every
    step, configs/render/3dgrt.yaml:6 + base_gs.yaml:88) + trace + trace_bwd."""
    import torch

    import threedgrt_tracer

    sc = make_scene(args.workload)
    n, H, W = sc.n, sc.height, sc.width
    tracer = threedgrt_tracer.Tracer({"render": {"min_transmittance": 0.001}})
    ot = tracer.tracer_wrapper
    particles = torch.from_numpy(sc.particles).to(dev)
    sph = torch.from_numpy(sc.sph).to(dev)
    pos, dns, rot, scl = (particles[:, 0:3].contiguous(), particles[:, 3:4].contiguous(), particles[:, 4:8].contiguous(),
                          particles[:, 8:11].contiguous())
    ro_np, rd_np = sc.rays()
    rays_o, rays_d = torch.from_numpy(ro_np).to(dev), torch.from_numpy(rd_np).to(dev)
    n_views = 100
    c2ws = [torch.from_numpy(np.asarray(sc.camera(i, n_views), np.float32))[None] for i in range(n_views)]
    gen = torch.Generator(device=dev).manual_seed(1234)
    d_rgb = torch.randn((1, H, W, 3), device=dev, generator=gen)
    d_alpha = torch.randn((1, H, W, 1), device=dev, generator=gen)
    d_dist = 0.05 * torch.randn((1, H, W, 1), device=dev, generator=gen)
    d_nrm = torch.zeros((1, H, W, 3), device=dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    stage = {"build_bvh": [], "trace": [], "trace_bwd": []}
    last = {}  # the latest step's outputs (fresh tensors every step)

    def view_of(step):
        return (step * world + rank) % n_views

    def step_device(step, timed=False):
        evs = [torch.cuda.Event(enable_timing=True) for _ in range(4)] if timed else None
        if timed:
            evs[0].record()
        ot.build_bvh(pos, rot, scl, dns, True, False)
        if timed:
            evs[1].record()
        c2w = c2ws[view_of(step)]
        feat, alpha, hit, nrm, hits, vis = ot.trace(step, c2w, rays_o, rays_d, particles, sph, 0, sc.sph_degree, 0.001)
        if timed:
            evs[2].record()
        dp, ds = ot.trace_bwd(step, c2w, rays_o, rays_d, feat, alpha, hit, nrm, particles, sph, d_rgb, d_alpha, d_dist, d_nrm, 0, sc.sph_degree, 0.001)
        last.update(rgb=feat, alpha=alpha, dist=hit, normals=nrm, hits=hits, visibility=vis, d_particles=dp, d_sph=ds)
        if timed:
            evs[3].record()
            torch.cuda.synchronize(dev)
            for k, (a, b) in zip(stage, zip(evs[:-1], evs[1:])):
                stage[k].append(a.elapsed_time(b))
        if world > 1:
            dist.all_reduce(dp)
            dist.all_reduce(ds)
        return feat

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local_rank)
    if rank == 0 and not sub:
        sampler.start()
    n_steps, n_warm = (min(args.steps, 10), min(args.warmup, 3)) if sub else (args.steps, args.warmup)
    for s in range(n_warm):
        step_device(s)
    barrier()
    ctx = ot.native_context(dev)
    launches0 = ctx.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n_steps)]
    for s in range(n_steps):
        flush.fill_(float(s))
        ev[s][0].record()
        step_device(n_warm + s)
        ev[s][1].record()
    barrier()
    if args.dump_outputs and rank == 0 and not sub:
        dump_outputs(args.dump_outputs, last)
    clocks = sampler.stop() if (rank == 0 and not sub) else None
    total_ms = torch.tensor([float(sum(a.elapsed_time(b) for a, b in ev))], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    launches = ctx.launch_count() - launches0
    for s in range(min(n_steps, 10)):
        flush.fill_(float(s))
        step_device(n_warm + s, timed=True)
    value = world * n_steps / (total_ms / 1000.0)
    stage_mean = {k: float(np.mean(v)) for k, v in stage.items()}
    grt_work = None
    if rank == 0:
        try:  # SURVEY 8d "3DGRT work units": counted on the device for the last view (debug entry point, outside every timed region)
            wc = ot.trace_counters(c2ws[view_of(n_warm + n_steps - 1)], rays_o, rays_d, particles, sph, sc.sph_degree, 0.001)
            peak_hbm, peak_src = load_peaks()
            rays_n = max(wc["rays"], 1)
            t_tr, t_bw = stage_mean["trace"] * 1e-3, stage_mean["trace_bwd"] * 1e-3
            fwd_bytes = wc["accepted_hits"] * 240 + wc["node_visits"] * 64 + 48 * rays_n
            bwd_bytes = wc["accepted_hits"] * (240 + 44 + 192) + 64 * rays_n
            grt_work = {"counters": wc, "rays_per_s_forward": rays_n / t_tr, "accepted_hits_per_s_forward": wc["accepted_hits"] / t_tr,
                        "node_visits_per_ray": wc["node_visits"] / rays_n, "box_tests_per_ray": wc["box_tests"] / rays_n,
                        "proxy_tests_per_ray": wc["proxy_tests"] / rays_n, "queries_per_ray": wc["queries"] / rays_n,
                        "accepted_hits_per_ray": wc["accepted_hits"] / rays_n,
                        "algorithmic_bytes": {"trace": fwd_bytes, "trace_bwd": bwd_bytes,
                                              "model": "trace: hits x 240 B (record + SH) + node visits x 64 B (two child boxes per node record; one "
                                                       "fetch per warp for packet-walked rays) + 48 B per ray; trace_bwd: hits x (240 + 44 + 192) B "
                                                       "(re-read + gradient RMW) + 64 B per ray (SURVEY 8d)"},
                        "achieved_gbs": {"trace": fwd_bytes / t_tr / 1e9, "trace_bwd": bwd_bytes / t_bw / 1e9},
                        "hbm_frac": {"trace": fwd_bytes / t_tr / 1e9 / peak_hbm, "trace_bwd": bwd_bytes / t_bw / 1e9 / peak_hbm},
                        "peak": peak_hbm, "peak_source": peak_src,
                        "note": "the traversal is latency / issue bound, not HBM bound: the byte figure is the SURVEY's work model, "
                                "reported beside rays/s, hits/s and node visits per ray"}
        except Exception as e:  # noqa: BLE001
            grt_work = {"unavailable": repr(e)}
    if sub:  # sub-record of the default c2 line: device-timed only
        return {"workload": sc.name + " via 3dgrt", "value": value, "unit": UNIT, "n_gpus": world, "steps": n_steps, "ms_per_step": total_ms / n_steps,
                "stage_ms": stage_mean, "gaussians": n, "rays": H * W, "work": grt_work,
                "note": "BASELINE configs[3]: the C2 scene through the 3DGRT path (software LBVH); step = build_bvh + trace + trace_bwd"}

    # e2e through Tracer.build_acc + Tracer.render + loss.backward with the camera batch from pinned host memory
    class _G:
        positions = pos.clone().requires_grad_(True)
        density = dns.clone().requires_grad_(True)
        rotation = rot.clone().requires_grad_(True)
        scale = scl.clone().requires_grad_(True)
        _f = sph.clone().requires_grad_(True)
        n_active_features = sc.sph_degree
        num_gaussians = n
        rotation_activation = scale_activation = density_activation = staticmethod(lambda t: t)
        get_rotation = staticmethod(lambda: _G.rotation)
        get_scale = staticmethod(lambda: _G.scale)
        get_density = staticmethod(lambda: _G.density)
        get_features = staticmethod(lambda: _G._f)

    pin_o, pin_d = torch.from_numpy(ro_np).pin_memory(), torch.from_numpy(rd_np).pin_memory()
    pin_gt = torch.rand((1, H, W, 3)).pin_memory()
    grads = [_G.positions, _G.density, _G.rotation, _G.scale, _G._f]

    class _B:
        pass

    feed = HostFeed(torch, dev, [pin_o, pin_d, pin_gt])

    def step_e2e(step):
        b = _B()
        b.rays_ori, b.rays_dir, gt = feed.take()
        b.T_to_world = c2ws[view_of(step)].to(dev)
        for g in grads:
            g.grad = None
        tracer.build_acc(_G, rebuild=True)
        out = tracer.render(_G, b, train=True, frame_id=step)
        loss = (out["pred_features"] - gt).abs().mean() + 0.01 * out["pred_opacity"].mean()
        loss.backward()
        if world > 1:
            for g in grads:
                dist.all_reduce(g.grad)
        return feed.give_loss(loss)

    e2e_steps = max(5, args.steps // 2)
    for s in range(min(args.warmup, 3)):
        step_e2e(s)
    barrier()
    t0 = time.perf_counter()
    for s in range(e2e_steps):
        step_e2e(args.warmup + s)
    feed.drain()
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * e2e_steps / float(e2e_s.item())
    h2d = int(pin_o.numel() * 4 + pin_d.numel() * 4 + pin_gt.numel() * 4)
    if rank == 0:
        peak, peak_src = load_peaks()
        stage_ms = {k: float(np.mean(v)) for k, v in stage.items()}
        dom = max(stage_ms, key=lambda k: stage_ms[k])
        P_ = H * W
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": total_ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": sc.name + " via 3dgrt", "gaussians": n, "resolution": [W, H], "path": "3dgrt (software LBVH)",
                       "step": "build_bvh + trace + trace_bwd", "l2": "flushed between timed steps (256 MiB fill)", "N": n, "P": P_},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "steps": e2e_steps,
                    "api": "threedgrt_tracer.Tracer.build_acc + render + loss.backward",
                    "feed": "pinned host -> device on a copy stream, one step ahead; loss read back one step later"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": (grt_work or {}).get("achieved_gbs", {}).get(dom), "peak": peak, "unit": "GB/s",
                         "frac": (grt_work or {}).get("hbm_frac", {}).get(dom), "traffic": None,
                         "peak_source": peak_src, "kernel_ms": stage_ms[dom],
                         "note": "traversal is latency / issue bound; achieved = SURVEY 8d's work-unit bytes (see `work`) over the live kernel time"},
            "work": grt_work,
            "stage_ms": stage_ms,
        }
        if not args.no_cpu_baseline:
            fps, _ = grt_cpu_port_frames_per_s(sc, args.cpu_ray_stride, frames=1)
            line["cpu_baseline"] = {"value": fps, "unit": UNIT, "cores": os.cpu_count() or 1, "kind": "port",
                                    "sample": f"every {args.cpu_ray_stride}th ray of one view, brute force over all particles, fwd+bwd, extrapolated"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def gut_device_loop(torch, dist, args, rank, world, dev, workload, steps, warmup, stage_pass=True, zero_dist_grad=False, dump_dir=None):
    """Device-timed 3DGUT loop on one workload: `warmup` untimed + `steps` timed view-steps per rank (one view forward + backward each), L2
    flushed between steps, per-step CUDA events, MAX over ranks.  With world > 1 every rank renders a different camera and the gradients are
    summed every `--accumulate` view-steps (a step's batch = accumulate x world views; DESIGN.md section 8): `compact` all-gathers each
    view's [N,4] radiance gradient asynchronously (it overlaps the next view's render), all-reduces the accumulated [N,12] once and rebuilds
    the [N,48] SH gradient; `allreduce` all-reduces [N,60] once per batch.  `dump_dir`: rank 0 writes the last timed step's outputs there."""
    import scenes
    import threedgut_tracer
    from threedgut_tracer.tracer import fromOpenCVPinholeCameraModelParameters, ShutterType

    sc = make_scene(workload)
    n, H, W = sc.n, sc.height, sc.width
    tracer = threedgut_tracer.Tracer({"render": {"enable_kernel_timings": False}})
    raster = tracer.tracer_wrapper
    particles = torch.from_numpy(sc.particles).to(dev)
    sph = torch.from_numpy(sc.sph).to(dev)
    ro_np, rd_np = sc.rays()
    rays_o, rays_d = torch.from_numpy(ro_np).to(dev), torch.from_numpy(rd_np).to(dev)
    sensor = fromOpenCVPinholeCameraModelParameters(np.array([W, H]), ShutterType.GLOBAL, np.array([sc.cx, sc.cy], np.float32),
                                                    np.array([sc.fx, sc.fy], np.float32), np.zeros(6, np.float32), np.zeros(2, np.float32),
                                                    np.zeros(4, np.float32))
    n_views = 100
    poses = [scenes.pose7_from_c2w(sc.camera(i, n_views)) for i in range(n_views)]
    gen = torch.Generator(device=dev).manual_seed(1234)
    d_rgba = torch.randn((H, W, 4), device=dev, generator=gen)
    d_dist = 0.05 * torch.randn((H, W, 1), device=dev, generator=gen)
    if zero_dist_grad:  # what autograd hands trace_bwd when the loss does not use pred_dist (the reference's default training loss)
        d_dist = torch.zeros_like(d_dist)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)  # > 126 MB L2
    V = max(1, args.accumulate) if world > 1 else 1

    def view_of(step, r=None):  # disjoint cameras per rank
        return (step * world + (rank if r is None else r)) % n_views

    grad_flat = torch.empty(n * 60, dtype=torch.float32, device=dev)  # [N,12] and [N,48] views of one bucket: one all-reduce
    grad_views = (grad_flat[: n * 12].view(n, 12), grad_flat[n * 12:].view(n, 48))
    grad_tmp = (torch.empty((n, 12), device=dev), torch.empty((n, 48), device=dev)) if (world > 1 and V > 1 and args.exchange == "allreduce") else None
    compact = None
    if world > 1 and args.exchange == "compact":
        import view_parallel

        compact = view_parallel.CompactGradientExchange(raster, n, dev, views_per_rank=V)
        pos_table = np.stack([raster.sensor_position(sensor, p, p, W, H) for p in poses]).astype(np.float32)  # every rank knows every pose
    xev = []  # (start, end) events around the exposed part of the exchange, filled only in the stage pass
    last = {}  # the latest step's forward outputs (fresh tensors every step)

    def step_device(step, time_exchange=False):
        pose = poses[view_of(step)]
        slot = step % V
        rgba, dst, hits, vis = raster.trace(step, sc.sph_degree, particles, sph, rays_o, rays_d, None, sensor, 0, 1, pose, pose)
        last.update(rgba=rgba, dist=dst, hits=hits, visibility=vis)
        if compact is not None:
            # 64 B instead of 240 B per Gaussian on the wire: all-reduce d_particles, all-gather the radiance gradients, rebuild d_sph
            raster.trace_bwd_compact(step, sc.sph_degree, particles, sph, rays_o, rays_d, None, sensor, 0, 1, pose, pose, rgba, d_rgba, dst,
                                     d_dist, out=compact.out(slot))
            compact.submit(slot)
            if slot == V - 1:
                first = step - (V - 1)
                idx = [view_of(first + j, r) for j in range(V) for r in range(world)]  # slot-major, rank-minor
                if time_exchange:
                    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    a.record()
                out = compact.finish(sc.sph_degree, particles, pos_table[idx])
                if time_exchange:
                    b.record()
                    xev.append((a, b))
                return out
            return None
        if world > 1 and slot > 0:
            raster.trace_bwd(step, sc.sph_degree, particles, sph, rays_o, rays_d, None, sensor, 0, 1, pose, pose, rgba, d_rgba, dst, d_dist, out=grad_tmp)
            grad_views[0].add_(grad_tmp[0])
            grad_views[1].add_(grad_tmp[1])
        else:
            raster.trace_bwd(step, sc.sph_degree, particles, sph, rays_o, rays_d, None, sensor, 0, 1, pose, pose, rgba, d_rgba, dst, d_dist,
                             out=grad_views)
        if world > 1 and slot == V - 1:
            if time_exchange:
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a.record()
            dist.all_reduce(grad_flat)
            if time_exchange:
                b.record()
                xev.append((a, b))
        return grad_views

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    ctx = raster.native_context(dev)
    steps = max(V, (steps // V) * V)      # whole batches only
    warmup = ((warmup + V - 1) // V) * V
    for s_ in range(warmup):
        step_device(s_)
    barrier()
    launches0 = ctx.launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    for s_ in range(steps):
        flush.fill_(float(s_))  # L2 flush between timed iterations, outside the per-step event pair
        ev[s_][0].record()
        grads = step_device(warmup + s_)
        ev[s_][1].record()
    barrier()
    if dump_dir is not None and rank == 0:  # before the stage pass below reuses the gradient buffers
        if grads is not None:
            last.update(d_particles=grads[0], d_sph=grads[1])
        dump_outputs(dump_dir, last)
    step_ms = np.array([a.elapsed_time(b) for a, b in ev], dtype=np.float64)
    total_ms = torch.tensor([float(step_ms.sum())], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    launches = ctx.launch_count() - launches0
    stats = ctx.stats()
    stage_ms, exchange = None, None
    if stage_pass:
        # separate short pass with per-stage CUDA events (they add host syncs, so never inside the timed region)
        ctx.set_timings(2)
        ctx.collect_stage_times()
        k = max(V, (min(steps, 20) // V) * V)
        for s_ in range(k):
            flush.fill_(float(s_))
            step_device(warmup + s_, time_exchange=True)
        barrier()
        stage_ms = ctx.collect_stage_times()
        ctx.set_timings(0)
        if world > 1 and xev:
            xms = float(np.mean([a.elapsed_time(b) for a, b in xev]))
            wire = compact.bytes_on_wire() if compact is not None else int(2 * (world - 1) / world * 240 * n)
            exchange = {"kind": args.exchange, "views_per_rank_per_batch": V, "exposed_ms_per_batch": xms, "exposed_ms_per_view": xms / V,
                        "bytes_on_wire_per_rank_per_batch": wire, "bus_gbs_over_exposed_time": wire / (xms * 1e-3) / 1e9 if xms > 0 else None,
                        "note": "exposed = the step's all-reduce + waiting for the (already running) all-gathers + the SH rebuild kernel, "
                                "CUDA events on the compute stream; the all-gathers of earlier views of the batch overlap the next view's render"}
    value = world * steps / (total_ms / 1000.0)
    return {"value": value, "total_ms": total_ms, "steps": steps, "warmup": warmup, "launches": launches, "stats": stats, "stage_ms": stage_ms,
            "exchange": exchange, "accumulate": V,
            "objs": dict(sc=sc, tracer=tracer, raster=raster, ctx=ctx, particles=particles, sph=sph, rays_o=rays_o, rays_d=rays_d, poses=poses,
                         d_rgba=d_rgba, d_dist=d_dist, flush=flush, view_of=view_of, barrier=barrier, sensor=sensor)}



def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2")
    ap.add_argument("--cpu-tile-stride", type=int, default=16)
    ap.add_argument("--cpu-ray-stride", type=int, default=2048)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-reference-gpu", action="store_true", help="skip the reference_gpu block (the reference's own kernels timed on this GPU)")
    ap.add_argument("--exchange", default="compact", choices=["compact", "allreduce"],
                    help="multi-GPU gradient exchange of the 3DGUT path: compact = all-reduce [N,12] + all-gather [N,4] + rebuild of the SH "
                         "gradient (64 B per Gaussian on the wire), allreduce = one all-reduce of [N,60] (240 B)")
    ap.add_argument("--accumulate", type=int, default=4,
                    help="multi-GPU: view-steps per rank between two gradient exchanges (a batch = accumulate x world views); ignored at N=1")
    ap.add_argument("--profile-host", default=None, help="write a cProfile of the end-to-end loop's host side to this file (diagnostic; the e2e number of such a run is not a bench value)")
    ap.add_argument("--sub-records", default="train_default,c3,c4", help="which sub-records the default c2 line carries (comma list)")
    ap.add_argument("--no-sub-records", action="store_true", help="skip the c3 (6M Gaussians) and c4 (3DGRT) sub-records of the default c2 line")
    ap.add_argument("--dump-outputs", default=None, metavar="DIR",
                    help="after the timed steps, write what the last timed step computed (rendered images, visibility, gradients) as "
                         "DIR/<name>.npy, float32, at most 64 MiB in all (larger arrays keep a fixed sample of rows); inputs are seeded")
    args = ap.parse_args()

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback (use --impl reference for the CPU port)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist

        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    import b200_native as nat  # noqa: F401
    import scenes
    import threedgut_tracer  # noqa: F401

    if args.workload.startswith("c4"):
        run_grt(args, rank, local_rank, world, dev, dist)
        return
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()  # runs through warm-up and the timed region (both under load)
    main_run = gut_device_loop(torch, dist, args, rank, world, dev, args.workload, args.steps, args.warmup, stage_pass=True,
                               dump_dir=args.dump_outputs)
    clocks = sampler.stop() if rank == 0 else None
    o = main_run["objs"]
    sc, tracer, raster, ctx, particles, sph, rays_o, rays_d, poses, d_rgba, d_dist, flush, view_of = (
        o["sc"], o["tracer"], o["raster"], o["ctx"], o["particles"], o["sph"], o["rays_o"], o["rays_d"], o["poses"], o["d_rgba"], o["d_dist"],
        o["flush"], o["view_of"])
    n, H, W, n_views = sc.n, sc.height, sc.width, 100
    ro_np, rd_np = sc.rays()
    total_ms, launches, stats, stage_ms, value = main_run["total_ms"], main_run["launches"], main_run["stats"], main_run["stage_ms"], main_run["value"]
    barrier = o["barrier"]
    work, fma_peak = None, None
    if rank == 0:
        try:  # debug entry points, outside every timed region: work counters of the last frame + FP32 FMA peak of this GPU
            work = ctx.work_counters(particles.data_ptr(), rays_o.data_ptr(), rays_d.data_ptr())
            fma_peak = ctx.fma_peak_tflops()
        except RuntimeError as e:
            print(f"bench.py: work counters unavailable: {e}", file=sys.stderr)

    # ---- end to end through the public API: Tracer.render + loss.backward, camera batch from pinned host memory
    class _G:
        positions = particles[:, 0:3].clone().requires_grad_(True)
        _d = particles[:, 3:4].clone().requires_grad_(True)
        _r = particles[:, 4:8].clone().requires_grad_(True)
        _s = particles[:, 8:11].clone().requires_grad_(True)
        _f = sph.clone().requires_grad_(True)
        n_active_features = sc.sph_degree
        ray_feature_dim = 3
        num_gaussians = n
        get_rotation = staticmethod(lambda: _G._r)
        get_scale = staticmethod(lambda: _G._s)
        get_density = staticmethod(lambda: _G._d)
        get_features = staticmethod(lambda: _G._f)

    pin_o, pin_d = torch.from_numpy(ro_np).pin_memory(), torch.from_numpy(rd_np).pin_memory()
    pin_gt = torch.rand((1, H, W, 3)).pin_memory()
    intr = dict(resolution=np.array([W, H]), shutter_type="GLOBAL", principal_point=np.array([sc.cx, sc.cy], np.float32),
                focal_length=np.array([sc.fx, sc.fy], np.float32), radial_coeffs=np.zeros(6, np.float32),
                tangential_coeffs=np.zeros(2, np.float32), thin_prism_coeffs=np.zeros(4, np.float32))

    class _B:
        T_to_world_end = None
        rays_in_world_space = False
        intrinsics = None
        intrinsics_OpenCVPinholeCameraModelParameters = intr

    c2ws = [torch.from_numpy(np.asarray(sc.camera(i, n_views), np.float32))[None] for i in range(n_views)]
    grads = [_G.positions, _G._d, _G._r, _G._s, _G._f]

    feed = HostFeed(torch, dev, [pin_o, pin_d, pin_gt])

    def step_e2e(step):
        b = _B()
        b.rays_ori, b.rays_dir, gt = feed.take()
        b.T_to_world = c2ws[view_of(step)]
        for g in grads:
            g.grad = None
        out = tracer.render(_G, b, train=True, frame_id=step)
        loss = (out["pred_features"] - gt).abs().mean() + 0.01 * out["pred_opacity"].mean()
        loss.backward()
        if world > 1:
            for g in grads:
                dist.all_reduce(g.grad)
        return feed.give_loss(loss)  # D2H read of the step's result (pinned slot, consumed one step later)

    e2e_steps = max(10, args.steps // 2)
    for s in range(min(args.warmup, 5)):
        step_e2e(s)
    barrier()
    t0 = time.perf_counter()
    prof = None
    if args.profile_host:
        import cProfile
        prof = cProfile.Profile()
        prof.enable()
    for s in range(e2e_steps):
        step_e2e(args.warmup + s)
    if prof is not None:
        prof.disable()
        import io, pstats
        buf = io.StringIO()
        pstats.Stats(prof, stream=buf).sort_stats("cumulative").print_stats(70)
        pstats.Stats(prof, stream=buf).sort_stats("tottime").print_stats(40)
        with open(args.profile_host, "w") as f:
            f.write(f"steps {e2e_steps}\n" + buf.getvalue())
    e2e_host_ms = (time.perf_counter() - t0) * 1e3 / e2e_steps  # host time to ISSUE a step (includes the forward's wait on the list total)
    feed.drain()
    barrier()
    e2e_s = torch.tensor([time.perf_counter() - t0], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * e2e_steps / float(e2e_s.item())
    h2d = int(pin_o.numel() * 4 + pin_d.numel() * 4 + pin_gt.numel() * 4)

    # ---- measurements beside the metric (rank 0, N = 1): the reference's own kernels on this GPU, optimizer step, image loss
    extras = {}
    peak, peak_src = load_peaks()
    if rank == 0 and world == 1:
        if not args.no_reference_gpu:
            rg = time_reference_gpu(torch, dev, sc, poses, particles, sph, rays_o, rays_d, d_rgba, d_dist, flush, view_of, steps=min(args.steps, 30))
            if rg is not None:
                extras["reference_gpu"] = rg
                if "value" in rg:
                    ours_map = {"project": "project", "prepare_expand": "scan", "expand": "expand", "sort": "sort+tile_ranges", "render": "render",
                                "render_backward": "render_backward", "project_backward": "project_backward"}
                    ours_stage = dict(stage_ms)
                    ours_stage["sort+tile_ranges"] = stage_ms["sort"] + stage_ms["tile_ranges"]
                    extras["vs_reference_gpu"] = {"speedup_device_timed": value / rg["value"],
                                                  "per_stage_ours_over_reference_ms": {k: [ours_stage[v], rg["stage_ms"][k]] for k, v in ours_map.items()}}
        extras["optimizer_step"] = time_optimizer_step(torch, dev, n, flush, peak, peak_src)
        extras["image_loss"] = time_image_loss(torch, dev, H, W, flush, peak, peak_src)

    # ---- sub-records of the default line (same process, same ranks, short runs; never part of `value`): BASELINE configs[2] (C3: 6M
    # Gaussians at 1237x822, the configuration the 1->8 GPU curve is named on) and, at N=1, configs[3] (C4: the C2 scene through 3DGRT)
    sub_records = {}
    run_info = {k: v for k, v in main_run.items() if k != "objs"}
    sc_name = sc.name
    if args.workload == "c2" and not args.no_sub_records:
        del main_run, o, tracer, raster, ctx, particles, sph, rays_o, rays_d, d_rgba, d_dist, flush, feed, _G, grads
        torch.cuda.empty_cache()
        want_sub = set(args.sub_records.split(","))
        if world == 1 and "train_default" in want_sub:
            td = gut_device_loop(torch, dist, args, rank, world, dev, "c2", steps=min(args.steps, 50), warmup=5, stage_pass=True, zero_dist_grad=True)
            sub_records["train_default"] = {"workload": td["objs"]["sc"].name, "value": td["value"], "unit": UNIT, "steps": td["steps"],
                                            "ms_per_step": td["total_ms"] / td["steps"], "stage_ms": td["stage_ms"],
                                            "note": "the headline loop with a ZERO distance gradient (a loss on rgb / opacity only, the reference's default "
                                                    "training loss): renderBackward then skips the depth branch of the adjoint; `value` keeps random "
                                                    "gradients on every output (rgba and distance), the harder case"}
            del td
            torch.cuda.empty_cache()
        if "c3" in want_sub:
            c3 = gut_device_loop(torch, dist, args, rank, world, dev, "c3", steps=max(2 * args.accumulate, 12), warmup=4, stage_pass=True)
            sub_records["c3"] = {"workload": c3["objs"]["sc"].name, "value": c3["value"], "unit": UNIT, "n_gpus": world, "steps": c3["steps"],
                                 "ms_per_step": c3["total_ms"] / c3["steps"], "stage_ms": c3["stage_ms"], "exchange": c3["exchange"],
                                 "N": c3["stats"]["N"], "V": c3["stats"]["V"], "I": c3["stats"]["I"], "T": c3["stats"]["T"],
                                 "note": "BASELINE configs[2]: 6M Gaussians, 1237x822; same loop, timing and exchange as the headline, fewer steps"}
            del c3
            torch.cuda.empty_cache()
        if world == 1 and "c4" in want_sub:
            sub_records["c4"] = run_grt(args, rank, local_rank, world, dev, dist, sub=True)

    if rank == 0:
        N_, I_, V_, T_, P_ = stats["N"], stats["I"], stats["V"], stats["T"], H * W
        # algorithmic bytes per launch (SURVEY.md 8d bracketed terms; DESIGN.md section 4)
        stage_bytes = {
            "project": 92 * N_ + 204 * V_,
            "scan": 8 * N_,
            "expand": 8 * N_ + 36 * V_ + 12 * I_,
            "sort": (8 + 24 * ((32 + int(np.ceil(np.log2(max(T_, 2)))) + 7) // 8)) * I_,
            "tile_ranges": 8 * I_ + 8 * T_,
            "render": 8 * T_ + 64 * I_ + 48 * P_,
            "render_backward": 8 * T_ + 64 * I_ + 64 * P_ + 112 * V_,
            "project_backward": 4 * N_ + 444 * V_ + 112 * N_,
        }
        dom = max(stage_ms, key=lambda k: stage_ms[k])
        dom_ms = stage_ms[dom]
        traffic = None  # dram__bytes_read+write of that kernel from the committed ncu --set full capture of this workload
        tpath = os.path.join(ROOT, "profiles", "r02_traffic.json")
        if os.path.exists(tpath):
            tj = json.load(open(tpath))
            if tj.get("workload") == sc_name:
                traffic = tj["dram_bytes_per_launch"].get({"render": "render_forward"}.get(dom, dom))
        achieved = stage_bytes[dom] / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else 0.0
        # SURVEY 8d "Algorithmic FLOPs for G6/G7": 65 per pair test + 30 per accepted hit (forward) / 400 per accepted hit (adjoint), with the
        # pair tests of the REFERENCE's loop (every live pixel tests every list entry) counted on the device for this frame, over the live
        # kernel times; the denominator is the FMA micro-benchmark run in this process
        fp32 = None
        if work is not None:
            f_fwd = 65.0 * work["tests_ref"] + 30.0 * work["hits"]
            f_bwd = 65.0 * work["tests_ref"] + 400.0 * work["hits"]
            t_fwd, t_bwd = stage_ms["render"] * 1e-3, stage_ms["render_backward"] * 1e-3
            fp32 = {"unit": "TFLOP/s", "peak": fma_peak, "peak_source": "FMA micro-benchmark in this run (gutb200_debug_fma_peak: 8 chains/thread, 2 flops/FMA)",
                    "formula": "(65*tests_ref + 30*hits) / t_render ; (65*tests_ref + 400*hits) / t_render_backward (SURVEY 8d)",
                    "render": {"achieved": f_fwd / t_fwd / 1e12, "frac": f_fwd / t_fwd / 1e12 / fma_peak if fma_peak else None},
                    "render_backward": {"achieved": f_bwd / t_bwd / 1e12, "frac": f_bwd / t_bwd / 1e12 / fma_peak if fma_peak else None},
                    "work": work,
                    "executed": {"forward_lane_tests": work["tests_exec"], "backward_lane_tests_whole_warp_walk": work["bwd_lanes"],
                                 "forward_warp_iterations": work["fwd_iters"],
                                 "backward_warp_iterations": {"quarter_warp_walk (default)": work["iters8"], "half_warp_walk": work["iters16"],
                                                              "whole_warp_walk": work["hit_iters"]},
                                 "gradient_rows_flushed": {"quarter": work["sub8_hits"], "half": work["sub16_hits"], "whole": work["hit_iters"]},
                                 "hit_lanes_per_whole_warp_iteration": work["hits"] / max(work["hit_iters"], 1)}}
        frame_bytes = 356 * N_ + 796 * V_ + (156 + 24 * 6) * I_ + 24 * T_ + 136 * P_
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": run_info["steps"], "warmup": run_info["warmup"],
            "ms_per_step": total_ms / run_info["steps"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": sc_name, "gaussians": n, "resolution": [W, H], "path": "3dgut", "step": "one view per rank, forward + backward",
                       "views_per_step": world, "views_per_batch": world * run_info["accumulate"],
                       "parallelism": f"view-parallel dp{world}, gradients summed every {run_info['accumulate']} view-steps" if world > 1 else "single",
                       "exchange": (args.exchange if world > 1 else "none"), "l2": "flushed between timed steps (256 MiB fill)",
                       "N": N_, "V": V_, "I": I_, "T": T_, "P": P_},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4, "steps": e2e_steps, "host_issue_ms_per_step": e2e_host_ms,
                    "api": "threedgut_tracer.Tracer.render + loss.backward",
                    "feed": "pinned host -> device on a copy stream, one step ahead; loss read back one step later"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": int(stage_bytes[dom]),
                         "kernel_ms": dom_ms,
                         "note": "render/render_backward are FP32-issue bound (SURVEY 8d): the HBM fraction is reported as required; "
                                 "roofline_fp32 (work counters and FMA peak both measured in this run) is the figure that bounds them"},
            "roofline_fp32": fp32,
            "stage_ms": stage_ms,
            "frame_algorithmic_gbs": frame_bytes / (total_ms / run_info["steps"] * 1e-3) / 1e9,
        }
        if run_info["exchange"] is not None:
            line["exchange"] = run_info["exchange"]
        line.update(sub_records)
        line.update(extras)
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            sc_cpu = make_scene(args.workload)
            fps, _ = cpu_port_frames_per_s(sc_cpu, 1, frames=1, warm=0)
            line["cpu_baseline"] = {"value": fps, "unit": UNIT, "cores": cores, "kind": "port",
                                    "sample": "1 whole view (every tile) through the CPU port: projection + binning + compositing forward + backward, OpenMP over tiles"}
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()

if __name__ == "__main__":
    main()
