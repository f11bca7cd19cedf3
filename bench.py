#!/usr/bin/env python
"""Benchmark of the hot path: fwd+bwd Mpixels/s of the differentiable rasteriser (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our sm_100a path
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's CPU path on the host cores

Workload (N = 1): BASELINE.json configs[4] - S-mesh(708): 1,002,528-triangle closed torus, 2048x2048, C = 3, Gouraud
vertex colours, sigma = 1 edge-overdraw antialiasing, dense image_b; one "step" = per-iteration refresh of ij/colours
+ gradient clear + renderScene (forward) + renderScene_B (adjoint) of the rank's views (--views-per-gpu, default 1;
`--workload c4` = BASELINE configs[3]: 8 views per GPU of the 200k-triangle mesh at 512x512, an RGB and a depth render
each).  N > 1: weak scaling over the batch-of-views axis (same mesh, different cameras), plus ONE NCCL all-reduce per
step of the gradient of the shared parameter (vertex colours, colors_b[V,C]); ij_b is per view.  The all-reduce runs on a
communication stream and only the colour readers of the NEXT forward wait for it (deodr_b200_workspace_set_colors_ready),
so it overlaps that forward's binning and z pass.

One JSON line on rank 0; keys follow the driver contract, plus `roofline`, `cpu_baseline`, `e2e`, `clocks`.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (torus n, width, height, textured, nb_colors, description)
    "c5": (708, 2048, 2048, False, 3, "1M-tri synthetic torus mesh (T=1002528), 2048x2048, C=3, sigma=1, fwd+bwd"),
    "c3": (158, 1024, 1024, True, 3, "50k-tri textured torus mesh (T=49928), 1024x1024, bilinear UV, sigma=1, fwd+bwd"),
    "c4": (316, 512, 512, False, 3, "200k-tri torus mesh (T=199712), 512x512 RGB view, sigma=1, fwd+bwd"),
    "c2": (23, 640, 480, False, 3, "1k-tri torus mesh (T=1058; stand-in for the 1048-face hand mesh), 640x480, fwd+bwd"),
    "c3u": (158, 1024, 1024, False, 3, "c3 without the texture (development A/B)"),
    "c5t": (708, 2048, 2048, True, 3, "c5 with a 512x512 texture on every triangle (development A/B)"),
    "dev": (100, 512, 512, False, 3, "development-size torus"),
}
METRIC = "fwd+bwd Mpixels/s"
UNIT = "Mpixels/s"
SIGMA = 1.0


def algorithmic_bytes(scene):
    """SURVEY.md section 8(d): canonical layout, every plane / record touched once per direction."""
    P, C = scene.height * scene.width, scene.nb_colors
    T, V, U = scene.faces.shape[0], scene.depths.shape[0], scene.uv.shape[0]
    b_fwd = P * (4 * C + 8 + 4) + T * (12 + 3 + 2) + V * (16 + 8 + 4 * C)
    b_bwd = b_fwd + V * (8 + 4 * C)
    if scene.textured.any():
        tex = scene.texture.size * 4
        b_fwd += T * 12 + U * 8 + V * 4 + tex
        b_bwd += T * 12 + U * 8 + V * 4 + tex + U * 8 + V * 4 + tex
    return b_fwd, b_bwd


def kernel_algorithmic_bytes(scene):
    """Share of the SURVEY section 8(d) byte budget each raster kernel is responsible for (per launch = one view):
    every framebuffer plane / primitive record / vertex record counted once, in the kernel that has to touch it."""
    P, C = scene.height * scene.width, scene.nb_colors
    T, V, U = scene.faces.shape[0], scene.depths.shape[0], scene.uv.shape[0]
    tex = scene.texture.size * 4 if scene.textured.any() else 0
    tex_terms = (T * 12 + U * 8 + V * 4 + tex) if tex else 0
    return {
        # the single binning pass: faces + flags (17 T) and ij + depths (24 V) read (its 64-byte records are overhead)
        "bin": T * 17 + V * 24,
        # z-buffer (8) + face / owner id (4) written; faces + flags (17 T) and ij + depths (24 V) read
        "tile_z": P * 12 + T * 17 + V * 24,
        # image written (4C), vertex colours read (+ uv / shade / texture)
        "shade": P * 4 * C + V * 4 * C + tex_terms,
        # image_b (4C) + owner (4) + z (8) read, geometry + colours read, gradients written
        "small_tri_bwd": P * (4 * C + 12) + T * 17 + V * (24 + 4 * C) + V * (8 + 4 * C) + tex_terms + (U * 8 + V * 4 + tex if tex else 0),
        "interior_bwd": P * (4 * C + 12) + T * 17 + V * (24 + 4 * C) + V * (8 + 4 * C) + tex_terms + (U * 8 + V * 4 + tex if tex else 0),
    }


def measured_peak_gbs():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region through NVML (every ~2 ms; nvidia-smi's 100 ms
    loop is too coarse for a region of a few tens of milliseconds).  Falls back to one nvidia-smi query."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown"}

    def __init__(self, index: int):
        self.index = index
        self.samples = []
        self.mask = 0
        self.stop_flag = False
        self.thread = None
        self.nvml = None
        self.sm_max = None
        try:
            import pynvml

            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def _loop(self):
        nv = self.nvml
        while not self.stop_flag:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)))
                self.mask |= int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self.nvml:
            self.thread = threading.Thread(target=self._loop, daemon=True)
            self.thread.start()

    def stop(self):
        if self.thread:
            self.stop_flag = True
            self.thread.join(timeout=1)
            reasons = sorted(name for bit, name in self.REASONS.items() if self.mask & bit)
            return {"sm_mhz": statistics.median(self.samples) if self.samples else None, "sm_max_mhz": self.sm_max,
                    "samples": len(self.samples), "reasons": reasons, "source": "nvml, 2 ms period, timed region only"}
        try:
            out = subprocess.run(["nvidia-smi", f"--id={self.index}", "--query-gpu=clocks.sm,clocks.max.sm",
                                  "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
            sm, smax = [float(x) for x in out.strip().split(",")]
            return {"sm_mhz": sm, "sm_max_mhz": smax, "samples": 1, "reasons": [], "source": "nvidia-smi after the region"}
        except Exception:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["clock query unavailable"]}


def build_scene(workload: str, view: int, n_views: int):
    from deodr_b200.scenes import torus_scene

    n, W, H, textured, C, _ = WORKLOADS[workload]
    return torus_scene(n, W, H, view=view, n_views=n_views, textured=textured, nb_colors=C)


# ------------------------------------------------------------------------------------------------- our arm


def run_ours(args):
    import torch
    import torch.distributed as dist

    from deodr_b200.distributed import allreduce_flat
    from deodr_b200.renderer import DeviceScene, Renderer

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
    dev = torch.device(f"cuda:{local}")

    per_gpu = args.views_per_gpu if args.views_per_gpu > 0 else (8 if args.workload == "c4" else 1)
    n_views = per_gpu * max(world, 1)
    depth_too = args.workload == "c4"  # configs[3]: "depth+RGB"
    scenes = [build_scene(args.workload, view=rank * per_gpu + v, n_views=n_views) for v in range(per_gpu)]
    if depth_too:
        for v in range(per_gpu):
            d = build_scene(args.workload, view=rank * per_gpu + v, n_views=n_views)
            d.nb_colors, d.colors = 1, np.ascontiguousarray(d.depths[:, None])
            d.background_color = np.array([float(d.depths.max())])
            d.texture = np.zeros((2, 2, 1))
            scenes.append(d)
    scene = scenes[0]
    H, W, C = scene.height, scene.width, scene.nb_colors
    P = H * W
    renderer = Renderer(local)
    dss = [DeviceScene(s, dev) for s in scenes]
    ij_dev = [ds.t["ij"].clone() for ds in dss]
    colors_dev = [ds.t["colors"].clone() for ds in dss]
    rng = np.random.default_rng(1 + rank)
    image_bs = [torch.from_numpy(rng.random((s.height, s.width, s.nb_colors), dtype=np.float32) * 2 - 1).to(dev)
                for s in scenes]
    # gradient slots: ONE flat buffer (callers clear scene.*_b before every backward: one memset); the gradients of
    # the parameters the views share (colours per render kind, uv, shade, texture) are shared views of it, ij_b is
    # per view - the `+=` of deodr/mesh_fitter.py:518-527 happens in place
    kinds, total = {}, 0
    for ds in dss:  # shared blocks first: they form the prefix that is all-reduced
        if ds.nb_colors not in kinds:
            kinds[ds.nb_colors] = {}
            for k, n in (("colors_b", "colors"), ("uv_b", "uv"), ("shade_b", "shade"), ("texture_b", "texture")):
                kinds[ds.nb_colors][k] = (total, ds.t[n].shape)
                total += int(np.prod(ds.t[n].shape))
    shared_end = total
    layout = []
    for ds in dss:
        layout.append((total, ds.t["ij"].shape))
        total += int(np.prod(ds.t["ij"].shape))
    flat = torch.zeros(total, dtype=torch.float32, device=dev)
    view_of = lambda off, shape: flat[off:off + int(np.prod(shape))].view(shape)  # noqa: E731
    grads = []
    for i, ds in enumerate(dss):
        g = {k: view_of(*kinds[ds.nb_colors][k]) for k in ("colors_b", "uv_b", "shade_b", "texture_b")}
        g["ij_b"] = view_of(*layout[i])
        grads.append(g)
    outs = None
    # (high priority: the collective's few CTAs and the colour update behind it must not queue behind the binning pass)
    comm = torch.cuda.Stream(device=dev, priority=-1) if world > 1 else None
    ev_bwd = torch.cuda.Event()
    ev_colors = torch.cuda.Event()
    overlap = world > 1 and not args.no_overlap

    def compute(wait_colors=True):
        """The device work of one fitting step on the compute stream: refresh, clear, forward, adjoint."""
        nonlocal outs
        for ds, ij, col in zip(dss, ij_dev, colors_dev):      # per-iteration refresh of the optimised inputs
            ds.update(ij=ij)
        if overlap:
            # the colours are written by the "optimiser" on the communication stream (after the all-reduce of the
            # previous step): only the kernels of this forward that READ colours wait for that, and colors_b - which the
            # communication stream zeroes once the all-reduce has consumed it - is only touched after that wait
            if wait_colors:
                renderer.set_colors_ready(ev_colors)
            flat[shared_end:].zero_()                         # the per-view ij_b
        else:
            for ds, col in zip(dss, colors_dev):
                ds.update(colors=col)
            flat.zero_()                                      # callers clear scene.*_b before every backward
        outs = renderer.render_views(dss, SIGMA, out=outs)
        renderer.render_b_views(dss, SIGMA, outs, image_bs, grads)

    def compute_head():
        """N > 1, replayed: the colour-independent head of the step (refresh of ij, clear of ij_b, binning) ..."""
        nonlocal outs
        for ds, ij in zip(dss, ij_dev):
            ds.update(ij=ij)
        flat[shared_end:].zero_()
        outs = renderer.render_views(dss, SIGMA, out=outs, part="geometry")

    def compute_tail():
        """... and the rest of it (colour readers of the forward, adjoint), behind the wait for the colours."""
        nonlocal outs
        outs = renderer.render_views(dss, SIGMA, out=outs, part="resume")
        renderer.render_b_views(dss, SIGMA, outs, image_bs, grads)

    def communicate():
        """One flat all-reduce of every shared gradient + the optimiser's colour update, on the communication stream."""
        if world == 1:
            return
        if overlap:
            ev_bwd.record()
            with torch.cuda.stream(comm):
                comm.wait_event(ev_bwd)
                # deodr_b200.distributed: ONE flat collective; a synchronous op is enqueued on the current (= the
                # communication) stream, without the hop through the process group's own stream
                allreduce_flat([flat[:shared_end]])
                for ds, col in zip(dss, colors_dev):           # stand-in for the optimiser's colour update
                    ds.update(colors=col)
                flat[:shared_end].zero_()
                ev_colors.record(comm)
        else:
            allreduce_flat([flat[:shared_end]])                # shared-parameter gradients, one call per step

    def step():
        compute()
        communicate()

    def fence():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if overlap:
        ev_colors.record(comm)
    for _ in range(args.warmup):
        step()
    if overlap:
        torch.cuda.current_stream().wait_stream(comm)
    fence()

    # ---- the timed region replays the step as CUDA graphs (nothing inside the passes touches the host: deferred
    # verdicts, checked after the region).  --eager times the plain calls instead (also the fallback when a capture fails).
    graph, graph_head, graph_note = None, None, None

    def replay():
        """One step as graph replays.  N > 1: the collective stays outside the graphs and the step is TWO graphs with an
        ordinary stream wait for the colours between them - an event wait captured INSIDE one graph of the whole step
        (an external event wait node) holds back the launch of that whole graph until the all-reduce of the step before
        has finished (measured, 2 GPUs: 0.411 ms per step against 0.387 ms for the plain calls), which is exactly the
        overlap the wait was meant to keep."""
        if graph_head is not None:
            graph_head.replay()
            torch.cuda.current_stream().wait_event(ev_colors)
        graph.replay()
        communicate()

    if not args.eager:
        try:
            renderer.set_deferred(True)
            cap = torch.cuda.Stream(device=dev)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.stream(cap):
                if overlap:
                    graph_head = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(graph_head, stream=cap, capture_error_mode="thread_local"):
                        compute_head()
                    with torch.cuda.graph(graph, stream=cap, capture_error_mode="thread_local"):
                        compute_tail()
                else:
                    with torch.cuda.graph(graph, stream=cap, capture_error_mode="thread_local"):
                        compute()
            for _ in range(2):
                replay()
            if overlap:
                torch.cuda.current_stream().wait_stream(comm)
            fence()
            renderer.status()
        except Exception as exc:  # capture is an optimisation of the launch path, never a requirement
            graph = graph_head = None
            graph_note = f"capture failed, eager calls timed instead: {type(exc).__name__}: {str(exc)[:200]}"
            renderer.set_deferred(False)
            torch.cuda.synchronize()
            if overlap:
                ev_colors.record(comm)
            step()
            fence()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    side = torch.cuda.Stream(device=dev) if args.side_stream else None
    if side is not None:  # (A/B: the steps on a non-default stream, where DEODR_B200_GRAPHS=1 can capture them)
        side.wait_stream(torch.cuda.current_stream())
        torch.cuda.set_stream(side)
        for _ in range(3):
            step()
        fence()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    if graph is not None:
        for _ in range(args.steps):
            replay()
        if overlap:
            torch.cuda.current_stream().wait_stream(comm)
    else:
        for _ in range(args.steps):
            step()
        if overlap:
            torch.cuda.current_stream().wait_stream(comm)
    stop.record()
    fence()
    elapsed_ms = start.elapsed_time(stop)
    clocks = sampler.stop() if rank == 0 else None
    if graph is not None:
        renderer.status()  # raises if a replayed pass overflowed its plan (its results would be void)
        renderer.set_deferred(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outs, grads, len(scenes))
    if world > 1:
        t = torch.tensor([elapsed_ms], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        elapsed_ms = float(t.item())
    ms_per_step = elapsed_ms / args.steps
    pixels_per_step = world * sum(s.height * s.width for s in scenes)
    value = pixels_per_step / (ms_per_step * 1e-3) / 1e6

    # ---- second region, same process, same K steps through the plain (eager) calls with the library's per-kernel CUDA
    # events switched on: kernel durations for the roofline, launch count, and the eager step time next to the replayed one
    if overlap:
        ev_colors.record(comm)
    step()
    fence()
    renderer.timing_enable(14 * args.steps * len(dss) + 16)
    launches0 = renderer.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        step()
    if overlap:
        torch.cuda.current_stream().wait_stream(comm)
    e1.record()
    fence()
    eager_ms = e0.elapsed_time(e1) / args.steps
    launches = renderer.launches - launches0
    phases = renderer.timing_collect()
    renderer.timing_enable(0)
    if graph is None:
        graph_note = graph_note or "--eager"

    # ---- per-kernel durations inside the timed region -> roofline of the dominant kernel
    per_phase = {}
    for name, ms in phases:
        per_phase.setdefault(name, []).append(ms)
    phase_ms = {k: statistics.mean(v) for k, v in per_phase.items()}
    b_fwd = sum(algorithmic_bytes(s)[0] for s in scenes)
    b_bwd = sum(algorithmic_bytes(s)[1] for s in scenes)
    kernel_bytes = kernel_algorithmic_bytes(scene)
    if "shade" not in phase_ms:  # the colour pass ran as the z pass's epilogue: one kernel owns both byte budgets
        kernel_bytes["tile_z"] += kernel_bytes["shade"]
    peak, peak_src = measured_peak_gbs()
    roofline = None
    # The forward's z pass and shading run back to back on the caller's stream, so their event brackets are their
    # own durations; the three adjoint kernels run CONCURRENTLY on forked streams (their brackets overlap and sum to
    # more than the backward pass), so they are reported in phase_ms but not used as the roofline kernel.
    raster = {k: v for k, v in phase_ms.items() if k in ("tile_z", "shade", "bin")}
    if raster:
        kernel = max(raster, key=raster.get)
        t_k, b_k = raster[kernel], kernel_bytes[kernel]
        achieved = b_k / (t_k * 1e-3) / 1e9
        traffic, traffic_src, step_traffic = None, None, None
        try:
            doc = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
            traffic = doc.get(args.workload, {}).get(kernel)
            step_traffic = doc.get(args.workload, {}).get("step")  # every kernel of one forward + adjoint
            traffic_src = doc.get("source")
        except Exception:
            pass
        roofline = {
            "bound": "hbm", "kernel": kernel, "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
            "frac": round(achieved / peak, 4), "traffic": traffic, "traffic_source": traffic_src,
            "peak_source": peak_src,
            "algorithmic_bytes_per_launch": b_k, "kernel_ms": round(t_k, 4),
            "phase_ms": {k: round(v, 4) for k, v in phase_ms.items()},
            "phase_note": "measured in the eager region that follows the timed one (same process, same K steps), per launch (one view); edge_bin/edge_tile_sort overlap tile_z..shade; edge_bwd, interior_bwd "
                          "and small_tri_bwd overlap each other (forked streams): brackets, not exclusive times; "
                          "`plan` only appears when a plan was (re)built",
            "step_algorithmic_bytes": b_fwd + b_bwd,
            "step_frac_of_peak": round((b_fwd + b_bwd) / (ms_per_step * 1e-3) / 1e9 / peak, 4),
            # DRAM traffic of all kernels of one view's forward + adjoint in the same ncu capture (one view per step only)
            "step_traffic": step_traffic if len(scenes) == 1 else None,
        }

    # ---- end to end through the reference-facing plugin call with HOST (numpy fp64) buffers
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, scene, world, dev)

    # ---- CPU baseline beside it: rank 0, N = 1 only
    cpu_baseline = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu_baseline = time_cpu(scene, threads=1, repeats=1)

    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64 geometry/z + f32 colours/gradients", "data": "synthetic",
        "config": {
            "workload": f"{args.workload}: {WORKLOADS[args.workload][5]}",
            "triangles": int(scene.faces.shape[0]), "vertices": int(scene.depths.shape[0]), "height": H, "width": W,
            "nb_colors": C, "sigma": SIGMA, "views_per_gpu": per_gpu,
            "renders_per_view": "RGB (C=3) + depth (C=1)" if depth_too else "RGB (C=3)" if C == 3 else f"C={C}",
            "parallelism": f"views x{world}" + (" + NCCL all-reduce of the shared gradients" +
                                                (" overlapped with the next forward (colours-ready event)" if overlap else "")
                                                if world > 1 else ""),
            "timed_region": (("CUDA graph replay of the step's device work" +
                              (", collective outside the graphs" +
                               (" (binning graph | wait for the colours | raster + adjoint graph)" if graph_head is not None else "")
                               if world > 1 else ""))
                             if graph is not None else f"eager calls ({graph_note})"),
            "eager_ms_per_step": round(eager_ms, 4),
            "l2_policy": "inputs larger than L2: each step touches >= %.0f MB (algorithmic) vs 126 MB L2" % ((b_fwd + b_bwd) / 1e6),
        },
        "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e,
        "clocks": clocks,
    }
    print(json.dumps(line), flush=True)


DUMP_BYTES = 64 << 20


def dump_outputs(path, outs, grads, n_views):
    """Writes what the last timed step returned to its caller - per view the image and z-buffer of the forward and the
    gradients of the adjoint - as <path>/<name>.npy, flattened, in the float32 / float64 they were computed in.
    One process only (main() refuses the option otherwise).

    Pixels that no triangle covers have a z of +inf; the z-buffer is written with 0 there and <name>_finite.npy holds
    1.0 where z is finite, so that every file is finite.  Each output gets an equal share of DUMP_BYTES; a larger one
    is reduced to the elements at np.sort(np.random.default_rng(0).choice(n, k, replace=False)), the same sample in
    every run, so that two builds can be compared output for output."""
    os.makedirs(path, exist_ok=True)
    arrays = {}
    for v in range(n_views):
        arrays[f"view{v}_image"] = outs[v]["image"]
        z = outs[v]["z_buffer"]
        finite = z.isfinite()
        arrays[f"view{v}_z_buffer"] = z.where(finite, z.new_zeros(()))
        arrays[f"view{v}_z_buffer_finite"] = finite.double()  # float64 like z: the same sample of pixels
        for name in ("ij_b", "colors_b", "uv_b", "shade_b", "texture_b"):
            if grads[v][name].numel():
                arrays[f"view{v}_{name}"] = grads[v][name]
    share = DUMP_BYTES // len(arrays)
    total = 0
    for name, t in arrays.items():
        a = t.detach().reshape(-1).cpu().numpy()
        k = share // a.itemsize
        if a.size > k:
            a = a[np.sort(np.random.default_rng(0).choice(a.size, k, replace=False))]
        assert a.dtype in (np.float32, np.float64) and np.isfinite(a).all(), name
        np.save(os.path.join(path, f"{name}.npy"), a)
        total += a.nbytes
    assert total <= DUMP_BYTES, f"dumped {total} bytes"


def run_e2e(args, scene, world, dev):
    """Same metric through renderSceneCpp / renderSceneBCpp (deodr_b200.differentiable_renderer_cython): numpy fp64
    host arrays in, numpy fp64 host arrays out, host<->device copies inside the timed region."""
    import torch
    import torch.distributed as dist

    from deodr_b200 import differentiable_renderer_cython as shim
    from deodr_b200.differentiable_renderer import Scene2D

    H, W, C = scene.height, scene.width, scene.nb_colors
    s2 = Scene2D(**{k: getattr(scene, k) for k in (
        "faces", "faces_uv", "ij", "depths", "textured", "uv", "shade", "colors", "shaded", "edgeflags", "height",
        "width", "nb_colors", "texture", "background_image", "background_color", "clockwise", "backface_culling",
        "strict_edge", "perspective_correct", "integer_pixel_centers")})
    image = np.empty((H, W, C))
    z = np.empty((H, W))
    image_b = np.random.default_rng(1).random((H, W, C)) * 2 - 1
    steps = max(1, min(args.steps, args.e2e_steps))

    def step():
        s2.clear_gradients()
        shim.renderSceneCpp(s2, SIGMA, image, z)
        shim.renderSceneBCpp(s2, SIGMA, image, z, image_b)

    for _ in range(min(args.warmup, 2)):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    torch.cuda.synchronize()
    dt = (time.perf_counter() - t0) / steps
    if world > 1:
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    # bytes that cross PCIe per step (counted from the arrays the host path copies, host_api.cu): the scene in its
    # canonical device layout once (the adjoint call finds it unchanged in the pinned mirror), image_b as fp32;
    # image as fp32, z_buffer as fp64, the five gradient arrays as fp32.
    canon = {"faces": 4, "faces_uv": 4, "ij": 8, "depths": 8, "uv": 8, "colors": 4, "shade": 4, "edgeflags": 1,
             "textured": 1, "shaded": 1, "texture": 4}
    scene_bytes = sum(np.asarray(getattr(scene, k)).size * w for k, w in canon.items())
    bg = scene.background_image if scene.background_image is not None else scene.background_color
    scene_bytes += np.asarray(bg).size * 4
    grads_bytes = 4 * (s2.ij_b.size + s2.colors_b.size + s2.uv_b.size + s2.shade_b.size + s2.texture_b.size)
    h2d = scene_bytes + image_b.size * 4
    d2h = image.size * 4 + z.size * 8 + grads_bytes
    return {"value": round(world * H * W / dt / 1e6, 2), "unit": UNIT, "ms_per_step": round(dt * 1e3, 3),
            "steps": steps, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "api": "clear_gradients + renderSceneCpp + renderSceneBCpp (numpy fp64 host buffers in and out; staged through "
                   "pinned memory by copy threads, every input copied to the device every step)"}


# ------------------------------------------------------------------------------------------- CPU (reference) arm


def time_cpu(scene, threads: int, repeats: int):
    """fwd+bwd of the SAME scene on the host cores with the reference core (oracle/_ref) or, if it is not built, the
    C restatement (oracle port).  `threads` independent copies run concurrently (ctypes releases the GIL)."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle.oracle import Oracle, available

    kind = "reference" if available("reference") else "port"
    oracle = Oracle(kind)
    H, W, C = scene.height, scene.width, scene.nb_colors
    image_b = np.random.default_rng(1).random((H, W, C)) * 2 - 1

    def one(_):
        image, z = oracle.render(scene, SIGMA)
        oracle.render_b(scene, SIGMA, image, z, image_b)

    times = []
    with ThreadPoolExecutor(max_workers=threads) as pool:
        for _ in range(repeats):
            t0 = time.perf_counter()
            list(pool.map(one, range(threads)))
            times.append(time.perf_counter() - t0)
    dt = statistics.median(times)
    return {"value": round(threads * H * W / dt / 1e6, 3), "unit": UNIT, "cores": threads, "kind": kind,
            "sample": f"{threads} x 1 view fwd+bwd of the same workload, {repeats} repeat(s), {dt:.2f} s each",
            "seconds_per_step": round(dt, 3), "host_cpus": os.cpu_count()}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return  # the reference has no GPU / multi-process path: rank 0 alone measures the host
    scene = build_scene(args.workload, view=0, n_views=max(world, 1))
    threads = max(1, min(os.cpu_count() or 1, args.cpu_threads))
    for _ in range(min(args.warmup, 1)):
        time_cpu(scene, threads, 1)
    repeats = max(1, min(args.steps, args.ref_steps))
    res = time_cpu(scene, threads, repeats)
    line = {
        "impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": world,
        # the steps actually TIMED (bounded sample: one step = `threads` concurrent fwd+bwd of the workload's view)
        "steps": repeats, "steps_requested": args.steps, "warmup": min(args.warmup, 1), "ms_per_step": round(res["seconds_per_step"] * 1e3, 2),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {WORKLOADS[args.workload][5]}", "threads": threads,
                   "bounded_sample": res["sample"]},
        "cpu_baseline": {k: res[k] for k in ("value", "unit", "cores", "kind", "sample")},
        "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c5", choices=sorted(WORKLOADS))
    ap.add_argument("--views-per-gpu", type=int, default=0, help="views rendered per step and GPU (0: 8 for c4, else 1)")
    ap.add_argument("--side-stream", action="store_true", help="run the timed steps on a non-default stream (A/B)")
    ap.add_argument("--eager", action="store_true", help="time the plain calls instead of a CUDA-graph replay of them")
    ap.add_argument("--graph", action="store_true", help="(default) kept for compatibility")
    ap.add_argument("--no-overlap", action="store_true", help="N > 1: all-reduce on the compute stream (A/B)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-steps", type=int, default=10, help="cap on the e2e (host-buffer) timed steps")
    ap.add_argument("--ref-steps", type=int, default=5, help="cap on the bounded reference-arm repeats")
    ap.add_argument("--cpu-threads", type=int, default=64, help="cap on the reference-arm host threads")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (seeded sample of large ones)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.gpus > 1 or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        # with N > 1 the shared gradients are all-reduced and cleared on the communication stream inside the step,
        # so the arrays a caller receives are not left in place after it
        ap.error("--dump-outputs needs --impl ours in a single process (--gpus 1)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    import __graft_entry__ as entry

    if not os.path.exists(entry.LIB):
        entry.build()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
