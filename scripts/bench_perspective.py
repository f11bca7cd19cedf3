#!/usr/bin/env python
"""Cost of perspective-correct interpolation: ms per forward + adjoint step, replayed from a CUDA graph as bench.py
times its steps, for the same scene with and without perspective_correct.  The perspective step adds the depths_b
output (deodr_b200_render_b_views_depths); the projection that would consume it is not part of the step.

    python scripts/bench_perspective.py [--steps 20] [--warmup 3]

Prints one JSON line per scene, and the GPU name and power limit first (they are part of every number)."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from deodr_b200.renderer import DeviceScene, Renderer  # noqa: E402
from deodr_b200.scenes import dense_image_b, torus_scene  # noqa: E402

SCENES = {
    "c5": dict(n=708, width=2048, height=2048, views=1, textured=False),          # 1M triangles, 2048^2
    "textured_50k": dict(n=158, width=1024, height=1024, views=1, textured=True),  # 50k triangles, 1024^2
    "views_8x200k": dict(n=316, width=512, height=512, views=8, textured=False),   # 8 views of 200k triangles, 512^2
}


def gpu_description():
    name = torch.cuda.get_device_name(0)
    try:
        power = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        power = "unknown"
    return {"gpu": name, "power_limit": power}


def time_step(cfg, persp, steps, warmup):
    r = Renderer(0)
    scenes = []
    for v in range(cfg["views"]):
        s = torus_scene(cfg["n"], cfg["width"], cfg["height"], view=v, n_views=cfg["views"], textured=cfg["textured"])
        s.perspective_correct = persp
        scenes.append(s)
    dss = [DeviceScene(s, "cuda:0") for s in scenes]
    image_b = torch.from_numpy(dense_image_b(np.zeros((cfg["height"], cfg["width"], 3)), seed=3).astype(np.float32)).cuda()
    image_bs = [image_b] * len(dss)
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        out = r.render_views(dss, 1.0)  # builds the plans
        grads = r.render_b_views(dss, 1.0, out, image_bs, depths_b=persp)
        torch.cuda.synchronize()
        r.set_deferred(True)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=stream):
            for g in grads:
                for t in g.values():
                    t.zero_()
            r.render_views(dss, 1.0, out=out)
            r.render_b_views(dss, 1.0, out, image_bs, grads, depths_b=persp)
        for _ in range(warmup):
            graph.replay()
        torch.cuda.synchronize()
        times = []
        for _ in range(steps):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(stream)
            graph.replay()
            b.record(stream)
            b.synchronize()
            times.append(a.elapsed_time(b))
        r.status()
        r.set_deferred(False)
    return float(np.median(times)), float(np.min(times))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--scenes", default=",".join(SCENES))
    args = ap.parse_args()
    print(json.dumps(gpu_description()), flush=True)
    for name in args.scenes.split(","):
        cfg = SCENES[name]
        row = {"scene": name}
        for persp in (False, True):
            med, best = time_step(cfg, persp, args.steps, args.warmup)
            key = "perspective" if persp else "affine"
            row[key + "_ms_median"], row[key + "_ms_min"] = round(med, 4), round(best, 4)
        row["ratio_median"] = round(row["perspective_ms_median"] / row["affine_ms_median"], 3)
        print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
