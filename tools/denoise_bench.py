#!/usr/bin/env python
"""Cost and effect of the denoiser (pt_render_features + pt_denoise), one JSON line per measurement.

    python tools/denoise_bench.py [--repeats R] [--out FILE]

  gpu        card name and power limit (nvidia-smi, read only)
  time       per size (1280x720, 1920x1080, 3840x2160): pt_render_features at 4 spp and pt_denoise with 5 passes on a
             10_final frame, and the 16-spp renders whose noise the filter removes (10_final; the Yoimiya stand-in of
             tests/helpers.py (yoimiya_ground_full) with mesh_camera).  CUDA events on the stream, median of --repeats calls after a warm-up
             call.  Each filter figure is given twice: "warm" = back-to-back calls (the 1080p working set, 48 B per pixel
             per pass, fits the 126 MB L2), "l2_flushed" = a 256 MB buffer is overwritten before every timed call.
  rmse       RMSE of the linear mean against a 4096-spp render of the same scene (other seed) at 4, 16, 64, 256 spp,
             noisy and denoised (4-spp features, 5 passes), for 10_final and the Yoimiya stand-in at 640x360.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))

SIZES = [(1280, 720), (1920, 1080), (3840, 2160)]
DEPTH = 32


def scene(name, size):
    import learn_path_tracing_b200 as L
    from learn_path_tracing_b200 import scenes
    if name == "10_final":
        world, cam = scenes.scene_10_final(size)
        return world, cam, L.PT_SHADE_V2
    from helpers import mesh_camera, stand_in_world
    return stand_in_world("yoimiya_ground_full"), mesh_camera(size), L.PT_SHADE_LEGACY


def timed(fn, repeats, flush=None):
    import torch
    fn()  # warm-up
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(repeats):
        if flush is not None:
            flush.add_(1.0)
        ev0.record()
        fn()
        ev1.record()
        ev1.synchronize()
        ms.append(ev0.elapsed_time(ev1))
    return statistics.median(ms)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--repeats", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import numpy as np
    import torch
    import learn_path_tracing_b200 as L
    from multi_device_bench import gpu_info

    lines = []

    def emit(d):
        print(json.dumps(d), flush=True)
        lines.append(d)

    emit({"gpu": gpu_info()})
    ctx = L.default_context()
    flush = torch.zeros(64 << 20, dtype=torch.float32, device="cuda")  # 256 MB, twice the L2
    for W, H in SIZES:
        world, cam, model = scene("10_final", (W, H))
        sc, cs = world.device_scene(ctx), cam.to_struct()
        r = L.Renderer(W, H, ctx, want_sq=True)
        r.render(sc, cs, 16, DEPTH, model, seed=1, want_stats=False)
        r.features(sc, cs, 4, 1)

        def feats():
            r.feature_planes.zero_()
            r.features(sc, cs, 4, 1)

        def den():
            r.denoised(iterations=5)

        row = {"size": f"{W}x{H}", "pixels": W * H}
        for tag, fl in (("warm", None), ("l2_flushed", flush)):
            row[f"features_4spp_ms_{tag}"] = timed(feats, args.repeats, fl)
            row[f"denoise_5pass_ms_{tag}"] = timed(den, args.repeats, fl)
        row["denoise_dram_bytes_per_pass"] = 48 * W * H  # colour in + colour out + guides, 16 B each per pixel
        for name in ("10_final", "yoimiya_stand_in"):
            world, cam, model = scene(name, (W, H))
            sc2, cs2 = world.device_scene(ctx), cam.to_struct()
            r2 = L.Renderer(W, H, ctx)

            def render():
                r2.clear()
                r2.render(sc2, cs2, 16, DEPTH, model, seed=1, want_stats=False)

            row[f"render_16spp_ms_{name}"] = timed(render, max(3, args.repeats // 2), flush)
            del r2
        emit({"time": row})
        del r
        torch.cuda.empty_cache()

    W, H = 640, 360
    for name in ("10_final", "yoimiya_stand_in"):
        world, cam, model = scene(name, (W, H))
        sc, cs = world.device_scene(ctx), cam.to_struct()
        ref = L.Renderer(W, H, ctx)
        ref.render(sc, cs, 4096, DEPTH, model, seed=1234)
        ref = ref.accum.cpu().numpy()[:, :3] / 4096
        row = {"scene": name, "size": f"{W}x{H}", "reference_spp": 4096}
        for spp in (4, 16, 64, 256):
            r = L.Renderer(W, H, ctx, want_sq=True)
            r.render(sc, cs, spp, DEPTH, model, seed=1)
            r.features(sc, cs, 4, 1, 0, 0, model)
            noisy = r.accum.cpu().numpy()[:, :3] / spp
            den = r.denoised().cpu().numpy()[:, :3]
            row[f"rmse_noisy_{spp}"] = float(np.sqrt(np.mean((noisy - ref) ** 2)))
            row[f"rmse_denoised_{spp}"] = float(np.sqrt(np.mean((den - ref) ** 2)))
        emit({"rmse": row})
    if args.out:
        with open(args.out, "w") as f:
            for d in lines:
                f.write(json.dumps(d) + "\n")


if __name__ == "__main__":
    main()
