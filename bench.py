#!/usr/bin/env python
"""bench.py — benchmark of the path-tracing hot path (BASELINE.json metric: Mpaths/s and Mrays/s per scene).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload NAME] [--only]
                    [--dump-outputs DIR]

One "step" = one complete render of a workload (every sample of every pixel) through pt_render, or one pass of
the fixed ray batch through pt_trace_batch_device.

The JSON line's HEADLINE (metric / value / ms_per_step / roofline / e2e / cpu_baseline) is the north-star workload
`10_final_720p_8192` = BASELINE configs[0] exactly: taichi_pathtracer/10_final (RTIOW random-spheres scene, 486 spheres,
defocus blur) at the script's 1280x720, 8192 spp, depth 32.  The same line carries `workloads`: one entry per other
BASELINE config — `8_refract_1080p` (configs[1]), `yoimiya_1080p` (configs[2]), `zhongli_4k_4096` (configs[3]),
`intersect_10m` (configs[4]) — each with value / ms_per_step / roofline / e2e measured the same way (K timed steps).
`--only` measures just `--workload`.

--dump-outputs DIR writes what the last timed step of `--workload` computed, as the caller of that path receives it, to
DIR/<name>.npy: `accum.npy` (a render: the [H*W, 4] float32 accumulator, RGB sums over all samples + the count of
contributing paths) or `t.npy`, `prim.npy`, `uv.npy` (the ray batch: hit distance, primitive id as float64, barycentrics).
Inputs are seeded, so two builds can be compared output for output.  Past 64 MB the same seeded sample of rows is written
for every array, with the row numbers in `sample_rows.npy`.  N > 1: rank 0's arrays (for a render, the reduced image).

N > 1 (torchrun, one rank per GPU): STRONG scaling for every workload — the job is fixed, the scene is replicated, the
samples of every pixel (the rays of the batch) are split N ways, and the per-GPU accumulators are summed onto rank 0 by
NCCL reduces inside the timed region (the ray batch needs no collective).

--impl reference times the CPU oracle (the reference's algorithm restated in C + OpenMP, all host cores) on a bounded
sample of the same workload: the reference itself (Python + Taichi) cannot be installed here (DESIGN.md section 1).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (scene, W, H, spp of the whole job, depth)
    "10_final_720p_8192": ("10_final", 1280, 720, 8192, 32),    # BASELINE configs[0]: the script's own resolution/spp/depth
    "8_refract_1080p": ("8_refract", 1920, 1080, 256, 50),      # configs[1]
    "yoimiya_1080p": ("cache:yoimiya_ground_full", 1920, 1080, 512, 32),      # configs[2]
    "zhongli_4k_4096": ("cache:zhongli_full", 3840, 2160, 4096, 32),          # configs[3]
    "ganyu_4k_4096": ("cache:ganyu_full", 3840, 2160, 4096, 32),              # configs[3], the other model
    # reduced forms for quick A/B runs (not bench lines)
    "10_final_720p": ("10_final", 1280, 720, 256, 32),
    "9_dof_720p": ("9_dof", 1280, 720, 256, 32),
    "zhongli_4k": ("cache:zhongli_full", 3840, 2160, 64, 32),
}
# BASELINE configs[4]: synthetic 10M-triangle scene, 64Mi-ray intersection-only batch
INTERSECT = {"intersect_10m": (10_000_000, 64 * 2**20, 12345, 54321, 0.004),
             "intersect_1m": (1_000_000, 8 * 2**20, 12345, 54321, 0.0086)}
SPP_OVERRIDE = 0   # --spp: A/B runs at another sample count (e.g. the per-GPU share of a split frame); never a bench line
HEADLINE = "10_final_720p_8192"
OTHERS = ["8_refract_1080p", "yoimiya_1080p", "zhongli_4k_4096", "intersect_10m"]
KERNEL_OF = {"10_final_720p_8192": "k_paths_persist<V2>", "10_final_720p": "k_paths_persist<V2>", "8_refract_1080p": "k_paths_persist<V2>",
             "yoimiya_1080p": "k_paths_persist<LEGACY>", "zhongli_4k_4096": "k_paths_persist<LEGACY>", "zhongli_4k": "k_paths_persist<LEGACY>",
             "ganyu_4k_4096": "k_paths_persist<LEGACY>", "intersect_10m": "k_trace_persist<QNODES>"}
# algorithmic HBM bytes (SURVEY 8d): per ray segment / per path
B_PER_SEGMENT = 160  # extend 48 (read o|d 32, write hit 16) + shade 112 (read o|d 32 + throughput 16 + hit 16, write successor 48)
B_PER_PATH = 24      # fp32 RGB accumulate read-modify-write
L2_BYTES = 126e6
DUMP_BYTES = 63 * 10**6   # --dump-outputs: rows written in all; with the .npy headers the dump stays under 64 MB


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def kernel_source_hash():
    """Hash of the kernel sources the library is built from: profiles/ncu_counters.json is only quoted when it was
    captured from the same sources (tools/ncu_capture.sh stamps it)."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "learn_path_tracing_b200", "csrc")
    for fn in sorted(os.listdir(d)):
        if fn.endswith((".cu", ".cuh", ".h")) or fn == "Makefile":
            with open(os.path.join(d, fn), "rb") as f:
                h.update(fn.encode() + b"\0" + f.read())
    return h.hexdigest()[:16]


def ncu_counters(workload):
    """(counters of the dominant kernel captured by tools/ncu_capture.sh, or None, and where from / why not)."""
    p = os.path.join(ROOT, "profiles", "ncu_counters.json")
    if not os.path.exists(p):
        return None, "profiles/ncu_counters.json missing"
    with open(p) as f:
        d = json.load(f)
    if d.get("kernel_source_hash") != kernel_source_hash():
        return None, (f"profiles/ncu_counters.json is stale (captured from kernel sources {d.get('kernel_source_hash')}, "
                      f"this library is built from {kernel_source_hash()}): refused")
    return d.get("workloads", {}).get(workload), "profiles/ncu_counters.json"


class ClockSampler(threading.Thread):
    """Samples SM clocks / throttle reasons with NVML every 100 ms while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self.stop_flag = index, [], set(), None, False
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.ok = True
        except Exception:
            pass

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40,
                 "hw_power_brake_slowdown": 0x80, "sw_power_cap": 0x4}
        while not self.stop_flag:
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for k, bit in names.items():
                    if r & bit:
                        self.reasons.add(k)
            except Exception:
                pass
            time.sleep(0.1)

    def result(self):
        self.stop_flag = True
        if not self.ok or not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml_unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def workload_config(name):
    """The workload as both arms describe it (identical dict on the `ours` and the `reference` line)."""
    if name in INTERSECT:
        n_tri, n_rays, seed_t, seed_r, edge = INTERSECT[name]
        return {"workload": name, "triangles": n_tri, "rays": n_rays, "edge_scale": edge, "seeds": [seed_t, seed_r]}
    scene, W, H, spp, depth = WORKLOADS[name]
    spp = SPP_OVERRIDE or spp
    return {"workload": name, "scene": scene, "width": W, "height": H, "spp": spp, "max_depth": depth,
            "l2": "GPU arm: 252 MB fill between timed steps; CPU arm: not applicable"}


def build_workload(name):
    """-> (world, camera, W, H, spp, depth, shading model)"""
    import learn_path_tracing_b200 as L
    from learn_path_tracing_b200 import scenes
    scene, W, H, spp, depth = WORKLOADS[name]
    spp = SPP_OVERRIDE or spp
    if scene.startswith("cache:"):
        from learn_path_tracing_b200 import legacy, scene_cache
        path = os.path.join(ROOT, "scenes_cache", scene[6:] + ".npz")
        if not os.path.exists(path):
            raise FileNotFoundError(f"{path} missing (python tools/prepare_assets.py needs the reference checkout)")
        world = scene_cache.load_cache(path)
        cam = legacy.Camera((W, H))       # 15_module.py:1068-1072
        cam.set_fov(30)
        cam.set_position(legacy.Vec3f([0, 8, -30]))
        cam.look_at(legacy.Vec3f([0, 8, 0]))
        return world, cam, W, H, spp, depth, L.PT_SHADE_LEGACY
    world, cam = scenes.SCENES[scene]((W, H))
    return world, cam, W, H, spp, depth, L.PT_SHADE_V2


def oracle_scene(world, model):
    from oracle import ptoracle as O
    import learn_path_tracing_b200 as L
    return O.scene_from_legacy_world(world) if model == L.PT_SHADE_LEGACY else O.scene_from_world(world)


def cpu_baseline_run(world, cam, W, H, depth, target_seconds, threads=0, model=0):
    """Times the oracle (kind 'port': the reference's algorithm in C + OpenMP) on a bounded sample."""
    from oracle import ptoracle as O
    sc = oracle_scene(world, model)
    cs = cam.to_struct()
    t0 = time.perf_counter()
    O.render(sc, cs, W, H, 1, depth, model, seed=1, threads=threads)
    t1 = time.perf_counter() - t0
    spp = int(max(1, min(1024, target_seconds / max(t1, 1e-3))))
    t0 = time.perf_counter()
    _, _, st = O.render(sc, cs, W, H, spp, depth, model, seed=1, threads=threads)
    dt = time.perf_counter() - t0
    cores = O.num_threads() if threads <= 0 else threads
    return {"mpaths": st.paths / dt / 1e6, "mrays": st.segments / dt / 1e6, "seconds": dt, "spp": spp, "cores": cores}


def cpu_note(model):
    import learn_path_tracing_b200 as L
    return ("unpruned stack walk of the stored SAH tree, texture fetch per candidate" if model == L.PT_SHADE_LEGACY
            else "brute-force sphere loop per bounce")


# ---------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """The reference arm: the CPU restatement of the reference's algorithm on the host cores, rank 0 only."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    name = args.workload
    if name in INTERSECT:
        raise SystemExit("--impl reference: use a render workload (the intersect entry carries its own cpu_baseline)")
    world, cam, W, H, spp, depth, model = build_workload(name)
    per_step = 8.0
    vals = []
    for i in range(args.warmup + args.steps):
        r = cpu_baseline_run(world, cam, W, H, depth, per_step if i >= args.warmup else 1.0, model=model)
        if i >= args.warmup:
            vals.append(r)
    v = float(np.mean([r["mpaths"] for r in vals]))
    ms = float(np.mean([r["seconds"] for r in vals]) * 1e3)
    sample = (f"{name}: {W}x{H}, {vals[-1]['spp']} spp per step (of {spp}), depth {depth}; OpenMP C restatement of the "
              f"reference algorithm ({cpu_note(model)}); Taichi is not installable, rate on a bounded sample")
    line = {
        "impl": "reference", "metric": "Mpaths/s", "value": v, "unit": "Mpaths/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(name),
        "mrays_per_s": float(np.mean([r["mrays"] for r in vals])),
        "cpu_baseline": {"value": v, "unit": "Mpaths/s", "cores": vals[-1]["cores"], "kind": "port", "sample": sample},
        "e2e": {"value": v, "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
class Dist:
    def __init__(self):
        import torch
        self.torch = torch
        self.world_size = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the path tracer has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        if self.world_size > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
        self.flush = torch.empty(int(2 * L2_BYTES) // 4, dtype=torch.float32, device="cuda")

    def barrier(self):
        if self.world_size > 1:
            import torch.distributed as dist
            dist.barrier()

    def _all(self, x, op):
        if self.world_size == 1:
            return float(x)
        import torch.distributed as dist
        t = self.torch.tensor([float(x)], dtype=self.torch.float64, device="cuda")
        dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
        return float(t.item())

    def max_f(self, x):
        return self._all(x, "MAX")

    def sum_f(self, x):
        return self._all(x, "SUM")

    def close(self):
        if self.world_size > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()


def dump_outputs(directory, rows, arrays):
    """Saves each device array of `arrays` (all with `rows` rows) as <directory>/<name>.npy; over DUMP_BYTES, the rows of
    one seeded sample (row numbers in sample_rows.npy)."""
    import torch
    os.makedirs(directory, exist_ok=True)
    per_row = sum(a.element_size() * (a.numel() // rows) for a in arrays.values())
    if per_row * rows > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(rows, DUMP_BYTES // (per_row + 8), replace=False))
        np.save(os.path.join(directory, "sample_rows.npy"), keep.astype(np.float64))
        idx = torch.from_numpy(keep).to(next(iter(arrays.values())).device)
        arrays = {k: a[idx] for k, a in arrays.items()}
    for k, a in arrays.items():
        np.save(os.path.join(directory, k + ".npy"), a.cpu().numpy())


def issue_entry(nc):
    if not nc:
        return None
    ia, lanes = nc.get("issue_active_pct"), nc.get("lanes_per_instruction")
    return {"bound": "issue", "issue_active_pct": ia, "lanes_per_instruction": lanes,
            "useful_lane_issue_frac": (ia / 100.0) * (lanes / 32.0) if ia and lanes else None,
            "l1tex_data_pipe_pct": nc.get("l1tex_data_pipe_pct"), "long_scoreboard_warps_per_issue": nc.get("long_scoreboard"),
            "source": nc.get("summary"), "captured_from_sources": kernel_source_hash()}


def measure_render(D, name, steps, warmup, args, cpu_seconds=0.0, dump=None):
    """One render workload on D.world_size GPUs (strong scaling: the job's spp split over the ranks)."""
    import learn_path_tracing_b200 as L
    from learn_path_tracing_b200.multigpu import render_split_reduce, split_samples
    torch = D.torch
    world, cam, W, H, spp, depth, model = build_workload(name)
    ws, rank = D.world_size, D.rank
    ctx = L.default_context()
    scene = world.device_scene(ctx)
    cs = cam.to_struct()
    r = L.Renderer(W, H, ctx)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kw = dict(mode=args.mode, shade_min=args.shade_min, serve_min=args.serve_min)
    bands = args.bands if ws > 1 else 1

    def step():
        r.clear()
        render_split_reduce(r, scene, cs, spp, depth, model, 1, bands=bands, **kw)

    for _ in range(max(warmup, 3)):
        step()
    sampler = ClockSampler(D.local_rank)
    sampler.start()
    times = []
    for _ in range(steps):
        D.flush.fill_(1.0)  # evict L2 between timed iterations
        torch.cuda.synchronize()
        D.barrier()
        ev0.record()
        step()
        ev1.record()
        torch.cuda.synchronize()
        times.append(ev0.elapsed_time(ev1))
    clocks = sampler.result()
    if dump and rank == 0:
        dump_outputs(dump, W * H, {"accum": r.accum})
    t_local = float(sum(times))
    t_max = D.max_f(t_local)
    my_off, my_spp = split_samples(spp, ws, rank)
    # kernel-only time of this rank's share (the event pair around the launch inside pt_render) and the traversal
    # counters, from two extra untimed renders
    r.clear()
    stc = r.render(scene, cs, my_spp, depth, model, seed=1, spp_offset=my_off, flags=L.PT_FLAG_COUNTERS, **kw)
    r.clear()
    stt = r.render(scene, cs, my_spp, depth, model, seed=1, spp_offset=my_off, flags=L.PT_FLAG_TIMING, **kw)
    seg_rank = float(stt.segments)
    seg_total = D.sum_f(seg_rank)
    paths_total = float(W) * H * spp

    # ---- end to end through the public API with host buffers: scene upload + build + render (+ reduce) + host image
    legacy_scene = model == L.PT_SHADE_LEGACY
    if legacy_scene:
        h2d = sum(m["positions"].nbytes + m["normals"].nbytes + m["texture_coords"].nbytes + m["indices"].nbytes
                  for m in world.meshes) + world._atlas[0].nbytes + (world._env[0].nbytes if world._env else 0) + 128
    else:
        cr, mats = world.arrays()
        h2d = cr.nbytes + mats.nbytes + 64 + 64
    d2h = W * H * 3 * 4
    e_times, img = [], None
    for i in range(2 + min(max(steps, 3), 5)):
        world._scene = None  # force re-upload + rebuild: the scene starts on the host every step
        torch.cuda.synchronize()
        D.barrier()
        t0 = time.perf_counter()
        img = L.render_distributed(world, cam, spp=spp, propagate_limit=depth, seed=1, ctx=ctx, bands=bands)
        dt = time.perf_counter() - t0
        if i >= 2:  # two untimed calls: pinned-host and device caching allocators warm up
            e_times.append(dt)
    if rank == 0:
        assert img.shape == (W, H, 3) and np.isfinite(img).all()
    e_t = D.max_f(float(np.median(e_times)))   # median of 3-5 timed calls shrugs off a host hiccup
    e2e = {"value": paths_total / e_t / 1e6, "unit": "Mpaths/s", "h2d_bytes_per_step": int(h2d * ws), "d2h_bytes_per_step": int(d2h),
           "ms": e_t * 1e3, "through": "learn_path_tracing_b200.render_distributed(world, camera): host scene in, host image out"}

    peak, peak_kind = measured_peaks()
    paths_rank = float(W) * H * my_spp
    ms_kernel = float(stt.ms_shade)  # events around the one k_paths_persist launch of this rank's share
    bytes_launch = B_PER_SEGMENT * seg_rank + B_PER_PATH * paths_rank
    achieved = bytes_launch / (ms_kernel * 1e-3) / 1e9
    nodes_seg = stc.nodes_visited / max(stc.segments, 1)
    prims_seg = stc.prims_tested / max(stc.segments, 1)
    flops_seg = nodes_seg * 36.0 + prims_seg * (45.0 if legacy_scene else 17.0) + 280.0
    try:
        fp32_peak = ctx.measure_fp32_peak()
    except Exception:
        fp32_peak = None
    fp32_achieved = seg_rank * flops_seg / (ms_kernel * 1e-3) / 1e12
    nc, nc_src = ncu_counters(name)
    frac = achieved / peak
    roof = {"bound": "hbm", "kernel": KERNEL_OF.get(name, "k_paths_persist"), "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": frac, "traffic": nc.get("dram_bytes_per_launch") if nc else None, "traffic_source": nc_src,
            "traffic_captured_as": nc.get("captured_as") if nc else None,
            "peak_kind": peak_kind, "avg_launch_ms": ms_kernel, "algorithmic_bytes_per_launch": bytes_launch,
            "algorithmic_bytes": "SURVEY 8d: 160 B per ray segment + 24 B per path = what a split wavefront moves through HBM. "
                                 "NOMINAL for this kernel: a path lives in registers from its camera ray to its last segment, so the "
                                 "measured DRAM traffic (`traffic`) is a small fraction of this figure and HBM is not what limits it",
            "limiter": "instruction issue at partially filled warps + L1/L2 latency (roofline_issue, roofline_fp32)"}
    if frac > 1.0:
        roof["note"] = "frac > 1: the SURVEY 8d accounting does not describe this kernel (it never writes path state to HBM)"
    entry = {
        "metric": "Mpaths/s", "value": paths_total * steps / (t_max * 1e-3) / 1e6, "unit": "Mpaths/s",
        "ms_per_step": t_max / steps, "steps": steps, "warmup": max(warmup, 3),
        "mrays_per_s": seg_total * steps / (t_max * 1e-3) / 1e6,
        "segments_per_path": seg_total / paths_total,
        "config": workload_config(name),
        "parallelism": f"samples split x{ws} (strong), scene replicated" + ((f", one NCCL reduce (rgb) behind the render on the same stream" if bands == 1 else f", NCCL reduce in {bands} row bands overlapped with rendering") if ws > 1 else ""),
        "mode": int(stt.reserved[0]),
        "e2e": e2e, "gpu_launches": steps * bands, "clocks": clocks,
        "roofline": roof, "roofline_issue": issue_entry(nc),
        "roofline_fp32": {"bound": "fp32", "achieved": fp32_achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                          "frac": (fp32_achieved / fp32_peak) if fp32_peak else None, "flops_per_segment": flops_seg,
                          "nodes_per_segment": nodes_seg, "prims_per_segment": prims_seg,
                          "accounting": "36 flop per BVH2 node visit + 17 per sphere / 45 per triangle test + 280 shading (SURVEY 8d)"},
        "kernel_ms_rank0": ms_kernel, "step_ms_rank0": t_local / steps, "cpu_baseline": None,
    }
    if cpu_seconds > 0 and ws == 1:
        cpu = cpu_baseline_run(world, cam, W, H, depth, cpu_seconds, model=model)
        entry["cpu_baseline"] = {"value": cpu["mpaths"], "unit": "Mpaths/s", "cores": cpu["cores"], "kind": "port",
                                 "sample": f"{W}x{H}, {cpu['spp']} spp (of {spp}), depth {depth}, {cpu['seconds']:.1f} s of the OpenMP C "
                                           f"oracle (reference algorithm: {cpu_note(model)})",
                                 "mrays_per_s": cpu["mrays"]}
    world._scene = None
    del r, scene
    return entry


def measure_intersect(D, name, steps, warmup, args, dump=None):
    """BASELINE configs[4]: fixed ray batch against an LBVH over random triangles, intersection only.  Rays and
    triangles come from counter-based device generators (bit-identical to the oracle's); N > 1 shards the batch by ray
    ranges, no collective."""
    import learn_path_tracing_b200 as L
    from oracle import ptoracle as O
    torch = D.torch
    n_tri, n_rays, seed_t, seed_r, edge = INTERSECT[name]
    ws, rank = D.world_size, D.rank
    ctx = L.default_context()
    sc = L.Scene(ctx)
    t0 = time.perf_counter()
    sc.set_random_triangles(n_tri, seed_t, edge)
    sc.build()
    build_s = time.perf_counter() - t0
    n_local = n_rays // ws
    rays = torch.empty((2 * n_rays, 4), dtype=torch.float32, device="cuda")
    ctx.random_rays_device(rays.data_ptr(), n_rays, seed_r)
    my = rays[2 * rank * n_local: 2 * (rank + 1) * n_local]
    hits = torch.empty((n_local, 4), dtype=torch.float32, device="cuda")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(max(warmup, 3)):
        ctx.trace_batch_device(sc, my.data_ptr(), n_local, hits.data_ptr(), args.trace_flags)
    sampler = ClockSampler(D.local_rank)
    sampler.start()
    times = []
    for _ in range(steps):
        D.flush.fill_(1.0)
        torch.cuda.synchronize()
        D.barrier()
        ev0.record()
        ctx.trace_batch_device(sc, my.data_ptr(), n_local, hits.data_ptr(), args.trace_flags)
        ev1.record()
        torch.cuda.synchronize()
        times.append(ev0.elapsed_time(ev1))
    clocks = sampler.result()
    if dump and rank == 0:
        dump_outputs(dump, n_local, {"t": hits[:, 0], "prim": hits.view(torch.int32)[:, 1].double(), "uv": hits[:, 2:4]})
    t_local = float(sum(times))
    t_max = D.max_f(t_local)
    st = ctx.trace_batch_device(sc, my.data_ptr(), n_local, hits.data_ptr(), L.PT_FLAG_COUNTERS | args.trace_flags)
    st_plain = ctx.trace_batch_device(sc, my.data_ptr(), n_local, hits.data_ptr(), args.trace_flags)  # sort / traversal split
    # e2e: host ray buffer in, host ids/t out (pt_trace_batch), on a bounded slice
    n_e = min(n_local, 16 * 2**20)
    rays_h = my[:2 * n_e].cpu().numpy().reshape(n_e, 8)
    ids_h, t_h = np.zeros(n_e, np.int32), np.zeros(n_e, np.float32)   # the caller's result arrays, reused every call
    te = []
    for i in range(4):
        t0 = time.perf_counter()
        ctx.trace_batch(sc, rays_h, out=(ids_h, t_h))
        if i:  # the first call allocates the pinned / device staging of the context
            te.append(time.perf_counter() - t0)
    e_t = D.max_f(min(te))
    peak, peak_kind = measured_peaks()
    nodes_per_ray = st.nodes_visited / n_local
    tris_per_ray = st.prims_tested / n_local
    bytes_per_ray = 32 + 8 + 64 * nodes_per_ray + 48 * tris_per_ray
    ms_kernel = float(st_plain.ms_extend)
    achieved = bytes_per_ray * n_local / (ms_kernel * 1e-3) / 1e9
    nc, nc_src = ncu_counters(name)
    roof = {"bound": "hbm", "kernel": KERNEL_OF.get(name, "k_trace_persist"), "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "traffic": nc.get("dram_bytes_per_launch") if nc else None, "traffic_source": nc_src,
            "traffic_captured_as": nc.get("captured_as") if nc else None,
            "peak_kind": peak_kind, "avg_launch_ms": ms_kernel,
            "step_ms": {"ray_sort": st_plain.ms_other, "traversal": st_plain.ms_extend, "step": t_local / steps},
            "algorithmic_bytes_per_launch": bytes_per_ray * n_local,
            "algorithmic_bytes": f"SURVEY 8d: 32 + 8 + 64*{nodes_per_ray:.1f} nodes + 48*{tris_per_ray:.2f} triangles = {bytes_per_ray:.0f} B/ray "
                                 "(counts from a counter-instrumented run). NOMINAL: the kernel reads 32-byte quantised nodes and the ray "
                                 "sort turns most fetches into L1/L2 hits, so the measured DRAM traffic (`traffic`) is far lower",
            "compulsory_40B_per_ray": {"achieved": 40.0 * n_local / (ms_kernel * 1e-3) / 1e9},
            "limiter": "L1 data pipe + L2 latency on dependent node fetches (roofline_issue)"}
    if nc and nc.get("dram_bytes_per_launch") and ws == 1:
        dram = nc["dram_bytes_per_launch"] / (ms_kernel * 1e-3) / 1e9
        roof["measured_dram"] = {"achieved": dram, "frac": dram / peak, "unit": "GB/s",
                                 "note": "ncu dram__bytes of the captured launch over this run's kernel time"}
    if roof["frac"] > 1.0:
        roof["note"] = "frac > 1: the SURVEY 8d accounting does not describe this kernel (most node fetches never reach HBM)"
    entry = {
        "metric": "Mrays/s", "value": n_local * ws * steps / (t_max * 1e-3) / 1e6, "unit": "Mrays/s",
        "ms_per_step": t_max / steps, "steps": steps, "warmup": max(warmup, 3),
        "config": workload_config(name), "parallelism": f"ray ranges x{ws} (strong), no collective", "lbvh_build_s": build_s,
        "hit_fraction": float((ids_h >= 0).mean()),
        "e2e": {"value": n_e * ws / e_t / 1e6, "unit": "Mrays/s", "h2d_bytes_per_step": int(n_e * 32 * ws),
                "d2h_bytes_per_step": int(n_e * 8 * ws), "through": f"Context.trace_batch (pt_trace_batch): {n_e} host rays in, host ids / t out"},
        "gpu_launches": steps * 4, "clocks": clocks, "roofline": roof, "roofline_issue": issue_entry(nc), "cpu_baseline": None,
    }
    if rank == 0 and ws == 1 and not args.no_cpu:
        # CPU baseline: the oracle walking the SAME LBVH with the reference triangle test, bounded ray sample
        n_c = 2**18
        nodes, _ = sc.bvh_download()
        tris = O.random_triangles(n_tri, seed_t, edge)
        t0 = time.perf_counter()
        oid, ot, _ = O.trace_bvh2(nodes, tris, rays_h[:n_c])
        cpu_s = time.perf_counter() - t0
        entry["ids_equal_to_oracle"] = float((ids_h[:n_c] == oid).mean())
        entry["cpu_baseline"] = {"value": n_c / cpu_s / 1e6, "unit": "Mrays/s", "cores": O.num_threads(), "kind": "port",
                                 "sample": f"{n_c} rays of the same batch, oracle walking the same LBVH with the reference triangle test, {cpu_s:.1f} s"}
    sc.close()
    del rays, hits, my
    torch.cuda.empty_cache()
    return entry


def measure(D, name, steps, warmup, args, cpu_seconds=0.0, dump=None):
    if name in INTERSECT:
        return measure_intersect(D, name, steps, warmup, args, dump)
    return measure_render(D, name, steps, warmup, args, cpu_seconds, dump)


def merge_clocks(a, b):
    if not b or b.get("sm_mhz") is None:
        return a
    if not a or a.get("sm_mhz") is None:
        return b
    return {"sm_mhz": min(a["sm_mhz"], b["sm_mhz"]), "sm_max_mhz": a["sm_max_mhz"],
            "reasons": sorted(set(a["reasons"]) | set(b["reasons"]))}


def run_ours(args):
    D = Dist()
    head = measure(D, args.workload, args.steps, args.warmup, args, cpu_seconds=0.0 if args.no_cpu else 12.0,
                   dump=args.dump_outputs)
    others = {}
    if not args.only:
        for name in OTHERS:
            if name == args.workload:
                continue
            try:
                others[name] = measure(D, name, args.steps, args.warmup, args)
            except FileNotFoundError as e:  # scene caches are derived from the reference checkout (tools/prepare_assets.py)
                others[name] = {"unavailable": str(e)}
    if D.rank == 0:
        clocks = head["clocks"]
        for e in others.values():
            clocks = merge_clocks(clocks, e.get("clocks"))
        line = {
            "metric": head["metric"], "value": head["value"], "unit": head["unit"], "n_gpus": D.world_size,
            "steps": head["steps"], "warmup": head["warmup"], "ms_per_step": head["ms_per_step"],
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": head["config"],
        }
        for k, v in head.items():
            if k not in line and k != "clocks":
                line[k] = v
        line["clocks"] = clocks  # lowest median SM clock and the union of throttle reasons over all timed regions
        line["gpu_launches"] = int(head["gpu_launches"] + sum(e.get("gpu_launches", 0) for e in others.values()))
        line["workloads"] = others
        line["library"] = {"kernel_source_hash": kernel_source_hash()}
        print(json.dumps(line), flush=True)
    D.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=HEADLINE, choices=sorted(WORKLOADS) + sorted(INTERSECT))
    ap.add_argument("--only", action="store_true", help="measure --workload alone (no `workloads` entries)")
    ap.add_argument("--mode", type=int, default=0, help="render mode: 0 auto (= 3 persistent), 1 split kernels, 2 K-step fused, 3 persistent")
    ap.add_argument("--bands", type=int, default=1, help="N > 1: row bands per frame, the reduce of a band overlapping the rendering of the next "
                    "(measured on 2 B200s: 1 band 34.9 / 4 bands 33.6 / 8 bands 31.5 Gpaths/s on 8_refract, 9.6 / 8.2 / 7.3 on Yoimiya: every band "
                    "pays the ramp-up and tail of its own persistent launch, the reduce it hides is ~0.1 ms; hence 1)")
    ap.add_argument("--shade-min", type=int, default=0, help="persistent mode: waiting lanes that trigger shading (0 = default)")
    ap.add_argument("--serve-min", type=int, default=0, help="persistent mode: waiting lanes that trigger a service (0 = default)")
    ap.add_argument("--trace-flags", type=int, default=0, help="intersect workloads: PT_FLAG_* for pt_trace_batch_device")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline leg (profiling runs)")
    ap.add_argument("--spp", type=int, default=0, help="A/B runs only: override the workload's samples per pixel (config.spp shows it)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of --workload computed to DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    global SPP_OVERRIDE
    SPP_OVERRIDE = max(0, args.spp)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
