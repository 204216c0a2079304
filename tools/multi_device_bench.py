#!/usr/bin/env python
"""Strong scaling of the single-process multi-GPU path (MultiRenderer / pt_multi_render), one JSON line per
(workload, N), N in {1, 2, 4, 8} capped at the visible device count.

    python tools/multi_device_bench.py [--steps K] [--warmup W] [--repeats R] [--workloads a,b] [--torchrun]

Workloads come from bench.build_workload: 10_final_720p_8192 and 8_refract_1080p always, yoimiya_1080p and
zhongli_4k_4096 when scenes_cache/ holds them ("not available" otherwise).  A step is one whole frame: clear the root's
accumulator, pt_multi_render over devices 0 .. N-1, timed with CUDA events on the root stream after a warm-up and an L2
flush on every device, as bench.py times its steps.  Every line carries
  value          Mpaths/s (median over --repeats runs of K steps; `runs` lists them all)
  scaling        value / value at N = 1
  max_member_ms  the slowest member's render (PtStats.ms_total, one extra frame with stats): reduce + chaining is
                 ms_per_step - max_member_ms
  gpu            card name and power limit (nvidia-smi, read only)
--torchrun also runs `torchrun --nproc-per-node N bench.py --gpus N --workload X --only` for the same workloads and N
and prints its result line under {"torchrun": ...}, so that both multi-GPU paths are measured on the same box.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402

ALWAYS = ["10_final_720p_8192", "8_refract_1080p"]
IF_CACHED = ["yoimiya_1080p", "zhongli_4k_4096"]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                             text=True, timeout=60).stdout.strip().splitlines()
        return [dict(zip(("name", "power_limit"), (x.strip() for x in line.split(",")))) for line in out]
    except Exception as e:  # the number is still a number; say why the card is not named
        return [{"error": str(e)}]


def measure(name, n, steps, warmup, repeats):
    import torch
    import learn_path_tracing_b200 as L
    world, cam, W, H, spp, depth, model = bench.build_workload(name)
    ctx = L.default_context()
    r = L.MultiRenderer(W, H, list(range(n)), ctx)
    scene = world.device_scene(ctx)
    cs = cam.to_struct()
    flush = [torch.empty(int(2 * bench.L2_BYTES) // 4, dtype=torch.float32, device=f"cuda:{d}") for d in range(n)]
    stream = torch.cuda.current_stream(r.accum.device)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def step():
        r.clear()
        r.render(scene, cs, spp, depth, model, seed=1, spp_offset=0, want_stats=False)

    for _ in range(max(warmup, 1)):
        step()
    runs, per_step = [], []
    for _ in range(repeats):
        t = 0.0
        for _ in range(steps):
            for f in flush:
                f.fill_(1.0)
            for d in range(n):
                torch.cuda.synchronize(d)
            ev0.record(stream)
            step()
            ev1.record(stream)
            ev1.synchronize()
            t += ev0.elapsed_time(ev1)
        per_step.append(t / steps)
        runs.append(float(W) * H * spp * steps / (t * 1e-3) / 1e6)
    r.clear()
    r.render(scene, cs, spp, depth, model, seed=1, spp_offset=0, want_stats=True)
    member_ms = [float(s.ms_total) for s in r.member_stats]
    out = {"value": statistics.median(runs), "runs": runs, "ms_per_step": statistics.median(per_step),
           "max_member_ms": max(member_ms), "member_ms": member_ms}
    del r, scene
    world._scene = None
    torch.cuda.empty_cache()
    return out


def torchrun_line(name, n, steps, warmup):
    cmd = [sys.executable, "-m", "torch.distributed.run", "--standalone", "--nproc-per-node", str(n),
           os.path.join(ROOT, "bench.py"), "--gpus", str(n), "--workload", name, "--only", "--no-cpu",
           "--steps", str(steps), "--warmup", str(warmup)]
    p = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT)
    lines = [x for x in p.stdout.splitlines() if x.startswith("{")]
    if p.returncode != 0 or not lines:
        return {"error": f"rc {p.returncode}", "stderr_tail": p.stderr[-2000:]}
    d = json.loads(lines[-1])
    return {"value": d["value"], "ms_per_step": d["ms_per_step"], "n_gpus": d["n_gpus"], "parallelism": d.get("parallelism")}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--workloads", default=",".join(ALWAYS + IF_CACHED))
    ap.add_argument("--torchrun", action="store_true")
    args = ap.parse_args()
    import torch
    n_dev = torch.cuda.device_count()
    if n_dev < 1:
        raise SystemExit("no CUDA device visible: this measurement needs the GPUs it measures")
    ns = [n for n in (1, 2, 4, 8) if n <= n_dev]
    gpu = gpu_info()
    unavailable = {}
    for name in args.workloads.split(","):
        base = None
        for n in ns:
            line = {"tool": "multi_device_bench", "workload": name, "n_gpus": n, "visible_gpus": n_dev, "gpu": gpu,
                    "path": "MultiRenderer (pt_multi_render: one process, peer-memory reduce)", "unit": "Mpaths/s",
                    "steps": args.steps, "warmup": args.warmup, "repeats": args.repeats}
            try:
                m = measure(name, n, args.steps, args.warmup, args.repeats)
            except FileNotFoundError as e:
                line["unavailable"] = unavailable[name] = "not available: " + str(e).replace(ROOT + os.sep, "")
                print(json.dumps(line), flush=True)
                break
            base = m["value"] if n == 1 else base
            line.update(m)
            line["scaling"] = m["value"] / base if base else None
            line["reduce_and_chaining_ms"] = m["ms_per_step"] - m["max_member_ms"]
            print(json.dumps(line), flush=True)
    if args.torchrun:
        for name in args.workloads.split(","):
            if name in unavailable:
                print(json.dumps({"torchrun": {"unavailable": unavailable[name]}, "workload": name, "gpu": gpu}), flush=True)
                continue
            base = None
            for n in ns:
                t = torchrun_line(name, n, args.steps, args.warmup)
                if "value" in t:
                    base = t["value"] if n == 1 else base
                    t["scaling"] = t["value"] / base if base else None
                print(json.dumps({"torchrun": t, "workload": name, "n_gpus": n, "gpu": gpu}), flush=True)


if __name__ == "__main__":
    main()
