"""bench.py's contract on the CPU: the reference arm prints the driver's JSON line (rank 0 only under torchrun), both arms
describe a workload with the SAME config dict, and ncu counters captured from other kernel sources are refused."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import bench  # noqa: E402

KEYS = {"impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
        "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"}


def _run(env_extra, *args):
    env = dict(os.environ, **env_extra)
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, env=env, timeout=600)


def test_reference_arm_prints_the_contract_line():
    p = _run({}, "--impl", "reference", "--workload", "9_dof_720p", "--steps", "1", "--warmup", "0", "--gpus", "1")
    assert p.returncode == 0, p.stderr[-2000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    assert KEYS <= set(line) and line["impl"] == "reference" and line["metric"] == "Mpaths/s" and line["value"] > 0
    assert line["config"] == bench.workload_config("9_dof_720p")          # what the `ours` arm prints for the same workload
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": "Mpaths/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["higher_is_better"] is True and line["vs_baseline"] is None and line["scaling"] == "strong"


def test_reference_arm_other_ranks_exit_silently():
    p = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0")
    assert p.returncode == 0 and p.stdout.strip() == ""


def test_default_headline_is_configs0_and_every_config_is_a_workload():
    assert bench.HEADLINE == "10_final_720p_8192" and bench.WORKLOADS[bench.HEADLINE] == ("10_final", 1280, 720, 8192, 32)
    assert bench.OTHERS == ["8_refract_1080p", "yoimiya_1080p", "zhongli_4k_4096", "intersect_10m"]
    assert bench.WORKLOADS["8_refract_1080p"][1:] == (1920, 1080, 256, 50) and bench.WORKLOADS["yoimiya_1080p"][1:] == (1920, 1080, 512, 32)
    assert bench.WORKLOADS["zhongli_4k_4096"][1:] == (3840, 2160, 4096, 32) and bench.INTERSECT["intersect_10m"][:2] == (10_000_000, 64 * 2**20)


def test_stale_ncu_counters_are_refused(tmp_path, monkeypatch):
    prof = tmp_path / "profiles"
    prof.mkdir()
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    monkeypatch.setattr(bench, "kernel_source_hash", lambda: "aaaa")
    assert bench.ncu_counters("yoimiya_1080p")[0] is None                  # no file
    (prof / "ncu_counters.json").write_text(json.dumps({"kernel_source_hash": "bbbb", "workloads": {"yoimiya_1080p": {"issue_active_pct": 70}}}))
    nc, why = bench.ncu_counters("yoimiya_1080p")
    assert nc is None and "stale" in why
    (prof / "ncu_counters.json").write_text(json.dumps({"kernel_source_hash": "aaaa", "workloads": {"yoimiya_1080p": {"issue_active_pct": 70}}}))
    assert bench.ncu_counters("yoimiya_1080p")[0] == {"issue_active_pct": 70}


import numpy as np  # noqa: E402
import pytest  # noqa: E402


def test_dump_outputs_writes_every_array_or_one_seeded_sample_of_rows(tmp_path, monkeypatch):
    import torch
    arrays = {"a": torch.arange(4000, dtype=torch.float32).reshape(1000, 4), "p": torch.arange(1000, dtype=torch.float64)}
    bench.dump_outputs(str(tmp_path / "all"), 1000, arrays)
    assert sorted(os.listdir(tmp_path / "all")) == ["a.npy", "p.npy"]
    assert np.array_equal(np.load(tmp_path / "all" / "a.npy"), arrays["a"].numpy())
    monkeypatch.setattr(bench, "DUMP_BYTES", 100 * (16 + 8 + 8))
    for d in ("one", "two"):
        bench.dump_outputs(str(tmp_path / d), 1000, arrays)
    rows = np.load(tmp_path / "one" / "sample_rows.npy")
    assert len(rows) == 100 and np.all(np.diff(rows) > 0) and np.array_equal(rows, np.load(tmp_path / "two" / "sample_rows.npy"))
    a, p = np.load(tmp_path / "one" / "a.npy"), np.load(tmp_path / "one" / "p.npy")
    assert a.dtype == np.float32 and p.dtype == np.float64
    assert np.array_equal(a, arrays["a"].numpy()[rows.astype(np.int64)]) and np.array_equal(p, rows)
    assert sum(os.path.getsize(tmp_path / "one" / f) for f in os.listdir(tmp_path / "one")) <= 100 * 32 + 3 * 128


def test_steps_below_one_are_refused():
    p = _run({}, "--impl", "reference", "--steps", "0")
    assert p.returncode != 0 and "--steps" in p.stderr


@pytest.mark.gpu
def test_ours_arm_prints_the_contract_line_on_the_gpu(tmp_path):
    """`bench.py --workload X --only` on the GPU: every key the driver reads is there, the roofline block carries the
    achieved / peak / frac / traffic fields, e2e counts host<->device bytes, clocks were sampled during the timed region;
    --dump-outputs writes the accumulator of the last timed step."""
    p = _run({}, "--workload", "9_dof_720p", "--only", "--steps", "2", "--warmup", "3", "--no-cpu", "--dump-outputs", str(tmp_path))
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout.strip().splitlines()[-1])
    need = (KEYS - {"impl"}) | {"clocks", "roofline", "roofline_fp32", "mrays_per_s", "workloads", "library"}
    assert need <= set(line), need - set(line)
    assert line["n_gpus"] == 1 and line["steps"] == 2 and line["warmup"] == 3 and line["scaling"] == "strong"
    assert line["config"] == bench.workload_config("9_dof_720p") and line["workloads"] == {}
    r = line["roofline"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic", "kernel", "avg_launch_ms"} <= set(r) and r["bound"] == "hbm"
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["unit"] == "GB/s"
    e = line["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] == 1280 * 720 * 3 * 4
    assert e["value"] <= 1.05 * line["value"]            # end to end cannot beat the device-resident rate
    assert line["gpu_launches"] == 2 and line["value"] > 1000 and line["clocks"]["sm_max_mhz"]
    assert line["library"]["kernel_source_hash"] == bench.kernel_source_hash()
    acc = np.load(tmp_path / "accum.npy")
    assert sorted(os.listdir(tmp_path)) == ["accum.npy"] and acc.dtype == np.float32 and acc.shape == (1280 * 720, 4)
    assert np.isfinite(acc).all() and acc[:, 3].max() <= 256 and acc[:, :3].mean() > 0   # 256 spp: one whole render
