"""The benchmark contract on the CPU side: the committed JSON lines of the round carry every key the driver reads, the
reference arm prints the GPU arm's config object, and a non-zero rank of the reference arm exits quietly."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
LINES = os.path.join(ROOT, "profiles", "r2_bench")
KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
        "dtype", "data", "config", "e2e", "gpu_launches", "clocks", "roofline"}


def _line(name):
    with open(os.path.join(LINES, name)) as f:
        return json.loads(f.read())


@pytest.mark.parametrize("name", ["bench_c1.json", "bench_c2.json", "bench_c3.json", "bench_c4.json", "bench_c5.json"])
def test_committed_bench_lines_carry_the_contract(name):
    d = _line(name)
    assert KEYS <= set(d), KEYS - set(d)
    assert d["metric"] == "frames_per_s" and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and d["dtype"] == "int16"
    assert d["value"] > 0 and d["gpu_launches"] > 0 and d["steps"] >= 1 and d["warmup"] >= 3
    frames = d["config"].get("job_frames") or d["config"]["frames_per_step_per_gpu"] * d["n_gpus"]   # c5: the whole job is a step
    assert abs(d["value"] - frames / d["ms_per_step"] * 1e3) <= 1e-6 * d["value"]
    e = d["e2e"]
    assert e["value"] > 0 and e["h2d_bytes_per_step"] > 0 and e["d2h_bytes_per_step"] > 0 and e["value"] != d["value"]
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert abs(r["achieved"] - r["algorithmic_bytes_per_run"] / (r["ms_per_run"] * 1e-3) / 1e9) <= 1e-9 * r["achieved"]
    assert abs(sum(r["groups_ms_per_run"].values()) - r["ms_per_run"]) <= 1e-9
    assert d["clocks"]["sm_mhz"] > 0 and not set(d["clocks"]["reasons"]) & {"hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown"}
    assert d["scaling"] == ("strong" if name == "bench_c5.json" else "weak")
    if name != "bench_c5.json":   # (the c5 line is taken with --no-cpu)
        c = d["cpu_baseline"]
        assert c["kind"] == "port" and c["cores"] >= 1 and c["value"] > 0 and c["parity_check"]["ok"] is True


def test_reference_arm_line_matches_the_gpu_arm():
    ref, gpu = _line("bench_c3_reference_arm.json"), _line("bench_c3.json")
    assert ref["impl"] == "reference" and ref["config"] == gpu["config"]
    for k in ("metric", "unit", "higher_is_better", "dtype", "scaling"):
        assert ref[k] == gpu[k], k
    assert ref["e2e"] == {"value": ref["value"], "unit": ref["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert ref["cpu_baseline"]["value"] == ref["value"] and ref["gpu_launches"] == 0


@pytest.mark.parametrize("config", ["c1", "c4"])
def test_dump_outputs_within_budget(tmp_path, config):
    """--dump-outputs with every frame at max_points (a stand-in for the pipeline whose values depend on the frame slot):
    float32 / float64 files only, at most 64 MB in all, the same frame sample on every run, counts.npy the counts handed
    in, and frameNNN_<key>.npy the values fetch(NNN) returned for <key>."""
    import re
    import numpy as np
    import bench

    class Pipe:
        def fetch(self, f):
            W, H, m = bench.W, bench.H, bench.MAX_POINTS
            i = np.arange(W * H, dtype=np.int64).reshape(H, W)
            xy = np.arange(2 * m).reshape(m, 2) * 0.25 + f
            return dict(left_rect=((i[..., None] * 3 + np.arange(3) + f) % 256).astype(np.uint8),
                        depth=(i % 977 + f).astype(np.float32) / 7, disp16=((i * 37 + f) % 65536 - 32768).astype(np.int16),
                        points_2d=xy if config == "c1" else xy.astype(np.float32),   # Simple: float64, Steger: float32
                        points_3d=np.arange(3 * m).reshape(m, 3) * 0.125 - f)

    bench.select_config(config)
    counts = (np.arange(bench.CFG["frames"]) * 7919 % 20001).astype(np.int32)
    listings = []
    for run in ("a", "b"):
        d = tmp_path / run
        bench.dump_outputs(str(d), Pipe(), counts)
        files = sorted(os.listdir(d))
        assert sum(os.path.getsize(d / f) for f in files) <= 64 * 10 ** 6
        assert np.array_equal(np.load(d / "counts.npy"), counts) and np.load(d / "counts.npy").dtype == np.float64
        slots = set()
        for f in files:
            if f == "counts.npy":
                continue
            m = re.fullmatch(r"frame(\d{3})_(\w+)\.npy", f)
            assert m, f
            slots.add(int(m.group(1)))
            got, want = np.load(d / f), Pipe().fetch(int(m.group(1)))[m.group(2)]
            assert got.dtype == (np.float64 if want.dtype == np.float64 else np.float32), f
            assert got.shape == want.shape and np.array_equal(got, want), f
        assert slots and len(files) == 1 + 5 * len(slots)
        listings.append(files)
    assert listings[0] == listings[1]


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT="29533")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "1"], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ""
