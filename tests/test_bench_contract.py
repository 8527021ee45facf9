"""CPU: the reference arm of bench.py (`--impl reference`) prints the contracted JSON line without touching a GPU.
GPU: `--dump-outputs` writes the same arrays on every run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_the_contracted_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0",
                          "--rows", "3000", "--cpu-seconds", "2"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["metric"] == "row_x_group_x_feature_scores_per_sec" and line["unit"] == "scores/s"
    assert line["higher_is_better"] is True and line["value"] > 0 and line["gpu_launches"] == 0
    assert line["config"]["workload"].startswith("C2:")
    cb = line["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == line["value"] and "rows" in cb["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "scores/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def _bench_dump(out_dir, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1",
                          "--rows", "20000", "--configs", "none", "--no-e2e", "--no-cpu", "--no-parity", "--dump-outputs", str(out_dir)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and [c["name"] for c in line["configs"]] == ["C2"]
    return line


@pytest.mark.gpu
def test_dump_outputs_are_the_same_on_every_run(tmp_path):
    # --dump-outputs: what the last timed step computed, seeded inputs, so that two runs (or two builds) compare array for array
    dirs = [tmp_path / "run0", tmp_path / "run1"]
    lines = [_bench_dump(d, 2) for d in dirs]
    one = _bench_dump(tmp_path / "one_step", 1)
    # --steps sets the number of timed steps: every step is the same sweep, so two steps launch twice the kernels of one
    assert lines[0]["gpu_launches"] == lines[1]["gpu_launches"] == 2 * one["gpu_launches"] > 0
    names = sorted(os.listdir(dirs[0]))
    assert names == sorted(os.listdir(dirs[1])) == ["C2_%s.npy" % n for n in ("assignments", "group_ids", "group_sizes", "scores", "suffstats")]
    assert sum(os.path.getsize(dirs[0] / n) for n in names) <= 64e6
    for n in names:
        a, b = np.load(dirs[0] / n), np.load(dirs[1] / n)
        assert a.dtype in (np.float32, np.float64) and a.size > 0, n
        assert np.array_equal(a, b), n
    assign = np.load(dirs[0] / "C2_assignments.npy")
    gids, sizes = np.load(dirs[0] / "C2_group_ids.npy"), np.load(dirs[0] / "C2_group_sizes.npy")
    assert assign.shape == (20000,) and sizes.sum() == 20000
    # one capture of one state: every group's size is the number of rows the assignments put in it
    assert set(np.unique(assign)) <= set(gids)
    assert np.array_equal(np.array([(assign == g).sum() for g in gids]), sizes)
    assert np.load(dirs[0] / "C2_scores.npy").shape[1] == 200
