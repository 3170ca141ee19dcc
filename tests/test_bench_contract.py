"""bench.py's CPU arm (`--impl reference`) runs without a GPU: check that it prints ONE JSON line with the contract's keys.
(The GPU arm is exercised by the driver; its extra keys are listed here so that a rename shows up in review.)"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config"}
GPU_ARM_KEYS = BASE_KEYS | {"clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline"}


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--cpu-rows", "4000", "--trees", "4",
                          "--depth", "4", "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["unit"] == "records/s" and d["value"] > 0 and "workload" in d["config"]
    assert {"value", "unit", "cores", "kind", "sample"} <= set(d["cpu_baseline"]) and d["cpu_baseline"]["kind"] == "port"
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0 and d["e2e"]["value"] == d["value"]


def test_reference_arm_sets_its_thread_count_and_honours_warmup():
    # torchrun exports OMP_NUM_THREADS=1 to its workers: the CPU arm must not inherit it (SCALE_r01: the N>1 arms timed out)
    env = dict(os.environ, OMP_NUM_THREADS="1", RANK="0", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--workload", "cicids_script",
                          "--cpu-rows", "3000", "--trees", "3", "--depth", "3", "--steps", "1", "--warmup", "2"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][0])
    cores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else os.cpu_count()
    assert d["cpu_baseline"]["cores"] == cores and d["warmup"] == 2 and d["n_gpus"] == 2
    assert d["config"]["name"] == "cicids_script" and d["config"]["sample_rows"] == 3000 and d["config"]["classes"] == 14


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def _dump(tmp_path, tag, *args):
    out = tmp_path / tag
    run = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args, "--dump-outputs", str(out)],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert run.returncode == 0, run.stderr[-2000:]
    files = sorted(os.listdir(out))
    assert sum(os.path.getsize(out / f) for f in files) <= 64 << 20
    arrays = {f[:-4]: np.load(out / f) for f in files}
    assert all(v.dtype in (np.float32, np.float64) for v in arrays.values())
    return arrays


def _assert_same(a, b):
    assert sorted(a) == sorted(b)
    for k in a:
        assert np.array_equal(a[k], b[k]), k


def test_reference_arm_dumps_the_same_outputs_whatever_the_step_count(tmp_path):
    args = ["--impl", "reference", "--cpu-rows", "4000", "--trees", "4", "--depth", "4"]
    a = _dump(tmp_path, "a", *args, "--steps", "1", "--warmup", "0")
    b = _dump(tmp_path, "b", *args, "--steps", "2", "--warmup", "1")
    _assert_same(a, b)
    assert {"prediction", "macro_f1", "forest_nid", "forest_counts", "forest_mask"} <= set(a) and len(a["prediction"]) > 900


@pytest.mark.gpu
def test_gpu_arm_dumps_the_same_outputs_whatever_the_step_count(tmp_path):
    args = ["--rows", "30000", "--trees", "4", "--depth", "6", "--no-cpu-baseline"]
    a = _dump(tmp_path, "a", *args, "--steps", "1", "--warmup", "0")
    b = _dump(tmp_path, "b", *args, "--steps", "3", "--warmup", "2")
    _assert_same(a, b)
    assert np.array_equal(a["prediction"], a["e2e_prediction"]) and len(a["prediction"]) > 6000
    C = a["confusion"].shape[0]                                 # confusion[label, prediction] over the same test rows
    assert a["probability"].shape == a["rawPrediction"].shape == (len(a["prediction"]), C)
    assert np.array_equal(a["confusion"].sum(0), np.bincount(a["prediction"].astype(np.int64), minlength=C))


def test_gpu_arm_keys_are_emitted_by_bench_source():
    src = open(os.path.join(ROOT, "bench.py")).read()
    for k in GPU_ARM_KEYS | {"traffic", "frac", "peak", "achieved", "bound", "h2d_bytes_per_step", "d2h_bytes_per_step", "sm_mhz",
                             "dram_frac", "lsu_pct", "labels_equal", "forest_equal", "forest_hash"}:
        assert '"%s"' % k in src, k
