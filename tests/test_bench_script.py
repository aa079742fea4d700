"""bench.py's own code paths (argument handling, world generation, stepping through the public Pipeline API, byte accounting, parity record, the cpu_baseline
leg with the reference binary, the JSON line as the last line of stdout, a quiet stderr) on the CPU stand-in: tests/bench_dry_run.py swaps the library and
pretends a device is there. The numbers mean nothing; a typo in the script would otherwise only show on the GPU box at the end of a round."""
import json, os, subprocess, sys
import pytest
from arriba_b200 import _build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bench_script_runs_on_the_stand_in(hostsim_lib, tmp_path):
    env = dict(os.environ, ARB_BENCH_DIR=str(tmp_path), PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "bench_dry_run.py"), "--workload", "tiny_20k", "--steps", "2", "--warmup", "1"], env=env, capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])          # the JSON line is the LAST line of stdout
    assert len(r.stderr.splitlines()) < 40                         # the library's per-row warnings went to its log file
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "clocks", "e2e", "gpu_launches", "roofline", "cpu_baseline", "parity"):
        assert key in line, key
    assert line["steps"] == 2 and line["warmup"] == 1 and line["n_gpus"] == 1 and line["unit"] == "reads/s" and line["gpu_launches"] > 0
    e = line["e2e"]
    assert e["h2d_bytes_per_step"] == sum(e["h2d_bytes_are"].values()) > 0 and e["d2h_bytes_per_step"] == sum(e["d2h_bytes_are"].values()) > 0
    assert abs(line["value"] - line["fragments_per_step"] / (line["ms_per_step"] * 1e-3)) < 1e-6 * line["value"]
    assert {"bound", "achieved", "peak", "unit", "frac", "traffic"} <= set(line["roofline"]) and {"value", "unit", "cores", "kind", "sample"} <= set(line["cpu_baseline"])


def test_bench_dump_outputs(hostsim_lib, tmp_path):
    """--dump-outputs: the last timed step's candidate table and labels as float64 .npy files, the same for two runs with the same arguments"""
    import numpy as np
    env = dict(os.environ, ARB_BENCH_DIR=str(tmp_path), PYTHONPATH=ROOT)
    dumps = []
    for run, steps in (("a", "1"), ("b", "2")):
        d = str(tmp_path / run)
        r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "bench_dry_run.py"), "--workload", "tiny_20k", "--steps", steps, "--warmup", "0", "--no-cpu-baseline",
                            "--dump-outputs", d], env=env, capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == int(steps)
        dumps.append({f: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))})
    assert sorted(dumps[0]) == sorted(dumps[1]) and "candidates.filter.npy" in dumps[0] and "fragments.label.npy" in dumps[0]
    assert sum(a.nbytes for a in dumps[0].values()) <= 64 << 20
    for f, a in dumps[0].items():
        assert a.dtype == np.float64 and np.array_equal(a, dumps[1][f]), f
    assert len(dumps[0]["fragments.label.npy"]) > 10000


@pytest.mark.skipif(not _build.oracle_available(), reason="needs the reference binary, which oracle/Makefile builds from the reference sources")
def test_reference_arm_line(tmp_path):
    env = dict(os.environ, ARB_BENCH_DIR=str(tmp_path), PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", "tiny_20k", "--steps", "1", "--warmup", "0"], env=env, capture_output=True, text=True, timeout=900, cwd=str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["value"] > 0 and line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["value"] == line["value"]
