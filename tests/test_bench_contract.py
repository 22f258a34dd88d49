"""bench.py's reference arm runs on the CPU (the C oracle stands in for the Dart reference), so its side of the JSON
contract can be checked here: one line, the arm's keys, and that a rank other than 0 prints nothing."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(env_extra, *args):
    env = dict(os.environ, B200Z_REF_UNITS="64", B200Z_CACHE=os.path.join(ROOT, ".pytest_cache", "b200z_cache"), **env_extra)
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *args], capture_output=True,
                       text=True, env=env, cwd=ROOT, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return [ln for ln in p.stdout.splitlines() if ln.strip()]


def test_reference_arm_line():
    lines = run({}, "--steps", "2", "--warmup", "1")
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "inflate_uncompressed_GBps" and d["unit"] == "GB/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload"].startswith("gzip-multimember-64KiB")


def test_reference_arm_other_ranks_are_silent():
    assert run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"}, "--gpus", "2", "--steps", "1", "--warmup", "1") == []


def test_bad_arguments_are_refused():
    for args in (["--steps", "0"], ["--dump-outputs", "out"], ["--config", "3", "--dump-outputs", "out"]):
        p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", *args], capture_output=True,
                           text=True, cwd=ROOT, timeout=60)
        assert p.returncode == 2 and "error" in p.stderr, args
    assert not os.path.exists(os.path.join(ROOT, "out"))


def test_dump_outputs(tmp_path):
    """--dump-outputs: float arrays only, the same sample of units every time, exact values, and at the default size
    (16 384 units) at most 64 MB in all."""
    import numpy as np
    import bench  # (the repository root is on sys.path: conftest.py)
    n = 200
    rng = np.random.default_rng(1)
    full = rng.integers(0, 256, size=n * bench.UNIT, dtype=np.uint8)
    status, out_len, in_used = np.zeros(n, np.int32), np.full(n, bench.UNIT, np.int32), rng.integers(1, 65536, n).astype(np.int32)
    for d in (tmp_path / "a", tmp_path / "b"):
        bench.dump_outputs(str(d), full, status, out_len, in_used)
    a = {f.stem: np.load(f) for f in (tmp_path / "a").iterdir()}
    assert sorted(a) == ["decoded_sample", "decoded_sample_units", "in_used", "out_len", "status"]
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    for f in (tmp_path / "b").iterdir():
        assert np.array_equal(np.load(f), a[f.stem])
    units = a["decoded_sample_units"].astype(np.int64)
    assert len(units) == bench.DUMP_UNITS and len(set(units)) == len(units) and (np.diff(units) > 0).all()
    assert np.array_equal(a["decoded_sample"], full.reshape(n, bench.UNIT)[units])
    assert np.array_equal(a["in_used"], in_used) and np.array_equal(a["out_len"], out_len) and not a["status"].any()
    assert bench.DUMP_UNITS * bench.UNIT * 4 + 3 * 4 * 16384 + 8 * bench.DUMP_UNITS <= 64e6
