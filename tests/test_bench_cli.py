"""bench.py's command line on the CPU arm (--impl reference): --steps sets the number of timed steps and
--dump-outputs writes what the last step computed, the same for the same arguments and within the size cap."""
import json
import os
import subprocess
import sys

import numpy as np

from cnosdb_b200 import datagen

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference"] + list(args),
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def test_scan_dump_is_the_same_for_the_same_arguments(tmp_path):
    lines = [run_bench("--series", "3000", "--steps", "3", "--warmup", "1", "--dump-outputs", str(tmp_path / d))
             for d in ("a", "b")]
    assert all(ln["steps"] == 3 and "3 of 3 steps timed" in ln["cpu_baseline"]["sample"] for ln in lines)
    names = sorted(os.listdir(tmp_path / "a"))
    assert names == sorted(os.listdir(tmp_path / "b"))
    assert {"c1_count.npy", "c1_count_valid.npy", "c2_mean.npy", "c2_mean_valid.npy"} <= set(names)
    for n in names:
        a, b = np.load(tmp_path / "a" / n), np.load(tmp_path / "b" / n)
        assert a.dtype in (np.float32, np.float64)
        np.testing.assert_array_equal(a, b)
    assert np.load(tmp_path / "a" / "c1_count_valid.npy").any()


def test_decode_only_steps_and_exact_timestamps(tmp_path):
    line = run_bench("--workload", "C1", "--steps", "4", "--warmup", "1", "--dump-outputs", str(tmp_path))
    assert line["steps"] == 4
    hi, lo = np.load(tmp_path / "page0_values_hi.npy"), np.load(tmp_path / "page0_values_lo.npy")
    ts = ((hi.astype(np.uint64) << np.uint64(32)) | lo.astype(np.uint64)).view(np.int64)
    assert ts.size == 10_000 and ts[0] == datagen.TSBS_T0 and (np.diff(ts) == datagen.TSBS_STEP).all()


def test_dump_over_the_cap_is_a_fixed_sample(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 8192)
    arrays = {"v": np.arange(2000, dtype=np.float64).reshape(20, 100), "v_valid": np.ones((20, 100), np.float32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
        assert sum(os.path.getsize(tmp_path / d / n) for n in os.listdir(tmp_path / d)) <= 8192
    v = np.load(tmp_path / "a" / "v.npy")
    assert 0 < v.size < 2000 and (np.diff(v) > 0).all()  # positions kept in order
    np.testing.assert_array_equal(v, np.load(tmp_path / "b" / "v.npy"))
    assert np.load(tmp_path / "a" / "v_valid.npy").size == v.size
