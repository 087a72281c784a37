"""bench.py --dump-outputs without a GPU: the writer's dtypes and size cap, the fixed env sample, and the argument checks."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_write_outputs_dtypes_and_cap(tmp_path):
    bench.write_outputs(str(tmp_path / "out"), {"params": np.ones(3, np.float32), "action": np.array([1, 2], np.int32),
                                                "terminal": np.array([0, 1], np.uint8), "key": np.array([2**40 + 1], np.int64)})
    got = {f[:-4]: np.load(tmp_path / "out" / f) for f in os.listdir(tmp_path / "out")}
    assert sorted(got) == ["action", "key", "params", "terminal"]
    assert got["params"].dtype == np.float32
    assert all(got[k].dtype == np.float64 for k in ("action", "terminal", "key"))
    assert got["key"][0] == 2**40 + 1
    with pytest.raises(ValueError):
        bench.write_outputs(str(tmp_path / "big"), {"x": np.zeros(bench.DUMP_MAX_BYTES // 4 + 1, np.float32)})
    assert not (tmp_path / "big").exists()


def test_dump_env_sample_is_fixed():
    assert np.array_equal(bench.dump_env_sample(100), np.arange(100))
    a, b = bench.dump_env_sample(65536), bench.dump_env_sample(65536)
    assert a.size == bench.DUMP_ENVS and np.array_equal(a, b) and np.all(np.diff(a) > 0) and a[-1] < 65536


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "x"]])
def test_bench_rejects_bad_arguments(argv):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "error" in r.stderr
