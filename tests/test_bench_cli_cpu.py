"""bench.py's command line and --dump-outputs writer.  CPU only."""
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_writes_every_result_field(tmp_path):
    import bench
    from cartographer_b200._lib import RESULT2D_DTYPE
    rec = np.zeros(3, RESULT2D_DTYPE)
    rec["found"] = [1, 0, 1]
    rec["score"] = np.float32([0.625, 0.0, 0.71875])
    rec["pose_estimate"] = [[1.0, -2.5, 0.125], [0, 0, 0], [3.0, 4.0, -1.0]]
    rec["best_scan_index"] = [7, 0, 2147483647]
    bench.dump_outputs(str(tmp_path / "out"), rec)
    assert sorted(os.listdir(tmp_path / "out")) == sorted(n + ".npy" for n in RESULT2D_DTYPE.names)
    score = np.load(tmp_path / "out" / "score.npy")
    assert score.dtype == np.float32 and np.array_equal(score, rec["score"])
    for name in RESULT2D_DTYPE.names:
        a = np.load(tmp_path / "out" / (name + ".npy"))
        assert a.dtype in (np.float32, np.float64) and a.shape == rec[name].shape
        assert np.array_equal(a, rec[name])


def _bench(*argv):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *argv],
                          capture_output=True, text=True, timeout=120)


def test_bench_rejects_zero_steps():
    out = _bench("--steps", "0")
    assert out.returncode == 2 and "--steps" in out.stderr


def test_bench_rejects_dump_outside_config_2(tmp_path):
    out = _bench("--config", "1", "--dump-outputs", str(tmp_path))
    assert out.returncode == 2 and "--dump-outputs" in out.stderr
    out = _bench("--impl", "reference", "--dump-outputs", str(tmp_path))
    assert out.returncode == 2 and "--dump-outputs" in out.stderr
