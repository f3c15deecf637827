"""bench.py --dump-outputs: what the timed path computed in its last step, reproducible from run to run."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, *args):
    subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "256", "--warmup", "0",
                    "--dump-outputs", str(out_dir), *args], check=True, capture_output=True, cwd=ROOT, timeout=600)
    return np.load(os.path.join(str(out_dir), "ao.npy"))


def _oracle_frame0():
    import bench
    from oracle.oracle import Oracle
    return Oracle(256, 256, intensity=bench.INTENSITY).run(bench.make_depth(256, 256, 0)).astype(np.float32)


def test_reference_arm_dump_is_the_oracle_output_and_reproducible(tmp_path):
    a = _bench(tmp_path / "a", "--impl", "reference", "--steps", "2")
    b = _bench(tmp_path / "b", "--impl", "reference", "--steps", "2")
    assert a.dtype == np.float32 and a.shape == (256, 256)
    assert np.array_equal(a, b)
    assert np.array_equal(a, _oracle_frame0())


def test_dump_above_the_budget_is_a_fixed_sample(tmp_path, monkeypatch):
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 40_000)
    a = np.arange(100 * 100, dtype=np.float64).reshape(100, 100)
    bench.dump_output(str(tmp_path / "a"), "x", a)
    bench.dump_output(str(tmp_path / "b"), "x", a)
    got = np.load(str(tmp_path / "a" / "x.npy"))
    assert os.path.getsize(str(tmp_path / "a" / "x.npy")) <= 40_000
    assert got.dtype == np.float32 and got.ndim == 1 and np.all(np.diff(got) > 0)     # sorted positions of a ramp
    assert np.array_equal(got, np.load(str(tmp_path / "b" / "x.npy")))


@pytest.mark.gpu
def test_gpu_dump_is_the_last_timed_step(tmp_path):
    """9 steps over 8 rotating depth frames: the last step renders frame 0 again, whose AO the oracle gives."""
    got = _bench(tmp_path / "gpu", "--steps", "9", "--quick", "--no-cpu")
    assert np.array_equal(got, _oracle_frame0())
