"""bench.py's command line and output dump (CPU-only: the timed run itself needs a GPU)."""
import importlib.util
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    spec = importlib.util.spec_from_file_location("bench", os.path.join(ROOT, "bench.py"))
    bench = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(bench)
    return bench


def test_steps_below_one_are_rejected():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 2 and "--steps must be at least 1" in res.stdout, res.stdout


def test_dump_outputs_writes_float64_arrays(tmp_path):
    class Ct:                          # stands in for engine.Ciphertext: numpy() gives the active limbs as uint64
        def __init__(self, a):
            self.a = a

        def numpy(self):
            return self.a

    rng = np.random.default_rng(0)
    grad = rng.integers(0, 1 << 60, size=(1, 2, 2, 64), dtype=np.uint64)
    neww = rng.integers(0, 1 << 60, size=(1, 2, 1, 64), dtype=np.uint64)
    weights = rng.uniform(-1, 1, 8)
    grad[0, 0, 0, :3] = [(1 << 60) - 1, (1 << 53) + 1, 1]     # words float64 alone would round
    _bench().dump_outputs(str(tmp_path / "out"), Ct(grad), Ct(neww), weights)
    out = tmp_path / "out"
    assert sorted(os.listdir(out)) == ["gradient_ct_hi.npy", "gradient_ct_lo.npy", "weights.npy",
                                       "weights_ct_hi.npy", "weights_ct_lo.npy"]
    for name, want in (("gradient_ct", grad), ("weights_ct", neww)):
        hi, lo = np.load(out / (name + "_hi.npy")), np.load(out / (name + "_lo.npy"))
        assert hi.dtype == lo.dtype == np.float64 and hi.shape == lo.shape == want.shape
        assert np.array_equal((hi.astype(np.uint64) << np.uint64(30)) | lo.astype(np.uint64), want)   # exact round trip
    got = np.load(out / "weights.npy")
    assert got.dtype == np.float64 and np.array_equal(got, weights)


def test_dump_outputs_with_ncu_is_rejected():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--ncu", "--dump-outputs", "unused"],
                         stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    assert res.returncode == 2 and "--dump-outputs" in res.stdout, res.stdout
