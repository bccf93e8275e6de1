"""bench.py on the B200 at a small domain: --steps sets the number of timed proofs, and --dump-outputs writes the proof of
the last timed step (the verified one), identical from run to run."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(out_dir, steps):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--log-n", "12", "--steps", str(steps), "--warmup", "1",
                          "--no-extras", "--no-cpu", "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=900, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    return json.loads(lines[0])


def test_bench_steps_and_dumped_proof(tmp_path):
    one, two = run_bench(tmp_path / "one", 1), run_bench(tmp_path / "two", 2)
    assert one["steps"] == 1 and two["steps"] == 2
    assert two["gpu_launches"] == 2 * one["gpu_launches"] > 0
    assert one["verified"]["proof_equals_known_discrete_logs"] and two["verified"]["proof_equals_known_discrete_logs"]
    # BLS12-381 affine points in 32-bit limbs: G1 = 2 x 12 words, G2 = 4 x 12 words
    for name, words in (("proof_a", 24), ("proof_b", 48), ("proof_c", 24)):
        a, b = np.load(tmp_path / "one" / f"{name}.npy"), np.load(tmp_path / "two" / f"{name}.npy")
        assert a.dtype == np.float64 and a.shape == (words,) and a.any(), name
        assert np.array_equal(a, b) and np.array_equal(a, np.floor(a)) and a.max() < 2**32, name
