"""bench.py --dump-outputs: the tracker results of the last timed step, written as float64 .npy files, are the same from
run to run (the inputs depend on the arguments only and the solve sums are reduced in a fixed order), so that the outputs
of two builds can be compared file by file."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

STREAMS, STEPS = 16, 3


def run_bench(out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(STEPS), "--warmup", "3",
                        "--streams", str(STREAMS), "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


def test_dump_outputs_repeat_exactly(tmp_path):
    a, b = tmp_path / "a", tmp_path / "b"
    res = run_bench(a)
    run_bench(b)
    assert res["steps"] == STEPS and res["config"]["streams_per_gpu"] == STREAMS
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b))
    assert {"poses.npy", "summary_final_cost.npy", "summary_iterations.npy", "summary_termination.npy"} <= set(names)
    total = 0
    for n in names:
        x, y = np.load(a / n), np.load(b / n)
        assert x.dtype == np.float64 and x.shape == ((STREAMS, 7) if n == "poses.npy" else (STREAMS, 3)), (n, x.shape)
        np.testing.assert_array_equal(x, y, err_msg=n)
        total += x.nbytes
    assert total <= 64 << 20
    poses = np.load(a / "poses.npy")
    assert np.allclose(np.linalg.norm(poses[:, :4], axis=1), 1.0)
    # the last timed step (frame 6) is no key frame: every stream solved every level from real points and stopped on a
    # convergence test or the iteration limit (terminations 1..5)
    term = np.load(a / "summary_termination.npy")
    assert (np.load(a / "summary_n_residuals.npy") > 0).all() and ((term >= 1) & (term <= 5)).all(), term
