"""bench.py --dump-outputs on the GPU: the files hold what the last timed step returned, checked against the CPU
oracle stepping the same inputs."""

import json
import os
import subprocess
import sys
import tempfile

import numpy as np
import pytest

from conftest import ROOT
from oracle import oracle as O

pytestmark = pytest.mark.gpu

NAMES = ("state", "reward", "done", "truncated", "step_count", "lengths")


def test_dump_outputs_hold_the_last_timed_step():
    from ac_solver_b200.synthetic import random_actions, random_presentations

    rows, mrl, horizon = 1 << 16, 36, 200
    with tempfile.TemporaryDirectory() as d:
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0",
                              "--rows", str(rows), "--cpu-sample-rows", "2048", "--skip-bfs", "--skip-greedy",
                              "--skip-vecenv", "--skip-ppo", "--skip-barcode", "--skip-python-baseline",
                              "--dump-outputs", d], capture_output=True, text=True, timeout=600)
        assert out.returncode == 0, out.stderr
        lines = [l for l in out.stdout.splitlines() if l.strip()]
        assert len(lines) == 1 and json.loads(lines[0])["steps"] == 1
        assert sorted(os.listdir(d)) == sorted(n + ".npy" for n in NAMES)
        got = {n: np.load(os.path.join(d, n + ".npy")) for n in NAMES}
    assert all(a.dtype == np.float32 and len(a) == rows for a in got.values())
    # the one timed step ran on state buffer 0: the seed-0 presentations, the seed-1 actions, step counters at 0
    state = random_presentations(rows, mrl, seed=0)
    step_count = np.zeros(rows, np.int32)
    reward, done, trunc, lens, status = O.env_step_batch(state, random_actions(rows, seed=1), step_count, horizon)
    ok = status == 0
    assert ok.sum() > rows // 2
    assert np.array_equal(got["state"], state)
    for name, exp in (("reward", reward), ("done", done), ("truncated", trunc), ("step_count", step_count),
                      ("lengths", lens)):
        assert np.array_equal(got[name][ok], exp[ok]), name
