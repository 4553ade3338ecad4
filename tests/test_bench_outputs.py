"""bench.py --dump-outputs writes the scores and norms of the last timed step, the inputs are the same from run to run, and
--steps sets the number of timed steps (the launches of the timed region scale with it)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu


def _bench(steps, out, *extra):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "1", "--workload", "512",
           "--no-workloads", "--no-cpu-baseline", "--no-refgpu", "--no-numa-bind", "--dump-outputs", str(out), *extra]
    p = subprocess.run(cmd, cwd=ROOT, env=dict(os.environ, BENCH_NO_CLOCKS="1"), stdout=subprocess.PIPE, check=True, text=True)
    return json.loads(p.stdout.strip().splitlines()[-1])


def test_dump_outputs_and_steps(tmp_path):
    one, two = _bench(1, tmp_path / "a"), _bench(2, tmp_path / "b")
    assert one["steps"] == 1 and two["steps"] == 2
    assert two["gpu_launches"] == 2 * one["gpu_launches"] > 0
    a, b = np.load(tmp_path / "a" / "scores.npy"), np.load(tmp_path / "b" / "scores.npy")
    n = one["config"]["pairs_per_step_per_gpu"]
    assert a.dtype == np.float64 and a.shape == (n,)
    assert np.all((a > 0) & (a <= 100)) and np.unique(a).size > 1
    assert np.array_equal(a, b)
    assert a[0] == one["scores"]["first"] and a[-1] == one["scores"]["last"]
    na, nb = np.load(tmp_path / "a" / "norms.npy"), np.load(tmp_path / "b" / "norms.npy")
    assert na.dtype == np.float64 and na.shape == (n, 108) and np.all(np.isfinite(na)) and np.any(na != 0)
    assert np.array_equal(na, nb)
    # the shard API scores the same seeded pairs in the same order: same scores, bit for bit, and no norms
    sh = _bench(1, tmp_path / "s", "--shard-api")
    assert sh["steps"] == 1 and sorted(os.listdir(tmp_path / "s")) == ["scores.npy"]
    assert np.array_equal(np.load(tmp_path / "s" / "scores.npy"), a)
