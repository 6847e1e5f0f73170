"""bench.py --dump-outputs: two runs with the same arguments write the same arrays, float32 and under 64 MB in all; --steps
is the number of timed steps; and what is written is the state after the last timed step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

pytestmark = pytest.mark.gpu


def run_bench(out, *args):
    proc = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--no-extra", "--dump-outputs", str(out)] + list(args),
                          cwd=os.path.dirname(out), capture_output=True, text=True, timeout=600)
    assert proc.returncode == 0, proc.stderr[-3000:]
    return json.loads(proc.stdout.strip().splitlines()[-1])


def load(d):
    return {f: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dumped_outputs_repeat_from_run_to_run(tmp_path):
    a = run_bench(tmp_path / "a", "--steps", "7", "--warmup", "3")
    run_bench(tmp_path / "b", "--steps", "7", "--warmup", "3")
    assert a["steps"] == a["timed"]["steps"] == 7 and a["gpu_launches"] == 7
    da, db = load(tmp_path / "a"), load(tmp_path / "b")
    assert sorted(da) == sorted(db) == sorted(k + ".npy" for k in ("reward", "terminated", "win", "target_find", "obs", "state"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in da) <= 64e6
    for f in da:
        assert da[f].dtype == np.float32 and len(da[f]) > 200_000, f
        assert np.array_equal(da[f], db[f]), f
    assert da["obs.npy"].shape[1:] == (3, 4)


def test_dump_is_the_state_after_the_last_timed_step(tmp_path):
    """c3 draws its policy in the kernel, keyed by env id, episode and time step, so its outputs depend only on how many
    steps were taken: 1 (launch count probe) + warm-up + burn-in (6000 rounded up to whole K-step replays) + K timed.
    K=7, W=3 and K=6, W=10 both take 6017 steps and must agree; K=7, W=4 takes one more and must not.  A dump taken before
    the timed replay would compare 6010 with 6011 steps instead."""
    run_bench(tmp_path / "k7w3", "--workload", "c3", "--steps", "7", "--warmup", "3")
    run_bench(tmp_path / "k6w10", "--workload", "c3", "--steps", "6", "--warmup", "10")
    run_bench(tmp_path / "k7w4", "--workload", "c3", "--steps", "7", "--warmup", "4")
    a, b, c = load(tmp_path / "k7w3"), load(tmp_path / "k6w10"), load(tmp_path / "k7w4")
    assert sorted(a) == sorted(b) == sorted(c)
    for f in a:
        assert np.array_equal(a[f], b[f]), f
    assert not np.array_equal(a["state.npy"], c["state.npy"])
