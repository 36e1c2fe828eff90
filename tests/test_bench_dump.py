"""bench.py --dump-outputs and --steps on the CPU arm, and the size cap of the dump (no GPU needed)."""
import os
import subprocess
import sys

import numpy as np

from tests.helpers import ROOT

sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _reference_dump(out, steps):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--envs", "64",
                        "--steps", str(steps), "--warmup", "1", "--dump-outputs", str(out)],
                       capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    return {k: np.load(os.path.join(out, k + ".npy")) for k in ("obs", "reward", "done")}


def test_reference_arm_dump_is_reproducible_and_follows_steps(tmp_path):
    a = _reference_dump(tmp_path / "a", 3)
    b = _reference_dump(tmp_path / "b", 3)
    c = _reference_dump(tmp_path / "c", 4)
    assert a["obs"].shape == (64, 76) and a["reward"].shape == (64,) and a["done"].shape == (64,)
    assert all(x.dtype == np.float32 for x in a.values()) and np.isfinite(a["obs"]).all()
    for k in a:
        assert np.array_equal(a[k], b[k]), k                  # same arguments, same inputs, same outputs
    assert not np.array_equal(a["obs"], c["obs"])             # one more timed step, another last step


def test_dump_keeps_the_same_seeded_rows_under_the_cap(tmp_path, monkeypatch):
    n, d = 1000, 76
    obs = np.arange(n * d, dtype=np.float32).reshape(n, d)
    rew = np.arange(n, dtype=np.float32)
    monkeypatch.setattr(bench, "DUMP_LIMIT_BYTES", 100 * (d + 1) * 4 + 2 * 1024)
    bench.dump_outputs(str(tmp_path / "a"), {"obs": obs, "reward": rew})
    bench.dump_outputs(str(tmp_path / "b"), {"obs": obs, "reward": rew})
    o, r = np.load(tmp_path / "a" / "obs.npy"), np.load(tmp_path / "a" / "reward.npy")
    assert o.shape == (100, d) and r.shape == (100,)
    assert np.array_equal(o[:, 0] / d, r)                     # the same rows in every array
    assert np.array_equal(o, np.load(tmp_path / "b" / "obs.npy"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in ("obs.npy", "reward.npy")) <= bench.DUMP_LIMIT_BYTES
    bench.dump_outputs(str(tmp_path / "c"), {"obs": obs[:50], "reward": rew[:50]})     # under the cap: all rows
    assert np.array_equal(np.load(tmp_path / "c" / "obs.npy"), obs[:50])


def test_steps_below_one_is_rejected():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True,
                       text=True, cwd=ROOT, timeout=120)
    assert p.returncode == 2 and "--steps" in p.stderr
