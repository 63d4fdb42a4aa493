"""GPU: bench.py --dump-outputs writes what the last timed step computed (float32 / float64 .npy files, < 64 MB): the
workload's start states, chained steps and normalised advantages, the same bits on every run with the same arguments.
--steps is the number of timed steps: the timed region issues `steps` times the launches of one step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(steps, dump=None):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--batch", "4096",
           "--cpu-batch", "0", "--no-e2e"] + (["--dump-outputs", dump] if dump else [])
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_dump_outputs_repeatable_and_steps_counted(tmp_path):
    a, b = str(tmp_path / "a"), str(tmp_path / "b")
    la, lb, l1 = _bench(2, a), _bench(2, b), _bench(1)
    assert la["steps"] == lb["steps"] == 2 and l1["steps"] == 1
    assert la["gpu_launches"] == 2 * l1["gpu_launches"] > 0
    names = sorted(os.listdir(a))
    assert names == sorted(os.listdir(b))
    assert {"obs.npy", "act.npy", "nextobs.npy", "rew.npy", "adv.npy", "cret.npy", "length.npy",
            "adv_stats_sums.npy"} <= set(names)
    total = 0
    for f in names:
        x, y = np.load(os.path.join(a, f)), np.load(os.path.join(b, f))
        assert x.dtype in (np.float32, np.float64), f
        assert x.dtype == y.dtype and np.array_equal(x, y, equal_nan=True), f
        total += os.path.getsize(os.path.join(a, f))
    assert total < 64e6

    # the contents, checked against what bench.py's workload feeds in and against relations the dump code does not
    # compute: at 4096 start states every path is in the sample, in order
    z = {f[:-4]: np.load(os.path.join(a, f)) for f in names}
    from cmbpo_b200 import workload as wl
    dyn = wl.make_problem(0, 17, 6, hidden=(512, 512), task="HalfCheetahSafe-v2")[0]
    start, _ = wl.make_states(100, 4096, 17, 6, dyn)
    assert np.array_equal(z["path_index"], np.arange(4096))
    length = z["length"].astype(np.int64)
    alive = np.arange(z["obs"].shape[1])[None, :] < length[:, None]
    assert length.min() > 0 and z["adv_stats_sums"][0] == length.sum()
    assert np.array_equal(z["obs"][:, 0], start)
    chained = alive[:, 1:]                                   # step t + 1 starts from the state step t predicted
    assert np.array_equal(z["obs"][:, 1:][chained], z["nextobs"][:, :-1][chained])
    for f in ("obs", "nextobs", "act", "rew", "adv", "cret", "term"):
        assert np.isfinite(z[f]).all() and not z[f][~alive].any(), f
    adv, cadv = z["adv"][alive].astype(np.float64), z["cadv"][alive].astype(np.float64)
    assert abs(adv.mean()) < 1e-3 and abs(adv.std() - 1.0) < 1e-3      # normalised: what the caller receives
    assert abs(cadv.mean()) < 1e-3                                       # centred
