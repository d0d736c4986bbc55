"""bench.py --dump-outputs: the arrays of the headline path's last step, identical from run to run at equal arguments
(seeded data and keys, run-to-run deterministic kernels), so that two builds can be compared output for output."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, steps):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "c1", "--steps", str(steps), "--warmup", "3",
           "--no-e2e", "--no-cpu-baseline", "--dump-outputs", str(out_dir)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return {p.stem: np.load(p) for p in sorted(out_dir.glob("*.npy"))}


def test_bench_dump_outputs_repeat(cuda, tmp_path):
    a = _bench(tmp_path / "a", 7)
    b = _bench(tmp_path / "b", 7)
    c = _bench(tmp_path / "c", 8)
    assert {"loss", "n_examples", "rng_key", "optim_m", "optim_v", "param_w_loc", "param_intercept_loc"} <= set(a)
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    assert set(a) == set(b) == set(c)
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert np.isfinite(a["loss"]).all() and a["n_examples"][0] > 0
    # one more timed step is one more update: the state moves
    assert not np.array_equal(a["rng_key"], c["rng_key"]) and not np.array_equal(a["param_w_loc"], c["param_w_loc"])
