"""GPU: ``bench.py --dump-outputs DIR`` on the training workload (B = 2 episodes keeps it short): exactly ``--steps``
timed steps, then the last one's loss, BatchNorm running statistics, gradients and parameters as float .npy files of
64 MB at most.  Every step starts from the same state, so runs with different numbers of steps dump the same step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench_dump(out, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "3",
                        "--no-secondary", "--no-library-bar", "--no-cpu-baseline", "--dump-outputs", str(out)],
                       cwd=ROOT, capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, AVDN_BENCH_BATCH="2"))
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps and line["config"]["per_gpu_batch"] == 2
    return {f[:-4]: np.load(out / f) for f in os.listdir(out)}


@pytest.mark.gpu
def test_dump_outputs_of_the_training_step(built_lib, tmp_path):
    a = _bench_dump(tmp_path / "a", 1)
    assert sorted(a) == ["et_grad", "et_param", "loss", "trunk_bn_running", "trunk_grad", "trunk_param"]
    assert a["loss"].dtype == np.float64 and a["loss"].shape == (1,)
    for name, x in a.items():
        assert x.dtype in (np.float32, np.float64) and np.isfinite(x).all(), name
        assert np.abs(x).max() > 0, name
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    # two more timed steps before the dumped one: the same state and batch, so the same outputs up to the order of
    # atomic reductions (a step taken from another state moves parameters by ~lr = 1e-5 and gradients far more)
    b = _bench_dump(tmp_path / "b", 3)
    for name in a:
        tol = 1e-6 if name.endswith("_param") or name == "loss" else 1e-5
        err = np.abs(a[name].astype(np.float64) - b[name]).max() / np.abs(a[name]).max()
        assert err <= tol, (name, err)
