"""bench.py --dump-outputs on the GPU: the last timed generation's outputs, the same from run to run."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import rel_err

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.gpu
def test_dump_outputs_repeat_with_the_same_arguments(tmp_path):
    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "cartpole", "--steps", "3",
                            "--warmup", "0", "--table-log2", "20", "--no-extras", "--no-cpu-baseline",
                            "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600, cwd=ROOT)
        assert r.returncode == 0, r.stderr[-2000:]
        dumps.append({f: np.load(out / f) for f in os.listdir(out)})
    a, b = dumps
    assert set(a) == {"policy.npy", "population_returns.npy", "episode_reward.npy", "best_reward.npy",
                      "best_policy.npy"}
    assert a["population_returns.npy"].shape == (4096, 1) and a["policy.npy"].shape == (4610,)
    for name in a:
        assert a[name].dtype in (np.float32, np.float64), name
        assert rel_err(a[name], b[name]) < 1e-5, name
