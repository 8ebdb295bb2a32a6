"""GPU: the B200 arm of bench.py prints one line that satisfies the contract validator, for the default workload (shrunk) and the two
secondary configs (shrunk); e2e crosses host buffers."""
import json
import os
import subprocess
import sys

import pytest

from tests.test_bench_contract import validate_line

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("cfg,extra", [("idqn", ["--envs", "256", "--batch", "64", "--buffer", "1024"]), ("vdn15", ["--envs", "128", "--batch", "32", "--buffer", "512"]),
                                       ("ia2c", ["--envs", "512"])])
def test_b200_arm_line(cfg, extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", cfg, "--steps", "2", "--warmup", "3", "--no-cpu-baseline"] + extra,
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    validate_line(d)
    assert d["n_gpus"] == 1 and d["env_steps_timed"] > 0
    assert 0.2 * d["value"] < d["e2e"]["value"] <= 1.1 * d["value"]


def test_dump_outputs_repeat_and_follow_steps(tmp_path):
    """--dump-outputs: two runs with the same arguments write the same arrays (seeded inputs, reductions in a fixed order); one more timed step
    changes them."""
    import numpy as np

    dumps = {}
    for name, steps in (("a", 2), ("b", 2), ("c", 3)):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "idqn", "--envs", "256", "--batch", "64", "--buffer", "1024",
                              "--steps", str(steps), "--warmup", "3", "--no-cpu-baseline", "--no-e2e", "--dump-outputs", str(tmp_path / name)],
                             capture_output=True, text=True, timeout=900)
        assert out.returncode == 0, out.stderr[-3000:]
        assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
        dumps[name] = {f[:-4]: np.load(tmp_path / name / f) for f in sorted(os.listdir(tmp_path / name))}
    a, b, c = dumps["a"], dumps["b"], dumps["c"]
    assert {"theta", "theta_target", "metrics", "episode_length", "episode_return", "episodes_obs", "episodes_act"} <= set(a)
    assert all(v.dtype == np.float32 for v in a.values()) and sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a["episode_length"].shape == (256,) and a["episodes_obs"].shape == (256, 2, 26, 15) and a["episode_length"].sum() > 0
    assert a.keys() == b.keys() and all(np.array_equal(a[k], b[k]) for k in a), [k for k in a if not np.array_equal(a[k], b[k])]
    assert not np.array_equal(a["theta"], c["theta"])
