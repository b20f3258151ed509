"""GPU: `bench.py --dump-outputs` writes what the last timed actor step returned.  A small run of the headline workload
is checked bit for bit against the same actor steps replayed through the host API (one te_step per actor step, a greedy
decision every `spacing` steps counted from the start of each of bench's pre-roll / warm-up / timed ranges)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402

E, PREROLL, WARMUP, STEPS = 256, 7, 2, 5


@pytest.mark.parametrize("launches", [[], ["--no-multi"]], ids=["multi", "one_per_step"])
def test_dump_is_the_last_timed_step(tmp_path, launches):
    from traffic_env_b200 import VecTrafficEnv
    out = tmp_path / "dump"
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--envs", str(E), "--preroll", str(PREROLL),
           "--warmup", str(WARMUP), "--steps", str(STEPS), "--no-e2e", "--no-cpu-baseline", "--no-secondary",
           "--dump-outputs", str(out)] + launches
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout + res.stderr
    assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == STEPS
    w = bench.WORKLOADS["grid10x10_L500_greedy"]
    env = VecTrafficEnv(m=w["m"], n=w["n"], length=w["length"], num_envs=E, local_cars_per_sec=w["lcps"],
                        arrivals="philox", seed=2026, ticks_per_step=bench.K_TICKS, remi=True)
    env.reset()
    for n in (PREROLL, WARMUP, STEPS):
        for s in range(n):
            if s % bench.SPACING == 0:
                act = env.greedy_actions().copy()
            obs, rew, done = env.step(act)
    assert obs.any() and rew.any()
    assert (np.load(out / "env_index.npy") == np.arange(E)).all()
    for name, want in (("obs", obs), ("reward", rew), ("done", done), ("actions", act)):
        got = np.load(out / (name + ".npy"))
        assert got.dtype == np.float32 and got.tobytes() == want.astype(np.float32).tobytes(), name
    env.close()
