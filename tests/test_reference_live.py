"""Build-container only (marker `reference`; skipped where /root/reference is absent, e.g. on the GPU box).

(a) the C oracle against the LIVE unmodified reference (numba), tick by tick, on grids / seeds / flags that are
    NOT among the committed fixtures - fresh evidence every run that oracle/traffic_oracle.c restates
    gym_traffic/envs/traffic_env.py:224-248 exactly (ring indices, obs, waiting, rewards, done, x and v bits);
(b) the reference's own launcher and baseline agents (traffic_test.py, alg_flags.py,
    gym_traffic/algorithms/{fixed,random,greedy,const0,const1,spacedgreedy}.py) import UNCHANGED on top of the drop-in
    gym_traffic package, `traffic_test.make_env()` builds the reference's own wrapper chain around the drop-in
    TrafficEnv, and - in this GPU-less container - the first call that needs the device fails with the library's
    "no CUDA device" error and nothing else (no CPU fallback).
"""
import os
import subprocess
import sys

import numpy as np
import pytest

from tests.golden_util import tick_digest

pytestmark = pytest.mark.reference
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (m, n, length, ticks, local_cars_per_sec, light period, seed, learn_switch, poisson)
LIVE_CASES = [
    (5, 4, 300, 300, 0.30, 17, 101, False, True),
    (2, 5, 90, 400, 1.00, 60, 102, False, True),     # heavy overflow: short roads, long reds, stepping past `done`
    (7, 7, 400, 200, 0.25, 23, 103, False, True),
    (3, 3, 250, 400, 0.40, 9, 104, True, True),      # learn_switch
    (4, 3, 200, 300, 0.30, 13, 105, False, False),   # regular arrivals
]


@pytest.mark.parametrize("case", LIVE_CASES, ids=lambda c: "%dx%d_L%d_seed%d" % (c[0], c[1], c[2], c[6]))
def test_oracle_vs_reference_live(case):
    from oracle import ref_harness as rh
    from oracle.gen_golden import set_flags
    from oracle.oracle import OracleEnv
    m, n, length, ticks, lcps, period, seed, learn_switch, poisson = case
    ref = rh.load()
    set_flags(ref, local_cars_per_sec=lcps, learn_switch=learn_switch, poisson=poisson)
    try:
        np.random.seed(seed)
        env = rh.make_env(ref, m, n, length, seed=seed)
        sched = rh.record_schedule(ref, m, n, ticks, seed=seed)
        env.reset()
        o = OracleEnv(m, n, float(length), 0.5, learn_switch=learn_switch)
        o.reset(env.current_phase.copy())
        rng = np.random.RandomState(seed + 1)
        overflow_ticks = 0
        for t in range(ticks):
            if t % period == 0:
                a = rng.randint(2, size=m * n).astype(np.int32)
            obs, rew, done, _ = env.step(a)
            od = o.step(a, sched[t])
            xs, vs = rh.live_state(env)
            oxs, ovs = o.live_state()
            dr = tick_digest(env.leading, env.lastcar, env.obs, env.waiting, env.passed_dst, rew, done, xs, vs)
            do = tick_digest(o.leading, o.lastcar, o.obs, o.waiting, o.passed_dst, o.rewards, od, oxs, ovs)
            assert dr == do, "tick %d: oracle diverges from the live reference" % t
            overflow_ticks += int(done)
        assert env.generated_cars == o.generated_cars == sum(len(s) for s in sched)
        if (m, n) == (2, 5):
            assert overflow_ticks > 20, "the heavy case is meant to overflow"
    finally:
        set_flags(ref)


def test_oracle_clock_past_2_24_vs_reference_live():
    """The np.float32 episode clock near 2^24, validate mode: the reference adds 1 per tick to a float32 clock (under
    NumPy 2 it stays float32), so it stops at 16777216, and cars born after that leave with trip time 0.  The oracle's
    clock (to_set_steps, then its own tick rule) and its trip times must equal the reference's, tick by tick."""
    from oracle import ref_harness as rh
    from oracle.gen_golden import set_flags
    from oracle.oracle import OracleEnv
    m, n, length, ticks, seed = 3, 3, 100, 200, 106
    start = np.float32(2 ** 24 - 20)
    ref = rh.load()
    set_flags(ref, local_cars_per_sec=0.2, mode="validate")
    try:
        np.random.seed(seed)
        env = rh.make_env(ref, m, n, length, seed=seed)
        sched = rh.record_schedule(ref, m, n, ticks, seed=seed)
        env.reset()
        env.steps = start
        o = OracleEnv(m, n, float(length), 0.5, validate=True)
        o.reset(env.current_phase.copy())
        o.steps = start
        rng = np.random.RandomState(seed + 1)
        for t in range(ticks):
            if t % 11 == 0:
                a = rng.randint(2, size=m * n).astype(np.int32)
            obs, rew, done, _ = env.step(a)
            od = o.step(a, sched[t])
            assert type(env.steps) is np.float32 and env.steps.tobytes() == np.float32(o.steps).tobytes(), t
            xs, vs = rh.live_state(env)
            oxs, ovs = o.live_state()
            dr = tick_digest(env.leading, env.lastcar, env.obs, env.waiting, env.passed_dst, rew, done, xs, vs)
            do = tick_digest(o.leading, o.lastcar, o.obs, o.waiting, o.passed_dst, o.rewards, od, oxs, ovs)
            assert dr == do, "tick %d: oracle diverges from the live reference" % t
        assert float(env.steps) == 2.0 ** 24
        want = np.asarray(env.trip_times, np.float64)
        assert want.tobytes() == o.trip_times().tobytes()
        assert (want == 0.0).any() and (want > 0.0).any(), "cars born before and after the clock stopped are meant to leave"
    finally:
        set_flags(ref)


_LAUNCHER_SCRIPT = r"""
import importlib, os, sys, types
sys.path.insert(0, %(root)r)
os.environ.setdefault("NUMBA_CACHE_DIR", "/tmp/traffic_env_numba_cache")
for stub in ("tensorflow", "matplotlib", "matplotlib.pyplot"):     # inert: the baseline agents import but never use them
    try:
        importlib.import_module(stub)
    except Exception:
        sys.modules[stub] = types.ModuleType(stub)
sys.path.insert(0, os.path.join(%(root)r, 'tests', 'support', 'gym_compat'))   # the only stand-in: an old-API gym
import traffic_env_b200.install as inst
dropin = inst.install(reference_dir=%(ref)r)
sys.argv = ["traffic_test.py", "--trainer", "fixed"]
import traffic_test, alg_flags, args
ref = os.path.realpath(%(ref)r)
for mod in (traffic_test, alg_flags, args):
    assert os.path.realpath(mod.__file__).startswith(ref), mod.__file__
for name in ("fixed", "random", "greedy", "const0", "const1", "spacedgreedy"):
    mod = importlib.import_module("gym_traffic.algorithms." + name)
    assert os.path.realpath(mod.__file__).startswith(ref), mod.__file__
    assert callable(mod.run)
for name in ("warmup", "history", "gspace"):
    mod = importlib.import_module("gym_traffic.wrappers." + name)
    assert os.path.realpath(mod.__file__).startswith(ref), mod.__file__
import gym_traffic, gym_traffic.envs.traffic_env as te, gym_traffic.envs.roadgraph as rg, gym_traffic.spaces.gspace as gs
for mod in (gym_traffic, te, rg, gs):
    assert os.path.realpath(mod.__file__).startswith(os.path.realpath(dropin)), mod.__file__
from gym_traffic.envs.traffic_env import cars_on_roads          # greedy.py:4 imports it by name
args.parse_flags()                                              # traffic_test.py:94
assert args.FLAGS.light_iterations == 10 and args.FLAGS.episode_len == 120
env = traffic_test.make_env()                                   # the reference's own wrapper chain
chain = []
e = env
while True:
    chain.append(type(e).__name__)
    if e is e.unwrapped: break
    e = e.env
assert chain == ["Remi", "Repeater", "TrafficEnv"], chain
assert type(env).__module__ == "traffic_test" and type(env.unwrapped).__module__ == "gym_traffic.envs.traffic_env"
assert env.action_space.shape == [9] and env.observation_space.shape == [81] and env.reward_size == 9
from traffic_env_b200 import TrafficB200Error
import ctypes
try:
    ctypes.CDLL("libcuda.so.1"); have_driver = True
except OSError:
    have_driver = False
try:
    obs = env.reset()
except TrafficB200Error as ex:
    assert "no CUDA device" in str(ex), str(ex)
    print("LAUNCHER_OK no-device")
else:
    # a GPU is present: run the reference's own `fixed` agent loop body for one episode
    total = 0.0
    for i in range(args.FLAGS.episode_len):
        a = __import__("numpy").ones(9) if importlib.import_module("gym_traffic.algorithms.fixed").phase(i) else __import__("numpy").zeros(9)
        obs, reward, done, info = env.step(a)
        total += float(reward.mean())
        if done: break
    print("LAUNCHER_OK device", total)
"""


def test_reference_launcher_imports_over_dropin():
    from oracle import ref_harness as rh
    script = _LAUNCHER_SCRIPT % {"root": ROOT, "ref": rh.REFERENCE_DIR}
    res = subprocess.run([sys.executable, "-c", script], capture_output=True, text=True, cwd="/tmp", timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "LAUNCHER_OK" in res.stdout, res.stdout + res.stderr
