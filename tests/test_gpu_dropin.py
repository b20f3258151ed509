"""GPU: the drop-in gym_traffic package (TrafficEnv facade + wrappers) behaves like the reference's.

The reference tree is not on the GPU box, so the agents' loops (algorithms/fixed.py:9-23,
greedy.py:7-19, random.py:6-16) are restated here as their env-facing contract."""
import os
import sys

import numpy as np
import pytest

from tests.golden_util import live_walk, tick_digest

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


@pytest.fixture(scope="module")
def dropin():
    from tests.support import install_dropin
    install_dropin()
    import gym
    import gym_traffic  # noqa: F401
    from args import FLAGS
    from gym_traffic.envs.roadgraph import GridRoad
    FLAGS.local_cars_per_sec, FLAGS.rate, FLAGS.poisson, FLAGS.entry, FLAGS.learn_switch = 0.12, 0.5, True, "all", False
    return gym, GridRoad, FLAGS


def new_env(gym, GridRoad, m=3, n=3, length=250, seed=0):
    env = gym.make("traffic-v0")
    env.set_graph(GridRoad(m, n, length))
    env.seed_generator(seed)
    env.reset_entrypoints()
    return env


def test_kat_through_the_facade(dropin):
    """SURVEY.md 8c recipe, verbatim, on the drop-in: np.random.seed(0), seed_generator(0), fixed policy.
    The facade feeds the device the reference's own MT19937 arrival stream, so every tick digest of the
    golden run (ints and float bits) must match."""
    gym, GridRoad, FLAGS = dropin
    g = np.load(os.path.join(GOLDEN, "kat_fixed_3x3.npz"))
    np.random.seed(0)
    u = new_env(gym, GridRoad)
    u.reset()
    assert list(u.current_phase) == [0, 1, 1, 0, 1, 1, 1, 1, 1]
    for t in range(1200):
        a = np.ones(9, np.int32) if ((t // 10) % 6) >= 3 else np.zeros(9, np.int32)
        obs, rew, done, info = u.step(a)
        assert obs is u.obs and rew is u.rewards and info is None  # same buffers every call (traffic_env.py:248)
        if t % 50 == 49 or t < 20:
            u.sync_counters()
            st = u._snapshot()
            xs, vs = live_walk(st["leading"][0], st["lastcar"][0], st["x"][0], st["v"][0])
            d = tick_digest(st["leading"][0], st["lastcar"][0], obs, u.waiting, u.passed_dst, rew, done, xs, vs)
            assert d == g["digests"][t], "tick %d" % t
    assert u.generated_cars == 859 and float(u.steps) == 1200.0
    assert u.cars_on_roads().shape == (3, 3, 4)
    assert u.state.shape == (48, 10, 20)


def test_fused_wrappers_match_tick_loop(dropin):
    """Remi(Repeater(10)) with the fused single-launch Repeater == the same wrappers forced onto the
    reference's tick-by-tick loop (rendering flag disables fusion), action types as the agents send them."""
    gym, GridRoad, FLAGS = dropin
    from traffic_env_b200.wrappers import Remi, Repeater

    def build(fused):
        np.random.seed(3)
        base = new_env(gym, GridRoad, seed=11)
        if not fused:
            base.rendering = True           # per-tick rendering requested: Repeater must not fuse ...
            base.render = lambda *a, **k: None  # ... and the (absent) viewer is stubbed out
        return Remi(Repeater(10)(base)), base

    fa, fb = build(True)
    ta, tb = build(False)
    np.random.seed(21)
    o1 = fa.reset()
    np.random.seed(21)   # GSpace.sample() draws phases and the first action from the global RNG
    o2 = ta.reset()
    assert o1.dtype == np.float32 and o1.shape == (81,) and o1.tobytes() == o2.tobytes()
    rng = np.random.RandomState(0)
    sent = [lambda: rng.rand(9) < 0.5,                       # bool (a3c)
            lambda: rng.randint(2, size=9).astype(np.int32),  # int32 (dqn)
            lambda: rng.randint(2, size=9).astype(np.float64),  # float64 (fixed / const)
            lambda: rng.randint(2, size=9).astype(np.int8),   # int8 (cem)
            lambda: tuple(int(v) for v in rng.randint(2, size=9))]  # tuple (UnGSpaceWrapper)
    for s in range(40):
        a = sent[s % len(sent)]()
        x1, r1, d1, _ = fa.step(a)
        x2, r2, d2, _ = ta.step(a)
        assert x1.tobytes() == np.asarray(x2, np.float32).tobytes(), s
        assert np.asarray(r1).tobytes() == np.asarray(r2).tobytes() and d1 == d2, s
    assert fa.reward_size == 9 and fa.observation_space.shape == [81] and fa.action_space.size == 9


def test_fused_wrappers_match_tick_loop_past_clock_limit(dropin, monkeypatch):
    """Remi(Repeater(10)), fused and on the tick loop, from an episode clock of 2^24 - 40: the float32 clock stops at 2^24
    on both paths, one float32 add per tick.  Heavy arrivals make fused steps overflow, and such a step reads back the
    ticks it ran; the count must come from the device, not from the clock, or the injected arrival schedule goes out of
    step with the device.  A short schedule window makes the host send a new window every few steps."""
    gym, GridRoad, FLAGS = dropin
    from gym_traffic.envs import traffic_env as te
    from traffic_env_b200.wrappers import Remi, Repeater
    monkeypatch.setattr(te, "_WINDOW", 48)
    monkeypatch.setattr(FLAGS, "local_cars_per_sec", 0.35)
    start = np.float32(2 ** 24 - 40)

    def build(fused):
        np.random.seed(3)
        base = new_env(gym, GridRoad, seed=11)
        if not fused:
            base.rendering = True
            base.render = lambda *a, **k: None
        return Remi(Repeater(10)(base)), base

    (fa, fb), (ta, tb) = build(True), build(False)
    for env, base in ((fa, fb), (ta, tb)):
        np.random.seed(21)
        env.reset()          # (Repeater's reset runs a first actor step)
        base.steps = start
        st = base._sim.get_state(0, 1)
        st["steps"][:] = start
        base._sim.set_state(st)
    ticks0 = int(tb._sim.stats()["ticks"])
    assert fb._sim.stats()["ticks"] == ticks0
    rng = np.random.RandomState(5)
    fused_overflows = 0
    for s in range(60):
        a = rng.randint(2, size=9) if s % 7 else np.zeros(9, np.int32)
        x1, r1, d1, _ = fa.step(a)
        x2, r2, d2, _ = ta.step(a)
        assert x1.tobytes() == np.asarray(x2, np.float32).tobytes(), s
        assert np.asarray(r1).tobytes() == np.asarray(r2).tobytes() and d1 == d2, s
        fused_overflows += int(d1)
        ticks = int(tb._sim.stats()["ticks"]) - ticks0
        want = np.float32(min(float(start) + ticks, 2.0 ** 24))   # +1 per tick in float32: exact up to 2^24, then stuck
        assert type(fb.steps) is np.float32 and fb.steps == tb.steps == want, (s, float(fb.steps), float(tb.steps), float(want))
        assert fb._sim.get_state(0, 1)["steps"][0] == want, s
        assert fb._sim.stats()["ticks"] == ticks0 + ticks, s
        assert fb._sim.stats()["cars_generated"] == tb._sim.stats()["cars_generated"], s
    assert fused_overflows > 3 and float(fb.steps) == 2.0 ** 24


def test_agent_loop_contracts(dropin):
    gym, GridRoad, FLAGS = dropin
    from tests.support.wrappers_ref import make_env
    FLAGS.light_iterations = 10
    env = make_env(seed=5)
    # fixed.py: float64 0./1. actions alternating every `spacing` steps
    actions = np.zeros((2, *env.action_space.shape))
    actions[1, :] = 1
    obs = env.reset()
    total = 0.0
    for i in range(30):
        obs, reward, done, info = env.step(actions[int((i % 6) >= 3)])
        total += np.mean(reward)
        assert reward.shape == (9,) and reward.dtype == np.float32
        if done:
            break
    # greedy.py: cars_on_roads().dot([1,1,-1,-1]) < 0 every `spacing` steps
    env.reset()
    for i in range(30):
        counts = env.unwrapped.cars_on_roads()
        if i % 3 == 0:
            action = env.action_space.to_action(counts.dot([1, 1, -1, -1]) < 0)
        obs, reward, done, info = env.step(action)
        if done:
            break
    # random.py
    env.reset()
    for i in range(10):
        obs, reward, done, info = env.step(env.action_space.sample())
    assert np.isfinite(obs).all()


def test_writes_to_obs_views_reach_the_device(dropin):
    gym, GridRoad, FLAGS = dropin
    np.random.seed(1)
    u = new_env(gym, GridRoad, seed=2)
    u.reset()
    u.current_phase[:] = 1
    u.elapsed[:] = 3
    u.step(np.ones(9, np.int32))   # no change of phase: elapsed keeps counting from the written value
    assert list(u.current_phase) == [1] * 9 and list(u.elapsed) == [4] * 9


def test_full_wrapper_stack_and_launcher(dropin):
    """traffic_test.make_env's optional layers (Warmup, Localize, Squish, History, UnGSpace) on the B200 env, and
    the baseline-controller launcher."""
    gym, GridRoad, FLAGS = dropin
    from tests.support.wrappers_ref import make_env
    np.random.seed(4)
    env = make_env(seed=1, light_iterations=10, warmup_lights=2, local_weight=3, history=4)
    obs = env.reset()
    assert obs.shape == (4, 81) and env.observation_space.shape == [4, 81]
    o2, r, d, _ = env.step(np.zeros(9))
    assert o2.shape == (4, 81) and (o2[:3] == obs[1:]).all()       # history slides by one
    assert r.shape == (9,)
    # Localize: own reward counted local_weight times
    base_r = env.unwrapped.rewards.copy()
    want = np.mean(np.diag(base_r) * 2 + base_r, axis=1) / 3
    assert np.allclose(r, want)
    np.random.seed(5)
    single = make_env(seed=2, light_iterations=10, squish_rewards=True, single_agent=True)
    single.reset()
    o, r, d, _ = single.step(5)                                     # Discrete(9) index (UnGSpaceWrapper semantics)
    assert list(single.unwrapped.current_phase) == [1] * 9          # a one-element action broadcasts, as in the reference
    assert np.isscalar(r) or np.ndim(r) == 0
    assert single.action_space.n == 9
    from tests.support import run_baselines as run
    for trainer in ("fixed", "greedy", "random", "const0", "const1"):
        mean = run.main(["--trainer", trainer, "--episodes", "2", "--episode_secs", "100"])
        assert np.isfinite(mean)


def test_random_entry_sides(dropin):
    """FLAGS.entry == 'random' (traffic_env.py:390): the open sides change with reset_entrypoints()."""
    gym, GridRoad, FLAGS = dropin
    FLAGS.entry = "random"
    try:
        np.random.seed(11)
        u = new_env(gym, GridRoad, seed=3)
        seen = set()
        for _ in range(4):
            u.reset_entrypoints()
            u.reset()
            for _ in range(30):
                u.step(np.zeros(9))
            seen.add(tuple(u.graph.entrypoints))
            counts = u.cars_on_roads()
            assert counts.sum() >= 0
        assert len(seen) >= 2
    finally:
        FLAGS.entry = "all"


def test_random_entry_matches_reference_recording(dropin):
    """FLAGS.entry == 'random' across four episodes, against a recording of the unmodified reference
    (tests/golden/entry_random_3x3.npz): the open sides are re-drawn by reset_entrypoints() while the arrival
    generator carries on - the drop-in must make the same arrivals and reach the same state on every tick."""
    gym, GridRoad, FLAGS = dropin
    g = np.load(os.path.join(GOLDEN, "entry_random_3x3.npz"))
    FLAGS.entry, FLAGS.local_cars_per_sec = "random", 0.3
    try:
        np.random.seed(2)
        u = new_env(gym, GridRoad, seed=21)
        T = int(g["ticks_per_episode"])
        eoff = np.concatenate([[0], np.cumsum(g["entry_sizes"])])
        i = 0
        for ep in range(int(g["episodes"])):
            u.reset_entrypoints()
            assert list(u.graph.entrypoints) == list(g["entries"][eoff[ep]:eoff[ep + 1]])
            u.reset()
            assert (u.current_phase == g["init_phases"][ep]).all()
            for t in range(T):
                obs, rew, done, _ = u.step(g["actions"][i].astype(np.int32))
                if t % 10 == 9 or t < 3:
                    u.sync_counters()
                    st = u._snapshot()
                    xs, vs = live_walk(st["leading"][0], st["lastcar"][0], st["x"][0], st["v"][0])
                    d = tick_digest(st["leading"][0], st["lastcar"][0], obs, u.waiting, u.passed_dst, rew, done, xs, vs)
                    assert d == g["digests"][i], "episode %d tick %d" % (ep, t)
                assert done == bool(g["dones"][i])
                i += 1
    finally:
        FLAGS.entry, FLAGS.local_cars_per_sec = "all", 0.12


@pytest.mark.parametrize("learn_switch", [False, True])
def test_fused_step_host_mirror_equals_device_state(dropin, learn_switch):
    """The fused Repeater step refreshes the caller-visible int32 obs (detected | phase | elapsed) from closed
    forms on the host when no ring overflowed; with TRAFFIC_B200_NO_HOST_MIRROR it reads the device state back
    instead.  Both must agree at every step, including steps that overflow and resets in between."""
    gym, GridRoad, FLAGS = dropin
    from traffic_env_b200.wrappers import Remi, Repeater
    old_ls, old_rate = FLAGS.learn_switch, FLAGS.local_cars_per_sec
    FLAGS.learn_switch, FLAGS.local_cars_per_sec = learn_switch, 0.35   # heavy arrivals: some steps overflow
    try:
        def run(mirror_off):
            if mirror_off:
                os.environ["TRAFFIC_B200_NO_HOST_MIRROR"] = "1"
            try:
                np.random.seed(4)
                base = new_env(gym, GridRoad, seed=21)
                env = Remi(Repeater(10)(base))
                rng = np.random.RandomState(8)
                out = []
                env.reset()
                for s in range(150):
                    a = rng.randint(2, size=9) if s % 4 else rng.rand(9) < 0.5
                    obs, rew, done, _ = env.step(a)
                    out.append((obs.copy(), rew.copy(), done, base.obs.copy(), float(base.steps)))
                    if done:
                        env.reset()
                return out
            finally:
                os.environ.pop("TRAFFIC_B200_NO_HOST_MIRROR", None)
        fast, slow = run(False), run(True)
        assert any(d for _, _, d, _, _ in fast) and not all(d for _, _, d, _, _ in fast)
        for s, (f, g) in enumerate(zip(fast, slow)):
            assert f[0].tobytes() == g[0].tobytes() and f[1].tobytes() == g[1].tobytes() and f[2] == g[2], s
            assert (f[3] == g[3]).all() and f[4] == g[4], s
    finally:
        FLAGS.learn_switch, FLAGS.local_cars_per_sec = old_ls, old_rate
