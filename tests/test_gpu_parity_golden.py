"""GPU: the CUDA path against the reference's golden vectors and against the oracle, tick by tick.

Integer state (ring indices, car counts, passed/detected/waiting, light phases, done) and the
float state (x, v of every live car) are compared BIT-EXACT: the device reproduces numba's
float/double operation mix and glibc's powf (see traffic_env_b200/csrc/te_math.cuh)."""
import glob
import os

import numpy as np
import pytest

from tests.golden_util import live_walk, tick_digest, unpack_schedule

pytestmark = pytest.mark.gpu

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RAW = sorted(p for p in glob.glob(os.path.join(GOLDEN, "*.npz")) if str(np.load(p)["kind"]) == "raw")
WRAPPED = sorted(p for p in glob.glob(os.path.join(GOLDEN, "*.npz")) if str(np.load(p)["kind"]) == "wrapped")


def make_env(g, num_envs=1, **kw):
    from traffic_env_b200 import VecTrafficEnv
    return VecTrafficEnv(m=int(g["m"]), n=int(g["n"]), length=float(g["length"]), rate=float(g["rate"]),
                         num_envs=num_envs, arrivals="injected",
                         learn_switch=bool(g["learn_switch"]) if "learn_switch" in g else False,
                         entry=int(g["entry_spec"]) if "entry_spec" in g else "all", **kw)


@pytest.mark.parametrize("path", RAW, ids=[os.path.basename(p)[:-4] for p in RAW])
def test_raw_ticks_bit_exact(path):
    """te_step_raw == bare TrafficEnv._step, every tick, including ticks after an overflow."""
    g = np.load(path)
    env = make_env(g, remi=False)
    assert (env.entrypoints == g["entrypoints"]).all()
    sched = unpack_schedule(g["sched_off"], g["sched_roads"])
    env.set_arrivals([sched])
    env.reset(init_phase=g["init_phase"][None])
    T = int(g["ticks"])
    for t in range(T):
        obs, rew, done = env.step_raw(g["actions"][t][None])
        st = env.get_state(0, 1)
        xs, vs = live_walk(st["leading"][0], st["lastcar"][0], st["x"][0], st["v"][0])
        d = tick_digest(st["leading"][0], st["lastcar"][0], obs[0], st["waiting"][0], st["passed_dst"][0],
                        rew[0], done[0], xs, vs)
        if d != g["digests"][t]:
            key = "ck%d_x" % (t + 1)
            detail = ""
            if key in g:
                detail = " max|dx|=%g" % np.abs(xs - g[key]).max() if xs.shape == g[key].shape else " live count differs"
            pytest.fail("first divergent tick %d of %s%s (done %d vs %d)" % (t, os.path.basename(path), detail,
                                                                         done[0], g["dones"][t]))
    stats = env.stats()
    assert stats["cars_generated"] == int(g["generated"][-1])
    assert stats["ticks"] == T


@pytest.mark.parametrize("path", WRAPPED, ids=[os.path.basename(p)[:-4] for p in WRAPPED])
def test_fused_actor_steps_bit_exact(path):
    """te_step(K) == Remi(Repeater(K)) of traffic_test.py for a batch of envs in one launch."""
    g = np.load(path)
    K, S, E = int(g["K"]), int(g["actor_steps"]), int(g["n_envs"])
    env = make_env(g, num_envs=E, remi=True, ticks_per_step=K)
    scheds = []
    for e in range(E):
        lo, hi = g["sched_roads_off"][e], g["sched_roads_off"][e + 1]
        scheds.append(unpack_schedule(g["sched_off"][e], g["sched_roads"][lo:hi]))
    env.set_arrivals(scheds)
    env.reset(init_phase=g["init_phase"])
    for s in range(S):
        obs, rew, done = env.step(g["actions"][s])
        assert obs.tobytes() == g["obs"][:, s].tobytes(), "obs differ at actor step %d" % s
        assert rew.tobytes() == g["reward"][:, s].tobytes(), "reward differs at actor step %d" % s
        assert (done == g["done"][:, s]).all(), "done differs at actor step %d" % s
    st = env.get_state()
    for e in range(E):
        xs, vs = live_walk(st["leading"][e], st["lastcar"][e], st["x"][e], st["v"][e])
        assert xs.tobytes() == g["fin%d_x" % e].tobytes() and vs.tobytes() == g["fin%d_v" % e].tobytes()
        assert (st["leading"][e] == g["fin%d_leading" % e]).all() and (st["lastcar"][e] == g["fin%d_lastcar" % e]).all()
        r, I = env.train_roads, env.intersections
        assert (st["obs"][e][r:] == g["fin%d_obs" % e][r:]).all()  # detected | phase | elapsed


def test_raw_and_fused_agree():
    """K raw ticks + remi_reward == one fused actor step, on the same schedule."""
    g = np.load(os.path.join(GOLDEN, "wrapped_3x3_cfg2.npz"))
    K, E = int(g["K"]), int(g["n_envs"])
    scheds = []
    for e in range(E):
        lo, hi = g["sched_roads_off"][e], g["sched_roads_off"][e + 1]
        scheds.append(unpack_schedule(g["sched_off"][e], g["sched_roads"][lo:hi]))
    a = make_env(g, num_envs=E, remi=True, ticks_per_step=K)
    b = make_env(g, num_envs=E, remi=False)
    for env in (a, b):
        env.set_arrivals(scheds)
        env.reset(init_phase=g["init_phase"])
    for s in range(6):  # the first steps never overflow in this fixture
        obs, rew, done = a.step(g["actions"][s])
        assert not done.any()
        for _ in range(K):
            b.step_raw(g["actions"][s])
        rb = b.remi_reward()
        assert rew.tobytes() == rb.tobytes()
    sa, sb = a.get_state(), b.get_state()
    for k in ("leading", "lastcar", "waiting", "passed_dst"):
        assert (sa[k] == sb[k]).all(), k


def test_validate_mode_trip_times():
    """TE_VALIDATE: per-car birth ticks travel with the cars; trip times of cars leaving the map equal the
    reference's advance_hack list (traffic_env.py:139-157), values and order."""
    g = np.load(os.path.join(GOLDEN, "validate_3x3.npz"))
    env = make_env(g, remi=False, validate=True)
    sched = unpack_schedule(g["sched_off"], g["sched_roads"])
    env.set_arrivals([sched])
    env.reset(init_phase=g["init_phase"][None])
    got = []
    for t in range(int(g["ticks"])):
        obs, rew, done = env.step_raw(g["actions"][t][None])
        if t % 97 == 0:
            got.extend(env.trip_times(clear=True)[1])
    envs, trips = env.trip_times(clear=True)
    got.extend(trips)
    want = g["trip_times"]
    assert len(want) > 50
    assert np.asarray(got, np.float64).tobytes() == want.tobytes()
    st = env.get_state(0, 1)
    assert (st["leading"][0] == g["ck600_leading"]).all()


def test_validate_mode_fused_steps_same_trips():
    """The fused K-tick launch records the same trips as K raw ticks."""
    g = np.load(os.path.join(GOLDEN, "validate_3x3.npz"))
    sched = unpack_schedule(g["sched_off"], g["sched_roads"])
    a = make_env(g, remi=False, validate=True)
    b = make_env(g, remi=False, validate=True, ticks_per_step=10)
    for env in (a, b):
        env.set_arrivals([sched])
        env.reset(init_phase=g["init_phase"][None])
    for s in range(40):
        act = g["actions"][10 * s][None]
        for _ in range(10):
            a.step_raw(act)
        _, _, done = b.step(act)
        assert not done[0]
    ta, tb = a.trip_times()[1], b.trip_times()[1]
    assert len(ta) > 20 and ta.tobytes() == tb.tobytes()


def test_fused_learn_switch_matches_raw_ticks():
    """learn_switch=True: the action toggles the phase on EVERY tick of the actor step (traffic_env.py:225-227);
    the fused launch derives phase/elapsed of the later ticks in closed form - compare with K raw ticks."""
    g = np.load(os.path.join(GOLDEN, "learnswitch_2x3.npz"))
    sched = unpack_schedule(g["sched_off"], g["sched_roads"])
    K = 7
    a = make_env(g, remi=False)
    b = make_env(g, remi=False, ticks_per_step=K)
    for env in (a, b):
        env.set_arrivals([sched])
        env.reset(init_phase=g["init_phase"][None])
    rng = np.random.RandomState(3)
    checked = 0
    for s in range(60):
        act = rng.randint(2, size=(1, 6))
        tot, done_raw, obs_passed = np.zeros(6, np.float32), False, np.zeros(24, np.float32)
        for k in range(K):
            o, r, d = a.step_raw(act)
            tot += r[0]
            obs_passed += o[0][:24]
            if d[0]:
                done_raw = True
                break
        if done_raw:
            # the raw env stopped early like Repeater does; re-align the fused env on the same number of ticks
            of, rf, df = b.step(act, k=k + 1)
        else:
            of, rf, df = b.step(act)
        assert bool(df[0]) == done_raw
        assert rf[0].tobytes() == tot.tobytes()
        assert of[0][:24].tobytes() == obs_passed.tobytes()
        sa, sb = a.get_state(), b.get_state()
        for key in ("leading", "lastcar", "waiting", "passed_dst"):
            assert (sa[key] == sb[key]).all(), (s, key)
        assert (sa["obs"][0][24:] == sb["obs"][0][24:]).all(), s   # detected | phase | elapsed
        checked += 1
    assert checked == 60


# 11x11: 544 rows in the 768-row validate kernel; 13x13 fills it (14x14 and larger are refused)
VALIDATE_ROWS = [(10, 10, 50.0, 3), (6, 5, 90.0, 4), (11, 11, 50.0, 2), (13, 13, 50.0, 2)]
VALIDATE_VARIANTS = {(10, 10): 512, (6, 5): 256, (11, 11): 768, (13, 13): 768}


@pytest.mark.parametrize("m,n,L,E", VALIDATE_ROWS)
def test_validate_mode_larger_grids_vs_oracle(m, n, L, E):
    """TE_VALIDATE on the larger kernel variants (third shared-memory plane): trip times of cars leaving the map
    and the ring state against the oracle in validate mode, injected arrivals, 320 raw ticks."""
    from oracle.oracle import OracleEnv
    from traffic_env_b200 import VecTrafficEnv
    from tests.golden_util import live_walk
    rng = np.random.RandomState(100 * m + n)
    T = 320
    env = VecTrafficEnv(m=m, n=n, length=L, num_envs=E, arrivals="injected", remi=False, validate=True)
    v = env.step_variant()
    assert (v["kind"], v["max_threads"]) == ("validate", VALIDATE_VARIANTS[(m, n)])
    I = env.intersections
    scheds = [[list(rng.choice(env.entrypoints, size=rng.poisson(1.5))) for _ in range(T)] for _ in range(E)]
    init = rng.randint(2, size=(E, I))
    env.set_arrivals(scheds)
    env.reset(init_phase=init)
    oracles = []
    for e in range(E):
        o = OracleEnv(m, n, L, 0.5, validate=True)
        o.reset(init[e])
        oracles.append(o)
    act = rng.randint(2, size=(E, I))
    for t in range(T):
        if t % 10 == 0:
            act = rng.randint(2, size=(E, I))
        obs, rew, done = env.step_raw(act)
        for e, o in enumerate(oracles):
            o.step(act[e], scheds[e][t])
            assert (obs[e] == o.obs).all(), (e, t)
    envs, trips = env.trip_times()
    st = env.get_state()
    total = 0
    for e, o in enumerate(oracles):
        want = np.asarray(o.trip_times(), np.float64)
        got = np.asarray(trips[np.asarray(envs) == e], np.float64)
        assert got.tobytes() == want.tobytes(), e
        total += len(want)
        gx, gv = live_walk(st["leading"][e], st["lastcar"][e], st["x"][e], st["v"][e])
        ox, ov = o.live_state()
        assert gx.tobytes() == ox.tobytes() and gv.tobytes() == ov.tobytes()
    assert total > 20
