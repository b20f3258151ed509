"""GPU: the per-env episode clock `steps` past 2^24.

The reference adds 1 to an np.float32 clock once per tick (traffic_env.py:247; float32 under NumPy 2), so the clock stops
at 2^24 = 16777216, a clock of 2^22 or more with a fractional part rounds at every tick, and a negative clock below -2^24
stops too.  Birth ticks (validate mode) are the clock at the start of the car's tick, and a trip time is (clock - birth)
/ 2.  Every entry point that advances the clock is compared here with the oracle, bit for bit, from start clocks on both
sides of those limits."""
import numpy as np
import pytest

from oracle.oracle import OracleEnv
from tests.golden_util import live_walk
from tests.test_gpu_fuzz_state import variant_of
from tests.test_gpu_hardening import ARCH_ODD

pytestmark = pytest.mark.gpu

SEED = 29
HANDLES = {   # Philox arrivals with remi; one handle per kernel kind
    "3x3_grouped96": dict(m=3, n=3, length=250.0, E=6, lcps=0.5, variant=("grouped", 96)),   # two envs per CTA
    "10x10_tame512": dict(m=10, n=10, length=500.0, E=2, lcps=0.15, variant=("tame", 512)),
    "7x7_checked256": dict(m=7, n=7, length=200.0, E=2, lcps=0.4, rate=0.4, archetype=ARCH_ODD, variant=("checked", 256)),
    "3x3_validate256": dict(m=3, n=3, length=80.0, E=3, lcps=0.3, validate=True, variant=("validate", 256)),
    "10x10_validate512": dict(m=10, n=10, length=50.0, E=2, lcps=0.2, validate=True, variant=("validate", 512)),
}
# start clocks: even envs start at the row's clock, odd envs at its negation (so envs sharing a CTA have different clocks)
CLOCKS = {"0": 0.0, "1.5": 1.5, "2^24-37": 2.0 ** 24 - 37, "2^24-1": 2.0 ** 24 - 1, "2^24": 2.0 ** 24, "2^24+2": 2.0 ** 24 + 2,
          "2^25-4": 2.0 ** 25 - 4, "2^23-4.5": 2.0 ** 23 - 4.5, "-2^24-10": -2.0 ** 24 - 10, "3e38": 3e38}


def make_handle(h, clock):
    from traffic_env_b200 import VecTrafficEnv
    from traffic_env_b200.arrivals import gap_cdf
    m, n, L, E, rate = h["m"], h["n"], h["length"], h["E"], h.get("rate", 0.5)
    kw = dict(archetype=np.asarray(h["archetype"], np.float32)) if "archetype" in h else {}
    env = VecTrafficEnv(m=m, n=n, length=L, num_envs=E, rate=rate, arrivals="philox", seed=SEED,
                        local_cars_per_sec=h["lcps"], ticks_per_step=10, remi=True, validate=h.get("validate", False), **kw)
    assert variant_of(env) == h["variant"]
    init = np.random.RandomState(E).randint(2, size=(E, m * n))
    env.reset(init_phase=init)
    clocks = np.where(np.arange(E) % 2 == 0, np.float32(clock), -np.float32(clock)).astype(np.float32)
    st = env.get_state()
    st["steps"] = clocks
    env.set_state(st)
    assert env.get_state()["steps"].tobytes() == clocks.tobytes()
    cdf = gap_cdf(env.cars_per_sec * rate)
    oracles = []
    for e in range(E):
        o = OracleEnv(m, n, L, rate, validate=h.get("validate", False))
        if "archetype" in h:
            o.set_archetype(np.asarray(h["archetype"], np.float32))
        o.reset(init[e])
        o.philox_seed(SEED, e, cdf)
        o.steps = clocks[e]
        oracles.append(o)
    return env, oracles


def assert_clocks(env, oracles, tag):
    got = env.get_state()["steps"]
    for e, o in enumerate(oracles):
        assert got[e:e + 1].tobytes() == np.float32(o.steps).tobytes(), "%s: env %d clock %r, oracle %r" % (
            tag, e, float(got[e]), float(o.steps))


def assert_final_state(env, oracles):
    st = env.get_state()
    for e, o in enumerate(oracles):
        assert (st["leading"][e] == o.leading).all() and (st["lastcar"][e] == o.lastcar).all(), e
        gx, gv = live_walk(st["leading"][e], st["lastcar"][e], st["x"][e], st["v"][e])
        ox, ov = o.live_state()
        assert gx.tobytes() == ox.tobytes() and gv.tobytes() == ov.tobytes(), e


@pytest.mark.parametrize("clock", list(CLOCKS.values()), ids=list(CLOCKS))
@pytest.mark.parametrize("handle", list(HANDLES))
def test_clock_on_every_entry_point_vs_oracle(handle, clock):
    """Fused steps of 10, 7 and 20 ticks (20: the float route), a six-step greedy launch with a second decision inside
    it, a masked step over half the envs, a wire step and a raw tick, twice over: after every call the clock of every
    env equals the oracle's bit for bit, as do the observation, reward and done of the envs stepped."""
    h = HANDLES[handle]
    env, oracles = make_handle(h, clock)
    E, I, K = h["E"], h["m"] * h["n"], 10
    rng = np.random.RandomState(7)
    multi_done = 0

    def fused(obs, rew, done, e, act_e, k, tag):
        oo, orw, od = oracles[e].actor_step_philox(np.asarray(act_e, np.int32), k, use_remi=True)
        assert obs[e].tobytes() == oo.tobytes() and rew[e].tobytes() == orw.tobytes() and bool(done[e]) == od, (tag, e)

    for rnd in range(2):
        act = rng.randint(2, size=(E, I)).astype(np.uint8)
        for k in (10, 7, 20):
            obs, rew, done = env.step(act, k=k)
            for e in range(E):
                fused(obs, rew, done, e, act[e], k, "step k=%d round %d" % (k, rnd))
            assert_clocks(env, oracles, "step k=%d round %d" % (k, rnd))
        acts, obs6, rew6, done6 = env.step_multi(6, controller="greedy", spacing=3)
        for j in range(6):
            for e, o in enumerate(oracles):
                a = acts[j // 3, e]
                if j % 3 == 0:   # the device controller == greedy.py:14-16 on the oracle's counts at that moment
                    assert (a == (o.cars_on_roads().reshape(-1, 4).dot([1, 1, -1, -1]) < 0)).all(), (rnd, j, e)
                fused(obs6[j], rew6[j], done6[j], e, a, K, "step_multi actor step %d round %d" % (j, rnd))
            multi_done += int(done6[j].sum()) if j < 5 else 0
        assert_clocks(env, oracles, "step_multi round %d" % rnd)
        mask = np.arange(E) % 2 == rnd % 2
        obs, rew, done = env.step_masked(act, mask)
        for e in np.nonzero(mask)[0]:
            fused(obs, rew, done, e, act[e], K, "step_masked round %d" % rnd)
        assert_clocks(env, oracles, "step_masked round %d" % rnd)
        env.step_wire(act)
        obs, rew, done = env.expand_wire()
        for e in range(E):
            fused(obs, rew, done, e, act[e], K, "step_wire round %d" % rnd)
        assert_clocks(env, oracles, "step_wire round %d" % rnd)
        obs, rew, done = env.step_raw(act)
        for e, o in enumerate(oracles):
            od = o.step(act[e], o.philox_arrivals())
            assert (obs[e] == o.obs).all() and rew[e].tobytes() == o.rewards.tobytes() and bool(done[e]) == od, (rnd, e)
        assert_clocks(env, oracles, "step_raw round %d" % rnd)
    assert_final_state(env, oracles)
    assert multi_done > 0, "the test is meant to stop envs inside a multi-step launch (overflow break)"
    if h.get("validate"):
        envs, trips = env.trip_times()
        total = 0
        for e, o in enumerate(oracles):
            want = o.trip_times()
            assert np.asarray(trips[envs == e], np.float64).tobytes() == want.tobytes(), e
            total += len(want)
        assert total > 0


def birth_ticks(env, oracles):
    """(device, oracle) birth ticks of every live car, road by road in ring order: the w plane of the snapshot records
    and the oracle's state[road, 9, slot]."""
    lay = env.snapshot_layout
    rec = env.save_envs()
    st = env.get_state()
    R = env.roads
    out = []
    for e, o in enumerate(oracles):
        w = rec[e, lay.w:lay.w + R * 20 * 4].view(np.float32).reshape(R, 20)
        gw, _ = live_walk(st["leading"][e], st["lastcar"][e], w, w)
        ow, _ = live_walk(o.leading, o.lastcar, o.state[:, 9, :], o.state[:, 9, :])
        out.append((gw, ow))
    return out


@pytest.mark.parametrize("m,n,L,E,lcps,S", [(3, 3, 250.0, 3, 0.12, 60), (10, 10, 100.0, 2, 0.08, 60)])
def test_validate_trips_across_the_clock_limit(m, n, L, E, lcps, S):
    """Validate mode from 2^24 - 150: cars born before the clock stops and after it leave the map.  Trip times (per env,
    in order) and the birth tick of every live car equal the oracle's bit for bit; the cars born after the clock stopped
    leave with a trip time of exactly 0."""
    from traffic_env_b200 import VecTrafficEnv
    from traffic_env_b200.arrivals import gap_cdf
    start = np.float32(2 ** 24 - 150)
    env = VecTrafficEnv(m=m, n=n, length=L, num_envs=E, arrivals="philox", seed=SEED, local_cars_per_sec=lcps,
                        ticks_per_step=10, remi=True, validate=True)
    init = np.random.RandomState(3).randint(2, size=(E, m * n))
    env.reset(init_phase=init)
    st = env.get_state()
    st["steps"][:] = start
    env.set_state(st)
    cdf = gap_cdf(env.cars_per_sec * 0.5)
    oracles = []
    for e in range(E):
        o = OracleEnv(m, n, L, 0.5, validate=True)
        o.reset(init[e])
        o.philox_seed(SEED, e, cdf)
        o.steps = start
        oracles.append(o)
    rng = np.random.RandomState(11)
    got = [[] for _ in range(E)]
    for s in range(S):
        if s % 3 == 0:
            act = rng.randint(2, size=(E, m * n))
        obs, rew, done = env.step(act)
        for e, o in enumerate(oracles):
            oo, orw, od = o.actor_step_philox(act[e], 10, use_remi=True)
            assert obs[e].tobytes() == oo.tobytes() and rew[e].tobytes() == orw.tobytes() and bool(done[e]) == od, (s, e)
        envs, trips = env.trip_times(clear=True)
        for e in range(E):
            got[e].extend(trips[envs == e])
        if s % 10 == 9:
            for e, (gw, ow) in enumerate(birth_ticks(env, oracles)):
                assert gw.tobytes() == ow.tobytes(), "step %d env %d: birth ticks %s, oracle %s" % (s, e, gw[:8], ow[:8])
    assert_clocks(env, oracles, "end")
    assert_final_state(env, oracles)
    alltrips = []
    for e, o in enumerate(oracles):
        want = o.trip_times()
        assert np.asarray(got[e], np.float64).tobytes() == want.tobytes(), e
        alltrips.extend(want)
    alltrips = np.asarray(alltrips)
    assert (alltrips == 0.0).any(), "cars born after the clock stopped are meant to leave the map"
    assert (alltrips > 0.0).any()
    assert float(oracles[0].steps) == 2.0 ** 24
