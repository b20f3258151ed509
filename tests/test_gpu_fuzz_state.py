"""GPU: random ring states (wrapped rings, full rings, several cars crossing the end of a road in one
tick, collisions, stale counters) set on the device and on the oracle, stepped tick by tick, compared
bit for bit.  Exercises the parts the recorded trajectories reach rarely: ring overflow on transfer in
both road-index orders, multi-pop ticks (ordered-transfer fallback), the wrapped-ring `waiting` quirk
(traffic_env.py:210), `detected` staying stale on empty roads."""
import numpy as np
import pytest

from oracle.oracle import OracleEnv
from tests.golden_util import live_walk

pytestmark = pytest.mark.gpu

ARCH = np.array([0.0, 11.11, 4.0, 3.0, 4.0, 13.89, 6.0, 2.0, 1.0, 0.0], np.float32)
CAP = 20


def random_env_state(rng, R, r, I, L, dense):
    leading = rng.randint(1, CAP, size=R).astype(np.int32)
    n = rng.randint(0, 19, size=R) if dense else rng.choice([0, 1, 2, 5, 17, 18], size=R)
    lastcar = ((leading - 1 + n) % 19 + 1).astype(np.int32)
    x = np.full((R, CAP), np.nan, np.float32)
    v = np.full((R, CAP), np.nan, np.float32)
    for e in range(R):
        s = int(leading[e])
        x[e, s] = np.inf if e >= r else np.float32(rng.uniform(0, 2 * L))
        v[e, s] = 0.0
        pos = np.float32(rng.uniform(L - 20, L + 7) if rng.rand() < 0.7 else rng.uniform(0, L))
        for k in range(int(n[e])):
            s = 1 if s + 1 >= CAP else s + 1
            x[e, s] = pos
            v[e, s] = np.float32(0.0 if rng.rand() < 0.4 else rng.uniform(0, 15))
            gap = rng.choice([5.0, 5.5, 7.0, 3.0, 12.0, 30.0], p=[0.35, 0.2, 0.15, 0.05, 0.15, 0.1])
            pos = np.float32(pos - gap * rng.uniform(0.9, 1.1))
    obs = np.zeros(2 * r + 2 * I, np.int32)
    obs[r:2 * r] = rng.randint(0, 5, size=r)              # stale `detected`
    obs[2 * r:2 * r + I] = rng.randint(0, 2, size=I)      # phase
    obs[2 * r + I:] = rng.randint(0, 12, size=I)          # elapsed
    waiting = rng.randint(0, 3, size=r).astype(np.int32)
    passed_dst = rng.randint(0, 2, size=I).astype(np.uint8)
    return dict(leading=leading, lastcar=lastcar, x=x, v=v, obs=obs, waiting=waiting, passed_dst=passed_dst)


def load_oracle(o, st, arch=ARCH):
    """The state `st` (random_env_state) into OracleEnv `o`, whose cars have the archetype `arch` (the handle's)."""
    R = o.roads
    o.leading[:] = st["leading"]
    o.lastcar[:] = st["lastcar"]
    o.state[:] = np.nan
    for e in range(R):
        s = int(st["leading"][e])
        o.state[e, :, s] = 0.0
        o.state[e, 0, s] = st["x"][e, s]
        while s != int(st["lastcar"][e]):
            s = 1 if s + 1 >= CAP else s + 1
            o.state[e, :, s] = arch
            o.state[e, 0, s] = st["x"][e, s]
            o.state[e, 1, s] = st["v"][e, s]
    o.obs[:] = st["obs"]
    o.waiting[:] = st["waiting"]
    o.passed_dst[:] = st["passed_dst"]


FUZZ_ROWS = [
    (3, 3, 250.0, 96, True, False), (3, 3, 250.0, 96, False, False), (3, 3, 250.0, 64, True, True),
    (2, 3, 100.0, 64, True, False), (1, 1, 60.0, 32, True, False), (10, 10, 500.0, 6, True, False),
    (4, 2, 80.0, 48, False, True), (3, 2, 123.456, 64, True, False), (2, 2, 77.7, 48, True, False),
    # one grid per tame kernel variant: tame 128 / grouped 160 / tame 256 / 512 / 768 / 1024
    (5, 5, 150.0, 8, True, False), (4, 4, 90.0, 8, True, False), (7, 7, 120.0, 4, True, False),
    (10, 11, 100.0, 3, True, False), (13, 13, 100.0, 2, True, False), (15, 15, 100.0, 2, False, False),
    # tame 64 (one env per CTA: sharing a CTA would save no lanes); grouped 256 with G = 4 and a last CTA holding two
    # envs; grouped 64 with G = 3 and a last CTA holding one env
    (4, 3, 90.0, 20, True, False), (2, 5, 80.0, 30, True, False), (1, 3, 70.0, 31, True, False)]
# the step-kernel instantiation (kind, MAXT) each grid of FUZZ_ROWS runs
FUZZ_VARIANTS = {(3, 3): ("grouped", 96), (2, 3): ("grouped", 160), (1, 1): ("grouped", 64), (10, 10): ("tame", 512),
                 (4, 2): ("grouped", 96), (3, 2): ("grouped", 160), (2, 2): ("grouped", 96), (5, 5): ("tame", 128),
                 (4, 4): ("grouped", 160), (7, 7): ("tame", 256), (10, 11): ("tame", 512), (13, 13): ("tame", 768),
                 (15, 15): ("tame", 1024), (4, 3): ("tame", 64), (2, 5): ("grouped", 256), (1, 3): ("grouped", 64)}


def variant_of(env):
    v = env.step_variant()
    return v["kind"], v["max_threads"]


@pytest.mark.parametrize("m,n,L,E,dense,ordered", FUZZ_ROWS)
def test_random_states_tick_by_tick(m, n, L, E, dense, ordered):
    from traffic_env_b200 import VecTrafficEnv
    rng = np.random.RandomState(1000 * m + 10 * n + int(dense) + 2 * int(ordered))
    T = 4
    env = VecTrafficEnv(m=m, n=n, length=L, num_envs=E, arrivals="injected", remi=False, ordered_transfers=ordered)
    assert variant_of(env) == FUZZ_VARIANTS[(m, n)]
    R, r, I = env.roads, env.train_roads, env.intersections
    states = [random_env_state(rng, R, r, I, L, dense) for _ in range(E)]
    scheds = [[list(rng.choice(env.entrypoints, size=rng.randint(0, 4))) for _ in range(T)] for _ in range(E)]
    actions = rng.randint(0, 2, size=(T, E, I))
    env.set_arrivals(scheds)
    env.set_state({k: np.stack([s[k] for s in states]) for k in states[0]} | {"steps": np.zeros(E, np.float32)})
    oracles = []
    for e in range(E):
        o = OracleEnv(m, n, L, 0.5)
        load_oracle(o, states[e])
        oracles.append(o)
    # round trip of the state through the device
    st = env.get_state()
    for e in range(E):
        assert (st["leading"][e] == states[e]["leading"]).all() and (st["lastcar"][e] == states[e]["lastcar"]).all()
        a, b = live_walk(st["leading"][e], st["lastcar"][e], st["x"][e], st["v"][e])
        c, d = live_walk(states[e]["leading"], states[e]["lastcar"], states[e]["x"], states[e]["v"])
        assert a.tobytes() == c.tobytes() and b.tobytes() == d.tobytes()
    multi_pop = 0
    for t in range(T):
        obs, rew, done = env.step_raw(actions[t])
        st = env.get_state()
        for e, o in enumerate(oracles):
            before = o.leading.copy()
            od = o.step(actions[t, e], scheds[e][t])
            multi_pop += int((((o.leading - before) % 19) >= 2).sum())
            tag = "env %d tick %d" % (e, t)
            assert (st["leading"][e] == o.leading).all(), tag + " leading"
            assert (st["lastcar"][e] == o.lastcar).all(), tag + " lastcar"
            assert (obs[e] == o.obs).all(), tag + " obs"
            assert (st["waiting"][e] == o.waiting).all(), tag + " waiting"
            assert (st["passed_dst"][e] == o.passed_dst).all(), tag + " passed_dst"
            assert rew[e].tobytes() == o.rewards.tobytes(), tag + " rewards"
            assert bool(done[e]) == od, tag + " done"
            gx, gv = live_walk(st["leading"][e], st["lastcar"][e], st["x"][e], st["v"][e])
            ox, ov = o.live_state()
            assert gx.tobytes() == ox.tobytes() and gv.tobytes() == ov.tobytes(), tag + " car state"
    assert env.is_tame() and variant_of(env) == FUZZ_VARIANTS[(m, n)]
    stats = env.stats()
    assert stats["overflows"] == sum(o.overflows for o in oracles)
    assert stats["vehicle_updates"] == sum(o.vehicle_updates for o in oracles)
    if dense and m * n > 1:
        assert multi_pop > 0, "fuzz did not produce a multi-pop tick"
        if not ordered:
            assert stats["seq_fallback_ticks"] > 0, "ordered-transfer fallback never triggered"
