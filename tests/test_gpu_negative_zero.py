"""GPU: a car at x = -0 is not tame.  The tame kernels move a car whose step dx is <= 0 by keeping its x, where the
reference adds gate * dx = +-0; the two differ only at x = -0 (-0 + +0 = +0).  The dynamics never produce -0, so such a
car can only come from te_set_state, a snapshot record or an archetype with x_new = -0, and each of them must move the
handle to the checked kernels, whose ticks then match the oracle bit for bit."""
import numpy as np
import pytest

from oracle.oracle import OracleEnv
from tests.golden_util import live_walk
from tests.test_gpu_fuzz_state import load_oracle, random_env_state

pytestmark = pytest.mark.gpu

STATE_KEYS = ("leading", "lastcar", "x", "v", "obs", "waiting", "passed_dst")


def negative_zero_cars(states, rng, R):
    """x = -0 (bits 0x80000000) for the front car of a few roads of every other env; returns how many"""
    n = 0
    for st in states[::2]:
        for rd in rng.choice(R, size=min(R, 4), replace=False):
            ld, lc = int(st["leading"][rd]), int(st["lastcar"][rd])
            if ld == lc:
                continue
            sl = 1 if ld + 1 >= 20 else ld + 1
            st["x"][rd, sl] = np.float32(-0.0)
            st["v"][rd, sl] = np.float32(0.0)
            n += 1
    return n


def run_against_oracle(env, rng, m, n, L, E, T, start):
    R, I = env.roads, env.intersections
    scheds = [[list(rng.choice(env.entrypoints, size=rng.randint(0, 3))) for _ in range(T)] for _ in range(E)]
    env.set_arrivals(scheds, first_tick=0)
    oracles = []
    for e in range(E):
        o = OracleEnv(m, n, L, 0.5)
        load_oracle(o, {k: start[k][e] for k in STATE_KEYS})
        oracles.append(o)
    for t in range(T):
        act = rng.randint(0, 2, size=(E, I))
        obs, rew, done = env.step_raw(act)
        st = env.get_state()
        for e, o in enumerate(oracles):
            od = o.step(act[e], scheds[e][t])
            tag = "env %d tick %d" % (e, t)
            assert (st["leading"][e] == o.leading).all() and (st["lastcar"][e] == o.lastcar).all(), tag + " rings"
            assert (obs[e] == o.obs).all(), tag + " obs"
            assert rew[e].tobytes() == o.rewards.tobytes(), tag + " rewards"
            assert bool(done[e]) == od, tag + " done"
            gx, gv = live_walk(st["leading"][e], st["lastcar"][e], st["x"][e], st["v"][e])
            ox, ov = o.live_state()
            assert gx.tobytes() == ox.tobytes() and gv.tobytes() == ov.tobytes(), tag + " car state"


@pytest.mark.parametrize("m,n,L,E", [(3, 3, 250.0, 20), (10, 10, 120.0, 4)])
def test_negative_zero_car_through_set_state_leaves_tame_mode(m, n, L, E):
    from traffic_env_b200 import VecTrafficEnv
    rng = np.random.RandomState(11 * m + n)
    env = VecTrafficEnv(m=m, n=n, length=L, num_envs=E, arrivals="injected", remi=False)
    R, r, I = env.roads, env.train_roads, env.intersections
    assert env.is_tame()
    states = [random_env_state(rng, R, r, I, L, True) for _ in range(E)]
    assert negative_zero_cars(states, rng, R) > 0
    env.set_state({k: np.stack([s[k] for s in states]) for k in states[0]} | {"steps": np.zeros(E, np.float32)})
    assert not env.is_tame()
    st0 = env.get_state()
    run_against_oracle(env, rng, m, n, L, E, 5, st0)


@pytest.mark.parametrize("m,n,L,E", [(3, 3, 250.0, 12), (10, 10, 120.0, 3)])
def test_negative_zero_car_in_a_record_leaves_tame_mode(m, n, L, E):
    from traffic_env_b200 import VecTrafficEnv
    rng = np.random.RandomState(13 * m + n)
    env = VecTrafficEnv(m=m, n=n, length=L, num_envs=E, arrivals="injected", remi=False)
    R, r, I = env.roads, env.train_roads, env.intersections
    states = [random_env_state(rng, R, r, I, L, True) for _ in range(E)]
    env.set_state({k: np.stack([s[k] for s in states]) for k in states[0]} | {"steps": np.zeros(E, np.float32)})
    assert env.is_tame()
    rec = env.save_envs()
    lay = env.snapshot_layout
    nz = 0
    for e in range(0, E, 2):
        xv = rec[e, lay.x:lay.x + R * 80].view(np.uint32).reshape(R, 20)
        vv = rec[e, lay.v:lay.v + R * 80].view(np.float32).reshape(R, 20)
        for rd in range(R):
            ld, lc = int(xv[rd, 0] & 0xff), int((xv[rd, 0] >> 8) & 0xff)
            if ld != lc:
                sl = 1 if ld + 1 >= 20 else ld + 1
                xv[rd, sl] = 0x80000000
                vv[rd, sl] = 0.0
                nz += 1
                break
    assert nz > 0
    env.load_envs(rec)
    assert not env.is_tame()
    st0 = env.get_state()
    run_against_oracle(env, rng, m, n, L, E, 5, st0)


def test_negative_zero_entry_position_is_not_a_tame_archetype():
    from traffic_env_b200 import ARCHETYPE, VecTrafficEnv
    assert VecTrafficEnv(m=3, n=3, num_envs=4, arrivals="injected").is_tame()
    arch = ARCHETYPE.copy()
    arch[0] = np.float32(-0.0)
    assert not VecTrafficEnv(m=3, n=3, num_envs=4, arrivals="injected", archetype=arch).is_tame()
