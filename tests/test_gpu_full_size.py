"""GPU: the headline workload at BASELINE.json's full size (16384 envs of the 10x10 grid) through
size-independent properties, plus exact replay of sampled envs on the oracle."""
import numpy as np
import pytest

from oracle.oracle import OracleEnv

pytestmark = pytest.mark.gpu

E, M, N, L, LCPS, K = 16384, 10, 10, 500.0, 0.12, 10


@pytest.fixture(scope="module")
def big():
    from traffic_env_b200 import VecTrafficEnv
    env = VecTrafficEnv(m=M, n=N, length=L, num_envs=E, arrivals="philox", seed=2026, local_cars_per_sec=LCPS,
                        ticks_per_step=K, remi=True)
    env.reset(init_phase=np.zeros((E, M * N), np.uint8))
    acts = []
    for s in range(40):
        if s % 3 == 0:
            a = env.greedy_actions().copy()
        acts.append(a)
        env.step(a)
    return env, acts


def test_car_conservation(big):
    """generated = live + exited + dropped, summed over all 16384 envs."""
    env, _ = big
    st = env.stats()
    live = int(env.cars_on_roads_flat().sum())
    assert st["cars_generated"] > 5_000_000
    assert st["cars_generated"] == live + st["cars_exited"] + st["overflows"]


def test_ring_invariants(big):
    env, _ = big
    c = env.cars_on_roads_flat()
    assert c.min() >= 0 and c.max() <= 18
    st = env.get_state(0, 256)
    assert st["leading"].min() >= 1 and st["leading"].max() <= 19
    assert st["lastcar"].min() >= 1 and st["lastcar"].max() <= 19
    # cars on a road are ordered front to back (x non-increasing along the ring) in the vast majority of roads
    bad = tot = 0
    for e in range(16):
        for rd in range(env.roads):
            s, xs = int(st["leading"][e, rd]), []
            while s != int(st["lastcar"][e, rd]):
                s = 1 if s + 1 >= 20 else s + 1
                xs.append(st["x"][e, rd, s])
            if len(xs) > 1:
                tot += 1
                bad += int((np.diff(np.asarray(xs)) > 0).any())
    assert tot > 1000 and bad == 0


def test_sampled_envs_replay_on_oracle(big):
    """12 of the 16384 envs, chosen across the batch, replayed from scratch on the CPU oracle with the same
    Philox stream and the recorded actions: final ring indices and car state bit-exact."""
    from traffic_env_b200.arrivals import gap_cdf
    from tests.golden_util import live_walk
    env, acts = big
    cdf = gap_cdf(env.cars_per_sec * 0.5)
    for e in (0, 1, 777, 4095, 4096, 8191, 9000, 12345, 16000, 16381, 16382, 16383):
        o = OracleEnv(M, N, L, 0.5)
        o.reset(np.zeros(M * N, np.int32))
        o.philox_seed(2026, e, cdf)
        for a in acts:
            o.actor_step_philox(a[e], K, use_remi=True)
        st = env.get_state(e, 1)
        assert (st["leading"][0] == o.leading).all() and (st["lastcar"][0] == o.lastcar).all(), e
        gx, gv = live_walk(st["leading"][0], st["lastcar"][0], st["x"][0], st["v"][0])
        ox, ov = o.live_state()
        assert gx.tobytes() == ox.tobytes() and gv.tobytes() == ov.tobytes(), e
        assert float(st["steps"][0]) == float(o.steps)


def test_state_round_trip_is_idempotent(big):
    env, _ = big
    ids = range(100, 164)
    rec = env.save_envs(ids)
    a = env.get_state(100, 64)
    env.set_state(a, env_begin=100)
    b = env.get_state(100, 64)
    for k in ("leading", "lastcar", "obs", "waiting", "passed_dst"):
        assert (a[k] == b[k]).all(), k
    assert env.save_envs(ids).tobytes() == rec.tobytes()
