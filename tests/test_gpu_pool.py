"""GPU: config 5 - learner-style rollout loops (a3c.epoch contract, a3c.py:52-63) from several Python threads, each on
its own single-env proxy (traffic_env_b200.pool.EnvPool), the device stepping whichever slots have an action ready with
one masked launch.  Every slot's trajectory is checked against the CPU oracle with the slot's Philox key."""
import threading
import time

import numpy as np
import pytest

from oracle.oracle import OracleEnv

pytestmark = pytest.mark.gpu

KW = dict(m=3, n=3, length=250.0, arrivals="philox", local_cars_per_sec=0.3, ticks_per_step=10)


def rollout(env, slot, seed, steps, out, delay=0.0, k_ticks=10):
    """a3c.epoch restated: obs = env.reset(); y = policy(obs); new_obs, reward, done, _ = env.step(y) - with every
    observation / reward / done compared, on the spot, with an OracleEnv driven by the same actions (k_ticks: the pool's
    ticks per actor step)."""
    from traffic_env_b200.arrivals import gap_cdf
    rng = np.random.RandomState(100 + slot)
    w = rng.standard_normal((env.observation_space.size, env.action_space.size)).astype(np.float32)
    o = OracleEnv(3, 3, 250.0, 0.5)
    o.philox_seed(seed, slot, gap_cdf(KW["local_cars_per_sec"] * 3 * 4 * 0.5))

    def reset():
        ph, first = rng.randint(2, size=9), rng.randint(2, size=9)
        obs = env.reset(init_phase=ph, first_action=first)
        o.reset(ph)
        oo, _, _ = o.actor_step_philox(first, k_ticks, use_remi=True)
        assert obs.tobytes() == oo.tobytes(), "slot %d: reset observation" % slot
        return obs
    try:
        obs = reset()
        n_done = 0
        for t in range(steps):
            y = (obs @ w) < 0                      # bool vector, like tf.less in algorithms/util.py:114
            new_obs, reward, done, _ = env.step(y)
            oo, orw, od = o.actor_step_philox(y, k_ticks, use_remi=True)
            assert new_obs.tobytes() == oo.tobytes() and reward.tobytes() == orw.tobytes() and done == od, \
                "slot %d diverges from the oracle at step %d" % (slot, t)
            assert new_obs.shape == (81,) and new_obs.dtype == np.float32 and reward.shape == (9,) and y.dtype == np.bool_
            obs = new_obs
            if done:
                n_done += 1
                obs = reset()
            if delay:
                time.sleep(delay)
        out[slot] = ("ok", time.perf_counter(), n_done)
    except BaseException as ex:  # surfaced by the main thread
        out[slot] = ("fail", repr(ex), 0)
    finally:
        env.close()


def run_pool(T, steps, seed, delays=None, k_ticks=10):
    from traffic_env_b200.pool import EnvPool
    pool = EnvPool(T, seed=seed, **dict(KW, ticks_per_step=k_ticks))
    out = {}
    threads = [threading.Thread(target=rollout, args=(pool.slot(i), i, seed, steps[i], out, (delays or {}).get(i, 0.0),
                                                      k_ticks))
               for i in range(T)]
    t0 = time.perf_counter()
    for th in threads:
        th.start()
    for th in threads:
        th.join(timeout=180)
        assert not th.is_alive()
    for i in range(T):
        assert out[i][0] == "ok", out[i]
    return pool, out, t0


def test_every_slot_matches_the_oracle_from_threads():
    T, S = 8, 60
    pool, out, _ = run_pool(T, [S] * T, seed=3)
    # ready slots share launches: fewer launches than single-env steps, every step served
    assert pool.stepped >= T * S and pool.launches <= pool.stepped
    assert pool.vec.stats()["actor_steps"] == pool.stepped


def test_every_slot_matches_the_oracle_on_the_float_route():
    """20 ticks per actor step: too long for a wire record, so the pool's masked launches take the float route, which
    must write no row of a slot it did not step (other slots' threads read theirs meanwhile)."""
    T, S = 8, 60
    pool, out, _ = run_pool(T, [S] * T, seed=3, k_ticks=20)
    assert pool.stepped >= T * S and pool.launches <= pool.stepped
    assert pool.vec.stats()["actor_steps"] == pool.stepped


def test_a_slow_learner_only_delays_itself():
    """No lock-step round: seven fast threads finish their rollouts while the slow one (a learner busy with its
    gradient step, a3c.py:129-137) has barely started; all eight trajectories still match the oracle."""
    T = 8
    steps = [400] * T
    steps[5] = 6
    pool, out, t0 = run_pool(T, steps, seed=9, delays={5: 0.25})
    fast_done = max(out[i][1] for i in range(T) if i != 5) - t0
    slow_done = out[5][1] - t0
    assert slow_done > 1.4
    assert fast_done < slow_done - 0.3, (fast_done, slow_done)


def test_heavy_traffic_resets_inside_rollouts():
    """Dense arrivals: rings overflow, slots reset at different times (masked resets next to masked steps)."""
    from traffic_env_b200.pool import EnvPool
    global KW
    old = dict(KW)
    KW["local_cars_per_sec"] = 0.9
    try:
        T, S = 6, 80
        pool, out, _ = run_pool(T, [S] * T, seed=5)
        assert sum(out[i][2] for i in range(T)) > 0, "the test is meant to see episodes end on overflow"
    finally:
        KW.clear()
        KW.update(old)
