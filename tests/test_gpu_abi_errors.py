"""GPU: error behaviour of the C ABI - bad arguments are reported through the return code and te_last_error(),
simulation overflow is data."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def test_argument_errors_are_reported():
    from traffic_env_b200 import TrafficB200Error, VecTrafficEnv
    env = VecTrafficEnv(m=3, n=3, num_envs=4, arrivals="injected")
    with pytest.raises(TrafficB200Error, match="no arrival schedule"):
        env.step(np.zeros((4, 9)))
    with pytest.raises(TrafficB200Error, match="not an entry road"):
        env.set_arrivals([[[1]], [[]], [[]], [[]]])          # road 1 is interior
    env.set_arrivals([[[0, 3]], [[]], [[]], [[]]])
    with pytest.raises(TrafficB200Error, match="k_ticks"):
        env.step(np.zeros((4, 9)), k=65)
    with pytest.raises(TrafficB200Error, match="out of bounds"):
        env.get_state(2, 3)
    before = env.save_envs()
    st = env.get_state()
    st["leading"][3, 0] = 0                                  # the last env only: the earlier ones are not written either
    with pytest.raises(TrafficB200Error, match="ring index"):
        env.set_state(st)
    assert env.save_envs().tobytes() == before.tobytes()
    st = env.get_state()
    st["obs"][3, env.train_roads] = 256                      # detected of road 0: one byte of the row header
    with pytest.raises(TrafficB200Error, match="detected"):
        env.set_state(st)
    assert env.save_envs().tobytes() == before.tobytes()
    st = env.get_state()
    st["passed_dst"][1, 2] = 2
    env.set_state(st)
    assert env.get_state()["passed_dst"][1, 2] == 1
    with pytest.raises(TrafficB200Error, match="TE_VALIDATE"):
        env.trip_times()
    obs, rew, done = env.step(np.zeros((4, 9)))              # still usable after the errors
    assert obs.shape == (4, 81) and not done.any()
    with pytest.raises(TrafficB200Error, match="exceed one CTA|shared memory"):
        VecTrafficEnv(m=20, n=20, num_envs=1)
    with pytest.raises(TrafficB200Error, match="Philox arrivals need"):
        VecTrafficEnv(m=3, n=3, num_envs=1, entry=0b1111)     # every side closed: nowhere to arrive


def test_overflow_is_data_not_an_error():
    from traffic_env_b200 import VecTrafficEnv
    env = VecTrafficEnv(m=1, n=1, length=60.0, num_envs=2, arrivals="injected", remi=False)
    sched = [[[0, 0, 0]] * 40, [[]] * 40]                     # env 0: three cars per tick on one entry road
    env.set_arrivals(sched)
    env.reset(init_phase=np.ones((2, 1)))
    saw = False
    for t in range(12):
        obs, rew, done = env.step_raw(np.ones((2, 1)))         # phase 1 == E/W roads red
        if done[0]:
            saw = True
            assert rew[0, 0] <= -10.0 and rew[0, 0] % 10 == 0
        assert not done[1] and rew[1, 0] == 0.0
    assert saw and env.stats()["overflows"] > 0


def test_two_handles_from_two_threads():
    """Handles are independent (a3c.py:69-72 steps its envs from several Python threads)."""
    import threading
    from traffic_env_b200 import VecTrafficEnv
    outs = {}

    def work(seed):
        env = VecTrafficEnv(m=3, n=3, num_envs=16, arrivals="philox", seed=seed)
        env.reset(init_phase=np.zeros((16, 9)))
        tot = 0.0
        for s in range(30):
            obs, rew, done = env.step(np.full((16, 9), s % 2))
            tot += float(obs.sum())
        outs[seed] = (tot, env.stats()["vehicle_updates"])

    ths = [threading.Thread(target=work, args=(s,)) for s in (1, 2, 1)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    work(1)
    ref1 = outs[1]
    work(2)
    assert outs[2][1] > 0 and outs[1] == ref1   # same seed, same result, regardless of concurrent handles
