"""GPU: snapshot records (te_save_envs / te_load_envs).  Rewind, resume on a fresh handle, gather / scatter, both
memory routes, rejection of bad records with the batch left untouched, and the tame-mode rule."""

import numpy as np
import pytest

from oracle.oracle import OracleEnv
from tests.golden_util import live_walk
from tests.test_gpu_fuzz_state import load_oracle, random_env_state

pytestmark = pytest.mark.gpu

STATE_KEYS = ("leading", "lastcar", "x", "v", "obs", "waiting", "passed_dst", "steps")


def same_state(a, b, rows_a=slice(None), rows_b=slice(None)):
    return all(a[k][rows_a].tobytes() == b[k][rows_b].tobytes() for k in STATE_KEYS)


def run_window(env, n, multi):
    """n actor steps under the greedy controller; every output as bytes."""
    out = []
    if multi:
        for _ in range(n):
            act, obs, rew, done = env.step_multi(2, controller="greedy")
            out += [act.tobytes(), obs.tobytes(), rew.tobytes(), done.tobytes()]
    else:
        for _ in range(n):
            act = env.greedy_actions()
            obs, rew, done = env.step(act)
            out += [act.tobytes(), obs.tobytes(), rew.tobytes(), done.tobytes()]
    return out


def injected_schedule(env, rng, ticks):
    return [[list(rng.choice(env.entrypoints, size=rng.randint(0, 3))) for _ in range(ticks)] for _ in range(env.num_envs)]


@pytest.mark.parametrize("name,kw,multi", [
    ("3x3", dict(m=3, n=3, num_envs=66, local_cars_per_sec=0.4), True),
    ("10x10", dict(m=10, n=10, length=500.0, num_envs=6, local_cars_per_sec=0.3), True),
    ("auto_reset", dict(m=3, n=3, num_envs=40, local_cars_per_sec=0.5, auto_reset=True, episode_len=3), False),
    ("validate", dict(m=3, n=3, num_envs=40, local_cars_per_sec=0.3, validate=True), True),
    ("learn_switch", dict(m=3, n=3, num_envs=40, local_cars_per_sec=0.4, learn_switch=True), True),
    ("injected", dict(m=3, n=3, num_envs=24, arrivals="injected"), True)])
def test_rewind_replays_bit_for_bit(name, kw, multi):
    from traffic_env_b200 import VecTrafficEnv
    env = VecTrafficEnv(seed=11, ticks_per_step=5, **kw)
    if kw.get("arrivals") == "injected":
        env.set_arrivals(injected_schedule(env, np.random.RandomState(3), 200))
    env.reset()
    run_window(env, 30, multi)                         # pre-roll (long enough for trips to end in validate mode)
    validate = kw.get("validate", False)
    if validate:
        env.trip_times(clear=True)
    rec = env.save_envs()
    ep0 = env.stats()["episodes"]
    first = run_window(env, 7, multi)
    st1, rec1 = env.get_state(), env.save_envs()
    ep1 = env.stats()["episodes"]
    trips1 = env.trip_times(clear=True) if validate else None
    env.load_envs(rec)
    assert env.save_envs().tobytes() == rec.tobytes()
    second = run_window(env, 7, multi)
    st2, rec2 = env.get_state(), env.save_envs()
    assert len(first) == len(second)
    for i, (a, b) in enumerate(zip(first, second)):
        assert a == b, "%s: output %d of the replay differs" % (name, i)
    assert same_state(st1, st2), name + ": final state"
    assert rec1.tobytes() == rec2.tobytes(), name + ": final records (return statistics, arrival stream, clocks)"
    if kw.get("auto_reset"):
        assert ep1 - ep0 > 0 and env.stats()["episodes"] - ep1 == ep1 - ep0, "same reset points"
    if validate:
        trips2 = env.trip_times(clear=True)
        assert len(trips1[0]) > 0
        assert trips1[0].tobytes() == trips2[0].tobytes() and trips1[1].tobytes() == trips2[1].tobytes()


@pytest.mark.parametrize("base", [0, 4096])
def test_resume_on_a_fresh_handle(base):
    """Save on handle A, load into a new handle B with the same config, seed and env_id_base (one rank of a sharded
    run when base > 0): B continues A's trajectory bit for bit."""
    from traffic_env_b200 import VecTrafficEnv
    kw = dict(m=3, n=3, num_envs=50, seed=5, env_id_base=base, local_cars_per_sec=0.4, ticks_per_step=5)
    a = VecTrafficEnv(**kw)
    a.reset()
    run_window(a, 5, True)
    rec = a.save_envs()
    ref = run_window(a, 6, True)
    b = VecTrafficEnv(**kw)
    b.load_envs(rec)
    assert run_window(b, 6, True) == ref
    assert same_state(a.get_state(), b.get_state())
    # another env_id_base keys another arrival stream: the same state diverges
    c = VecTrafficEnv(**dict(kw, env_id_base=base + 50))
    c.load_envs(rec)
    assert run_window(c, 6, True) != ref


def test_gather_and_scatter():
    from traffic_env_b200 import VecTrafficEnv
    kw = dict(m=3, n=3, num_envs=12, seed=2, local_cars_per_sec=0.5, ticks_per_step=5)
    env, twin = VecTrafficEnv(**kw), VecTrafficEnv(**kw)
    for e in (env, twin):
        e.reset()
        run_window(e, 5, True)
    src, dst = [5, 2, 9, 5], [0, 1, 3, 7]
    before = env.get_state()
    rec = env.save_envs(src)
    assert rec.shape == (4, env.snapshot_layout.stride)
    env.load_envs(rec, env_ids=dst)
    after, tw = env.get_state(), twin.get_state()
    for s, d in zip(src, dst):
        assert same_state(after, before, d, s), "env %d is not a copy of env %d" % (d, s)
    rest = [e for e in range(12) if e not in dst]
    assert same_state(after, tw, rest, rest)
    assert env.save_envs(rest).tobytes() == twin.save_envs(rest).tobytes()
    # the envs not named keep stepping like the untouched twin
    act = np.random.RandomState(0).randint(0, 2, size=(12, 9))
    for _ in range(4):
        o1, r1, d1 = (x.copy() for x in env.step(act))
        o2, r2, d2 = twin.step(act)
        assert o1[rest].tobytes() == o2[rest].tobytes() and r1[rest].tobytes() == r2[rest].tobytes()
        assert d1[rest].tobytes() == d2[rest].tobytes()
    assert env.save_envs(rest).tobytes() == twin.save_envs(rest).tobytes()
    # without arrivals the state is the whole future: with equal actions a copy steps exactly like its source
    quiet = VecTrafficEnv(**dict(kw, arrivals="none"))
    quiet.load_envs(env.save_envs())
    quiet.load_envs(quiet.save_envs(src), env_ids=dst)
    for _ in range(4):
        obs, rew, done = quiet.step(act[:1].repeat(12, axis=0))
        for s, d in zip(src, dst):
            assert obs[d].tobytes() == obs[s].tobytes() and rew[d].tobytes() == rew[s].tobytes() and done[d] == done[s]
    st = quiet.get_state()
    for s, d in zip(src, dst):
        assert same_state(st, st, d, s)


def test_host_and_device_records_agree():
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("torch without CUDA")
    from traffic_env_b200 import VecTrafficEnv
    E = 40
    env = VecTrafficEnv(m=3, n=3, num_envs=E, seed=9, local_cars_per_sec=0.4, ticks_per_step=5)
    env.reset()
    run_window(env, 3, True)
    stride = env.snapshot_layout.stride
    host = env.save_envs()
    dev = torch.empty((E, stride), dtype=torch.uint8, device="cuda")
    env.save_envs(out=dev)
    torch.cuda.synchronize()
    assert dev.cpu().numpy().tobytes() == host.tobytes()
    ids = [3, 3, 17, 0]
    dsub = torch.empty((4, stride), dtype=torch.uint8, device="cuda")
    env.save_envs(ids, out=dsub.data_ptr())
    torch.cuda.synchronize()
    assert dsub.cpu().numpy().tobytes() == host[ids].tobytes()
    # a save queued on a torch stream right behind a device step, no synchronisation in between: the post-step state
    s = torch.cuda.Stream()
    n = 3
    act = torch.empty((E, 9), dtype=torch.uint8, device="cuda")
    obs = torch.empty((n, E, env.obs_len), dtype=torch.float32, device="cuda")
    rew = torch.empty((n, E, 9), dtype=torch.float32, device="cuda")
    done = torch.empty((n, E), dtype=torch.uint8, device="cuda")
    after = torch.empty((E, stride), dtype=torch.uint8, device="cuda")
    with torch.cuda.stream(s):
        env.step_multi_device(n, act, obs, rew, done, controller="greedy", stream=s.cuda_stream)
        env.save_envs(out=after, stream=s.cuda_stream)
    s.synchronize()
    assert after.cpu().numpy().tobytes() == env.save_envs().tobytes()
    assert after.cpu().numpy().tobytes() != host.tobytes()
    # device records load like host ones
    env.load_envs(dev)
    assert env.save_envs().tobytes() == host.tobytes()


def test_bad_records_are_rejected_and_change_nothing():
    from traffic_env_b200 import VecTrafficEnv, _lib
    from traffic_env_b200._lib import TE_HOST, TrafficB200Error
    E = 8
    env = VecTrafficEnv(m=3, n=3, num_envs=E, seed=4, local_cars_per_sec=0.5, ticks_per_step=5)
    env.reset()
    run_window(env, 3, True)
    lay = env.snapshot_layout
    good = env.save_envs()
    other = VecTrafficEnv(m=4, n=4, num_envs=2)
    four = other.save_envs()

    def rejected(records, match, env_ids=None):
        with pytest.raises(TrafficB200Error, match=match):
            env.load_envs(records, env_ids=env_ids)
        assert env.save_envs().tobytes() == good.tobytes(), "a rejected load changed the batch"

    rejected(np.ascontiguousarray(four[:1, :lay.stride]), r"record 0 .*dimensions", env_ids=[0])
    bad = good.copy()
    bad[3, 0] ^= 1
    rejected(bad, r"record 3 \(for env 3\).*magic")
    for value, field in ((0, "leading"), (20, "leading")):
        bad = good.copy()
        bad[5, lay.x + 7 * 80] = value                  # road 7's header word: leading is its low byte
        rejected(bad, r"record 5 .*%s" % field)
    bad = good.copy()
    bad[2, lay.x + 3 * 80 + 1] = 0                      # lastcar = 0
    rejected(bad, r"record 2 .*lastcar")
    bad = good.copy()
    bad[1, lay.x + 3] = 1                               # top byte of road 0's header word
    rejected(bad, r"record 1 .*top byte")
    bad = good.copy()
    bad[6, lay.phase + 4] = 2
    rejected(bad, r"record 6 .*phase")
    bad = good.copy()
    bad[4, lay.passed_dst] = 7
    bad[6, lay.phase] = 2
    rejected(bad, r"record 4 \(for env 4\).*passed_dst")  # the first bad record is named
    rejected(good[:2], r"outside", env_ids=[0, E])
    rejected(good[:2], r"outside", env_ids=[-1, 0])
    rejected(good[:2], r"twice", env_ids=[1, 1])
    L = _lib.load()
    with pytest.raises(TrafficB200Error, match="negative"):
        _lib.check(L.te_load_envs(env._h, None, -1, good.ctypes.data, TE_HOST, None))
    with pytest.raises(TrafficB200Error, match="negative"):
        _lib.check(L.te_save_envs(env._h, None, -1, good.ctypes.data, TE_HOST, None))
    with pytest.raises(TrafficB200Error, match="outside"):
        env.save_envs([0, E])
    assert env.save_envs().tobytes() == good.tobytes()


@pytest.mark.parametrize("m,n,L,E", [(3, 3, 250.0, 12), (10, 10, 120.0, 3)])
def test_tame_mode_follows_the_records(m, n, L, E):
    """Records of a tame handle keep the destination tame; a record with one wild car moves the handle to the checked
    kernels, whose ticks then match the oracle bit for bit."""
    from traffic_env_b200 import VecTrafficEnv
    rng = np.random.RandomState(7 * m + n)
    T = 5
    env = VecTrafficEnv(m=m, n=n, length=L, num_envs=E, arrivals="injected", remi=False)
    R, r, I = env.roads, env.train_roads, env.intersections
    states = [random_env_state(rng, R, r, I, L, True) for _ in range(E)]
    env.set_state({k: np.stack([s[k] for s in states]) for k in states[0]} | {"steps": np.zeros(E, np.float32)})
    assert env.is_tame()
    rec = env.save_envs()
    env.load_envs(rec[::-1].copy())
    assert env.is_tame()
    lay = env.snapshot_layout
    wild = rec.copy()
    nwild = 0
    for e in range(0, E, 2):
        xv = wild[e, lay.x:lay.x + R * 80].view(np.uint32).reshape(R, 20)
        vv = wild[e, lay.v:lay.v + R * 80].view(np.float32).reshape(R, 20)
        for rd in range(R):
            ld, lc = int(xv[rd, 0] & 0xff), int((xv[rd, 0] >> 8) & 0xff)
            if ld != lc:
                vv[rd, 1 if ld + 1 >= 20 else ld + 1] = np.float32([200.0, 1e-35][nwild % 2])
                nwild += 1
                break
    assert nwild > 0
    env.load_envs(wild)
    assert not env.is_tame()
    st0 = env.get_state()
    scheds = injected_schedule(env, rng, T)
    env.set_arrivals(scheds)
    oracles = []
    for e in range(E):
        o = OracleEnv(m, n, L, 0.5)
        load_oracle(o, {k: st0[k][e] for k in STATE_KEYS})
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
