"""GPU: round-2 hardening - trajectories with a non-default archetype (delta != 4; T and rate not powers of two: the
longer arithmetic forms of te_math.cuh) against the oracle, a steady-state replay of sampled envs out of the full
16384-env headline batch, a stress test aimed at the two hazards the kernel names (phase-C slot reuse -> ordered-transfer
fallback; tick-stamped early break) on the 16/24/32-warp CTA variants, and the stricter argument checks of the C ABI."""
import numpy as np
import pytest

from oracle.oracle import OracleEnv
from tests.golden_util import live_walk
from tests.test_gpu_fuzz_state import load_oracle, random_env_state, variant_of

pytestmark = pytest.mark.gpu

# x, v, l, a, delta, v0, b, T, s0, w
ARCH_ODD = [0.0, 9.5, 4.5, 2.2, 3.5, 15.3, 4.1, 1.7, 1.5, 0.0]        # nothing a power of two, delta != 4
ARCH_DELTA4 = [0.0, 11.11, 4.0, 3.0, 4.0, 13.89, 6.0, 1.3, 1.0, 0.0]  # delta == 4 but T (and the rates used) not powers of two
ARCH_POW2 = [0.0, 12.0, 5.0, 1.5, 2.0, 17.0, 3.0, 2.0, 2.0, 0.0]      # T, rate powers of two, delta != 4
NONDEFAULT_ARCH_ROWS = [
    (ARCH_ODD, 0.4, 3, 3, 250.0, 0.25, 24), (ARCH_DELTA4, 0.3, 2, 3, 140.0, 0.4, 24), (ARCH_POW2, 0.5, 4, 4, 200.0, 0.2, 24),
    # the checked 256 / 768 / 1024 kernels, a few envs each
    (ARCH_ODD, 0.4, 7, 7, 200.0, 0.25, 4), (ARCH_DELTA4, 0.3, 13, 13, 140.0, 0.4, 2), (ARCH_ODD, 0.4, 15, 15, 150.0, 0.25, 2)]
NONDEFAULT_ARCH_VARIANTS = {(3, 3): ("checked", 64), (2, 3): ("checked", 64), (4, 4): ("checked", 128),
                            (7, 7): ("checked", 256), (13, 13): ("checked", 768), (15, 15): ("checked", 1024)}


@pytest.mark.parametrize("arch,rate,m,n,L,lcps,E", NONDEFAULT_ARCH_ROWS)
def test_nondefault_archetype_trajectories(arch, rate, m, n, L, lcps, E):
    from traffic_env_b200 import VecTrafficEnv
    from traffic_env_b200.arrivals import gap_cdf
    K, S = 10, 45
    arch = np.asarray(arch, np.float32)
    env = VecTrafficEnv(m=m, n=n, length=L, num_envs=E, rate=rate, arrivals="philox", seed=77, local_cars_per_sec=lcps,
                        ticks_per_step=K, remi=True, archetype=arch)
    # (is_tame() may hold: an archetype inside the tame ranges still runs the checked form unless it is the reference's)
    assert variant_of(env) == NONDEFAULT_ARCH_VARIANTS[(m, n)]
    rng = np.random.RandomState(5)
    I = m * n
    init = rng.randint(2, size=(E, I))
    env.reset(init_phase=init)
    cdf = gap_cdf(env.cars_per_sec * rate)
    oracles = []
    for e in range(E):
        o = OracleEnv(m, n, L, rate)
        o.set_archetype(arch)
        o.reset(init[e])
        o.philox_seed(77, e, cdf)
        oracles.append(o)
    cars = 0
    for s in range(S):
        if s % 4 == 0:
            act = rng.randint(2, size=(E, I))
        obs, rew, done = env.step(act)
        for e, o in enumerate(oracles):
            oo, orw, od = o.actor_step_philox(act[e], K, use_remi=True)
            assert obs[e].tobytes() == oo.tobytes() and rew[e].tobytes() == orw.tobytes() and bool(done[e]) == od, (e, s)
    st = env.get_state()
    for e, o in enumerate(oracles):
        assert (st["leading"][e] == o.leading).all() and (st["lastcar"][e] == o.lastcar).all()
        gx, gv = live_walk(st["leading"][e], st["lastcar"][e], st["x"][e], st["v"][e])
        ox, ov = o.live_state()
        assert gx.tobytes() == ox.tobytes() and gv.tobytes() == ov.tobytes(), e
        cars += len(ox)
    assert cars > 20 * E, "the test is meant to have traffic on the map"
    assert env.stats()["vehicle_updates"] == sum(o.vehicle_updates for o in oracles)
    assert env.stats()["arrival_saturations"] == 0


def test_headline_steady_state_replay_16384():
    """The bench workload at full size, 300 actor steps into its ring-capacity-bound steady state (overflow in a third
    of the steps, early breaks): 32 envs spread over the batch replayed from scratch on the oracle - every sampled
    env's final ring indices, car state (bits), tick count and the last observation must match."""
    from traffic_env_b200 import VecTrafficEnv
    from traffic_env_b200.arrivals import gap_cdf
    E, M, N, L, K, S = 16384, 10, 10, 500.0, 10, 300
    env = VecTrafficEnv(m=M, n=N, length=L, num_envs=E, arrivals="philox", seed=2026, local_cars_per_sec=0.12,
                        ticks_per_step=K, remi=True)
    env.reset(init_phase=np.zeros((E, M * N), np.uint8))
    ids = np.unique(np.concatenate([np.arange(0, E, 529), [1, E - 2, E - 1]]))[:32]
    acts = np.zeros((S, len(ids), M * N), np.uint8)
    last_obs = None
    overflow_steps = 0
    for s in range(S):
        if s % 3 == 0:
            a = env.greedy_actions().copy()
        acts[s] = a[ids]
        obs, rew, done = env.step(a)
        overflow_steps += int(done[ids].sum())
        last_obs = obs[ids].copy()
    cdf = gap_cdf(env.cars_per_sec * 0.5)
    assert overflow_steps > 100, "the steady state is meant to overflow often"
    for j, e in enumerate(ids):
        o = OracleEnv(M, N, L, 0.5)
        o.reset(np.zeros(M * N, np.int32))
        o.philox_seed(2026, int(e), cdf)
        for s in range(S):
            oo, orw, od = o.actor_step_philox(acts[s, j], K, use_remi=True)
        st = env.get_state(int(e), 1)
        assert (st["leading"][0] == o.leading).all() and (st["lastcar"][0] == o.lastcar).all(), e
        gx, gv = live_walk(st["leading"][0], st["lastcar"][0], st["x"][0], st["v"][0])
        ox, ov = o.live_state()
        assert gx.tobytes() == ox.tobytes() and gv.tobytes() == ov.tobytes(), e
        assert float(st["steps"][0]) == float(o.steps), e
        assert last_obs[j].tobytes() == oo.tobytes(), e
        assert len(ox) > 2500
    assert env.stats()["arrival_saturations"] == 0


@pytest.mark.parametrize("m,n,L,E,multi", [(10, 10, 60.0, 40, False), (13, 13, 60.0, 24, False), (15, 15, 60.0, 16, False),
                                           (10, 10, 60.0, 24, True), (3, 3, 60.0, 90, True), (4, 4, 60.0, 31, True)])
def test_transfer_hazards_under_load(m, n, L, E, multi):
    """16-, 24- and 32-warp CTAs (512 / 768 / 1024-thread variants) and shared CTAs (3x3, 4x4), many co-resident envs,
    short roads packed with cars near the road end: most ticks pop two or more cars per road, so the parallel transfer
    phase keeps meeting the slot-reuse hazard (-> strict-order fallback on that tick) and rings overflow (-> tick-stamped
    early break of the fused step).  Fused K-tick steps - one per launch, or two per launch (te_step_multi: the
    ordered-transfer stamps then have to survive the step boundary) - against the oracle's tick loop; raw ticks are
    covered by test_gpu_fuzz_state."""
    from traffic_env_b200 import VecTrafficEnv
    rng = np.random.RandomState(31 * m + n)
    K, S = 6, 4
    env = VecTrafficEnv(m=m, n=n, length=L, num_envs=E, arrivals="injected", remi=True, ticks_per_step=K)
    R, r, I = env.roads, env.train_roads, env.intersections
    states = [random_env_state(rng, R, r, I, L, True) for _ in range(E)]
    T = K * S
    scheds = [[list(rng.choice(env.entrypoints, size=rng.randint(0, 5))) for _ in range(T)] for _ in range(E)]
    env.set_arrivals(scheds)
    env.set_state({k: np.stack([s[k] for s in states]) for k in states[0]} | {"steps": np.zeros(E, np.float32)})
    oracles = []
    for e in range(E):
        o = OracleEnv(m, n, L, 0.5)
        load_oracle(o, states[e])
        oracles.append(o)
    cursor = np.zeros(E, np.int64)         # arrival-process tick of each env (advances by the ticks actually run)
    multi_pop = breaks = 0
    for s in range(S):
        if multi and s % 2 == 1:
            obs, rew, done = obs2[1], rew2[1], done2[1]          # second actor step of the launch, same action
        else:
            act = rng.randint(0, 2, size=(E, I))
            if multi:
                _, obs2, rew2, done2 = env.step_multi(2, actions=act, controller="given")
                obs, rew, done = obs2[0], rew2[0], done2[0]
            else:
                obs, rew, done = env.step(act)
        st = env.get_state() if (not multi or s % 2 == 1) else None    # (the state is that after the whole launch)
        for e, o in enumerate(oracles):
            passed = np.zeros(r, np.float32)
            od = False
            for k in range(K):
                before = o.leading.copy()
                od = o.step(act[e], scheds[e][cursor[e]] if cursor[e] < T else [])
                multi_pop += int((((o.leading - before) % 19) >= 2).sum())
                cursor[e] += 1
                passed += o.passed
                if od:
                    breaks += int(k < K - 1)
                    break
            orw = o.remi_reward().copy()
            o.passed_dst[:] = 0
            tag = "env %d step %d" % (e, s)
            assert bool(done[e]) == od, tag
            assert obs[e, :r].tobytes() == passed.tobytes(), tag + " passed"
            assert (obs[e, r:2 * r] == o.detected).all(), tag + " detected"
            assert rew[e].tobytes() == orw.tobytes(), tag + " reward"
            if st is not None:
                assert (st["leading"][e] == o.leading).all() and (st["lastcar"][e] == o.lastcar).all(), tag + " rings"
                gx, gv = live_walk(st["leading"][e], st["lastcar"][e], st["x"][e], st["v"][e])
                ox, ov = o.live_state()
                assert gx.tobytes() == ox.tobytes() and gv.tobytes() == ov.tobytes(), tag + " car state"
    stats = env.stats()
    assert multi_pop > E * R // 200 and breaks > 0
    assert stats["seq_fallback_ticks"] > (E // 4 if R > 200 else 0), "the ordered-transfer fallback is meant to fire"
    assert stats["overflows"] == sum(o.overflows for o in oracles)


def test_strict_argument_checks():
    from traffic_env_b200 import TrafficB200Error, VecTrafficEnv
    env = VecTrafficEnv(m=3, n=3, num_envs=2, arrivals="injected")
    H = 4
    roads = np.array([0, 3, 6], np.int16)
    ok = np.array([[0, 1, 1, 2, 3], [3, 3, 3, 3, 3]], np.int64)
    env.set_arrivals_csr(ok, roads, H)
    for bad, what in ((np.array([[0, 1, 1, 2, 4], [3, 3, 3, 3, 3]], np.int64), "beyond num_roads"),
                      (np.array([[-1, 1, 1, 2, 3], [3, 3, 3, 3, 3]], np.int64), "outside"),
                      (np.array([[0, 1, 1, 2, 3], [5, 5, 5, 5, 5]], np.int64), "outside|beyond"),
                      (np.array([[0, 2, 1, 2, 3], [3, 3, 3, 3, 3]], np.int64), "not monotone")):
        with pytest.raises(TrafficB200Error, match=what):
            env.set_arrivals_csr(bad, roads, H)
    obs, rew, done = env.step(np.zeros((2, 9)))     # the old (valid) schedule is still in place
    assert env.stats()["cars_generated"] == 3
    for kw, what in ((dict(length=10.0), "maximum displacement"), (dict(rate=0.0), "finite and positive"),
                     (dict(length=float("nan")), "finite and positive"),
                     (dict(archetype=[0, 11.11, 4, 3, 4, 0.0, 6, 2, 1, 0]), "v0"),
                     (dict(archetype=[0, 11.11, 4, 3, 4, 13.89, float("inf"), 2, 1, 0]), "finite")):
        with pytest.raises(TrafficB200Error, match=what):
            VecTrafficEnv(m=2, n=2, num_envs=1, **kw)


def test_wire_records_equal_float_outputs():
    """The compact wire format of the host path: te_step_wire records (host and device memory) expand to exactly the
    float obs / reward / done of te_step; steps of more than 13 ticks (passed counts no longer fit a byte) take the float
    path and still agree with the device-buffer launch; remi off (overflow penalties of -10 n travel as f32)."""
    import ctypes as C
    import torch
    from traffic_env_b200 import TrafficB200Error, VecTrafficEnv
    from traffic_env_b200._lib import TE_DEVICE, check
    E = 4096 + 11
    kw = dict(m=3, n=3, length=250.0, num_envs=E, arrivals="philox", seed=5, local_cars_per_sec=0.6, ticks_per_step=10)
    for remi in (True, False):
        a, b, d = VecTrafficEnv(remi=remi, **kw), VecTrafficEnv(remi=remi, **kw), VecTrafficEnv(remi=remi, **kw)
        rng = np.random.RandomState(8)
        init = rng.randint(2, size=(E, 9))
        for env in (a, b, d):
            env.reset(init_phase=init)
        dev = torch.device("cuda", 0)
        d_rec = torch.zeros((E, a.wire.stride), dtype=torch.uint8, device=dev)
        saw_done = False
        for s in range(14):
            act = rng.randint(2, size=(E, 9)).astype(np.uint8)
            k = 14 if s == 9 else (3 if s == 5 else None)     # one step on the float path, one short step
            obs, rew, done = a.step(act, k=k)
            if k == 14:
                with pytest.raises(TrafficB200Error, match="k_ticks"):
                    b.step_wire(act, k=14)
                o2, r2, d2 = b.step(act, k=14)
                o2, r2, d2 = o2.copy(), r2.copy(), d2.copy()
                d.step(act, k=14)
            else:
                rec = b.step_wire(act, k=k)
                assert rec["passed"].dtype == np.uint8 and rec["light"].dtype == np.float32
                assert (rec["passed"].astype(np.float32) == obs[:, :36]).all()
                o2, r2, d2 = b.expand_wire()
                check(d._L.te_step_wire(d._h, torch.from_numpy(act).to(dev).data_ptr(), d.ticks_per_step if k is None else k,
                                        d_rec.data_ptr(), TE_DEVICE, None))
                d.synchronize()
                assert d_rec.cpu().numpy()[:, :a.wire.done + 1].tobytes() == b._wire_buf[:, :a.wire.done + 1].tobytes(), s
            assert obs.tobytes() == o2.tobytes() and rew.tobytes() == r2.tobytes() and done.tobytes() == d2.tobytes(), s
            saw_done = saw_done or bool(done.any())
        assert saw_done, "the test is meant to include ring overflows"
        assert a.stats()["vehicle_updates"] == b.stats()["vehicle_updates"] == d.stats()["vehicle_updates"]


@pytest.mark.parametrize("m,n,L,E,lcps,extra", [
    (3, 3, 250.0, 301, 0.5, {}), (10, 10, 500.0, 6, 0.3, {}), (2, 2, 120.0, 77, 0.9, {}), (4, 4, 150.0, 33, 0.4, {}),
    (3, 3, 250.0, 65, 0.5, {"learn_switch": True}), (3, 3, 250.0, 40, 0.15, {"validate": True}), (3, 3, 250.0, 50, 0.5, {"remi": False})])
def test_multi_step_launch_equals_single_steps(m, n, L, E, lcps, extra):
    """te_step_multi (n actor steps per launch, greedy controller evaluated in the kernel or a given action) produces,
    actor step by actor step, exactly what n te_step calls with the same action produce - host and device buffers -
    including overflow steps (early break) in the middle of a launch and an env count that leaves a partial CTA."""
    import torch
    from traffic_env_b200 import VecTrafficEnv
    kw = dict(m=m, n=n, length=L, num_envs=E, arrivals="philox", seed=11, local_cars_per_sec=lcps, ticks_per_step=10, remi=True)
    kw.update(extra)
    a, b, d = VecTrafficEnv(**kw), VecTrafficEnv(**kw), VecTrafficEnv(**kw)
    I = m * n
    rng = np.random.RandomState(3)
    init = rng.randint(2, size=(E, I))
    for env in (a, b, d):
        env.reset(init_phase=init)
    dev = torch.device("cuda", 0)
    NS = 6 if (m, n) == (4, 4) else 3          # 6 x 10 ticks: close to the 64-tick limit of one launch
    d_act = torch.zeros((E, I), dtype=torch.uint8, device=dev)
    d_obs = torch.zeros((NS, E, a.obs_len), dtype=torch.float32, device=dev)
    d_rew = torch.zeros((NS, E, I), dtype=torch.float32, device=dev)
    d_done = torch.zeros((NS, E), dtype=torch.uint8, device=dev)
    saw_done = 0
    for launch in range(24 if extra.get("validate") else 14):
        ctrl = "greedy" if launch % 3 != 2 else "given"
        ns = NS if launch % 4 != 3 else 2
        if launch == 5:
            ns = 1
        if ctrl == "greedy":
            act = a.greedy_actions().copy()
            act_b, obs_b, rew_b, done_b = b.step_multi(ns, controller="greedy")
            d.step_multi_device(ns, d_act, d_obs, d_rew, d_done, controller="greedy")
        else:
            act = rng.randint(2, size=(E, I)).astype(np.uint8)
            act_b, obs_b, rew_b, done_b = b.step_multi(ns, actions=act, controller="given")
            d_act.copy_(torch.from_numpy(act))
            d.step_multi_device(ns, d_act, d_obs, d_rew, d_done, controller="given")
        d.synchronize()
        assert (act_b != 0).tobytes() == (act != 0).tobytes(), launch
        assert (d_act.cpu().numpy() != 0).tobytes() == (act != 0).tobytes(), launch
        for j in range(ns):
            obs, rew, done = a.step(act)
            assert obs.tobytes() == obs_b[j].tobytes() and rew.tobytes() == rew_b[j].tobytes() and done.tobytes() == done_b[j].tobytes(), (launch, j)
            assert obs.tobytes() == d_obs[j].cpu().numpy().tobytes() and rew.tobytes() == d_rew[j].cpu().numpy().tobytes() \
                and done.tobytes() == d_done[j].cpu().numpy().tobytes(), (launch, j)
            saw_done += int(done.sum())
    sa, sb, sd = a.get_state(), b.get_state(), d.get_state()
    for k in ("leading", "lastcar", "obs", "waiting", "passed_dst", "steps"):
        assert (sa[k] == sb[k]).all() and (sa[k] == sd[k]).all(), k
    for e in range(E):
        xa, va = live_walk(sa["leading"][e], sa["lastcar"][e], sa["x"][e], sa["v"][e])
        xb, vb = live_walk(sb["leading"][e], sb["lastcar"][e], sb["x"][e], sb["v"][e])
        xd, vd = live_walk(sd["leading"][e], sd["lastcar"][e], sd["x"][e], sd["v"][e])
        assert xa.tobytes() == xb.tobytes() == xd.tobytes() and va.tobytes() == vb.tobytes() == vd.tobytes(), e
    sta, stb, std = a.stats(), b.stats(), d.stats()
    for k in ("ticks", "actor_steps", "vehicle_updates", "overflows", "cars_generated", "cars_exited"):
        assert sta[k] == stb[k] == std[k], k
    assert saw_done > 0 or extra.get("validate"), "the test is meant to include overflow steps"
    if extra.get("validate"):
        (ea, ta), (eb, tb), (ed, td) = a.trip_times(), b.trip_times(), d.trip_times()
        assert len(ta) > 0 and ea.tobytes() == eb.tobytes() == ed.tobytes() and ta.tobytes() == tb.tobytes() == td.tobytes()


@pytest.mark.parametrize("m,n,L,E", [(3, 3, 250.0, 37), (10, 10, 500.0, 5), (2, 2, 100.0, 31)])
def test_masked_step_touches_only_the_masked_envs(m, n, L, E):
    """te_step_masked: the masked envs advance exactly as the oracle does, the others keep their state, their arrival
    stream and their rows of the output arrays - for single envs of a shared CTA (two default-grid envs per CTA) too."""
    from traffic_env_b200 import VecTrafficEnv
    from traffic_env_b200.arrivals import gap_cdf
    K, I = 10, m * n
    env = VecTrafficEnv(m=m, n=n, length=L, num_envs=E, arrivals="philox", seed=21, local_cars_per_sec=0.4,
                        ticks_per_step=K, remi=True)
    rng = np.random.RandomState(2)
    init = rng.randint(2, size=(E, I))
    env.reset(init_phase=init)
    cdf = gap_cdf(env.cars_per_sec * 0.5)
    oracles = []
    for e in range(E):
        o = OracleEnv(m, n, L, 0.5)
        o.reset(init[e])
        o.philox_seed(21, e, cdf)
        oracles.append(o)
    for s in range(40):
        mask = rng.rand(E) < (0.5 if s % 5 else 0.08)
        if s == 7:
            mask[:] = False
        act = rng.randint(2, size=(E, I))
        sentinel = env._obs.copy()
        obs, rew, done = env.step_masked(act, mask)
        for e, o in enumerate(oracles):
            if mask[e]:
                oo, orw, od = o.actor_step_philox(act[e], K, use_remi=True)
                assert obs[e].tobytes() == oo.tobytes() and rew[e].tobytes() == orw.tobytes() and bool(done[e]) == od, (e, s)
            else:
                assert obs[e].tobytes() == sentinel[e].tobytes(), (e, s)
    st = env.get_state()
    for e, o in enumerate(oracles):
        assert (st["leading"][e] == o.leading).all() and (st["lastcar"][e] == o.lastcar).all(), e
        gx, gv = live_walk(st["leading"][e], st["lastcar"][e], st["x"][e], st["v"][e])
        ox, ov = o.live_state()
        assert gx.tobytes() == ox.tobytes() and gv.tobytes() == ov.tobytes(), e
        assert float(st["steps"][e]) == float(o.steps), e
    assert env.stats()["vehicle_updates"] == sum(o.vehicle_updates for o in oracles)


def test_multi_step_wire_records():
    """step_multi_wire == step_multi, field by field (records [n_steps, E, stride])."""
    from traffic_env_b200 import VecTrafficEnv
    E = 1000
    kw = dict(m=3, n=3, length=250.0, num_envs=E, arrivals="philox", seed=4, local_cars_per_sec=0.5, ticks_per_step=10, remi=True)
    a, b = VecTrafficEnv(**kw), VecTrafficEnv(**kw)
    init = np.random.RandomState(1).randint(2, size=(E, 9))
    a.reset(init_phase=init)
    b.reset(init_phase=init)
    for launch in range(8):
        act_a, obs, rew, done = a.step_multi(3, controller="greedy")
        act_b, rec = b.step_multi_wire(3, controller="greedy")
        assert act_a.tobytes() == act_b.tobytes()
        assert (rec["passed"].astype(np.float32) == obs[:, :, :36]).all() and (rec["detected"].astype(np.float32) == obs[:, :, 36:72]).all()
        assert rec["light"].tobytes() == np.ascontiguousarray(obs[:, :, 72:]).tobytes()
        assert rec["reward"].tobytes() == rew.tobytes() and (rec["done"] == done).all()
    assert a.stats()["vehicle_updates"] == b.stats()["vehicle_updates"] > 0


def test_lazy_results_and_both_host_transports(monkeypatch):
    """step(lazy=True) / step_multi(lazy=True) deliver WireResults whose lazily expanded observation equals the eager
    float arrays, and the two transports of the eager host path (wire records expanded on the host; float arrays written
    by the copy engine, TE_HOST_FLOAT_DMA) give identical bytes - single and multi-step."""
    from traffic_env_b200 import VecTrafficEnv, WireResult
    E = 2500
    kw = dict(m=3, n=3, length=250.0, num_envs=E, arrivals="philox", seed=6, local_cars_per_sec=0.5, ticks_per_step=10, remi=True)
    monkeypatch.setenv("TE_HOST_FLOAT_DMA", "0")
    a, lz = VecTrafficEnv(**kw), VecTrafficEnv(**kw)
    monkeypatch.setenv("TE_HOST_FLOAT_DMA", "1")
    b = VecTrafficEnv(**kw)
    init = np.random.RandomState(1).randint(2, size=(E, 9))
    for env in (a, b, lz):
        env.reset(init_phase=init)
    rng = np.random.RandomState(2)
    for s in range(10):
        if s % 2 == 0:
            act = rng.randint(2, size=(E, 9)).astype(np.uint8)
            oa, ra, da = a.step(act)
            ob, rb, db = b.step(act)
            res = lz.step(act, lazy=True)
            assert isinstance(res, WireResult)
            assert oa.tobytes() == ob.tobytes() and ra.tobytes() == rb.tobytes() and da.tobytes() == db.tobytes(), s
            assert res.obs_of([0, 7, E - 1]).tobytes() == oa[[0, 7, E - 1]].tobytes()
            ol, rl, dl = res
            assert ol.tobytes() == oa.tobytes() and rl.tobytes() == ra.tobytes() and dl.tobytes() == da.tobytes(), s
        else:
            xa, oa, ra, da = a.step_multi(3, controller="greedy")
            xb, ob, rb, db = b.step_multi(3, controller="greedy")
            xl, res = lz.step_multi(3, controller="greedy", lazy=True)
            assert xa.tobytes() == xb.tobytes() == xl.tobytes()
            assert oa.tobytes() == ob.tobytes() and ra.tobytes() == rb.tobytes() and da.tobytes() == db.tobytes(), s
            assert res.obs.tobytes() == oa.tobytes() and res.reward.tobytes() == ra.tobytes() and (res.done == da).all(), s
            assert res.obs_of([3, 4], step=2).tobytes() == oa[2, [3, 4]].tobytes()
    assert a.stats()["vehicle_updates"] == b.stats()["vehicle_updates"] == lz.stats()["vehicle_updates"] > 0


def test_multi_step_argument_errors():
    from traffic_env_b200 import TrafficB200Error, VecTrafficEnv
    env = VecTrafficEnv(m=3, n=3, num_envs=8, arrivals="philox", ticks_per_step=10)
    with pytest.raises(TrafficB200Error, match="n_steps"):
        env.step_multi(7, controller="greedy")              # 70 ticks > 64 per launch
    with pytest.raises(TrafficB200Error, match="n_steps"):
        env.step_multi(0, controller="greedy")
    act, obs, rew, done = env.step_multi(6, controller="greedy")
    assert obs.shape == (6, 8, 81) and rew.shape == (6, 8, 9) and done.shape == (6, 8)
    auto = VecTrafficEnv(m=3, n=3, num_envs=8, arrivals="philox", ticks_per_step=10, auto_reset=True, episode_len=5)
    with pytest.raises(TrafficB200Error, match="TE_AUTO_RESET"):
        auto.step_multi(3, controller="greedy")
    o, r, d = auto.step(np.zeros((8, 9)))                   # single steps are what such a handle is for
    assert o.shape == (8, 81)


WILD_CAR_ROWS = [(3, 3, 250.0, 66), (10, 10, 120.0, 6), (1, 1, 60.0, 8),
                 # the checked 64 / 256 / 768 / 1024 kernels with the reference's archetype (pow2 and powf4 shortcuts on)
                 (4, 3, 90.0, 12), (7, 7, 120.0, 4), (13, 13, 100.0, 2), (15, 15, 100.0, 2)]
# (kind, MAXT) of the step kernel before and after the wild cars
WILD_CAR_VARIANTS = {(3, 3): (("grouped", 96), ("checked", 64)), (10, 10): (("tame", 512), ("checked", 512)),
                     (1, 1): (("grouped", 64), ("checked", 64)), (4, 3): (("tame", 64), ("checked", 64)),
                     (7, 7): (("tame", 256), ("checked", 256)), (13, 13): (("tame", 768), ("checked", 768)),
                     (15, 15): (("tame", 1024), ("checked", 1024))}


@pytest.mark.parametrize("m,n,L,E", WILD_CAR_ROWS)
def test_wild_car_moves_the_handle_to_the_checked_kernels(m, n, L, E):
    """A handle runs the kernels without the per-car validity predicate only while every car it was ever given is tame
    (te_is_tame, include/traffic_b200.h).  Tame random states first (is_tame stays set, two shared-CTA envs per CTA on
    the 3x3 grid), then the same states with a few cars at speeds outside the tame range - float products that round
    (1e-35, 3e-31, subnormal 1e-42: the generic routine decides) or above the handle's speed cap (200 m/s): the handle
    must leave the tame mode and every tick must still match the oracle bit for bit.  (Speeds that overflow to NaN state
    are compared - NaN payloads aside - at the level of the update in test_gpu_math.py::test_idm_adversarial_operands.)"""
    from traffic_env_b200 import VecTrafficEnv
    rng = np.random.RandomState(5 * m + n)
    T = 6
    env = VecTrafficEnv(m=m, n=n, length=L, num_envs=E, arrivals="injected", remi=False)
    R, r, I = env.roads, env.train_roads, env.intersections
    assert env.is_tame()
    for wild in (False, True):
        states = [random_env_state(rng, R, r, I, L, True) for _ in range(E)]
        nwild = 0
        if wild:
            for st in states[::2]:
                for rd in rng.choice(R, size=min(R, 6), replace=False):
                    ld, lc = int(st["leading"][rd]), int(st["lastcar"][rd])
                    if ld == lc:
                        continue
                    sl = 1 if ld + 1 >= 20 else ld + 1
                    st["v"][rd, sl] = np.float32(rng.choice([1e-35, 1e-42, 200.0, 3e-31]))
                    nwild += 1
            assert nwild > 0
        scheds = [[list(rng.choice(env.entrypoints, size=rng.randint(0, 3))) for _ in range(T)] for _ in range(E)]
        env.set_arrivals(scheds, first_tick=T if wild else 0)     # (the envs' arrival clocks are at T after the first pass)
        env.set_state({k: np.stack([s[k] for s in states]) for k in states[0]} | {"steps": np.zeros(E, np.float32)})
        assert env.is_tame() == (not wild)
        assert variant_of(env) == WILD_CAR_VARIANTS[(m, n)][int(wild)]
        oracles = []
        for e in range(E):
            o = OracleEnv(m, n, L, 0.5)
            load_oracle(o, states[e])
            oracles.append(o)
        for t in range(T):
            act = rng.randint(0, 2, size=(E, I))
            obs, rew, done = env.step_raw(act)
            st = env.get_state()
            for e, o in enumerate(oracles):
                od = o.step(act[e], scheds[e][t])
                tag = "wild %s env %d tick %d" % (wild, e, t)
                assert (st["leading"][e] == o.leading).all() and (st["lastcar"][e] == o.lastcar).all(), tag + " rings"
                assert (obs[e] == o.obs).all(), tag + " obs"
                assert rew[e].tobytes() == o.rewards.tobytes(), tag + " rewards"
                assert bool(done[e]) == od, tag + " done"
                gx, gv = live_walk(st["leading"][e], st["lastcar"][e], st["x"][e], st["v"][e])
                ox, ov = o.live_state()
                assert gx.tobytes() == ox.tobytes() and gv.tobytes() == ov.tobytes(), tag + " car state"
    # a tame state afterwards does not bring the unchecked kernels back (cars given earlier may still be on the roads)
    assert not env.is_tame()


CONTROLLER_ROWS = [
    (3, 3, 250.0, 301, 0.5, {}), (10, 10, 500.0, 6, 0.3, {}), (2, 2, 120.0, 77, 0.9, {}), (4, 4, 150.0, 33, 0.4, {}),
    (3, 3, 250.0, 65, 0.5, {"learn_switch": True}), (3, 3, 250.0, 40, 0.15, {"validate": True}), (3, 3, 250.0, 50, 0.5, {"remi": False}),
    (3, 3, 250.0, 64, 0.12, {"ticks_per_step": 4}),
    # a non-tame archetype: the decisions are taken inside the checked 256 kernel
    (7, 7, 150.0, 6, 0.9, {"archetype": ARCH_ODD, "rate": 0.4})]


@pytest.mark.parametrize("m,n,L,E,lcps,extra", CONTROLLER_ROWS)
def test_controller_decisions_inside_a_launch(m, n, L, E, lcps, extra):
    """te_set_controller_spacing: one te_step_multi launch that holds several greedy decisions (a new one every
    `spacing` actor steps, evaluated in the kernel on the live rings) produces exactly what one launch per decision
    produces - actions of every decision, every actor step's obs / reward / done, host buffers, device buffers and wire
    records, final car state and counters - including overflow steps (early break: the envs of a CTA then decide at
    different ticks of the launch), learn_switch (the light toggles from the decision tick on), validate mode, a spacing
    that does not divide the launch, and going back to one decision per launch on the same handle."""
    import torch
    from traffic_env_b200 import VecTrafficEnv
    kw = dict(m=m, n=n, length=L, num_envs=E, arrivals="philox", seed=23, local_cars_per_sec=lcps, ticks_per_step=10, remi=True)
    kw.update(extra)
    K = kw["ticks_per_step"]
    a, b, d, w = (VecTrafficEnv(**kw) for _ in range(4))
    I = m * n
    init = np.random.RandomState(5).randint(2, size=(E, I))
    for env in (a, b, d, w):
        env.reset(init_phase=init)
    if "archetype" in extra:
        assert variant_of(a) == ("checked", 256)
    dev = torch.device("cuda", 0)
    NMAX = 64 // K
    d_act = torch.zeros((NMAX, E, I), dtype=torch.uint8, device=dev)
    d_obs = torch.zeros((NMAX, E, a.obs_len), dtype=torch.float32, device=dev)
    d_rew = torch.zeros((NMAX, E, I), dtype=torch.float32, device=dev)
    d_done = torch.zeros((NMAX, E), dtype=torch.uint8, device=dev)
    saw_done = 0
    plans = [(6, 3), (6, 2), (5, 3), (6, 1), (4, 3), (3, None), (6, 3), (2, 5), (6, 4)] if K == 10 else [(16, 3), (12, 5), (16, 4), (9, None)]
    for rep in range(3 if not extra.get("validate") else 4):
        for ns, sp in plans:
            ns = min(ns, NMAX)
            act_b, obs_b, rew_b, done_b = b.step_multi(ns, controller="greedy", spacing=sp)
            d.step_multi_device(ns, d_act, d_obs, d_rew, d_done, controller="greedy", spacing=sp)
            act_w, rec = w.step_multi_wire(ns, controller="greedy", spacing=sp)
            d.synchronize()
            seg = ns if sp is None else sp
            ndec = (ns + seg - 1) // seg
            act_b = act_b.reshape(ndec, E, I)
            act_w = act_w.reshape(ndec, E, I)
            j = 0
            for dec in range(ndec):
                cnt = min(seg, ns - j)
                act_a, obs_a, rew_a, done_a = a.step_multi(cnt, controller="greedy")       # one launch per decision
                tag = (rep, ns, sp, dec)
                assert act_a.tobytes() == act_b[dec].tobytes() == act_w[dec].tobytes(), tag
                assert act_a.tobytes() == d_act[dec].cpu().numpy().tobytes(), tag
                for q in range(cnt):
                    assert obs_a[q].tobytes() == obs_b[j].tobytes() and rew_a[q].tobytes() == rew_b[j].tobytes() \
                        and done_a[q].tobytes() == done_b[j].tobytes(), tag + (q,)
                    assert obs_a[q].tobytes() == d_obs[j].cpu().numpy().tobytes() and rew_a[q].tobytes() == d_rew[j].cpu().numpy().tobytes() \
                        and done_a[q].tobytes() == d_done[j].cpu().numpy().tobytes(), tag + (q,)
                    assert rec["reward"][j].tobytes() == rew_a[q].tobytes() and (rec["done"][j] == done_a[q]).all(), tag + (q,)
                    assert rec["light"][j].tobytes() == np.ascontiguousarray(obs_a[q][:, 2 * a.train_roads:]).tobytes(), tag + (q,)
                    saw_done += int(done_a[q].sum())
                    j += 1
    sa = a.get_state()
    for other in (b, d, w):
        so = other.get_state()
        for k in ("leading", "lastcar", "obs", "waiting", "passed_dst", "steps"):
            assert (sa[k] == so[k]).all(), k
        for e in range(E):
            xa, va = live_walk(sa["leading"][e], sa["lastcar"][e], sa["x"][e], sa["v"][e])
            xo, vo = live_walk(so["leading"][e], so["lastcar"][e], so["x"][e], so["v"][e])
            assert xa.tobytes() == xo.tobytes() and va.tobytes() == vo.tobytes(), e
        sta, sto = a.stats(), other.stats()
        for k in ("ticks", "actor_steps", "vehicle_updates", "overflows", "cars_generated", "cars_exited"):
            assert sta[k] == sto[k], k
    assert saw_done > 0 or extra.get("validate") or K != 10, "the test is meant to include overflow steps"
    if extra.get("validate"):
        (ea, ta), (eb, tb) = a.trip_times(), b.trip_times()
        assert len(ta) > 0 and ea.tobytes() == eb.tobytes() and ta.tobytes() == tb.tobytes()
