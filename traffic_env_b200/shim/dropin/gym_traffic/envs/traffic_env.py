"""TrafficEnv: the reference's gym environment (gym_traffic/envs/traffic_env.py:221-394) as a thin
host object over ONE env instance of the B200 simulator.  Same attribute and method names, same
in-place `obs` / `rewards` buffers (with `passed`, `detected`, `current_phase`, `elapsed` as views,
traffic_env.py:372-376), same flags (FLAGS.rate / poisson / entry / learn_switch /
local_cars_per_sec, written FLAGS.cars_per_sec), so the reference's wrappers and agents run
unchanged on top.  Every tick is one te_step_raw launch; the fused K-tick path is
traffic_env_b200.wrappers.Repeater / VecTrafficEnv.

Not provided: the pyglet renderer (traffic_env.py:285-359) and the raw `state[R,10,20]` array as a
live buffer (a snapshot is available as `.state`).
"""
import os

import gym
import numpy as np
from args import FLAGS, add_argument

from gym_traffic.spaces.gspace import GSpace
from traffic_env_b200 import VecTrafficEnv
from traffic_env_b200.host_arrivals import ArrivalStream
from traffic_env_b200.vec_env import ARCHETYPE, inv_popcount as _inv_popcount

add_argument('--local_cars_per_sec', 0.12, type=float)
add_argument('--rate', 0.5, type=float)
add_argument('--poisson', True, type=bool)
add_argument('--entry', 'all')
add_argument('--learn_switch', False, type=bool)

THRESH = 0.2
PASSING_REWARD = 0
YELLOW_TICKS = 6
DECEL_PENALTY = False
OVERFLOW_PENALTY = 10
CAPACITY = 20
EPS = 1e-8

params = 10
xi, vi, li, ai, deltai, v0i, bi, ti, s0i, wi = range(params)
archetypes = ARCHETYPE.reshape(1, params).copy()

_WINDOW = 4096  # ticks of arrival schedule handed to the device at a time


def inv_popcount(inv_i):
    return np.uint32(_inv_popcount(inv_i))


def cars_on_roads(leading, lastcar):
    """Cars per road from the ring indices (traffic_env.py:214-218); algorithms/greedy.py imports this."""
    leading, lastcar = np.asarray(leading), np.asarray(lastcar)
    return (lastcar - leading + (CAPACITY - 1) * (leading > lastcar)).astype(np.int32)


def clock_after(steps, ticks):
    """The np.float32 clock after `ticks` ticks of the reference's `self.steps += 1` (traffic_env.py:247): one float32
    add per tick, so the clock stops at 2^24 - the rule the device's clock follows too."""
    steps = np.float32(steps)
    for _ in range(int(ticks)):
        steps = np.float32(steps + np.float32(1))
    return steps


def _mode():
    try:
        return FLAGS.mode
    except AttributeError:  # alg_flags not imported: the reference would raise here (SURVEY.md section 5)
        return 'train'


class TrafficEnv(gym.Env):
    metadata = {'render.modes': ['human']}

    # ------------------------------------------------------------------ construction
    def set_graph(self, graph):
        self.viewer = None
        self.graph = graph
        r, i = graph.train_roads, graph.intersections
        self.action_space = GSpace([i], np.int32(2))
        self.observation_space = GSpace([2 * r + 2 * i], np.int32(1))
        self.obs = np.zeros(2 * r + 2 * i, dtype=np.int32)
        self.passed = self.obs[:r]
        self.detected = self.obs[r:2 * r]
        self.current_phase = self.obs[2 * r:2 * r + i]
        self.elapsed = self.obs[-i:]
        self.waiting = np.zeros(r, dtype=np.int32)
        self.rewards = np.zeros(i, dtype=np.float32)
        self.reward_size = self.rewards.size
        self.passed_dst = np.zeros(i, dtype=np.bool_)
        self.trip_times = []
        self.steps = np.float32(0)
        self.generated_cars = 0
        self._sim = None
        self._seed = None
        self._seeded = False
        self._done_u8 = np.zeros(1, np.uint8)
        self.reset_entrypoints()

    def seed_generator(self, seed=None):
        if seed is None:
            seed = int.from_bytes(os.urandom(4), "little")
        self._seed = seed
        self._seeded = True
        self._stream = None  # built lazily: FLAGS.cars_per_sec may still change (reset_entrypoints)
        self._win_snapshot = None
        if getattr(self, "_sim", None) is not None:
            self._sched_end = self._ticks_total  # drop what the old generator had scheduled ahead
            self._window = []

    def reset_entrypoints(self):
        if FLAGS.entry == "random":
            spec = int(np.random.randint(0b1111, dtype='uint32'))
        elif FLAGS.entry == "one":
            spec = 0b1110
        else:
            spec = 0
        self._spec = spec
        self.graph.generate_entrypoints(spec)
        FLAGS.cars_per_sec = FLAGS.local_cars_per_sec * self.graph.m * inv_popcount(spec)
        if getattr(self, "_sim", None) is not None and self._sim_key() != self._key:
            # the open sides changed.  The reference keeps its generator (same RandomState, same rate) and simply
            # draws future cars from the new entry list: rewind the pre-drawn window to the current tick first.
            consumed = self._ticks_total - self._sched_begin
            if getattr(self, "_stream", None) is not None:
                self._stream.restore(self._win_snapshot)
                self._stream.window(consumed)                      # re-draw what was executed, old entry list
                self._stream.entrypoints = np.asarray(self.graph.entrypoints)
            old = self._sim
            carry = (self._ticks_total, old.get_state(0, 1))
            old.close()
            self._sim = None
            self._device()                                         # new handle: new entry tables
            self._ticks_total = self._sched_begin = self._sched_end = 0
            self._sim.set_state(carry[1])
            self._mirror[:] = self.obs

    # ------------------------------------------------------------------ device plumbing
    def _sim_key(self):
        return (self.graph.m, self.graph.n, float(self.graph.len), float(FLAGS.rate), bool(FLAGS.learn_switch),
                self._spec, _mode() == 'validate')

    def _device(self):
        if self._sim is None:
            g = self.graph
            self._key = self._sim_key()
            self._sim = VecTrafficEnv(m=g.m, n=g.n, length=float(g.len), num_envs=1, rate=float(FLAGS.rate),
                                      remi=False, learn_switch=bool(FLAGS.learn_switch), arrivals="injected",
                                      validate=(_mode() == 'validate'),
                                      entry=self._spec, device=int(os.environ.get("TRAFFIC_B200_DEVICE", "0")))
            assert (self._sim.nexts == g.nexts).all() and (self._sim.entrypoints == g.entrypoints).all()
            self._sched_begin = self._sched_end = self._ticks_total = 0
            self._window = []
            self._sim.set_arrivals([[]])
            self._mirror = self.obs.copy()
        return self._sim

    def _ensure_schedule(self, ticks):
        """Keep the device's injected arrival window ahead of the arrival-process clock."""
        if self._ticks_total + ticks <= self._sched_end:
            return
        if not self._seeded:
            self.seed_generator()
        if self._stream is None:
            self._stream = ArrivalStream(self._seed, self.graph.entrypoints, FLAGS.cars_per_sec, FLAGS.rate,
                                         poisson=bool(FLAGS.poisson))
        # the window must start at the current clock: keep the not-yet-consumed tail of the old window
        consumed = self._ticks_total - self._sched_begin
        tail = self._window[consumed:] if self._sched_end > self._ticks_total else []
        # snapshot of the stream at the start of the new window (= at the current tick): rewind, replay what ran
        if getattr(self, "_win_snapshot", None) is not None and self._window:
            self._stream.restore(self._win_snapshot)
            self._stream.window(consumed)
            tail = []
        self._win_snapshot = self._stream.snapshot()
        fresh = self._stream.window(max(_WINDOW, ticks) - len(tail))
        self._window = tail + fresh
        self._sched_begin = self._ticks_total
        self._sched_end = self._sched_begin + len(self._window)
        self._sim.set_arrivals([self._window], first_tick=self._sched_begin)

    def _pull(self, obs_raw, rewards, ticks):
        if self._key[-1]:  # validate mode: trip times of the cars that left the map (traffic_env.py:154)
            self.trip_times.extend(np.float32(t) for t in self._sim.trip_times(clear=True)[1])
        self.obs[:] = obs_raw
        self._mirror[:] = obs_raw
        self.rewards[:] = rewards
        self._ticks_total += ticks
        self.steps = clock_after(self.steps, ticks)

    def _as_action(self, action):
        """Truthiness per intersection, with numpy broadcasting like the reference's logical_xor(current_phase, action)
        (traffic_env.py:229): a one-element action (UnGSpaceWrapper's unravelled index) applies to every light."""
        a = np.asarray(action).astype(bool)
        return np.broadcast_to(a.reshape(-1), (self.graph.intersections,)).reshape(1, -1)

    def _push_if_dirty(self):
        """`obs` aliases live state in the reference (current_phase, elapsed, detected are views the callers
        may write, e.g. to force a light phase).  If the host copy was modified since the last step, send
        it to the device before stepping."""
        r = self.graph.train_roads
        if np.array_equal(self.obs[r:], self._mirror[r:]):
            return
        st = self._sim.get_state(0, 1)
        st["obs"][0, r:] = self.obs[r:]
        self._sim.set_state(st)
        self._mirror[:] = self.obs

    # ------------------------------------------------------------------ gym API
    def _reset(self):
        sim = self._device()
        self.steps = np.float32(0)
        self.generated_cars = 0
        self.current_phase[:] = self.action_space.sample()
        sim.reset(init_phase=self.current_phase[None])
        self.elapsed[:] = 0
        self.passed[:] = 0
        self.passed_dst[:] = False
        self.waiting[:] = 0
        self._mirror[:] = self.obs
        return self.obs

    def _step(self, action):
        sim = self._device()
        self._ensure_schedule(1)
        self._push_if_dirty()
        obs, rew, done = sim.step_raw(self._as_action(action))
        self._pull(obs[0], rew[0], 1)
        return self.obs, self.rewards, bool(done[0]), None

    def step_repeated(self, action, repeat_count):
        """Repeater(repeat_count)._step fused into one launch (traffic_test.py:37-56): returns the float
        observation [passed summed | detected | elapsed/100 * (2*phase-1)], the summed env reward and done.

        The int32 `obs` views the callers hold (current_phase, elapsed, detected) are refreshed WITHOUT reading
        the device state back when all `repeat_count` ticks ran (no ring overflow): the light state of a constant
        action is a closed form of the tick count (traffic_env.py:225-232) and `detected` comes back in the float
        observation.  A step that overflowed (the tick loop stopped early) reads the state from the device."""
        sim = self._device()
        self._ensure_schedule(repeat_count)
        self._push_if_dirty()
        act = self._as_action(action)
        obs, rew, done = sim.step(act, k=repeat_count)
        r, i = self.graph.train_roads, self.graph.intersections
        if not done[0] and not self._key[-1] and not os.environ.get("TRAFFIC_B200_NO_HOST_MIRROR"):
            a = act[0].astype(np.int32)
            raw = self._mirror.copy()
            ph, el = raw[2 * r:2 * r + i], raw[2 * r + i:]
            if FLAGS.learn_switch:                       # the action toggles: elapsed restarts at every tick it is set
                el[:] = np.where(a != 0, 0, el + repeat_count)
                ph[:] = ph ^ (a * (repeat_count & 1))
            else:                                        # first tick: change = phase xor action, then `action` holds
                el[:] = (el + 1) * (ph == a) + (repeat_count - 1)
                ph[:] = a
            raw[:r] = 0      # per-tick `passed` of the last tick is not kept by the fused path
            raw[r:2 * r] = obs[0, r:2 * r].astype(np.int32)
            ticks = repeat_count
        else:
            st = sim.get_state(0, 1)
            raw = st["obs"][0]
            raw[:r] = 0
            # the ticks the launch ran, from the device's tick count (the clock stops at 2^24: its change is no count)
            ticks = int(sim.stats()["ticks"]) - self._ticks_total
        self._pull(raw, rew[0], ticks)
        return obs[0].copy(), self.rewards, bool(done[0])

    def cars_on_roads(self):
        c = self._device().cars_on_roads_flat()[0]
        g = self.graph
        return np.transpose(np.reshape(c[:g.train_roads], [4, g.m, g.n]), (1, 2, 0))

    def remi_reward(self):
        self.rewards[:] = self._device().remi_reward()[0]
        self.passed_dst[:] = False
        self.waiting[:] = 0
        return self.rewards

    def _render(self, mode='human', close=False):
        if close:
            return None
        raise NotImplementedError("the pyglet viewer of the reference (traffic_env.py:285-359) is not part of the B200 path")

    # ------------------------------------------------------------------ state snapshots (host copies)
    def _snapshot(self):
        return self._device().get_state(0, 1)

    @property
    def leading(self):
        return self._snapshot()["leading"][0]

    @property
    def lastcar(self):
        return self._snapshot()["lastcar"][0]

    @property
    def state(self):
        """float32[R, 10, 20] snapshot in the reference layout; only live slots and the leading slot carry data."""
        st = self._snapshot()
        R = self.graph.roads
        out = np.full((R, params, CAPACITY), np.nan, dtype=np.float32)
        out[:, xi, :] = st["x"][0]
        out[:, vi, :] = st["v"][0]
        for p in (li, ai, deltai, v0i, bi, ti, s0i):
            out[:, p, :] = ARCHETYPE[p]
        ld = st["leading"][0]
        out[np.arange(R), vi, ld] = 0.0
        out[np.arange(R), li, ld] = 0.0
        return out

    def sync_counters(self):
        """Refresh `waiting` / `passed_dst` (kept on the device between remi_reward calls)."""
        st = self._snapshot()
        self.waiting[:] = st["waiting"][0]
        self.passed_dst[:] = st["passed_dst"][0].astype(bool)
        self.generated_cars = int(self._device().stats()["cars_generated"])
        return self
