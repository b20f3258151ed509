"""VecTrafficEnv: E independent traffic-env instances advanced by one CUDA kernel launch.

Host-side mirror of the reference's TrafficEnv (gym_traffic/envs/traffic_env.py:221-394)
plus the Repeater/Remi wrappers that sit on its tick loop (traffic_test.py:27-64), for a
batch of env instances.  All simulation work happens in libtraffic_b200.so (sm_100a CUDA,
C ABI in include/traffic_b200.h); this class only marshals buffers.
"""
import ctypes as C

import numpy as np

from . import _lib
from ._lib import (TE_CTRL_GIVEN, TE_CTRL_GREEDY, TE_ARRIVALS_INJECTED, TE_ARRIVALS_NONE, TE_ARRIVALS_PHILOX, TE_AUTO_RESET, TE_CAP, TE_DEVICE,
                   TE_HOST, TE_LEARN_SWITCH, TE_ORDERED_TRANSFERS, TE_REMI, TE_VALIDATE, check)

ARCHETYPE = np.array([0.0, 11.11, 4.0, 3.0, 4.0, 13.89, 6.0, 2.0, 1.0, 0.0], dtype=np.float32)  # traffic_env.py:35-43


def inv_popcount(spec):
    """Open sides of the grid (traffic_env.py:180-185: popcount of the inverted low 4 bits)."""
    return bin((~int(spec)) & 0b1111).count("1")


def entry_spec_of(entry):
    if isinstance(entry, str):
        if entry == "all":
            return 0
        if entry == "one":
            return 0b1110  # traffic_env.py:391
        raise ValueError("entry must be 'all', 'one' or an integer side mask")
    return int(entry)


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return int(a.data_ptr())  # torch tensor


class WireResult(object):
    """Results of an actor step (or of the n actor steps of one launch) as they arrived in host memory: compact wire
    records.  `reward` f32[..., E, I], `done` u8[..., E], `passed` / `detected` u8[..., E, r] and `light` f32[..., E, I] are
    views into the page-locked record buffer; the float observation of the reference's Repeater (traffic_test.py:37-56:
    float32[2r + I] = passed | detected | light) is expanded LAZILY: `obs` expands everything on first access (C, cached),
    `obs_of(env_ids)` only the rows asked for.  Unpacking `obs, reward, done = result` works like the eager API."""

    def __init__(self, env, buf):
        self._env, self._buf, self._obs = env, buf, None
        v = env._wire_views(buf)
        self.passed, self.detected, self.light, self.reward, self.done = (v[k] for k in ("passed", "detected", "light", "reward", "done"))

    @property
    def obs(self):
        if self._obs is None:
            e = self._env
            lead = self._buf.shape[:-2]
            n = int(np.prod(lead)) * e.num_envs if lead else e.num_envs
            obs = np.empty(lead + (e.num_envs, e.obs_len), np.float32)
            rew = np.empty(lead + (e.num_envs, e.intersections), np.float32)
            done = np.empty(lead + (e.num_envs,), np.uint8)
            check(e._L.te_expand_wire(e._h, self._buf.ctypes.data, n, obs.ctypes.data, rew.ctypes.data, done.ctypes.data))
            self._obs = obs
        return self._obs

    def obs_of(self, env_ids, step=None):
        """float32[len(env_ids), 2r + I] for the given envs (of actor step `step` for a multi-step result)."""
        ids = np.asarray(env_ids, dtype=np.int64).reshape(-1)
        sel = (ids,) if step is None else (step, ids)
        return np.concatenate([self.passed[sel].astype(np.float32), self.detected[sel].astype(np.float32), self.light[sel]], axis=-1)

    def __iter__(self):
        return iter((self.obs, self.reward, self.done))


class VecTrafficEnv(object):
    def __init__(self, m=3, n=3, length=250.0, num_envs=1, rate=0.5, ticks_per_step=10, remi=True,
                 learn_switch=False, auto_reset=False, validate=False, arrivals="philox", local_cars_per_sec=0.12,
                 entry="all", seed=0, env_id_base=0, device=0, episode_len=0, gamma=0.8, archetype=None,
                 ordered_transfers=False):
        L = _lib.load()
        cfg = _lib.default_config()
        cfg.m, cfg.n, cfg.length, cfg.rate = int(m), int(n), float(length), float(rate)
        cfg.num_envs, cfg.env_id_base, cfg.device = int(num_envs), int(env_id_base), int(device)
        cfg.flags = ((TE_REMI if remi else 0) | (TE_LEARN_SWITCH if learn_switch else 0) |
                     (TE_AUTO_RESET if auto_reset else 0) | (TE_VALIDATE if validate else 0) |
                     (TE_ORDERED_TRANSFERS if ordered_transfers else 0))
        cfg.entry_spec = entry_spec_of(entry)
        cfg.arrival_mode = {"philox": TE_ARRIVALS_PHILOX, "injected": TE_ARRIVALS_INJECTED,
                            "none": TE_ARRIVALS_NONE}[arrivals]
        # FLAGS.cars_per_sec = local_cars_per_sec * m * inv_popcount(spec)  (traffic_env.py:394)
        self.cars_per_sec = float(local_cars_per_sec) * int(m) * inv_popcount(cfg.entry_spec)
        cfg.cars_per_tick = self.cars_per_sec * float(rate)
        cfg.seed, cfg.episode_len, cfg.gamma = int(seed), int(episode_len), float(gamma)
        arch = ARCHETYPE if archetype is None else np.asarray(archetype, dtype=np.float32)
        for i in range(_lib.TE_PARAMS):
            cfg.archetype[i] = float(arch[i])
        self._L = L
        self._h = C.c_void_p()
        check(L.te_create(C.byref(cfg), C.byref(self._h)))
        d = _lib.TeDims()
        check(L.te_get_dims(self._h, C.byref(d)))
        self.m, self.n = d.m, d.n
        self.intersections, self.train_roads, self.roads = d.intersections, d.train_roads, d.roads
        self.roads_padded = d.roads_padded
        self.num_envs, self.num_entry = d.num_envs, d.num_entry
        self.obs_raw_len, self.obs_len = d.obs_raw, d.obs_actor
        self.ticks_per_step = int(ticks_per_step)
        self.device = int(device)
        self.remi = bool(remi)
        self.auto_reset = bool(auto_reset)
        wl = _lib.TeWireLayout()
        check(L.te_wire_layout(self._h, C.byref(wl)))
        self.wire = wl
        self.dest = np.empty(self.roads, np.int32)
        self.nexts = np.empty(self.roads, np.int32)
        self.phases = np.empty(self.roads, np.int32)
        self.entrypoints = np.empty(self.num_entry, np.int32)
        check(L.te_get_topology(self._h, self.dest.ctypes.data, self.nexts.ctypes.data, self.phases.ctypes.data,
                                self.entrypoints.ctypes.data))
        E, I = self.num_envs, self.intersections
        # result / action buffers live in page-locked host memory owned by this object
        self._pinned = []
        self._obs = self._host_array((E, self.obs_len), np.float32)
        self._obs_raw = self._host_array((E, self.obs_raw_len), np.int32)
        self._reward = self._host_array((E, I), np.float32)
        self._done = self._host_array((E,), np.uint8)
        self._act = self._host_array((E, I), np.uint8)
        self._cars = self._host_array((E, self.roads), np.int32)
        self._wire_buf = None   # page-locked record buffer, allocated on first step_wire()

    def _host_array(self, shape, dtype):
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        ptr = C.c_void_p()
        check(self._L.te_host_alloc(max(n, 16), C.byref(ptr)))
        self._pinned.append(ptr)
        buf = (C.c_ubyte * max(n, 16)).from_address(ptr.value)
        return np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._L.te_destroy(self._h)
            self._h = C.c_void_p()
            for name in ("_obs", "_obs_raw", "_reward", "_done", "_act", "_cars", "_wire_buf", "_multi", "_multi_wire"):
                setattr(self, name, None)
            for ptr in self._pinned:
                self._L.te_host_free(ptr)
            self._pinned = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ------------------------------------------------------------ helpers
    def _actions(self, actions):
        """Any array-like of truthy values (bool from A3C, int32 from DQN, float64 from `fixed`, ...) -> the page-locked
        uint8 action buffer.  Bytes are copied as they are: the device tests `!= 0` itself."""
        a = np.asarray(actions)
        if a.dtype == np.bool_ or a.dtype == np.uint8:
            np.copyto(self._act.view(a.dtype), a.reshape(self.num_envs, self.intersections))
        else:
            np.not_equal(a.reshape(self.num_envs, self.intersections), 0, out=self._act.view(np.bool_))
        return self._act

    # ------------------------------------------------------------ reference API, batched
    def reset(self, mask=None, init_phase=None):
        """TrafficEnv._reset for the masked envs (all when mask is None)."""
        mk = None if mask is None else np.ascontiguousarray(np.asarray(mask).astype(bool), dtype=np.uint8)
        ip = None if init_phase is None else np.ascontiguousarray(
            np.asarray(init_phase).astype(bool).reshape(self.num_envs, self.intersections), dtype=np.uint8)
        check(self._L.te_reset(self._h, _ptr(mk), _ptr(ip), TE_HOST, None))

    def set_arrivals(self, schedules, first_tick=0):
        """schedules[e][t] = ordered entry-road ids of env e at arrival-process tick first_tick + t."""
        E = self.num_envs
        assert len(schedules) == E
        horizon = max(len(s) for s in schedules)
        off = np.zeros((E, horizon + 1), dtype=np.int64)
        roads = []
        base = 0
        for e, s in enumerate(schedules):
            off[e, 0] = base
            for t in range(horizon):
                if t < len(s):
                    roads.extend(int(x) for x in s[t])
                    base += len(s[t])
                off[e, t + 1] = base
        roads = np.asarray(roads, dtype=np.int16)
        self.set_arrivals_csr(off, roads, horizon, first_tick)

    def set_arrivals_csr(self, offsets, roads, horizon, first_tick=0):
        offsets = np.ascontiguousarray(offsets, dtype=np.int64)
        roads = np.ascontiguousarray(roads, dtype=np.int16)
        assert offsets.size == self.num_envs * (horizon + 1)
        nroads = roads.size
        if roads.size == 0:
            roads = np.zeros(1, np.int16)
        check(self._L.te_set_arrivals(self._h, offsets.ctypes.data, roads.ctypes.data, int(nroads), int(first_tick),
                                      int(horizon)))

    def step(self, actions, k=None, lazy=False):
        """One actor step (Repeater(k) [+ Remi]) for every env; returns (obs, reward, done) host arrays
        that are reused between calls, like the reference's in-place obs/rewards buffers.  lazy=True: a WireResult - the
        results stay in the compact form they crossed PCIe in and the float observation is expanded on demand."""
        if lazy:
            self.step_wire(actions, k)
            return WireResult(self, self._wire_buf)
        a = self._actions(actions)
        k = self.ticks_per_step if k is None else int(k)
        check(self._L.te_step(self._h, a.ctypes.data, k, self._obs.ctypes.data, self._reward.ctypes.data,
                              self._done.ctypes.data, TE_HOST, None))
        return self._obs, self._reward, self._done

    def step_masked(self, actions, env_mask, k=None):
        """step() for the envs whose mask entry is non-zero only (te_step_masked); the rows of the others in the returned
        (reused) arrays keep what they held."""
        a = self._actions(actions)
        m = np.ascontiguousarray(np.asarray(env_mask).astype(bool), dtype=np.uint8)
        k = self.ticks_per_step if k is None else int(k)
        check(self._L.te_step_masked(self._h, a.ctypes.data, m.ctypes.data, k, self._obs.ctypes.data,
                                     self._reward.ctypes.data, self._done.ctypes.data, TE_HOST, None))
        return self._obs, self._reward, self._done

    def _controller_spacing(self, spacing, n_steps, controller):
        """te_set_controller_spacing when it changed; the action buffer te_step_multi reads / writes."""
        spacing = 0 if (spacing is None or controller != "greedy") else int(spacing)
        if spacing != getattr(self, "_spacing", 0):
            check(self._L.te_set_controller_spacing(self._h, spacing))
            self._spacing = spacing
        if spacing == 0:
            return self._act
        ndec = (n_steps + spacing - 1) // spacing
        if getattr(self, "_act_multi_n", 0) < ndec:
            self._act_multi = self._host_array((ndec, self.num_envs, self.intersections), np.uint8)
            self._act_multi_n = ndec
        return self._act_multi[:ndec]

    def step_multi(self, n_steps, actions=None, controller="greedy", k=None, lazy=False, spacing=None):
        """n_steps actor steps in one launch (te_step_multi), host buffers: returns
        (actions uint8[E, I], obs float[n_steps, E, 2r+I], reward float[n_steps, E, I], done uint8[n_steps, E]).
        controller "greedy": the kernel evaluates algorithms/greedy.py:14-16 at launch - and again every `spacing` actor
        steps when spacing is given (greedy.py's --spacing; actions is then uint8[ceil(n_steps / spacing), E, I]);
        "given": `actions` holds for the whole launch.  lazy=True: (actions, WireResult) - see step()."""
        k = self.ticks_per_step if k is None else int(k)
        n_steps = int(n_steps)
        if lazy:
            act, _ = self.step_multi_wire(n_steps, actions, controller, k, spacing)
            return act, WireResult(self, self._multi_wire[:n_steps])
        if getattr(self, "_multi_n", 0) < n_steps:
            E, I = self.num_envs, self.intersections
            self._multi = (self._host_array((n_steps, E, self.obs_len), np.float32),
                           self._host_array((n_steps, E, I), np.float32), self._host_array((n_steps, E), np.uint8))
            self._multi_n = n_steps
        obs, rew, done = (x[:n_steps] for x in self._multi)
        act = self._controller_spacing(spacing, n_steps, controller)
        if controller == "greedy":
            ctrl = TE_CTRL_GREEDY
        else:
            ctrl = TE_CTRL_GIVEN
            self._actions(actions)
        check(self._L.te_step_multi(self._h, n_steps, ctrl, act.ctypes.data, k, obs.ctypes.data, rew.ctypes.data,
                                    done.ctypes.data, TE_HOST, None))
        return act, obs, rew, done

    def _wire_views(self, w):
        """dict of views into a record buffer [..., E, stride]."""
        r, I, wl = self.train_roads, self.intersections, self.wire
        return {"passed": w[..., wl.passed:wl.passed + r], "detected": w[..., wl.detected:wl.detected + r],
                "light": w[..., wl.light:wl.light + 4 * I].view(np.float32),
                "reward": w[..., wl.reward:wl.reward + 4 * I].view(np.float32), "done": w[..., wl.done]}

    def step_multi_wire(self, n_steps, actions=None, controller="greedy", k=None, spacing=None):
        """step_multi with the results left as wire records: (actions, dict of views [n_steps, E, ...])."""
        k = self.ticks_per_step if k is None else int(k)
        n_steps = int(n_steps)
        if getattr(self, "_multi_wire_n", 0) < n_steps:
            self._multi_wire = self._host_array((n_steps, self.num_envs, self.wire.stride), np.uint8)
            self._multi_wire_n = n_steps
        buf = self._multi_wire[:n_steps]
        act = self._controller_spacing(spacing, n_steps, controller)
        if controller != "greedy":
            self._actions(actions)
        check(self._L.te_step_multi_wire(self._h, n_steps, TE_CTRL_GREEDY if controller == "greedy" else TE_CTRL_GIVEN,
                                         act.ctypes.data, k, buf.ctypes.data, TE_HOST, None))
        return act, self._wire_views(buf)

    def step_multi_device(self, n_steps, actions, obs, reward, done, controller="greedy", k=None, stream=None, spacing=None):
        """te_step_multi on caller-owned device buffers ([n_steps, E, ...] outputs; `actions` [E, I] - with spacing:
        [ceil(n_steps / spacing), E, I] - is written by the greedy controller or read when controller == "given");
        asynchronous."""
        k = self.ticks_per_step if k is None else int(k)
        self._controller_spacing(spacing, int(n_steps), controller)
        check(self._L.te_step_multi(self._h, int(n_steps), TE_CTRL_GREEDY if controller == "greedy" else TE_CTRL_GIVEN,
                                    _ptr(actions), k, _ptr(obs), _ptr(reward), _ptr(done), TE_DEVICE, stream))

    def step_wire(self, actions, k=None):
        """step() with the results left in the compact wire format (te_step_wire): a dict of views into one page-locked
        record buffer - passed u8[E, r], detected u8[E, r], light f32[E, I], reward f32[E, I], done u8[E] - for consumers
        that feed a policy directly; `expand_wire()` gives the float arrays of step()."""
        a = self._actions(actions)
        k = self.ticks_per_step if k is None else int(k)
        E, r, I, wl = self.num_envs, self.train_roads, self.intersections, self.wire
        if self._wire_buf is None:
            self._wire_buf = self._host_array((E, wl.stride), np.uint8)
        check(self._L.te_step_wire(self._h, a.ctypes.data, k, self._wire_buf.ctypes.data, TE_HOST, None))
        return self._wire_views(self._wire_buf)

    def expand_wire(self, env_begin=0, count=None):
        """Float (obs, reward, done) of step() from the records of the last step_wire()."""
        count = self.num_envs - env_begin if count is None else count
        rec = self._wire_buf[env_begin:env_begin + count]
        obs, rew, done = self._obs[env_begin:env_begin + count], self._reward[env_begin:env_begin + count], self._done[env_begin:env_begin + count]
        check(self._L.te_expand_wire(self._h, rec.ctypes.data, count, obs.ctypes.data, rew.ctypes.data, done.ctypes.data))
        return obs, rew, done

    def d2h_bytes_per_step(self, k=None):
        """Bytes te_step(TE_HOST) moves device -> host per actor step."""
        k = self.ticks_per_step if k is None else int(k)
        E = self.num_envs
        if k <= self.wire.max_k_ticks:
            return E * self.wire.stride
        return E * (self.obs_len * 4 + self.intersections * 4 + 1)

    def host_float_dma(self):
        """True when te_step(TE_HOST) delivers float outputs through the copy engine instead of expanding wire records
        on the host, as the library decided at te_create (few host cores per GPU, or TE_HOST_FLOAT_DMA=1)."""
        return bool(self.wire.host_float_dma)

    def host_path_note(self):
        return ("compact wire records of %d B per env (u8 passed / detected, f32 light / reward, u8 done) expanded on the "
                "host into float obs[%d] / reward[%d] / done by the handle's helper threads" %
                (self.wire.stride, self.obs_len, self.intersections))

    def step_raw(self, actions):
        """One physics tick (bare TrafficEnv._step); obs is int32 passed|detected|phase|elapsed."""
        a = self._actions(actions)
        check(self._L.te_step_raw(self._h, a.ctypes.data, self._obs_raw.ctypes.data, self._reward.ctypes.data,
                                  self._done.ctypes.data, TE_HOST, None))
        return self._obs_raw, self._reward, self._done

    def step_device(self, actions, obs, reward, done, k=None, stream=None):
        """Same as step() on caller-owned device buffers (torch CUDA tensors or raw pointers); asynchronous."""
        k = self.ticks_per_step if k is None else int(k)
        check(self._L.te_step(self._h, _ptr(actions), k, _ptr(obs), _ptr(reward), _ptr(done), TE_DEVICE, stream))

    def step_pinned(self, actions, obs, reward, done, k=None):
        """step() on caller-owned HOST buffers (e.g. pinned torch tensors); synchronous."""
        k = self.ticks_per_step if k is None else int(k)
        check(self._L.te_step(self._h, _ptr(actions), k, _ptr(obs), _ptr(reward), _ptr(done), TE_HOST, None))

    def remi_reward(self):
        out = np.empty((self.num_envs, self.intersections), np.float32)
        check(self._L.te_remi_reward(self._h, out.ctypes.data, TE_HOST, None))
        return out

    def cars_on_roads_flat(self):
        check(self._L.te_cars_on_roads(self._h, self._cars.ctypes.data, TE_HOST, None))
        return self._cars

    def cars_on_roads(self):
        """[E, m, n, 4] like TrafficEnv.cars_on_roads (traffic_env.py:255-257)."""
        c = self.cars_on_roads_flat()[:, :self.train_roads]
        return np.transpose(c.reshape(self.num_envs, 4, self.m, self.n), (0, 2, 3, 1))

    def host_buffer(self, shape, dtype):
        """A page-locked host array owned by this env (te_host_alloc): for actions and results that cross PCIe every step."""
        return self._host_array(tuple(shape), dtype)

    def greedy_actions(self, out=None, stream=None):
        """algorithms/greedy.py:14-16 for every env; a new host array by default, into the host array `out` (uint8[E, I],
        C-contiguous; page-locked memory from host_buffer() avoids a staging copy), or into a device buffer `out`."""
        if out is None or isinstance(out, np.ndarray):
            if out is None:
                out = np.empty((self.num_envs, self.intersections), np.uint8)
            assert out.dtype == np.uint8 and out.flags.c_contiguous and out.size == self.num_envs * self.intersections
            check(self._L.te_greedy_actions(self._h, out.ctypes.data, TE_HOST, None))
            return out
        check(self._L.te_greedy_actions(self._h, _ptr(out), TE_DEVICE, stream))
        return out

    # ------------------------------------------------------------ state / stats
    def get_state(self, env_begin=0, count=None):
        count = self.num_envs - env_begin if count is None else count
        R, r, I = self.roads, self.train_roads, self.intersections
        st = dict(leading=np.empty((count, R), np.int32), lastcar=np.empty((count, R), np.int32),
                  x=np.empty((count, R, TE_CAP), np.float32), v=np.empty((count, R, TE_CAP), np.float32),
                  obs=np.empty((count, 2 * r + 2 * I), np.int32), waiting=np.empty((count, r), np.int32),
                  passed_dst=np.empty((count, I), np.uint8), steps=np.empty(count, np.float32))
        check(self._L.te_get_state(self._h, env_begin, count, *[st[k].ctypes.data for k in
                                   ("leading", "lastcar", "x", "v", "obs", "waiting", "passed_dst", "steps")]))
        return st

    def set_state(self, st, env_begin=0):
        count = st["leading"].shape[0]
        arrs = [np.ascontiguousarray(st[k], dtype=dt) for k, dt in
                (("leading", np.int32), ("lastcar", np.int32), ("x", np.float32), ("v", np.float32),
                 ("obs", np.int32), ("waiting", np.int32), ("passed_dst", np.uint8), ("steps", np.float32))]
        check(self._L.te_set_state(self._h, env_begin, count, *[a.ctypes.data for a in arrs]))

    # ------------------------------------------------------------ snapshot records
    @property
    def snapshot_layout(self):
        """Byte layout of one snapshot record (te_snapshot_layout): stride and the offsets of x, v, w (-1 without
        validate), phase, elapsed, passed_dst and the library-private scalars."""
        lay = _lib.TeSnapshotLayout()
        check(self._L.te_snapshot_layout(self._h, C.byref(lay)))
        return lay

    def _env_ids(self, env_ids, count=None):
        """(int32 id array or None, count) for te_save_envs / te_load_envs; None stands for envs [0, count)."""
        if env_ids is None:
            return None, self.num_envs if count is None else count
        ids = np.ascontiguousarray(np.asarray(env_ids, dtype=np.int64).reshape(-1), dtype=np.int32)
        return ids, ids.size

    def save_envs(self, env_ids=None, out=None, stream=None):
        """Snapshot records of the listed envs (all when env_ids is None; duplicates allowed), one row of
        snapshot_layout.stride bytes per id.  out None: a new uint8[count, stride] host array (synchronous); a host array:
        filled in place; a CUDA torch tensor or a raw device pointer: written on the device, asynchronously on `stream`
        (a cudaStream_t as int, None = the handle's stream) after the steps queued there before it."""
        ids, count = self._env_ids(env_ids)
        stride = self.snapshot_layout.stride
        if out is None or isinstance(out, np.ndarray):
            if out is None:
                out = np.empty((count, stride), np.uint8)
            assert out.flags.c_contiguous and out.nbytes == count * stride, "out must be C-contiguous [count, stride] bytes"
            check(self._L.te_save_envs(self._h, _ptr(ids), count, out.ctypes.data, TE_HOST, None))
            return out
        if not isinstance(out, int):
            assert out.is_cuda and out.is_contiguous() and out.numel() * out.element_size() >= count * stride, \
                "out must be a contiguous CUDA tensor of at least count * stride bytes"
        check(self._L.te_save_envs(self._h, _ptr(ids), count, out if isinstance(out, int) else _ptr(out), TE_DEVICE,
                                   stream))
        return out

    def load_envs(self, records, env_ids=None):
        """Load snapshot records (a host array or CUDA torch tensor of [count, stride] bytes) into the listed envs, record j
        into env env_ids[j] (envs [0, count) when env_ids is None).  Synchronous; every record is checked first, and a bad
        one raises TrafficB200Error with every env left as it was."""
        stride = self.snapshot_layout.stride
        if isinstance(records, np.ndarray):
            rec = np.ascontiguousarray(records).view(np.uint8).reshape(-1)
            mem, ptr, nbytes = TE_HOST, rec.ctypes.data, rec.nbytes
        else:
            assert records.is_cuda and records.is_contiguous(), "device records must be a contiguous CUDA tensor"
            mem, ptr, nbytes = TE_DEVICE, _ptr(records), records.numel() * records.element_size()
        ids, count = self._env_ids(env_ids, nbytes // stride)
        if nbytes < count * stride or (env_ids is None and nbytes != count * stride):
            raise ValueError("records hold %d bytes; %d records of %d bytes expected" % (nbytes, count, stride))
        check(self._L.te_load_envs(self._h, _ptr(ids), count, ptr, mem, None))

    def trip_times(self, clear=True):
        """Validate mode: (env ids, trip times in seconds) of the cars that left the map since the last clear."""
        n = C.c_int64()
        check(self._L.te_get_trip_times(self._h, None, None, 0, C.byref(n), 0))
        envs = np.empty(n.value, np.int32)
        trips = np.empty(n.value, np.float32)
        rc = check(self._L.te_get_trip_times(self._h, envs.ctypes.data, trips.ctypes.data, n.value, C.byref(n), int(clear)))
        if rc > 0:
            import warnings
            warnings.warn(self._L.te_last_error().decode("utf-8", "replace"))
        return envs, trips

    def is_tame(self):
        """True while the handle runs the kernels without the per-car validity predicate (te_is_tame)."""
        t = C.c_int32(0)
        check(self._L.te_is_tame(self._h, C.byref(t), None))
        return bool(t.value)

    def tame_speed_cap(self):
        """Largest car speed te_set_state accepts without leaving the tame mode (0.0: archetype outside the ranges)."""
        t, cap = C.c_int32(0), C.c_float(0)
        check(self._L.te_is_tame(self._h, C.byref(t), C.byref(cap)))
        return float(cap.value)

    def stats(self):
        s = _lib.TeStats()
        check(self._L.te_get_stats(self._h, C.byref(s)))
        return {k: getattr(s, k) for k, _ in s._fields_}

    def last_kernel_ms(self):
        ms = C.c_float()
        check(self._L.te_last_kernel_ms(self._h, C.byref(ms)))
        return ms.value

    def stage_bandwidth(self, repeats=5):
        """GB/s of the step kernel's bulk-TMA stage-in + flush with no ticks in between (te_stage_bandwidth)."""
        out = C.c_double()
        check(self._L.te_stage_bandwidth(self._h, int(repeats), C.byref(out)))
        return out.value

    def synchronize(self):
        check(self._L.te_synchronize(self._h))


def idm_arithmetic_peak(device=0, rate=0.5, archetype=None, iters=4000, form=-1, warps_per_sm=None):
    """vehicle-updates/s of the IDM arithmetic alone, registers only, every lane busy (te_idm_peak_form).  form -1: the
    form the step kernels run for this archetype on a tame handle (5 or 0); 0: the general checked form (the denominator
    of the round-1 figures); 5: the tame form.  Any other form raises.  warps_per_sm None: the better of 32 warps per SM
    (the step kernels' occupancy) and 64."""
    L = _lib.load()
    arch = np.ascontiguousarray(ARCHETYPE if archetype is None else archetype, dtype=np.float32)
    best = 0.0
    for w in ((32, 0) if warps_per_sm is None else (int(warps_per_sm),)):
        out = C.c_double()
        check(L.te_idm_peak_form(int(device), arch.ctypes.data, float(rate), int(iters), int(form), w, C.byref(out)))
        best = max(best, out.value)
    return best
