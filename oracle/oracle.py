"""ctypes binding of oracle/libtraffic_oracle.so - TEST INFRASTRUCTURE ONLY.

The CPU restatement of the reference tick (oracle/traffic_oracle.c).  Imported
by tests/, __graft_entry__.smoke() and bench.py's cpu_baseline/--impl reference
legs as the *checker* / reported baseline; never by traffic_env_b200/.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libtraffic_oracle.so")
_lib = None

PARAMS, CAP = 10, 20


def build(force=False):
    src = os.path.join(_HERE, "traffic_oracle.c")
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", _HERE] + (["-B"] if force else []))
    return _SO


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_SO)
        vp, i32, f32 = C.c_void_p, C.c_int, C.c_float
        pi = C.POINTER(C.c_int)
        pf = C.POINTER(C.c_float)
        L.to_create.restype = vp
        L.to_create.argtypes = [i32, i32, f32, f32, i32, i32]
        L.to_destroy.argtypes = [vp]
        L.to_reset.argtypes = [vp, pi]
        L.to_step.restype = i32
        L.to_step.argtypes = [vp, pi, pi, i32]
        L.to_remi.argtypes = [vp]
        L.to_cars_on_roads.argtypes = [vp, pi]
        L.to_generate_entrypoints.argtypes = [vp, C.c_uint]
        L.to_dim.restype = i32
        L.to_dim.argtypes = [vp, i32]
        for name, rt in (("to_state", pf), ("to_leading", pi), ("to_lastcar", pi), ("to_obs", pi),
                         ("to_waiting", pi), ("to_rewards", pf), ("to_passed_dst", C.POINTER(C.c_ubyte)),
                         ("to_dest", pi), ("to_nexts", pi), ("to_phases", pi), ("to_entry", pi)):
            getattr(L, name).restype = rt
            getattr(L, name).argtypes = [vp]
        L.to_steps.restype = f32
        L.to_steps.argtypes = [vp]
        L.to_set_steps.argtypes = [vp, f32]
        for name in ("to_generated", "to_vehicle_updates", "to_overflows"):
            getattr(L, name).restype = C.c_long
            getattr(L, name).argtypes = [vp]
        L.to_trip_times.restype = C.c_long
        L.to_trip_times.argtypes = [vp, C.POINTER(C.c_double), C.c_long]
        L.to_set_archetype.argtypes = [vp, pf]
        L.to_powf_restated.restype = f32
        L.to_powf_restated.argtypes = [f32, f32]
        L.to_powf_libm.restype = f32
        L.to_powf_libm.argtypes = [f32, f32]
        L.to_powf_compare.restype = C.c_long
        L.to_powf_compare.argtypes = [pf, C.c_long, f32, C.POINTER(C.c_long)]
        L.to_sim_kernel.argtypes = [f32, f32, f32, f32, pf, pf, pf]
        L.to_sim_bulk.argtypes = [f32, pf, pf, pf, pf, pf, pf, C.c_long, pf, pf]
        L.to_powf_bulk.argtypes = [pf, f32, C.c_long, pf]
        L.to_philox4x32_10.argtypes = [C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]
        L.to_philox_seed.argtypes = [vp, C.c_uint32, C.c_uint32, C.POINTER(C.c_uint32), i32]
        L.to_philox_arrivals.restype = i32
        L.to_philox_arrivals.argtypes = [vp, pi, i32]
        L.to_actor_step_philox.restype = i32
        L.to_actor_step_philox.argtypes = [vp, pi, i32, i32, pf, pf]
        _lib = L
    return _lib


def _view(ptr, shape, dtype):
    n = int(np.prod(shape))
    arr = np.ctypeslib.as_array(ptr, shape=(n,))
    return arr.view(dtype).reshape(shape) if arr.dtype != dtype else arr.reshape(shape)


class OracleEnv(object):
    """Single env with the reference's attribute names (traffic_env.py:361-382)."""

    def __init__(self, m=3, n=3, length=250.0, rate=0.5, learn_switch=False, validate=False):
        L = lib()
        self._L = L
        self._h = L.to_create(m, n, float(length), float(rate), int(learn_switch), int(validate))
        self.m, self.n = m, n
        self.intersections = L.to_dim(self._h, 5)
        self.train_roads = L.to_dim(self._h, 3)
        self.roads = L.to_dim(self._h, 4)
        R, r, I = self.roads, self.train_roads, self.intersections
        self.state = _view(L.to_state(self._h), (R, PARAMS, CAP), np.float32)
        self.leading = _view(L.to_leading(self._h), (R,), np.int32)
        self.lastcar = _view(L.to_lastcar(self._h), (R,), np.int32)
        self.obs = _view(L.to_obs(self._h), (2 * r + 2 * I,), np.int32)
        self.passed = self.obs[:r]
        self.detected = self.obs[r:2 * r]
        self.current_phase = self.obs[2 * r:2 * r + I]
        self.elapsed = self.obs[2 * r + I:]
        self.waiting = _view(L.to_waiting(self._h), (r,), np.int32)
        self.rewards = _view(L.to_rewards(self._h), (I,), np.float32)
        self.passed_dst = _view(L.to_passed_dst(self._h), (I,), np.uint8)
        self.dest = _view(L.to_dest(self._h), (R,), np.int32)
        self.nexts = _view(L.to_nexts(self._h), (R,), np.int32)
        self.phases = _view(L.to_phases(self._h), (R,), np.int32)
        self._gap_cdf = None

    def __del__(self):
        try:
            self._L.to_destroy(self._h)
        except Exception:
            pass

    @property
    def entrypoints(self):
        ne = self._L.to_dim(self._h, 6)
        return _view(self._L.to_entry(self._h), (2 * self.m + 2 * self.n,), np.int32)[:ne].copy()

    def generate_entrypoints(self, spec):
        self._L.to_generate_entrypoints(self._h, int(spec))

    def reset(self, init_phase=None):
        if init_phase is None:
            self._L.to_reset(self._h, None)
        else:
            p = np.ascontiguousarray(init_phase, dtype=np.int32)
            self._L.to_reset(self._h, p.ctypes.data_as(C.POINTER(C.c_int)))

    def step(self, action, arrivals=()):
        a = np.ascontiguousarray(np.asarray(action).astype(bool), dtype=np.int32)
        ar = np.ascontiguousarray(arrivals, dtype=np.int32)
        return bool(self._L.to_step(self._h, a.ctypes.data_as(C.POINTER(C.c_int)),
                                    ar.ctypes.data_as(C.POINTER(C.c_int)), int(ar.size)))

    def remi_reward(self):
        self._L.to_remi(self._h)
        return self.rewards

    def cars_on_roads_flat(self):
        out = np.empty(self.roads, dtype=np.int32)
        self._L.to_cars_on_roads(self._h, out.ctypes.data_as(C.POINTER(C.c_int)))
        return out

    def cars_on_roads(self):
        return np.transpose(np.reshape(self.cars_on_roads_flat()[:self.train_roads], [4, self.m, self.n]), (1, 2, 0))

    @property
    def steps(self):
        return self._L.to_steps(self._h)

    @steps.setter
    def steps(self, value):
        """Start the np.float32 clock anywhere (as a reference env's `steps` attribute can be set)."""
        self._L.to_set_steps(self._h, float(np.float32(value)))

    @property
    def generated_cars(self):
        return self._L.to_generated(self._h)

    @property
    def vehicle_updates(self):
        return self._L.to_vehicle_updates(self._h)

    @property
    def overflows(self):
        return self._L.to_overflows(self._h)

    def trip_times(self):
        n = self._L.to_trip_times(self._h, None, 0)
        out = np.empty(n, dtype=np.float64)
        if n:
            self._L.to_trip_times(self._h, out.ctypes.data_as(C.POINTER(C.c_double)), n)
        return out

    def set_archetype(self, arch):
        a = np.ascontiguousarray(arch, dtype=np.float32)
        assert a.size == PARAMS
        self._L.to_set_archetype(self._h, a.ctypes.data_as(C.POINTER(C.c_float)))

    # ---- counter-based arrivals (shared definition with the CUDA path)
    def philox_seed(self, seed, env_id, gap_cdf):
        self._gap_cdf = np.ascontiguousarray(gap_cdf, dtype=np.uint32)  # keep alive
        self._L.to_philox_seed(self._h, int(seed), int(env_id),
                               self._gap_cdf.ctypes.data_as(C.POINTER(C.c_uint32)), int(self._gap_cdf.size))

    def philox_arrivals(self, cap=4096):
        buf = np.empty(cap, dtype=np.int32)
        n = self._L.to_philox_arrivals(self._h, buf.ctypes.data_as(C.POINTER(C.c_int)), cap)
        return buf[:n].copy()

    def actor_step_philox(self, action, K, use_remi=True):
        r, I = self.train_roads, self.intersections
        a = np.ascontiguousarray(np.asarray(action).astype(bool), dtype=np.int32)
        obs = np.empty(2 * r + I, dtype=np.float32)
        rew = np.empty(I, dtype=np.float32)
        done = self._L.to_actor_step_philox(self._h, a.ctypes.data_as(C.POINTER(C.c_int)), int(K), int(use_remi),
                                            obs.ctypes.data_as(C.POINTER(C.c_float)),
                                            rew.ctypes.data_as(C.POINTER(C.c_float)))
        return obs, rew, bool(done)

    def live_state(self):
        """Ring-order walk of live slots, road-major (x, v) as float32 arrays."""
        xs, vs = [], []
        for e in range(self.roads):
            s = int(self.leading[e])
            while s != int(self.lastcar[e]):
                s = 1 if s + 1 >= CAP else s + 1
                xs.append(self.state[e, 0, s])
                vs.append(self.state[e, 1, s])
        return np.asarray(xs, dtype=np.float32), np.asarray(vs, dtype=np.float32)


def powf_compare(x, y):
    """#mismatches between host libm powf and the restated glibc algorithm."""
    L = lib()
    x = np.ascontiguousarray(x, dtype=np.float32)
    first = C.c_long(-1)
    bad = L.to_powf_compare(x.ctypes.data_as(C.POINTER(C.c_float)), x.size, float(y), C.byref(first))
    return int(bad), int(first.value)


def sim_one(rate, xL, vL, lL, x, v, arch):
    L = lib()
    cx, cv = C.c_float(x), C.c_float(v)
    a = np.ascontiguousarray(arch, dtype=np.float32)
    L.to_sim_kernel(float(rate), float(xL), float(vL), float(lL), C.byref(cx), C.byref(cv),
                    a.ctypes.data_as(C.POINTER(C.c_float)))
    return np.float32(cx.value), np.float32(cv.value)


def philox4x32_10(ctr, key):
    L = lib()
    c = (C.c_uint32 * 4)(*[int(v) & 0xFFFFFFFF for v in ctr])
    k = (C.c_uint32 * 2)(*[int(v) & 0xFFFFFFFF for v in key])
    o = (C.c_uint32 * 4)()
    L.to_philox4x32_10(c, k, o)
    return [int(v) for v in o]


def _pf(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def sim_bulk(rate, xL, vL, lL, x, v, arch):
    """Oracle IDM update (traffic_env.py:50-62) for arrays of (leader, follower) pairs."""
    L = lib()
    arrs = [np.ascontiguousarray(a, dtype=np.float32) for a in (xL, vL, lL, x, v)]
    a = np.ascontiguousarray(arch, dtype=np.float32)
    n = arrs[0].size
    xo, vo = np.empty(n, np.float32), np.empty(n, np.float32)
    L.to_sim_bulk(float(rate), *[_pf(t) for t in arrs], _pf(a), n, _pf(xo), _pf(vo))
    return xo, vo


def powf_bulk(x, y):
    """Host libm powf (what numba calls for float32 ** float32)."""
    L = lib()
    x = np.ascontiguousarray(x, dtype=np.float32)
    out = np.empty_like(x)
    L.to_powf_bulk(_pf(x), float(y), x.size, _pf(out))
    return out
