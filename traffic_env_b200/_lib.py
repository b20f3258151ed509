"""ctypes binding of libtraffic_b200.so (C ABI: include/traffic_b200.h).

The library is the product: if it is missing, cannot be loaded, or finds no CUDA
device, importing/creating fails loudly - there is no CPU fallback.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libtraffic_b200.so")
if os.environ.get("TRAFFIC_B200_SO"):
    # developer switch for A/B measurements of kernel variants (tools/ab_variants.py): another build of the SAME library
    SO_PATH = os.path.abspath(os.environ["TRAFFIC_B200_SO"])

TE_HOST, TE_DEVICE = 0, 1
TE_LEARN_SWITCH, TE_REMI, TE_AUTO_RESET, TE_VALIDATE, TE_ORDERED_TRANSFERS = 1, 2, 4, 8, 16
TE_ARRIVALS_NONE, TE_ARRIVALS_INJECTED, TE_ARRIVALS_PHILOX = 0, 1, 2
TE_PARAMS, TE_CAP = 10, 20
TE_CTRL_GIVEN, TE_CTRL_GREEDY = 0, 1

EXPORTS = [
    "te_default_config", "te_device_count", "te_create", "te_destroy", "te_get_dims", "te_last_error", "te_get_topology",
    "te_reset", "te_set_arrivals", "te_step", "te_step_masked", "te_step_multi", "te_step_multi_wire", "te_step_wire",
    "te_pool_create", "te_pool_destroy", "te_pool_step", "te_pool_reset", "te_pool_cars", "te_pool_counters", "te_pool_last_error", "te_wire_layout", "te_expand_wire", "te_step_raw", "te_remi_reward", "te_cars_on_roads",
    "te_greedy_actions", "te_get_state", "te_set_state", "te_get_stats", "te_get_trip_times",
    "te_synchronize", "te_host_alloc", "te_host_free", "te_last_kernel_ms", "te_stage_bandwidth", "te_idm_peak_form", "te_test_powf", "te_test_idm", "te_test_idm_tame", "te_is_tame", "te_tame_speed_cap", "te_set_controller_spacing", "te_test_powf4_exhaustive", "te_test_philox",
    "te_snapshot_layout", "te_save_envs", "te_load_envs",
]


class TeConfig(C.Structure):
    _fields_ = [
        ("struct_size", C.c_int32), ("m", C.c_int32), ("n", C.c_int32), ("length", C.c_float),
        ("rate", C.c_float), ("num_envs", C.c_int32), ("env_id_base", C.c_int64), ("device", C.c_int32),
        ("flags", C.c_int32), ("entry_spec", C.c_uint32), ("arrival_mode", C.c_int32),
        ("cars_per_tick", C.c_double), ("seed", C.c_uint64), ("episode_len", C.c_int32), ("gamma", C.c_float),
        ("archetype", C.c_float * TE_PARAMS),
    ]


class TeDims(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("m", "n", "intersections", "train_roads", "roads", "roads_padded",
                                         "num_envs", "num_entry", "obs_raw", "obs_actor")]


class TeStats(C.Structure):
    _fields_ = [
        ("ticks", C.c_uint64), ("actor_steps", C.c_uint64), ("vehicle_updates", C.c_uint64),
        ("overflows", C.c_uint64), ("cars_generated", C.c_uint64), ("episodes", C.c_uint64),
        ("return_sum", C.c_double), ("disc_return_sum", C.c_double), ("seq_fallback_ticks", C.c_uint64),
        ("cars_exited", C.c_uint64), ("arrival_saturations", C.c_uint64),
    ]


class TeWireLayout(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("stride", "passed", "detected", "light", "reward", "done", "max_k_ticks",
                                            "host_float_dma")]


class TeSnapshotLayout(C.Structure):
    _fields_ = [(k, C.c_int32) for k in ("stride", "x", "v", "w", "phase", "elapsed", "passed_dst", "scalars")]


class TrafficB200Error(RuntimeError):
    pass


_lib = None


def load():
    """Load the shared library (building is __graft_entry__.build()'s / build.py's job)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(SO_PATH):
        raise TrafficB200Error(
            "%s not found: build it with `python -m traffic_env_b200.build` (nvcc, sm_100a). "
            "There is no CPU fallback." % SO_PATH)
    L = C.CDLL(SO_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.te_default_config.argtypes = [C.POINTER(TeConfig)]
    L.te_default_config.restype = None
    L.te_create.argtypes = [C.POINTER(TeConfig), C.POINTER(vp)]
    L.te_destroy.argtypes = [vp]
    L.te_get_dims.argtypes = [vp, C.POINTER(TeDims)]
    L.te_last_error.restype = C.c_char_p
    L.te_get_topology.argtypes = [vp, vp, vp, vp, vp]
    L.te_reset.argtypes = [vp, vp, vp, C.c_int, vp]
    L.te_set_arrivals.argtypes = [vp, vp, vp, i64, i64, i32]
    L.te_device_count.argtypes = [C.POINTER(i32)]
    L.te_step.argtypes = [vp, vp, i32, vp, vp, vp, C.c_int, vp]
    L.te_step_raw.argtypes = [vp, vp, vp, vp, vp, C.c_int, vp]
    L.te_step_wire.argtypes = [vp, vp, i32, vp, C.c_int, vp]
    L.te_step_masked.argtypes = [vp, vp, vp, i32, vp, vp, vp, C.c_int, vp]
    L.te_step_multi.argtypes = [vp, i32, i32, vp, i32, vp, vp, vp, C.c_int, vp]
    L.te_step_multi_wire.argtypes = [vp, i32, i32, vp, i32, vp, C.c_int, vp]
    L.te_pool_create.argtypes = [vp, i32, i32, C.POINTER(vp)]
    L.te_pool_destroy.argtypes = [vp]
    L.te_pool_step.argtypes = [vp, i32, vp, vp, vp, vp]
    L.te_pool_reset.argtypes = [vp, i32, vp]
    L.te_pool_cars.argtypes = [vp, i32, vp]
    L.te_pool_counters.argtypes = [vp, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.te_pool_last_error.argtypes = [vp]
    L.te_pool_last_error.restype = C.c_char_p
    L.te_wire_layout.argtypes = [vp, C.POINTER(TeWireLayout)]
    L.te_expand_wire.argtypes = [vp, vp, i32, vp, vp, vp]
    L.te_remi_reward.argtypes = [vp, vp, C.c_int, vp]
    L.te_cars_on_roads.argtypes = [vp, vp, C.c_int, vp]
    L.te_greedy_actions.argtypes = [vp, vp, C.c_int, vp]
    L.te_get_state.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    L.te_set_state.argtypes = [vp, i32, i32, vp, vp, vp, vp, vp, vp, vp, vp]
    L.te_get_stats.argtypes = [vp, C.POINTER(TeStats)]
    L.te_get_trip_times.argtypes = [vp, vp, vp, i64, C.POINTER(i64), C.c_int]
    L.te_synchronize.argtypes = [vp]
    L.te_last_kernel_ms.argtypes = [vp, C.POINTER(C.c_float)]
    L.te_host_alloc.argtypes = [C.c_uint64, C.POINTER(vp)]
    L.te_host_free.argtypes = [vp]
    L.te_stage_bandwidth.argtypes = [vp, i32, C.POINTER(C.c_double)]
    L.te_idm_peak_form.argtypes = [C.c_int, vp, C.c_float, i32, i32, i32, C.POINTER(C.c_double)]
    L.te_test_powf.argtypes = [C.c_int, vp, C.c_float, vp, i64]
    L.te_test_idm.argtypes = [C.c_int, C.c_float, vp, vp, vp, vp, vp, vp, vp, vp, i64]
    L.te_test_idm_tame.argtypes = [C.c_int, C.c_float, vp, vp, vp, vp, vp, vp, vp, vp, i64]
    L.te_set_controller_spacing.argtypes = [vp, i32]
    L.te_tame_speed_cap.argtypes = [vp, C.c_float, C.c_float, C.POINTER(C.c_float)]
    L.te_is_tame.argtypes = [vp, C.POINTER(i32), C.POINTER(C.c_float)]
    L.te_test_powf4_exhaustive.argtypes = [C.c_int, C.c_uint64, vp]
    L.te_test_philox.argtypes = [C.c_int, vp, vp, vp]
    L.te_snapshot_layout.argtypes = [vp, C.POINTER(TeSnapshotLayout)]
    L.te_save_envs.argtypes = [vp, vp, i32, vp, C.c_int, vp]
    L.te_load_envs.argtypes = [vp, vp, i32, vp, C.c_int, vp]
    for name in EXPORTS:
        if name not in ("te_default_config", "te_last_error", "te_pool_last_error"):
            getattr(L, name).restype = C.c_int
    _lib = L
    return L


def check(rc):
    """C ABI convention: 0 = ok, < 0 = error (te_last_error has the text), > 0 = ok with a warning."""
    if rc < 0:
        raise TrafficB200Error(load().te_last_error().decode("utf-8", "replace"))
    return rc


def device_count():
    """CUDA devices visible to libtraffic_b200.so (0 when there is no driver / device); never raises."""
    try:
        n = C.c_int32(0)
        load().te_device_count(C.byref(n))
        return int(n.value)
    except Exception:
        return 0


def default_config():
    cfg = TeConfig()
    load().te_default_config(C.byref(cfg))
    return cfg
