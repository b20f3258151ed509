"""traffic_env_b200 - B200 (sm_100a) implementation of the traffic-env simulation step.

Drop-in for the hot path of samanklesaria/traffic-env: gym_traffic/envs/traffic_env.py
(TrafficEnv._step and friends), gym_traffic/envs/roadgraph.py (GridRoad) and the
Repeater/Remi wrappers of traffic_test.py.  The simulation runs in
libtraffic_b200.so (hand-written CUDA, C ABI in include/traffic_b200.h).
"""
from ._lib import TrafficB200Error, load as load_library, SO_PATH  # noqa: F401
from .vec_env import VecTrafficEnv, WireResult, inv_popcount, plan_step_variant, ARCHETYPE  # noqa: F401

__all__ = ["VecTrafficEnv", "WireResult", "TrafficB200Error", "load_library", "inv_popcount", "plan_step_variant", "ARCHETYPE", "SO_PATH"]
