"""GPU: a live handle runs the step kernel te_plan_step_variant names for its configuration, and the one it names for
wild = 1 once a wild car was loaded; a configuration no kernel has room for is refused with the largest one named."""
import numpy as np
import pytest

from tests.test_gpu_fuzz_state import random_env_state
from tests.test_kernel_variants_cpu import oracle_rows

pytestmark = pytest.mark.gpu


def test_live_handles_run_the_planned_variant():
    from traffic_env_b200 import VecTrafficEnv, plan_step_variant
    seen = set()
    for _, kw, _ in oracle_rows():
        kw = dict(kw, num_envs=1, arrivals="injected", remi=False)
        cfg = repr(sorted((k, np.asarray(v).tolist()) for k, v in kw.items()))
        if cfg in seen:
            continue
        seen.add(cfg)
        env = VecTrafficEnv(**kw)
        assert env.step_variant() == plan_step_variant(**kw), kw
        R, r, I, L = env.roads, env.train_roads, env.intersections, kw["length"]
        st = random_env_state(np.random.RandomState(len(seen)), R, r, I, L, True)
        rd = next(rd for rd in range(R) if st["leading"][rd] != st["lastcar"][rd])
        st["v"][rd, st["leading"][rd] % 19 + 1] = np.float32(1e-35)     # the leader's follower: a wild speed
        env.set_state({k: v[None] for k, v in st.items()} | {"steps": np.zeros(1, np.float32)})
        assert not env.is_tame()
        assert env.step_variant() == plan_step_variant(wild=True, **kw), kw
        env.close()
    assert len(seen) >= 25


def test_validate_handle_too_large_for_every_variant_is_refused():
    from traffic_env_b200 import TrafficB200Error, VecTrafficEnv
    with pytest.raises(TrafficB200Error, match=r"te_create: 1024 roads exceed the largest validate-mode kernel variant "
                                                r"\(te_step_kernel<768, 1, validate>\)"):
        VecTrafficEnv(m=15, n=15, validate=True)
