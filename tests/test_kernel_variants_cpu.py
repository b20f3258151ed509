"""CPU: the step kernel is compiled as a fixed set of instantiations, te_step_kernel<MAXT, MINB, VALIDATE, TAME, GROUPED>,
and te_create picks one from the grid, the archetype, the validate flag and whether a wild car was ever loaded.  Every
instantiation must be reachable, and every one must be run by a GPU test that compares it with the oracle: a kernel no
test runs can be wrong without the suite noticing.  The layout rules (te_plan_step_variant) need no device."""
import pytest

from tests.test_gpu_fuzz_state import FUZZ_ROWS, FUZZ_VARIANTS
from tests.test_gpu_hardening import (ARCH_ODD, NONDEFAULT_ARCH_ROWS, NONDEFAULT_ARCH_VARIANTS, WILD_CAR_ROWS,
                                      WILD_CAR_VARIANTS)
from tests.test_gpu_parity_golden import VALIDATE_ROWS, VALIDATE_VARIANTS

NON_TAME = dict(archetype=ARCH_ODD, rate=0.4)


def key(v):
    return v["kind"], v["max_threads"], v["min_blocks"]


def name(k):
    return "te_step_kernel<%d, %d> (%s)" % (k[1], k[2], k[0])


def compiled():
    from traffic_env_b200 import _lib
    return [key(v) for v in _lib.step_variants()]


def oracle_rows():
    """(test, VecTrafficEnv kwargs, wild) of every row of the GPU tests that compare the step kernel with the oracle;
    the wild-car test runs each of its grids both before and after the wild load."""
    for m, n, L, E, _, ordered in FUZZ_ROWS:
        yield "fuzz", dict(m=m, n=n, length=L, num_envs=E, ordered_transfers=ordered), False
    for arch, rate, m, n, L, _, E in NONDEFAULT_ARCH_ROWS:
        yield "nondefault archetype", dict(m=m, n=n, length=L, num_envs=E, rate=rate, archetype=arch), False
    for m, n, L, E in WILD_CAR_ROWS:
        for wild in (False, True):
            yield "wild car", dict(m=m, n=n, length=L, num_envs=E), wild
    for m, n, L, E in VALIDATE_ROWS:
        yield "validate", dict(m=m, n=n, length=L, num_envs=E, validate=True), False


def test_variant_table():
    from traffic_env_b200 import _lib
    variants = _lib.step_variants()
    assert len(variants) == 19 and len(set(map(key, variants))) == 19
    assert all(v["roads"] == v["roads_padded"] == v["envs_per_cta"] == v["threads"] == 0 for v in variants)
    assert ("grouped", 128, 8) not in map(key, variants)       # no grid reaches it
    assert not any(v["validate"] and (v["tame"] or v["grouped"]) for v in variants)
    assert all(v["tame"] for v in variants if v["grouped"])


def test_every_variant_is_reachable():
    """Grids up to 32 x 32 with the reference's archetype, a non-tame archetype, after a wild car, and in validate mode."""
    from traffic_env_b200 import TrafficB200Error, plan_step_variant
    reached, refused = set(), 0
    for m in range(1, 33):
        for n in range(1, 33):
            for kw in ({}, NON_TAME, {"wild": True}, {"validate": True}):
                try:
                    v = plan_step_variant(m=m, n=n, length=1000.0, **kw)
                except TrafficB200Error as ex:
                    assert "exceed" in str(ex), str(ex)
                    refused += 1
                    continue
                assert v["threads"] <= v["max_threads"] and v["threads"] % 32 == 0
                assert v["envs_per_cta"] == 1 or (v["grouped"] and 2 <= v["envs_per_cta"] <= 4)
                assert v["threads"] >= v["envs_per_cta"] * v["roads"]
                assert v["roads"] == 4 * m * n + 2 * (m + n) and v["roads_padded"] >= v["roads"]
                reached.add(key(v))
    table = compiled()
    assert reached <= set(table)
    missing = [name(k) for k in table if k not in reached]
    assert not missing, "compiled but reached by no grid: " + ", ".join(missing)
    assert refused > 0


def test_planner_follows_the_handle_rules():
    """Spot checks of the rules te_create documents: the default 3x3 grid shares a CTA between two envs, a wild car
    moves a handle to the one-env checked kernels, and grids past a variant's capacity are refused naming it."""
    from traffic_env_b200 import TrafficB200Error, plan_step_variant
    v = plan_step_variant()
    assert (key(v), v["roads"], v["roads_padded"], v["envs_per_cta"], v["threads"]) == (("grouped", 96, 10), 48, 64, 2, 96)
    v = plan_step_variant(wild=True)
    assert (key(v), v["envs_per_cta"], v["threads"]) == (("checked", 64, 16), 1, 64)
    v = plan_step_variant(m=10, n=10, length=500.0)
    assert (key(v), v["roads"], v["threads"]) == (("tame", 512, 2), 440, 512)
    assert plan_step_variant(m=11, n=11, validate=True)["threads"] == 544
    with pytest.raises(TrafficB200Error, match=r"te_step_kernel<768, 1, validate>"):
        plan_step_variant(m=15, n=15, validate=True)
    with pytest.raises(TrafficB200Error, match="exceed one CTA"):
        plan_step_variant(m=16, n=16)
    with pytest.raises(TrafficB200Error, match="road length"):
        plan_step_variant(length=5.0)


def test_oracle_tests_run_every_variant():
    from traffic_env_b200 import plan_step_variant
    covered = {}
    for test, kw, wild in oracle_rows():
        covered.setdefault(key(plan_step_variant(wild=wild, **kw)), test)
    missing = [name(k) for k in compiled() if k not in covered]
    assert not missing, "never compared with the oracle: " + ", ".join(missing)


def test_rows_state_the_variant_the_planner_picks():
    """The (kind, MAXT) each GPU row asserts on its live handle is what the layout rules give for it."""
    from traffic_env_b200 import plan_step_variant

    def km(**kw):
        v = plan_step_variant(**kw)
        return v["kind"], v["max_threads"]
    for m, n, L, E, _, _ in FUZZ_ROWS:
        assert km(m=m, n=n, length=L, num_envs=E) == FUZZ_VARIANTS[(m, n)], (m, n)
    for arch, rate, m, n, L, _, E in NONDEFAULT_ARCH_ROWS:
        assert km(m=m, n=n, length=L, num_envs=E, rate=rate, archetype=arch) == NONDEFAULT_ARCH_VARIANTS[(m, n)], (m, n)
    for m, n, L, E in WILD_CAR_ROWS:
        assert tuple(km(m=m, n=n, length=L, wild=w) for w in (False, True)) == WILD_CAR_VARIANTS[(m, n)], (m, n)
    for m, n, L, E in VALIDATE_ROWS:
        assert km(m=m, n=n, length=L, validate=True) == ("validate", VALIDATE_VARIANTS[(m, n)]), (m, n)
