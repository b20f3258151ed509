"""CPU: the C-ABI library loads, exports every symbol include/traffic_b200.h declares, and refuses to
run without a CUDA device (no compute calls here)."""
import ctypes as C
import os
import re

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    txt = open(os.path.join(ROOT, "include", "traffic_b200.h")).read()
    txt = re.sub(r"/\*.*?\*/", "", txt, flags=re.S)
    return sorted(set(re.findall(r"\b(te_[a-z0-9_]+)\s*\(", txt)))


def test_library_exports_every_declared_symbol():
    from traffic_env_b200 import _lib, build
    build.build()
    L = _lib.load()
    names = declared_symbols()
    assert len(names) >= 20
    missing = [n for n in names if not hasattr(L, n)]
    assert not missing, missing
    assert sorted(_lib.EXPORTS) == names


def test_config_struct_matches_header():
    from traffic_env_b200 import _lib
    cfg = _lib.default_config()
    assert cfg.struct_size == C.sizeof(_lib.TeConfig)
    assert (cfg.m, cfg.n, cfg.length, cfg.rate) == (3, 3, 250.0, 0.5)
    assert [round(cfg.archetype[i], 2) for i in range(10)] == [0.0, 11.11, 4.0, 3.0, 4.0, 13.89, 6.0, 2.0, 1.0, 0.0]
    assert cfg.cars_per_tick == pytest.approx(0.72)


def test_no_cpu_fallback():
    """Without a GPU the product path must fail loudly, never compute on the host."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from traffic_env_b200 import TrafficB200Error, VecTrafficEnv
    with pytest.raises(TrafficB200Error, match="no CUDA device"):
        VecTrafficEnv()


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "traffic_env_b200")
    for dp, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                txt = open(os.path.join(dp, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt and "libtraffic_oracle" not in txt, f


def test_gap_cdf_table_properties():
    import numpy as np
    from traffic_env_b200.arrivals import gap_cdf
    for rate in (0.72, 2.4, 0.05):
        t = gap_cdf(rate)
        assert t.size > 4 and (np.diff(t.astype(np.int64)) >= 0).all()
        # P(gap = 0) = 1 - exp(-rate / 2)
        assert abs(t[0] / 2 ** 32 - (1 - np.exp(-0.5 * rate))) < 1e-9
        mean_gap = float(((2 ** 32 - t.astype(np.float64)) / 2 ** 32).sum())  # sum_k P(gap > k)
        assert abs(mean_gap - (1 / rate)) < 0.15 + 0.02 / rate


def test_idm_peak_form_rejects_unknown_forms():
    """The micro-kernel times form 5 (tame), form 0 (general) or, for -1, the one the step kernels run; any other form
    is refused with a message naming the accepted ones, before a device is touched."""
    import numpy as np
    from traffic_env_b200 import _lib
    L = _lib.load()
    arch = np.array(_lib.default_config().archetype, np.float32)
    for form in (1, 2, 3, 4, 6):
        out = C.c_double(-1.0)
        assert L.te_idm_peak_form(0, arch.ctypes.data, 0.5, 100, form, 0, C.byref(out)) < 0
        msg = L.te_last_error().decode()
        assert "form %d" % form in msg and "-1 = " in msg and "0 = general" in msg and "5 = tame" in msg, msg
        assert out.value == -1.0


def test_step_variant_queries_need_no_device():
    """te_step_variants and te_plan_step_variant answer from the host tables; te_get_step_variant needs a handle."""
    from traffic_env_b200 import _lib
    L = _lib.load()
    n = C.c_int32(-1)
    assert L.te_step_variants(None, 0, C.byref(n)) == 0 and n.value == 19
    assert L.te_step_variants(None, 1, C.byref(n)) < 0
    two = (_lib.TeStepVariant * 2)()
    assert L.te_step_variants(two, 2, C.byref(n)) == 0 and n.value == 19 and two[1].max_threads > 0
    out = _lib.TeStepVariant()
    cfg = _lib.default_config()
    assert L.te_plan_step_variant(C.byref(cfg), 0, C.byref(out)) == 0
    assert (out.max_threads, out.min_blocks, out.tame, out.grouped, out.envs_per_cta, out.threads) == (96, 10, 1, 1, 2, 96)
    assert L.te_plan_step_variant(C.byref(cfg), 1, C.byref(out)) == 0
    assert (out.max_threads, out.tame, out.grouped, out.envs_per_cta, out.threads) == (64, 0, 0, 1, 64)
    assert L.te_plan_step_variant(None, 0, C.byref(out)) < 0
    cfg.struct_size = 8
    assert L.te_plan_step_variant(C.byref(cfg), 0, C.byref(out)) < 0 and "size mismatch" in L.te_last_error().decode()
    assert L.te_get_step_variant(None, C.byref(out)) < 0 and "null argument" in L.te_last_error().decode()
