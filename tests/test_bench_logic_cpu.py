"""CPU: host-side logic of bench.py that the driver relies on - both arms print the same static `config`, the row padding
rule mirrors te_create's, and the ncu traffic figure is refused when the kernel sources have changed since the capture."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _args(**kw):
    a = argparse.Namespace(gpus=1, steps=20, warmup=5, impl="b200", workload="grid10x10_L500_greedy", envs=0, preroll=-1,
                           no_cpu_baseline=False, no_e2e=False, no_secondary=False, no_multi=False, cpu_seconds=12.0)
    for k, v in kw.items():
        setattr(a, k, v)
    return a


def test_both_arms_print_the_same_config():
    for wl in bench.WORKLOADS:
        w = bench.WORKLOADS[wl]
        ours = bench.bench_config(_args(workload=wl), w, w["envs"])
        ref = bench.bench_config(_args(workload=wl, impl="reference", gpus=8), w, w["envs"])
        assert ours == ref and json.dumps(ours) == json.dumps(ref)
        assert ours["workload"] == wl and "steady_state_cars_per_env" not in ours      # measured values live outside config
        assert ours["envs_per_gpu"] == w["envs"]


def test_row_padding_rule_matches_te_create():
    # R = 4 m n + 2 m + 2 n padded to 32, or to 128 when that costs at most 20 % (te_api.cu)
    assert bench.rows_padded(dict(m=3, n=3)) == 64            # 48 roads
    assert bench.rows_padded(dict(m=10, n=10)) == 512         # 440 roads
    assert bench.rows_padded(dict(m=7, n=7)) == 256           # 224 roads
    assert bench.rows_padded(dict(m=5, n=5)) == 128           # 120 roads
    assert bench.rows_padded(dict(m=1, n=1)) == 32            # 8 roads


def test_traffic_figure_is_refused_when_sources_changed(tmp_path, monkeypatch):
    sha = bench.kernel_source_sha()
    assert len(sha) == 16 and sha == bench.kernel_source_sha()
    prof = tmp_path / "profiles"
    prof.mkdir()
    monkeypatch.setattr(bench, "ROOT", str(tmp_path))
    monkeypatch.setattr(bench, "kernel_source_sha", lambda: sha)
    (prof / "traffic_bytes.json").write_text(json.dumps({"w": {"dram_bytes_per_launch": 123, "kernel_source_sha": sha, "capture": "x"}}))
    assert bench.measured_traffic("w")[0] == 123
    assert bench.measured_traffic("other")[0] is None
    monkeypatch.setattr(bench, "kernel_source_sha", lambda: "0" * 16)
    val, why = bench.measured_traffic("w")
    assert val is None and "stale" in why


def test_launch_plan_keeps_decisions_on_the_same_steps():
    """bench.launch_plan: whatever the launch length and wherever a range starts, the launches cover exactly the
    requested steps, "greedy" launches start on a decision step and hold whole decisions (except at the end of the range),
    and the set of decision steps is the same as with one launch per decision."""
    sp = bench.SPACING
    for spl in (sp, 2 * sp, 4 * sp):
        for s0 in range(0, 8):
            for n in range(0, 30):
                plan = bench.launch_plan(s0, n, spl)
                assert sum(k for k, _ in plan) == n and all(k >= 1 for k, _ in plan)
                s, decisions = s0, []
                for k, ctrl in plan:
                    if ctrl == "greedy":
                        assert s % sp == 0 and k <= spl
                        decisions += list(range(s, s + k, sp))
                    else:
                        assert s % sp != 0 and k <= sp - s % sp      # finishes the decision in force, never crosses one
                    s += k
                assert decisions == [t for t in range(s0, s0 + n) if t % sp == 0]
    assert bench.launch_plan(0, 21, 6) == [(6, "greedy"), (6, "greedy"), (6, "greedy"), (3, "greedy")]
    assert bench.launch_plan(4, 10, 6) == [(2, "given"), (6, "greedy"), (2, "greedy")]


def test_dump_outputs_rows_and_budget(tmp_path):
    """bench.dump_outputs: every array as float32 .npy holding the same env rows (listed in env_index.npy, float64) -
    all of them when they fit the byte budget, else a seeded sample that is the same every time - within the budget."""
    rng = np.random.RandomState(1)
    E = 1000
    arrays = {"obs": rng.rand(E, 81).astype(np.float32), "reward": rng.rand(E, 9).astype(np.float32),
              "done": rng.randint(2, size=E).astype(np.uint8), "actions": rng.randint(2, size=(E, 9)).astype(np.uint8)}
    for budget in (10 ** 6, 10 ** 5):
        dumps = []
        for rep in range(2):
            out = tmp_path / ("%d_%d" % (budget, rep))
            bench.dump_outputs(str(out), arrays, max_bytes=budget)
            assert sorted(os.listdir(out)) == sorted(n + ".npy" for n in list(arrays) + ["env_index"])
            assert sum(os.path.getsize(out / f) for f in os.listdir(out)) <= budget
            idx = np.load(out / "env_index.npy")
            assert idx.dtype == np.float64 and (np.diff(idx) > 0).all() and 0 <= idx[0] and idx[-1] < E
            rows = idx.astype(np.int64)
            for name, arr in arrays.items():
                got = np.load(out / (name + ".npy"))
                assert got.dtype == np.float32 and (got == arr[rows]).all()
            dumps.append(rows)
        assert (dumps[0] == dumps[1]).all()
        assert (len(dumps[0]) == E) == (budget == 10 ** 6) and len(dumps[0]) > E // 10
