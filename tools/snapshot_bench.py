"""Bandwidth of snapshot records (te_save_envs / te_load_envs, device records) on two workloads, beside the stage-in /
flush bandwidth of the step kernel (te_stage_bandwidth) measured in the same run:

  headline: 16384 envs, 10x10 grid, L = 500, after a 300-actor-step greedy pre-roll (as bench.py's flagship workload);
  grid3x3 : 131072 envs, 3x3 grid, L = 250, after a 150-step pre-roll.

Both working sets (about 1.2 GB of records plus the same again of env state) are far above L2.  Save is timed with CUDA
events around back-to-back launches on one stream; load (synchronous: check pass, status word to the host, scatter
pass) with the host clock around whole calls, and its two kernels with torch.profiler in a separate pass.  GB/s =
2 x count x stride / kernel time.  Also times one rewind of the headline batch (a load) against the pre-roll it replaces.
Prints one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

WORKLOADS = {
    "headline": dict(m=10, n=10, length=500.0, envs=16384, preroll=300),
    "grid3x3": dict(m=3, n=3, length=250.0, envs=131072, preroll=150),
}


def card():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception:
        pl = "unknown"
    return name, pl


def preroll(env, steps, torch, s):
    """`steps` greedy actor steps (decision every 3 steps, 6 per launch) on device buffers on stream s; returns ms."""
    E, I = env.num_envs, env.intersections
    n = 6
    act = torch.empty((2, E, I), dtype=torch.uint8, device="cuda")
    obs = torch.empty((n, E, env.obs_len), dtype=torch.float32, device="cuda")
    rew = torch.empty((n, E, I), dtype=torch.float32, device="cuda")
    done = torch.empty((n, E), dtype=torch.uint8, device="cuda")
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    left = steps
    while left > 0:
        k = min(n, left)
        env.step_multi_device(k, act, obs[:k], rew[:k], done[:k], controller="greedy", stream=s.cuda_stream, spacing=3)
        left -= k
    e1.record(s)
    e1.synchronize()
    return e0.elapsed_time(e1)


def measure(name, w, iters, torch):
    from traffic_env_b200 import VecTrafficEnv
    env = VecTrafficEnv(m=w["m"], n=w["n"], length=w["length"], num_envs=w["envs"], arrivals="philox", seed=1,
                        local_cars_per_sec=0.12, ticks_per_step=10)
    env.reset()
    # one explicit stream for every launch and event (stream 0 would mean the handle's own stream to the library)
    s = torch.cuda.Stream()
    preroll_ms = preroll(env, w["preroll"], torch, s)
    E, stride = env.num_envs, env.snapshot_layout.stride
    rec_bytes = E * stride
    recs = torch.empty((E, stride), dtype=torch.uint8, device="cuda")
    stage = env.stage_bandwidth(repeats=50)
    # save: back-to-back launches on one stream
    for _ in range(5):
        env.save_envs(out=recs, stream=s.cuda_stream)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(s)
    for _ in range(iters):
        env.save_envs(out=recs, stream=s.cuda_stream)
    e1.record(s)
    e1.synchronize()
    save_ms = e0.elapsed_time(e1) / iters
    snap = recs.clone()
    # load: whole synchronous calls
    for _ in range(3):
        env.load_envs(recs)
    t0 = time.perf_counter()
    for _ in range(iters):
        env.load_envs(recs)
    load_call_ms = (time.perf_counter() - t0) * 1e3 / iters
    # the two kernels of a load, and the save kernel, from a profiled pass of their own
    from torch.profiler import ProfilerActivity, profile
    n_prof = 20
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n_prof):
            env.load_envs(recs)
            env.save_envs(out=recs, stream=s.cuda_stream)
        torch.cuda.synchronize()
    ker = {}
    for ev in prof.events():
        for k in ("te_snap_check_kernel", "te_snap_load_kernel", "te_snap_save_kernel"):
            if k in ev.name and ev.device_type.name == "CUDA":
                ker.setdefault(k, []).append(ev.device_time)
    ker_ms = {k: sum(v) / len(v) / 1e3 for k, v in ker.items()}
    if len(ker_ms) < 3:
        raise SystemExit("snapshot_bench: the profiler saw no snapshot kernels (%s)" % sorted(ker_ms))
    load_kernels_ms = ker_ms["te_snap_check_kernel"] + ker_ms["te_snap_load_kernel"]
    # the last load restored the saved state: a fresh save reproduces the records
    env.load_envs(snap)
    env.save_envs(out=recs, stream=s.cuda_stream)
    torch.cuda.synchronize()
    assert torch.equal(recs, snap), "a load + save round trip changed the records"
    # one rewind of the batch (a load from device records) against the pre-roll it replaces
    t0 = time.perf_counter()
    env.load_envs(snap)
    rewind_ms = (time.perf_counter() - t0) * 1e3
    gbs = lambda ms: 2.0 * rec_bytes / (ms * 1e-3) / 1e9
    out = {
        "envs": E, "grid": "%dx%d" % (w["m"], w["n"]), "length": w["length"], "stride_bytes": stride,
        "records_gb": rec_bytes / 1e9, "iters": iters,
        "save_ms": save_ms, "save_gbps": gbs(save_ms),
        "save_kernel_ms_profiled": ker_ms["te_snap_save_kernel"],
        "load_call_ms": load_call_ms, "load_call_gbps": gbs(load_call_ms),
        "load_check_kernel_ms": ker_ms["te_snap_check_kernel"], "load_scatter_kernel_ms": ker_ms["te_snap_load_kernel"],
        "load_kernels_gbps": gbs(load_kernels_ms), "load_scatter_gbps": gbs(ker_ms["te_snap_load_kernel"]),
        "stage_bandwidth_gbps": stage,
        "preroll_actor_steps": w["preroll"], "preroll_ms": preroll_ms, "rewind_load_ms": rewind_ms,
    }
    env.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--iters", type=int, default=300, help="timed calls per figure")
    ap.add_argument("--workloads", default="headline,grid3x3")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("snapshot_bench: needs a CUDA device (there is no CPU path)")
    name, pl = card()
    res = {"tool": "snapshot_bench", "gpu": name, "power_limit": pl}
    for wname in a.workloads.split(","):
        res[wname] = measure(wname, WORKLOADS[wname], a.iters, torch)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
