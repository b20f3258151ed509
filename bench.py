"""bench.py - vehicle-updates/s of the traffic-env simulation step on B200.

Headline workload (BASELINE.json configs[2], the config the target is quoted on): 10x10 grid, long
roads (L = 500 m), 16384 env instances per GPU, greedy light controller recomputed every 3
actor steps (algorithms/greedy.py:13-16 with --spacing 3), Philox arrivals at the reference's
stock --local_cars_per_sec 0.12, Remi(Repeater(10)) semantics, envs pre-rolled to the
ring-capacity-bound steady state (see DESIGN.md "headline workload").  A step = one actor step
(10 physics ticks unless a ring overflows) of every env; the controller runs inside the kernel, and one te_step_multi
launch holds as many decisions as fit its 64 ticks: 6 actor steps = 2 greedy decisions (--launch-steps 3: one decision
per launch; --no-multi: one te_step launch per step + a controller kernel every third).

After the timed region a `secondary` block puts the other BASELINE configs on the same record (every rank takes
part, values are whole-job aggregates): the default 3x3 grid at 131072 envs per GPU (config 4: 2^20 envs at
--gpus 8) with the greedy controller and, as config 4 prescribes, with a random policy + auto-reset; the headline
workload with auto-reset (what every reference agent does on `done`); the learner-style rollouts of config 5; the
single-env drop-in of config 1; and a per-rank parity spot check against the CPU oracle.

  python bench.py [--gpus N] [--steps K] [--warmup W]           our arm (one rank per GPU under torchrun)
  python bench.py --impl reference ...                          the CPU arm: the oracle port on the host cores
  python bench.py ... --dump-outputs DIR                        also write what the last timed step computed (rank 0)

Prints ONE JSON line (rank 0).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: grid, road length, arrival rate, default envs per GPU, pre-roll actor steps, policy, reset
    "grid10x10_L500_greedy": dict(m=10, n=10, length=500.0, lcps=0.12, envs=16384, preroll=300),
    "grid3x3_L250_greedy": dict(m=3, n=3, length=250.0, lcps=0.12, envs=131072, preroll=150),
}
K_TICKS = 10      # FLAGS.light_iterations = light_secs / rate = 5 / 0.5 (traffic_test.py:21)
SPACING = 3       # FLAGS.spacing (alg_flags.py:22)
MAX_LAUNCH_TICKS = 64   # te_step_multi: n_steps * k_ticks <= 64
EPISODE_LEN = 120  # FLAGS.episode_len = episode_secs / light_secs = 600 / 5 (traffic_test.py:12-20)
OPS_PER_UPDATE = 34  # SURVEY.md 8a: arithmetic ops of one sim() element


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="grid10x10_L500_greedy", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=0, help="env instances per GPU (default: the workload's)")
    ap.add_argument("--preroll", type=int, default=-1)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--launch-steps", type=int, default=0, help="actor steps per te_step_multi launch (a multiple of the "
                    "controller spacing; default: as many decisions as fit the 64 ticks of a launch = 6; 3 = one decision per launch)")
    ap.add_argument("--no-multi", action="store_true", help="one launch per actor step + a separate greedy-controller "
                    "kernel every `spacing` steps (round-1 scheme) instead of te_step_multi")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last of them computed "
                    "(rank 0: obs, reward, done and the actions in force, one row per env) as DIR/<name>.npy, so that two "
                    "builds can be compared on the same inputs; a seeded sample of the env rows when all exceed 64 MB")
    a = ap.parse_args()
    if a.dump_outputs and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return a


DUMP_MAX_BYTES = 64 * 10 ** 6


def dump_outputs(path, arrays, max_bytes=DUMP_MAX_BYTES, seed=0):
    """Writes every [E, ...] host array of `arrays` as path/<name>.npy in float32, plus path/env_index.npy (float64): the
    env rows written.  All E rows when they fit `max_bytes`, else the same seeded sample of rows from every array."""
    E = len(next(iter(arrays.values())))
    row_bytes = 8 + sum(4 * int(np.prod(a.shape[1:])) for a in arrays.values())
    n = min(E, (max_bytes - 256 * (len(arrays) + 1)) // row_bytes)       # 256: room for each file's .npy header
    idx = np.arange(E) if n == E else np.sort(np.random.RandomState(seed).choice(E, n, replace=False))
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "env_index.npy"), idx.astype(np.float64))
    for name, arr in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.ascontiguousarray(arr[idx], dtype=np.float32))


# --------------------------------------------------------------------------- clocks
class ClockSampler(object):
    """nvidia-smi sampling during the timed region (B200_PROFILING.md clocks line)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def mark(self):
        return len(self.rows)

    def stop(self, first=0, last=None):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = self.rows[first:last] if (last is not None and last - first >= 3) else self.rows
        sm = [float(r[1]) for r in rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            if len(r) >= 9:
                for nm, val in zip(names, r[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------- CPU arm (oracle port)
def _cpu_worker(args):
    """One env of the workload on one core: pre-roll, then timed actor steps.  Returns (vehicle_updates, seconds,
    env_ticks, actor_steps)."""
    wl, seed, preroll, budget_s, min_steps, policy = args
    from oracle.oracle import OracleEnv
    from traffic_env_b200.arrivals import gap_cdf
    w = WORKLOADS[wl]
    I = w["m"] * w["n"]
    o = OracleEnv(w["m"], w["n"], w["length"], 0.5)
    o.reset(np.zeros(I, np.int32))
    cps = w["lcps"] * w["m"] * 4
    o.philox_seed(2026, seed, gap_cdf(cps * 0.5))
    act = np.zeros(I, np.int32)
    ones = np.ones(I, np.int32)

    def run(nsteps, deadline=None):
        nonlocal act
        done_steps = 0
        for s in range(nsteps):
            if policy == "fixed":
                act = ones if (s % (2 * SPACING)) >= SPACING else ones * 0    # fixed.py:6-7
            elif s % SPACING == 0:
                act = (o.cars_on_roads().reshape(-1, 4).dot([1, 1, -1, -1]) < 0).astype(np.int32)
            o.actor_step_philox(act, K_TICKS, use_remi=True)
            done_steps += 1
            if deadline is not None and done_steps >= min_steps and time.perf_counter() > deadline:
                break
        return done_steps

    run(preroll)
    vu0, t0 = o.vehicle_updates, time.perf_counter()
    tick0 = o.steps
    n = run(10 ** 9, deadline=t0 + budget_s)
    dt = time.perf_counter() - t0
    return o.vehicle_updates - vu0, dt, float(o.steps - tick0), n


def cpu_run(wl, cores, preroll, budget_s, min_steps=3, policy="greedy"):
    import multiprocessing as mp
    jobs = [(wl, i, preroll, budget_s, min_steps, policy) for i in range(cores)]
    if cores == 1:
        res = [_cpu_worker(jobs[0])]
    else:
        with mp.get_context("fork").Pool(cores) as pool:
            res = pool.map(_cpu_worker, jobs)
    vu = sum(r[0] for r in res)
    wall = max(r[1] for r in res)
    return dict(vehicle_updates=vu, seconds=wall, value=vu / wall, env_ticks=sum(r[2] for r in res),
                actor_steps=sum(r[3] for r in res))


def reference_arm(a):
    """The reference's CPU implementation of the path, timed on the host cores.  The reference is Python +
    numba and cannot travel to the GPU box, so this is its C restatement (oracle/, kind "port"), one
    independent env per core (the reference has no intra-env parallelism).  profiles/cpu_reference_numba.json holds
    the unmodified numba reference timed beside this port in the build container (the port is 6-11 x faster)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as orc
    orc.build()
    cores = os.cpu_count() or 1
    w = WORKLOADS[a.workload]
    per_step = []
    preroll = 60  # bounded: enough for the first cars to cross several intersections
    cpu_run(a.workload, 1, 2, 0.01, 1)  # warm the page cache / library load
    t0 = time.perf_counter()
    tot_vu, tot_s, tot_ticks, tot_steps = 0, 0.0, 0.0, 0
    budget = max(1.0, min(20.0, 150.0 / max(1, a.steps + a.warmup)))
    for s in range(a.warmup + a.steps):
        r = cpu_run(a.workload, cores, preroll, budget)
        if s >= a.warmup:
            tot_vu += r["vehicle_updates"]; tot_s += r["seconds"]; tot_ticks += r["env_ticks"]; tot_steps += r["actor_steps"]
            per_step.append(r["seconds"])
    value = tot_vu / tot_s
    sample = ("%d independent envs (one per core) of %s, %d-actor-step pre-roll then ~%.1f s of actor steps per bench step"
              % (cores, a.workload, preroll, budget))
    line = {
        "impl": "reference", "metric": "vehicle_updates_per_sec", "value": value, "unit": "vehicle-updates/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * tot_s / max(1, a.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
        "config": bench_config(a, w, w["envs"] if not a.envs else a.envs),
        "env_steps_per_sec": {"ticks": tot_ticks / tot_s, "actor_steps": tot_steps / tot_s},
        "cpu_baseline": {"value": value, "unit": "vehicle-updates/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "vehicle-updates/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": time.perf_counter() - t0,
    }
    print(json.dumps(line), flush=True)


def rows_padded(w):
    """The device's row padding rule (te_api.cu: te_create): roads padded to 32, or to 128 when that costs <= 20 %."""
    R = w["m"] * w["n"] * 4 + 2 * w["m"] + 2 * w["n"]
    rp, rp128 = (R + 31) // 32 * 32, (R + 127) // 128 * 128
    return rp128 if rp128 * 5 <= R * 6 else rp


def bench_config(a, w, envs):
    """Static description of the workload: identical in both arms (measured quantities live outside `config`)."""
    return {"workload": a.workload, "grid": "%dx%d" % (w["m"], w["n"]), "road_length_m": w["length"],
            "envs_per_gpu": envs, "policy": "greedy(spacing=%d)" % SPACING, "ticks_per_actor_step": K_TICKS,
            "arrivals": "philox, local_cars_per_sec=%.2f (reference default)" % w["lcps"],
            "wrappers": "Remi(Repeater(10))",
            "launches": "te_step_multi with the controller in the kernel: a new greedy decision every %d actor steps, as many "
                        "decisions per launch as fit its %d ticks (--launch-steps; default 6 actor steps = 2 decisions)" % (SPACING, MAX_LAUNCH_TICKS),
            "reset": "none (env keeps stepping after overflow, as the bare reference env does); pre-rolled into the "
                     "ring-capacity-bound steady state: ~48 % mean ring occupancy, NOT near-full in the mean (DESIGN.md 7); "
                     "the auto-reset variant is secondary.headline_auto_reset",
            "l2": "inputs larger than L2: state is %.2f GB per GPU against the 126 MB L2" % (envs * rows_padded(w) * 160 / 1e9)}


def kernel_source_sha():
    h = hashlib.sha256()
    d = os.path.join(ROOT, "traffic_env_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


def measured_traffic(workload):
    """dram bytes per launch from the committed ncu capture - only when it was taken from these very kernel sources."""
    tp = os.path.join(ROOT, "profiles", "traffic_bytes.json")
    try:
        rec = json.load(open(tp)).get(workload)
    except Exception:
        return None, "no profiles/traffic_bytes.json"
    if not isinstance(rec, dict):
        return None, "no capture for this workload"
    if rec.get("kernel_source_sha") != kernel_source_sha():
        return None, "stale: captured from kernel sources %s, current %s" % (rec.get("kernel_source_sha"), kernel_source_sha())
    return rec.get("dram_bytes_per_launch"), "ncu --set full, %s" % rec.get("capture", "profiles/")


# --------------------------------------------------------------------------- our arm
class Ctx(object):
    pass


def setup_dist():
    # helper threads of the host path (they expand wire records while the GPU works): what the host can spare per rank
    world = int(os.environ.get("WORLD_SIZE", "1"))
    os.environ.setdefault("TE_HOST_THREADS", str(max(2, min(8, (os.cpu_count() or 4) // max(world, 1) - 1))))
    import torch
    import torch.distributed as dist
    c = Ctx()
    c.torch, c.dist = torch, dist
    c.rank = int(os.environ.get("RANK", "0"))
    c.world = int(os.environ.get("WORLD_SIZE", "1"))
    c.local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the product path has no CPU fallback")
    torch.cuda.set_device(c.local)
    c.dev = torch.device("cuda", c.local)
    if c.world > 1:
        # stdout carries exactly one JSON line: whatever NCCL prints while the communicator comes up (its
        # "NCCL version ..." banner at NCCL_DEBUG=VERSION/WARN) is sent to stderr by pointing fd 1 at fd 2 meanwhile
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=c.dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    c.tstream = torch.cuda.Stream(device=c.dev)   # a dedicated (non-default) stream: kernels and CUDA events go here
    c.stream = c.tstream.cuda_stream
    return c


def barrier(c):
    c.torch.cuda.synchronize()
    if c.world > 1:
        c.dist.barrier()
    c.torch.cuda.synchronize()


def allreduce(c, vals, op="sum"):
    t = c.torch.tensor([float(v) for v in vals], dtype=c.torch.float64, device=c.dev)
    if c.world > 1:
        c.dist.all_reduce(t, op=c.dist.ReduceOp.SUM if op == "sum" else (c.dist.ReduceOp.MAX if op == "max" else c.dist.ReduceOp.MIN))
    return [float(x) for x in t.tolist()]


def launch_plan(s0, n, spl, spacing=SPACING):
    """The te_step_multi launches that cover actor steps [s0, s0 + n): a list of (steps, controller).  A launch starts at a
    controller decision (step index divisible by `spacing`) and holds up to `spl` steps - spl / spacing decisions, taken
    inside the kernel; a range that starts between two decisions first finishes the current one ("given": the action in
    force).  Decisions therefore fall on the same step indices whatever the launch length."""
    plan, s = [], s0
    while s < s0 + n:
        if s % spacing == 0:
            k, ctrl = min(spl, s0 + n - s), "greedy"
        else:
            k, ctrl = min(spacing - s % spacing, s0 + n - s), "given"
        plan.append((k, ctrl))
        s += k
    return plan


class Runner(object):
    """One batched env on this rank plus its device-resident and host-side step loops."""

    def __init__(self, c, w, E, policy="greedy", auto_reset=False, episode_len=0, multi=True, launch_steps=0):
        from traffic_env_b200 import VecTrafficEnv
        torch = c.torch
        self.c, self.w, self.E, self.policy = c, w, E, policy
        # greedy decisions hold for `spacing` actor steps (greedy.py:14-16): those steps are ONE te_step_multi launch with
        # the controller evaluated in the kernel (not for TE_AUTO_RESET handles, which reset between te_step calls)
        self.multi = bool(multi) and policy == "greedy" and not auto_reset
        # ... and a launch holds as many decisions as fit its 64 ticks (te_set_controller_spacing: the controller is
        # re-evaluated inside the kernel every `spacing` steps): 6 actor steps = 2 decisions at 10 ticks per step
        fit = max(SPACING, MAX_LAUNCH_TICKS // K_TICKS // SPACING * SPACING)
        self.spl = (min(fit, max(SPACING, launch_steps // SPACING * SPACING)) if launch_steps else fit) if self.multi else 1
        self.env = VecTrafficEnv(m=w["m"], n=w["n"], length=w["length"], num_envs=E, local_cars_per_sec=w["lcps"],
                                 arrivals="philox", seed=2026, env_id_base=c.rank * E, device=c.local,
                                 ticks_per_step=K_TICKS, remi=True, auto_reset=auto_reset, episode_len=episode_len)
        env = self.env
        self.I, self.OL = env.intersections, env.obs_len
        ns = self.spl
        self.ndec = (ns + SPACING - 1) // SPACING
        self.d_acts = torch.zeros((self.ndec, E, self.I), dtype=torch.uint8, device=c.dev)   # one block per decision of a launch
        self.d_act = self.d_acts[0]                                                           # the action in force
        self.d_obs = torch.empty((ns, E, self.OL), dtype=torch.float32, device=c.dev)
        self.d_rew = torch.empty((ns, E, self.I), dtype=torch.float32, device=c.dev)
        self.d_done = torch.empty((ns, E), dtype=torch.uint8, device=c.dev)
        self.launches = 0
        self.h_act = env.host_buffer((E, self.I), np.uint8)     # page-locked: the agent's actions cross PCIe from here
        self.h_act[:] = 0
        if policy == "random":
            g = torch.Generator(device=c.dev).manual_seed(1234 + c.rank)
            self.d_rand = torch.randint(0, 2, (8, E, self.I), dtype=torch.uint8, device=c.dev, generator=g)
            self.h_rand = self.d_rand.cpu().numpy()
        env.reset()
        torch.cuda.synchronize()

    def device_steps(self, n, s0=0):
        """n actor steps of every env, device-resident; returns nothing (asynchronous)."""
        if not self.multi:
            for s in range(s0, s0 + n):
                self.device_step(s)
            return
        for k, ctrl in launch_plan(s0, n, self.spl):
            if ctrl == "greedy":
                self.env.step_multi_device(k, self.d_acts, self.d_obs, self.d_rew, self.d_done, controller="greedy",
                                           spacing=SPACING, stream=self.c.stream)
                self.d_act = self.d_acts[(k - 1) // SPACING]
            else:
                self.env.step_multi_device(k, self.d_act, self.d_obs, self.d_rew, self.d_done, controller="given", stream=self.c.stream)
            self.launches += 1

    def host_steps(self, n, s0=0):
        if not self.multi:
            acc = 0.0
            for s in range(s0, s0 + n):
                acc += self.host_step(s)
            return acc
        acc = 0.0
        for k, ctrl in launch_plan(s0, n, self.spl):
            if ctrl == "greedy":
                act, obs, rew, done = self.env.step_multi(k, controller="greedy", spacing=SPACING)
                self.h_act[:] = act[-1]
            else:
                act, obs, rew, done = self.env.step_multi(k, actions=self.h_act, controller="given")
            for j in range(k):
                acc += float(rew[j, 0, 0]) + float(obs[j, 0, 0])   # every actor step's result is read on the host
        return acc

    def host_steps_agent(self, n, s0=0, lazy=True):
        """The greedy AGENT on the host, as algorithms/greedy.py:13-17 runs it: every `spacing` actor steps it asks the env
        for its decision (the ring counts stay on the device: te_greedy_actions evaluates greedy.py:14-16 there and copies
        the actions device -> host), then steps with THAT action: actions host -> device from page-locked memory, one
        te_step_multi launch for the steps the decision holds for, every actor step's results device -> host."""
        acc = 0.0
        for k, ctrl in launch_plan(s0, n, SPACING):     # one launch per decision: the agent decides on the host
            if ctrl == "greedy":
                self.env.greedy_actions(out=self.h_act)
            if lazy:
                act, res = self.env.step_multi(k, actions=self.h_act, controller="given", lazy=True)
                for j in range(k):
                    acc += float(res.reward[j, 0, 0]) + float(res.obs_of([0], step=j)[0, 0])
            else:
                act, obs, rew, done = self.env.step_multi(k, actions=self.h_act, controller="given")
                for j in range(k):
                    acc += float(rew[j, 0, 0]) + float(obs[j, 0, 0])
        return acc

    def host_steps_wire(self, n, s0=0):
        """host_steps through the lazy form of the same calls (step(..., lazy=True) / step_multi(..., lazy=True)): every
        env's results arrive in page-locked host memory as compact wire records, the float observation is expanded on
        demand - here for one env per actor step, which is also read."""
        acc = 0.0
        if self.policy == "greedy" and self.multi:
            for k, ctrl in launch_plan(s0, n, self.spl):
                if ctrl == "greedy":
                    act, res = self.env.step_multi(k, controller="greedy", spacing=SPACING, lazy=True)
                    self.h_act[:] = act[-1]
                else:
                    act, res = self.env.step_multi(k, actions=self.h_act, controller="given", lazy=True)
                for j in range(k):
                    acc += float(res.reward[j, 0, 0]) + float(res.obs_of([0], step=j)[0, 0])
            return acc
        for s in range(s0, s0 + n):         # one te_step per actor step
            if self.policy == "greedy":
                if s % SPACING == 0:
                    self.h_act[:] = self.env.greedy_actions()
                a = self.h_act
            else:
                a = self.h_rand[s % 8]
            res = self.env.step(a, lazy=True)
            acc += float(res.reward[0, 0]) + float(res.obs_of([0])[0, 0])
        return acc

    def device_step(self, s):
        if self.policy == "greedy":
            if s % SPACING == 0:
                self.env.greedy_actions(out=self.d_act, stream=self.c.stream)
                self.launches += 1
            act = self.d_act
        else:
            act = self.d_rand[s % 8]
        self.env.step_device(act, self.d_obs[0], self.d_rew[0], self.d_done[0], stream=self.c.stream)
        self.launches += 1 + (1 if self.env_auto_reset else 0)

    @property
    def env_auto_reset(self):
        return bool(getattr(self.env, "auto_reset", False))

    def host_step(self, s):
        """The agent loop on the batched env through the public host API: actions host -> device, obs / reward / done
        device -> host every step; the greedy controller's output (te_greedy_actions) comes back every `spacing` steps."""
        if self.policy == "greedy":
            if s % SPACING == 0:
                self.h_act[:] = self.env.greedy_actions()
            act = self.h_act
        else:
            act = self.h_rand[s % 8]
        obs, rew, done = self.env.step(act)
        return float(rew[0, 0]) + float(obs[0, 0])  # the result is read on the host

    def timed_device(self, steps, warmup):
        c, env = self.c, self.env
        with c.torch.cuda.stream(c.tstream):
            self.device_steps(warmup)
            barrier(c)
            st0 = env.stats()
            self.launches = 0
            ev0, ev1 = c.torch.cuda.Event(enable_timing=True), c.torch.cuda.Event(enable_timing=True)
            barrier(c)
            ev0.record(c.tstream)
            self.device_steps(steps)
            ev1.record(c.tstream)
            barrier(c)
        ms = ev0.elapsed_time(ev1)
        st1 = env.stats()
        d = {k: st1[k] - st0[k] for k in ("vehicle_updates", "ticks", "actor_steps", "cars_generated", "overflows",
                                          "seq_fallback_ticks", "episodes")}
        tot = allreduce(c, [d["vehicle_updates"], d["ticks"], d["actor_steps"], d["cars_generated"], d["overflows"], d["episodes"]])
        ms_max = allreduce(c, [ms], "max")[0]
        return dict(ms=ms_max, local=d, vu=tot[0], ticks=tot[1], asteps=tot[2], gen=tot[3], ovf=tot[4], episodes=tot[5],
                    launches=self.launches)

    def last_step_outputs(self, steps):
        """On the host: what the last actor step of device_steps(steps) returned to its caller - obs, reward and done of
        every env, and the actions in force during that step.  Valid until the next device_steps call."""
        j = launch_plan(0, steps, self.spl)[-1][0] - 1 if self.multi else 0      # its slot in the last launch's outputs
        self.c.torch.cuda.synchronize()
        return {"obs": self.d_obs[j].cpu().numpy(), "reward": self.d_rew[j].cpu().numpy(),
                "done": self.d_done[j].cpu().numpy(), "actions": self.d_act.cpu().numpy()}

    def timed_host(self, steps, warmup, wire=False, agent=False):
        """agent=True: actions come from the host every decision (host_steps_agent); else the controller runs in the kernel."""
        c, env = self.c, self.env
        agent = agent and self.policy == "greedy" and self.multi
        if agent:
            run = lambda n: self.host_steps_agent(n, lazy=wire)     # noqa: E731
        else:
            run = self.host_steps_wire if wire else self.host_steps
        run(max(warmup, self.spl))     # at least one full-size launch: the page-locked result buffers grow on first use
        barrier(c)
        b0 = env.stats()["vehicle_updates"]
        t0 = time.perf_counter()
        run(steps)
        c.torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        vu = allreduce(c, [env.stats()["vehicle_updates"] - b0])[0]
        t = allreduce(c, [dt], "max")[0]
        E, I, OL = self.E, self.I, self.OL
        if agent:
            h2d, calls = E * I // SPACING, 2.0 / SPACING            # actions up once per decision; greedy_actions + step_multi
        elif self.multi:
            h2d, calls = 0, 1.0 / self.spl                           # controller in the kernel: nothing goes up
        else:
            h2d, calls = E * I, 1.0 + (1.0 / SPACING if self.policy == "greedy" else 0.0)
        return {"value": vu / t, "unit": "vehicle-updates/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int((env.d2h_bytes_per_step() if wire or not env.host_float_dma() else E * (OL * 4 + I * 4 + 1))
                                          + (E * I // SPACING if self.policy == "greedy" else 0)),
                "steps": steps, "host_calls_per_step": calls}

    def kernel_times(self, n):
        """Mean duration of one step-kernel launch (CUDA events on the launch stream, te_last_kernel_ms) and the
        vehicle-updates it processed; a launch is `steps_per_launch` actor steps."""
        kms, kvu = [], []
        spl = self.spl
        with self.c.torch.cuda.stream(self.c.tstream):
            for i in range(n):
                b0 = self.env.stats()["vehicle_updates"]
                self.device_steps(spl, i * spl)
                kms.append(self.env.last_kernel_ms())
                kvu.append(self.env.stats()["vehicle_updates"] - b0)
        return float(np.mean(kms)), float(np.mean(kvu))

    def occupancy(self):
        """Ring occupancy of the current state of this rank's envs (cars per road; a ring holds at most 18)."""
        cars = self.env.cars_on_roads_flat()
        r = self.env.train_roads
        tr, ex = cars[:, :r], cars[:, r:]
        hist = np.bincount(cars.reshape(-1), minlength=19)[:19]
        return {"cars_per_env": float(cars.sum(axis=1).mean()), "mean_cars_per_train_road": float(tr.mean()),
                "mean_cars_per_exit_road": float(ex.mean()), "frac_rings_ge_14": float((cars >= 14).mean()),
                "frac_rings_full_18": float((cars >= 18).mean()), "mean_ring_occupancy_frac": float(cars.mean() / 18.0),
                "hist_cars_per_road_0_to_18": [int(x) for x in hist]}

    def close(self):
        self.env.close()
        for k in ("d_act", "d_acts", "d_obs", "d_rew", "d_done", "d_rand"):
            if hasattr(self, k):
                delattr(self, k)
        self.c.torch.cuda.empty_cache()


def parity_spot(c, w, E, steps=30, nspot=4):
    """On THIS rank: `nspot` global env ids of the default-grid workload (first, last and two in between of the rank's
    block) stepped through the host API inside the full E-env batch and replayed on the CPU oracle with the same Philox
    key (seed, GLOBAL env id): actions, observations, rewards, done flags and the final car state must be bit-equal."""
    from oracle.oracle import OracleEnv
    from traffic_env_b200.arrivals import gap_cdf
    from traffic_env_b200 import VecTrafficEnv
    env = VecTrafficEnv(m=w["m"], n=w["n"], length=w["length"], num_envs=E, local_cars_per_sec=w["lcps"],
                        arrivals="philox", seed=2026, env_id_base=c.rank * E, device=c.local, ticks_per_step=K_TICKS,
                        remi=True)
    I = env.intersections
    env.reset()
    ids = sorted(set([0, E // 3, (2 * E) // 3, E - 1]))[:nspot]
    cdf = gap_cdf(env.cars_per_sec * 0.5)
    orc = []
    for e in ids:
        st = env.get_state(e, 1)
        o = OracleEnv(w["m"], w["n"], w["length"], 0.5)
        o.reset(st["obs"][0, 2 * env.train_roads:2 * env.train_roads + I])   # the Philox-drawn initial phases
        o.philox_seed(2026, c.rank * E + e, cdf)
        orc.append(o)
    ok = True
    act = np.zeros((E, I), np.uint8)
    oact = [np.zeros(I, np.int32) for _ in ids]
    for s in range(steps):
        if s % SPACING == 0:
            act[:] = env.greedy_actions()
            for j, o in enumerate(orc):
                oact[j] = (o.cars_on_roads().reshape(-1, 4).dot([1, 1, -1, -1]) < 0).astype(np.int32)
        obs, rew, done = env.step(act)
        for j, (e, o) in enumerate(zip(ids, orc)):
            oo, orw, od = o.actor_step_philox(oact[j], K_TICKS, use_remi=True)
            ok = ok and (act[e] == oact[j]).all() and obs[e].tobytes() == oo.tobytes() and \
                rew[e].tobytes() == orw.tobytes() and bool(done[e]) == od
    for e, o in zip(ids, orc):
        st = env.get_state(e, 1)
        ok = ok and (st["leading"][0] == o.leading).all() and (st["lastcar"][0] == o.lastcar).all()
        xs, vs = o.live_state()
        gx, gv = [], []
        for rd in range(env.roads):
            sl = int(st["leading"][0, rd])
            while sl != int(st["lastcar"][0, rd]):
                sl = 1 if sl + 1 >= 20 else sl + 1
                gx.append(st["x"][0, rd, sl]); gv.append(st["v"][0, rd, sl])
        ok = ok and np.asarray(gx, np.float32).tobytes() == xs.tobytes() and np.asarray(gv, np.float32).tobytes() == vs.tobytes()
    env.close()
    return bool(ok), [int(c.rank * E + e) for e in ids]


def single_env_dropin(steps_budget_s=3.0):
    """BASELINE.json configs[0] on the drop-in: gym.make('traffic-v0') + Remi(Repeater(10)), `fixed` policy
    (algorithms/fixed.py:6-17, spacing 3), episodes of 120 actor steps, MT19937 arrivals replayed on the host.
    The gym / args stand-ins come from tests/support (the GPU box has neither gym nor the reference)."""
    from tests.support import install_dropin
    install_dropin()
    import gym
    import gym_traffic  # noqa: F401
    from args import FLAGS
    from gym_traffic.envs.roadgraph import GridRoad
    from traffic_env_b200.wrappers import Remi, Repeater
    FLAGS.local_cars_per_sec, FLAGS.rate, FLAGS.poisson, FLAGS.entry, FLAGS.learn_switch = 0.12, 0.5, True, "all", False
    np.random.seed(0)
    base = gym.make("traffic-v0")
    base.set_graph(GridRoad(3, 3, 250))
    base.seed_generator(0)
    base.reset_entrypoints()
    env = Remi(Repeater(K_TICKS)(base))
    acts = [np.zeros(9), np.ones(9)]

    def episode():
        env.reset()
        n = 0
        for i in range(EPISODE_LEN):
            obs, rew, done, info = env.step(acts[int((i % (2 * SPACING)) >= SPACING)])
            n += 1
            if done:
                break
        return n
    episode()   # creates the CUDA context / handle
    t0, n = time.perf_counter(), 0
    while time.perf_counter() - t0 < steps_budget_s:
        n += episode()
    dt = time.perf_counter() - t0
    return {"actor_steps_per_sec": n / dt, "ticks_per_sec": n * K_TICKS / dt, "episodes_of": EPISODE_LEN,
            "what": "one env, Remi(Repeater(10)) over the drop-in TrafficEnv, `fixed` policy, one fused launch per actor "
                    "step, MT19937 arrival generator replayed on the host (launch- and host-bound: one CTA on the GPU)"}


def secondary_block(c, a, arith_peak):
    """Everything BASELINE.json names besides the headline line; runs after the timed region."""
    out = {}
    steps, warm = max(6, min(a.steps, 20)), max(3, min(a.warmup, 5))
    w3 = WORKLOADS["grid3x3_L250_greedy"]
    E3 = w3["envs"]
    # (iv) parity spot check on every rank, inside the full-size batch
    ok, ids = parity_spot(c, w3, E3)
    allok = allreduce(c, [1.0 if ok else 0.0], "min")[0] == 1.0
    out["parity_spot"] = {"ok": bool(allok), "ranks": c.world, "global_env_ids_rank0": ids, "actor_steps": 30,
                          "what": "4 envs of each rank's 131072-env default-grid batch vs the CPU oracle (same Philox key): "
                                  "actions, obs, reward, done every step and the final car state, bit for bit; min over ranks"}
    # (i) default grid, 131072 envs per GPU: greedy / no reset (kernel-quality number, comparable across rounds) ...
    r3 = Runner(c, w3, E3, policy="greedy", multi=not a.no_multi, launch_steps=a.launch_steps)
    with c.torch.cuda.stream(c.tstream):
        r3.device_steps(w3["preroll"])
    d = r3.timed_device(steps, warm)
    k_ms, k_vu = r3.kernel_times(min(steps, 8))
    e2e_float = r3.timed_host(max(3, steps // 2), 3, agent=True)
    e2e = r3.timed_host(max(3, steps // 2), 3, wire=True, agent=True)
    e2e_dc = r3.timed_host(max(3, steps // 2), 3, wire=True)
    occ = r3.occupancy()
    out["grid3x3_L250_greedy"] = {
        "value": d["vu"] / (d["ms"] * 1e-3), "unit": "vehicle-updates/s", "envs_per_gpu": E3, "envs_total": E3 * c.world,
        "ms_per_step": d["ms"] / steps, "steps": steps, "e2e": e2e, "e2e_float": e2e_float, "e2e_device_controller": e2e_dc,
        "kernel_ms": k_ms,
        "env_actor_steps_per_sec": d["asteps"] / (d["ms"] * 1e-3),
        "roofline_compute": {"achieved": k_vu / (k_ms * 1e-3), "peak": arith_peak,
                             "frac": (k_vu / (k_ms * 1e-3) / arith_peak) if arith_peak else None},
        "cars_per_env": occ["cars_per_env"], "policy": "greedy(spacing=3), no reset, %d-step pre-roll" % w3["preroll"]}
    r3.close()
    # ... and as BASELINE config 4 prescribes: random policy, auto-reset (overflow or 120 actor steps)
    r4 = Runner(c, w3, E3, policy="random", auto_reset=True, episode_len=EPISODE_LEN)
    with c.torch.cuda.stream(c.tstream):
        r4.device_steps(EPISODE_LEN + 17)     # past the first synchronous episode boundary
    d = r4.timed_device(steps, warm)
    e2e_float = r4.timed_host(max(3, steps // 2), 3)
    e2e = r4.timed_host(max(3, steps // 2), 3, wire=True)
    occ = r4.occupancy()
    st = r4.env.stats()
    out["config4_grid3x3_random_autoreset"] = {
        "value": d["vu"] / (d["ms"] * 1e-3), "unit": "vehicle-updates/s", "envs_per_gpu": E3, "envs_total": E3 * c.world,
        "ms_per_step": d["ms"] / steps, "steps": steps, "e2e": e2e, "e2e_float": e2e_float,
        "env_actor_steps_per_sec": d["asteps"] / (d["ms"] * 1e-3), "cars_per_env": occ["cars_per_env"],
        "episodes_closed_rank0": int(st["episodes"]),
        "mean_episode_return_rank0": (st["return_sum"] / st["episodes"]) if st["episodes"] else None,
        "policy": "uniform random actions per intersection per actor step (device-resident), TE_AUTO_RESET, episode_len 120"}
    r4.close()
    # (ii) the headline workload the way every reference agent runs it: reset on `done` or after 120 actor steps
    wh = WORKLOADS[a.workload]
    Eh = a.envs or wh["envs"]
    rh = Runner(c, wh, Eh, policy="greedy", auto_reset=True, episode_len=EPISODE_LEN)
    with c.torch.cuda.stream(c.tstream):
        rh.device_steps(EPISODE_LEN + 40)
    d = rh.timed_device(steps, warm)
    occ = rh.occupancy()
    out["headline_auto_reset"] = {
        "value": d["vu"] / (d["ms"] * 1e-3), "unit": "vehicle-updates/s", "envs_per_gpu": Eh, "ms_per_step": d["ms"] / steps,
        "ticks_per_actor_step": d["ticks"] / max(d["asteps"], 1.0), "overflows_per_actor_step": d["ovf"] / max(d["asteps"], 1.0),
        "episodes_closed_in_timed_region": d["episodes"], "occupancy_rank0": occ,
        "what": "%s with TE_AUTO_RESET + episode_len 120 (envs restart empty, desynchronised by overflow resets)" % a.workload}
    rh.close()
    # (iii) config 5: learner-style rollouts (a3c.py:52-63 contract) - rank 0; (v) config 1: the single-env drop-in
    if c.rank == 0:
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        try:
            import rollout_bench as rb
            roll = {"device": rb.run_device(E3, 120)}
            for T in (4, 16, 64):
                roll["threads_%d" % T] = rb.run_threads(T, 120)
            out["config5_rollout"] = roll
        except Exception as ex:  # the bench line must survive a failure of an auxiliary measurement
            out["config5_rollout"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
        try:
            out["config1_single_env_dropin"] = single_env_dropin()
            from oracle import oracle as orc
            orc.build()
            r1 = cpu_run("grid3x3_L250_greedy", 1, 30, 3.0, policy="fixed")
            out["config1_single_env_dropin"]["cpu_port_one_core"] = {
                "actor_steps_per_sec": r1["actor_steps"] / r1["seconds"], "vehicle_updates_per_sec": r1["value"],
                "what": "oracle port, same grid and policy, no reset; the unmodified numba reference: profiles/cpu_reference_numba.json"}
        except Exception as ex:
            out["config1_single_env_dropin"] = {"error": "%s: %s" % (type(ex).__name__, ex)}
    barrier(c)
    return out


def b200_arm(a):
    c = setup_dist()
    torch = c.torch
    w = WORKLOADS[a.workload]
    E = a.envs or w["envs"]
    preroll = w["preroll"] if a.preroll < 0 else a.preroll
    run = Runner(c, w, E, policy="greedy", multi=not a.no_multi, launch_steps=a.launch_steps)
    env = run.env
    I, OL = run.I, run.OL
    sampler = ClockSampler(c.local)
    if c.rank == 0:
        sampler.start()   # nvidia-smi needs a few hundred ms to deliver its first sample; the pre-roll, the warm-up
                          # and the timed region run the same kernel back to back, so all samples are under load
    with torch.cuda.stream(c.tstream):
        run.device_steps(preroll)
    torch.cuda.synchronize()
    occ = run.occupancy()
    d = run.timed_device(a.steps, a.warmup)
    mark = sampler.mark()
    if a.dump_outputs and c.rank == 0:
        dump_outputs(a.dump_outputs, run.last_step_outputs(a.steps))
    ms_max, n_launch = d["ms"], d["launches"]
    vu_all, ticks_all, asteps_all, gen_all, ovf_all = d["vu"], d["ticks"], d["asteps"], d["gen"], d["ovf"]
    loc = d["local"]

    # per-launch kernel time (CUDA events on the launch stream, separate pass so the sync does not sit in the timed region)
    k_ms, k_vu = run.kernel_times(min(a.steps, 10))
    spl = run.spl                                          # actor steps per launch
    cars_env = k_vu / E / spl / (loc["ticks"] / max(loc["actor_steps"], 1))
    R, r = env.roads, env.train_roads
    arr_per_step = loc["cars_generated"] / max(loc["actor_steps"], 1)
    # SURVEY.md 8d per env and LAUNCH: car state and ring indices read + written once, phase/elapsed r/w, actions; per
    # actor step of the launch: observation, reward, done, arrivals
    bytes_env = 2 * (8 * cars_env + 8 * R) + 4 * I + 2 * 8 * I + spl * (4 * (2 * r + I) + 4 * I + 1 + 2 * arr_per_step)
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = bytes_env * E / (k_ms * 1e-3) / 1e9
    traffic, traffic_note = measured_traffic(a.workload)

    # end to end through the public API with HOST buffers: what the greedy agent does (greedy.py:13-17)
    # `e2e` / `e2e_float`: the AGENT is on the host - its actions go host -> device every decision, every actor step's results
    # come device -> host; `e2e_device_controller`: the same with the controller inside the kernel (nothing goes up).
    e2e = e2e_float = e2e_dc = None
    if not a.no_e2e:
        e2e_float = run.timed_host(max(10, a.steps), max(3, min(a.warmup, 5)), agent=True)
        e2e = run.timed_host(max(10, a.steps), max(3, min(a.warmup, 5)), wire=True, agent=True)
        e2e_dc = run.timed_host(max(10, a.steps), max(3, min(a.warmup, 5)), wire=True)
        e2e["api"] = ("the greedy agent on the host (greedy.py:13-17): every %d actor steps VecTrafficEnv.greedy_actions(out=pinned) "
                      "(greedy.py:14-16 evaluated on the device-resident ring counts, actions device -> host), then "
                      "VecTrafficEnv.step_multi(%d, actions=pinned, controller='given', lazy=True) -> te_step_multi_wire(TE_HOST): "
                      "actions host -> device from page-locked memory, one launch for the steps the decision holds for; per actor "
                      "step the results of EVERY env arrive in page-locked host memory as compact wire records (%d B per env: u8 "
                      "passed / detected, f32 light / reward, u8 done - lossless: the counts are small integers); the float "
                      "observation is expanded on demand (WireResult.obs / obs_of), here for one env per step, and read" %
                      (SPACING, SPACING, env.wire.stride))
        e2e_dc["api"] = ("VecTrafficEnv.step_multi(%d, controller='greedy', spacing=%d, lazy=True): the controller runs inside the "
                         "kernel (no host -> device traffic; the chosen actions come back), %d actor steps per launch, results as "
                         "for e2e" % (run.spl, SPACING, run.spl))
        e2e_float["api"] = ("the eager form of the e2e call (lazy=False): every env's float obs[%d] / reward / done in host "
                            "memory every actor step - %s" % (env.obs_len, "float arrays written by the copy engine (few host "
                            "cores per GPU)" if env.host_float_dma() else "wire records expanded by %s helper threads of the handle "
                            "while the next slices are simulated" % os.environ.get("TE_HOST_THREADS")))
    clocks = sampler.stop(0, mark) if c.rank == 0 else None

    cpu = None
    if c.rank == 0 and c.world == 1 and not a.no_cpu_baseline:
        from oracle import oracle as orc
        orc.build()
        r1 = cpu_run(a.workload, 1, 60, a.cpu_seconds)
        cpu = {"value": r1["value"], "unit": "vehicle-updates/s", "cores": 1, "kind": "port",
               "sample": "1 env of %s on 1 core (oracle/traffic_oracle.c): 60-actor-step pre-roll, then %.0f s of "
               "actor steps (%d steps); `--impl reference` runs the same port on all %d host cores" %
               (a.workload, r1["seconds"], r1["actor_steps"], os.cpu_count() or 1)}

    barrier(c)
    flush_gbs = env.stage_bandwidth(5) if c.rank == 0 else None
    arith_peak = arith_peak_general = None
    if c.rank == 0:
        from traffic_env_b200.vec_env import idm_arithmetic_peak
        arith_peak = idm_arithmetic_peak(device=c.local)                     # the form the step kernels run (tame handle)
        arith_peak_general = idm_arithmetic_peak(device=c.local, form=0)     # general checked form: round 1's denominator
    arith_peak = allreduce(c, [arith_peak or 0.0], "max")[0]
    run.close()
    secondary = None
    if not a.no_secondary:
        secondary = secondary_block(c, a, arith_peak)
    if c.rank == 0:
        sec = ms_max * 1e-3
        value = vu_all / sec
        fp32_peak = 148 * 128 * 2 * (clocks["sm_mhz"] or 1965.0) * 1e6 if clocks else None
        line = {
            "metric": "vehicle_updates_per_sec", "value": value, "unit": "vehicle-updates/s", "n_gpus": c.world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_max / a.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic",
            "config": bench_config(a, w, E),
            "env_steps_per_sec": {"ticks": ticks_all / sec, "actor_steps": asteps_all / sec},
            "ticks_per_actor_step": ticks_all / max(asteps_all, 1.0), "overflows_per_actor_step": ovf_all / max(asteps_all, 1.0),
            "ordered_transfer_ticks_frac_rank0": loc["seq_fallback_ticks"] / max(loc["ticks"], 1),
            "steady_state_occupancy_rank0": occ,
            "target_8gpu": 1e11, "frac_of_per_gpu_target": value / c.world / 1.25e10,
            "clocks": clocks, "e2e": e2e, "e2e_float": e2e_float, "e2e_device_controller": e2e_dc, "gpu_launches": n_launch,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "traffic_source": traffic_note, "kernel": "te_step_kernel", "kernel_ms": k_ms,
                         "actor_steps_per_launch": spl, "algorithmic_bytes_per_env_launch": bytes_env, "cars_per_env": cars_env,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s",
                         "note": "the fused K-tick kernel is issue/FP64-pipe bound, not HBM bound (SURVEY.md 8d); see roofline_issue"},
            "roofline_flush": {"bound": "hbm", "achieved": flush_gbs, "peak": peak, "unit": "GB/s", "frac": flush_gbs / peak,
                               "what": "the step kernel's bulk-TMA stage-in + flush alone (te_stage_kernel: same CTA shape "
                               "and shared-memory footprint, no ticks), read + written bytes"},
            "roofline_compute": {"bound": "idm arithmetic (registers only, all lanes busy: te_idm_peak_form micro-kernel, the "
                                 "form of the update the step kernel runs - compile-time archetype, no validity predicate - at "
                                 "the better of 32 and 64 warps per SM)",
                                 "achieved": k_vu / (k_ms * 1e-3), "peak": arith_peak,
                                 "unit": "vehicle-updates/s", "frac": k_vu / (k_ms * 1e-3) / arith_peak,
                                 "peak_general_checked_form": arith_peak_general,
                                 "frac_of_general_checked_form": k_vu / (k_ms * 1e-3) / arith_peak_general,
                                 "note": "round 1 and the round-2 profiles before the tame mode quote fractions of the "
                                 "general checked form's rate"},
            "roofline_issue": {"ops_per_vehicle_update": OPS_PER_UPDATE,
                               "achieved_gops": k_vu * OPS_PER_UPDATE / (k_ms * 1e-3) / 1e9,
                               "fp32_peak_gops_nominal_at_clock": fp32_peak / 1e9 if fp32_peak else None},
            "cpu_baseline": cpu,
            "secondary": secondary,
        }
        print(json.dumps(line), flush=True)
    if c.world > 1:
        c.dist.destroy_process_group()


def main():
    a = parse()
    if a.impl == "reference":
        reference_arm(a)
    else:
        b200_arm(a)


if __name__ == "__main__":
    main()
