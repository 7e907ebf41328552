#!/usr/bin/env python
"""bench.py — so100 env-steps/s at 65 536 envs/GPU (BASELINE.json metric), one process per GPU.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--task Env01] [--envs-per-gpu 65536]
                    [--dump-outputs DIR]

A "step" is one `so100_step` launch over every env of this rank: pre-step task logic, 16 physics substeps,
obs / reward / termination / TimeLimit and in-kernel auto-reset.  Inputs (actions) are resident in HBM when the timed
region starts; `e2e` repeats the measurement through the host-buffer C-ABI call (pinned host actions in, host
obs / reward / done out, copies inside the timed region).  Rank 0 prints ONE JSON line.

`--dump-outputs DIR` writes what the last timed step returned (see `dump_outputs`).  The inputs depend on the
arguments only, so two builds run with the same arguments can be compared output for output.  bench.py writes nothing
into the source tree (which may be read-only): the CPU leg's -march=native oracle is compiled into the temp directory.

`--impl reference`: the reference's CPU path.  MuJoCo is not installable in this image (no wheel, no network), so the
timed engine is the repo's fp64 C oracle (kind "port") on all host cores, on a bounded sample of the same workload.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # no __pycache__ in the source tree either

# Algorithmic work per env step (DESIGN.md "Roofline arithmetic"; tools/count_flops.cpp counts the generic recursion with
# the shipped sweep schedule: 5 Gauss-Seidel sweeps on the first substep of an env step, 3 on the other 15)
FLOP_PER_ENV_STEP = {1: 56900.0, 2: 56900.0, 5: 57200.0, 6: 56900.0}
BYTES_PER_ENV_STEP = {1: 338.0, 2: 362.0, 5: 420.0, 6: 362.0}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--task", default="Env01")
    ap.add_argument("--envs-per-gpu", type=int, default=65536)
    ap.add_argument("--cpu-envs", type=int, default=0, help="envs in the CPU sample (default: 256 per host thread)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--subproc-harness", type=float, default=0.0, help=argparse.SUPPRESS)  # internal: run the SubprocVecEnv-style CPU harness for this many seconds
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--e2e-device-buffers", default="", choices=["", "in", "out", "both"], help=argparse.SUPPRESS)  # experiment: the pipeline without the host link (needs SO100_HOST_ALLOW_DEVICE=1); not an e2e number
    ap.add_argument("--e2e-groups", type=int, default=8, help="env groups of the pipelined host path (so100_step_host_async)")
    ap.add_argument("--no-tasks", action="store_true", help="skip the Env02 / Env05 records (BASELINE configs 3, 4)")
    ap.add_argument("--no-ppo", action="store_true", help="skip the Env05 PPO record (BASELINE config 5)")
    ap.add_argument("--no-contact", action="store_true", help="skip the record of the opt-in arm-floor contact physics (SO100_FLAG_ARM_CONTACT)")
    ap.add_argument("--flags", type=int, default=0, help="SO100_FLAG_* bits for the env (e.g. 16 = no arm-floor contact)")
    ap.add_argument("--dump-outputs", metavar="DIR", default="",
                    help="write the arrays the last timed step returned as DIR/<name>.npy (float32 / float64, at most 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def workload(args) -> str:
    return (f"{args.task}, {args.envs_per_gpu} envs/GPU, U(-1,1) random actions, 16 substeps/step, in-kernel auto-reset, "
            "episode clocks staggered over the TimeLimit (decorrelated start)")


class ClockSampler:
    """Samples SM clock and throttle reasons with nvidia-smi WHILE the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._pump, daemon=True).start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for k, name in enumerate(names):
                if len(r) > 3 + k and r[3 + k].lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_oracle_rate(task: int, n_envs: int, seconds: float, threads: int):
    """env-steps/s of the fp64 C oracle on `threads` host threads (bounded sample)."""
    import numpy as np
    from oracle import pyoracle
    from oracle.pyoracle import Oracle
    from so100_mujoco_rl_b200.model import load_model
    from so100_mujoco_rl_b200.tasks import make_task_cfg
    pyoracle.use_native_build()  # -O3 -march=native for the timed CPU leg (BASELINE.md §3)
    o = Oracle(load_model().to_ctypes(), make_task_cfg(task, n_envs, seed=0))
    o.reset(nthreads=threads)
    rng = np.random.default_rng(0)
    acts = [rng.uniform(-1, 1, (n_envs, 6)).astype(np.float32) for _ in range(8)]
    o.step(acts[0], nthreads=threads)  # warm-up
    t0, k = time.perf_counter(), 0
    while True:
        o.step(acts[k % 8], nthreads=threads)
        k += 1
        dt = time.perf_counter() - t0
        if dt >= seconds:
            break
    return n_envs * k / dt, k, dt


def _subproc_worker(conn, task: int, seed: int):
    """One env per process, stepped on request (SB3 SubprocVecEnv's worker loop)."""
    import numpy as np
    from oracle import pyoracle
    from oracle.pyoracle import Oracle
    from so100_mujoco_rl_b200.model import load_model
    from so100_mujoco_rl_b200.tasks import make_task_cfg
    pyoracle.use_native_build()
    o = Oracle(load_model().to_ctypes(), make_task_cfg(task, 1, seed=seed, env_offset=seed))
    conn.send(o.reset())
    while True:
        a = conn.recv()
        if a is None:
            break
        obs, rew, term, trunc, *_ = o.step(np.asarray(a, dtype=np.float32).reshape(1, 6))
        conn.send((obs, float(rew[0]), bool(term[0] or trunc[0])))


def subproc_harness(task: int, seconds: float) -> dict:
    """The reference's CPU architecture at scale: one process per host core, one env each, an action pipe down and an
    (obs, reward, done) pipe up every step (Stable-Baselines3 SubprocVecEnv), oracle physics in the workers."""
    import multiprocessing as mp
    import numpy as np
    ctx = mp.get_context("fork")
    n = os.cpu_count() or 1
    pipes, procs = [], []
    for i in range(n):
        a, b = ctx.Pipe()
        pr = ctx.Process(target=_subproc_worker, args=(b, task, i), daemon=True)
        pr.start()
        pipes.append(a); procs.append(pr)
    for c in pipes:
        c.recv()
    rng = np.random.default_rng(0)
    acts = rng.uniform(-1, 1, (64, n, 6)).astype(np.float32)
    for k in range(20):  # warm-up
        for i, c in enumerate(pipes):
            c.send(acts[k % 64, i])
        for c in pipes:
            c.recv()
    t0, k = time.perf_counter(), 0
    while time.perf_counter() - t0 < seconds:
        for i, c in enumerate(pipes):
            c.send(acts[k % 64, i])
        for c in pipes:
            c.recv()
        k += 1
    dt = time.perf_counter() - t0
    for c in pipes:
        c.send(None)
    for pr in procs:
        pr.join(timeout=5)
    return {"value": n * k / dt, "unit": "env-steps/s", "processes": n, "seconds": dt}


def run_reference(args, rank: int):
    """Reference arm: the CPU path on the host's cores (oracle port; see module docstring)."""
    if rank != 0:
        return
    import numpy as np
    from oracle import pyoracle
    from oracle.pyoracle import Oracle, lib
    from so100_mujoco_rl_b200.model import load_model
    from so100_mujoco_rl_b200.tasks import MAX_EPISODE_STEPS, make_task_cfg, task_id
    native = pyoracle.use_native_build()  # -O3 -march=native for the timed CPU leg (BASELINE.md §3)
    task = task_id(args.task)
    threads = lib().orc_hw_threads()
    n = args.cpu_envs or 256 * threads
    o = Oracle(load_model().to_ctypes(), make_task_cfg(task, n, seed=0, flags=args.flags))
    o.reset(nthreads=threads)
    for i in range(n):  # the same decorrelated start as the GPU arm: episode clocks staggered over the TimeLimit
        st = o.state(i)
        st.elapsed_steps = (i * 2654435761) % MAX_EPISODE_STEPS[task]
        st.time = st.elapsed_steps * 0.032
        st.target_time = st.time
    rng = np.random.default_rng(0)
    acts = [rng.uniform(-1, 1, (n, 6)).astype(np.float32) for _ in range(8)]
    for w in range(max(args.warmup, 3)):
        o.step(acts[w % 8], nthreads=threads)
    t0 = time.perf_counter()
    for k in range(args.steps):
        out = o.step(acts[k % 8], nthreads=threads)
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(STEP_OUTPUTS, out)))
    value = n * args.steps / dt
    sample = f"{n} envs x {args.steps} steps of the {args.envs_per_gpu}-env workload, fp64 C oracle{' -O3 -march=native' if native else ''} (MuJoCo not installable here), {threads} threads"
    line = {
        "impl": "reference", "metric": "so100 env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * dt / args.steps, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload(args), "envs_per_gpu": args.envs_per_gpu, "task": args.task, "env_flags": args.flags},
        "cpu_baseline": {"value": value, "unit": "env-steps/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def emit(line: dict):
    """The contract is ONE JSON line on stdout; everything else (NCCL banner, torchrun notices) goes to stderr."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


# libraries (NCCL prints its version banner) write to fd 1: keep the real stdout aside and point fd 1 at stderr
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)

DUMP_BUDGET_BYTES = 64_000_000  # all ranks' files together, .npy headers included


def dump_outputs(out_dir: str, outputs: dict, rank: int = 0, world: int = 1):
    """Writes one step's outputs (name -> array with one row per env of this rank) as out_dir/<name>.npy: float64 stays
    float64, everything else becomes float32 (flags and episode lengths are small integers, exact in float32).
    terminal_obs / ep_return / ep_len are only defined where the episode ended in that step; their other rows hold
    whatever an earlier step left there and are written as 0.  With several ranks each writes its own env shard with a
    _rank<r> suffix.  When a rank's arrays exceed its share of DUMP_BUDGET_BYTES, the same fixed, seeded sample of env rows is kept
    in every array, in env order, and env_index<suffix>.npy lists the (local) rows kept."""
    import numpy as np
    arrays = {k: np.asarray(v) for k, v in outputs.items()}
    arrays = {k: v.astype(np.float64 if v.dtype == np.float64 else np.float32) for k, v in arrays.items()}
    ended = (arrays["terminated"] + arrays["truncated"]) > 0
    for k in ("terminal_obs", "ep_return", "ep_len"):
        arrays[k][~ended] = 0
    n = len(ended)
    row_bytes = sum(v[:1].nbytes for v in arrays.values())
    keep = min(n, (DUMP_BUDGET_BYTES // world - 4096) // (row_bytes + 8))  # 4 KiB: the headers; 8 B: env_index
    if keep < n:
        rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: v[rows] for k, v in arrays.items()}
        arrays["env_index"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    suffix = f"_rank{rank}" if world > 1 else ""
    for k, v in arrays.items():
        np.save(os.path.join(out_dir, f"{k}{suffix}.npy"), v)


# what one env step returns, in the order of `Oracle.step`'s tuple and of the fields of a StepResult
STEP_OUTPUTS = ("obs", "reward", "terminated", "truncated", "terminal_obs", "ep_return", "ep_len")


def profile_lookup(task: int, n: int, build_id: str):
    """ncu-derived figures of one step_kernel launch (profiles/step_kernel_profile.json, written by
    tools/ncu_to_profile.py from an `ncu --set full` capture), valid only for the sources they were measured on."""
    try:
        entries = json.load(open(os.path.join(ROOT, "profiles", "step_kernel_profile.json")))["entries"]
    except Exception:  # noqa: BLE001
        return None, True
    same = [e for e in entries if e.get("task") == task and e.get("envs") == n]
    for e in same:
        if e.get("csrc_hash") == build_id:
            return e, False
    return (same[-1] if same else None), True


def pin_to_gpu_numa_node(local_rank: int):
    """Run this rank's host threads (and hence its first-touch pinned allocations) on the NUMA node of its GPU."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(local_rank).pci_bus_id
        dom = getattr(torch.cuda.get_device_properties(local_rank), "pci_domain_id", 0)
        dev = getattr(torch.cuda.get_device_properties(local_rank), "pci_device_id", 0)
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{dev:02x}.0/numa_node"
        node = int(open(path).read().strip())
        if node < 0:
            return {"numa_node": node, "pinned": False}
        cpus = []
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus += list(range(int(a), int(b or a) + 1))
        allowed = sorted(set(cpus) & os.sched_getaffinity(0))
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"numa_node": node, "pinned": bool(allowed), "cpus": len(allowed)}
    except Exception as e:  # noqa: BLE001 - a hint, never fatal
        return {"numa_node": None, "pinned": False, "why": f"{type(e).__name__}"[:60]}


def timed_steps(env, ring, steps, flush, torch, before=None):
    """`steps` env.step launches, each bracketed by CUDA events on the launch stream, L2 flushed in between."""
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    out = []
    for k in range(steps):
        a = ring[k % len(ring)]
        if before is not None:
            a = before(k, a)
        flush.zero_()  # evict the env state from L2 between timed iterations
        ev[k][0].record()
        r = env.step(a)
        ev[k][1].record()
        out.append(r)
    return ev, out


def main():
    args = parse()
    if args.subproc_harness > 0:  # child invocation: no torch / CUDA in this process, workers are forked
        from so100_mujoco_rl_b200.tasks import task_id
        emit(subproc_harness(task_id(args.task), args.subproc_harness))
        return
    rank, local_rank, world = (int(os.environ.get(k, d)) for k, d in (("RANK", "0"), ("LOCAL_RANK", "0"), ("WORLD_SIZE", "1")))
    if args.impl == "reference":
        run_reference(args, rank)
        return

    import torch
    import torch.distributed as dist
    from so100_mujoco_rl_b200 import _native
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    from so100_mujoco_rl_b200.sharding import max_over_ranks
    from so100_mujoco_rl_b200.tasks import MAX_EPISODE_STEPS, OBS_DIM, task_id

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path (use --impl reference for the CPU arm)")
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if args.gpus > 1 and world == 1:
        raise SystemExit("launch multi-GPU runs with torch.distributed.run (one process per GPU)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa = pin_to_gpu_numa_node(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    task = task_id(args.task)
    n = args.envs_per_gpu
    steps, warmup = args.steps, max(args.warmup, 3)
    build_id = _native.lib().so100_build_id().decode()
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)      # > 126 MB L2
    g = torch.Generator(device=dev).manual_seed(1 + rank)
    ring = [torch.rand((n, 6), device=dev, generator=g) * 2 - 1 for _ in range(64)]  # U(-1,1) actions, resident in HBM

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def fresh_env(t, seed=0, flags=None):
        """Env-sharded (no collective on the step path), started from a DECORRELATED state: episode clocks staggered over
        the whole TimeLimit, then 64 untimed steps, so truncations + in-kernel resets run inside the timed region at
        their steady rate and no env is in its post-reset transient."""
        e = BatchedSo100Env(t, n, device=local_rank, seed=seed, env_offset=rank * n, flags=args.flags if flags is None else flags)
        e.reset()
        e.stagger_episodes()
        for w in range(64):
            e.step(ring[w % 64])
        return e

    # The clock sampler starts FIRST and the GPU is kept busy (the FP32 peak probe: no env state involved) until nvidia-smi
    # has delivered a sample and at least half a second has passed: on a fresh box the first nvidia-smi call takes longer
    # than the whole timed region, and a GPU coming out of idle clocks is not what the metric is about.  The same probe
    # runs for a quarter of a second after the timed region, so that the 100 ms sampling grid has points under load on
    # both sides of it; every sample kept was taken between the first and the last of these launches.
    import ctypes
    sampler = ClockSampler(local_rank)
    sampler.start()

    def spin(seconds, need_sample=False):
        tf_ = ctypes.c_double(0.0)
        t_end, t_max = time.perf_counter() + seconds, time.perf_counter() + 6.0
        while time.perf_counter() < t_end or (need_sample and not sampler.rows and time.perf_counter() < t_max):
            _native.check(_native.lib().so100_bench_fp32_peak(local_rank, 4096, ctypes.byref(tf_)))

    env = fresh_env(task)
    spin(0.5, need_sample=True)
    sampler.rows.clear()  # (samples from before the GPU was under load)
    for w in range(warmup):
        env.step(ring[w % 64])
    launches0 = env.stats()["launches"]
    barrier()
    t_wall0 = time.perf_counter()
    ev, res = timed_steps(env, ring, steps, flush, torch)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    spin(0.25)
    clocks = sampler.stop()
    total_ms = sum(a.elapsed_time(b) for a, b in ev)
    launches = env.stats()["launches"] - launches0
    stats = env.stats()
    if args.dump_outputs:  # before the e2e legs step this env further
        dump_outputs(args.dump_outputs, {k: getattr(res[-1], k).cpu().numpy() for k in STEP_OUTPUTS}, rank, world)

    # ---- end to end through the host-buffer C ABI (host actions in, host obs / reward / flags out, every step)
    e2e = None
    if not args.no_e2e:
        od = OBS_DIM[task]
        host = env.alloc_host()
        host_ring = [r.cpu().pin_memory() for r in ring[:8]]
        if args.e2e_device_buffers in ("out", "both"):
            host = {k: v.to(dev) for k, v in host.items()}
        if args.e2e_device_buffers in ("in", "both"):
            host_ring = ring[:8]
        st_ptr = torch.cuda.current_stream(dev).cuda_stream
        # (a) the synchronous call (what the SB3 VecEnv adapter makes): one launch, phases in series
        sync_s = float("nan")
        if not args.e2e_device_buffers:
            for w in range(max(warmup, 8)):
                env.step_host(host, actions=host_ring[w % 8])
            barrier()
            t0 = time.perf_counter()
            for k in range(steps):
                env.step_host(host, actions=host_ring[k % 8])
            barrier()
            sync_s = time.perf_counter() - t0
        # (b) the pipelined call: G env groups in rotation, each step of a group = its action rows in from pinned host
        # memory, its obs / reward / flag rows back into pinned host memory; the host waits for a group's rows before it
        # issues that group's next step (the policy's data dependency), while the other groups keep the GPU and both
        # directions of the link busy; groups are served in completion order (so100_step_host_wait_any)
        G = max(1, min(args.e2e_groups, 16))
        env.host_groups(G)
        def rotate(nsteps):
            """Every group takes `nsteps` steps; a group's next step is issued as soon as ITS previous rows are on the host."""
            count = [1] * G
            for g_ in range(G):
                env.step_host_async(host, g_, actions=host_ring[0], stream=st_ptr)
            left = G * nsteps
            while left:
                g_ = env.step_host_wait_any()
                left -= 1
                if count[g_] < nsteps:
                    env.step_host_async(host, g_, actions=host_ring[count[g_] % 8], stream=st_ptr)
                    count[g_] += 1

        rotate(max(warmup, 8))
        barrier()
        t0 = time.perf_counter()
        rotate(steps)
        barrier()
        pipe_s = time.perf_counter() - t0
        done_rows = float((host["terminated"] | host["truncated"]).sum())
        env.host_groups(1)
        # (c) what the host link alone could carry: the per-step payloads in both directions at once by copy engine, no
        # kernel, no dependency between the directions - on every rank at the same time (tools/pcie_bw.py's measurement)
        link_ms = float("nan")
        if not args.e2e_device_buffers:
            in_b, out_b = n * 6 * 4, n * (od * 4 + 6)
            h_in, h_out = torch.empty(in_b, dtype=torch.uint8).pin_memory(), torch.empty(out_b, dtype=torch.uint8).pin_memory()
            d_in, d_out = torch.empty(in_b, dtype=torch.uint8, device=dev), torch.empty(out_b, dtype=torch.uint8, device=dev)
            s1, s2 = torch.cuda.Stream(dev), torch.cuda.Stream(dev)

            def both(reps):
                for _ in range(reps):
                    with torch.cuda.stream(s1):
                        d_in.copy_(h_in, non_blocking=True)
                    with torch.cuda.stream(s2):
                        h_out.copy_(d_out, non_blocking=True)
            both(20)
            torch.cuda.synchronize(dev)
            barrier()
            t0 = time.perf_counter()
            both(200)
            torch.cuda.synchronize(dev)
            link_ms = (time.perf_counter() - t0) / 200 * 1e3
        # bytes per step: actions in; obs + reward + terminated + truncated out, plus the terminal rows
        # (terminal_obs + ep_return + ep_len) of the ~n/max_steps envs whose episode ended in that step
        per_done = od * 4 + 8
        e2e = {"pipe_s": max_over_ranks(pipe_s, dev), "sync_s": max_over_ranks(sync_s, dev), "groups": G, "h2d": n * 6 * 4,
               "d2h": n * (od * 4 + 4 + 1 + 1) + int(round(n / MAX_EPISODE_STEPS[task])) * per_done, "done_rows_last_step": done_rows,
               "link_ms": max_over_ranks(link_ms, dev)}

    total_ms = max_over_ranks(total_ms, dev)

    # ---- BASELINE configs 3 and 4: Env02 with a scripted-reach subset (relocations/s), Env05 (lost-cube resets/s)
    tasks_rec = None
    if not args.no_tasks:
        from so100_mujoco_rl_b200.scripted import reach_actions
        tasks_rec = {}
        for name, t in (("Env02", 2), ("Env05", 5)):
            e = fresh_env(t, seed=3)
            ksteps, kscr = max(20, min(steps, 50)), (min(2048, n) if t == 2 else 0)
            obs = e.obs.clone()
            aux_prev = e.get_state()["aux"][:3].clone() if t == 2 else None
            ms = reloc = dones = 0
            for k in range(ksteps + 5):
                a = ring[(k + 7) % 64].clone()
                if kscr:  # the scripted envs servo onto their block; the controller is host-side tooling, outside the timing
                    a[:kscr] = reach_actions(e, obs, kscr)
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(); r = e.step(a); e1.record()
                obs = r.obs.clone()
                e1.synchronize()
                if k >= 5:
                    ms += e0.elapsed_time(e1)
                    dones += int((r.terminated | r.truncated).sum())
                if t == 2:
                    aux = e.get_state()["aux"][:3]
                    if k >= 5:
                        reloc += int(((aux - aux_prev).abs().sum(0) > 0).sum()) - int((r.terminated | r.truncated).sum())
                    aux_prev = aux.clone()
            ms = max_over_ranks(ms, dev)
            rec = {"envs_per_gpu": n, "steps": ksteps, "ms_per_step": ms / ksteps, "env_steps_per_s": n * world * ksteps / (ms * 1e-3),
                   "episode_resets_per_s_rank0": dones / (ms * 1e-3)}
            if t == 2:
                rec.update({"scripted_envs": kscr, "relocations_rank0": reloc, "relocations_per_s_rank0": reloc / (ms * 1e-3)})
            tasks_rec[name] = rec
            e.close()

    # ---- the opt-in arm-floor contact physics (the reference's jaw-pad colliders): what the same workload costs with it
    contact_rec = None
    if not args.no_contact and not (args.flags & 16):
        e = fresh_env(task, seed=0, flags=args.flags | 16)
        ksteps = 10
        evc, resc = timed_steps(e, ring, ksteps, flush, torch)
        torch.cuda.synchronize(dev)
        ms = max_over_ranks(sum(a.elapsed_time(b) for a, b in evc), dev)
        touching = float(((e.get_state()["counters"][1] & 16) != 0).float().mean())
        below = float((resc[-1].obs[:, 14] < 0).float().mean()) if task != 5 else None
        below_off = float((res[-1].obs[:, 14] < 0).float().mean()) if task != 5 else None
        st_c = e.stats()
        contact_rec = {"flag": "SO100_FLAG_ARM_CONTACT", "ms_per_step": ms / ksteps, "env_steps_per_s": n * world * ksteps / (ms * 1e-3),
                       "slowdown_vs_default": (ms / ksteps) / (total_ms / steps), "envs_touching_floor_frac": touching,
                       "end_effector_below_floor_frac": below, "end_effector_below_floor_frac_without_contact": below_off,
                       "solver_unconverged": st_c["solver_unconverged"], "nan_resets": st_c["nan_resets"]}
        e.close()

    # ---- BASELINE config 5: Env05 PPO rollout + update (fused learner), env-sharded, one flat all-reduce per minibatch
    ppo_rec = None
    if not args.no_ppo:
        from so100_mujoco_rl_b200.ppo import FusedPPO, PPOConfig
        e = BatchedSo100Env(5, n, device=local_rank, seed=0, env_offset=rank * n, flags=args.flags)
        cfg = PPOConfig(n_steps=32, n_minibatches=8, n_epochs=10, seed=0)
        algo = FusedPPO(e, cfg, env_offset=rank * n)
        algo.learn(total_samples=n * world * cfg.n_steps, log_every=0, callback=lambda r_: None)   # warm-up iteration
        s0, r0, u0 = algo.stats.samples, algo.stats.rollout_s, algo.stats.update_s
        iters = 2
        barrier()
        t0 = time.perf_counter()
        algo.learn(total_samples=s0 + iters * n * world * cfg.n_steps, log_every=0, callback=lambda r_: None)
        barrier()
        dt = max_over_ranks(time.perf_counter() - t0, dev)
        ppo_rec = {"task": "Env05", "envs_per_gpu": n, "n_steps": cfg.n_steps, "n_minibatches": cfg.n_minibatches, "n_epochs": cfg.n_epochs,
                   "iterations": iters, "samples_per_s": (algo.stats.samples - s0) / dt, "rollout_s_per_iter": (algo.stats.rollout_s - r0) / iters,
                   "update_s_per_iter": (algo.stats.update_s - u0) / iters,
                   "mean_step_reward": algo.stats.history[-1]["mean_step_reward"]}
        e.close()

    if rank == 0:
        total_envs = n * world
        value = total_envs * steps / (total_ms * 1e-3)
        per_gpu = value / world
        tf = ctypes.c_double(0.0)
        _native.check(_native.lib().so100_bench_fp32_peak(local_rank, 4096, ctypes.byref(tf)))
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak, hbm_src = (peaks["hbm_gbs"], "of measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "of fallback")
        ach_tf = per_gpu * FLOP_PER_ENV_STEP[task] / 1e12
        ach_gb = per_gpu * BYTES_PER_ENV_STEP[task] / 1e9
        prof, stale = profile_lookup(task, n, build_id)
        dones_in_region = int(sum(int((r.terminated | r.truncated).sum()) for r in res[-1:]))
        line = {
            "metric": "so100 env-steps/sec", "value": value, "unit": "env-steps/s", "n_gpus": world, "steps": steps,
            "warmup": warmup, "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": workload(args), "envs_per_gpu": n, "task": args.task, "l2": "flushed between timed steps (256 MiB memset)",
                       "parallelism": f"env-sharded x{world}, no collective on the step path",
                       "env_flags": args.flags, "episodes_ended_in_last_timed_step_rank0": dones_in_region},
            "roofline": {"bound": "fp32", "achieved": ach_tf, "peak": tf.value, "unit": "TFLOP/s",
                         "frac": ach_tf / tf.value if tf.value else None,
                         # dram__bytes_read.sum + dram__bytes_write.sum of ONE step_kernel launch from an `ncu --set full` capture of
                         # this library build (profiles/step_kernel_profile.json); null + stale when the sources have changed since
                         "traffic": (prof or {}).get("traffic_bytes") if not stale else None,
                         "peak_source": "FFMA probe measured in this run (so100_bench_fp32_peak); nominal 74.5",
                         "flop_per_env_step": FLOP_PER_ENV_STEP[task],
                         "frac_is": "useful algorithmic FLOP of the generic recursion per second / FFMA peak (not pipe utilisation)",
                         "executed_flop_per_env_step": (prof or {}).get("executed_flop_per_env_step"),
                         "executed_frac": (per_gpu * prof["executed_flop_per_env_step"] / 1e12 / tf.value
                                           if prof and prof.get("executed_flop_per_env_step") and tf.value else None),
                         "pipe_fma_pct": (prof or {}).get("pipe_fma_pct"), "issue_active_pct": (prof or {}).get("issue_active_pct"),
                         "profile": {"file": "profiles/step_kernel_profile.json", "csrc_hash": (prof or {}).get("csrc_hash"),
                                     "build_id": build_id, "stale": stale}},
            "roofline_hbm": {"bound": "hbm", "achieved": ach_gb, "peak": hbm_peak, "unit": "GB/s", "frac": ach_gb / hbm_peak,
                             "peak_source": hbm_src, "bytes_per_env_step": BYTES_PER_ENV_STEP[task]},
            "gpu_launches": launches,
            "clocks": clocks,
            "wall_s_timed_region": t_wall,
            "solver_unconverged": stats["solver_unconverged"], "nan_resets": stats["nan_resets"],
            "host": numa,
        }
        if e2e:
            line["e2e"] = {"value": total_envs * steps / e2e["pipe_s"], "unit": "env-steps/s",
                           "h2d_bytes_per_step": e2e["h2d"], "d2h_bytes_per_step": e2e["d2h"],
                           "how": f"so100_step_host_async / _wait over {e2e['groups']} env groups in rotation (pinned host buffers in place "
                                  "over the host link; every group's rows are on the host before its next step is issued)",
                           "groups": e2e["groups"]}
            if e2e["link_ms"] == e2e["link_ms"]:  # (not NaN) the link alone, all ranks copying at once
                ceiling = total_envs / (e2e["link_ms"] * 1e-3)
                line["e2e"]["host_link"] = {"ms_per_step_both_directions": e2e["link_ms"], "ceiling_env_steps_per_s": ceiling,
                                            "frac_of_ceiling": line["e2e"]["value"] / ceiling,
                                            "how": "per-step payloads H2D and D2H at once by copy engine from / to pinned memory, no kernel, "
                                                   "every rank at the same time (max over ranks)"}
            line["e2e_sync"] = {"value": total_envs * steps / e2e["sync_s"], "unit": "env-steps/s",
                                "how": "so100_step_host: one synchronous call per step for the whole batch (the SB3 VecEnv adapter's call)"}
        if tasks_rec:
            line["tasks"] = tasks_rec
        if ppo_rec:
            line["ppo"] = ppo_rec
        if contact_rec:
            line["arm_floor_contact"] = contact_rec
        if world == 1 and not args.no_cpu_baseline:
            threads = os.cpu_count() or 1
            ncpu = args.cpu_envs or 256 * threads
            rate, k, dt = cpu_oracle_rate(task, ncpu, 12.0, threads)
            one, k1, dt1 = cpu_oracle_rate(task, 1, 2.0, 1)  # BASELINE config 1: ONE env on one core, as the reference steps it
            line["cpu_baseline"] = {"value": rate, "unit": "env-steps/s", "cores": threads, "kind": "port",
                                    "sample": f"{ncpu} envs x {k} steps ({dt:.1f} s) of the same workload on the fp64 C oracle",
                                    "per_core": rate / threads, "single_env_single_core": one}
            try:  # the reference's own architecture at scale (north star): SubprocVecEnv over the host's cores, fresh process
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--subproc-harness", "3", "--task", args.task],
                                   capture_output=True, text=True, timeout=120)
                line["cpu_baseline"]["subproc_vec_env"] = json.loads(r.stdout.strip().splitlines()[-1])
            except Exception as e:  # noqa: BLE001 - a reported extra, never fatal
                line["cpu_baseline"]["subproc_vec_env"] = {"error": f"{type(e).__name__}: {e}"[:200]}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
