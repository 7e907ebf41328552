"""A/B of two builds of libso100_b200.so in one process, with bench.py's method.

    python tools/bench_ab.py OLD.so NEW.so [--rounds 7] [--out profiles/r3_substep_instructions_ab.json]

Each library gets its own envs: Env01 / Env02 / Env05 at 65 536 envs on the default kernel, Env02 with the arm-floor
contact (SO100_FLAG_ARM_CONTACT) and Env01 with per-env dynamics parameters (the PARAMS kernels).  Every env starts
decorrelated (episode clocks staggered over the TimeLimit, then 64 untimed steps); each timed step is bracketed by CUDA
events with L2 flushed in between by a 256 MiB memset.  The libraries are timed in alternating rounds, the order
swapped every round, so that clock and neighbour drift hits both alike; the figure per round is the mean step time of
its timed steps, and the result is the median over rounds with the spread (min, max) beside it, and b / a - 1 within
each round.  The card's name, power limit and maximum SM clock are read with a query-only nvidia-smi call in the same
run.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

# (label, task, flags, per-env parameters, timed steps per round: the contact path is ~10x slower per step)
CONFIGS = [("Env01", 1, 0, False, 200), ("Env02", 2, 0, False, 200), ("Env05", 5, 0, False, 200),
           ("Env02_arm_contact", 2, 16, False, 20), ("Env01_params", 1, 0, True, 200)]
PARAMS = "kp=0.7:1.3,damping=0.8:1.2,forcerange=0.8:1.0,frictionloss=0.5:2"


def card() -> dict:
    out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, timeout=60).stdout.strip()
    name, power, sm = (x.strip() for x in out.split(","))
    return {"name": name, "power_limit": power, "sm_max_clock": sm}


def load(path: str):
    """The ctypes handle of the library at `path`, configured like the package's own (a second library is a second
    dlopen of a different file: both stay loaded side by side)."""
    from so100_mujoco_rl_b200 import _native
    _native.LIB_PATH, _native._lib = os.path.abspath(path), None
    return _native.lib()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("lib_a", help="baseline library")
    ap.add_argument("lib_b", help="candidate library")
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--only", default=None, help="comma-separated config labels (default: all)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_ab.py measures the GPU: no CUDA device")
    from so100_mujoco_rl_b200 import _native
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    from so100_mujoco_rl_b200.randomization import ParamRanges

    n, dev = args.envs, torch.device("cuda", 0)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    g = torch.Generator(device=dev).manual_seed(1)
    ring = [torch.rand((n, 6), device=dev, generator=g) * 2 - 1 for _ in range(64)]
    configs = [c for c in CONFIGS if args.only is None or c[0] in args.only.split(",")]
    libs = {"a": load(args.lib_a), "b": load(args.lib_b)}

    def fresh(lib, task, flags, params):
        _native._lib = lib  # BatchedSo100Env binds the library current at construction
        e = BatchedSo100Env(task, n, device=0, seed=0, flags=flags, param_ranges=ParamRanges.parse(PARAMS) if params else None)
        e.reset()
        e.stagger_episodes()
        for w in range(64):
            e.step(ring[w % 64])
        return e

    def timed(e, steps, k0):
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for k in range(steps):
            flush.zero_()
            ev[k][0].record()
            e.step(ring[(k0 + k) % 64])
            ev[k][1].record()
        torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in ev) / steps

    result = {"card": card(), "envs": n, "libs": {"a": os.path.basename(args.lib_a), "b": os.path.basename(args.lib_b)},
              "build_ids": {k: L.so100_build_id().decode() for k, L in libs.items()},
              "method": "decorrelated start (staggered episode clocks + 64 steps), L2 flushed between timed steps (256 MiB memset), "
                        "CUDA events per step; libraries alternated in rounds (order swapped every round); per round the mean "
                        "step time, reported as the median over rounds with min / max", "rounds": args.rounds, "configs": {}}
    for label, task, flags, params, steps in configs:
        envs = {k: fresh(L, task, flags, params) for k, L in libs.items()}
        for k, e in envs.items():  # warm-up of the timed shape
            timed(e, 10, 0)
        rounds = {"a": [], "b": []}
        for rnd in range(args.rounds):
            for k in (("a", "b") if rnd % 2 == 0 else ("b", "a")):
                rounds[k].append(timed(envs[k], steps, rnd * steps))
        run = {"timed_steps_per_round": steps, "kernel_variant": {k: e.kernel_variant for k, e in envs.items()}}
        for k, r in rounds.items():
            run[k] = {"median_ms": statistics.median(r), "min_ms": min(r), "max_ms": max(r), "rounds_ms": r}
        run["b_vs_a"] = run["b"]["median_ms"] / run["a"]["median_ms"] - 1
        # the same within each round (a and b back to back): the round-to-round drift cancels
        run["b_vs_a_per_round"] = [y / x - 1 for x, y in zip(rounds["a"], rounds["b"])]
        # spread: the larger relative half-width (max - min) / 2 / median of the two libraries' rounds
        run["spread"] = max((run[k]["max_ms"] - run[k]["min_ms"]) / 2 / run[k]["median_ms"] for k in ("a", "b"))
        result["configs"][label] = run
        print(f"{label:20s} a {run['a']['median_ms']:.4f} ms  b {run['b']['median_ms']:.4f} ms  b/a-1 {100 * run['b_vs_a']:+.2f} %"
              f"  spread +-{100 * run['spread']:.2f} %", flush=True)
        for e in envs.values():
            e.close()
    print(json.dumps(result, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
