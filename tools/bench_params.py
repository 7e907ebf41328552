"""Cost of per-env dynamics randomisation (so100_set_param_ranges) on the env step.

Env01 at 65 536 envs with bench.py's method: episode clocks staggered over the TimeLimit and 64 untimed steps (a
decorrelated start), L2 flushed between timed steps (256 MiB memset), every step bracketed by CUDA events.  Three
configurations share one process and are timed in alternating rounds, so that clock and neighbour drift hits them alike:
  default  - no ranges: the default kernels;
  unit     - every range [1, 1]: the per-env kernels on the model's values (the pure kernel overhead);
  typical  - kp 0.7:1.3, damping 0.8:1.2, forcerange 0.8:1.0, frictionloss 0.5:2 (the values differ per env and are
             redrawn at the resets inside the timed window).
The same three again with SO100_FLAG_ARM_CONTACT.  The card's name, power limit and maximum SM clock are read with a
query-only nvidia-smi call and written beside the numbers.

    python tools/bench_params.py --out profiles/params_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

TYPICAL = "kp=0.7:1.3,damping=0.8:1.2,forcerange=0.8:1.0,frictionloss=0.5:2"


def card() -> dict:
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, sm = (x.strip() for x in out.split(","))
        return {"name": name, "power_limit": power, "sm_max_clock": sm}
    except Exception as e:  # noqa: BLE001
        return {"name": None, "why": f"{type(e).__name__}: {e}"[:120]}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--steps", type=int, default=100, help="timed steps per configuration and round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--contact-steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_params.py measures the GPU: no CUDA device")
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    from so100_mujoco_rl_b200.randomization import ParamRanges
    from so100_mujoco_rl_b200.tasks import FLAG_ARM_CONTACT

    n, dev = args.envs, torch.device("cuda", 0)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    g = torch.Generator(device=dev).manual_seed(1)
    ring = [torch.rand((n, 6), device=dev, generator=g) * 2 - 1 for _ in range(64)]
    configs = {"default": None, "unit": ParamRanges(), "typical": ParamRanges.parse(TYPICAL)}

    def fresh(flags, ranges):
        e = BatchedSo100Env(1, n, device=0, seed=0, flags=flags, param_ranges=ranges)
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
        return [a.elapsed_time(b) for a, b in ev]

    result = {"card": card(), "task": "Env01", "envs": n, "method": "decorrelated start (staggered episode clocks + 64 steps), "
              "L2 flushed between timed steps, CUDA events per step, configurations alternated in rounds", "runs": {}}
    for label, flags, steps in (("no_contact", 0, args.steps), ("arm_contact", FLAG_ARM_CONTACT, args.contact_steps)):
        envs = {name: fresh(flags, r) for name, r in configs.items()}
        times = {name: [] for name in configs}
        for rnd in range(args.rounds):
            for name, e in envs.items():
                times[name] += timed(e, steps, rnd * steps)
        run = {}
        for name, t in times.items():
            t = sorted(t)
            run[name] = {"mean_ms": sum(t) / len(t), "median_ms": t[len(t) // 2], "p10_ms": t[len(t) // 10], "p90_ms": t[9 * len(t) // 10],
                         "steps": len(t), "kernel_variant": envs[name].kernel_variant}
        for name in ("unit", "typical"):
            run[name]["median_vs_default"] = run[name]["median_ms"] / run["default"]["median_ms"] - 1
        result["runs"][label] = run
        for e in envs.values():
            e.close()
    print(json.dumps(result, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
