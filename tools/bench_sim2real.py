"""Cost of actuator latency and joint-angle observation noise (so100_set_sim2real) on the env step.

Env01 and Env05 at 65 536 envs with bench.py's method: episode clocks staggered over the TimeLimit and 64 untimed steps
(a decorrelated start), L2 flushed between timed steps (256 MiB memset), every step bracketed by CUDA events.  The
configurations of one task share one process and are timed in alternating rounds, so that clock and neighbour drift
hits them alike:
  default  - nothing set: the default kernels;
  ranges   - typical param ranges only (the per-env kernels as tools/bench_params.py measured them);
  latency  - latency 0:16 only (every env redraws d at its resets inside the timed window);
  noise    - joint-angle noise only, std 0.01 rad (Env01 only: Env05 refuses noise);
  all      - ranges, latency 0:16 and noise together (Env05: ranges and latency).
The same again with SO100_FLAG_ARM_CONTACT.  The ranges-only case is set against profiles/r3_params_bench.json, which
measured the per-env kernels before they carried latency and noise.  The card's name, power limit and maximum SM clock
are read with a query-only nvidia-smi call and written beside the numbers.

    python tools/bench_sim2real.py --out profiles/r3_sim2real_bench.json
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_params import TYPICAL, card  # noqa: E402


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
        raise SystemExit("bench_sim2real.py measures the GPU: no CUDA device")
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    from so100_mujoco_rl_b200.randomization import ParamRanges, Sim2Real
    from so100_mujoco_rl_b200.tasks import FLAG_ARM_CONTACT

    n, dev = args.envs, torch.device("cuda", 0)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    g = torch.Generator(device=dev).manual_seed(1)
    ring = [torch.rand((n, 6), device=dev, generator=g) * 2 - 1 for _ in range(64)]
    ranges = ParamRanges.parse(TYPICAL)

    def configs(task):
        c = {"default": (None, None), "ranges": (ranges, None), "latency": (None, Sim2Real(latency=(0, 16)))}
        if task != 5:
            c["noise"] = (None, Sim2Real(obs_noise=0.01))
            c["all"] = (ranges, Sim2Real(latency=(0, 16), obs_noise=0.01))
        else:
            c["all"] = (ranges, Sim2Real(latency=(0, 16)))
        return c

    def fresh(task, flags, cfg):
        e = BatchedSo100Env(task, n, device=0, seed=0, flags=flags, param_ranges=cfg[0], sim2real=cfg[1])
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

    result = {"card": card(), "envs": n, "method": "decorrelated start (staggered episode clocks + 64 steps), L2 flushed "
              "between timed steps, CUDA events per step, configurations of a task alternated in rounds",
              "ranges": TYPICAL, "latency": [0, 16], "obs_noise": 0.01, "runs": {}}
    for task, tname in ((1, "Env01"), (5, "Env05")):
        for label, flags, steps in (("no_contact", 0, args.steps), ("arm_contact", FLAG_ARM_CONTACT, args.contact_steps)):
            cfgs = configs(task)
            envs = {name: fresh(task, flags, c) for name, c in cfgs.items()}
            times = {name: [] for name in cfgs}
            for rnd in range(args.rounds):
                for name, e in envs.items():
                    times[name] += timed(e, steps, rnd * steps)
            run = {}
            for name, t in times.items():
                t = sorted(t)
                run[name] = {"mean_ms": sum(t) / len(t), "median_ms": t[len(t) // 2], "p10_ms": t[len(t) // 10],
                             "p90_ms": t[9 * len(t) // 10], "steps": len(t), "kernel_variant": envs[name].kernel_variant}
            for name in run:
                if name != "default":
                    run[name]["median_vs_default"] = run[name]["median_ms"] / run["default"]["median_ms"] - 1
            result["runs"][f"{tname}_{label}"] = run
            for e in envs.values():
                e.close()
    ref_path = os.path.join(ROOT, "profiles", "r3_params_bench.json")
    if os.path.exists(ref_path):  # the per-env kernels before latency and noise, same method, Env01
        ref = json.load(open(ref_path))
        cmp = {}
        for label in ("no_contact", "arm_contact"):
            r = ref["runs"][label]
            now = result["runs"][f"Env01_{label}"]
            cmp[label] = {"r3_params_typical_vs_default": r["typical"]["median_vs_default"],
                          "now_ranges_vs_default": now["ranges"]["median_vs_default"],
                          "r3_params_typical_median_ms": r["typical"]["median_ms"], "now_ranges_median_ms": now["ranges"]["median_ms"],
                          "r3_params_default_median_ms": r["default"]["median_ms"], "now_default_median_ms": now["default"]["median_ms"]}
        result["ranges_only_vs_r3_params_bench"] = {"card_then": ref.get("card"), **cmp}
    print(json.dumps(result, indent=1))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)


if __name__ == "__main__":
    main()
