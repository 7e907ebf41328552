#!/usr/bin/env python
"""Cost and effect of gSDE exploration (so100_ppo_sde_act / so100_ppo_sde_grad, DESIGN.md §7d).

Kernel times (CUDA events around `--launches` back-to-back launches, median over `--rounds` rounds; the plain and the gSDE
call alternate within every round, so clock and neighbour drift hit them alike; inputs are not flushed from L2, as in a
rollout, where the env step has just written the observations):
  act   - so100_ppo_act vs so100_ppo_sde_act at 65 536 and 262 144 envs, obs_dim 8 (Env05), stochastic, every output
          written; the tcgen05 kernel in this process, the mma.sync kernel (SO100_PPO_ACT_MMA=1, read once per process)
          in a child process run the same way;
  grad  - so100_ppo_grad vs so100_ppo_sde_grad on a minibatch of 262 144 of 2^21 samples (the trainer's geometry).
Learner (Env05, 65 536 envs, n_steps 32, SB3 defaults otherwise): FusedPPO rollout and update seconds per iteration, and
per seed (--seeds) SB3's default exploration against --use-sde --log-std-init -2: the mean step reward at fixed sample
counts and the mean |a_t - a_t-1| of the clipped rollout actions over consecutive steps of one episode.
The card's name, power limit and maximum SM clock are read with a query-only nvidia-smi call in the same run.

    python tools/bench_sde.py --out profiles/r3_sde_bench.json
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
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_params import card  # noqa: E402


def _policy_params(od, use_sde, dev):
    import torch

    from so100_mujoco_rl_b200.ppo import MlpPolicy, pack_params
    torch.manual_seed(0)
    p = MlpPolicy(od, 6, log_std_init=-2.0 if use_sde else 0.0, use_sde=use_sde)
    with torch.no_grad():
        for t in p.parameters():
            t.add_(0.1 * torch.randn_like(t))
    return pack_params(p).to(dev)


def _timed(fn, launches):
    import torch
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(launches):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / launches


def act_times(sizes, od, rounds, launches):
    """{n: {"plain_ms", "sde_ms"}}: medians over rounds, plain and gSDE alternating."""
    import torch

    from so100_mujoco_rl_b200 import _native
    L, check = _native.lib(), _native.check
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    P = {False: _policy_params(od, False, dev), True: _policy_params(od, True, dev)}
    out = {}
    for n in sizes:
        obs = torch.randn(n, od, device=dev)
        bufs = [torch.empty(n, 6, device=dev), torch.empty(n, 6, device=dev), torch.empty(n, device=dev), torch.empty(n, device=dev),
                torch.empty(n, od, device=dev)]
        ptrs = [b.data_ptr() for b in bufs]
        key = [0]

        def call(sde):
            key[0] += 1
            fn = L.so100_ppo_sde_act if sde else L.so100_ppo_act
            check(fn(od, P[sde].data_ptr(), obs.data_ptr(), n, 1, 0, key[0], 0, *ptrs, st))
        for sde in (False, True):   # warm-up: module load, shared-memory opt-in
            for _ in range(5):
                call(sde)
        torch.cuda.synchronize()
        t = {False: [], True: []}
        for _ in range(rounds):
            for sde in (False, True):
                t[sde].append(_timed(lambda: call(sde), launches))
        out[str(n)] = {"plain_ms": statistics.median(t[False]), "sde_ms": statistics.median(t[True]),
                       "plain_rounds_ms": t[False], "sde_rounds_ms": t[True]}
    return out


def grad_times(od, S, mb, rounds, launches):
    import torch

    from so100_mujoco_rl_b200 import _native
    L, check = _native.lib(), _native.check
    dev = torch.device("cuda", 0)
    st = torch.cuda.current_stream().cuda_stream
    g = torch.Generator(device=dev).manual_seed(0)
    obs, act = torch.randn(S, od, device=dev, generator=g), torch.randn(S, 6, device=dev, generator=g) * 0.3
    logp, adv, ret = torch.randn(S, device=dev, generator=g) - 2.0, torch.randn(S, device=dev, generator=g), torch.randn(S, device=dev, generator=g)
    perm = torch.randperm(S, device=dev, generator=g)
    state = {}
    for sde in (False, True):
        P = _policy_params(od, sde, dev)
        wsf = L.so100_ppo_sde_workspace_floats if sde else L.so100_ppo_workspace_floats
        state[sde] = (P, torch.zeros(int(wsf(od)), device=dev), torch.zeros(P.numel(), device=dev), torch.zeros(3, device=dev))
    k = [0]

    def call(sde):
        P, ws, grad, loss = state[sde]
        j = k[0] % (S // mb)
        k[0] += 1
        idx = perm[j * mb:(j + 1) * mb]
        fn = L.so100_ppo_sde_grad if sde else L.so100_ppo_grad
        check(fn(od, P.data_ptr(), obs.data_ptr(), act.data_ptr(), logp.data_ptr(), adv.data_ptr(), ret.data_ptr(), idx.data_ptr(), mb, 0.2, 0.5,
                 0.0, 1, ws.data_ptr(), grad.data_ptr(), loss.data_ptr(), st))
    for sde in (False, True):
        for _ in range(3):
            call(sde)
    torch.cuda.synchronize()
    t = {False: [], True: []}
    for _ in range(rounds):
        for sde in (False, True):
            t[sde].append(_timed(lambda: call(sde), launches))
    return {"minibatch": mb, "samples": S, "plain_ms": statistics.median(t[False]), "sde_ms": statistics.median(t[True]),
            "plain_rounds_ms": t[False], "sde_rounds_ms": t[True]}


def learner_runs(envs, seeds, iters, report_every):
    """Env05 FusedPPO, SB3 defaults vs gSDE with log_std_init -2: timings and the effect on rewards and action changes."""
    import torch

    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    from so100_mujoco_rl_b200.ppo import FusedPPO, PPOConfig
    configs = {"default": dict(), "sde": dict(use_sde=True, log_std_init=-2.0)}
    out = {k: [] for k in configs}
    for seed in range(seeds):
        for name, kw in configs.items():   # the two configurations alternate seed by seed
            env = BatchedSo100Env(5, envs, device=0, seed=100 + seed)
            lr = FusedPPO(env, PPOConfig(n_steps=32, seed=seed, **kw))
            recs = []

            def cb(rec):
                b = lr.buf
                a = b["act"].clamp(-1.0, 1.0)
                same_ep = (1.0 - b["done"][:-1])[..., None]   # a_t and a_t+1 belong to one episode unless it ended at t
                dact = float(((a[1:] - a[:-1]).abs() * same_ep).sum() / (same_ep.sum() * 6))
                recs.append({"iter": rec["iter"], "samples": rec["samples"], "mean_step_reward": rec["mean_step_reward"],
                             "mean_abs_action_change": dact, "log_std_mean": rec["log_std_mean"],
                             "rollout_s": rec["rollout_s"], "update_s": rec["update_s"]})
            lr.learn(total_samples=iters * 32 * envs, log_every=0, callback=cb)
            env.close()
            timed = recs[2:]   # first iterations include module loads
            out[name].append({"seed": seed, "rollout_s_per_iter": statistics.median(r["rollout_s"] for r in timed),
                              "update_s_per_iter": statistics.median(r["update_s"] for r in timed),
                              "at": [r for r in recs if r["iter"] % report_every == 0 or r["iter"] == 1]})
            torch.cuda.synchronize()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--seeds", type=int, default=3)
    ap.add_argument("--iters", type=int, default=60, help="learner iterations per run (n_steps 32 x envs samples each)")
    ap.add_argument("--report-every", type=int, default=10)
    ap.add_argument("--act-only", action="store_true", help="child mode: print the act timings as JSON and exit")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    sizes, od = (65536, 262144), 8
    if args.act_only:
        print(json.dumps(act_times(sizes, od, args.rounds, args.launches)))
        return
    res = {"card": card(), "obs_dim": od}
    res["act_tc"] = act_times(sizes, od, args.rounds, args.launches)
    env = dict(os.environ, SO100_PPO_ACT_MMA="1")
    child = subprocess.run([sys.executable, os.path.abspath(__file__), "--act-only", "--rounds", str(args.rounds), "--launches", str(args.launches)],
                           env=env, capture_output=True, text=True, check=True, timeout=1800)
    res["act_mma"] = json.loads(child.stdout.strip().splitlines()[-1])
    res["grad"] = grad_times(od, 2 ** 21, 2 ** 18, args.rounds, max(5, args.launches // 5))
    res["learner_env05"] = learner_runs(args.envs, args.seeds, args.iters, args.report_every)
    res["card_after"] = card()
    txt = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")
    summary = {k: {n: (v["plain_ms"], v["sde_ms"]) for n, v in res[k].items()} for k in ("act_tc", "act_mma")}
    summary["grad"] = (res["grad"]["plain_ms"], res["grad"]["sde_ms"])
    for name, runs in res["learner_env05"].items():
        summary[name] = [(r["rollout_s_per_iter"], r["update_s_per_iter"], r["at"][-1]["mean_step_reward"], r["at"][-1]["mean_abs_action_change"])
                         for r in runs]
    print(json.dumps({"card": res["card"], **summary}))


if __name__ == "__main__":
    main()
