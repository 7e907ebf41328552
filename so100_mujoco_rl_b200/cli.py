"""Command surface of the reference's `main.py` for the batched backend:  `-a PPO [-m MODEL] train -e EnvXX`.

Reference: src/so100_mujoco_rl/main.py:241-284 (`cli` group with -a/--algorithm and -m/--model, sub-commands
train | test | record, each with -e/--environment).  Here `train` builds the batched simulator instead of `gym.make`:
  * `--trainer native` (default): the GPU-resident PPO of so100_mujoco_rl_b200/ppo.py (SB3-default hyper-parameters);
  * `--trainer sb3`: hands a `So100VecEnv` to stable_baselines3 exactly as main.py:56-64 does (needs SB3 installed).
`test` and `record` drive an interactive viewer / a video encoder in the reference (main.py:78-171); rendering is outside
the hot path, so they only evaluate the policy head-less and report returns.

    python -m so100_mujoco_rl_b200.cli -a PPO train -e Env01 --num-envs 4096 --total-timesteps 20000000
"""
from __future__ import annotations

import json
import os
import time

import click


@click.group()
@click.option("-a", "--algorithm", default="PPO", show_default=True, help="RL algorithm (main.py:242-249); the native trainer implements PPO")
@click.option("-m", "--model", "model_path", default=None, help="path of a saved policy to continue from / evaluate (main.py:250-256)")
@click.pass_context
def cli(ctx, algorithm, model_path):
    ctx.ensure_object(dict)
    ctx.obj["ALGORITHM_NAME"], ctx.obj["MODEL_PATH"] = algorithm, model_path


@cli.command()
@click.option("-e", "--environment", required=True, help="Env01 | Env02 | Env05 (or the -v1 ids)")
@click.option("--num-envs", default=4096, show_default=True)
@click.option("--device", default=0, show_default=True)
@click.option("--trainer", type=click.Choice(["native", "sb3"]), default="native", show_default=True)
@click.option("--total-timesteps", default=20_000_000, show_default=True)
@click.option("--n-steps", default=32, show_default=True)
@click.option("--seed", default=0, show_default=True)
@click.option("--out", default="models", show_default=True, help="output folder (reference: models/<Env>_<Algo>/)")
@click.option("--learner", "learner_kind", type=click.Choice(["fused", "torch"]), default="fused", show_default=True,
              help="fused = hand-written PPO kernels (include/so100_ppo.h); torch = the PyTorch reference learner")
@click.option("--eval-freq", default=2_000_000, show_default=True, help="samples between evaluations (main.py:221 uses 20000 for its single env)")
@click.option("--eval-envs", default=64, show_default=True, help="envs of the evaluation simulator (0 = no evaluation)")
@click.option("--eval-steps", default=0, show_default=True, help="env steps per evaluation (0 = the task's TimeLimit: one full episode per env)")
@click.option("--save-freq", default=4_000_000, show_default=True, help="samples between checkpoints (main.py:228 uses 40000 for its single env)")
@click.option("--tensorboard-log", default="logs", show_default=True, help="TensorBoard folder (main.py:30, :62); empty = off")
@click.option("--randomize", "randomize", default=None,
              help="per-env dynamics randomisation of the training simulator, redrawn at every episode reset, e.g. "
                   "'kp=0.7:1.3,damping=0.8:1.2,forcerange=0.8:1.0,frictionloss=0.5:2' (scales of the model's values); "
                   "evaluation stays on the model's dynamics")
@click.option("--latency", "latency", default=None,
              help="actuator latency of the training simulator in substeps (2 ms each), LO:HI, drawn per env at every "
                   "episode reset: a new servo target acts from that substep of the env step; evaluation stays exact")
@click.option("--obs-noise", "obs_noise", default=None, type=float,
              help="std (rad) of Gaussian noise on the observed joint angles of the training simulator (Env01/02/06); "
                   "evaluation stays exact")
@click.option("--use-sde", "use_sde", is_flag=True, default=False,
              help="generalized State-Dependent Exploration (SB3 use_sde): action noise h E from the policy's last hidden layer, "
                   "E redrawn per env once per rollout; smooth commands instead of per-step jitter")
@click.option("--sde-sample-freq", "sde_sample_freq", default=None, type=int,
              help="with --use-sde: redraw the exploration matrices every N rollout steps (SB3 sde_sample_freq; default -1 = once per rollout)")
@click.option("--log-std-init", "log_std_init", default=0.0, show_default=True, type=float,
              help="initial log_std of the policy (SB3 policy kwarg log_std_init); gSDE runs usually start lower, e.g. -2")
@click.pass_context
def train(ctx, environment, num_envs, device, trainer, total_timesteps, n_steps, seed, out, learner_kind, eval_freq, eval_envs,
          eval_steps, save_freq, tensorboard_log, randomize, latency, obs_noise, use_sde, sde_sample_freq, log_std_init):
    algo = ctx.obj["ALGORITHM_NAME"]
    if trainer != "sb3" and algo != "PPO":  # refuse before anything is created on disk
        raise click.UsageError("the native trainer implements PPO; use --trainer sb3 for other algorithms")
    if sde_sample_freq is not None and not use_sde:
        raise click.BadParameter("needs --use-sde", param_hint="--sde-sample-freq")
    if sde_sample_freq is None:
        sde_sample_freq = -1
    elif sde_sample_freq == 0 or sde_sample_freq < -1:
        raise click.BadParameter("must be a positive number of steps or -1 (once per rollout)", param_hint="--sde-sample-freq")
    ckpt = None
    if ctx.obj["MODEL_PATH"] and trainer != "sb3":  # a run resumes with the exploration it was trained with
        ckpt, saved_sde = _load_checkpoint(ctx.obj["MODEL_PATH"])
        if saved_sde != use_sde:
            raise click.UsageError(f"{ctx.obj['MODEL_PATH']} holds a {'gSDE' if saved_sde else 'plain Gaussian'} policy: "
                                   f"{'add' if saved_sde else 'drop'} --use-sde to continue it")
    ranges = None
    if randomize:
        from .randomization import ParamRanges
        try:
            ranges = ParamRanges.parse(randomize)
        except ValueError as e:
            raise click.BadParameter(str(e), param_hint="--randomize") from None
    sim2real = None
    if latency is not None or obs_noise is not None:
        from .randomization import Sim2Real
        from .tasks import task_id
        try:
            lat = Sim2Real.parse_latency(latency) if latency is not None else (0, 0)
        except ValueError as e:
            raise click.BadParameter(str(e), param_hint="--latency") from None
        try:
            sim2real = Sim2Real(latency=lat, obs_noise=obs_noise or 0.0)
            sim2real.validate(task=task_id(environment))
        except ValueError as e:
            raise click.BadParameter(str(e), param_hint="--obs-noise" if str(e).startswith("obs_noise") else "--latency") from None
    folder = os.path.join(out, f"{environment}_{algo}")
    os.makedirs(folder, exist_ok=True)
    if trainer == "sb3":
        import stable_baselines3  # noqa: F401  (as main.py:258-262 validates the algorithm name)
        from .vec_env import So100VecEnv
        env = So100VecEnv(environment, num_envs, device=device, seed=seed, param_ranges=ranges, sim2real=sim2real)
        cls = getattr(stable_baselines3, algo)
        kw = {}
        if use_sde:
            kw.update(use_sde=True, sde_sample_freq=sde_sample_freq)
        if log_std_init != 0.0:
            kw["policy_kwargs"] = dict(log_std_init=log_std_init)
        model = cls("MlpPolicy", env, device="cpu", n_steps=n_steps, verbose=1, **kw) if not ctx.obj["MODEL_PATH"] \
            else cls.load(ctx.obj["MODEL_PATH"], env=env, **kw)
        model.learn(total_timesteps=total_timesteps)
        model.save(os.path.join(folder, "final_model"))
        return
    import torch
    from .batched_env import BatchedSo100Env
    from .callbacks import TrainCallbacks
    from .ppo import PPO, FusedPPO, PPOConfig
    env = BatchedSo100Env(environment, num_envs, device=device, seed=seed, param_ranges=ranges, sim2real=sim2real)
    cfg = PPOConfig(n_steps=n_steps, seed=seed, use_sde=use_sde, sde_sample_freq=sde_sample_freq, log_std_init=log_std_init)
    learner = FusedPPO(env, cfg) if learner_kind == "fused" else PPO(env, cfg)
    if ctx.obj["MODEL_PATH"]:  # main.py:201-207: continue from a saved model (weights; a .pt also restores Adam and the counters)
        path = ctx.obj["MODEL_PATH"]
        full = ckpt.get("learner")
        if full is not None:
            learner.load_state_dict(full)
        else:
            learner.load_policy(_load_policy(path, env.obs_dim, env.device))
        # the simulator continues where the checkpoint left it (same episodes, same RNG tick) when it has the same shape;
        # otherwise the run restarts its envs under a different seed so that it does not replay the original draws
        es = ckpt.get("env")
        if es is not None and es.get("num_envs") == env.num_envs:
            env.set_state(es["state"]); env.tick = int(es["tick"])
            if es.get("params") is not None:  # the same per-env dynamics as when it was saved (and its ranges unless --randomize is given)
                if env.param_ranges is None:
                    from .randomization import ParamRanges
                    env.set_param_ranges(ParamRanges.from_dict(es["param_ranges"]))
                env.set_params(es["params"])
            if es.get("actuator") is not None:  # the same latencies and previous targets (and its config unless --latency / --obs-noise is given)
                if env.sim2real is None:
                    from .randomization import Sim2Real
                    env.set_sim2real(Sim2Real.from_dict(es["sim2real"]))
                env.set_actuator_state(es["actuator"])
            learner.obs = env.obs   # (stale by one step at most: refreshed by the first env.step of the next rollout)
        else:
            env.seed(seed + 1_000_003)
            learner.obs = env.reset() if learner_kind == "fused" else env.reset().clone()
    # main.py:211-232: EvalCallback(eval_freq=20000) + reward threshold 6000 + no-improvement stop, CheckpointCallback(40000)
    eval_env = BatchedSo100Env(environment, eval_envs, device=device, seed=seed + 1) if eval_envs > 0 else None
    eval_steps = eval_steps or env.max_episode_steps
    cb = TrainCallbacks(learner, folder, f"{environment}_{algo}", eval_env=eval_env, eval_freq=eval_freq, eval_steps=eval_steps,
                        save_freq=save_freq, tensorboard_dir=tensorboard_log or None)
    t0 = time.time()
    stats = learner.learn(total_timesteps, log_every=0, callback=cb, additional=bool(ctx.obj["MODEL_PATH"]))  # SB3 restarts its count per learn() call
    cb.save("final_model")
    cb.close()
    click.echo(json.dumps({"samples": stats.samples, "wall_s": time.time() - t0, "rollout_s": stats.rollout_s, "update_s": stats.update_s,
                           "best_eval": cb.best, "stopped": cb.stop_reason, "last": stats.history[-1] if stats.history else None}))


def _load_checkpoint(path):
    """(the .pt checkpoint or {} for a .zip, whether its policy is gSDE's): a gSDE policy's log_std is [64, 6]."""
    import torch
    from .callbacks import load_sb3_zip
    if path.endswith(".zip"):
        return {}, load_sb3_zip(path)["log_std"].dim() == 2
    ckpt = torch.load(path, map_location="cpu")
    return ckpt, ckpt["policy"]["log_std"].dim() == 2


def _load_policy(path, obs_dim, device):
    """A policy saved by this package (.pt) or a Stable-Baselines3 style archive (.zip, policy.pth inside); plain or gSDE,
    told apart by the shape of log_std."""
    import torch
    from .callbacks import load_sb3_zip
    from .ppo import MlpPolicy
    sd = load_sb3_zip(path) if path.endswith(".zip") else torch.load(path, map_location="cpu")["policy"]
    policy = MlpPolicy(obs_dim, 6, use_sde=sd["log_std"].dim() == 2)
    if path.endswith(".zip"):
        policy.load_state_dict_sb3(sd)
    else:
        policy.load_state_dict(sd)
    return policy.to(device)


def _evaluate(ctx, environment, num_envs, device, steps, video_dir=None):
    """Deterministic policy for `steps` steps; with `video_dir` env 0 is rasterised every step (render.py) into
    `<video_dir>/rec-<env>-step-0-to-step-<steps>.mp4`, the file name VecVideoRecorder gives it in the reference."""
    import torch
    from .batched_env import BatchedSo100Env
    from .ppo import MlpPolicy  # noqa: F401  (torch.load of a pickled policy needs the class importable)
    if not ctx.obj["MODEL_PATH"]:
        raise click.UsageError("-m/--model is required")
    env = BatchedSo100Env(environment, num_envs, device=device, seed=123)
    policy = _load_policy(ctx.obj["MODEL_PATH"], env.obs_dim, env.device)
    obs, total = env.reset(), torch.zeros(num_envs, device=env.device)
    sink = renderer = None
    if video_dir:
        from .render import SceneRenderer, VideoSink
        renderer = SceneRenderer(env.spec)
        sink = VideoSink(video_dir, f"rec-{environment}", 0, steps, renderer.w, renderer.h)
    with torch.no_grad():
        for t in range(steps):
            a, _, _ = policy.act(obs, deterministic=True)
            r = env.step(torch.clamp(a, -1, 1))
            obs = r.obs
            total += r.reward
            if sink is not None:
                st = env.get_state()
                sink.write(renderer.render(st["qpos"][:, 0].cpu().numpy(), st["block"][:3, 0].cpu().numpy(),
                                           text=f"{environment}  step {t + 1}  return {float(total[0]):.2f}"))
    out = {"env": environment, "steps": steps, "mean_return": float(total.mean()), "mean_step_reward": float(total.mean()) / steps}
    if sink is not None:
        sink.close()
        out["video"] = sink.path
    click.echo(json.dumps(out))


@cli.command()
@click.option("-e", "--environment", required=True)
@click.option("--num-envs", default=256, show_default=True)
@click.option("--device", default=0, show_default=True)
@click.option("--steps", default=3000, show_default=True)
@click.option("--video-dir", default=None, help="also rasterise env 0 into a video in this directory")
@click.pass_context
def test(ctx, environment, num_envs, device, steps, video_dir):
    """main.py:78-124 opens an interactive MuJoCo viewer and loops predict -> step; head-less here: the deterministic
    policy's mean return over --steps steps, optionally with the rasterised video of env 0."""
    _evaluate(ctx, environment, num_envs, device, steps, video_dir)


@cli.command()
@click.option("-e", "--environment", required=True)
@click.option("--num-envs", default=1, show_default=True)
@click.option("--device", default=0, show_default=True)
@click.option("--video-dir", default="recordings", show_default=True, help="RECORDING_DIR of the reference (main.py:30)")
@click.pass_context
def record(ctx, environment, num_envs, device, video_dir):
    """main.py:127-171: 3000 steps of the policy recorded to `recordings/rec-<env>-step-0-to-step-3000.mp4`, drawn by the
    head-less software rasteriser (render.py) instead of MuJoCo's GL renderer."""
    _evaluate(ctx, environment, num_envs, device, 3000, video_dir)


if __name__ == "__main__":
    cli(obj={})
