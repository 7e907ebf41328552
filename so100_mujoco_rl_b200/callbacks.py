"""Checkpoint / evaluation / early-stop / TensorBoard plumbing around the learners, mirroring the reference's `train`
(src/so100_mujoco_rl/main.py:211-238): `EvalCallback(eval_freq=20000, best_model_save_path=models/<Env>_<Algo>)` with
`StopTrainingOnRewardThreshold(6000)` on a new best and `StopTrainingOnNoModelImprovement(max_no_improvement_evals=5,
min_evals=10000)` after every evaluation, `CheckpointCallback(save_freq=40000, name_prefix=<Env>_<Algo>_cp_)`, and
`tensorboard_log="logs"` with SB3's scalar names.  Frequencies are in SAMPLES here (SB3 counts callback calls, i.e.
steps of its single env, so the numbers mean the same thing).

Policies are saved twice: `<name>.pt` (this package's own checkpoint) and `<name>.zip`, a Stable-Baselines3 style
archive holding `policy.pth` under SB3's ActorCriticPolicy parameter names, which
`stable_baselines3.PPO("MlpPolicy", env).set_parameters("<name>.zip", exact_match=False)` loads as is (SURVEY.md §8 f1).
"""
from __future__ import annotations

import io
import json
import os
import time
import zipfile

import torch

SB3_VERSION = "2.6.0"  # the reference's pin (pixi.lock:2674)


def export_sb3_zip(path: str, sb3_state_dict: dict, meta: dict | None = None) -> str:
    """SB3 `save_to_zip_file` layout: data (JSON), policy.pth, pytorch_variables.pth, _stable_baselines3_version."""
    def blob(obj) -> bytes:
        buf = io.BytesIO()
        torch.save(obj, buf)
        return buf.getvalue()

    path = path if path.endswith(".zip") else path + ".zip"
    with zipfile.ZipFile(path, "w") as z:
        z.writestr("data", json.dumps({"policy_class": "stable_baselines3.common.policies.ActorCriticPolicy",
                                       "net_arch": {"pi": [64, 64], "vf": [64, 64]}, "activation_fn": "Tanh", **(meta or {})}))
        z.writestr("policy.pth", blob({k: v.detach().cpu() for k, v in sb3_state_dict.items()}))
        z.writestr("pytorch_variables.pth", blob(None))
        z.writestr("_stable_baselines3_version", SB3_VERSION)
    return path


def load_sb3_zip(path: str) -> dict:
    with zipfile.ZipFile(path) as z:
        return torch.load(io.BytesIO(z.read("policy.pth")), map_location="cpu")


@torch.no_grad()
def evaluate_policy(policy, env, n_steps: int) -> dict:
    """Deterministic roll-out of `policy` (an MlpPolicy) on `env` (BatchedSo100Env-like) for n_steps env steps.
    The score (`mean_return`) is ONE quantity whatever the episode length: every env's reward accumulated over the fixed
    horizon, averaged over envs (episodes that end inside the horizon simply continue into their next episode).  With
    n_steps = the task's TimeLimit this is EvalCallback's mean episode reward for tasks that never terminate early."""
    obs = env.reset()
    total = torch.zeros(env.num_envs, device=obs.device)
    ers, cnt = 0.0, 0.0
    for _ in range(n_steps):
        a, _, _ = policy.act(obs, deterministic=True)
        r = env.step(torch.clamp(a, -1.0, 1.0))
        done = (r.terminated.bool() | r.truncated.bool()).float()
        total += r.reward
        ers += float((r.ep_return * done).sum()); cnt += float(done.sum())
        obs = r.obs
    mean_return = float(total.mean())
    return {"mean_return": mean_return, "mean_step_reward": mean_return / n_steps, "mean_ep_return": ers / cnt if cnt else None,
            "episodes": int(cnt)}


class TrainCallbacks:
    """Call once per learner iteration with the learner's record (`learn(callback=cb)`); returns nothing, sets
    `.stop` when a stop condition of main.py:211-216 fires (the caller's loop checks it)."""

    def __init__(self, learner, folder: str, prefix: str, eval_env=None, eval_freq: int = 20000, eval_steps: int = 256,
                 save_freq: int = 40000, reward_threshold: float = 6000.0, max_no_improvement_evals: int = 5,
                 min_evals: int = 10000, tensorboard_dir: str | None = "logs", verbose: bool = True):
        self.learner, self.folder, self.prefix, self.eval_env = learner, folder, prefix, eval_env
        self.eval_freq, self.eval_steps, self.save_freq = int(eval_freq), int(eval_steps), int(save_freq)
        self.reward_threshold, self.max_no_improvement_evals, self.min_evals = reward_threshold, max_no_improvement_evals, min_evals
        self.best, self.n_evals, self.no_improvement, self.stop, self.stop_reason = None, 0, 0, False, None
        self._next_eval, self._next_save, self._t0 = self.eval_freq, self.save_freq, time.time()
        self.verbose, self.evals, self.checkpoints = verbose, [], []
        os.makedirs(folder, exist_ok=True)
        self.tb = None
        if tensorboard_dir:
            try:
                from torch.utils.tensorboard import SummaryWriter
                self.tb = SummaryWriter(os.path.join(tensorboard_dir, prefix))
            except Exception:  # noqa: BLE001 - TensorBoard is optional
                self.tb = None

    def save(self, name: str) -> str:
        pol = self.learner.policy
        base = os.path.join(self.folder, name)
        ckpt = {"policy": pol.state_dict(), "samples": self.learner.stats.samples}
        if hasattr(self.learner, "state_dict"):  # optimizer moments and counters
            ckpt["learner"] = self.learner.state_dict()
        env = getattr(self.learner, "env", None)
        if env is not None and hasattr(env, "get_state") and hasattr(env, "tick"):  # simulator state: the resumed run continues the same episodes
            ckpt["env"] = {"state": {k: v.cpu() for k, v in env.get_state().items()}, "tick": env.tick, "num_envs": env.num_envs}
            ranges = getattr(env, "param_ranges", None)  # per-env dynamics (randomization.py): resumed with the same values
            ckpt["env"]["param_ranges"] = ranges.to_dict() if ranges is not None else None
            ckpt["env"]["params"] = {k: v.cpu() for k, v in env.get_params().items()} if ranges is not None else None
            s2r = getattr(env, "sim2real", None)  # actuator latency / observation noise: resumed with the same actuator state
            ckpt["env"]["sim2real"] = s2r.to_dict() if s2r is not None else None
            ckpt["env"]["actuator"] = {k: v.cpu() for k, v in env.get_actuator_state().items()} if s2r is not None else None
        torch.save(ckpt, base + ".pt")
        meta = {"num_timesteps": self.learner.stats.samples}
        cfg = getattr(self.learner, "cfg", None)
        if getattr(cfg, "use_sde", False):  # SB3 reads these from `data`; policy.pth holds the [64, 6] log_std
            meta.update(use_sde=True, sde_sample_freq=cfg.sde_sample_freq)
        export_sb3_zip(base + ".zip", pol.state_dict_sb3(), meta)
        return base

    def __call__(self, rec: dict) -> None:
        n = rec["samples"]
        if self.tb is not None:  # SB3's logger keys
            for key, val in (("rollout/ep_rew_mean", rec.get("ep_return_mean")), ("rollout/ep_len_mean", rec.get("ep_len_mean")),
                             ("rollout/mean_step_reward", rec.get("mean_step_reward")), ("train/policy_gradient_loss", rec.get("pg_loss")),
                             ("train/value_loss", rec.get("v_loss")), ("train/approx_kl", rec.get("approx_kl")),
                             ("train/log_std", rec.get("log_std_mean")), ("time/fps", n / max(time.time() - self._t0, 1e-9))):
                if val is not None:
                    self.tb.add_scalar(key, val, n)
        if self.save_freq and n >= self._next_save:  # CheckpointCallback
            self.checkpoints.append(self.save(f"{self.prefix}_cp__{n}_steps"))
            self._next_save += self.save_freq * max(1, (n - self._next_save) // self.save_freq + 1)
        if self.eval_env is not None and self.eval_freq and n >= self._next_eval:  # EvalCallback
            self._next_eval += self.eval_freq * max(1, (n - self._next_eval) // self.eval_freq + 1)
            ev = evaluate_policy(self.learner.policy, self.eval_env, self.eval_steps)
            score = ev["mean_return"]   # fixed-horizon return: the same quantity at every evaluation
            self.n_evals += 1
            self.evals.append({"samples": n, "score": score, **ev})
            if self.tb is not None:
                self.tb.add_scalar("eval/mean_reward", score, n)
            if self.best is None or score > self.best:
                self.best, self.no_improvement = score, 0
                self.save("best_model")
                if score >= self.reward_threshold:  # StopTrainingOnRewardThreshold (callback_on_new_best)
                    self.stop, self.stop_reason = True, f"mean reward {score:.2f} reached the threshold {self.reward_threshold}"
            else:
                self.no_improvement += 1
            # StopTrainingOnNoModelImprovement (callback_after_eval)
            if self.n_evals > self.min_evals and self.no_improvement > self.max_no_improvement_evals:
                self.stop, self.stop_reason = True, f"no improvement in {self.no_improvement} evaluations"
            if self.verbose:
                print(json.dumps({"eval": self.evals[-1], "best": self.best}), flush=True)
        if self.verbose and (rec["iter"] % 10 == 0 or rec["iter"] == 1):
            print(json.dumps(rec), flush=True)

    def close(self):
        if self.tb is not None:
            self.tb.close()
