"""`So100VecEnv` — the drop-in seam: a Stable-Baselines3 `VecEnv` over the batched GPU simulator.

The reference builds ONE `gym.make(env)` and lets SB3 wrap it in a 1-env `DummyVecEnv`
(src/so100_mujoco_rl/main.py:56-64, :182-189).  SB3 also accepts any object implementing its `VecEnv` interface and
uses it as is; this class is that object for N environments stepped by one kernel launch.  Semantics reproduced:

  * `reset()` -> float32 [N, obs_dim];  `step_async(a)` / `step_wait()` -> (obs, rewards, dones, infos)
  * auto-reset (DummyVecEnv.step_wait): for a finished env the returned obs is the first obs of the next episode and
    `infos[i]["terminal_observation"]` the last one; `infos[i]["TimeLimit.truncated"] = truncated and not terminated`
    (gymnasium TimeLimit at 4000 / 6000 steps, src/so100_mujoco_rl/__init__.py:5-45)
  * `infos[i]["episode"] = {"r", "l", "t"}` as the reference's `Monitor(env)` wrapper adds (main.py:183)

If stable_baselines3 is importable the class derives from its `VecEnv` (isinstance checks pass); otherwise it is a
structurally identical stand-in, so the host logic is testable without SB3.
"""
from __future__ import annotations

import time
from typing import Any, Sequence

import numpy as np

from .model import load_model
from .spaces import action_space, observation_space
from .tasks import MAX_EPISODE_STEPS, OBS_DIM, task_id

try:  # pragma: no cover - SB3 is not installed in the build image
    from stable_baselines3.common.vec_env import VecEnv as _VecEnvBase  # type: ignore
except Exception:  # noqa: BLE001
    _VecEnvBase = object


class TorchBackend:
    """Host-buffer face of BatchedSo100Env for the adapter: numpy in, numpy out, pinned staging buffers."""

    def __init__(self, env_id, num_envs, device=0, seed=0, env_offset=0, flags=0, max_episode_steps=None, param_ranges=None,
                 sim2real=None):
        from .batched_env import BatchedSo100Env  # needs CUDA; imported lazily so that CPU-only tooling can import this module
        self.env = BatchedSo100Env(env_id, num_envs, device=device, seed=seed, env_offset=env_offset, flags=flags,
                                   max_episode_steps=max_episode_steps, param_ranges=param_ranges, sim2real=sim2real)
        self.host = self.env.alloc_host()
        self.np = {k: v.numpy() for k, v in self.host.items()}

    def reset_np(self) -> np.ndarray:
        self.env.reset_host(self.host)
        return self.np["obs"]

    def step_np(self, actions: np.ndarray):
        self.np["actions"][...] = actions
        self.env.step_host(self.host)
        h = self.np
        return (h["obs"], h["reward"], h["terminated"], h["truncated"], h["terminal_obs"], h["ep_return"], h["ep_len"])

    def seed(self, seed: int):
        self.env.seed(seed)

    def close(self):
        self.env.close()


class So100VecEnv(_VecEnvBase):
    metadata = {"render_modes": ["human", "rgb_array", "depth_array"], "render_fps": 31}  # env_base_01.py:26-33

    def __init__(self, env_id: str | int, num_envs: int, device: int = 0, seed: int = 0, backend: Any = None,
                 clip_actions: bool = True, max_episode_steps: int | None = None, param_ranges=None, sim2real=None):
        self.task = task_id(env_id)
        self.env_id = env_id
        spec = load_model()
        obs_space, act_space = observation_space(self.task, spec), action_space()
        self.render_mode = None
        if _VecEnvBase is not object:  # pragma: no cover
            super().__init__(num_envs, obs_space, act_space)
        else:
            self.num_envs = int(num_envs)
            self.observation_space = obs_space
            self.action_space = act_space
            self.reset_infos = [{} for _ in range(num_envs)]
            self._seeds = [None for _ in range(num_envs)]
            self._options = [{} for _ in range(num_envs)]
        self.max_episode_steps = int(max_episode_steps or MAX_EPISODE_STEPS[self.task])
        self.clip_actions = clip_actions
        self._backend = backend if backend is not None else TorchBackend(
            env_id, num_envs, device=device, seed=seed, max_episode_steps=self.max_episode_steps, param_ranges=param_ranges,
            sim2real=sim2real)
        self._actions = None
        self._t0 = time.time()
        self.obs_dim = OBS_DIM[self.task]

    # ---- VecEnv core
    def reset(self) -> np.ndarray:
        obs = self._backend.reset_np()
        self.reset_infos = [{} for _ in range(self.num_envs)]
        self._seeds = [None for _ in range(self.num_envs)]
        self._options = [{} for _ in range(self.num_envs)]
        return np.array(obs, dtype=np.float32, copy=True)

    def step_async(self, actions: np.ndarray) -> None:
        a = np.asarray(actions, dtype=np.float32).reshape(self.num_envs, 6)
        if self.clip_actions:  # SB3 clips Box actions before calling; repeat for other callers
            a = np.clip(a, -1.0, 1.0)
        self._actions = a

    def step_wait(self):
        if self._actions is None:
            raise RuntimeError("step_wait() called without step_async()")
        obs, rew, term, trunc, tobs, ep_ret, ep_len = self._backend.step_np(self._actions)
        self._actions = None
        dones = (term != 0) | (trunc != 0)
        infos: list[dict] = [{} for _ in range(self.num_envs)]
        if dones.any():
            now = round(time.time() - self._t0, 6)
            for i in np.flatnonzero(dones):
                infos[i] = {
                    "terminal_observation": np.array(tobs[i], dtype=np.float32, copy=True),
                    "TimeLimit.truncated": bool(trunc[i]) and not bool(term[i]),
                    "episode": {"r": float(ep_ret[i]), "l": int(ep_len[i]), "t": now},
                }
        return (np.array(obs, dtype=np.float32, copy=True), np.array(rew, dtype=np.float32, copy=True),
                np.array(dones, dtype=bool, copy=True), infos)

    def step(self, actions: np.ndarray):
        self.step_async(actions)
        return self.step_wait()

    def close(self) -> None:
        if self._backend is not None:
            self._backend.close()
            self._backend = None

    # ---- the rest of the VecEnv contract
    def _indices(self, indices) -> Sequence[int]:
        if indices is None:
            return range(self.num_envs)
        if isinstance(indices, int):
            return [indices]
        return indices

    def get_attr(self, attr_name: str, indices=None) -> list:
        val = getattr(self, attr_name)
        return [val for _ in self._indices(indices)]

    def set_attr(self, attr_name: str, value: Any, indices=None) -> None:
        setattr(self, attr_name, value)

    def env_method(self, method_name: str, *method_args, indices=None, **method_kwargs) -> list:
        raise NotImplementedError(f"env_method({method_name!r}): the batched simulator has no per-env Python objects")

    def env_is_wrapped(self, wrapper_class, indices=None) -> list:
        return [False for _ in self._indices(indices)]

    def seed(self, seed: int | None = None):
        """SB3 semantics: env i gets seed + i at its next reset.  Here the device RNG is counter-based and keyed by
        (seed, global env id, tick), so one re-keying serves every env with its own stream."""
        self._seeds = [None if seed is None else seed + i for i in range(self.num_envs)]
        if seed is not None and hasattr(self._backend, "seed"):
            self._backend.seed(int(seed))
        return list(self._seeds)

    def set_options(self, options=None) -> None:
        self._options = [options or {} for _ in range(self.num_envs)]

    def get_images(self):
        return [None for _ in range(self.num_envs)]

    def render(self, mode: str | None = None):
        return None  # rendering is outside the hot path (SURVEY.md §8: out of scope)
