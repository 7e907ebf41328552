"""`BatchedSo100Env` — torch-tensor front end of the batched so100 simulator (one instance = one GPU, one task).

It mirrors the reference env's surface for N environments at once
(src/so100_mujoco_rl/envs/env01_v1.py:15-63, env02_v1.py:18-81, env03_v1.py:124-215, env05_v1.py:32-75):
`reset()` -> obs, `step(actions)` -> (obs, reward, terminated, truncated), with SB3 VecEnv auto-reset semantics
(finished envs return the first observation of their next episode; the last observation of the finished episode
is in `terminal_obs`).  All tensors live on the env's CUDA device; the work is enqueued on torch's current stream
through the C ABI (include/so100_b200.h).  PyTorch is only the owner of device memory and streams here.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass

import numpy as np
import torch

from . import _native
from .model import ModelSpec, load_model
from .randomization import ACTUATOR_NAMES, PARAM_NAMES, ParamRanges, Sim2Real, So100ActuatorView, So100ParamView
from .tasks import MAX_EPISODE_STEPS, OBS_DIM, make_task_cfg, task_id

NJ = 6


@dataclass
class StepResult:
    obs: torch.Tensor           # [N, obs_dim] f32 (first obs of the next episode where done)
    reward: torch.Tensor        # [N] f32
    terminated: torch.Tensor    # [N] u8
    truncated: torch.Tensor     # [N] u8  (TimeLimit.truncated: truncated and not terminated)
    terminal_obs: torch.Tensor  # [N, obs_dim] f32, rows valid where terminated|truncated
    ep_return: torch.Tensor     # [N] f32, valid where done
    ep_len: torch.Tensor        # [N] i32, valid where done


class HostBuffers(dict):
    """Page-locked host arrays of one env batch (`BatchedSo100Env.alloc_host`).  Their addresses are cached: the ctypes
    call is on the per-step path of the host-side caller."""
    _ORDER = ("actions", "obs", "reward", "terminated", "truncated", "terminal_obs", "ep_return", "ep_len")

    def ptrs(self, with_terminal: bool = True) -> tuple:
        key = "_p1" if with_terminal else "_p0"
        p = self.__dict__.get(key)
        if p is None:
            p = tuple(self[k].data_ptr() if (with_terminal or i < 5) else None for i, k in enumerate(self._ORDER))
            self.__dict__[key] = p
        return p


def _host_ptrs(host: dict, with_terminal: bool) -> tuple:
    if isinstance(host, HostBuffers):
        return host.ptrs(with_terminal)
    return tuple(host[k].data_ptr() if (with_terminal or i < 5) else None for i, k in enumerate(HostBuffers._ORDER))


class BatchedSo100Env:
    def __init__(self, env: str | int, num_envs: int, device: int | str | torch.device = 0, seed: int = 0,
                 env_offset: int = 0, flags: int = 0, model: ModelSpec | None = None,
                 max_episode_steps: int | None = None, param_ranges: ParamRanges | None = None,
                 sim2real: Sim2Real | None = None):
        self.task = task_id(env)
        self.num_envs = int(num_envs)
        self.obs_dim = OBS_DIM[self.task]
        self.act_dim = NJ
        self.max_episode_steps = int(max_episode_steps or MAX_EPISODE_STEPS[self.task])
        self.spec = model or load_model()
        dev = torch.device(device if not isinstance(device, int) else f"cuda:{device}")
        if dev.type != "cuda":
            raise ValueError("BatchedSo100Env runs on CUDA devices only (there is no CPU path)")
        if not torch.cuda.is_available():
            raise RuntimeError("CUDA is not available: BatchedSo100Env has no CPU fallback")
        self.device = torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())
        self._L = _native.lib()
        self._model_ct = self.spec.to_ctypes()
        self._cfg_ct = make_task_cfg(self.task, self.num_envs, seed=seed, env_offset=env_offset, flags=flags,
                                     max_episode_steps=self.max_episode_steps)
        h = ctypes.c_void_p()
        _native.check(self._L.so100_create(ctypes.byref(self._model_ct), ctypes.byref(self._cfg_ct),
                                           self.device.index, ctypes.byref(h)))
        self._h = h
        self._any_group = ctypes.c_int(-1)
        n, od = self.num_envs, self.obs_dim
        f32 = dict(dtype=torch.float32, device=self.device)
        self.obs = torch.zeros((n, od), **f32)
        self.reward = torch.zeros(n, **f32)
        self.terminated = torch.zeros(n, dtype=torch.uint8, device=self.device)
        self.truncated = torch.zeros(n, dtype=torch.uint8, device=self.device)
        self.terminal_obs = torch.zeros((n, od), **f32)
        self.ep_return = torch.zeros(n, **f32)
        self.ep_len = torch.zeros(n, dtype=torch.int32, device=self.device)
        self.param_ranges: ParamRanges | None = None
        if param_ranges is not None:
            self.set_param_ranges(param_ranges)
        self.sim2real: Sim2Real | None = None
        if sim2real is not None:
            self.set_sim2real(sim2real)

    # ---- lifecycle
    def close(self):
        if getattr(self, "_h", None):
            self._L.so100_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    # ---- env API
    def reset(self, mask: torch.Tensor | None = None) -> torch.Tensor:
        mp = None
        if mask is not None:
            mask = mask.to(device=self.device, dtype=torch.uint8).contiguous()
            if mask.numel() != self.num_envs:
                raise ValueError("mask must have num_envs elements")
            mp = mask.data_ptr()
        _native.check(self._L.so100_reset(self._h, mp, self.obs.data_ptr(), self._stream()))
        return self.obs

    def step(self, actions: torch.Tensor) -> StepResult:
        if actions.device != self.device or actions.dtype != torch.float32:
            actions = actions.to(device=self.device, dtype=torch.float32)
        actions = actions.contiguous()
        if actions.shape != (self.num_envs, NJ):
            raise ValueError(f"actions must have shape ({self.num_envs}, {NJ})")
        _native.check(self._L.so100_step(
            self._h, actions.data_ptr(), self.obs.data_ptr(), self.reward.data_ptr(), self.terminated.data_ptr(),
            self.truncated.data_ptr(), self.terminal_obs.data_ptr(), self.ep_return.data_ptr(), self.ep_len.data_ptr(),
            self._stream()))
        return StepResult(self.obs, self.reward, self.terminated, self.truncated, self.terminal_obs, self.ep_return,
                          self.ep_len)

    def step_substeps(self, ctrl: torch.Tensor, n_substeps: int = 1) -> None:
        """Debug / parity triage: n x mj_step under absolute servo targets ctrl [N, 6]; no task logic (see the header)."""
        ctrl = ctrl.to(device=self.device, dtype=torch.float32).contiguous()
        if ctrl.shape != (self.num_envs, NJ):
            raise ValueError(f"ctrl must have shape ({self.num_envs}, {NJ})")
        _native.check(self._L.so100_step_substeps(self._h, ctrl.data_ptr(), int(n_substeps), self._stream()))

    # ---- host-buffer path (the reference-facing call: numpy in / numpy out, copies inside the library)
    def alloc_host(self) -> "HostBuffers":
        n, od = self.num_envs, self.obs_dim
        pin = dict(pin_memory=True)
        return HostBuffers({
            "actions": torch.zeros((n, NJ), dtype=torch.float32, **pin),
            "obs": torch.zeros((n, od), dtype=torch.float32, **pin),
            "reward": torch.zeros(n, dtype=torch.float32, **pin),
            "terminated": torch.zeros(n, dtype=torch.uint8, **pin),
            "truncated": torch.zeros(n, dtype=torch.uint8, **pin),
            "terminal_obs": torch.zeros((n, od), dtype=torch.float32, **pin),
            "ep_return": torch.zeros(n, dtype=torch.float32, **pin),
            "ep_len": torch.zeros(n, dtype=torch.int32, **pin),
        })

    def reset_host(self, host: dict) -> torch.Tensor:
        _native.check(self._L.so100_reset_host(self._h, host["obs"].data_ptr(), self._stream()))
        return host["obs"]

    def step_host(self, host: dict, with_terminal: bool = True, actions: torch.Tensor | None = None) -> dict:
        """actions are read from host['actions'] (or from `actions`, a host float32 [N, 6] tensor); results land in the
        other host buffers (synchronous).  With pinned buffers the kernel reads / writes them in place over the host link."""
        act = host["actions"] if actions is None else actions
        if act.device.type != "cpu" or act.dtype != torch.float32 or not act.is_contiguous() or act.shape != (self.num_envs, NJ):
            raise ValueError(f"host actions must be a contiguous CPU float32 tensor of shape ({self.num_envs}, {NJ})")
        p = _host_ptrs(host, with_terminal)
        _native.check(self._L.so100_step_host(self._h, act.data_ptr(), p[1], p[2], p[3], p[4], p[5], p[6], p[7], self._stream()))
        return host

    def stagger_episodes(self, seed: int = 0) -> None:
        """Spread the envs' episode clocks uniformly over [0, max_episode_steps) (a scrambled assignment, so every CTA of
        envs sees the same mix): TimeLimit truncations and the in-kernel resets then arrive at a steady rate of
        num_envs / max_episode_steps per step instead of all at once.  Env05's retarget clock is kept consistent."""
        st = self.get_state()
        i = torch.arange(self.num_envs, device=self.device, dtype=torch.int64)
        el = ((i * 2654435761 + seed * 40503) % self.max_episode_steps).to(torch.int32)
        st["counters"][0] = el
        st["counters"][3] = el
        self.set_state({"counters": st["counters"]})

    # ---- pipelined host path: env groups stepped asynchronously (include/so100_b200.h, so100_step_host_async)
    def host_groups(self, n_groups: int) -> list[tuple[int, int]]:
        """Split the envs into n_groups contiguous ranges; returns their (lo, hi) env indices."""
        _native.check(self._L.so100_host_groups(self._h, int(n_groups)))
        out = []
        for g in range(int(n_groups)):
            lo, hi = ctypes.c_int(0), ctypes.c_int(0)
            _native.check(self._L.so100_host_group_range(self._h, g, ctypes.byref(lo), ctypes.byref(hi)))
            out.append((int(lo.value), int(hi.value)))
        return out

    def step_host_async(self, host: dict, group: int, with_terminal: bool = True, actions: torch.Tensor | None = None,
                        stream: int | None = None) -> None:
        """Enqueue one step of env group `group`: its rows of host['actions'] (or of `actions`, a pinned [N, 6] float32
        tensor) in, its rows of the other (pinned) host buffers out; returns immediately.  `step_host_wait(group)` blocks
        until those rows have landed.  `stream` (a cudaStream_t as int) saves the lookup of torch's current stream."""
        p = _host_ptrs(host, with_terminal)
        rc = self._L.so100_step_host_async(self._h, group, p[0] if actions is None else actions.data_ptr(), p[1], p[2], p[3], p[4],
                                           p[5], p[6], p[7], self._stream() if stream is None else stream)
        if rc < 0:
            _native.check(rc)

    def step_host_wait(self, group: int) -> None:
        rc = self._L.so100_step_host_wait(self._h, group)
        if rc < 0:
            _native.check(rc)

    def step_host_wait_any(self) -> int:
        """Block until any group with a step in flight has finished; returns its index (-1 if nothing is in flight)."""
        g = self._any_group
        rc = self._L.so100_step_host_wait_any(self._h, ctypes.byref(g))
        if rc < 0:
            _native.check(rc)
        return g.value

    # ---- state access (parity tests, checkpoints)
    _STATE_FIELDS = {"qpos": (6, torch.float32), "qvel": (6, torch.float32), "qacc_warm": (6, torch.float32), "qpos_comp": (6, torch.float32),
                     "block": (4, torch.float32), "snap": (12, torch.float32), "aux": (24, torch.float32),
                     "counters": (4, torch.int32), "ep_return": (1, torch.float32)}

    def get_state(self) -> dict:
        """Structure-of-arrays copies: field[k, env]."""
        out, view = {}, _native.StateView()
        for name, (k, dt) in self._STATE_FIELDS.items():
            out[name] = torch.zeros((k, self.num_envs), dtype=dt, device=self.device)
            setattr(view, name, out[name].data_ptr())
        _native.check(self._L.so100_get_state(self._h, ctypes.byref(view), self._stream()))
        return out

    def set_state(self, state: dict):
        view, keep = _native.StateView(), []
        for name, t in state.items():
            k, dt = self._STATE_FIELDS[name]
            t = t.to(device=self.device, dtype=dt).reshape(k, self.num_envs).contiguous()
            keep.append(t)
            setattr(view, name, t.data_ptr())
        _native.check(self._L.so100_set_state(self._h, ctypes.byref(view), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    # ---- per-env dynamics randomisation (randomization.py; include/so100_b200.h, so100_set_param_ranges)
    def set_param_ranges(self, ranges: ParamRanges | None) -> None:
        """Redraw kp, kv, forcerange and friction loss of every env at each of its episode resets from these scale ranges;
        None switches back to the model's constants.  The first call starts every env from the model's values; a later
        change of ranges applies from each env's next reset."""
        if ranges is None:
            _native.check(self._L.so100_set_param_ranges(self._h, None))
        else:
            r = ranges.to_ctypes()
            _native.check(self._L.so100_set_param_ranges(self._h, ctypes.byref(r)))
        self.param_ranges = ranges

    def get_params(self) -> dict:
        """Every env's current values: {kp, kv, force_lo, force_hi, frictionloss} -> float32 [6, N] copies."""
        out = {k: torch.zeros((NJ, self.num_envs), dtype=torch.float32, device=self.device) for k in PARAM_NAMES}
        view = So100ParamView(*(out[k].data_ptr() for k in PARAM_NAMES))
        _native.check(self._L.so100_get_env_params(self._h, ctypes.byref(view), self._stream()))
        return out

    def set_params(self, params: dict) -> None:
        """Overwrite some or all of the per-env values ([6, N] each); they hold until each env's next reset."""
        view, keep = So100ParamView(), []
        for name, t in params.items():
            if name not in PARAM_NAMES:
                raise KeyError(f"unknown parameter {name!r}; expected one of {PARAM_NAMES}")
            t = t.to(device=self.device, dtype=torch.float32).reshape(NJ, self.num_envs).contiguous()
            keep.append(t)
            setattr(view, name, t.data_ptr())
        _native.check(self._L.so100_set_env_params(self._h, ctypes.byref(view), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    # ---- actuator latency and joint-angle observation noise (randomization.py; include/so100_b200.h, so100_set_sim2real)
    def set_sim2real(self, cfg: Sim2Real | None) -> None:
        """Draw every env's actuator latency from cfg.latency at each of its episode resets and add Gaussian noise of std
        cfg.obs_noise to the observed joint angles from the next step; None switches both off.  The first call starts
        every env at latency 0 with its current position as the previous servo target."""
        if cfg is None:
            _native.check(self._L.so100_set_sim2real(self._h, None))
        else:
            cfg.validate(nsubstep=self.spec.nsubstep, task=self.task)
            c = cfg.to_ctypes()
            _native.check(self._L.so100_set_sim2real(self._h, ctypes.byref(c)))
        self.sim2real = cfg

    def get_actuator_state(self) -> dict:
        """Every env's actuator state: {latency: int32 [N]} and, Env01/02/06, {ctrl_prev_hi, ctrl_prev_lo: float32 [6, N]}
        (the previous servo target; Env05's is aux[0:6] of the state)."""
        names = ACTUATOR_NAMES if self.task != 5 else ACTUATOR_NAMES[:1]
        out = {k: torch.zeros(self.num_envs if k == "latency" else (NJ, self.num_envs),
                              dtype=torch.int32 if k == "latency" else torch.float32, device=self.device) for k in names}
        view = So100ActuatorView(*(out[k].data_ptr() if k in out else None for k in ACTUATOR_NAMES))
        _native.check(self._L.so100_get_actuator_state(self._h, ctypes.byref(view), self._stream()))
        return out

    def set_actuator_state(self, state: dict) -> None:
        """Overwrite some or all of the actuator state; the values hold until each env's next reset."""
        view, keep = So100ActuatorView(), []
        for name, t in state.items():
            if name not in ACTUATOR_NAMES:
                raise KeyError(f"unknown actuator field {name!r}; expected one of {ACTUATOR_NAMES}")
            if name == "latency":
                t = t.to(device=self.device, dtype=torch.int32).reshape(self.num_envs).contiguous()
            else:
                t = t.to(device=self.device, dtype=torch.float32).reshape(NJ, self.num_envs).contiguous()
            keep.append(t)
            setattr(view, name, t.data_ptr())
        _native.check(self._L.so100_set_actuator_state(self._h, ctypes.byref(view), self._stream()))
        torch.cuda.current_stream(self.device).synchronize()

    @property
    def tick(self) -> int:
        t = ctypes.c_int64(0)
        _native.check(self._L.so100_get_tick(self._h, ctypes.byref(t)))
        return int(t.value)

    @tick.setter
    def tick(self, v: int):
        _native.check(self._L.so100_set_tick(self._h, int(v)))

    def seed(self, seed: int) -> None:
        """Re-key the device RNG (reset draws, Env02 relocations, Env05 targets and noise); the tick restarts at 0."""
        _native.check(self._L.so100_set_seed(self._h, int(seed) & 0xFFFFFFFFFFFFFFFF))
        self.tick = 0

    def derived(self):
        a, b, c = np.zeros(NJ), np.zeros(NJ), np.zeros(NJ)
        dp = lambda x: x.ctypes.data_as(ctypes.POINTER(ctypes.c_double))  # noqa: E731
        _native.check(self._L.so100_get_derived(self._h, dp(a), dp(b), dp(c)))
        return a, b, c

    @property
    def kernel_variant(self) -> str:
        return "specialised" if _native.check(self._L.so100_kernel_variant(self._h)) == 1 else "generic"

    def stats(self) -> dict:
        a, b, c = ctypes.c_int64(0), ctypes.c_int64(0), ctypes.c_int64(0)
        _native.check(self._L.so100_get_stats(self._h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
        return {"launches": int(a.value), "solver_unconverged": int(b.value), "nan_resets": int(c.value)}

    def forward_dynamics(self, qpos: torch.Tensor, qvel: torch.Tensor, ctrl: torch.Tensor):
        """Debug/parity entry: SoA [6, n] inputs -> M [21, n], bias [6, n], qacc [6, n], kin [18, n]."""
        n = qpos.shape[1]
        args = [x.to(device=self.device, dtype=torch.float32).contiguous() for x in (qpos, qvel, ctrl)]
        f32 = dict(dtype=torch.float32, device=self.device)
        M, bias, qacc, kin = (torch.zeros((k, n), **f32) for k in (21, 6, 6, 18))
        _native.check(self._L.so100_forward_dynamics(self._h, n, args[0].data_ptr(), args[1].data_ptr(),
                                                     args[2].data_ptr(), M.data_ptr(), bias.data_ptr(),
                                                     qacc.data_ptr(), kin.data_ptr(), self._stream()))
        return M, bias, qacc, kin
