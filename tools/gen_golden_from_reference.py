#!/usr/bin/env python
"""Generates tests/golden/ref_env0{1,2,5,6}.npz by running the REFERENCE'S OWN Python task logic, unmodified, and
tests/golden/ref_mjcf.npz, the reference's scene as the MJCF reader parses it.

Runs only in the build container (it imports from /root/reference); the fixtures travel, this script's inputs do not.

What is real and what is stubbed
  * REAL: the reference's env classes — So100BaseEnv (envs/env_base_01.py), Env01 (env01_v1.py), Env02 (env02_v1.py),
    Env03/Env05 (env03_v1.py, env05_v1.py), Env06 (env06_v1.py, env_base_06.py), So100OffscreenBaseEnv's projection (env_base_02.py:85-127) and utils.py —
    imported from /root/reference/src and executed as they are: reward, observation, reset, block scripting,
    re-projection, lost-cube termination.
  * STUBBED (not installable offline): `mujoco`, `gymnasium`, `ultralytics`, `glfw`.  The stub `mujoco.mj_step`
    advances the arm with the repo's fp64 oracle physics (n-1 substeps, kinematics, 1 substep: so xpos/xmat are one
    substep stale exactly as MuJoCo leaves them) and the free block along z with the oracle's floor-contact restatement;
    `mj_resetData` zero-fills like MuJoCo; `MujocoEnv.reset` is
    gymnasium's (`mj_resetData` + `reset_model`); TimeLimit / auto-reset follow gymnasium + SB3 DummyVecEnv.
    => these fixtures pin the TASK LOGIC (the part the reference itself owns); the physics stays "parity unpinned".
  * RNG: the reference draws from the global np.random; here np.random.uniform / randint are patched to serve the
    repo's counter-based Philox draws in the reference's own call order (incl. the discarded theta of env01_v1.py:46),
    so the oracle and the kernels can replay the identical random numbers.
  * Env05 cannot be constructed in the reference without GL + YOLO weights, and env_base_02.py:89 uses an un-imported
    CAMERA_NAME (SURVEY Q15): the harness builds the object without So100OffscreenBaseEnv.__init__ and injects
    CAMERA_NAME = utils.CAMERA_NAME, i.e. the evident intent.
"""
from __future__ import annotations

import os
import sys
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF_SRC = "/root/reference/src"
sys.path.insert(0, ROOT)

from oracle.pyoracle import Oracle, philox  # noqa: E402
from so100_mujoco_rl_b200.model import BODY_NAMES, JOINT_NAMES, load_model, reference_scene_path  # noqa: E402
from so100_mujoco_rl_b200.tasks import FLAG_ARM_CONTACT, make_task_cfg  # noqa: E402

SPEC = load_model(reference_scene_path())
PHYS = Oracle(SPEC.to_ctypes(), make_task_cfg(1, 1, flags=FLAG_ARM_CONTACT))  # the reference's scene: pads collide with the floor
PREFIX = "so100_"

# ----------------------------------------------------------------------------------------------- RNG bridge
STREAM_RESET, STREAM_TASK, STREAM_NOISE, STREAM_API_RESET, STREAM_RESET_NOISE = 0, 1, 2, 3, 4


class RngBridge:
    def __init__(self):
        self.seed = self.env = self.tick = 0
        self.phase_stream = STREAM_API_RESET
        self.slots = {}

    def context(self, seed, env, tick, phase_stream):
        self.seed, self.env, self.tick, self.phase_stream = seed, env, tick, phase_stream
        self.slots = {}

    def _next(self, stream):
        k = self.slots.get(stream, 0)
        self.slots[stream] = k + 1
        assert k < 4, "more than 4 draws on one Philox block"
        return int(philox(self.seed, self.env, self.tick, stream)[k])

    def uniform(self, lo, hi):
        u = (self._next(self.phase_stream) >> 8) / 16777216.0
        return lo + (hi - lo) * u

    def randint(self, lo, hi):
        raw = self._next(self.phase_stream)
        return lo + ((raw * (hi - lo)) >> 32)


RNG = RngBridge()
np.random.uniform = RNG.uniform
np.random.randint = RNG.randint


# ----------------------------------------------------------------------------------------------- stub mujoco
class _Named:
    def __init__(self, **kw):
        self.__dict__.update(kw)


class _Actuator:
    def __init__(self, data, j):
        object.__setattr__(self, "_d", data)
        object.__setattr__(self, "_j", j)

    def __setattr__(self, k, v):
        assert k == "ctrl"
        self._d.ctrl[self._j] = float(v)

    @property
    def ctrl(self):
        return self._d.ctrl[self._j:self._j + 1]


class MjData:
    def __init__(self, model):
        self.model = model
        self.qpos = np.zeros(13); self.qvel = np.zeros(12); self.ctrl = np.zeros(6)
        self.qfrc_applied = np.zeros(12); self.warm = np.zeros(6)
        self.xpos = np.zeros((9, 3)); self.xmat = np.zeros((9, 9))
        self.cam_xpos = np.zeros((1, 3)); self.cam_xmat = np.zeros((1, 9))
        self.time = 0.0
        self.qpos[9] = 1.0  # free-joint quaternion of qpos0

    def joint(self, name):
        if name == "block_a_joint":
            return _Named(qpos=self.qpos[6:13], qvel=self.qvel[6:12], qfrc_applied=self.qfrc_applied[6:12])
        j = JOINT_NAMES.index(name[len(PREFIX):])
        return _Named(qpos=self.qpos[j:j + 1], qvel=self.qvel[j:j + 1], qfrc_applied=self.qfrc_applied[j:j + 1])

    def body(self, name):
        bid = 8 if name == "block_a" else 2 + BODY_NAMES.index(name[len(PREFIX):])
        return _Named(xpos=self.xpos[bid], xmat=self.xmat[bid], id=bid)

    def actuator(self, name):
        return _Actuator(self, JOINT_NAMES.index(name[len(PREFIX):]))

    def camera(self, name):
        assert name == "so100_end_point_camera"
        return _Named(xpos=self.cam_xpos[0], xmat=self.cam_xmat[0], id=0)


class MjModel:
    def __init__(self):
        self.njnt = 7
        self.jnt_range = np.vstack([SPEC.jnt_range, [[0.0, 0.0]]])
        self.opt = _Named(timestep=SPEC.timestep, gravity=np.array(SPEC.gravity))
        self.body_mass = np.array([0, 0, *SPEC.body_mass, 0.008])
        self.cam_fovy = np.array([SPEC.cam_fovy_deg])
        self.vis = _Named(global_=_Named(offwidth=640, offheight=480))

    @staticmethod
    def from_xml_path(path):
        assert path.endswith(("env01.xml", "env06.xml"))  # env06.xml is byte-identical to env01.xml
        return MjModel()

    def body(self, name):
        return _Named(id=8 if name == "block_a" else 2 + BODY_NAMES.index(name[len(PREFIX):]))

    def camera(self, name):
        return _Named(id=0)


def mj_id2name(model, objtype, i):
    return PREFIX + JOINT_NAMES[i] if i < 6 else "block_a_joint"


def mj_resetData(model, d):
    for a in (d.qpos, d.qvel, d.ctrl, d.qfrc_applied, d.warm, d.xpos, d.xmat, d.cam_xpos, d.cam_xmat):
        a[...] = 0.0
    d.qpos[9] = 1.0
    d.time = 0.0


def _kinematics(d):
    k = PHYS.fk(d.qpos[:6])
    d.xpos[2:8] = k["xpos"]; d.xmat[2:8] = k["xmat"]
    d.xpos[8] = d.qpos[6:9]
    d.xmat[8] = np.eye(3).ravel()
    d.cam_xpos[0] = k["cam_xpos"]; d.cam_xmat[0] = k["cam_xmat"]


def mj_step(model, d, nstep=1):
    """nstep x mj_step for this scene: arm = oracle physics; block = the oracle's free-box-on-a-plane restatement
    (gravity + qfrc_applied + soft floor contact along z; Env05 cancels gravity and zeroes the velocity itself)."""
    def advance(n):
        q, v, w = PHYS.substeps(d.qpos[:6], d.qvel[:6], d.warm, d.ctrl, n)
        d.qpos[:6], d.qvel[:6], d.warm[:] = q, v, w
        d.qpos[8], d.qvel[8] = PHYS.block_substeps(d.qpos[8], d.qvel[8], n, fz_applied=d.qfrc_applied[8])

    advance(nstep - 1)
    _kinematics(d)  # forward quantities of the LAST substep are computed before its integration
    advance(1)
    d.time += nstep * model.opt.timestep


def _install_stubs():
    mj = types.ModuleType("mujoco")
    mj.MjModel, mj.MjData = MjModel, MjData
    mj.mj_id2name, mj.mj_resetData, mj.mj_step = mj_id2name, mj_resetData, mj_step
    mj.mj_rnePostConstraint = lambda m, d: None
    mj.mjtObj = _Named(mjOBJ_JOINT=3)
    mj.mjtGridPos = _Named(mjGRID_TOPRIGHT=1)
    mj.mjtCamera = _Named(mjCAMERA_FIXED=2)
    mj.MjvCamera = lambda: _Named(type=0, fixedcamid=0)
    sys.modules["mujoco"] = mj

    class Box:
        def __init__(self, low, high, dtype=np.float32):
            self.low, self.high, self.dtype = np.asarray(low, dtype), np.asarray(high, dtype), dtype
            self.shape = self.low.shape

    class EzPickle:
        def __init__(self, *a, **k):
            pass

    class MujocoEnv:
        """gymnasium.envs.mujoco.MujocoEnv reduced to what the reference touches (gymnasium 1.1.1 semantics)."""

        def __init__(self, model_path, frame_skip, observation_space, default_camera_config=None, width=480,
                     height=480, render_mode=None, **kwargs):
            self.model = MjModel.from_xml_path(model_path)
            self.data = MjData(self.model)
            self.frame_skip, self.observation_space, self.render_mode = frame_skip, observation_space, render_mode
            self.mujoco_renderer = _Named(viewer=None)
            self._set_action_space()

        def reset(self, *, seed=None, options=None):
            mj_resetData(self.model, self.data)
            return self.reset_model(), {}

    g = types.ModuleType("gymnasium")
    g.utils = types.ModuleType("gymnasium.utils"); g.utils.EzPickle = EzPickle
    g.spaces = types.ModuleType("gymnasium.spaces"); g.spaces.Box = Box
    g.envs = types.ModuleType("gymnasium.envs")
    g.envs.mujoco = types.ModuleType("gymnasium.envs.mujoco"); g.envs.mujoco.MujocoEnv = MujocoEnv
    g.envs.mujoco.mujoco_rendering = types.ModuleType("gymnasium.envs.mujoco.mujoco_rendering")
    g.envs.mujoco.mujoco_rendering.OffScreenViewer = object
    g.envs.registration = types.ModuleType("gymnasium.envs.registration")
    for n in ("make", "pprint_registry", "register", "registry", "spec"):
        setattr(g.envs.registration, n, lambda *a, **k: None)
    for name, mod in (("gymnasium", g), ("gymnasium.utils", g.utils), ("gymnasium.spaces", g.spaces),
                      ("gymnasium.envs", g.envs), ("gymnasium.envs.mujoco", g.envs.mujoco),
                      ("gymnasium.envs.mujoco.mujoco_rendering", g.envs.mujoco.mujoco_rendering),
                      ("gymnasium.envs.registration", g.envs.registration)):
        sys.modules[name] = mod
    ul = types.ModuleType("ultralytics"); ul.YOLO = lambda *a, **k: None
    sys.modules["ultralytics"] = ul
    sys.modules["glfw"] = types.ModuleType("glfw")


def make_env(task):
    if task == 1:
        from so100_mujoco_rl.envs.env01_v1 import Env01
        return Env01()
    if task == 2:
        from so100_mujoco_rl.envs.env02_v1 import Env02
        return Env02()
    if task == 6:
        from so100_mujoco_rl.envs.env06_v1 import Env06
        return Env06()
    import so100_mujoco_rl.envs.env_base_02 as b2
    from so100_mujoco_rl.envs.env05_v1 import Env05
    from so100_mujoco_rl.envs.env_base_01 import So100BaseEnv
    from so100_mujoco_rl.envs.utils import CAMERA_NAME
    b2.CAMERA_NAME = CAMERA_NAME  # SURVEY Q15: used at env_base_02.py:89-90 but never imported there
    env = Env05.__new__(Env05)    # skip So100OffscreenBaseEnv.__init__ (GL viewer + YOLO weights)
    So100BaseEnv.__init__(env, "./model/env01.xml")
    env._set_initial_values()                                       # env_base_02.py:32
    env.offscreen_viewer = _Named(get_end_camera=lambda: _Named(fixedcamid=0))
    env.data.joint("block_a_joint").qpos[0:3] = env.block_target    # env_base_02.py:51
    inner = env._get_obs

    def get_obs_on_noise_stream():  # instrumentation only: draws made inside _get_obs come from the noise stream
        saved = RNG.phase_stream
        RNG.phase_stream = STREAM_NOISE if saved == STREAM_TASK else STREAM_RESET_NOISE
        try:
            return inner()
        finally:
            RNG.phase_stream = saved
    env._get_obs = get_obs_on_noise_stream
    return env


def rollout(task, n_envs, steps, seed, max_episode_steps, action_seed):
    envs = [make_env(task) for _ in range(n_envs)]
    od = 8 if task == 5 else 15
    rng = np.random.default_rng(action_seed)
    actions = rng.uniform(-1, 1, (steps, n_envs, 6)).astype(np.float32)
    if task == 5:
        actions[:, : n_envs // 2] *= 0.15  # gentle actions keep the cube in view; the others lose it and terminate
    obs0 = np.zeros((n_envs, od), np.float32)
    obs = np.zeros((steps, n_envs, od), np.float32); tobs = np.zeros_like(obs)
    rew = np.zeros((steps, n_envs)); term = np.zeros((steps, n_envs), np.uint8); trunc = np.zeros_like(term)
    elapsed = np.zeros(n_envs, int)
    for i, e in enumerate(envs):
        RNG.context(seed, i, 0, STREAM_API_RESET)
        obs0[i] = e.reset()[0]
    for t in range(steps):
        tick = t + 1
        for i, e in enumerate(envs):
            RNG.context(seed, i, tick, STREAM_TASK)
            ob, r, te, _, _ = e.step(actions[t, i].astype(np.float64))
            elapsed[i] += 1
            tr = elapsed[i] >= max_episode_steps            # gymnasium TimeLimit
            rew[t, i], term[t, i], trunc[t, i] = float(r), te, (tr and not te)
            if te or tr:                                    # SB3 DummyVecEnv.step_wait
                tobs[t, i] = ob
                RNG.context(seed, i, tick, STREAM_RESET)
                ob = e.reset()[0]
                elapsed[i] = 0
            obs[t, i] = ob
    return dict(actions=actions, obs0=obs0, obs=obs, terminal_obs=tobs, reward=rew, terminated=term, truncated=trunc,
                seed=np.int64(seed), max_episode_steps=np.int64(max_episode_steps), task=np.int64(task))


MJCF_FIELDS = ("body_pos", "body_quat", "body_ipos", "body_iquat", "body_mass", "body_inertia", "jnt_axis", "jnt_range",
               "jnt_armature", "jnt_frictionloss", "act_kp", "act_dampratio", "act_ctrlrange", "act_forcerange",
               "cam_pos", "cam_quat", "ee_offset", "gravity", "cam_fovy_deg", "timestep")


def main():
    _install_stubs()
    sys.path.insert(0, REF_SRC)
    out = os.path.join(ROOT, "tests", "golden")
    os.makedirs(out, exist_ok=True)
    # the reference's MJCF as load_model reads it: tests/test_model.py checks the committed mesh-free scene against it
    np.savez_compressed(os.path.join(out, "ref_mjcf.npz"), **{f: np.asarray(getattr(SPEC, f)) for f in MJCF_FIELDS})
    for task, n, steps, limit in ((1, 6, 90, 40), (2, 6, 90, 35), (5, 8, 140, 100), (6, 6, 90, 35)):
        d = rollout(task, n, steps, seed=1234 + task, max_episode_steps=limit, action_seed=task)
        path = os.path.join(out, f"ref_env0{task}.npz")
        np.savez_compressed(path, **d)
        print(f"Env0{task}: {n} envs x {steps} steps, {int(d['terminated'].sum())} terminations, "
              f"{int(d['truncated'].sum())} truncations, reward range [{d['reward'].min():.3f}, {d['reward'].max():.3f}] -> {path}")


if __name__ == "__main__":
    main()
