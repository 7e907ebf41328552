"""ctypes binding of the CPU fp64 oracle (oracle/libso100_oracle.so).  TEST INFRASTRUCTURE ONLY.

Importable only from tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference legs.
The product package (so100_mujoco_rl_b200) never imports this module.
"""
from __future__ import annotations

import ctypes
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB_PATH = os.path.join(_HERE, "libso100_oracle.so")
NJ = 6


class OrcKin(ctypes.Structure):
    _fields_ = [
        ("xpos", (ctypes.c_double * 3) * NJ), ("xmat", (ctypes.c_double * 9) * NJ),
        ("xaxis", (ctypes.c_double * 3) * NJ), ("xipos", (ctypes.c_double * 3) * NJ),
        ("ximat", (ctypes.c_double * 9) * NJ),
        ("end_pos", ctypes.c_double * 3), ("wrist_pos", ctypes.c_double * 3),
        ("cam_xpos", ctypes.c_double * 3), ("cam_xmat", ctypes.c_double * 9),
    ]


class OrcEnvState(ctypes.Structure):
    _fields_ = [
        ("qpos", ctypes.c_double * NJ), ("qvel", ctypes.c_double * NJ), ("qacc_warm", ctypes.c_double * NJ),
        ("ctrl", ctypes.c_double * NJ), ("time", ctypes.c_double), ("block", ctypes.c_double * 3),
        ("block_vz", ctypes.c_double),
        ("end_pos", ctypes.c_double * 3), ("wrist_pos", ctypes.c_double * 3), ("block_xpos", ctypes.c_double * 3),
        ("cam_xpos", ctypes.c_double * 3), ("cam_xmat", ctypes.c_double * 9),
        ("task_block_pos", ctypes.c_double * 3), ("last_block_pos", ctypes.c_double * 3),
        ("cmd", ctypes.c_double * NJ), ("last_angvel", ctypes.c_double * NJ), ("target", ctypes.c_double * 3),
        ("target_dt", ctypes.c_double), ("target_time", ctypes.c_double), ("last_centre", ctypes.c_double * 2),
        ("elapsed_steps", ctypes.c_int32), ("ever_stepped", ctypes.c_int32), ("has_last_block", ctypes.c_int32),
        ("angvel_valid", ctypes.c_int32), ("centre_valid", ctypes.c_int32), ("miss_count", ctypes.c_int32),
        ("ep_return", ctypes.c_double),
    ]


def build(force: bool = False) -> str:
    src = os.path.join(_HERE, "so100_oracle.c")
    if force or not os.path.exists(_LIB_PATH) or os.path.getmtime(_LIB_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _LIB_PATH


_lib = None


def _native_build() -> str | None:
    """-O3 -march=native build for the TIMED CPU legs of bench.py (BASELINE.md §3), compiled on the machine it runs on
    (the portable oracle build that the tests use stays -O2 -ffp-contract=off so that the committed fixtures reproduce bit
    for bit).
    The library goes to a private directory under the temp directory, named after the host's CPU flags and the
    oracle's sources, so that the source tree is never written and may be read-only."""
    import hashlib
    import tempfile
    try:
        cpu = next(ln for ln in open("/proc/cpuinfo") if ln.startswith("flags"))
    except Exception:  # noqa: BLE001
        cpu = "unknown"
    src = os.path.join(_HERE, "so100_oracle.c")
    h = hashlib.sha1(cpu.encode())
    for f in (src, os.path.join(_HERE, "so100_oracle.h")):
        h.update(open(f, "rb").read())
    d = os.path.join(tempfile.gettempdir(), f"so100_oracle_{os.getuid()}")
    out = os.path.join(d, f"libso100_oracle_native_{h.hexdigest()[:12]}.so")
    try:
        os.makedirs(d, mode=0o700, exist_ok=True)
        if os.stat(d).st_uid != os.getuid():
            return None  # someone else's directory: do not load a library from it
        if not os.path.exists(out):
            tmp = f"{out}.{os.getpid()}"
            subprocess.check_call(["gcc", "-O3", "-march=native", "-pthread", "-fPIC", "-std=c11", "-D_GNU_SOURCE", "-shared",
                                   "-o", tmp, src, "-lm"], stderr=subprocess.DEVNULL)
            os.replace(tmp, out)  # atomic: a concurrent process never loads a half-written file
    except Exception:  # noqa: BLE001 - no compiler or no writable temp directory: time the portable build instead
        return None
    return out


def use_native_build() -> bool:
    """Switch this process to the -O3 -march=native oracle (call before the first Oracle is created)."""
    global _LIB_PATH, _lib
    p = _native_build()
    if p is None:
        return False
    _LIB_PATH, _lib = p, None
    return True


def lib():
    global _lib
    if _lib is None:
        if os.path.basename(_LIB_PATH) == "libso100_oracle.so":
            build()
        L = ctypes.CDLL(_LIB_PATH)
        dp, fp, u8p, i32p = (ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_float),
                             ctypes.POINTER(ctypes.c_uint8), ctypes.POINTER(ctypes.c_int32))
        L.orc_create.restype = ctypes.c_void_p
        L.orc_create.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
        L.orc_destroy.argtypes = [ctypes.c_void_p]
        L.orc_obs_dim.argtypes = [ctypes.c_void_p]
        L.orc_get_derived.argtypes = [ctypes.c_void_p, dp, dp, dp]
        L.orc_state.restype = ctypes.POINTER(OrcEnvState)
        L.orc_state.argtypes = [ctypes.c_void_p, ctypes.c_int]
        L.orc_get_tick.restype = ctypes.c_int64
        L.orc_get_tick.argtypes = [ctypes.c_void_p]
        L.orc_set_tick.argtypes = [ctypes.c_void_p, ctypes.c_int64]
        L.orc_fk.argtypes = [ctypes.c_void_p, dp, ctypes.POINTER(OrcKin)]
        L.orc_mass_matrix.argtypes = [ctypes.c_void_p, dp, dp]
        L.orc_bias.argtypes = [ctypes.c_void_p, dp, dp, dp]
        L.orc_contacts.argtypes = [ctypes.c_void_p, dp, dp, dp, i32p]
        L.orc_body_invweight0.argtypes = [ctypes.c_void_p, dp]
        L.orc_forward.argtypes = [ctypes.c_void_p, dp, dp, dp, dp, dp, dp, dp, i32p]
        L.orc_substeps.argtypes = [ctypes.c_void_p, dp, dp, dp, dp, ctypes.c_int]
        L.orc_energy.argtypes = [ctypes.c_void_p, dp, dp, dp, dp]
        L.orc_block_substeps.argtypes = [ctypes.c_void_p, dp, dp, ctypes.c_double, ctypes.c_int]
        L.orc_reset.argtypes = [ctypes.c_void_p, u8p, fp, ctypes.c_int]
        L.orc_step.argtypes = [ctypes.c_void_p, fp, fp, dp, u8p, u8p, fp, dp, i32p, ctypes.c_int]
        L.orc_set_state_soa.argtypes = [ctypes.c_void_p] + [ctypes.c_void_p] * 9
        L.orc_get_state_soa.argtypes = [ctypes.c_void_p, dp, dp, dp]
        L.orc_philox.argtypes = [ctypes.c_uint64, ctypes.c_uint32, ctypes.c_uint32, ctypes.c_uint32,
                                 ctypes.POINTER(ctypes.c_uint32)]
        L.orc_hw_threads.restype = ctypes.c_int
        _lib = L
    return _lib


def _d(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def philox(seed: int, env_id: int, tick: int, stream: int) -> np.ndarray:
    out = (ctypes.c_uint32 * 4)()
    lib().orc_philox(seed, env_id, tick, stream, out)
    return np.array(list(out), dtype=np.uint32)


class Oracle:
    """fp64 CPU restatement of the so100 hot path (physics building blocks + Env01/02/05 reset/step)."""

    def __init__(self, model_ct, cfg_ct):
        self._L = lib()
        assert self._L.orc_sizeof_model() == ctypes.sizeof(model_ct), "so100_model layout mismatch"
        assert self._L.orc_sizeof_task_cfg() == ctypes.sizeof(cfg_ct), "so100_task_cfg layout mismatch"
        assert self._L.orc_sizeof_env_state() == ctypes.sizeof(OrcEnvState), "orc_env_state layout mismatch"
        self._m, self._c = model_ct, cfg_ct
        self._h = self._L.orc_create(ctypes.byref(model_ct), ctypes.byref(cfg_ct))
        if not self._h:
            raise ValueError("orc_create rejected the model / task configuration")
        self.num_envs = int(cfg_ct.num_envs)
        self.obs_dim = int(self._L.orc_obs_dim(self._h))
        self.task = int(cfg_ct.task)

    def close(self):
        if self._h:
            self._L.orc_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- physics building blocks
    def derived(self):
        m0, kv, iw = np.zeros(NJ), np.zeros(NJ), np.zeros(NJ)
        self._L.orc_get_derived(self._h, _d(m0), _d(kv), _d(iw))
        return m0, kv, iw

    def fk(self, qpos) -> dict:
        q = np.ascontiguousarray(qpos, dtype=np.float64)
        k = OrcKin()
        self._L.orc_fk(self._h, _d(q), ctypes.byref(k))
        out = {}
        for name, _ in OrcKin._fields_:
            out[name] = np.array(getattr(k, name), dtype=np.float64)
        return out

    def mass_matrix(self, qpos) -> np.ndarray:
        q = np.ascontiguousarray(qpos, dtype=np.float64)
        M = np.zeros((NJ, NJ))
        self._L.orc_mass_matrix(self._h, _d(q), _d(M))
        return M

    def bias(self, qpos, qvel) -> np.ndarray:
        q = np.ascontiguousarray(qpos, dtype=np.float64)
        v = np.ascontiguousarray(qvel, dtype=np.float64)
        b = np.zeros(NJ)
        self._L.orc_bias(self._h, _d(q), _d(v), _d(b))
        return b

    def forward(self, qpos, qvel, ctrl, warm=None):
        q = np.ascontiguousarray(qpos, dtype=np.float64)
        v = np.ascontiguousarray(qvel, dtype=np.float64)
        c = np.ascontiguousarray(ctrl, dtype=np.float64)
        w = None if warm is None else np.ascontiguousarray(warm, dtype=np.float64)
        qacc, qs, qc = np.zeros(NJ), np.zeros(NJ), np.zeros(NJ)
        it = ctypes.c_int32(0)
        self._L.orc_forward(self._h, _d(q), _d(v), _d(c), None if w is None else _d(w), _d(qacc), _d(qs), _d(qc),
                            ctypes.byref(it))
        return qacc, qs, qc, int(it.value)

    def contacts(self, qpos):
        """Pad <-> floor contacts of one configuration: (pos [n, 3], dist [n], body [n])."""
        q = np.ascontiguousarray(qpos, dtype=np.float64)
        pos, dist, body = np.zeros((32, 3)), np.zeros(32), np.zeros(32, dtype=np.int32)
        n = self._L.orc_contacts(self._h, _d(q), _d(pos), _d(dist), body.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)))
        return pos[:n], dist[:n], body[:n]

    def body_invweight0(self) -> np.ndarray:
        t = np.zeros(NJ)
        self._L.orc_body_invweight0(self._h, _d(t))
        return t

    def substeps(self, qpos, qvel, warm, ctrl, n):
        q = np.array(qpos, dtype=np.float64)
        v = np.array(qvel, dtype=np.float64)
        w = np.array(warm, dtype=np.float64)
        c = np.ascontiguousarray(ctrl, dtype=np.float64)
        self._L.orc_substeps(self._h, _d(q), _d(v), _d(w), _d(c), int(n))
        return q, v, w

    def block_substeps(self, z: float, vz: float, n: int, fz_applied: float = 0.0):
        """n mj_step substeps of the free block's z coordinate (gravity + applied force + floor contact)."""
        zz, vv = ctypes.c_double(z), ctypes.c_double(vz)
        self._L.orc_block_substeps(self._h, ctypes.byref(zz), ctypes.byref(vv), float(fz_applied), int(n))
        return zz.value, vv.value

    def energy(self, qpos, qvel):
        q = np.ascontiguousarray(qpos, dtype=np.float64)
        v = np.ascontiguousarray(qvel, dtype=np.float64)
        T, V = ctypes.c_double(0), ctypes.c_double(0)
        self._L.orc_energy(self._h, _d(q), _d(v), ctypes.byref(T), ctypes.byref(V))
        return T.value, V.value

    # ---- env API
    @property
    def tick(self) -> int:
        return int(self._L.orc_get_tick(self._h))

    @tick.setter
    def tick(self, v: int):
        self._L.orc_set_tick(self._h, int(v))

    def state(self, env: int) -> OrcEnvState:
        p = self._L.orc_state(self._h, int(env))
        if not p:
            raise IndexError(env)
        return p.contents

    def reset(self, mask=None, nthreads: int = 1) -> np.ndarray:
        obs = np.zeros((self.num_envs, self.obs_dim), dtype=np.float32)
        mp = None
        if mask is not None:
            mask = np.ascontiguousarray(mask, dtype=np.uint8)
            mp = mask.ctypes.data_as(ctypes.POINTER(ctypes.c_uint8))
        self._L.orc_reset(self._h, mp, obs.ctypes.data_as(ctypes.POINTER(ctypes.c_float)), nthreads)
        return obs

    def step(self, actions, nthreads: int = 1):
        a = np.ascontiguousarray(actions, dtype=np.float32).reshape(self.num_envs, NJ)
        n, od = self.num_envs, self.obs_dim
        obs = np.zeros((n, od), dtype=np.float32)
        term_obs = np.zeros((n, od), dtype=np.float32)
        rew, ep_ret = np.zeros(n), np.zeros(n)
        term, trunc = np.zeros(n, dtype=np.uint8), np.zeros(n, dtype=np.uint8)
        ep_len = np.zeros(n, dtype=np.int32)
        fp, u8p = ctypes.POINTER(ctypes.c_float), ctypes.POINTER(ctypes.c_uint8)
        self._L.orc_step(self._h, a.ctypes.data_as(fp), obs.ctypes.data_as(fp), _d(rew), term.ctypes.data_as(u8p),
                         trunc.ctypes.data_as(u8p), term_obs.ctypes.data_as(fp), _d(ep_ret),
                         ep_len.ctypes.data_as(ctypes.POINTER(ctypes.c_int32)), nthreads)
        return obs, rew, term, trunc, term_obs, ep_ret, ep_len

    def set_state_soa(self, state: dict) -> None:
        """Adopt a state of the CUDA path: `state` maps so100_state_view field names to [k, N] float32 / int32 arrays
        (what `BatchedSo100Env.get_state()` returns, moved to the host)."""
        keep, ptr = [], {}
        for name, dt in (("qpos", np.float32), ("qvel", np.float32), ("qacc_warm", np.float32), ("qpos_comp", np.float32),
                         ("block", np.float32), ("snap", np.float32), ("aux", np.float32), ("counters", np.int32),
                         ("ep_return", np.float32)):
            a = state.get(name)
            if a is None:
                ptr[name] = None
                continue
            a = np.ascontiguousarray(a, dtype=dt)
            assert a.shape[-1] == self.num_envs, name
            keep.append(a)
            ptr[name] = a.ctypes.data
        self._L.orc_set_state_soa(self._h, ptr["qpos"], ptr["qvel"], ptr["qacc_warm"], ptr["qpos_comp"], ptr["block"], ptr["snap"],
                                  ptr["aux"], ptr["counters"], ptr["ep_return"])

    def get_state_soa(self):
        """(qpos [6, N], qvel [6, N], block [4, N]) as float64."""
        q, v, b = np.zeros((NJ, self.num_envs)), np.zeros((NJ, self.num_envs)), np.zeros((4, self.num_envs))
        self._L.orc_get_state_soa(self._h, _d(q), _d(v), _d(b))
        return q, v, b

    def gather(self, field: str) -> np.ndarray:
        """Stack one orc_env_state field over all envs -> [N, ...]."""
        return np.array([np.array(getattr(self.state(i), field)) for i in range(self.num_envs)])
