"""ctypes loader of libso100_b200.so — the C ABI declared in include/so100_b200.h.

There is NO fallback: if the library has not been built (`python __graft_entry__.py build`) the import of anything that
needs it raises, and every call that needs a GPU raises `So100Error` when CUDA reports a failure.
"""
from __future__ import annotations

import ctypes
import os

from .model import So100Model
from .tasks import So100TaskCfg

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SO100_B200_LIB") or os.path.join(PKG_DIR, "libso100_b200.so")  # override: kernel experiments only

# every symbol include/so100_b200.h declares (tests/test_abi.py checks the two lists against each other)
EXPORTS = [
    "so100_abi_version", "so100_last_error", "so100_build_id", "so100_obs_dim", "so100_act_dim", "so100_create", "so100_destroy",
    "so100_reset", "so100_step", "so100_reset_host", "so100_step_host", "so100_get_state", "so100_set_state",
    "so100_get_tick", "so100_set_tick", "so100_forward_dynamics", "so100_host_forward", "so100_host_substeps", "so100_get_derived",
    "so100_get_stats", "so100_bench_fp32_peak", "so100_host_constants", "so100_kernel_variant",
    "so100_host_solver_constants", "so100_set_seed", "so100_step_substeps",
    "so100_host_groups", "so100_host_group_range", "so100_step_host_async", "so100_step_host_wait", "so100_step_host_wait_any",
    "so100_set_param_ranges", "so100_get_env_params", "so100_set_env_params",
    "so100_set_sim2real", "so100_get_actuator_state", "so100_set_actuator_state",
    # include/so100_ppo.h
    "so100_ppo_param_count", "so100_ppo_workspace_floats", "so100_ppo_act", "so100_ppo_post_step", "so100_ppo_gae",
    "so100_ppo_grad", "so100_ppo_adam", "so100_ppo_permutation",
    "so100_ppo_sde_param_count", "so100_ppo_sde_workspace_floats", "so100_ppo_sde_act", "so100_ppo_sde_grad",
]


class So100Error(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libso100_b200 error {code}: {msg}")
        self.code = code


class StateView(ctypes.Structure):
    """ctypes mirror of `so100_state_view`."""
    _fields_ = [(n, ctypes.c_void_p) for n in
                ("qpos", "qvel", "qacc_warm", "qpos_comp", "block", "snap", "aux", "counters", "ep_return")]


_lib = None


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build the CUDA extension first (python -c 'import __graft_entry__ as g; g.build()'). "
            "so100_mujoco_rl_b200 has no CPU or PyTorch fallback.")
    L = ctypes.CDLL(LIB_PATH)
    vp, ci = ctypes.c_void_p, ctypes.c_int
    dp = ctypes.POINTER(ctypes.c_double)
    i64p = ctypes.POINTER(ctypes.c_int64)
    L.so100_abi_version.restype = ci
    L.so100_last_error.restype = ctypes.c_char_p
    L.so100_build_id.restype = ctypes.c_char_p
    L.so100_obs_dim.argtypes = [ci]
    L.so100_act_dim.argtypes = [ci]
    L.so100_create.argtypes = [ctypes.POINTER(So100Model), ctypes.POINTER(So100TaskCfg), ci, ctypes.POINTER(vp)]
    L.so100_destroy.argtypes = [vp]
    L.so100_destroy.restype = None
    L.so100_reset.argtypes = [vp, vp, vp, vp]
    L.so100_step.argtypes = [vp] + [vp] * 8 + [vp]
    L.so100_step_substeps.argtypes = [vp, vp, ci, vp]
    L.so100_reset_host.argtypes = [vp, vp, vp]
    L.so100_step_host.argtypes = [vp] + [vp] * 8 + [vp]
    L.so100_host_groups.argtypes = [vp, ci]
    L.so100_host_group_range.argtypes = [vp, ci, ctypes.POINTER(ci), ctypes.POINTER(ci)]
    L.so100_step_host_async.argtypes = [vp, ci] + [vp] * 8 + [vp]
    L.so100_step_host_wait.argtypes = [vp, ci]
    L.so100_step_host_wait_any.argtypes = [vp, ctypes.POINTER(ci)]
    from .randomization import So100ActuatorView, So100ParamRanges, So100ParamView, So100Sim2Real
    L.so100_set_param_ranges.argtypes = [vp, ctypes.POINTER(So100ParamRanges)]
    L.so100_get_env_params.argtypes = [vp, ctypes.POINTER(So100ParamView), vp]
    L.so100_set_env_params.argtypes = [vp, ctypes.POINTER(So100ParamView), vp]
    L.so100_set_sim2real.argtypes = [vp, ctypes.POINTER(So100Sim2Real)]
    L.so100_get_actuator_state.argtypes = [vp, ctypes.POINTER(So100ActuatorView), vp]
    L.so100_set_actuator_state.argtypes = [vp, ctypes.POINTER(So100ActuatorView), vp]
    L.so100_get_state.argtypes = [vp, ctypes.POINTER(StateView), vp]
    L.so100_set_state.argtypes = [vp, ctypes.POINTER(StateView), vp]
    L.so100_get_tick.argtypes = [vp, i64p]
    L.so100_set_tick.argtypes = [vp, ctypes.c_int64]
    L.so100_set_seed.argtypes = [vp, ctypes.c_uint64]
    L.so100_forward_dynamics.argtypes = [vp, ci] + [vp] * 7 + [vp]
    L.so100_host_forward.argtypes = [ctypes.POINTER(So100Model), ci, dp, dp, dp, dp, dp, dp, dp, ci, ci]
    L.so100_host_substeps.argtypes = [ctypes.POINTER(So100Model), ci, dp, dp, dp, dp, ci, ci, i64p]
    L.so100_host_constants.argtypes = [ctypes.POINTER(So100Model), dp]
    L.so100_host_solver_constants.argtypes = [ctypes.POINTER(So100Model), ctypes.POINTER(ctypes.c_float), ci]
    L.so100_kernel_variant.argtypes = [vp]
    L.so100_get_derived.argtypes = [vp, dp, dp, dp]
    L.so100_get_stats.argtypes = [vp, i64p, i64p, i64p]
    L.so100_bench_fp32_peak.argtypes = [ci, ci, dp]
    cf, u32, u64, i64 = ctypes.c_float, ctypes.c_uint32, ctypes.c_uint64, ctypes.c_int64
    L.so100_ppo_param_count.argtypes = [ci]
    L.so100_ppo_workspace_floats.argtypes = [ci]
    L.so100_ppo_act.argtypes = [ci, vp, vp, ci, u64, i64, u32, ci, vp, vp, vp, vp, vp, vp]
    L.so100_ppo_post_step.argtypes = [ci, vp, ci, vp, vp, vp, vp, vp, vp, cf, vp, vp, vp, vp]
    L.so100_ppo_gae.argtypes = [vp, vp, vp, vp, ci, ci, cf, cf, vp, vp, vp]
    L.so100_ppo_grad.argtypes = [ci, vp, vp, vp, vp, vp, vp, vp, ci, cf, cf, cf, ci, vp, vp, vp, vp]
    L.so100_ppo_permutation.argtypes = [ci, u64, vp, vp]
    L.so100_ppo_adam.argtypes = [ci, vp, vp, vp, vp, vp, cf, cf, cf, cf, cf, cf, vp]
    L.so100_ppo_sde_param_count.argtypes = [ci]
    L.so100_ppo_sde_workspace_floats.argtypes = [ci]
    L.so100_ppo_sde_act.argtypes = L.so100_ppo_act.argtypes
    L.so100_ppo_sde_grad.argtypes = L.so100_ppo_grad.argtypes
    for name in EXPORTS:
        if name not in ("so100_last_error", "so100_destroy", "so100_build_id"):
            getattr(L, name).restype = ci
    L.so100_ppo_workspace_floats.restype = i64
    L.so100_ppo_sde_workspace_floats.restype = i64
    if L.so100_abi_version() != 3:
        raise ImportError("libso100_b200.so has an unexpected ABI version; rebuild it")
    _lib = L
    return L


def check(rc: int) -> int:
    if rc < 0:
        raise So100Error(rc, lib().so100_last_error().decode("utf-8", "replace"))
    return rc
