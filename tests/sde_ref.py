"""Host recomputation of the gSDE exploration matrices of so100_ppo_sde_act (include/so100_ppo.h, "Draw layout"):
normal i = 64 j + k of an env is position i % 4 of Philox block (seed, env, noise_key, 0x5D00 + i / 4), through the same
Box-Muller transform as box_muller_ref.z_host (fp64 from the kernel's fp32 uniforms)."""
import numpy as np

SDE_STREAM = 0x5D00
HID, ACT = 64, 6


def sde_z_host(seed, env_id, key):
    """z[k][j] (fp64, [64, 6]) of one env and the Box-Muller radius each carries."""
    from oracle.pyoracle import philox
    w = np.concatenate([philox(seed, env_id, key, SDE_STREAM + b) for b in range(HID * ACT // 4)])
    f = (w >> np.uint32(8)).astype(np.float32)
    u1 = (f[0::2] + np.float32(0.5)) * np.float32(1.0 / 16777216.0)
    u2 = f[1::2] * np.float32(1.0 / 16777216.0)
    rad = np.sqrt(-2.0 * np.log(u1.astype(np.float64)))
    ang = 2.0 * np.pi * u2.astype(np.float64)
    z = np.empty(HID * ACT)
    z[0::2], z[1::2] = rad * np.cos(ang), rad * np.sin(ang)
    # normal i = 64 j + k  ->  [k][j]
    return z.reshape(ACT, HID).T.copy(), np.repeat(rad, 2).reshape(ACT, HID).T.copy()
