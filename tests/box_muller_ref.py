"""Host recomputation of the kernels' Box-Muller normals (the PPO act kernel's action noise and the env step's observation
noise use the same transform): the Philox words come from the fp64 oracle's restatement of the generator, and the
transform runs in fp64 from the kernel's fp32 uniforms."""
import numpy as np


def z_host(seed, env_id, tick, stream):
    """z[0..5] of the kernel's Box-Muller draw, in fp64 from the kernel's fp32 uniforms, and the radii they carry."""
    from oracle.pyoracle import philox
    w = np.concatenate([philox(seed, env_id, tick, stream), philox(seed, env_id, tick, stream + 1)])[:6]
    f = (w >> np.uint32(8)).astype(np.float32)
    u1 = (f[0::2] + np.float32(0.5)) * np.float32(1.0 / 16777216.0)  # fp32, as the kernel rounds it
    u2 = f[1::2] * np.float32(1.0 / 16777216.0)
    rad = np.sqrt(-2.0 * np.log(u1.astype(np.float64)))
    ang = 2.0 * np.pi * u2.astype(np.float64)
    z = np.empty(6)
    z[0::2], z[1::2] = rad * np.cos(ang), rad * np.sin(ang)
    return z, np.repeat(rad, 2)


def noise_tolerance(sigma, rad, noise, obs):
    """|device - host| bound of fp32(q + fp32(sigma z)), from the CUDA math library's documented maximum errors:
    logf 1 ulp, sqrtf correctly rounded (0.5 ulp), sincospif 1 ulp, fp32 products / sums 0.5 ulp each.
      rad:  -2 logf(u1) is off by <= 2^-23 relative, sqrtf halves that and adds 2^-24     -> <= 2^-23 rad
      z:    rad (cos + dcos) with |dcos| <= 1 ulp <= 2^-23, the product rounded (2^-24)  -> <= 2.5 * 2^-23 rad
    The kernel's sigma z and q + sigma z are each rounded once, the host's once more from fp64: one ulp of each on top.
    A factor 2 on the z bound leaves room for the host's own fp64 rounding (~2^-52)."""
    eps = 2.0 ** -23
    return sigma * 5.0 * eps * rad + np.spacing(np.abs(noise).astype(np.float32)) + np.spacing(np.abs(obs).astype(np.float32))
