"""Fused PPO kernels (include/so100_ppo.h) against plain float64 references of the same operations, at the sizes the
trainer launches and at the edges of the C ABI.

test_gpu_ppo.py compares the kernels with torch fp32 at small sizes.  Here every reference is float64 and every
tolerance is an error bound derived from the fp32 computation the kernel does (running-error analysis): the bound is
evaluated per element from the fp64 magnitudes of the same computation, so a kernel that is wrong by more than its
own rounding fails, and one that is right passes whatever the data.  Units:
  U          = 2^-23: one fp32 ulp relative.  A full ulp (not half) per rounding also covers the tensor cores' fp32
               accumulation, which may truncate instead of rounding to nearest.
  EPS_3XTF32 = 3 * 2^-20: error of one 3xTF32 product a b = hi hi + hi lo + lo hi.  hi keeps 11 significant bits, so
               |lo| < 2^-10 |x|; the tensor core truncates lo to 11 bits (< 2^-20 |x| lost) in each of the two cross
               terms, and lo lo (< 2^-20 |ab|) is dropped (so100_ppo_kernels.cuh, split_tf32).
  CUDA math library maximum errors (CUDA C Programming Guide, "Mathematical functions"): tanhf 2 ulp, expf 2 ulp,
               logf 1 ulp, sincospif 1 ulp, powf 4 ulp, rsqrtf 2 ulp; sqrtf and '/' are correctly rounded (the library
               is built without fast-math).
Each test prints its largest observed error beside its bound (pytest -s).  The bounds are worst cases: every rounding
error at its maximum and of the same sign, and input errors carried through |W| (the L1 row norms of W2 and W3 are
~10, so the forward-pass bound grows ~100x over the two layers after the first).  Measured on an NVIDIA B200 (1000 W
power limit), observed / bound is 0.2-0.5 for GAE and Adam (short chains of roundings), 0.04-0.2 for the action noise,
and 1e-2 to 1e-6 for the forward pass and the gradient, whose errors are sums of thousands of nearly independent
roundings that cancel.  The dense checks therefore catch gross errors (a wrong branch, wrong or duplicated samples,
a wrong tile); the placement, chunking and noise tests pin the rest bit for bit or to a few ulps.
"""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from box_muller_ref import noise_tolerance, z_host

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

U = 2.0 ** -23
EPS_3XTF32 = 3.0 * 2.0 ** -20
LOG_SQRT_2PI = 0.5 * math.log(2.0 * math.pi)
GT = 32          # samples per tile of the gradient kernel
ACT_TILE = 128   # samples per tile of the tcgen05 inference kernel
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    from so100_mujoco_rl_b200 import _native
    return _native.lib(), _native.check


def _st():
    return torch.cuda.current_stream().cuda_stream


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _report(what, err, bound):
    """One line per check: the largest |kernel - fp64| and the largest ratio to its bound."""
    err, bound = np.asarray(err, dtype=np.float64), np.asarray(bound, dtype=np.float64)
    ratio = float(np.max(err / np.maximum(bound, 1e-300))) if err.size else 0.0
    print(f"[fp64] {what}: max err {float(err.max()) if err.size else 0.0:.3e}  max bound {float(bound.max()) if bound.size else 0.0:.3e}"
          f"  max err/bound {ratio:.3e}")
    return ratio


def _params(od, seed, scale=1.0):
    """A policy away from SB3's tiny-gain initialisation (every path carries signal), packed as the kernels read it."""
    from so100_mujoco_rl_b200.ppo import MlpPolicy, pack_params
    torch.manual_seed(seed)
    p = MlpPolicy(od, 6)
    with torch.no_grad():
        for t in p.parameters():
            t.add_(scale * 0.1 * torch.randn_like(t))
        p.log_std.add_(0.3 * torch.randn(6))
    return pack_params(p)


def _blocks(flat, od):
    """Named views (param_layout order) into a flat parameter vector."""
    from so100_mujoco_rl_b200.ppo import param_layout
    out, o = {}, 0
    for name, shape in param_layout(od):
        k = int(np.prod(shape))
        out[name] = flat[o:o + k].view(shape)
        o += k
    assert o == flat.numel()
    return out


def _c(k):
    """Relative error of a k-long 3xTF32 dot product plus a bias, accumulated in fp32, per unit of sum |terms|."""
    return EPS_3XTF32 + (k + 1) * U


def _tower64(B, t, x):
    """fp64 forward pass of one tower; differentiable when B's tensors are."""
    h1 = torch.tanh(x @ B[f"{t}.W1"].T + B[f"{t}.b1"])
    h2 = torch.tanh(h1 @ B[f"{t}.W2"].T + B[f"{t}.b2"])
    return h1, h2, h2 @ B[f"{t}.W3"].T + B[f"{t}.b3"]


def _tower_bound(B, t, x, h1, h2):
    """Running-error bound of the kernels' fp32 forward pass of one tower, element by element.
      layer:  |dz| <= |W| |dx| + c(K) (|W| |x| + |b|)   (3xTF32 products, K + 1 fp32 additions; K = 16 for the padded
              first layer, 64 after it.  The fp32 FMA heads and value_one are covered by the same bound.)
      tanhf:  |dh| <= |dz| + 2 ulp(h)                       (tanh is 1-Lipschitz)."""
    W1, b1, W2, b2, W3, b3 = (B[f"{t}.{k}"].abs() for k in ("W1", "b1", "W2", "b2", "W3", "b3"))
    e1 = _c(16) * (x.abs() @ W1.T + b1) + 2 * U * h1.abs()
    e2 = e1 @ W2.T + _c(64) * (h1.abs() @ W2.T + b2) + 2 * U * h2.abs()
    eo = e2 @ W3.T + _c(64) * (h2.abs() @ W3.T + b3)
    return e1, e2, eo


# ------------------------------------------------------------------------------------------------ 1. so100_ppo_act
ACT_OD = (1, 8, 15, 16)
ACT_N = ("1", "127", "129", "65536", "multi")


def _act_n(label):
    # multi: at least two tiles for every CTA of the persistent grid (2 CTAs per SM) plus a ragged last tile
    return 2 * _sms() * ACT_TILE * 2 + 77 if label == "multi" else int(label)


def _act_offset(label):
    # a large env_offset for the multi-tile case: the Philox counter crosses 2^31 inside the first CTA's tiles
    return {"multi": 2 ** 31 - 3 * ACT_TILE - 5, "65536": 0}.get(label, 12345)


_ACT_CHILD = r"""
import sys
import numpy as np
import torch
root, inp, outp = sys.argv[1:4]
sys.path.insert(0, root)
from so100_mujoco_rl_b200 import _native
L = _native.lib()
st = torch.cuda.current_stream().cuda_stream
src = np.load(inp)
chunk = 2 * torch.cuda.get_device_properties(0).multi_processor_count * 128   # one tile per CTA
names = ("a", "c", "lp", "v", "oc")
out = {}


def run(od, P, obs, n, seed, off, tick, det):
    f = dict(device="cuda", dtype=torch.float32)
    res = [torch.full((n, 6), float("nan"), **f), torch.full((n, 6), float("nan"), **f), torch.full((n,), float("nan"), **f),
           torch.full((n,), float("nan"), **f), torch.full((n, od), float("nan"), **f)]
    _native.check(L.so100_ppo_act(od, P.data_ptr(), obs.data_ptr(), n, seed, off, tick, det, *(t.data_ptr() for t in res), st))
    return [t.cpu().numpy() for t in res]


for key in src["keys"]:
    od, n, seed, off, tick = (int(x) for x in src[key + "__meta"])
    P, obs = torch.from_numpy(src[key + "__P"]).cuda(), torch.from_numpy(src[key + "__obs"]).cuda()
    for tag, det in (("det", 1), ("sto", 0)):
        for name, arr in zip(names, run(od, P, obs, n, seed, off, tick, det)):
            out[key + "__" + tag + "__" + name] = arr
    parts = [run(od, P, obs[c0:c0 + chunk].contiguous(), min(chunk, n - c0), seed, off + c0, tick, 0) for c0 in range(0, n, chunk)]
    for i, name in enumerate(names):
        out[key + "__chunk__" + name] = np.concatenate([p[i] for p in parts])
torch.cuda.synchronize()
np.savez(outp, **out)
"""


@pytest.fixture(scope="module")
def act_runs(tmp_path_factory):
    """Both inference kernels on every (obs_dim, n) case: deterministic, stochastic, and the stochastic call again as
    chunks of one tile per CTA.  SO100_PPO_ACT_MMA is read once per process, hence one subprocess per kernel."""
    d = tmp_path_factory.mktemp("act")
    inputs, keys = {}, []
    for od in ACT_OD:
        P = _params(od, seed=100 + od).numpy()
        for i, label in enumerate(ACT_N):
            n, key = _act_n(label), f"{od}_{label}"
            rng = np.random.default_rng(1000 * od + i)
            inputs[key + "__P"] = P
            inputs[key + "__obs"] = (2.0 * rng.standard_normal((n, od))).astype(np.float32)
            inputs[key + "__meta"] = np.array([od, n, 0x5EED0000 + od, _act_offset(label), 40 + i], dtype=np.int64)
            keys.append(key)
    inputs["keys"] = np.array(keys)
    inp = str(d / "in.npz")
    np.savez(inp, **inputs)
    res = {}
    for path in ("tc", "mma"):
        env = dict(os.environ)
        env.pop("SO100_PPO_ACT_MMA", None)
        if path == "mma":
            env["SO100_PPO_ACT_MMA"] = "1"
        outp = str(d / f"{path}.npz")
        subprocess.run([sys.executable, "-c", _ACT_CHILD, ROOT, inp, outp], check=True, env=env, timeout=600)
        res[path] = dict(np.load(outp))
    return inputs, res


def _case(act_runs, path, od, label):
    inputs, res = act_runs
    key = f"{od}_{label}"
    od_, n, seed, off, tick = (int(x) for x in inputs[key + "__meta"])
    got = {k[len(key) + 2:]: v for k, v in res[path].items() if k.startswith(key + "__")}
    return inputs[key + "__P"], inputs[key + "__obs"], n, seed, off, tick, got


def _act_fp64(P, obs, od):
    B = _blocks(torch.from_numpy(P).cuda().double(), od)
    x = torch.from_numpy(obs).cuda().double()
    out = {}
    for t in ("pi", "vf"):
        h1, h2, o = _tower64(B, t, x)
        out[t] = (o, _tower_bound(B, t, x, h1, h2)[2])
    return out["pi"][0].cpu().numpy(), out["pi"][1].cpu().numpy(), out["vf"][0][:, 0].cpu().numpy(), out["vf"][1][:, 0].cpu().numpy(), \
        B["log_std"].cpu().numpy()


def _noise_envs(n):
    """A few hundred envs spread over tiles and CTAs: both ends, tile edges, the first tile of the second pass."""
    c = 2 * _sms() * ACT_TILE
    pick = set(np.linspace(0, n - 1, 240).astype(np.int64).tolist())
    pick |= {g for g in (0, 1, 127, 128, 129, c - 1, c, c + 1, 2 * c, n - 78, n - 2, n - 1) if 0 <= g < n}
    return np.array(sorted(pick))


@pytest.mark.parametrize("label", ACT_N)
@pytest.mark.parametrize("od", ACT_OD)
@pytest.mark.parametrize("path", ["tc", "mma"])
def test_act_matches_the_fp64_forward_pass(act_runs, path, od, label):
    """Deterministic mode returns the fp64 mean, value and log-prob within the forward-pass bound of _tower_bound.
    log-prob = sum_k (-ls_k - log sqrt(2 pi)): 18 fp32 roundings of partial sums <= sum_k (|ls_k| + log sqrt(2 pi)).
    The stochastic call returns the same value bits, act_clip = clip(act_raw) and obs_copy = obs bit for bit."""
    P, obs, n, seed, off, tick, got = _case(act_runs, path, od, label)
    mean, e_mean, val, e_val, ls = _act_fp64(P, obs, od)
    err_m, err_v = np.abs(got["det__a"] - mean), np.abs(got["det__v"] - val)
    _report(f"act {path} od={od} n={n} mean", err_m, e_mean)
    _report(f"act {path} od={od} n={n} value", err_v, e_val)
    assert (err_m <= e_mean).all(), np.unravel_index(np.argmax(err_m - e_mean), err_m.shape)
    assert (err_v <= e_val).all(), int(np.argmax(err_v - e_val))
    lp = float(np.sum(-ls - LOG_SQRT_2PI))
    assert np.all(np.abs(got["det__lp"] - lp) <= 18 * U * float(np.sum(np.abs(ls) + LOG_SQRT_2PI)))
    for tag in ("det", "sto"):
        assert np.array_equal(got[tag + "__oc"].view(np.int32), obs.view(np.int32))
        assert np.array_equal(got[tag + "__c"].view(np.int32), np.clip(got[tag + "__a"], -1.0, 1.0).view(np.int32))
    assert np.array_equal(got["sto__v"].view(np.int32), got["det__v"].view(np.int32))


@pytest.mark.parametrize("label", ACT_N)
@pytest.mark.parametrize("od", [8, 16])
@pytest.mark.parametrize("path", ["tc", "mma"])
def test_act_noise_is_the_documented_philox_box_muller_draw(act_runs, path, od, label):
    """(a - mean_det) / exp(log_std) against z_host(seed, env_offset + env, tick, 0x5050) (with the 0x5051 block).
    Bound in action space: box_muller_ref.noise_tolerance(sigma, rad, sigma z, a) for fp32(mean + fp32(sigma z)), plus
    2 ulp of sigma times |z| <= rad because the kernel's sigma is expf(log_std).  The log-prob of the draw is
    sum_k (-z_k^2 / 2 - ls_k - log sqrt(2 pi)) within sum_k |z_k| dz_k (dz = 5 ulp rad, noise_tolerance's z bound) plus
    24 roundings of partial sums <= sum_k (z_k^2 / 2 + |ls_k| + log sqrt(2 pi))."""
    P, obs, n, seed, off, tick, got = _case(act_runs, path, od, label)
    ls = _blocks(torch.from_numpy(P).double(), od)["log_std"].numpy()
    sig = np.exp(ls)
    worst_z = worst_lp = 0.0
    for g in _noise_envs(n):
        z, rad = z_host(seed, int(off + g) & 0xFFFFFFFF, tick, 0x5050)
        a, m = got["sto__a"][g].astype(np.float64), got["det__a"][g].astype(np.float64)
        tol = noise_tolerance(sig, rad, sig * z, got["sto__a"][g]) + 2 * U * sig * rad
        dz = np.abs((a - m) / sig - z)
        worst_z = max(worst_z, float(np.max(dz / (tol / sig))))
        assert (dz <= tol / sig).all(), (g, (a - m) / sig, z, tol / sig)
        lp = float(np.sum(-0.5 * z * z - ls - LOG_SQRT_2PI))
        e_lp = float(np.sum(np.abs(z) * 5 * U * rad)) + 24 * U * float(np.sum(0.5 * z * z + np.abs(ls) + LOG_SQRT_2PI))
        worst_lp = max(worst_lp, abs(float(got["sto__lp"][g]) - lp) / e_lp)
        assert abs(float(got["sto__lp"][g]) - lp) <= e_lp, (g, got["sto__lp"][g], lp, e_lp)
    print(f"[fp64] act noise {path} od={od} n={n}: max err/bound z {worst_z:.3e}, log-prob {worst_lp:.3e}")


@pytest.mark.parametrize("od", ACT_OD)
@pytest.mark.parametrize("path", ["tc", "mma"])
def test_act_single_call_equals_one_tile_per_cta_chunks_bitwise(act_runs, path, od):
    """A persistent CTA that serves several tiles (mbarrier phase, TMEM reuse, second pass of the tile loop) gives the
    bits that chunks of at most 2 SMs x 128 envs (one tile per CTA) give, with matching env_offset, on every output."""
    P, obs, n, seed, off, tick, got = _case(act_runs, path, od, "multi")
    for name in ("a", "c", "lp", "v", "oc"):
        a, b = got["sto__" + name], got["chunk__" + name]
        assert a.shape == b.shape and np.array_equal(a.view(np.int32), b.view(np.int32)), name


# ------------------------------------------------------------------------------------------------ 2. so100_ppo_grad
def _grad_data(od, S, seed, clip=0.2):
    """Rollout-like buffers: actions drawn from the policy, old log-probs from a perturbed policy (ratios on both
    sides of the clip range), then nudged so that no ratio lies within 1e-4 of 1 +- clip: which branch of the
    surrogate a sample takes must not depend on rounding."""
    P = _params(od, seed=seed).cuda()
    g = torch.Generator(device="cuda").manual_seed(seed)
    obs = torch.randn(S, od, device="cuda", generator=g)
    B = _blocks(P.double(), od)
    with torch.no_grad():
        mean = _tower64(B, "pi", obs.double())[2]
        sig = B["log_std"].exp()
        act = (mean + sig * torch.randn(S, 6, device="cuda", generator=g, dtype=torch.float64)).float()
        lp_of = lambda m: (-0.5 * ((act.double() - m) / sig) ** 2 - B["log_std"] - LOG_SQRT_2PI).sum(-1)  # noqa: E731
        logp_old = lp_of(mean + 0.15 * torch.randn(S, 6, device="cuda", generator=g, dtype=torch.float64)).float()
        for _ in range(3):
            ratio = torch.exp(lp_of(mean) - logp_old.double())
            near = ((ratio - (1 - clip)).abs() < 1e-4) | ((ratio - (1 + clip)).abs() < 1e-4)
            logp_old = torch.where(near, logp_old - 1e-3, logp_old)
        assert not bool(near.any())
    adv = torch.randn(S, device="cuda", generator=g) * 2 + 0.3
    ret = torch.randn(S, device="cuda", generator=g)
    return P, obs, act, logp_old, adv, ret


def _kernel_grad(od, P, obs, act, logp_old, adv, ret, idx, clip, vf_coef, ent_coef, normalize):
    L, check = _lib()
    ws = torch.zeros(int(L.so100_ppo_workspace_floats(od)), device="cuda")
    grad, loss = torch.full((P.numel(),), float("nan"), device="cuda"), torch.full((3,), float("nan"), device="cuda")
    check(L.so100_ppo_grad(od, P.data_ptr(), obs.data_ptr(), act.data_ptr(), logp_old.data_ptr(), adv.data_ptr(), ret.data_ptr(),
                           idx.data_ptr(), idx.numel(), clip, vf_coef, ent_coef, normalize, ws.data_ptr(), grad.data_ptr(), loss.data_ptr(), _st()))
    return grad, loss


def _sb3_grad64(od, P, x, act, lpo, adv, ret, clip, vf_coef, ent_coef, normalize, divisor=None):
    """SB3 PPO.train's loss for one minibatch in float64 through autograd (stable_baselines3/ppo/ppo.py): advantages
    normalised when there is more than one, clipped surrogate, MSE value loss, entropy bonus.  divisor replaces the
    minibatch mean's 1/len by 1/divisor (one sample of a larger minibatch)."""
    flat = P.double().clone().requires_grad_(True)
    B = _blocks(flat, od)
    a = adv
    if normalize and a.numel() > 1:
        a = (a - a.mean()) / (a.std() + 1e-8)
    mean, ls = _tower64(B, "pi", x)[2], B["log_std"]
    value = _tower64(B, "vf", x)[2][:, 0]
    logp = (-((act - mean) ** 2) / (2 * torch.exp(2 * ls)) - ls - LOG_SQRT_2PI).sum(-1)
    lr = logp - lpo
    ratio = torch.exp(lr)
    k = float(divisor or x.shape[0])
    pg = -torch.min(a * ratio, a * torch.clamp(ratio, 1 - clip, 1 + clip)).sum() / k
    vl = ((value - ret) ** 2).sum() / k
    ent = (0.5 + LOG_SQRT_2PI + ls).sum() * (x.shape[0] / k)
    (pg + vf_coef * vl - ent_coef * ent).backward()
    return flat.grad.detach(), torch.stack([pg.detach(), vl.detach(), ((ratio - 1) - lr).sum().detach() / k])


def _grad_bound(od, P, x, act, lpo, adv, ret, clip, vf_coef, ent_coef, normalize, divisor, depth):
    """Element-wise bound of |kernel - fp64| for the gradient and the three losses (running-error analysis of the
    kernel's fp32 computation; every quantity carries its magnitude and a bound of its error).
      forward:  _tower_bound -> e(mean), e(value), e(h1), e(h2).
      loss:     d = act - mean (+1 ulp);  log-prob: 22 roundings of partial sums <= sum_k (d^2 / 2 sigma^2 + |ls| + c)
                plus sum_k |d_k| e(d_k) / sigma_k^2;  ratio = expf(lp - old): e(ratio) = ratio (e(lr) + 3 ulp);
                normalised A = (adv - fp32(mean)) * fp32(rstd): e(A) = rstd 2^-24 |mean| + 3 ulp |A| (the statistics
                themselves are fp64);  g = A ratio on the active branch;  d loss / d out per sample: 4 more roundings.
                A sample whose A is within e(A) of 0 outside the clip range may take either branch: |A| + e(A) times
                ratio is allowed for it.
      backward: through the heads (fp32 FMA, <= 6 terms) and 1 - h2^2:  10 ulp and 2 |h2| e(h2);  through W2
                (3xTF32, K = 64) and 1 - h1^2: c(64) + 3 ulp and 2 |h1| e(h1); propagated errors through |W|.
      sums over the minibatch: every weight-gradient entry is a sum of per-sample terms accumulated in fp32 along a
                chain of `depth` additions (a tile's samples, the CTA's tiles, then the CTAs' partials in the reduction):
                depth ulp of sum |terms| plus the per-sample errors."""
    B = _blocks(P.double(), od)
    m = x.shape[0]
    with torch.no_grad():
        res = {}
        h1p, h2p, mean = _tower64(B, "pi", x)
        h1v, h2v, vout = _tower64(B, "vf", x)
        e1p, e2p, em = _tower_bound(B, "pi", x, h1p, h2p)
        e1v, e2v, ev = _tower_bound(B, "vf", x, h1v, h2v)
        value, ev = vout[:, 0], ev[:, 0]
        ls = B["log_std"]
        isig2 = torch.exp(-2 * ls)
        d = act - mean
        e_d = em + U * d.abs()
        T_lp = (0.5 * d * d * isig2 + ls.abs() + LOG_SQRT_2PI).sum(-1)
        lp = (-0.5 * d * d * isig2 - ls - LOG_SQRT_2PI).sum(-1)
        e_lp = (d.abs() * isig2 * e_d).sum(-1) + 22 * U * T_lp
        lr = lp - lpo
        e_lr = e_lp + U * (lp.abs() + lpo.abs())
        ratio = torch.exp(lr)
        e_ratio = ratio * (e_lr + 3 * U) * (1 + 2 * e_lr)
        if normalize and m > 1:
            mu, rstd = adv.mean(), 1.0 / (adv.std() + 1e-8)
            A = (adv - mu) * rstd
            e_A = rstd * 2.0 ** -24 * mu.abs() + 3 * U * A.abs()
        else:
            A, e_A = adv, torch.zeros_like(adv)
        inside = (ratio >= 1 - clip) & (ratio <= 1 + clip)
        x1, x2 = A * ratio, A * ratio.clamp(1 - clip, 1 + clip)
        active = (inside | (x1 < x2)).double()
        either = (~inside & (A.abs() <= e_A)).double()
        e_g = active * (A.abs() * e_ratio + ratio * e_A + U * x1.abs()) + either * (A.abs() + e_A) * ratio * (1 + e_lr)
        dlp = -A * ratio * active / divisor
        e_dlp = e_g / divisor + 2 * U * dlp.abs()
        dout = dlp[:, None] * d * isig2
        e_dout = e_dlp[:, None] * d.abs() * isig2 + dlp.abs()[:, None] * e_d * isig2 + 4 * U * dout.abs()
        q_ls = d * d * isig2 - 1
        mag_ls = dlp.abs()[:, None] * q_ls.abs() + ent_coef / divisor
        e_ls = e_dlp[:, None] * q_ls.abs() + dlp.abs()[:, None] * 2 * d.abs() * isig2 * e_d \
            + 6 * U * (dlp.abs()[:, None] * (d * d * isig2 + 1) + ent_coef / divisor)
        e_v = value - ret
        dv = 2 * e_v * vf_coef / divisor
        e_dv = 2 * vf_coef / divisor * ev + 4 * U * dv.abs()
        c_w = EPS_3XTF32 + depth * U
        c_s = depth * U
        for t, G, E, h1, h2, e1, e2 in (("pi", dout.abs(), e_dout, h1p, h2p, e1p, e2p), ("vf", dv.abs()[:, None], e_dv[:, None], h1v, h2v, e1v, e2v)):
            W2a, W3a = B[f"{t}.W2"].abs(), B[f"{t}.W3"].abs()
            q2 = G @ W3a
            sd2 = 1 - h2 * h2
            G2 = q2 * sd2
            E2 = (E @ W3a) * sd2 + q2 * 2 * h2.abs() * e2 + 10 * U * q2
            q1 = G2 @ W2a
            sd1 = 1 - h1 * h1
            G1 = q1 * sd1
            E1 = (E2 @ W2a) * sd1 + q1 * 2 * h1.abs() * e1 + (_c(64) + 3 * U) * q1
            res[f"{t}.W3"] = E.T @ h2.abs() + G.T @ e2 + c_s * (G.T @ h2.abs())
            res[f"{t}.b3"] = E.sum(0) + c_s * G.sum(0)
            res[f"{t}.W2"] = E2.T @ h1.abs() + G2.T @ e1 + c_w * (G2.T @ h1.abs())
            res[f"{t}.b2"] = E2.sum(0) + c_s * G2.sum(0)
            res[f"{t}.W1"] = E1.T @ x.abs() + c_w * (G1.T @ x.abs())
            res[f"{t}.b1"] = E1.sum(0) + c_s * G1.sum(0)
        res["log_std"] = e_ls.sum(0) + c_s * mag_ls.sum(0)
        from so100_mujoco_rl_b200.ppo import param_layout
        tol = torch.cat([res[name].reshape(-1) for name, _ in param_layout(od)])
        pmin = torch.minimum(x1, x2).abs()
        e_pg = ((A.abs() * e_ratio + ratio * e_A + 2 * U * x1.abs()).sum() + (c_s + 2 * U) * pmin.sum()) / divisor \
            + (either * (A.abs() + e_A) * ratio * (1 + e_lr)).sum() / divisor
        e_vl = ((2 * e_v.abs() * ev + 2 * U * e_v * e_v).sum() + (c_s + 2 * U) * (e_v * e_v).sum()) / divisor
        kl = (ratio - 1) - lr
        e_kl = ((e_ratio + e_lr + 2 * U * ((ratio - 1).abs() + lr.abs())).sum() + (c_s + 2 * U) * kl.abs().sum()) / divisor
    return tol, torch.stack([e_pg, e_vl, e_kl])


def _depth(mb):
    """Longest fp32 accumulation chain of a gradient entry: a tile's 32 samples, the tiles of the busiest CTA, the
    partials of every CTA (reduce_kernel), plus the 4 sample groups / 3 MMAs per product."""
    ntiles = (mb + GT - 1) // GT
    grid = min(ntiles, 2 * _sms())
    return GT + (ntiles + grid - 1) // grid + grid + 4


def _check_grad(what, od, grad, loss, g64, l64, tol, ltol):
    from so100_mujoco_rl_b200.ppo import param_layout
    err = (grad.double() - g64).abs()
    o = 0
    for name, shape in param_layout(od):
        k = int(np.prod(shape))
        e, b = err[o:o + k], tol[o:o + k]
        _report(f"grad {what} {name} (|g64| max {float(g64[o:o + k].abs().max()):.2e})", e.cpu().numpy(), b.cpu().numpy())
        assert bool((e <= b).all()), (name, float((e - b).max()), int(torch.argmax(e - b)))
        o += k
    lerr = (loss.double() - l64).abs()
    _report(f"grad {what} losses", lerr.cpu().numpy(), ltol.cpu().numpy())
    assert bool((lerr <= ltol).all()), (loss.tolist(), l64.tolist(), ltol.tolist())


def _dense_case(od, S, mb, normalize, ent_coef, seed=7, clip=0.2, vf_coef=0.5):
    P, obs, act, lpo, adv, ret = _grad_data(od, S, seed, clip)
    g = torch.Generator(device="cuda").manual_seed(seed + 1)
    idx = torch.randperm(S, device="cuda", generator=g)[:mb]
    grad, loss = _kernel_grad(od, P, obs, act, lpo, adv, ret, idx, clip, vf_coef, ent_coef, normalize)
    x, a64, l64_, adv64, ret64 = obs[idx].double(), act[idx].double(), lpo[idx].double(), adv[idx].double(), ret[idx].double()
    g64, loss64 = _sb3_grad64(od, P, x, a64, l64_, adv64, ret64, clip, vf_coef, ent_coef, normalize)
    tol, ltol = _grad_bound(od, P, x, a64, l64_, adv64, ret64, clip, vf_coef, ent_coef, normalize, mb, _depth(mb))
    return grad, loss, g64, loss64, tol, ltol, (P, obs, act, lpo, adv, ret, idx)


GRAD_CASES = {  # od, S, mb (a function of the SM count), normalize, ent_coef
    "production-normalised": (8, 2 ** 21, lambda s: 2 ** 18, 1, 0.0),
    "production-raw": (8, 2 ** 21, lambda s: 2 ** 18, 0, 0.0),
    "od1": (1, 60_000, lambda s: 40_000, 1, 0.0),
    "od15-entropy": (15, 60_000, lambda s: 40_000, 1, 0.01),
    "od16-ragged-entropy": (16, 100_000, lambda s: 3 * 2 * s * GT + 17, 1, 0.01),
}


@pytest.mark.parametrize("case", list(GRAD_CASES))
def test_grad_matches_fp64_autograd(case):
    """Every parameter block and the three losses within _grad_bound of the fp64 autograd of SB3's loss, at the
    trainer's shape (obs_dim 8, 2^21 samples, minibatch 2^18: ~28 tiles per CTA) and at the obs_dim / ragged edges;
    both branches of the clipped surrogate are exercised."""
    od, S, mbf, normalize, ent_coef = GRAD_CASES[case]
    mb = mbf(_sms())
    grad, loss, g64, l64, tol, ltol, data = _dense_case(od, S, mb, normalize, ent_coef)
    P, obs, act, lpo, adv, ret, idx = data
    with torch.no_grad():
        mean = _tower64(_blocks(P.double(), od), "pi", obs[idx].double())[2]
        ls = _blocks(P.double(), od)["log_std"]
        ratio = torch.exp((-0.5 * ((act[idx].double() - mean) / ls.exp()) ** 2 - ls - LOG_SQRT_2PI).sum(-1) - lpo[idx].double())
    frac_clipped = float(((ratio - 1).abs() > 0.2).double().mean())
    assert 0.05 < frac_clipped < 0.95, frac_clipped
    _check_grad(f"{case} mb={mb}", od, grad, loss, g64, l64, tol, ltol)


def _placement_positions(mb):
    ntiles = (mb + GT - 1) // GT
    grid = min(ntiles, 2 * _sms())
    last_tile_cta0 = ((ntiles - 1) // grid) * grid      # CTA 0 serves the most tiles; its last one
    pos = {0, 31, 32, mb - 1, grid * GT, grid * GT + 5, last_tile_cta0 * GT, min(last_tile_cta0 * GT + 7, mb - 1)}
    return sorted(p for p in pos if 0 <= p < mb)


PLACEMENT_MB = ("1", "31", "32", "33", "2sm32-1", "2sm32+1", "262144")


def _placement_mb(label):
    s = _sms()
    return {"2sm32-1": 2 * s * GT - 1, "2sm32+1": 2 * s * GT + 1}.get(label) or int(label)


@pytest.mark.parametrize("label", PLACEMENT_MB)
def test_grad_single_sample_is_placement_independent_bitwise(label):
    """normalize = 0, vf_coef = 0, ent_coef = 0, advantage 0 everywhere except sample j, which appears once in idx.
    Every other sample then contributes exact zeros (A = 0 takes the tie branch with g = 0), so the gradient must have
    the same bits wherever j sits: first / last sample of a tile, first tile of the grid's second pass, last tile of the
    busiest CTA, last sample.  It must also be the fp64 single-sample gradient / mb within _grad_bound (one sample:
    no accumulation beyond the 3 MMAs of its product).  A dropped, duplicated or misplaced sample fails outright."""
    od, S = 8, 2 ** 18 + 4096
    mb = _placement_mb(label)
    P, obs, act, lpo, adv, ret = _grad_data(od, S, seed=11)
    with torch.no_grad():  # j: a sample whose ratio is inside the clip range, so that its gradient is not zero
        B = _blocks(P.double(), od)
        tail = torch.arange(S - 64, S, device="cuda")
        mean = _tower64(B, "pi", obs[tail].double())[2]
        ratio = torch.exp((-0.5 * ((act[tail].double() - mean) / B["log_std"].exp()) ** 2 - B["log_std"] - LOG_SQRT_2PI).sum(-1) - lpo[tail].double())
        j = int(tail[torch.nonzero((ratio - 1).abs() < 0.15)[-1, 0]])
    adv = torch.zeros_like(adv)
    adv[j] = 1.7
    filler = torch.randperm(S - 1, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))[:mb]
    filler = filler + (filler >= j).long()    # every sample but j
    ref = None
    for p in _placement_positions(mb):
        idx = filler.clone()
        idx[p] = j
        grad, _ = _kernel_grad(od, P, obs, act, lpo, adv, ret, idx, 0.2, 0.0, 0.0, 0)
        if ref is None:
            ref = grad
            assert bool(grad.abs().max() > 0)
        else:
            assert torch.equal(grad.view(torch.int32), ref.view(torch.int32)), (mb, p)
    one = torch.tensor([j], device="cuda")
    x, a64, l64_, adv64, ret64 = obs[one].double(), act[one].double(), lpo[one].double(), adv[one].double(), ret[one].double()
    g64, _ = _sb3_grad64(od, P, x, a64, l64_, adv64, ret64, 0.2, 0.0, 0.0, 0, divisor=mb)
    tol, _ = _grad_bound(od, P, x, a64, l64_, adv64, ret64, 0.2, 0.0, 0.0, 0, mb, 3)
    err = (ref.double() - g64).abs()
    _report(f"grad single sample mb={mb}", err.cpu().numpy(), tol.cpu().numpy())
    assert bool((err <= tol).all()), (float((err - tol).max()), int(torch.argmax(err - tol)))


@pytest.mark.parametrize("kind", ["mb1", "mb2", "constant", "offset"])
def test_grad_advantage_normalisation_edges(kind):
    """Against fp64 with normalize = 1:
      mb1:      one sample keeps its raw advantage (SB3 normalises only when len(advantages) > 1);
      mb2:      the unbiased std of two samples;
      constant: every advantage equal (negative, so that the padding slots of the ragged last tile, whose advantage 0
                normalises to +3e7, would take the active branch if they were not masked): the kernel's fp64 statistics
                give A = 0 exactly, so the policy tower and log_std get exact zeros (torch fp32 would not: an fp32 mean
                of 50 000 equal values is not exact);
      offset:   1e3 + N(0, 1): fp32(mean) is off by up to 2^-24 1e3 = 6e-5 std, which _grad_bound carries in e(A)."""
    od, S = 8, 60_000
    mb = {"mb1": 1, "mb2": 2}.get(kind, 50_000)
    P, obs, act, lpo, adv, ret = _grad_data(od, S, seed=13)
    if kind == "constant":
        adv = torch.full_like(adv, -0.3)
    elif kind == "offset":
        adv = 1e3 + torch.randn(S, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2))
    idx = torch.randperm(S, device="cuda", generator=torch.Generator(device="cuda").manual_seed(4))
    if mb <= 2:  # samples inside the clip range: their policy gradient is not zero
        with torch.no_grad():
            B = _blocks(P.double(), od)
            mean = _tower64(B, "pi", obs[idx].double())[2]
            ratio = torch.exp((-0.5 * ((act[idx].double() - mean) / B["log_std"].exp()) ** 2 - B["log_std"] - LOG_SQRT_2PI).sum(-1) - lpo[idx].double())
            idx = idx[(ratio - 1).abs() < 0.15]
    idx = idx[:mb].contiguous()
    grad, loss = _kernel_grad(od, P, obs, act, lpo, adv, ret, idx, 0.2, 0.5, 0.0, 1)
    x, a64, l64_, adv64, ret64 = obs[idx].double(), act[idx].double(), lpo[idx].double(), adv[idx].double(), ret[idx].double()
    g64, l64 = _sb3_grad64(od, P, x, a64, l64_, adv64, ret64, 0.2, 0.5, 0.0, 1)
    tol, ltol = _grad_bound(od, P, x, a64, l64_, adv64, ret64, 0.2, 0.5, 0.0, 1, mb, _depth(mb))
    assert bool(torch.isfinite(grad).all()) and bool(torch.isfinite(loss).all())
    if kind == "mb1":
        assert bool(_blocks(grad, od)["pi.W2"].abs().max() > 0)   # the policy gradient is not silently zeroed
    if kind == "constant":
        B = _blocks(grad, od)
        assert all(bool((B[k] == 0).all()) for k in B if k.startswith("pi.") or k == "log_std")
        assert float(loss[0]) == 0.0
    _check_grad(f"normalisation {kind} mb={mb}", od, grad, loss, g64, l64, tol, ltol)


# ------------------------------------------------------------------------------------------------ 3. GAE, post_step
def _gae64(rew, val, done, last, gamma, lam):
    """SB3 RolloutBuffer.compute_returns_and_advantage in fp64, with the running-error bound of the kernel's fp32
    recursion: delta = r + fp32(gamma nxt) nonterm - v (3 roundings of |gamma nxt|, |r + .|, |delta|); last = delta +
    fp32(gamma lam) nonterm last (the propagated error times gamma lam, 2 roundings of |gamma lam last|, 1 of |last|);
    ret = last + v (1 rounding)."""
    T = rew.shape[0]
    adv, e_adv = np.zeros_like(rew), np.zeros_like(rew)
    a, e = np.zeros(rew.shape[1]), np.zeros(rew.shape[1])
    gl = gamma * lam
    for t in reversed(range(T)):
        nxt = last if t == T - 1 else val[t + 1]
        nt = 1.0 - done[t]
        c = rew[t] + gamma * nxt * nt
        delta = c - val[t]
        e_delta = U * (np.abs(gamma * nxt) + np.abs(c) + np.abs(delta))
        a_new = delta + gl * nt * a
        e = e_delta + gl * nt * e + U * (2 * np.abs(gl * nt * a) + np.abs(a_new))
        a = a_new
        adv[t], e_adv[t] = a, e
    ret = adv + val
    return adv, ret, e_adv, e_adv + U * np.abs(ret)


@pytest.mark.parametrize("pattern", ["none", "all", "last", "random"])
@pytest.mark.parametrize("T,N", [(2048, 1), (32, 65536), (1, 300)])
def test_gae_matches_fp64(T, N, pattern):
    L, check = _lib()
    rng = np.random.default_rng(T + N)
    rew = rng.standard_normal((T, N)).astype(np.float32)
    val = (3 * rng.standard_normal((T, N))).astype(np.float32)
    last = (3 * rng.standard_normal(N)).astype(np.float32)
    done = {"none": np.zeros((T, N)), "all": np.ones((T, N)), "random": (rng.random((T, N)) < 0.05) * 1.0,
            "last": np.concatenate([np.zeros((T - 1, N)), np.ones((1, N))])}[pattern].astype(np.float32)
    gamma, lam = np.float32(0.99), np.float32(0.95)
    dev = [torch.from_numpy(v).cuda() for v in (rew, val, done, last)]
    adv, ret = torch.full((T, N), float("nan"), device="cuda"), torch.full((T, N), float("nan"), device="cuda")
    check(L.so100_ppo_gae(*(t.data_ptr() for t in dev), T, N, float(gamma), float(lam), adv.data_ptr(), ret.data_ptr(), _st()))
    a64, r64, ea, er = _gae64(*(v.astype(np.float64) for v in (rew, val, done, last)), float(gamma), float(lam))
    da, dr = np.abs(adv.cpu().numpy() - a64), np.abs(ret.cpu().numpy() - r64)
    _report(f"gae T={T} N={N} {pattern} adv", da, ea)
    assert (da <= ea).all() and (dr <= er).all()


def test_post_step_matches_fp64():
    """n = 65 613 rows, ~1 % truncated and ~1 % terminated.  reward_out = r + gamma V(terminal_obs) on truncated rows,
    with V in fp64 and the bound of _tower_bound (value_one is fp32 FMA) plus the roundings of gamma V and r + .;
    a truncated row whose terminal observation is NaN keeps its reward bits (a non-finite bootstrap never enters
    the returns, as in the torch learner); NaN, inf or garbage on rows that were not truncated changes nothing.
    acc (fp64, accumulated onto its previous value) = the fp64 sums of the raw rewards, of ep_return and ep_len over
    finished episodes and of their count, within 5 ulp (the warp's fp32 shuffle tree)
    of each warp's sum |terms|; the episode count is exact."""
    L, check = _lib()
    od, n, gamma = 15, 65536 + 77, np.float32(0.99)
    P = _params(od, seed=21)
    rng = np.random.default_rng(5)
    r = rng.standard_normal(n).astype(np.float32)
    u = rng.random(n)
    trunc = (u < 0.01).astype(np.uint8)
    term = ((u >= 0.01) & (u < 0.02)).astype(np.uint8)
    tobs = (2 * rng.standard_normal((n, od))).astype(np.float32)
    tr_rows = np.flatnonzero(trunc)
    nan_rows = tr_rows[::7]
    tobs[nan_rows, 3] = np.nan
    other = np.flatnonzero(trunc == 0)
    tobs[other[::3]] = np.nan
    tobs[other[1::3], 0] = np.inf
    tobs[other[2::3]] = 1e30
    epr = (50 * rng.standard_normal(n)).astype(np.float32)
    epl = rng.integers(1, 10_000_000, n).astype(np.int32)
    acc0 = np.array([1.5, -2.0, 3.0, 4.0])
    dev = {k: torch.from_numpy(v).cuda() for k, v in dict(r=r, term=term, trunc=trunc, tobs=tobs, epr=epr, epl=epl, acc=acc0).items()}
    ro, do = torch.full((n,), float("nan"), device="cuda"), torch.full((n,), float("nan"), device="cuda")
    check(L.so100_ppo_post_step(od, P.cuda().data_ptr(), n, dev["r"].data_ptr(), dev["term"].data_ptr(), dev["trunc"].data_ptr(),
                                dev["tobs"].data_ptr(), dev["epr"].data_ptr(), dev["epl"].data_ptr(), float(gamma), ro.data_ptr(),
                                do.data_ptr(), dev["acc"].data_ptr(), _st()))
    ro, do, acc = ro.cpu().numpy(), do.cpu().numpy(), dev["acc"].cpu().numpy()
    done = (trunc | term).astype(bool)
    assert np.array_equal(do, done.astype(np.float32))
    boot_rows = np.setdiff1d(tr_rows, nan_rows)
    assert boot_rows.size > 300 and nan_rows.size > 50
    keep = np.setdiff1d(np.arange(n), boot_rows)
    assert np.array_equal(ro[keep].view(np.int32), r[keep].view(np.int32))
    B = _blocks(P.double().cuda(), od)
    x = torch.from_numpy(tobs[boot_rows]).cuda().double()
    h1, h2, v = _tower64(B, "vf", x)
    ev = _tower_bound(B, "vf", x, h1, h2)[2][:, 0].cpu().numpy()
    v = v[:, 0].cpu().numpy()
    g = float(gamma)
    want = r[boot_rows] + g * v
    tol = g * ev + U * np.abs(g * v) + U * np.abs(want)
    err = np.abs(ro[boot_rows] - want)
    _report("post_step bootstrap", err, tol)
    assert (err <= tol).all()
    # acc: per-warp fp32 tree sums (5 levels), fp64 across warps and blocks
    cols = [r.astype(np.float64), np.where(done, epr, 0).astype(np.float64), np.where(done, epl, 0).astype(np.float64), done * 1.0]
    pad = (-n) % 32
    for k, c in enumerate(cols):
        want_k = acc0[k] + c.sum()
        bound = 5 * U * np.abs(np.concatenate([c, np.zeros(pad)])).reshape(-1, 32).sum(1).sum()
        _report(f"post_step acc[{k}]", [abs(acc[k] - want_k)], [bound])
        assert abs(acc[k] - want_k) <= bound + 4 * np.spacing(abs(want_k)), (k, acc[k], want_k, bound)
    assert acc[3] == acc0[3] + done.sum()


# ------------------------------------------------------------------------------------------------ 3. Adam
def _adam_step64(p, m, v, grad, t, gscale, max_norm, lr, b1, b2, eps):
    """One clip_grad_norm_ + Adam step in fp64 from the kernel's own state (so errors do not compound), and a bound
    of |kernel - fp64| for p, m, v:
      norm: fp32 sum of squares along a chain of ceil(n / 1024) + 5 + 32 additions, plus the square's rounding ->
            relative e(s); e(norm) = e(s) / 2 + 1 ulp; clip coefficient max / (norm + 1e-6): + 2 ulp;  g = grad coef: 2 ulp;
      m, v: 3 and 4 roundings of their terms, plus the propagated e(g);
      bias corrections 1 - powf(b, t): 4 ulp of b^t, which is relative 4 ulp b^t / (1 - b^t) (large at t = 1);
      step = lr / bc1 m / (sqrtf(v) rsqrtf(bc2) + eps): e(sqrt v) = min(e(v) / 2 sqrt(v), sqrt(e(v))) + 1 ulp, rsqrtf 2 ulp,
            2 more roundings;  p - step: one ulp of p."""
    g = grad * gscale
    n = g.numel()
    s = (g * g).sum()
    norm = s.sqrt()
    depth = -(-n // 1024) + 5 + 32
    e_norm_rel = 0.5 * (depth + 2) * U + U
    if max_norm > 0:
        coef = torch.clamp(max_norm / (norm + 1e-6), max=1.0)
        e_coef_rel = (e_norm_rel + 2 * U) if bool(coef < 1) else 0.0
    else:
        coef, e_coef_rel = torch.ones((), dtype=torch.float64, device=g.device), 0.0
    g = g * coef
    e_g = g.abs() * (e_coef_rel + 2 * U)
    m1 = b1 * m + (1 - b1) * g
    e_m = 3 * U * (b1 * m.abs() + (1 - b1) * g.abs()) + (1 - b1) * e_g
    v1 = b2 * v + (1 - b2) * g * g
    e_v = 4 * U * (b2 * v + (1 - b2) * g * g) + (1 - b2) * 2 * g.abs() * e_g
    pw1, pw2 = b1 ** t, b2 ** t
    bc1, bc2 = 1 - pw1, 1 - pw2
    e_bc1, e_bc2 = (4 * U * pw1 + U * bc1) / bc1, (4 * U * pw2 + U * bc2) / bc2
    ss = lr / bc1
    sq = v1.sqrt()
    e_sq = torch.minimum(0.5 * e_v / sq.clamp_min(1e-300), e_v.sqrt()) + U * sq
    rs = 1.0 / math.sqrt(bc2)
    denom = sq * rs + eps
    e_den = e_sq * rs + sq * rs * (0.5 * e_bc2 + 3 * U) + U * denom
    step = ss * m1 / denom
    e_step = step.abs() * (e_bc1 + U + e_den / denom + 2 * U) + ss * e_m / denom
    p1 = p - step
    return p1, m1, v1, e_step + U * p1.abs(), e_m, e_v


@pytest.mark.parametrize("max_norm,gscale", [(0.5, 1.0), (0.5, 0.125), (0.0, 1.0)])
@pytest.mark.parametrize("n", [1, 1023, 1025, 9933, 10829])
def test_adam_matches_fp64_clip_and_adam(n, max_norm, gscale):
    """300 steps, then 50 more resumed at step_count = 10 000; gradients alternate below and above the clip threshold
    (max_norm 0.5); gscale 1/8 is applied to sums of 8 gradients (the all-reduce of 8 ranks); max_norm 0 is "no
    clipping".  Each step is compared with an fp64 step from the kernel's previous state: the parameter change
    relative to lr, and the moments, within _adam_step64's bound."""
    L, check = _lib()
    lr, b1, b2, eps = 3e-4, 0.9, 0.999, 1e-5
    b1_, b2_, eps_ = (float(np.float32(x)) for x in (b1, b2, eps))   # the fp32 values the kernel receives
    g = torch.Generator(device="cuda").manual_seed(n)
    p = torch.randn(n, device="cuda", generator=g)
    m, v = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    step = torch.zeros(1, device="cuda", dtype=torch.int32)
    ratios, clipped = [], []
    thr = 0.5 / math.sqrt(n)
    for k in range(350):
        if k == 300:
            step.fill_(10_000)
        t = int(step.item()) + 1 if k in (0, 300) else t + 1
        scale = thr * (0.3, 3.0, 30.0, 0.9)[k % 4]
        if gscale == 1.0:
            grad = torch.randn(n, device="cuda", generator=g) * scale
        else:
            grad = (torch.randn(8, n, device="cuda", generator=g) * scale / math.sqrt(8)).sum(0) / float(gscale) * 0.125 * 8
        p0, m0, v0 = p.double(), m.double(), v.double()
        check(L.so100_ppo_adam(n, p.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), step.data_ptr(), gscale, max_norm, lr, b1, b2, eps, _st()))
        p1, m1, v1, ep, em, ev = _adam_step64(p0, m0, v0, grad.double(), t, gscale, max_norm, float(np.float32(lr)), b1_, b2_, eps_)
        ratios.append(torch.stack([((p.double() - p1).abs() / ep).max(), ((m.double() - m1).abs() / em.clamp_min(1e-300)).max(),
                                   ((v.double() - v1).abs() / ev.clamp_min(1e-300)).max(), ((p.double() - p1).abs() / lr).max(), (ep / lr).max()]))
        clipped.append(bool(max_norm > 0) and float((grad.double() * gscale).norm()) > max_norm)
    r = torch.stack(ratios).cpu().numpy()
    print(f"[fp64] adam n={n} max_norm={max_norm} gscale={gscale}: max |dp err| / lr {r[:, 3].max():.3e}  max bound / lr {r[:, 4].max():.3e}"
          f"  max err/bound p {r[:, 0].max():.3e} m {r[:, 1].max():.3e} v {r[:, 2].max():.3e}")
    bad = np.argwhere(r[:, :3] > 1.0)
    assert bad.size == 0, (bad[:5].tolist(), r[bad[0][0]].tolist())
    assert int(step.item()) == 10_050
    if max_norm > 0 and n > 1:
        assert any(clipped) and not all(clipped)
