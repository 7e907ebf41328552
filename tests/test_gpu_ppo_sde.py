"""gSDE entry points of the fused PPO learner (so100_ppo_sde_act, so100_ppo_sde_grad; include/so100_ppo.h) against
float64 restatements of SB3's StateDependentNoiseDistribution, and the learners and CLI built on them.

Tolerances are running-error bounds of the kernels' fp32 computation in the units of test_gpu_ppo_fp64.py (U = 2^-23,
EPS_3XTF32, the CUDA math library's ulp figures), evaluated element by element from the fp64 magnitudes:
  h (the policy tower's h2) carries _tower_bound's e2;  std = expf(log_std), S = expf(2 log_std): 2 ulp each;
  z: 2.5 ulp of its Box-Muller radius (box_muller_ref.noise_tolerance);  E = fl(std z): one more rounding;
  noise and var: four fp32 FMA chains of 16 terms and 3 additions: 20 ulp of the sum of |terms|.
The bounds are worst cases dominated by the forward pass's (test_gpu_ppo_fp64.py); measured on an NVIDIA B200 (1000 W
power limit), observed / bound is at most ~2e-3 for the noise and the log-prob and ~5e-4 for the gradient.  A wrong draw,
key, feature or sample gives errors of order one; the bitwise tests (keys, env_offset splits, placements) pin the rest.
"""
import math
import os
import subprocess
import sys

import numpy as np
import pytest

from sde_ref import sde_z_host
from test_gpu_ppo_fp64 import EPS_3XTF32, U, _c, _depth, _report, _sms, _st, _tower64, _tower_bound  # noqa: F401

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

LOG_SQRT_2PI = 0.5 * math.log(2.0 * math.pi)
SDE_EPS = 1e-6
GT = 32
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    from so100_mujoco_rl_b200 import _native
    return _native.lib(), _native.check


def _sde_params(od, seed, log_std_init=-1.0):
    """A gSDE policy away from the initialisation (every path carries signal), packed as the kernels read it."""
    from so100_mujoco_rl_b200.ppo import MlpPolicy, pack_params
    torch.manual_seed(seed)
    p = MlpPolicy(od, 6, log_std_init=log_std_init, use_sde=True)
    with torch.no_grad():
        for t in p.parameters():
            t.add_(0.1 * torch.randn_like(t))
        p.log_std.add_(0.3 * torch.randn(64, 6))
    return pack_params(p)


def _plain_of(P_sde):
    """The plain layout with the same towers (every offset before log_std is shared) and some log_std[6]."""
    return torch.cat([P_sde[:-384], torch.linspace(-0.5, 0.3, 6)])


def _blocks(flat, od, use_sde=True):
    from so100_mujoco_rl_b200.ppo import param_layout
    out, o = {}, 0
    for name, shape in param_layout(od, use_sde=use_sde):
        k = int(np.prod(shape))
        out[name] = flat[o:o + k].view(shape)
        o += k
    assert o == flat.numel()
    return out


# ------------------------------------------------------------------------------------------------ 1. so100_ppo_sde_act
ACT_OD = (1, 8, 15, 16)
ACT_N = (1, 127, 129, 65536)
KEY = 0xA5A5
_CHILD = r"""
import sys
import numpy as np
import torch
root, inp, outp = sys.argv[1:4]
sys.path.insert(0, root)
from so100_mujoco_rl_b200 import _native
L = _native.lib()
st = torch.cuda.current_stream().cuda_stream
src = np.load(inp)
out = {}


def run(fn, od, P, obs, n, seed, off, key, det):
    f = dict(device="cuda", dtype=torch.float32)
    res = [torch.full((n, 6), float("nan"), **f), torch.full((n, 6), float("nan"), **f), torch.full((n,), float("nan"), **f),
           torch.full((n,), float("nan"), **f), torch.full((n, od), float("nan"), **f)]
    _native.check(fn(od, P.data_ptr(), obs.data_ptr(), n, seed, off, key, det, *(t.data_ptr() for t in res), st))
    return [t.cpu().numpy() for t in res]


for case in src["keys"]:
    od, n, seed, off, key = (int(x) for x in src[case + "__meta"])
    P, Pp, obs = (torch.from_numpy(src[case + s]).cuda() for s in ("__P", "__Pplain", "__obs"))
    runs = {"plain_det": run(L.so100_ppo_act, od, Pp, obs, n, seed, off, 77, 1),
            "det": run(L.so100_ppo_sde_act, od, P, obs, n, seed, off, key, 1),
            "sto": run(L.so100_ppo_sde_act, od, P, obs, n, seed, off, key, 0),
            "rep": run(L.so100_ppo_sde_act, od, P, obs, n, seed, off, key, 0),
            "other": run(L.so100_ppo_sde_act, od, P, obs, n, seed, off, key + 1, 0)}
    c = max(1, n // 3)   # three env_offset ranges
    parts = [run(L.so100_ppo_sde_act, od, P, obs[c0:c0 + c].contiguous(), min(c, n - c0), seed, off + c0, key, 0) for c0 in range(0, n, c)]
    runs["split"] = [np.concatenate([p[i] for p in parts]) for i in range(5)]
    for tag, r in runs.items():
        for name, arr in zip(("a", "c", "lp", "v", "oc"), r):
            out[case + "__" + tag + "__" + name] = arr
torch.cuda.synchronize()
np.savez(outp, **out)
"""


@pytest.fixture(scope="module")
def sde_runs(tmp_path_factory):
    """Both inference kernels on every (obs_dim, n) case.  SO100_PPO_ACT_MMA is read once per process: one child each."""
    d = tmp_path_factory.mktemp("sde_act")
    inputs, keys = {}, []
    for od in ACT_OD:
        P = _sde_params(od, seed=200 + od)
        for i, n in enumerate(ACT_N):
            case = f"{od}_{n}"
            rng = np.random.default_rng(31 * od + i)
            inputs[case + "__P"], inputs[case + "__Pplain"] = P.numpy(), _plain_of(P).numpy()
            inputs[case + "__obs"] = (2.0 * rng.standard_normal((n, od))).astype(np.float32)
            inputs[case + "__meta"] = np.array([od, n, 0x5DE00000 + od, 4321 + 7 * i, KEY + i], dtype=np.int64)
            keys.append(case)
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
        subprocess.run([sys.executable, "-c", _CHILD, ROOT, inp, outp], check=True, env=env, timeout=900)
        res[path] = dict(np.load(outp))
    return inputs, res


def _case(sde_runs, path, od, n):
    inputs, res = sde_runs
    case = f"{od}_{n}"
    _, _, seed, off, key = (int(x) for x in inputs[case + "__meta"])
    got = {k[len(case) + 2:]: v for k, v in res[path].items() if k.startswith(case + "__")}
    return inputs[case + "__P"], inputs[case + "__obs"], seed, off, key, got


@pytest.mark.parametrize("n", ACT_N)
@pytest.mark.parametrize("od", ACT_OD)
@pytest.mark.parametrize("path", ["tc", "mma"])
def test_sde_deterministic_equals_plain_act_bitwise(sde_runs, path, od, n):
    """deterministic = 1: act_raw (the mean), act_clip, value and obs_copy have so100_ppo_act's bits on the same towers;
    the stochastic calls return the same value and obs_copy bits, and act_clip = clip(act_raw)."""
    P, obs, seed, off, key, got = _case(sde_runs, path, od, n)
    for name in ("a", "c", "v", "oc"):
        assert np.array_equal(got["det__" + name].view(np.int32), got["plain_det__" + name].view(np.int32)), name
    for tag in ("sto", "other", "split"):
        assert np.array_equal(got[tag + "__v"].view(np.int32), got["det__v"].view(np.int32))
        assert np.array_equal(got[tag + "__oc"].view(np.int32), obs.view(np.int32))
        assert np.array_equal(got[tag + "__c"].view(np.int32), np.clip(got[tag + "__a"], -1.0, 1.0).view(np.int32))


def _h64(P, obs, od):
    B = _blocks(torch.from_numpy(P).cuda().double(), od)
    x = torch.from_numpy(obs).cuda().double()
    h1, h2, _ = _tower64(B, "pi", x)
    e2 = _tower_bound(B, "pi", x, h1, h2)[1]
    return h2.cpu().numpy(), e2.cpu().numpy(), B["log_std"].cpu().numpy()


def _logp_bound(d, var, e_var):
    """|kernel - fp64| of sum_j [-d^2 / 2v - log(v) / 2 - log sqrt(2 pi)], v = var + 1e-6, at the kernel's own (a, mean)
    (d exact in fp64): r_v = e(var) / v + 1 ulp;  d^2 / v: r_v + 5 ulp;  logf: 1 ulp, and r_v / 2 through the log;
    24 roundings of partial sums."""
    v = var + SDE_EPS
    r_v = e_var / v + U
    q, lg = 0.5 * d * d / v, 0.5 * np.log(v)
    return np.sum(q * (r_v + 5 * U) + 0.5 * r_v + 2 * U * np.abs(lg), -1) + 24 * U * np.sum(q + np.abs(lg) + LOG_SQRT_2PI, -1)


def _var_bound(h, e2, S):
    """var = sum_k fl(h_k^2) S_kj: the input error 2 |h| e2 + e2^2, S's 2 ulp, h^2's rounding and the chains' 20 ulp."""
    return (2 * np.abs(h) * e2 + e2 * e2) @ S + 23 * U * ((h * h) @ S)


def _pick(n):
    c = 2 * _sms() * 128
    return np.array(sorted({g for g in list(np.linspace(0, n - 1, 40).astype(int)) + [0, 1, 63, 64, 127, 128, c - 1, c, n - 1] if 0 <= g < n}))


@pytest.mark.parametrize("n", ACT_N)
@pytest.mark.parametrize("od", [8, 16])
@pytest.mark.parametrize("path", ["tc", "mma"])
def test_sde_noise_is_h_times_the_documented_draw(sde_runs, path, od, n):
    """act_raw - mean against the fp64 h E with E = exp(log_std) z rebuilt on the host from the header's draw layout,
    within (per action j)  sum_k e2_k |E_kj| + sum_k |h_k| std_kj (5 ulp rad + 3 ulp |z|) + 20 ulp sum_k |h_k E_kj| +
    1 ulp |a| (the rounding of mean + noise).  The log-prob of the stochastic and of the deterministic call against the fp64
    gSDE log-prob at the kernel's own (action, mean), within _logp_bound."""
    P, obs, seed, off, key, got = _case(sde_runs, path, od, n)
    h, e2, ls = _h64(P, obs, od)
    std, S = np.exp(ls), np.exp(2 * ls)
    var = (h * h) @ S
    e_var = _var_bound(h, e2, S)
    worst = worst_lp = 0.0
    for g in _pick(n):
        z, rad = sde_z_host(seed, int(off + g) & 0xFFFFFFFF, key)
        E = std * z
        noise64 = h[g] @ E
        a, m = got["sto__a"][g].astype(np.float64), got["det__a"][g].astype(np.float64)
        tol = e2[g] @ np.abs(E) + np.abs(h[g]) @ (std * (5 * U * rad + 3 * U * np.abs(z))) + 20 * U * (np.abs(h[g]) @ np.abs(E)) + U * np.abs(a)
        err = np.abs((a - m) - noise64)
        worst = max(worst, float(np.max(err / tol)))
        assert (err <= tol).all(), (g, a - m, noise64, tol)
        lp64 = np.sum(-0.5 * (a - m) ** 2 / (var[g] + SDE_EPS) - 0.5 * np.log(var[g] + SDE_EPS) - LOG_SQRT_2PI)
        e_lp = _logp_bound(a - m, var[g], e_var[g])
        worst_lp = max(worst_lp, abs(float(got["sto__lp"][g]) - lp64) / e_lp)
        assert abs(float(got["sto__lp"][g]) - lp64) <= e_lp, (g, got["sto__lp"][g], lp64, e_lp)
    lp_det64 = np.sum(-0.5 * np.log(var + SDE_EPS) - LOG_SQRT_2PI, -1)
    e_det = _logp_bound(np.zeros_like(var), var, e_var)
    assert (np.abs(got["det__lp"] - lp_det64) <= e_det).all()
    print(f"[fp64] sde noise {path} od={od} n={n}: max err/bound noise {worst:.3e}, log-prob {worst_lp:.3e}")


@pytest.mark.parametrize("od", ACT_OD)
def test_sde_tc_and_mma_paths_agree(sde_runs, od):
    """The two inference kernels draw the same E: their noises (act_raw - mean) differ by no more than twice the part of
    the noise bound that does not cancel between them (h's error and the chains' rounding, with |z| < 5.8 for every 24-bit
    uniform) plus the rounding of each mean + noise; their log-probs by their two _logp_bound plus what the noise
    difference moves d^2 / 2v."""
    n = 65536
    P, obs, seed, off, key, tc = _case(sde_runs, "tc", od, n)
    mma = _case(sde_runs, "mma", od, n)[5]
    h, e2, ls = _h64(P, obs, od)
    E_max = np.exp(ls) * 5.8
    n_tc, n_mma = (r["sto__a"].astype(np.float64) - r["det__a"] for r in (tc, mma))
    tol = 2 * (e2 @ E_max + 20 * U * (np.abs(h) @ E_max)) + U * (np.abs(tc["sto__a"]) + np.abs(mma["sto__a"]))
    dn = np.abs(n_tc - n_mma)
    _report(f"sde tc vs mma noise od={od}", dn, tol)
    assert (dn <= tol).all()
    S = np.exp(2 * ls)
    var, e_var = (h * h) @ S, _var_bound(h, e2, S)
    slack = np.sum((np.abs(n_tc) + 0.5 * dn) * dn / (var + SDE_EPS), -1)
    dlp = np.abs(tc["sto__lp"].astype(np.float64) - mma["sto__lp"])
    assert (dlp <= _logp_bound(n_tc, var, e_var) + _logp_bound(n_mma, var, e_var) + slack).all()


@pytest.mark.parametrize("od", ACT_OD)
@pytest.mark.parametrize("path", ["tc", "mma"])
def test_sde_keys_repeat_differ_and_split_by_env_offset(sde_runs, path, od):
    """The same noise key gives the same bits on a repeat call; another key other noise; a call split into three
    env_offset ranges the single call's bits on every output."""
    for n in ACT_N:
        got = _case(sde_runs, path, od, n)[5]
        for name in ("a", "c", "lp", "v", "oc"):
            assert np.array_equal(got["rep__" + name].view(np.int32), got["sto__" + name].view(np.int32)), (n, name)
            assert np.array_equal(got["split__" + name].view(np.int32), got["sto__" + name].view(np.int32)), (n, name)
        assert (got["other__a"] != got["sto__a"]).mean() > 0.99


def test_sde_noise_is_standard_normal_over_a_million_samples():
    """(a - mean)_j / sqrt(var_j), var from the fp64 h, over 2^20 envs with varied observations and log_std: six KS tests
    against N(0, 1), and the standardised noise of different actions of one env is uncorrelated."""
    from scipy import stats
    L, check = _lib()
    od, n = 15, 2 ** 20
    P = _sde_params(od, seed=5, log_std_init=-1.5).cuda()
    obs = 2.0 * torch.randn(n, od, device="cuda", generator=torch.Generator(device="cuda").manual_seed(9))
    a, m = torch.empty(n, 6, device="cuda"), torch.empty(n, 6, device="cuda")
    check(L.so100_ppo_sde_act(od, P.data_ptr(), obs.data_ptr(), n, 99, 0, 3, 0, a.data_ptr(), None, None, None, None, _st()))
    check(L.so100_ppo_sde_act(od, P.data_ptr(), obs.data_ptr(), n, 99, 0, 3, 1, m.data_ptr(), None, None, None, None, _st()))
    B = _blocks(P.double(), od)
    h = _tower64(B, "pi", obs.double())[1]
    var = (h * h) @ torch.exp(2 * B["log_std"])
    zs = ((a.double() - m.double()) / var.sqrt()).cpu().numpy()
    for j in range(6):
        p = stats.kstest(zs[:, j], "norm").pvalue
        print(f"[ks] action {j}: p = {p:.3f}")
        assert p > 1e-3, (j, p)
    c = np.corrcoef(zs.T)
    assert np.abs(c - np.eye(6)).max() < 5.0 / math.sqrt(n)


# ------------------------------------------------------------------------------------------------ 2. so100_ppo_sde_grad
def _grad_data(od, S, seed, clip=0.2):
    """Rollout-like buffers for a gSDE policy: actions from Normal(mean, scale(h)), old log-probs from a perturbed mean,
    nudged so that no ratio lies within 1e-4 of 1 +- clip."""
    P = _sde_params(od, seed=seed).cuda()
    g = torch.Generator(device="cuda").manual_seed(seed)
    obs = torch.randn(S, od, device="cuda", generator=g)
    B = _blocks(P.double(), od)
    with torch.no_grad():
        _, h, mean = _tower64(B, "pi", obs.double())
        var = (h * h) @ torch.exp(2 * B["log_std"]) + SDE_EPS
        act = (mean + var.sqrt() * torch.randn(S, 6, device="cuda", generator=g, dtype=torch.float64)).float()
        lp_of = lambda mu: (-0.5 * (act.double() - mu) ** 2 / var - 0.5 * torch.log(var) - LOG_SQRT_2PI).sum(-1)  # noqa: E731
        logp_old = lp_of(mean + 0.15 * var.sqrt() * torch.randn(S, 6, device="cuda", generator=g, dtype=torch.float64)).float()
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
    ws = torch.zeros(int(L.so100_ppo_sde_workspace_floats(od)), device="cuda")
    grad, loss = torch.full((P.numel(),), float("nan"), device="cuda"), torch.full((3,), float("nan"), device="cuda")
    check(L.so100_ppo_sde_grad(od, P.data_ptr(), obs.data_ptr(), act.data_ptr(), logp_old.data_ptr(), adv.data_ptr(), ret.data_ptr(),
                               idx.data_ptr(), idx.numel(), clip, vf_coef, ent_coef, normalize, ws.data_ptr(), grad.data_ptr(), loss.data_ptr(), _st()))
    return grad, loss


def _sb3_sde_grad64(od, P, x, act, lpo, adv, ret, clip, vf_coef, ent_coef, normalize, divisor=None):
    """SB3 PPO.train's loss with use_sde=True for one minibatch in fp64 through autograd: the StateDependentNoiseDistribution's
    log-prob and entropy with h detached in the variance (learn_features=False)."""
    flat = P.double().clone().requires_grad_(True)
    B = _blocks(flat, od)
    a = adv
    if normalize and a.numel() > 1:
        a = (a - a.mean()) / (a.std() + 1e-8)
    _, h, mean = _tower64(B, "pi", x)
    scale = torch.sqrt((h.detach() ** 2) @ torch.exp(B["log_std"]) ** 2 + SDE_EPS)
    value = _tower64(B, "vf", x)[2][:, 0]
    logp = (-((act - mean) ** 2) / (2 * scale ** 2) - torch.log(scale) - LOG_SQRT_2PI).sum(-1)
    lr = logp - lpo
    ratio = torch.exp(lr)
    k = float(divisor or x.shape[0])
    pg = -torch.min(a * ratio, a * torch.clamp(ratio, 1 - clip, 1 + clip)).sum() / k
    vl = ((value - ret) ** 2).sum() / k
    ent = (0.5 + LOG_SQRT_2PI + torch.log(scale)).sum() / k
    (pg + vf_coef * vl - ent_coef * ent).backward()
    return flat.grad.detach(), torch.stack([pg.detach(), vl.detach(), ((ratio - 1) - lr).sum().detach() / k])


def _sde_grad_bound(od, P, x, act, lpo, adv, ret, clip, vf_coef, ent_coef, normalize, divisor, depth):
    """Element-wise bound of |kernel - fp64| (test_gpu_ppo_fp64._grad_bound with the gSDE distribution):
      var = sum_k fl(h^2) S: _var_bound; v = var + 1e-6, r_v = e(var) / v + 1 ulp;  1 / v: r_v + 1 ulp.
      log-prob: sum_j |d| e(d) / v + d^2 / 2v (r_v + 5 ulp) + r_v / 2 + 2 ulp |log v / 2|, plus 22 ulp of the terms.
      dL/dmean = dlp d / v;  dL/dvar = (dlp (d^2 / v - 1) - ent_coef / mb) / 2v, each with its inputs' errors + 6 ulp.
      d log_std_kj = 2 S_kj sum_s dvar_sj h_sk^2: the errors of dvar and of h^2 (2 |h| e2 + e2^2), S's 2 ulp, the chain."""
    B = _blocks(P.double(), od)
    m = x.shape[0]
    with torch.no_grad():
        res = {}
        h1p, h2p, mean = _tower64(B, "pi", x)
        h1v, h2v, vout = _tower64(B, "vf", x)
        e1p, e2p, em = _tower_bound(B, "pi", x, h1p, h2p)
        e1v, e2v, ev = _tower_bound(B, "vf", x, h1v, h2v)
        value, ev = vout[:, 0], ev[:, 0]
        S = torch.exp(2 * B["log_std"])
        h2sq, e_h2sq = h2p * h2p, 2 * h2p.abs() * e2p + e2p * e2p
        var = h2sq @ S
        e_var = e_h2sq @ S + 23 * U * (h2sq @ S)
        v = var + SDE_EPS
        r_v = e_var / v + U
        isig2 = 1.0 / v
        d = act - mean
        e_d = em + U * d.abs()
        lg = 0.5 * torch.log(v)
        T_lp = (0.5 * d * d * isig2 + lg.abs() + LOG_SQRT_2PI).sum(-1)
        lp = (-0.5 * d * d * isig2 - lg - LOG_SQRT_2PI).sum(-1)
        e_lp = (d.abs() * isig2 * e_d + 0.5 * d * d * isig2 * (r_v + 5 * U) + 0.5 * r_v + 2 * U * lg.abs()).sum(-1) + 22 * U * T_lp
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
        r_is = r_v + U
        dout = dlp[:, None] * d * isig2
        e_dout = e_dlp[:, None] * d.abs() * isig2 + dlp.abs()[:, None] * (e_d + d.abs() * r_is) * isig2 + 4 * U * dout.abs()
        q = d * d * isig2 - 1
        e_q = 2 * d.abs() * isig2 * e_d + d * d * isig2 * (r_is + 2 * U) + U * q.abs()
        ent = ent_coef / divisor
        dvar = 0.5 * (dlp[:, None] * q - ent) * isig2
        e_dvar = 0.5 * isig2 * (e_dlp[:, None] * q.abs() + dlp.abs()[:, None] * e_q + (dlp.abs()[:, None] * q.abs() + ent) * (r_is + 6 * U))
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
        res["log_std"] = 2 * S * ((h2sq.T @ e_dvar) + (e_h2sq.T @ dvar.abs()) + (c_s + 8 * U) * (h2sq.T @ dvar.abs()))
        from so100_mujoco_rl_b200.ppo import param_layout
        tol = torch.cat([res[name].reshape(-1) for name, _ in param_layout(od, use_sde=True)])
        pmin = torch.minimum(x1, x2).abs()
        e_pg = ((A.abs() * e_ratio + ratio * e_A + 2 * U * x1.abs()).sum() + (c_s + 2 * U) * pmin.sum()) / divisor \
            + (either * (A.abs() + e_A) * ratio * (1 + e_lr)).sum() / divisor
        e_vl = ((2 * e_v.abs() * ev + 2 * U * e_v * e_v).sum() + (c_s + 2 * U) * (e_v * e_v).sum()) / divisor
        kl = (ratio - 1) - lr
        e_kl = ((e_ratio + e_lr + 2 * U * ((ratio - 1).abs() + lr.abs())).sum() + (c_s + 2 * U) * kl.abs().sum()) / divisor
    return tol, torch.stack([e_pg, e_vl, e_kl])


def _check_grad(what, od, grad, loss, g64, l64, tol, ltol):
    from so100_mujoco_rl_b200.ppo import param_layout
    err = (grad.double() - g64).abs()
    o = 0
    for name, shape in param_layout(od, use_sde=True):
        k = int(np.prod(shape))
        e, b = err[o:o + k], tol[o:o + k]
        _report(f"sde grad {what} {name} (|g64| max {float(g64[o:o + k].abs().max()):.2e})", e.cpu().numpy(), b.cpu().numpy())
        assert bool((e <= b).all()), (name, float((e - b).max()), int(torch.argmax(e - b)))
        o += k
    lerr = (loss.double() - l64).abs()
    _report(f"sde grad {what} losses", lerr.cpu().numpy(), ltol.cpu().numpy())
    assert bool((lerr <= ltol).all()), (loss.tolist(), l64.tolist(), ltol.tolist())


GRAD_MB = (1, 31, 33, 4096, 262144)


@pytest.mark.parametrize("ent_coef", [0.0, 0.01])
@pytest.mark.parametrize("normalize", [1, 0])
@pytest.mark.parametrize("mb", GRAD_MB)
def test_sde_grad_matches_fp64_autograd(mb, normalize, ent_coef):
    """Every parameter block (the [64, 6] log_std included) and the three losses within _sde_grad_bound of the fp64 autograd
    of SB3's gSDE loss; the result is bit-identical on a rerun."""
    od, S = 8, (2 ** 21 if mb > 4096 else 60_000)
    P, obs, act, lpo, adv, ret = _grad_data(od, S, seed=17 + mb)
    idx = torch.randperm(S, device="cuda", generator=torch.Generator(device="cuda").manual_seed(mb))[:mb].contiguous()
    grad, loss = _kernel_grad(od, P, obs, act, lpo, adv, ret, idx, 0.2, 0.5, ent_coef, normalize)
    grad2, loss2 = _kernel_grad(od, P, obs, act, lpo, adv, ret, idx, 0.2, 0.5, ent_coef, normalize)
    assert torch.equal(grad.view(torch.int32), grad2.view(torch.int32)) and torch.equal(loss.view(torch.int32), loss2.view(torch.int32))
    x, a64, l64_, adv64, ret64 = obs[idx].double(), act[idx].double(), lpo[idx].double(), adv[idx].double(), ret[idx].double()
    g64, l64 = _sb3_sde_grad64(od, P, x, a64, l64_, adv64, ret64, 0.2, 0.5, ent_coef, normalize)
    tol, ltol = _sde_grad_bound(od, P, x, a64, l64_, adv64, ret64, 0.2, 0.5, ent_coef, normalize, mb, _depth(mb))
    assert bool(torch.isfinite(grad).all())
    if mb >= 4096:
        assert float(_blocks(grad, od)["log_std"].abs().max()) > 0
    _check_grad(f"mb={mb} norm={normalize} ent={ent_coef}", od, grad, loss, g64, l64, tol, ltol)


@pytest.mark.parametrize("mb", [33, 2 * 148 * GT + 1, 262144])
def test_sde_grad_single_sample_is_placement_independent_bitwise(mb):
    """normalize = 0, vf_coef = 0, ent_coef = 0 and a zero advantage everywhere but sample j: every other sample adds exact
    zeros (to dL/dmean and to dL/dvar), so the gradient has the same bits wherever j sits in the minibatch, and it is the
    fp64 single-sample gradient / mb within the bound."""
    od, S = 8, 2 ** 18 + 4096
    P, obs, act, lpo, adv, ret = _grad_data(od, S, seed=23)
    with torch.no_grad():
        B = _blocks(P.double(), od)
        tail = torch.arange(S - 64, S, device="cuda")
        _, h, mean = _tower64(B, "pi", obs[tail].double())
        var = (h * h) @ torch.exp(2 * B["log_std"]) + SDE_EPS
        ratio = torch.exp((-0.5 * (act[tail].double() - mean) ** 2 / var - 0.5 * torch.log(var) - LOG_SQRT_2PI).sum(-1) - lpo[tail].double())
        j = int(tail[torch.nonzero((ratio - 1).abs() < 0.15)[-1, 0]])
    adv = torch.zeros_like(adv)
    adv[j] = 1.7
    filler = torch.randperm(S - 1, device="cuda", generator=torch.Generator(device="cuda").manual_seed(3))[:mb]
    filler = filler + (filler >= j).long()
    ntiles = (mb + GT - 1) // GT
    grid = min(ntiles, 2 * _sms())
    positions = sorted({p for p in (0, 31, 32, mb - 1, grid * GT, ((ntiles - 1) // grid) * grid * GT) if 0 <= p < mb})
    ref = None
    for p in positions:
        idx = filler.clone()
        idx[p] = j
        grad, _ = _kernel_grad(od, P, obs, act, lpo, adv, ret, idx, 0.2, 0.0, 0.0, 0)
        if ref is None:
            ref = grad
            assert float(_blocks(grad, od)["log_std"].abs().max()) > 0
        else:
            assert torch.equal(grad.view(torch.int32), ref.view(torch.int32)), (mb, p)
    one = torch.tensor([j], device="cuda")
    x, a64, l64_, adv64, ret64 = obs[one].double(), act[one].double(), lpo[one].double(), adv[one].double(), ret[one].double()
    g64, _ = _sb3_sde_grad64(od, P, x, a64, l64_, adv64, ret64, 0.2, 0.0, 0.0, 0, divisor=mb)
    tol, _ = _sde_grad_bound(od, P, x, a64, l64_, adv64, ret64, 0.2, 0.0, 0.0, 0, mb, 3)
    err = (ref.double() - g64).abs()
    _report(f"sde grad single sample mb={mb}", err.cpu().numpy(), tol.cpu().numpy())
    assert bool((err <= tol).all()), (float((err - tol).max()), int(torch.argmax(err - tol)))


# ------------------------------------------------------------------------------------------------ 3. learners and CLI
def test_fused_sde_tracks_the_torch_learner_and_learns():
    """FusedPPO(use_sde) and PPO(use_sde) start from identical weights; one fused minibatch step equals the torch step on
    the fused rollout; a short Env01 run improves the per-step reward."""
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    from so100_mujoco_rl_b200.ppo import PPO, FusedPPO, PPOConfig, pack_params
    cfg = PPOConfig(n_steps=16, n_minibatches=4, n_epochs=4, seed=0, cuda_graph=False, use_sde=True, log_std_init=-2.0)
    env = BatchedSo100Env(1, 2048, device=0, seed=1)
    fused = FusedPPO(env, cfg)
    ref = PPO(BatchedSo100Env(1, 2048, device=0, seed=1), cfg)
    assert fused.params.numel() == 11207 and torch.equal(fused.params, pack_params(ref.policy))
    adv, ret = fused.collect()
    total = adv.numel()
    idx = torch.randperm(total, device="cuda")[: total // 4]
    flat = {k: v.view(total, *v.shape[2:]) for k, v in fused.buf.items()}
    ref._last_info = torch.zeros(3, device="cuda")
    ref._minibatch_step(idx, flat, adv.reshape(-1), ret.reshape(-1))
    fused.minibatch_step(idx, adv, ret)
    assert torch.allclose(fused.params, pack_params(ref.policy), atol=2e-6)
    assert torch.allclose(fused.loss, ref._last_info, rtol=1e-3, atol=1e-5)
    hist = []
    fused.learn(total_samples=2048 * 16 * 60, log_every=0, callback=hist.append)
    first, last = np.mean([h["mean_step_reward"] for h in hist[:3]]), np.mean([h["mean_step_reward"] for h in hist[-3:]])
    print(f"[sde learn] Env01 mean step reward {first:.4f} -> {last:.4f}")
    assert last > first + 0.2, (first, last)
    assert all(math.isfinite(h["pg_loss"]) and math.isfinite(h["log_std_mean"]) for h in hist)
    env.close()


def test_fused_sde_rollout_keys_and_state_roundtrip():
    """Within a rollout the exploration matrices stay put (freq -1) or change every sde_sample_freq steps; act() reuses the
    key in use whatever the tick; the learner state round trip resumes bit-exactly."""
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    from so100_mujoco_rl_b200.ppo import FusedPPO, PPOConfig
    cfg = PPOConfig(n_steps=8, n_minibatches=2, n_epochs=2, seed=3, use_sde=True, sde_sample_freq=4, log_std_init=-1.0)
    a = FusedPPO(BatchedSo100Env(5, 512, device=0, seed=2), cfg)
    keys = []
    orig = a._act_fn
    a._act_fn = lambda *args: (keys.append(int(args[6])), orig(*args))[1]
    a.collect()
    t0 = a.tick - 8
    assert keys == [t0 + 1] * 4 + [t0 + 5] * 4 + [a.tick]   # (the last call is the deterministic bootstrap value)
    a._act_fn = orig
    obs = torch.randn(100, a.od, device="cuda")
    x1, x2 = a.act(obs), a.act(obs)
    assert x1[0].view(torch.int32).equal(x2[0].view(torch.int32)) and a.sde_key == t0 + 5
    a.learn(total_samples=512 * 8 * 3, log_every=0, callback=lambda r: None)
    sd = a.state_dict()
    assert sd["config"]["use_sde"] and sd["config"]["sde_sample_freq"] == 4
    b = FusedPPO(BatchedSo100Env(5, 512, device=0, seed=2), cfg)
    b.load_state_dict({k: (v.cpu() if torch.is_tensor(v) else v) for k, v in sd.items()})
    assert torch.equal(a.params, b.params) and torch.equal(a.exp_avg, b.exp_avg) and b.tick == a.tick and b.sde_key == a.sde_key
    assert a.act(obs)[0].view(torch.int32).equal(b.act(obs)[0].view(torch.int32))
    for k in a.buf:
        b.buf[k].copy_(a.buf[k])
    idx = torch.randperm(a.adv.numel(), device="cuda")[:1024]
    a.minibatch_step(idx, a.adv, a.ret); b.minibatch_step(idx, a.adv, a.ret)
    assert torch.equal(a.params, b.params)


def test_cli_train_use_sde_writes_a_gsde_zip_and_evaluates(tmp_path):
    import io
    import json
    import zipfile

    from click.testing import CliRunner

    from so100_mujoco_rl_b200.cli import cli
    out = tmp_path / "models"
    r = CliRunner().invoke(cli, ["-a", "PPO", "train", "-e", "Env01", "--num-envs", "256", "--total-timesteps", str(256 * 32 * 2),
                                 "--out", str(out), "--eval-envs", "0", "--tensorboard-log", "", "--use-sde", "--sde-sample-freq", "8",
                                 "--log-std-init", "-2"], obj={})
    assert r.exit_code == 0, (r.output, r.exception)
    folder = out / "Env01_PPO"
    with zipfile.ZipFile(folder / "final_model.zip") as z:
        data = json.loads(z.read("data"))
        sd = torch.load(io.BytesIO(z.read("policy.pth")))
    assert data["use_sde"] is True and data["sde_sample_freq"] == 8 and sd["log_std"].shape == (64, 6)
    for f in ("final_model.zip", "final_model.pt"):
        e = CliRunner().invoke(cli, ["-m", str(folder / f), "test", "-e", "Env01", "--num-envs", "8", "--steps", "20"], obj={})
        assert e.exit_code == 0, (f, e.output, e.exception)
        assert math.isfinite(json.loads(e.output.strip().splitlines()[-1])["mean_return"])
    # resuming it without --use-sde is refused; with it, it continues
    bad = CliRunner().invoke(cli, ["-m", str(folder / "final_model.pt"), "train", "-e", "Env01", "--num-envs", "256", "--out", str(out)], obj={})
    assert bad.exit_code != 0 and "--use-sde" in bad.output
    ok = CliRunner().invoke(cli, ["-m", str(folder / "final_model.pt"), "train", "-e", "Env01", "--num-envs", "256", "--total-timesteps",
                                  str(256 * 32), "--out", str(out), "--eval-envs", "0", "--tensorboard-log", "", "--use-sde"], obj={})
    assert ok.exit_code == 0, (ok.output, ok.exception)
