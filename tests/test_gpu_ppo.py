"""Fused PPO kernels (include/so100_ppo.h, through the C ABI) against the plain PyTorch fp32 reference of the same ops:
rollout inference, TimeLimit bootstrap, GAE, the minibatch gradient (autograd of the SB3 loss) and clip + Adam.

Tolerances are fp32 re-association only: the kernels and torch compute the same fp32 formulas in different orders.
"""
import math

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu


def _lib():
    from so100_mujoco_rl_b200 import _native
    return _native.lib(), _native.check


def _policy(od, seed=0, scale=1.0):
    from so100_mujoco_rl_b200.ppo import MlpPolicy
    torch.manual_seed(seed)
    p = MlpPolicy(od, 6).cuda()
    with torch.no_grad():
        for t in p.parameters():  # away from the tiny-gain initialisation so every path carries signal
            t.add_(scale * 0.1 * torch.randn_like(t))
    return p


def _st():
    return torch.cuda.current_stream().cuda_stream


@pytest.mark.parametrize("od,n", [(15, 1000), (8, 65)])
def test_act_matches_torch_forward(od, n):
    from so100_mujoco_rl_b200.ppo import pack_params
    L, check = _lib()
    pol = _policy(od)
    P = pack_params(pol)
    assert P.numel() == L.so100_ppo_param_count(od)
    obs = torch.randn(n, od, device="cuda")
    f = dict(device="cuda", dtype=torch.float32)
    a, c, lp, v, oc = torch.zeros(n, 6, **f), torch.zeros(n, 6, **f), torch.zeros(n, **f), torch.zeros(n, **f), torch.zeros(n, od, **f)
    check(L.so100_ppo_act(od, P.data_ptr(), obs.data_ptr(), n, 7, 0, 3, 0, a.data_ptr(), c.data_ptr(), lp.data_ptr(), v.data_ptr(), oc.data_ptr(), _st()))
    with torch.no_grad():
        mean, log_std = pol.dist_params(obs)
        assert torch.allclose(v, pol.value(obs), atol=2e-5)
        assert torch.allclose(lp, pol.log_prob(mean, log_std, a), atol=2e-4)      # log-prob of the action it drew
    assert torch.equal(oc, obs) and torch.equal(c, a.clamp(-1, 1))
    z = ((a - mean) / log_std.exp()).detach().flatten().cpu().numpy()                       # the noise it used is N(0, 1)
    if n >= 1000:
        assert abs(z.mean()) < 0.05 and abs(z.std() - 1) < 0.05 and abs((z ** 3).mean()) < 0.15
    # deterministic mode returns the mean; same (seed, env, tick) -> same draw; other tick -> other draw
    a2, a3, a4 = torch.zeros_like(a), torch.zeros_like(a), torch.zeros_like(a)
    check(L.so100_ppo_act(od, P.data_ptr(), obs.data_ptr(), n, 7, 0, 3, 1, a2.data_ptr(), None, None, None, None, _st()))
    check(L.so100_ppo_act(od, P.data_ptr(), obs.data_ptr(), n, 7, 0, 3, 0, a3.data_ptr(), None, None, None, None, _st()))
    check(L.so100_ppo_act(od, P.data_ptr(), obs.data_ptr(), n, 7, 0, 4, 0, a4.data_ptr(), None, None, None, None, _st()))
    assert torch.allclose(a2, mean, atol=2e-5) and torch.equal(a3, a) and not torch.equal(a4, a)
    # sharding: env_offset shifts the stream, so rank r's envs draw what a single process would draw for them
    a5 = torch.zeros(n - 10, 6, **f)
    check(L.so100_ppo_act(od, P.data_ptr(), obs[10:].contiguous().data_ptr(), n - 10, 7, 10, 3, 0, a5.data_ptr(), None, None, None, None, _st()))
    assert torch.equal(a5, a[10:])


def test_gae_and_post_step_match_torch():
    from so100_mujoco_rl_b200.ppo import compute_gae, pack_params
    L, check = _lib()
    od, T, N = 15, 9, 777
    pol = _policy(od)
    P = pack_params(pol)
    g = torch.Generator(device="cuda").manual_seed(1)
    rew, val = torch.randn(T, N, device="cuda", generator=g), torch.randn(T, N, device="cuda", generator=g)
    done = (torch.rand(T, N, device="cuda", generator=g) < 0.15).float()
    last = torch.randn(N, device="cuda", generator=g)
    adv, ret = torch.zeros_like(rew), torch.zeros_like(rew)
    check(L.so100_ppo_gae(rew.data_ptr(), val.data_ptr(), done.data_ptr(), last.data_ptr(), T, N, 0.99, 0.95, adv.data_ptr(), ret.data_ptr(), _st()))
    adv_t, ret_t = compute_gae(rew, val, done, last, 0.99, 0.95)
    assert torch.allclose(adv, adv_t, atol=2e-5) and torch.allclose(ret, ret_t, atol=2e-5)
    # post_step: bootstrap only where truncated, done = term | trunc, Monitor sums
    r = torch.randn(N, device="cuda", generator=g)
    term = (torch.rand(N, device="cuda", generator=g) < 0.1).to(torch.uint8)
    trunc = ((torch.rand(N, device="cuda", generator=g) < 0.1) & (term == 0)).to(torch.uint8)
    tobs = torch.randn(N, od, device="cuda", generator=g)
    epr, epl = torch.randn(N, device="cuda", generator=g), torch.randint(1, 4000, (N,), device="cuda", dtype=torch.int32)
    ro, do = torch.zeros(N, device="cuda"), torch.zeros(N, device="cuda")
    acc = torch.zeros(4, device="cuda", dtype=torch.float64)
    check(L.so100_ppo_post_step(od, P.data_ptr(), N, r.data_ptr(), term.data_ptr(), trunc.data_ptr(), tobs.data_ptr(), epr.data_ptr(),
                                epl.data_ptr(), 0.99, ro.data_ptr(), do.data_ptr(), acc.data_ptr(), _st()))
    with torch.no_grad():
        expect = torch.where(trunc.bool(), r + 0.99 * pol.value(tobs), r)
    d = (term | trunc).bool()
    assert torch.allclose(ro, expect, atol=2e-5) and torch.equal(do, d.float())
    assert torch.allclose(acc, torch.stack([r.double().sum(), epr[d].double().sum(), epl[d].double().sum(), d.double().sum()]), rtol=1e-6)


def _torch_minibatch_grad(pol, obs, act, logp_old, adv, ret, idx, clip, vf_coef, ent_coef, normalize):
    """SB3 PPO.train's loss for one minibatch, through autograd (stable_baselines3/ppo/ppo.py)."""
    for p in pol.parameters():
        p.grad = None
    a = adv[idx]
    if normalize and a.numel() > 1:
        a = (a - a.mean()) / (a.std() + 1e-8)
    v, logp, ent = pol.evaluate(obs[idx], act[idx])
    lr = logp - logp_old[idx]
    ratio = torch.exp(lr)
    pg = -torch.min(a * ratio, a * torch.clamp(ratio, 1 - clip, 1 + clip)).mean()
    vl = torch.nn.functional.mse_loss(v, ret[idx])
    (pg + vf_coef * vl - ent_coef * ent.mean()).backward()
    from so100_mujoco_rl_b200.ppo import _policy_tensors
    g = torch.cat([t.grad.reshape(-1) for t in _policy_tensors(pol)])
    return g, torch.stack([pg.detach(), vl.detach(), ((ratio - 1) - lr).mean().detach()])


@pytest.mark.parametrize("od,S,mb,normalize,ent_coef", [(15, 4096, 2048, 1, 0.0), (8, 3000, 1000, 1, 0.01), (15, 50000, 32768, 0, 0.0)])
def test_minibatch_gradient_matches_autograd(od, S, mb, normalize, ent_coef):
    from so100_mujoco_rl_b200.ppo import pack_params
    L, check = _lib()
    pol = _policy(od, seed=3)
    P = pack_params(pol)
    g = torch.Generator(device="cuda").manual_seed(5)
    obs = torch.randn(S, od, device="cuda", generator=g)
    with torch.no_grad():
        mean, log_std = pol.dist_params(obs)
        act = mean + log_std.exp() * torch.randn(S, 6, device="cuda", generator=g)
        # old log-probs from a perturbed policy so that ratios spread over both sides of the clip range
        logp_old = pol.log_prob(mean + 0.15 * torch.randn(S, 6, device="cuda", generator=g), log_std, act)
    adv, ret = torch.randn(S, device="cuda", generator=g) * 2 + 0.3, torch.randn(S, device="cuda", generator=g)
    idx = torch.randperm(S, device="cuda", generator=g)[:mb]
    ws = torch.zeros(int(L.so100_ppo_workspace_floats(od)), device="cuda")
    grad, loss = torch.zeros(P.numel(), device="cuda"), torch.zeros(3, device="cuda")
    check(L.so100_ppo_grad(od, P.data_ptr(), obs.data_ptr(), act.data_ptr(), logp_old.data_ptr(), adv.data_ptr(), ret.data_ptr(),
                           idx.data_ptr(), mb, 0.2, 0.5, ent_coef, normalize, ws.data_ptr(), grad.data_ptr(), loss.data_ptr(), _st()))
    gt, lt = _torch_minibatch_grad(pol, obs, act, logp_old, adv, ret, idx, 0.2, 0.5, ent_coef, bool(normalize))
    frac_clipped = float(((torch.exp(pol.log_prob(*pol.dist_params(obs[idx]), act[idx]) - logp_old[idx]) - 1).abs() > 0.2).float().mean())
    assert 0.05 < frac_clipped < 0.95                                                 # both branches of the surrogate are exercised
    err = (grad - gt).abs().max().item()
    assert err < 2e-5 * max(1.0, gt.abs().max().item()), (err, gt.abs().max().item())
    assert torch.allclose(loss, lt, rtol=2e-4, atol=2e-6)
    # deterministic: the same call gives bit-identical gradients
    grad2 = torch.zeros_like(grad)
    check(L.so100_ppo_grad(od, P.data_ptr(), obs.data_ptr(), act.data_ptr(), logp_old.data_ptr(), adv.data_ptr(), ret.data_ptr(),
                           idx.data_ptr(), mb, 0.2, 0.5, ent_coef, normalize, ws.data_ptr(), grad2.data_ptr(), loss.data_ptr(), _st()))
    assert torch.equal(grad, grad2)


def test_adam_matches_torch_clip_and_adam():
    L, check = _lib()
    n = 10829
    g = torch.Generator(device="cuda").manual_seed(2)
    p0 = torch.randn(n, device="cuda", generator=g)
    p_t = torch.nn.Parameter(p0.clone())
    opt = torch.optim.Adam([p_t], lr=3e-4, eps=1e-5)
    p, m, v = p0.clone(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    step = torch.zeros(1, device="cuda", dtype=torch.int32)
    for k in range(5):
        grad = torch.randn(n, device="cuda", generator=g) * (0.001 if k == 2 else 0.05)  # step 2 is below the clip threshold
        p_t.grad = grad.clone()
        torch.nn.utils.clip_grad_norm_([p_t], 0.5)
        opt.step()
        check(L.so100_ppo_adam(n, p.data_ptr(), grad.data_ptr(), m.data_ptr(), v.data_ptr(), step.data_ptr(), 1.0, 0.5, 3e-4, 0.9, 0.999, 1e-5, _st()))
        assert torch.allclose(p, p_t.detach(), atol=1e-6), k
    assert int(step.item()) == 5


def test_fused_ppo_tracks_the_torch_learner_and_learns():
    """Same seed, same env seed: the first update of FusedPPO and of the torch PPO start from identical weights; after
    training the fused learner must have improved Env01's per-step reward like the torch one does."""
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    from so100_mujoco_rl_b200.ppo import PPO, FusedPPO, PPOConfig, pack_params
    cfg = PPOConfig(n_steps=16, n_minibatches=4, n_epochs=4, seed=0, cuda_graph=False)
    env = BatchedSo100Env(1, 2048, device=0, seed=1)
    fused = FusedPPO(env, cfg)
    ref = PPO(BatchedSo100Env(1, 2048, device=0, seed=1), cfg)
    assert torch.equal(fused.params, pack_params(ref.policy))
    # one fused minibatch step == one torch minibatch step on the fused learner's own rollout
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
    assert last > first + 0.2, (first, last)
    assert all(math.isfinite(h["pg_loss"]) and math.isfinite(h["v_loss"]) for h in hist)
    env.close()


@pytest.mark.parametrize("n", [1, 2, 3, 1000, 4096, 65536, 65537, 2 ** 20 - 1, 65536 * 32 + 17])
def test_permutation_is_a_bijection_and_depends_on_the_key(n):
    L, check = _lib()
    a, b = torch.zeros(n, dtype=torch.int64, device="cuda"), torch.zeros(n, dtype=torch.int64, device="cuda")
    check(L.so100_ppo_permutation(n, 12345, a.data_ptr(), _st()))
    check(L.so100_ppo_permutation(n, 12346, b.data_ptr(), _st()))
    assert torch.equal(torch.sort(a).values, torch.arange(n, device="cuda"))
    assert torch.equal(torch.sort(b).values, torch.arange(n, device="cuda"))
    if n >= 1000:
        assert (a != b).float().mean() > 0.99 and (a != torch.arange(n, device="cuda")).float().mean() > 0.99
        # no structure a minibatch could inherit: neighbouring positions map far apart, halves are balanced
        x = a.double()
        tol = 4.0 / n ** 0.5 + 0.005  # 4 sigma of an ideal random permutation
        assert abs(float(torch.corrcoef(torch.stack([x[:-1], x[1:]]))[0, 1])) < tol
        assert abs(float((a[: n // 2] < n // 2).float().mean()) - 0.5) < tol


def test_fused_learner_state_roundtrip_resumes_bit_exactly():
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    from so100_mujoco_rl_b200.ppo import FusedPPO, PPOConfig
    cfg = PPOConfig(n_steps=8, n_minibatches=2, n_epochs=2, seed=3)
    a = FusedPPO(BatchedSo100Env(5, 512, device=0, seed=2), cfg)
    a.learn(total_samples=512 * 8 * 3, log_every=0, callback=lambda r: None)
    sd = a.state_dict()
    b = FusedPPO(BatchedSo100Env(5, 512, device=0, seed=2), cfg)
    b.load_state_dict({k: (v.cpu() if torch.is_tensor(v) else v) for k, v in sd.items()})   # as read back from a .pt file
    assert torch.equal(a.params, b.params) and torch.equal(a.exp_avg, b.exp_avg) and int(b.step_count) == int(a.step_count)
    assert b.stats.samples == a.stats.samples and b.tick == a.tick
    # the same minibatch on the same rollout data moves both learners identically
    for k in a.buf:
        b.buf[k].copy_(a.buf[k])
    idx = torch.randperm(a.adv.numel(), device="cuda")[:1024]
    a.minibatch_step(idx, a.adv, a.ret); b.minibatch_step(idx, a.adv, a.ret)
    assert torch.equal(a.params, b.params)


def test_torch_learner_resume_keeps_adam_state_under_cuda_graph():
    """ADVICE r1: with cuda_graph=True the graph is built lazily on the first update(), AFTER load_state_dict; the
    warm-up steps of the capture must not wipe the restored Adam moments / step.  The resumed learner's next update
    has to equal the uninterrupted learner's."""
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    from so100_mujoco_rl_b200.ppo import PPO, PPOConfig, pack_params
    # one minibatch per epoch: the update then does not depend on which permutation torch.randperm draws (capturing a
    # graph touches the CUDA generator's bookkeeping, so the two learners need not draw the same one)
    cfg = PPOConfig(n_steps=4, n_minibatches=1, n_epochs=2, seed=5, cuda_graph=True)
    a = PPO(BatchedSo100Env(1, 256, device=0, seed=9), cfg)
    a.learn(total_samples=256 * 4 * 2, log_every=0, callback=lambda r: None)
    import io
    f = io.BytesIO()
    torch.save(a.state_dict(), f)    # as a checkpoint file: state_dict() itself aliases the live tensors
    sd = torch.load(io.BytesIO(f.getvalue()), map_location="cpu")
    b = PPO(BatchedSo100Env(1, 256, device=0, seed=9), cfg)
    b.load_state_dict(sd)
    for k in a.buf:
        b.buf[k].copy_(a.buf[k])
    adv, ret = torch.randn_like(a.buf["rew"]), torch.randn_like(a.buf["rew"])
    torch.manual_seed(123); a.update(adv, ret)
    torch.manual_seed(123); b.update(adv, ret)   # builds b's graph here, after the restore
    sa, sb = a.opt.state_dict()["state"], b.opt.state_dict()["state"]
    assert all(float(sa[k]["step"]) == float(sb[k]["step"]) for k in sa), "Adam step was reset by the graph capture"
    assert all(torch.allclose(sa[k]["exp_avg"], sb[k]["exp_avg"], atol=1e-6) for k in sa)
    assert all(torch.allclose(sa[k]["exp_avg_sq"], sb[k]["exp_avg_sq"], atol=1e-8, rtol=1e-4) for k in sa)
    assert torch.allclose(pack_params(a.policy), pack_params(b.policy), atol=2e-5)
    # and it matters: a learner that restarts Adam from zero lands elsewhere
    c = PPO(BatchedSo100Env(1, 256, device=0, seed=9), cfg)
    c.policy.load_state_dict(sd["policy"])
    for k in a.buf:
        c.buf[k].copy_(a.buf[k])
    c.update(adv, ret)
    assert not torch.allclose(pack_params(a.policy), pack_params(c.policy), atol=2e-5)


_ACT_SNIPPET = r"""
import sys, numpy as np, torch
sys.path.insert(0, {root!r})
from so100_mujoco_rl_b200 import _native
from so100_mujoco_rl_b200.ppo import MlpPolicy, pack_params
L = _native.lib()
od, n = {od}, {n}
torch.manual_seed(0)
p = MlpPolicy(od, 6).cuda()
with torch.no_grad():
    for t in p.parameters():
        t.add_(0.1 * torch.randn_like(t))
P = pack_params(p)
obs = torch.randn(n, od, device="cuda")
f = dict(device="cuda", dtype=torch.float32)
a, lp, v = torch.zeros(n, 6, **f), torch.zeros(n, **f), torch.zeros(n, **f)
_native.check(L.so100_ppo_act(od, P.data_ptr(), obs.data_ptr(), n, 7, 0, 3, 0, a.data_ptr(), None, lp.data_ptr(), v.data_ptr(), None,
                              torch.cuda.current_stream().cuda_stream))
torch.cuda.synchronize()
np.savez({out!r}, a=a.cpu().numpy(), lp=lp.cpu().numpy(), v=v.cpu().numpy())
"""


@pytest.mark.parametrize("od,n", [(15, 777), (8, 4096), (16, 300_000)])
def test_act_tcgen05_and_mma_kernels_agree(od, n, tmp_path):
    """The rollout-inference kernel on tcgen05 / TMEM (the default) and the warp-level mma.sync one (SO100_PPO_ACT_MMA=1,
    read once per process, hence the subprocesses) compute the same fp32-level forward pass: same noise, values and
    log-probs to re-association error."""
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    res = {}
    for tag, env in (("tc", {}), ("mma", {"SO100_PPO_ACT_MMA": "1"})):
        out = str(tmp_path / f"act_{tag}.npz")
        e = dict(os.environ, **env)
        e.pop("SO100_PPO_ACT_MMA", None) if not env else None
        subprocess.run([sys.executable, "-c", _ACT_SNIPPET.format(root=root, od=od, n=n, out=out)], check=True, env=e, timeout=300)
        res[tag] = np.load(out)
    assert np.abs(res["tc"]["v"] - res["mma"]["v"]).max() < 2e-5
    assert np.abs(res["tc"]["a"] - res["mma"]["a"]).max() < 2e-5
    assert np.abs(res["tc"]["lp"] - res["mma"]["lp"]).max() < 2e-4
