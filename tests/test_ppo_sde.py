"""gSDE (SB3 use_sde=True) on the host: the torch policy against a direct fp64 restatement of SB3's
StateDependentNoiseDistribution, the flat parameter layout against the C ABI, the noise-key schedule, the torch learner on
the CPU toy env, the CLI's flag checks and the argument checks of the _sde_ entry points.  No GPU needed."""
import math

import numpy as np
import pytest
import torch

from so100_mujoco_rl_b200.ppo import PPO, SDE_EPS, MlpPolicy, PPOConfig, pack_params, param_layout, sde_noise_key, unpack_params
from test_ppo import ToyEnv

LOG_SQRT_2PI = 0.5 * math.log(2 * math.pi)


def _sb3_sde64(policy, obs, actions, mats):
    """SB3 2.6.0 StateDependentNoiseDistribution (full_std, no expln, learn_features=False) in fp64, written out:
    h = latent_pi, var_j = sum_k h_k^2 exp(log_std_kj)^2, scale = sqrt(var + eps); noise = h E[env]."""
    with torch.no_grad():
        x = obs.double()
        h = torch.tanh(torch.tanh(x @ policy.pi[0].weight.double().T + policy.pi[0].bias.double()) @ policy.pi[2].weight.double().T
                       + policy.pi[2].bias.double())
        mean = h @ policy.action_net.weight.double().T + policy.action_net.bias.double()
        std = torch.exp(policy.log_std.double())
        var = (h * h) @ (std * std)
        scale = torch.sqrt(var + SDE_EPS)
        a = actions.double()
        logp = (-((a - mean) ** 2) / (2 * scale ** 2) - torch.log(scale) - LOG_SQRT_2PI).sum(-1)
        ent = (0.5 + LOG_SQRT_2PI + torch.log(scale)).sum(-1)
        noise = torch.einsum("nk,nkj->nj", h, mats.double())
    return mean, logp, ent, noise


def _sde_policy(od=15, seed=0, log_std_init=-1.0):
    torch.manual_seed(seed)
    p = MlpPolicy(od, 6, log_std_init=log_std_init, use_sde=True)
    with torch.no_grad():
        for t in p.parameters():
            t.add_(0.1 * torch.randn_like(t))
    return p


def test_sde_policy_matches_sb3_formulas_in_fp64():
    p = _sde_policy()
    assert p.log_std.shape == (64, 6)
    obs = torch.randn(33, 15)
    p.reset_noise(33)
    assert p.exploration_matrices.shape == (33, 64, 6) and p.exploration_mat.shape == (64, 6)
    a, logp, v = p.act(obs)
    v2, logp2, ent = p.evaluate(obs, a)
    mean64, logp64, ent64, noise64 = _sb3_sde64(p, obs, a, p.exploration_matrices)
    mean = p.dist_params(obs)[0]
    assert torch.allclose((a - mean).double(), noise64, atol=1e-5)
    assert torch.allclose(logp.double(), logp64, atol=1e-4) and torch.allclose(logp2.double(), logp64, atol=1e-4)
    assert torch.allclose(ent.double(), ent64, atol=1e-5) and torch.allclose(v, v2)
    # the matrices are Normal(0, exp(log_std)): standardised, they are N(0, 1)
    z = (p.exploration_matrices / torch.exp(p.log_std.detach())).flatten().double()
    assert abs(float(z.mean())) < 0.02 and abs(float(z.std()) - 1) < 0.02
    # deterministic gives the mean; a batch that is not one per env uses the shared matrix (SB3 get_noise)
    assert torch.equal(p.act(obs, deterministic=True)[0], mean)
    a1 = p.act(obs[:5])[0]
    assert torch.allclose((a1 - mean[:5]).double(), _sb3_sde64(p, obs[:5], a1, p.exploration_mat.expand(5, 64, 6))[3], atol=1e-5)


def test_sde_variance_sends_gradient_to_log_std_only():
    """learn_features=False: the log-prob's dependence on the variance reaches log_std, never the policy tower."""
    p = _sde_policy(seed=1)
    obs, act = torch.randn(17, 15), torch.randn(17, 6)
    _, logp, ent = p.evaluate(obs, act)
    g_tower = torch.autograd.grad(ent.sum(), [p.pi[0].weight, p.pi[2].weight, p.log_std], allow_unused=True)
    assert g_tower[0] is None and g_tower[1] is None and float(g_tower[2].abs().sum()) > 0
    # and the mean path is the plain one: with log_std frozen, d logp / d tower = that of Normal(mean, fixed scale)
    mean, ls = p.dist_params(obs)
    ls = ls.detach()
    ref = (-((act - mean) ** 2) / (2 * torch.exp(2 * ls)) - ls - LOG_SQRT_2PI).sum()
    g1 = torch.autograd.grad(logp.sum(), p.pi[2].weight, retain_graph=True)[0]
    g2 = torch.autograd.grad(ref, p.pi[2].weight)[0]
    assert torch.allclose(g1, g2, atol=1e-5)


def test_sde_flat_layout_matches_the_c_abi(native_lib):
    for od, expect in ((15, 11207), (8, 10311)):
        assert native_lib.so100_ppo_sde_param_count(od) == expect
        assert sum(int(np.prod(s)) for _, s in param_layout(od, use_sde=True)) == expect
        # every entry before log_std sits where the plain layout has it
        assert param_layout(od, use_sde=True)[:-1] == param_layout(od)[:-1]
        p = _sde_policy(od)
        flat = pack_params(p)
        assert flat.numel() == expect and torch.equal(flat[-384:].view(64, 6), p.log_std.detach())
        q = unpack_params(flat * 2, MlpPolicy(od, 6, use_sde=True))
        assert torch.equal(q.log_std, 2 * p.log_std) and torch.equal(q.pi[0].weight, 2 * p.pi[0].weight)
        assert torch.equal(pack_params(q), flat * 2)
        with pytest.raises(AssertionError):
            unpack_params(flat, MlpPolicy(od, 6))
    assert native_lib.so100_ppo_sde_param_count(0) < 0 and native_lib.so100_ppo_sde_param_count(17) < 0
    assert native_lib.so100_ppo_sde_workspace_floats(15) >= 1024 * (11207 + 4)
    assert native_lib.so100_ppo_sde_workspace_floats(17) < 0


def test_sde_state_dict_keeps_sb3_names():
    p = _sde_policy()
    sd = p.state_dict_sb3()
    assert set(sd) == set(MlpPolicy(15, 6).state_dict_sb3()) and sd["log_std"].shape == (64, 6)
    q = MlpPolicy(15, 6, use_sde=True).load_state_dict_sb3(sd)
    assert torch.equal(pack_params(q), pack_params(p))


@pytest.mark.parametrize("freq,expect", [
    (-1, [1, 1, 1, 1, 1, 1, 1, 1, 1]),
    (1, [1, 2, 3, 4, 5, 6, 7, 8, 9]),
    (4, [1, 1, 1, 1, 5, 5, 5, 5, 9]),
])
def test_noise_key_schedule(freq, expect):
    """Rollout steps t = 0..8 at ticks 1..9: a fresh key (the tick) at t = 0 and, with freq > 0, wherever t % freq == 0."""
    key, got = 12345, []
    for t in range(9):
        key = sde_noise_key(t, t + 1, freq, key)
        got.append(key)
    assert got == expect
    # the next rollout starts a fresh draw even with freq = -1
    assert sde_noise_key(0, 100, -1, key) == 100


def test_torch_learner_with_sde_learns_and_redraws_per_schedule(monkeypatch):
    env = ToyEnv(256)
    cfg = PPOConfig(n_steps=16, n_epochs=4, n_minibatches=4, lr=3e-3, seed=1, use_sde=True, log_std_init=-2.0)
    algo = PPO(env, cfg)
    assert algo.policy.use_sde and float(algo.policy.log_std.mean()) == -2.0
    draws = []
    orig = algo.policy.reset_noise
    monkeypatch.setattr(algo.policy, "reset_noise", lambda n: (draws.append(n), orig(n)))
    hist = []
    algo.learn(total_samples=256 * 16 * 30, log_every=0, callback=hist.append)
    assert draws == [256] * 30                                   # once per rollout (sde_sample_freq = -1)
    first, last = np.mean([h["mean_step_reward"] for h in hist[:3]]), np.mean([h["mean_step_reward"] for h in hist[-3:]])
    assert last > first + 0.3, (first, last)
    assert all(np.isfinite(h["log_std_mean"]) for h in hist)
    draws.clear()
    algo.cfg.sde_sample_freq = 4
    algo.learn(total_samples=256 * 16, log_every=0, callback=lambda r: None, additional=True)
    assert len(draws) == 4                                       # t = 0, 4, 8, 12


def test_sde_checkpoint_and_zip_carry_the_config(tmp_path):
    import json
    import zipfile

    from so100_mujoco_rl_b200.callbacks import TrainCallbacks, load_sb3_zip
    cfg = PPOConfig(n_steps=8, n_epochs=1, n_minibatches=1, seed=4, cuda_graph=False, use_sde=True, sde_sample_freq=4, log_std_init=-1.5)
    a = PPO(ToyEnv(32, limit=8, seed=1), cfg)
    a.learn(total_samples=32 * 8 * 2, log_every=0, callback=lambda r: None)
    cb = TrainCallbacks(a, str(tmp_path), "Toy", eval_env=None, save_freq=0, tensorboard_dir=None, verbose=False)
    cb.save("ckpt")
    ck = torch.load(tmp_path / "ckpt.pt")
    assert ck["learner"]["config"]["use_sde"] is True and ck["learner"]["config"]["sde_sample_freq"] == 4
    assert ck["policy"]["log_std"].shape == (64, 6)
    with zipfile.ZipFile(tmp_path / "ckpt.zip") as z:
        data = json.loads(z.read("data"))
    assert data["use_sde"] is True and data["sde_sample_freq"] == 4
    assert load_sb3_zip(str(tmp_path / "ckpt.zip"))["log_std"].shape == (64, 6)
    b = PPO(ToyEnv(32, limit=8, seed=1), cfg)
    b.load_state_dict(ck["learner"])
    assert torch.equal(pack_params(a.policy), pack_params(b.policy))


# ------------------------------------------------------------------------------------------------ CLI
click = pytest.importorskip("click")


def _invoke(args):
    from click.testing import CliRunner

    from so100_mujoco_rl_b200.cli import cli
    return CliRunner().invoke(cli, args, obj={})


def test_cli_sde_flags():
    h = _invoke(["train", "--help"]).output
    for token in ("--use-sde", "--sde-sample-freq", "--log-std-init"):
        assert token in h
    r = _invoke(["train", "-e", "Env01", "--sde-sample-freq", "4"])
    assert r.exit_code != 0 and "--sde-sample-freq" in r.output and "--use-sde" in r.output
    r = _invoke(["train", "-e", "Env01", "--use-sde", "--sde-sample-freq", "0"])
    assert r.exit_code != 0 and "--sde-sample-freq" in r.output


@pytest.mark.parametrize("saved_sde", [True, False])
@pytest.mark.parametrize("fmt", ["pt", "zip"])
def test_cli_resume_refuses_a_different_policy_kind(tmp_path, saved_sde, fmt):
    from so100_mujoco_rl_b200.callbacks import export_sb3_zip
    p = MlpPolicy(15, 6, use_sde=saved_sde)
    path = str(tmp_path / f"m.{fmt}")
    if fmt == "pt":
        torch.save({"policy": p.state_dict()}, path)
    else:
        export_sb3_zip(path, p.state_dict_sb3())
    args = ["-m", path, "train", "-e", "Env01", "--num-envs", "8", "--out", str(tmp_path / "o")] + ([] if saved_sde else ["--use-sde"])
    r = _invoke(args)
    assert r.exit_code != 0 and "--use-sde" in r.output, r.output
    assert ("add --use-sde" if saved_sde else "drop --use-sde") in r.output


def test_load_policy_recognises_sde_by_log_std_shape(tmp_path):
    from so100_mujoco_rl_b200.callbacks import export_sb3_zip
    from so100_mujoco_rl_b200.cli import _load_policy
    p = _sde_policy()
    torch.save({"policy": p.state_dict()}, tmp_path / "m.pt")
    export_sb3_zip(str(tmp_path / "m.zip"), p.state_dict_sb3())
    obs = torch.randn(4, 15)
    for f in ("m.pt", "m.zip"):
        q = _load_policy(str(tmp_path / f), 15, "cpu")
        assert q.use_sde and torch.equal(q.act(obs, deterministic=True)[0], p.act(obs, deterministic=True)[0])


# ------------------------------------------------------------------------------------------------ C ABI arguments
def test_sde_entry_points_reject_bad_arguments(native_lib):
    """SO100_ERR_ARG (-1) before any CUDA call: unsupported obs_dim, NULL pointers, n <= 0 / mb <= 0."""
    L = native_lib
    fake = 4096   # never dereferenced: the argument checks come first
    act = lambda od, P, obs, n: L.so100_ppo_sde_act(od, P, obs, n, 0, 0, 1, 0, None, None, None, None, None, None)  # noqa: E731
    assert act(0, fake, fake, 8) == -1 and act(17, fake, fake, 8) == -1
    assert act(15, None, fake, 8) == -1 and act(15, fake, None, 8) == -1
    assert act(15, fake, fake, 0) == -1 and act(15, fake, fake, -3) == -1

    def grad(od=15, mb=8, null=None):
        ptrs = [fake] * 7
        if null is not None and null < 7:
            ptrs[null] = None
        P, obs, a, lpo, adv, ret, idx = ptrs
        ws = None if null == 7 else fake
        g = None if null == 8 else fake
        return L.so100_ppo_sde_grad(od, P, obs, a, lpo, adv, ret, idx, mb, 0.2, 0.5, 0.0, 1, ws, g, None, None)
    assert grad(od=0) == -1 and grad(od=17) == -1
    assert grad(mb=0) == -1 and grad(mb=-1) == -1
    for k in range(9):
        assert grad(null=k) == -1, k
