"""Host logic of the GPU PPO learner on CPU tensors: GAE against the textbook recursion, SB3-compatible export,
TimeLimit bootstrap, and that it actually learns a toy batched task."""
from types import SimpleNamespace

import numpy as np
import pytest
import torch

from so100_mujoco_rl_b200.ppo import PPO, MlpPolicy, PPOConfig, compute_gae


def test_gae_matches_reference_recursion():
    torch.manual_seed(0)
    T, N, g, lam = 7, 5, 0.99, 0.95
    r, v = torch.randn(T, N), torch.randn(T, N)
    d = (torch.rand(T, N) < 0.2).float()
    last = torch.randn(N)
    adv, ret = compute_gae(r, v, d, last, g, lam)
    for n in range(N):
        a_next, expect = 0.0, np.zeros(T)
        for t in reversed(range(T)):
            nv = last[n].item() if t == T - 1 else v[t + 1, n].item()
            nt = 1.0 - d[t, n].item()
            delta = r[t, n].item() + g * nv * nt - v[t, n].item()
            a_next = delta + g * lam * nt * a_next
            expect[t] = a_next
        assert np.allclose(adv[:, n].numpy(), expect, atol=1e-5)
    assert torch.allclose(ret, adv + v)


def test_policy_matches_sb3_defaults_and_export_names():
    p = MlpPolicy(15, 6)
    n_params = sum(x.numel() for x in p.parameters())
    assert n_params == 5574 + 5249 + 6  # SURVEY §8e: pi 15-64-64-6, vf 15-64-64-1, log_std
    sd = p.state_dict_sb3()
    assert set(sd) == {"log_std", "mlp_extractor.policy_net.0.weight", "mlp_extractor.policy_net.0.bias",
                       "mlp_extractor.policy_net.2.weight", "mlp_extractor.policy_net.2.bias",
                       "mlp_extractor.value_net.0.weight", "mlp_extractor.value_net.0.bias",
                       "mlp_extractor.value_net.2.weight", "mlp_extractor.value_net.2.bias",
                       "action_net.weight", "action_net.bias", "value_net.weight", "value_net.bias"}
    assert sd["action_net.weight"].shape == (6, 64) and float(p.log_std.abs().sum()) == 0.0
    obs = torch.randn(9, 15)
    a, logp, v = p.act(obs)
    v2, logp2, ent = p.evaluate(obs, a)
    assert torch.allclose(logp, logp2, atol=1e-6) and torch.allclose(v, v2)
    assert torch.allclose(ent, torch.full((9,), 6 * (0.5 + 0.5 * np.log(2 * np.pi))), atol=1e-6)


class ToyEnv:
    """N independent 1-step-memory tasks: reward = -|a - target(obs)|^2, episodes of `limit` steps (truncation)."""

    def __init__(self, n, limit=16, seed=0):
        self.num_envs, self.obs_dim, self.act_dim, self.device = n, 15, 6, torch.device("cpu")
        self.g = torch.Generator().manual_seed(seed)
        self.limit = limit
        self.t = torch.zeros(n, dtype=torch.int32)
        self.ret = torch.zeros(n)

    def _obs(self):
        return torch.rand((self.num_envs, self.obs_dim), generator=self.g) * 2 - 1

    def reset(self):
        self.obs = self._obs()
        return self.obs

    def step(self, a):
        rew = -((a - 0.5 * self.obs[:, :6]) ** 2).sum(-1)
        self.t += 1
        self.ret += rew
        trunc = self.t >= self.limit
        term_obs = self._obs()
        nxt = self._obs()
        ep_ret, ep_len = self.ret.clone(), self.t.clone()
        self.ret[trunc] = 0; self.t[trunc] = 0
        self.obs = nxt
        return SimpleNamespace(obs=nxt, reward=rew, terminated=torch.zeros_like(trunc, dtype=torch.uint8),
                               truncated=trunc.to(torch.uint8), terminal_obs=term_obs, ep_return=ep_ret, ep_len=ep_len)


def test_ppo_learns_a_toy_task():
    env = ToyEnv(256)
    algo = PPO(env, PPOConfig(n_steps=16, n_epochs=4, n_minibatches=4, lr=3e-3, seed=1))
    hist = []
    algo.learn(total_samples=256 * 16 * 30, log_every=0, callback=hist.append)
    first, last = np.mean([h["mean_step_reward"] for h in hist[:3]]), np.mean([h["mean_step_reward"] for h in hist[-3:]])
    assert last > first + 0.3, (first, last)
    assert hist[-1]["episodes"] > 0 and hist[-1]["ep_len_mean"] == 16
    assert algo.stats.samples == 256 * 16 * 30


def test_one_sample_minibatches_stay_finite():
    """num_envs * n_steps = 8 with 8 minibatches: every minibatch holds one sample.  SB3 2.x leaves a lone advantage
    unnormalised (the std of one sample is NaN); the learner must do the same and keep finite weights and losses."""
    from so100_mujoco_rl_b200.ppo import pack_params
    algo = PPO(ToyEnv(4, limit=4), PPOConfig(n_steps=2, n_epochs=2, n_minibatches=8, seed=6))
    p0 = pack_params(algo.policy)
    hist = []
    algo.learn(total_samples=4 * 2 * 3, log_every=0, callback=hist.append)
    p1 = pack_params(algo.policy)
    assert torch.isfinite(p1).all() and not torch.equal(p0, p1)
    assert all(np.isfinite(h["pg_loss"]) and np.isfinite(h["v_loss"]) and np.isfinite(h["approx_kl"]) for h in hist)
    assert any(h["pg_loss"] != 0.0 for h in hist)   # the policy gradient is not zeroed


def test_truncation_bootstraps_with_terminal_value():
    env = ToyEnv(8, limit=2)
    algo = PPO(env, PPOConfig(n_steps=2, n_epochs=1, n_minibatches=1))
    with torch.no_grad():
        for p in algo.policy.value_net.parameters():
            p.fill_(0.0)
        algo.policy.value_net.bias.fill_(3.0)  # V(s) = 3 everywhere
    adv, ret = algo.collect()
    # step 2 of every env is a truncation: its stored reward carries gamma * V(terminal) = 0.99 * 3
    r_env = algo.buf["rew"][1]
    assert (algo.buf["done"][1] == 1).all()
    assert ((r_env - 0.99 * 3.0) <= 1e-6).all()  # raw toy rewards are <= 0


def test_flat_parameter_layout_matches_the_c_abi(native_lib):
    """pack_params / unpack_params / param_layout agree with so100_ppo_param_count (include/so100_ppo.h)."""
    from so100_mujoco_rl_b200.ppo import pack_params, param_layout, unpack_params
    for od, expect in ((15, 10829), (8, 9933)):
        assert native_lib.so100_ppo_param_count(od) == expect
        assert sum(int(np.prod(s)) for _, s in param_layout(od)) == expect
        p = MlpPolicy(od, 6)
        flat = pack_params(p)
        assert flat.numel() == expect and torch.equal(flat[-6:], p.log_std.detach())
        assert torch.equal(flat[:64 * od].view(64, od), p.pi[0].weight.detach())
        q = unpack_params(flat * 2, MlpPolicy(od, 6))
        assert torch.equal(q.value_net.weight, 2 * p.value_net.weight) and torch.equal(q.pi[2].bias, 2 * p.pi[2].bias)
    assert native_lib.so100_ppo_param_count(17) < 0 and native_lib.so100_ppo_workspace_floats(15) >= 1024 * 10833


def test_callbacks_checkpoint_eval_and_sb3_zip(tmp_path):
    """main.py:211-232 plumbing on the toy task: checkpoints at save_freq, best_model on improvement, early stop at the
    reward threshold, and the SB3-style zip round-trips through SB3's parameter names."""
    from so100_mujoco_rl_b200.callbacks import TrainCallbacks, load_sb3_zip
    env, eval_env = ToyEnv(64, limit=8), ToyEnv(32, limit=8, seed=5)
    algo = PPO(env, PPOConfig(n_steps=8, n_epochs=2, n_minibatches=2, lr=3e-3, seed=2))
    cb = TrainCallbacks(algo, str(tmp_path), "Toy_PPO", eval_env=eval_env, eval_freq=1024, eval_steps=16, save_freq=2048,
                        reward_threshold=-1e9, tensorboard_dir=str(tmp_path / "logs"), verbose=False)
    algo.learn(total_samples=64 * 8 * 40, log_every=0, callback=cb)
    cb.close()
    assert cb.stop and "threshold" in cb.stop_reason and algo.stats.samples == 1024   # stopped at the first evaluation
    assert (tmp_path / "best_model.zip").exists() and (tmp_path / "best_model.pt").exists()
    sd = load_sb3_zip(str(tmp_path / "best_model.zip"))
    assert set(sd) == set(algo.policy.state_dict_sb3())
    q = MlpPolicy(15, 6).load_state_dict_sb3(sd)
    obs = torch.randn(5, 15)
    assert torch.allclose(q.act(obs, deterministic=True)[0], algo.policy.act(obs, deterministic=True)[0])
    # without a reachable threshold: checkpoints accumulate and training runs to the end
    algo2 = PPO(ToyEnv(64, limit=8), PPOConfig(n_steps=8, n_epochs=1, n_minibatches=1, seed=3))
    cb2 = TrainCallbacks(algo2, str(tmp_path / "b"), "Toy_PPO", eval_env=eval_env, eval_freq=1024, eval_steps=16, save_freq=1024,
                         tensorboard_dir=None, verbose=False)
    algo2.learn(total_samples=64 * 8 * 8, log_every=0, callback=cb2)
    assert not cb2.stop and len(cb2.checkpoints) == 4 and len(cb2.evals) == 4
    assert (tmp_path / "b" / "Toy_PPO_cp__1024_steps.zip").exists()
    assert any((tmp_path / "logs" / "Toy_PPO").iterdir())                                  # TensorBoard event file


def test_checkpoint_resume_restores_optimizer_and_counters(tmp_path):
    from so100_mujoco_rl_b200.callbacks import TrainCallbacks
    from so100_mujoco_rl_b200.ppo import pack_params
    cfg = PPOConfig(n_steps=8, n_epochs=1, n_minibatches=1, seed=4, cuda_graph=False)
    a = PPO(ToyEnv(32, limit=8, seed=1), cfg)
    a.learn(total_samples=32 * 8 * 2, log_every=0, callback=lambda r: None)
    cb = TrainCallbacks(a, str(tmp_path), "Toy", eval_env=None, save_freq=0, tensorboard_dir=None, verbose=False)
    cb.save("ckpt")
    sd = torch.load(tmp_path / "ckpt.pt")["learner"]
    b = PPO(ToyEnv(32, limit=8, seed=1), cfg)
    b.load_state_dict(sd)
    assert torch.equal(pack_params(a.policy), pack_params(b.policy)) and b.stats.samples == a.stats.samples
    sa, sb = a.opt.state_dict()["state"], b.opt.state_dict()["state"]
    assert all(torch.equal(sa[k]["exp_avg"], sb[k]["exp_avg"]) and torch.equal(sa[k]["step"], sb[k]["step"]) for k in sa)
