"""GPU-resident PPO for the batched so100 envs — the caller side of the seam at scale (SURVEY.md §8 f1).

The reference trains with `stable_baselines3.PPO("MlpPolicy", env, device='cpu')` on ONE env
(src/so100_mujoco_rl/main.py:56-64, 234-238).  SB3's rollout loop is per-env Python and its buffers are numpy, which caps
a 65 536-env simulator at a few 10^5 samples/s; this learner keeps observations, actions, the rollout buffer, GAE and
the updates on the GPU and drives `BatchedSo100Env` tensors directly.  Hyper-parameters and network are SB3 2.6.0's
PPO/MlpPolicy defaults (2x64 tanh, separate policy/value towers, state-independent log_std initialised at 0,
orthogonal init, Adam 3e-4 eps 1e-5, gamma 0.99, lambda 0.95, clip 0.2, vf_coef 0.5, ent_coef 0, max_grad_norm 0.5,
10 epochs, per-minibatch advantage normalisation, bootstrap of TimeLimit truncations with V(terminal_obs)); only the
batch geometry differs (n_steps x num_envs samples per rollout, large minibatches).  `state_dict_sb3()` exports the
weights under SB3's parameter names so that `PPO.load`-style tooling can consume them.

Two learners share the hyper-parameters, the rollout geometry and the `learn()` loop:
  * `PPO`       — plain PyTorch fp32 (autograd, torch.optim.Adam, optionally replayed as a CUDA graph).  It is the
                  numerical REFERENCE of the fused path and the only one that runs on CPU tensors (host-logic tests).
  * `FusedPPO`  — the product path on a GPU: hand-written kernels behind include/so100_ppo.h do the rollout inference
                  (`so100_ppo_act`), the TimeLimit bootstrap + statistics (`so100_ppo_post_step`), GAE, one fused
                  forward + loss + backward per minibatch (`so100_ppo_grad`) and clip + Adam (`so100_ppo_adam`); torch only
                  owns the buffers, draws the minibatch permutation and runs the NCCL all-reduce.

Both support SB3's `use_sde=True` / `sde_sample_freq` (generalized State-Dependent Exploration, DESIGN.md §7d): the action
noise is h E with h the policy tower's last hidden layer and E a 64x6 matrix per env redrawn once per rollout (or every
`sde_sample_freq` steps), so the commanded actions change only as fast as the state does.

Data parallel: one process per GPU, each with its own env shard; gradients are averaged with ONE flat all-reduce per
minibatch (NCCL over NVLink; ~10 k fp32 values, latency bound).  The env step path itself has no collective.
"""
from __future__ import annotations

import dataclasses
import math
import time
from dataclasses import dataclass, field

import torch
import torch.distributed as dist
from torch import nn


def _ortho(layer: nn.Linear, gain: float) -> nn.Linear:
    nn.init.orthogonal_(layer.weight, gain=gain)
    nn.init.zeros_(layer.bias)
    return layer


SDE_EPS = 1e-6  # StateDependentNoiseDistribution.epsilon


class MlpPolicy(nn.Module):
    """SB3 ActorCriticPolicy with net_arch dict(pi=[64, 64], vf=[64, 64]), tanh, DiagGaussian head; with use_sde=True
    SB3's StateDependentNoiseDistribution (full_std, no expln, learn_features=False): log_std is [hidden, act_dim]."""

    def __init__(self, obs_dim: int, act_dim: int, hidden: int = 64, log_std_init: float = 0.0, use_sde: bool = False):
        super().__init__()
        g = math.sqrt(2.0)
        self.pi = nn.Sequential(_ortho(nn.Linear(obs_dim, hidden), g), nn.Tanh(), _ortho(nn.Linear(hidden, hidden), g), nn.Tanh())
        self.vf = nn.Sequential(_ortho(nn.Linear(obs_dim, hidden), g), nn.Tanh(), _ortho(nn.Linear(hidden, hidden), g), nn.Tanh())
        self.action_net = _ortho(nn.Linear(hidden, act_dim), 0.01)
        self.value_net = _ortho(nn.Linear(hidden, 1), 1.0)
        self.use_sde = bool(use_sde)
        self.log_std = nn.Parameter(torch.full((hidden, act_dim) if self.use_sde else (act_dim,), float(log_std_init)))
        self.exploration_mat = self.exploration_matrices = None  # gSDE: drawn by reset_noise

    def value(self, obs: torch.Tensor) -> torch.Tensor:
        return self.value_net(self.vf(obs)).squeeze(-1)

    def _dist(self, obs: torch.Tensor):
        """(h, mean, log scale): the log scale is log_std itself, or per sample for gSDE: 0.5 log(h^2 exp(2 log_std) + eps),
        with h detached (learn_features=False: the variance sends gradient to log_std only)."""
        h = self.pi(obs)
        mean = self.action_net(h)
        if not self.use_sde:
            return h, mean, self.log_std
        var = (h.detach() ** 2) @ torch.exp(self.log_std) ** 2
        return h, mean, 0.5 * torch.log(var + SDE_EPS)

    def dist_params(self, obs: torch.Tensor):
        _, mean, log_std = self._dist(obs)
        return mean, log_std

    def reset_noise(self, n_envs: int = 1) -> None:
        """StateDependentNoiseDistribution.sample_weights: E ~ Normal(0, exp(log_std)), one matrix per env (and one shared)."""
        with torch.no_grad():
            std = torch.exp(self.log_std)
            self.exploration_mat = std * torch.randn_like(std)
            self.exploration_matrices = std * torch.randn((n_envs, *std.shape), device=std.device, dtype=std.dtype)

    def sde_noise(self, h: torch.Tensor) -> torch.Tensor:
        """h E per sample (SB3 get_noise): bmm with the per-env matrices, or the shared matrix when the batch differs."""
        if self.exploration_mat is None:
            self.reset_noise(h.shape[0])
        h = h.detach()
        if h.shape[0] == 1 or h.shape[0] != self.exploration_matrices.shape[0]:
            return h @ self.exploration_mat
        return torch.bmm(h.unsqueeze(1), self.exploration_matrices).squeeze(1)

    @staticmethod
    def log_prob(mean, log_std, actions):
        var = torch.exp(2 * log_std)
        return (-((actions - mean) ** 2) / (2 * var) - log_std - 0.5 * math.log(2 * math.pi)).sum(-1)

    def act(self, obs: torch.Tensor, deterministic: bool = False):
        h, mean, log_std = self._dist(obs)
        if deterministic:
            a = mean
        elif self.use_sde:
            a = mean + self.sde_noise(h)
        else:
            a = mean + torch.exp(log_std) * torch.randn_like(mean)
        return a, self.log_prob(mean, log_std, a), self.value(obs)

    def evaluate(self, obs, actions):
        mean, log_std = self.dist_params(obs)
        entropy = (0.5 + 0.5 * math.log(2 * math.pi) + log_std).sum(-1).expand(obs.shape[0])
        return self.value(obs), self.log_prob(mean, log_std, actions), entropy

    def load_state_dict_sb3(self, sd: dict) -> "MlpPolicy":
        """Inverse of state_dict_sb3: accepts a stable_baselines3 ActorCriticPolicy state dict (policy.pth of a .zip)."""
        with torch.no_grad():
            self.log_std.copy_(sd["log_std"])
            for name, seq in (("policy_net", self.pi), ("value_net", self.vf)):
                for idx in (0, 2):
                    seq[idx].weight.copy_(sd[f"mlp_extractor.{name}.{idx}.weight"])
                    seq[idx].bias.copy_(sd[f"mlp_extractor.{name}.{idx}.bias"])
            for name, lin in (("action_net", self.action_net), ("value_net", self.value_net)):
                lin.weight.copy_(sd[f"{name}.weight"])
                lin.bias.copy_(sd[f"{name}.bias"])
        return self

    def state_dict_sb3(self) -> dict:
        """Weights under stable_baselines3.common.policies.ActorCriticPolicy's parameter names."""
        sd = {"log_std": self.log_std.detach().clone()}
        for name, seq in (("policy_net", self.pi), ("value_net", self.vf)):
            for idx in (0, 2):
                sd[f"mlp_extractor.{name}.{idx}.weight"] = seq[idx].weight.detach().clone()
                sd[f"mlp_extractor.{name}.{idx}.bias"] = seq[idx].bias.detach().clone()
        for name, lin in (("action_net", self.action_net), ("value_net", self.value_net)):
            sd[f"{name}.weight"] = lin.weight.detach().clone()
            sd[f"{name}.bias"] = lin.bias.detach().clone()
        return sd


def compute_gae(rewards, values, dones, last_value, gamma: float, lam: float):
    """SB3 RolloutBuffer.compute_returns_and_advantage on [T, N] tensors.  dones[t] = episode ended AT step t
    (the value after it belongs to the next episode)."""
    T = rewards.shape[0]
    adv = torch.zeros_like(rewards)
    last = torch.zeros_like(last_value)
    for t in reversed(range(T)):
        nxt = last_value if t == T - 1 else values[t + 1]
        nonterm = 1.0 - dones[t]
        delta = rewards[t] + gamma * nxt * nonterm - values[t]
        last = delta + gamma * lam * nonterm * last
        adv[t] = last
    return adv, adv + values


def param_layout(obs_dim: int, act_dim: int = 6, hidden: int = 64, use_sde: bool = False):
    """(name, shape) in the order of the flat parameter vector of include/so100_ppo.h (gSDE: log_std [hidden, act_dim])."""
    out = []
    for tower, nout in (("pi", act_dim), ("vf", 1)):
        out += [(f"{tower}.W1", (hidden, obs_dim)), (f"{tower}.b1", (hidden,)), (f"{tower}.W2", (hidden, hidden)),
                (f"{tower}.b2", (hidden,)), (f"{tower}.W3", (nout, hidden)), (f"{tower}.b3", (nout,))]
    return out + [("log_std", (hidden, act_dim) if use_sde else (act_dim,))]


def sde_redraw(t: int, sample_freq: int) -> bool:
    """SB3 collect_rollouts: reset_noise at the start of every rollout and, when sample_freq > 0, at every rollout step t
    with t % sample_freq == 0."""
    return t == 0 or (sample_freq > 0 and t % sample_freq == 0)


def sde_noise_key(t: int, tick: int, sample_freq: int, key: int) -> int:
    """Noise key of the exploration matrices at rollout step t: the current tick where a fresh draw starts, else the key
    in use."""
    return tick if sde_redraw(t, sample_freq) else key


def _policy_tensors(policy: "MlpPolicy"):
    return [policy.pi[0].weight, policy.pi[0].bias, policy.pi[2].weight, policy.pi[2].bias, policy.action_net.weight,
            policy.action_net.bias, policy.vf[0].weight, policy.vf[0].bias, policy.vf[2].weight, policy.vf[2].bias,
            policy.value_net.weight, policy.value_net.bias, policy.log_std]


def pack_params(policy: "MlpPolicy") -> torch.Tensor:
    """MlpPolicy -> flat float32 vector in the layout of include/so100_ppo.h."""
    return torch.cat([t.detach().reshape(-1).float() for t in _policy_tensors(policy)])


def unpack_params(flat: torch.Tensor, policy: "MlpPolicy") -> "MlpPolicy":
    o = 0
    with torch.no_grad():
        for t in _policy_tensors(policy):
            k = t.numel()
            t.copy_(flat[o:o + k].view_as(t))
            o += k
    assert o == flat.numel()
    return policy


@dataclass
class PPOConfig:
    n_steps: int = 32
    n_epochs: int = 10
    n_minibatches: int = 8
    gamma: float = 0.99
    gae_lambda: float = 0.95
    clip_range: float = 0.2
    vf_coef: float = 0.5
    ent_coef: float = 0.0
    max_grad_norm: float = 0.5
    lr: float = 3e-4
    normalize_advantage: bool = True
    seed: int = 0
    cuda_graph: bool = True  # capture one optimiser step (the 2x64 MLPs are launch-bound: ~10x faster updates)
    use_sde: bool = False    # gSDE exploration (SB3 use_sde)
    sde_sample_freq: int = -1  # redraw the exploration matrices every n steps; -1: once per rollout (SB3 sde_sample_freq)
    log_std_init: float = 0.0  # SB3's policy kwarg, for both distributions


@dataclass
class PPOStats:
    iterations: int = 0
    samples: int = 0
    rollout_s: float = 0.0
    update_s: float = 0.0
    history: list = field(default_factory=list)  # per iteration: dict(mean_step_reward, ep_return_mean, ep_len_mean, ...)


class _LearnLoop:
    def _sync(self):
        if self.device.type == "cuda":
            torch.cuda.synchronize(self.device)

    def learn(self, total_samples: int, log_every: int = 10, callback=None, additional: bool = False) -> PPOStats:
        """Run until `stats.samples` reaches total_samples; with additional=True until total_samples MORE have been drawn
        (SB3's `learn(total_timesteps)` restarts its count on every call: what a resumed `train -m ...` wants)."""
        per_iter = self.cfg.n_steps * self.env.num_envs * self.world
        if additional:
            total_samples = self.stats.samples + total_samples
        while self.stats.samples < total_samples:
            self._sync(); t0 = time.perf_counter()
            adv, ret = self.collect()
            self._sync(); t1 = time.perf_counter()
            info = self.update(adv, ret)
            self._sync(); t2 = time.perf_counter()
            s = self.stats
            s.iterations += 1; s.samples += per_iter; s.rollout_s += t1 - t0; s.update_s += t2 - t1
            raw, ers, els, cnt = (float(x) for x in self._acc.tolist())
            self._acc.zero_()
            rec = {"iter": s.iterations, "samples": s.samples, "mean_step_reward": raw / (self.cfg.n_steps * self.env.num_envs),
                   "ep_return_mean": ers / cnt if cnt else None, "ep_len_mean": els / cnt if cnt else None,
                   "episodes": int(cnt), "log_std_mean": self._log_std_mean(), "rollout_s": t1 - t0, "update_s": t2 - t1, **info}
            s.history.append(rec)
            if callback is not None:
                callback(rec)
                if getattr(callback, "stop", False):  # callbacks.TrainCallbacks: reward threshold / no improvement
                    break
            elif log_every and s.iterations % log_every == 0:
                print(rec, flush=True)
        return self.stats


class PPO(_LearnLoop):
    """`env` is a BatchedSo100Env-like object: .num_envs, .obs_dim, .act_dim, .device, reset() -> obs [N, od],
    step(actions [N, 6]) -> object with obs, reward, terminated, truncated, terminal_obs, ep_return, ep_len."""

    def __init__(self, env, cfg: PPOConfig | None = None):
        self.env, self.cfg = env, cfg or PPOConfig()
        self.device = env.device
        torch.manual_seed(self.cfg.seed)
        self.policy = MlpPolicy(env.obs_dim, env.act_dim, log_std_init=self.cfg.log_std_init, use_sde=self.cfg.use_sde).to(self.device)
        self.opt = torch.optim.Adam(self.policy.parameters(), lr=self.cfg.lr, eps=1e-5,
                                    capturable=self.device.type == "cuda" and self.cfg.cuda_graph)
        self.world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        if self.world > 1:  # identical initial weights on every rank
            for p in self.policy.parameters():
                dist.broadcast(p.data, src=0)
            # ... but different exploration noise: every rank owns different envs (the fused learner keys its noise by the
            # global env id; here torch's generator is re-seeded per rank once the shared initialisation is done)
            torch.manual_seed(self.cfg.seed + 7919 * (dist.get_rank() + 1))
        self.obs = env.reset().clone()
        self.stats = PPOStats()
        n, T, od, ad = env.num_envs, self.cfg.n_steps, env.obs_dim, env.act_dim
        f = dict(device=self.device, dtype=torch.float32)
        self.buf = {"obs": torch.zeros((T, n, od), **f), "act": torch.zeros((T, n, ad), **f), "logp": torch.zeros((T, n), **f),
                    "val": torch.zeros((T, n), **f), "rew": torch.zeros((T, n), **f), "done": torch.zeros((T, n), **f)}
        self._acc = torch.zeros(4, device=self.device, dtype=torch.float64)  # raw reward sum, ep return sum, ep len sum, episodes

    @torch.no_grad()
    def collect(self):
        cfg, b = self.cfg, self.buf
        for t in range(cfg.n_steps):
            if cfg.use_sde and sde_redraw(t, cfg.sde_sample_freq):
                self.policy.reset_noise(self.env.num_envs)
            a, logp, v = self.policy.act(self.obs)
            b["obs"][t], b["act"][t], b["logp"][t], b["val"][t] = self.obs, a, logp, v
            r = self.env.step(torch.clamp(a, -1.0, 1.0))  # SB3 clips Box actions before env.step (logp is of the raw action)
            # no host synchronisation inside the rollout loop: masks instead of branches, statistics stay on the device
            rew = r.reward.clone()
            term, trunc = r.terminated.bool(), r.truncated.bool()
            done = term | trunc
            self._acc[0] += rew.sum()
            # TimeLimit: bootstrap with the value of the terminal observation (SB3 on_policy_algorithm); rows of envs
            # that did not finish hold stale (finite) data and are masked out
            boot = cfg.gamma * self.policy.value(r.terminal_obs)
            rew = torch.where(trunc & torch.isfinite(boot), rew + boot, rew)
            b["rew"][t], b["done"][t] = rew, done.float()
            df = done.float()
            self._acc[1] += (r.ep_return * df).sum(); self._acc[2] += (r.ep_len.float() * df).sum(); self._acc[3] += df.sum()
            self.obs = r.obs.clone()
        last_value = self.policy.value(self.obs)
        adv, ret = compute_gae(b["rew"], b["val"], b["done"], last_value, cfg.gamma, cfg.gae_lambda)
        return adv, ret

    def _allreduce_grads(self):
        if self.world == 1:
            return
        flat = torch.cat([p.grad.reshape(-1) for p in self.policy.parameters()])
        dist.all_reduce(flat)
        flat /= self.world
        o = 0
        for p in self.policy.parameters():
            k = p.numel()
            p.grad.copy_(flat[o:o + k].view_as(p))
            o += k

    def _minibatch_step(self, idx, flat, adv, ret):
        cfg = self.cfg
        a = adv[idx]
        if cfg.normalize_advantage and a.numel() > 1:  # SB3 2.x: the std of one sample is NaN, so it is left raw
            a = (a - a.mean()) / (a.std() + 1e-8)
        v, logp, ent = self.policy.evaluate(flat["obs"][idx], flat["act"][idx])
        lr = logp - flat["logp"][idx]
        ratio = torch.exp(lr)
        pg = -torch.min(a * ratio, a * torch.clamp(ratio, 1 - cfg.clip_range, 1 + cfg.clip_range)).mean()
        vl = torch.nn.functional.mse_loss(v, ret[idx])
        loss = pg + cfg.vf_coef * vl - cfg.ent_coef * ent.mean()
        self.opt.zero_grad(set_to_none=False)
        loss.backward()
        self._allreduce_grads()
        nn.utils.clip_grad_norm_(self.policy.parameters(), cfg.max_grad_norm)
        self.opt.step()
        self._last_info.copy_(torch.stack([pg.detach(), vl.detach(), ((ratio - 1) - lr).mean().detach()]))

    def _restore_optimizer(self, saved: dict) -> None:
        """Write a saved `opt.state_dict()` back IN PLACE (a captured graph holds the addresses of the live state
        tensors); entries the snapshot lacks (fresh optimiser) restart from zero."""
        params = [p for g in self.opt.param_groups for p in g["params"]]
        for i, p in enumerate(params):
            old = saved["state"].get(i, {})
            for k, v in self.opt.state.get(p, {}).items():
                if torch.is_tensor(v):
                    if k in old:
                        v.copy_(torch.as_tensor(old[k]).to(device=v.device, dtype=v.dtype))
                    else:
                        v.zero_()

    def _build_graph(self, flat, mb):
        """Capture one minibatch step on static tensors; replayed n_epochs * n_minibatches times per iteration.
        Weights AND optimiser state (Adam moments, step: possibly restored from a checkpoint before the first update)
        are snapshotted before the warm-up steps and written back after capture."""
        import copy
        self._idx = torch.zeros(mb, dtype=torch.long, device=self.device)
        side = torch.cuda.Stream(self.device)
        side.wait_stream(torch.cuda.current_stream(self.device))
        saved = {k: v.clone() for k, v in self.policy.state_dict().items()}
        saved_opt = copy.deepcopy(self.opt.state_dict())
        with torch.cuda.stream(side):  # warm-up outside capture (allocations, optimizer state)
            for _ in range(3):
                self._minibatch_step(self._idx, flat, self._adv, self._ret)
        torch.cuda.current_stream(self.device).wait_stream(side)
        self._graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(self._graph):
            self._minibatch_step(self._idx, flat, self._adv, self._ret)
        self.policy.load_state_dict(saved)  # undo the warm-up updates
        self._restore_optimizer(saved_opt)

    def update(self, adv, ret):
        cfg, b = self.cfg, self.buf
        T, n = b["rew"].shape
        flat = {k: v.view(T * n, *v.shape[2:]) for k, v in b.items()}
        total = T * n
        mb = total // cfg.n_minibatches
        if not hasattr(self, "_adv"):
            self._adv, self._ret = torch.zeros(total, device=self.device), torch.zeros(total, device=self.device)
            self._last_info = torch.zeros(3, device=self.device)
            self._graph = None
            if cfg.cuda_graph and self.device.type == "cuda":
                try:
                    self._build_graph(flat, mb)
                except Exception as e:  # noqa: BLE001  - fall back to eager updates, loudly
                    print(f"[ppo] CUDA-graph capture failed ({type(e).__name__}: {e}); using eager updates", flush=True)
                    self._graph = None
        self._adv.copy_(adv.reshape(-1)); self._ret.copy_(ret.reshape(-1))
        for _ in range(cfg.n_epochs):
            perm = torch.randperm(total, device=self.device)
            for k in range(cfg.n_minibatches):
                idx = perm[k * mb:(k + 1) * mb]
                if self._graph is not None:
                    self._idx.copy_(idx)
                    self._graph.replay()
                else:
                    self._minibatch_step(idx, flat, self._adv, self._ret)
        pg, vl, kl = self._last_info.tolist()
        return {"pg_loss": pg, "v_loss": vl, "approx_kl": kl}

    def _log_std_mean(self) -> float:
        return float(self.policy.log_std.mean())

    def load_policy(self, policy: MlpPolicy) -> None:
        self.policy.load_state_dict(policy.state_dict())

    def state_dict(self) -> dict:
        """Everything a resumed run needs: weights, Adam moments and step, sample counter."""
        return {"kind": "torch", "policy": self.policy.state_dict(), "optimizer": self.opt.state_dict(), "samples": self.stats.samples,
                "config": dataclasses.asdict(self.cfg)}

    def load_state_dict(self, sd: dict) -> None:
        self.policy.load_state_dict(sd["policy"])
        if sd.get("kind") == "torch" and "optimizer" in sd:
            self.opt.load_state_dict(sd["optimizer"])
        self.stats.samples = int(sd.get("samples", 0))


class FusedPPO(_LearnLoop):
    """PPO on the hand-written kernels of include/so100_ppo.h; same interface and hyper-parameters as `PPO`.

    `env` must be a `BatchedSo100Env` (CUDA tensors with stable addresses: the kernels read `env.obs` etc. in place).
    Initial weights are those `PPO` would start from for the same seed (torch's orthogonal init), so the two learners
    can be compared step by step."""

    def __init__(self, env, cfg: PPOConfig | None = None, env_offset: int = 0):
        import ctypes

        from . import _native
        self.env, self.cfg = env, cfg or PPOConfig()
        self.device = env.device
        if self.device.type != "cuda":
            raise ValueError("FusedPPO runs on CUDA devices only (use PPO for CPU tensors)")
        self._L, self._check, self._ct = _native.lib(), _native.check, ctypes
        self.od, n, T = env.obs_dim, env.num_envs, self.cfg.n_steps
        self.sde = bool(self.cfg.use_sde)  # gSDE: the _sde_ entry points for act and grad, the shared ones for the rest
        self._act_fn = self._L.so100_ppo_sde_act if self.sde else self._L.so100_ppo_act
        self._grad_fn = self._L.so100_ppo_sde_grad if self.sde else self._L.so100_ppo_grad
        self.n_params = self._check((self._L.so100_ppo_sde_param_count if self.sde else self._L.so100_ppo_param_count)(self.od))
        self.n_log_std = 64 * env.act_dim if self.sde else env.act_dim
        torch.manual_seed(self.cfg.seed)
        self.params = pack_params(self._new_policy()).to(self.device)
        self.world = dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1
        if self.world > 1:
            dist.broadcast(self.params, src=0)
        f = dict(device=self.device, dtype=torch.float32)
        self.exp_avg, self.exp_avg_sq = torch.zeros(self.n_params, **f), torch.zeros(self.n_params, **f)
        self.grad = torch.zeros(self.n_params, **f)
        self.step_count = torch.zeros(1, device=self.device, dtype=torch.int32)
        ws = self._L.so100_ppo_sde_workspace_floats if self.sde else self._L.so100_ppo_workspace_floats
        self.workspace = torch.zeros(int(ws(self.od)), **f)
        self.loss = torch.zeros(3, **f)
        self.buf = {"obs": torch.zeros((T, n, self.od), **f), "act": torch.zeros((T, n, env.act_dim), **f), "logp": torch.zeros((T, n), **f),
                    "val": torch.zeros((T, n), **f), "rew": torch.zeros((T, n), **f), "done": torch.zeros((T, n), **f)}
        self.adv, self.ret = torch.zeros((T, n), **f), torch.zeros((T, n), **f)
        self.act_clip, self.last_val = torch.zeros((n, env.act_dim), **f), torch.zeros(n, **f)
        self._acc = torch.zeros(4, device=self.device, dtype=torch.float64)
        self.env_offset, self.tick = int(env_offset), 0
        self.sde_key = 0  # gSDE: noise key of the exploration matrices in use
        self._perm, self._epoch = None, 0
        self.obs = env.reset()
        self.stats = PPOStats()

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _new_policy(self) -> MlpPolicy:
        return MlpPolicy(self.od, 6, log_std_init=self.cfg.log_std_init, use_sde=self.sde)

    def act(self, obs: torch.Tensor, deterministic: bool = False):
        """Policy inference on arbitrary observations [n, od] -> (raw action, clipped action, log-prob, value).
        gSDE draws with the exploration matrices in use (those of the last rollout step)."""
        n = obs.shape[0]
        f = dict(device=self.device, dtype=torch.float32)
        a, c, lp, v = torch.empty((n, 6), **f), torch.empty((n, 6), **f), torch.empty(n, **f), torch.empty(n, **f)
        self.tick += 1
        self._check(self._act_fn(self.od, self.params.data_ptr(), obs.contiguous().data_ptr(), n, self.cfg.seed, self.env_offset,
                                 self.sde_key if self.sde else self.tick, int(deterministic), a.data_ptr(), c.data_ptr(), lp.data_ptr(),
                                 v.data_ptr(), None, self._stream()))
        return a, c, lp, v

    @torch.no_grad()
    def collect(self):
        cfg, b, L, st, P = self.cfg, self.buf, self._L, self._stream(), self.params.data_ptr()
        n = self.env.num_envs
        for t in range(cfg.n_steps):
            self.tick += 1
            key = self.tick
            if self.sde:
                key = self.sde_key = sde_noise_key(t, self.tick, cfg.sde_sample_freq, self.sde_key)
            self._check(self._act_fn(self.od, P, self.obs.data_ptr(), n, cfg.seed, self.env_offset, key, 0, b["act"][t].data_ptr(),
                                     self.act_clip.data_ptr(), b["logp"][t].data_ptr(), b["val"][t].data_ptr(), b["obs"][t].data_ptr(), st))
            r = self.env.step(self.act_clip)  # SB3 clips Box actions before env.step (the log-prob is of the raw action)
            self._check(L.so100_ppo_post_step(self.od, P, n, r.reward.data_ptr(), r.terminated.data_ptr(), r.truncated.data_ptr(),
                                              r.terminal_obs.data_ptr(), r.ep_return.data_ptr(), r.ep_len.data_ptr(), cfg.gamma,
                                              b["rew"][t].data_ptr(), b["done"][t].data_ptr(), self._acc.data_ptr(), st))
            self.obs = r.obs
        self._check(self._act_fn(self.od, P, self.obs.data_ptr(), n, cfg.seed, self.env_offset, self.tick, 1, None, None, None,
                                 self.last_val.data_ptr(), None, st))
        self._check(L.so100_ppo_gae(b["rew"].data_ptr(), b["val"].data_ptr(), b["done"].data_ptr(), self.last_val.data_ptr(), cfg.n_steps, n,
                                    cfg.gamma, cfg.gae_lambda, self.adv.data_ptr(), self.ret.data_ptr(), st))
        return self.adv, self.ret

    def minibatch_step(self, idx: torch.Tensor, adv: torch.Tensor, ret: torch.Tensor):
        """One optimiser step on the samples idx (int64, device) of the flattened rollout buffers."""
        cfg, b, L, st = self.cfg, self.buf, self._L, self._stream()
        self._check(self._grad_fn(self.od, self.params.data_ptr(), b["obs"].data_ptr(), b["act"].data_ptr(), b["logp"].data_ptr(),
                                     adv.data_ptr(), ret.data_ptr(), idx.data_ptr(), idx.numel(), cfg.clip_range, cfg.vf_coef, cfg.ent_coef,
                                     int(cfg.normalize_advantage), self.workspace.data_ptr(), self.grad.data_ptr(), self.loss.data_ptr(), st))
        if self.world > 1:
            dist.all_reduce(self.grad)  # ~10^4 floats over NVLink: latency bound
        self._check(L.so100_ppo_adam(self.n_params, self.params.data_ptr(), self.grad.data_ptr(), self.exp_avg.data_ptr(),
                                     self.exp_avg_sq.data_ptr(), self.step_count.data_ptr(), 1.0 / self.world, cfg.max_grad_norm, cfg.lr,
                                     0.9, 0.999, 1e-5, st))

    def update(self, adv, ret):
        cfg = self.cfg
        total = adv.numel()
        mb = total // cfg.n_minibatches
        if self._perm is None or self._perm.numel() != total:
            self._perm = torch.empty(total, dtype=torch.int64, device=self.device)
        for _ in range(cfg.n_epochs):
            self._epoch += 1  # a fresh keyed permutation per epoch (SB3: np.random.permutation in RolloutBuffer.get)
            key = (cfg.seed * 0x9E3779B97F4A7C15 + self._epoch * 0xD1B54A32D192ED03) & 0xFFFFFFFFFFFFFFFF
            self._check(self._L.so100_ppo_permutation(total, key, self._perm.data_ptr(), self._stream()))
            for k in range(cfg.n_minibatches):
                self.minibatch_step(self._perm[k * mb:(k + 1) * mb], adv, ret)
        pg, vl, kl = self.loss.tolist()
        return {"pg_loss": pg, "v_loss": vl, "approx_kl": kl}

    def _log_std_mean(self) -> float:
        return float(self.params[-self.n_log_std:].mean())

    def load_policy(self, policy: MlpPolicy) -> None:
        """Continue from the weights of a torch MlpPolicy (Adam moments restart)."""
        if policy.use_sde != self.sde:
            raise ValueError(f"the policy {'uses' if policy.use_sde else 'does not use'} gSDE and the learner {'does' if self.sde else 'does not'}")
        self.params.copy_(pack_params(policy).to(self.device))
        self.exp_avg.zero_(); self.exp_avg_sq.zero_(); self.step_count.zero_()

    def state_dict(self) -> dict:
        """Everything a resumed run needs: weights (as an MlpPolicy state dict), Adam moments and step, counters."""
        return {"kind": "fused", "policy": self.policy.state_dict(), "exp_avg": self.exp_avg.clone(), "exp_avg_sq": self.exp_avg_sq.clone(),
                "step_count": int(self.step_count.item()), "tick": self.tick, "epoch": self._epoch, "samples": self.stats.samples,
                "sde_key": self.sde_key, "config": dataclasses.asdict(self.cfg)}

    def load_state_dict(self, sd: dict) -> None:
        pol = self._new_policy()
        pol.load_state_dict(sd["policy"])
        self.load_policy(pol)
        if sd.get("kind") == "fused":
            self.exp_avg.copy_(sd["exp_avg"].to(self.device)); self.exp_avg_sq.copy_(sd["exp_avg_sq"].to(self.device))
            self.step_count.fill_(int(sd["step_count"]))
            self.tick, self._epoch = int(sd.get("tick", 0)), int(sd.get("epoch", 0))
            self.sde_key = int(sd.get("sde_key", 0))
        self.stats.samples = int(sd.get("samples", 0))

    @property
    def policy(self) -> MlpPolicy:
        """The current weights as a torch MlpPolicy (export, evaluation, tests)."""
        return unpack_params(self.params, self._new_policy().to(self.device))
