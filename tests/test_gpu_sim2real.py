"""Actuator latency and joint-angle observation noise (so100_set_sim2real) on the GPU.

The contract pinned here:
  * latency [0, 0] and zero noise give the default ctx's bits, alone and with unit param ranges;
  * noise is output only, and is the documented function of (seed, global env id, tick, stream), recomputed on the host;
  * latencies are drawn at resets only, as documented, and a latency-d step composes exactly from two substeps calls;
  * with latency, the envs track an fp64 replay of the same servo targets;
  * every bit-exact contract of the library (shards, env groups, host paths, reruns, state round trips) still holds.
"""
import ctypes

import numpy as np
import pytest

from box_muller_ref import noise_tolerance as _noise_tolerance
from box_muller_ref import z_host as _z_host
from conftest import make_oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

STREAM_LAT_AUTO, STREAM_LAT_API = 14, 22
STREAM_OBS_STEP, STREAM_OBS_AUTO, STREAM_OBS_API = 24, 26, 28
ARM = ("qpos", "qpos_comp", "qvel", "qacc_warm", "snap")
SIGMA = [0.01, 0.02, 0.0, 0.03, 0.005, 0.04]  # joint 2 without noise: its column keeps its bits
TOL_Q, TOL_V = 2e-5, 1e-3  # test_gpu_parity.py's trajectory tolerances


def _s2r(latency=(0, 0), noise=0.0):
    from so100_mujoco_rl_b200.randomization import Sim2Real
    return Sim2Real(latency=latency, obs_noise=noise)


def _flags(contact=False, generic=False):
    from so100_mujoco_rl_b200.tasks import FLAG_ARM_CONTACT, FLAG_GENERIC_KERNEL
    return (FLAG_ARM_CONTACT if contact else 0) | (FLAG_GENERIC_KERNEL if generic else 0)


def _env(task, n, seed=5, **kw):
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    return BatchedSo100Env(task, n, device=0, seed=seed, **kw)


def _bits(t):
    t = t.contiguous()
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _same(a, b):
    return torch.equal(_bits(a), _bits(b))


def _same_dict(a, b):
    return all(_same(a[k], b[k]) for k in a)


def _actions(rng, n):
    return torch.from_numpy(rng.uniform(-1, 1, (n, 6)).astype(np.float32)).cuda()


def _driven_actions(rng, n):
    """Random actions with the Pitch pushed down: a good share of the arms reach the floor."""
    a = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
    a[:, 1] = np.clip(a[:, 1] + 0.6, -1, 1)
    return torch.from_numpy(a).cuda()


def _outputs_done_masked(r):
    """Outputs with the rows that are only defined for finished envs zeroed elsewhere."""
    done = (r.terminated | r.truncated).bool()
    tobs = torch.where(done[:, None], r.terminal_obs, torch.zeros_like(r.terminal_obs))
    epr = torch.where(done, r.ep_return, torch.zeros_like(r.ep_return))
    epl = torch.where(done, r.ep_len, torch.zeros_like(r.ep_len))
    return [r.obs.clone(), r.reward.clone(), r.terminated.clone(), r.truncated.clone(), tobs, epr, epl]


# ------------------------------------------------------------------------------------------------ host recomputation
def _latency_expected(seed, env_ids, tick, stream, lo, hi):
    from oracle.pyoracle import philox
    x = np.array([philox(seed, int(i), tick, stream)[0] for i in env_ids], dtype=np.uint64)
    return (lo + ((x * np.uint64(hi - lo + 1)) >> np.uint64(32))).astype(np.int32)


def _check_noisy_rows(got, clean, seed, env_ids, tick, stream, sigma):
    """got / clean: [k, >= 6] rows (numpy float32) of the noisy and the noise-free ctx for global env ids env_ids."""
    sig32 = np.asarray(sigma, dtype=np.float32)
    for row_g, row_c, i in zip(got, clean, env_ids):
        z, rad = _z_host(seed, int(i), tick, stream)
        noise = (sig32.astype(np.float64) * z).astype(np.float32)
        want = (row_c[:6].astype(np.float64) + noise.astype(np.float64)).astype(np.float32)
        tol = _noise_tolerance(sig32.astype(np.float64), rad, noise, want)
        on = sig32 != 0
        assert (np.abs(row_g[:6][on].astype(np.float64) - want[on]) <= tol[on]).all(), (i, row_g[:6], want, tol)
        assert (row_g[:6][~on].view(np.int32) == row_c[:6][~on].view(np.int32)).all()
        assert (row_g[6:].view(np.int32) == row_c[6:].view(np.int32)).all()


# ------------------------------------------------------------------------------------------------ 1. identity
@pytest.mark.parametrize("task", [1, 2, 5, 6])
@pytest.mark.parametrize("contact", [False, True])
def test_zero_latency_and_noise_give_the_default_bits(task, contact):
    """300 steps under a short TimeLimit, half on so100_step, half on so100_step_host; alone and with unit ranges."""
    from so100_mujoco_rl_b200.randomization import ParamRanges
    n, limit = 512, 23 if task != 5 else 41
    kw = dict(flags=_flags(contact), max_episode_steps=limit)
    envs = [_env(task, n, **kw), _env(task, n, sim2real=_s2r(), **kw), _env(task, n, sim2real=_s2r(), param_ranges=ParamRanges(), **kw)]
    assert all(e.kernel_variant == "specialised" for e in envs)
    first = [e.reset() for e in envs]
    assert all(_same(first[0], o) for o in first[1:])
    rng = np.random.default_rng(task)
    hosts = [e.alloc_host() for e in envs]
    dones = 0
    for t in range(300):
        act = (_driven_actions if contact else _actions)(rng, n)
        if t < 150:
            outs = [_outputs_done_masked(e.step(act)) for e in envs]
            dones += int((outs[0][2] | outs[0][3]).sum())
        else:
            outs = []
            for e, h in zip(envs, hosts):
                h["actions"].copy_(act.cpu())
                e.step_host(h)
                outs.append([h[k].clone() for k in ("obs", "reward", "terminated", "truncated", "terminal_obs", "ep_return")])
        assert all(_same(x, y) for o in outs[1:] for x, y in zip(outs[0], o)), f"step {t}"
    assert dones > 2 * n
    st = envs[0].get_state()
    assert all(_same_dict(st, e.get_state()) for e in envs[1:])
    assert (envs[1].get_actuator_state()["latency"] == 0).all()


# ------------------------------------------------------------------------------------------------ 2. noise
@pytest.mark.parametrize("task", [1, 2, 6])
def test_noise_is_output_only_and_matches_the_host_draws(task):
    n, seed, limit = 512, 21, 9
    a = _env(task, n, seed=seed, max_episode_steps=limit, sim2real=_s2r(noise=SIGMA))
    b = _env(task, n, seed=seed, max_episode_steps=limit)
    oa, ob = a.reset().cpu().numpy(), b.reset().cpu().numpy()
    rows = np.arange(0, n, 7)
    _check_noisy_rows(oa[rows], ob[rows], seed, rows, 0, STREAM_OBS_API, SIGMA)
    rng = np.random.default_rng(2)
    checked = dict(step=0, terminal=0, auto=0, api=0)
    for t in range(40):
        act = _actions(rng, n)
        ra, rb = a.step(act), b.step(act)
        for x, y in zip(_outputs_done_masked(ra)[1:], _outputs_done_masked(rb)[1:]):
            if x.dim() == 2:
                assert _same(x[:, 6:], y[:, 6:]), f"step {t}"
            else:
                assert _same(x, y), f"step {t}"
        assert _same(ra.obs[:, 6:], rb.obs[:, 6:])
        assert _same_dict(a.get_state(), b.get_state()), f"step {t}"
        tick = a.tick
        done = (ra.terminated | ra.truncated).cpu().numpy().astype(bool)
        ga, gb = ra.obs.cpu().numpy(), rb.obs.cpu().numpy()
        live = np.flatnonzero(~done)[::11]
        _check_noisy_rows(ga[live], gb[live], seed, live, tick, STREAM_OBS_STEP, SIGMA)
        checked["step"] += len(live)
        ids = np.flatnonzero(done)[:40]
        if len(ids):
            ta, tb = ra.terminal_obs.cpu().numpy(), rb.terminal_obs.cpu().numpy()
            _check_noisy_rows(ta[ids], tb[ids], seed, ids, tick, STREAM_OBS_STEP, SIGMA)
            _check_noisy_rows(ga[ids], gb[ids], seed, ids, tick, STREAM_OBS_AUTO, SIGMA)
            checked["terminal"] += len(ids); checked["auto"] += len(ids)
        if t == 20:  # masked so100_reset in the middle of the run
            mask = torch.from_numpy(rng.random(n) < 0.3).cuda()
            ma, mb = a.reset(mask).cpu().numpy(), b.reset(mask).cpu().numpy()
            ids = np.flatnonzero(mask.cpu().numpy())[:60]
            _check_noisy_rows(ma[ids], mb[ids], seed, ids, a.tick, STREAM_OBS_API, SIGMA)
            checked["api"] += len(ids)
    assert min(checked.values()) > 30, checked


def test_noise_is_standard_normal_per_joint():
    from scipy import stats
    n, seed = 65536, 3
    a = _env(1, n, seed=seed, sim2real=_s2r(noise=SIGMA))
    b = _env(1, n, seed=seed)
    a.reset(); b.reset()
    rng = np.random.default_rng(9)
    z = [[] for _ in range(6)]
    for _ in range(4):
        act = _actions(rng, n)
        ga, gb = a.step(act).obs.cpu().numpy().astype(np.float64), b.step(act).obs.cpu().numpy().astype(np.float64)
        for j in range(6):
            if SIGMA[j] > 0:
                z[j].append((ga[:, j] - gb[:, j]) / float(np.float32(SIGMA[j])))
            else:
                assert (ga[:, j] == gb[:, j]).all()
    pooled = []
    for j in range(6):
        if SIGMA[j] > 0:
            zj = np.concatenate(z[j])
            assert stats.kstest(zj, "norm").pvalue > 1e-4, j
            pooled.append(zj)
    pooled = np.concatenate(pooled)
    assert pooled.size >= 10 ** 6
    assert stats.kstest(pooled, "norm").pvalue > 1e-4


def test_env05_refuses_noise():
    from so100_mujoco_rl_b200._native import lib
    env = _env(5, 256)
    c = _s2r().to_ctypes()
    c.obs_noise[3] = 0.01
    assert lib().so100_set_sim2real(env._h, ctypes.byref(c)) == -1
    assert b"Env05" in lib().so100_last_error()
    with pytest.raises(ValueError):
        env.set_sim2real(_s2r(noise=0.01))
    env.set_sim2real(_s2r(latency=(0, 16)))  # latency alone is fine
    assert set(env.get_actuator_state()) == {"latency"}


# ------------------------------------------------------------------------------------------------ 3. latency draws
def test_latency_draws_are_reproducible_uniform_and_change_only_at_resets():
    from scipy import stats
    n, seed, lo, hi = 65536, 7, 3, 11
    env = _env(1, n, seed=seed, max_episode_steps=10, sim2real=_s2r(latency=(lo, hi)))
    assert (env.get_actuator_state()["latency"] == 0).all()  # until each env's next reset
    env.reset()
    d0 = env.get_actuator_state()["latency"].cpu().numpy()
    rng = np.random.default_rng(3)
    sample = np.unique(np.concatenate([rng.choice(n, 300, replace=False), [0, n - 1]]))
    assert (d0[sample] == _latency_expected(seed, sample, 0, STREAM_LAT_API, lo, hi)).all()
    counts = np.bincount(d0 - lo, minlength=hi - lo + 1)
    assert d0.min() == lo and d0.max() == hi and counts.size == hi - lo + 1
    assert stats.chisquare(counts).pvalue > 1e-4
    st = env.get_state()
    cp = env.get_actuator_state()
    assert _same(cp["ctrl_prev_hi"], st["qpos"]) and (cp["ctrl_prev_lo"] == 0).all()  # the reset pose
    env.stagger_episodes(seed=1)
    prev = d0
    for t in range(12):
        q_start = env.get_state()["qpos"]
        res = env.step(_actions(rng, n))
        done = (res.terminated | res.truncated).cpu().numpy().astype(bool)
        act = env.get_actuator_state()
        cur = act["latency"].cpu().numpy()
        assert 0.05 * n < done.sum() < 0.15 * n
        assert (cur[~done] == prev[~done]).all(), f"step {t}"
        ids = np.flatnonzero(done)
        assert (cur[ids[:200]] == _latency_expected(seed, ids[:200], env.tick, STREAM_LAT_AUTO, lo, hi)).all()
        assert (cur[ids] != prev[ids]).mean() > 0.8  # 1 / 9 of the redraws repeat the old value
        # ctrl_prev: this step's target (hi = the step's start position) where the env ran on, the reset pose where it reset
        dm = torch.from_numpy(done).cuda()
        q_now = env.get_state()["qpos"]
        assert _same(act["ctrl_prev_hi"][:, ~dm], q_start[:, ~dm])
        assert _same(act["ctrl_prev_hi"][:, dm], q_now[:, dm]) and (act["ctrl_prev_lo"][:, dm] == 0).all()
        prev = cur
    mask = torch.from_numpy(rng.random(n) < 0.3).cuda()
    env.reset(mask)
    cur = env.get_actuator_state()["latency"].cpu().numpy()
    m = mask.cpu().numpy().astype(bool)
    assert (cur[~m] == prev[~m]).all()
    ids = np.flatnonzero(m)[:200]
    assert (cur[ids] == _latency_expected(seed, ids, env.tick, STREAM_LAT_API, lo, hi)).all()


def test_latency_draws_use_the_global_env_id():
    n, seed, off = 300, 4, 1000
    env = _env(2, n, seed=seed, env_offset=off, sim2real=_s2r(latency=(0, 16)))
    env.reset()
    d = env.get_actuator_state()["latency"].cpu().numpy()
    assert (d == _latency_expected(seed, np.arange(off, off + n), 0, STREAM_LAT_API, 0, 16)).all()


# ------------------------------------------------------------------------------------------------ 4. / 5. exactness
def test_latency_step_composes_from_two_substeps_calls_env05():
    """Generic kernel with arm contact: the step and so100_step_substeps run the same physics<> instantiation."""
    nsub, reps = 16, 8
    n = (nsub + 1) * reps
    flags = _flags(contact=True, generic=True)
    env = _env(5, n, seed=4, flags=flags, max_episode_steps=100000, sim2real=_s2r(latency=(0, nsub)))
    plain = _env(5, n, seed=4, flags=flags, max_episode_steps=100000)
    assert env.kernel_variant == plain.kernel_variant == "generic"
    env.reset()
    rng = np.random.default_rng(1)
    for _ in range(40):
        env.step(_driven_actions(rng, n))
    d = torch.arange(n, device="cuda", dtype=torch.int32) % (nsub + 1)
    env.set_actuator_state({"latency": d})
    st = env.get_state()
    res = env.step(_driven_actions(rng, n))
    end = env.get_state()
    done = (res.terminated | res.truncated).bool()
    prev_cmd, new_cmd = st["aux"][:6].T.contiguous(), end["aux"][:6].T.contiguous()  # Env05's command before / after
    touching = int(((st["counters"][1] & 16) != 0).sum())
    print(f"{touching} of {n} envs touch the floor")
    assert touching > 0
    compared = 0
    for k in range(nsub + 1):
        plain.set_state(st)
        if k > 0:
            plain.step_substeps(prev_cmd, k)
        if k < nsub:
            plain.step_substeps(new_cmd, nsub - k)
        got = plain.get_state()
        cols = ((d == k) & ~done).nonzero().flatten()
        for f in ARM:
            assert _same(got[f][:, cols], end[f][:, cols]), (k, f)
        compared += len(cols)
    assert compared > 0.9 * n


@pytest.mark.parametrize("task", [1, 2, 6])
def test_full_latency_first_step_is_a_zero_action_step(task):
    n, seed = 1024, 8
    env = _env(task, n, seed=seed, sim2real=_s2r(latency=(16, 16)))
    ref = _env(task, n, seed=seed)
    assert _same(env.reset(), ref.reset())
    rng = np.random.default_rng(task)
    ra, rb = env.step(_actions(rng, n)), ref.step(torch.zeros((n, 6), device="cuda"))
    assert all(_same(x, y) for x, y in zip(_outputs_done_masked(ra), _outputs_done_masked(rb)))
    assert _same_dict(env.get_state(), ref.get_state())


# ------------------------------------------------------------------------------------------------ 6. oracle tracking
@pytest.mark.parametrize("task", [1, 2, 5, 6])
def test_latency_tracks_an_fp64_replay(task):
    """The fp64 replay composes Oracle.substeps: d substeps on the previous target, 16 - d on the new one.  Envs that reset
    are re-synchronised to the device's reset state (the draws are checked above)."""
    from so100_mujoco_rl_b200.tasks import JOINT_STEP_SCALE
    n, steps, limit = 256, 300, 100
    env = _env(task, n, seed=11, max_episode_steps=limit, sim2real=_s2r(latency=(0, 16)))
    o = make_oracle(task, 1)
    env.reset()
    st = env.get_state()
    q, v, w = (st[k].cpu().numpy().T.astype(np.float64) for k in ("qpos", "qvel", "qacc_warm"))
    prev = st["qpos"].cpu().numpy().T.astype(np.float64) if task != 5 else st["aux"][:6].cpu().numpy().T.astype(np.float64)
    rng = np.random.default_rng(5)
    worst_q = worst_v = 0.0
    resets = 0
    for t in range(steps):
        d = env.get_actuator_state()["latency"].cpu().numpy()
        a = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
        r = env.step(torch.from_numpy(a).cuda())
        st = env.get_state()
        done = (r.terminated | r.truncated).cpu().numpy().astype(bool)
        if task == 5:
            new = st["aux"][:6].cpu().numpy().T.astype(np.float64)  # the device's fp32 commands
        for i in range(n):
            tgt = q[i] + a[i].astype(np.float64) * JOINT_STEP_SCALE if task != 5 else new[i]
            if d[i] > 0:
                q[i], v[i], w[i] = o.substeps(q[i], v[i], w[i], prev[i], int(d[i]))
            if d[i] < 16:
                q[i], v[i], w[i] = o.substeps(q[i], v[i], w[i], tgt, 16 - int(d[i]))
            prev[i] = tgt
        gq, gv = st["qpos"].cpu().numpy().T, st["qvel"].cpu().numpy().T
        ok = ~done  # (every env truncates at once at the TimeLimit)
        if ok.any():
            worst_q = max(worst_q, float(np.abs(gq[ok] - q[ok]).max()))
            worst_v = max(worst_v, float(np.abs(gv[ok] - v[ok]).max()))
        if done.any():
            resets += int(done.sum())
            q[done], v[done] = gq[done], gv[done]
            w[done] = st["qacc_warm"].cpu().numpy().T[done]
            prev[done] = gq[done] if task != 5 else st["aux"][:6].cpu().numpy().T[done]
    print(f"task {task}: max|dq| {worst_q:.2e} max|dv| {worst_v:.2e} resets {resets}")
    assert resets >= n
    assert worst_q < TOL_Q and worst_v < TOL_V


# ------------------------------------------------------------------------------------------------ 7. library contracts
def _run(env, rng_seed, steps, n, contact=False):
    rng = np.random.default_rng(rng_seed)
    return [_outputs_done_masked(env.step((_driven_actions if contact else _actions)(rng, n))) for _ in range(steps)]


ALL = dict(latency=(0, 16), noise=SIGMA)


@pytest.mark.parametrize("contact", [False, True])
def test_shards_equal_the_full_batch(contact):
    from so100_mujoco_rl_b200.randomization import ParamRanges
    n, lim = 512, 20
    kw = dict(seed=9, flags=_flags(contact), max_episode_steps=lim, sim2real=_s2r(**ALL),
              param_ranges=ParamRanges.parse("kp=0.7:1.3,frictionloss=0.5:2"))
    full = _env(2, n, **kw)
    parts = [_env(2, 300, env_offset=0, **kw), _env(2, 212, env_offset=300, **kw)]
    full.reset(); [p.reset() for p in parts]
    full.stagger_episodes(seed=2)
    st, ac = full.get_state(), full.get_actuator_state()
    for p, sl in ((parts[0], slice(0, 300)), (parts[1], slice(300, n))):
        p.set_state({k: v[:, sl] for k, v in st.items()})
        p.set_actuator_state({k: (v[sl] if v.dim() == 1 else v[:, sl]) for k, v in ac.items()})
    rng = np.random.default_rng(4)
    for t in range(60):
        act = (_driven_actions if contact else _actions)(rng, n)
        fo = _outputs_done_masked(full.step(act))
        po = [_outputs_done_masked(parts[0].step(act[:300])), _outputs_done_masked(parts[1].step(act[300:]))]
        assert all(_same(f, torch.cat([po[0][k], po[1][k]])) for k, f in enumerate(fo)), f"step {t}"
    fa = full.get_actuator_state()
    pa = [p.get_actuator_state() for p in parts]
    assert all(_same(fa[k], torch.cat([pa[0][k], pa[1][k]], dim=-1)) for k in fa)


def test_async_groups_host_paths_rerun_and_roundtrip_are_bit_exact():
    from so100_mujoco_rl_b200.randomization import ParamRanges
    n, lim = 1024, 15
    kw = dict(seed=6, max_episode_steps=lim, sim2real=_s2r(**ALL), param_ranges=ParamRanges.parse("kp=0.7:1.3"))
    a, b, p = _env(6, n, **kw), _env(6, n, **kw), _env(6, n, **kw)
    for e in (a, b, p):
        e.reset(); e.stagger_episodes(seed=3)
    ha, hb = a.alloc_host(), b.alloc_host()
    hp = {k: torch.zeros_like(v) for k, v in p.alloc_host().items()}  # pageable
    assert not hp["obs"].is_pinned()
    groups = b.host_groups(4)
    rng = np.random.default_rng(8)
    keys = ("obs", "reward", "terminated", "truncated", "terminal_obs")
    for t in range(40):
        act = _actions(rng, n).cpu()
        for h in (ha, hb, hp):
            h["actions"].copy_(act)
        a.step_host(ha); p.step_host(hp)
        for g in range(len(groups)):
            b.step_host_async(hb, g)
        for g in range(len(groups)):
            b.step_host_wait(g)
        done = (ha["terminated"] | ha["truncated"]).bool()
        for k in keys:
            x, y, z = ha[k], hb[k], hp[k]
            if k == "terminal_obs":
                x, y, z = x[done], y[done], z[done]
            assert _same(x, y) and _same(x, z), f"{k} step {t}"
    for e in (b, p):
        assert _same_dict(a.get_actuator_state(), e.get_actuator_state()) and _same_dict(a.get_state(), e.get_state())
    # same-seed rerun on the device path
    c = _env(6, n, **kw)
    c.reset(); c.stagger_episodes(seed=3)
    rng = np.random.default_rng(8)
    for t in range(40):
        c.step(_actions(rng, n))
    assert _same_dict(a.get_actuator_state(), c.get_actuator_state()) and _same_dict(a.get_state(), c.get_state())
    # state + actuator state + params + tick into a fresh ctx: it continues bit for bit
    saved = (c.get_state(), c.get_actuator_state(), c.get_params(), c.tick)
    ref = _run(c, 21, 30, n)
    d = _env(6, n, **kw)
    d.set_state(saved[0]); d.set_actuator_state(saved[1]); d.set_params(saved[2]); d.tick = saved[3]
    got = _run(d, 21, 30, n)
    assert all(_same(x, y) for ro, go in zip(ref, got) for x, y in zip(ro, go))
    assert _same_dict(c.get_actuator_state(), d.get_actuator_state())


def test_set_actuator_state_holds_until_reset_and_switching_off_restores_the_default_kernel():
    from so100_mujoco_rl_b200._native import So100Error
    n = 512
    env = _env(1, n, seed=1, max_episode_steps=100000, sim2real=_s2r(latency=(0, 4)))
    env.reset()
    mine = torch.full((n,), 13, dtype=torch.int32, device="cuda")
    env.set_actuator_state({"latency": mine})
    _run(env, 1, 10, n)
    assert _same(env.get_actuator_state()["latency"], mine)
    mask = torch.zeros(n, dtype=torch.uint8, device="cuda")
    mask[::3] = 1
    env.reset(mask)
    after = env.get_actuator_state()["latency"]
    keep = mask == 0
    assert _same(after[keep], mine[keep]) and (after[~keep] <= 4).all()
    # off: the default kernel, bit for bit with a default ctx from the same state
    env.set_sim2real(None)
    with pytest.raises(So100Error):
        env.get_actuator_state()
    with pytest.raises(So100Error):
        env.set_actuator_state({"latency": mine})
    ref = _env(1, n, seed=1, max_episode_steps=100000)
    ref.set_state(env.get_state()); ref.tick = env.tick
    assert all(_same(x, y) for ro, go in zip(_run(ref, 5, 20, n), _run(env, 5, 20, n)) for x, y in zip(ro, go))
    assert _same_dict(ref.get_state(), env.get_state())
    # ranges on and sim2real off, then ranges off too
    from so100_mujoco_rl_b200.randomization import ParamRanges
    env.set_sim2real(_s2r(latency=(2, 2)))
    env.set_param_ranges(ParamRanges())
    env.set_param_ranges(None)
    with pytest.raises(So100Error):
        env.get_params()
    assert (env.get_actuator_state()["latency"] == 0).all()  # the first set: d = 0 until the next reset
    env.set_sim2real(None)
    env.set_param_ranges(None)
    assert all(_same(x, y) for ro, go in zip(_run(ref, 6, 10, n), _run(env, 6, 10, n)) for x, y in zip(ro, go))


def test_bad_configs_and_group_steps_in_flight_are_refused():
    from so100_mujoco_rl_b200._native import So100Error, lib
    from so100_mujoco_rl_b200.randomization import So100ActuatorView, So100Sim2Real
    env = _env(1, 512, sim2real=_s2r())
    L = lib()
    for lat in ((-1, 2), (3, 2), (0, 17)):
        c = _s2r().to_ctypes()
        c.latency[0], c.latency[1] = lat
        assert L.so100_set_sim2real(env._h, ctypes.byref(c)) == -1
    for bad in (-0.1, float("nan"), float("inf"), 1e39):
        c = _s2r().to_ctypes()
        c.obs_noise[4] = bad
        assert L.so100_set_sim2real(env._h, ctypes.byref(c)) == -1
    c = _s2r().to_ctypes()
    c.struct_size = ctypes.sizeof(So100Sim2Real) - 8
    assert L.so100_set_sim2real(env._h, ctypes.byref(c)) == -1
    off = _env(1, 512)
    v = So100ActuatorView()
    assert L.so100_get_actuator_state(off._h, ctypes.byref(v), None) == -4  # SO100_ERR_STATE: no config set
    env.reset()
    h = env.alloc_host()
    env.host_groups(2)
    env.step_host_async(h, 0)
    with pytest.raises(So100Error):
        env.get_actuator_state()
    with pytest.raises(So100Error):
        env.set_sim2real(None)
    env.step_host_wait(0)
    env.get_actuator_state()


# ------------------------------------------------------------------------------------------------ 8. CLI
def test_cli_train_latency_and_noise_checkpoint_and_resume(tmp_path):
    from click.testing import CliRunner
    from so100_mujoco_rl_b200.cli import cli
    common = ["-e", "Env01", "--num-envs", "256", "--n-steps", "8", "--eval-envs", "0", "--tensorboard-log", "",
              "--save-freq", "1000000000", "--out", str(tmp_path)]
    res = CliRunner().invoke(cli, ["-a", "PPO", "train", *common, "--total-timesteps", "4096", "--latency", "0:8", "--obs-noise", "0.01"],
                             obj={}, catch_exceptions=False)
    assert res.exit_code == 0, res.output
    path = tmp_path / "Env01_PPO" / "final_model.pt"
    ck = torch.load(path, map_location="cpu", weights_only=False)
    assert ck["env"]["sim2real"] == {"latency": [0, 8], "obs_noise": [0.01] * 6}
    A = ck["env"]["actuator"]
    assert set(A) == {"latency", "ctrl_prev_hi", "ctrl_prev_lo"} and A["latency"].shape == (256,) and A["ctrl_prev_hi"].shape == (6, 256)
    assert int(A["latency"].min()) >= 0 and int(A["latency"].max()) <= 8 and len(set(A["latency"].tolist())) > 1
    out2 = tmp_path / "resumed"
    res = CliRunner().invoke(cli, ["-a", "PPO", "-m", str(path), "train", *common[:-2], "--out", str(out2), "--total-timesteps", "0"],
                             obj={}, catch_exceptions=False)
    assert res.exit_code == 0, res.output
    ck2 = torch.load(out2 / "Env01_PPO" / "final_model.pt", map_location="cpu", weights_only=False)
    assert ck2["env"]["sim2real"] == ck["env"]["sim2real"] and ck2["env"]["tick"] == ck["env"]["tick"]
    assert all(_same(ck2["env"]["actuator"][k], A[k]) for k in A)
    assert all(_same(ck2["env"]["state"][k], ck["env"]["state"][k]) for k in ck["env"]["state"])
    bad = CliRunner().invoke(cli, ["-a", "PPO", "train", "-e", "Env05", *common[2:], "--obs-noise", "0.01"], obj={})
    assert bad.exit_code != 0
