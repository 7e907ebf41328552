"""Per-env dynamics randomisation (so100_set_param_ranges) on the GPU.

Each env of a ctx with ranges set holds its own fp32 kp, kv, forcerange and friction loss and redraws them at every
episode reset.  The contract pinned here:
  * unit ranges give the default ctx's bits (the per-env kernels do the same arithmetic on the same values);
  * the draws are the documented function of (seed, global env id, tick, stream), reproduced on the host, and they change
    exactly for the envs that reset;
  * env i steps bit for bit like env i of a plain ctx whose model carries env i's values, and tracks the fp64 oracle built
    from that model;
  * every bit-exact contract of the library (shards, env groups, reruns, state round trips) holds under randomisation.
"""
import copy
import ctypes

import numpy as np
import pytest

from conftest import make_oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

STATE = ("qpos", "qpos_comp", "qvel", "qacc_warm", "block", "snap", "aux", "counters", "ep_return")
WIDE = "kp=0.5:2,damping=0.5:2,forcerange=0.8:1.2,frictionloss=0.5:2"
TYPICAL = "kp=0.7:1.3,damping=0.8:1.2,forcerange=0.8:1.0,frictionloss=0.5:2"
STREAM_AUTO, STREAM_API = 8, 16
TOL_Q, TOL_V, TOL_OBS = 2e-5, 1e-3, 2e-5  # test_gpu_parity.py's trajectory tolerances


def _ranges(spec=TYPICAL):
    from so100_mujoco_rl_b200.randomization import ParamRanges
    return ParamRanges.parse(spec)


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
    """Random actions with the Pitch pushed down: a good share of the arms reach the floor (test_gpu_contact_kernel.py)."""
    a = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
    a[:, 1] = np.clip(a[:, 1] + 0.6, -1, 1)
    return torch.from_numpy(a).cuda()


def _outputs(r):
    return [t.clone() for t in (r.obs, r.reward, r.terminated, r.truncated)]


def _params_mat(p):
    """{kp, kv, force_lo, force_hi, frictionloss} [6, N] -> [30, N]"""
    return torch.cat([p[k] for k in ("kp", "kv", "force_lo", "force_hi", "frictionloss")], dim=0)


def _expected(seed, env_ids, tick, stream, ranges, base):
    """Host recomputation of the draws: 6 Philox blocks per env, numpy float32 (every operation rounded on its own)."""
    from oracle.pyoracle import philox
    lo, hi = ranges.lo_hi_f32()
    kp0, kv0, flo0, fhi0, fl0 = (base[6 * k: 6 * k + 6] for k in range(5))
    out = []
    for i in env_ids:
        x = np.concatenate([philox(seed, int(i), tick, stream + k) for k in range(6)])
        u = (x >> np.uint32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)
        s = lo + (hi - lo) * u
        kp, sd, sf, sl = s[:6], s[6:12], s[12:18], s[18:24]
        out.append(np.concatenate([kp0 * kp, (kv0 * np.sqrt(kp)) * sd, flo0 * sf, fhi0 * sf, fl0 * sl]))
    return np.stack(out, axis=1)  # [30, len(env_ids)]


def _base(env):
    """The ctx's fp32 constants: what every env holds right after the first so100_set_param_ranges."""
    p = _params_mat(env.get_params()).cpu().numpy()
    assert (p == p[:, :1]).all()
    return p[:, 0].copy()


def _plain_spec(spec, P, i):
    """The so100 model carrying env i's values (P: get_params() on the host)."""
    m = copy.deepcopy(spec)
    m.act_kp = np.array(P["kp"][:, i], dtype=np.float64)
    m.act_dampratio = np.zeros(6)
    m.act_kv = np.array(P["kv"][:, i], dtype=np.float64)
    m.act_forcerange = np.stack([P["force_lo"][:, i], P["force_hi"][:, i]], axis=1).astype(np.float64)
    m.jnt_frictionloss = np.array(P["frictionloss"][:, i], dtype=np.float64)
    return m


def _col(st, i):
    return {k: v[:, i:i + 1].clone() for k, v in st.items()}


# ------------------------------------------------------------------------------------------------ identity
@pytest.mark.parametrize("task", [1, 2, 5, 6])
@pytest.mark.parametrize("contact", [False, True])
def test_unit_ranges_give_the_default_bits(task, contact):
    """300 steps under a short TimeLimit (every env resets many times), half on so100_step, half on so100_step_host."""
    from so100_mujoco_rl_b200.randomization import ParamRanges
    n, limit = 512, 23 if task != 5 else 41
    a = _env(task, n, flags=_flags(contact), max_episode_steps=limit)
    b = _env(task, n, flags=_flags(contact), max_episode_steps=limit, param_ranges=ParamRanges())
    assert a.kernel_variant == b.kernel_variant == "specialised"
    assert _same(a.reset(), b.reset())
    rng = np.random.default_rng(task)
    ha, hb = a.alloc_host(), b.alloc_host()
    dones = 0
    for t in range(300):
        act = (_driven_actions if contact else _actions)(rng, n)
        if t < 150:
            ra, rb = a.step(act), b.step(act)
            oa, ob = _outputs(ra), _outputs(rb)
            assert _same(ra.terminal_obs, rb.terminal_obs) and _same(ra.ep_return, rb.ep_return)
            dones += int((ra.terminated | ra.truncated).sum())
        else:
            ha["actions"].copy_(act.cpu()); hb["actions"].copy_(act.cpu())
            a.step_host(ha); b.step_host(hb)
            oa = [ha[k].clone() for k in ("obs", "reward", "terminated", "truncated", "terminal_obs", "ep_return")]
            ob = [hb[k].clone() for k in ("obs", "reward", "terminated", "truncated", "terminal_obs", "ep_return")]
        assert all(_same(x, y) for x, y in zip(oa, ob)), f"step {t}"
    assert dones > 2 * n
    assert _same_dict(a.get_state(), b.get_state())
    base = _base_values(b)
    assert (_params_mat(b.get_params()).cpu().numpy() == base[:, None]).all()  # unit scales: the model's values, bit for bit


def _base_values(env):
    import so100_mujoco_rl_b200._native as nat
    out = (ctypes.c_float * 146)()
    nat.check(nat.lib().so100_host_solver_constants(ctypes.byref(env._model_ct), out, 146))
    c = np.array(out, dtype=np.float32)
    # flat layout (include/so100_b200.h): ConC (16 x 6; fr_loss is row 2), then kp, kv, ctrl_lo, ctrl_hi, frc_lo, frc_hi
    kp, kv, flo, fhi = c[96:102], c[102:108], c[120:126], c[126:132]
    return np.concatenate([kp, kv, flo, fhi, c[12:18]])


# ------------------------------------------------------------------------------------------------ draws
def test_draws_are_reproducible_uniform_and_change_exactly_at_resets():
    from scipy import stats
    n, seed = 65536, 7
    r = _ranges()
    env = _env(1, n, seed=seed, max_episode_steps=10)
    env.set_param_ranges(r)
    base = _base(env)
    assert (base == _base_values(env)).all()
    env.reset()
    p0 = _params_mat(env.get_params()).cpu().numpy()
    rng = np.random.default_rng(3)
    sample = np.unique(np.concatenate([rng.choice(n, 200, replace=False), [0, n - 1]]))
    assert (p0[:, sample] == _expected(seed, sample, 0, STREAM_API, r, base)).all()
    # every scale in its range, and uniform (KS over all joints of 65 536 envs)
    lo, hi = r.lo_hi_f32()
    s_kp = p0[0:6] / base[0:6, None].astype(np.float64)
    scales = {0: s_kp, 1: p0[6:12] / (base[6:12, None] * np.sqrt(s_kp)), 2: p0[12:18] / base[12:18, None].astype(np.float64),
              3: p0[24:30] / base[24:30, None].astype(np.float64)}
    for g, s in scales.items():
        l, h = lo[6 * g: 6 * g + 6, None].astype(np.float64), hi[6 * g: 6 * g + 6, None].astype(np.float64)
        assert (s >= l * (1 - 1e-6)).all() and (s <= h * (1 + 1e-6)).all()
        pval = stats.kstest(((s - l) / (h - l)).ravel(), "uniform").pvalue
        assert pval > 1e-4, (g, pval)
    # auto-resets: staggered episode clocks, so that a tenth of the envs resets on every step
    env.stagger_episodes(seed=1)
    prev = p0
    for t in range(1, 13):
        res = env.step(_actions(rng, n))
        done = (res.terminated | res.truncated).cpu().numpy().astype(bool)
        cur = _params_mat(env.get_params()).cpu().numpy()
        changed = (cur != prev).any(axis=0)
        assert 0.05 * n < done.sum() < 0.15 * n
        assert (changed == done).all(), f"step {t}"
        ids = np.flatnonzero(done)[:64]
        assert (cur[:, ids] == _expected(seed, ids, env.tick, STREAM_AUTO, r, base)).all()
        prev = cur
    # masked so100_reset: exactly the masked envs redraw
    mask = torch.from_numpy(rng.random(n) < 0.3).cuda()
    env.reset(mask)
    cur = _params_mat(env.get_params()).cpu().numpy()
    m = mask.cpu().numpy()
    assert ((cur != prev).any(axis=0) == m).all()
    ids = np.flatnonzero(m)[:64]
    assert (cur[:, ids] == _expected(seed, ids, env.tick, STREAM_API, r, base)).all()
    # a new seed gives new draws
    env.seed(99)
    env.reset()
    p1 = _params_mat(env.get_params()).cpu().numpy()
    assert (p1 != p0).any(axis=0).mean() > 0.999
    assert (p1[:, sample] == _expected(99, sample, 0, STREAM_API, r, base)).all()
    env.close()


def test_draws_use_the_global_env_id():
    n, seed, off = 300, 4, 1000
    r = _ranges(WIDE)
    env = _env(2, n, seed=seed, env_offset=off, param_ranges=r)
    base = _base_values(env)
    env.reset()
    p = _params_mat(env.get_params()).cpu().numpy()
    assert (p == _expected(seed, np.arange(off, off + n), 0, STREAM_API, r, base)).all()


# ------------------------------------------------------------------------------------------------ exact replay
def _replay(task, contact, spec):
    n, seed, steps = 1024, 3, 200
    flags = _flags(contact=contact, generic=True)
    env = _env(task, n, seed=seed, flags=flags, max_episode_steps=100000, param_ranges=_ranges(WIDE))
    assert env.kernel_variant == "generic"
    env.reset()
    rng = np.random.default_rng(task + 10 * contact)
    if contact:  # drive the arms into the floor first (no episode ends: Env01/02/06 never terminate, the TimeLimit is far)
        for _ in range(60):
            env.step(_driven_actions(rng, n))
    st, tick = env.get_state(), env.tick
    P = {k: v.cpu().numpy() for k, v in env.get_params().items()}
    if contact:
        touching = np.flatnonzero((st["counters"][1] & 16).cpu().numpy() != 0)
        assert len(touching) > 0.1 * n
        ids = list(rng.choice(touching, 6, replace=False)) + [0, n - 1]
    else:
        ids = list(rng.choice(n, 6, replace=False)) + [0, n - 1]
    small = {}
    for i in ids:
        s = _env(task, 1, seed=seed, env_offset=int(i), flags=flags, max_episode_steps=100000, model=_plain_spec(spec, P, i))
        s.set_state(_col(st, i))
        s.tick = tick
        small[i] = s
    live = set(ids)
    touched = compared = 0
    for t in range(steps):
        act = (_driven_actions if contact else _actions)(rng, n)
        r = env.step(act)
        big = _outputs(r)
        if contact:
            touched += int(((env.get_state()["counters"][1] & 16) != 0).sum())
        for i in list(live):
            o = _outputs(small[i].step(act[i:i + 1]))
            assert all(_same(x[i:i + 1], y) for x, y in zip(big, o)), f"env {i} step {t}"
            compared += 1
            if bool(r.terminated[i] | r.truncated[i]):
                live.discard(i)  # the big ctx redraws at the reset, the plain one keeps its model
    end = env.get_state()
    for i in live:
        assert _same_dict(_col(end, i), small[i].get_state()), f"env {i}"
    assert compared >= 30 * len(ids)  # Env05 ends episodes early (block lost for 30 steps); the others run the whole window
    if contact:
        assert touched > 0.1 * n * steps


@pytest.mark.parametrize("task", [1, 2, 5, 6])
def test_env_replays_bit_exactly_on_a_plain_ctx_with_its_values(task, spec):
    _replay(task, False, spec)


@pytest.mark.parametrize("task", [1, 2])
def test_env_replays_bit_exactly_on_a_plain_ctx_with_arm_contact(task, spec):
    """The contact solve (cooperative and serial) takes the env's own friction loss."""
    _replay(task, True, spec)


@pytest.mark.parametrize("task", [1, 2])
def test_randomised_envs_track_the_oracle_built_from_their_models(task, spec):
    n, seed, steps = 64, 11, 200
    env = _env(task, n, seed=seed, param_ranges=_ranges(WIDE))
    env.reset()
    P = {k: v.cpu().numpy() for k, v in env.get_params().items()}
    orc = [make_oracle(task, 1, seed=seed, env_offset=i, spec=_plain_spec(spec, P, i)) for i in range(n)]
    obs_o = np.concatenate([o.reset() for o in orc])
    assert np.abs(env.obs.cpu().numpy() - obs_o).max() < 1e-6
    rng = np.random.default_rng(5)
    worst = 0.0
    for t in range(steps):
        a = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
        r = env.step(torch.from_numpy(a).cuda())
        outs = [o.step(a[i:i + 1]) for i, o in enumerate(orc)]
        assert not (r.terminated | r.truncated).any()
        worst = max(worst, float(np.abs(r.obs.cpu().numpy() - np.concatenate([x[0] for x in outs])).max()))
    st = env.get_state()
    dq = max(float(np.abs(st["qpos"][:, i].cpu().numpy() - o.gather("qpos")[0]).max()) for i, o in enumerate(orc))
    dv = max(float(np.abs(st["qvel"][:, i].cpu().numpy() - o.gather("qvel")[0]).max()) for i, o in enumerate(orc))
    print(f"task {task}: max|dq| {dq:.2e} max|dv| {dv:.2e} max|dobs| {worst:.2e}")
    assert dq < TOL_Q and dv < TOL_V and worst < TOL_OBS


def test_specialised_and_generic_randomised_kernels_agree():
    n, steps = 512, 100
    a = _env(1, n, seed=2, param_ranges=_ranges(WIDE))
    b = _env(1, n, seed=2, flags=_flags(generic=True), param_ranges=_ranges(WIDE))
    assert a.kernel_variant == "specialised" and b.kernel_variant == "generic"
    a.reset(); b.reset()
    assert _same_dict(a.get_params(), b.get_params())
    rng = np.random.default_rng(1)
    for _ in range(steps):
        act = _actions(rng, n)
        ra, rb = a.step(act), b.step(act)
        assert torch.equal(ra.terminated, rb.terminated)
    sa, sb = a.get_state(), b.get_state()
    assert (sa["qpos"] - sb["qpos"]).abs().max() < 2e-5
    assert (sa["qvel"] - sb["qvel"]).abs().max() < 1e-3


# ------------------------------------------------------------------------------------------------ bit-exact contracts
def _run(env, rng_seed, steps, n, contact=False):
    rng = np.random.default_rng(rng_seed)
    outs = []
    for _ in range(steps):
        outs.append(_outputs(env.step((_driven_actions if contact else _actions)(rng, n))))
    return outs


@pytest.mark.parametrize("contact", [False, True])
def test_shards_equal_the_full_batch(contact):
    n, lim = 512, 20
    kw = dict(seed=9, flags=_flags(contact), max_episode_steps=lim, param_ranges=_ranges(WIDE))
    full = _env(2, n, **kw)
    parts = [_env(2, 300, env_offset=0, **kw), _env(2, 212, env_offset=300, **kw)]
    full.reset(); [p.reset() for p in parts]
    full.stagger_episodes(seed=2)
    st = full.get_state()
    parts[0].set_state({k: v[:, :300] for k, v in st.items()}); parts[1].set_state({k: v[:, 300:] for k, v in st.items()})
    rng = np.random.default_rng(4)
    for t in range(60):
        act = (_driven_actions if contact else _actions)(rng, n)
        fo = _outputs(full.step(act))
        po = [_outputs(parts[0].step(act[:300])), _outputs(parts[1].step(act[300:]))]
        assert all(_same(f, torch.cat([po[0][k], po[1][k]])) for k, f in enumerate(fo)), f"step {t}"
    fp = full.get_params()
    pp = [p.get_params() for p in parts]
    assert all(_same(fp[k], torch.cat([pp[0][k], pp[1][k]], dim=1)) for k in fp)


def test_async_groups_rerun_and_state_roundtrip_are_bit_exact():
    n, lim = 1024, 15
    kw = dict(seed=6, max_episode_steps=lim, param_ranges=_ranges(WIDE))
    a, b = _env(6, n, **kw), _env(6, n, **kw)
    a.reset(); b.reset()
    a.stagger_episodes(seed=3); b.stagger_episodes(seed=3)
    ha, hb = a.alloc_host(), b.alloc_host()
    groups = b.host_groups(4)
    rng = np.random.default_rng(8)
    for t in range(40):
        act = _actions(rng, n).cpu()
        ha["actions"].copy_(act); hb["actions"].copy_(act)
        a.step_host(ha)
        for g in range(len(groups)):
            b.step_host_async(hb, g)
        for g in range(len(groups)):
            b.step_host_wait(g)
        for k in ("obs", "reward", "terminated", "truncated"):
            assert _same(ha[k], hb[k]), f"{k} step {t}"
    assert _same_dict(a.get_params(), b.get_params()) and _same_dict(a.get_state(), b.get_state())
    # same-seed rerun from the start, and a save / restore of state + params + tick followed by continuation
    c = _env(6, n, **kw)
    c.reset(); c.stagger_episodes(seed=3)
    rng = np.random.default_rng(8)
    for t in range(40):
        c.step(_actions(rng, n))
    assert _same_dict(a.get_params(), c.get_params()) and _same_dict(a.get_state(), c.get_state())
    saved = (c.get_state(), c.get_params(), c.tick)
    ref = _run(c, 21, 30, n)
    d = _env(6, n, **kw)
    d.set_state(saved[0]); d.set_params(saved[1]); d.tick = saved[2]
    got = _run(d, 21, 30, n)
    assert all(_same(x, y) for ro, go in zip(ref, got) for x, y in zip(ro, go))
    assert _same_dict(c.get_params(), d.get_params())


@pytest.mark.parametrize("contact", [False, True])
def test_substeps_equal_the_plain_model_ctx(contact, spec):
    n = 256
    flags = _flags(contact=contact, generic=True)
    env = _env(1, n, seed=12, flags=flags, param_ranges=_ranges(WIDE))
    env.reset()
    rng = np.random.default_rng(2)
    for _ in range(30):
        env.step(_driven_actions(rng, n))
    st, tick = env.get_state(), env.tick
    P = {k: v.cpu().numpy() for k, v in env.get_params().items()}
    ctrl = torch.from_numpy(rng.uniform(-1.5, 1.5, (n, 6)).astype(np.float32)).cuda()
    ctrl[:, 1] = -1.2  # Pitch down: arms into the floor
    env.step_substeps(ctrl, 160)
    end = env.get_state()
    for i in [0, 17, 200, n - 1]:
        s = _env(1, 1, seed=12, env_offset=i, flags=flags, model=_plain_spec(spec, P, i))
        s.set_state(_col(st, i)); s.tick = tick
        s.step_substeps(ctrl[i:i + 1], 160)
        assert _same_dict(_col(end, i), s.get_state()), f"env {i}"
    assert env.tick == tick
    assert _same_dict(env.get_params(), {k: torch.from_numpy(v).cuda() for k, v in P.items()})  # substeps never redraw


# ------------------------------------------------------------------------------------------------ explicit values, off
def test_set_params_hold_until_reset_and_switching_off_restores_the_default_kernel():
    from so100_mujoco_rl_b200._native import So100Error
    n = 512
    env = _env(1, n, seed=1, max_episode_steps=100000, param_ranges=_ranges())
    env.reset()
    mine = {k: v * 0.9 for k, v in env.get_params().items()}
    env.set_params({"kp": mine["kp"], "frictionloss": mine["frictionloss"]})
    got = env.get_params()
    assert _same(got["kp"], mine["kp"]) and _same(got["frictionloss"], mine["frictionloss"])
    assert not _same(got["kv"], mine["kv"])
    _run(env, 1, 10, n)
    assert _same(env.get_params()["kp"], mine["kp"])
    mask = torch.zeros(n, dtype=torch.uint8, device="cuda")
    mask[::3] = 1
    env.reset(mask)
    after = env.get_params()["kp"]
    keep = mask.cpu().numpy() == 0
    assert _same(after[:, keep], mine["kp"][:, keep]) and (after[:, ~keep] != mine["kp"][:, ~keep]).any(dim=0).all()
    # off: the model's constants and the default kernel, bit for bit with a default ctx from the same state
    env.set_param_ranges(None)
    with pytest.raises(So100Error):
        env.get_params()
    with pytest.raises(So100Error):
        env.set_params({"kp": mine["kp"]})
    ref = _env(1, n, seed=1, max_episode_steps=100000)
    ref.set_state(env.get_state()); ref.tick = env.tick
    assert all(_same(x, y) for ro, go in zip(_run(ref, 5, 20, n), _run(env, 5, 20, n)) for x, y in zip(ro, go))
    assert _same_dict(ref.get_state(), env.get_state())
    # on again: every env starts from the model's values
    env.set_param_ranges(_ranges())
    assert (_params_mat(env.get_params()).cpu().numpy() == _base_values(env)[:, None]).all()


def test_bad_ranges_and_group_steps_in_flight_are_refused():
    from so100_mujoco_rl_b200._native import So100Error, lib
    from so100_mujoco_rl_b200.randomization import So100ParamRanges
    env = _env(1, 512, param_ranges=_ranges())
    L = lib()
    r = _ranges().to_ctypes()
    r.kp[2][0] = 0.0
    assert L.so100_set_param_ranges(env._h, ctypes.byref(r)) == -1
    r = _ranges().to_ctypes()
    r.damping[0][0], r.damping[0][1] = 1.2, 1.1
    assert L.so100_set_param_ranges(env._h, ctypes.byref(r)) == -1
    r = _ranges().to_ctypes()
    r.frictionloss[1][1] = float("inf")
    assert L.so100_set_param_ranges(env._h, ctypes.byref(r)) == -1
    r = _ranges().to_ctypes()
    r.struct_size = ctypes.sizeof(So100ParamRanges) - 8
    assert L.so100_set_param_ranges(env._h, ctypes.byref(r)) == -1
    env.reset()
    h = env.alloc_host()
    env.host_groups(2)
    env.step_host_async(h, 0)
    with pytest.raises(So100Error):
        env.get_params()
    with pytest.raises(So100Error):
        env.set_param_ranges(None)
    env.step_host_wait(0)
    env.get_params()


# ------------------------------------------------------------------------------------------------ CLI
def test_cli_train_randomize_checkpoints_and_resumes_the_per_env_values(tmp_path):
    from click.testing import CliRunner
    from so100_mujoco_rl_b200.cli import cli
    common = ["-e", "Env01", "--num-envs", "256", "--n-steps", "8", "--eval-envs", "0", "--tensorboard-log", "",
              "--save-freq", "1000000000", "--out", str(tmp_path)]
    res = CliRunner().invoke(cli, ["-a", "PPO", "train", *common, "--total-timesteps", "4096", "--randomize", TYPICAL],
                             obj={}, catch_exceptions=False)
    assert res.exit_code == 0, res.output
    path = tmp_path / "Env01_PPO" / "final_model.pt"
    ck = torch.load(path, map_location="cpu", weights_only=False)
    P = ck["env"]["params"]
    assert set(P) == {"kp", "kv", "force_lo", "force_hi", "frictionloss"} and P["kp"].shape == (6, 256)
    assert ck["env"]["param_ranges"]["kp"] == [[0.7, 1.3]] * 6
    assert (P["kp"] != P["kp"][:, :1]).any()  # drawn per env
    # resume (no --randomize: the checkpoint's ranges) with nothing more to learn: the saved simulator is the restored one
    out2 = tmp_path / "resumed"
    res = CliRunner().invoke(cli, ["-a", "PPO", "-m", str(path), "train", *common[:-2], "--out", str(out2), "--total-timesteps", "0"],
                             obj={}, catch_exceptions=False)
    assert res.exit_code == 0, res.output
    ck2 = torch.load(out2 / "Env01_PPO" / "final_model.pt", map_location="cpu", weights_only=False)
    assert ck2["env"]["param_ranges"] == ck["env"]["param_ranges"] and ck2["env"]["tick"] == ck["env"]["tick"]
    assert all(_same(ck2["env"]["params"][k], P[k]) for k in P)
    assert all(_same(ck2["env"]["state"][k], ck["env"]["state"][k]) for k in ck["env"]["state"])
