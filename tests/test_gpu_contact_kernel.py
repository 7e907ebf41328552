"""The arm-floor contact kernel (SO100_FLAG_ARM_CONTACT) at the bit level.

Every substep a CTA hands the touching envs slots of a 48-slot shared-memory pool, solves the filled slots cooperatively
(eight lanes per env, four envs per warp in lockstep), and serves what the pool cannot take with the out-of-line serial
solve on the env's own thread.  Both solves converge in double far below fp32 resolution before the result is rounded to
float, so an env's bits must not depend on which path served it, which slot or warp it had, or what its neighbours in
the CTA do.  The tests below pin that contract where the kernel could break it - a CTA with more than 48 touching envs,
a ragged last CTA whose tail threads shadow a touching env, more than eight corners at once, the pool-less substeps entry,
the generic kernel - and the library's bit-exact contracts (determinism, state round trip, host path, env groups,
sharding) under the contact flag.  Tolerance tests (against the fp64 oracle) cover the two entries the parity suite does
not reach: so100_step_substeps and the generic kernel with contact.
"""
import numpy as np
import pytest

from conftest import make_oracle

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

F_TOUCH = 16        # counters[1] bit: a jaw pad touched the floor in the env's last substep
CTA, POOL = 256, 48  # envs per CTA, contact-solve slots per CTA (csrc/so100_b200.cu kBlock / kPoolSlots)
K = 8               # env steps compared bit for bit
STATE = ("qpos", "qpos_comp", "qvel", "qacc_warm")
TOL_Q = 2e-5


def _flags(generic=False):
    from so100_mujoco_rl_b200.tasks import FLAG_ARM_CONTACT, FLAG_GENERIC_KERNEL
    return FLAG_ARM_CONTACT | (FLAG_GENERIC_KERNEL if generic else 0)


def _env(task, n, seed=5, flags=None, **kw):
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    return BatchedSo100Env(task, n, device=0, seed=seed, flags=_flags() if flags is None else flags, **kw)


def _bits(t):
    """The raw bits of a tensor (float comparisons would call -0.0 and 0.0 equal)."""
    t = t.contiguous()
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _same(a, b):
    return torch.equal(_bits(a), _bits(b))


def _touch(st):
    return (st["counters"][1] & F_TOUCH) != 0


def _col(st, i):
    return {k: v[:, i].clone() for k, v in st.items()}


def _stack(cols):
    return {k: torch.stack([c[k] for c in cols], dim=1).contiguous() for k in cols[0]}


def _slice(st, lo, hi):
    return {k: v[:, lo:hi].contiguous() for k, v in st.items()}


def _driven_actions(rng, n):
    """test_arm_floor_contact_parity's recipe: random actions, Pitch pushed down in the first half of the envs."""
    a = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
    a[: n // 2, 1] = np.clip(a[: n // 2, 1] + 0.6, -1, 1)
    return torch.from_numpy(a).cuda()


_DRIVEN = {}


def _driven(task, n, steps=80, generic=False):
    """(state, tick) of n envs after `steps` driven steps: a good share of them rest on or slide along the floor."""
    key = (task, n, steps, generic)
    if key not in _DRIVEN:
        env = _env(task, n, flags=_flags(generic))
        env.reset()
        rng = np.random.default_rng(8)
        for _ in range(steps):
            env.step(_driven_actions(rng, n))
        _DRIVEN[key] = (env.get_state(), env.tick)
        env.close()
    return _DRIVEN[key]


def _filler(task):
    """A contact-free column: the task's reset pose (arm clear of the floor), held there by zero actions."""
    env = _env(task, 1, seed=99)
    env.reset()
    c = _col(env.get_state(), 0)
    env.close()
    return c


def _run(env, actions):
    """Step through `actions`; per step the outputs and the state fields, env-major ([n, ...])."""
    out = []
    for a in actions:
        r = env.step(a)
        st = env.get_state()
        rec = {"obs": r.obs.clone(), "reward": r.reward.clone(), "terminated": r.terminated.clone(), "truncated": r.truncated.clone(),
               "touch": _touch(st)}
        rec.update({k: st[k].T.contiguous() for k in STATE})
        out.append(rec)
    return out


def _assert_rows_equal(got, i, ref, j, what):
    """Row i of run `got` equals row j of run `ref` in every output and state field, at every step."""
    for t, (g, r) in enumerate(zip(got, ref)):
        for k in ("obs", "reward", "terminated", "truncated") + STATE:
            assert _same(g[k][i], r[k][j]), f"{what}: step {t}, {k} of env {i} differs"


# ------------------------------------------------------------------------------------------------ 1. identical envs


@pytest.fixture(scope="module")
def resting_env01():
    """One Env01 state resting on the floor with 1..8 pad corners at most 4 mm deep (checked with the oracle's
    contacts), episode clock at 0 so that no TimeLimit reset draws from the RNG in the compared window."""
    st, _ = _driven(1, CTA, steps=100)
    o = make_oracle(1, 1, flags=_flags())
    q = (st["qpos"].double() - st["qpos_comp"].double()).cpu().numpy().T
    for i in np.flatnonzero(_touch(st).cpu().numpy()):
        d = o.contacts(q[i])[1]
        if 0 < len(d) <= 8 and d.min() > -0.004:
            c = _col(st, i)
            c["counters"][0] = 0
            return c
    pytest.fail("no env of the driven batch rests on the floor with 1..8 corners")


def _push(rng):
    """One action row: random, Pitch pushed down so that the contact persists."""
    a = rng.uniform(-0.5, 0.5, 6).astype(np.float32)
    a[1] = 0.6
    return a


def _reference_run(task, touching, actions_row, flags=None):
    """A full CTA (no tail threads): env 0 holds `touching`, the other 255 the contact-free filler with zero actions,
    so env 0 is the CTA's only pool request and takes the cooperative solve."""
    env = _env(task, CTA, flags=flags)
    env.set_state(_stack([touching] + [_filler(task)] * (CTA - 1)))
    acts = []
    for a in actions_row:
        x = torch.zeros((CTA, 6), device="cuda")
        x[0] = torch.from_numpy(a)
        acts.append(x)
    out = _run(env, acts)
    env.close()
    return out


@pytest.mark.parametrize("n", [1, 256, 1000])
def test_identical_touching_envs_give_identical_bits(resting_env01, n):
    """The same touching state and actions in every env: n = 256 is one CTA of 256 touching envs (208 of them beyond the
    pool), n = 1000 three full CTAs and a ragged one of 232 envs, n = 1 one live thread and 255 tail threads.  Every env
    must reproduce, bit for bit, the env that had the pool to itself."""
    rng = np.random.default_rng(4)
    rows = [_push(rng) for _ in range(K)]
    ref = _reference_run(1, resting_env01, rows)
    for t, r in enumerate(ref):
        assert bool(r["touch"][0]), f"the reference env left the floor at step {t}"
        assert not r["touch"][1:].any(), "a filler env touched the floor"
    free = _reference_run(1, resting_env01, rows, flags=0)
    assert not _same(free[-1]["qpos"][0], ref[-1]["qpos"][0])   # the contact changed the trajectory

    env = _env(1, n)
    env.set_state(_stack([resting_env01] * n))
    got = _run(env, [torch.from_numpy(a).cuda().expand(n, 6).contiguous() for a in rows])
    assert all(bool(g["touch"].all()) for g in got)
    for i in range(n):
        _assert_rows_equal(got, i, ref, 0, f"{n} identical envs")
    env.close()


# ------------------------------------------------------------------------------------------------ 2. mixed batch


def test_mixed_batch_equals_single_env_runs():
    """512 Env02 envs driven into the floor, then K more steps.  Envs of the CTA whose touching envs overflow the pool,
    envs clear of the floor and the last env, each replayed from the saved state at local index 0 of a 256-env ctx
    (env_offset = its index: the same RNG stream) among contact-free fillers, must give the same bits."""
    n = 512
    st, tick = _driven(2, n)
    per_cta = _touch(st).reshape(n // CTA, CTA).sum(dim=1).cpu().numpy()
    assert per_cta.max() > POOL, f"touching envs per CTA {per_cta}: no CTA overflows the pool"
    full = _env(2, n)
    full.set_state(st)
    full.tick = tick
    rng = np.random.default_rng(21)
    acts = [_driven_actions(rng, n) for _ in range(K)]
    ref = _run(full, acts)
    full.close()

    over = int(np.argmax(per_cta))
    touching = np.flatnonzero(_touch(st).cpu().numpy())
    touching = touching[(touching // CTA) == over]
    clear = np.flatnonzero(~_touch(st).cpu().numpy())
    pick = sorted(set(touching[np.linspace(0, len(touching) - 1, 10).astype(int)].tolist())
                  | set(clear[np.linspace(0, len(clear) - 1, 5).astype(int)].tolist()) | {n - 1})
    filler = _filler(2)
    for i in pick:
        env = _env(2, CTA, env_offset=i)
        env.set_state(_stack([_col(st, i)] + [filler] * (CTA - 1)))
        env.tick = tick
        got = _run(env, [torch.cat([a[i:i + 1], torch.zeros((CTA - 1, 6), device="cuda")]) for a in acts])
        assert not any(bool(g["touch"][1:].any()) for g in got), "a filler env touched the floor"
        _assert_rows_equal(got, 0, ref, i, f"env {i} alone")
        env.close()


# ------------------------------------------------------------------------------------------------ 3. bit-exact contracts


def _touch_frac(run):
    return float(torch.stack([r["touch"] for r in run]).float().mean())


def _assert_runs_equal(a, b, what):
    for t, (x, y) in enumerate(zip(a, b)):
        for k in ("obs", "reward", "terminated", "truncated") + STATE:
            assert _same(x[k], y[k]), f"{what}: step {t}, {k} differs"


def _loaded(task, n, st, tick, **kw):
    env = _env(task, n, **kw)
    env.set_state(st)
    env.tick = tick
    return env


@pytest.mark.parametrize("task", [1, 2, 5, 6])
def test_same_seed_gives_the_same_bits_under_contact(task):
    n = 512
    st, tick = _driven(task, n)
    rng = np.random.default_rng(3)
    acts = [_driven_actions(rng, n) for _ in range(K)]
    a, b = _loaded(task, n, st, tick), _loaded(task, n, st, tick)
    ra, rb = _run(a, acts), _run(b, acts)
    assert _touch_frac(ra) > 0.05
    _assert_runs_equal(ra, rb, "two ctxs")
    sa, sb = a.get_state(), b.get_state()
    for k in sa:
        assert _same(sa[k], sb[k]), k


@pytest.mark.parametrize("task", [1, 2, 5, 6])
def test_state_roundtrip_replays_bit_exactly_under_contact(task):
    n = 512
    st, tick = _driven(task, n)
    rng = np.random.default_rng(5)
    acts = [_driven_actions(rng, n) for _ in range(K + 3)]
    env = _loaded(task, n, st, tick)
    _run(env, acts[:3])
    snap, t0 = env.get_state(), env.tick
    first = _run(env, acts[3:])
    env.set_state(snap)
    env.tick = t0
    second = _run(env, acts[3:])
    assert _touch_frac(first) > 0.05
    _assert_runs_equal(first, second, "replay")


def test_host_path_equals_device_path_under_contact():
    """N = 300: a ragged last CTA.  Pinned buffers (one zero-copy launch) and pageable ones (copy pipeline)."""
    import ctypes
    from so100_mujoco_rl_b200 import _native
    n = 300
    st, tick = _driven(1, 512)
    st = _slice(st, 0, n)
    dev, pin, page = (_loaded(1, n, st, tick) for _ in range(3))
    host = pin.alloc_host()
    od = page.obs_dim
    buf = {"obs": np.zeros((n, od), np.float32), "reward": np.zeros(n, np.float32), "terminated": np.zeros(n, np.uint8),
           "truncated": np.zeros(n, np.uint8)}
    p = lambda a: a.ctypes.data_as(ctypes.c_void_p)  # noqa: E731
    rng = np.random.default_rng(6)
    touching = 0
    for t in range(K):
        a = _driven_actions(rng, n)
        r = dev.step(a)
        host["actions"].copy_(a.cpu())
        pin.step_host(host)
        act = a.cpu().numpy()
        _native.check(page._L.so100_step_host(page._h, p(act), p(buf["obs"]), p(buf["reward"]), p(buf["terminated"]),
                                              p(buf["truncated"]), None, None, None, None))
        for k in ("obs", "reward", "terminated", "truncated"):
            assert _same(getattr(r, k).cpu(), host[k]), (t, k, "pinned")
            assert _same(getattr(r, k).cpu(), torch.from_numpy(buf[k])), (t, k, "pageable")
        touching += int(_touch(dev.get_state()).sum())
    assert touching > 0.05 * K * n
    sd, sp, sq = dev.get_state(), pin.get_state(), page.get_state()
    for k in sd:
        assert _same(sd[k], sp[k]) and _same(sd[k], sq[k]), k


def test_async_groups_equal_the_full_batch_under_contact():
    """N = 1000 Env02 envs in 3 env groups, a 20-step TimeLimit with staggered episode clocks: terminal rows on every step
    (70 % of the envs end an episode in the window), while the envs that have not been reset yet keep touching the floor
    (a reset puts the arm back in its pose clear of the floor)."""
    n, groups, limit, steps = 1000, 3, 20, 14
    st, tick = _driven(2, n)
    st = {k: v.clone() for k, v in st.items()}
    st["counters"][0] = torch.arange(n, device="cuda", dtype=torch.int32) % limit
    e1, e2 = _loaded(2, n, st, tick, max_episode_steps=limit), _loaded(2, n, st, tick, max_episode_steps=limit)
    h1, h2 = e1.alloc_host(), e2.alloc_host()
    e2.host_groups(groups)
    rng = np.random.default_rng(7)
    touching = ndone = 0
    for t in range(steps):
        a = _driven_actions(rng, n).cpu()
        h1["actions"].copy_(a); h2["actions"].copy_(a)
        e1.step_host(h1)
        for g in (range(groups) if t % 2 else reversed(range(groups))):
            e2.step_host_async(h2, g)
        for g in range(groups):
            e2.step_host_wait(g)
        for k in ("obs", "reward", "terminated", "truncated"):
            assert _same(h1[k], h2[k]), (t, k)
        done = (h1["terminated"] | h1["truncated"]).bool()
        ndone += int(done.sum())
        for k in ("terminal_obs", "ep_return", "ep_len"):
            assert _same(h1[k][done], h2[k][done]), (t, k)
        touching += int(_touch(e1.get_state()).sum())
    assert ndone >= n // 2 and touching > 0.05 * steps * n
    s1, s2 = e1.get_state(), e2.get_state()
    for k in s1:
        assert _same(s1[k], s2[k]), k


def test_env_offset_sharding_under_contact():
    """Shards of 300 + 212 envs (env_offset 0 / 300) against one ctx of 512: the shards cut a CTA of touching envs in two
    and end in ragged CTAs."""
    n, cut = 512, 300
    st, tick = _driven(2, n)
    full = _loaded(2, n, st, tick)
    lo = _loaded(2, cut, _slice(st, 0, cut), tick)
    hi = _loaded(2, n - cut, _slice(st, cut, n), tick, env_offset=cut)
    rng = np.random.default_rng(9)
    acts = [_driven_actions(rng, n) for _ in range(K)]
    rf = _run(full, acts)
    rl = _run(lo, [a[:cut].contiguous() for a in acts])
    rh = _run(hi, [a[cut:].contiguous() for a in acts])
    assert _touch_frac(rf) > 0.05
    joined = [{k: torch.cat([x[k], y[k]]) for k in x} for x, y in zip(rl, rh)]
    _assert_runs_equal(rf, joined, "300 + 212 shards")


# ------------------------------------------------------------------------------------------------ 4. substeps entry


def _contact_free(o, rng, lo, hi, n):
    """n joint configurations whose jaw pads are clear of the floor."""
    out = []
    while len(out) < n:
        q = rng.uniform(lo, hi)
        if len(o.contacts(q)[1]) == 0:
            out.append(q)
    return np.array(out)


def _touching(o, rng, lo, hi, n, max_con=8, max_depth=0.004):
    """n configurations with 1..max_con pad corners up to max_depth below the floor."""
    out = []
    while len(out) < n:
        q = rng.uniform(lo, hi)
        d = o.contacts(q)[1]
        if 0 < len(d) <= max_con and d.min() > -max_depth:
            out.append(q)
    return np.array(out)


def _many_corners(o, rng, lo, hi, n):
    """n configurations with 9..16 pad corners at most 4 mm below the floor (both jaws flat on it): a random pose with
    more than 8 corners, lifted by one joint until the deepest corner is within 4 mm."""
    out = []
    while len(out) < n:
        q = rng.uniform(lo, hi)
        if len(o.contacts(q)[1]) <= 8:
            continue
        for j in (1, 2, 3):
            for s in np.linspace(-0.3, 0.3, 61):
                qq = q.copy()
                qq[j] += s
                d = o.contacts(qq)[1]
                if 8 < len(d) <= 16 and d.min() > -0.004:
                    out.append(qq)
                    break
            else:
                continue
            break
    return np.array(out)


def _substep_states(spec):
    """512 Env01 configurations: 256 clear of the floor (random velocities), 224 with 1..8 pad corners in it and 32 with
    more than 8 (at rest); servo targets near the pose, Pitch pushed down for the touching ones."""
    o = make_oracle(1, 1, flags=_flags())
    rng = np.random.default_rng(12)
    lo, hi = spec.jnt_range[:, 0], spec.jnt_range[:, 1]
    q = np.concatenate([_contact_free(o, rng, lo, hi, 256), _touching(o, rng, lo, hi, 224), _many_corners(o, rng, lo, hi, 32)])
    v = np.zeros_like(q)
    v[:256] = rng.normal(0, 0.5, (256, 6))
    a = rng.uniform(-1, 1, q.shape)
    a[256:, 1] = np.clip(a[256:, 1] + 0.6, -1, 1)
    q, v = q.astype(np.float32), v.astype(np.float32)
    ctrl = (q + a * 0.075).astype(np.float32)
    return q, v, ctrl


@pytest.mark.parametrize("contact", [True, False])
@pytest.mark.parametrize("nsub", [16, 160])
def test_step_substeps_tracks_the_oracle(spec, contact, nsub):
    """so100_step_substeps (no pool: every contact solve is the serial one) against Oracle.substeps in fp64, in the
    form of test_host_substeps_track_the_oracle_through_contact.  It advances physics only: the tick and the episode
    clocks stay, and `snap` holds the kinematics of the last substep's start state."""
    n = 512
    q, v, ctrl = _substep_states(spec)
    flags = _flags() if contact else 0
    base = _filler(1)
    st = _stack([base] * n)
    st["qpos"] = torch.from_numpy(q.T.copy()).cuda()
    st["qvel"] = torch.from_numpy(v.T.copy()).cuda()
    st["qacc_warm"].zero_(); st["qpos_comp"].zero_()
    st["counters"][0] = 3
    envs = []
    for m in (nsub, nsub - 1):   # the second one stops at the start of the first one's last substep
        env = _env(1, n, flags=flags)
        env.set_state(st)
        env.tick = 5
        env.step_substeps(torch.from_numpy(ctrl), m)
        assert env.tick == 5
        envs.append(env.get_state())
    sa, sb = envs
    assert (sa["counters"][0] == 3).all()
    o = make_oracle(1, 1, flags=flags)
    qg = (sa["qpos"].double() - sa["qpos_comp"].double()).cpu().numpy().T
    vg = sa["qvel"].cpu().numpy().T
    dq, dv = np.zeros(n), np.zeros(n)
    for i in range(n):
        qo, vo, _ = o.substeps(q[i], v[i], np.zeros(6), ctrl[i], nsub)
        dq[i], dv[i] = np.abs(qg[i] - qo).max(), np.abs(vg[i] - vo).max()
    if contact:
        assert (_touch(sa).cpu().numpy()[256:].mean() > 0.5)
    print(f"substeps {nsub} contact {contact}: |dq| median {np.median(dq):.2e} p99 {np.quantile(dq, 0.99):.2e} max {dq.max():.2e}; "
          f"|dv| median {np.median(dv):.2e} p99 {np.quantile(dv, 0.99):.2e}")
    assert np.median(dq) < 2e-7 and np.quantile(dq, 0.99) < 2e-6 and (dq > TOL_Q).mean() < 1e-2
    assert np.median(dv) < 1e-5 and np.quantile(dv, 0.99) < 1e-4
    # the snapshot: end-effector point and wrist height at the last substep's start state, the block where it was then
    snap = sa["snap"].cpu().numpy()
    qs = (sb["qpos"].double() - sb["qpos_comp"].double()).cpu().numpy().T
    for i in range(0, n, 8):
        k = o.fk(qs[i])
        assert np.abs(snap[:3, i] - k["end_pos"]).max() < 2e-6 and abs(snap[3, i] - k["wrist_pos"][2]) < 2e-6, i
    assert _same(sa["snap"][4:7], sb["block"][:3])


# ------------------------------------------------------------------------------------------------ 5. serial == cooperative


def test_serial_solve_equals_cooperative_solve_on_the_device():
    """Env05 on the generic kernel: so100_step and so100_step_substeps both run physics<5, false, true>, and Env05's
    open-loop ctrl (aux[0:6] + a * step_scale, no low part) can be handed to the substeps entry as it is.  Env 0 alone
    among contact-free envs takes the pool's cooperative solve in so100_step; the substeps entry has no pool and takes the
    serial solve.  The results must be the same bits."""
    from so100_mujoco_rl_b200.tasks import JOINT_STEP_SCALE
    st, _ = _driven(5, CTA, generic=True)
    o = make_oracle(5, 1, flags=_flags())
    q = (st["qpos"].double() - st["qpos_comp"].double()).cpu().numpy().T
    idx = [i for i in np.flatnonzero(_touch(st).cpu().numpy()) if 0 < len(o.contacts(q[i])[1]) <= 8]
    assert idx, "no env of the driven batch touches the floor with 1..8 corners"
    filler = _filler(5)
    a = np.zeros(6, np.float32)
    a[1] = 0.3
    tried = 0
    for i in idx[:4]:
        c = _col(st, i)
        c["counters"][2] = 0   # no lost-cube termination (and reset) in the step
        s0 = _stack([c] + [filler] * (CTA - 1))
        A = _env(5, CTA, flags=_flags(generic=True))
        B = _env(5, CTA, flags=_flags(generic=True))
        assert A.kernel_variant == "generic"
        A.set_state(s0); B.set_state(s0)
        act = torch.zeros((CTA, 6), device="cuda")
        act[0] = torch.from_numpy(a)
        A.step(act)
        # the kernel computes aux + a * step_scale as one fused multiply-add: the exact sum, rounded once to fp32
        aux = s0["aux"][:6].cpu().numpy().T.astype(np.float64)
        ctrl = (aux + act.cpu().numpy().astype(np.float64) * np.float64(np.float32(JOINT_STEP_SCALE))).astype(np.float32)
        B.step_substeps(torch.from_numpy(ctrl), 16)
        sa, sb = A.get_state(), B.get_state()
        assert bool(_touch(sa)[0]) and bool(_touch(sb)[0])
        assert not _touch(sa)[1:].any()
        for k in STATE:
            assert _same(sa[k][:, 0], sb[k][:, 0]), (i, k)
        tried += 1
        A.close(); B.close()
    assert tried >= 1


# ------------------------------------------------------------------------------------------------ 6. generic kernel


def _contact_parity(task, steps, flags, model=None):
    n, seed = 512, 5
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    env = BatchedSo100Env(task, n, device=0, seed=seed, flags=flags, model=model)
    assert env.kernel_variant == "generic"
    o = make_oracle(task, n, seed=seed, flags=flags, spec=model)
    assert np.abs(env.reset().cpu().numpy() - o.reset(nthreads=0)).max() < 1e-6
    rng = np.random.default_rng(8)
    dq, touching, below = [], 0, 0
    for t in range(steps):
        a = _driven_actions(rng, n)
        r = env.step(a)
        oo, ro, to, co, *_ = o.step(a.cpu().numpy(), nthreads=0)
        assert (r.terminated.cpu().numpy() == to).all() and (r.truncated.cpu().numpy() == co).all()
        st = env.get_state()
        qg = st["qpos"].cpu().numpy().astype(np.float64) - st["qpos_comp"].cpu().numpy()
        dq.append(np.abs(qg - o.get_state_soa()[0]).max(axis=0))
        touching += int(_touch(st).sum())
        below += int((r.obs[:, 14] < 0).sum())
    dq = np.array(dq)
    rate = float((dq > TOL_Q).mean())
    print(f"task {task} generic kernel with contact: {touching / (steps * n):.1%} touching; |dq| median {np.median(dq):.2e} "
          f"p90 {np.quantile(dq, 0.9):.2e} max {dq.max():.2e}; rate {rate:.2e}")
    assert touching > 0.05 * steps * n
    assert below == 0
    assert np.median(dq) < 1e-6 and np.quantile(dq, 0.9) < 5e-6
    assert rate < 0.05
    s = env.stats()
    assert s["nan_resets"] == 0 and s["solver_unconverged"] <= 5
    env.close()


@pytest.mark.parametrize("task", [1, 2])
def test_generic_kernel_with_contact_tracks_the_oracle(task):
    _contact_parity(task, 60, _flags(generic=True))


def test_other_mjcf_numbers_with_contact_track_the_oracle(spec):
    """The modified model of test_other_mjcf_numbers_run_on_the_generic_kernel_and_track_the_oracle, with the pads."""
    import copy
    m = copy.deepcopy(spec)
    m.body_mass = m.body_mass * np.array([1.3, 0.8, 1.1, 1.5, 0.7, 2.0])
    m.body_inertia = m.body_inertia * 1.2
    m.act_kp = m.act_kp * np.array([0.8, 1.2, 1.0, 0.6, 1.5, 1.0])
    m.jnt_frictionloss = m.jnt_frictionloss * np.array([0.5, 1.0, 2.0, 1.0, 0.3, 1.0])
    m.jnt_range = m.jnt_range * 0.9
    m.jnt_solimp_limit = m.jnt_solimp_limit.copy(); m.jnt_solimp_limit[:, 4] = 3.0
    m.contact_solref = np.array([0.03, 1.0]); m.block_friction = 0.7; m.block_half_z = 0.015
    _contact_parity(2, 60, _flags(), model=m)


def test_specialised_and_generic_contact_kernels_agree():
    """Both integrate the same fp32 model with the same contact path, their dynamics rounded differently (generated
    straight-line code against the generic recursion), over 100 driven Env05 steps.  An env that never touched the floor
    stays within fp32 rounding of its twin, as test_specialised_and_generic_kernels_agree asserts without contact.  An env
    that did can meet a make / break or stick / slip transition (or come to rest in a joint's friction dead band) on the
    other side of a substep boundary in the two roundings, and the twins then part for good: those are bounded in the
    quantile + rate form of test_arm_floor_contact_parity, as each kernel's distance to the oracle is."""
    n, steps = 512, 100
    a_env, b_env = _env(5, n, seed=3), _env(5, n, seed=3, flags=_flags(generic=True))
    assert a_env.kernel_variant == "specialised" and b_env.kernel_variant == "generic"
    a_env.reset(); b_env.reset()
    rng = np.random.default_rng(0)
    touched = torch.zeros(n, dtype=torch.bool, device="cuda")
    dq, flags_differ = [], torch.zeros(n, dtype=torch.bool, device="cuda")
    for _ in range(steps):
        act = _driven_actions(rng, n)
        ra, rb = a_env.step(act), b_env.step(act)
        flags_differ |= (ra.terminated != rb.terminated) | (ra.truncated != rb.truncated)
        sa, sb = a_env.get_state(), b_env.get_state()
        touched |= _touch(sa) | _touch(sb)
        qa = sa["qpos"].double() - sa["qpos_comp"].double()
        qb = sb["qpos"].double() - sb["qpos_comp"].double()
        dq.append((qa - qb).abs().max(dim=0).values)
    dq = torch.stack(dq).cpu().numpy()          # [step, env]
    clear = ~touched.cpu().numpy()
    rate = float((dq > TOL_Q).mean())
    parted = int((dq.max(axis=0) > TOL_Q).sum())
    print(f"specialised vs generic with contact: {int((~touched).sum())} envs never touched (max |dq| {dq[:, clear].max():.2e}); "
          f"all envs: |dq| median {np.median(dq):.2e} p90 {np.quantile(dq, 0.9):.2e} max {dq.max():.2e}, rate {rate:.2e}, "
          f"{parted} envs part by > {TOL_Q:g}, all of them touched: {bool(not (clear & (dq.max(axis=0) > TOL_Q)).any())}")
    assert touched.float().mean() > 0.2 and clear.sum() > 0.1 * n
    assert dq[:, clear].max() < TOL_Q                                           # fp32 rounding of each other
    assert (sa["qvel"] - sb["qvel"]).abs().max(dim=0).values[~touched].max() < 1e-3
    assert not flags_differ[~touched].any()
    assert np.median(dq) < 1e-6 and np.quantile(dq, 0.9) < 5e-6 and rate < 0.05
