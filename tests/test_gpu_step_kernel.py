"""The default env-step kernel, step_kernel<TASK, SPEC = true, PADS = false, PARAMS>, one or two substeps at a time.

The kernel that bench.py times is also the one that keeps changing.  The trajectory parity suite (test_gpu_parity.py)
runs it over 16-substep steps, where the servo equilibrium hides errors in M and the bias, and where chaotic
amplification forces quantile tolerances.  Here the same kernel runs ONE or TWO substeps per env step:
so100_create picks the specialised kernel by comparing the dynamics and solver constants, and nsubstep is not among
them (test_short_step_ctx_runs_the_default_kernel guards this).  Substep 0 gets the first substep's 5 Gauss-Seidel
sweeps, substep 1 the other substeps' 3.  After one or two substeps nothing has bifurcated, so the kernel is held to
max-norm bounds derived from fp32 rounding, against so100_host_substeps variant 0: the same templates and sweep
schedule in fp64, which test_host_dyn.py ties to the independent oracle at 1e-10 .. 1e-14.

Also here: the warp-uniform limit rows (solve_qacc<float, true>) bit for bit against a 1-env run whatever the warp's
other lanes hold, and the counters of ragged launches.  Every measured worst error is kept next to its bound by
test_gpu_parity._record, as step_kernel_*.json beside the parity suite's figures.
"""
import copy
import ctypes
import dataclasses

import numpy as np
import pytest

from test_gpu_parity import _record

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

TASKS = (1, 2, 5, 6)
STATE = ("qpos", "qpos_comp", "qvel", "qacc_warm", "block", "snap", "aux", "counters", "ep_return")
WIDE = "kp=0.5:2,damping=0.5:2,forcerange=0.8:1.2,frictionloss=0.5:2"
UNIT = "kp=1:1,damping=1:1,forcerange=1:1,frictionloss=1:1"
FAR = 1 << 30          # TimeLimit of the short-step ctxs: no truncation, so no reset draws from the RNG
STEP_SCALE = np.float32(0.075)
U = 2.0 ** -24         # fp32 unit roundoff


# ------------------------------------------------------------------------------------------------ helpers
def _env(spec, task, n, nsub=16, seed=3, env_offset=0, flags=0, ranges=None, max_episode_steps=FAR):
    from so100_mujoco_rl_b200.batched_env import BatchedSo100Env
    env = BatchedSo100Env(task, n, device=0, seed=seed, env_offset=env_offset, flags=flags,
                          model=dataclasses.replace(spec, nsubstep=nsub), max_episode_steps=max_episode_steps)
    if ranges is not None:
        from so100_mujoco_rl_b200.randomization import ParamRanges
        env.set_param_ranges(ParamRanges.parse(ranges))
    return env


def _bits(t):
    t = t.contiguous()
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _dp(x):
    return x.ctypes.data_as(ctypes.POINTER(ctypes.c_double))


def _f32(x):
    return np.asarray(x, dtype=np.float32).astype(np.float64)


def _ref_model(spec, kv, P=None, i=None):
    """The host reference model: the so100 model with the actuator, limit and friction constants the kernel holds in fp32
    (an env's own get_params values with P), evaluated in fp64.  No pads: the default kernel has no arm-floor contact."""
    m = copy.deepcopy(spec)
    m.jnt_range = _f32(spec.jnt_range)
    m.act_ctrlrange = _f32(spec.act_ctrlrange)
    m.act_dampratio = np.zeros(6)
    if P is None:
        m.act_kp, m.act_kv = _f32(spec.act_kp), _f32(kv)
        m.act_forcerange, m.jnt_frictionloss = _f32(spec.act_forcerange), _f32(spec.jnt_frictionloss)
    else:
        m.act_kp, m.act_kv = _f32(P["kp"][:, i]), _f32(P["kv"][:, i])
        m.act_forcerange = np.stack([_f32(P["force_lo"][:, i]), _f32(P["force_hi"][:, i])], axis=1)
        m.jnt_frictionloss = _f32(P["frictionloss"][:, i])
    ct = m.to_ctypes()
    ct.n_pad = 0
    return ct


def _host_substeps(m, q, v, w, ctrl, nsub, variant):
    """so100_host_substeps on [n, 6] fp64 copies; returns (qpos, qvel, qacc, stats)."""
    from so100_mujoco_rl_b200 import _native
    q, v, w = (np.ascontiguousarray(x, dtype=np.float64).copy() for x in (q, v, w))
    c = np.ascontiguousarray(ctrl, dtype=np.float64)
    st = np.zeros(5, dtype=np.int64)
    _native.check(_native.lib().so100_host_substeps(ctypes.byref(m), len(q), _dp(q), _dp(v), _dp(w), _dp(c), int(nsub), int(variant),
                                                    st.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))))
    return q, v, w, st


def _host_forward(m, q, v):
    """fp64 M (packed lower triangle) and bias of the generic templates."""
    from so100_mujoco_rl_b200 import _native
    q, v = (np.ascontiguousarray(x, dtype=np.float64) for x in (q, v))
    n = len(q)
    M, b = np.zeros((n, 21)), np.zeros((n, 6))
    _native.check(_native.lib().so100_host_forward(ctypes.byref(m), n, _dp(q), _dp(v), _dp(q), _dp(M), _dp(b), None, None, 1, 0))
    return M, b


def _unpack(Mp):
    M = np.zeros((len(Mp), 6, 6))
    k = 0
    for r in range(6):
        for c in range(r + 1):
            M[:, r, c] = M[:, c, r] = Mp[:, k]
            k += 1
    return M


def _round32(x):
    """Correctly rounded fp32 of an exact value given as a float64 pair (s + e, |e| <= ulp(s) / 2)."""
    s, e = x
    r = s.astype(np.float32)
    d = s - r.astype(np.float64)                    # exact: the rounding residue of s
    half = np.abs(np.spacing(r).astype(np.float64)) / 2
    tie = (np.abs(d) == half) & (e != 0)            # s sits on a midpoint: the tail decides the direction
    up = np.nextafter(r, np.where(d + e > 0, np.float32(np.inf), np.float32(-np.inf)))
    return np.where(tie, up, r)


def _two_sum(a, b):
    s = a + b
    bb = s - a
    return s, (a - (s - bb)) + (b - bb)


_BULK = {}


def _bulk_state(spec, task, n):
    """A decorrelated state, built as in test_parity_at_baseline_size: staggered episode clocks, then 100 steps of random
    actions on a 16-substep ctx (the distribution bench.py times; joint-limit rows are common)."""
    key = (task, n)
    if key not in _BULK:
        env = _env(spec, task, n, 16, seed=0, max_episode_steps=None)
        env.reset()
        env.stagger_episodes()
        g = torch.Generator(device="cuda").manual_seed(7)
        for _ in range(100):
            env.step(torch.rand((n, 6), device="cuda", generator=g) * 2 - 1)
        _BULK[key] = {k: v.cpu().numpy().copy() for k, v in env.get_state().items()}
        env.close()
    return {k: v.copy() for k, v in _BULK[key].items()}


def _crafted(spec, task, base, rng):
    """Edge inputs, one env per row: per dof j the joint below lo / above hi at depths across the solimp width
    (impedance ramp and saturation), velocity into and out of the limit, |dist| within ulps of 0 with a nonzero
    qpos_comp (the compensated presence test decides), exactly on a limit, servo targets beyond ctrlrange and within an
    ulp of it, torque beyond forcerange, stick and slip, large velocities, and warm starts exact / zero / 100x off.
    Returns (state columns [k, m], actions [m, 6], warm-start mode per env)."""
    lo32, hi32 = spec.jnt_range[:, 0].astype(np.float32), spec.jnt_range[:, 1].astype(np.float32)
    clo32, chi32 = spec.act_ctrlrange[:, 0].astype(np.float32), spec.act_ctrlrange[:, 1].astype(np.float32)
    rows = []

    def add(q=None, qc=None, v=None, a=None, aux=None, warm="bulk"):
        q0 = (lo32 + (hi32 - lo32) * rng.uniform(0.25, 0.75, 6)).astype(np.float32)
        r = dict(q=q0, qc=np.zeros(6, np.float32), v=rng.normal(0, 0.5, 6).astype(np.float32),
                 a=rng.uniform(-1, 1, 6).astype(np.float32), aux=None, warm=warm)
        for k, x in (("q", q), ("qc", qc), ("v", v), ("a", a), ("aux", aux)):
            if x is not None:
                r[k] = x
        rows.append(r)

    def with_dof(j, **kw):
        out = {}
        for k, x in kw.items():
            if k == "warm":
                out[k] = x
                continue
            z = (lo32 + (hi32 - lo32) * rng.uniform(0.25, 0.75, 6)).astype(np.float32) if k == "q" else (
                np.zeros(6, np.float32) if k == "qc" else (rng.normal(0, 0.5, 6).astype(np.float32) if k == "v" else rng.uniform(-1, 1, 6).astype(np.float32)))
            z[j] = x
            out[k] = z
        return out

    for j in range(6):
        for side, lim in ((-1, lo32[j]), (1, hi32[j])):
            for depth in (1e-6, 3e-4, 1e-3, 3e-3, 0.03):          # solimp width 1e-3: ramp, its end and saturation
                for vin in (2.0, -2.0):                            # into the limit / out of it
                    add(**with_dof(j, q=np.float32(lim + side * depth), v=np.float32(side * vin)))
            for k in (-3, -1, 0, 1, 3):                            # within ulps of the limit, nonzero compensation
                qj = lim
                for _ in range(abs(k)):   # (at lo = 0: steps of 1e-8, clear of subnormals)
                    qj = np.nextafter(qj, np.float32(np.inf if k > 0 else -np.inf)) if lim != 0 else np.float32(qj + np.sign(k) * 1e-8)
                ulp = float(np.spacing(np.float32(max(abs(float(lim)), 1e-3))))
                for qcj in (0.3 * ulp, -0.3 * ulp, 0.49 * ulp) if lim != 0 else (1e-9, -1e-9, 3e-8):
                    add(**with_dof(j, q=np.float32(qj), qc=np.float32(qcj), v=np.float32(side * 0.7)))
        # servo torque far beyond forcerange (Env05: target through aux) and large velocities (large bias terms)
        add(**with_dof(j, v=np.float32(25.0)))
        add(**with_dof(j, v=np.float32(-25.0), a=np.float32(1.0)))
        add(**with_dof(j, a=np.float32(0.004)))                    # inside the friction deadband (stick)
        add(**with_dof(j, a=np.float32(-0.9)))                     # well outside (slip)
    add(v=rng.normal(0, 12.0, 6).astype(np.float32))
    add(q=lo32 - np.float32(2e-3), v=np.full(6, -1.0, np.float32))  # rows on every dof
    add(q=hi32 + np.float32(2e-3), v=np.full(6, -1.0, np.float32))
    for warm in ("exact", "zero", "x100"):
        for _ in range(6):
            add(warm=warm)
        add(q=lo32 - np.float32(5e-4), v=np.full(6, -1.0, np.float32), warm=warm)
    # servo targets beyond ctrlrange and within an ulp of it: Env01/02/06 reach ctrlrange only where the joint range
    # touches it (the target is q + 0.075 a); Env05 sets any target through aux
    for j in range(6):
        for lim, sgn in ((clo32[j], -1), (chi32[j], 1)):
            if task == 5:
                for t in (lim + sgn * 0.2, np.nextafter(lim, np.float32(sgn * np.inf)), lim, np.nextafter(lim, np.float32(-sgn * np.inf))):
                    aux = np.zeros(6, np.float32)
                    aux[j] = t
                    add(**with_dof(j, a=np.float32(0.0)), aux=aux)
                aux = np.zeros(6, np.float32)
                aux[j] = lim - sgn * np.float32(1.5)
                add(**with_dof(j, a=np.float32(0.0)), aux=aux)     # |kp (target - q)| far beyond forcerange
            elif (sgn < 0 and lim == lo32[j]) or (sgn > 0 and lim == hi32[j]):
                for qj in (lim, np.nextafter(lim, np.float32(-sgn * np.inf))):
                    for aj in (sgn * 1.0, np.float32(0.0), sgn * 1e-6):
                        add(**with_dof(j, q=np.float32(qj), a=np.float32(aj), v=np.float32(0.0)))
    m = len(rows)
    st = {k: np.repeat(v[:, :1], m, axis=1).copy() for k, v in base.items()}
    st["qpos"] = np.stack([r["q"] for r in rows], axis=1)
    st["qpos_comp"] = np.stack([r["qc"] for r in rows], axis=1)
    st["qvel"] = np.stack([r["v"] for r in rows], axis=1)
    st["qacc_warm"] = np.zeros((6, m), np.float32)
    if task == 5:
        st["aux"][:6] = np.stack([r["aux"] if r["aux"] is not None else r["q"] for r in rows], axis=1)
    return st, np.stack([r["a"] for r in rows]), np.array([r["warm"] for r in rows])


def _prepare(st, task):
    """Keep the step free of RNG-drawing events: episode clock 0 under a far TimeLimit, Env05's lost-cube counter 0,
    Env02's stale end-effector far from the block (no relocation)."""
    st["counters"][0] = 0
    st["counters"][2] = 0
    if task in (2, 6):
        st["snap"][0:3] = 50.0
    return st


def _targets(task, st, act, out):
    """Servo target pairs (ctrl_hi, ctrl_lo) as the kernel forms them, and their exact fp64 sum (the reference's ctrl)."""
    q = st["qpos"].T.astype(np.float32)
    qc = st["qpos_comp"].T.astype(np.float32)
    if task == 5:
        hi = out["aux"][:6].T.astype(np.float32)          # the kernel stores the command it used: aux[0:6]
        lo = np.zeros_like(hi)
    else:
        hi = q
        lo = _round32(_two_sum(act.astype(np.float64) * np.float64(STEP_SCALE), -qc.astype(np.float64)))  # fma(a, s, -qc)
    return hi, lo, hi.astype(np.float64) + lo.astype(np.float64)


def _device_target(hi, lo, clo, chi):
    """The kernel's effective target: its `in` test on the fp32 sum, then the pair or the clamped sum."""
    s = (hi + lo).astype(np.float32)
    inside = (s >= clo) & (s <= chi)
    return np.where(inside, hi.astype(np.float64) + lo.astype(np.float64), np.clip(s, clo, chi).astype(np.float64))


# ------------------------------------------------------------------------------------------------ 1. the right kernel
@pytest.mark.parametrize("task", TASKS)
def test_short_step_ctx_runs_the_default_kernel(spec, task):
    """The fp64 tests below drive the shipped kernel one or two substeps at a time through a ctx with nsubstep 1 or 2.
    That only tests the default kernel while so100_create leaves nsubstep out of its specialisation check: if it ever
    takes it in, this fails here instead of the tests below silently checking the generic kernel."""
    from so100_mujoco_rl_b200.tasks import FLAG_GENERIC_KERNEL
    for nsub in (1, 2, 16):
        for ranges in (None, UNIT):
            env = _env(spec, task, 64, nsub, ranges=ranges)
            assert env.kernel_variant == "specialised", (task, nsub, ranges)
            env.close()
        env = _env(spec, task, 64, nsub, flags=FLAG_GENERIC_KERNEL)
        assert env.kernel_variant == "generic", (task, nsub)
        env.close()


# ------------------------------------------------------------------------------------------------ 2. one and two substeps vs fp64
def _bounds(mref, q_true, v, w_in, a_ref, kv, kp, frc, ctrl, dtarget):
    """Per-env max-norm bound on |qacc - qacc_fp64| after the first substep, from fp32 rounding.

    The projected Gauss-Seidel iterates towards the minimiser of  a'Ma/2 - b'a + (per-dof friction and limit rows); the
    rows are separable convex functions, so the minimiser moves by at most ||M^-1||_inf times a change of b (or of M a).
    M = armature (0.1 per dof) + a PSD link inertia, so ||M^-1||_2 <= 10 and cond(M) < 1.3; ||M^-1||_inf and the smallest
    diagonal entry m are taken from each env's fp64 M.
      * b = clamp(kp (target - q) - kv v) - bias.  The generated dynamics run on MUFU sin/cos (2^-21.2 each; a link's
        rotation enters a torque through at most 5 joints) and on constants rounded to fp32 (2^-24, ~20 operations
        deep): 5 * 2^-21.2 + 20 * 2^-24 < 2^-18, relative to the magnitudes summed, 1 + |bias| + |kv v| + ||M|| |a|.
      * The servo term rounds kp (target - q) and the target pair (cl + qc, a fma or a mul and a sub): 4 * 2^-24 kp |e|.
        The kernel's `in` test runs on the fp32 sum ctrl_hi + ctrl_lo: a sum within an ulp of ctrlrange can take the
        other branch than the exact sum.  Such envs are identified from the inputs (dtarget = |kernel's target - exact
        target|, zero for every other env) and carry kp dtarget in their bound.
      * The sweeps run in fp32: a coordinate update sums up to 6 products of magnitude |b| + ||M|| |a| and divides by m,
        ~16 roundings: 2^-20 (1 + |b| + ||M|| |a|) / m, plus 2^-20 |a| for the row terms (xl ~ |a| where a row is active).
        A 1e2-off warm start leaves at most an ulp of itself: 2^-24 |w|.
    The limit-row presence test needs no split: the reference carries the fp32 limits, q - lo is exact near a limit
    (Sterbenz), so (q - lo) - qc has the sign of the exact q - qc - lo (asserted per sample by _presence_agrees)."""
    Mp, bias = _host_forward(mref, q_true, v)
    M = _unpack(Mp)
    minv = np.abs(np.linalg.inv(M)).sum(axis=2).max(axis=1)
    mnorm = np.abs(M).sum(axis=2).max(axis=1)
    mmin = np.diagonal(M, axis1=1, axis2=2).min(axis=1)
    amax = np.abs(a_ref).max(axis=1)
    serv = kp * np.abs(ctrl - q_true)
    kvv = np.abs(kv * v)
    bsz = np.minimum(serv + kvv, frc).max(axis=1) + np.abs(bias).max(axis=1)
    db = 2.0 ** -18 * (1 + np.abs(bias).max(axis=1) + kvv.max(axis=1) + mnorm * amax) + 4 * U * serv.max(axis=1) \
        + (kp * dtarget).max(axis=1)
    gs = 2.0 ** -20 * ((1 + bsz + mnorm * amax) / mmin + amax)
    return minv * db + gs + U * np.abs(w_in).max(axis=1)


def _presence_agrees(q, qc, lo, hi):
    """The kernel's compensated presence test in fp32 against the exact one, per (env, dof)."""
    q32, qc32 = q.astype(np.float32), qc.astype(np.float32)
    dev = (((q32 - lo) - qc32) < 0) | (((hi - q32) + qc32) < 0)
    qt = q.astype(np.float64) - qc.astype(np.float64)
    ref = (qt - lo < 0) | (hi - qt < 0)
    return dev == ref


def _run_short(spec, task, nsub, st, act, ranges=None, P=None):
    env = _env(spec, task, st["qpos"].shape[1], nsub, ranges=ranges)
    if ranges is not None:
        env.reset()          # draws every env's values from the ranges
    env.set_state({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in st.items()})
    if P is not None:
        env.set_params({k: torch.from_numpy(v) for k, v in P.items()})
    s0 = env.stats()
    r = env.step(torch.from_numpy(np.ascontiguousarray(act)).cuda())
    assert int(r.terminated.sum()) == 0 and int(r.truncated.sum()) == 0, "an RNG-drawing reset entered the comparison"
    out = {k: v.cpu().numpy() for k, v in env.get_state().items()}
    obs = r.obs.cpu().numpy()
    Pd = {k: v.cpu().numpy() for k, v in env.get_params().items()} if ranges is not None else None
    s1 = env.stats()
    env.close()
    return out, obs, Pd, s1["solver_unconverged"] - s0["solver_unconverged"], s1["nan_resets"] - s0["nan_resets"]


def _inputs(spec, task, params, rng):
    if params:
        base = _bulk_state(spec, task, 4096)
        cols = rng.choice(4096, 24, replace=False)
        bulk = {k: v[:, cols].copy() for k, v in base.items()}
        cr, cact, cw = _crafted(spec, task, bulk, rng)
        on = np.flatnonzero((cr["qpos_comp"] != 0).any(axis=0))     # the compensated presence test: keep them all
        rest = np.setdiff1d(np.arange(cr["qpos"].shape[1]), on)
        pick = np.concatenate([on, rng.choice(rest, 40, replace=False)])
        cr = {k: v[:, pick] for k, v in cr.items()}
        cact, cw = cact[pick], cw[pick]
    else:
        n = 65536 if task == 1 else 4096
        bulk = _bulk_state(spec, task, n)
        cr, cact, cw = _crafted(spec, task, bulk, rng)
    nb = bulk["qpos"].shape[1]
    st = {k: np.concatenate([bulk[k], cr[k]], axis=1) for k in bulk}
    act = np.concatenate([rng.uniform(-1, 1, (nb, 6)).astype(np.float32), cact])
    warm = np.concatenate([np.array(["bulk"] * nb), cw])
    return _prepare(st, task), act, warm


@pytest.mark.parametrize("params", [False, True], ids=["default", "params"])
@pytest.mark.parametrize("task", TASKS)
def test_one_and_two_substeps_match_fp64(spec, native_lib, task, params):
    """qacc, qvel and qpos after one and after two substeps of the shipped kernel, against the fp64 reference on the same
    inputs and sweep schedule, bounded per env by _bounds (max-norms, no quantiles); the integration bit for bit; the
    snapshot kinematics against the oracle; the block's floor contact against the oracle."""
    from conftest import make_oracle
    rng = np.random.default_rng(100 + task + 10 * params)
    st, act, warm = _inputs(spec, task, params, rng)
    n = st["qpos"].shape[1]
    probe = _env(spec, task, 1, 1)
    kv = probe.derived()[1]
    probe.close()
    lo, hi = _f32(spec.jnt_range[:, 0]), _f32(spec.jnt_range[:, 1])
    clo, chi = spec.act_ctrlrange[:, 0].astype(np.float32), spec.act_ctrlrange[:, 1].astype(np.float32)
    q32, qc32 = st["qpos"].T, st["qpos_comp"].T
    q_true = q32.astype(np.float64) - qc32.astype(np.float64)
    v_in = st["qvel"].T.astype(np.float64)
    assert _presence_agrees(q32, qc32, lo, hi).all()
    on_limit = (((q32 - lo.astype(np.float32)) == 0) | ((hi.astype(np.float32) - q32) == 0)) & (qc32 != 0)
    assert on_limit.sum() >= 6

    ranges = WIDE if params else None
    # per-env reference models (PARAMS: each env's own drawn values); a dry run fixes the drawn values and the Env05 command
    out1, _, P, _, _ = _run_short(spec, task, 1, st, act, ranges=ranges)
    models = [_ref_model(spec, kv, P, i) for i in range(n)] if params else [_ref_model(spec, kv)]
    kpv = (P["kp"].T if params else np.tile(_f32(spec.act_kp), (n, 1))).astype(np.float64)
    kvv = (P["kv"].T if params else np.tile(_f32(kv), (n, 1))).astype(np.float64)
    hi_c, lo_c, ctrl = _targets(task, st, act, out1)
    frc = (np.maximum(np.abs(P["force_lo"]), np.abs(P["force_hi"])).T if params else
           np.tile(np.abs(_f32(spec.act_forcerange)).max(axis=1), (n, 1))).astype(np.float64)
    sl = lambda i: slice(None) if i is None else slice(i, i + 1)  # noqa: E731
    dtarget = np.abs(_device_target(hi_c, lo_c, clo, chi) - np.clip(ctrl, clo.astype(np.float64), chi.astype(np.float64)))

    def ref(nsub, w, variant):
        if not params:
            return _host_substeps(models[0], q_true, v_in, w, ctrl, nsub, variant)
        parts = [_host_substeps(models[i], q_true[i:i + 1], v_in[i:i + 1], w[i:i + 1], ctrl[i:i + 1], nsub, variant) for i in range(n)]
        return tuple(np.concatenate([p[k] for p in parts]) if k < 3 else sum(p[3] for p in parts) for k in range(4))

    # warm starts: the state's own, zero, exact (fp32 of the fp64 solution) or 100x off
    w = st["qacc_warm"].T.astype(np.float64).copy()
    a_star = ref(1, w, 0)[2]
    w[warm == "zero"] = 0.0
    w[warm == "exact"] = _f32(a_star[warm == "exact"])
    w[warm == "x100"] = _f32(100.0 * a_star[warm == "x100"])
    st["qacc_warm"] = w.T.astype(np.float32).copy()

    rec = dict(envs=n, split_ctrl_envs=int((dtarget > 0).any(axis=1).sum()), on_limit_samples=int(on_limit.sum()))
    tol_prev = None
    for nsub in (1, 2):
        out, obs, P2, unconv, nan = _run_short(spec, task, nsub, st, act, ranges=ranges, P=P)
        assert nan == 0
        qr, vr, ar, sr = ref(nsub, w, 0)
        q3, v3, a3, _ = ref(nsub, w, 3)
        if nsub == 1:
            assert unconv == sr[4], "solver_unconverged differs from the fp64 reference's count"
        a_dev = out["qacc_warm"].T.astype(np.float64)
        v_dev = out["qvel"].T.astype(np.float64)
        q_dev = out["qpos"].T.astype(np.float64) - out["qpos_comp"].T.astype(np.float64)
        tol_a = np.concatenate([_bounds(models[i if params else 0], *(x[sl(i)] for x in (q_true, v_in, w, ar, kvv, kpv, frc, ctrl, dtarget)))
                                for i in (range(n) if params else [None])])
        h = spec.timestep
        if nsub == 1:
            tol1 = tol_a
            tol_v = h * tol_a + U * (np.abs(vr).max(axis=1) + 1e-30) * 2
            tol_q = h * tol_v + 1e-12
        else:
            # the second substep starts from states that differ by h dqacc (qvel) and h^2 dqacc (qpos): with the stiffest
            # terms (limit row damping B = 2 / (dmax tc) = 105 s^-1, kv / m <= 70 s^-1) that moves qacc by < 0.25 dqacc_1
            tol_a = tol_a + 0.25 * tol1
            tol_v = h * (tol1 + tol_a) + U * (np.abs(vr).max(axis=1) + 1e-30) * 4
            tol_q = h * tol_v + h * (h * tol1) + 1e-12
        ea = np.abs(a_dev - ar).max(axis=1)
        ev = np.abs(v_dev - vr).max(axis=1)
        eq = np.abs(q_dev - qr).max(axis=1)
        e3 = np.abs(a3 - ar).max(axis=1)
        rec.update({f"nsub{nsub}_qacc_err_max": ea.max(), f"nsub{nsub}_qacc_err_over_bound_max": (ea / tol_a).max(),
                    f"nsub{nsub}_qacc_bound_median": np.median(tol_a), f"nsub{nsub}_qacc_err_host_fp32_mufu_max": e3.max(),
                    f"nsub{nsub}_qacc_err_host_fp32_mufu_over_bound_max": (e3 / tol_a).max(),
                    f"nsub{nsub}_qvel_err_over_bound_max": (ev / tol_v).max(), f"nsub{nsub}_qpos_err_over_bound_max": (eq / tol_q).max(),
                    f"nsub{nsub}_qpos_err_max": eq.max(), f"nsub{nsub}_unconverged": unconv})
        worst = int(np.argmax(ea / tol_a))
        assert (ea <= tol_a).all(), f"nsub {nsub}: env {worst} ({warm[worst]}) |dqacc| {ea[worst]:.3e} > bound {tol_a[worst]:.3e}"
        assert (ev <= tol_v).all(), f"nsub {nsub}: |dqvel| / bound {(ev / tol_v).max():.3g}"
        assert (eq <= tol_q).all(), f"nsub {nsub}: |dqpos| / bound {(eq / tol_q).max():.3g}"

        if nsub == 1:
            _integration_is_exact(st, out, h)
            _snapshot_matches_oracle(spec, task, st, out, rng)
            if task != 5:
                o = make_oracle(task, 1)
                blk_in, blk = st["block"], out["block"]
                idx = rng.choice(n, min(n, 512), replace=False)
                ref_b = np.array([o.block_substeps(float(blk_in[2, i]), float(blk_in[3, i]), 1) for i in idx])
                dz, dvz = np.abs(blk[2, idx] - ref_b[:, 0]), np.abs(blk[3, idx] - ref_b[:, 1])
                # vz' = vz + h a: a and its terms (|aref| <= B |vz| + K imp |dist| ~ 30 m/s^2 resting) in fp32, ~16 roundings
                # (2^-16 relative); z' = z + h vz' rounds to half an ulp of 0.01
                tol_vz = h * 2.0 ** -16 * 30 + U * np.abs(blk_in[3, idx]).max()
                tol_z = float(np.spacing(np.float32(0.01))) + h * tol_vz
                rec.update(block_dz_max=dz.max(), block_dvz_max=dvz.max(), block_dz_bound=tol_z, block_dvz_bound=tol_vz)
                assert dz.max() <= tol_z and dvz.max() <= tol_vz
                assert (blk[:2] == blk_in[:2]).all()
    _record(f"step_kernel_fp64_task{task}_{'params' if params else 'default'}", **rec)


def _integration_is_exact(st, out, h):
    """Given the kernel's own qacc: qvel' = fl(v + h w) (one FFMA) and the compensated position sum with its
    __fmul_rn / __fsub_rn / __fadd_rn, bit for bit."""
    h32 = np.float32(h)
    v, q, qc = st["qvel"], st["qpos"], st["qpos_comp"]
    w = out["qacc_warm"]
    v1 = _round32(_two_sum(v.astype(np.float64), np.float64(h32) * w.astype(np.float64)))   # h w is exact in fp64
    assert np.array_equal(v1.view(np.int32), out["qvel"].view(np.int32)), "qvel' != fl(qvel + h qacc)"
    with np.errstate(over="ignore", invalid="ignore"):
        y = (h32 * v1).astype(np.float32) - qc
        s1 = (q + y).astype(np.float32)
        qc1 = ((s1 - q).astype(np.float32) - y).astype(np.float32)
    assert np.array_equal(s1.view(np.int32), out["qpos"].view(np.int32)), "qpos' differs from the compensated sum"
    assert np.array_equal(qc1.view(np.int32), out["qpos_comp"].view(np.int32)), "qpos_comp' differs from the compensated sum"


def _snapshot_matches_oracle(spec, task, st, out, rng):
    """With one substep the stored kinematics are the start state's: oracle.fk(q - qc), within the MUFU bound of
    DESIGN §4.1 (< 3e-7 m; camera rotation entries: 5 joint rotations of 2^-21.2 each, < 3e-6)."""
    from conftest import make_oracle
    o = make_oracle(task, 1)
    n = st["qpos"].shape[1]
    idx = rng.choice(n, min(n, 1024), replace=False)
    qt = st["qpos"].astype(np.float64) - st["qpos_comp"].astype(np.float64)
    dpos = drot = 0.0
    for i in idx:
        k = o.fk(qt[:, i])
        s = out["snap"][:, i]
        if task == 5:
            dpos = max(dpos, np.abs(s[0:3] - k["cam_xpos"]).max())
            drot = max(drot, np.abs(s[3:12] - k["cam_xmat"]).max())
        else:
            dpos = max(dpos, np.abs(s[0:3] - k["end_pos"]).max(), abs(s[3] - k["wrist_pos"][2]))
            assert (s[4:7] == st["block"][:3, i]).all()   # the block's pose at the substep's start
    assert dpos < 3e-7 and drot < 3e-6, (dpos, drot)


def test_solver_unconverged_counts_each_env_once(spec, native_lib):
    """Warm starts on a ladder of magnitudes: the large ones exhaust the 7 extra sweeps.  The kernel's solver_unconverged
    must equal the number of envs the fp64 reference leaves unconverged (same schedule, same test), and that number
    must be the envs with the largest warm starts."""
    task, n = 1, 256
    rng = np.random.default_rng(4)
    st = _prepare(_bulk_state(spec, task, 4096), task)
    st = {k: v[:, :n].copy() for k, v in st.items()}
    mag = 10.0 ** np.linspace(0, 30, n)
    sign = rng.choice([-1.0, 1.0], (n, 6))
    st["qacc_warm"] = (mag[:, None] * sign).T.astype(np.float32)
    act = rng.uniform(-1, 1, (n, 6)).astype(np.float32)
    probe = _env(spec, task, 1, 1)
    kv = probe.derived()[1]
    probe.close()
    _, _, _, unconv, _ = _run_short(spec, task, 1, st, act)
    q_true = st["qpos"].T.astype(np.float64) - st["qpos_comp"].T.astype(np.float64)
    hi_c, lo_c, ctrl = _targets(task, st, act, None)
    _, _, _, sr = _host_substeps(_ref_model(spec, kv), q_true, st["qvel"].T, st["qacc_warm"].T, ctrl, 1, 0)
    _record("step_kernel_unconverged_ladder", envs=n, kernel=unconv, fp64_reference=int(sr[4]))
    assert sr[4] > 10 and sr[4] < n - 10
    assert unconv == sr[4]


# ------------------------------------------------------------------------------------------------ 3. warp composition
def _probe_states(spec, base, rng):
    """Probe envs: no limit row, a row on each single dof (ending active / inactive), rows on all dofs, and one whose
    warm start is 1e8 off (it alone takes extra sweeps)."""
    lo32, hi32 = spec.jnt_range[:, 0].astype(np.float32), spec.jnt_range[:, 1].astype(np.float32)
    mid = ((lo32 + hi32) / 2).astype(np.float32)
    probes = []

    def make(q, v, w=None):
        s = {k: v_[:, :1].copy() for k, v_ in base.items()}
        s["qpos"][:, 0] = q
        s["qpos_comp"][:, 0] = 0.0
        s["qvel"][:, 0] = v
        s["qacc_warm"][:, 0] = 0.0 if w is None else w
        probes.append(s)

    make(mid, np.zeros(6, np.float32))
    for j in range(6):
        q = mid.copy()
        v = np.zeros(6, np.float32)
        q[j] = lo32[j] - np.float32(1e-3)
        v[j] = np.float32(-0.5 if j % 2 == 0 else 4.0)     # into the limit (row stays active) / out of it (ends inactive)
        make(q, v)
    make(lo32 - np.float32(1e-3), np.full(6, -0.3, np.float32))
    make(mid, np.zeros(6, np.float32), w=np.float32(1e8) * np.array([1, -1, 1, -1, 1, -1], np.float32))
    return probes


def _fill(spec, kind, m, base, rng):
    lo32, hi32 = spec.jnt_range[:, 0].astype(np.float32), spec.jnt_range[:, 1].astype(np.float32)
    s = {k: np.repeat(v[:, :1], m, axis=1).copy() for k, v in base.items()}
    q = (lo32[:, None] + (hi32 - lo32)[:, None] * rng.uniform(0.2, 0.8, (6, m))).astype(np.float32)
    if kind == "all":
        q = np.where(rng.random((6, m)) < 0.5, lo32[:, None] - 2e-3, hi32[:, None] + 2e-3).astype(np.float32)
    elif kind in ("mix", "nan"):
        r = rng.random((6, m))
        q = np.where(r < 0.15, lo32[:, None] - 1e-3, np.where(r > 0.85, hi32[:, None] + 1e-3, q)).astype(np.float32)
    s["qpos"], s["qpos_comp"] = q, np.zeros((6, m), np.float32)
    s["qvel"] = rng.normal(0, 1, (6, m)).astype(np.float32)
    s["qacc_warm"] = np.zeros((6, m), np.float32)
    if kind == "nan":
        s["qvel"][2, m // 2] = np.nan
        s["qpos"][4, (m // 2 + 1) % m] = np.inf
    return s


def _run_steps(spec, task, st, acts, env_offset, ranges, flags=0):
    n = st["qpos"].shape[1]
    env = _env(spec, task, n, 16, seed=9, env_offset=env_offset, ranges=ranges, flags=flags, max_episode_steps=FAR)
    env.set_state({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in st.items()})
    outs = []
    for a in acts:
        r = env.step(torch.from_numpy(np.ascontiguousarray(a)).cuda())
        outs.append([_bits(t).clone() for t in (r.obs, r.reward, r.terminated, r.truncated)])
    final = {k: _bits(v) for k, v in env.get_state().items()}
    env.close()
    return outs, final


@pytest.mark.parametrize("ranges", [None, UNIT], ids=["default", "unit_params"])
@pytest.mark.parametrize("task", TASKS)
def test_warp_neighbours_do_not_change_an_env(spec, native_lib, task, ranges):
    """WARP_ROWS: the limit rows are swept on warp-uniform branches, for every dof on which ANY lane has a row; a lane
    without one keeps its values through selects.  DESIGN §4.1 states the results are bit for bit the per-lane
    branch's whatever the neighbours do.  Each probe runs 8 steps at lanes 0, 17 and 31 of a warp whose other lanes have
    no rows, rows on every dof, a random mix, or one non-finite env, and as the last env of ragged launches (tail
    threads shadow it); its outputs and state must equal, as int32 bits, its run in a 1-env ctx.  The probe's global
    env id is fixed through env_offset, so that any RNG-keyed draw is the same in every placement."""
    rng = np.random.default_rng(50 + task)
    base = _prepare(_bulk_state(spec, task, 4096), task)
    probes = _probe_states(spec, base, rng)
    G = 5000
    checked = 0
    for p, ps in enumerate(probes):
        acts = [rng.uniform(-1, 1, (1, 6)).astype(np.float32) for _ in range(8)]
        ref_outs, ref_final = _run_steps(spec, task, ps, acts, G, ranges)
        placements = [(kind, lane, 32) for kind in ("none", "all", "mix", "nan") for lane in (0, 17, 31)]
        placements += [("mix", n - 1, n) for n in (33, 257, 1000)]
        for kind, lane, n in placements:
            st = _fill(spec, kind if kind != "none" else "none", n, base, rng)
            for k in st:
                st[k][:, lane] = ps[k][:, 0]
            A = [np.concatenate([rng.uniform(-1, 1, (lane, 6)).astype(np.float32), a, rng.uniform(-1, 1, (n - lane - 1, 6)).astype(np.float32)]) for a in acts]
            outs, final = _run_steps(spec, task, st, A, G - lane, ranges)
            for t, (o, r) in enumerate(zip(outs, ref_outs)):
                assert torch.equal(o[0][lane], r[0][0]) and torch.equal(o[1][lane], r[1][0]), (p, kind, lane, n, t)
                assert torch.equal(o[2][lane], r[2][0]) and torch.equal(o[3][lane], r[3][0]), (p, kind, lane, n, t)
            for k in STATE:
                assert torch.equal(final[k][:, lane], ref_final[k][:, 0]), (p, kind, lane, n, k)
            checked += 1
    _record(f"step_kernel_warp_task{task}_{'unit' if ranges else 'default'}", probes=len(probes), placements=checked)


# ------------------------------------------------------------------------------------------------ 4. tail threads
@pytest.mark.parametrize("n", [257, 1000])
def test_ragged_tail_counts_once_and_writes_nothing_beyond_n(spec, native_lib, n):
    """The last CTA's tail threads shadow the last env.  Made non-finite, that env raises nan_resets by exactly 1;
    made unconverged (a 1e30 warm start), solver_unconverged by exactly 1 - not once per shadowing thread.  The
    caller's output rows past n (a guard region) stay untouched."""
    from so100_mujoco_rl_b200 import _native
    task, G = 1, 300
    base = _prepare(_bulk_state(spec, task, 4096), task)
    for case in ("nan", "unconverged"):
        st = {k: v[:, :n].copy() for k, v in base.items()}
        st["qacc_warm"][:] = 0.0
        if case == "nan":
            st["qvel"][3, n - 1] = np.nan
        else:
            st["qacc_warm"][:, n - 1] = np.float32(1e30)
        env = _env(spec, task, n, 1)
        env.set_state({k: torch.from_numpy(np.ascontiguousarray(v)) for k, v in st.items()})
        f32 = dict(dtype=torch.float32, device="cuda")
        obs, tobs = torch.full((n + G, 15), 7.0, **f32), torch.full((n + G, 15), 7.0, **f32)
        rew, epr = torch.full((n + G,), 7.0, **f32), torch.full((n + G,), 7.0, **f32)
        term, trunc = (torch.full((n + G,), 7, dtype=torch.uint8, device="cuda") for _ in range(2))
        epl = torch.full((n + G,), 7, dtype=torch.int32, device="cuda")
        act = torch.zeros((n + G, 6), **f32)
        s0 = env.stats()
        _native.check(env._L.so100_step(env._h, act.data_ptr(), obs.data_ptr(), rew.data_ptr(), term.data_ptr(), trunc.data_ptr(),
                                        tobs.data_ptr(), epr.data_ptr(), epl.data_ptr(), torch.cuda.current_stream().cuda_stream))
        torch.cuda.synchronize()
        s1 = env.stats()
        dn, du = s1["nan_resets"] - s0["nan_resets"], s1["solver_unconverged"] - s0["solver_unconverged"]
        _record(f"step_kernel_tail_{case}_n{n}", nan_resets=dn, solver_unconverged=du)
        if case == "nan":
            assert dn == 1 and int(term[:n].sum()) == 1 and int(term[n - 1]) == 1
        else:
            assert du == 1 and dn == 0
        for t, fill in ((obs, 7.0), (tobs, 7.0), (rew, 7.0), (epr, 7.0), (term, 7), (trunc, 7), (epl, 7)):
            assert (t[n:] == fill).all(), "a tail thread wrote past the last env"
        env.close()
