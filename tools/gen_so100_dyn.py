#!/usr/bin/env python
"""Emits so100_mujoco_rl_b200/csrc/so100_dyn_gen.cuh: the so100 arm's bias forces and joint-space inertia as
straight-line code specialised to the MJCF's numbers ("model parsed once on the host").

How: the SAME recursion as csrc/so100_dyn.cuh (link-local RNEA + composite rigid bodies) is executed symbolically on a
hash-consed expression DAG whose leaves are sin/cos of the joint angles, the joint velocities and link constants
derived from the ones the library computes (so100_host_constants).  Every link frame is first turned about its joint
axis (`reframe`, in fp64, rounded to fp32 once) so that each constant rotation is Rx(alpha) Rz(theta) with alpha a
quarter turn up to ~1e-5 rad; the Rz(theta) is merged with the joint angle by the angle-addition identity.  Folding
then removes every multiplication by 0.0f / 1.0f / -1.0f and every addition of 0, common sub-expressions are shared,
and a*b+c is emitted as an fma.  Bias forces and M do not depend on the frames, so both kernels compute the same
model; only the fp32 rounding differs.  Every operation is emitted explicitly (so_fma / so_mul / so_add / so_sub), so
no kernel that inlines the code can contract it differently from another.

The generated header also carries the fp64 constants it was built from; so100_create compares them with the model it
is given and launches the generic kernel when they differ (any other MJCF still works, only slower).

    python tools/gen_so100_dyn.py            # rewrite the header
    python tools/gen_so100_dyn.py --check    # exit 1 if the committed header is stale
"""
from __future__ import annotations

import argparse
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, "so100_mujoco_rl_b200", "csrc", "so100_dyn_gen.cuh")
NJ = 6


# ------------------------------------------------------------------------------------------- expression DAG
class G:
    """Hash-consed DAG.  A value is (sign, node id); node kinds: const, var, add, sub, mul."""

    def __init__(self):
        self.nodes = []  # (kind, a, b) with a/b = node ids, or payload for const/var
        self.memo = {}
        self.region = None  # the part of the recursion being built: its operations are counted under this name
        self.node_region = []

    def _mk(self, key):
        if key not in self.memo:
            self.memo[key] = len(self.nodes)
            self.nodes.append(key)
            self.node_region.append(self.region)
        return self.memo[key]

    def const(self, x):
        x = float(np.float32(x))
        if x == 0.0:
            return V(self, 1, self._mk(("const", 0.0, None)))
        return V(self, 1 if x > 0 else -1, self._mk(("const", abs(x), None)))

    def var(self, name):
        return V(self, 1, self._mk(("var", name, None)))

    def is_const(self, nid):
        return self.nodes[nid][0] == "const"

    def cval(self, nid):
        return self.nodes[nid][1]


class V:
    __slots__ = ("g", "s", "n")

    def __init__(self, g, s, n):
        self.g, self.s, self.n = g, s, n

    # ---- helpers
    def _w(self, o):
        return o if isinstance(o, V) else self.g.const(o)

    def is_zero(self):
        return self.g.is_const(self.n) and self.g.cval(self.n) == 0.0

    def cv(self):
        return self.s * self.g.cval(self.n) if self.g.is_const(self.n) else None

    def __neg__(self):
        return V(self.g, -self.s, self.n)

    def __add__(self, o):
        o = self._w(o)
        if self.is_zero():
            return o
        if o.is_zero():
            return self
        a, b = self.cv(), o.cv()
        if a is not None and b is not None:
            return self.g.const(a + b)
        if self.n == o.n:
            return self * 2.0 if self.s == o.s else self.g.const(0.0)
        if self.s == o.s:
            x, y = sorted((self.n, o.n))
            return V(self.g, self.s, self.g._mk(("add", x, y)))
        # s*(a - b): keep the sign of the first operand outside
        pos, neg = (self, o) if self.s > 0 else (o, self)
        return V(self.g, 1, self.g._mk(("sub", pos.n, neg.n)))

    __radd__ = __add__

    def __sub__(self, o):
        return self + (-self._w(o))

    def __rsub__(self, o):
        return self._w(o) + (-self)

    def __mul__(self, o):
        o = self._w(o)
        if self.is_zero() or o.is_zero():
            return self.g.const(0.0)
        a, b = self.cv(), o.cv()
        if a is not None and b is not None:
            return self.g.const(a * b)
        if a is not None and abs(a) == 1.0:
            return V(self.g, o.s * (1 if a > 0 else -1), o.n)
        if b is not None and abs(b) == 1.0:
            return V(self.g, self.s * (1 if b > 0 else -1), self.n)
        x, y = sorted((self.n, o.n))
        return V(self.g, self.s * o.s, self.g._mk(("mul", x, y)))

    __rmul__ = __mul__


# ------------------------------------------------------------------------------------------- the recursion (mirrors so100_dyn.cuh)
def cross(a, b):
    return [a[1] * b[2] - a[2] * b[1], a[2] * b[0] - a[0] * b[2], a[0] * b[1] - a[1] * b[0]]


def vadd(a, b):
    return [x + y for x, y in zip(a, b)]


def _rz(c, s):
    return np.array([[c, -s, 0.0], [s, c, 0.0], [0.0, 0.0, 1.0]])


QUARTER = [(1.0, 0.0), (0.0, 1.0), (-1.0, 0.0), (0.0, -1.0)]  # exact cos, sin of k * 90 degrees
SNAP = 1e-9  # fp64 residue of the MJCF's quaternions, far below fp32 rounding: treated as 0


def _sym(I):
    return np.array([[I[0], I[3], I[4]], [I[3], I[1], I[5]], [I[4], I[5], I[2]]])


def reframe(flat):
    """The link constants in modified-DH-like frames, in fp64.

    Each link frame may turn about its own joint axis (and the base frame about gravity) without changing bias or M.
    Frame i is turned by phi_i so that the constant rotation of link i + 1 is Rx(alpha) Rz(theta): a rotation about x
    whose alpha is a quarter turn up to ~1e-5 rad, then a turn about the joint axis that merges with the joint angle.
    phi_0 .. phi_4 are exact quarter turns (the inertial constants are only permuted); the last link is turned by its
    own small residual so that it needs no merge, and link 0's rotation goes into the base frame (gravity rotates).
    Each frame's origin may also slide along its joint axis: it moves to where link i + 1's origin has z = 0.
    Returns per link (ct, st, (ca, sa) or None, p, m, h, I, arm) and a0."""
    R = [np.array(flat[23 * i:23 * i + 9]).reshape(3, 3) for i in range(NJ)]
    phi = []
    for i in range(NJ - 1):
        Rn = R[i + 1]
        k = 0 if Rn[0, 2] == 0 and Rn[1, 2] == 0 else round(np.degrees(np.arctan2(Rn[0, 2], -Rn[1, 2])) / 90) % 4
        phi.append(_rz(*QUARTER[k]))
    R5 = phi[-1].T @ R[-1]
    b = np.arctan2(R5[2, 0], R5[2, 1])
    phi.append(_rz(np.cos(b), -np.sin(b)))
    base = R[0] @ phi[0]
    rot, p, h, S, m = [], [], [], [], [flat[23 * i + 12] for i in range(NJ)]
    for i in range(NJ):
        f = flat[23 * i:23 * i + 23]
        Rp = np.eye(3) if i == 0 else phi[i - 1].T @ R[i] @ phi[i]
        ct, st, ca, sa = (0.0 if abs(x) < SNAP else x for x in (Rp[0, 0], -Rp[0, 1], Rp[2, 2], -Rp[1, 2]))
        Rx = np.array([[1.0, 0.0, 0.0], [0.0, ca, -sa], [0.0, sa, ca]])
        assert np.abs(Rx @ _rz(ct, st) - Rp).max() < SNAP, f"link {i}: constant rotation is not Rx(alpha) Rz(theta)"
        rot.append((ct, st, ca, sa))
        p.append(np.array(f[9:12]) if i == 0 else phi[i - 1].T @ np.array(f[9:12]))  # link 0's origin is never used
        h.append(phi[i].T @ np.array(f[13:16]))
        S.append(phi[i].T @ _sym(f[16:22]) @ phi[i])
    # frame i's origin slides along its joint axis onto the plane z = 0 of link i + 1's origin; the inertia moves to the
    # new origin (about o' = o + d z: I' = I + (|h'|^2 - |h|^2) / m E - (h' h'^T - h h^T) / m, h' = h - m d z)
    for i in range(NJ - 1):
        d = p[i + 1][2]
        p[i + 1] = np.array([p[i + 1][0], p[i + 1][1], 0.0])
        if i > 0:
            p[i] = p[i] + d * np.array([0.0, -rot[i][3], rot[i][2]])
        hn = h[i] - np.array([0.0, 0.0, m[i] * d])
        S[i] = S[i] + (hn @ hn - h[i] @ h[i]) / m[i] * np.eye(3) - (np.outer(hn, hn) - np.outer(h[i], h[i])) / m[i]
        h[i] = hn
    links = []
    for i in range(NJ):
        ct, st, ca, sa = rot[i]
        I = [S[i][0, 0], S[i][1, 1], S[i][2, 2], S[i][0, 1], S[i][0, 2], S[i][1, 2]]
        links.append((ct, st, None if (ca, sa) == (1.0, 0.0) else (ca, sa), list(p[i]), m[i], list(h[i]), I, flat[23 * i + 22]))
    a0 = base.T @ np.array(flat[138:141])
    return links, [0.0 if abs(x) < SNAP * abs(a0).max() else x for x in a0]


class Link:
    def __init__(self, g, frame, sj, cj):
        ct, st, rx, p, m, h, I, arm = frame
        r32 = lambda v: [float(np.float32(x)) for x in v]  # noqa: E731
        self.p, self.m, self.h, self.I, self.arm = r32(p), r32([m])[0], r32(h), r32(I), r32([arm])[0]
        # the turn about the joint axis merges with the joint angle: Rz(theta) Rz(q) = Rz(theta + q)
        ct, st = r32([ct, st])
        self.planar = (ct, st) != (1.0, 0.0)
        self.s, self.c = (sj * ct + cj * st, cj * ct - sj * st) if self.planar else (sj, cj)
        if rx is None:
            self.R = None
        else:
            ca, sa = r32(rx)
            self.R = np.array([[1.0, 0.0, 0.0], [0.0, ca, -sa], [0.0, sa, ca]])

    def to_parent(self, v):
        x, y, z = self.c * v[0] - self.s * v[1], self.s * v[0] + self.c * v[1], v[2]
        if self.R is None:
            return [x, y, z]
        R = self.R
        return [x * R[r, 0] + y * R[r, 1] + z * R[r, 2] for r in range(3)]

    def to_child(self, v):
        if self.R is None:
            x, y, z = v
        else:
            R = self.R
            x, y, z = (v[0] * R[0, k] + v[1] * R[1, k] + v[2] * R[2, k] for k in range(3))
        return [self.c * x + self.s * y, self.c * y - self.s * x, z]


def sym_mv(I, v):
    return [I[0] * v[0] + I[3] * v[1] + I[4] * v[2], I[3] * v[0] + I[1] * v[1] + I[5] * v[2],
            I[4] * v[0] + I[5] * v[1] + I[2] * v[2]]


def add_composite(L, m, h, I, pm, ph, pI):
    s, c = L.s, L.c
    c2, s2 = c * c - s * s, (c * s) * 2.0
    av, bv = (I[0] + I[1]) * 0.5, (I[0] - I[1]) * 0.5
    xx, yy, xy = av + bv * c2 - I[3] * s2, av - bv * c2 + I[3] * s2, bv * s2 + I[3] * c2
    xz, yz, zz = c * I[4] - s * I[5], s * I[4] + c * I[5], I[2]
    if L.R is None:
        J = [xx, yy, zz, xy, xz, yz]
    else:
        R = L.R
        S = [[xx, xy, xz], [xy, yy, yz], [xz, yz, zz]]
        T = [[sum((S[k][j] * R[r, k] for k in range(3)), 0.0) for j in range(3)] for r in range(3)]  # R*S
        Jm = lambda a, b: sum((T[a][k] * R[b, k] for k in range(3)), 0.0)  # noqa: E731  (R*S*R^T)[a][b]
        J = [Jm(0, 0), Jm(1, 1), Jm(2, 2), Jm(0, 1), Jm(0, 2), Jm(1, 2)]
    hr = L.to_parent(h)
    p = L.p
    t = [hr[k] * 2.0 + m * p[k] for k in range(3)]
    pt = p[0] * t[0] + p[1] * t[1] + p[2] * t[2]
    nI = [pI[0] + J[0] + pt - t[0] * p[0], pI[1] + J[1] + pt - t[1] * p[1], pI[2] + J[2] + pt - t[2] * p[2],
          pI[3] + J[3] - (t[1] * p[0] + t[0] * p[1]) * 0.5, pI[4] + J[4] - (t[2] * p[0] + t[0] * p[2]) * 0.5,
          pI[5] + J[5] - (t[2] * p[1] + t[1] * p[2]) * 0.5]
    nh = [ph[k] + hr[k] + m * p[k] for k in range(3)]
    return pm + m, nh, nI


def build(flat):
    g = G()
    g.region = "RNE forward"  # including the planar merges of the joint angles
    s = [g.var(f"s[{i}]") for i in range(NJ)]
    c = [g.var(f"c[{i}]") for i in range(NJ)]
    qd = [g.var(f"qd[{i}]") for i in range(NJ)]
    K = lambda x: g.const(x)  # noqa: E731
    frames, a0 = reframe(flat)
    links = [Link(g, frames[i], s[i], c[i]) for i in range(NJ)]
    for L in links:
        L.p = [K(x) for x in L.p]; L.h = [K(x) for x in L.h]; L.I = [K(x) for x in L.I]
        L.m = K(L.m); L.arm = K(L.arm)
        if L.R is not None:
            L.R = np.array([[K(x) for x in row] for row in L.R], dtype=object)
    a0 = [K(x) for x in a0]
    zero = K(0.0)
    w, wd, a = [zero] * 3, [zero] * 3, a0
    f, n = [None] * NJ, [None] * NJ
    for i, L in enumerate(links):
        ap = a
        if i > 0:
            ap = vadd(vadd(a, cross(wd, L.p)), cross(w, cross(w, L.p)))
        wl, wdl, al = L.to_child(w), L.to_child(wd), L.to_child(ap)
        wdl = [wdl[0] + qd[i] * wl[1], wdl[1] - qd[i] * wl[0], wdl[2]]
        wl = [wl[0], wl[1], wl[2] + qd[i]]
        f[i] = vadd(vadd([L.m * x for x in al], cross(wdl, L.h)), cross(wl, cross(wl, L.h)))
        n[i] = vadd(vadd(sym_mv(L.I, wdl), cross(wl, sym_mv(L.I, wl))), cross(L.h, al))
        w, wd, a = wl, wdl, al
    bias, M = [None] * NJ, {}
    cm, ch, cI = links[-1].m, links[-1].h, links[-1].I
    for i in range(NJ - 1, -1, -1):
        bias[i] = n[i][2]
        g.region = "M entries"
        M[(i, i)] = cI[2] + links[i].arm
        cf, cn = [-ch[1], ch[0], zero], [cI[4], cI[5], cI[2]]
        for j in range(i - 1, -1, -1):
            Lc = links[j + 1]
            cf = Lc.to_parent(cf)
            cn = vadd(Lc.to_parent(cn), cross(Lc.p, cf))
            M[(i, j)] = cn[2]
        if i > 0:
            L = links[i]
            g.region = "RNE backward"
            fp = L.to_parent(f[i])
            npv = vadd(L.to_parent(n[i]), cross(L.p, fp))
            f[i - 1] = vadd(f[i - 1], fp)
            n[i - 1] = vadd(n[i - 1], npv)
            g.region = "composite inertia"
            cm, ch, cI = add_composite(L, cm, ch, cI, links[i - 1].m, links[i - 1].h, links[i - 1].I)
    outs = [(f"bias[{i}]", bias[i]) for i in range(NJ)]
    outs += [(f"M[{i * (i + 1) // 2 + j}]", M[(i, j)]) for i in range(NJ) for j in range(i + 1)]
    return g, outs, [L.planar for L in links]


# ------------------------------------------------------------------------------------------- emission
def f32_lit(x):
    return f"{float(np.float32(x)).hex()}f" if x not in (0.0,) else "0.0f"


def emit(g, outs):
    live, stack = set(), [v.n for _, v in outs]
    while stack:
        n = stack.pop()
        if n in live:
            continue
        live.add(n)
        k, a, b = g.nodes[n]
        if k in ("add", "sub", "mul"):
            stack += [a, b]
    uses = {}
    for n in live:
        k, a, b = g.nodes[n]
        if k in ("add", "sub", "mul"):
            uses[a] = uses.get(a, 0) + 1
            uses[b] = uses.get(b, 0) + 1
    for _, v in outs:
        uses[v.n] = uses.get(v.n, 0) + 1
    # a mul that feeds exactly one add/sub is fused into it (one product per fma); then a mul whose every consumer is an
    # add/sub with no product fused yet is formed inside each of them (k fma instead of one mul and k additions)
    consumers = {}
    for n in sorted(live):
        k, a, b = g.nodes[n]
        if k in ("add", "sub", "mul"):
            consumers.setdefault(a, []).append(n); consumers.setdefault(b, []).append(n)
    fuse_into = {}  # add/sub node -> the mul it forms
    for n in sorted(live):
        k, a, b = g.nodes[n]
        if k in ("add", "sub"):
            for x in (a, b):
                if g.nodes[x][0] == "mul" and uses.get(x, 0) == 1:
                    fuse_into[n] = x
                    break
    outn = {v.n for _, v in outs}
    for n in sorted(live):
        cs = consumers.get(n, [])
        if (g.nodes[n][0] == "mul" and len(cs) > 1 and n not in outn
                and all(g.nodes[x][0] in ("add", "sub") and x not in fuse_into for x in cs)):
            for x in cs:
                fuse_into[x] = n
    fused = set(fuse_into.values())

    def ref(n):
        k, a, b = g.nodes[n]
        if k == "const":
            return f"T({f32_lit(a)})"
        if k == "var":
            return a
        return f"t{n}"

    nop = {r: {"fma": 0, "mul": 0, "add": 0} for r in dict.fromkeys(g.node_region)}  # regions in recursion order
    lines = []
    for n in sorted(live):
        k, a, b = g.nodes[n]
        if k in ("const", "var") or n in fused:
            continue
        cnt = nop[g.node_region[n]]
        if k == "mul":
            lines.append(f"  const T t{n} = so_mul({ref(a)}, {ref(b)});"); cnt["mul"] += 1
            continue
        if n in fuse_into:
            m = fuse_into[n]
            fa, o = m == a, b if m == a else a
            _, x, y = g.nodes[m]
            if k == "add":
                e = f"so_fma({ref(x)}, {ref(y)}, {ref(o)})"
            elif fa:   # m - o
                e = f"so_fma({ref(x)}, {ref(y)}, -{ref(o)})"
            else:      # o - m
                e = f"so_fma(-{ref(x)}, {ref(y)}, {ref(o)})"
            cnt["fma"] += 1
        else:
            e = f"so_{k}({ref(a)}, {ref(b)})"; cnt["add"] += 1
        lines.append(f"  const T t{n} = {e};")
    for name, v in outs:
        lines.append(f"  {name} = {'-' if v.s < 0 else ''}{ref(v.n)};")
    return lines, nop


def host_constants():
    from so100_mujoco_rl_b200 import _native
    from so100_mujoco_rl_b200.model import load_model
    L = _native.lib()
    m = load_model().to_ctypes()
    out = (ctypes.c_double * 141)()
    L.so100_host_constants.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_double)]
    _native.check(L.so100_host_constants(ctypes.byref(m), out))
    return list(out)


N_SOLVER = 16 * NJ + 6 * NJ + 1 + 13
CON_FIELDS = ["fr_D", "fr_B", "fr_loss", "lo", "hi", "lim_B", "lim_K", "invw", "imp0", "imp1", "imp_w", "imp_mid", "imp_pow",
              "imp_rw", "imp_rmid", "imp_r1mid"]
ACT_FIELDS = ["kp", "kv", "ctrl_lo", "ctrl_hi", "frc_lo", "frc_hi"]
BLK_FIELDS = ["half_z", "gz", "K", "B", "lam_scale", "imp0", "imp1", "imp_w", "imp_rw", "imp_mid", "imp_rmid", "imp_r1mid", "imp_pow"]


def host_solver_constants():
    """fp32 solver / servo constants in the ConC<float> + ActC<float> layout (so100_host_solver_constants)."""
    from so100_mujoco_rl_b200 import _native
    from so100_mujoco_rl_b200.model import load_model
    L = _native.lib()
    m = load_model().to_ctypes()
    out = (ctypes.c_float * N_SOLVER)()
    L.so100_host_solver_constants.argtypes = [ctypes.c_void_p, ctypes.POINTER(ctypes.c_float), ctypes.c_int]
    _native.check(L.so100_host_solver_constants(ctypes.byref(m), out, N_SOLVER))
    return [float(x) for x in out]


def f32lit(x: float) -> str:
    return float(np.float32(x)).hex() + "f"


def render_solver(sflat):
    rows = lambda k: "{" + ", ".join(f32lit(v) for v in sflat[k * NJ:(k + 1) * NJ]) + "}"  # noqa: E731
    con = ",\n      ".join(f"/* {name} */ {rows(k)}" for k, name in enumerate(CON_FIELDS))
    act = ",\n      ".join(f"/* {name} */ {rows(len(CON_FIELDS) + k)}" for k, name in enumerate(ACT_FIELDS))
    blk = ", ".join(f"/* {name} */ {f32lit(sflat[22 * NJ + 1 + k])}" for k, name in enumerate(BLK_FIELDS))
    hexs = ",\n    ".join(", ".join(f32lit(x) for x in sflat[i:i + 6]) for i in range(0, N_SOLVER, 6))
    return f"""
// fp32 solver / servo constants (ConC<float> then ActC<float>, so100_host_solver_constants layout); compared exactly too.
#define SO100_GEN_NS {N_SOLVER}
static const float kGenSolverConstants[SO100_GEN_NS] = {{
    {hexs}}};

// The same numbers as literals: after unrolling they become immediates of the solver / servo instructions.
SO_HD void so100_gen_solver_constants(ConC<float>& K, ActC<float>& A, BlkC<float>& Bk) {{
  K = ConC<float>{{
      {con}}};
  A = ActC<float>{{
      {act},
      /* h */ {f32lit(sflat[22 * NJ])}}};
  Bk = BlkC<float>{{{blk}}};
}}
"""


def render():
    flat = host_constants()
    sflat = host_solver_constants()
    g, outs, planar = build(flat)
    lines, by_region = emit(g, outs)
    nop = {k: sum(r[k] for r in by_region.values()) for k in ("fma", "mul", "add")}
    hexd = ",\n    ".join(", ".join(float(x).hex() for x in flat[i:i + 4]) for i in range(0, 141, 4))
    total = nop["fma"] + nop["mul"] + nop["add"]
    regions = "\n".join(f"//   {name:18s} {r['fma']:4d} fma + {r['mul']:4d} mul + {r['add']:4d} add/sub = {sum(r.values()):4d}"
                        for name, r in by_region.items())
    hdr = f"""// GENERATED by tools/gen_so100_dyn.py from so100_mujoco_rl_b200/assets/so100_scene.xml — do not edit.
// so100 arm: bias[6] = RNE(q, qd, 0) incl. gravity and M[21] = joint-space inertia (packed lower triangle, armature
// included), specialised to the model's fp32 constants.  Same recursion as so100_dyn.cuh::dyn_bias_mass.
// Straight-line: {nop['fma']} fma + {nop['mul']} mul + {nop['add']} add/sub = {total} instructions
// ({2 * nop['fma'] + nop['mul'] + nop['add']} FLOP); planar-merged links: {[i for i, p in enumerate(planar) if p]}.
// By the part of the recursion that creates each operation:
{regions}
#pragma once
#include "so100_dyn.cuh"

// fp64 constants this file was generated from (so100_host_constants layout); so100_create compares them exactly.
static const double kGenDynConstants[SO100_GEN_N] = {{
    {hexd}}};

template <typename T>
SO_HD void dyn_bias_mass_so100(const T* s, const T* c, const T* qd, T* bias, T* M) {{
"""
    return hdr + "\n".join(lines) + "\n}\n" + render_solver(sflat), nop


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--check", action="store_true")
    args = ap.parse_args()
    txt, nop = render()
    if args.check:
        cur = open(OUT).read() if os.path.exists(OUT) else ""
        if cur != txt:
            print("so100_dyn_gen.cuh is stale: run python tools/gen_so100_dyn.py")
            sys.exit(1)
        print("so100_dyn_gen.cuh is up to date")
        return
    open(OUT, "w").write(txt)
    print(f"wrote {OUT}: {nop}")


if __name__ == "__main__":
    main()
