// so100_dyn.cuh — arm dynamics of the so100 chain as straight-line recursions in LINK-LOCAL frames.
//
// This is the B200 restatement of what MuJoCo's mj_fwdPosition / mj_fwdVelocity compute for this model
// (mj_kinematics, mj_crb, mj_rne; reference call site: mujoco.mj_step at
// src/so100_mujoco_rl/envs/env01_v1.py:26, env02_v1.py:39, env03_v1.py:142).  It is NOT MuJoCo's formulation:
//   * every link frame is re-based on the host so that its hinge turns about the local +z axis; crossing a joint is
//     then a constant 3x3 times a planar (c,s) rotation, and no world-frame kinematics is needed in the substep loop;
//   * bias forces: recursive Newton-Euler with the spatial inertia (m, h = m*com, I about the joint origin);
//   * joint-space inertia: composite rigid bodies accumulated tip -> base in the same backward sweep;
//   * everything lives in registers of ONE thread per environment; loops are fully unrolled.
// The same templates run on the host in double (T = double) to derive MuJoCo's compile-time constants
// (dof_M0, dof_invweight0, actuator kv) and on the device in float.
#pragma once

#include <cmath>

#ifdef __CUDACC__
#define SO_HD __host__ __device__ __forceinline__
#else
#define SO_HD inline
#endif

#define SO_NJ 6

struct SoTrue { static constexpr bool value = true; };
struct SoFalse { static constexpr bool value = false; };

SO_HD float so_fma(float a, float b, float c) { return fmaf(a, b, c); }
SO_HD double so_fma(double a, double b, double c) { return a * b + c; }
template <typename T>
SO_HD T so_fma(T a, T b, T c) { return a * b + c; }

// A separate multiplication / addition that ptxas may not contract into an fma: the generated dynamics says where it
// fuses, so every kernel that inlines it rounds the same way whatever the surrounding code.
#ifdef __CUDA_ARCH__
SO_HD float so_mul(float a, float b) { return __fmul_rn(a, b); }
SO_HD float so_add(float a, float b) { return __fadd_rn(a, b); }
SO_HD float so_sub(float a, float b) { return __fsub_rn(a, b); }
#endif
template <typename T>
SO_HD T so_mul(T a, T b) { return a * b; }
template <typename T>
SO_HD T so_add(T a, T b) { return a + b; }
template <typename T>
SO_HD T so_sub(T a, T b) { return a - b; }

// sin/cos of a joint angle inside the substep loop.  Device fp32: MUFU.SIN / MUFU.COS (|err| <= 2^-21.2 on [-pi, pi],
// CUDA C Programming Guide table of intrinsics; joint ranges of this model stay inside +-3.1416).  A 4e-7 error in
// sin/cos moves a gravity torque of <= 1 N m by 4e-7 N m, i.e. the servo's equilibrium by 1e-8 rad; the task
// kinematics (end-effector / camera pose) by < 3e-7 m.  -DSO100_ACCURATE_SINCOS restores sincosf().
SO_HD void so_sincos(float x, float* s, float* c) {
#if defined(__CUDA_ARCH__) && !defined(SO100_ACCURATE_SINCOS)
  __sincosf(x, s, c);
#elif defined(__CUDA_ARCH__)
  sincosf(x, s, c);
#else
  *s = std::sin(x); *c = std::cos(x);
#endif
}
SO_HD void so_sincos(double x, double* s, double* c) { *s = std::sin(x); *c = std::cos(x); }

template <typename T>
struct LinkC {
  T R[9];  // parent <- child constant rotation (row-major), before the joint rotation
  T p[3];  // child origin in the parent frame
  T m;     // mass
  T h[3];  // m * com (child frame)
  T I[6];  // inertia about the joint origin, child frame: xx yy zz xy xz yz
  T arm;   // armature
};

template <typename T>
struct DynC {
  LinkC<T> L[SO_NJ];
  T a0[3];  // acceleration of the base frame = -gravity, in base coordinates
};

// packed lower triangle, i >= j
SO_HD constexpr int midx(int i, int j) { return i * (i + 1) / 2 + j; }

template <typename T>
SO_HD void cross3(const T* a, const T* b, T* o) {
  T x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  o[0] = x; o[1] = y; o[2] = z;
}
// o += a x b
template <typename T>
SO_HD void cross3_acc(const T* a, const T* b, T* o) {
  T x = a[1] * b[2] - a[2] * b[1], y = a[2] * b[0] - a[0] * b[2], z = a[0] * b[1] - a[1] * b[0];
  o[0] += x; o[1] += y; o[2] += z;
}
// child -> parent:  o = R * Rz(c,s) * v
template <typename T>
SO_HD void to_parent(const T* R, T s, T c, const T* v, T* o) {
  T x = c * v[0] - s * v[1], y = s * v[0] + c * v[1], z = v[2];
  T o0 = R[0] * x + R[1] * y + R[2] * z, o1 = R[3] * x + R[4] * y + R[5] * z, o2 = R[6] * x + R[7] * y + R[8] * z;
  o[0] = o0; o[1] = o1; o[2] = o2;
}
// parent -> child:  o = Rz(c,s)^T * R^T * v
template <typename T>
SO_HD void to_child(const T* R, T s, T c, const T* v, T* o) {
  T x = R[0] * v[0] + R[3] * v[1] + R[6] * v[2], y = R[1] * v[0] + R[4] * v[1] + R[7] * v[2],
    z = R[2] * v[0] + R[5] * v[1] + R[8] * v[2];
  o[0] = c * x + s * y; o[1] = c * y - s * x; o[2] = z;
}
template <typename T>
SO_HD void sym_mv(const T* I, const T* v, T* o) {  // I: xx yy zz xy xz yz
  T x = I[0] * v[0] + I[3] * v[1] + I[4] * v[2], y = I[3] * v[0] + I[1] * v[1] + I[5] * v[2],
    z = I[4] * v[0] + I[5] * v[1] + I[2] * v[2];
  o[0] = x; o[1] = y; o[2] = z;
}

// Move a composite spatial inertia (m, h, I about the child origin, child frame) into the parent frame about the
// parent origin and ADD it to (pm, ph, pI).
template <typename T>
SO_HD void add_composite(const LinkC<T>& L, T s, T c, T m, const T* h, const T* I, T& pm, T* ph, T* pI) {
  // 1) planar rotation Rz(q) of the symmetric tensor (double-angle form)
  T c2 = c * c - s * s, s2 = T(2) * c * s;
  T av = T(0.5) * (I[0] + I[1]), bv = T(0.5) * (I[0] - I[1]);
  T xx = av + bv * c2 - I[3] * s2, yy = av - bv * c2 + I[3] * s2, xy = bv * s2 + I[3] * c2;
  T xz = c * I[4] - s * I[5], yz = s * I[4] + c * I[5], zz = I[2];
  // 2) constant rotation: J = R * I1 * R^T
  const T* R = L.R;
  T t0[3], t1[3], t2[3];  // rows of R*I1
  for (int r = 0; r < 3; r++) {
    T a = R[3 * r], b = R[3 * r + 1], d = R[3 * r + 2];
    T u0 = a * xx + b * xy + d * xz, u1 = a * xy + b * yy + d * yz, u2 = a * xz + b * yz + d * zz;
    if (r == 0) { t0[0] = u0; t0[1] = u1; t0[2] = u2; }
    else if (r == 1) { t1[0] = u0; t1[1] = u1; t1[2] = u2; }
    else { t2[0] = u0; t2[1] = u1; t2[2] = u2; }
  }
  T Jxx = t0[0] * R[0] + t0[1] * R[1] + t0[2] * R[2];
  T Jyy = t1[0] * R[3] + t1[1] * R[4] + t1[2] * R[5];
  T Jzz = t2[0] * R[6] + t2[1] * R[7] + t2[2] * R[8];
  T Jxy = t0[0] * R[3] + t0[1] * R[4] + t0[2] * R[5];
  T Jxz = t0[0] * R[6] + t0[1] * R[7] + t0[2] * R[8];
  T Jyz = t1[0] * R[6] + t1[1] * R[7] + t1[2] * R[8];
  // 3) first moment, then the shift of the reference point by p (parallel-axis with a non-central first moment):
  //    I' = J + (p.t) 1 - (p t^T + t p^T)/2,   t = 2 h_r + m p
  T hr[3];
  to_parent(R, s, c, h, hr);
  const T* p = L.p;
  T tx = T(2) * hr[0] + m * p[0], ty = T(2) * hr[1] + m * p[1], tz = T(2) * hr[2] + m * p[2];
  T pt = p[0] * tx + p[1] * ty + p[2] * tz;
  pI[0] += Jxx + pt - p[0] * tx;
  pI[1] += Jyy + pt - p[1] * ty;
  pI[2] += Jzz + pt - p[2] * tz;
  pI[3] += Jxy - T(0.5) * (p[0] * ty + p[1] * tx);
  pI[4] += Jxz - T(0.5) * (p[0] * tz + p[2] * tx);
  pI[5] += Jyz - T(0.5) * (p[1] * tz + p[2] * ty);
  ph[0] += hr[0] + m * p[0]; ph[1] += hr[1] + m * p[1]; ph[2] += hr[2] + m * p[2];
  pm += m;
}

// bias[6] = RNE(q, qd, qdd = 0) incl. gravity;  M[21] = joint-space inertia incl. armature (packed lower triangle).
template <typename T>
SO_HD void dyn_bias_mass(const DynC<T>& C, const T* s, const T* c, const T* qd, T* bias, T* M) {
  T f[SO_NJ][3], n[SO_NJ][3];
  {
    T w[3] = {T(0), T(0), T(0)}, wd[3] = {T(0), T(0), T(0)}, a[3] = {C.a0[0], C.a0[1], C.a0[2]};
#pragma unroll
    for (int i = 0; i < SO_NJ; i++) {
      const LinkC<T>& L = C.L[i];
      T ap[3] = {a[0], a[1], a[2]};
      if (i > 0) {  // origin of link i rides on link i-1 at offset p
        T t[3];
        cross3_acc(wd, L.p, ap);
        cross3(w, L.p, t);
        cross3_acc(w, t, ap);
      }
      T wl[3], wdl[3], al[3];
      to_child(L.R, s[i], c[i], w, wl);
      to_child(L.R, s[i], c[i], wd, wdl);
      to_child(L.R, s[i], c[i], ap, al);
      wdl[0] += qd[i] * wl[1];  // (E^T w_parent) x (e_z qd)
      wdl[1] -= qd[i] * wl[0];
      wl[2] += qd[i];
      // f = m a + wd x h + w x (w x h);   n = I wd + w x (I w) + h x a     (about the joint origin)
      T t[3], Iw[3];
      f[i][0] = L.m * al[0]; f[i][1] = L.m * al[1]; f[i][2] = L.m * al[2];
      cross3_acc(wdl, L.h, f[i]);
      cross3(wl, L.h, t);
      cross3_acc(wl, t, f[i]);
      sym_mv(L.I, wdl, n[i]);
      sym_mv(L.I, wl, Iw);
      cross3_acc(wl, Iw, n[i]);
      cross3_acc(L.h, al, n[i]);
#pragma unroll
      for (int k = 0; k < 3; k++) { w[k] = wl[k]; wd[k] = wdl[k]; a[k] = al[k]; }
    }
  }
  // backward sweep: wrench accumulation (bias) + composite inertia and its columns (M)
  T cm = C.L[SO_NJ - 1].m, ch[3], cI[6];
#pragma unroll
  for (int k = 0; k < 3; k++) ch[k] = C.L[SO_NJ - 1].h[k];
#pragma unroll
  for (int k = 0; k < 6; k++) cI[k] = C.L[SO_NJ - 1].I[k];
#pragma unroll
  for (int i = SO_NJ - 1; i >= 0; i--) {
    bias[i] = n[i][2];
    M[midx(i, i)] = cI[2] + C.L[i].arm;
    // unit acceleration about local z of the composite body: force (e_z x h), moment I e_z
    T cf[3] = {-ch[1], ch[0], T(0)}, cn[3] = {cI[4], cI[5], cI[2]};
#pragma unroll
    for (int j = i - 1; j >= 0; j--) {
      const LinkC<T>& Lc = C.L[j + 1];
      to_parent(Lc.R, s[j + 1], c[j + 1], cf, cf);
      to_parent(Lc.R, s[j + 1], c[j + 1], cn, cn);
      cross3_acc(Lc.p, cf, cn);
      M[midx(i, j)] = cn[2];
    }
    if (i > 0) {
      const LinkC<T>& L = C.L[i];
      T fp[3], np[3];
      to_parent(L.R, s[i], c[i], f[i], fp);
      to_parent(L.R, s[i], c[i], n[i], np);
      cross3_acc(L.p, fp, np);
#pragma unroll
      for (int k = 0; k < 3; k++) { f[i - 1][k] += fp[k]; n[i - 1][k] += np[k]; }
      T pm = C.L[i - 1].m, ph[3], pI[6];
#pragma unroll
      for (int k = 0; k < 3; k++) ph[k] = C.L[i - 1].h[k];
#pragma unroll
      for (int k = 0; k < 6; k++) pI[k] = C.L[i - 1].I[k];
      add_composite(L, s[i], c[i], cm, ch, cI, pm, ph, pI);
      cm = pm;
#pragma unroll
      for (int k = 0; k < 3; k++) ch[k] = ph[k];
#pragma unroll
      for (int k = 0; k < 6; k++) cI[k] = pI[k];
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Soft constraints (MuJoCo friction-loss + joint-limit rows, SURVEY.md Appendix B.6/B.7) and their solve.
template <typename T>
struct ConC {
  T fr_D[SO_NJ], fr_B[SO_NJ], fr_loss[SO_NJ];  // friction-loss row: D = 1/R, aref = -B*qd, |force| <= loss
  T lo[SO_NJ], hi[SO_NJ];                      // joint range
  T lim_B[SO_NJ], lim_K[SO_NJ], invw[SO_NJ];   // limit row: aref = -B*(J qd) - K*imp*dist, R = (1-imp)/imp*invw
  T imp0[SO_NJ], imp1[SO_NJ], imp_w[SO_NJ], imp_mid[SO_NJ], imp_pow[SO_NJ];
  T imp_rw[SO_NJ], imp_rmid[SO_NJ], imp_r1mid[SO_NJ];  // 1/width, 1/mid, 1/(1-mid): no divisions on the device
};

// Position servo + integrator constants (MuJoCo actuator gainprm/biasprm, ctrlrange, forcerange; SURVEY.md B.4)
template <typename T>
struct ActC {
  T kp[SO_NJ], kv[SO_NJ], ctrl_lo[SO_NJ], ctrl_hi[SO_NJ], frc_lo[SO_NJ], frc_hi[SO_NJ];
  T h;  // timestep
};

// Free block resting on the floor plane, reduced to its z coordinate (exact by symmetry: DESIGN.md "Block-floor
// contact", which restates the MuJoCo contact semantics this folds).  All contact rows are identical, so the
// constrained acceleration is closed form:  a = (g + lam aref) / (1 + lam),  lam = lam_scale * imp / (1 - imp),
// lam_scale = rows / (2 mu^2 (1 + mu^2)) = 4 for 4 corner contacts x 4 pyramid rows at mu = 1.
template <typename T>
struct BlkC {
  T half_z, gz, K, B, lam_scale;
  T imp0, imp1, imp_w, imp_rw, imp_mid, imp_rmid, imp_r1mid, imp_pow;
};

template <typename T>
SO_HD T so_pow(T x, T p) {
#ifdef __CUDA_ARCH__
  return (sizeof(T) == 4) ? (T)powf((float)x, (float)p) : (T)pow((double)x, (double)p);
#else
  return (T)std::pow((double)x, (double)p);
#endif
}

// MuJoCo getimpedance with margin 0: d0 at dist 0 rising to d1 at |dist| >= width along a power-law sigmoid
template <typename T>
SO_HD T impedance_f(T d0, T d1, T w, T rw, T mid, T rmid, T r1mid, T p, T dist) {
  if (d0 == d1 || w <= T(1e-15)) return T(0.5) * (d0 + d1);
  T x = (dist < 0 ? -dist : dist) * rw;
  if (x >= T(1)) return d1;
  if (x <= T(0)) return d0;
  T y;
  if (p == T(1)) y = x;
  else if (p == T(2)) y = (x <= mid) ? x * x * rmid : T(1) - (T(1) - x) * (T(1) - x) * r1mid;
  else if (x <= mid) y = so_pow(x, p) / so_pow(mid, p - T(1));
  else y = T(1) - so_pow(T(1) - x, p) / so_pow(T(1) - mid, p - T(1));
  return d0 + y * (d1 - d0);
}
template <typename T>
SO_HD T impedance(const ConC<T>& K, int j, T dist) {
  return impedance_f(K.imp0[j], K.imp1[j], K.imp_w[j], K.imp_rw[j], K.imp_mid[j], K.imp_rmid[j], K.imp_r1mid[j], K.imp_pow[j], dist);
}

#ifdef __CUDACC__
#define SO_NOINLINE __host__ __device__ __noinline__
#else
#define SO_NOINLINE
#endif
SO_HD float so_clamp(float x, float lo, float hi) {
#ifdef __CUDA_ARCH__
  return fminf(fmaxf(x, lo), hi);
#else
  return x < lo ? lo : (x > hi ? hi : x);
#endif
}
SO_HD double so_clamp(double x, double lo, double hi) { return x < lo ? lo : (x > hi ? hi : x); }
template <typename T>
SO_HD T so_clamp(T x, T lo, T hi) { return x < lo ? lo : (x > hi ? hi : x); }
// 1/x for the solver's preconditioners (1/M_jj, 1/(M_jj + D)): MUFU.RCP, <= 1 ulp.  A relative error eps here moves the
// Gauss-Seidel fixed point by eps relative, i.e. by the same amount as one fp32 rounding of the result.
SO_HD float so_rcp(float x) {
#ifdef __CUDA_ARCH__
  float r;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
#else
  return 1.0f / x;
#endif
}
template <typename T>
SO_HD T so_rcp(T x) { return T(1) / x; }
SO_HD float so_rsqrt(float x) {
#ifdef __CUDA_ARCH__
  return rsqrtf(x);
#else
  return 1.0f / std::sqrt(x);
#endif
}
SO_HD double so_rsqrt(double x) { return 1.0 / sqrt(x); }
template <typename T>
SO_HD T so_rsqrt(T x) { return T(1) / T(sqrt((double)x)); }

// One mj_step of the block's z coordinate: soft floor contact + gravity, semi-implicit Euler.
template <typename T>
SO_HD void block_substep(const BlkC<T>& Kb, T h, T& z, T& vz) {
  T a = Kb.gz, dist = z - Kb.half_z;
  if (!(dist > T(0))) {  // mjc_PlaneBox keeps the corner contacts while dist <= margin = 0
    T imp = impedance_f(Kb.imp0, Kb.imp1, Kb.imp_w, Kb.imp_rw, Kb.imp_mid, Kb.imp_rmid, Kb.imp_r1mid, Kb.imp_pow, dist);
    T aref = -Kb.B * vz - Kb.K * imp * dist;
    T lam = Kb.lam_scale * imp * so_rcp(T(1) - imp);
    if (Kb.gz < aref) a = (Kb.gz + lam * aref) * so_rcp(T(1) + lam);  // rows active iff J a - aref < 0
  }
  vz += h * a;
  z += h * vz;
}

// Friction-loss row on one dof: the exact minimiser over x of  m x^2/2 - c x + huber_f(x - af)  is closed form,
//   t = c - m af;  F = clamp(t * D/(m+D), -loss, loss);  x = af + (t - F)/m        (used inline in solve_qacc)

// Joint j is outside its range: one unilateral limit row (MuJoCo mj_instantiateLimit) joins the friction row on this
// dof.  Evaluated ONCE per substep; the sweeps only see (xl, sDl, rm2, kap2).  With random actions the arm sits on
// its limits often (several start poses are on them), so this is not a cold path.
template <typename T>
SO_HD void limit_row(const ConC<T>& K, int j, T m, T q, T qc, T qd, T& xl, T& sDl, T& rm2, T& kap2) {
  T dlo = (q - K.lo[j]) - qc, dhi = (K.hi[j] - q) + qc;  // true qpos = q - qc (compensated sum)
  T side = dlo < T(0) ? T(1) : T(-1), dist = dlo < T(0) ? dlo : dhi;
  T imp = impedance(K, j, dist);
  T R = (T(1) - imp) * K.invw[j] * so_rcp(imp);
  R = R < T(1e-15) ? T(1e-15) : R;
  T Dl = so_rcp(R);
  xl = side * (-K.lim_B[j] * (side * qd) - K.lim_K[j] * imp * dist);  // row active while side*(x - xl) < 0
  sDl = side * Dl;
  T m2 = m + Dl;
  rm2 = so_rcp(m2);
  kap2 = K.fr_D[j] * so_rcp(m2 + K.fr_D[j]);
}

// Projected Gauss-Seidel on   min_a  a^T M a / 2 - b^T a + sum_j [ friction_j(a_j) + limit_j(a_j) ]:
// every constraint row touches ONE dof, so each coordinate update is the exact 1-D minimiser.  M ~ armature-dominated
// (cond < 1.3) => contraction ~1e-2 per sweep (measured against the fp64 Newton oracle, see DESIGN.md).
// a[] holds the warm start on entry and the solution on exit; returns the largest update of the LAST sweep.
// qc[] is the compensation term of the fp32 position integration (zeros when T = double).  loss[] is the friction loss of
// the dofs: K.fr_loss, or an env's own values (so100_set_param_ranges).
// WARP_ROWS (device, all 32 lanes converged at the call): the limit rows are set up and swept per dof on a warp-uniform
// branch, taken when ANY lane of the warp has a row on that dof; lanes without one keep their values through selects
// (sDl = 0 makes the row's activity test false), so every lane's result is bit for bit the per-lane branch's.
template <typename T, bool WARP_ROWS = false>
SO_HD T solve_qacc(const ConC<T>& K, const T* loss, const T* M, const T* b, const T* q, const T* qc, const T* qd, T* a, int sweeps) {
  // per-dof constants of this substep.  Friction row only:  t = c - m af,  x = af + (t - clamp(t kap, +-loss)) / m
  //   = (af + t rm) - clamp(t kr, +-lr)   with kr = kap rm, lr = loss rm;  bp = b - m af folds "- m af" into the sum.
  T af[SO_NJ], rm[SO_NJ], kr[SO_NJ], lr[SO_NJ], bp[SO_NJ], xl[SO_NJ], sDl[SO_NJ], rm2[SO_NJ], kap2[SO_NJ], dl[SO_NJ];
  unsigned own = 0u;  // WARP_ROWS: bit j = this lane's joint j is outside its range
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) {
    T m = M[midx(j, j)];
    af[j] = -K.fr_B[j] * qd[j];
    rm[j] = so_rcp(m);
    kr[j] = K.fr_D[j] * so_rcp(m + K.fr_D[j]) * rm[j];
    lr[j] = loss[j] * rm[j];
    bp[j] = b[j] - m * af[j];
    const bool out = (q[j] - K.lo[j]) - qc[j] < T(0) || (K.hi[j] - q[j]) + qc[j] < T(0);
    if (WARP_ROWS) {
      own |= out ? 1u << j : 0u;
    } else {
      xl[j] = T(0); sDl[j] = T(0); rm2[j] = T(0); kap2[j] = T(0); dl[j] = T(0);
      if (out) {
        limit_row(K, j, m, q[j], qc[j], qd[j], xl[j], sDl[j], rm2[j], kap2[j]);
        dl[j] = (sDl[j] < T(0) ? -sDl[j] : sDl[j]) * (xl[j] - af[j]);  // t with the limit row active = t + Dl (xl - af)
      }
    }
  }
  unsigned rows = own;  // WARP_ROWS: bit j = some lane of the warp has a limit row on dof j (xl .. dl are set only then)
#ifdef __CUDA_ARCH__
  if (WARP_ROWS) rows = __reduce_or_sync(0xffffffffu, own);
#endif
  if (WARP_ROWS) {
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) {
      if (rows & (1u << j)) {
        T xl_, sDl_, rm2_, kap2_;
        limit_row(K, j, M[midx(j, j)], q[j], qc[j], qd[j], xl_, sDl_, rm2_, kap2_);
        const T dl_ = (sDl_ < T(0) ? -sDl_ : sDl_) * (xl_ - af[j]);
        const bool mine = own & (1u << j);
        xl[j] = mine ? xl_ : T(0); sDl[j] = mine ? sDl_ : T(0); rm2[j] = mine ? rm2_ : T(0); kap2[j] = mine ? kap2_ : T(0);
        dl[j] = mine ? dl_ : T(0);
      }
    }
  }
  T last = T(0), amax = T(1);  // amax: scale of the iterate, refreshed by every tracked sweep (a warm start left by a
                               // contact solve can be 100x the contact-free solution)
  // one Gauss-Seidel sweep; TRACK: also return the largest coordinate update
  auto sweep = [&](auto track) -> T {
    constexpr bool TRACK = decltype(track)::value;
    T big = T(0);
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) {
      // t = bp_j - sum_{k != j} M_jk a_k; the coordinate updated last (j - 1) enters last: one fma on the critical path
      constexpr int NJ = SO_NJ;
      const int prev = (j + NJ - 1) % NJ;
      T t = bp[j];
#pragma unroll
      for (int k = 0; k < SO_NJ; k++) {
        if (k == j || k == prev) continue;
        t -= (k < j ? M[midx(j, k)] : M[midx(k, j)]) * a[k];
      }
      t -= (prev < j ? M[midx(j, prev)] : M[midx(prev, j)]) * a[prev];
      T x = so_fma(t, rm[j], af[j]) - so_clamp(t * kr[j], -lr[j], lr[j]);
      if (WARP_ROWS ? (rows & (1u << j)) != 0u : sDl[j] != T(0)) {  // limit row present: active iff the limit-free minimiser violates it
        T t2 = t + dl[j];
        T x2 = af[j] + (t2 - so_clamp(t2 * kap2[j], -loss[j], loss[j])) * rm2[j];
        x = sDl[j] * (x - xl[j]) < T(0) ? x2 : x;
      }
      if (TRACK) {
        T d = x - a[j];
        d = d < T(0) ? -d : d;
        big = d > big ? d : big;
        const T ax = x < T(0) ? -x : x;
        amax = ax > amax ? ax : amax;
      }
      a[j] = x;
    }
    return big;
  };
  // fixed schedule: sweeps-1 plain sweeps, then the last scheduled one with bookkeeping, then (rare, per-lane) extra
  // sweeps while the last one still moved qacc by > 1e-3 relative
#pragma unroll 1
  for (int sw = 0; sw < sweeps - 1; sw++) sweep(SoFalse());
#pragma unroll 1
  for (int sw = 0; sw < 7; sw++) {
    amax = T(1);
    last = sweep(SoTrue());
    if (!(last > T(1e-3) * amax)) break;
  }
  return last;
}

// ---------------------------------------------------------------------------------------------------------------
// World kinematics of the points the tasks look at (done once per env step, in the last substep: SURVEY Q3).
template <typename T>
struct KinC {
  T base_R[9], base_p[3];
  int ee_body, wrist_body, cam_body;
  T ee_off[3], cam_pos[3], cam_R[9];
};
template <typename T>
struct KinOut { T end_pos[3], wrist[3], cam_pos[3], cam_R[9]; };

template <typename T>
SO_HD void mat_vec(const T* R, const T* v, T* o) {
  T x = R[0] * v[0] + R[1] * v[1] + R[2] * v[2], y = R[3] * v[0] + R[4] * v[1] + R[5] * v[2],
    z = R[6] * v[0] + R[7] * v[1] + R[8] * v[2];
  o[0] = x; o[1] = y; o[2] = z;
}
template <typename T>
SO_HD void mat_mul(const T* A, const T* B, T* o) {
  T r[9];
#pragma unroll
  for (int i = 0; i < 3; i++)
#pragma unroll
    for (int j = 0; j < 3; j++) r[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
#pragma unroll
  for (int i = 0; i < 9; i++) o[i] = r[i];
}

template <typename T, bool WANT_CAM>
SO_HD void task_kinematics(const DynC<T>& C, const KinC<T>& Kc, const T* s, const T* c, KinOut<T>& out) {
  T R[9], o[3];
#pragma unroll
  for (int k = 0; k < 9; k++) R[k] = Kc.base_R[k];
#pragma unroll
  for (int k = 0; k < 3; k++) o[k] = Kc.base_p[k];
#pragma unroll
  for (int i = 0; i < SO_NJ; i++) {
    const LinkC<T>& L = C.L[i];
    if (i > Kc.ee_body && i > Kc.wrist_body && (!WANT_CAM || i > Kc.cam_body)) break;
    T t[3];
    mat_vec(R, L.p, t);
    o[0] += t[0]; o[1] += t[1]; o[2] += t[2];
    mat_mul(R, L.R, R);
#pragma unroll
    for (int r = 0; r < 3; r++) {  // R <- R * Rz(q_i)
      T x = R[3 * r], y = R[3 * r + 1];
      R[3 * r] = c[i] * x + s[i] * y;
      R[3 * r + 1] = c[i] * y - s[i] * x;
    }
    if (i == Kc.wrist_body) { out.wrist[0] = o[0]; out.wrist[1] = o[1]; out.wrist[2] = o[2]; }
    if (i == Kc.ee_body) {
      mat_vec(R, Kc.ee_off, t);
      out.end_pos[0] = o[0] + t[0]; out.end_pos[1] = o[1] + t[1]; out.end_pos[2] = o[2] + t[2];
    }
    if (WANT_CAM && i == Kc.cam_body) {
      mat_vec(R, Kc.cam_pos, t);
      out.cam_pos[0] = o[0] + t[0]; out.cam_pos[1] = o[1] + t[1]; out.cam_pos[2] = o[2] + t[2];
      mat_mul(R, Kc.cam_R, out.cam_R);
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------
// Arm <-> floor contact: the jaws' primitive box colliders ("pads", so_arm100_camera.xml:60-61, :108-111, :120-123 of
// the reference) against the floor plane z = 0 (env01.xml:39).  MuJoCo semantics (mjc_PlaneBox, mj_instantiateContact,
// mj_makeImpedance; DESIGN.md "Arm-floor contact"): every box corner below the plane is a contact with condim 3 and a
// pyramidal cone, i.e. four unilateral rows  J_n +- mu J_t1, J_n +- mu J_t2  with dense Jacobians,
// aref = -B (J qd) - K imp(dist) dist  and  R = (1 - imp)/imp * 2 mu^2 (1 + mu^2) body_invweight0.  The rows couple all
// joints with a stiffness of ~3e3 against an inertia of ~0.1, which is what Newton's method is for: the per-dof
// Gauss-Seidel of solve_qacc stays the path of envs that touch nothing, envs with a penetrating corner take
// contact_solve() instead.
#define SO_MAX_PAD 8
#define SO_MAX_CON 16  // contacts the out-of-line solve keeps (4 per pad possible; > 4 at once is 0.3 % of the touching envs, > 8 unseen)

template <typename T>
struct PadC {
  int n;                     // pads, sorted by link; 0 = no arm <-> floor contact
  int first[SO_NJ + 1];      // pads of link i are [first[i], first[i + 1])
  T p[SO_MAX_PAD][3];        // box centre in the (re-based) link frame
  T A[SO_MAX_PAD][9];        // half-extent vectors: A[3 r + m] = component r of box axis m times its half size
  T diag[SO_MAX_PAD];        // 2 mu^2 (1 + mu^2) body_invweight0_trans(link):  R = (1 - imp)/imp * diag
  T K, B, mu;                // contact reference (mixed solref, refsafe) and sliding friction of the pair
  T imp0, imp1, imp_w, imp_rw, imp_mid, imp_rmid, imp_r1mid, imp_pow;  // mixed + clamped solimp and reciprocals
};

// Broad phase, every substep, every env: does ANY pad corner lie below the floor?  Only the z row of each link's world
// rotation and the z of its origin are propagated (~16 operations per link), then per pad the height of its lowest
// corner  cz - sum_m |w . A_m|.  Exact: bit k of the result is set iff contact_solve would find a contact on pad k.
template <typename T>
SO_HD unsigned pads_touch(const DynC<T>& C, const KinC<T>& Kc, const PadC<T>& P, const T* s, const T* c, T margin = T(0)) {
  T w0 = Kc.base_R[6], w1 = Kc.base_R[7], w2 = Kc.base_R[8], oz = Kc.base_p[2];
  unsigned touch = 0u;
#pragma unroll
  for (int i = 0; i < SO_NJ; i++) {
    const LinkC<T>& L = C.L[i];
    oz += w0 * L.p[0] + w1 * L.p[1] + w2 * L.p[2];
    const T t0 = w0 * L.R[0] + w1 * L.R[3] + w2 * L.R[6], t1 = w0 * L.R[1] + w1 * L.R[4] + w2 * L.R[7],
            t2 = w0 * L.R[2] + w1 * L.R[5] + w2 * L.R[8];
    w0 = c[i] * t0 + s[i] * t1; w1 = c[i] * t1 - s[i] * t0; w2 = t2;
    for (int k = P.first[i]; k < P.first[i + 1]; k++) {
      const T cz = oz + w0 * P.p[k][0] + w1 * P.p[k][1] + w2 * P.p[k][2];
      T ext = T(0);
#pragma unroll
      for (int m = 0; m < 3; m++) {
        const T u = w0 * P.A[k][m] + w1 * P.A[k][3 + m] + w2 * P.A[k][6 + m];
        ext += u < T(0) ? -u : u;
      }
      touch |= (cz - ext < margin) ? (1u << k) : 0u;
    }
  }
  return touch;
}

// ---- storage of the SERIAL contact solve (contact_newton: the host's fp64 path and the device's fallback).  It keeps, per
// contact, its three Jacobian rows (float), four parameters (c0, b_y, b_x, D: float), six residual / slope values for the
// line search (double), and the 6x6 Hessian (double), in the thread's local memory.  The device's normal path is the
// cooperative solve further down, whose storage is a CoopSlot in shared memory.
template <typename TC, int NC>
struct ContactLocal {
  static constexpr int kMaxCon = NC;
  TC jf[NC * 18], pf[NC * 4];
  double rd[NC * 6], hd[21];
  SO_HD TC& J(int c, int axis, int j) { return jf[(c * 3 + axis) * 6 + j]; }
  SO_HD TC& par(int c, int m) { return pf[c * 4 + m]; }
  SO_HD double& res(int c, int m) { return rd[c * 6 + m]; }
  SO_HD double& H(int k) { return hd[k]; }
};
// In-place Cholesky of the packed lower-triangular 6x6 SPD matrix held by the store, then solve H x = r.
template <typename T, typename Store>
SO_HD bool chol_solve6(Store& S, const T* r, T* x) {
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) {
    T d = S.H(midx(j, j));
#pragma unroll
    for (int k = 0; k < j; k++) { const T l = S.H(midx(j, k)); d -= l * l; }
    if (!(d > T(0))) return false;
    const T rd = so_rsqrt(d);
    S.H(midx(j, j)) = rd;  // the diagonal holds 1 / L_jj
#pragma unroll
    for (int i = j + 1; i < SO_NJ; i++) {
      T v = S.H(midx(i, j));
#pragma unroll
      for (int k = 0; k < j; k++) v -= S.H(midx(i, k)) * S.H(midx(j, k));
      S.H(midx(i, j)) = v * rd;
    }
  }
  T y[SO_NJ];
#pragma unroll
  for (int i = 0; i < SO_NJ; i++) {
    T v = r[i];
#pragma unroll
    for (int k = 0; k < i; k++) v -= S.H(midx(i, k)) * y[k];
    y[i] = v * S.H(midx(i, i));
  }
#pragma unroll
  for (int i = SO_NJ - 1; i >= 0; i--) {
    T v = y[i];
#pragma unroll
    for (int k = i + 1; k < SO_NJ; k++) v -= S.H(midx(k, i)) * x[k];
    x[i] = v * S.H(midx(i, i));
  }
  return true;
}

// Kinematics of the contact path: world frames of the links from ACCURATE sin / cos, the pads' penetrating corners
// (MuJoCo mjc_PlaneBox), and per contact its three Jacobian rows and row parameters written into the store.
// Returns the number of contacts; -1 (and nothing usable in the store) if more than Store::kMaxCon corners penetrate.
template <typename TC, typename Store>
SO_HD int contact_setup(const DynC<TC>& C, const KinC<TC>& Kc, const PadC<TC>& P, Store& S, const TC* s, const TC* c, const TC* qd,
                        unsigned pad_mask) {
  constexpr int NC = Store::kMaxCon;
  int nc = 0;
  {
    // ---- world kinematics: joint axes (local +z of each link), link origins; contacts of the pads on the way
    TC zax[SO_NJ][3], org[SO_NJ][3], W[9], o[3];
#pragma unroll
    for (int k = 0; k < 9; k++) W[k] = Kc.base_R[k];
#pragma unroll
    for (int k = 0; k < 3; k++) o[k] = Kc.base_p[k];
#pragma unroll
    for (int i = 0; i < SO_NJ; i++) {
      const LinkC<TC>& L = C.L[i];
      TC t[3];
      mat_vec(W, L.p, t);
      o[0] += t[0]; o[1] += t[1]; o[2] += t[2];
      mat_mul(W, L.R, W);
#pragma unroll
      for (int r = 0; r < 3; r++) {  // W <- W * Rz(q_i)
        const TC x = W[3 * r], y = W[3 * r + 1];
        W[3 * r] = c[i] * x + s[i] * y;
        W[3 * r + 1] = c[i] * y - s[i] * x;
      }
#pragma unroll
      for (int k = 0; k < 3; k++) { zax[i][k] = W[3 * k + 2]; org[i][k] = o[k]; }
      for (int k = P.first[i]; k < P.first[i + 1]; k++) {
        if (!(pad_mask >> k & 1u)) continue;  // the broad phase saw this pad's lowest corner above the floor
        TC cw[3], h[3][3];  // box centre and half-extent vectors in the world
        mat_vec(W, P.p[k], cw);
        cw[0] += o[0]; cw[1] += o[1]; cw[2] += o[2];
#pragma unroll
        for (int m = 0; m < 3; m++) {
          const TC v[3] = {P.A[k][m], P.A[k][3 + m], P.A[k][6 + m]};
          mat_vec(W, v, h[m]);
        }
        int found = 0;
        for (int ci = 0; ci < 8 && found < 4; ci++) {  // MuJoCo mjc_PlaneBox: corners in index order, at most 4
          const TC s0 = (ci & 1) ? TC(1) : TC(-1), s1 = (ci & 2) ? TC(1) : TC(-1), s2 = (ci & 4) ? TC(1) : TC(-1);
          const TC ld = s0 * h[0][2] + s1 * h[1][2] + s2 * h[2][2];
          const TC dist = cw[2] + ld;
          if (dist > TC(0) || ld > TC(0)) continue;
          found++;
          if (!(dist < TC(0))) continue;  // in the gap: detected, not instantiated
          if (nc >= NC) return -1;
          const TC px = cw[0] + s0 * h[0][0] + s1 * h[1][0] + s2 * h[2][0], py = cw[1] + s0 * h[0][1] + s1 * h[1][1] + s2 * h[2][1],
                   pz = TC(0.5) * dist;  // corner - n dist / 2
          // point Jacobian, columns j <= i:  z_j x (pos - o_j);  velocity of the point
          TC vx = TC(0), vy = TC(0), vz = TC(0);
#pragma unroll
          for (int j = 0; j < SO_NJ; j++) {
            const bool on = j <= i;
            const TC dx = px - org[j][0], dy = py - org[j][1], dz = pz - org[j][2];
            const TC jx = on ? zax[j][1] * dz - zax[j][2] * dy : TC(0), jy = on ? zax[j][2] * dx - zax[j][0] * dz : TC(0),
                     jz = on ? zax[j][0] * dy - zax[j][1] * dx : TC(0);
            S.J(nc, 0, j) = jz; S.J(nc, 1, j) = jy; S.J(nc, 2, j) = jx;
            vx += jx * qd[j]; vy += jy * qd[j]; vz += jz * qd[j];
          }
          const TC imp = impedance_f(P.imp0, P.imp1, P.imp_w, P.imp_rw, P.imp_mid, P.imp_rmid, P.imp_r1mid, P.imp_pow, dist);
          TC R = (TC(1) - imp) * P.diag[k] / imp;
          R = R < TC(1e-15) ? TC(1e-15) : R;
          // aref of row (sigma, t) = c0 - sigma b_t,  c0 = -B vz - K imp dist,  b_t = B mu v_t
          S.par(nc, 0) = -P.K * imp * dist - P.B * vz;
          S.par(nc, 1) = P.B * P.mu * vy;
          S.par(nc, 2) = P.B * P.mu * vx;
          S.par(nc, 3) = TC(1) / R;
          nc++;
        }
      }
    }
  }
  return nc;
}

// qacc of an env whose pads touch the floor: primal Newton on the full convex problem
//   min_a  1/2 a'Ma - b'a + sum_j [friction_j(a_j) + limit_j(a_j)] + sum_contacts sum_4 rows  D/2 min(0, J a - aref)^2
// with the exact generalised Hessian, a Cholesky solve per iteration, and an exact line search: phi'(alpha) along the
// Newton direction is piecewise linear and increasing, and it is evaluated from stored row residuals and slopes (no
// Jacobians), so a safeguarded Newton iteration on it costs a few operations per row.  If no row switched state along
// the step, the step ended on the minimiser of the quadratic piece it started in and the solve is finished.
//
// Two number types.  TC is the kernel's own (float on the device): constants, the substep's inputs, the contact geometry
// and Jacobians.  The SOLVE (residuals, gradient, Hessian, Cholesky, line search) runs in double: the Hessian
// M + sum D J J' mixes a stiffness of ~250 with an inertia of 0.1, so a float solve leaves ~1e-3 of every step in the
// soft directions; measured on 1 024 envs x 16 steps against the fp64 oracle (tools/contact_precision.py): float solve
// p99.9 |dq| 5.7e-4 rad, double solve 2.7e-7.  B200 issues DFMA at half the FFMA rate.
//
// s, c must be ACCURATE sin / cos of the joint angles (not MUFU's): a resting contact penetrates ~2e-7 m.
// Returns the number of gradient/Hessian evaluations (0: no corner is below the floor), negated if the iteration cap
// was hit or the Hessian was not positive definite; *overflow is set if more than Store::kMaxCon corners penetrated
// (the solve is then not attempted with this store: the caller retries with a larger one).
template <typename TC, typename Store>
SO_HD int contact_newton(const DynC<TC>& C, const KinC<TC>& Kc, const PadC<TC>& P, const ConC<TC>& K, const TC* loss, Store& S, const TC* s, const TC* c,
                         const TC* q, const TC* qc, const TC* qd, const TC* M, const TC* b, TC* a, unsigned pad_mask, bool exact_in,
                         int* overflow, int* ls_evals) {
  typedef double T;
  const int nc = contact_setup<TC>(C, Kc, P, S, s, c, qd, pad_mask);
  if (nc < 0) { *overflow = 1; return 0; }
  if (nc == 0) return 0;
  // per-dof rows (the ones solve_qacc handles): friction loss, and the limit row of a joint outside its range
  TC af[SO_NJ], xl[SO_NJ], sDl[SO_NJ];
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) {
    af[j] = -K.fr_B[j] * qd[j];
    xl[j] = TC(0); sDl[j] = TC(0);
    if ((q[j] - K.lo[j]) - qc[j] < TC(0) || (K.hi[j] - q[j]) + qc[j] < TC(0)) {
      TC rm2, kap2;
      limit_row(K, j, M[midx(j, j)], q[j], qc[j], qd[j], xl[j], sDl[j], rm2, kap2);
    }
  }
  const T mu = P.mu;
  // gradient at x and generalised Hessian (into the store); the contact residuals (e, ty, tx) are kept for the line
  // search: rows of contact k are  e + ty, e - ty, e + tx, e - tx, each active iff < 0
  auto eval = [&](const T* x, T* g) {
#pragma unroll
    for (int k = 0; k < 21; k++) S.H(k) = (T)M[k];
#pragma unroll
    for (int i = 0; i < SO_NJ; i++) {
      T v = -(T)b[i];
#pragma unroll
      for (int j = 0; j < SO_NJ; j++) v += (T)(j <= i ? M[midx(i, j)] : M[midx(j, i)]) * x[j];
      const T fD = K.fr_D[i], fL = loss[i];
      const T t = fD * (x[i] - (T)af[i]);  // Huber friction row: force -clamp(D r, +-loss)
      if (t > -fL && t < fL) { v += t; S.H(midx(i, i)) += fD; }
      else v += t < T(0) ? -fL : fL;
      if (sDl[i] != TC(0) && (T)sDl[i] * (x[i] - (T)xl[i]) < T(0)) {  // limit row active
        const T Dl = sDl[i] < TC(0) ? -(T)sDl[i] : (T)sDl[i];
        v += Dl * (x[i] - (T)xl[i]);
        S.H(midx(i, i)) += Dl;
      }
      g[i] = v;
    }
    for (int k = 0; k < nc; k++) {
      T Jz[SO_NJ], Jy[SO_NJ], Jx[SO_NJ], jx = T(0), jy = T(0), jz = T(0);
#pragma unroll
      for (int j = 0; j < SO_NJ; j++) {
        Jz[j] = S.J(k, 0, j); Jy[j] = S.J(k, 1, j); Jx[j] = S.J(k, 2, j);
        jz += Jz[j] * x[j]; jy += Jy[j] * x[j]; jx += Jx[j] * x[j];
      }
      const T e = jz - (T)S.par(k, 0), ty = mu * jy + (T)S.par(k, 1), tx = mu * jx + (T)S.par(k, 2);
      S.res(k, 0) = e; S.res(k, 1) = ty; S.res(k, 2) = tx;
      const T r1 = e + ty, r2 = e - ty, r3 = e + tx, r4 = e - tx;
      const T a1 = r1 < T(0) ? T(1) : T(0), a2 = r2 < T(0) ? T(1) : T(0), a3 = r3 < T(0) ? T(1) : T(0), a4 = r4 < T(0) ? T(1) : T(0);
      const T nact = a1 + a2 + a3 + a4;
      if (nact == T(0)) continue;
      const T D = S.par(k, 3);
      const T gz = D * (a1 * r1 + a2 * r2 + a3 * r3 + a4 * r4), gy = D * mu * (a1 * r1 - a2 * r2), gx = D * mu * (a3 * r3 - a4 * r4);
      const T hzz = D * nact, hzy = D * mu * (a1 - a2), hyy = D * mu * mu * (a1 + a2), hzx = D * mu * (a3 - a4), hxx = D * mu * mu * (a3 + a4);
#pragma unroll
      for (int i = 0; i < SO_NJ; i++) {
        g[i] += gz * Jz[i] + gy * Jy[i] + gx * Jx[i];
        const T uz = hzz * Jz[i] + hzy * Jy[i] + hzx * Jx[i], uy = hzy * Jz[i] + hyy * Jy[i], ux = hzx * Jz[i] + hxx * Jx[i];
#pragma unroll
        for (int j = 0; j <= i; j++) S.H(midx(i, j)) += uz * Jz[j] + uy * Jy[j] + ux * Jx[j];
      }
    }
  };
  const T tol = exact_in ? T(1e-13) : T(1e-9);    // relative size of the last Newton step (fp32 inputs: no point below 1e-9)
  const T lstol = exact_in ? T(1e-12) : T(1e-8);  // |phi'(alpha)| / |phi'(0)| at which the line search stops
  const T atol = exact_in ? T(1e-14) : T(1e-10);  // ... or when its Newton iteration on alpha no longer moves
  T x[SO_NJ], g[SO_NJ];
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) x[j] = a[j];
  int evals = 0, nls = 0;
  bool ok = false;
  for (int it = 0; it < 30 && !ok; it++) {
    eval(x, g);
    evals++;
    T p[SO_NJ], ng[SO_NJ], d0 = T(0), pMp = T(0), ds = T(0), pmax = T(0), xmax = T(1);
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) ng[j] = -g[j];
    if (!chol_solve6<T>(S, ng, p)) { evals = -evals; break; }
#pragma unroll
    for (int i = 0; i < SO_NJ; i++) {
      T v = T(0), w = -(T)b[i];
#pragma unroll
      for (int j = 0; j < SO_NJ; j++) {
        const T mij = j <= i ? M[midx(i, j)] : M[midx(j, i)];
        v += mij * p[j]; w += mij * x[j];
      }
      pMp += p[i] * v;
      ds += w * p[i];  // smooth part of phi'(0)
      d0 += g[i] * p[i];
      const T ap = p[i] < T(0) ? -p[i] : p[i], ax = x[i] < T(0) ? -x[i] : x[i];
      pmax = ap > pmax ? ap : pmax; xmax = ax > xmax ? ax : xmax;
    }
    if (!(d0 < T(0))) { ok = true; break; }  // stationary to rounding
    for (int k = 0; k < nc; k++) {  // slopes of the contact residuals along p
      T jx = T(0), jy = T(0), jz = T(0);
#pragma unroll
      for (int j = 0; j < SO_NJ; j++) { jz += (T)S.J(k, 0, j) * p[j]; jy += (T)S.J(k, 1, j) * p[j]; jx += (T)S.J(k, 2, j) * p[j]; }
      S.res(k, 3) = jz; S.res(k, 4) = mu * jy; S.res(k, 5) = mu * jx;
    }
    // phi'(alpha) and phi''(alpha): phi' is piecewise linear and increasing, so Newton on it is exact within a piece.
    // `same` reports whether every row is in the state it had at alpha = 0.
    auto dphi = [&](T al, T& curv, bool& same) -> T {
      T d = ds + al * pMp, cv = pMp;
      same = true;
#pragma unroll
      for (int j = 0; j < SO_NJ; j++) {
        const T fD = K.fr_D[j], fL = loss[j];
        const T r0 = x[j] - (T)af[j], t0 = fD * r0, t = fD * (r0 + al * p[j]);
        const bool q0 = t0 > -fL && t0 < fL, q1 = t > -fL && t < fL;
        if (q1) { d += t * p[j]; cv += fD * p[j] * p[j]; }
        else d += (t < T(0) ? -fL : fL) * p[j];
        same = same && (q0 == q1) && (q1 || ((t0 < T(0)) == (t < T(0))));
        if (sDl[j] != TC(0)) {
          const T sd = sDl[j], l0 = x[j] - (T)xl[j], l1 = l0 + al * p[j];
          const bool b0 = sd * l0 < T(0), b1 = sd * l1 < T(0);
          if (b1) { const T Dl = sd < T(0) ? -sd : sd; d += Dl * l1 * p[j]; cv += Dl * p[j] * p[j]; }
          same = same && (b0 == b1);
        }
      }
      for (int k = 0; k < nc; k++) {
        const T e0 = S.res(k, 0), ty0 = S.res(k, 1), tx0 = S.res(k, 2), se = S.res(k, 3), sty = S.res(k, 4), stx = S.res(k, 5);
        const T e = e0 + al * se, ty = ty0 + al * sty, tx = tx0 + al * stx;
        const T r[4] = {e + ty, e - ty, e + tx, e - tx};
        const T r00[4] = {e0 + ty0, e0 - ty0, e0 + tx0, e0 - tx0};
        const T sl[4] = {se + sty, se - sty, se + stx, se - stx};
        const T D = S.par(k, 3);
#pragma unroll
        for (int m = 0; m < 4; m++) {
          if (r[m] < T(0)) { d += D * r[m] * sl[m]; cv += D * sl[m] * sl[m]; }
          same = same && ((r[m] < T(0)) == (r00[m] < T(0)));
        }
      }
      curv = cv;
      return d;
    };
    T lo = T(0), dlo = d0, hi = T(-1), dhi = T(0), alpha = T(1);
    bool same = false;
    for (int ls = 0; ls < 24; ls++) {
      T cv;
      const T d = dphi(alpha, cv, same);
      nls++;
      const T ad = d < T(0) ? -d : d;
      if (ad <= lstol * -d0) break;
      if (d < T(0)) { lo = alpha; dlo = d; } else { hi = alpha; dhi = d; }
      T an = alpha - d / cv;                                        // exact if no row switches in between
      const bool inside = an > lo && (hi < T(0) || an < hi);
      if (!inside) an = hi < T(0) ? T(2) * alpha : lo + (hi - lo) * (-dlo) / (dhi - dlo);
      const T da = an - alpha;
      alpha = an;
      if ((da < T(0) ? -da : da) <= atol * alpha) { dphi(alpha, cv, same); break; }
    }
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) x[j] += alpha * p[j];
    // the minimiser of the quadratic piece x started in, reached without any row switching state: done
    ok = same || alpha * pmax <= tol * xmax;
  }
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) a[j] = (TC)x[j];
  if (ls_evals) *ls_evals = nls;
  if (evals > 0 && !ok) evals = -evals;
  return evals;
}

template <typename T>
struct ContactIO {  // inputs / output of the out-of-line solve, copied once at the call site (keeps the hot path's arrays in registers)
  T s[SO_NJ], c[SO_NJ], q[SO_NJ], qc[SO_NJ], qd[SO_NJ], M[21], b[SO_NJ];
  T a[SO_NJ];       // in: warm start (previous qacc); out: qacc
};

// The solve with thread-local storage for up to SO_MAX_CON contacts, out of line: the host path, and on the device the
// fallback of a lane that found no slot in the shared-memory pool or more corners than a slot holds.
template <typename TC>
SO_HD int contact_solve_local(const DynC<TC>& C, const KinC<TC>& Kc, const PadC<TC>& P, const ConC<TC>& K, const TC* loss, ContactIO<TC>& io,
                              unsigned pad_mask, int* overflow, int* ls_evals) {
  ContactLocal<TC, SO_MAX_CON> S;
  int over = 0;
  const int st = contact_newton<TC>(C, Kc, P, K, loss, S, io.s, io.c, io.q, io.qc, io.qd, io.M, io.b, io.a, pad_mask, sizeof(TC) == 8, &over, ls_evals);
  if (over && overflow) *overflow = 1;
  return over ? -1 : st;
}
template <typename TC>
SO_NOINLINE int contact_solve(const DynC<TC>& C, const KinC<TC>& Kc, const PadC<TC>& P, const ConC<TC>& K, ContactIO<TC>& io,
                               unsigned pad_mask, int* overflow = nullptr, int* ls_evals = nullptr) {
  return contact_solve_local<TC>(C, Kc, P, K, K.fr_loss, io, pad_mask, overflow, ls_evals);
}
// The same with the env's own friction loss (so100_set_param_ranges): a separate function, so that the call of the
// model-constant solve above keeps its signature.  loss[] is copied to the callee's frame (a cold path).
template <typename TC>
SO_NOINLINE int contact_solve_loss(const DynC<TC>& C, const KinC<TC>& Kc, const PadC<TC>& P, const ConC<TC>& K, const TC* loss, ContactIO<TC>& io,
                                   unsigned pad_mask, int* overflow) {
  return contact_solve_local<TC>(C, Kc, P, K, loss, io, pad_mask, overflow, nullptr);
}

// ---------------------------------------------------------------------------------------------------------------
// The contact solve spread over a GROUP of lanes.  contact_newton above is one thread's serial chain of ~30 k
// instructions per solve, sixteen of them in a row per env step, with one or two such warps per SM: nothing hides its
// latency (DESIGN.md "Arm-floor contact").  Here the same Newton iteration runs on kCoopLanes lanes per env: the lanes
// split the contacts (residuals, activity, slopes, line-search rows), the 21 Hessian entries, the 6 gradient entries and
// the rows of M p / M x; one lane does the 6x6 Cholesky.  Lanes only talk through the env's SLOT (shared memory on the
// device), in phases separated by a group barrier, and every phase is a function of (slot, lane): the device runs the
// lanes of a phase in parallel, the host (tests, so100_host_substeps) runs them one after the other and gets
// bit-identical numbers.
//
// A slot is self-contained (the solve reads nothing else): it is filled by the env's own thread (coop_fill: accurate
// kinematics, contact enumeration, Jacobians, row parameters, the substep's M, b, per-dof rows and warm start).
constexpr int kCoopLanes = 8;
constexpr int kCoopCon = 8;  // contacts per slot (== kCoopLanes: one lane per contact)

struct CoopSlot {  // slot-major storage: consecutive words of one slot are consecutive in memory (the lanes of a group read different words)
  float* f;
  double* d;
  // float words
  static constexpr int kJ = 0, kPar = kJ + kCoopCon * 18, kM = kPar + kCoopCon * 4, kB = kM + 21, kAf = kB + 6, kXl = kAf + 6, kSDl = kXl + 6,
                       kX0 = kSDl + 6, kFrD = kX0 + 6, kFrL = kFrD + 6, kMu = kFrL + 6, kNc = kMu + 1, kAct = kNc + 1, kFloats = kAct + kCoopCon;
  // double words
  static constexpr int kX = 0, kG = 6, kP = 12, kH = 18, kRes = 39, kDiag = kRes + kCoopCon * 6, kRed = kDiag + 6, kSc = kRed + kCoopLanes * 2,
                       kDoubles = kSc + 12;
  static_assert(kFloats % 2 == 1 && kDoubles % 2 == 1, "odd slot sizes spread the slots of a warp over the shared-memory banks");
  SO_HD float& F(int w) const { return f[w]; }
  SO_HD double& D(int w) const { return d[w]; }
  SO_HD float& J(int c, int axis, int j) const { return f[kJ + (c * 3 + axis) * 6 + j]; }
  SO_HD float& par(int c, int m) const { return f[kPar + c * 4 + m]; }
  SO_HD double& res(int c, int m) const { return d[kRes + c * 6 + m]; }
  SO_HD double& sc(int k) const { return d[kSc + k]; }
};
// sc[10]: state of the solve (0 running, 1 converged, 2 failed: Hessian not positive definite / iteration cap)

// the store interface of contact_setup over a slot
struct CoopStore {
  static constexpr int kMaxCon = kCoopCon;
  CoopSlot s;
  SO_HD float& J(int c, int axis, int j) { return s.J(c, axis, j); }
  SO_HD float& par(int c, int m) { return s.par(c, m); }
};

// Fill a slot (the env's own thread).  Returns the number of contacts: 0 = the accurate kinematics found no corner below
// the floor (no solve), -1 = more than kCoopCon corners (the caller takes the out-of-line serial solve).
SO_HD int coop_fill(const DynC<float>& C, const KinC<float>& Kc, const PadC<float>& P, const ConC<float>& K, const float* loss, const CoopSlot& S, const float* s,
                    const float* c, const float* q, const float* qc, const float* qd, const float* M, const float* b, const float* a0,
                    unsigned pad_mask) {
  CoopStore st{S};
  const int nc = contact_setup<float>(C, Kc, P, st, s, c, qd, pad_mask);
  S.F(CoopSlot::kNc) = (float)(nc > 0 ? nc : 0);
  if (nc <= 0) return nc;
#pragma unroll
  for (int k = 0; k < 21; k++) S.F(CoopSlot::kM + k) = M[k];
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) {
    float xl = 0.0f, sDl = 0.0f;
    if ((q[j] - K.lo[j]) - qc[j] < 0.0f || (K.hi[j] - q[j]) + qc[j] < 0.0f) {
      float rm2, kap2;
      limit_row(K, j, M[midx(j, j)], q[j], qc[j], qd[j], xl, sDl, rm2, kap2);
    }
    S.F(CoopSlot::kB + j) = b[j]; S.F(CoopSlot::kAf + j) = -K.fr_B[j] * qd[j]; S.F(CoopSlot::kXl + j) = xl; S.F(CoopSlot::kSDl + j) = sDl;
    S.F(CoopSlot::kX0 + j) = a0[j]; S.F(CoopSlot::kFrD + j) = K.fr_D[j]; S.F(CoopSlot::kFrL + j) = loss[j];
  }
  S.F(CoopSlot::kMu) = P.mu;
  return nc;
}

// ---- phases.  `lane` in [0, kCoopLanes).  P1-P3 and P7 exchange through the slot (a group barrier after each); P4 and
// the line search keep their rows in the lane's registers (CoopLane) and exchange through butterfly reductions over the
// group's lanes (coop_sum / coop_max / coop_all: shuffles on the device, loops on the host - the same additions in the
// same order, and a + b == b + a, so every lane ends with the same bits).
//
// P1: lane = contact: residuals at x, the rows' activity and the contact's gradient coefficients;
//     lane = dof: x (first iteration: the warm start), smooth + per-dof part of the gradient, per-dof curvature
SO_HD void coop_p1(const CoopSlot& S, int lane, bool first) {
  const int nc = (int)S.F(CoopSlot::kNc);
  const double mu = (double)S.F(CoopSlot::kMu);
  double x[SO_NJ];
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) x[j] = first ? (double)S.F(CoopSlot::kX0 + j) : S.D(CoopSlot::kX + j);
  if (lane < nc) {
    double jz = 0.0, jy = 0.0, jx = 0.0;
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) { jz += (double)S.J(lane, 0, j) * x[j]; jy += (double)S.J(lane, 1, j) * x[j]; jx += (double)S.J(lane, 2, j) * x[j]; }
    const double e = jz - (double)S.par(lane, 0), ty = mu * jy + (double)S.par(lane, 1), tx = mu * jx + (double)S.par(lane, 2), D = (double)S.par(lane, 3);
    const double r1 = e + ty, r2 = e - ty, r3 = e + tx, r4 = e - tx;
    const double a1 = r1 < 0.0 ? 1.0 : 0.0, a2 = r2 < 0.0 ? 1.0 : 0.0, a3 = r3 < 0.0 ? 1.0 : 0.0, a4 = r4 < 0.0 ? 1.0 : 0.0;
    S.res(lane, 0) = e; S.res(lane, 1) = ty; S.res(lane, 2) = tx;
    S.res(lane, 3) = D * (a1 * r1 + a2 * r2 + a3 * r3 + a4 * r4); S.res(lane, 4) = D * mu * (a1 * r1 - a2 * r2); S.res(lane, 5) = D * mu * (a3 * r3 - a4 * r4);
    S.F(CoopSlot::kAct + lane) = (float)((r1 < 0.0 ? 1 : 0) | (r2 < 0.0 ? 2 : 0) | (r3 < 0.0 ? 4 : 0) | (r4 < 0.0 ? 8 : 0));
  }
  if (lane < SO_NJ) {
    const int i = lane;
    double v = -(double)S.F(CoopSlot::kB + i);
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) v += (double)S.F(CoopSlot::kM + (j <= i ? midx(i, j) : midx(j, i))) * x[j];
    const double xi = first ? (double)S.F(CoopSlot::kX0 + i) : S.D(CoopSlot::kX + i);
    const double fD = (double)S.F(CoopSlot::kFrD + i), fL = (double)S.F(CoopSlot::kFrL + i);
    const double t = fD * (xi - (double)S.F(CoopSlot::kAf + i));  // Huber friction row: force -clamp(D r, +-loss)
    double cv = 0.0;
    if (t > -fL && t < fL) { v += t; cv = fD; }
    else v += t < 0.0 ? -fL : fL;
    const double sd = (double)S.F(CoopSlot::kSDl + i), xl = (double)S.F(CoopSlot::kXl + i);
    if (sd != 0.0 && sd * (xi - xl) < 0.0) { const double Dl = sd < 0.0 ? -sd : sd; v += Dl * (xi - xl); cv += Dl; }  // limit row active
    S.D(CoopSlot::kG + i) = v;
    S.D(CoopSlot::kDiag + i) = cv;
    if (first) S.D(CoopSlot::kX + i) = xi;
  }
  if (first && lane == kCoopLanes - 1) S.sc(10) = 0.0;
}
// P2: the generalised Hessian's 21 entries over the lanes, and the contacts' part of the gradient (lane = dof)
SO_HD void coop_p2(const CoopSlot& S, int lane) {
  const int nc = (int)S.F(CoopSlot::kNc);
  const double mu = (double)S.F(CoopSlot::kMu);
  int ei[3], ej[3];
  double h[3];
#pragma unroll
  for (int m = 0; m < 3; m++) {
    const int k = lane + m * kCoopLanes;  // entry k = midx(i, j); k >= 21: this lane has no m-th entry
    int i = 0;
#pragma unroll
    for (int r = 1; r < SO_NJ; r++) i += (k >= midx(r, 0)) ? 1 : 0;
    ei[m] = i; ej[m] = k < 21 ? k - midx(i, 0) : 0;
    h[m] = k < 21 ? (double)S.F(CoopSlot::kM + k) + (i == ej[m] ? S.D(CoopSlot::kDiag + i) : 0.0) : 0.0;
  }
  double g = lane < SO_NJ ? S.D(CoopSlot::kG + lane) : 0.0;
  const int gl = lane < SO_NJ ? lane : 0;
  for (int c = 0; c < nc; c++) {
    const int act = (int)S.F(CoopSlot::kAct + c);
    if (act == 0) continue;
    const double D = (double)S.par(c, 3), Dm = D * mu, Dmm = Dm * mu;
    const double a1 = (act & 1) ? 1.0 : 0.0, a2 = (act & 2) ? 1.0 : 0.0, a3 = (act & 4) ? 1.0 : 0.0, a4 = (act & 8) ? 1.0 : 0.0;
    const double hzz = D * (a1 + a2 + a3 + a4), hzy = Dm * (a1 - a2), hyy = Dmm * (a1 + a2), hzx = Dm * (a3 - a4), hxx = Dmm * (a3 + a4);
#pragma unroll
    for (int m = 0; m < 3; m++) {
      const double zi = S.J(c, 0, ei[m]), yi = S.J(c, 1, ei[m]), xi = S.J(c, 2, ei[m]), zj = S.J(c, 0, ej[m]), yj = S.J(c, 1, ej[m]), xj = S.J(c, 2, ej[m]);
      h[m] += (hzz * zi + hzy * yi + hzx * xi) * zj + (hzy * zi + hyy * yi) * yj + (hzx * zi + hxx * xi) * xj;
    }
    g += S.res(c, 3) * (double)S.J(c, 0, gl) + S.res(c, 4) * (double)S.J(c, 1, gl) + S.res(c, 5) * (double)S.J(c, 2, gl);
  }
#pragma unroll
  for (int m = 0; m < 3; m++)
    if (lane + m * kCoopLanes < 21) S.D(CoopSlot::kH + lane + m * kCoopLanes) = h[m];
  if (lane < SO_NJ) S.D(CoopSlot::kG + lane) = g;
}
// 1/sqrt(x) to double rounding from the float unit's estimate and two Newton steps (a libm sqrt + divide is ~120 instructions)
SO_HD double coop_rsqrt(double x) {
  double y = (double)so_rsqrt((float)x);
  const double hx = 0.5 * x;
  y = y * (1.5 - hx * y * y);
  y = y * (1.5 - hx * y * y);
  return y;
}
// P3 (lane 0): Cholesky and the Newton direction p = -H^-1 g, written out as straight-line code on named scalars (generated:
// a loop nest over a local array is not reliably unrolled here, and an array in local memory puts an L1 round trip behind
// every step of the dependent chain)
SO_HD void coop_p3(const CoopSlot& S, int lane) {
  if (lane != 0) return;
  double h0 = S.D(CoopSlot::kH + 0);
  double h1 = S.D(CoopSlot::kH + 1);
  double h2 = S.D(CoopSlot::kH + 2);
  double h3 = S.D(CoopSlot::kH + 3);
  double h4 = S.D(CoopSlot::kH + 4);
  double h5 = S.D(CoopSlot::kH + 5);
  double h6 = S.D(CoopSlot::kH + 6);
  double h7 = S.D(CoopSlot::kH + 7);
  double h8 = S.D(CoopSlot::kH + 8);
  double h9 = S.D(CoopSlot::kH + 9);
  double h10 = S.D(CoopSlot::kH + 10);
  double h11 = S.D(CoopSlot::kH + 11);
  double h12 = S.D(CoopSlot::kH + 12);
  double h13 = S.D(CoopSlot::kH + 13);
  double h14 = S.D(CoopSlot::kH + 14);
  double h15 = S.D(CoopSlot::kH + 15);
  double h16 = S.D(CoopSlot::kH + 16);
  double h17 = S.D(CoopSlot::kH + 17);
  double h18 = S.D(CoopSlot::kH + 18);
  double h19 = S.D(CoopSlot::kH + 19);
  double h20 = S.D(CoopSlot::kH + 20);
  bool ok = true;
  ok = ok && h0 > 0.0;
  h0 = coop_rsqrt(h0 > 0.0 ? h0 : 1.0);  // the diagonal holds 1 / L_00
  h1 *= h0;
  h3 *= h0;
  h6 *= h0;
  h10 *= h0;
  h15 *= h0;
  h2 -= h1 * h1;
  ok = ok && h2 > 0.0;
  h2 = coop_rsqrt(h2 > 0.0 ? h2 : 1.0);  // the diagonal holds 1 / L_11
  h4 -= h3 * h1;
  h4 *= h2;
  h7 -= h6 * h1;
  h7 *= h2;
  h11 -= h10 * h1;
  h11 *= h2;
  h16 -= h15 * h1;
  h16 *= h2;
  h5 -= h3 * h3;
  h5 -= h4 * h4;
  ok = ok && h5 > 0.0;
  h5 = coop_rsqrt(h5 > 0.0 ? h5 : 1.0);  // the diagonal holds 1 / L_22
  h8 -= h6 * h3;
  h8 -= h7 * h4;
  h8 *= h5;
  h12 -= h10 * h3;
  h12 -= h11 * h4;
  h12 *= h5;
  h17 -= h15 * h3;
  h17 -= h16 * h4;
  h17 *= h5;
  h9 -= h6 * h6;
  h9 -= h7 * h7;
  h9 -= h8 * h8;
  ok = ok && h9 > 0.0;
  h9 = coop_rsqrt(h9 > 0.0 ? h9 : 1.0);  // the diagonal holds 1 / L_33
  h13 -= h10 * h6;
  h13 -= h11 * h7;
  h13 -= h12 * h8;
  h13 *= h9;
  h18 -= h15 * h6;
  h18 -= h16 * h7;
  h18 -= h17 * h8;
  h18 *= h9;
  h14 -= h10 * h10;
  h14 -= h11 * h11;
  h14 -= h12 * h12;
  h14 -= h13 * h13;
  ok = ok && h14 > 0.0;
  h14 = coop_rsqrt(h14 > 0.0 ? h14 : 1.0);  // the diagonal holds 1 / L_44
  h19 -= h15 * h10;
  h19 -= h16 * h11;
  h19 -= h17 * h12;
  h19 -= h18 * h13;
  h19 *= h14;
  h20 -= h15 * h15;
  h20 -= h16 * h16;
  h20 -= h17 * h17;
  h20 -= h18 * h18;
  h20 -= h19 * h19;
  ok = ok && h20 > 0.0;
  h20 = coop_rsqrt(h20 > 0.0 ? h20 : 1.0);  // the diagonal holds 1 / L_55
  if (!ok) { S.sc(10) = 2.0; return; }
  double y0 = -S.D(CoopSlot::kG + 0);
  y0 *= h0;
  double y1 = -S.D(CoopSlot::kG + 1);
  y1 -= h1 * y0;
  y1 *= h2;
  double y2 = -S.D(CoopSlot::kG + 2);
  y2 -= h3 * y0;
  y2 -= h4 * y1;
  y2 *= h5;
  double y3 = -S.D(CoopSlot::kG + 3);
  y3 -= h6 * y0;
  y3 -= h7 * y1;
  y3 -= h8 * y2;
  y3 *= h9;
  double y4 = -S.D(CoopSlot::kG + 4);
  y4 -= h10 * y0;
  y4 -= h11 * y1;
  y4 -= h12 * y2;
  y4 -= h13 * y3;
  y4 *= h14;
  double y5 = -S.D(CoopSlot::kG + 5);
  y5 -= h15 * y0;
  y5 -= h16 * y1;
  y5 -= h17 * y2;
  y5 -= h18 * y3;
  y5 -= h19 * y4;
  y5 *= h20;
  double p5 = y5;
  p5 *= h20;
  double p4 = y4;
  p4 -= h19 * p5;
  p4 *= h14;
  double p3 = y3;
  p3 -= h13 * p4;
  p3 -= h18 * p5;
  p3 *= h9;
  double p2 = y2;
  p2 -= h8 * p3;
  p2 -= h12 * p4;
  p2 -= h17 * p5;
  p2 *= h5;
  double p1 = y1;
  p1 -= h4 * p2;
  p1 -= h7 * p3;
  p1 -= h11 * p4;
  p1 -= h16 * p5;
  p1 *= h2;
  double p0 = y0;
  p0 -= h1 * p1;
  p0 -= h3 * p2;
  p0 -= h6 * p3;
  p0 -= h10 * p4;
  p0 -= h15 * p5;
  p0 *= h0;
  S.D(CoopSlot::kP + 0) = p0;
  S.D(CoopSlot::kP + 1) = p1;
  S.D(CoopSlot::kP + 2) = p2;
  S.D(CoopSlot::kP + 3) = p3;
  S.D(CoopSlot::kP + 4) = p4;
  S.D(CoopSlot::kP + 5) = p5;
}

// one lane's registers from P4 to P7: its rows of the line search (dof `lane`: friction + limit; contact `lane`: four
// pyramid rows) and the scalars every lane of the group holds identically
struct CoopLane {
  double fD, fL, r0, pj, sdl, l0;         // dof rows (fD = 0, sdl = 0: none)
  double e0, ty0, tx0, se, sty, stx, D;   // contact rows (D = 0: none)
  double d0, pMp, ds, pmax, xmax;         // P4: this lane's terms; after the reduction: g.p, p'Mp, (Mx - b).p, max |p|, max(1, |x|)
  double alpha, lo, dlo, hi, dhi;         // line-search bracket
  int ls;                                 // 0 searching, 1 accepted and no row switched along the step, 2 accepted
};
// P4: slopes of this lane's contact residuals along p, its dof rows, and the i-th terms of g.p, p'Mp and (Mx - b).p
SO_HD void coop_p4(const CoopSlot& S, int lane, CoopLane& L) {
  const int nc = (int)S.F(CoopSlot::kNc);
  const double mu = (double)S.F(CoopSlot::kMu);
  double p[SO_NJ];
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) p[j] = S.D(CoopSlot::kP + j);
  L.e0 = L.ty0 = L.tx0 = L.se = L.sty = L.stx = L.D = 0.0;
  if (lane < nc) {
    double jz = 0.0, jy = 0.0, jx = 0.0;
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) { jz += (double)S.J(lane, 0, j) * p[j]; jy += (double)S.J(lane, 1, j) * p[j]; jx += (double)S.J(lane, 2, j) * p[j]; }
    L.se = jz; L.sty = mu * jy; L.stx = mu * jx;
    L.e0 = S.res(lane, 0); L.ty0 = S.res(lane, 1); L.tx0 = S.res(lane, 2); L.D = (double)S.par(lane, 3);
  }
  L.fD = L.fL = L.r0 = L.pj = L.sdl = L.l0 = 0.0;
  L.d0 = L.pMp = L.ds = L.pmax = L.xmax = 0.0;
  if (lane < SO_NJ) {
    const int i = lane;
    double v = 0.0, w = -(double)S.F(CoopSlot::kB + i);
    const double pi = S.D(CoopSlot::kP + i), xi = S.D(CoopSlot::kX + i);
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) {
      const double mij = (double)S.F(CoopSlot::kM + (j <= i ? midx(i, j) : midx(j, i)));
      v += mij * p[j]; w += mij * S.D(CoopSlot::kX + j);
    }
    L.d0 = S.D(CoopSlot::kG + i) * pi; L.pMp = pi * v; L.ds = w * pi;
    L.pmax = pi < 0.0 ? -pi : pi; L.xmax = xi < 0.0 ? -xi : xi;
    L.fD = (double)S.F(CoopSlot::kFrD + i); L.fL = (double)S.F(CoopSlot::kFrL + i); L.r0 = xi - (double)S.F(CoopSlot::kAf + i); L.pj = pi;
    L.sdl = (double)S.F(CoopSlot::kSDl + i); L.l0 = xi - (double)S.F(CoopSlot::kXl + i);
  }
}
// after the reduction of P4's terms: start the line search at alpha = 1.  Returns false if x is stationary to rounding.
SO_HD bool coop_ls_begin(CoopLane& L) {
  L.xmax = L.xmax > 1.0 ? L.xmax : 1.0;
  L.alpha = 1.0; L.lo = 0.0; L.dlo = L.d0; L.hi = -1.0; L.dhi = 0.0; L.ls = 0;
  return L.d0 < 0.0;
}
// this lane's share of phi'(alpha), phi''(alpha) and of "every row is in the state it had at alpha = 0"
SO_HD void coop_ls_eval(const CoopLane& L, double& d, double& cv, bool& same) {
  const double al = L.alpha;
  d = 0.0; cv = 0.0; same = true;
  {
    const double t0 = L.fD * L.r0, t = L.fD * (L.r0 + al * L.pj);
    const bool q0 = t0 > -L.fL && t0 < L.fL, q1 = t > -L.fL && t < L.fL;
    if (q1) { d += t * L.pj; cv += L.fD * L.pj * L.pj; }
    else d += (t < 0.0 ? -L.fL : L.fL) * L.pj;
    same = same && (q0 == q1) && (q1 || ((t0 < 0.0) == (t < 0.0)));
    if (L.sdl != 0.0) {
      const double l1 = L.l0 + al * L.pj;
      const bool b0 = L.sdl * L.l0 < 0.0, b1 = L.sdl * l1 < 0.0;
      if (b1) { const double Dl = L.sdl < 0.0 ? -L.sdl : L.sdl; d += Dl * l1 * L.pj; cv += Dl * L.pj * L.pj; }
      same = same && (b0 == b1);
    }
  }
  {
    const double e = L.e0 + al * L.se, ty = L.ty0 + al * L.sty, tx = L.tx0 + al * L.stx;
    const double r[4] = {e + ty, e - ty, e + tx, e - tx}, r00[4] = {L.e0 + L.ty0, L.e0 - L.ty0, L.e0 + L.tx0, L.e0 - L.tx0},
                 sl[4] = {L.se + L.sty, L.se - L.sty, L.se + L.stx, L.se - L.stx};
#pragma unroll
    for (int m = 0; m < 4; m++) {
      if (r[m] < 0.0) { d += L.D * r[m] * sl[m]; cv += L.D * sl[m] * sl[m]; }
      same = same && ((r[m] < 0.0) == (r00[m] < 0.0));
    }
  }
}
// (every lane, identically) with the reduced phi', phi'' and flag: accept alpha, or the next alpha of the safeguarded
// Newton iteration on phi' (piecewise linear and increasing: Newton is exact within a piece)
SO_HD void coop_ls_decide(CoopLane& L, double dsum, double cvsum, bool same, double lstol, double atol_, int ls_iter) {
  const double alpha = L.alpha, d = L.ds + alpha * L.pMp + dsum, cv = L.pMp + cvsum;
  const double ad = d < 0.0 ? -d : d;
  bool done = ad <= lstol * -L.d0 || ls_iter >= 23;
  if (!done) {
    if (d < 0.0) { L.lo = alpha; L.dlo = d; } else { L.hi = alpha; L.dhi = d; }
    double an = alpha - d / cv;  // exact if no row switches in between
    const bool inside = an > L.lo && (L.hi < 0.0 || an < L.hi);
    if (!inside) an = L.hi < 0.0 ? 2.0 * alpha : L.lo + (L.hi - L.lo) * (-L.dlo) / (L.dhi - L.dlo);
    const double da = an - alpha;
    L.alpha = an;
    if ((da < 0.0 ? -da : da) <= atol_ * an) { done = true; same = false; }  // alpha converged to rounding: the flag belongs to the previous point
  }
  if (done) L.ls = same ? 1 : 2;
}
// P7: take the step (lane = dof).  Returns (every lane, identically) whether the solve is finished: the minimiser of the
// quadratic piece x started in was reached without any row switching state, or the step is below the tolerance.
SO_HD bool coop_p7(const CoopSlot& S, int lane, const CoopLane& L, double tol) {
  if (lane < SO_NJ) S.D(CoopSlot::kX + lane) += L.alpha * L.pj;
  return L.ls == 1 || L.alpha * L.pmax <= tol * L.xmax;
}

struct CoopTol { double tol, lstol, atol_; };
SO_HD CoopTol coop_tolerances() { return CoopTol{1e-9, 1e-8, 1e-10}; }  // fp32 inputs (contact_newton's exact_in = false)
constexpr int kCoopMaxIter = 30, kCoopMaxLs = 24;

// host: the phases with the lanes in sequence, the reductions as the device's butterflies.  Returns the number of
// gradient/Hessian evaluations, negated if the solve did not converge (iteration cap, indefinite Hessian).
inline void coop_host_sum(double* v) {
  for (int k = 1; k < kCoopLanes; k <<= 1) { double t[kCoopLanes]; for (int l = 0; l < kCoopLanes; l++) t[l] = v[l] + v[l ^ k]; for (int l = 0; l < kCoopLanes; l++) v[l] = t[l]; }
}
inline void coop_host_max(double* v) {
  for (int k = 1; k < kCoopLanes; k <<= 1) { double t[kCoopLanes]; for (int l = 0; l < kCoopLanes; l++) t[l] = v[l] > v[l ^ k] ? v[l] : v[l ^ k]; for (int l = 0; l < kCoopLanes; l++) v[l] = t[l]; }
}
inline int coop_solve_host(const CoopSlot& S, int* ls_evals = nullptr) {
  CoopTol T = coop_tolerances();
  static const double lstol_env = getenv("SO100_COOP_LSTOL") ? atof(getenv("SO100_COOP_LSTOL")) : 0.0;  // experiments
  if (lstol_env > 0.0) T.lstol = lstol_env;
  CoopLane L[kCoopLanes];
  int evals = 0, nls = 0;
  bool conv = false;
  for (int it = 0; it < kCoopMaxIter && !conv; it++) {
    for (int l = 0; l < kCoopLanes; l++) coop_p1(S, l, it == 0);
    for (int l = 0; l < kCoopLanes; l++) coop_p2(S, l);
    for (int l = 0; l < kCoopLanes; l++) coop_p3(S, l);
    evals++;
    if (S.sc(10) != 0.0) break;
    for (int l = 0; l < kCoopLanes; l++) coop_p4(S, l, L[l]);
    {
      double a[kCoopLanes], b[kCoopLanes], c[kCoopLanes], d[kCoopLanes], e[kCoopLanes];
      for (int l = 0; l < kCoopLanes; l++) { a[l] = L[l].d0; b[l] = L[l].pMp; c[l] = L[l].ds; d[l] = L[l].pmax; e[l] = L[l].xmax; }
      coop_host_sum(a); coop_host_sum(b); coop_host_sum(c); coop_host_max(d); coop_host_max(e);
      for (int l = 0; l < kCoopLanes; l++) { L[l].d0 = a[l]; L[l].pMp = b[l]; L[l].ds = c[l]; L[l].pmax = d[l]; L[l].xmax = e[l]; }
    }
    bool descent = true;
    for (int l = 0; l < kCoopLanes; l++) descent = coop_ls_begin(L[l]);
    if (!descent) { conv = true; break; }  // stationary to rounding
    for (int ls = 0; ls < kCoopMaxLs && L[0].ls == 0; ls++) {
      double d[kCoopLanes], cv[kCoopLanes];
      bool same = true;
      for (int l = 0; l < kCoopLanes; l++) { bool s1; coop_ls_eval(L[l], d[l], cv[l], s1); same = same && s1; }
      coop_host_sum(d); coop_host_sum(cv);
      for (int l = 0; l < kCoopLanes; l++) coop_ls_decide(L[l], d[l], cv[l], same, T.lstol, T.atol_, ls);
      nls++;
    }
    for (int l = 0; l < kCoopLanes; l++) conv = coop_p7(S, l, L[l], T.tol);
  }
  if (S.sc(10) == 0.0) S.sc(10) = conv ? 1.0 : 2.0;
  if (ls_evals) *ls_evals = nls;
  return S.sc(10) == 1.0 ? evals : -evals;
}

#ifdef __CUDACC__
// device: one WARP runs the solves of four slots in lockstep, kCoopLanes lanes each (sf == nullptr: this group has no
// slot).  All control flow is warp-uniform - a group that is finished, or waiting for the others' line searches, skips the
// phase bodies - so the four solves cost the longest of them, not their sum (groups that diverge are serialised by the
// hardware).  Out of line: the solve's registers are its own (the caller is the step kernel at its 128-register cap).
__device__ __forceinline__ double coop_shfl_xor(double v, int k) { return __shfl_xor_sync(0xffffffffu, v, k); }
__device__ __forceinline__ double coop_sum(double v) {
#pragma unroll
  for (int k = 1; k < kCoopLanes; k <<= 1) v += coop_shfl_xor(v, k);
  return v;
}
__device__ __forceinline__ double coop_max(double v) {
#pragma unroll
  for (int k = 1; k < kCoopLanes; k <<= 1) { const double o = coop_shfl_xor(v, k); v = v > o ? v : o; }
  return v;
}
__device__ __noinline__ void coop_solve_warp(float* sf, double* sd, int lane, int gshift) {
  const CoopSlot S{sf, sd};
  const CoopTol T = coop_tolerances();
  bool active = sf != nullptr, conv = false;
  CoopLane L;
  for (int it = 0; it < kCoopMaxIter; it++) {
    if (!__any_sync(0xffffffffu, active)) break;
    if (active) coop_p1(S, lane, it == 0);
    __syncwarp();
    if (active) coop_p2(S, lane);
    __syncwarp();
    if (active) coop_p3(S, lane);
    __syncwarp();
    if (active && S.sc(10) != 0.0) active = false;  // Hessian not positive definite
    if (active) coop_p4(S, lane, L);
    else { L.d0 = L.pMp = L.ds = L.pmax = L.xmax = 0.0; L.fD = L.fL = L.r0 = L.pj = L.sdl = L.l0 = 0.0; L.e0 = L.ty0 = L.tx0 = L.se = L.sty = L.stx = L.D = 0.0; }
    L.d0 = coop_sum(L.d0); L.pMp = coop_sum(L.pMp); L.ds = coop_sum(L.ds); L.pmax = coop_max(L.pmax); L.xmax = coop_max(L.xmax);
    const bool descent = coop_ls_begin(L);
    if (active && !descent) { active = false; conv = true; }  // stationary to rounding
    if (!active) L.ls = 2;
    for (int ls = 0; ls < kCoopMaxLs; ls++) {
      if (!__any_sync(0xffffffffu, L.ls == 0)) break;
      double d, cv;
      bool same;
      coop_ls_eval(L, d, cv, same);
      d = coop_sum(d); cv = coop_sum(cv);
      same = ((__ballot_sync(0xffffffffu, same) >> gshift) & 0xffu) == 0xffu;
      if (L.ls == 0) coop_ls_decide(L, d, cv, same, T.lstol, T.atol_, ls);
    }
    if (active) {
      conv = coop_p7(S, lane, L, T.tol);
      if (conv) active = false;
    }
    __syncwarp();
  }
  if (sf != nullptr && lane == 0 && S.sc(10) == 0.0) S.sc(10) = conv ? 1.0 : 2.0;
}
#endif
