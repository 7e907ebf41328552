// so100_b200.cu — libso100_b200.so: C ABI (include/so100_b200.h) + sm_100a kernels of the batched so100 env step.
//
// One thread owns one environment for the whole env step: it loads the env's structure-of-arrays state (coalesced),
// runs the task's pre-step logic, 16 physics substeps entirely in registers (so100_dyn.cuh), the observation /
// reward / termination / TimeLimit logic and the in-kernel auto-reset, and stores the state back.  Observations and
// actions cross the ABI as row-major [N, dim] fp32; they are staged through shared memory so that global accesses
// stay coalesced.  No tensor cores: nothing here is a large dense contraction (6x6 systems per env).
//
// Reference behaviour replaced (paths relative to the reference repo, src/so100_mujoco_rl/):
//   envs/env01_v1.py:15-63, envs/env02_v1.py:18-81, envs/env03_v1.py:35-215, envs/env05_v1.py:32-75,
//   envs/env_base_01.py:107-270, envs/env_base_02.py:85-127, __init__.py:5-45, and mujoco.mj_step (3rd party).
#include <cuda_runtime.h>
#include <limits.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <cmath>
#include <new>
#include <string>

#include "../../include/so100_b200.h"
#include "../../include/so100_ppo.h"
#include "so100_dyn.cuh"
#define SO100_GEN_N SO100_N_DYN_CONSTANTS
#include "so100_dyn_gen.cuh"  // model-specialised straight-line dynamics (tools/gen_so100_dyn.py)

// ------------------------------------------------------------------------------------------------ error plumbing
static thread_local std::string g_err;
static int fail(int code, const std::string& msg) { g_err = msg; return code; }
#define CU(call)                                                                                      \
  do {                                                                                                \
    cudaError_t e_ = (call);                                                                          \
    if (e_ != cudaSuccess)                                                                            \
      return fail(SO100_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_));                \
  } while (0)

// ------------------------------------------------------------------------------------------------ device constants
// Launch shape (tunable at build time for experiments; defaults are the measured best, see profiles/).
#ifndef SO100_BLOCK
#define SO100_BLOCK 256
#endif
#ifndef SO100_MINBLOCKS
#define SO100_MINBLOCKS 2
#endif
#ifndef SO100_SYNC
#define SO100_SYNC 1   // __syncthreads() per substep: keeps a CTA's warps on the same stretch of straight-line code (i-cache)
#endif
constexpr int kBlock = SO100_BLOCK;  // threads per CTA, one env each
#ifndef SO100_SWEEPS_FIRST
#define SO100_SWEEPS_FIRST 5  // Gauss-Seidel sweeps scheduled on the first substep of an env step (ctrl has just jumped) ...
#define SO100_SWEEPS_REST 3   // ... and on the other 15 (warm start within a few %); more follow per lane while a sweep still moves qacc by > 1e-3
#endif
#define SO100_TOUCH_MARGIN 2e-6f   // broad-phase margin [m] over the MUFU sin/cos error (see physics<>)
constexpr int kMaxStart = SO100_MAX_START;
constexpr int kSnap = 12, kAux = 24, kCnt = 4;
enum { F_EVER_STEPPED = 1, F_HAS_LAST_BLOCK = 2, F_ANGVEL_VALID = 4, F_CENTRE_VALID = 8,
       F_TOUCH = 16 };  // F_TOUCH: a jaw pad touched the floor in the env's last substep (scheduling hint only, no effect on results)
enum { STREAM_RESET = 0, STREAM_TASK = 1, STREAM_NOISE = 2, STREAM_API_RESET = 3, STREAM_RESET_NOISE = 4,
       STREAM_PARAM_RESET = 8, STREAM_PARAM_API_RESET = 16,  // per-env parameters: streams 8..13 (auto-reset) and 16..21 (so100_reset)
       STREAM_LAT_RESET = 14, STREAM_LAT_API_RESET = 22,     // actuator latency: auto-reset, so100_reset
       STREAM_OBS_NOISE = 24, STREAM_OBS_RESET_NOISE = 26, STREAM_OBS_API_NOISE = 28 };  // joint-angle noise, 2 streams each

struct TaskC {
  int task, n, max_steps, n_start, lost_limit, nsub;
  int contact_warps;  // warps of a CTA over which the touching envs are dealt (1..8)
  unsigned flags;
  unsigned seed_lo, seed_hi;
  long long env_offset;
  float dt_env, step_scale;
  ActC<float> act;                     // servo gains, clamps, timestep
  BlkC<float> blk;                     // block <-> floor contact
  float pen_lo[SO_NJ], pen_hi[SO_NJ];  // joint-penalty thresholds, env_base_01.py:155-156
  float rest[SO_NJ], start05[SO_NJ];
  float dist_lo, dist_hi, theta_half, reach;
  float space_s[2][3], space_e[2][3], speed_min, speed_max, ramp, res_w, res_h, fy, noise;
};

struct Consts {
  DynC<float> dyn;
  ConC<float> con;
  KinC<float> kin;
  PadC<float> pad;
  TaskC t;
};

struct Bufs {
  float *qpos, *qvel, *warm, *qcomp, *block, *snap, *aux, *ep_return;
  int* cnt;
  const float* start_tab;  // [n_start][6]
  unsigned long long* stats;  // [0] solver non-converged, [1] nan resets, [2] contact solves that dropped corners (> SO_MAX_CON)
};

// Per-env dynamics parameters (so100_set_param_ranges), drawn at every episode reset.  p: [kParams][n] device array,
// rows kp[6], kv[6], force_lo[6], force_hi[6], frictionloss[6]; nullptr while ranges are off.  lo / hi: fp32 scale
// ranges in draw order, kp[6], damping[6], forcerange[6], frictionloss[6].
// Actuator latency and joint-angle observation noise (so100_set_sim2real) travel here as well: latency [n] (substeps;
// nullptr while no sim2real config is set), ctrl_prev [2][6][n] (Env01/02/06: the previous step's (ctrl_hi, ctrl_lo);
// nullptr for Env05, whose previous target is aux[0:6]), the latency range drawn at resets, and the noise std per joint.
// Any of the three settings selects the per-env kernels; while ranges are off, p holds the model's constants and
// lo = hi = 1, which the reset-time draw reproduces bit for bit.
constexpr int kParams = 5 * SO_NJ, kParamDraws = 4 * SO_NJ;
struct ParamIO {
  float* p;
  float lo[kParamDraws], hi[kParamDraws];
  int* latency;
  float* ctrl_prev;
  int lat_lo, lat_hi;
  float noise[SO_NJ];
  int noise_on;  // some noise[j] != 0
};

struct StepIO {
  const float* actions;
  float *obs, *reward, *terminal_obs, *ep_return_out;
  uint8_t *terminated, *truncated;
  int* ep_len_out;
  unsigned tick;
  int env_lo, env_hi;   // this launch covers envs [env_lo, env_hi) (the host path pipelines chunks)
  int* any_done;        // optional: set to 1 if any env of the launch finished an episode
};

// ------------------------------------------------------------------------------------------------ device helpers
__device__ __forceinline__ uint4 philox4x32(unsigned k0, unsigned k1, unsigned c0, unsigned c1, unsigned c2, unsigned c3) {
#pragma unroll
  for (int r = 0; r < 10; r++) {
    unsigned hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    unsigned hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    unsigned n0 = hi1 ^ c1 ^ k0, n2 = hi0 ^ c3 ^ k1;
    c0 = n0; c1 = lo1; c2 = n2; c3 = lo0;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  return make_uint4(c0, c1, c2, c3);
}
__device__ __forceinline__ float u01(unsigned x) { return (float)(x >> 8) * (1.0f / 16777216.0f); }
__device__ __forceinline__ uint4 draw(const TaskC& t, int env, unsigned tick, unsigned stream) {
  return philox4x32(t.seed_lo, t.seed_hi, (unsigned)(t.env_offset + env), tick, stream, 0u);
}
__device__ __forceinline__ float clampf(float x, float lo, float hi) { return fminf(fmaxf(x, lo), hi); }

struct EnvRegs {  // everything one env carries through a step, in registers
  float q[SO_NJ], v[SO_NJ], w[SO_NJ];
  float qc[SO_NJ];  // Kahan compensation of the qpos integration (qpos = q - qc to ~2^-48)
  float blk[3], bvz;  // block position, z velocity
  float snap[kSnap];
  float aux[kAux];
  int elapsed, flags, miss, t0step;
  float ep_ret;
};

template <int TASK>
__device__ __forceinline__ void load_env(const Bufs& B, int n, int i, EnvRegs& e) {
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) { e.q[j] = B.qpos[j * n + i]; e.v[j] = B.qvel[j * n + i]; e.w[j] = B.warm[j * n + i]; e.qc[j] = B.qcomp[j * n + i]; }
#pragma unroll
  for (int k = 0; k < 3; k++) e.blk[k] = B.block[k * n + i];
  e.bvz = TASK == 5 ? 0.0f : B.block[3 * n + i];
  constexpr int ns = TASK == 5 ? 12 : 7, na = TASK == 5 ? 18 : ((TASK == 2 || TASK == 6) ? 6 : 0);
#pragma unroll
  for (int k = 0; k < ns; k++) e.snap[k] = B.snap[k * n + i];
#pragma unroll
  for (int k = 0; k < na; k++) e.aux[k] = B.aux[k * n + i];
  e.elapsed = B.cnt[i]; e.flags = B.cnt[n + i];
  if (TASK == 5) { e.miss = B.cnt[2 * n + i]; e.t0step = B.cnt[3 * n + i]; }
  e.ep_ret = B.ep_return[i];
}
template <int TASK>
__device__ __forceinline__ void store_env(const Bufs& B, int n, int i, const EnvRegs& e) {
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) { B.qpos[j * n + i] = e.q[j]; B.qvel[j * n + i] = e.v[j]; B.warm[j * n + i] = e.w[j]; B.qcomp[j * n + i] = e.qc[j]; }
#pragma unroll
  for (int k = 0; k < 3; k++) B.block[k * n + i] = e.blk[k];
  if (TASK != 5) B.block[3 * n + i] = e.bvz;
  constexpr int ns = TASK == 5 ? 12 : 7, na = TASK == 5 ? 18 : ((TASK == 2 || TASK == 6) ? 6 : 0);
#pragma unroll
  for (int k = 0; k < ns; k++) B.snap[k * n + i] = e.snap[k];
#pragma unroll
  for (int k = 0; k < na; k++) B.aux[k * n + i] = e.aux[k];
  B.cnt[i] = e.elapsed; B.cnt[n + i] = e.flags;
  if (TASK == 5) { B.cnt[2 * n + i] = e.miss; B.cnt[3 * n + i] = e.t0step; }
  B.ep_return[i] = e.ep_ret;
}

// snapshot layout  Env01/02: end_pos[0..2], wrist_z[3], block_xpos[4..6];  Env05: cam_xpos[0..2], cam_xmat[3..11]
// aux layout       Env02: task_block_pos[0..2], last_block_pos[3..5]
//                  Env05: cmd[0..5], last_angvel[6..11], target[12..14], target_dt[15], last_centre[16..17]

template <int TASK>
__device__ __forceinline__ void take_snapshot(const Consts& C, const float* s, const float* c, EnvRegs& e) {
  KinOut<float> ko;
  task_kinematics<float, TASK == 5>(C.dyn, C.kin, s, c, ko);
  if (TASK == 5) {
#pragma unroll
    for (int k = 0; k < 3; k++) e.snap[k] = ko.cam_pos[k];
#pragma unroll
    for (int k = 0; k < 9; k++) e.snap[3 + k] = ko.cam_R[k];
  } else {
#pragma unroll
    for (int k = 0; k < 3; k++) { e.snap[k] = ko.end_pos[k]; e.snap[4 + k] = e.blk[k]; }
    e.snap[3] = ko.wrist[2];
  }
}

__device__ __forceinline__ void place_block(const TaskC& t, const uint4& r, float* blk) {
  // env01_v1.py:45-49 / env02_v1.py:55-59; draw slot 1 is the reference's discarded theta
  float dist = t.dist_lo + (t.dist_hi - t.dist_lo) * u01(r.x);
  float theta = -1.57079632679489662f + (-t.theta_half + 2.0f * t.theta_half * u01(r.z));
  float sn, cs;
  sincosf(theta, &sn, &cs);
  blk[0] = dist * cs; blk[1] = dist * sn; blk[2] = 0.0f;
}

// env_base_02.py:88-127 on the stale camera pose; returns detection flag, centre in (cx, cy) before noise
__device__ __forceinline__ bool project05(const TaskC& t, const EnvRegs& e, float& cx, float& cy) {
  float rx = e.blk[0] - e.snap[0], ry = e.blk[1] - e.snap[1], rz = e.blk[2] - e.snap[2];
  const float* R = &e.snap[3];
  float x = R[0] * rx + R[3] * ry + R[6] * rz, y = R[1] * rx + R[4] * ry + R[7] * rz, z = R[2] * rx + R[5] * ry + R[8] * rz;
  float u = __fdiv_rn(t.fy * x, z) + 0.5f * t.res_w, v = __fdiv_rn(t.fy * y, z) + 0.5f * t.res_h;
  if (isnan(u) || isnan(v)) return false;
  u = truncf(u); v = truncf(v);
  if (u < 0.0f || u >= t.res_w || v < 0.0f || v >= t.res_h) return false;
  cx = (t.res_w - u) / t.res_w; cy = (t.res_h - v) / t.res_h;
  return true;
}

template <int TASK>
__device__ __forceinline__ void write_obs(const TaskC& t, EnvRegs& e, int env, unsigned tick, unsigned noise_stream, float* o) {
  if (TASK == 5) {  // env05_v1.py:32-75: commanded angles + noisy projected centre, or (-1,-1)
    float cx = -1.0f, cy = -1.0f, px, py;
    if (project05(t, e, px, py)) {
      uint4 r = draw(t, env, tick, noise_stream);
      cx = px + (-t.noise + 2.0f * t.noise * u01(r.x));
      cy = py + (-t.noise + 2.0f * t.noise * u01(r.y));
    }
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) o[j] = e.aux[j];
    o[6] = cx; o[7] = cy;
  } else {  // env_base_01.py:241-270
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) o[j] = e.q[j];
#pragma unroll
    for (int k = 0; k < 3; k++) { o[6 + k] = e.snap[4 + k] - e.snap[k]; o[9 + k] = e.snap[4 + k]; o[12 + k] = e.snap[k]; }
  }
}

// MujocoEnv.reset = mj_resetData + reset_model; kinematics stay ZERO because the reference never calls mj_forward
template <int TASK>
__device__ __forceinline__ void reset_env(const Consts& C, const Bufs& B, EnvRegs& e, int env, unsigned tick, unsigned stream, float* obs) {
  const TaskC& t = C.t;
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) { e.q[j] = 0.0f; e.v[j] = 0.0f; e.w[j] = 0.0f; e.qc[j] = 0.0f; }
#pragma unroll
  for (int k = 0; k < kSnap; k++) e.snap[k] = 0.0f;
  e.elapsed = 0; e.ep_ret = 0.0f; e.bvz = 0.0f;  // mj_resetData zeroes qvel
  e.flags &= ~F_TOUCH;
  if (TASK == 1) {  // env01_v1.py:39-63
    uint4 r = draw(t, env, tick, stream);
    place_block(t, r, e.blk);
    int idx = (int)__umulhi(r.w, (unsigned)t.n_start);
#pragma unroll
    for (int j = 0; j < SO_NJ - 1; j++) e.q[j] = B.start_tab[idx * SO_NJ + j];  // Jaw keeps qpos0
  } else if (TASK == 2 || TASK == 6) {  // env02_v1.py:70-81 + :52-68 (env06_v1.py:53-82 is the same code)
    uint4 r = draw(t, env, tick, stream);
    float prev[3] = {e.aux[0], e.aux[1], e.aux[2]};
    place_block(t, r, e.blk);
    bool has = e.flags & F_HAS_LAST_BLOCK;
#pragma unroll
    for (int k = 0; k < 3; k++) { e.aux[3 + k] = has ? prev[k] : e.blk[k]; e.aux[k] = e.blk[k]; }
    e.flags |= F_HAS_LAST_BLOCK;
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) e.q[j] = t.rest[j];
  } else {  // env03_v1.py:203-215 + :35-57
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) { e.q[j] = t.start05[j]; e.aux[j] = t.start05[j]; }
#pragma unroll
    for (int k = 0; k < 3; k++) { e.aux[12 + k] = 0.5f * (t.space_s[0][k] + t.space_s[1][k]); e.blk[k] = e.aux[12 + k]; }
    e.aux[15] = 0.01f; e.t0step = 0; e.miss = 0;
    e.flags &= ~F_CENTRE_VALID;
  }
  if (t.flags & SO100_FLAG_FRESH_FK_ON_RESET) {
    float s[SO_NJ], c[SO_NJ];
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) sincosf(e.q[j], &s[j], &c[j]);
    take_snapshot<TASK>(C, s, c, e);
  }
  write_obs<TASK>(t, e, env, tick, STREAM_RESET_NOISE, obs);
}

// Draws env `env`'s dynamics parameters: 6 Philox blocks on streams stream..stream+5 give 24 uniforms in draw order;
// scale s = lo + (hi - lo) u; kp = kp0 s_kp, kv = kv0 sqrt(s_kp) s_d, force = force0 s_f, frictionloss = loss0 s_fl, from the
// ctx's fp32 constants, every operation rounded on its own (no contraction), so that the host reproduces the bits.
__device__ __forceinline__ void draw_params(const Consts& C, const ParamIO& P, int env, unsigned tick, unsigned stream) {
  const TaskC& t = C.t;
  const int n = t.n;
  float s[kParamDraws];
#pragma unroll
  for (int k = 0; k < kParamDraws / 4; k++) {
    const uint4 r = draw(t, env, tick, stream + k);
    const unsigned x[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
    for (int m = 0; m < 4; m++) s[4 * k + m] = __fadd_rn(P.lo[4 * k + m], __fmul_rn(__fsub_rn(P.hi[4 * k + m], P.lo[4 * k + m]), u01(x[m])));
  }
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) {
    P.p[j * n + env] = __fmul_rn(t.act.kp[j], s[j]);
    P.p[(SO_NJ + j) * n + env] = __fmul_rn(__fmul_rn(t.act.kv[j], sqrtf(s[j])), s[SO_NJ + j]);
    P.p[(2 * SO_NJ + j) * n + env] = __fmul_rn(t.act.frc_lo[j], s[2 * SO_NJ + j]);
    P.p[(3 * SO_NJ + j) * n + env] = __fmul_rn(t.act.frc_hi[j], s[2 * SO_NJ + j]);
    P.p[(4 * SO_NJ + j) * n + env] = __fmul_rn(C.con.fr_loss[j], s[3 * SO_NJ + j]);
  }
}

// Actuator state at an episode reset (so100_set_sim2real): a new latency d = lo + umulhi(x, hi - lo + 1) from one Philox
// block on `stream`, and the previous servo target becomes the reset pose, (q, 0) for Env01/02/06 (Env05's is aux[0:6],
// which reset_env already set to the start pose): a delayed servo holds the pose instead of chasing ctrl = 0.
template <int TASK>
__device__ __forceinline__ void reset_actuator(const TaskC& t, const ParamIO& P, const EnvRegs& e, int env, unsigned tick, unsigned stream) {
  const uint4 r = draw(t, env, tick, stream);
  P.latency[env] = P.lat_lo + (int)__umulhi(r.x, (unsigned)(P.lat_hi - P.lat_lo + 1));
  if (TASK != 5) {
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) { P.ctrl_prev[j * t.n + env] = e.q[j]; P.ctrl_prev[(SO_NJ + j) * t.n + env] = 0.0f; }
  }
}

// Joint-angle observation noise (Env01/02/06): o[j] = q_j + sigma_j z_j, z standard normals by the Box-Muller transform of
// act_kernel (so100_ppo_kernels.cuh) on Philox blocks stream, stream + 1; z[0..5] of the 8 it gives.  A joint with
// sigma_j == 0 keeps its bits (no 0 * z is added).  Output only: nothing the env carries depends on it.
__device__ __forceinline__ void obs_noise(const TaskC& t, const ParamIO& P, int env, unsigned tick, unsigned stream, float* o) {
  const uint4 r0 = draw(t, env, tick, stream), r1 = draw(t, env, tick, stream + 1);
  const unsigned w[SO_NJ] = {r0.x, r0.y, r0.z, r0.w, r1.x, r1.y};  // (u1, u2) pairs; block 1's (z, w) would give z[6..7]
  float z[SO_NJ];
#pragma unroll
  for (int k = 0; k < SO_NJ / 2; k++) {
    const float u1 = ((float)(w[2 * k] >> 8) + 0.5f) * (1.0f / 16777216.0f), u2 = (float)(w[2 * k + 1] >> 8) * (1.0f / 16777216.0f);
    const float rad = sqrtf(-2.0f * logf(u1));
    float sn, cs;
    sincospif(2.0f * u2, &sn, &cs);
    z[2 * k] = rad * cs; z[2 * k + 1] = rad * sn;
  }
#pragma unroll
  for (int j = 0; j < SO_NJ; j++)
    if (P.noise[j] != 0.0f) o[j] = __fadd_rn(o[j], __fmul_rn(P.noise[j], z[j]));
}

__device__ __forceinline__ float joint_penalty(const TaskC& t, const float* ang) {  // env_base_01.py:144-163
  float r = 0.0f;
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) {
    if (ang[j] < t.pen_lo[j]) r -= (t.pen_lo[j] - ang[j]) * 10.0f;
    else if (ang[j] > t.pen_hi[j]) r -= (ang[j] - t.pen_hi[j]) * 10.0f;
  }
  return r;
}

// env_base_01.py:180-239 evaluated BEFORE the physics step on the previous step's (stale) kinematics
__device__ __forceinline__ float reward_reach(const TaskC& t, EnvRegs& e, bool in_reach) {
  const float PI07 = 2.19911485751285527f;  // 0.7*pi
  float dx = e.snap[4] - e.snap[0], dy = e.snap[5] - e.snap[1], dz = e.snap[6] - e.snap[2];
  float distance = sqrtf(dx * dx + dy * dy + dz * dz);
  bool ever = e.flags & F_EVER_STEPPED;
  float r = 0.0f;
  if (e.snap[5] < -0.1f && ever && e.q[1] < -PI07) r += (e.q[1] + PI07) * 0.7f;
  if (ever && e.snap[2] < 0.02f) r += (e.snap[2] - 0.02f) * 20.0f;
  if (ever && e.snap[3] < 0.08f) r += clampf((e.snap[3] - 0.08f) * 10.0f, -0.8f, 0.8f);
  r += fminf(-distance + 0.02f, 0.0f) * 0.5f;
  if (in_reach) {  // Env06: env_base_06.py:149-162
    float jn = clampf((e.q[5] + 0.2f) / 2.2f, 0.0f, 1.0f);
    r += 100.0f / (1.0f + expf(-10.0f * (jn - 0.3f)));
  }
  r += joint_penalty(t, e.q);
  e.flags |= F_EVER_STEPPED;
  return r;
}

// Shared-memory pool of contact-solve slots of one CTA (CoopSlot in so100_dyn.cuh, slot-major).  Slots are handed out
// anew in every substep from one of two counters used in alternation: cnt[sub & 1] serves substep `sub`, and thread 0
// clears the other one right after the substep's CTA barrier, a full substep before it is used again.
constexpr int kPoolSlots = 48;
struct ContactPool {
  float* f;
  double* d;
  int* cnt;
  int nslot;  // 0: no pool (debug kernels): every contact solve takes the out-of-line serial path
  __device__ __forceinline__ CoopSlot slot(int k) const { return CoopSlot{f + k * CoopSlot::kFloats, d + k * CoopSlot::kDoubles}; }
};
constexpr size_t kPoolBytes = (size_t)kPoolSlots * (CoopSlot::kDoubles * 8 + CoopSlot::kFloats * 4);

// 16 x mj_step on the arm.  ctrl is constant over the env step, so kp*clip(ctrl) is hoisted.
// ctrl is carried as an unevaluated sum ctrl_hi + ctrl_lo so that Env01/02's closed loop ctrl = qpos + a*0.075 does not
// round the 0.075-rad increment to the ulp of a 3-rad angle (that rounding random-walks qpos in a neutrally stable loop).
// PARAMS: the env's own kp, kv, forcerange and friction loss (ParamIO; pv = p + env, rows n apart) replace the model's,
// read once and held in registers over the substeps; every other constant stays the model's.
// Actuator latency (PARAMS only): (ctrl_hi, ctrl_lo) drive substeps 0 .. d-1, and at substep d (0 < d < nsub) the control
// switches to the step's own target, reloaded from `next` (Env01/02/06: the env's ctrl_prev column, rows n apart, where the
// step stored it; Env05: its new command, ctrl_lo 0) so that only one control pair is held over the loop.  Substep d gets
// the first substep's sweeps: the control jumps there.  d = 0 and next = nullptr: no switch.
template <int TASK, bool SPEC, bool PADS, bool PARAMS>
__device__ __forceinline__ void physics(const Consts& C, const Bufs& B, EnvRegs& e, const float* ctrl_hi, const float* ctrl_lo, bool live, int nsub,
                                        const ContactPool& pool, const float* pv, int d_switch = 0, const float* next = nullptr) {
  const TaskC& t = C.t;
  // SPEC: the solver / servo constants of the so100 MJCF are literals (immediates after unrolling), not constant-bank loads
  ConC<float> Kg;
  ActC<float> Ag;
  BlkC<float> Bg;
  if (SPEC) so100_gen_solver_constants(Kg, Ag, Bg);
  const ConC<float>& K = SPEC ? Kg : C.con;
  const ActC<float>& A = SPEC ? Ag : t.act;
  const BlkC<float>& Kb = SPEC ? Bg : t.blk;
  const bool block_moves = TASK != 5 && !(t.flags & SO100_FLAG_STATIC_BLOCK);  // Env05 scripts its block (env03_v1.py:95-122)
  float pkp[SO_NJ], pkv[SO_NJ], pflo[SO_NJ], pfhi[SO_NJ], ploss[SO_NJ];
  if (PARAMS) {
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) {
      pkp[j] = pv[j * t.n]; pkv[j] = pv[(SO_NJ + j) * t.n]; pflo[j] = pv[(2 * SO_NJ + j) * t.n];
      pfhi[j] = pv[(3 * SO_NJ + j) * t.n]; ploss[j] = pv[(4 * SO_NJ + j) * t.n];
    }
  }
  const float* loss = PARAMS ? ploss : K.fr_loss;
  float cc[SO_NJ], cl[SO_NJ];
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) {
    float sum = ctrl_hi[j] + ctrl_lo[j];
    bool in = sum >= A.ctrl_lo[j] && sum <= A.ctrl_hi[j];
    cc[j] = in ? ctrl_hi[j] : clampf(sum, A.ctrl_lo[j], A.ctrl_hi[j]);
    cl[j] = in ? ctrl_lo[j] : 0.0f;
  }
  bool unconverged = false;
#pragma unroll 1
  for (int sub = 0; sub < nsub; sub++) {
    __syncthreads();  // keeps a CTA's warps on the same stretch of straight-line code (i-cache), and orders the pool's slot counters
    if (PADS && pool.nslot && threadIdx.x == 0) pool.cnt[(sub + 1) & 1] = 0;
    if (PARAMS && sub == d_switch && sub > 0) {
#pragma unroll
      for (int j = 0; j < SO_NJ; j++) {
        const float hi = TASK == 5 ? next[j] : next[j * t.n], lo = TASK == 5 ? 0.0f : next[(SO_NJ + j) * t.n];
        const float sum = hi + lo;
        const bool in = sum >= A.ctrl_lo[j] && sum <= A.ctrl_hi[j];
        cc[j] = in ? hi : clampf(sum, A.ctrl_lo[j], A.ctrl_hi[j]);
        cl[j] = in ? lo : 0.0f;
      }
    }
    const int sweeps = (sub == 0 || (PARAMS && sub == d_switch)) ? SO100_SWEEPS_FIRST : SO100_SWEEPS_REST;
    float s[SO_NJ], c[SO_NJ], bias[SO_NJ], M[21], b[SO_NJ];
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) so_sincos(e.q[j], &s[j], &c[j]);
    if (sub == nsub - 1) take_snapshot<TASK>(C, s, c, e);  // kinematics of the LAST substep's start state (Q3)
    if (SPEC) dyn_bias_mass_so100<float>(s, c, e.v, bias, M);  // constants folded at build time (so100 MJCF)
    else dyn_bias_mass<float>(C.dyn, s, c, e.v, bias, M);       // any other model: constants from the ctx
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) {
      float f = (PARAMS ? pkp[j] : A.kp[j]) * ((cc[j] - e.q[j]) + (cl[j] + e.qc[j])) - (PARAMS ? pkv[j] : A.kv[j]) * e.v[j];  // differences first: no cancellation
      b[j] = clampf(f, PARAMS ? pflo[j] : A.frc_lo[j], PARAMS ? pfhi[j] : A.frc_hi[j]) - bias[j];
    }
    // ctrl changes once per env step, so the first substep's warm start is far: 5 sweeps (each contracts the error
    // ~100x); afterwards qacc moves a few % per substep: 3 sweeps.  The solver adds per-lane sweeps if the last one
    // still moved qacc by > 1e-3.  (Extrapolating the warm start to save a sweep was measured: no faster, 6x less
    // accurate - profiles/r1_variants.md.)
    // envs with a pad corner below the floor take the Newton path on the full problem (dense contact rows); the rest
    // keep the per-dof Gauss-Seidel.  e.w enters both as the warm start (the previous substep's qacc).
    // The broad phase runs on the substep's MUFU sin/cos, whose 2^-21 error moves a pad corner by up to ~1.5e-7 m - as
    // much as a resting contact penetrates (~2e-7 m) - so it asks with a margin, and the contact path redoes its own
    // kinematics with sincosf of the compensated angle: without that, resting contacts flicker on and off from substep to
    // substep (measured: p99.9 |dq| 9e-4 rad against the oracle instead of 3e-7, tools/contact_precision.py).
    // A tail thread (!live, shadowing the launch's last env) never touches: it asks for no pool slot, so that a touching
    // last env cannot fill its CTA's pool with copies of itself and push the CTA's real touching envs to the serial solve.
    unsigned touch = PADS && C.pad.n > 0 ? pads_touch<float>(C.dyn, C.kin, C.pad, s, c, SO100_TOUCH_MARGIN) : 0u;
    if (!live) touch = 0u;
    if (PADS && sub == nsub - 1) e.flags = touch ? (e.flags | F_TOUCH) : (e.flags & ~F_TOUCH);
    float d = 0.0f;
    bool solved = false;
    const unsigned tmask = PADS ? __ballot_sync(0xffffffffu, touch != 0u) : 0u;
    if (PADS) {
      // Phase A, the touching env's own thread: a pool slot (one atomic per warp), accurate trigonometry, the contacts
      // with their Jacobians and row parameters, and the substep's M, b, per-dof rows and warm start -> the slot.
      int myslot = -1;
      if (tmask) {  // (warp-uniform) some lane touches
        int slot = kPoolSlots;
        if (pool.nslot) {
          const int lane = threadIdx.x & 31, leader = __ffs(tmask) - 1;
          int base = 0;
          if (lane == leader) base = atomicAdd(&pool.cnt[sub & 1], __popc(tmask));
          base = __shfl_sync(0xffffffffu, base, leader);
          slot = base + __popc(tmask & ((1u << lane) - 1u));
        }
        if (touch) {
          float cs[SO_NJ], cc_[SO_NJ];
#pragma unroll
          for (int j = 0; j < SO_NJ; j++) {
            float sj, cj;
            sincosf(e.q[j], &sj, &cj);
            cs[j] = fmaf(-e.qc[j], cj, sj); cc_[j] = fmaf(e.qc[j], sj, cj);  // sin / cos of q - qc to first order in qc (|qc| < 2e-7)
          }
          bool serial = slot >= pool.nslot;  // pool exhausted (> kPoolSlots touching envs in this CTA)
          if (!serial) {
            const int nc = coop_fill(C.dyn, C.kin, C.pad, C.con, PARAMS ? ploss : C.con.fr_loss, pool.slot(slot), cs, cc_, e.q, e.qc, e.v, M, b, e.w, touch);
            serial = nc < 0;            // > kCoopCon corners at once
            if (nc > 0) myslot = slot;  // nc == 0: the accurate kinematics found no corner below the floor after all
          }
          if (serial) {  // thread-local storage, one thread, out of line
            ContactIO<float> cio;
#pragma unroll
            for (int j = 0; j < SO_NJ; j++) { cio.s[j] = cs[j]; cio.c[j] = cc_[j]; cio.q[j] = e.q[j]; cio.qc[j] = e.qc[j]; cio.qd[j] = e.v[j]; cio.b[j] = b[j]; cio.a[j] = e.w[j]; }
#pragma unroll
            for (int k = 0; k < 21; k++) cio.M[k] = M[k];
            int over = 0;
            int st;
            if (PARAMS) {
              float lc[SO_NJ];  // a copy for the out-of-line call: ploss itself stays in registers
#pragma unroll
              for (int j = 0; j < SO_NJ; j++) lc[j] = ploss[j];
              st = contact_solve_loss<float>(C.dyn, C.kin, C.pad, C.con, lc, cio, touch, &over);
            } else st = contact_solve<float>(C.dyn, C.kin, C.pad, C.con, cio, touch, &over);
            if (over && live) atomicAdd(&B.stats[2], 1ULL);
            if (st != 0 && !over) {
#pragma unroll
              for (int j = 0; j < SO_NJ; j++) e.w[j] = cio.a[j];
            }
            if (over) st = 0;  // > SO_MAX_CON corners (never seen): counted, and this substep falls back to the contact-free solve
            solved = st != 0;
            if (st < 0) d = 1e30f;  // iteration cap / indefinite Hessian: counted with the Gauss-Seidel's unconverged substeps
          }
        }
      }
      // every other env: the per-dof Gauss-Seidel, BEFORE the cooperative phase, so that M and b are dead across it
      if (!solved && myslot < 0) {
        d = solve_qacc<float>(K, loss, M, b, e.q, e.qc, e.v, e.w, sweeps);
        solved = true;
      }
      // Phase B, the whole CTA: groups of kCoopLanes threads run the Newton solves of the filled slots.  Consecutive slots
      // go to different warps (slot = 8 * (group within its warp) + warp), so a few touching envs occupy every scheduler.
      if (pool.nslot) {
        __syncthreads();
        const int nfill = min(pool.cnt[sub & 1], pool.nslot);  // CTA-uniform
        if (nfill > 0) {
          const int g = threadIdx.x / kCoopLanes, glane = threadIdx.x % kCoopLanes, gw = g & 3;
          constexpr int kGroups = kBlock / kCoopLanes;
          for (int base = 0; base < nfill; base += kGroups) {
            if (base + (g >> 2) < nfill) {  // (warp-uniform) the warp's first group has a slot
              const int sl = base + gw * (kGroups / 4) + (g >> 2);
              float* sf = nullptr;
              double* sd = nullptr;
              if (sl < nfill && pool.slot(sl).F(CoopSlot::kNc) > 0.0f) { sf = pool.slot(sl).f; sd = pool.slot(sl).d; }
              coop_solve_warp(sf, sd, glane, 8 * gw);
            }
          }
          __syncthreads();
          if (myslot >= 0) {
            const CoopSlot S = pool.slot(myslot);
#pragma unroll
            for (int j = 0; j < SO_NJ; j++) e.w[j] = (float)S.D(CoopSlot::kX + j);
            solved = true;
            if (S.sc(10) != 1.0) d = 1e30f;
          }
        }
      }
    }
    if (!PADS) d = solve_qacc<float>(K, loss, M, b, e.q, e.qc, e.v, e.w, sweeps);
    float amax = 1.0f;
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) {
      amax = fmaxf(amax, fabsf(e.w[j]));
      e.v[j] += A.h * e.w[j];   // mj_Euler (semi-implicit; no joint damping in this model)
      float y = __fsub_rn(__fmul_rn(A.h, e.v[j]), e.qc[j]);  // compensated sum: 16 000 substeps of 1e-5 rad increments on |q| ~ 3
      float s1 = __fadd_rn(e.q[j], y);
      e.qc[j] = __fsub_rn(__fsub_rn(s1, e.q[j]), y);
      e.q[j] = s1;
    }
    unconverged |= d > 2e-3f * amax;
    if (block_moves) block_substep<float>(Kb, A.h, e.blk[2], e.bvz);  // after the snapshot: xpos is of the substep's start
  }
  // the last sweep's largest update bounds the error BEFORE that sweep; the sweep itself contracts it ~100x more
  if (unconverged && live) atomicAdd(&B.stats[0], 1ULL);
}

// ------------------------------------------------------------------------------------------------ kernels
template <int TASK, bool SPEC, bool PADS, bool PARAMS>
__global__ void __launch_bounds__(kBlock, SO100_MINBLOCKS) step_kernel(const __grid_constant__ Consts C, const Bufs B, const StepIO io,
                                                                        const __grid_constant__ ParamIO par) {
  constexpr int OD = TASK == 5 ? 8 : 15;
  __shared__ __align__(16) float sh[kBlock * OD];
  static_assert((kBlock * OD) % 4 == 0, "obs rows of a CTA must be a whole number of float4");
  const TaskC& t = C.t;
  const int n = t.n, base = io.env_lo + blockIdx.x * kBlock, hi = io.env_hi;
  const unsigned tick = io.tick;
  // Envs whose jaw pads touched the floor last step take the contact path in most substeps of this one (~4-10 % of the
  // envs under random actions).  The CTA re-deals its 256 envs to its threads with the touching ones first (a stable
  // partition on the hint bit) and deals those round-robin over W warps: phase A of the contact path (the env's own
  // thread fills its slot) then costs every warp a few lanes instead of one warp all of its lanes.  `slot` is the env
  // this thread now owns.
  __shared__ unsigned short perm[kBlock];
  __shared__ int warp_cnt[kBlock / 32];
  __shared__ int pool_cnt[2];
  extern __shared__ double pool_mem[];  // kPoolBytes when the model has pads, else nothing
  const ContactPool pool{reinterpret_cast<float*>(pool_mem + (size_t)kPoolSlots * CoopSlot::kDoubles), pool_mem, pool_cnt,
                         PADS && C.pad.n > 0 ? kPoolSlots : 0};
  if (threadIdx.x < 2) pool_cnt[threadIdx.x] = 0;
  int slot = threadIdx.x;
  if (PADS && C.pad.n > 0) {  // (compile-time for the default kernel: thread t owns env t, every access coalesced)
    const int mine = base + (int)threadIdx.x;
    const bool hint = mine < hi && (B.cnt[n + mine] & F_TOUCH);
    const unsigned bal = __ballot_sync(0xffffffffu, hint);
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    if (lane == 0) warp_cnt[wid] = __popc(bal);
    __syncthreads();
    int before = 0, total = 0;  // touching envs in earlier warps / in the CTA
#pragma unroll
    for (int w = 0; w < kBlock / 32; w++) { const int cw = warp_cnt[w]; total += cw; before += w < wid ? cw : 0; }
    const int rank_t = before + __popc(bal & ((1u << lane) - 1u));  // rank among the touching envs
    // Touching env r goes to lane r / W of warp r % W (W = contact_warps): warp w < W holds c_w = ceil((total - w) / W) of
    // them in its first lanes.  The other envs fill the remaining lanes in their original order, so their state accesses
    // stay (piecewise) coalesced.  With fewer than 32 * W positions for the touching ones (never at W = 8) the rest queue
    // behind them in order as well.
    const int W = t.contact_warps, cap = 32 * W;
    int dest;
    if (hint && rank_t < cap) dest = (rank_t % W) * 32 + rank_t / W;
    else {
      const int dealt = total < cap ? total : cap;
      int k = hint ? (rank_t - cap) : (total - dealt) + ((int)threadIdx.x - rank_t);  // rank among the envs that are not dealt
      dest = 0;
#pragma unroll
      for (int w = 0; w < kBlock / 32; w++) {
        int cw = w < W ? (dealt - w + W - 1) / W : 0;
        cw = cw < 0 ? 0 : (cw > 32 ? 32 : cw);
        const int free_w = 32 - cw;
        if (k >= 0 && k < free_w) dest = w * 32 + cw + k;
        k -= free_w;
      }
    }
    perm[dest] = (unsigned short)threadIdx.x;
    __syncthreads();
    slot = perm[threadIdx.x];
  }
  const bool live = base + slot < hi;
  const int i = live ? base + slot : hi - 1;  // tail threads shadow the last env (they must reach every barrier); nothing they compute is stored
  // coalesced load of the CTA's action rows through shared memory
  for (int k = threadIdx.x; k < kBlock * SO_NJ; k += kBlock) {
    int g = base * SO_NJ + k;
    sh[k] = g < hi * SO_NJ ? io.actions[g] : 0.0f;
  }
  __syncthreads();
  float a[SO_NJ];
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) {
    a[j] = sh[slot * SO_NJ + j];
    if (t.flags & SO100_FLAG_CLIP_ACTIONS) a[j] = clampf(a[j], -1.0f, 1.0f);
  }
  __syncthreads();
  float obs[OD];
  {
    EnvRegs e;
    load_env<TASK>(B, n, i, e);
    // actuator state, loaded with the env state: a later first touch of cold memory waits out the drain of whatever the
    // L2 holds dirty (measured under bench.py's L2 flush: +30 us per step when these loads came just before physics<>)
    int d = 0;
    float ph[SO_NJ], pl[SO_NJ];
    if (PARAMS && par.latency) {
      d = par.latency[i];
      if (TASK != 5) {
#pragma unroll
        for (int j = 0; j < SO_NJ; j++) { ph[j] = par.ctrl_prev[j * n + i]; pl[j] = par.ctrl_prev[(SO_NJ + j) * n + i]; }
      }
    }
    float rew, ctrl[SO_NJ], ctrl_lo[SO_NJ];
    bool term = false;
    if (TASK == 1 || TASK == 2 || TASK == 6) {
      bool in_reach = false;
      if (TASK == 6) {  // env06_v1.py:19, on the stale kinematics
        float dx = e.snap[4] - e.snap[0], dy = e.snap[5] - e.snap[1], dz = e.snap[6] - e.snap[2];
        in_reach = sqrtf(dx * dx + dy * dy + dz * dz) < t.reach;
      }
      rew = reward_reach(t, e, in_reach);
      if (TASK == 6 && in_reach) {  // env06_v1.py:30-38: bonus, the block stays where it is
        float bx = e.aux[0] - e.aux[3], by = e.aux[1] - e.aux[4], bz = e.aux[2] - e.aux[5];
        rew += sqrtf(bx * bx + by * by + bz * bz) * 20.0f;
      }
#pragma unroll
      for (int j = 0; j < SO_NJ; j++) { ctrl[j] = e.q[j]; ctrl_lo[j] = a[j] * t.step_scale - e.qc[j]; }  // closed loop on qpos (Q6)
      if (TASK == 2) {  // env02_v1.py:29-37, reach test on stale kinematics
        float dx = e.snap[4] - e.snap[0], dy = e.snap[5] - e.snap[1], dz = e.snap[6] - e.snap[2];
        if (sqrtf(dx * dx + dy * dy + dz * dz) < t.reach) {
          float bx = e.aux[0] - e.aux[3], by = e.aux[1] - e.aux[4], bz = e.aux[2] - e.aux[5];
          rew += sqrtf(bx * bx + by * by + bz * bz) * 20.0f;
          uint4 r = draw(t, i, tick, STREAM_TASK);
#pragma unroll
          for (int k = 0; k < 3; k++) e.aux[3 + k] = e.aux[k];
          place_block(t, r, e.blk);
#pragma unroll
          for (int k = 0; k < 3; k++) e.aux[k] = e.blk[k];
        }
      }
      if (PARAMS && par.latency) {  // the previous target drives substeps 0 .. d-1; this step's target goes to ctrl_prev
        float* cp = par.ctrl_prev + i;
#pragma unroll
        for (int j = 0; j < SO_NJ; j++) {
          if (live) { cp[j * n] = ctrl[j]; cp[(SO_NJ + j) * n] = ctrl_lo[j]; }
          if (d > 0) { ctrl[j] = ph[j]; ctrl_lo[j] = pl[j]; }
        }
      }
      physics<TASK, SPEC, PADS, PARAMS>(C, B, e, ctrl, ctrl_lo, live, t.nsub, pool, PARAMS ? par.p + i : nullptr, d,
                                        PARAMS && par.latency ? par.ctrl_prev + i : nullptr);
      write_obs<TASK>(t, e, i, tick, STREAM_NOISE, obs);
      if (PARAMS && par.noise_on) obs_noise(t, par, i, tick, STREAM_OBS_NOISE, obs);
    } else {  // env03_v1.py:124-201
      float time = (float)e.elapsed * t.dt_env;
      float f = fminf(time / t.ramp, 1.0f);
      float smin[3], smax[3];
#pragma unroll
      for (int k = 0; k < 3; k++) {
        smin[k] = t.space_s[0][k] + f * (t.space_e[0][k] - t.space_s[0][k]);
        smax[k] = t.space_s[1][k] + f * (t.space_e[1][k] - t.space_s[1][k]);
      }
      float speed = f <= 0.05f ? t.speed_min : t.speed_min + (f - 0.05f) * (t.speed_max - t.speed_min) / (1.0f - 0.05f);
      float dx = e.aux[12] - e.blk[0], dy = e.aux[13] - e.blk[1], dz = e.aux[14] - e.blk[2];
      float dist = sqrtf(dx * dx + dy * dy + dz * dz);
      if (!((float)(e.elapsed - e.t0step) * t.dt_env < e.aux[15] && dist > 0.02f)) {  // :77-93
        uint4 r = draw(t, i, tick, STREAM_TASK);
        e.aux[12] = smin[0] + (smax[0] - smin[0]) * u01(r.x);
        e.aux[13] = smin[1] + (smax[1] - smin[1]) * u01(r.y);
        e.aux[14] = smin[2] + (smax[2] - smin[2]) * u01(r.z);
        e.aux[15] = 1.2f + (5.1f - 1.2f) * u01(r.w);
        e.t0step = e.elapsed;
      }
      dx = e.aux[12] - e.blk[0]; dy = e.aux[13] - e.blk[1]; dz = e.aux[14] - e.blk[2];  // :95-122
      dist = sqrtf(dx * dx + dy * dy + dz * dz);
      if (dist > 0.0f) {
        float sd = fminf(speed * t.act.h, dist) / dist;
        e.blk[0] += dx * sd; e.blk[1] += dy * sd; e.blk[2] += dz * sd;
      }
      float newcmd[SO_NJ];
#pragma unroll
      for (int j = 0; j < SO_NJ; j++) { newcmd[j] = e.aux[j] + a[j] * t.step_scale; ctrl[j] = newcmd[j]; ctrl_lo[j] = 0.0f; }  // open loop (Q6)
      if (PARAMS && d > 0) {  // the previous command drives substeps 0 .. d-1
#pragma unroll
        for (int j = 0; j < SO_NJ; j++) ctrl[j] = e.aux[j];
      }
      physics<TASK, SPEC, PADS, PARAMS>(C, B, e, ctrl, ctrl_lo, live, t.nsub, pool, PARAMS ? par.p + i : nullptr, d, newcmd);
      write_obs<TASK>(t, e, i, tick, STREAM_NOISE, obs);
      if (obs[6] == -1.0f && obs[7] == -1.0f) {  // :152-164
        if (e.miss > t.lost_limit) term = true;
        e.miss += 1;
      } else { e.aux[16] = obs[6]; e.aux[17] = obs[7]; e.flags |= F_CENTRE_VALID; e.miss = 0; }
      rew = 0.5f;
      if (e.flags & F_CENTRE_VALID) {
        float ex = 0.5f - e.aux[16], ey = 0.5f - e.aux[17];
        rew -= sqrtf(ex * ex + ey * ey);
      }
      rew += joint_penalty(t, e.aux);  // on the commanded (old) angles, Q7
      float pen = 0.0f;
#pragma unroll
      for (int j = 0; j < SO_NJ; j++) {  // env_base_01.py:165-178 with timestep 0.002 (Q8)
        float av = (newcmd[j] - e.aux[j]) / t.act.h;
        if (e.flags & F_ANGVEL_VALID) pen += fabsf(av - e.aux[6 + j]) * 0.0025f;
        e.aux[6 + j] = av;
      }
      e.flags |= F_ANGVEL_VALID;
      rew += -pen * f;
      obs[6] *= 5.0f; obs[7] *= 5.0f;
#pragma unroll
      for (int j = 0; j < SO_NJ; j++) e.aux[j] = newcmd[j];
    }
    // MuJoCo's mj_checkPos/Vel analogue: a non-finite state forces a reset (counted, never trapped)
    float chk = 0.0f;
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) chk += e.q[j] + e.v[j];
    bool bad = !isfinite(chk);
    if (bad && live) atomicAdd(&B.stats[1], 1ULL);
    // A blown-up env ends its episode as TERMINATED (never truncated: a learner bootstraps truncations with
    // V(terminal_obs)), with a finite reward and, below, a finite terminal observation (the reset one).
    if (bad) { term = true; if (!isfinite(rew)) rew = 0.0f; }
    e.elapsed += 1;
    e.ep_ret += rew;
    bool trunc = e.elapsed >= t.max_steps;  // gymnasium TimeLimit
    if (live) {
      io.reward[i] = rew;
      io.terminated[i] = term ? 1 : 0;
      io.truncated[i] = (trunc && !term) ? 1 : 0;
    }
    if (term || trunc) {
      if (live && io.terminal_obs && !bad) {
#pragma unroll
        for (int k = 0; k < OD; k++) io.terminal_obs[(size_t)i * OD + k] = obs[k];
      }
      if (live && io.ep_return_out) io.ep_return_out[i] = e.ep_ret;
      if (live && io.ep_len_out) io.ep_len_out[i] = e.elapsed;
      if (live && io.any_done) *io.any_done = 1;
      reset_env<TASK>(C, B, e, i, tick, STREAM_RESET, obs);
      if (PARAMS && live) draw_params(C, par, i, tick, STREAM_PARAM_RESET);
      if (PARAMS && live && par.latency) reset_actuator<TASK>(t, par, e, i, tick, STREAM_LAT_RESET);
      if (PARAMS && TASK != 5 && par.noise_on) obs_noise(t, par, i, tick, STREAM_OBS_RESET_NOISE, obs);
      if (live && io.terminal_obs && bad) {
#pragma unroll
        for (int k = 0; k < OD; k++) io.terminal_obs[(size_t)i * OD + k] = obs[k];
      }
    }
    if (live) store_env<TASK>(B, n, i, e);
#pragma unroll
    for (int k = 0; k < OD; k++) sh[slot * OD + k] = obs[k];
  }
  __syncthreads();
  // the CTA's obs rows are one contiguous, 16-byte aligned span (kBlock * OD floats): 512 bytes per warp instruction
  // (on the host path these stores cross the link; larger write bursts pack into fuller PCIe packets)
  if (base + kBlock <= hi) {
    float4* dst = reinterpret_cast<float4*>(io.obs + (size_t)base * OD);
    const float4* src = reinterpret_cast<const float4*>(sh);
    for (int k = threadIdx.x; k < kBlock * OD / 4; k += kBlock) dst[k] = src[k];
  } else {
    for (int k = threadIdx.x; k < kBlock * OD; k += kBlock) {
      size_t g = (size_t)base * OD + k;
      if (g < (size_t)hi * OD) io.obs[g] = sh[k];
    }
  }
}

template <int TASK>
__global__ void __launch_bounds__(kBlock) reset_kernel(const __grid_constant__ Consts C, const Bufs B, const uint8_t* mask, float* obs_out, unsigned tick,
                                                       const __grid_constant__ ParamIO par) {
  constexpr int OD = TASK == 5 ? 8 : 15;
  const int n = C.t.n, i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= n || (mask && !mask[i])) return;
  EnvRegs e;
  load_env<TASK>(B, n, i, e);
  float obs[OD];
  reset_env<TASK>(C, B, e, i, tick, STREAM_API_RESET, obs);
  if (par.p) draw_params(C, par, i, tick, STREAM_PARAM_API_RESET);
  if (par.latency) reset_actuator<TASK>(C.t, par, e, i, tick, STREAM_LAT_API_RESET);
  if (TASK != 5 && par.noise_on) obs_noise(C.t, par, i, tick, STREAM_OBS_API_NOISE, obs);
  store_env<TASK>(B, n, i, e);
#pragma unroll
  for (int k = 0; k < OD; k++) obs_out[(size_t)i * OD + k] = obs[k];
}

// ctrl_prev at the first so100_set_sim2real: the exact current position, (qpos, -qpos_comp); m = 6 n
__global__ void __launch_bounds__(kBlock) actuator_init_kernel(const float* qpos, const float* qcomp, float* ctrl_prev, int m) {
  const int k = blockIdx.x * kBlock + threadIdx.x;
  if (k >= m) return;
  ctrl_prev[k] = qpos[k];
  ctrl_prev[m + k] = -qcomp[k];
}

// debug / parity triage: n x mj_step under a given ctrl, no task logic (no reward / obs / counters / reset); the snapshot
// is refreshed with the kinematics of the last substep's start state, as in a full env step
template <int TASK, bool SPEC, bool PARAMS>
__global__ void __launch_bounds__(kBlock, SO100_MINBLOCKS) substeps_kernel(const __grid_constant__ Consts C, const Bufs B, const float* ctrl, int nsub,
                                                                           const float* par) {
  const int n = C.t.n, base = blockIdx.x * kBlock;
  const bool live = base + (int)threadIdx.x < n;
  const int i = live ? base + (int)threadIdx.x : n - 1;  // tail threads shadow the last env (physics has CTA barriers)
  EnvRegs e;
  load_env<TASK>(B, n, i, e);
  float ch[SO_NJ], cl[SO_NJ];
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) { ch[j] = ctrl[(size_t)i * SO_NJ + j]; cl[j] = 0.0f; }
  physics<TASK, SPEC, true, PARAMS>(C, B, e, ch, cl, live, nsub, ContactPool{nullptr, nullptr, nullptr, 0}, PARAMS ? par + i : nullptr);
  if (live) store_env<TASK>(B, n, i, e);
}

// debug / parity: one cold-start forward-dynamics evaluation per sample
__global__ void __launch_bounds__(kBlock) forward_kernel(const __grid_constant__ Consts C, int n, const float* qpos, const float* qvel, const float* ctrl,
                                                          float* M_out, float* bias_out, float* qacc_out, float* kin_out) {
  int i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= n) return;
  const TaskC& t = C.t;
  float q[SO_NJ], v[SO_NJ], s[SO_NJ], c[SO_NJ], bias[SO_NJ], M[21], b[SO_NJ], a[SO_NJ];
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) { q[j] = qpos[j * n + i]; v[j] = qvel[j * n + i]; sincosf(q[j], &s[j], &c[j]); a[j] = 0.0f; }
  dyn_bias_mass<float>(C.dyn, s, c, v, bias, M);
#pragma unroll
  for (int j = 0; j < SO_NJ; j++) {
    float f = t.act.kp[j] * clampf(ctrl[j * n + i], t.act.ctrl_lo[j], t.act.ctrl_hi[j]) - t.act.kp[j] * q[j] - t.act.kv[j] * v[j];
    b[j] = clampf(f, t.act.frc_lo[j], t.act.frc_hi[j]) - bias[j];
  }
  float zc[SO_NJ] = {0, 0, 0, 0, 0, 0};
  if (C.pad.n > 0 && pads_touch<float>(C.dyn, C.kin, C.pad, s, c)) {
    ContactIO<float> cio;
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) { cio.s[j] = s[j]; cio.c[j] = c[j]; cio.q[j] = q[j]; cio.qc[j] = 0.0f; cio.qd[j] = v[j]; cio.b[j] = b[j]; cio.a[j] = 0.0f; }
#pragma unroll
    for (int k = 0; k < 21; k++) cio.M[k] = M[k];
    contact_solve<float>(C.dyn, C.kin, C.pad, C.con, cio, ~0u);
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) a[j] = cio.a[j];
  } else solve_qacc<float>(C.con, C.con.fr_loss, M, b, q, zc, v, a, 12);
  if (M_out)
#pragma unroll
    for (int k = 0; k < 21; k++) M_out[k * n + i] = M[k];
  if (bias_out)
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) bias_out[j * n + i] = bias[j];
  if (qacc_out)
#pragma unroll
    for (int j = 0; j < SO_NJ; j++) qacc_out[j * n + i] = a[j];
  if (kin_out) {
    KinOut<float> ko;
    task_kinematics<float, true>(C.dyn, C.kin, s, c, ko);
#pragma unroll
    for (int k = 0; k < 3; k++) { kin_out[k * n + i] = ko.end_pos[k]; kin_out[(3 + k) * n + i] = ko.wrist[k]; kin_out[(6 + k) * n + i] = ko.cam_pos[k]; }
#pragma unroll
    for (int k = 0; k < 9; k++) kin_out[(9 + k) * n + i] = ko.cam_R[k];
  }
}

// FP32 peak probe: 8 independent FFMA chains per thread, operands in registers
__global__ void __launch_bounds__(256) ffma_peak_kernel(float* out, int iters, float a, float b) {
  float x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
  for (int i = 0; i < iters; i++) {
#pragma unroll
    for (int k = 0; k < 16; k++) {
      x0 = fmaf(x0, a, b); x1 = fmaf(x1, a, b); x2 = fmaf(x2, a, b); x3 = fmaf(x3, a, b);
      x4 = fmaf(x4, a, b); x5 = fmaf(x5, a, b); x6 = fmaf(x6, a, b); x7 = fmaf(x7, a, b);
    }
  }
  float s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
  if (s == 12345.678f) out[0] = s;  // never true in practice; keeps the chains alive
}

// ------------------------------------------------------------------------------------------------ host: model -> constants
namespace {

struct V3 { double v[3]; };
void qnorm(const double* q, double* o) {
  double n = std::sqrt(q[0] * q[0] + q[1] * q[1] + q[2] * q[2] + q[3] * q[3]);
  for (int i = 0; i < 4; i++) o[i] = q[i] / n;
}
void q2m(const double* q, double* R) {
  double w = q[0], x = q[1], y = q[2], z = q[3];
  R[0] = w * w + x * x - y * y - z * z; R[1] = 2 * (x * y - w * z); R[2] = 2 * (x * z + w * y);
  R[3] = 2 * (x * y + w * z); R[4] = w * w - x * x + y * y - z * z; R[5] = 2 * (y * z - w * x);
  R[6] = 2 * (x * z - w * y); R[7] = 2 * (y * z + w * x); R[8] = w * w - x * x - y * y + z * z;
}
void mmul(const double* A, const double* B, double* o) {
  double r[9];
  for (int i = 0; i < 3; i++)
    for (int j = 0; j < 3; j++) r[3 * i + j] = A[3 * i] * B[j] + A[3 * i + 1] * B[3 + j] + A[3 * i + 2] * B[6 + j];
  memcpy(o, r, sizeof r);
}
void mtrans(const double* A, double* o) {
  double r[9];
  for (int i = 0; i < 3; i++) for (int j = 0; j < 3; j++) r[3 * i + j] = A[3 * j + i];
  memcpy(o, r, sizeof r);
}
void mvec(const double* A, const double* v, double* o) {
  double r[3];
  for (int i = 0; i < 3; i++) r[i] = A[3 * i] * v[0] + A[3 * i + 1] * v[1] + A[3 * i + 2] * v[2];
  memcpy(o, r, sizeof r);
}
// proper rotation P with P e_z = axis (columns a, b, axis)
bool axis_frame(const double* ax_in, double* P) {
  double n = std::sqrt(ax_in[0] * ax_in[0] + ax_in[1] * ax_in[1] + ax_in[2] * ax_in[2]);
  if (!(n > 1e-12)) return false;
  double u[3] = {ax_in[0] / n, ax_in[1] / n, ax_in[2] / n};
  // exact cyclic permutations for coordinate axes keep the constants free of rounding noise
  if (u[0] == 1 && u[1] == 0 && u[2] == 0) { double Q[9] = {0, 0, 1, 1, 0, 0, 0, 1, 0}; memcpy(P, Q, sizeof Q); return true; }
  if (u[0] == 0 && u[1] == 1 && u[2] == 0) { double Q[9] = {0, 1, 0, 0, 0, 1, 1, 0, 0}; memcpy(P, Q, sizeof Q); return true; }
  if (u[0] == 0 && u[1] == 0 && u[2] == 1) { double Q[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1}; memcpy(P, Q, sizeof Q); return true; }
  double t[3] = {1, 0, 0};
  if (std::fabs(u[0]) > 0.9) { t[0] = 0; t[1] = 1; }
  double d = t[0] * u[0] + t[1] * u[1] + t[2] * u[2];
  double a[3] = {t[0] - d * u[0], t[1] - d * u[1], t[2] - d * u[2]};
  double an = std::sqrt(a[0] * a[0] + a[1] * a[1] + a[2] * a[2]);
  for (int k = 0; k < 3; k++) a[k] /= an;
  double b[3] = {u[1] * a[2] - u[2] * a[1], u[2] * a[0] - u[0] * a[2], u[0] * a[1] - u[1] * a[0]};
  for (int r = 0; r < 3; r++) { P[3 * r] = a[r]; P[3 * r + 1] = b[r]; P[3 * r + 2] = u[r]; }
  return true;
}

struct HostModel {
  DynC<double> dyn;
  ConC<double> con;
  KinC<double> kin;
  PadC<double> pad;
  double dof_M0[SO_NJ], kv[SO_NJ], invw[SO_NJ], body_tran[SO_NJ];
};

template <typename A, typename B>
void cast_arr(const A* a, B* b, int n) { for (int i = 0; i < n; i++) b[i] = (B)a[i]; }
void cast_pad(const PadC<double>& s, PadC<float>& d) {
  d.n = s.n;
  memcpy(d.first, s.first, sizeof d.first);
  cast_arr(&s.p[0][0], &d.p[0][0], SO_MAX_PAD * 3); cast_arr(&s.A[0][0], &d.A[0][0], SO_MAX_PAD * 9); cast_arr(s.diag, d.diag, SO_MAX_PAD);
  d.K = (float)s.K; d.B = (float)s.B; d.mu = (float)s.mu;
  d.imp0 = (float)s.imp0; d.imp1 = (float)s.imp1; d.imp_w = (float)s.imp_w; d.imp_rw = (float)s.imp_rw; d.imp_mid = (float)s.imp_mid;
  d.imp_rmid = (float)s.imp_rmid; d.imp_r1mid = (float)s.imp_r1mid; d.imp_pow = (float)s.imp_pow;
}

int build_host_model(const so100_model& m, HostModel& H) {
  double Pprev[9] = {1, 0, 0, 0, 1, 0, 0, 0, 1};
  double Pall[SO_NJ][9];
  for (int i = 0; i < SO_NJ; i++) {
    double P[9], Pt[9], bq[4], Rfix[9], T[9];
    if (!axis_frame(m.jnt_axis[i], P)) return fail(SO100_ERR_MODEL, "joint axis of zero length");
    memcpy(Pall[i], P, sizeof P);
    qnorm(m.body_quat[i], bq);
    q2m(bq, Rfix);
    mtrans(Pprev, Pt);
    mmul(Pt, Rfix, T);
    mmul(T, P, H.dyn.L[i].R);              // R' = P_{i-1}^T Rfix P_i
    mvec(Pt, m.body_pos[i], H.dyn.L[i].p);  // p' = P_{i-1}^T p
    // inertia about the COM in the re-based child frame, then about the joint origin
    double iq[4], Riq[9], A[9], At[9], Ic[9], D[9] = {0}, com[3];
    qnorm(m.body_iquat[i], iq);
    q2m(iq, Riq);
    mtrans(P, Pt);
    mmul(Pt, Riq, A);
    D[0] = m.body_inertia[i][0]; D[4] = m.body_inertia[i][1]; D[8] = m.body_inertia[i][2];
    mmul(A, D, T);
    mtrans(A, At);
    mmul(T, At, Ic);
    mvec(Pt, m.body_ipos[i], com);
    double mass = m.body_mass[i], c2 = com[0] * com[0] + com[1] * com[1] + com[2] * com[2];
    if (!(mass > 0)) return fail(SO100_ERR_MODEL, "body mass must be positive");
    LinkC<double>& L = H.dyn.L[i];
    L.m = mass;
    for (int k = 0; k < 3; k++) L.h[k] = mass * com[k];
    L.I[0] = Ic[0] + mass * (c2 - com[0] * com[0]);
    L.I[1] = Ic[4] + mass * (c2 - com[1] * com[1]);
    L.I[2] = Ic[8] + mass * (c2 - com[2] * com[2]);
    L.I[3] = Ic[1] - mass * com[0] * com[1];
    L.I[4] = Ic[2] - mass * com[0] * com[2];
    L.I[5] = Ic[5] - mass * com[1] * com[2];
    L.arm = m.jnt_armature[i];
    memcpy(Pprev, P, sizeof P);
  }
  double bq[4], Rb[9], Rbt[9], g[3] = {-m.gravity[0], -m.gravity[1], -m.gravity[2]};
  qnorm(m.base_quat, bq);
  q2m(bq, Rb);
  mtrans(Rb, Rbt);
  mvec(Rbt, g, H.dyn.a0);
  memcpy(H.kin.base_R, Rb, sizeof Rb);
  memcpy(H.kin.base_p, m.base_pos, sizeof(double) * 3);
  if (m.ee_body < 0 || m.ee_body >= SO_NJ || m.wrist_body < 0 || m.wrist_body >= SO_NJ || m.cam_body < 0 || m.cam_body >= SO_NJ)
    return fail(SO100_ERR_MODEL, "ee_body / wrist_body / cam_body out of range");
  H.kin.ee_body = m.ee_body; H.kin.wrist_body = m.wrist_body; H.kin.cam_body = m.cam_body;
  double Pt[9], cq[4], Rc[9];
  mtrans(Pall[m.ee_body], Pt);
  mvec(Pt, m.ee_offset, H.kin.ee_off);
  mtrans(Pall[m.cam_body], Pt);
  mvec(Pt, m.cam_pos, H.kin.cam_pos);
  qnorm(m.cam_quat, cq);
  q2m(cq, Rc);
  mmul(Pt, Rc, H.kin.cam_R);

  // mj_setConst analogue at qpos0 = 0: dof_M0, dof_invweight0 (diag of M^-1), kv from dampratio
  double s0[SO_NJ] = {0}, c0[SO_NJ] = {1, 1, 1, 1, 1, 1}, v0[SO_NJ] = {0}, bias[SO_NJ], Mp[21], Mf[36], Lc[36] = {0};
  dyn_bias_mass<double>(H.dyn, s0, c0, v0, bias, Mp);
  for (int i = 0; i < SO_NJ; i++) for (int j = 0; j <= i; j++) Mf[i * 6 + j] = Mf[j * 6 + i] = Mp[midx(i, j)];
  for (int j = 0; j < SO_NJ; j++) {
    double d = Mf[j * 6 + j];
    for (int k = 0; k < j; k++) d -= Lc[j * 6 + k] * Lc[j * 6 + k];
    if (!(d > 0)) return fail(SO100_ERR_MODEL, "mass matrix at qpos0 is not positive definite");
    Lc[j * 6 + j] = std::sqrt(d);
    for (int i = j + 1; i < SO_NJ; i++) {
      double sv = Mf[i * 6 + j];
      for (int k = 0; k < j; k++) sv -= Lc[i * 6 + k] * Lc[j * 6 + k];
      Lc[i * 6 + j] = sv / Lc[j * 6 + j];
    }
  }
  for (int j = 0; j < SO_NJ; j++) {
    double y[SO_NJ], x[SO_NJ];
    for (int i = 0; i < SO_NJ; i++) {
      double sv = (i == j) ? 1.0 : 0.0;
      for (int k = 0; k < i; k++) sv -= Lc[i * 6 + k] * y[k];
      y[i] = sv / Lc[i * 6 + i];
    }
    for (int i = SO_NJ - 1; i >= 0; i--) {
      double sv = y[i];
      for (int k = i + 1; k < SO_NJ; k++) sv -= Lc[k * 6 + i] * x[k];
      x[i] = sv / Lc[i * 6 + i];
    }
    H.invw[j] = x[j];
    H.dof_M0[j] = Mf[j * 6 + j];
    H.kv[j] = m.act_dampratio[j] > 0 ? m.act_dampratio[j] * 2 * std::sqrt(m.act_kp[j] * H.dof_M0[j]) : m.act_kv[j];
  }
  // constraint constants (SURVEY B.6)
  for (int j = 0; j < SO_NJ; j++) {
    auto kb = [&](const double* solref, const double* solimp, double& K, double& Bv) {
      double tc = solref[0], dr = solref[1], dmax = solimp[1];
      if (tc > 0) {
        if (tc < 2 * m.timestep) tc = 2 * m.timestep;  // refsafe
        K = 1.0 / std::fmax(1e-15, dmax * dmax * tc * tc * dr * dr);
        Bv = 2.0 / std::fmax(1e-15, dmax * tc);
      } else { K = -solref[0] / (dmax * dmax); Bv = -solref[1] / dmax; }
    };
    double K, Bv;
    kb(m.dof_solref_friction[j], m.dof_solimp_friction[j], K, Bv);
    const double* si = m.dof_solimp_friction[j];
    double imp = (si[0] == si[1] || si[2] <= 1e-15) ? 0.5 * (si[0] + si[1]) : si[0];  // impedance at pos = 0
    double Rf = std::fmax(1e-15, (1 - imp) / imp * H.invw[j]);
    H.con.fr_D[j] = 1.0 / Rf; H.con.fr_B[j] = Bv; H.con.fr_loss[j] = m.jnt_frictionloss[j] > 0 ? m.jnt_frictionloss[j] : 0.0;
    kb(m.jnt_solref_limit[j], m.jnt_solimp_limit[j], K, Bv);
    H.con.lim_B[j] = Bv; H.con.lim_K[j] = K; H.con.invw[j] = H.invw[j];
    H.con.lo[j] = m.jnt_range[j][0]; H.con.hi[j] = m.jnt_range[j][1];
    if (!(H.con.hi[j] > H.con.lo[j])) return fail(SO100_ERR_MODEL, "joint range must have hi > lo");
    const double* sl = m.jnt_solimp_limit[j];
    H.con.imp0[j] = sl[0]; H.con.imp1[j] = sl[1]; H.con.imp_w[j] = sl[2]; H.con.imp_mid[j] = sl[3]; H.con.imp_pow[j] = sl[4];
    H.con.imp_rw[j] = sl[2] > 1e-15 ? 1.0 / sl[2] : 0.0;
    H.con.imp_rmid[j] = sl[3] > 0 ? 1.0 / sl[3] : 0.0;
    H.con.imp_r1mid[j] = sl[3] < 1 ? 1.0 / (1.0 - sl[3]) : 0.0;
  }
  // body_invweight0 (mj_setConst): mean diagonal of Jv M^-1 Jv^T, Jv = translational Jacobian of the link COM at qpos0
  {
    double W[9], o[3], zax[SO_NJ][3], org[SO_NJ][3];
    memcpy(W, H.kin.base_R, sizeof W);
    memcpy(o, H.kin.base_p, sizeof o);
    for (int i = 0; i < SO_NJ; i++) {  // q = 0: every joint rotation is the identity
      const LinkC<double>& L = H.dyn.L[i];
      double t[3];
      mvec(W, L.p, t);
      for (int k = 0; k < 3; k++) o[k] += t[k];
      mmul(W, L.R, W);
      for (int k = 0; k < 3; k++) { zax[i][k] = W[3 * k + 2]; org[i][k] = o[k]; }
      double com_l[3] = {L.h[0] / L.m, L.h[1] / L.m, L.h[2] / L.m}, com[3];
      mvec(W, com_l, com);
      for (int k = 0; k < 3; k++) com[k] += o[k];
      double tr = 0;
      for (int cidx = 0; cidx < 3; cidx++) {
        double Jr[SO_NJ] = {0}, y[SO_NJ], x[SO_NJ];
        for (int j = 0; j <= i; j++) {
          double d[3] = {com[0] - org[j][0], com[1] - org[j][1], com[2] - org[j][2]};
          double col[3] = {zax[j][1] * d[2] - zax[j][2] * d[1], zax[j][2] * d[0] - zax[j][0] * d[2], zax[j][0] * d[1] - zax[j][1] * d[0]};
          Jr[j] = col[cidx];
        }
        for (int a = 0; a < SO_NJ; a++) {
          double sv = Jr[a];
          for (int k = 0; k < a; k++) sv -= Lc[a * 6 + k] * y[k];
          y[a] = sv / Lc[a * 6 + a];
        }
        for (int a = SO_NJ - 1; a >= 0; a--) {
          double sv = y[a];
          for (int k = a + 1; k < SO_NJ; k++) sv -= Lc[k * 6 + a] * x[k];
          x[a] = sv / Lc[a * 6 + a];
        }
        for (int j = 0; j < SO_NJ; j++) tr += Jr[j] * x[j];
      }
      H.body_tran[i] = std::fmax(1e-15, tr / 3);
    }
  }
  // arm <-> floor pads in the re-based link frames, sorted by link; pair parameters mixed like mj_contactParam
  // (equal priority and solmix: mean solref / solimp, max friction) and clamped like getsolparam
  {
    PadC<double>& Pd = H.pad;
    memset(&Pd, 0, sizeof Pd);
    if (m.n_pad < 0 || m.n_pad > SO_MAX_PAD) return fail(SO100_ERR_MODEL, "n_pad out of range");
    double solref[2], solimp[5];
    for (int i = 0; i < 2; i++) solref[i] = 0.5 * (m.pad_solref[i] + m.floor_solref[i]);
    for (int i = 0; i < 5; i++) solimp[i] = 0.5 * (m.pad_solimp[i] + m.floor_solimp[i]);
    solimp[0] = std::fmin(0.9999, std::fmax(0.0001, solimp[0]));
    solimp[1] = std::fmin(0.9999, std::fmax(0.0001, solimp[1]));
    solimp[2] = std::fmax(0.0, solimp[2]);
    solimp[3] = std::fmin(0.9999, std::fmax(0.0001, solimp[3]));
    solimp[4] = std::fmax(1.0, solimp[4]);
    const double mu = std::fmax(m.pad_friction, m.floor_friction);
    double tc = solref[0], dr = solref[1], dmax = solimp[1];
    if (tc > 0) {
      if (tc < 2 * m.timestep) tc = 2 * m.timestep;  // refsafe
      Pd.K = 1.0 / std::fmax(1e-15, dmax * dmax * tc * tc * dr * dr);
      Pd.B = 2.0 / std::fmax(1e-15, dmax * tc);
    } else { Pd.K = -solref[0] / (dmax * dmax); Pd.B = -solref[1] / dmax; }
    Pd.mu = mu;
    Pd.imp0 = solimp[0]; Pd.imp1 = solimp[1]; Pd.imp_w = solimp[2]; Pd.imp_mid = solimp[3]; Pd.imp_pow = solimp[4];
    Pd.imp_rw = solimp[2] > 1e-15 ? 1.0 / solimp[2] : 0.0;
    Pd.imp_rmid = 1.0 / solimp[3];
    Pd.imp_r1mid = 1.0 / (1.0 - solimp[3]);
    int k = 0;
    for (int i = 0; i < SO_NJ; i++) {
      Pd.first[i] = k;
      for (int q = 0; q < m.n_pad; q++) {
        if (m.pad_body[q] < 0 || m.pad_body[q] >= SO_NJ) return fail(SO100_ERR_MODEL, "pad_body out of range");
        if (m.pad_body[q] != i) continue;
        if (!(m.pad_size[q][0] > 0 && m.pad_size[q][1] > 0 && m.pad_size[q][2] > 0) || !(mu > 0)) return fail(SO100_ERR_MODEL, "pad sizes and friction must be positive");
        double Pt[9];
        mtrans(Pall[i], Pt);
        mvec(Pt, m.pad_pos[q], Pd.p[k]);
        for (int a = 0; a < 3; a++)
          for (int r = 0; r < 3; r++) Pd.A[k][3 * r + a] = Pt[3 * r + a] * m.pad_size[q][a];  // P^T e_a size_a
        Pd.diag[k] = 2 * mu * mu * (1 + mu * mu) * H.body_tran[i];
        k++;
      }
    }
    Pd.first[SO_NJ] = k;
    Pd.n = k;
  }
  return SO100_OK;
}

// fp64 -> fp32 physics constants as the kernels consume them (link constants, task kinematics, pads)
void physics_constants_f32(const HostModel& H, Consts& C) {
  for (int i = 0; i < SO_NJ; i++) {
    const LinkC<double>& s = H.dyn.L[i];
    LinkC<float>& d = C.dyn.L[i];
    cast_arr(s.R, d.R, 9); cast_arr(s.p, d.p, 3); cast_arr(s.h, d.h, 3); cast_arr(s.I, d.I, 6);
    d.m = (float)s.m; d.arm = (float)s.arm;
  }
  cast_arr(H.dyn.a0, C.dyn.a0, 3);
  cast_arr(H.kin.base_R, C.kin.base_R, 9); cast_arr(H.kin.base_p, C.kin.base_p, 3);
  cast_arr(H.kin.ee_off, C.kin.ee_off, 3); cast_arr(H.kin.cam_pos, C.kin.cam_pos, 3); cast_arr(H.kin.cam_R, C.kin.cam_R, 9);
  C.kin.ee_body = H.kin.ee_body; C.kin.wrist_body = H.kin.wrist_body; C.kin.cam_body = H.kin.cam_body;
  cast_pad(H.pad, C.pad);
}

// fp32 solver / servo constants exactly as the kernels consume them (also what so100_dyn_gen.cuh bakes in)
void solver_constants_f32(const so100_model& m, const HostModel& H, ConC<float>& K, ActC<float>& A, BlkC<float>& Bk) {
#define CASTF(f) cast_arr(H.con.f, K.f, SO_NJ)
  CASTF(fr_D); CASTF(fr_B); CASTF(fr_loss); CASTF(lo); CASTF(hi); CASTF(lim_B); CASTF(lim_K); CASTF(invw);
  CASTF(imp0); CASTF(imp1); CASTF(imp_w); CASTF(imp_mid); CASTF(imp_pow); CASTF(imp_rw); CASTF(imp_rmid); CASTF(imp_r1mid);
#undef CASTF
  for (int j = 0; j < SO_NJ; j++) {
    A.kp[j] = (float)m.act_kp[j]; A.kv[j] = (float)H.kv[j];
    A.ctrl_lo[j] = (float)m.act_ctrlrange[j][0]; A.ctrl_hi[j] = (float)m.act_ctrlrange[j][1];
    A.frc_lo[j] = (float)m.act_forcerange[j][0]; A.frc_hi[j] = (float)m.act_forcerange[j][1];
  }
  A.h = (float)m.timestep;
  // block <-> floor contact (csrc/so100_dyn.cuh:block_substep; MuJoCo semantics in DESIGN.md "Block-floor contact")
  {
    double tc = m.contact_solref[0], dr = m.contact_solref[1], dmax = m.contact_solimp[1], Kc, Bc;
    if (tc > 0) {
      if (tc < 2 * m.timestep) tc = 2 * m.timestep;  // refsafe
      Kc = 1.0 / std::fmax(1e-15, dmax * dmax * tc * tc * dr * dr);
      Bc = 2.0 / std::fmax(1e-15, dmax * tc);
    } else { Kc = -m.contact_solref[0] / (dmax * dmax); Bc = -m.contact_solref[1] / dmax; }
    const double mu = m.block_friction, rows = 4.0 * (m.block_ncon > 0 ? m.block_ncon : 0);
    const double* si = m.contact_solimp;
    Bk.half_z = (float)m.block_half_z; Bk.gz = (float)m.gravity[2]; Bk.K = (float)Kc; Bk.B = (float)Bc;
    Bk.lam_scale = (float)(mu > 0 ? rows / (2 * mu * mu * (1 + mu * mu)) : 0.0);
    Bk.imp0 = (float)si[0]; Bk.imp1 = (float)si[1]; Bk.imp_w = (float)si[2]; Bk.imp_mid = (float)si[3]; Bk.imp_pow = (float)si[4];
    Bk.imp_rw = (float)(si[2] > 1e-15 ? 1.0 / si[2] : 0.0);
    Bk.imp_rmid = (float)(si[3] > 0 ? 1.0 / si[3] : 0.0);
    Bk.imp_r1mid = (float)(si[3] < 1 ? 1.0 / (1.0 - si[3]) : 0.0);
  }
}
static_assert(sizeof(ConC<float>) == 16 * SO_NJ * 4 && sizeof(ActC<float>) == (6 * SO_NJ + 1) * 4 && sizeof(BlkC<float>) == 13 * 4, "flat float layout");
constexpr int kNSolverConstants = 16 * SO_NJ + 6 * SO_NJ + 1 + 13;
void flatten_solver(const ConC<float>& K, const ActC<float>& A, const BlkC<float>& Bk, float* out) {
  memcpy(out, &K, sizeof K);
  memcpy(out + 16 * SO_NJ, &A, sizeof A);
  memcpy(out + 16 * SO_NJ + 6 * SO_NJ + 1, &Bk, sizeof Bk);
}

}  // namespace

// Host emulation of physics<>'s substep loop with the generic templates, in T = float (what the generic kernel
// computes, incl. the compensated position sum) or T = double.  No GPU needed: the CPU-side development and test
// vehicle of the contact path.  stats: [0] contact substeps, [1] gradient/Hessian evaluations, [2] line-search
// evaluations, [3] largest evaluation count of one solve, [4] unconverged solves.
// The cooperative solve on the host (fp32 only; kNoCoop: not applicable - fp64 emulation, > kCoopCon corners, or
// SO100_HOST_SERIAL_CONTACT set - and the caller takes the serial solve).
constexpr int kNoCoop = INT_MIN;
static int host_coop_solve(const DynC<double>&, const KinC<double>&, const PadC<double>&, const ConC<double>&, ContactIO<double>&, unsigned, int*) { return kNoCoop; }
static int host_coop_solve(const DynC<float>& D, const KinC<float>& Kn, const PadC<float>& P, const ConC<float>& K, ContactIO<float>& io, unsigned touch,
                           int* nls) {
  static const bool serial = getenv("SO100_HOST_SERIAL_CONTACT") != nullptr;
  if (serial) return kNoCoop;
  float sf[CoopSlot::kFloats];
  double sd[CoopSlot::kDoubles];
  memset(sf, 0, sizeof sf); memset(sd, 0, sizeof sd);
  const CoopSlot S{sf, sd};
  const int nc = coop_fill(D, Kn, P, K, K.fr_loss, S, io.s, io.c, io.q, io.qc, io.qd, io.M, io.b, io.a, touch);
  if (nc < 0) return kNoCoop;
  if (nc == 0) return 0;
  const int st = coop_solve_host(S, nls);
  for (int j = 0; j < SO_NJ; j++) io.a[j] = (float)S.D(CoopSlot::kX + j);
  return st;
}

template <typename T>
static void host_substeps_t(const DynC<T>& D, const KinC<T>& Kn, const PadC<T>& P, const ConC<T>& K, const ActC<T>& A, int n, double* qpos,
                            double* qvel, double* warm, const double* ctrl, int nsub, int64_t* stats, bool coarse_sincos = false) {
  for (int i = 0; i < n; i++) {
    T q[SO_NJ], qc[SO_NJ], v[SO_NJ], w[SO_NJ], cc[SO_NJ];
    for (int j = 0; j < SO_NJ; j++) {
      q[j] = (T)qpos[6 * i + j]; qc[j] = (T)((double)q[j] - qpos[6 * i + j]);  // q - qc = the fp64 input
      v[j] = (T)qvel[6 * i + j]; w[j] = (T)warm[6 * i + j];
      cc[j] = (T)std::fmin(std::fmax(ctrl[6 * i + j], (double)A.ctrl_lo[j]), (double)A.ctrl_hi[j]);
    }
    for (int sub = 0; sub < nsub; sub++) {
      T s[SO_NJ], c[SO_NJ], bias[SO_NJ], M[21], b[SO_NJ];
      for (int j = 0; j < SO_NJ; j++) { s[j] = (T)std::sin((double)q[j] - (double)qc[j]); c[j] = (T)std::cos((double)q[j] - (double)qc[j]); }
      if (coarse_sincos) {  // sin/cos of the fp32 angle quantised to 2^-22: the accuracy class of MUFU.SIN / MUFU.COS (__sincosf)
        for (int j = 0; j < SO_NJ; j++) {
          s[j] = (T)(std::round(std::sin((double)q[j]) * 4194304.0) / 4194304.0);
          c[j] = (T)(std::round(std::cos((double)q[j]) * 4194304.0) / 4194304.0);
        }
      }
      dyn_bias_mass<T>(D, s, c, v, bias, M);
      for (int j = 0; j < SO_NJ; j++) {
        T f = A.kp[j] * ((cc[j] - q[j]) + qc[j]) - A.kv[j] * v[j];
        b[j] = so_clamp(f, A.frc_lo[j], A.frc_hi[j]) - bias[j];
      }
      const unsigned touch = P.n > 0 ? pads_touch<T>(D, Kn, P, s, c, sizeof(T) == 4 ? T(SO100_TOUCH_MARGIN) : T(0)) : 0u;
      bool solved = false;
      if (touch) {
        ContactIO<T> cio;
        for (int j = 0; j < SO_NJ; j++) { cio.s[j] = s[j]; cio.c[j] = c[j]; cio.q[j] = q[j]; cio.qc[j] = qc[j]; cio.qd[j] = v[j]; cio.b[j] = b[j]; cio.a[j] = w[j]; }
        // the contact geometry always gets correctly rounded sin/cos of the compensated angle (see physics<>)
        for (int j = 0; j < SO_NJ; j++) { cio.s[j] = (T)std::sin((double)q[j] - (double)qc[j]); cio.c[j] = (T)std::cos((double)q[j] - (double)qc[j]); }
        memcpy(cio.M, M, sizeof M);
        int nls = 0;
        int over = 0;
        int st = host_coop_solve(D, Kn, P, K, cio, touch, &nls);  // fp32: the device's cooperative solve, lanes in sequence
        if (st == kNoCoop) st = contact_solve<T>(D, Kn, P, K, cio, touch, &over, &nls);
        solved = st != 0;
        if (solved) memcpy(w, cio.a, sizeof w);
        if (stats && solved) {
          const int ev = st < 0 ? -st : st;
          stats[0] += 1; stats[1] += ev; stats[2] += nls;
          if (ev > stats[3]) stats[3] = ev;
          if (st < 0) stats[4] += 1;
        }
      }
      if (!solved) {
        static const int sw0 = getenv("SO100_SWEEPS0") ? atoi(getenv("SO100_SWEEPS0")) : SO100_SWEEPS_FIRST, sw1 = getenv("SO100_SWEEPS1") ? atoi(getenv("SO100_SWEEPS1")) : SO100_SWEEPS_REST;
        const T dlast = solve_qacc<T>(K, K.fr_loss, M, b, q, qc, v, w, sub == 0 ? sw0 : sw1);
        T amax = T(1);
        for (int j = 0; j < SO_NJ; j++) amax = std::fmax(amax, std::fabs(w[j]));
        if (stats && dlast > T(2e-3) * amax) stats[4] += 1;  // as physics<> counts Gauss-Seidel substeps that were still moving
      }
      for (int j = 0; j < SO_NJ; j++) {
        v[j] += A.h * w[j];
        if (sizeof(T) == 4) {  // compensated position sum, as in physics<>
          volatile T y = A.h * v[j] - qc[j];
          volatile T s1 = q[j] + y;
          volatile T t = s1 - q[j];
          qc[j] = t - y;
          q[j] = s1;
        } else q[j] += A.h * v[j];
      }
    }
    for (int j = 0; j < SO_NJ; j++) { qpos[6 * i + j] = (double)q[j] - (double)qc[j]; qvel[6 * i + j] = v[j]; warm[6 * i + j] = w[j]; }
  }
}

// ------------------------------------------------------------------------------------------------ ctx
static void flatten_dyn(const DynC<double>& D, double* out) {
  int k = 0;
  for (int i = 0; i < SO_NJ; i++) {
    const LinkC<double>& L = D.L[i];
    for (int a = 0; a < 9; a++) out[k++] = L.R[a];
    for (int a = 0; a < 3; a++) out[k++] = L.p[a];
    out[k++] = L.m;
    for (int a = 0; a < 3; a++) out[k++] = L.h[a];
    for (int a = 0; a < 6; a++) out[k++] = L.I[a];
    out[k++] = L.arm;
  }
  for (int a = 0; a < 3; a++) out[k++] = D.a0[a];
}

struct so100_ctx {
  int device = 0, n = 0, task = 0, obs_dim = 0;
  Consts C;
  HostModel H;
  Bufs B{};
  float* start_tab = nullptr;
  int64_t tick = 0, launches = 0;
  bool specialised = false;  // model == the constants baked into so100_dyn_gen.cuh
  ParamIO par{};             // per-env kernels' data; par.p == nullptr: the default kernels (neither ranges nor a sim2real config set)
  bool ranges_on = false;    // so100_set_param_ranges set (else par.p, if allocated, holds the model's constants, lo = hi = 1)
  // staging for the *_host entry points
  float *h_act = nullptr, *h_obs = nullptr, *h_rew = nullptr, *h_tobs = nullptr, *h_epr = nullptr;
  uint8_t *h_term = nullptr, *h_trunc = nullptr;
  int* h_epl = nullptr;
  // host path.  Pinned host buffers: the kernel reads the actions and writes obs / reward / flags / terminal rows
  // straight through the host link (zero-copy), one launch per call.  Pageable buffers: chunks of envs on helper
  // streams so that H2D, kernel and D2H overlap.
  static constexpr int kMaxChunks = 16;
  int n_chunks = 2;
  bool zero_copy = true;
  cudaStream_t hs[kMaxChunks] = {};
  cudaEvent_t ev_start = nullptr, ev_done[kMaxChunks] = {};
  int *d_any_done = nullptr, *p_any_done = nullptr;  // device flag + pinned host copy (the zero-copy path writes the latter)
  // env groups of the asynchronous host path (so100_host_groups / so100_step_host_async / so100_step_host_wait):
  // contiguous CTA-aligned env ranges, each with its own stream, completion event and step counter
  static constexpr int kMaxGroups = SO100_MAX_GROUPS;
  int n_groups = 1, g_lo[kMaxGroups] = {}, g_hi[kMaxGroups] = {};
  int64_t g_tick[kMaxGroups] = {};
  bool g_pending[kMaxGroups] = {};
  int g_next = 0;  // where so100_step_host_wait_any resumes its scan
  // async path: a group's action rows come in by copy engine (measured 5 % faster than loads over the link from the SMs, whose
  // read requests queue behind the other groups' posted obs writes: profiles/r2_e2e_groups.txt); obs go out as stores from
  // the kernel.  A/B knobs SO100_ASYNC_H2D_COPY / SO100_ASYNC_D2H_COPY.
  bool async_h2d_copy = true, async_d2h_copy = false;
  bool g_fork_needed[kMaxGroups] = {};  // work enqueued on a caller stream since this group's last async step (reset, set_state, ...)
  cudaStream_t gs[kMaxGroups] = {};
  cudaEvent_t g_done[kMaxGroups] = {}, g_fork = nullptr;
};

static void free_ctx(so100_ctx* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  void* ptrs[] = {c->B.qpos, c->B.qvel, c->B.warm, c->B.qcomp, c->B.block, c->B.snap, c->B.aux, c->B.ep_return, c->B.cnt, c->B.stats,
                  c->start_tab, c->par.p, c->par.latency, c->par.ctrl_prev, c->h_act, c->h_obs, c->h_rew, c->h_tobs, c->h_epr, c->h_term, c->h_trunc, c->h_epl};
  for (void* p : ptrs) if (p) cudaFree(p);
  if (c->d_any_done) cudaFree(c->d_any_done);
  if (c->p_any_done) cudaFreeHost(c->p_any_done);
  for (int k = 0; k < so100_ctx::kMaxChunks; k++) {
    if (c->hs[k]) cudaStreamDestroy(c->hs[k]);
    if (c->ev_done[k]) cudaEventDestroy(c->ev_done[k]);
  }
  if (c->ev_start) cudaEventDestroy(c->ev_start);
  for (int k = 0; k < so100_ctx::kMaxGroups; k++) {
    if (c->gs[k]) cudaStreamDestroy(c->gs[k]);
    if (c->g_done[k]) cudaEventDestroy(c->g_done[k]);
  }
  if (c->g_fork) cudaEventDestroy(c->g_fork);
  delete c;
}

static void mark_caller_stream_work(so100_ctx* c) {
  for (int g = 0; g < so100_ctx::kMaxGroups; g++) c->g_fork_needed[g] = true;
}

extern "C" {

#ifndef SO100_CSRC_HASH
#define SO100_CSRC_HASH "unknown"
#endif
int so100_abi_version(void) { return SO100_ABI_VERSION; }
const char* so100_build_id(void) { return SO100_CSRC_HASH; }
const char* so100_last_error(void) { return g_err.c_str(); }
int so100_obs_dim(int task) {
  if (task == SO100_TASK_ENV01 || task == SO100_TASK_ENV02 || task == SO100_TASK_ENV06) return 15;
  if (task == SO100_TASK_ENV05) return 8;
  return fail(SO100_ERR_ARG, "unknown task");
}
int so100_act_dim(int task) { return so100_obs_dim(task) < 0 ? SO100_ERR_ARG : SO_NJ; }

int so100_create(const so100_model* m, const so100_task_cfg* cfg, int device, so100_ctx** out) {
  if (!m || !cfg || !out) return fail(SO100_ERR_ARG, "null argument");
  *out = nullptr;
  if (m->struct_size != (int)sizeof(so100_model)) return fail(SO100_ERR_ARG, "so100_model.struct_size mismatch");
  if (cfg->struct_size != (int)sizeof(so100_task_cfg)) return fail(SO100_ERR_ARG, "so100_task_cfg.struct_size mismatch");
  if (so100_obs_dim(cfg->task) < 0) return SO100_ERR_ARG;
  if (cfg->num_envs <= 0) return fail(SO100_ERR_ARG, "num_envs must be positive");
  if (cfg->max_episode_steps <= 0) return fail(SO100_ERR_ARG, "max_episode_steps must be positive");
  if (cfg->task == SO100_TASK_ENV01 && (cfg->n_start <= 0 || cfg->n_start > kMaxStart)) return fail(SO100_ERR_ARG, "n_start out of range");
  if (m->nsubstep <= 0 || !(m->timestep > 0)) return fail(SO100_ERR_MODEL, "nsubstep / timestep must be positive");
  if (!(m->block_mass > 0) || !(m->block_half_z > 0) || m->block_ncon < 0) return fail(SO100_ERR_MODEL, "block mass / half size must be positive");
  int ndev = 0;
  CU(cudaGetDeviceCount(&ndev));
  if (device < 0 || device >= ndev) return fail(SO100_ERR_ARG, "no such CUDA device");
  CU(cudaSetDevice(device));
  so100_ctx* c = new (std::nothrow) so100_ctx();
  if (!c) return fail(SO100_ERR_CUDA, "out of host memory");
  c->device = device; c->n = cfg->num_envs; c->task = cfg->task; c->obs_dim = so100_obs_dim(cfg->task);
  int rc = build_host_model(*m, c->H);
  if (rc != SO100_OK) { delete c; return rc; }
  {
    double flat[SO100_N_DYN_CONSTANTS];
    flatten_dyn(c->H.dyn, flat);
    ConC<float> K;
    ActC<float> A;
    BlkC<float> Bk;
    float sflat[kNSolverConstants];
    solver_constants_f32(*m, c->H, K, A, Bk);
    flatten_solver(K, A, Bk, sflat);
    static_assert(SO100_GEN_NS == kNSolverConstants, "so100_dyn_gen.cuh is stale: run tools/gen_so100_dyn.py");
    c->specialised = memcmp(flat, kGenDynConstants, sizeof flat) == 0 && memcmp(sflat, kGenSolverConstants, sizeof sflat) == 0 &&
                     !(cfg->flags & SO100_FLAG_GENERIC_KERNEL);
  }
  // fp64 -> fp32 constants
  Consts& C = c->C;
  memset(&C, 0, sizeof C);
  physics_constants_f32(c->H, C);
  if (!(cfg->flags & SO100_FLAG_ARM_CONTACT)) { C.pad.n = 0; for (int i = 0; i <= SO_NJ; i++) C.pad.first[i] = 0; }
  TaskC& t = C.t;
  t.task = cfg->task; t.n = cfg->num_envs; t.max_steps = cfg->max_episode_steps; t.n_start = cfg->n_start;
  t.lost_limit = cfg->lost_limit; t.nsub = m->nsubstep; t.flags = cfg->flags;
  t.contact_warps = kBlock / 32;  // measured (65 536 envs, cooperative solve): 1.375 / 1.373 / 1.340 ms with 1 / 4 / 8
  if (const char* e = getenv("SO100_CONTACT_WARPS")) { const int v = atoi(e); if (v >= 1 && v <= kBlock / 32) t.contact_warps = v; }  // tuning knob
  t.seed_lo = (unsigned)(cfg->seed & 0xFFFFFFFFull); t.seed_hi = (unsigned)(cfg->seed >> 32);
  t.env_offset = cfg->env_offset;
  t.dt_env = (float)(m->timestep * m->nsubstep); t.step_scale = (float)cfg->joint_step_scale;
  solver_constants_f32(*m, c->H, C.con, t.act, t.blk);
  for (int j = 0; j < SO_NJ; j++) {
    double lo = m->jnt_range[j][0], hi = m->jnt_range[j][1];
    t.pen_lo[j] = (float)(lo + 0.05 * (hi - lo)); t.pen_hi[j] = (float)(hi - 0.05 * (hi - lo));
    t.rest[j] = (float)cfg->rest_position[j]; t.start05[j] = (float)cfg->start_position05[j];
  }
  t.dist_lo = (float)cfg->block_dist_range[0]; t.dist_hi = (float)cfg->block_dist_range[1];
  t.theta_half = (float)cfg->block_theta_half; t.reach = (float)cfg->reach_threshold;
  for (int a = 0; a < 2; a++) for (int k = 0; k < 3; k++) { t.space_s[a][k] = (float)cfg->block_space_start[a][k]; t.space_e[a][k] = (float)cfg->block_space_end[a][k]; }
  t.speed_min = (float)cfg->block_speed_min; t.speed_max = (float)cfg->block_speed_max; t.ramp = (float)cfg->ramp_seconds;
  t.res_w = (float)cfg->cam_res_w; t.res_h = (float)cfg->cam_res_h; t.noise = (float)cfg->obs_noise;
  t.fy = (float)(0.5 * cfg->cam_res_h / std::tan(m->cam_fovy_deg * 3.14159265358979323846 / 180.0 / 2));  // env_base_02.py:100

  const size_t n = (size_t)c->n;
  auto alloc = [&](void** p, size_t bytes) -> bool {
    if (cudaMalloc(p, bytes) != cudaSuccess) return false;
    return cudaMemset(*p, 0, bytes) == cudaSuccess;
  };
  bool ok = alloc((void**)&c->B.qpos, 6 * n * 4) && alloc((void**)&c->B.qvel, 6 * n * 4) && alloc((void**)&c->B.warm, 6 * n * 4) && alloc((void**)&c->B.qcomp, 6 * n * 4) &&
            alloc((void**)&c->B.block, 4 * n * 4) && alloc((void**)&c->B.snap, kSnap * n * 4) && alloc((void**)&c->B.aux, kAux * n * 4) &&
            alloc((void**)&c->B.ep_return, n * 4) && alloc((void**)&c->B.cnt, kCnt * n * 4) && alloc((void**)&c->B.stats, 4 * 8) &&
            alloc((void**)&c->start_tab, kMaxStart * SO_NJ * 4);
  if (!ok) { std::string e = cudaGetErrorString(cudaGetLastError()); free_ctx(c); return fail(SO100_ERR_CUDA, "cudaMalloc: " + e); }
  float tab[kMaxStart * SO_NJ];
  for (int i = 0; i < kMaxStart; i++) for (int j = 0; j < SO_NJ; j++) tab[i * SO_NJ + j] = (float)cfg->start_positions[i][j];
  if (cudaMemcpy(c->start_tab, tab, sizeof tab, cudaMemcpyHostToDevice) != cudaSuccess) { free_ctx(c); return fail(SO100_ERR_CUDA, "cudaMemcpy(start table)"); }
  c->B.start_tab = c->start_tab;
  c->n_groups = 1; c->g_lo[0] = 0; c->g_hi[0] = c->n;
  {  // the contact pool is > 48 KB of dynamic shared memory: opt in, per device, for this task's step kernels
    cudaError_t e1 = cudaSuccess, e2 = cudaSuccess;
#define SO100_OPT(T)                                                                                                              \
  e1 = cudaFuncSetAttribute(step_kernel<T, true, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPoolBytes);  \
  e2 = cudaFuncSetAttribute(step_kernel<T, false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPoolBytes); \
  if (e1 == cudaSuccess) e1 = cudaFuncSetAttribute(step_kernel<T, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPoolBytes); \
  if (e2 == cudaSuccess) e2 = cudaFuncSetAttribute(step_kernel<T, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kPoolBytes)
    switch (c->task) {
      case 1: SO100_OPT(1); break;
      case 2: SO100_OPT(2); break;
      case 6: SO100_OPT(6); break;
      default: SO100_OPT(5); break;
    }
#undef SO100_OPT
    if (e1 != cudaSuccess || e2 != cudaSuccess) { free_ctx(c); return fail(SO100_ERR_CUDA, "cudaFuncSetAttribute(MaxDynamicSharedMemorySize)"); }
  }
  *out = c;
  return SO100_OK;
}

void so100_destroy(so100_ctx* ctx) { free_ctx(ctx); }

static inline int grid_for(int n) { return (n + kBlock - 1) / kBlock; }

int so100_reset(so100_ctx* c, const uint8_t* mask_dev, float* obs_dev, void* stream) {
  if (!c || !obs_dev) return fail(SO100_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  unsigned tick = (unsigned)c->tick;
  switch (c->task) {
    case 1: reset_kernel<1><<<grid_for(c->n), kBlock, 0, st>>>(c->C, c->B, mask_dev, obs_dev, tick, c->par); break;
    case 2: reset_kernel<2><<<grid_for(c->n), kBlock, 0, st>>>(c->C, c->B, mask_dev, obs_dev, tick, c->par); break;
    case 6: reset_kernel<6><<<grid_for(c->n), kBlock, 0, st>>>(c->C, c->B, mask_dev, obs_dev, tick, c->par); break;
    default: reset_kernel<5><<<grid_for(c->n), kBlock, 0, st>>>(c->C, c->B, mask_dev, obs_dev, tick, c->par); break;
  }
  c->launches++;
  mark_caller_stream_work(c);
  CU(cudaGetLastError());
  return SO100_OK;
}

static int launch_step(so100_ctx* c, const StepIO& io, cudaStream_t st) {
  const int g = grid_for(io.env_hi - io.env_lo);
  const bool pads = c->C.pad.n > 0;
  const size_t dyn = pads ? kPoolBytes : 0;
  // three variants per task: model-specialised without / with the arm-floor contact path, and the generic one (any model, with it);
  // each again with per-env dynamics parameters while ranges are set
#define SO100_VARIANTS(T, P)                                                                                  \
  do {                                                                                                        \
    if (c->specialised && !pads) step_kernel<T, true, false, P><<<g, kBlock, 0, st>>>(c->C, c->B, io, c->par);        \
    else if (c->specialised) step_kernel<T, true, true, P><<<g, kBlock, dyn, st>>>(c->C, c->B, io, c->par);           \
    else step_kernel<T, false, true, P><<<g, kBlock, dyn, st>>>(c->C, c->B, io, c->par);                              \
  } while (0)
#define SO100_LAUNCH(T)                     \
  do {                                      \
    if (c->par.p) SO100_VARIANTS(T, true);  \
    else SO100_VARIANTS(T, false);          \
  } while (0)
  switch (c->task) {
    case 1: SO100_LAUNCH(1); break;
    case 2: SO100_LAUNCH(2); break;
    case 6: SO100_LAUNCH(6); break;
    default: SO100_LAUNCH(5); break;
  }
#undef SO100_LAUNCH
#undef SO100_VARIANTS
  c->launches++;
  CU(cudaGetLastError());
  return SO100_OK;
}

// a full step needs every env group at the same step count (they share the RNG tick)
static int groups_in_step(so100_ctx* c) {
  for (int g = 0; g < c->n_groups; g++) {
    if (c->g_pending[g]) return fail(SO100_ERR_STATE, "an asynchronous group step is in flight: call so100_step_host_wait first");
    if (c->g_tick[g] != c->tick) return fail(SO100_ERR_STATE, "env groups are at different step counts: advance the lagging groups first");
  }
  return SO100_OK;
}
static void set_all_ticks(so100_ctx* c, int64_t tick) {
  c->tick = tick;
  for (int g = 0; g < so100_ctx::kMaxGroups; g++) c->g_tick[g] = tick;
}

int so100_step(so100_ctx* c, const float* actions_dev, float* obs_dev, float* reward_dev, uint8_t* terminated_dev,
               uint8_t* truncated_dev, float* terminal_obs_dev, float* ep_return_dev, int32_t* ep_len_dev, void* stream) {
  if (!c || !actions_dev || !obs_dev || !reward_dev || !terminated_dev || !truncated_dev) return fail(SO100_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  if (int rc = groups_in_step(c)) return rc;
  set_all_ticks(c, c->tick + 1);
  StepIO io{actions_dev, obs_dev, reward_dev, terminal_obs_dev, ep_return_dev, terminated_dev, truncated_dev, ep_len_dev, (unsigned)c->tick, 0, c->n, nullptr};
  mark_caller_stream_work(c);
  return launch_step(c, io, st);
}

int so100_step_substeps(so100_ctx* c, const float* ctrl_dev, int n_substeps, void* stream) {
  if (!c || !ctrl_dev || n_substeps <= 0) return fail(SO100_ERR_ARG, "bad argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  const int g = grid_for(c->n);
#define SO100_SUBSTEPS(T, S)                                                                                   \
  do {                                                                                                         \
    if (c->par.p) substeps_kernel<T, S, true><<<g, kBlock, 0, st>>>(c->C, c->B, ctrl_dev, n_substeps, c->par.p); \
    else substeps_kernel<T, S, false><<<g, kBlock, 0, st>>>(c->C, c->B, ctrl_dev, n_substeps, nullptr);        \
  } while (0)
  switch (c->task) {  // a debug entry: always the generic recursion (the same mathematics; csrc/so100_dyn.cuh)
    case 1: SO100_SUBSTEPS(1, false); break;
    case 2: SO100_SUBSTEPS(2, false); break;
    case 6: SO100_SUBSTEPS(6, false); break;
    default: SO100_SUBSTEPS(5, false); break;
  }
#undef SO100_SUBSTEPS
  mark_caller_stream_work(c);
  c->launches++;
  CU(cudaGetLastError());
  return SO100_OK;
}

static int ensure_staging(so100_ctx* c) {
  if (c->h_act) return SO100_OK;
  size_t n = (size_t)c->n, od = (size_t)c->obs_dim;
  CU(cudaMalloc((void**)&c->h_act, n * SO_NJ * 4));
  CU(cudaMalloc((void**)&c->h_obs, n * od * 4));
  CU(cudaMalloc((void**)&c->h_tobs, n * od * 4));
  CU(cudaMalloc((void**)&c->h_rew, n * 4));
  CU(cudaMalloc((void**)&c->h_epr, n * 4));
  CU(cudaMalloc((void**)&c->h_epl, n * 4));
  CU(cudaMalloc((void**)&c->h_term, n));
  CU(cudaMalloc((void**)&c->h_trunc, n));
  CU(cudaMalloc((void**)&c->d_any_done, sizeof(int)));
  CU(cudaMallocHost((void**)&c->p_any_done, sizeof(int)));
  if (const char* e = getenv("SO100_HOST_ZEROCOPY")) c->zero_copy = atoi(e) != 0;  // A/B knob (default on)
  if (const char* e = getenv("SO100_HOST_CHUNKS")) {  // tuning knob of the host path (default 2: measured best of 1..8, profiles/r1_e2e_chunks.txt)
    int v = atoi(e);
    if (v >= 1 && v <= so100_ctx::kMaxChunks) c->n_chunks = v;
  }
  for (int k = 0; k < so100_ctx::kMaxChunks; k++) {
    CU(cudaStreamCreateWithFlags(&c->hs[k], cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&c->ev_done[k], cudaEventDisableTiming));
  }
  CU(cudaEventCreateWithFlags(&c->ev_start, cudaEventDisableTiming));
  for (int k = 0; k < so100_ctx::kMaxGroups; k++) {
    CU(cudaStreamCreateWithFlags(&c->gs[k], cudaStreamNonBlocking));
    CU(cudaEventCreateWithFlags(&c->g_done[k], cudaEventDisableTiming));
  }
  CU(cudaEventCreateWithFlags(&c->g_fork, cudaEventDisableTiming));
  if (const char* e = getenv("SO100_ASYNC_H2D_COPY")) c->async_h2d_copy = atoi(e) != 0;
  if (const char* e = getenv("SO100_ASYNC_D2H_COPY")) c->async_d2h_copy = atoi(e) != 0;
  return SO100_OK;
}

int so100_reset_host(so100_ctx* c, float* obs_host, void* stream) {
  if (!c || !obs_host) return fail(SO100_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  int rc = ensure_staging(c);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  rc = so100_reset(c, nullptr, c->h_obs, stream);
  if (rc) return rc;
  CU(cudaMemcpyAsync(obs_host, c->h_obs, (size_t)c->n * c->obs_dim * 4, cudaMemcpyDeviceToHost, st));
  CU(cudaStreamSynchronize(st));
  return SO100_OK;
}

// Pageable host buffers: chunked H2D -> step_kernel -> D2H pipeline, forked from `st` onto the helper streams.
static int enqueue_host_pipeline(so100_ctx* c, cudaStream_t st, const float* actions_host, float* obs_host, float* reward_host,
                                 uint8_t* terminated_host, uint8_t* truncated_host, bool want_term) {
  const size_t od = (size_t)c->obs_dim;
  // chunks are multiples of the CTA size; small batches are not worth splitting
  int nchunk = c->n >= 4 * 4096 ? c->n_chunks : 1;
  int per = ((c->n + nchunk - 1) / nchunk + kBlock - 1) / kBlock * kBlock;
  CU(cudaMemsetAsync(c->d_any_done, 0, sizeof(int), st));
  CU(cudaEventRecord(c->ev_start, st));
  for (int k = 0; k < nchunk; k++) {
    int lo = k * per, hi = lo + per < c->n ? lo + per : c->n;
    if (lo >= hi) { nchunk = k; break; }
    cudaStream_t hs = c->hs[k];
    size_t cnt = (size_t)(hi - lo);
    CU(cudaStreamWaitEvent(hs, c->ev_start, 0));
    CU(cudaMemcpyAsync(c->h_act + (size_t)lo * SO_NJ, actions_host + (size_t)lo * SO_NJ, cnt * SO_NJ * 4, cudaMemcpyHostToDevice, hs));
    StepIO io{c->h_act, c->h_obs, c->h_rew, want_term ? c->h_tobs : nullptr, want_term ? c->h_epr : nullptr, c->h_term, c->h_trunc,
              want_term ? c->h_epl : nullptr, (unsigned)c->tick, lo, hi, c->d_any_done};
    int rc = launch_step(c, io, hs);
    if (rc) return rc;
    CU(cudaMemcpyAsync(obs_host + (size_t)lo * od, c->h_obs + (size_t)lo * od, cnt * od * 4, cudaMemcpyDeviceToHost, hs));
    CU(cudaMemcpyAsync(reward_host + lo, c->h_rew + lo, cnt * 4, cudaMemcpyDeviceToHost, hs));
    CU(cudaMemcpyAsync(terminated_host + lo, c->h_term + lo, cnt, cudaMemcpyDeviceToHost, hs));
    CU(cudaMemcpyAsync(truncated_host + lo, c->h_trunc + lo, cnt, cudaMemcpyDeviceToHost, hs));
    CU(cudaEventRecord(c->ev_done[k], hs));
  }
  for (int k = 0; k < nchunk; k++) CU(cudaStreamWaitEvent(st, c->ev_done[k], 0));
  CU(cudaMemcpyAsync(c->p_any_done, c->d_any_done, sizeof(int), cudaMemcpyDeviceToHost, st));
  return SO100_OK;
}

// device-visible alias of a pinned (page-locked, mapped) host pointer, or nullptr for pageable memory
static void* mapped_alias(const void* host) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, host) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  if (a.type == cudaMemoryTypeDevice && getenv("SO100_HOST_ALLOW_DEVICE")) return a.devicePointer;  // pipeline experiments without the link
  if (a.type != cudaMemoryTypeHost || !a.devicePointer) return nullptr;
  return a.devicePointer;
}

// Device-visible aliases of one set of host buffers; ok = every mandatory buffer (and every optional one that was
// given) is page-locked and mapped, so one launch can read / write them in place.
struct HostAlias {
  const float* act; float *obs, *rew, *tobs, *epr; uint8_t *term, *trunc; int* epl; bool ok;
};
static HostAlias alias_host(const float* actions_host, float* obs_host, float* reward_host, uint8_t* terminated_host, uint8_t* truncated_host,
                            float* terminal_obs_host, float* ep_return_host, int32_t* ep_len_host) {
  HostAlias a{};
  a.act = (const float*)mapped_alias(actions_host);
  a.obs = a.act ? (float*)mapped_alias(obs_host) : nullptr;
  a.rew = a.obs ? (float*)mapped_alias(reward_host) : nullptr;
  a.term = a.rew ? (uint8_t*)mapped_alias(terminated_host) : nullptr;
  a.trunc = a.term ? (uint8_t*)mapped_alias(truncated_host) : nullptr;
  a.ok = a.trunc != nullptr;
  if (a.ok && terminal_obs_host) a.ok = (a.tobs = (float*)mapped_alias(terminal_obs_host)) != nullptr;
  if (a.ok && ep_return_host) a.ok = (a.epr = (float*)mapped_alias(ep_return_host)) != nullptr;
  if (a.ok && ep_len_host) a.ok = (a.epl = (int*)mapped_alias(ep_len_host)) != nullptr;
  return a;
}

int so100_step_host(so100_ctx* c, const float* actions_host, float* obs_host, float* reward_host, uint8_t* terminated_host,
                    uint8_t* truncated_host, float* terminal_obs_host, float* ep_return_host, int32_t* ep_len_host, void* stream) {
  if (!c || !actions_host || !obs_host || !reward_host || !terminated_host || !truncated_host) return fail(SO100_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  int rc = ensure_staging(c);
  if (rc) return rc;
  if ((rc = groups_in_step(c))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t od = (size_t)c->obs_dim;
  const bool want_term = terminal_obs_host || ep_return_host || ep_len_host;
  set_all_ticks(c, c->tick + 1);
  HostAlias z{};
  if (c->zero_copy) z = alias_host(actions_host, obs_host, reward_host, terminated_host, truncated_host, terminal_obs_host, ep_return_host, ep_len_host);
  if (z.ok) {
    // zero-copy: ONE launch.  Each CTA pulls its action rows over the host link when it starts and posts its obs /
    // reward / flag rows (and, for envs whose episode ended, the terminal rows) when it ends.  65 536 envs are a single
    // wave of CTAs, so the three phases are in series: actions in, ~85 us of arithmetic, results out; the pipelined
    // alternative is so100_step_host_async over env groups.
    StepIO io{z.act, z.obs, z.rew, z.tobs, z.epr, z.term, z.trunc, z.epl, (unsigned)c->tick, 0, c->n, nullptr};
    rc = launch_step(c, io, st);
    if (rc) return rc;
    CU(cudaStreamSynchronize(st));
    return SO100_OK;
  }
  rc = enqueue_host_pipeline(c, st, actions_host, obs_host, reward_host, terminated_host, truncated_host, want_term);
  if (rc) return rc;
  CU(cudaStreamSynchronize(st));
  if (want_term && *c->p_any_done) {  // the terminal rows are only meaningful for envs that finished: copy them only then
    size_t n = (size_t)c->n;
    if (terminal_obs_host) CU(cudaMemcpyAsync(terminal_obs_host, c->h_tobs, n * od * 4, cudaMemcpyDeviceToHost, st));
    if (ep_return_host) CU(cudaMemcpyAsync(ep_return_host, c->h_epr, n * 4, cudaMemcpyDeviceToHost, st));
    if (ep_len_host) CU(cudaMemcpyAsync(ep_len_host, c->h_epl, n * 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
  }
  return SO100_OK;
}

// ---- asynchronous host path over env groups
int so100_host_groups(so100_ctx* c, int n_groups) {
  if (!c || n_groups < 1 || n_groups > so100_ctx::kMaxGroups) return fail(SO100_ERR_ARG, "n_groups out of range");
  if (int rc = groups_in_step(c)) return rc;
  const int ctas = grid_for(c->n);
  if (n_groups > ctas) return fail(SO100_ERR_ARG, "more groups than CTAs of envs");
  for (int g = 0; g < n_groups; g++) {  // balanced, CTA-aligned, contiguous
    c->g_lo[g] = (int)((int64_t)ctas * g / n_groups) * kBlock;
    int hi = (int)((int64_t)ctas * (g + 1) / n_groups) * kBlock;
    c->g_hi[g] = hi < c->n ? hi : c->n;
  }
  c->n_groups = n_groups;
  return SO100_OK;
}
int so100_host_group_range(so100_ctx* c, int group, int* env_lo, int* env_hi) {
  if (!c || group < 0 || group >= c->n_groups) return fail(SO100_ERR_ARG, "no such env group");
  if (env_lo) *env_lo = c->g_lo[group];
  if (env_hi) *env_hi = c->g_hi[group];
  return SO100_OK;
}

int so100_step_host_async(so100_ctx* c, int group, const float* actions_host, float* obs_host, float* reward_host, uint8_t* terminated_host,
                          uint8_t* truncated_host, float* terminal_obs_host, float* ep_return_host, int32_t* ep_len_host, void* stream) {
  if (!c || !actions_host || !obs_host || !reward_host || !terminated_host || !truncated_host) return fail(SO100_ERR_ARG, "null argument");
  if (group < 0 || group >= c->n_groups) return fail(SO100_ERR_ARG, "no such env group");
  if (c->g_pending[group]) return fail(SO100_ERR_STATE, "this group already has a step in flight: call so100_step_host_wait first");
  CU(cudaSetDevice(c->device));
  int rc = ensure_staging(c);
  if (rc) return rc;
  HostAlias z = alias_host(actions_host, obs_host, reward_host, terminated_host, truncated_host, terminal_obs_host, ep_return_host, ep_len_host);
  if (!z.ok) return fail(SO100_ERR_ARG, "so100_step_host_async needs page-locked (pinned / registered) host buffers");
  cudaStream_t gs = c->gs[group];
  if (c->g_fork_needed[group]) {  // order after what the library has enqueued on the caller's stream (a reset, a set_state)
    CU(cudaEventRecord(c->g_fork, (cudaStream_t)stream));
    CU(cudaStreamWaitEvent(gs, c->g_fork, 0));
    c->g_fork_needed[group] = false;
  }
  c->g_tick[group] += 1;
  if (c->g_tick[group] > c->tick) c->tick = c->g_tick[group];
  const int lo = c->g_lo[group], hi = c->g_hi[group];
  const size_t cnt = (size_t)(hi - lo), od = (size_t)c->obs_dim;
  const float* act = z.act;
  float* obs = z.obs;
  if (c->async_h2d_copy) {  // the group's action rows by copy engine instead of loads over the link from the SMs
    CU(cudaMemcpyAsync(c->h_act + (size_t)lo * SO_NJ, actions_host + (size_t)lo * SO_NJ, cnt * SO_NJ * 4, cudaMemcpyHostToDevice, gs));
    act = c->h_act;
  }
  if (c->async_d2h_copy) obs = c->h_obs;
  StepIO io{act, obs, z.rew, z.tobs, z.epr, z.term, z.trunc, z.epl, (unsigned)c->g_tick[group], lo, hi, nullptr};
  rc = launch_step(c, io, gs);
  if (rc) return rc;
  if (c->async_d2h_copy) CU(cudaMemcpyAsync(obs_host + (size_t)lo * od, c->h_obs + (size_t)lo * od, cnt * od * 4, cudaMemcpyDeviceToHost, gs));
  CU(cudaEventRecord(c->g_done[group], gs));
  c->g_pending[group] = true;
  return SO100_OK;
}

int so100_step_host_wait(so100_ctx* c, int group) {
  if (!c || group < 0 || group >= c->n_groups) return fail(SO100_ERR_ARG, "no such env group");
  if (!c->g_pending[group]) return SO100_OK;
  CU(cudaEventSynchronize(c->g_done[group]));
  c->g_pending[group] = false;
  return SO100_OK;
}

int so100_step_host_wait_any(so100_ctx* c, int* group_out) {
  if (!c || !group_out) return fail(SO100_ERR_ARG, "null argument");
  int pending = 0;
  for (int g = 0; g < c->n_groups; g++) pending += c->g_pending[g] ? 1 : 0;
  *group_out = -1;
  if (!pending) return SO100_OK;
  CU(cudaSetDevice(c->device));
  for (int g = c->g_next;; g = (g + 1) % c->n_groups) {  // round-robin from the group after the last one returned
    if (!c->g_pending[g]) continue;
    cudaError_t e = cudaEventQuery(c->g_done[g]);
    if (e == cudaSuccess) {
      c->g_pending[g] = false;
      c->g_next = (g + 1) % c->n_groups;
      *group_out = g;
      return SO100_OK;
    }
    if (e != cudaErrorNotReady) return fail(SO100_ERR_CUDA, std::string("cudaEventQuery: ") + cudaGetErrorString(e));
  }
}

static int copy_state(so100_ctx* c, const so100_state_view* v, void* stream, bool get) {
  if (!c || !v) return fail(SO100_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  size_t n = (size_t)c->n;
  struct { void* ext; void* in; size_t bytes; } f[] = {
      {v->qpos, c->B.qpos, 6 * n * 4}, {v->qvel, c->B.qvel, 6 * n * 4}, {v->qacc_warm, c->B.warm, 6 * n * 4}, {v->qpos_comp, c->B.qcomp, 6 * n * 4},
      {v->block, c->B.block, 4 * n * 4}, {v->snap, c->B.snap, kSnap * n * 4}, {v->aux, c->B.aux, kAux * n * 4},
      {v->counters, c->B.cnt, kCnt * n * 4}, {v->ep_return, c->B.ep_return, n * 4}};
  for (auto& x : f) {
    if (!x.ext) continue;
    if (get) CU(cudaMemcpyAsync(x.ext, x.in, x.bytes, cudaMemcpyDeviceToDevice, st));
    else CU(cudaMemcpyAsync(x.in, x.ext, x.bytes, cudaMemcpyDeviceToDevice, st));
  }
  mark_caller_stream_work(c);  // (a get must also be ordered before a later group step overwrites the state)
  return SO100_OK;
}
int so100_get_state(so100_ctx* c, const so100_state_view* v, void* stream) { return copy_state(c, v, stream, true); }
int so100_set_state(so100_ctx* c, const so100_state_view* v, void* stream) { return copy_state(c, v, stream, false); }

int so100_get_tick(so100_ctx* c, int64_t* tick) {
  if (!c || !tick) return fail(SO100_ERR_ARG, "null argument");
  *tick = c->tick;
  return SO100_OK;
}
int so100_set_tick(so100_ctx* c, int64_t tick) {
  if (!c || tick < 0) return fail(SO100_ERR_ARG, "bad argument");
  set_all_ticks(c, tick);
  return SO100_OK;
}

int so100_set_seed(so100_ctx* c, uint64_t seed) {
  if (!c) return fail(SO100_ERR_ARG, "null argument");
  c->C.t.seed_lo = (unsigned)(seed & 0xFFFFFFFFull);  // the constants travel by value with every launch
  c->C.t.seed_hi = (unsigned)(seed >> 32);
  return SO100_OK;
}

// ---- per-env dynamics parameters, actuator latency, joint-angle observation noise
static bool group_step_in_flight(const so100_ctx* c) {
  for (int g = 0; g < c->n_groups; g++) if (c->g_pending[g]) return true;
  return false;
}

// every env's parameters = the ctx's constants, and lo = hi = 1 (what the reset-time draw then reproduces); allocates
// the array on first use
static int fill_model_params(so100_ctx* c) {
  const size_t n = (size_t)c->n;
  float* d = c->par.p;
  if (!d) CU(cudaMalloc((void**)&d, kParams * n * 4));
  float* h = (float*)malloc(kParams * n * 4);
  if (!h) { if (!c->par.p) cudaFree(d); return fail(SO100_ERR_CUDA, "out of host memory"); }
  const TaskC& t = c->C.t;
  for (int j = 0; j < SO_NJ; j++) {
    const float v[5] = {t.act.kp[j], t.act.kv[j], t.act.frc_lo[j], t.act.frc_hi[j], c->C.con.fr_loss[j]};
    for (int k = 0; k < 5; k++) for (size_t i = 0; i < n; i++) h[(k * SO_NJ + j) * n + i] = v[k];
  }
  const cudaError_t e = cudaMemcpy(d, h, kParams * n * 4, cudaMemcpyHostToDevice);
  free(h);
  if (e != cudaSuccess) { if (!c->par.p) cudaFree(d); return fail(SO100_ERR_CUDA, std::string("cudaMemcpy(params): ") + cudaGetErrorString(e)); }
  c->par.p = d;
  for (int k = 0; k < kParamDraws; k++) c->par.lo[k] = c->par.hi[k] = 1.0f;
  return SO100_OK;
}

static int free_model_params(so100_ctx* c) {
  if (c->par.p) {
    CU(cudaDeviceSynchronize());  // no launch may still read the array
    CU(cudaFree(c->par.p));
    c->par.p = nullptr;
  }
  return SO100_OK;
}

int so100_set_param_ranges(so100_ctx* c, const so100_param_ranges* r) {
  if (!c) return fail(SO100_ERR_ARG, "null argument");
  if (group_step_in_flight(c)) return fail(SO100_ERR_STATE, "an asynchronous group step is in flight: call so100_step_host_wait first");
  CU(cudaSetDevice(c->device));
  if (!r) {  // off: the model's constants, and the default kernels again unless a sim2real config keeps the per-env ones
    c->ranges_on = false;
    if (!c->par.latency) return free_model_params(c);
    CU(cudaDeviceSynchronize());
    return fill_model_params(c);
  }
  if (r->struct_size != (int)sizeof(so100_param_ranges)) return fail(SO100_ERR_ARG, "so100_param_ranges.struct_size mismatch");
  const double(*rows[4])[2] = {r->kp, r->damping, r->forcerange, r->frictionloss};
  const char* names[4] = {"kp", "damping", "forcerange", "frictionloss"};
  const bool positive[4] = {true, false, true, false};
  float lo[kParamDraws], hi[kParamDraws];
  for (int g = 0; g < 4; g++) {
    for (int j = 0; j < SO_NJ; j++) {
      const double a = rows[g][j][0], b = rows[g][j][1];
      if (!std::isfinite((float)a) || !std::isfinite((float)b) || !(a <= b))
        return fail(SO100_ERR_ARG, std::string(names[g]) + ": every range needs finite bounds with lo <= hi");
      if (positive[g] ? !(a > 0) : !(a >= 0)) return fail(SO100_ERR_ARG, std::string(names[g]) + (positive[g] ? ": lo must be > 0" : ": lo must be >= 0"));
      lo[g * SO_NJ + j] = (float)a; hi[g * SO_NJ + j] = (float)b;
    }
  }
  // first set: every env starts from the ctx's own constants and keeps them until its next reset (a sim2real config
  // already holds them there)
  if (!c->par.p) if (int rc = fill_model_params(c)) return rc;
  memcpy(c->par.lo, lo, sizeof lo);  // the ranges travel by value with every launch: they apply from each env's next reset
  memcpy(c->par.hi, hi, sizeof hi);
  c->ranges_on = true;
  return SO100_OK;
}

static int copy_params(so100_ctx* c, const so100_param_view* v, void* stream, bool get) {
  if (!c || !v) return fail(SO100_ERR_ARG, "null argument");
  if (group_step_in_flight(c)) return fail(SO100_ERR_STATE, "an asynchronous group step is in flight: call so100_step_host_wait first");
  if (!c->ranges_on) return fail(SO100_ERR_STATE, "per-env parameters are off: call so100_set_param_ranges first");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = (size_t)c->n, rows = SO_NJ * n;
  float* f[5] = {v->kp, v->kv, v->force_lo, v->force_hi, v->frictionloss};
  for (int k = 0; k < 5; k++) {
    if (!f[k]) continue;
    if (get) CU(cudaMemcpyAsync(f[k], c->par.p + k * rows, rows * 4, cudaMemcpyDeviceToDevice, st));
    else CU(cudaMemcpyAsync(c->par.p + k * rows, f[k], rows * 4, cudaMemcpyDeviceToDevice, st));
  }
  mark_caller_stream_work(c);
  return SO100_OK;
}
int so100_get_env_params(so100_ctx* c, const so100_param_view* v, void* stream) { return copy_params(c, v, stream, true); }
int so100_set_env_params(so100_ctx* c, const so100_param_view* v, void* stream) { return copy_params(c, v, stream, false); }

int so100_set_sim2real(so100_ctx* c, const so100_sim2real* cfg) {
  if (!c) return fail(SO100_ERR_ARG, "null argument");
  if (group_step_in_flight(c)) return fail(SO100_ERR_STATE, "an asynchronous group step is in flight: call so100_step_host_wait first");
  CU(cudaSetDevice(c->device));
  if (!cfg) {  // off: no latency, no noise; the default kernels again unless ranges keep the per-env ones
    if (c->par.latency) {
      CU(cudaDeviceSynchronize());
      CU(cudaFree(c->par.latency));
      if (c->par.ctrl_prev) CU(cudaFree(c->par.ctrl_prev));
      c->par.latency = nullptr; c->par.ctrl_prev = nullptr;
    }
    c->par.lat_lo = c->par.lat_hi = 0;
    for (int j = 0; j < SO_NJ; j++) c->par.noise[j] = 0.0f;
    c->par.noise_on = 0;
    return c->ranges_on ? SO100_OK : free_model_params(c);
  }
  if (cfg->struct_size != (int)sizeof(so100_sim2real)) return fail(SO100_ERR_ARG, "so100_sim2real.struct_size mismatch");
  const int nsub = c->C.t.nsub;
  if (!(0 <= cfg->latency[0] && cfg->latency[0] <= cfg->latency[1] && cfg->latency[1] <= nsub))
    return fail(SO100_ERR_ARG, "latency: need 0 <= lo <= hi <= nsubstep (" + std::to_string(nsub) + ")");
  float noise[SO_NJ];
  int noise_on = 0;
  for (int j = 0; j < SO_NJ; j++) {
    const double s = cfg->obs_noise[j];
    if (!std::isfinite((float)s) || !(s >= 0)) return fail(SO100_ERR_ARG, "obs_noise: every std must be finite and >= 0");
    noise[j] = (float)s;
    noise_on |= noise[j] != 0.0f;
  }
  if (noise_on && c->task == SO100_TASK_ENV05)
    return fail(SO100_ERR_ARG, "obs_noise: Env05 observes its commanded angles, which carry no noise");
  if (!c->par.p) if (int rc = fill_model_params(c)) return rc;
  if (!c->par.latency) {  // first set: every env at d = 0, and its previous target the exact current position (q, -qc)
    const size_t n = (size_t)c->n;
    CU(cudaDeviceSynchronize());  // the state as the caller's queued work leaves it
    CU(cudaMalloc((void**)&c->par.latency, n * 4));
    CU(cudaMemset(c->par.latency, 0, n * 4));
    if (c->task != SO100_TASK_ENV05) {
      CU(cudaMalloc((void**)&c->par.ctrl_prev, 2 * SO_NJ * n * 4));
      actuator_init_kernel<<<grid_for(c->n * SO_NJ), kBlock>>>(c->B.qpos, c->B.qcomp, c->par.ctrl_prev, c->n * SO_NJ);
      CU(cudaGetLastError());
    }
    CU(cudaDeviceSynchronize());
  }
  c->par.lat_lo = cfg->latency[0]; c->par.lat_hi = cfg->latency[1];  // by value with every launch: from each env's next reset
  for (int j = 0; j < SO_NJ; j++) c->par.noise[j] = noise[j];       // from the next step
  c->par.noise_on = noise_on;
  return SO100_OK;
}

static int copy_actuator(so100_ctx* c, const so100_actuator_view* v, void* stream, bool get) {
  if (!c || !v) return fail(SO100_ERR_ARG, "null argument");
  if (group_step_in_flight(c)) return fail(SO100_ERR_STATE, "an asynchronous group step is in flight: call so100_step_host_wait first");
  if (!c->par.latency) return fail(SO100_ERR_STATE, "latency is off: call so100_set_sim2real first");
  if (!c->par.ctrl_prev && (v->ctrl_prev_hi || v->ctrl_prev_lo))
    return fail(SO100_ERR_ARG, "Env05 has no ctrl_prev: its previous target is aux[0:6] of the state");
  CU(cudaSetDevice(c->device));
  cudaStream_t st = (cudaStream_t)stream;
  const size_t n = (size_t)c->n, rows = SO_NJ * n;
  void* dev[3] = {c->par.latency, c->par.ctrl_prev, c->par.ctrl_prev ? c->par.ctrl_prev + rows : nullptr};
  void* usr[3] = {v->latency, v->ctrl_prev_hi, v->ctrl_prev_lo};
  const size_t bytes[3] = {n * 4, rows * 4, rows * 4};
  for (int k = 0; k < 3; k++) {
    if (!usr[k]) continue;
    if (get) CU(cudaMemcpyAsync(usr[k], dev[k], bytes[k], cudaMemcpyDeviceToDevice, st));
    else CU(cudaMemcpyAsync(dev[k], usr[k], bytes[k], cudaMemcpyDeviceToDevice, st));
  }
  mark_caller_stream_work(c);
  return SO100_OK;
}
int so100_get_actuator_state(so100_ctx* c, const so100_actuator_view* v, void* stream) { return copy_actuator(c, v, stream, true); }
int so100_set_actuator_state(so100_ctx* c, const so100_actuator_view* v, void* stream) { return copy_actuator(c, v, stream, false); }

int so100_forward_dynamics(so100_ctx* c, int n, const float* qpos_dev, const float* qvel_dev, const float* ctrl_dev,
                           float* M_dev, float* bias_dev, float* qacc_dev, float* kin_dev, void* stream) {
  if (!c || n <= 0 || !qpos_dev || !qvel_dev || !ctrl_dev) return fail(SO100_ERR_ARG, "bad argument");
  CU(cudaSetDevice(c->device));
  forward_kernel<<<grid_for(n), kBlock, 0, (cudaStream_t)stream>>>(c->C, n, qpos_dev, qvel_dev, ctrl_dev, M_dev, bias_dev, qacc_dev, kin_dev);
  c->launches++;
  CU(cudaGetLastError());
  return SO100_OK;
}

int so100_host_constants(const so100_model* m, double* out) {
  if (!m || !out) return fail(SO100_ERR_ARG, "null argument");
  if (m->struct_size != (int)sizeof(so100_model)) return fail(SO100_ERR_ARG, "so100_model.struct_size mismatch");
  HostModel H;
  int rc = build_host_model(*m, H);
  if (rc) return rc;
  flatten_dyn(H.dyn, out);
  return SO100_OK;
}

int so100_host_solver_constants(const so100_model* m, float* out, int n_out) {
  if (!m || !out) return fail(SO100_ERR_ARG, "null argument");
  if (m->struct_size != (int)sizeof(so100_model)) return fail(SO100_ERR_ARG, "so100_model.struct_size mismatch");
  if (n_out != kNSolverConstants) return fail(SO100_ERR_ARG, "n_out must be SO100_N_SOLVER_CONSTANTS");
  HostModel H;
  int rc = build_host_model(*m, H);
  if (rc) return rc;
  ConC<float> K;
  ActC<float> A;
  BlkC<float> Bk;
  solver_constants_f32(*m, H, K, A, Bk);
  flatten_solver(K, A, Bk, out);
  return SO100_OK;
}

int so100_host_forward(const so100_model* m, int n, const double* qpos, const double* qvel, const double* ctrl, double* M_out,
                       double* bias_out, double* qacc_out, double* kin_out, int sweeps, int variant) {
  if (!m || n <= 0 || !qpos || !qvel || !ctrl) return fail(SO100_ERR_ARG, "bad argument");
  if (m->struct_size != (int)sizeof(so100_model)) return fail(SO100_ERR_ARG, "so100_model.struct_size mismatch");
  HostModel H;
  int rc = build_host_model(*m, H);
  if (rc) return rc;
  if (variant == 1) {
    double flat[SO100_N_DYN_CONSTANTS];
    flatten_dyn(H.dyn, flat);
    if (memcmp(flat, kGenDynConstants, sizeof flat) != 0) return fail(SO100_ERR_MODEL, "model differs from the constants baked into so100_dyn_gen.cuh");
  } else if (variant != 0 && variant != 2) return fail(SO100_ERR_ARG, "variant must be 0 (generic, fp64), 1 (specialised, fp64) or 2 (generic, fp32)");
  if (variant == 2) {  // the generic recursion in fp32 on the host: what the kernels compute, without a GPU
    static Consts Cf;  // (large: keep it off the stack)
    memset(&Cf, 0, sizeof Cf);
    physics_constants_f32(H, Cf);
    ActC<float> A;
    BlkC<float> Bk;
    solver_constants_f32(*m, H, Cf.con, A, Bk);
    for (int i = 0; i < n; i++) {
      float q[SO_NJ], v[SO_NJ], s[SO_NJ], c[SO_NJ], bias[SO_NJ], M[21], b[SO_NJ], a[SO_NJ] = {0};
      for (int j = 0; j < SO_NJ; j++) { q[j] = (float)qpos[6 * i + j]; v[j] = (float)qvel[6 * i + j]; s[j] = std::sin(q[j]); c[j] = std::cos(q[j]); }
      dyn_bias_mass<float>(Cf.dyn, s, c, v, bias, M);
      for (int j = 0; j < SO_NJ; j++) {
        float cc = std::fmin(std::fmax((float)ctrl[6 * i + j], A.ctrl_lo[j]), A.ctrl_hi[j]);
        float f = A.kp[j] * cc - A.kp[j] * q[j] - A.kv[j] * v[j];
        b[j] = std::fmin(std::fmax(f, A.frc_lo[j]), A.frc_hi[j]) - bias[j];
      }
      const float zc[SO_NJ] = {0, 0, 0, 0, 0, 0};
      int st = 0;
      if (Cf.pad.n > 0 && pads_touch<float>(Cf.dyn, Cf.kin, Cf.pad, s, c)) {
        ContactIO<float> cio;
        for (int j = 0; j < SO_NJ; j++) { cio.s[j] = s[j]; cio.c[j] = c[j]; cio.q[j] = q[j]; cio.qc[j] = 0; cio.qd[j] = v[j]; cio.b[j] = b[j]; cio.a[j] = 0; }
        memcpy(cio.M, M, sizeof M);
        st = contact_solve<float>(Cf.dyn, Cf.kin, Cf.pad, Cf.con, cio, ~0u);
        memcpy(a, cio.a, sizeof a);
      } else solve_qacc<float>(Cf.con, Cf.con.fr_loss, M, b, q, zc, v, a, sweeps > 0 ? sweeps : 1);
      if (M_out) for (int k = 0; k < 21; k++) M_out[21 * i + k] = M[k];
      if (bias_out) for (int j = 0; j < SO_NJ; j++) bias_out[6 * i + j] = bias[j];
      if (qacc_out) for (int j = 0; j < SO_NJ; j++) qacc_out[6 * i + j] = a[j];
    }
    return SO100_OK;
  }
  for (int i = 0; i < n; i++) {
    const double *q = qpos + 6 * i, *v = qvel + 6 * i, *u = ctrl + 6 * i;
    double s[SO_NJ], c[SO_NJ], bias[SO_NJ], M[21], b[SO_NJ], a[SO_NJ] = {0};
    for (int j = 0; j < SO_NJ; j++) { s[j] = std::sin(q[j]); c[j] = std::cos(q[j]); }
    if (variant == 1) dyn_bias_mass_so100<double>(s, c, v, bias, M);
    else dyn_bias_mass<double>(H.dyn, s, c, v, bias, M);
    for (int j = 0; j < SO_NJ; j++) {
      double cc = std::fmin(std::fmax(u[j], m->act_ctrlrange[j][0]), m->act_ctrlrange[j][1]);
      double f = m->act_kp[j] * cc - m->act_kp[j] * q[j] - H.kv[j] * v[j];
      b[j] = std::fmin(std::fmax(f, m->act_forcerange[j][0]), m->act_forcerange[j][1]) - bias[j];
    }
    const double zc[SO_NJ] = {0, 0, 0, 0, 0, 0};
    if (H.pad.n > 0 && pads_touch<double>(H.dyn, H.kin, H.pad, s, c)) {
      ContactIO<double> cio;
      for (int j = 0; j < SO_NJ; j++) { cio.s[j] = s[j]; cio.c[j] = c[j]; cio.q[j] = q[j]; cio.qc[j] = 0; cio.qd[j] = v[j]; cio.b[j] = b[j]; cio.a[j] = 0; }
      memcpy(cio.M, M, sizeof M);
      contact_solve<double>(H.dyn, H.kin, H.pad, H.con, cio, ~0u);
      memcpy(a, cio.a, sizeof a);
    } else solve_qacc<double>(H.con, H.con.fr_loss, M, b, q, zc, v, a, sweeps > 0 ? sweeps : 1);
    if (M_out) memcpy(M_out + 21 * i, M, sizeof M);
    if (bias_out) memcpy(bias_out + 6 * i, bias, sizeof bias);
    if (qacc_out) memcpy(qacc_out + 6 * i, a, sizeof a);
    if (kin_out) {
      KinOut<double> ko;
      task_kinematics<double, true>(H.dyn, H.kin, s, c, ko);
      memcpy(kin_out + 18 * i, ko.end_pos, 24); memcpy(kin_out + 18 * i + 3, ko.wrist, 24);
      memcpy(kin_out + 18 * i + 6, ko.cam_pos, 24); memcpy(kin_out + 18 * i + 9, ko.cam_R, 72);
    }
  }
  return SO100_OK;
}

int so100_host_substeps(const so100_model* m, int n, double* qpos, double* qvel, double* qacc_warm, const double* ctrl, int n_substeps,
                        int variant, int64_t* stats) {
  if (!m || n <= 0 || !qpos || !qvel || !qacc_warm || !ctrl || n_substeps <= 0) return fail(SO100_ERR_ARG, "bad argument");
  if (m->struct_size != (int)sizeof(so100_model)) return fail(SO100_ERR_ARG, "so100_model.struct_size mismatch");
  if (variant != 0 && variant != 2 && variant != 3) return fail(SO100_ERR_ARG, "variant must be 0 (fp64), 2 (fp32) or 3 (fp32, MUFU-class sin/cos)");
  HostModel H;
  int rc = build_host_model(*m, H);
  if (rc) return rc;
  if (stats) memset(stats, 0, 5 * sizeof(int64_t));
  static Consts Cf;
  memset(&Cf, 0, sizeof Cf);
  physics_constants_f32(H, Cf);
  ActC<float> Af;
  BlkC<float> Bk;
  solver_constants_f32(*m, H, Cf.con, Af, Bk);
  if (variant >= 2) { host_substeps_t<float>(Cf.dyn, Cf.kin, Cf.pad, Cf.con, Af, n, qpos, qvel, qacc_warm, ctrl, n_substeps, stats, variant == 3); return SO100_OK; }
  ActC<double> Ad;
  for (int j = 0; j < SO_NJ; j++) {
    Ad.kp[j] = m->act_kp[j]; Ad.kv[j] = H.kv[j]; Ad.ctrl_lo[j] = m->act_ctrlrange[j][0]; Ad.ctrl_hi[j] = m->act_ctrlrange[j][1];
    Ad.frc_lo[j] = m->act_forcerange[j][0]; Ad.frc_hi[j] = m->act_forcerange[j][1];
  }
  Ad.h = m->timestep;
  host_substeps_t<double>(H.dyn, H.kin, H.pad, H.con, Ad, n, qpos, qvel, qacc_warm, ctrl, n_substeps, stats);
  return SO100_OK;
}

int so100_get_derived(so100_ctx* c, double* dof_M0, double* kv, double* invweight0) {
  if (!c) return fail(SO100_ERR_ARG, "null argument");
  for (int j = 0; j < SO_NJ; j++) {
    if (dof_M0) dof_M0[j] = c->H.dof_M0[j];
    if (kv) kv[j] = c->H.kv[j];
    if (invweight0) invweight0[j] = c->H.invw[j];
  }
  return SO100_OK;
}

int so100_kernel_variant(so100_ctx* c) {
  if (!c) return fail(SO100_ERR_ARG, "null argument");
  return c->specialised ? 1 : 0;
}

int so100_get_stats(so100_ctx* c, int64_t* launches, int64_t* solver_fallbacks, int64_t* nan_resets) {
  if (!c) return fail(SO100_ERR_ARG, "null argument");
  CU(cudaSetDevice(c->device));
  unsigned long long s[2];
  CU(cudaMemcpy(s, c->B.stats, sizeof s, cudaMemcpyDeviceToHost));
  if (launches) *launches = c->launches;
  if (solver_fallbacks) *solver_fallbacks = (int64_t)s[0];
  if (nan_resets) *nan_resets = (int64_t)s[1];
  return SO100_OK;
}

int so100_bench_fp32_peak(int device, int iters, double* tflops_out) {
  if (!tflops_out || iters <= 0) return fail(SO100_ERR_ARG, "bad argument");
  CU(cudaSetDevice(device));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, device));
  float* d = nullptr;
  CU(cudaMalloc((void**)&d, 4));
  const int blocks = prop.multiProcessorCount * 8, threads = 256;
  cudaEvent_t e0, e1;
  CU(cudaEventCreate(&e0));
  CU(cudaEventCreate(&e1));
  double best = 0;
  for (int rep = 0; rep < 5; rep++) {
    CU(cudaEventRecord(e0));
    ffma_peak_kernel<<<blocks, threads>>>(d, iters, 0.999f, 0.001f);
    CU(cudaEventRecord(e1));
    CU(cudaEventSynchronize(e1));
    float ms = 0;
    CU(cudaEventElapsedTime(&ms, e0, e1));
    double fl = 2.0 * 8 * 16 * (double)iters * blocks * threads;
    if (rep > 0 && ms > 0) best = std::fmax(best, fl / (ms * 1e-3) / 1e12);
  }
  cudaEventDestroy(e0); cudaEventDestroy(e1); cudaFree(d);
  *tflops_out = best;
  return SO100_OK;
}

}  // extern "C"

#include "so100_ppo_kernels.cuh"  // fused PPO learner kernels + their C ABI (include/so100_ppo.h)
