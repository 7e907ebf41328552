// so100_ppo_kernels.cuh — fused PPO learner kernels (C ABI: include/so100_ppo.h); included by so100_b200.cu.
//
// What SB3 runs as ~60 small PyTorch kernels per minibatch (policy.evaluate_actions, the losses, loss.backward(),
// clip_grad_norm_, Adam.step; reference call site: stable_baselines3.PPO(...).learn, src/so100_mujoco_rl/main.py:56-64,
// 234-238) is ONE gradient kernel plus two tiny ones here.  The policy is SB3's default MlpPolicy: two separate
// 2x64 tanh towers (pi: od -> 64 -> 64 -> 6, vf: od -> 64 -> 64 -> 1) and a state-independent log_std.
//
// Gradient kernel: persistent CTAs (one per SM, 256 threads), each looping over tiles of 64 samples.  Both towers'
// weights stay in shared memory for the whole kernel (88 KB); a tile's activations live in shared memory in two
// layouts, [feature][sample] for the forward / back-propagation products and [sample][feature] for the weight-gradient
// products, so that every product is a 64x64x64 GEMM with both operands K-major.  The GEMMs run on the tensor cores
// as warp-level m16n8k8 TF32 MMAs with the 3xTF32 split (x = hi + lo, D += lo*hi + hi*lo + hi*hi, fp32 accumulate),
// which keeps fp32-level parity against torch's autograd; each warp owns a 16x32 slab of the output, and every
// fragment load is a conflict-free 4-byte shared load (row stride 72 = 8 mod 32).  The first version of this kernel did
// the same products on the FP32 pipes with 4x4 register tiles and was bound by shared-memory bandwidth (one 16-byte
// load per 8 FMAs; profiles/r1_ppo_grad_ncu_raw.csv); the MMA path moves 5x fewer bytes per flop.  Weight gradients
// accumulate in REGISTERS (MMA accumulator fragments) across all tiles of the CTA and leave the SM once, as per-CTA
// partials; a second kernel adds the partials in a fixed order, so the result is deterministic.  A tcgen05 / TMEM
// version is the step after this one (DESIGN.md §4.2).
#pragma once
#include "so100_tc.cuh"

namespace ppo {

constexpr int HID = SO100_PPO_HIDDEN, ACT = SO100_PPO_ACT, TB = SO100_PPO_TILE, NT = 256, K1 = 16;
constexpr int LD = 72;    // row stride of every K-major 64-column matrix in shared memory: 72 = 8 (mod 32) makes the MMA
                          // fragment loads (4 k-rows x 8 consecutive columns per warp) hit 32 distinct banks
constexpr int LDXT = 24;  // same property for the [sample][input feature] copy (16 columns)
constexpr float LOG_SQRT_2PI = 0.91893853320467274178f;

struct Layout {  // offsets into the flat parameter vector
  int od, W1[2], b1[2], W2[2], b2[2], W3[2], b3[2], log_std, total;
};
// sde: gSDE's log_std[HID][ACT] in place of log_std[ACT]; every offset before it is the same in both layouts
__host__ __device__ inline Layout make_layout(int od, bool sde = false) {
  Layout L;
  L.od = od;
  int o = 0;
  for (int t = 0; t < 2; t++) {
    const int nout = t == 0 ? ACT : 1;
    L.W1[t] = o; o += HID * od;
    L.b1[t] = o; o += HID;
    L.W2[t] = o; o += HID * HID;
    L.b2[t] = o; o += HID;
    L.W3[t] = o; o += nout * HID;
    L.b3[t] = o; o += nout;
  }
  L.log_std = o; o += sde ? HID * ACT : ACT;
  L.total = o;
  return L;
}

// shared-memory image of one tower's weights
struct TowerS {
  float* W1t;  // [K1][LD]    W1t[k][m] = W1[m][k], rows k >= od are zero
  float* W2t;  // [HID][LD]   W2t[k][m] = W2[m][k]
  float* W2n;  // [HID][LD]   W2 as stored, [out][in]
  float* W3;   // [nout][HID]
  float *b1, *b2, *b3;
};
constexpr int tower_floats(bool with_w2n) { return K1 * LD + HID * LD + (with_w2n ? HID * LD : 0) + 8 * HID + HID + HID + 8; }

__device__ inline float* carve_tower(float* p, TowerS& T, bool with_w2n) {
  T.W1t = p; p += K1 * LD;
  T.W2t = p; p += HID * LD;
  T.W2n = with_w2n ? p : nullptr; p += with_w2n ? HID * LD : 0;
  T.W3 = p; p += 8 * HID;
  T.b1 = p; p += HID;
  T.b2 = p; p += HID;
  T.b3 = p; p += 8;
  return p;
}
__device__ inline void load_tower(const Layout& L, const float* P, int t, TowerS& T, bool with_w2n) {
  const int od = L.od, nout = t == 0 ? ACT : 1, tid = threadIdx.x, nt = blockDim.x;
  for (int e = tid; e < K1 * HID; e += nt) { int k = e / HID, m = e % HID; T.W1t[k * LD + m] = k < od ? P[L.W1[t] + m * od + k] : 0.0f; }
  for (int e = tid; e < HID * HID; e += nt) {
    int k = e / HID, m = e % HID;
    T.W2t[k * LD + m] = P[L.W2[t] + m * HID + k];
    if (with_w2n) T.W2n[k * LD + m] = P[L.W2[t] + e];
  }
  for (int e = tid; e < 8 * HID; e += nt) T.W3[e] = e < nout * HID ? P[L.W3[t] + e] : 0.0f;
  for (int e = tid; e < HID; e += nt) { T.b1[e] = P[L.b1[t] + e]; T.b2[e] = P[L.b2[t] + e]; }
  for (int e = tid; e < 8; e += nt) T.b3[e] = e < nout ? P[L.b3[t] + e] : 0.0f;
}

// ---- warp-level tensor-core tile: D(16 x 8*NTILE) += A(16 x K) B(K x 8*NTILE), both operands K-major in shared memory
// (At[k][m], Bm[k][n]).  Lane (g = lane / 4, t = lane % 4) owns rows m0 + g + 8 i (i = 0, 1) and, in n-tile j, columns
// n0 + 8 j + 2 t + e (e = 0, 1): acc[j][2 i + e]  (PTX ISA, mma.m16n8k8 .tf32 fragment layouts).
struct Own {
  int m0, n0, g, t;
  __device__ __forceinline__ int row(int i) const { return m0 + g + 8 * i; }
  __device__ __forceinline__ int col(int j, int e) const { return n0 + 8 * j + 2 * t + e; }
};
__device__ __forceinline__ Own own_64x64() {  // 8 warps: 4 along M x 2 along N, each 16 x 32
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  return Own{16 * (w & 3), 32 * (w >> 2), lane >> 2, lane & 3};
}
// 3xTF32 operand split.  The tensor core reads only the upper 19 bits of an fp32 operand (sign, exponent, 10 mantissa
// bits), so "hi" is x itself as far as the MMA is concerned; lo = x - trunc19(x) is exact in fp32 (two instructions;
// cvt.rna.tf32 is emulated with ~8 on this architecture) and is itself truncated by the hardware to 11 significant bits:
// the neglected lo*lo term is at most 2^-20 relative per product (truncation keeps its sign, so it under-estimates |ab|
// by up to ~1e-6; the gradient test bounds the total at 2e-5 of the largest entry).
__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = __float_as_uint(x);
  lo = __float_as_uint(x - __uint_as_float(hi & 0xFFFFE000u));
}
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], const uint32_t (&b)[2]) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b[0]), "r"(b[1]));
}
template <int K, int NTILE, int lda, int ldb>
__device__ __forceinline__ void gemm_mma(const float* __restrict__ At, const float* __restrict__ Bm, const Own& o, float (&acc)[NTILE][4]) {
#pragma unroll 2
  for (int k0 = 0; k0 < K; k0 += 8) {
    const float* ap = At + (k0 + o.t) * lda + o.m0 + o.g;
    uint32_t ah[4], al[4];
    split_tf32(ap[0], ah[0], al[0]);
    split_tf32(ap[8], ah[1], al[1]);
    split_tf32(ap[4 * lda], ah[2], al[2]);
    split_tf32(ap[4 * lda + 8], ah[3], al[3]);
    const float* bp = Bm + (k0 + o.t) * ldb + o.n0 + o.g;
#pragma unroll
    for (int j = 0; j < NTILE; j++) {
      uint32_t bh[2], bl[2];
      split_tf32(bp[8 * j], bh[0], bl[0]);
      split_tf32(bp[4 * ldb + 8 * j], bh[1], bl[1]);
      mma_tf32(acc[j], al, bh);  // small terms first
      mma_tf32(acc[j], ah, bl);
      mma_tf32(acc[j], ah, bh);
    }
  }
}
template <int NTILE>
__device__ __forceinline__ void zero_acc(float (&a)[NTILE][4]) {
#pragma unroll
  for (int j = 0; j < NTILE; j++)
#pragma unroll
    for (int q = 0; q < 4; q++) a[j][q] = 0.0f;
}
// h = tanh(acc + bias[row]) -> H[row][col] ([feature][sample]) and, if HT, HT[col][row] ([sample][feature]); both ld = LD
__device__ __forceinline__ void store_tanh(const float (&acc)[4][4], const float* bias, const Own& o, float* H, float* HT) {
#pragma unroll
  for (int i = 0; i < 2; i++) {
    const int r = o.row(i);
    const float bi = bias[r];
#pragma unroll
    for (int j = 0; j < 4; j++) {
      const float h0 = tanhf(acc[j][2 * i] + bi), h1 = tanhf(acc[j][2 * i + 1] + bi);
      const int c = o.col(j, 0);
      *reinterpret_cast<float2*>(H + r * LD + c) = make_float2(h0, h1);
      if (HT) { HT[c * LD + r] = h0; HT[(c + 1) * LD + r] = h1; }
    }
  }
}
// two hidden layers of one tower on the tile in X ([K1][LD]); leaves H1, H2 (and the transposed copies when given)
__device__ __forceinline__ void tower_forward(const TowerS& T, const float* X, float* H1, float* H1T, float* H2, float* H2T, const Own& o) {
  float acc[4][4];
  zero_acc(acc);
  gemm_mma<K1, 4, LD, LD>(T.W1t, X, o, acc);
  store_tanh(acc, T.b1, o, H1, H1T);
  __syncthreads();
  zero_acc(acc);
  gemm_mma<HID, 4, LD, LD>(T.W2t, H1, o, acc);
  store_tanh(acc, T.b2, o, H2, H2T);
  __syncthreads();
}
// out[o][s] = b3[o] + sum_k W3[o][k] H2[k][s].  The 64-long sums are split over four thread groups (16 k each, NOUT
// independent chains per thread) and combined through `scratch` ([4][8][TB]); ends with the block synchronised.
template <int NOUT>
__device__ __forceinline__ void head_forward(const TowerS& T, const float* H2, float* out, float* scratch) {
  const int kg = threadIdx.x >> 6, s = threadIdx.x & 63;
  float acc[NOUT];
#pragma unroll
  for (int o = 0; o < NOUT; o++) acc[o] = 0.0f;
#pragma unroll
  for (int k = 16 * kg; k < 16 * kg + 16; k++) {
    const float h = H2[k * LD + s];
#pragma unroll
    for (int o = 0; o < NOUT; o++) acc[o] = fmaf(T.W3[o * HID + k], h, acc[o]);
  }
#pragma unroll
  for (int o = 0; o < NOUT; o++) scratch[(kg * 8 + o) * TB + s] = acc[o];
  __syncthreads();
  for (int e = threadIdx.x; e < NOUT * TB; e += NT) {
    const int o = e / TB, c = e % TB;
    out[e] = T.b3[o] + ((scratch[o * TB + c] + scratch[(8 + o) * TB + c]) + (scratch[(16 + o) * TB + c] + scratch[(24 + o) * TB + c]));
  }
  __syncthreads();
}

// ------------------------------------------------------------------------------------------------ gSDE (DESIGN.md §7d)
// SB3's StateDependentNoiseDistribution (full_std, no expln, learn_features=False): with h = the policy tower's last
// hidden layer, the action is mean + h E, E[k][j] = exp(log_std[k][j]) z[k][j] drawn per env, and the distribution is
// Normal(mean, sqrt(var + 1e-6)) with var_j = sum_k h_k^2 S[k][j], S = exp(2 log_std).  E is never stored: normal number
// i = 64 j + k of an env is position i % 4 of Philox block (seed, env_offset + env, noise_key, 0x5D00 + i / 4, 0), through
// the Box-Muller transform of the plain noise (words 0,1 and 2,3).  Both inference kernels and the gradient kernel split
// the 64 features into four groups of 16, each an fp32 FMA chain from zero in ascending k, combined as (g0 + g1) + (g2 + g3).
constexpr unsigned kSdeStream = 0x5D00u;
constexpr float kSdeEps = 1e-6f;

// group [k0, k0 + 16) of the noise sum_k h_k fl(std_kj z_kj) (when `noise`; else zeros) and of var_j = sum_k fl(h_k^2) S_kj.
// The Box-Muller lines restate the act kernels' own (left in place there, so that their plain instantiations keep their SASS).
__device__ __forceinline__ void sde_partial(const float (&h)[16], int k0, unsigned seed_lo, unsigned seed_hi, unsigned env, unsigned key, bool noise,
                                            const float* sstd, const float* sS, float (&nz)[ACT], float (&vr)[ACT]) {
#pragma unroll
  for (int j = 0; j < ACT; j++) { nz[j] = 0.0f; vr[j] = 0.0f; }
#pragma unroll
  for (int k = 0; k < 16; k++) {
    const float h2 = h[k] * h[k];
#pragma unroll
    for (int j = 0; j < ACT; j++) vr[j] = fmaf(h2, sS[(k0 + k) * ACT + j], vr[j]);
  }
  if (!noise) return;
#pragma unroll 1
  for (int j = 0; j < ACT; j++) {
#pragma unroll
    for (int b = 0; b < 4; b++) {
      const uint4 r = philox4x32(seed_lo, seed_hi, env, key, kSdeStream + 16u * j + (unsigned)(k0 >> 2) + b, 0u);
      const unsigned w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
      for (int q = 0; q < 2; q++) {
        const float u1 = ((float)(w[2 * q] >> 8) + 0.5f) * (1.0f / 16777216.0f), u2 = (float)(w[2 * q + 1] >> 8) * (1.0f / 16777216.0f);
        const float rad = sqrtf(-2.0f * logf(u1));
        float sn, cs;
        sincospif(2.0f * u2, &sn, &cs);
        const int k = 4 * b + 2 * q;
        nz[j] = fmaf(h[k], sstd[(k0 + k) * ACT + j] * (rad * cs), nz[j]);
        nz[j] = fmaf(h[k + 1], sstd[(k0 + k + 1) * ACT + j] * (rad * sn), nz[j]);
      }
    }
  }
}
// one action's term of the gSDE log-prob, given isig2 = 1 / (var + 1e-6)
__device__ __forceinline__ float sde_logp_term(float d, float v, float isig2) { return -0.5f * d * d * isig2 - 0.5f * logf(v) - LOG_SQRT_2PI; }

// ------------------------------------------------------------------------------------------------ rollout inference
constexpr int kActSmemFloats = 2 * tower_floats(false) + K1 * LD + 2 * HID * LD + 8 * TB + 32 * TB + 8;
constexpr int kActSmemFloatsSde = kActSmemFloats + 2 * HID * ACT;  // + std and S; the partials reuse H1
static_assert(4 * 2 * ACT * TB <= HID * LD, "act_kernel<SDE>: the partials fit the H1 buffer");

template <bool SDE>
__global__ void __launch_bounds__(NT) act_kernel(Layout L, const float* __restrict__ P, const float* __restrict__ obs, int n, unsigned seed_lo,
                                                 unsigned seed_hi, long long env_offset, unsigned tick, int deterministic, float* act_raw,
                                                 float* act_clip, float* logp, float* value, float* obs_copy) {
  extern __shared__ __align__(16) float sm[];
  TowerS T[2];
  float* p = carve_tower(sm, T[0], false);
  p = carve_tower(p, T[1], false);
  float* X = p; p += K1 * LD;
  float* H1 = p; p += HID * LD;
  float* H2 = p; p += HID * LD;
  float* out = p; p += 8 * TB;
  float* scratch = p; p += 32 * TB;
  float* ls = p;
  float* sstd = ls + 8;             // (SDE) exp(log_std) [HID][ACT]
  float* sS = sstd + HID * ACT;     // (SDE) exp(2 log_std)
  const int tid = threadIdx.x, od = L.od;
  load_tower(L, P, 0, T[0], false);
  load_tower(L, P, 1, T[1], false);
  if constexpr (SDE) {
    for (int e = tid; e < HID * ACT; e += NT) { sstd[e] = expf(P[L.log_std + e]); sS[e] = expf(2.0f * P[L.log_std + e]); }
  } else {
    if (tid < ACT) ls[tid] = P[L.log_std + tid];
  }
  const Own o = own_64x64();
  const int ntiles = (n + TB - 1) / TB;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {  // persistent: the weights are staged once per CTA
    const int base = tile * TB;
    __syncthreads();
    for (int e = tid; e < TB * K1; e += NT) {
      const int s = e / K1, f = e % K1, g = base + s;
      float v = 0.0f;
      if (g < n && f < od) {
        v = obs[(size_t)g * od + f];
        if (obs_copy) obs_copy[(size_t)g * od + f] = v;
      }
      X[f * LD + s] = v;
    }
    __syncthreads();
    tower_forward(T[1], X, H1, nullptr, H2, nullptr, o);
    head_forward<1>(T[1], H2, out + 7 * TB, scratch);  // value in row 7
    tower_forward(T[0], X, H1, nullptr, H2, nullptr, o);
    head_forward<ACT>(T[0], H2, out, scratch);
    if constexpr (SDE) {  // thread (q, s): feature group q of sample s; partials -> the H1 buffer (h1 is dead) [4][2 ACT][TB]
      const int q = tid >> 6, s = tid & 63, g = base + s;
      float h[16], nz[ACT], vr[ACT];
#pragma unroll
      for (int k = 0; k < 16; k++) h[k] = H2[(16 * q + k) * LD + s];
      sde_partial(h, 16 * q, seed_lo, seed_hi, (unsigned)(env_offset + g), tick, !deterministic && g < n, sstd, sS, nz, vr);
#pragma unroll
      for (int j = 0; j < ACT; j++) { H1[(q * 2 * ACT + j) * TB + s] = nz[j]; H1[(q * 2 * ACT + ACT + j) * TB + s] = vr[j]; }
      __syncthreads();
      if (tid < TB && base + tid < n) {
        const int g = base + tid;
        auto sum4 = [&](int r) { return (H1[r * TB + tid] + H1[(2 * ACT + r) * TB + tid]) + (H1[(4 * ACT + r) * TB + tid] + H1[(6 * ACT + r) * TB + tid]); };
        float lp = 0.0f;
#pragma unroll
        for (int k = 0; k < ACT; k++) {
          const float mean = out[k * TB + tid], a = deterministic ? mean : mean + sum4(k);
          const float v = sum4(ACT + k) + kSdeEps, d = a - mean;
          lp += sde_logp_term(d, v, 1.0f / v);
          if (act_raw) act_raw[(size_t)g * ACT + k] = a;
          if (act_clip) act_clip[(size_t)g * ACT + k] = fminf(fmaxf(a, -1.0f), 1.0f);
        }
        if (logp) logp[g] = lp;
        if (value) value[g] = out[7 * TB + tid];
      }
      continue;
    }
    if (tid < TB && base + tid < n) {
      const int g = base + tid;
      float eps[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      if (!deterministic) {  // 8 standard normals from two Philox blocks (Box-Muller)
#pragma unroll
        for (int b = 0; b < 2; b++) {
          const uint4 r = philox4x32(seed_lo, seed_hi, (unsigned)(env_offset + g), tick, 0x5050u + b, 0u);
          const unsigned w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
          for (int q = 0; q < 2; q++) {
            const float u1 = ((float)(w[2 * q] >> 8) + 0.5f) * (1.0f / 16777216.0f), u2 = (float)(w[2 * q + 1] >> 8) * (1.0f / 16777216.0f);
            const float rad = sqrtf(-2.0f * logf(u1));
            float sn, cs;
            sincospif(2.0f * u2, &sn, &cs);
            eps[4 * b + 2 * q] = rad * cs; eps[4 * b + 2 * q + 1] = rad * sn;
          }
        }
      }
      float lp = 0.0f;
#pragma unroll
      for (int k = 0; k < ACT; k++) {
        const float mean = out[k * TB + tid], a = mean + expf(ls[k]) * eps[k];
        lp += -0.5f * eps[k] * eps[k] - ls[k] - LOG_SQRT_2PI;  // (a - mean)^2 / (2 sigma^2) = eps^2 / 2
        if (act_raw) act_raw[(size_t)g * ACT + k] = a;
        if (act_clip) act_clip[(size_t)g * ACT + k] = fminf(fmaxf(a, -1.0f), 1.0f);
      }
      if (logp) logp[g] = lp;
      if (value) value[g] = out[7 * TB + tid];
    }
  }
}

// ------------------------------------------------------------------------------------------------ rollout inference, tcgen05
// The same computation on the 5th-generation tensor cores (csrc/so100_tc.cuh): tiles of 128 samples, D[sample][feature] =
// act[sample][k] W[feature][k] issued by ONE thread as tcgen05.mma kind::tf32 with M = 128.  The ACTIVATIONS NEVER TOUCH
// SHARED MEMORY: the A operand of every product is read from TMEM (row = TMEM lane = sample, K along the columns), where
// the thread that owns the sample has put it with tcgen05.st - the observation row at the start of a tile, then after
// each layer tcgen05.ld of its accumulator row -> bias + tanh -> the 3xTF32 split (hi and lo copies, made ONCE per value)
// -> tcgen05.st of its row of the next layer's A.  Only the weights sit in shared memory (hi and lo images in the no-
// swizzle K-major layout, 96 KB), so TWO CTAs share an SM (and its 512 TMEM columns: 256 each) and one's epilogue overlaps
// the other's MMAs.  The two warpgroups of a CTA split a layer's 64 columns.  Per tile and tower: layer 1 (6 MMAs), layer 2
// (24), head (24, N = 16); one mbarrier, committed after every layer.  Persistent over tiles.
constexpr int TM = 128, NTC = 256;
struct ActTc {  // byte offsets into dynamic shared memory
  static constexpr int W1 = 0;                         // [tower][hi, lo][64 x 16]
  static constexpr int W2 = W1 + 2 * 2 * 64 * 16 * 4;  // [tower][hi, lo][64 x 64]
  static constexpr int W3 = W2 + 2 * 2 * 64 * 64 * 4;  // [tower][hi, lo][16 x 64]
  static constexpr int BIAS = W3 + 2 * 2 * 16 * 64 * 4;  // b1[2][64], b2[2][64], b3[2][8], log_std[8]
  static constexpr int BAR = BIAS + (2 * 64 + 2 * 64 + 16 + 8) * 4;
  static constexpr int BYTES = BAR + 16;
  // gSDE only: exp(log_std) and exp(2 log_std) [64][6], then warpgroup 1's partials [2 ACT][128]
  static constexpr int SDE_STD = BYTES, SDE_S = SDE_STD + 64 * 6 * 4, SDE_X = SDE_S + 64 * 6 * 4;
  static constexpr int BYTES_SDE = SDE_X + 2 * 6 * 128 * 4;
  // TMEM columns (256 per CTA)
  static constexpr uint32_t cD = 0, cAh = 64, cAl = 128, cXh = 192, cXl = 208, cHead = 224;
};
static_assert(2 * (ActTc::BYTES + 1024) <= 227 * 1024, "act_kernel_tc: two CTAs per SM");
static_assert(2 * (ActTc::BYTES_SDE + 1024) <= 227 * 1024, "act_kernel_tc<SDE>: two CTAs per SM");

// one layer's epilogue for this thread's half of the 64 columns: h = tanh(D + bias) -> hi / lo rows of the next layer's A (TMEM)
__device__ __forceinline__ void tc_epilogue_tanh(uint32_t tmem_row, int col0, const float* bias) {
#pragma unroll
  for (int c0 = col0; c0 < col0 + 32; c0 += 16) {
    float v[16], hi[16], lo[16];
    tc::tmem_ld16(tmem_row + ActTc::cD + c0, v);
#pragma unroll
    for (int i = 0; i < 16; i++) tc::split(tanhf(v[i] + bias[c0 + i]), hi[i], lo[i]);
    tc::tmem_st16(tmem_row + ActTc::cAh + c0, hi);
    tc::tmem_st16(tmem_row + ActTc::cAl + c0, lo);
  }
  tc::tmem_st_wait();
}
// D (+)= A B^T over K with the 3xTF32 split (small terms first); A (hi at column ah, lo at al) in TMEM, B in shared memory
template <int NROWS_B, int K>
__device__ __forceinline__ void tc_gemm3(uint32_t tmem_d, uint32_t ah, uint32_t al, uint32_t bh, uint32_t bl, uint32_t idesc) {
#pragma unroll
  for (int k0 = 0; k0 < K; k0 += 8) {
    tc::mma_tf32_ts(tmem_d, al + k0, tc::op_desc<NROWS_B>(bh, k0 / 4), idesc, k0 > 0);
    tc::mma_tf32_ts(tmem_d, ah + k0, tc::op_desc<NROWS_B>(bl, k0 / 4), idesc, true);
    tc::mma_tf32_ts(tmem_d, ah + k0, tc::op_desc<NROWS_B>(bh, k0 / 4), idesc, true);
  }
}

template <bool SDE>
__global__ void __launch_bounds__(NTC, 2) act_kernel_tc(Layout L, const float* __restrict__ P, const float* __restrict__ obs, int n, unsigned seed_lo,
                                                        unsigned seed_hi, long long env_offset, unsigned tick, int deterministic, float* act_raw,
                                                        float* act_clip, float* logp, float* value, float* obs_copy) {
  extern __shared__ __align__(128) unsigned char smc[];
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, od = L.od;
  const int row = tid & (TM - 1), half = tid >> 7;  // TMEM lane = sample of the tile; which half of a layer's columns
  float* bias = reinterpret_cast<float*>(smc + ActTc::BIAS);
  float *b1 = bias, *b2 = bias + 128, *b3 = bias + 256, *ls = bias + 272;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smc + ActTc::BAR);
  auto W1 = [&](int t, int lo) { return smc + ActTc::W1 + (2 * t + lo) * 64 * 16 * 4; };
  auto W2 = [&](int t, int lo) { return smc + ActTc::W2 + (2 * t + lo) * 64 * 64 * 4; };
  auto W3 = [&](int t, int lo) { return smc + ActTc::W3 + (2 * t + lo) * 16 * 64 * 4; };

  if (tid == 0) { tc::bar_init(bar, 1); tc::bar_init_fence(); }
  if (warp == 0) tc::tmem_alloc<256>(&tmem_slot);
  // weights -> hi / lo operand images (once per CTA)
  for (int t = 0; t < 2; t++) {
    const int nout = t == 0 ? ACT : 1;
    for (int e = tid; e < HID * K1; e += NTC) {
      const int m = e / K1, k = e % K1;
      float hi, lo;
      tc::split(k < od ? P[L.W1[t] + m * od + k] : 0.0f, hi, lo);
      const int off = tc::op_offset<64>(m, k);
      *reinterpret_cast<float*>(W1(t, 0) + off) = hi; *reinterpret_cast<float*>(W1(t, 1) + off) = lo;
    }
    for (int e = tid; e < HID * HID; e += NTC) {
      float hi, lo;
      tc::split(P[L.W2[t] + e], hi, lo);
      const int off = tc::op_offset<64>(e / HID, e % HID);
      *reinterpret_cast<float*>(W2(t, 0) + off) = hi; *reinterpret_cast<float*>(W2(t, 1) + off) = lo;
    }
    for (int e = tid; e < 16 * HID; e += NTC) {
      float hi, lo;
      tc::split(e < nout * HID ? P[L.W3[t] + e] : 0.0f, hi, lo);
      const int off = tc::op_offset<16>(e / HID, e % HID);
      *reinterpret_cast<float*>(W3(t, 0) + off) = hi; *reinterpret_cast<float*>(W3(t, 1) + off) = lo;
    }
    for (int e = tid; e < HID; e += NTC) { b1[64 * t + e] = P[L.b1[t] + e]; b2[64 * t + e] = P[L.b2[t] + e]; }
    for (int e = tid; e < 8; e += NTC) b3[8 * t + e] = e < nout ? P[L.b3[t] + e] : 0.0f;
  }
  float* sstd = reinterpret_cast<float*>(smc + ActTc::SDE_STD);
  float* sS = reinterpret_cast<float*>(smc + ActTc::SDE_S);
  float* xch = reinterpret_cast<float*>(smc + ActTc::SDE_X);
  if constexpr (SDE) {
    for (int e = tid; e < HID * ACT; e += NTC) { sstd[e] = expf(P[L.log_std + e]); sS[e] = expf(2.0f * P[L.log_std + e]); }
  } else {
    if (tid < 8) ls[tid] = tid < ACT ? P[L.log_std + tid] : 0.0f;
  }
  tc::fence_smem_to_mma();
  tc::fence_before_sync();
  __syncthreads();
  tc::fence_after_sync();
  const uint32_t tmem = tmem_slot, tmem_row = tmem + ((uint32_t)(32 * (warp & 3)) << 16);
  uint32_t phase = 0;
  const int ntiles = (n + TM - 1) / TM;
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    const int base = tile * TM, g = base + row;
    {  // this sample's observation row -> the hi (warpgroup 0) or lo (warpgroup 1) copy of X in TMEM; padding columns zero
      float x[16];
#pragma unroll
      for (int k = 0; k < 16; k++) x[k] = (g < n && k < od) ? obs[(size_t)g * od + k] : 0.0f;
      if (half == 0 && obs_copy && g < n) {
#pragma unroll
        for (int k = 0; k < 16; k++)
          if (k < od) obs_copy[(size_t)g * od + k] = x[k];
      }
      float part[16];
#pragma unroll
      for (int k = 0; k < 16; k++) {
        float hi, lo;
        tc::split(x[k], hi, lo);
        part[k] = half ? lo : hi;
      }
      tc::tmem_st16(tmem_row + (half ? ActTc::cXl : ActTc::cXh), part);
      tc::tmem_st_wait();
    }
    tc::fence_before_sync();
    __syncthreads();
#pragma unroll 1
    for (int t = 1; t >= 0; t--) {  // value tower first, as in act_kernel
      if (tid == 0) {
        tc::fence_after_sync();
        tc_gemm3<64, K1>(tmem + ActTc::cD, tmem + ActTc::cXh, tmem + ActTc::cXl, tc::smem_u32(W1(t, 0)), tc::smem_u32(W1(t, 1)), tc::idesc_tf32(TM, 64));
        tc::mma_commit(bar);
      }
      tc::bar_wait(bar, phase); phase ^= 1;
      tc::fence_after_sync();
      tc_epilogue_tanh(tmem_row, 32 * half, b1 + 64 * t);
      tc::fence_before_sync();
      __syncthreads();
      if (tid == 0) {
        tc::fence_after_sync();
        tc_gemm3<64, HID>(tmem + ActTc::cD, tmem + ActTc::cAh, tmem + ActTc::cAl, tc::smem_u32(W2(t, 0)), tc::smem_u32(W2(t, 1)), tc::idesc_tf32(TM, 64));
        tc::mma_commit(bar);
      }
      tc::bar_wait(bar, phase); phase ^= 1;
      tc::fence_after_sync();
      tc_epilogue_tanh(tmem_row, 32 * half, b2 + 64 * t);  // h2 over h1: the layer-2 MMAs have finished reading it
      tc::fence_before_sync();
      __syncthreads();
      if (tid == 0) {
        tc::fence_after_sync();
        tc_gemm3<16, HID>(tmem + ActTc::cHead + 16 * t, tmem + ActTc::cAh, tmem + ActTc::cAl, tc::smem_u32(W3(t, 0)), tc::smem_u32(W3(t, 1)),
                          tc::idesc_tf32(TM, 16));
        tc::mma_commit(bar);
      }
      tc::bar_wait(bar, phase); phase ^= 1;  // the head has consumed h2: the next tower may overwrite A
      tc::fence_after_sync();
      __syncthreads();  // no thread is still polling this phase when the next commit arrives
    }
    // heads: warpgroup 0 samples the action from the six means, warpgroup 1 stores the value
    float o16[16];
    tc::tmem_ld16(tmem_row + ActTc::cHead + 16 * (half ? 1 : 0), o16);
    if constexpr (SDE) {  // the policy tower's h2 = hi + lo (exact) is still in TMEM: warpgroup w takes features 32 w .. 32 w + 31
      float nz[ACT], vr[ACT];
#pragma unroll
      for (int c = 0; c < 2; c++) {
        float hi[16], lo[16], h[16], pn[ACT], pv[ACT];
        tc::tmem_ld16(tmem_row + ActTc::cAh + 32 * half + 16 * c, hi);
        tc::tmem_ld16(tmem_row + ActTc::cAl + 32 * half + 16 * c, lo);
#pragma unroll
        for (int i = 0; i < 16; i++) h[i] = hi[i] + lo[i];
        sde_partial(h, 32 * half + 16 * c, seed_lo, seed_hi, (unsigned)(env_offset + g), tick, !deterministic && g < n, sstd, sS, pn, pv);
#pragma unroll
        for (int j = 0; j < ACT; j++) {
          if (c == 0) { nz[j] = pn[j]; vr[j] = pv[j]; }
          else { nz[j] = nz[j] + pn[j]; vr[j] = vr[j] + pv[j]; }
        }
      }
      if (half) {
#pragma unroll
        for (int j = 0; j < ACT; j++) { xch[j * TM + row] = nz[j]; xch[(ACT + j) * TM + row] = vr[j]; }
      }
      __syncthreads();
      if (g < n) {
        if (half) {
          if (value) value[g] = o16[0] + b3[8];
        } else {
          float lp = 0.0f;
#pragma unroll
          for (int k = 0; k < ACT; k++) {
            const float mean = o16[k] + b3[k], a = deterministic ? mean : mean + (nz[k] + xch[k * TM + row]);
            const float v = (vr[k] + xch[(ACT + k) * TM + row]) + kSdeEps, d = a - mean;
            lp += sde_logp_term(d, v, 1.0f / v);
            if (act_raw) act_raw[(size_t)g * ACT + k] = a;
            if (act_clip) act_clip[(size_t)g * ACT + k] = fminf(fmaxf(a, -1.0f), 1.0f);
          }
          if (logp) logp[g] = lp;
        }
      }
    } else if (g < n) {
      if (half) {
        if (value) value[g] = o16[0] + b3[8];
      } else {
        float eps[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (!deterministic) {  // 8 standard normals from two Philox blocks (Box-Muller), as act_kernel
#pragma unroll
          for (int b = 0; b < 2; b++) {
            const uint4 r = philox4x32(seed_lo, seed_hi, (unsigned)(env_offset + g), tick, 0x5050u + b, 0u);
            const unsigned w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
            for (int q = 0; q < 2; q++) {
              const float u1 = ((float)(w[2 * q] >> 8) + 0.5f) * (1.0f / 16777216.0f), u2 = (float)(w[2 * q + 1] >> 8) * (1.0f / 16777216.0f);
              const float rad = sqrtf(-2.0f * logf(u1));
              float sn, cs;
              sincospif(2.0f * u2, &sn, &cs);
              eps[4 * b + 2 * q] = rad * cs; eps[4 * b + 2 * q + 1] = rad * sn;
            }
          }
        }
        float lp = 0.0f;
#pragma unroll
        for (int k = 0; k < ACT; k++) {
          const float mean = o16[k] + b3[k], a = mean + expf(ls[k]) * eps[k];
          lp += -0.5f * eps[k] * eps[k] - ls[k] - LOG_SQRT_2PI;
          if (act_raw) act_raw[(size_t)g * ACT + k] = a;
          if (act_clip) act_clip[(size_t)g * ACT + k] = fminf(fmaxf(a, -1.0f), 1.0f);
        }
        if (logp) logp[g] = lp;
      }
    }
    tc::fence_before_sync();
    __syncthreads();  // every thread has read its head row: the next tile may overwrite TMEM
  }
  if (warp == 0) tc::tmem_free<256>(tmem);
}

// value tower for single rows, weights from global memory: used where truncations (rare) need V(terminal_obs)
__device__ inline float value_one(const Layout& L, const float* __restrict__ P, const float* __restrict__ x) {
  float h1[HID];
  for (int m = 0; m < HID; m++) {
    float s = P[L.b1[1] + m];
    for (int k = 0; k < L.od; k++) s = fmaf(P[L.W1[1] + m * L.od + k], x[k], s);
    h1[m] = tanhf(s);
  }
  float v = P[L.b3[1]];
  for (int m = 0; m < HID; m++) {
    float s = P[L.b2[1] + m];
    for (int k = 0; k < HID; k++) s = fmaf(P[L.W2[1] + m * HID + k], h1[k], s);
    v = fmaf(P[L.W3[1] + m], tanhf(s), v);
  }
  return v;
}

__global__ void __launch_bounds__(256) post_step_kernel(Layout L, const float* __restrict__ P, int n, const float* __restrict__ reward,
                                                        const uint8_t* __restrict__ term, const uint8_t* __restrict__ trunc,
                                                        const float* __restrict__ tobs, const float* __restrict__ ep_return,
                                                        const int32_t* __restrict__ ep_len, float gamma, float* reward_out, float* done_out,
                                                        double* acc) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  float r = 0.0f, er = 0.0f, el = 0.0f, dn = 0.0f;
  if (i < n) {
    r = reward[i];
    const bool tr = trunc[i] != 0, done = tr || term[i] != 0;
    float ro = r;
    if (tr) {  // TimeLimit bootstrap (SB3 on_policy_algorithm.collect_rollouts); a non-finite value never enters the returns
      const float boot = gamma * value_one(L, P, tobs + (size_t)i * L.od);
      if (isfinite(boot)) ro += boot;
    }
    reward_out[i] = ro;
    done_out[i] = done ? 1.0f : 0.0f;
    if (done) { er = ep_return[i]; el = (float)ep_len[i]; dn = 1.0f; }
  }
  __shared__ float red[4][8];
  float v[4] = {r, er, el, dn};
#pragma unroll
  for (int k = 0; k < 4; k++) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
    if ((threadIdx.x & 31) == 0) red[k][threadIdx.x >> 5] = v[k];
  }
  __syncthreads();
  if (threadIdx.x < 4) {
    double s = 0.0;
    for (int w = 0; w < 8; w++) s += (double)red[threadIdx.x][w];
    if (s != 0.0) atomicAdd(&acc[threadIdx.x], s);
  }
}

__global__ void __launch_bounds__(256) gae_kernel(const float* __restrict__ rew, const float* __restrict__ val, const float* __restrict__ done,
                                                  const float* __restrict__ last_val, int T, int N, float gamma, float lam, float* adv, float* ret) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  float last = 0.0f, nxt = last_val[i];
  for (int t = T - 1; t >= 0; t--) {
    const size_t o = (size_t)t * N + i;
    const float nonterm = 1.0f - done[o], v = val[o];
    const float delta = rew[o] + gamma * nxt * nonterm - v;
    last = delta + gamma * lam * nonterm * last;
    adv[o] = last;
    ret[o] = last + v;
    nxt = v;
  }
}

// ------------------------------------------------------------------------------------------------ minibatch sampling
// A keyed pseudo-random PERMUTATION of [0, n) computed element-wise (SB3 draws np.random.permutation per epoch): a
// 6-round balanced Feistel network on 2*ceil(bits/2) bits with cycle walking back into [0, n).  Every index appears
// exactly once per epoch whatever the key; one launch instead of torch.randperm's key generation + radix sort.
__device__ __forceinline__ unsigned feistel_round(unsigned x, unsigned k) {
  x = (x ^ k) * 0x9E3779B1u;
  x ^= x >> 15;
  x *= 0x85EBCA77u;
  x ^= x >> 13;
  return x;
}
__global__ void __launch_bounds__(256) permutation_kernel(int n, int half_bits, unsigned k0, unsigned k1, int64_t* out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned mask = (1u << half_bits) - 1u;
  unsigned x = (unsigned)i;
  do {  // cycle walking: the network permutes [0, 2^(2 half_bits)), which is < 4 n
    unsigned l = x >> half_bits, r = x & mask;
#pragma unroll
    for (int rd = 0; rd < 6; rd++) {
      const unsigned f = feistel_round(r, (rd & 1 ? k1 : k0) + 0x632BE5ABu * (unsigned)rd) & mask;
      const unsigned nl = r;
      r = l ^ f;
      l = nl;
    }
    x = (l << half_bits) | r;
  } while (x >= (unsigned)n);
  out[i] = (int64_t)x;
}

// ------------------------------------------------------------------------------------------------ minibatch gradient
// Per-CTA partial sums (fp64) of adv[idx] and its square over the minibatch; the gradient kernel combines the partials in
// a fixed order (deterministic) into mean and 1 / (unbiased std + 1e-8).
constexpr int kStatCtas = 128;
__global__ void __launch_bounds__(256) adv_stats_kernel(const float* __restrict__ adv, const int64_t* __restrict__ idx, int mb, double* part) {
  __shared__ double red[2][8];
  const int tid = threadIdx.x;
  double s = 0.0, q = 0.0;
  for (int e = blockIdx.x * 256 + tid; e < mb; e += gridDim.x * 256) { const double a = (double)adv[idx[e]]; s += a; q += a * a; }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) { s += __shfl_xor_sync(0xffffffffu, s, o); q += __shfl_xor_sync(0xffffffffu, q, o); }
  if ((tid & 31) == 0) { red[0][tid >> 5] = s; red[1][tid >> 5] = q; }
  __syncthreads();
  if (tid < 2) {
    double t = 0.0;
    for (int w = 0; w < 8; w++) t += red[tid][w];
    part[2 * blockIdx.x + tid] = t;
  }
}

// ---- geometry of the gradient kernel: tiles of GT = 32 samples so that TWO CTAs fit one SM (109 KB each) and overlap each
// other's barriers, loss phases and epilogues; [feature][sample] matrices use row stride LDG = 40 (= 8 mod 32)
constexpr int GT = 32, LDG = 40;
constexpr int kGradSmemFloats = 2 * tower_floats(false)  // weights of both towers (W2 once: the back-prop product reads it row-major)
                                + K1 * LDG               // X
                                + 2 * HID * LDG          // H1 (later dZ2), H2   [feature][sample]
                                + 3 * GT * LD            // H1T, dZ2T, dZ1T      [sample][feature]
                                + 8 * GT + 8 * GT        // head outputs, head gradients
                                + 6 * GT + 4 * GT + 32 * GT + 16;  // actions, (logp_old, adv, ret, valid), head scratch, log_std
static_assert(kGradSmemFloats * 4 <= 113 * 1024, "two gradient CTAs must fit one SM");
constexpr int kGradSmemFloatsSde = kGradSmemFloats + HID * ACT + 2 * ACT * GT;  // + S = exp(2 log_std), var and dL/dvar per sample
static_assert(kGradSmemFloatsSde * 4 <= 113 * 1024, "two gSDE gradient CTAs must fit one SM");
// the gSDE arrays behind log_std[16]: S = exp(2 log_std) [HID][ACT], var and dL/dvar [ACT][GT]
struct GradSde {
  float *S, *var, *dvar;
  __device__ __forceinline__ static GradSde at(float* ls) { return GradSde{ls + 16, ls + 16 + HID * ACT, ls + 16 + HID * ACT + ACT * GT}; }
};

// A given row-major (A[m][k] at Ar[m * lda + k]) instead of K-major: same MMA, 2-way conflicted fragment loads
template <int K, int NTILE, int lda, int ldb>
__device__ __forceinline__ void gemm_mma_rowA(const float* __restrict__ Ar, const float* __restrict__ Bm, const Own& o, float (&acc)[NTILE][4]) {
#pragma unroll 2
  for (int k0 = 0; k0 < K; k0 += 8) {
    const float* ap = Ar + (o.m0 + o.g) * lda + k0 + o.t;
    uint32_t ah[4], al[4];
    split_tf32(ap[0], ah[0], al[0]);
    split_tf32(ap[8 * lda], ah[1], al[1]);
    split_tf32(ap[4], ah[2], al[2]);
    split_tf32(ap[8 * lda + 4], ah[3], al[3]);
    const float* bp = Bm + (k0 + o.t) * ldb + o.n0 + o.g;
#pragma unroll
    for (int j = 0; j < NTILE; j++) {
      uint32_t bh[2], bl[2];
      split_tf32(bp[8 * j], bh[0], bl[0]);
      split_tf32(bp[4 * ldb + 8 * j], bh[1], bl[1]);
      mma_tf32(acc[j], al, bh);
      mma_tf32(acc[j], ah, bl);
      mma_tf32(acc[j], ah, bh);
    }
  }
}
// h = tanh(acc + bias[row]) for a 16 x 16 warp slab -> H[row][col] (ld LDG) and, if HT, HT[col][row] (ld LD)
__device__ __forceinline__ void store_tanh_g(const float (&acc)[2][4], const float* bias, const Own& o, float* H, float* HT) {
#pragma unroll
  for (int i = 0; i < 2; i++) {
    const int r = o.row(i);
    const float bi = bias[r];
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const float h0 = tanhf(acc[j][2 * i] + bi), h1 = tanhf(acc[j][2 * i + 1] + bi);
      const int c = o.col(j, 0);
      *reinterpret_cast<float2*>(H + r * LDG + c) = make_float2(h0, h1);
      if (HT) { HT[c * LD + r] = h0; HT[(c + 1) * LD + r] = h1; }
    }
  }
}
// out[o][s] = b3[o] + sum_k W3[o][k] H2[k][s] for GT samples: threads 0..127 = 4 k-groups x 32 samples; ends synchronised
template <int NOUT>
__device__ __forceinline__ void head_forward_g(const TowerS& T, const float* H2, float* out, float* scratch) {
  const int kg = threadIdx.x >> 5, s = threadIdx.x & 31;
  if (threadIdx.x < 4 * GT) {
    float acc[NOUT];
#pragma unroll
    for (int o = 0; o < NOUT; o++) acc[o] = 0.0f;
#pragma unroll
    for (int k = 16 * kg; k < 16 * kg + 16; k++) {
      const float h = H2[k * LDG + s];
#pragma unroll
      for (int o = 0; o < NOUT; o++) acc[o] = fmaf(T.W3[o * HID + k], h, acc[o]);
    }
#pragma unroll
    for (int o = 0; o < NOUT; o++) scratch[(kg * 8 + o) * GT + s] = acc[o];
  }
  __syncthreads();
  for (int e = threadIdx.x; e < NOUT * GT; e += NT) {
    const int o = e / GT, c = e % GT;
    out[e] = T.b3[o] + ((scratch[o * GT + c] + scratch[(8 + o) * GT + c]) + (scratch[(16 + o) * GT + c] + scratch[(24 + o) * GT + c]));
  }
  __syncthreads();
}

template <bool SDE>
__global__ void __launch_bounds__(NT, 2) grad_kernel(Layout L, const float* __restrict__ P, const float* __restrict__ obs, const float* __restrict__ act,
                                                    const float* __restrict__ logp_old, const float* __restrict__ adv, const float* __restrict__ ret,
                                                    const int64_t* __restrict__ idx, int mb, const double* __restrict__ adv_part, float clip,
                                                    float vf_coef, float ent_coef, int normalize, float* __restrict__ gpart) {
  extern __shared__ __align__(16) float sm[];
  TowerS T[2];
  float* p = carve_tower(sm, T[0], false);
  p = carve_tower(p, T[1], false);
  float* X = p; p += K1 * LDG;
  float* H1 = p; p += HID * LDG;   // h1, then dZ2 ([feature][sample]) once the second layer has consumed it
  float* H2 = p; p += HID * LDG;
  float* H1T = p; p += GT * LD;
  float* dZ2T = p; p += GT * LD;
  float* dZ1T = p; p += GT * LD;
  float* out = p; p += 8 * GT;
  float* dOut = p; p += 8 * GT;
  float* sAct = p; p += 6 * GT;
  float* sOld = p; p += GT;
  float* sAdv = p; p += GT;
  float* sRet = p; p += GT;
  float* sValid = p; p += GT;
  float* scratch = p; p += 32 * GT;
  float* ls = p;  // log_std[6]; (SDE) then the GradSde arrays (addressed only inside the SDE branches)

  const int tid = threadIdx.x, od = L.od, w = tid >> 5, lane = tid & 31;
  const Own oA{16 * (w & 3), 16 * (w >> 2), lane >> 2, lane & 3};  // 64 features x 32 samples: 16 x 16 per warp
  const Own oW{16 * (w & 3), 32 * (w >> 2), lane >> 2, lane & 3};  // dW2, 64 x 64: 16 x 32 per warp
  const Own o1{0, 8 * w, lane >> 2, lane & 3};                     // dW1^T, 16 inputs x 64 outputs: 16 x 8 per warp
  const int sg = tid >> 6, fk = tid & 63;  // (group of 8 samples, feature) mapping of the reductions over a tile's samples
  load_tower(L, P, 0, T[0], false);
  load_tower(L, P, 1, T[1], false);
  if constexpr (SDE) {
    float* sS = GradSde::at(ls).S;
    for (int e = tid; e < HID * ACT; e += NT) sS[e] = expf(2.0f * P[L.log_std + e]);
  } else {
    if (tid < ACT) ls[tid] = P[L.log_std + tid];
  }
  float a_mean = 0.0f, a_rstd = 1.0f;
  if (normalize) {  // every thread combines the partials in the same order: identical values everywhere
    double s1 = 0.0, s2 = 0.0;
    for (int c = 0; c < kStatCtas; c++) { s1 += adv_part[2 * c]; s2 += adv_part[2 * c + 1]; }
    const double mean = s1 / mb, var = fmax(s2 - s1 * mean, 0.0) / (mb > 1 ? mb - 1 : 1);
    a_mean = (float)mean;
    a_rstd = (float)(1.0 / (sqrt(var) + 1e-8));
  }
  const float inv_mb = 1.0f / (float)mb;

  // gradient accumulators, persistent over the CTA's tiles; each thread owns fixed parameters of both towers
  //   gW2 / gW1: the thread's MMA accumulator fragments of dW2 (dW1^T);  gW3p / gb2p / gb1p: partial sums over the thread's
  //   8-sample group (combined across the 4 groups at the end);  gOut / gLs / loss sums: per sample slot (threads 0..31)
  //   (SDE: gLs holds the partial sums of dvar_sj h2_sk^2 over the thread's 8-sample group for k = fk, all six j)
  float gW2[2][4][4], gW1[2][1][4], gW3p[ACT + 1], gb2p[2] = {0, 0}, gb1p[2] = {0, 0}, gOut[ACT + 1], gLs[ACT];
  float sPg = 0.0f, sV = 0.0f, sKl = 0.0f;
#pragma unroll
  for (int t = 0; t < 2; t++) {
    zero_acc(gW2[t]);
    zero_acc(gW1[t]);
  }
#pragma unroll
  for (int o = 0; o < ACT + 1; o++) { gW3p[o] = 0.0f; gOut[o] = 0.0f; }
#pragma unroll
  for (int o = 0; o < ACT; o++) gLs[o] = 0.0f;

  // ---- software-pipelined gather: the rows of tile i+1 are fetched (through indices loaded one tile earlier) while tile i
  //      is computed, so the idx -> obs dependent global loads never sit on the critical path
  const int ntiles = (mb + GT - 1) / GT;
  const int gs = tid >> 4, gf = tid & 15;      // this thread stages feature gf of samples gs and gs + 16
  int nidx[2] = {-1, -1}, nsi = -1;            // sample indices of the NEXT tile (-1 = past the end)
  float px[2] = {0.0f, 0.0f}, pa[ACT] = {0, 0, 0, 0, 0, 0}, pold = 0.0f, padv = 0.0f, pret = 0.0f, pvalid = 0.0f;
  auto load_indices = [&](int tile) {
#pragma unroll
    for (int j = 0; j < 2; j++) {
      const int g = tile * GT + gs + 16 * j;
      nidx[j] = (tile < ntiles && g < mb) ? (int)idx[g] : -1;
    }
    const int g = tile * GT + tid;
    nsi = (tid < GT && tile < ntiles && g < mb) ? (int)idx[g] : -1;
  };
  auto load_values = [&]() {
#pragma unroll
    for (int j = 0; j < 2; j++) px[j] = (nidx[j] >= 0 && gf < od) ? obs[(size_t)nidx[j] * od + gf] : 0.0f;
    if (tid < GT) {
      const bool valid = nsi >= 0;
      const size_t src = valid ? (size_t)nsi : 0;
#pragma unroll
      for (int k = 0; k < ACT; k++) pa[k] = valid ? act[src * ACT + k] : 0.0f;
      pold = valid ? logp_old[src] : 0.0f;
      padv = valid ? adv[src] : 0.0f;
      pret = valid ? ret[src] : 0.0f;
      pvalid = valid ? 1.0f : 0.0f;
    }
  };
  load_indices(blockIdx.x);
  load_values();
  load_indices(blockIdx.x + gridDim.x);
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
    __syncthreads();  // the previous tile's buffers are free (also orders the weight loads before first use)
#pragma unroll
    for (int j = 0; j < 2; j++) X[gf * LDG + gs + 16 * j] = px[j];
    if (tid < GT) {
#pragma unroll
      for (int k = 0; k < ACT; k++) sAct[k * GT + tid] = pa[k];
      sOld[tid] = pold; sAdv[tid] = padv; sRet[tid] = pret; sValid[tid] = pvalid;
    }
    load_values();                                 // rows of the next tile (indices arrived during the previous tile)
    load_indices(tile + 2 * (int)gridDim.x);       // indices of the tile after that
    __syncthreads();
#pragma unroll
    for (int t = 0; t < 2; t++) {  // unrolled: the accumulators of both towers stay in registers
      const TowerS& W = T[t];
      const int nout = t == 0 ? ACT : 1;
      {
        float acc[2][4];
        zero_acc(acc);
        gemm_mma<K1, 2, LD, LDG>(W.W1t, X, oA, acc);
        store_tanh_g(acc, W.b1, oA, H1, H1T);
        __syncthreads();
        zero_acc(acc);
        gemm_mma<HID, 2, LD, LDG>(W.W2t, H1, oA, acc);
        store_tanh_g(acc, W.b2, oA, H2, nullptr);
        __syncthreads();
      }
      if (t == 0) head_forward_g<ACT>(W, H2, out, scratch);
      else head_forward_g<1>(W, H2, out, scratch);
      if constexpr (SDE) {
        if (t == 0) {  // var[j][s] = sum_k fl(h2_ks^2) S_kj: the head's shape and order (4 groups of 16 k), h2^2 in, S as weights
          const GradSde X2 = GradSde::at(ls);
          const float *sS = X2.S;
          float* sVar = X2.var;
          const int kg = tid >> 5, s = tid & 31;
          if (tid < 4 * GT) {
            float acc[ACT];
#pragma unroll
            for (int j = 0; j < ACT; j++) acc[j] = 0.0f;
#pragma unroll
            for (int k = 16 * kg; k < 16 * kg + 16; k++) {
              const float h = H2[k * LDG + s], h2 = h * h;
#pragma unroll
              for (int j = 0; j < ACT; j++) acc[j] = fmaf(h2, sS[k * ACT + j], acc[j]);
            }
#pragma unroll
            for (int j = 0; j < ACT; j++) scratch[(kg * 8 + j) * GT + s] = acc[j];
          }
          __syncthreads();
          for (int e = tid; e < ACT * GT; e += NT) {
            const int j = e / GT, c = e % GT;
            sVar[e] = (scratch[j * GT + c] + scratch[(8 + j) * GT + c]) + (scratch[(16 + j) * GT + c] + scratch[(24 + j) * GT + c]);
          }
          __syncthreads();
        }
      }
      // ---- loss and its gradient with respect to the head outputs (one thread per sample)
      if (tid < GT) {
        const float valid = sValid[tid];
        if (t == 0) {
          float lp = 0.0f, d[ACT], isig2[ACT];
#pragma unroll
          for (int k = 0; k < ACT; k++) {
            if constexpr (SDE) {
              const float v = GradSde::at(ls).var[k * GT + tid] + kSdeEps;
              isig2[k] = 1.0f / v;
              d[k] = sAct[k * GT + tid] - out[k * GT + tid];
              lp += sde_logp_term(d[k], v, isig2[k]);
            } else {
              isig2[k] = expf(-2.0f * ls[k]);
              d[k] = sAct[k * GT + tid] - out[k * GT + tid];
              lp += -0.5f * d[k] * d[k] * isig2[k] - ls[k] - LOG_SQRT_2PI;
            }
          }
          const float lr = lp - sOld[tid], ratio = expf(lr);
          const float A = (sAdv[tid] - a_mean) * a_rstd;
          const float lo = 1.0f - clip, hi = 1.0f + clip;
          const float x1 = A * ratio, x2 = A * fminf(fmaxf(ratio, lo), hi);
          const bool inside = ratio >= lo && ratio <= hi;
          // d min(x1, x2) / d lp with torch's tie rule (half to each operand) and clamp's inclusive pass-through
          float g = 0.0f;
          if (x1 < x2) g = x1;
          else if (x1 > x2) g = inside ? x1 : 0.0f;
          else g = 0.5f * x1 + (inside ? 0.5f * x1 : 0.0f);
          const float dlp = -g * inv_mb * valid;
#pragma unroll
          for (int k = 0; k < ACT; k++) {
            const float dm = dlp * d[k] * isig2[k];
            dOut[k * GT + tid] = dm;
            gOut[k] += dm;  // d b3
            // d/d log_std of the diagonal Gaussian; for gSDE the same bracket is d/d log(var): dL/dvar = bracket / (2 var)
            if constexpr (SDE) GradSde::at(ls).dvar[k * GT + tid] = 0.5f * (dlp * (d[k] * d[k] * isig2[k] - 1.0f) - ent_coef * inv_mb * valid) * isig2[k];
            else gLs[k] += dlp * (d[k] * d[k] * isig2[k] - 1.0f) - ent_coef * inv_mb * valid;
          }
          sPg += -fminf(x1, x2) * valid;
          sKl += ((ratio - 1.0f) - lr) * valid;
        } else {
          const float e = out[tid] - sRet[tid], dv = 2.0f * e * vf_coef * inv_mb * valid;
          dOut[tid] = dv;
          gOut[ACT] += dv;
          sV += e * e * valid;
        }
      }
      __syncthreads();
      // ---- back through the head and the second tanh: dZ2 = (W3^T dOut) * (1 - H2^2) -> the H1 buffer ([feature][sample],
      //      h1 itself lives on in H1T) and dZ2T; H2 stays intact for the dW3 sums below
      {
        float w3[2][ACT];
#pragma unroll
        for (int i = 0; i < 2; i++)
#pragma unroll
          for (int q = 0; q < ACT; q++) w3[i][q] = q < nout ? W.W3[q * HID + oA.row(i)] : 0.0f;
#pragma unroll
        for (int j = 0; j < 2; j++) {
          const int c = oA.col(j, 0);
          float d[2][2] = {{0.0f, 0.0f}, {0.0f, 0.0f}};
#pragma unroll
          for (int q = 0; q < ACT; q++) {
            if (q >= nout) break;
            const float2 g2 = *reinterpret_cast<const float2*>(dOut + q * GT + c);
#pragma unroll
            for (int i = 0; i < 2; i++) { d[i][0] = fmaf(w3[i][q], g2.x, d[i][0]); d[i][1] = fmaf(w3[i][q], g2.y, d[i][1]); }
          }
#pragma unroll
          for (int i = 0; i < 2; i++) {
            const int r = oA.row(i);
            float2 h = *reinterpret_cast<const float2*>(H2 + r * LDG + c);
            h.x = d[i][0] * (1.0f - h.x * h.x); h.y = d[i][1] * (1.0f - h.y * h.y);
            *reinterpret_cast<float2*>(H1 + r * LDG + c) = h;
            dZ2T[c * LD + r] = h.x; dZ2T[(c + 1) * LD + r] = h.y;
          }
        }
      }
      __syncthreads();
      // ---- dZ1 = (W2^T dZ2) * (1 - h1^2) -> dZ1T only (nothing propagates to the observations); W2^T read from W2t row-major
      {
        float acc[2][4];
        zero_acc(acc);
        gemm_mma_rowA<HID, 2, LD, LDG>(W.W2t, H1, oA, acc);
#pragma unroll
        for (int i = 0; i < 2; i++) {
          const int r = oA.row(i);
#pragma unroll
          for (int j = 0; j < 2; j++) {
            const int c = oA.col(j, 0);
            const float h0 = H1T[c * LD + r], h1 = H1T[(c + 1) * LD + r];
            dZ1T[c * LD + r] = acc[j][2 * i] * (1.0f - h0 * h0);
            dZ1T[(c + 1) * LD + r] = acc[j][2 * i + 1] * (1.0f - h1 * h1);
          }
        }
      }
      __syncthreads();
      // ---- weight gradients (inner dimension = the tile's samples), accumulated in the persistent MMA fragments
      gemm_mma<GT, 4, LD, LD>(dZ2T, H1T, oW, gW2[t]);          // dW2[out][in] += dZ2[out][s] h1[in][s]
      gemm_mma_rowA<GT, 1, LDG, LD>(X, dZ1T, o1, gW1[t]);      // dW1^T[in][out] += X[in][s] dZ1[out][s]
      // dW3[o][k = fk] and the hidden biases: partial sums over this thread's 8 samples
#pragma unroll
      for (int s0 = 8 * sg; s0 < 8 * sg + 8; s0 += 4) {
        const float4 h4 = *reinterpret_cast<const float4*>(H2 + fk * LDG + s0);
        const float h[4] = {h4.x, h4.y, h4.z, h4.w};
#pragma unroll
        for (int i = 0; i < 4; i++) {
          gb2p[t] += dZ2T[(s0 + i) * LD + fk];
          gb1p[t] += dZ1T[(s0 + i) * LD + fk];
        }
#pragma unroll
        for (int q = 0; q < ACT; q++) {
          if (q >= nout) break;
          const float4 g4 = *reinterpret_cast<const float4*>(dOut + q * GT + s0);  // warp broadcast
          float& acc = gW3p[t == 0 ? q : ACT];
          acc = fmaf(g4.x, h[0], acc); acc = fmaf(g4.y, h[1], acc); acc = fmaf(g4.z, h[2], acc); acc = fmaf(g4.w, h[3], acc);
        }
        if constexpr (SDE) {
          if (t == 0) {  // sum_s dvar_sj fl(h2_sk^2): dW3's sum with h2^2 in place of h2
#pragma unroll
            for (int j = 0; j < ACT; j++) {
              const float4 g4 = *reinterpret_cast<const float4*>(GradSde::at(ls).dvar + j * GT + s0);
              float& acc = gLs[j];
              acc = fmaf(g4.x, h[0] * h[0], acc); acc = fmaf(g4.y, h[1] * h[1], acc); acc = fmaf(g4.z, h[2] * h[2], acc); acc = fmaf(g4.w, h[3] * h[3], acc);
            }
          }
        }
      }
      __syncthreads();  // the next tower (or tile) overwrites the activation buffers
    }
  }

  // ---- per-CTA partials: every parameter index is written by exactly one thread
  float* G = gpart + (size_t)blockIdx.x * (L.total + 4);
#pragma unroll
  for (int t = 0; t < 2; t++) {
#pragma unroll
    for (int i = 0; i < 2; i++) {
#pragma unroll
      for (int e = 0; e < 2; e++) {
#pragma unroll
        for (int j = 0; j < 4; j++) G[L.W2[t] + oW.row(i) * HID + oW.col(j, e)] = gW2[t][j][2 * i + e];
        if (o1.row(i) < od) G[L.W1[t] + o1.col(0, e) * od + o1.row(i)] = gW1[t][0][2 * i + e];  // fragment holds dW1^T[in][out]
      }
    }
  }
  __syncthreads();
  float* scr = H1T;  // H1T, dZ2T, dZ1T are contiguous and free now: combine the four sample groups / the 32 sample slots
#pragma unroll
  for (int o = 0; o < ACT + 1; o++) scr[(sg * 8 + o) * HID + fk] = gW3p[o];
#pragma unroll
  for (int t = 0; t < 2; t++) { scr[2048 + (2 * t) * 256 + sg * HID + fk] = gb2p[t]; scr[2048 + (2 * t + 1) * 256 + sg * HID + fk] = gb1p[t]; }
  if constexpr (SDE) {
    for (int j = 0; j < ACT; j++) scr[3072 + (sg * ACT + j) * HID + fk] = gLs[j];
  }
  __syncthreads();
  if constexpr (SDE) {  // d log_std_kj = 2 S_kj sum_s dvar_sj h2_sk^2, the four sample groups combined as for dW3
    for (int e = tid; e < HID * ACT; e += NT) {
      const int k = e / ACT, j = e % ACT;
      const float* q = scr + 3072 + j * HID + k;
      G[L.log_std + e] = 2.0f * GradSde::at(ls).S[e] * ((q[0] + q[ACT * HID]) + (q[2 * ACT * HID] + q[3 * ACT * HID]));
    }
  }
  for (int e = tid; e < (ACT + 1) * HID; e += NT) {
    const int o = e / HID, k = e % HID;
    const float v = (scr[o * HID + k] + scr[(8 + o) * HID + k]) + (scr[(16 + o) * HID + k] + scr[(24 + o) * HID + k]);
    G[(o < ACT ? L.W3[0] + o * HID : L.W3[1]) + k] = v;
  }
  {
    const int which = tid >> 6;  // 0: pi b2, 1: pi b1, 2: vf b2, 3: vf b1
    const float* q = scr + 2048 + which * 256;
    const float v = (q[fk] + q[HID + fk]) + (q[2 * HID + fk] + q[3 * HID + fk]);
    G[(which == 0 ? L.b2[0] : which == 1 ? L.b1[0] : which == 2 ? L.b2[1] : L.b1[1]) + fk] = v;
  }
  __syncthreads();
  if (tid < GT) {
#pragma unroll
    for (int o = 0; o < ACT; o++) { scr[o * GT + tid] = gOut[o]; scr[(ACT + o) * GT + tid] = gLs[o]; }
    scr[12 * GT + tid] = gOut[ACT]; scr[13 * GT + tid] = sPg; scr[14 * GT + tid] = sV; scr[15 * GT + tid] = sKl;
  }
  __syncthreads();
  if (tid < 16 && !(SDE && tid >= ACT && tid < 2 * ACT)) {  // (gSDE: log_std was written above)
    float v = 0.0f;
    for (int k = 0; k < GT; k++) v += scr[tid * GT + k];
    const int dst = tid < ACT ? L.b3[0] + tid : tid < 2 * ACT ? L.log_std + tid - ACT : tid == 12 ? L.b3[1] : L.total + tid - 13;
    G[dst] = v;
  }
}

// grad[i] = sum over CTAs of the partials (fixed order); loss_out = the three loss sums / mb
__global__ void __launch_bounds__(256) reduce_kernel(const float* __restrict__ gpart, int nparts, int total, int mb, float* grad, float* loss_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= total + 3) return;
  float s = 0.0f;
  for (int c = 0; c < nparts; c++) s += gpart[(size_t)c * (total + 4) + i];
  if (i < total) grad[i] = s;
  else if (loss_out) loss_out[i - total] = s / (float)mb;
}

// clip_grad_norm_ + Adam, single CTA (the parameter vector has ~10^4 entries)
__global__ void __launch_bounds__(1024) adam_kernel(int n, float* P, const float* __restrict__ grad, float* m, float* v, int32_t* step, float gscale,
                                                    float max_norm, float lr, float b1, float b2, float eps) {
  __shared__ float red[32];
  __shared__ float s_coef;
  const int tid = threadIdx.x;
  float q = 0.0f;
  for (int i = tid; i < n; i += 1024) { const float g = grad[i] * gscale; q = fmaf(g, g, q); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  if ((tid & 31) == 0) red[tid >> 5] = q;
  __syncthreads();
  if (tid == 0) {
    float s = 0.0f;
    for (int w = 0; w < 32; w++) s += red[w];
    const float norm = sqrtf(s);
    s_coef = max_norm > 0.0f ? fminf(max_norm / (norm + 1e-6f), 1.0f) : 1.0f;
    *step += 1;
  }
  __syncthreads();
  const float coef = s_coef * gscale;
  const int t = *step;
  const float bc1 = 1.0f - powf(b1, (float)t), bc2 = 1.0f - powf(b2, (float)t);
  const float step_size = lr / bc1, rsq_bc2 = rsqrtf(bc2);
  for (int i = tid; i < n; i += 1024) {
    const float g = grad[i] * coef;
    const float mi = b1 * m[i] + (1.0f - b1) * g, vi = b2 * v[i] + (1.0f - b2) * g * g;
    m[i] = mi; v[i] = vi;
    P[i] -= step_size * mi / (sqrtf(vi) * rsq_bc2 + eps);
  }
}

}  // namespace ppo

// ------------------------------------------------------------------------------------------------ C ABI
extern "C" {

int so100_ppo_param_count(int obs_dim) {
  if (obs_dim < 1 || obs_dim > ppo::K1) return fail(SO100_ERR_ARG, "obs_dim must be 1..16");
  return ppo::make_layout(obs_dim).total;
}
int64_t so100_ppo_workspace_floats(int obs_dim) {
  const int n = so100_ppo_param_count(obs_dim);
  return n < 0 ? n : (int64_t)SO100_PPO_MAX_CTAS * (n + 4) + 4 * ppo::kStatCtas;
}
int so100_ppo_sde_param_count(int obs_dim) {
  if (obs_dim < 1 || obs_dim > ppo::K1) return fail(SO100_ERR_ARG, "obs_dim must be 1..16");
  return ppo::make_layout(obs_dim, true).total;
}
int64_t so100_ppo_sde_workspace_floats(int obs_dim) {
  const int n = so100_ppo_sde_param_count(obs_dim);
  return n < 0 ? n : (int64_t)SO100_PPO_MAX_CTAS * (n + 4) + 4 * ppo::kStatCtas;
}

// The learner's buffers say which GPU they live on: make it current (the entry points take no device argument, and the
// caller's current device need not be the one its tensors are on).
static int ppo_use_device_of(const void* dev_ptr) {
  cudaPointerAttributes a;
  if (cudaPointerGetAttributes(&a, dev_ptr) != cudaSuccess || a.type != cudaMemoryTypeDevice) {
    cudaGetLastError();
    return fail(SO100_ERR_ARG, "expected a device pointer");
  }
  CU(cudaSetDevice(a.device));
  return SO100_OK;
}

static int ppo_smem_optin(const void* fn, int floats) {  // per device; the call is cheap, so it is simply repeated
  CU(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, floats * 4));
  return SO100_OK;
}

extern "C++" {
template <bool SDE>
static int ppo_act(int obs_dim, const float* params, const float* obs, int n, uint64_t seed, int64_t env_offset, uint32_t tick,
                   int deterministic, float* act_raw, float* act_clip, float* logp, float* value, float* obs_copy, void* stream) {
  if (so100_ppo_param_count(obs_dim) < 0) return SO100_ERR_ARG;
  if (!params || !obs || n <= 0) return fail(SO100_ERR_ARG, "bad argument");
  int rc = ppo_use_device_of(params);
  if (rc) return rc;
  int dev = 0, sms = 0;
  CU(cudaGetDevice(&dev));
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const ppo::Layout L = ppo::make_layout(obs_dim, SDE);
  static const bool use_mma = getenv("SO100_PPO_ACT_MMA") != nullptr;  // A/B knob: the warp-level mma.sync version
  if (!use_mma) {  // tcgen05 / TMEM: 128-sample tiles, two persistent CTAs per SM
    const int bytes = SDE ? ppo::ActTc::BYTES_SDE : ppo::ActTc::BYTES;
    CU(cudaFuncSetAttribute((const void*)ppo::act_kernel_tc<SDE>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    const int ntiles = (n + ppo::TM - 1) / ppo::TM, grid = ntiles < 2 * sms ? ntiles : 2 * sms;
    ppo::act_kernel_tc<SDE><<<grid, ppo::NTC, bytes, (cudaStream_t)stream>>>(
        L, params, obs, n, (unsigned)(seed & 0xFFFFFFFFull), (unsigned)(seed >> 32), env_offset, tick, deterministic,
        act_raw, act_clip, logp, value, obs_copy);
    CU(cudaGetLastError());
    return SO100_OK;
  }
  const int floats = SDE ? ppo::kActSmemFloatsSde : ppo::kActSmemFloats;
  rc = ppo_smem_optin((const void*)ppo::act_kernel<SDE>, floats);
  if (rc) return rc;
  const int ntiles = (n + ppo::TB - 1) / ppo::TB, grid = ntiles < 2 * sms ? ntiles : 2 * sms;  // ~103 KB of shared memory: two CTAs per SM
  ppo::act_kernel<SDE><<<grid, ppo::NT, floats * 4, (cudaStream_t)stream>>>(
      L, params, obs, n, (unsigned)(seed & 0xFFFFFFFFull), (unsigned)(seed >> 32), env_offset, tick, deterministic,
      act_raw, act_clip, logp, value, obs_copy);
  CU(cudaGetLastError());
  return SO100_OK;
}
}  // extern "C++"

int so100_ppo_act(int obs_dim, const float* params, const float* obs, int n, uint64_t seed, int64_t env_offset, uint32_t tick,
                  int deterministic, float* act_raw, float* act_clip, float* logp, float* value, float* obs_copy, void* stream) {
  return ppo_act<false>(obs_dim, params, obs, n, seed, env_offset, tick, deterministic, act_raw, act_clip, logp, value, obs_copy, stream);
}
int so100_ppo_sde_act(int obs_dim, const float* params, const float* obs, int n, uint64_t seed, int64_t env_offset, uint32_t noise_key,
                      int deterministic, float* act_raw, float* act_clip, float* logp, float* value, float* obs_copy, void* stream) {
  return ppo_act<true>(obs_dim, params, obs, n, seed, env_offset, noise_key, deterministic, act_raw, act_clip, logp, value, obs_copy, stream);
}

int so100_ppo_post_step(int obs_dim, const float* params, int n, const float* reward, const uint8_t* terminated, const uint8_t* truncated,
                        const float* terminal_obs, const float* ep_return, const int32_t* ep_len, float gamma, float* reward_out,
                        float* done_out, double* acc, void* stream) {
  if (so100_ppo_param_count(obs_dim) < 0) return SO100_ERR_ARG;
  if (!params || n <= 0 || !reward || !terminated || !truncated || !terminal_obs || !ep_return || !ep_len || !reward_out || !done_out || !acc)
    return fail(SO100_ERR_ARG, "bad argument");
  if (int rc = ppo_use_device_of(params)) return rc;
  ppo::post_step_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(ppo::make_layout(obs_dim), params, n, reward, terminated, truncated,
                                                                           terminal_obs, ep_return, ep_len, gamma, reward_out, done_out, acc);
  CU(cudaGetLastError());
  return SO100_OK;
}

int so100_ppo_gae(const float* rew, const float* val, const float* done, const float* last_val, int T, int N, float gamma, float lam,
                  float* adv, float* ret, void* stream) {
  if (!rew || !val || !done || !last_val || !adv || !ret || T <= 0 || N <= 0) return fail(SO100_ERR_ARG, "bad argument");
  if (int rc = ppo_use_device_of(rew)) return rc;
  ppo::gae_kernel<<<(N + 255) / 256, 256, 0, (cudaStream_t)stream>>>(rew, val, done, last_val, T, N, gamma, lam, adv, ret);
  CU(cudaGetLastError());
  return SO100_OK;
}

int so100_ppo_permutation(int n, uint64_t key, int64_t* idx_out, void* stream) {
  if (n <= 0 || !idx_out) return fail(SO100_ERR_ARG, "bad argument");
  if (int rc = ppo_use_device_of(idx_out)) return rc;
  int bits = 1;
  while ((1ll << bits) < (long long)n) bits++;
  const int half_bits = (bits + 1) / 2;
  ppo::permutation_kernel<<<(n + 255) / 256, 256, 0, (cudaStream_t)stream>>>(n, half_bits, (unsigned)(key & 0xFFFFFFFFull), (unsigned)(key >> 32), idx_out);
  CU(cudaGetLastError());
  return SO100_OK;
}

extern "C++" {
template <bool SDE>
static int ppo_grad(int obs_dim, const float* params, const float* obs, const float* act, const float* logp_old, const float* adv,
                    const float* ret, const int64_t* idx, int mb, float clip_range, float vf_coef, float ent_coef, int normalize,
                    float* workspace, float* grad, float* loss_out, void* stream) {
  if (so100_ppo_param_count(obs_dim) < 0) return SO100_ERR_ARG;
  if (!params || !obs || !act || !logp_old || !adv || !ret || !idx || mb <= 0 || !workspace || !grad) return fail(SO100_ERR_ARG, "bad argument");
  const ppo::Layout L = ppo::make_layout(obs_dim, SDE);
  const int smem_floats = SDE ? ppo::kGradSmemFloatsSde : ppo::kGradSmemFloats;
  int rc = ppo_use_device_of(params);
  if (rc) return rc;
  rc = ppo_smem_optin((const void*)ppo::grad_kernel<SDE>, smem_floats);
  if (rc) return rc;
  int dev = 0, sms = 0;
  CU(cudaGetDevice(&dev));
  CU(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
  const int ntiles = (mb + ppo::GT - 1) / ppo::GT;
  int grid = ntiles < 2 * sms ? ntiles : 2 * sms;  // persistent: two CTAs per SM
  if (grid > SO100_PPO_MAX_CTAS) grid = SO100_PPO_MAX_CTAS;
  cudaStream_t st = (cudaStream_t)stream;
  // fp64 partials behind the gradient partials; (total + 4) * MAX_CTAS floats is a multiple of 8 bytes
  double* stats = reinterpret_cast<double*>(workspace + (size_t)SO100_PPO_MAX_CTAS * (L.total + 4));
  normalize = normalize && mb > 1;  // SB3 normalises only when len(advantages) > 1: one sample keeps its raw advantage
  if (normalize) ppo::adv_stats_kernel<<<ppo::kStatCtas, 256, 0, st>>>(adv, idx, mb, stats);
  ppo::grad_kernel<SDE><<<grid, ppo::NT, smem_floats * 4, st>>>(L, params, obs, act, logp_old, adv, ret, idx, mb, stats, clip_range, vf_coef,
                                                               ent_coef, normalize, workspace);
  ppo::reduce_kernel<<<(L.total + 3 + 255) / 256, 256, 0, st>>>(workspace, grid, L.total, mb, grad, loss_out);
  CU(cudaGetLastError());
  return SO100_OK;
}
}  // extern "C++"

int so100_ppo_grad(int obs_dim, const float* params, const float* obs, const float* act, const float* logp_old, const float* adv,
                   const float* ret, const int64_t* idx, int mb, float clip_range, float vf_coef, float ent_coef, int normalize,
                   float* workspace, float* grad, float* loss_out, void* stream) {
  return ppo_grad<false>(obs_dim, params, obs, act, logp_old, adv, ret, idx, mb, clip_range, vf_coef, ent_coef, normalize, workspace, grad,
                         loss_out, stream);
}
int so100_ppo_sde_grad(int obs_dim, const float* params, const float* obs, const float* act, const float* logp_old, const float* adv,
                       const float* ret, const int64_t* idx, int mb, float clip_range, float vf_coef, float ent_coef, int normalize,
                       float* workspace, float* grad, float* loss_out, void* stream) {
  return ppo_grad<true>(obs_dim, params, obs, act, logp_old, adv, ret, idx, mb, clip_range, vf_coef, ent_coef, normalize, workspace, grad,
                        loss_out, stream);
}

int so100_ppo_adam(int n_params, float* params, const float* grad, float* exp_avg, float* exp_avg_sq, int32_t* step_count, float grad_scale,
                   float max_grad_norm, float lr, float beta1, float beta2, float eps, void* stream) {
  if (n_params <= 0 || !params || !grad || !exp_avg || !exp_avg_sq || !step_count) return fail(SO100_ERR_ARG, "bad argument");
  if (int rc = ppo_use_device_of(params)) return rc;
  ppo::adam_kernel<<<1, 1024, 0, (cudaStream_t)stream>>>(n_params, params, grad, exp_avg, exp_avg_sq, step_count, grad_scale, max_grad_norm, lr,
                                                          beta1, beta2, eps);
  CU(cudaGetLastError());
  return SO100_OK;
}

}  // extern "C"
