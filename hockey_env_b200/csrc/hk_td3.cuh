// hk_td3.cuh -- one TD3 learner update (DeviceTD3Learner.update, td3.py; the reference's TD3Learner.update,
// rl/td3/learner.py:55-219) as ONE sm_100a kernel launch: batch gather, target policy with clipped smoothing noise,
// twin-critic forward / backward / Adam, prioritized-replay importance weights and priority write-back, and -- on actor
// steps -- actor forward through the freshly updated Q1, actor backward / Adam and the Polyak updates of both target nets.
//
// Networks: the reference architecture only.  Actor 18 -> 256 -> 256 -> 4 (tanh after every layer); twin critic, each head
// 22 -> 256 -> 256 -> 1 (tanh, tanh, linear) on [obs, normalised action].
//
// Shape.  One thread-block cluster of kClusterMax = 16 CTAs (non-portable size; 8 when the device cannot co-schedule 16)
// of 256 threads.  The phases of the update are separated by hardware cluster barriers (barrier.cluster arrive.release /
// wait.acquire); activations, deltas and gradients travel between phases through a caller-owned scratch buffer in global
// memory (L2-resident: <= 24 MB at B = 1024), read with ld.global.cg so that no CTA can see a stale L1 line of data another
// CTA rewrote.  Work inside a phase is split three ways:
//   * unit slices: a 256-unit layer is 16 slices of 16 units.  The CTA that owns a slice computes those 16 output columns
//     for all B rows (forward: its 16 rows of W staged in shared memory; backward to the layer input: its 16 columns of
//     W), the matching 16 rows of dW and db, and the elementwise tanh derivatives.  Slice s belongs to CTA s mod size.
//   * rows: the narrow layers (actor fc3, 4 outputs; critic fc3, 1 output; the 4 action columns of the critic's fc1 in
//     the actor's backward pass) and the loss are a warp per row, dot products reduced by a fixed xor-shuffle tree.
//   * flat: Adam and Polyak are elementwise over the parameter vectors.
// So every output element is computed by exactly one thread in a fixed order whatever the cluster size, and the result
// does not depend on it.  A single cluster is bounded by latency, not by FMA throughput; the fp32 SIMT path keeps the
// learner equivalent to torch's fp32 learner (tensor cores are out of scope, DESIGN.md section 4.2).
//
// Numerics contract:
//  * Precision: fp32 throughout, like torch's fp32 learner with TF32 off.  The library builds with -fmad=false, so every
//    multiply-add of the GEMM loops is an explicit fmaf; tanh is tanhf.  Sums run in a fixed order (no float atomics):
//    the same inputs give bit-identical results run to run.  They are not torch's summation orders, so results agree with
//    torch to fp32 rounding, not bit for bit.
//  * Action normalisation: every critic forward applies TwinQNetwork's ((a - low) / range) * 2 - 1 from the critic's
//    action_low / action_range buffers (skipped, like torch, when a range entry is infinite); the actor's backward pass
//    multiplies the action gradient by 2 and divides it by range.
//  * Target noise: a' = clamp(target_actor(s') + clip(sigma * z, -clip, clip), -1, 1), z = four normals per row from one
//    Philox4x32-10 call hk::philox(seed, row, (uint32_t)ctr, HK_STREAM_TD3_TARGET | (uint32_t)(ctr >> 32) << 8) and
//    Box-Muller exactly as hk_actor.cuh's NoiseKey (u1 = ((a >> 8) + 1) 2^-24, u2 = (b >> 8) 2^-24); ctr is the arena's
//    noise counter, which every update advances.
//  * Loss: 0.5 (huber_w(q1, y) + huber_w(q2, y)), huber_w = weighted smooth-L1 with mean over B; y = r + gamma (1 - done)
//    min(Q1'(s', a'), Q2'(s', a')).  Actor loss -mean Q1(s, pi(s)) with the critic already stepped, as torch does.
//  * Adam (torch.optim.Adam, amsgrad off, betas 0.9 / 0.999, eps 1e-8): g += wd p; m = m + (1 - b1)(g - m);
//    v = b2 v + (1 - b2) g g; p -= (lr / (1 - b1^t)) * m / (sqrt(v) / sqrt(1 - b2^t) + eps).  The step counts t live
//    in the arena as int64 that the kernel increments (critic and actor separately); the bias corrections are computed in
//    double.  So a captured graph replays correctly.
//  * Polyak: tp = tp (1 - tau) + tau p over parameters (the critic's action buffers are not part of the arena).
//  * Prioritized batches: p_i = weight[idx_i] / sum over the batch (uniform 1 / B if the sum is not > 0), importance
//    weights w_i = (1 / (N p_i))^beta / max_j w_j (unnormalised if the max is not > 0); priorities
//    0.5 (|q1 - y| + |q2 - y|) clamped to [1e-6, 1e6] are written back, and for an index that occurs several times in the
//    batch the LAST occurrence wins.
#pragma once
#include <cooperative_groups.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace hk_td3 {

namespace cg = cooperative_groups;

constexpr int kObs = 18, kAct = 4, kH = 256, kQin = kObs + kAct;
constexpr int kObsLd = 20, kQinLd = 24;  // row strides of the staged inputs (zero padded to a multiple of 4)
constexpr int kMaxBatch = 1024;
constexpr int kThreads = 256;
constexpr int kSlice = 16;               // output units per slice
constexpr int kSlices = kH / kSlice;
constexpr int kClusterMax = 16;

// ---- arena: one fp32 block, offsets in floats; each net in state_dict order, row-major as torch stores it ---------------
// actor: fc1.weight [256,18], fc1.bias, fc2.weight [256,256], fc2.bias, fc3.weight [4,256], fc3.bias [4]
constexpr int kA_W1 = 0, kA_B1 = kA_W1 + kH * kObs, kA_W2 = kA_B1 + kH, kA_B2 = kA_W2 + kH * kH, kA_W3 = kA_B2 + kH,
              kA_B3 = kA_W3 + kAct * kH, kActorParams = kA_B3 + kAct;
// one critic head: fc1.weight [256,22], fc1.bias, fc2.weight, fc2.bias, fc3.weight [1,256], fc3.bias [1]; q1 then q2
constexpr int kQ_W1 = 0, kQ_B1 = kQ_W1 + kH * kQin, kQ_W2 = kQ_B1 + kH, kQ_B2 = kQ_W2 + kH * kH, kQ_W3 = kQ_B2 + kH,
              kQ_B3 = kQ_W3 + kH, kHeadParams = kQ_B3 + 1, kCriticParams = 2 * kHeadParams;
__host__ __device__ constexpr int64_t pad64(int64_t x) { return (x + 63) / 64 * 64; }
constexpr int64_t kOffActor = 0;
constexpr int64_t kOffCritic = kOffActor + pad64(kActorParams);
constexpr int64_t kOffTActor = kOffCritic + pad64(kCriticParams);
constexpr int64_t kOffTCritic = kOffTActor + pad64(kActorParams);
constexpr int64_t kOffMActor = kOffTCritic + pad64(kCriticParams);
constexpr int64_t kOffVActor = kOffMActor + pad64(kActorParams);
constexpr int64_t kOffMCritic = kOffVActor + pad64(kActorParams);
constexpr int64_t kOffVCritic = kOffMCritic + pad64(kCriticParams);
constexpr int64_t kOffCounters = kOffVCritic + pad64(kCriticParams);  // int64 [critic step, actor step, noise counter]
constexpr int64_t kArenaFloats = kOffCounters + 64;

// ---- scratch: offsets in floats, every region 256-byte aligned --------------------------------------------------------
struct Scratch {
  float *w, *r, *d, *y, *q, *dq, *closs, *aloss;          // [B] each; q, dq, closs [2][B] (head-major)
  float *s, *xc, *s2, *xt, *xp;                           // [B][20] obs, [B][24] [obs, norm a], [B][20] next obs,
                                                          // [B][24] [next obs, norm a'], [B][24] [obs, norm pi]
  float *ta1, *ta2, *tc1, *tc2, *c1, *c2, *d2, *d1;       // [B][256] target actor; [2][B][256] per head
  float *p1, *p2, *pi, *qa1, *qa2, *qd2, *qd1, *da3, *ad2, *ad1;  // actor step; pi, da3 [B][4]
  float *gA, *gC;                                         // gradients, laid out like the actor / critic parameters
  int64_t floats;
};
__host__ __device__ inline Scratch carve(float* base, int64_t B) {
  Scratch s;
  int64_t o = 0;
  auto take = [&](int64_t n) { float* p = base ? base + o : nullptr; o += pad64(n); return p; };
  const int64_t bh = B * kH;
  s.w = take(B); s.r = take(B); s.d = take(B); s.y = take(B);
  s.q = take(2 * B); s.dq = take(2 * B); s.closs = take(2 * B); s.aloss = take(B);
  s.s = take(B * kObsLd); s.xc = take(B * kQinLd); s.s2 = take(B * kObsLd); s.xt = take(B * kQinLd); s.xp = take(B * kQinLd);
  s.ta1 = take(bh); s.ta2 = take(bh); s.tc1 = take(2 * bh); s.tc2 = take(2 * bh);
  s.c1 = take(2 * bh); s.c2 = take(2 * bh); s.d2 = take(2 * bh); s.d1 = take(2 * bh);
  s.p1 = take(bh); s.p2 = take(bh); s.pi = take(B * kAct); s.qa1 = take(bh); s.qa2 = take(bh); s.qd2 = take(bh); s.qd1 = take(bh);
  s.da3 = take(B * kAct); s.ad2 = take(bh); s.ad1 = take(bh);
  s.gA = take(kActorParams); s.gC = take(kCriticParams);
  s.floats = o;
  return s;
}

struct Args {
  float* arena;
  float* scratch;
  const float *obs, *act, *rew, *nobs, *done;  // replay arrays [capacity, 18], [capacity, 4], [capacity], ...
  const long long* idx;                        // [B] rows of the batch
  float* pw;                                   // prioritized: the buffer's weights (NULL: uniform batch)
  const long long* pidx;                       // [B] indices into pw
  long long pn;                                // N of the importance weights (the buffer's size)
  const float *alow, *arange;                  // the critic's action_low / action_range buffers [4]
  float* losses;                               // [2]: actor loss (actor steps only), critic loss
  unsigned long long seed;
  int B, doActor;
  float gamma, tauA, tauC, lrA, lrC, wdA, wdC, beta, sigma, clip;
};

// ---- helpers ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ float ld(const float* p) { return __ldcg(p); }
__device__ __forceinline__ float4 ld4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ void clusterSync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ float warpSum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float normAct(float a, float low, float range, bool norm) {
  return norm ? ((a - low) / range) * 2.0f - 1.0f : a;
}

struct Smem {
  float S[kH * kSlice];             // staged operand [K][16]
  float part[kThreads * kSlice];    // partial sums of the column reductions
  float bias[kSlice];
  float red[kThreads];
};

// Y[r][j] = sum_k X[r][k] S[k][j] for the staged S [K][16] (K a multiple of 4), then epi(r, acc).  One row per thread.
template <class Epi>
__device__ __forceinline__ void mm16(const Smem& sm, const float* X, int ldx, int K, int B, Epi epi) {
  for (int r = threadIdx.x; r < B; r += kThreads) {
    float acc[kSlice];
#pragma unroll
    for (int j = 0; j < kSlice; ++j) acc[j] = 0.0f;
    const float* x = X + (int64_t)r * ldx;
#pragma unroll 2
    for (int k = 0; k < K; k += 4) {
      const float4 xv = ld4(x + k);
      const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const float4* s = reinterpret_cast<const float4*>(sm.S + (k + kk) * kSlice);
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const float4 w = s[q];
          acc[4 * q + 0] = fmaf(xs[kk], w.x, acc[4 * q + 0]);
          acc[4 * q + 1] = fmaf(xs[kk], w.y, acc[4 * q + 1]);
          acc[4 * q + 2] = fmaf(xs[kk], w.z, acc[4 * q + 2]);
          acc[4 * q + 3] = fmaf(xs[kk], w.w, acc[4 * q + 3]);
        }
      }
    }
    epi(r, acc);
  }
}

// S[k][j] = W[n0 + j][k] (k < K, zero up to Kp) and the 16 biases: the forward operand of units n0 .. n0 + 15
__device__ __forceinline__ void stageRows(Smem& sm, const float* W, const float* b, int K, int Kp, int n0) {
  __syncthreads();
  for (int i = threadIdx.x; i < kSlice * Kp; i += kThreads) {
    const int j = i / Kp, k = i - j * Kp;
    sm.S[k * kSlice + j] = k < K ? ld(W + (int64_t)(n0 + j) * K + k) : 0.0f;
  }
  if (threadIdx.x < kSlice) sm.bias[threadIdx.x] = ld(b + n0 + threadIdx.x);
  __syncthreads();
}
// S[n][j] = W[n][k0 + j], n < 256: the operand of the backward pass to input units k0 .. k0 + 15 of W [256, ldw]
__device__ __forceinline__ void stageCols(Smem& sm, const float* W, int ldw, int k0) {
  __syncthreads();
  for (int i = threadIdx.x; i < kH * kSlice; i += kThreads) {
    const int n = i / kSlice, j = i - n * kSlice;
    sm.S[i] = ld(W + (int64_t)n * ldw + k0 + j);
  }
  __syncthreads();
}

__device__ __forceinline__ void store16(float* y, const float* v) {
#pragma unroll
  for (int q = 0; q < 4; ++q) reinterpret_cast<float4*>(y)[q] = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
}

// Y[:, n0 .. n0 + 15] = tanh(X W^T + b) of a hidden layer W [256, K]
__device__ __forceinline__ void fwdSlice(Smem& sm, const float* W, const float* b, int K, int Kp, const float* X, int ldx, float* Y,
                                         int n0, int B) {
  stageRows(sm, W, b, K, Kp, n0);
  mm16(sm, X, ldx, Kp, B, [&](int r, float* acc) {
#pragma unroll
    for (int j = 0; j < kSlice; ++j) acc[j] = tanhf(acc[j] + sm.bias[j]);
    store16(Y + (int64_t)r * kH + n0, acc);
  });
}

// Out[:, k0 .. k0 + 15] = (D W)[:, k0 ..] * (1 - A^2): the delta at the tanh layer A feeding W [256, 256]
__device__ __forceinline__ void bwdSlice(Smem& sm, const float* W, const float* D, const float* A, float* Out, int k0, int B) {
  stageCols(sm, W, kH, k0);
  mm16(sm, D, kH, kH, B, [&](int r, float* acc) {
    const float* a = A + (int64_t)r * kH + k0;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const float4 y = ld4(a + 4 * q);
      acc[4 * q + 0] = acc[4 * q + 0] * (1.0f - y.x * y.x);
      acc[4 * q + 1] = acc[4 * q + 1] * (1.0f - y.y * y.y);
      acc[4 * q + 2] = acc[4 * q + 2] * (1.0f - y.z * y.z);
      acc[4 * q + 3] = acc[4 * q + 3] * (1.0f - y.w * y.w);
    }
    store16(Out + (int64_t)r * kH + k0, acc);
  });
}

// out[j] = sum_r a[r * as] X[r][c0 + j] (a == nullptr: weight 1), j < 16: 16 row groups, then a fixed-order combine
__device__ __forceinline__ void colsum16(Smem& sm, const float* X, int ldx, int c0, const float* a, int as, int B, float* out) {
  const int t = threadIdx.x, j = t & 15, g = t >> 4;
  float s = 0.0f;
  for (int r = g; r < B; r += 16) {
    const float x = ld(X + (int64_t)r * ldx + c0 + j);
    s = a ? fmaf(ld(a + (int64_t)r * as), x, s) : s + x;
  }
  __syncthreads();
  sm.part[g * 16 + j] = s;
  __syncthreads();
  if (t < 16) {
    float v = 0.0f;
    for (int q = 0; q < 16; ++q) v += sm.part[q * 16 + t];
    out[t] = v;
  }
}

// dW[n0 + j][k] = sum_r D[r][n0 + j] X[r][k], k < K (row-major [*, K] gradient block gW), and db[n0 + j] = sum_r D[r][n0 + j]
__device__ __forceinline__ void dwSlice(Smem& sm, const float* D, int n0, const float* X, int ldx, int K, int B, float* gW, float* gb) {
  const int t = threadIdx.x;
  const int kt = K > 32 ? kThreads : 32, groups = kThreads / kt, k = t % kt, g = t / kt;
  float e[kSlice], o[kSlice];  // even / odd rows of the group
#pragma unroll
  for (int j = 0; j < kSlice; ++j) e[j] = o[j] = 0.0f;
  if (k < K) {
    int r = g;
    for (; r + groups < B; r += 2 * groups) {
      const float x0 = ld(X + (int64_t)r * ldx + k), x1 = ld(X + (int64_t)(r + groups) * ldx + k);
      const float* d0 = D + (int64_t)r * kH + n0;
      const float* d1 = D + (int64_t)(r + groups) * kH + n0;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 a = ld4(d0 + 4 * q), b = ld4(d1 + 4 * q);
        e[4 * q + 0] = fmaf(a.x, x0, e[4 * q + 0]); o[4 * q + 0] = fmaf(b.x, x1, o[4 * q + 0]);
        e[4 * q + 1] = fmaf(a.y, x0, e[4 * q + 1]); o[4 * q + 1] = fmaf(b.y, x1, o[4 * q + 1]);
        e[4 * q + 2] = fmaf(a.z, x0, e[4 * q + 2]); o[4 * q + 2] = fmaf(b.z, x1, o[4 * q + 2]);
        e[4 * q + 3] = fmaf(a.w, x0, e[4 * q + 3]); o[4 * q + 3] = fmaf(b.w, x1, o[4 * q + 3]);
      }
    }
    if (r < B) {
      const float x0 = ld(X + (int64_t)r * ldx + k);
      const float* d0 = D + (int64_t)r * kH + n0;
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const float4 a = ld4(d0 + 4 * q);
        e[4 * q + 0] = fmaf(a.x, x0, e[4 * q + 0]);
        e[4 * q + 1] = fmaf(a.y, x0, e[4 * q + 1]);
        e[4 * q + 2] = fmaf(a.z, x0, e[4 * q + 2]);
        e[4 * q + 3] = fmaf(a.w, x0, e[4 * q + 3]);
      }
    }
  }
  if (groups == 1) {
    if (k < K)
#pragma unroll
      for (int j = 0; j < kSlice; ++j) gW[(int64_t)(n0 + j) * K + k] = e[j] + o[j];
  } else {
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kSlice; ++j) sm.part[(g * kSlice + j) * 32 + k] = e[j] + o[j];
    __syncthreads();
    for (int i = t; i < kSlice * 32; i += kThreads) {
      const int j = i >> 5, kk = i & 31;
      if (kk < K) {
        float v = 0.0f;
        for (int q = 0; q < groups; ++q) v += sm.part[(q * kSlice + j) * 32 + kk];
        gW[(int64_t)(n0 + j) * K + kk] = v;
      }
    }
  }
  colsum16(sm, D, kH, n0, nullptr, 0, B, gb + n0);
}

// warp-wide dot product of a 256-vector x with W row w (fixed xor tree: every lane gets the same sum)
__device__ __forceinline__ float dot256(const float* x, const float* w) {
  const int lane = threadIdx.x & 31;
  float s = 0.0f;
#pragma unroll
  for (int i = 0; i < kH / 32; ++i) s = fmaf(ld(x + lane + 32 * i), ld(w + lane + 32 * i), s);
  return warpSum(s);
}

__device__ __forceinline__ void adam(float* p, float* m, float* v, const float* g, int n, float lr, float wd, int64_t t, int gtid, int gstride) {
  const double bc1 = 1.0 - pow(0.9, (double)t), bc2 = 1.0 - pow(0.999, (double)t);
  const float stepSize = (float)((double)lr / bc1), bc2Sqrt = (float)sqrt(bc2);
  for (int i = gtid; i < n; i += gstride) {
    float gi = ld(g + i);
    const float pi = ld(p + i);
    if (wd != 0.0f) gi = gi + wd * pi;
    const float mi = ld(m + i) + 0.1f * (gi - ld(m + i));
    const float vi = ld(v + i) * 0.999f + 0.001f * gi * gi;
    m[i] = mi;
    v[i] = vi;
    p[i] = pi - stepSize * (mi / (sqrtf(vi) / bc2Sqrt + 1e-8f));
  }
}

__device__ __forceinline__ void polyak(float* tp, const float* p, int n, float tau, int gtid, int gstride) {
  const float keep = (float)(1.0 - (double)tau);
  for (int i = gtid; i < n; i += gstride) tp[i] = ld(tp + i) * keep + tau * ld(p + i);
}

// ---- the kernel -----------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kThreads, 1) k_td3_update(const Args a) {
  __shared__ __align__(16) Smem sm;
  const int nc = (int)cg::this_cluster().num_blocks(), c = (int)cg::this_cluster().block_rank();
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int B = a.B;
  const int gtid = c * kThreads + t, gstride = nc * kThreads;
  const int gwarp = c * (kThreads / 32) + warp, gwarps = nc * (kThreads / 32);
  const Scratch s = carve(a.scratch, B);
  float* arena = a.arena;
  long long* ctr = reinterpret_cast<long long*>(arena + kOffCounters);
  const long long tC = __ldcg(ctr) + 1, tA = __ldcg(ctr + 1) + 1, noiseCtr = __ldcg(ctr + 2);
  const float* actor = arena + kOffActor;
  float* critic = arena + kOffCritic;
  const float* tactor = arena + kOffTActor;
  const float* tcritic = arena + kOffTCritic;
  float low[kAct], range[kAct];
  bool norm = true;
#pragma unroll
  for (int j = 0; j < kAct; ++j) {
    low[j] = a.alow[j];
    range[j] = a.arange[j];
    norm = norm && !isinf(range[j]);
  }

  // ---- phase 0: gather the batch; CTA 0 computes the importance weights ----
  for (int r = gtid; r < B; r += gstride) {
    const long long ix = a.idx[r];
    const float* o = a.obs + ix * kObs;
    const float* o2 = a.nobs + ix * kObs;
    for (int k = 0; k < kObs; ++k) {
      const float v = o[k], v2 = o2[k];
      s.s[r * kObsLd + k] = v;
      s.xc[r * kQinLd + k] = v;
      s.s2[r * kObsLd + k] = v2;
      s.xt[r * kQinLd + k] = v2;
      s.xp[r * kQinLd + k] = v;
    }
    for (int k = kObs; k < kObsLd; ++k) s.s[r * kObsLd + k] = s.s2[r * kObsLd + k] = 0.0f;
    for (int j = 0; j < kAct; ++j) s.xc[r * kQinLd + kObs + j] = normAct(a.act[ix * kAct + j], low[j], range[j], norm);
    for (int k = kQin; k < kQinLd; ++k) s.xc[r * kQinLd + k] = s.xt[r * kQinLd + k] = s.xp[r * kQinLd + k] = 0.0f;
    s.r[r] = a.rew[ix];
    s.d[r] = a.done[ix];
  }
  if (c == 0) {
    if (a.pw) {
      float p[kMaxBatch / kThreads], sum = 0.0f;
#pragma unroll
      for (int q = 0; q < kMaxBatch / kThreads; ++q) {
        const int r = t + q * kThreads;
        p[q] = r < B ? __ldcg(a.pw + a.pidx[r]) : 0.0f;
        sum += p[q];
      }
      sm.red[t] = sum;
      __syncthreads();
      for (int h = kThreads / 2; h > 0; h >>= 1) {
        if (t < h) sm.red[t] += sm.red[t + h];
        __syncthreads();
      }
      const float tot = sm.red[0];
      __syncthreads();
      float wmax = 0.0f;
#pragma unroll
      for (int q = 0; q < kMaxBatch / kThreads; ++q) {
        const int r = t + q * kThreads;
        const float prob = tot > 0.0f ? p[q] / tot : 1.0f / (float)B;
        p[q] = powf(1.0f / (prob * (float)a.pn), a.beta);
        if (r < B) wmax = fmaxf(wmax, p[q]);
      }
      sm.red[t] = wmax;
      __syncthreads();
      for (int h = kThreads / 2; h > 0; h >>= 1) {
        if (t < h) sm.red[t] = fmaxf(sm.red[t], sm.red[t + h]);
        __syncthreads();
      }
      const float top = sm.red[0];
#pragma unroll
      for (int q = 0; q < kMaxBatch / kThreads; ++q) {
        const int r = t + q * kThreads;
        if (r < B) s.w[r] = top > 0.0f ? p[q] / top : p[q];
      }
    } else {
      for (int r = t; r < B; r += kThreads) s.w[r] = 1.0f;
    }
  }
  clusterSync();

  // ---- phase 1: target actor fc1 on s'; critic fc1 (both heads) on (s, a) ----
  for (int sl = c; sl < kSlices; sl += nc) {
    const int n0 = sl * kSlice;
    fwdSlice(sm, tactor + kA_W1, tactor + kA_B1, kObs, kObsLd, s.s2, kObsLd, s.ta1, n0, B);
    for (int h = 0; h < 2; ++h)
      fwdSlice(sm, critic + h * kHeadParams + kQ_W1, critic + h * kHeadParams + kQ_B1, kQin, kQinLd, s.xc, kQinLd, s.c1 + h * B * kH, n0, B);
  }
  clusterSync();
  // ---- phase 2: target actor fc2; critic fc2 ----
  for (int sl = c; sl < kSlices; sl += nc) {
    const int n0 = sl * kSlice;
    fwdSlice(sm, tactor + kA_W2, tactor + kA_B2, kH, kH, s.ta1, kH, s.ta2, n0, B);
    for (int h = 0; h < 2; ++h)
      fwdSlice(sm, critic + h * kHeadParams + kQ_W2, critic + h * kHeadParams + kQ_B2, kH, kH, s.c1 + h * B * kH, kH, s.c2 + h * B * kH, n0, B);
  }
  clusterSync();
  // ---- phase 3 (rows): a' = clamp(tanh(target fc3) + clipped noise, -1, 1); the target critic's input ----
  for (int r = gwarp; r < B; r += gwarps) {
    float v[kAct];
#pragma unroll
    for (int j = 0; j < kAct; ++j) v[j] = dot256(s.ta2 + (int64_t)r * kH, tactor + kA_W3 + j * kH);
    if (lane < kAct) {
      const hk::U4 u = hk::philox(a.seed, (uint64_t)r, (uint32_t)noiseCtr,
                                  (uint32_t)hk::HK_STREAM_TD3_TARGET | ((uint32_t)((unsigned long long)noiseCtr >> 32) << 8));
      float z0, z1, z2, z3;
      hk_actor::boxMuller(u.x, u.y, z0, z1);
      hk_actor::boxMuller(u.z, u.w, z2, z3);
      const float z = lane == 0 ? z0 : lane == 1 ? z1 : lane == 2 ? z2 : z3;
      const float va = lane == 0 ? v[0] : lane == 1 ? v[1] : lane == 2 ? v[2] : v[3];
      const float act = tanhf(va + ld(tactor + kA_B3 + lane));
      const float e = fminf(fmaxf(a.sigma * z, -a.clip), a.clip);
      const float an = fminf(fmaxf(act + e, -1.0f), 1.0f);
      s.xt[r * kQinLd + kObs + lane] = normAct(an, low[lane], range[lane], norm);
    }
  }
  clusterSync();
  // ---- phase 4: target critic fc1 on (s', a') ----
  for (int sl = c; sl < kSlices; sl += nc)
    for (int h = 0; h < 2; ++h)
      fwdSlice(sm, tcritic + h * kHeadParams + kQ_W1, tcritic + h * kHeadParams + kQ_B1, kQin, kQinLd, s.xt, kQinLd, s.tc1 + h * B * kH,
               sl * kSlice, B);
  clusterSync();
  // ---- phase 5: target critic fc2 ----
  for (int sl = c; sl < kSlices; sl += nc)
    for (int h = 0; h < 2; ++h)
      fwdSlice(sm, tcritic + h * kHeadParams + kQ_W2, tcritic + h * kHeadParams + kQ_B2, kH, kH, s.tc1 + h * B * kH, kH,
               s.tc2 + h * B * kH, sl * kSlice, B);
  clusterSync();
  // ---- phase 6 (rows): q1, q2, target y, loss terms, dL/dq, priorities ----
  for (int r = gwarp; r < B; r += gwarps) {
    float q[2], tq[2];
    for (int h = 0; h < 2; ++h) {
      q[h] = dot256(s.c2 + ((int64_t)h * B + r) * kH, critic + h * kHeadParams + kQ_W3) + ld(critic + h * kHeadParams + kQ_B3);
      tq[h] = dot256(s.tc2 + ((int64_t)h * B + r) * kH, tcritic + h * kHeadParams + kQ_W3) + ld(tcritic + h * kHeadParams + kQ_B3);
    }
    const float y = ld(s.r + r) + (a.gamma * (1.0f - ld(s.d + r))) * fminf(tq[0], tq[1]);
    const float w = ld(s.w + r), g = 0.5f / (float)B;
    if (lane == 0) {
      s.y[r] = y;
      for (int h = 0; h < 2; ++h) {
        const float dd = q[h] - y, ad = fabsf(dd);
        s.q[h * B + r] = q[h];
        s.closs[h * B + r] = ad < 1.0f ? ((0.5f * w) * dd) * dd : (ad - 0.5f) * w;
        s.dq[h * B + r] = g * (ad < 1.0f ? w * dd : w * copysignf(1.0f, dd));
      }
    }
    if (a.pw) {  // last occurrence of an index wins
      const long long ix = a.pidx[r];
      bool later = false;
      for (int r2 = r + 1 + lane; r2 < B && !later; r2 += 32) later = a.pidx[r2] == ix;
      if (!__any_sync(0xffffffffu, later) && lane == 0) {
        const float pr = 0.5f * (fabsf(q[0] - y) + fabsf(q[1] - y));
        a.pw[ix] = fminf(fmaxf(pr, 1e-6f), 1e6f);
      }
    }
  }
  clusterSync();
  // ---- phase 7: critic deltas at fc2, dW2 / db2 / dW3 of the owned slices; db3 and the critic loss on CTA 0 ----
  for (int sl = c; sl < kSlices; sl += nc) {
    const int k0 = sl * kSlice;
    for (int h = 0; h < 2; ++h) {
      const float* w3 = critic + h * kHeadParams + kQ_W3;
      const float* c2 = s.c2 + (int64_t)h * B * kH;
      float* d2 = s.d2 + (int64_t)h * B * kH;
      float* gh = s.gC + h * kHeadParams;
      for (int i = t; i < B * kSlice; i += kThreads) {
        const int r = i >> 4, j = i & 15;
        const float y = ld(c2 + (int64_t)r * kH + k0 + j);
        d2[(int64_t)r * kH + k0 + j] = (ld(s.dq + h * B + r) * ld(w3 + k0 + j)) * (1.0f - y * y);
      }
      __syncthreads();
      dwSlice(sm, d2, k0, s.c1 + (int64_t)h * B * kH, kH, kH, B, gh + kQ_W2, gh + kQ_B2);
      colsum16(sm, c2, kH, k0, s.dq + h * B, 1, B, gh + kQ_W3 + k0);
    }
  }
  if (c == 0 && warp < 2) {  // warp h: db3 of head h; then the loss
    float sd = 0.0f, sl = 0.0f, sl2 = 0.0f;
    for (int r = lane; r < B; r += 32) {
      sd += ld(s.dq + warp * B + r);
      sl += ld(s.closs + r);
      sl2 += ld(s.closs + B + r);
    }
    sd = warpSum(sd);
    sl = warpSum(sl);
    sl2 = warpSum(sl2);
    if (lane == 0) {
      s.gC[warp * kHeadParams + kQ_B3] = sd;
      if (warp == 0) a.losses[1] = 0.5f * (sl / (float)B + sl2 / (float)B);
    }
  }
  clusterSync();
  // ---- phase 8: critic deltas at fc1, dW1 / db1 ----
  for (int sl = c; sl < kSlices; sl += nc) {
    const int k0 = sl * kSlice;
    for (int h = 0; h < 2; ++h) {
      float* d1 = s.d1 + (int64_t)h * B * kH;
      bwdSlice(sm, critic + h * kHeadParams + kQ_W2, s.d2 + (int64_t)h * B * kH, s.c1 + (int64_t)h * B * kH, d1, k0, B);
      __syncthreads();
      dwSlice(sm, d1, k0, s.xc, kQinLd, kQin, B, s.gC + h * kHeadParams + kQ_W1, s.gC + h * kHeadParams + kQ_B1);
    }
  }
  clusterSync();
  // ---- phase 9: critic Adam ----
  adam(critic, arena + kOffMCritic, arena + kOffVCritic, s.gC, kCriticParams, a.lrC, a.wdC, tC, gtid, gstride);
  if (a.doActor) {
    float* actorW = arena + kOffActor;
    const float* q1 = critic;  // head 1, stepped
    clusterSync();
    // ---- phase 10, 11: pi hidden layers on s ----
    for (int sl = c; sl < kSlices; sl += nc) fwdSlice(sm, actor + kA_W1, actor + kA_B1, kObs, kObsLd, s.s, kObsLd, s.p1, sl * kSlice, B);
    clusterSync();
    for (int sl = c; sl < kSlices; sl += nc) fwdSlice(sm, actor + kA_W2, actor + kA_B2, kH, kH, s.p1, kH, s.p2, sl * kSlice, B);
    clusterSync();
    // ---- phase 12 (rows): pi = tanh(fc3); Q1's input [s, norm(pi)] ----
    for (int r = gwarp; r < B; r += gwarps) {
      float v[kAct];
#pragma unroll
      for (int j = 0; j < kAct; ++j) v[j] = dot256(s.p2 + (int64_t)r * kH, actor + kA_W3 + j * kH);
      if (lane < kAct) {
        const float va = lane == 0 ? v[0] : lane == 1 ? v[1] : lane == 2 ? v[2] : v[3];
        const float p = tanhf(va + ld(actor + kA_B3 + lane));
        s.pi[r * kAct + lane] = p;
        s.xp[r * kQinLd + kObs + lane] = normAct(p, low[lane], range[lane], norm);
      }
    }
    clusterSync();
    // ---- phase 13, 14: Q1 hidden layers on (s, pi); delta at fc2 for dL/dq = -1 / B ----
    for (int sl = c; sl < kSlices; sl += nc) fwdSlice(sm, q1 + kQ_W1, q1 + kQ_B1, kQin, kQinLd, s.xp, kQinLd, s.qa1, sl * kSlice, B);
    clusterSync();
    const float dqa = -1.0f / (float)B;
    for (int sl = c; sl < kSlices; sl += nc) {
      const int n0 = sl * kSlice;
      stageRows(sm, q1 + kQ_W2, q1 + kQ_B2, kH, kH, n0);
      mm16(sm, s.qa1, kH, kH, B, [&](int r, float* acc) {
        float dl[kSlice];
#pragma unroll
        for (int j = 0; j < kSlice; ++j) {
          acc[j] = tanhf(acc[j] + sm.bias[j]);
          dl[j] = (dqa * ld(q1 + kQ_W3 + n0 + j)) * (1.0f - acc[j] * acc[j]);
        }
        store16(s.qa2 + (int64_t)r * kH + n0, acc);
        store16(s.qd2 + (int64_t)r * kH + n0, dl);
      });
    }
    clusterSync();
    // ---- phase 15: Q1 delta at fc1 ----
    for (int sl = c; sl < kSlices; sl += nc) bwdSlice(sm, q1 + kQ_W2, s.qd2, s.qa1, s.qd1, sl * kSlice, B);
    clusterSync();
    // ---- phase 16 (rows): dL/dpi through Q1's action columns and the normalisation; delta at the actor's fc3; Q1 value ----
    for (int r = gwarp; r < B; r += gwarps) {
      float v[kAct];
#pragma unroll
      for (int j = 0; j < kAct; ++j) {  // column kObs + j of fc1.weight [256, 22]
        float sacc = 0.0f;
#pragma unroll
        for (int i = 0; i < kH / 32; ++i) {
          const int n = lane + 32 * i;
          sacc = fmaf(ld(s.qd1 + (int64_t)r * kH + n), ld(q1 + kQ_W1 + n * kQin + kObs + j), sacc);
        }
        v[j] = warpSum(sacc);
      }
      const float qv = dot256(s.qa2 + (int64_t)r * kH, q1 + kQ_W3) + ld(q1 + kQ_B3);
      if (lane == 0) s.aloss[r] = qv;
      if (lane < kAct) {
        const float gn = lane == 0 ? v[0] : lane == 1 ? v[1] : lane == 2 ? v[2] : v[3];
        const float ga = norm ? (gn * 2.0f) / range[lane] : gn;
        const float p = ld(s.pi + r * kAct + lane);
        s.da3[r * kAct + lane] = ga * (1.0f - p * p);
      }
    }
    clusterSync();
    // ---- phase 17: actor delta at fc2, dW2 / db2 / dW3; db3 and the actor loss on CTA 0 ----
    for (int sl = c; sl < kSlices; sl += nc) {
      const int k0 = sl * kSlice;
      for (int i = t; i < B * kSlice; i += kThreads) {
        const int r = i >> 4, j = i & 15;
        float g = 0.0f;
#pragma unroll
        for (int q = 0; q < kAct; ++q) g = fmaf(ld(s.da3 + r * kAct + q), ld(actor + kA_W3 + q * kH + k0 + j), g);
        const float y = ld(s.p2 + (int64_t)r * kH + k0 + j);
        s.ad2[(int64_t)r * kH + k0 + j] = g * (1.0f - y * y);
      }
      __syncthreads();
      dwSlice(sm, s.ad2, k0, s.p1, kH, kH, B, s.gA + kA_W2, s.gA + kA_B2);
      for (int q = 0; q < kAct; ++q) colsum16(sm, s.p2, kH, k0, s.da3 + q, kAct, B, s.gA + kA_W3 + q * kH + k0);
    }
    if (c == 0 && warp < kAct + 1) {  // warps 0..3: db3; warp 4: the actor loss
      float sacc = 0.0f;
      for (int r = lane; r < B; r += 32) sacc += warp < kAct ? ld(s.da3 + r * kAct + warp) : ld(s.aloss + r);
      sacc = warpSum(sacc);
      if (lane == 0) {
        if (warp < kAct) s.gA[kA_B3 + warp] = sacc;
        else a.losses[0] = -(sacc / (float)B);
      }
    }
    clusterSync();
    // ---- phase 18: actor delta at fc1, dW1 / db1 ----
    for (int sl = c; sl < kSlices; sl += nc) {
      const int k0 = sl * kSlice;
      bwdSlice(sm, actor + kA_W2, s.ad2, s.p1, s.ad1, k0, B);
      __syncthreads();
      dwSlice(sm, s.ad1, k0, s.s, kObsLd, kObs, B, s.gA + kA_W1, s.gA + kA_B1);
    }
    clusterSync();
    // ---- phase 19: actor Adam ----
    adam(actorW, arena + kOffMActor, arena + kOffVActor, s.gA, kActorParams, a.lrA, a.wdA, tA, gtid, gstride);
    clusterSync();
    // ---- phase 20: Polyak ----
    polyak(arena + kOffTActor, actorW, kActorParams, a.tauA, gtid, gstride);
    polyak(arena + kOffTCritic, critic, kCriticParams, a.tauC, gtid, gstride);
  }
  if (c == 0 && t == 0) {  // every CTA read the counters before its first cluster barrier
    ctr[0] = tC;
    if (a.doActor) ctr[1] = tA;
    ctr[2] = noiseCtr + 1;
  }
}

}  // namespace hk_td3
