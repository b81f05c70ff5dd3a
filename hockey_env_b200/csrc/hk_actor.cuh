// hk_actor.cuh -- the reference's TD3 actor (ActorNetwork.forward, rl/td3/networks.py:17-20:
// tanh(W3 tanh(W2 tanh(W1 obs + b1) + b2) + b3), 18 -> 256 -> 256 -> 4) as ONE fused sm_100a kernel on the 5th-generation
// tensor cores (BASELINE config 5: the actor consumes the env's observation tensor in place and writes the action tensor
// the next hk_step reads).
//
// This is the one GEMM-shaped op next to the env path, so it runs on tcgen05: a CTA owns 128 observation rows at a time
// (UMMA M = 128); the three weight matrices stay resident in shared memory (bf16, K-major, 8x16-byte core matrices, no
// swizzle) for the whole launch; `tcgen05.mma.cta_group::1.kind::f16` accumulates each layer in fp32 in tensor memory
// (TMEM); every thread owns one row: it reads its accumulator row back with `tcgen05.ld`, adds the bias, applies tanh and
// writes the activations straight into shared memory as the next layer's A operand, so the hidden activations never touch
// HBM and there is one launch instead of nine.  HBM traffic: 72 B in, 16 B out per row.
//
// Numerics: layer 1 (whose inputs are raw observations of magnitude up to ~10) runs in TF32 (kind::tf32, 11-bit
// significands), layers 2 and 3 (inputs in [-1, 1]) in bf16; fp32 accumulation and bias everywhere, tanh.approx.f32.  Mean
// |out - fp32| ~ 2.5e-3; a trained policy has steep regions where any rounding moves an output by ~0.1, so the check that
// matters is behavioural: same win rate as the fp32 module (tests/test_actor_kernel.py).
// Operand roundings, as measured on a B200 (tests/test_actor_numerics.py): the observations go through cvt.rna.tf32
// (nearest, ties away); W1 is packed as raw f32 bits and kind::tf32 drops their low 13 significand bits (truncation toward
// zero, not rounding); W2, W3 and the hidden activations are rounded to nearest even bf16.  tanh.approx.f32 showed a
// relative error of at most 2^-16.6 (the PTX ISA bounds it by 2^-10.987).  A float64 model of these roundings stays within
// RMS 3.5e-4 of the kernel on the trained policies.
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace hk_actor {

constexpr int kRows = 128;   // rows per tile = UMMA M
constexpr int kObs = 18;     // observation width
constexpr int kK1 = 24;      // layer-1 K, padded to three TF32 UMMA K-steps of 8
constexpr int kHidden = 256;
constexpr int kN3 = 16;      // layer-3 N, padded from 4 to the smallest UMMA N for M = 128
constexpr int kAct = 4;
constexpr int kThreads = 128;

// packed parameter block (packed by the host side, actor.py FusedActor.pack, or on the device, k_actor_pack): byte offsets
constexpr int kOffW1 = 0;                                // [kHidden x kK1]     tf32 (f32 bits), canonical K-major core-matrix order
constexpr int kOffW2 = kOffW1 + kHidden * kK1 * 4;       // [kHidden x kHidden] bf16
constexpr int kOffW3 = kOffW2 + kHidden * kHidden * 2;   // [kN3 x kHidden]     bf16 (rows 4..15 zero)
constexpr int kOffB1 = kOffW3 + kN3 * kHidden * 2;       // kHidden f32
constexpr int kOffB2 = kOffB1 + kHidden * 4;             // kHidden f32
constexpr int kOffB3 = kOffB2 + kHidden * 4;             // 16 f32 (4 used)
constexpr int kParamBytes = kOffB3 + 64;

// shared memory: the parameter block, then the A operands
constexpr int kOffA = kParamBytes;                       // [kRows x kHidden] bf16: layer-2 / layer-3 A operand
constexpr int kOffX = kOffA;                             // [kRows x kK1] tf32: layer-1 A operand (dead once layer 1 is done: aliased)
constexpr int kOffBar = kOffA + kRows * kHidden * 2;     // mbarrier (8 B) + TMEM base address (4 B)
constexpr int kSmemBytes = kOffBar + 16;

__device__ __forceinline__ uint32_t smemAddr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// UMMA shared-memory matrix descriptor, K-major, SWIZZLE_NONE: 8-row x 16-byte core matrices; `sbo` = byte distance between
// core matrices along M/N (8-row groups), `lbo` = byte distance between the two 16-byte K chunks of one K = 16 step
__device__ __forceinline__ uint64_t umaDesc(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | ((uint64_t)(lbo >> 4) << 16) | ((uint64_t)(sbo >> 4) << 32) | (1ull << 46);
}
// instruction descriptor: D = f32, A = B = bf16 (fmt 1) or tf32 (fmt 2), both K-major, M x N
__host__ __device__ constexpr uint32_t instrDesc(int m, int n, uint32_t fmt) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}
__device__ __forceinline__ void umma(uint32_t tmemD, uint64_t descA, uint64_t descB, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}\n" ::"r"(tmemD),
      "l"(descA), "l"(descB), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
__device__ __forceinline__ void ummaTf32(uint32_t tmemD, uint64_t descA, uint64_t descB, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, {%5, %5, %5, %5}, p;\n\t}\n" ::"r"(tmemD),
      "l"(descA), "l"(descB), "r"(idesc), "r"(accumulate), "r"(0u)
      : "memory");
}
__device__ __forceinline__ uint32_t toTf32(float x) {
  uint32_t y;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void ummaCommit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbarWait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}\n"
                 : "=r"(ok)
                 : "r"(bar), "r"(parity)
                 : "memory");
  } while (!ok);
}
__device__ __forceinline__ float tanhApprox(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t packBf16(float a, float b) {
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
// 32 consecutive accumulator columns of this thread's TMEM lane (= its row)
__device__ __forceinline__ void tmemLoad32(uint32_t taddr, float* v) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, "
      "%18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
        "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int k = 0; k < 32; ++k) v[k] = __uint_as_float(r[k]);
}

// hidden layer epilogue: this thread's 256 accumulator columns -> tanh(acc + bias) -> bf16 -> A operand row in smem
__device__ __forceinline__ void hiddenEpilogue(uint32_t taddr, const float* bias, unsigned char* sA) {
  const int t = threadIdx.x;
#pragma unroll 1
  for (int c = 0; c < kHidden / 32; ++c) {
    float v[32];
    tmemLoad32(taddr + (uint32_t)(c * 32), v);
#pragma unroll
    for (int q = 0; q < 4; ++q) {  // four 16-byte K chunks of 8 activations each
      uint32_t w[4];
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const int k = q * 8 + 2 * p;
        w[p] = packBf16(tanhApprox(v[k] + bias[c * 32 + k]), tanhApprox(v[k + 1] + bias[c * 32 + k + 1]));
      }
      // element (row t, column kc * 8 ..): chunk kc starts at kc * (kRows * 16) bytes, row t at + t * 16
      *reinterpret_cast<uint4*>(sA + (c * 4 + q) * (kRows * 16) + t * 16) = make_uint4(w[0], w[1], w[2], w[3]);
    }
  }
}

// Per-CTA state of the tile loop: the TMEM accumulator base, this warp's lanes of it, the mbarrier the MMAs commit to and
// the shared-memory addresses of the operands.
struct TileCtx {
  unsigned char* smem;
  uint32_t tmem, myT, barA, sW1, sW2, sW3, sX, sAa;
};

// the parameter block (global, L2-resident after the first CTA) -> shared memory.  The tile body's
// `fence.proxy.async.shared::cta`, executed by every thread after these writes, makes them visible to the tensor core.
__device__ __forceinline__ void loadParams(unsigned char* smem, const unsigned char* __restrict__ params) {
  for (int k = threadIdx.x; k < kParamBytes / 16; k += kThreads)
    reinterpret_cast<uint4*>(smem)[k] = reinterpret_cast<const uint4*>(params)[k];
}

// mbarrier init and the 512-column TMEM allocation (one warp: layer-1 accumulator [0,256), layer-2 [256,512), layer-3
// [0,16)); ends in a block barrier.  Free the columns with `actorTeardown`.
__device__ __forceinline__ TileCtx actorSetup(unsigned char* smem) {
  const int t = threadIdx.x, warp = t >> 5;
  uint64_t* bar = reinterpret_cast<uint64_t*>(smem + kOffBar);
  uint32_t* tmemSlot = reinterpret_cast<uint32_t*>(smem + kOffBar + 8);
  if (t == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smemAddr(bar)));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smemAddr(tmemSlot)), "r"(512));
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::);
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  TileCtx c;
  c.smem = smem;
  c.tmem = *tmemSlot;
  c.myT = c.tmem + ((uint32_t)(warp * 32) << 16);  // this warp's 32 TMEM lanes
  c.barA = smemAddr(bar);
  c.sW1 = smemAddr(smem + kOffW1);
  c.sW2 = smemAddr(smem + kOffW2);
  c.sW3 = smemAddr(smem + kOffW3);
  c.sX = smemAddr(smem + kOffX);
  c.sAa = smemAddr(smem + kOffA);
  return c;
}

__device__ __forceinline__ void actorTeardown(const TileCtx& c) {
  if ((threadIdx.x >> 5) == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(c.tmem), "r"(512));
}

// ---------------------------------------------------------------------------------------------------------------------
// Exploration / target-policy-smoothing noise in the layer-3 epilogue (the `kGaussian` instantiations):
//   act = clamp(tanh(MLP(obs)) + clip(sigma * z, -clip, clip), -1, 1),   z = four standard normals per row.
// Row i's normals come from ONE Philox4x32-10 call, hk::philox(seed, row0 + i, (uint32_t)ctr,
// HK_STREAM_ACTOR_NOISE | (uint32_t)(ctr >> 32) << 8), ctr = the call's counter (read from device memory, so a replayed
// graph draws fresh noise; the low 56 bits count), and Box-Muller on its words (x, y) -> z0, z1 and (z, w) -> z2, z3:
//   u1 = ((a >> 8) + 1) * 2^-24  in (0, 1]  (log finite),   u2 = (b >> 8) * 2^-24  in [0, 1),
//   r = sqrtf(-2 logf(u1)),   (z_even, z_odd) = (r cospif(2 u2), r sinpif(2 u2)).
// A row's noise depends on its key only: not on n, the tile order or (in the pool) the grouping; `row0` lets shards of
// one batch agree.  |z| <= sqrt(48 ln 2) ~ 5.77.
//
// Exploration (the `kExplore` instantiations): the same z drives a per-row AR(1) process whose state lives in device
// memory, with (rho, scale, clip) taken from a slot table in device memory (float4 {rho, scale, clip, reserved} per slot;
// the single-weight-set kernel reads slot 0, the pool kernel slot s for the rows of snapshot s):
//   x  = reset[i] ? 0 : state[i][j]
//   x' = fl(fl(rho * x) + fl(scale * z_j))        (rho == 0: x' = fl(scale * z_j); state and reset are not read)
//   state[i][j] = x',   act[i][j] = clamp(tanh(MLP(obs[i]))_j + clip(x', +-clip), -1, 1)
// rho = 0, scale = sigma is the Gaussian epilogue above bit for bit; OU noise dx = -theta x dt + sigma sqrt(dt) dW is
// rho = 1 - theta dt, scale = sigma sqrt(dt).  `state` is indexed by the local row i (not row0 + i), `reset` may be NULL.
// The table values are arithmetic operands only (never an index or a trip count), so any values are memory-safe.
enum NoiseMode { kPlain, kGaussian, kExplore };

struct NoiseKey {
  uint64_t seed;
  long long row0;
  uint32_t c2, c3;   // Philox counter words 2 and 3 (counter low word, stream tag | counter high bits << 8)
  float sigma, clip; // clip = +inf: no clip.  kExplore: sigma is the slot's scale
  float rho;                         // kExplore only: the slot's AR(1) coefficient
  float4* state;                     // kExplore only: [n] rows of 4 f32
  const uint8_t* reset;              // kExplore only: [n] or NULL
};

__device__ __forceinline__ NoiseKey noiseKey(uint64_t seed, const uint64_t* counter, float sigma, float clip, long long row0) {
  const uint64_t ctr = *counter;
  NoiseKey k;
  k.seed = seed;
  k.row0 = row0;
  k.c2 = (uint32_t)ctr;
  k.c3 = (uint32_t)hk::HK_STREAM_ACTOR_NOISE | ((uint32_t)(ctr >> 32) << 8);
  k.sigma = sigma;
  k.clip = clip;
  return k;
}

__device__ __forceinline__ void boxMuller(uint32_t a, uint32_t b, float& z0, float& z1) {
  const float u1 = (float)((a >> 8) + 1u) * (1.0f / 16777216.0f);
  const float u2 = (float)(b >> 8) * (1.0f / 16777216.0f);
  const float r = sqrtf(-2.0f * logf(u1));
  float s, c;
  sincospif(2.0f * u2, &s, &c);
  z0 = r * c;
  z1 = r * s;
}

__device__ __forceinline__ float addNoise(float a, float z, const NoiseKey& k) {
  const float e = fminf(fmaxf(k.sigma * z, -k.clip), k.clip);
  return fminf(fmaxf(a + e, -1.0f), 1.0f);
}

// kExplore: a slot {rho, scale, clip, reserved} of the table into the key
__device__ __forceinline__ void setSlot(NoiseKey& k, const float4& s) {
  k.rho = s.x;
  k.sigma = s.y;
  k.clip = s.z;
}

__device__ __forceinline__ NoiseKey exploreKey(uint64_t seed, const uint64_t* counter, const float4* slots, float4* state,
                                               const uint8_t* reset, long long row0) {
  NoiseKey k = noiseKey(seed, counter, 0.0f, 0.0f, row0);
  setSlot(k, slots[0]);
  k.state = state;
  k.reset = reset;
  return k;
}

// kExplore: one AR(1) step of row `row` (see NoiseKey); returns x', the pre-clip state, and stores it.  The products and
// the sum are rounded separately (__fmul_rn / __fadd_rn are never contracted into an FMA).
__device__ __forceinline__ float4 exploreStep(long long row, float z0, float z1, float z2, float z3, const NoiseKey& k) {
  float4 x = make_float4(__fmul_rn(k.sigma, z0), __fmul_rn(k.sigma, z1), __fmul_rn(k.sigma, z2), __fmul_rn(k.sigma, z3));
  if (k.rho != 0.0f) {
    float4 p = make_float4(0.0f, 0.0f, 0.0f, 0.0f);
    if (!(k.reset && k.reset[row])) p = k.state[row];
    x.x = __fadd_rn(__fmul_rn(k.rho, p.x), x.x);
    x.y = __fadd_rn(__fmul_rn(k.rho, p.y), x.y);
    x.z = __fadd_rn(__fmul_rn(k.rho, p.z), x.z);
    x.w = __fadd_rn(__fmul_rn(k.rho, p.w), x.w);
  }
  k.state[row] = x;
  return x;
}

__device__ __forceinline__ float addExplore(float a, float x, const NoiseKey& k) {
  const float e = fminf(fmaxf(x, -k.clip), k.clip);
  return fminf(fmaxf(a + e, -1.0f), 1.0f);
}

// One tile of 128 rows through the three layers with the weights now in shared memory.  Thread t owns TMEM lane t; `row`
// is the observation / action row it reads and writes, or -1 for a padding lane (zero input, nothing stored).  The only
// thing the callers differ in is how a thread finds its row.  Ends in a block barrier: on return every MMA of the tile
// has completed and every thread is done with the tile's shared memory (the weights may be replaced).  kGaussian adds the
// noise of `nk` to the four outputs, kExplore its AR(1) exploration noise (see NoiseKey); kPlain ignores `nk`.
template <NoiseMode kMode>
__device__ __forceinline__ void actorTile(const TileCtx& c, uint32_t& phase, const float* __restrict__ obs,
                                          float* __restrict__ act, int actStride, long long row, const NoiseKey& nk) {
  const int t = threadIdx.x;
  unsigned char* smem = c.smem;
  const uint32_t tmem = c.tmem, myT = c.myT, barA = c.barA;
  const float* b1 = reinterpret_cast<const float*>(smem + kOffB1);
  const float* b2 = reinterpret_cast<const float*>(smem + kOffB2);
  const float* b3 = reinterpret_cast<const float*>(smem + kOffB3);
  unsigned char* sA = smem + kOffA;
  // ---- this thread's observation row -> tf32 -> layer-1 A operand (K padded 18 -> 24 with zeros) ----
  float o[kK1];
#pragma unroll
  for (int k = 0; k < kK1; ++k) o[k] = 0.0f;
  if (row >= 0) {
    const float2* src = reinterpret_cast<const float2*>(obs + row * kObs);
#pragma unroll
    for (int k = 0; k < kObs / 2; ++k) {
      const float2 v = src[k];
      o[2 * k] = v.x;
      o[2 * k + 1] = v.y;
    }
  }
#pragma unroll
  for (int q = 0; q < kK1 / 4; ++q)  // 16-byte K chunks of four tf32 values: chunk q at q * (kRows * 16) bytes, row t at + t * 16
    *reinterpret_cast<uint4*>(smem + kOffX + q * (kRows * 16) + t * 16) =
        make_uint4(toTf32(o[4 * q]), toTf32(o[4 * q + 1]), toTf32(o[4 * q + 2]), toTf32(o[4 * q + 3]));
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy smem writes -> visible to the tensor core
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  // ---- layer 1 (TF32): D1[128 x 256] = X[128 x 24] W1^T ----
  if (t == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
    for (int ks = 0; ks < kK1 / 8; ++ks)
      ummaTf32(tmem, umaDesc(c.sX + ks * 2 * (kRows * 16), kRows * 16, 128), umaDesc(c.sW1 + ks * 2 * (kHidden * 16), kHidden * 16, 128),
               instrDesc(kRows, kHidden, 2), ks > 0);
    ummaCommit(barA);
  }
  mbarWait(barA, phase);
  phase ^= 1;
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  hiddenEpilogue(myT, b1, sA);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  // ---- layer 2: D2[128 x 256] = H1[128 x 256] W2^T ----
  if (t == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
    for (int ks = 0; ks < kHidden / 16; ++ks)
      umma(tmem + kHidden, umaDesc(c.sAa + ks * 2 * (kRows * 16), kRows * 16, 128),
           umaDesc(c.sW2 + ks * 2 * (kHidden * 16), kHidden * 16, 128), instrDesc(kRows, kHidden, 1), ks > 0);
    ummaCommit(barA);
  }
  mbarWait(barA, phase);
  phase ^= 1;
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  hiddenEpilogue(myT + kHidden, b2, sA);  // layer 2 has finished reading H1: its buffer takes H2
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  // ---- layer 3: D3[128 x 16] = H2[128 x 256] W3^T (4 real outputs) ----
  if (t == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
    for (int ks = 0; ks < kHidden / 16; ++ks)
      umma(tmem, umaDesc(c.sAa + ks * 2 * (kRows * 16), kRows * 16, 128), umaDesc(c.sW3 + ks * 2 * (kN3 * 16), kN3 * 16, 128),
           instrDesc(kRows, kN3, 1), ks > 0);
    ummaCommit(barA);
  }
  mbarWait(barA, phase);
  phase ^= 1;
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  {
    uint32_t r0, r1, r2, r3;
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];\n" : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(myT));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    if (row >= 0) {
      float* dst = act + row * actStride;
      if constexpr (kMode == kGaussian) {
        const hk::U4 w = hk::philox(nk.seed, (uint64_t)(nk.row0 + row), nk.c2, nk.c3);
        float z0, z1, z2, z3;
        boxMuller(w.x, w.y, z0, z1);
        boxMuller(w.z, w.w, z2, z3);
        dst[0] = addNoise(tanhApprox(__uint_as_float(r0) + b3[0]), z0, nk);
        dst[1] = addNoise(tanhApprox(__uint_as_float(r1) + b3[1]), z1, nk);
        dst[2] = addNoise(tanhApprox(__uint_as_float(r2) + b3[2]), z2, nk);
        dst[3] = addNoise(tanhApprox(__uint_as_float(r3) + b3[3]), z3, nk);
      } else if constexpr (kMode == kExplore) {
        const hk::U4 w = hk::philox(nk.seed, (uint64_t)(nk.row0 + row), nk.c2, nk.c3);
        float z0, z1, z2, z3;
        boxMuller(w.x, w.y, z0, z1);
        boxMuller(w.z, w.w, z2, z3);
        const float4 x = exploreStep(row, z0, z1, z2, z3, nk);
        dst[0] = addExplore(tanhApprox(__uint_as_float(r0) + b3[0]), x.x, nk);
        dst[1] = addExplore(tanhApprox(__uint_as_float(r1) + b3[1]), x.y, nk);
        dst[2] = addExplore(tanhApprox(__uint_as_float(r2) + b3[2]), x.z, nk);
        dst[3] = addExplore(tanhApprox(__uint_as_float(r3) + b3[3]), x.w, nk);
      } else {
        dst[0] = tanhApprox(__uint_as_float(r0) + b3[0]);
        dst[1] = tanhApprox(__uint_as_float(r1) + b3[1]);
        dst[2] = tanhApprox(__uint_as_float(r2) + b3[2]);
        dst[3] = tanhApprox(__uint_as_float(r3) + b3[3]);
      }
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();  // the next tile's layer 1 overwrites the columns layer 3 was just read from
}

// one weight set, rows 0..n-1 in order: tile `tile` holds rows tile * 128 + t
template <NoiseMode kMode>
__device__ __forceinline__ void actorMlp(const unsigned char* __restrict__ params, const float* __restrict__ obs,
                                         float* __restrict__ act, int actStride, long long n, const NoiseKey& nk) {
  extern __shared__ __align__(128) unsigned char smem[];
  loadParams(smem, params);  // once per CTA
  const TileCtx c = actorSetup(smem);
  uint32_t phase = 0;
  const long long tiles = (n + kRows - 1) / kRows;
  for (long long tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const long long row = tile * kRows + threadIdx.x;
    actorTile<kMode>(c, phase, obs, act, actStride, row < n ? row : -1, nk);
  }
  actorTeardown(c);
}

__global__ void __launch_bounds__(kThreads, 1) k_actor_mlp(const unsigned char* __restrict__ params, const float* __restrict__ obs,
                                                           float* __restrict__ act, int actStride, long long n) {
  actorMlp<kPlain>(params, obs, act, actStride, n, NoiseKey{});
}

__global__ void __launch_bounds__(kThreads, 1) k_actor_mlp_noisy(const unsigned char* __restrict__ params, const float* __restrict__ obs,
                                                                 float* __restrict__ act, int actStride, long long n, uint64_t seed,
                                                                 const uint64_t* __restrict__ counter, float sigma, float clip,
                                                                 long long row0) {
  actorMlp<kGaussian>(params, obs, act, actStride, n, noiseKey(seed, counter, sigma, clip, row0));
}

__global__ void __launch_bounds__(kThreads, 1) k_actor_mlp_explore(const unsigned char* __restrict__ params, const float* __restrict__ obs,
                                                                   float* __restrict__ act, int actStride, long long n, uint64_t seed,
                                                                   const uint64_t* __restrict__ counter, const float4* __restrict__ slots,
                                                                   float4* __restrict__ state, const uint8_t* __restrict__ reset,
                                                                   long long row0) {
  actorMlp<kExplore>(params, obs, act, actStride, n, exploreKey(seed, counter, slots, state, reset, row0));
}

// ---------------------------------------------------------------------------------------------------------------------
// Snapshot pool: act[i] = actor_{choice[i]}(obs[i]) for K weight sets laid out back to back (K blocks of kParamBytes),
// rows with choice[i] outside [0, K) untouched.  Rows are grouped by snapshot on the device, with no host sync:
//   cudaMemsetAsync(counts) -> k_pool_count (histogram) -> k_pool_scan (group and tile offsets, one block)
//   -> k_pool_scatter (row lists) -> k_actor_pool_mlp (persistent, tiles of one group share one weight set).
// Scratch layout (int32 words, caller-owned, poolScratchWords(n, K) of them):
//   counts[K] | groupOff[K + 1] | tileOff[K + 1] | cursor[K] | rows[n]
// groupOff[s] is where group s starts in rows[], tileOff[s] its first tile; tileOff[K] is the total tile count.
constexpr int kPoolMaxK = 4096;
constexpr int kPoolThreads = 256;        // count / scatter blocks
constexpr int kPoolItems = 8;            // rows per thread of one scatter block
constexpr int kScanThreads = 1024;

__host__ __device__ constexpr long long poolAlign4(long long words) { return (words + 3) & ~3LL; }  // 16-byte sections
__host__ __device__ inline long long poolOffGroup(int k) { return poolAlign4(k); }
__host__ __device__ inline long long poolOffTile(int k) { return poolOffGroup(k) + poolAlign4(k + 1); }
__host__ __device__ inline long long poolOffCursor(int k) { return poolOffTile(k) + poolAlign4(k + 1); }
__host__ __device__ inline long long poolOffRows(int k) { return poolOffCursor(k) + poolAlign4(k); }
__host__ __device__ inline long long poolScratchWords(long long n, int k) { return poolOffRows(k) + poolAlign4(n); }

// histogram of the valid choices: per-block counts in shared memory, then one global add per non-empty bin
__global__ void __launch_bounds__(kPoolThreads) k_pool_count(const int32_t* __restrict__ choice, long long n, int k,
                                                             int32_t* __restrict__ counts) {
  extern __shared__ int32_t hist[];
  for (int s = threadIdx.x; s < k; s += blockDim.x) hist[s] = 0;
  __syncthreads();
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const int c = choice[i];
    if (c >= 0 && c < k) atomicAdd(&hist[c], 1);
  }
  __syncthreads();
  for (int s = threadIdx.x; s < k; s += blockDim.x)
    if (hist[s]) atomicAdd(&counts[s], hist[s]);
}

// exclusive scans of the row counts and of the tile counts ceil(count / 128), one block; cursor[s] = groupOff[s]
__global__ void __launch_bounds__(kScanThreads) k_pool_scan(int32_t* __restrict__ scratch, int k) {
  __shared__ int2 warpSum[kScanThreads / 32];
  const int32_t* counts = scratch;
  int32_t* groupOff = scratch + poolOffGroup(k);
  int32_t* tileOff = scratch + poolOffTile(k);
  int32_t* cursor = scratch + poolOffCursor(k);
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const int per = (k + kScanThreads - 1) / kScanThreads;  // consecutive bins of this thread
  const int s0 = min(t * per, k), s1 = min(s0 + per, k);
  int2 mine = make_int2(0, 0);
  for (int s = s0; s < s1; ++s) {
    mine.x += counts[s];
    mine.y += (counts[s] + kRows - 1) / kRows;
  }
  int2 inc = mine;  // inclusive scan over the warp, then over the warp totals
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const int x = __shfl_up_sync(0xffffffffu, inc.x, d), y = __shfl_up_sync(0xffffffffu, inc.y, d);
    if (lane >= d) inc.x += x, inc.y += y;
  }
  if (lane == 31) warpSum[warp] = inc;
  __syncthreads();
  if (warp == 0) {
    int2 w = warpSum[lane];
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const int x = __shfl_up_sync(0xffffffffu, w.x, d), y = __shfl_up_sync(0xffffffffu, w.y, d);
      if (lane >= d) w.x += x, w.y += y;
    }
    warpSum[lane] = w;
  }
  __syncthreads();
  int2 run = make_int2(inc.x - mine.x, inc.y - mine.y);
  if (warp > 0) run.x += warpSum[warp - 1].x, run.y += warpSum[warp - 1].y;
  for (int s = s0; s < s1; ++s) {
    groupOff[s] = run.x;
    cursor[s] = run.x;
    tileOff[s] = run.y;
    run.x += counts[s];
    run.y += (counts[s] + kRows - 1) / kRows;
  }
  if (t == kScanThreads - 1) {
    groupOff[k] = run.x;
    tileOff[k] = run.y;
  }
}

// row lists: a block takes kPoolThreads * kPoolItems consecutive rows, ranks them per group in shared memory, reserves
// one range per non-empty group with a single atomic on that group's cursor and writes the row indices there
__global__ void __launch_bounds__(kPoolThreads) k_pool_scatter(const int32_t* __restrict__ choice, long long n, int k,
                                                               int32_t* __restrict__ scratch) {
  extern __shared__ int32_t sh[];  // hist[k] | base[k]
  int32_t* hist = sh;
  int32_t* base = sh + k;
  int32_t* cursor = scratch + poolOffCursor(k);
  int32_t* rows = scratch + poolOffRows(k);
  for (long long first = blockIdx.x * (long long)(kPoolThreads * kPoolItems); first < n;
       first += (long long)gridDim.x * (kPoolThreads * kPoolItems)) {
    for (int s = threadIdx.x; s < k; s += blockDim.x) hist[s] = 0;
    __syncthreads();
    int c[kPoolItems], rank[kPoolItems];
#pragma unroll
    for (int j = 0; j < kPoolItems; ++j) {
      const long long i = first + j * kPoolThreads + threadIdx.x;
      c[j] = i < n ? choice[i] : -1;
      rank[j] = (c[j] >= 0 && c[j] < k) ? atomicAdd(&hist[c[j]], 1) : -1;
    }
    __syncthreads();
    for (int s = threadIdx.x; s < k; s += blockDim.x)
      if (hist[s]) base[s] = atomicAdd(&cursor[s], hist[s]);
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kPoolItems; ++j)
      if (rank[j] >= 0) rows[base[c[j]] + rank[j]] = (int32_t)(first + j * kPoolThreads + threadIdx.x);
    __syncthreads();  // hist / base are reused by the next chunk
  }
}

// Persistent: CTA b walks the contiguous tile range [b T / G, (b + 1) T / G) of the T = tileOff[K] tiles, so it crosses few
// group boundaries; it copies a snapshot's weights into shared memory only when the group changes.  Tile j of group s holds
// rows[groupOff[s] + j * 128 + t]; lanes past the group's end are padding.
// kExplore: `slots` is the slot table (slot s for the rows of snapshot s); the other modes pass NULL.
template <NoiseMode kMode>
__device__ __forceinline__ void actorPoolMlp(const unsigned char* __restrict__ params, int k, const int32_t* __restrict__ scratch,
                                             const float* __restrict__ obs, float* __restrict__ act, int actStride,
                                             const NoiseKey& nk, const float4* __restrict__ slots) {
  extern __shared__ __align__(128) unsigned char smem[];
  const int32_t* groupOff = scratch + poolOffGroup(k);
  const int32_t* tileOff = scratch + poolOffTile(k);
  const int32_t* rows = scratch + poolOffRows(k);
  const long long total = tileOff[k];
  const long long t0 = total * blockIdx.x / gridDim.x, t1 = total * (blockIdx.x + 1) / gridDim.x;
  if (t0 >= t1) return;  // nothing to do: no TMEM allocated, no barrier entered
  const TileCtx c = actorSetup(smem);
  int lo = 0, hi = k - 1;  // the group of tile t0: the last s with tileOff[s] <= t0 (empty groups share their offset)
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (tileOff[mid] <= t0) lo = mid; else hi = mid - 1;
  }
  int s = lo, loaded = -1;
  uint32_t phase = 0;
  NoiseKey key = nk;
  for (long long tile = t0; tile < t1; ++tile) {
    while (tile >= tileOff[s + 1]) ++s;
    if (s != loaded) {
      // the previous tile (if any) ended with its layer-3 MMAs complete and a block barrier: the old weights are dead
      loadParams(smem, params + (size_t)s * kParamBytes);
      if constexpr (kMode == kExplore) setSlot(key, slots[s]);  // uniform over the tile: the rho == 0 branch does not diverge
      loaded = s;
    }
    const int local = (int)(tile - tileOff[s]) * kRows + threadIdx.x;
    const int count = groupOff[s + 1] - groupOff[s];
    actorTile<kMode>(c, phase, obs, act, actStride, local < count ? (long long)rows[groupOff[s] + local] : -1LL, key);
  }
  actorTeardown(c);
}

__global__ void __launch_bounds__(kThreads, 1) k_actor_pool_mlp(const unsigned char* __restrict__ params, int k,
                                                                const int32_t* __restrict__ scratch, const float* __restrict__ obs,
                                                                float* __restrict__ act, int actStride) {
  actorPoolMlp<kPlain>(params, k, scratch, obs, act, actStride, NoiseKey{}, nullptr);
}

__global__ void __launch_bounds__(kThreads, 1) k_actor_pool_mlp_noisy(const unsigned char* __restrict__ params, int k,
                                                                      const int32_t* __restrict__ scratch, const float* __restrict__ obs,
                                                                      float* __restrict__ act, int actStride, uint64_t seed,
                                                                      const uint64_t* __restrict__ counter, float sigma, float clip,
                                                                      long long row0) {
  actorPoolMlp<kGaussian>(params, k, scratch, obs, act, actStride, noiseKey(seed, counter, sigma, clip, row0), nullptr);
}

__global__ void __launch_bounds__(kThreads, 1) k_actor_pool_mlp_explore(const unsigned char* __restrict__ params, int k,
                                                                        const int32_t* __restrict__ scratch, const float* __restrict__ obs,
                                                                        float* __restrict__ act, int actStride, uint64_t seed,
                                                                        const uint64_t* __restrict__ counter, const float4* __restrict__ slots,
                                                                        float4* __restrict__ state, const uint8_t* __restrict__ reset,
                                                                        long long row0) {
  NoiseKey nk = noiseKey(seed, counter, 0.0f, 0.0f, row0);
  nk.state = state;
  nk.reset = reset;
  actorPoolMlp<kExplore>(params, k, scratch, obs, act, actStride, nk, slots);
}

// ---------------------------------------------------------------------------------------------------------------------
// Device-side pack: an ActorNetwork's fp32 parameters (fc1 [256, 18], fc2 [256, 256], fc3 [4, 256] row-major, biases)
// -> one kParamBytes block, byte-identical to actor.py FusedActor.pack.  Thread j writes 32-bit word j of the block:
// layer 1 as raw f32 bits, layers 2-3 as two bf16 (round to nearest even) of consecutive k, in K-major core-matrix order
// (element (n, k) of a [N, K] operand with e elements per 16-byte chunk at (k / e) * (N * 16) + n * 16 + (k % e) * size
// bytes), zeros in the padding (K 18 -> 24, fc3 rows 4 -> 16, b3 4 -> 16).
constexpr int kPackThreads = 256;
constexpr int kParamWords = kParamBytes / 4;

__device__ __forceinline__ uint32_t bf16Bits(float x) {
  const __nv_bfloat16 h = __float2bfloat16_rn(x);
  return (uint32_t)*reinterpret_cast<const uint16_t*>(&h);
}

// word `j` of a bf16 [nPad x kDim] operand (8 elements per chunk): elements (n, k), (n, k + 1) of w [nReal x kDim]
__device__ __forceinline__ uint32_t packBf16Word(const float* __restrict__ w, int j, int nPad, int nReal, int kDim) {
  const int chunk = j / (nPad * 4), rem = j % (nPad * 4);
  const int n = rem / 4, k = chunk * 8 + (rem % 4) * 2;
  if (n >= nReal) return 0u;
  return bf16Bits(w[n * kDim + k]) | (bf16Bits(w[n * kDim + k + 1]) << 16);
}

// word j < kParamWords of the packed block of one actor
__device__ __forceinline__ uint32_t packWord(const float* __restrict__ w1, const float* __restrict__ b1, const float* __restrict__ w2,
                                             const float* __restrict__ b2, const float* __restrict__ w3, const float* __restrict__ b3,
                                             int j) {
  uint32_t v;
  if (j < kOffW2 / 4) {  // layer 1: 4 f32 per chunk
    const int chunk = j / (kHidden * 4), rem = j % (kHidden * 4);
    const int n = rem / 4, k = chunk * 4 + rem % 4;
    v = k < kObs ? __float_as_uint(w1[n * kObs + k]) : 0u;
  } else if (j < kOffW3 / 4) {
    v = packBf16Word(w2, j - kOffW2 / 4, kHidden, kHidden, kHidden);
  } else if (j < kOffB1 / 4) {
    v = packBf16Word(w3, j - kOffW3 / 4, kN3, kAct, kHidden);
  } else if (j < kOffB2 / 4) {
    v = __float_as_uint(b1[j - kOffB1 / 4]);
  } else if (j < kOffB3 / 4) {
    v = __float_as_uint(b2[j - kOffB2 / 4]);
  } else {
    const int i = j - kOffB3 / 4;
    v = i < kAct ? __float_as_uint(b3[i]) : 0u;
  }
  return v;
}

__global__ void __launch_bounds__(kPackThreads) k_actor_pack(const float* __restrict__ w1, const float* __restrict__ b1,
                                                             const float* __restrict__ w2, const float* __restrict__ b2,
                                                             const float* __restrict__ w3, const float* __restrict__ b3,
                                                             uint32_t* __restrict__ out) {
  const int j = blockIdx.x * kPackThreads + threadIdx.x;
  if (j >= kParamWords) return;
  out[j] = packWord(w1, b1, w2, b2, w3, b3, j);
}

// K actors at once: slot s (blockIdx.y) of the pool table from the fp32 actor block at actors + s * stride, whose
// parameters lie back to back in state_dict order (fc1.weight, fc1.bias, fc2.weight, fc2.bias, fc3.weight, fc3.bias):
// exactly the actor block of a TD3 arena (hk_td3.cuh), so stride = the arena's size in floats packs a population.
constexpr int kActorFloats = kHidden * kObs + kHidden + kHidden * kHidden + kHidden + kAct * kHidden + kAct;
__global__ void __launch_bounds__(kPackThreads) k_actor_pack_many(const float* __restrict__ actors, long long stride,
                                                                  uint32_t* __restrict__ table) {
  const int j = blockIdx.x * kPackThreads + threadIdx.x;
  if (j >= kParamWords) return;
  const float* w1 = actors + (long long)blockIdx.y * stride;
  const float* b1 = w1 + kHidden * kObs;
  const float* w2 = b1 + kHidden;
  const float* b2 = w2 + kHidden * kHidden;
  const float* w3 = b2 + kHidden;
  const float* b3 = w3 + kAct * kHidden;
  table[(long long)blockIdx.y * kParamWords + j] = packWord(w1, b1, w2, b2, w3, b3, j);
}

}  // namespace hk_actor
