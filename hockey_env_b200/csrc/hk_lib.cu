// hk_lib.cu -- CUDA kernels and the C ABI (include/hockey_b200.h) of the batched HockeyEnv.
//
// One env per thread.  Each kernel stages the constant Scene into shared memory (polygon tables are
// indexed with per-lane indices in the narrow phase; shared memory serves divergent addresses far
// better than the constant cache), loads the env's 16 float4 groups with coalesced 128-bit
// accesses, runs hk::envTick and stores the groups back.  No tensor cores: the path is scalar
// fp32/fp64 integer-and-branch work (see DESIGN.md for the roofline discussion).
//
// Built for sm_100a only, with -fmad=false (see hk_math.cuh).  There is no CPU fallback in this
// library: without a CUDA device hk_create fails with HK_E_NODEVICE.
#include <cuda_runtime.h>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <cmath>
#include <string>

#include "../../include/hockey_b200.h"
#include "hk_tick.cuh"
#if !defined(HK_TU_INLINE)
#include "hk_actor.cuh"
#include "hk_td3.cuh"
#endif

using namespace hk;

namespace {

__constant__ Scene c_scene;

thread_local std::string g_err;
int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}
#define HK_CUDA(call)                                                                           \
  do {                                                                                          \
    cudaError_t _e = (call);                                                                    \
    if (_e != cudaSuccess)                                                                      \
      return fail(HK_E_CUDA, std::string(#call) + ": " + cudaGetErrorString(_e));               \
  } while (0)

struct DeviceGuard {
  int prev = -1;
  bool ok = true;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) ok = false;
    if (ok && prev != dev && cudaSetDevice(dev) != cudaSuccess) ok = false;
  }
  ~DeviceGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

constexpr int kBlock = 128;

__device__ __forceinline__ void stageScene(Scene* dst) {
  const uint32_t* src = reinterpret_cast<const uint32_t*>(&c_scene);
  uint32_t* d = reinterpret_cast<uint32_t*>(dst);
  for (int k = threadIdx.x; k < (int)(sizeof(Scene) / 4); k += blockDim.x) d[k] = src[k];
  __syncthreads();
}

__device__ __forceinline__ void loadEnv(const float4* __restrict__ core, int64_t n, int64_t i, Env& e) {
  F4 g[CORE_GROUPS];
#pragma unroll
  for (int k = 0; k < CORE_GROUPS; ++k) {
    // streaming (evict-first) accesses: at >= 262k envs the state stream would otherwise push the kernels' own code out of
    // L2 (ncu, k_fast at 1,048,576 envs: 18.6 cycles of no-instruction stall per issued instruction; profiles/README.md)
    float4 v = __ldcs(&core[(int64_t)k * n + i]);
    g[k] = F4{v.x, v.y, v.z, v.w};
  }
  groupsToEnv(g, e);
}
__device__ __forceinline__ void storeEnv(float4* __restrict__ core, int64_t n, int64_t i, const Env& e) {
  F4 g[CORE_GROUPS];
  envToGroups(e, g);
#pragma unroll
  for (int k = 0; k < CORE_GROUPS; ++k) __stcs(&core[(int64_t)k * n + i], make_float4(g[k].x, g[k].y, g[k].z, g[k].w));
}

__device__ __forceinline__ void flushInt(double* gstats, int slot, int v, int lane) {
  if (!__any_sync(0xffffffffu, v != 0)) return;  // most statistics are zero for a whole warp in most ticks
  int s = __reduce_add_sync(0xffffffffu, v);
  if (lane == 0 && s != 0) atomicAdd(&gstats[slot], (double)s);
}
__device__ __forceinline__ double warpSumD(double v) {
  for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
  return v;
}
// per-env contact reductions -> warp shuffles/redux, one atomic per warp and statistic
// The accumulators are replicated kStatsRows times (row = block index mod kStatsRows) so that the end-of-warp flushes of a
// whole grid do not queue up on sixteen addresses; readers sum the rows (k_sum_stats).
constexpr int kStatsRows = 64;
__device__ __forceinline__ double* statsRow(double* gstats) { return gstats + HK_STATS_DIM * (blockIdx.x & (kStatsRows - 1)); }
__device__ __forceinline__ void flushStats(double* gstats, const TickStats& st) {
  const int lane = threadIdx.x & 31;
  flushInt(gstats, 4, st.steps, lane);
  flushInt(gstats, 11, st.velIters, lane);
  flushInt(gstats, 9, st.touch1, lane);
  flushInt(gstats, 10, st.touch2, lane);
  flushInt(gstats, 12, st.toi, lane);
  flushInt(gstats, 13, st.overflow, lane);
  if (__any_sync(0xffffffffu, st.episodes != 0)) {
    flushInt(gstats, 0, st.episodes, lane);
    flushInt(gstats, 1, st.wins, lane);
    flushInt(gstats, 2, st.losses, lane);
    flushInt(gstats, 3, st.draws, lane);
    flushInt(gstats, 8, st.len, lane);
    double a = warpSumD(st.ret1), b = warpSumD(st.ret2), c = warpSumD(st.ret1sq);
    if (lane == 0) {
      atomicAdd(&gstats[5], a);
      atomicAdd(&gstats[6], b);
      atomicAdd(&gstats[7], c);
    }
  }
}

}  // namespace
namespace hkk {  // named: the struct is an argument of the launchers that cross the two passes of this file (hkinl, below)
struct KParams {
  float4* core;
  uint32_t* cache;
  double* stats;
  int32_t* queue;    // [5][n] env indices queued for the general tiers this tick, see Q_* below
  uint32_t* qctl;    // queue counters, see Q_* below
  unsigned long long* phaseClk;  // [2 tiers][4 phases] block-cycles spent per phase (diagnostics, hk_debug_phase_cycles)
  float* actBuf;     // [n,8] actions handed from k_fast to the general tiers
  uint32_t* trace;   // diagnostics (HK_LANE_TRACE=1): [n/32+8 warps][4] phase cycles, [n][2] per-env work record, [n/32+8 blocks][12] block stamps
  int64_t n;
  int64_t env_id_offset;
  Config cfg;
};
}  // namespace hkk
using hkk::KParams;
// This file is compiled TWICE (hockey_env_b200/build.py) and the two objects are linked into one library:
//   pass 1 (default)                         -- everything except the two kernels below; device helpers marked
//                                               HK_HD_NOINLINE stay functions (k_fast is 2.4x slower fully inlined);
//   pass 2 (-DHK_TU_INLINE -DHK_INLINE_ALL)  -- only k_general<1> and k_touch, with every helper inlined into the kernel;
//                                               built twice (HK_INL_NS / HK_GENERAL_BOUND): blocks of up to 384 threads at 168
//                                               registers, and blocks of up to 256 threads at up to 255 registers (-2.6 %)
//                                               (measured: general tier 0.462 -> 0.402 ms/tick at 65,536 envs, 2.61 ->
//                                               2.32 at 1,048,576; touch tier 1.01 -> 0.95; profiles/README.md r2n).
// Pass 1 reaches the kernels of pass 2 through these host functions; each pass has its own copy of the constant Scene.
#define HK_INL_DECLS                                                                                                              \
  cudaError_t setScene(const hk::Scene& S);                                                                                       \
  cudaError_t setMaxDynamicSmem(int bytes);                                                                                       \
  size_t staticSmemGeneral();                                                                                                     \
  void setCarveouts(int pctGeneral, int pctTouch);                                                                                \
  void launchGeneral1(unsigned grid, int block, size_t smem, cudaStream_t stream, const KParams& P, const hk::StepIO& io,         \
                      int unlimited, int lanesLog2, int firstClass, int phaseSync, int envWarps, int classWarps);                 \
  void launchTouch(unsigned grid, int block, cudaStream_t stream, const KParams& P, const hk::StepIO& io);
namespace hkinl { HK_INL_DECLS }     // pass 2:  k_general<1> bounded to 384 threads (168 registers), k_touch
namespace hkinl256 { HK_INL_DECLS }  // pass 2b: k_general<1> bounded to 256 threads (up to 255 registers): the blocks of batches <= 100k envs
#if !defined(HK_INL_NS)
#define HK_INL_NS hkinl
#endif
namespace {

constexpr int kSlowBlock = 384;  // one block per SM at 168 registers: all its warps walk the tick phases together
constexpr int kTouchBlock = 384; // threads per block of k_touch (pass 2): one block per SM at 166 registers

#if !defined(HK_TU_INLINE)
__global__ void __launch_bounds__(kBlock) k_create(KParams P) {
  __shared__ Scene S;
  stageScene(&S);
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  Env e;
  envCreate(S, P.cfg, e, (uint64_t)(P.env_id_offset + i));
  storeEnv(P.core, P.n, i, e);
}

__global__ void __launch_bounds__(kBlock) k_reset(KParams P, const uint8_t* mask, const int8_t* one_starting, const int64_t* seeds,
                                                  const uint8_t* modes, float* obs) {
  __shared__ Scene S;
  stageScene(&S);
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  if (mask && !mask[i]) return;
  Env e;
  loadEnv(P.core, P.n, i, e);
  envReset(S, P.cfg, e, (uint64_t)(P.env_id_offset + i), one_starting ? (int)one_starting[i] : -1, seeds ? seeds[i] : -1,
           modes ? (int)modes[i] : -1);
  storeEnv(P.core, P.n, i, e);
  if (obs) {
    float o[18];
    getObs(e, o);
    writeRow18(obs + 18 * i, o);
  }
}

__global__ void __launch_bounds__(kBlock) k_step(KParams P, StepIO io) {
  __shared__ Scene S;
  stageScene(&S);
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  TickStats st;
  tickStatsZero(st);
  if (i < P.n) {
    Env e;
    loadEnv(P.core, P.n, i, e);
    Cache cache;
    cache.base = P.cache + i;
    cache.stride = (size_t)P.n;
    envTick(S, P.cfg, cache, e, (uint64_t)(P.env_id_offset + i), (size_t)i, io, true, st);
    storeEnv(P.core, P.n, i, e);
  }
  flushStats(statsRow(P.stats), st);
}

#endif  // !HK_TU_INLINE
// ---- the per-tick pipeline: k_fast over all envs, then the general path over the queues (three-tier cascade) ----------------
// k_fast (tier 0) proves "nothing to solve" per env (hk_fast.cuh) and finishes those ticks with a small register
// footprint; every other env index is appended to the tier-1 queue (one atomic per warp).  The general path
// then runs on compacted queues, so lanes that iterate the contact solver sit next to each other instead of
// idling 30 neighbours (ncu, round 1: 1.6 active lanes per solver instruction in the monolithic kernel).
// queue layout: P.queue = [5][n] int32: rows 0-3 = tier-1 work classes (hk_fast.cuh bailClass), row 4 = tier 2.
// P.qctl = {count[0..3], tier-1 finished blocks, tier-2 count, tier-2 finished blocks, pad}.
enum { Q_CLASSES = 4, QC_DONE1 = 4, QC_COUNT2 = 5, QC_DONE2 = 6 };

// MINB = resident blocks per SM the register allocation aims at: 4 (120 registers, no spills) when the batch is one
// wave anyway, 5 (96 registers) when occupancy pays (measured: profiles/README.md r1e)
#if !defined(HK_TU_INLINE)
// BLOCK = 128: several independent blocks per SM (MINB of them).  BLOCK = kFastWide (batches of >= 16k envs): ONE block per
// SM whose warps walk the tick in three stages with block barriers in between (controllers | world step | epilogue).
// A large batch is many waves of blocks, so co-resident 128-thread blocks sit at unrelated places of a 140 KB kernel that
// has no loops to reuse and every block streams its own instructions from L2 (ncu, 1,048,576 envs: 18.6 cycles of
// no-instruction stall per issued instruction, 66 % of the kernel; 6.0 at 262,144; 1.7 at 65,536 where the single wave
// of blocks happens to run in step) -- with one wide block the fetched lines are shared by all the warps of the SM.
constexpr int kFastWide = 512;
template <int MINB, int BLOCK>
__global__ void __launch_bounds__(BLOCK, MINB) k_fast(KParams P, StepIO io) {
  constexpr bool kStaged = BLOCK > kBlock;
  __shared__ Scene S;
  __shared__ __align__(16) float sRows[BLOCK / 32][32 * 18];  // per warp: its 32 observation rows, staged for 128-bit stores
  stageScene(&S);
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool valid = i < P.n;
  TickStats st;
  tickStatsZero(st);
  bool ok = false, wroteFinal = false;
  int cls = 0;
  const bool stageRows = io.write != 0 && io.stageRows != 0;  // uniform
  float* const myRows = sRows[threadIdx.x >> 5];
  if (!kStaged) {
    if (valid) {
      Env e;
      loadEnv(P.core, P.n, i, e);
      e.bailKind = 15;
      ok = envTickFast(S, P.cfg, e, (uint64_t)(P.env_id_offset + i), (size_t)i, io, io.write != 0, st, stageRows ? &wroteFinal : nullptr);
      if (ok) {
        storeEnv(P.core, P.n, i, e);
        if (stageRows) getObs(e, myRows + 18 * (threadIdx.x & 31));
      } else {
        tickStatsZero(st);
        cls = bailClass(e.bailKind);
      }
    }
  } else {  // the same tick (hk_tick.cuh envTickFast), cut at its two call boundaries
    Env e;
    float a[8];
    int had1 = 0, had2 = 0;
    const uint64_t env_id = (uint64_t)(P.env_id_offset + i);
    if (valid) {
      loadEnv(P.core, P.n, i, e);
      e.bailKind = 15;
      policyActions(P.cfg, e, env_id, io.action ? io.action + (size_t)io.stride * i : nullptr, io.pol1, pol2Of(io, (size_t)i), a);
      had1 = e.has1;
      had2 = e.has2;
    }
    __syncthreads();
    if (valid) {
      ok = envStepFast(S, P.cfg, e, a);
      if (!ok && io.actBuf) {
        float4* ab = reinterpret_cast<float4*>(io.actBuf + 8 * i);
        ab[0] = make_float4(a[0], a[1], a[2], a[3]);
        ab[1] = make_float4(a[4], a[5], a[6], a[7]);
      }
    }
    __syncthreads();
    if (valid) {
      if (ok) {
        tickFinish(S, P.cfg, e, env_id, (size_t)i, io, io.write != 0, st, had1, had2, stageRows ? &wroteFinal : nullptr);
        storeEnv(P.core, P.n, i, e);
        if (stageRows) getObs(e, myRows + 18 * (threadIdx.x & 31));
      } else {
        cls = bailClass(e.bailKind);
      }
    }
  }
  if (stageRows) {  // the warp's envs are consecutive: write its finished rows front to back, 16 bytes per lane
    __syncwarp();
    const int64_t i0 = i - (threadIdx.x & 31);
    const unsigned okMask = __ballot_sync(0xffffffffu, ok), finMask = __ballot_sync(0xffffffffu, ok && !wroteFinal);
    if (okMask) warpStoreRows18(io.obs + 18 * i0, myRows, okMask);
    if (io.final_obs && finMask) warpStoreRows18(io.final_obs + 18 * i0, myRows, finMask);
  }
  const bool need = valid && !ok;
  const int lane = threadIdx.x & 31;
  if (__any_sync(0xffffffffu, need)) {
#pragma unroll
    for (int c = 0; c < Q_CLASSES; ++c) {
      const unsigned m = __ballot_sync(0xffffffffu, need && cls == c);
      if (m) {
        unsigned base = 0;
        if (lane == 0) base = atomicAdd(&P.qctl[c], (unsigned)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (need && cls == c) P.queue[(int64_t)c * P.n + base + __popc(m & ((1u << lane) - 1u))] = (int32_t)i;
      }
    }
  }
  flushStats(statsRow(P.stats), st);
}

#endif  // !HK_TU_INLINE
#if defined(HK_TU_INLINE)  // pass 2 only (see hkinl above)
// Touch tier: work class 0 of k_fast's queue (puck x racket contact ticks, i.e. every keep/shoot tick).  One contact,
// one manifold point, no continuous-collision event possible -- the lanes of a warp all walk the same short path
// (hk_fast.cuh worldStepTouch).  Envs whose proofs fail are appended to work class 3 for the general tier.
// One 384-thread block per SM (166 registers), staged like the wide k_fast: actions + Collide | island solve | proofs + epilogue.
__global__ void __launch_bounds__(kTouchBlock, 1) k_touch(KParams P, StepIO io) {
  __shared__ Scene S;
  stageScene(&S);
  const int lane = threadIdx.x & 31;
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const unsigned cnt = *((volatile uint32_t*)&P.qctl[0]);
  if ((int64_t)blockIdx.x * blockDim.x >= (int64_t)cnt) return;  // block-uniform
  const bool valid = j < (int64_t)cnt;
  TickStats st;
  tickStatsZero(st);
  Env e;
  Cache cache;
  float a[8];
  int had1 = 0, had2 = 0;
  int64_t i = 0;
  bool live = false;
  const float h = (float)(1.0 / HK_FPS);
  if (valid) {  // hk_tick.cuh envTickTouch / hk_fast.cuh envStepTouch, cut at their call boundaries
    i = P.queue[j];
    loadEnv(P.core, P.n, i, e);
    cache.base = P.cache + i;
    cache.stride = (size_t)P.n;
    const float4* ab = reinterpret_cast<const float4*>(io.actBuf + 8 * i);
    float4 lo = ab[0], hi = ab[1];
    a[0] = lo.x; a[1] = lo.y; a[2] = lo.z; a[3] = lo.w; a[4] = hi.x; a[5] = hi.y; a[6] = hi.z; a[7] = hi.w;
    e.bailKind = 15;
    policyAdvancePhases(P.cfg, e, (uint64_t)(P.env_id_offset + i), io.pol1, pol2Of(io, (size_t)i));
    had1 = e.has1;
    had2 = e.has2;
    envStepActions(S, P.cfg, e, a);
    e.sweepBudget = 1 << 20;
    e.allowToiEvents = true;
    e.aborted = false;
    live = worldStepTouchCollide(S, P.cfg, cache, e);
  }
  __syncthreads();
  if (live) live = worldStepTouchSolve(S, P.cfg, cache, e, h);
  __syncthreads();
  if (live) live = worldStepTouchFinish(S, cache, e);
  if (live) {
    envStepAfterWorld(e);
    tickFinish(S, P.cfg, e, (uint64_t)(P.env_id_offset + i), (size_t)i, io, io.write != 0, st, had1, had2);
    storeEnv(P.core, P.n, i, e);
  }
  const bool need = valid && !live;
  const unsigned m = __ballot_sync(0xffffffffu, need);
  if (m) {
    unsigned base = 0;
    if (lane == 0) base = atomicAdd(&P.qctl[Q_CLASSES - 1], (unsigned)__popc(m));
    base = __shfl_sync(0xffffffffu, base, 0);
    if (need) P.queue[(int64_t)(Q_CLASSES - 1) * P.n + base + __popc(m & ((1u << lane) - 1u))] = (int32_t)i;
  }
  flushStats(statsRow(P.stats), st);
}
#endif  // HK_TU_INLINE
// The general tier(s) run the same general path (generalTick below) over the class-sorted queue of k_fast:
//   k_general<1>, unlimited = 1 (the default, HK_TIERS=2): every queued env finishes its tick here.
//   k_general<1>, unlimited = 0 + k_general<2> (HK_TIERS=3; built and parity-tested, not the default at any batch size):
//                      tier 1 is budgeted -- a velocity solve must converge (fixed point / short cycle) within kMidSweeps
//                      sweeps and no continuous-collision EVENT may occur; otherwise the env is appended to the tier-2
//                      queue with nothing committed, and k_general<2> redoes its tick without limits, packed densely.
//   Every work class starts on a warp boundary, so the 32 lanes of a warp do the same kind of tick.
constexpr int kMidSweeps = 24;
// Velocity solves of a block are pooled in shared memory (phase 2 of k_general) and dealt to its warps as units of one
// loop shape each: a warp never runs two different 180-sweep loops one after the other unless the block holds more
// units than warps, and the lanes of a unit all execute the same register-resident loop.
struct SolveTask {   // multi-contact solve with a fixed-shape loop (solveKind 1..8)
  VC vcs[3];
  VelTriple v;
  int result, sweeps, kind;
};
struct Solve2Task {  // one contact, two manifold points
  VC vc;
  Vel A, B;
  int result, sweeps;
};
struct Solve1Task {  // one contact, one manifold point (95 % of the solves)
  VC1 vc;
  Vel A, B;
  int result, sweeps;
};
// Shared memory is taken out of L1, and the general path keeps its per-thread state (several KB) in local memory, i.e.
// in L1 (measured: profiles/README.md, carve-out sweep), so the pools are compact: one slot array for all multi-contact
// shapes (tagged with their kind), a small one for the two-point solves, 96 B per env lane for the one-point solves.
constexpr int kMultiSlots = 24;     // multi-contact tasks per block (<= 32: a warp finds its shape's tasks with one ballot); the rest is solved in place
constexpr int kTasksPerLane = 3;    // first-pass TOI evaluations a lane may file (phase 3)
constexpr size_t kRawMulti = sizeof(SolveTask) * kMultiSlots;
__host__ __device__ constexpr int twoPointSlots(int envLanes) { return envLanes / 8 < 16 ? 16 : envLanes / 8; }
__host__ __device__ constexpr size_t rawBytes(int envLanes) {  // dynamic shared memory of k_general for envLanes env lanes
  const size_t solve = kRawMulti + sizeof(Solve2Task) * (size_t)twoPointSlots(envLanes) + sizeof(Solve1Task) * (size_t)envLanes;
  const size_t toi = (sizeof(ToiTask) + sizeof(float)) * (size_t)envLanes * kTasksPerLane;
  return solve > toi ? solve : toi;
}
struct GenStamps {  // diagnostics: clock stamps of the phase boundaries of one general tick
  long long tc0, tc1, tc2, tc3, stampB, stampV, stampT, tf0, tfCommit, tfFinish, tfStore, tfFlush;
};
// Clock stamp AFTER a block barrier has completed.  BAR.SYNC.DEFER_BLOCKING does not hold the warp at the barrier
// instruction: the next CS2R issues at once and the warp only blocks at its next memory instruction (measured on B200,
// scripts/probes/bar_clock_probe.cu: a clock read right after __syncthreads() is 2 cycles after the one before it while
// the other warp is still 100k cycles away).  So the stamp is taken behind a shared-memory load whose value it needs.
__device__ __forceinline__ long long clockAfterBarrier(const Scene& S) {
  const unsigned v = *reinterpret_cast<const volatile unsigned*>(&S.puckRadius);
  long long t = 0;
  if (v != 0xFFFFFFFFu) t = clock64();  // never equal (a float radius): the branch only ties the stamp to the load
  return t;
}
// barrier among the threads that walk a general tick together: the whole block (k_general), or the general team of the
// fused rollout kernel (its first `nthr` threads; the other warps of that block run fast ticks meanwhile)
template <bool TEAM>
__device__ __forceinline__ void teamSync(int nthr) {
  if (TEAM) asm volatile("bar.sync 2, %0;" ::"r"(nthr) : "memory");
  else __syncthreads();
}
// One general tick for up to `envWarps` warps of envs (lane = env: `valid`, state index `i`, work class `cls`), walked
// phase by phase by `nthr` threads (threads 0 .. nthr-1 of the block, all of which must call this).
template <int TIER, bool TEAM>
__device__ __forceinline__ void generalTick(const KParams& P, const StepIO& io, const Scene& S, unsigned char* sRaw, const bool valid,
                                            const int64_t i, const int cls, const bool envWarp, const int64_t gw, const int unlimited,
                                            const int phaseSync, const int envWarps, const int nthr, const bool laneWrite,
                                            TickStats& st, bool& need, GenStamps& gs, unsigned long long* sSlowUnitP, unsigned* sFin) {
  const int envLanes = envWarps << 5;
  tickStatsZero(st);
  need = false;
  const int lane = threadIdx.x & 31;
  const int wib = threadIdx.x >> 5;
  // ---- the tick, phase by phase for the whole block (same code region at the same time on this SM) ----
  Env e;
  Cache cache;
  cache.base = P.cache + i;
  cache.stride = (size_t)P.n;
  int had1 = 0, had2 = 0;
  const uint64_t env_id = (uint64_t)(P.env_id_offset + i);
  const float dt = (float)(1.0 / HK_FPS);
  long long& tc0 = gs.tc0; tc0 = clock64();
  if (valid) {  // phase 1: policy, forces, keep/shoot, Collide
    loadEnv(P.core, P.n, i, e);
    float a[8];
    if (io.actBuf) {  // k_fast already ran the controllers for this tick
      const float4* ab = reinterpret_cast<const float4*>(io.actBuf + 8 * i);
      float4 lo = ab[0], hi = ab[1];
      a[0] = lo.x; a[1] = lo.y; a[2] = lo.z; a[3] = lo.w; a[4] = hi.x; a[5] = hi.y; a[6] = hi.z; a[7] = hi.w;
      policyAdvancePhases(P.cfg, e, env_id, io.pol1, pol2Of(io, (size_t)i));
    } else {
      policyActions(P.cfg, e, env_id, io.action ? io.action + (size_t)io.stride * i : nullptr, io.pol1, pol2Of(io, (size_t)i), a);
    }
    had1 = e.has1;
    had2 = e.has2;
    e.sweepBudget = (TIER == 1 && !unlimited) ? kMidSweeps : (1 << 20);
    e.allowToiEvents = TIER != 1 || unlimited;
    e.aborted = false;
    envStepActions(S, P.cfg, e, a);
    worldStepCollide(S, P.cfg, cache, e);
  }
  const long long tw1 = clock64();
  // phaseSync bit 0/1/2: block-wide barrier after Collide / after the island solve / after SolveTOI.  They keep the
  // warps of an SM in the same code region (shared instruction fetch); they are not needed for correctness.
  if (phaseSync & 1) teamSync<TEAM>(nthr);
  long long& tc1 = gs.tc1; tc1 = clockAfterBarrier(S);
  // ---- phase 2: island solve.  The velocity iterations of the whole block are pooled (see SolveTask): every lane files
  // its solve by loop shape, the warps of the block (helpers included) take one unit of one shape at a time.
  IslandCtx ctx;
  ctx.nvc = 0;
  long long &stampB = gs.stampB, &stampV = gs.stampV, &stampT = gs.stampT;  // diagnostics: block-level stamps inside phases 2 and 3
  stampB = stampV = stampT = 0;
  if (valid) solveIslandsBegin(S, cache, e, dt, ctx);
  {
    SolveTask* mtasks = reinterpret_cast<SolveTask*>(sRaw);
    Solve2Task* s2tasks = reinterpret_cast<Solve2Task*>(sRaw + kRawMulti);
    const int cap2 = twoPointSlots(envLanes);
    Solve1Task* s1tasks = reinterpret_cast<Solve1Task*>(sRaw + kRawMulti + sizeof(Solve2Task) * (size_t)cap2);
    // counts: multi kinds 1..8, one contact x 1 point, one contact x 2 points, all multi-contact slots handed out
    __shared__ int sKindCount[HK_MULTI_KINDS + 3];
    __shared__ unsigned short sList[2][kSlowBlock];  // one-point tasks still unfinished after a round (double buffer)
    __shared__ int sRound[5];                        // their count per round
    if (threadIdx.x < HK_MULTI_KINDS + 3) sKindCount[threadIdx.x] = 0;
    if (threadIdx.x < 5) sRound[threadIdx.x] = 0;
    if (threadIdx.x == 0) *sSlowUnitP = 0;
    teamSync<TEAM>(nthr);
    stampB = clockAfterBarrier(S);
    const int nwarps = nthr >> 5;
    const int budget = (TIER == 1 && !unlimited) ? kMidSweeps : (1 << 20);
    const bool pool1 = (phaseSync & 8) != 0;  // also pool the single-contact solves
    int kind = 0, slot = 0;  // kind 1..HK_MULTI_KINDS: multi; then single contact, 1 point; single contact, 2 points
    if (valid && ctx.nvc >= 2) {
      kind = solveKind(ctx.vcs, ctx.nvc);
      if (kind) {
        slot = atomicAdd(&sKindCount[HK_MULTI_KINDS + 2], 1);
        if (slot >= kMultiSlots) kind = 0;  // no room: solved in place
        else atomicAdd(&sKindCount[kind - 1], 1);
      }
    } else if (valid && ctx.nvc == 1 && pool1) {
      kind = HK_MULTI_KINDS + ctx.vcs[0].count;
      slot = atomicAdd(&sKindCount[kind - 1], 1);
      if (kind == HK_MULTI_KINDS + 2 && slot >= cap2) kind = 0;
    }
    if (kind == HK_MULTI_KINDS + 1) {
      Solve1Task& t = s1tasks[slot];
      t.vc = vc1Of(ctx.vcs[0]);
      t.A = loadVel(e, ctx.vcs[0].bA);
      t.B = loadVel(e, ctx.vcs[0].bB);
    } else if (kind == HK_MULTI_KINDS + 2) {
      Solve2Task& t = s2tasks[slot];
      t.vc = ctx.vcs[0];
      t.A = loadVel(e, ctx.vcs[0].bA);
      t.B = loadVel(e, ctx.vcs[0].bB);
    } else if (kind) {
      SolveTask& t = mtasks[slot];
      t.kind = kind;
      for (int k = 0; k < ctx.nvc; ++k) t.vcs[k] = ctx.vcs[k];
      t.v.b0 = loadVel(e, 0);
      t.v.b1 = loadVel(e, 1);
      t.v.b2 = loadVel(e, 2);
    }
    teamSync<TEAM>(nthr);
    {
      // unit list, identical in every warp: the multi-contact shapes that have tasks (heaviest loops first), then the
      // 2-point chunks, then the 1-point chunks; spare warps split the 1-point tasks into smaller chunks
      const int n1 = sKindCount[HK_MULTI_KINDS], n2 = min(sKindCount[HK_MULTI_KINDS + 1], cap2);
      const int nMulti = min(sKindCount[HK_MULTI_KINDS + 2], kMultiSlots);
      int nm = 0, mk_[HK_MULTI_KINDS];
#pragma unroll
      for (int q = 0; q < HK_MULTI_KINDS; ++q) {
        const int k = q == 0 ? 4 : (q == 1 ? 6 : (q == 2 ? 7 : (q == 3 ? 8 : (q == 4 ? 2 : (q == 5 ? 3 : (q == 6 ? 5 : 1))))));
        if (sKindCount[k - 1] > 0) mk_[nm++] = k;
      }
      const int c2 = (n2 + 31) >> 5;
      int c1 = (n1 + 31) >> 5;
      const int spare = nwarps - nm - c2;
      if (spare > c1) c1 = min(spare, (n1 + 3) >> 2);
      const int units = (phaseSync & 16) ? nm + c2 : nm + c2 + c1;
      // Re-packed one-point rounds (phaseSync bit 4): 92 % of the one-point solves end within ~30 sweeps, 8 % creep to
      // 180, so a chunk's lanes mostly idle behind its slowest one.  The warps that hold no multi-contact / two-point
      // unit run the one-point tasks in rounds of sweeps [0,12) [12,24) [24,48) [48,180) and re-pack the unfinished
      // tasks densely between rounds (exact: see runVelocityIterations1Range); they meet at a named barrier of their
      // own while the other warps work through the heavy units.
      const int wHeavy = !(phaseSync & 16) || units == 0 || nwarps == 1 ? 0 : min(units, max(1, nwarps / 2));
      const int uStride = (phaseSync & 16) ? max(wHeavy, 1) : nwarps;
      const bool heavyWarp = !(phaseSync & 16) || wib < wHeavy || nwarps == 1;
      // first round: unit w -> warp w; further rounds run backwards (the first warps hold the heavy multi-contact loops)
      for (int r = 0, u = wib; heavyWarp && u < units; ++r, u = r * uStride + ((r & 1) ? uStride - 1 - wib : wib)) {
        const long long tu0 = P.trace ? clock64() : 0;
        int utype = 10;  // diagnostics: 1..8 multi-contact shape, 9 two-point chunk, 10 one-point chunk, 11 in place
        if (u < nm) {
          utype = mk_[u];
          const int k = mk_[u];
          // this shape's tasks among the block's multi-contact slots: lane l takes the l-th of them
          const unsigned mine = __ballot_sync(0xffffffffu, lane < nMulti && mtasks[lane < nMulti ? lane : 0].kind == k);
          if (lane < __popc(mine)) {
            SolveTask& t = mtasks[__fns(mine, 0, lane + 1)];
            VelTriple v = t.v;
            int sweeps = 0;
            t.result = runVelocityIterationsKind(k, t.vcs, v, budget, 6 * 30, &sweeps);
            t.v = v;
            t.sweeps = sweeps;
          }
        } else if (u < nm + c2) {
          const int j = ((u - nm) << 5) + lane;
          if (j < n2) {
            Solve2Task& t = s2tasks[j];
            Vel A = t.A, B = t.B;
            int sweeps = 0;
            t.result = runVelocityIterations2Core(t.vc, A, B, budget, 6 * 30, &sweeps);
            t.A = A;
            t.B = B;
            t.sweeps = sweeps;
          }
        } else {
          const int c = u - nm - c2;
          const int lo = (int)(((long long)n1 * c) / c1), hi = (int)(((long long)n1 * (c + 1)) / c1);
          const int j = lo + lane;
          if (j < hi) {
            Solve1Task& t = s1tasks[j];
            Vel A = t.A, B = t.B;
            int sweeps = 0;
            t.result = runVelocityIterations1Core(t.vc, A, B, budget, 6 * 30, &sweeps);
            t.A = A;
            t.B = B;
            t.sweeps = sweeps;
          }
        }
        if (u >= nm && u < nm + c2) utype = 9;
        if (P.trace && lane == 0) atomicMax(sSlowUnitP, ((unsigned long long)(clock64() - tu0) << 8) | (unsigned)utype);
      }
      if ((phaseSync & 16) && wib >= wHeavy) {
        const long long tu0 = P.trace ? clock64() : 0;
        const int w1 = nwarps - wHeavy, myw = wib - wHeavy;
        int nA = n1, it0 = 0;
        for (int r = 0; r < 4 && nA > 0; ++r) {
          const int stop = r == 0 ? 12 : (r == 1 ? 24 : (r == 2 ? 48 : 6 * 30));
          const int chunks = (nA + 31) >> 5;
          for (int ch = myw; ch < chunks; ch += w1) {
            const int j = (ch << 5) + lane;
            if (j < nA) {
              const int idx = r == 0 ? j : (int)sList[r & 1][j];
              Solve1Task& t = s1tasks[idx];
              Vel A = t.A, B = t.B;
              int sweeps = 0;
              const int res = runVelocityIterations1Range(t.vc, A, B, budget, 6 * 30, it0, stop, &sweeps);
              t.A = A;
              t.B = B;
              if (res == HK_SOLVE_UNFINISHED) {
                sList[(r + 1) & 1][atomicAdd(&sRound[r + 1], 1)] = (unsigned short)idx;
              } else {
                t.result = res;
                t.sweeps = it0 + sweeps;
              }
            }
          }
          asm volatile("bar.sync 1, %0;" ::"r"(w1 * 32) : "memory");  // the one-point warps only
          nA = sRound[r + 1];
          it0 = stop;
        }
        if (P.trace && lane == 0) atomicMax(sSlowUnitP, ((unsigned long long)(clock64() - tu0) << 8) | 10u);
      }
    }
    int itc = 0;
    {
      const long long tu0 = P.trace ? clock64() : 0;
      const bool inPlace = valid && ctx.nvc > 0 && !kind;
      if (inPlace) itc = runVelocityIterations(e, ctx.vcs, ctx.nvc, 6 * 30);
      if (P.trace && __any_sync(0xffffffffu, inPlace) && lane == 0) atomicMax(sSlowUnitP, ((unsigned long long)(clock64() - tu0) << 8) | 11u);
    }
    teamSync<TEAM>(nthr);
    stampV = clockAfterBarrier(S);
    if (kind == HK_MULTI_KINDS + 1) {
      const Solve1Task& t = s1tasks[slot];
      ctx.vcs[0].pt[0].ni = t.vc.ni;
      ctx.vcs[0].pt[0].ti = t.vc.ti;
      storeVel(e, ctx.vcs[0].bA, t.A);
      storeVel(e, ctx.vcs[0].bB, t.B);
      e.nVelIters += (uint32_t)t.sweeps;
      itc = t.result;
    } else if (kind == HK_MULTI_KINDS + 2) {
      const Solve2Task& t = s2tasks[slot];
      ctx.vcs[0].pt[0].ni = t.vc.pt[0].ni;
      ctx.vcs[0].pt[0].ti = t.vc.pt[0].ti;
      ctx.vcs[0].pt[1].ni = t.vc.pt[1].ni;
      ctx.vcs[0].pt[1].ti = t.vc.pt[1].ti;
      storeVel(e, ctx.vcs[0].bA, t.A);
      storeVel(e, ctx.vcs[0].bB, t.B);
      e.nVelIters += (uint32_t)t.sweeps;
      itc = t.result;
    } else if (kind) {
      const SolveTask& t = mtasks[slot];
      for (int k = 0; k < ctx.nvc; ++k) {
        ctx.vcs[k].pt[0].ni = t.vcs[k].pt[0].ni;
        ctx.vcs[k].pt[0].ti = t.vcs[k].pt[0].ti;
        if (ctx.vcs[k].count == 2) {
          ctx.vcs[k].pt[1].ni = t.vcs[k].pt[1].ni;
          ctx.vcs[k].pt[1].ti = t.vcs[k].pt[1].ti;
        }
      }
      storeVel(e, 0, t.v.b0);
      storeVel(e, 1, t.v.b1);
      storeVel(e, 2, t.v.b2);
      e.nVelIters += (uint32_t)t.sweeps;
      itc = t.result;
    }
    if (valid) solveIslandsEnd(S, e, dt, 2 * 30, ctx, itc);
  }
  const long long tw2 = clock64();
  if (phaseSync & 2) teamSync<TEAM>(nthr);
  long long& tc2 = gs.tc2; tc2 = clockAfterBarrier(S);
  // phase 3a-3c: first-pass TOI evaluations of the whole block as one task list, one task per thread
  const bool wantToi = valid && !e.aborted && (e.exist & HK_PAIRS_TOI);
  {
    ToiTask* sTasks = reinterpret_cast<ToiTask*>(sRaw);  // worst case: every lane files all its tasks
    float* sAlpha = reinterpret_cast<float*>(sRaw + sizeof(ToiTask) * (size_t)envLanes * kTasksPerLane);
    __shared__ int sCount;
    if (threadIdx.x == 0) sCount = 0;
    teamSync<TEAM>(nthr);
    ToiTask mine[kTasksPerLane];
    int nMine = 0, base = 0;
    if (wantToi) {
      nMine = toiCollect(S, e, mine, kTasksPerLane);
      if (nMine > 0) {
        base = atomicAdd(&sCount, nMine);
        for (int k = 0; k < nMine; ++k) sTasks[base + k] = mine[k];
      }
    }
    teamSync<TEAM>(nthr);
    const int total = sCount;
    // tasks are dealt round-robin to the warps of the block (lane l of warp w takes task l * nwarps + w): the lanes
    // of a warp diverge inside b2TimeOfImpact, so a warp's time grows with the number of tasks it holds
    const int nwarps = nthr >> 5;
    for (int t = lane * nwarps + (threadIdx.x >> 5); t < total; t += nthr) sAlpha[t] = toiTaskRun(S, sTasks[t]);
    teamSync<TEAM>(nthr);
    stampT = clockAfterBarrier(S);
    for (int k = 0; k < nMine; ++k) {
      e.toiPre[mine[k].pid] = sAlpha[base + k];
      e.toiPreFlag |= 1u << mine[k].pid;
    }
  }
  const long long tw3a = clock64();
  if (wantToi) solveTOI(S, P.cfg, cache, e, dt, 6 * 30);  // phase 3d: events (rare) on top of the pre-seeded results
  const long long tw3 = clock64();
  if (P.trace && TIER == 1 && envWarp && lane == 0 && gw < P.n / 32 + 8) {
    uint32_t* w = P.trace + 4 * (size_t)gw;
    w[0] = (uint32_t)(tw1 - tc0);
    w[1] = (uint32_t)(tw2 - tc1);
    w[2] = (uint32_t)(tw3a - tc2);
    w[3] = (uint32_t)(tw3 - tw3a);
  }
  if (phaseSync & 4) teamSync<TEAM>(nthr);
  long long& tc3 = gs.tc3; tc3 = clockAfterBarrier(S);
  if (P.trace && (phaseSync & 4)) {  // diagnostics (HK_LANE_TRACE=1): block-wide max of per-lane TOI evaluation / event cycles
    __shared__ unsigned long long sMaxEval, sMaxEvent;
    if (threadIdx.x == 0) { sMaxEval = 0; sMaxEvent = 0; }
    teamSync<TEAM>(nthr);
    if (valid) {
      atomicMax(&sMaxEval, (unsigned long long)e.dbgEvalClk);
      atomicMax(&sMaxEvent, (unsigned long long)e.dbgEventClk);
    }
    teamSync<TEAM>(nthr);
    if (threadIdx.x == 0 && TIER == 1) {
      atomicAdd(&P.phaseClk[4], sMaxEval);
      atomicAdd(&P.phaseClk[5], sMaxEvent);
    }
  }
  if (P.trace && TIER == 1 && valid) {
    uint32_t* rec = P.trace + 4 * ((size_t)P.n / 32 + 8) + 2 * (size_t)i;
    rec[0] = (e.nVelIters & 0xFFFu) | ((e.nToiEvents & 0xFu) << 12) | ((uint32_t)(cls & 0xF) << 16) | ((e.dbgShape & 0xFFu) << 20) |
             (e.aborted ? 0x80000000u : 0u);
    rec[1] = (uint32_t)gw;
  }
  if (P.trace) {
    if (threadIdx.x < 4) sFin[threadIdx.x] = 0;
    teamSync<TEAM>(nthr);
  }
  if (io.waitFlag) {  // hk_step_host: this tick's rows of the fast tier are being copied into the host record the outputs go to
    if (threadIdx.x == 0)
      while (*((volatile const uint32_t*)io.waitFlag) != io.waitValue) __nanosleep(200);
    teamSync<TEAM>(nthr);
  }
  const long long tf0 = clockAfterBarrier(S);
  long long tf1 = tf0, tf2 = tf0;
  gs.tf0 = tf0;
  if (valid) {  // phase 4: commit, rewards, outputs, auto-reset, store
    if (!e.aborted) {
      worldStepFinish(cache, e);
      envStepAfterWorld(e);
      tf1 = clock64();
      if (P.trace && e.done) atomicAdd(&sFin[3], 1u);
      tickFinish(S, P.cfg, e, env_id, (size_t)i, io, laneWrite, st, had1, had2);
      tf2 = clock64();
      storeEnv(P.core, P.n, i, e);
    } else {
      need = true;
    }
  }
  __syncwarp();
  gs.tfCommit = tf1;
  gs.tfFinish = tf2;
  gs.tfStore = clock64();
  if (__any_sync(0xffffffffu, valid)) {
    if (TIER == 1 && !TEAM) {
      const unsigned m = __ballot_sync(0xffffffffu, need);
      if (m) {
        unsigned base = 0;
        if (lane == 0) base = atomicAdd(&P.qctl[QC_COUNT2], (unsigned)__popc(m));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (need) P.queue[(int64_t)Q_CLASSES * P.n + base + __popc(m & ((1u << lane) - 1u))] = (int32_t)i;
      }
    }
    flushInt(statsRow(P.stats), 14, st.steps, lane);  // env-ticks completed by the general tiers (units of work per launch)
    flushStats(statsRow(P.stats), st);
  }
  gs.tfFlush = clock64();
  if (P.trace && valid) {
    atomicMax(&sFin[0], (unsigned)(tf1 - tf0));
    atomicMax(&sFin[1], (unsigned)(tf2 - tf1));
    atomicMax(&sFin[2], (unsigned)(clock64() - tf2));
  }
}

template <int TIER>
#if !defined(HK_GENERAL_BOUND)
#define HK_GENERAL_BOUND kSlowBlock  // A/B switch: 256 lets ptxas use up to 255 registers (only valid for blocks <= 256 threads)
#endif
__global__ void __launch_bounds__(HK_GENERAL_BOUND, 1) k_general(KParams P, StepIO io, int unlimited, int lanesLog2, int firstClass, int phaseSync, int envWarps, int classWarps) {
  __shared__ Scene S;
  extern __shared__ __align__(16) unsigned char sRaw[];  // phase 2: solve tasks; phase 3: TOI tasks + results (rawBytes())
  stageScene(&S);
  const int lane = threadIdx.x & 31;
  // Up to envWarps warps of a block carry envs (fewer in the blocks of the TOI-heavy work classes, see below); the
  // others are helpers that only take part in the pooled phases (velocity solves, TOI evaluations).
  const int wib = threadIdx.x >> 5;
  bool envWarp = wib < envWarps;
  int64_t gw = (int64_t)blockIdx.x * envWarps + wib;  // global env-warp index (env warps only)
  const int envLanes = envWarps << 5;
  // Only the first 2^l lanes of an env warp carry an env; lanesLog2 packs l for the four work classes, 3 bits each
  // (tier 2: class 0's value).  Measured: full warps everywhere except 100k..200k envs (profiles/README.md).
  int cls = 0;
  bool valid = false;
  int64_t i = 0;
  if (TIER == 1 && classWarps) {
    // Class-homogeneous blocks.  A block waits for its slowest warp in every phase and the ticks of classes 1-3 (TOI
    // events) are about twice as long as those of class 0 (puck x racket), so a class-0 block carries twice the env
    // warps of the others.  classWarps > 0: env warps per block and class, 4 bits each (HK_CLASS_WARPS).
    // classWarps < 0: automatic -- the smallest b (class 0: 2b warps, others: b) for which the tick fits into
    // -classWarps blocks, i.e. one block per SM in a single wave; batches beyond that use full blocks.
    unsigned cnt[Q_CLASSES];
    int64_t nw[Q_CLASSES];
#pragma unroll
    for (int c = 0; c < Q_CLASSES; ++c) {
      cnt[c] = c < firstClass ? 0u : *((volatile uint32_t*)&P.qctl[c]);
      const int ll = (lanesLog2 >> (3 * c)) & 7;
      nw[c] = ((int64_t)cnt[c] + (1 << ll) - 1) >> ll;
    }
    int packed = classWarps;
    if (classWarps < 0) {
      const int maxW = envWarps, target = -classWarps;
      int b = 1;
      for (; b < maxW; ++b) {
        const int w0_ = min(2 * b, maxW);
        int64_t blocks = (nw[0] + w0_ - 1) / w0_;
#pragma unroll
        for (int c = 1; c < Q_CLASSES; ++c) blocks += (nw[c] + b - 1) / b;
        if (blocks <= target) break;
      }
      packed = min(2 * b, maxW) | (b << 4) | (b << 8) | (b << 12);
    }
    int64_t w0 = 0, b0 = 0;
    envWarp = false;
#pragma unroll
    for (int c = 0; c < Q_CLASSES; ++c) {
      const int ll = (lanesLog2 >> (3 * c)) & 7, lanes = 1 << ll;
      const int wpb = (packed >> (4 * c)) & 15;
      const int64_t nb = (nw[c] + wpb - 1) / wpb;
      if (!valid && (int64_t)blockIdx.x >= b0 && (int64_t)blockIdx.x < b0 + nb && wib < wpb) {
        const int64_t w = ((int64_t)blockIdx.x - b0) * wpb + wib;
        if (w < nw[c]) {
          envWarp = true;
          gw = w0 + w;
          const int64_t j = (w << ll) + lane;
          if (lane < lanes && j < (int64_t)cnt[c]) {
            valid = true;
            cls = c;
            i = P.queue[(int64_t)c * P.n + j];
          }
        }
      }
      w0 += nw[c];
      b0 += nb;
    }
  } else if (TIER == 1) {
    int64_t w0 = 0;
#pragma unroll
    for (int c = 0; c < Q_CLASSES; ++c) {
      const unsigned cnt = c < firstClass ? 0u : *((volatile uint32_t*)&P.qctl[c]);  // class 0 was k_touch's
      const int ll = (lanesLog2 >> (3 * c)) & 7, lanes = 1 << ll;
      const int64_t nw = ((int64_t)cnt + lanes - 1) >> ll;
      if (envWarp && !valid && gw >= w0 && gw < w0 + nw && lane < lanes) {
        const int64_t j = ((gw - w0) << ll) + lane;
        if (j < (int64_t)cnt) {
          valid = true;
          cls = c;
          i = P.queue[(int64_t)c * P.n + j];
        }
      }
      w0 += nw;
    }
  } else {
    const unsigned cnt = *((volatile uint32_t*)&P.qctl[QC_COUNT2]);
    const int ll = lanesLog2 & 7, lanes = 1 << ll;
    const int64_t j = (gw << ll) + lane;
    if (envWarp && lane < lanes && j < (int64_t)cnt) {
      valid = true;
      i = P.queue[(int64_t)Q_CLASSES * P.n + j];
    }
  }
  TickStats st;
  bool need = false;
  GenStamps gs;
  __shared__ unsigned long long sSlowUnit;  // diagnostics: (cycles << 8 | type) of the slowest pooled solve unit
  __shared__ unsigned sFin[4];              // diagnostics: block max of per-warp cycles in commit / tickFinish / store+flush, done lanes
  generalTick<TIER, false>(P, io, S, sRaw, valid, i, cls, envWarp, gw, unlimited, phaseSync, envWarps, (int)blockDim.x, io.write != 0, st,
                           need, gs, &sSlowUnit, sFin);
  const long long tc0 = gs.tc0, tc1 = gs.tc1, tc2 = gs.tc2, tc3 = gs.tc3, stampB = gs.stampB, stampV = gs.stampV, stampT = gs.stampT;

  // the last block to finish re-arms this tier's queue(s) for the next tick
  __syncthreads();
  if (threadIdx.x == 0) {
    if (__any_sync(1u, valid) || true) {
      long long tc4 = clockAfterBarrier(S);
      if (P.trace && TIER == 1 && blockIdx.x < P.n / 32 + 8) {
        uint32_t* w = P.trace + 4 * ((size_t)P.n / 32 + 8) + 2 * (size_t)P.n + 16 * (size_t)blockIdx.x;
        w[0] = (uint32_t)(tc1 - tc0);       // policy + Collide
        w[1] = (uint32_t)(stampB - tc1);    // solveIslandsBegin
        w[2] = (uint32_t)(stampV - stampB); // pooled velocity iterations
        w[3] = (uint32_t)(tc2 - stampV);    // solveIslandsEnd
        w[4] = (uint32_t)(stampT - tc2);    // TOI collect + first-pass evaluations
        w[5] = (uint32_t)(tc3 - stampT);    // TOI events
        w[6] = (uint32_t)(tc4 - tc3);       // finish
        unsigned sm;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(sm));
        w[7] = sm;
        unsigned long long gt;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(gt));
        w[8] = (uint32_t)gt;                // end time (ns, low word)
        w[9] = (uint32_t)(tc4 - tc0);
        w[10] = (uint32_t)(sSlowUnit >> 8);
        w[11] = (uint32_t)(sSlowUnit & 0xFF);
        w[12] = sFin[0];
        w[13] = sFin[1];
        w[14] = sFin[2];
        w[15] = sFin[3];
      }
      if (!P.trace && TIER == 1) {  // finish-phase split as warp 0 saw it: tc3->start, commit, tickFinish, store | flush, final barrier
        atomicAdd(&P.phaseClk[8], (unsigned long long)(gs.tf0 - tc3));
        atomicAdd(&P.phaseClk[9], (unsigned long long)(gs.tfCommit - gs.tf0));
        atomicAdd(&P.phaseClk[10], (unsigned long long)(gs.tfFinish - gs.tfCommit));
        atomicAdd(&P.phaseClk[11], (unsigned long long)(gs.tfStore - gs.tfFinish));
        atomicAdd(&P.phaseClk[12], (unsigned long long)(gs.tfFlush - gs.tfStore));
        atomicAdd(&P.phaseClk[13], (unsigned long long)(tc4 - gs.tfFlush));
      }
      unsigned long long* pc = P.phaseClk + 4 * (TIER - 1);
      atomicAdd(&pc[0], (unsigned long long)(tc1 - tc0));
      atomicAdd(&pc[1], (unsigned long long)(tc2 - tc1));
      atomicAdd(&pc[2], (unsigned long long)(tc3 - tc2));
      atomicAdd(&pc[3], (unsigned long long)(tc4 - tc3));
    }
    __threadfence();
    unsigned t = atomicAdd(&P.qctl[TIER == 1 ? QC_DONE1 : QC_DONE2], 1u);
    if (t == gridDim.x - 1) {
      if (TIER == 1) {
        for (int c = 0; c < Q_CLASSES; ++c) P.qctl[c] = 0;
        P.qctl[QC_DONE1] = 0;
      } else {
        P.qctl[QC_COUNT2] = 0;
        P.qctl[QC_DONE2] = 0;
      }
      __threadfence();
    }
  }
}

#if defined(HK_TU_INLINE)
}  // namespace
namespace HK_INL_NS {
cudaError_t setScene(const hk::Scene& S) { return cudaMemcpyToSymbol(c_scene, &S, sizeof(Scene)); }
cudaError_t setMaxDynamicSmem(int bytes) { return cudaFuncSetAttribute(k_general<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes); }
size_t staticSmemGeneral() {
  cudaFuncAttributes fa;
  return cudaFuncGetAttributes(&fa, k_general<1>) == cudaSuccess ? fa.sharedSizeBytes : sizeof(Scene) + 2048;
}
void setCarveouts(int pctGeneral, int pctTouch) {
  cudaFuncSetAttribute(k_general<1>, cudaFuncAttributePreferredSharedMemoryCarveout, pctGeneral);
  cudaFuncSetAttribute(k_touch, cudaFuncAttributePreferredSharedMemoryCarveout, pctTouch);
}
void launchGeneral1(unsigned grid, int block, size_t smem, cudaStream_t stream, const KParams& P, const hk::StepIO& io, int unlimited,
                    int lanesLog2, int firstClass, int phaseSync, int envWarps, int classWarps) {
  k_general<1><<<grid, block, smem, stream>>>(P, io, unlimited, lanesLog2, firstClass, phaseSync, envWarps, classWarps);
}
void launchTouch(unsigned grid, int block, cudaStream_t stream, const KParams& P, const hk::StepIO& io) {
  k_touch<<<grid, block, 0, stream>>>(P, io);
}
}  // namespace HK_INL_NS
#else  // pass 1: the rest of the file
// K fused ticks: body state stays in registers/local memory across ticks, HBM state traffic is paid once
__global__ void __launch_bounds__(kBlock) k_rollout(KParams P, StepIO io, int k_steps) {
  __shared__ Scene S;
  stageScene(&S);
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  TickStats st;
  tickStatsZero(st);
  if (i < P.n) {
    Env e;
    loadEnv(P.core, P.n, i, e);
    Cache cache;
    cache.base = P.cache + i;
    cache.stride = (size_t)P.n;
    for (int s = 0; s < k_steps; ++s)
      envTick(S, P.cfg, cache, e, (uint64_t)(P.env_id_offset + i), (size_t)i, io, s == k_steps - 1, st);
    storeEnv(P.core, P.n, i, e);
  }
  flushStats(statsRow(P.stats), st);
}

// ---- K fused ticks without a per-tick grid-wide join (hk_rollout) -------------------------------------------------------------
// A block owns a chunk of envs for all K ticks and alternates, at its own pace, between two phases:
//   * fast phase: its warps take batches of envs that are due for a fast attempt; every lane advances its env through up to
//     `fastRun` consecutive contact-free ticks with the state held in registers (nothing is re-read between ticks; the last
//     good state is written behind each tick) and re-queues it; an env whose proof fails is filed, by work class, for the
//     general phase.  The phase ends when no env is due for a fast attempt: fast envs run ahead, up to K ticks.
//   * general phase: rounds of one general tick (generalTick: Collide -> pooled island solve -> pooled TOI pass -> events
//     -> finish) for up to 384 filed envs, class by class, until nothing is filed; the envs go back to the fast queue.
// Envs are independent, so nothing waits for the slowest solve of "its" tick: the tick count of every env is tracked
// individually, there is no grid-wide join, and one block's long solve does not hold up the other 147.  (Running the two
// phases CONCURRENTLY on disjoint warps of the SM was measured and lost: the two code paths evict each other from the
// instruction cache and a general round takes 2.4 M cycles instead of 0.9 M, profiles/README.md.)
// Queues are rings in shared memory (publish = CAS on an empty slot, consume = reserve a range, then read each slot).
constexpr int kFusedChunk = 512;  // envs per chunk (ring capacity)
struct FusedShared {
  int fastRing[kFusedChunk];
  int genRing[Q_CLASSES][kFusedChunk];
  int remaining[kFusedChunk];  // ticks each env of the chunk still has to make
  unsigned fastHead, fastTail, genHead[Q_CLASSES], genTail[Q_CLASSES];
  int doneCount, roundActive, batch;
  int asgClass[kSlowBlock / 32], asgStart[kSlowBlock / 32], asgCount[kSlowBlock / 32];
};
__device__ __forceinline__ void ringPush(int* ring, unsigned* tail, int j) {
  const unsigned slot = atomicAdd(tail, 1u) % kFusedChunk;
  while (atomicCAS(&ring[slot], -1, j) != -1) {}  // the slot's previous entry (one lap ago) is consumed first
}
__device__ __forceinline__ int ringTake(int* ring, unsigned pos) {
  const unsigned slot = pos % kFusedChunk;
  int j;
  while ((j = atomicExch(&ring[slot], -1)) < 0) {}  // reserved by a producer, not written yet
  return j;
}
__global__ void __launch_bounds__(kSlowBlock, 1) k_rollout_fused(KParams P, StepIO io, int k_steps, int phaseSync, int chunk, int nChunks, int fastRun) {
  __shared__ Scene S;
  extern __shared__ __align__(16) unsigned char sRaw[];
  __shared__ FusedShared F;
  __shared__ unsigned long long sSlowUnit;
  __shared__ unsigned sFin[4];
  stageScene(&S);
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5;
  const int nwarps = blockDim.x >> 5;
  TickStats stFast;
  tickStatsZero(stFast);
  for (int c = blockIdx.x; c < nChunks; c += gridDim.x) {
    const int64_t lo = (int64_t)c * chunk;
    const int m = (int)(P.n - lo < (int64_t)chunk ? P.n - lo : (int64_t)chunk);
    for (int j = threadIdx.x; j < kFusedChunk; j += blockDim.x) {
      F.fastRing[j] = j < m ? j : -1;
      F.remaining[j] = k_steps;
#pragma unroll
      for (int q = 0; q < Q_CLASSES; ++q) F.genRing[q][j] = -1;
    }
    if (threadIdx.x == 0) {
      F.fastHead = 0;
      F.fastTail = (unsigned)m;
      for (int q = 0; q < Q_CLASSES; ++q) F.genHead[q] = F.genTail[q] = 0;
      F.doneCount = 0;
    }
    __syncthreads();
    for (;;) {
      // ---- fast phase: until no env is due for a fast attempt ----
      if (threadIdx.x == 0) {  // batches sized so that the envs due now are spread evenly over the warps
        const int due = (int)(F.fastTail - F.fastHead), waves = (due + blockDim.x - 1) / (int)blockDim.x;
        const int b = waves > 0 ? (due + nwarps * waves - 1) / (nwarps * waves) : 32;
        F.batch = b < 8 ? 8 : (b > 32 ? 32 : b);
      }
      __syncthreads();
      const long long tf0 = clock64();
      int batches = 0;
      for (;;) {
        int take = 0;
        unsigned h = 0;
        if (lane == 0) {
          for (;;) {
            const unsigned hh = *((volatile unsigned*)&F.fastHead), tt = *((volatile unsigned*)&F.fastTail);
            const int avail = (int)(tt - hh);
            if (avail <= 0) { take = -1; break; }
            const int want = avail < F.batch ? avail : F.batch;
            if (atomicCAS(&F.fastHead, hh, hh + (unsigned)want) == hh) { h = hh; take = want; break; }
          }
        }
        take = __shfl_sync(0xffffffffu, take, 0);
        h = __shfl_sync(0xffffffffu, h, 0);
        if (take < 0) break;
        ++batches;
        if (lane < take) {
          const int j = ringTake(F.fastRing, h + (unsigned)lane);
          const int64_t i = lo + j;
          const uint64_t env_id = (uint64_t)(P.env_id_offset + i);
          Env e;
          loadEnv(P.core, P.n, i, e);
          int rem = F.remaining[j];
          for (int it = 0;; ++it) {
            e.bailKind = 15;
            if (!envTickFast(S, P.cfg, e, env_id, (size_t)i, io, rem == 1 && io.obs != nullptr, stFast)) {
              F.remaining[j] = rem;
              const int q = bailClass(e.bailKind);
              ringPush(F.genRing[q], &F.genTail[q], j);  // read after the block-wide barrier that ends this phase
              break;
            }
            --rem;
            // the state as the next tick would load it: stored behind the tick, kept in registers for the next one
            F4 g[CORE_GROUPS];
            envToGroups(e, g);
#pragma unroll
            for (int k = 0; k < CORE_GROUPS; ++k) P.core[(int64_t)k * P.n + i] = make_float4(g[k].x, g[k].y, g[k].z, g[k].w);
            if (rem == 0 || it + 1 >= fastRun) {
              F.remaining[j] = rem;
              __threadfence_block();  // another warp may pick this env up within this phase
              if (rem > 0) ringPush(F.fastRing, &F.fastTail, j);
              else atomicAdd(&F.doneCount, 1);
              break;
            }
            groupsToEnv(g, e);
          }
        }
        __syncwarp();
      }
      // A warp that found the ring empty may leave while another one is still about to re-queue envs; those are picked
      // up in the next fast phase (after this block's general rounds), which keeps the phases strictly alternating.
      __syncthreads();
      if (P.phaseClk && lane == 0) {  // diagnostics (hk_debug_phase_cycles): fast batches, fast-phase cycles
        atomicAdd(&P.phaseClk[4], (unsigned long long)batches);
        if (threadIdx.x == 0) {
          atomicAdd(&P.phaseClk[5], 1ull);
          atomicAdd(&P.phaseClk[6], (unsigned long long)(clock64() - tf0));
        }
      }
      if (F.doneCount >= m) break;
      // ---- general phase: rounds of one general tick until nothing is filed ----
      for (;;) {
        const long long tr0 = clock64();
        if (threadIdx.x == 0) {
          int w = 0;
#pragma unroll
          for (int q = 0; q < Q_CLASSES; ++q) {
            int avail = (int)(F.genTail[q] - F.genHead[q]);
            while (avail > 0 && w < nwarps) {
              const int cnt = avail < 32 ? avail : 32;
              F.asgClass[w] = q;
              F.asgStart[w] = (int)F.genHead[q];
              F.asgCount[w] = cnt;
              F.genHead[q] += (unsigned)cnt;
              avail -= cnt;
              ++w;
            }
          }
          F.roundActive = w;
          for (; w < nwarps; ++w) F.asgCount[w] = 0;
        }
        __syncthreads();
        if (!F.roundActive) break;
        const int envWarps = F.roundActive;
        const int cnt = F.asgCount[wib], cls = F.asgClass[wib];
        const bool valid = lane < cnt;
        int j = 0;
        if (valid) j = ringTake(F.genRing[cls], (unsigned)F.asgStart[wib] + (unsigned)lane);
        const int64_t i = lo + j;
        bool need = false;
        GenStamps gs;
        TickStats st;
        generalTick<1, false>(P, io, S, sRaw, valid, i, cls, cnt > 0, (int64_t)wib, 1, phaseSync, envWarps, (int)blockDim.x,
                              valid && F.remaining[j] == 1 && io.obs != nullptr, st, need, gs, &sSlowUnit, sFin);
        if (valid) {
          const int rem = --F.remaining[j];
          if (rem > 0) ringPush(F.fastRing, &F.fastTail, j);
          else atomicAdd(&F.doneCount, 1);
        }
        __syncthreads();
        if (P.phaseClk) {  // diagnostics: rounds, their filled lanes, cycles in rounds
          if (lane == 0 && cnt > 0) atomicAdd(&P.phaseClk[1], (unsigned long long)cnt);
          if (threadIdx.x == 0) {
            atomicAdd(&P.phaseClk[0], 1ull);
            atomicAdd(&P.phaseClk[2], (unsigned long long)(clock64() - tr0));
          }
        }
      }
      if (F.doneCount >= m) break;
    }
    __syncthreads();
  }
  flushStats(statsRow(P.stats), stFast);
}

__global__ void __launch_bounds__(kBlock) k_get_obs(KParams P, float* obs, float* obs2) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  Env e;
  loadEnv(P.core, P.n, i, e);
  float o[18];
  if (obs) {
    getObs(e, o);
    writeRow18(obs + 18 * i, o);
  }
  if (obs2) {
    getObs2(e, o);
    writeRow18(obs2 + 18 * i, o);
  }
}

__global__ void __launch_bounds__(kBlock) k_get_info(KParams P, float* info, float* info2) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  Env e;
  loadEnv(P.core, P.n, i, e);
  double v[4];
  if (info) {
    getInfo(e, false, v);
    for (int k = 0; k < 4; ++k) info[4 * i + k] = (float)v[k];
  }
  if (info2) {
    getInfo(e, true, v);
    for (int k = 0; k < 4; ++k) info2[4 * i + k] = (float)v[k];
  }
}

__global__ void __launch_bounds__(kBlock) k_get_state(KParams P, uint32_t* rec) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  Env e;
  loadEnv(P.core, P.n, i, e);
  Cache cache;
  cache.base = P.cache + i;
  cache.stride = (size_t)P.n;
  uint32_t* r = rec + (size_t)HK_STATE_WORDS * i;
  packRecord(e, cache, r);
  r[HK_S_MODE] = modeWord(e, P.cfg.mode);
}

__global__ void __launch_bounds__(kBlock) k_set_state(KParams P, const uint32_t* rec) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  Env e;
  Cache cache;
  cache.base = P.cache + i;
  cache.stride = (size_t)P.n;
  const uint32_t* r = rec + (size_t)HK_STATE_WORDS * i;
  unpackRecord(r, e, cache);
  e.mode = modeOfWord(r[HK_S_MODE], P.cfg.mode);
  storeEnv(P.core, P.n, i, e);
}

__global__ void __launch_bounds__(kBlock) k_get_modes(KParams P, uint8_t* modes) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  Env e;
  loadEnv(P.core, P.n, i, e);
  modes[i] = (uint8_t)e.mode;
}

__global__ void __launch_bounds__(kBlock) k_set_obs_state(KParams P, const float* obs18) {
  __shared__ Scene S;
  stageScene(&S);
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= P.n) return;
  Env e;
  loadEnv(P.core, P.n, i, e);
  setObsState(S, e, obs18 + 18 * i, P.cfg.keep_mode);
  storeEnv(P.core, P.n, i, e);
}

}  // namespace

static long long g_shapedFor = -1;  // shapeKey() of the handle whose carve-out preferences are in force

struct hk_env {
  int64_t n;
  int device;
  int64_t env_id_offset;
  Config cfg;
  float4* core;
  uint32_t* cache;
  double* stats;
  int32_t* queue;
  uint32_t* qctl;
  unsigned long long* phaseClk;
  float* actBuf;
  uint32_t* trace;
  const uint8_t* pol2v = nullptr;  // hk_set_opponent_policies
  const uint8_t* resetModes = nullptr;  // hk_set_reset_modes
  bool fused = false;     // HK_FUSED=1: hk_rollout = ONE launch of k_rollout_fused instead of K x the per-tick cascade (measured
                          // slower on B200: profiles/README.md, fused rollout)
  int fusedFastRun = 4;   // HK_FUSED_FAST_RUN: consecutive fast ticks a lane takes with its state in registers before it is re-queued
  int sms = 148;
  int tiers;  // HK_TIERS=2 (default): fast + unlimited general tier; 3: fast + budgeted + unlimited
  bool mono;  // HK_MONO=1: single general kernel per tick (the round-1 baseline, kept for A/B measurements)
  KParams params() const {
    KParams P;
    P.core = core;
    P.cache = cache;
    P.stats = stats;
    P.queue = queue;
    P.qctl = qctl;
    P.phaseClk = phaseClk;
    P.actBuf = actBuf;
    P.trace = trace;
    P.n = n;
    P.env_id_offset = env_id_offset;
    P.cfg = cfg;
    return P;
  }
  unsigned grid() const { return (unsigned)((n + kBlock - 1) / kBlock); }
  // general tiers with 2^lanesLog2 envs per warp and envWarps env-carrying warps per block; tier 1: every work class
  // starts on a warp boundary -> up to 4 partly filled extra warps
  unsigned gridSlow(int lanesPacked, int envWarps, int classWarpsPacked = 0) const {
    int lanesLog2 = 5;
    for (int c = 0; c < Q_CLASSES; ++c) lanesLog2 = std::min(lanesLog2, (lanesPacked >> (3 * c)) & 7);
    int64_t warps = ((n + (1 << lanesLog2) - 1) >> lanesLog2) + 4;
    if (classWarpsPacked < 0)  // automatic shape: at most -classWarpsPacked blocks unless even full blocks do not fit
      return (unsigned)std::max<int64_t>(-classWarpsPacked, (warps + envWarps - 1) / envWarps + Q_CLASSES);
    if (classWarpsPacked > 0) {
      envWarps = 15;
      for (int c = 0; c < Q_CLASSES; ++c) envWarps = std::min(envWarps, (classWarpsPacked >> (4 * c)) & 15);
    }
    return (unsigned)((warps + envWarps - 1) / envWarps) + (classWarpsPacked ? Q_CLASSES : 0);
  }
  // Block shape of tier 1 (measured, profiles/README.md).  The warps of a block walk the tick phases together (shared
  // instruction fetch, pooled solver / TOI tasks), but a block also waits for its slowest warp in every phase.  Small
  // batches get ~one block per SM: few env warps plus helper warps for the pooled phases; batches that fill the GPU
  // get the largest block, all of it env warps.
  int envWarps1, block1;  // HK_ENV_WARPS / HK_SLOW_BLOCK override
  int classWarps1 = 0;    // HK_CLASS_WARPS: env warps per block and work class, 4 bits each (0: blocks cut from the sorted queue; < 0: automatic)
  int targetBlocks = 140; // HK_TARGET_BLOCKS: blocks the automatic shape aims at (one wave, one block per SM)
  void shapeTier1() {
    const int maxWarps = kSlowBlock / 32;
    envWarps1 = tiers == 3 ? 6 : (n < 100000 ? 5 : maxWarps);
    block1 = envWarps1 * 32;  // measured: helper warps do not pay (profiles/README.md)
    if (const char* e = getenv("HK_ENV_WARPS")) envWarps1 = atoi(e);
    if (const char* e = getenv("HK_SLOW_BLOCK")) block1 = atoi(e) / 32 * 32;
    if (envWarps1 < 1) envWarps1 = 1;
    if (envWarps1 > maxWarps) envWarps1 = maxWarps;
    if (block1 < envWarps1 * 32) block1 = envWarps1 * 32;
    if (block1 > kSlowBlock) block1 = kSlowBlock;
    if (const char* e = getenv("HK_TARGET_BLOCKS")) targetBlocks = atoi(e);
    // automatic class-homogeneous block shape (k_general) with up to envWarps1 env warps per block
    if (tiers == 2 && !getenv("HK_ENV_WARPS") && targetBlocks > 0) {
      envWarps1 = n <= 40000 ? 4 : (n <= 100000 ? 8 : maxWarps);
      if (const char* e = getenv("HK_AUTO_WARPS")) envWarps1 = std::min(maxWarps, std::max(1, atoi(e)));  // largest block of the automatic shape
      block1 = envWarps1 * 32;
      if (const char* e = getenv("HK_SLOW_BLOCK")) block1 = std::min(kSlowBlock, std::max(block1, atoi(e) / 32 * 32));
      classWarps1 = -targetBlocks;
    }
    if (const char* cw = getenv("HK_CLASS_WARPS")) {  // one hex digit (1..c) per class, e.g. "8444"; "0": sorted-queue cut
      int packed = 0, c = 0, mx = 0;
      for (; c < Q_CLASSES; ++c) {
        const int v = cw[c] >= '1' && cw[c] <= '9' ? cw[c] - '0' : (cw[c] >= 'a' && cw[c] <= 'c' ? cw[c] - 'a' + 10 : 0);
        if (!v) break;
        packed |= v << (4 * c);
        mx = std::max(mx, v);
      }
      if (c == Q_CLASSES) {
        classWarps1 = packed;
        envWarps1 = mx;
        block1 = std::max(mx * 32, getenv("HK_SLOW_BLOCK") ? std::min(kSlowBlock, atoi(getenv("HK_SLOW_BLOCK")) / 32 * 32) : 0);
      } else if (cw[0] == '0') {
        classWarps1 = 0;
        envWarps1 = n < 100000 ? 5 : maxWarps;
        block1 = envWarps1 * 32;
      }
    }
  }
  int blockTier2() const {
    int64_t b = ((int64_t)(0.06 * (double)n) / (2 * 148) + 31) / 32 * 32;
    if (b < 64) b = 64;
    if (b > kSlowBlock) b = kSlowBlock;
    return (int)b;
  }
  int lanes1, lanes2;  // log2 envs per warp in tier 1 / tier 2, 3 bits per work class (HK_LANES1 / HK_LANES2 / HK_CLASS_LANES override)
  bool touch;          // HK_TOUCH=0 disables the touch tier (A/B measurements)
  int phaseSync;       // HK_PHASE_SYNC: which phase barriers the general tiers keep (bit mask, see k_general)
  int launches;        // kernels per tick of the cascade
  // one tick: k_fast over all envs, k_touch over work class 0, the general tier(s) over the rest
  // The kernels keep several KB of per-thread state in local memory, i.e. in L1: ask for the smallest shared-memory
  // carve-out that holds the blocks an SM will actually run (the driver's default sizes it for the register-limited
  // block count, which at small blocks leaves almost no L1).  HK_CARVEOUT=0 keeps the driver default.
  bool carveout = true;
  long long shapeKey() const { return carveout ? ((long long)device << 56) ^ ((long long)block1 << 40) ^ ((long long)classWarps1 << 44) ^ (long long)gridSlow(lanes1, envWarps1, classWarps1) : -2; }
  int fastBlock = kBlock;  // threads per block of k_fast / k_touch (HK_FAST_BLOCK: 32..128)
  bool fastWide = false;   // k_fast as one staged 512-thread block per SM (HK_FAST_WIDE=0|1; default: from 16k envs)
  int fastWideBlock = kFastWide;  // its threads per block: the batch cut into whole waves of one block per SM (<= 512 threads)
  size_t staticSmem = sizeof(Scene) + 2048;  // static shared memory of k_general (queried at creation)
  size_t fastSmem = sizeof(Scene) + sizeof(float) * kBlock * 18;  // ... of k_fast
  // The carve-out preference is per-function, process-global state: it is set when a handle is created and again only
  // when the previous launch came from a handle with another shape (two handles of different batch sizes in one process).
  void shapeSharedMemory() const {
    if (!carveout) return;
    auto pct = [](size_t bytes) { return (int)std::min<size_t>(100, (bytes * 100 + 228 * 1024 - 1) / (228 * 1024)); };
    const size_t stat = staticSmem;
    const int perSm1 = std::max(1, std::min(65536 / (168 * block1), (int)((gridSlow(lanes1, envWarps1, classWarps1) + 147) / 148)));
    const int perSmAuto = std::max(1, (targetBlocks + sms - 1) / sms);  // automatic shape: blocks per SM the target asks for
    hkinl::setCarveouts(pct((rawBytes(envWarps1 * 32) + stat) * (classWarps1 < 0 ? perSmAuto : perSm1)), pct(stat));
    hkinl256::setCarveouts(pct((rawBytes(envWarps1 * 32) + stat) * (classWarps1 < 0 ? perSmAuto : perSm1)), pct(stat));
    cudaFuncSetAttribute(k_fast<4, kBlock>, cudaFuncAttributePreferredSharedMemoryCarveout, pct((fastSmem + 1024) * 4));
    cudaFuncSetAttribute(k_fast<5, kBlock>, cudaFuncAttributePreferredSharedMemoryCarveout, pct((fastSmem + 1024) * 5));
    cudaFuncSetAttribute(k_fast<1, kFastWide>, cudaFuncAttributePreferredSharedMemoryCarveout, pct(sizeof(Scene) + sizeof(float) * kFastWide * 18 + 1024));
    cudaFuncSetAttribute(k_rollout_fused, cudaFuncAttributePreferredSharedMemoryCarveout, pct(rawBytes(kSlowBlock) + stat + sizeof(FusedShared)));
  }
  // Per-kernel timing (hk_kernel_timing): CUDA events recorded on the launching stream around every kernel of a tick,
  // kTimedSteps ticks deep; off by default (an event record is not part of a plain hk_step).
  enum { kTimedSteps = 2048, kEventsPerStep = 5 };
  cudaEvent_t* events = nullptr;
  mutable int timedSteps = 0;
  void stamp(int k, cudaStream_t stream) const {
    if (events && timedSteps < kTimedSteps) cudaEventRecord(events[timedSteps * kEventsPerStep + k], stream);
  }
  // host-record path (hk_step_host): side stream for the DMA that overlaps the general tier
  cudaStream_t sideStream = nullptr;
  cudaEvent_t evTiers = nullptr, evCopy = nullptr;
  uint32_t* flagDev = nullptr;
  uint32_t* seqHost = nullptr;  // pinned table seq[k] = k: the source of the 4-byte "copy done" flag writes
  uint32_t hostTick = 0;
  void launchCascade(const StepIO& io, cudaStream_t stream, const StepIO* ioGeneral = nullptr, void (*between)(const hk_env*, cudaStream_t, void*) = nullptr,
                     void* betweenArg = nullptr) const {
    if (g_shapedFor != shapeKey()) {
      shapeSharedMemory();
      g_shapedFor = shapeKey();
    }
    if (trace) cudaMemsetAsync(trace, 0, sizeof(uint32_t) * (20 * ((size_t)n / 32 + 8) + 2 * (size_t)n), stream);
    stamp(0, stream);
    if (fastWide) k_fast<1, kFastWide><<<(unsigned)((n + fastWideBlock - 1) / fastWideBlock), fastWideBlock, 0, stream>>>(params(), io);
    else if (n < 100000) k_fast<4, kBlock><<<(unsigned)((n + fastBlock - 1) / fastBlock), fastBlock, 0, stream>>>(params(), io);
    else k_fast<5, kBlock><<<(unsigned)((n + fastBlock - 1) / fastBlock), fastBlock, 0, stream>>>(params(), io);
    stamp(1, stream);
    if (touch) hkinl::launchTouch((unsigned)((n + kTouchBlock - 1) / kTouchBlock), kTouchBlock, stream, params(), io);
    stamp(2, stream);
    if (between) between(this, stream, betweenArg);
    const StepIO& iog = ioGeneral ? *ioGeneral : io;
    const int b2 = blockTier2(), w2 = b2 / 32;
    (block1 <= 256 ? hkinl256::launchGeneral1 : hkinl::launchGeneral1)(gridSlow(lanes1, envWarps1, classWarps1), block1, rawBytes(envWarps1 * 32),
                                                                       stream, params(), iog, tiers == 2 ? 1 : 0, lanes1, touch ? 1 : 0, phaseSync,
                                                                       envWarps1, classWarps1);
    stamp(3, stream);
    if (tiers == 3) k_general<2><<<gridSlow(lanes2, w2), b2, rawBytes(b2), stream>>>(params(), iog, 1, lanes2, 0, phaseSync, w2, 0);
    stamp(4, stream);
    if (events && timedSteps < kTimedSteps) ++timedSteps;
  }
};

static bool validPolicy(int p) { return p >= HK_POLICY_EXTERNAL && p <= HK_POLICY_ZERO; }

__global__ void k_sum_stats(const double* rows, double* out) {  // <<<1, HK_STATS_DIM>>>
  double s = 0.0;
  for (int r = 0; r < kStatsRows; ++r) s += rows[HK_STATS_DIM * r + threadIdx.x];
  out[threadIdx.x] = s;
}

__global__ void k_check_codes(const uint8_t* codes, int64_t n, int maxCode, int* bad) {
  int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && codes[i] > maxCode) atomicAdd(bad, 1);
}
// one-time validation of the initial contents of a per-env code table (later rewrites are the caller's responsibility)
static int checkCodes(const hk_env* h, const uint8_t* codes_dev, int maxCode, const char* msg) {
  DeviceGuard guard(h->device);
  int* bad = nullptr;
  int hostBad = 0;
  HK_CUDA(cudaMalloc(&bad, sizeof(int)));
  cudaMemset(bad, 0, sizeof(int));
  k_check_codes<<<h->grid(), kBlock>>>(codes_dev, h->n, maxCode, bad);
  cudaError_t err = cudaMemcpy(&hostBad, bad, sizeof(int), cudaMemcpyDeviceToHost);
  cudaFree(bad);
  HK_CUDA(err);
  return hostBad ? fail(HK_E_INVALID, msg) : HK_OK;
}

extern "C" {

const char* hk_last_error(void) { return g_err.c_str(); }
const char* hk_version(void) { return "hockey_b200 0.1 (sm_100a, fmad=false)"; }

int hk_create(hk_env** out, int64_t n_envs, int mode, int keep_mode, int device, uint64_t seed, int64_t env_id_offset) {
  if (!out) return fail(HK_E_INVALID, "hk_create: out is NULL");
  *out = nullptr;
  if (n_envs <= 0) return fail(HK_E_INVALID, "hk_create: n_envs must be positive");
  if (mode < HK_MODE_NORMAL || mode > HK_MODE_TRAIN_DEFENSE)
    return fail(HK_E_INVALID, std::to_string(mode) + " is not a valid value for Mode");
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0)
    return fail(HK_E_NODEVICE, "hk_create: no CUDA device available (this library has no CPU fallback)");
  if (device < 0 || device >= count) return fail(HK_E_INVALID, "hk_create: bad device index");
  DeviceGuard guard(device);
  if (!guard.ok) return fail(HK_E_CUDA, "hk_create: cannot select device");
  hk_env* h = new hk_env();
  h->n = n_envs;
  h->device = device;
  h->env_id_offset = env_id_offset;
  h->cfg.mode = mode;
  h->cfg.keep_mode = keep_mode ? 1 : 0;
  h->cfg.max_timesteps = maxTimesteps(mode);
  h->cfg.seed = seed;
  h->core = nullptr;
  h->cache = nullptr;
  h->stats = nullptr;
  h->queue = nullptr;
  h->qctl = nullptr;
  h->phaseClk = nullptr;
  h->actBuf = nullptr;
  h->trace = nullptr;
  {
    const char* m = getenv("HK_MONO");
    h->mono = m && m[0] == '1';
    // measured (profiles/README.md, r1c sweeps): with pooled solves and the block-wide TOI pass the separate budgeted
    // tier no longer pays at any batch size (262,144 envs: 1.65 ms/tick with 2 tiers, 2.22 with 3); it stays available
    // through HK_TIERS=3.  Batches that fill the GPU several times over get the touch tier for the puck-racket ticks.
    const char* t = getenv("HK_TIERS");
    h->tiers = 2;
    if (t && (t[0] == '2' || t[0] == '3')) h->tiers = t[0] - '0';
    // envs per warp in the general tiers: dense warps once the batch can fill the GPU, sparse ones below that
    h->lanes1 = 5;  // measured: sparse warps only add instruction-fetch traffic (profiles/README.md)
    h->lanes2 = 5;
    if (const char* l1 = getenv("HK_LANES1")) h->lanes1 = atoi(l1);
    if (const char* l2 = getenv("HK_LANES2")) h->lanes2 = atoi(l2);
    if (h->lanes1 < 0 || h->lanes1 > 5) h->lanes1 = 5;
    if (h->lanes2 < 0 || h->lanes2 > 5) h->lanes2 = 5;
    h->lanes1 *= 01111;  // same value for the four work classes ...
    h->lanes2 *= 01111;
    // measured (r1c sweeps): around one general-tier wave per SM (100k..200k envs) half-filled warps for the two
    // TOI-heavy classes (racket / puck against statics) shorten the critical blocks (+4 %); elsewhere they cost
    if (n_envs >= 100000 && n_envs < 200000 && !getenv("HK_LANES1")) h->lanes1 = 5 | (5 << 3) | (4 << 6) | (4 << 9);
    if (const char* cl = getenv("HK_CLASS_LANES")) {  // ... or one digit per class, e.g. "5533"
      int packed = 0, c = 0;
      for (; c < Q_CLASSES && cl[c] >= '0' && cl[c] <= '5'; ++c) packed |= (cl[c] - '0') << (3 * c);
      if (c == Q_CLASSES) h->lanes1 = packed;
    }
    const char* tt = getenv("HK_TOUCH");
    h->touch = n_envs >= 750000;  // measured (profiles/README.md r1d): 524,288 envs are 2 % faster without it, 1,048,576 8 % faster with it
    if (tt && (tt[0] == '0' || tt[0] == '1')) h->touch = tt[0] == '1';
    if (const char* co = getenv("HK_CARVEOUT")) h->carveout = co[0] != '0';
    if (const char* fb = getenv("HK_FAST_BLOCK")) h->fastBlock = std::min(kBlock, std::max(32, atoi(fb) / 32 * 32));
    // measured (profiles/README.md r3d, r3f, r3k): with the block size fitted to whole waves the staged shape wins at every size
    // from 16k envs (-4 % at 16k, -8 % at 32k, -2 % at 65k, -5 % at 131k, -10 % at 262k, -45 % at 1,048,576)
    h->fastWide = n_envs >= 16000;
    if (const char* fw = getenv("HK_FAST_WIDE")) h->fastWide = fw[0] == '1';
    h->phaseSync = 31;  // bit 3 (8): pool the single-contact solves too (phase 2); bit 4 (16): re-packed one-point rounds
    if (const char* ps = getenv("HK_PHASE_SYNC")) h->phaseSync = atoi(ps) & 31;
    int sms = 148;
    if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms < 16) sms = 148;
    {  // wide k_fast: w = ceil(n / (sms * 512)) waves of one block per SM, block = ceil(n / (sms * w)) rounded up to a warp
      const int64_t waves = (n_envs + (int64_t)sms * kFastWide - 1) / ((int64_t)sms * kFastWide);
      const int64_t per = (n_envs + sms * waves - 1) / (sms * waves);
      h->fastWideBlock = (int)std::min<int64_t>(kFastWide, std::max<int64_t>(128, (per + 31) / 32 * 32));
      if (const char* fb = getenv("HK_FAST_WIDE_BLOCK")) h->fastWideBlock = std::min(kFastWide, std::max(32, atoi(fb) / 32 * 32));
    }
    cudaFuncAttributes fa;
    h->staticSmem = hkinl::staticSmemGeneral();
    if (cudaFuncGetAttributes(&fa, k_fast<4, kBlock>) == cudaSuccess) h->fastSmem = fa.sharedSizeBytes;
    h->sms = sms;
    if (const char* f = getenv("HK_FUSED")) h->fused = f[0] != '0';
    if (const char* g = getenv("HK_FUSED_FAST_RUN")) h->fusedFastRun = std::max(1, atoi(g));
    h->targetBlocks = sms;  // one general-tier block per SM in a single wave (measured: 148 > 140 > 132 on a 148-SM B200)
    h->shapeTier1();
    h->launches = h->mono ? 1 : 2 + (h->touch ? 1 : 0) + (h->tiers == 3 ? 1 : 0);
  }
  Scene S;
  std::memset(&S, 0, sizeof(S));
  scene_build::build(&S);
  cudaError_t err = cudaMemcpyToSymbol(c_scene, &S, sizeof(Scene));
  if (err == cudaSuccess) err = hkinl::setScene(S);
  if (err == cudaSuccess) err = hkinl::setMaxDynamicSmem((int)rawBytes(kSlowBlock));
  if (err == cudaSuccess) err = hkinl256::setScene(S);
  if (err == cudaSuccess) err = hkinl256::setMaxDynamicSmem((int)rawBytes(256));
  if (err == cudaSuccess) err = cudaFuncSetAttribute(k_general<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rawBytes(kSlowBlock));
  if (err == cudaSuccess) err = cudaFuncSetAttribute(k_rollout_fused, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rawBytes(kSlowBlock));
  if (err == cudaSuccess) err = cudaMalloc(&h->core, sizeof(float4) * CORE_GROUPS * (size_t)n_envs);
  if (err == cudaSuccess) err = cudaMalloc(&h->cache, sizeof(uint32_t) * 6 * N_PAIRS * (size_t)n_envs);
  if (err == cudaSuccess) err = cudaMalloc(&h->stats, sizeof(double) * HK_STATS_DIM * (kStatsRows + 1));  // rows + their sum
  if (err == cudaSuccess) err = cudaMalloc(&h->queue, sizeof(int32_t) * 5 * (size_t)n_envs);
  if (err == cudaSuccess) err = cudaMalloc(&h->qctl, sizeof(uint32_t) * 8);
  if (err == cudaSuccess) err = cudaMemset(h->qctl, 0, sizeof(uint32_t) * 8);
  if (err == cudaSuccess) err = cudaMalloc(&h->actBuf, sizeof(float) * 8 * (size_t)n_envs);
  if (err == cudaSuccess) err = cudaMalloc(&h->phaseClk, sizeof(unsigned long long) * 16);
  if (err == cudaSuccess) err = cudaMemset(h->phaseClk, 0, sizeof(unsigned long long) * 16);
  if (err == cudaSuccess && getenv("HK_LANE_TRACE")) err = cudaMalloc(&h->trace, sizeof(uint32_t) * (20 * ((size_t)n_envs / 32 + 8) + 2 * (size_t)n_envs));
  if (err == cudaSuccess) err = cudaMemset(h->cache, 0, sizeof(uint32_t) * 6 * N_PAIRS * (size_t)n_envs);
  if (err == cudaSuccess) err = cudaMemset(h->stats, 0, sizeof(double) * HK_STATS_DIM * (kStatsRows + 1));
  if (err == cudaSuccess) {
    k_create<<<h->grid(), kBlock>>>(h->params());
    err = cudaGetLastError();
  }
  if (err == cudaSuccess) err = cudaDeviceSynchronize();
  if (err != cudaSuccess) {
    std::string msg = std::string("hk_create: ") + cudaGetErrorString(err);
    cudaFree(h->core);
    cudaFree(h->cache);
    cudaFree(h->stats);
    cudaFree(h->queue);
    cudaFree(h->qctl);
    cudaFree(h->phaseClk);
    cudaFree(h->actBuf);
    cudaFree(h->trace);
    delete h;
    return fail(HK_E_CUDA, msg);
  }
  *out = h;
  return HK_OK;
}

int hk_destroy(hk_env* h) {
  if (!h) return HK_OK;
  DeviceGuard guard(h->device);
  cudaFree(h->core);
  cudaFree(h->cache);
  cudaFree(h->stats);
  cudaFree(h->queue);
  cudaFree(h->qctl);
  cudaFree(h->phaseClk);
  cudaFree(h->actBuf);
  cudaFree(h->trace);
  if (h->events) {
    for (int k = 0; k < hk_env::kTimedSteps * hk_env::kEventsPerStep; ++k) cudaEventDestroy(h->events[k]);
    delete[] h->events;
  }
  if (h->sideStream) {
    cudaStreamDestroy(h->sideStream);
    cudaEventDestroy(h->evTiers);
    cudaEventDestroy(h->evCopy);
    cudaFree(h->flagDev);
    cudaFreeHost(h->seqHost);
  }
  delete h;
  return HK_OK;
}

int64_t hk_num_envs(const hk_env* h) { return h ? h->n : 0; }

int hk_reset_seeded(hk_env* h, const uint8_t* mask_dev, const int8_t* one_starting_dev, const int64_t* seeds_dev, float* obs_dev,
                    void* stream) {
  if (!h) return fail(HK_E_INVALID, "hk_reset: NULL handle");
  DeviceGuard guard(h->device);
  k_reset<<<h->grid(), kBlock, 0, (cudaStream_t)stream>>>(h->params(), mask_dev, one_starting_dev, seeds_dev, h->resetModes, obs_dev);
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_reset(hk_env* h, const uint8_t* mask_dev, const int8_t* one_starting_dev, float* obs_dev, void* stream) {
  return hk_reset_seeded(h, mask_dev, one_starting_dev, nullptr, obs_dev, stream);
}

int hk_step(hk_env* h, const float* action_dev, int action_stride, int p1_policy, int p2_policy, int flags, float* obs_dev,
            float* obs2_dev, float* reward_dev, float* reward2_dev, uint8_t* done_dev, float* info_dev, float* info2_dev,
            float* final_obs_dev, void* stream) {
  if (!h) return fail(HK_E_INVALID, "hk_step: NULL handle");
  const bool perEnv = p2_policy == HK_POLICY_PER_ENV;
  if (!validPolicy(p1_policy) || !(validPolicy(p2_policy) || perEnv)) return fail(HK_E_INVALID, "hk_step: invalid policy id");
  if (perEnv && !h->pol2v) return fail(HK_E_INVALID, "hk_step: HK_POLICY_PER_ENV without hk_set_opponent_policies");
  if (!obs_dev) return fail(HK_E_INVALID, "hk_step: obs_dev is required");
  if ((((uintptr_t)info_dev | (uintptr_t)info2_dev) & 15u) != 0) return fail(HK_E_INVALID, "hk_step: info tensors must be 16-byte aligned");
  if ((((uintptr_t)obs_dev | (uintptr_t)obs2_dev | (uintptr_t)final_obs_dev) & 7u) != 0)
    return fail(HK_E_INVALID, "hk_step: observation tensors must be 8-byte aligned");
  if ((p1_policy == HK_POLICY_EXTERNAL || p2_policy == HK_POLICY_EXTERNAL) && !action_dev)
    return fail(HK_E_INVALID, "hk_step: action_dev is NULL but a policy is EXTERNAL");
  if (p1_policy == HK_POLICY_EXTERNAL && action_stride < 4) return fail(HK_E_INVALID, "hk_step: action_stride < 4");
  if (p2_policy == HK_POLICY_EXTERNAL && action_stride < 8)
    return fail(HK_E_INVALID, "hk_step: player 2 EXTERNAL needs action_stride >= 8");
  // per-env codes may contain EXTERNAL: those envs read columns 4..7
  if (perEnv && (!action_dev || action_stride < 8))
    return fail(HK_E_INVALID, "hk_step: HK_POLICY_PER_ENV needs action_dev with action_stride >= 8");
  DeviceGuard guard(h->device);
  StepIO io;
  io.action = action_dev;
  io.stride = action_stride;
  io.pol1 = p1_policy;
  io.pol2 = perEnv ? HK_POLICY_ZERO : p2_policy;
  io.pol2v = perEnv ? h->pol2v : nullptr;
  io.resetModes = h->resetModes;
  io.flags = flags;
  io.obs = obs_dev;
  io.obs2 = obs2_dev;
  io.reward = reward_dev;
  io.reward2 = reward2_dev;
  io.done = done_dev;
  io.info = info_dev;
  io.info2 = info2_dev;
  io.final_obs = final_obs_dev;
  io.write = 1;
  io.actBuf = nullptr;
  io.waitFlag = nullptr;
  io.waitValue = 0;
  // k_fast writes a warp's 32 rows with 128-bit stores when the row tensors are 16-byte aligned (torch tensors are)
  io.stageRows = (((uintptr_t)obs_dev | (uintptr_t)final_obs_dev) & 15u) == 0 ? 1 : 0;
  if (h->mono) {
    k_step<<<h->grid(), kBlock, 0, (cudaStream_t)stream>>>(h->params(), io);
  } else {
    io.actBuf = h->actBuf;
    h->launchCascade(io, (cudaStream_t)stream);
  }
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

// ---- host-record stepping ------------------------------------------------------------------------------------------------
// packed record: obs [n,18] f32 | reward [n] f32 | info [n,4] f32 | done [n] u8 (| final_obs [n,18] f32), sections 256-byte aligned
static int64_t recordLayout(int64_t n, int with_final_obs, int64_t off[5]) {
  auto up = [](int64_t x) { return (x + 255) / 256 * 256; };
  int64_t t = 0;
  off[0] = t; t += up(72 * n);
  off[1] = t; t += up(4 * n);
  off[2] = t; t += up(16 * n);
  off[3] = t; t += up(n);
  off[4] = t;
  if (with_final_obs) t += up(72 * n);
  return t;
}
int64_t hk_host_record_bytes(int64_t n_envs, int with_final_obs, int64_t* offsets5) {
  int64_t off[5];
  const int64_t t = recordLayout(n_envs, with_final_obs, off);
  if (offsets5) for (int k = 0; k < 5; ++k) offsets5[k] = off[k];
  return t;
}
static StepIO recordIO(const StepIO& base, uint8_t* rec, const int64_t off[5], int with_final_obs) {
  StepIO io = base;
  io.obs = reinterpret_cast<float*>(rec + off[0]);
  io.reward = reinterpret_cast<float*>(rec + off[1]);
  io.info = reinterpret_cast<float*>(rec + off[2]);
  io.done = rec + off[3];
  io.final_obs = with_final_obs ? reinterpret_cast<float*>(rec + off[4]) : nullptr;
  io.obs2 = io.reward2 = io.info2 = nullptr;
  return io;
}
struct HostCopyArgs {
  uint8_t* recDev;
  uint8_t* recHost;
  int64_t bytes;
};
static void copyFastRows(const hk_env* h, cudaStream_t stream, void* argp) {
  // The fast (and touch) tier's rows are complete: a copy engine moves the device record to the host while the general
  // tier runs; a 4-byte DMA write behind it raises the flag the general tier waits for before ITS rows go to the host.
  const HostCopyArgs* a = static_cast<const HostCopyArgs*>(argp);
  cudaEventRecord(h->evTiers, stream);
  cudaStreamWaitEvent(h->sideStream, h->evTiers, 0);
  cudaMemcpyAsync(a->recHost, a->recDev, (size_t)a->bytes, cudaMemcpyDeviceToHost, h->sideStream);
  cudaMemcpyAsync(h->flagDev, h->seqHost + (h->hostTick & 0xFFFFu), sizeof(uint32_t), cudaMemcpyHostToDevice, h->sideStream);
  cudaEventRecord(h->evCopy, h->sideStream);
}

int hk_step_host(hk_env* h, const float* action_host, int action_stride, int p1_policy, int p2_policy, int flags, float* action_dev,
                 uint8_t* record_dev, uint8_t* record_host, int with_final_obs, void* stream) {
  if (!h) return fail(HK_E_INVALID, "hk_step_host: NULL handle");
  if (!record_dev || !record_host) return fail(HK_E_INVALID, "hk_step_host: record_dev and record_host are required");
  const bool perEnv = p2_policy == HK_POLICY_PER_ENV;
  if (!validPolicy(p1_policy) || !(validPolicy(p2_policy) || perEnv)) return fail(HK_E_INVALID, "hk_step_host: invalid policy id");
  if (perEnv && !h->pol2v) return fail(HK_E_INVALID, "hk_step_host: HK_POLICY_PER_ENV without hk_set_opponent_policies");
  const bool ext = p1_policy == HK_POLICY_EXTERNAL || p2_policy == HK_POLICY_EXTERNAL || perEnv;
  if (ext && (!action_host || !action_dev)) return fail(HK_E_INVALID, "hk_step_host: action buffers are NULL but a policy is EXTERNAL");
  if (ext && (action_stride < 4 || ((p2_policy == HK_POLICY_EXTERNAL || perEnv) && action_stride < 8)))
    return fail(HK_E_INVALID, "hk_step_host: action_stride too small for the EXTERNAL policies");
  if ((((uintptr_t)record_dev | (uintptr_t)record_host) & 15u) != 0) return fail(HK_E_INVALID, "hk_step_host: records must be 16-byte aligned");
  DeviceGuard guard(h->device);
  cudaStream_t st = (cudaStream_t)stream;
  if (!h->sideStream) {
    HK_CUDA(cudaStreamCreateWithFlags(&h->sideStream, cudaStreamNonBlocking));
    HK_CUDA(cudaEventCreateWithFlags(&h->evTiers, cudaEventDisableTiming));
    HK_CUDA(cudaEventCreateWithFlags(&h->evCopy, cudaEventDisableTiming));
    HK_CUDA(cudaMalloc(&h->flagDev, sizeof(uint32_t)));
    HK_CUDA(cudaMemset(h->flagDev, 0xFF, sizeof(uint32_t)));
    HK_CUDA(cudaMallocHost(&h->seqHost, sizeof(uint32_t) * 65536));
    for (uint32_t k = 0; k < 65536; ++k) h->seqHost[k] = k;
  }
  int64_t off[5];
  const int64_t bytes = recordLayout(h->n, with_final_obs, off);
  if (ext) HK_CUDA(cudaMemcpyAsync(action_dev, action_host, sizeof(float) * (size_t)action_stride * (size_t)h->n, cudaMemcpyHostToDevice, st));
  StepIO io;
  std::memset(&io, 0, sizeof(io));
  io.action = ext ? action_dev : nullptr;
  io.stride = action_stride;
  io.pol1 = p1_policy;
  io.pol2 = perEnv ? HK_POLICY_ZERO : p2_policy;
  io.pol2v = perEnv ? h->pol2v : nullptr;
  io.resetModes = h->resetModes;
  io.flags = flags;
  io.write = 1;
  StepIO ioDev = recordIO(io, record_dev, off, with_final_obs);
  ioDev.stageRows = 1;
  if (h->mono) {  // single-kernel baseline: device record, then one copy
    k_step<<<h->grid(), kBlock, 0, st>>>(h->params(), ioDev);
    HK_CUDA(cudaMemcpyAsync(record_host, record_dev, (size_t)bytes, cudaMemcpyDeviceToHost, st));
  } else {
    ioDev.actBuf = h->actBuf;
    ++h->hostTick;
    StepIO ioHost = recordIO(ioDev, record_host, off, with_final_obs);  // the general tier stores straight into the mapped host record
    ioHost.waitFlag = h->flagDev;
    ioHost.waitValue = h->hostTick & 0xFFFFu;
    HostCopyArgs args{record_dev, record_host, bytes};
    h->launchCascade(ioDev, st, &ioHost, copyFastRows, &args);
    HK_CUDA(cudaStreamWaitEvent(st, h->evCopy, 0));  // whoever waits on `stream` also waits for the DMA
  }
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_set_opponent_policies(hk_env* h, const uint8_t* codes_dev) {
  if (!h) return fail(HK_E_INVALID, "hk_set_opponent_policies: NULL handle");
  if (codes_dev) {
    const int rc = checkCodes(h, codes_dev, HK_POLICY_ZERO, "hk_set_opponent_policies: codes must be HK_POLICY_EXTERNAL..HK_POLICY_ZERO");
    if (rc != HK_OK) return rc;
  }
  h->pol2v = codes_dev;
  return HK_OK;
}

int hk_set_reset_modes(hk_env* h, const uint8_t* modes_dev) {
  if (!h) return fail(HK_E_INVALID, "hk_set_reset_modes: NULL handle");
  if (modes_dev) {
    const int rc = checkCodes(h, modes_dev, HK_MODE_TRAIN_DEFENSE, "hk_set_reset_modes: modes must be HK_MODE_NORMAL..HK_MODE_TRAIN_DEFENSE");
    if (rc != HK_OK) return rc;
  }
  h->resetModes = modes_dev;
  return HK_OK;
}

int hk_get_modes(hk_env* h, uint8_t* modes_dev, void* stream) {
  if (!h || !modes_dev) return fail(HK_E_INVALID, "hk_get_modes: NULL argument");
  DeviceGuard guard(h->device);
  k_get_modes<<<h->grid(), kBlock, 0, (cudaStream_t)stream>>>(h->params(), modes_dev);
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_rollout(hk_env* h, int k_steps, int p1_policy, int p2_policy, float* obs_dev, void* stream) {
  if (!h) return fail(HK_E_INVALID, "hk_rollout: NULL handle");
  if (k_steps <= 0) return fail(HK_E_INVALID, "hk_rollout: k_steps must be positive");
  if (!validPolicy(p1_policy) || !validPolicy(p2_policy) || p1_policy == HK_POLICY_EXTERNAL || p2_policy == HK_POLICY_EXTERNAL)
    return fail(HK_E_INVALID, "hk_rollout: policies must be in-kernel (not EXTERNAL)");
  DeviceGuard guard(h->device);
  StepIO io;
  std::memset(&io, 0, sizeof(io));
  io.pol1 = p1_policy;
  io.pol2 = p2_policy;
  io.resetModes = h->resetModes;
  io.flags = HK_STEP_AUTORESET;
  io.obs = obs_dev;
  if (h->mono) {  // K ticks fused in one launch, state in registers between ticks (the round-1 baseline kernel)
    io.write = 1;
    k_rollout<<<h->grid(), kBlock, 0, (cudaStream_t)stream>>>(h->params(), io, k_steps);
  } else if (h->fused) {  // K ticks in ONE launch without a per-tick join: fast envs run ahead, slow ones are re-queued
    io.actBuf = h->actBuf;
    io.write = obs_dev ? 1 : 0;
    KParams P = h->params();
    P.trace = nullptr;
    int64_t chunk = (h->n + h->sms - 1) / h->sms;
    if (chunk > kFusedChunk) chunk = kFusedChunk;
    const int64_t nChunks = (h->n + chunk - 1) / chunk;
    k_rollout_fused<<<(unsigned)std::min<int64_t>(nChunks, h->sms), kSlowBlock, rawBytes(kSlowBlock), (cudaStream_t)stream>>>(
        P, io, k_steps, h->phaseSync, (int)chunk, (int)nChunks, h->fusedFastRun);
  } else {        // K ticks of the kernel cascade back to back; only the last tick writes its observation
    io.actBuf = h->actBuf;
    for (int s = 0; s < k_steps; ++s) {
      io.write = (s == k_steps - 1 && obs_dev) ? 1 : 0;
      h->launchCascade(io, (cudaStream_t)stream);
    }
  }
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_get_obs(hk_env* h, float* obs_dev, float* obs2_dev, void* stream) {
  if (!h) return fail(HK_E_INVALID, "hk_get_obs: NULL handle");
  DeviceGuard guard(h->device);
  k_get_obs<<<h->grid(), kBlock, 0, (cudaStream_t)stream>>>(h->params(), obs_dev, obs2_dev);
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_get_info(hk_env* h, float* info_dev, float* info2_dev, void* stream) {
  if (!h) return fail(HK_E_INVALID, "hk_get_info: NULL handle");
  DeviceGuard guard(h->device);
  k_get_info<<<h->grid(), kBlock, 0, (cudaStream_t)stream>>>(h->params(), info_dev, info2_dev);
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_get_state(hk_env* h, uint32_t* state_dev, void* stream) {
  if (!h || !state_dev) return fail(HK_E_INVALID, "hk_get_state: NULL argument");
  DeviceGuard guard(h->device);
  k_get_state<<<h->grid(), kBlock, 0, (cudaStream_t)stream>>>(h->params(), state_dev);
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_set_state(hk_env* h, const uint32_t* state_dev, void* stream) {
  if (!h || !state_dev) return fail(HK_E_INVALID, "hk_set_state: NULL argument");
  DeviceGuard guard(h->device);
  k_set_state<<<h->grid(), kBlock, 0, (cudaStream_t)stream>>>(h->params(), state_dev);
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_set_obs_state(hk_env* h, const float* obs18_dev, void* stream) {
  if (!h || !obs18_dev) return fail(HK_E_INVALID, "hk_set_obs_state: NULL argument");
  DeviceGuard guard(h->device);
  k_set_obs_state<<<h->grid(), kBlock, 0, (cudaStream_t)stream>>>(h->params(), obs18_dev);
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_get_stats(hk_env* h, double* out_host, void* stream) {
  if (!h || !out_host) return fail(HK_E_INVALID, "hk_get_stats: NULL argument");
  DeviceGuard guard(h->device);
  double* sum = h->stats + HK_STATS_DIM * kStatsRows;
  k_sum_stats<<<1, HK_STATS_DIM, 0, (cudaStream_t)stream>>>(h->stats, sum);
  HK_CUDA(cudaMemcpyAsync(out_host, sum, sizeof(double) * HK_STATS_DIM, cudaMemcpyDeviceToHost, (cudaStream_t)stream));
  HK_CUDA(cudaStreamSynchronize((cudaStream_t)stream));
  return HK_OK;
}

int hk_clear_stats(hk_env* h, void* stream) {
  if (!h) return fail(HK_E_INVALID, "hk_clear_stats: NULL handle");
  DeviceGuard guard(h->device);
  HK_CUDA(cudaMemsetAsync(h->stats, 0, sizeof(double) * HK_STATS_DIM * (kStatsRows + 1), (cudaStream_t)stream));
  return HK_OK;
}

int hk_copy_stats(hk_env* h, double* dst_dev, void* stream) {
  if (!h || !dst_dev) return fail(HK_E_INVALID, "hk_copy_stats: NULL argument");
  DeviceGuard guard(h->device);
  k_sum_stats<<<1, HK_STATS_DIM, 0, (cudaStream_t)stream>>>(h->stats, dst_dev);
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_debug_phase_cycles(hk_env* h, double* out_host8) {
  if (!h || !out_host8) return fail(HK_E_INVALID, "hk_debug_phase_cycles: NULL argument");
  DeviceGuard guard(h->device);
  unsigned long long v[16];
  HK_CUDA(cudaMemcpy(v, h->phaseClk, sizeof(v), cudaMemcpyDeviceToHost));
  for (int k = 0; k < 8; ++k) out_host8[k] = (double)v[k];
  return HK_OK;
}

int hk_debug_finish_cycles(hk_env* h, double* out_host6) {
  if (!h || !out_host6) return fail(HK_E_INVALID, "hk_debug_finish_cycles: NULL argument");
  DeviceGuard guard(h->device);
  unsigned long long v[16];
  HK_CUDA(cudaMemcpy(v, h->phaseClk, sizeof(v), cudaMemcpyDeviceToHost));
  for (int k = 0; k < 6; ++k) out_host6[k] = (double)v[8 + k];
  return HK_OK;
}

int hk_debug_lane_trace(hk_env* h, uint32_t* out_host, int64_t n_words) {
  if (!h || !out_host) return fail(HK_E_INVALID, "hk_debug_lane_trace: NULL argument");
  if (!h->trace) return fail(HK_E_INVALID, "hk_debug_lane_trace: create the env with HK_LANE_TRACE=1");
  const int64_t have = 20 * (h->n / 32 + 8) + 2 * h->n;
  DeviceGuard guard(h->device);
  HK_CUDA(cudaMemcpy(out_host, h->trace, sizeof(uint32_t) * (size_t)(n_words < have ? n_words : have), cudaMemcpyDeviceToHost));
  return HK_OK;
}

int hk_actor_param_bytes(void) { return hk_actor::kParamBytes; }

// validation shared by the plain and the noisy entry points (error messages name `who`); HK_OK or an error code
static int actorCheck(const char* who, const void* params_dev, const float* obs_dev, const float* act_dev, int act_stride, int64_t n) {
  if (!params_dev || !obs_dev || !act_dev) return fail(HK_E_INVALID, std::string(who) + ": NULL argument");
  if (n <= 0 || act_stride < hk_actor::kAct) return fail(HK_E_INVALID, std::string(who) + ": n must be positive and act_stride >= 4");
  if ((((uintptr_t)params_dev) & 15u) || (((uintptr_t)obs_dev) & 7u)) return fail(HK_E_INVALID, std::string(who) + ": params need 16-byte, obs 8-byte alignment");
  return HK_OK;
}

static int noiseCheck(const char* who, const uint64_t* counter_dev, float sigma, float clip, int64_t row0) {
  if (!counter_dev) return fail(HK_E_INVALID, std::string(who) + ": NULL argument");
  if (((uintptr_t)counter_dev) & 7u) return fail(HK_E_INVALID, std::string(who) + ": counter needs 8-byte alignment");
  if (!(sigma >= 0.0f) || std::isinf(sigma)) return fail(HK_E_INVALID, std::string(who) + ": sigma must be finite and >= 0");
  if (std::isnan(clip)) return fail(HK_E_INVALID, std::string(who) + ": clip must not be NaN");
  if (row0 < 0) return fail(HK_E_INVALID, std::string(who) + ": row0 must be >= 0");
  return HK_OK;
}

static int deviceCheck(const char* who, int device) {
  int count = 0;
  if (cudaGetDeviceCount(&count) != cudaSuccess || count == 0) return fail(HK_E_NODEVICE, std::string(who) + ": no CUDA device (there is no CPU fallback)");
  if (device < 0 || device >= count) return fail(HK_E_INVALID, std::string(who) + ": bad device index");
  return HK_OK;
}

// clip <= 0 or +inf: no clip (the kernel clamps to +-inf)
static float effectiveClip(float clip) { return clip > 0.0f ? clip : INFINITY; }

static int actorConfigure(const void* kernel, bool* configured, int device) {
  if (!configured[device & 63]) {
    HK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, hk_actor::kSmemBytes));
    configured[device & 63] = true;
  }
  return HK_OK;
}

static int actorSms(int device) {
  int sms = 148;
  if (cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, device) != cudaSuccess || sms < 1) sms = 148;
  return sms;
}

// One launch of the single-weight-set kernel; sigma == 0 runs the plain kernel (bit-identical to hk_actor_forward).
static int actorLaunch(const void* params_dev, const float* obs_dev, float* act_dev, int act_stride, int64_t n, bool noisy,
                       uint64_t seed, const uint64_t* counter_dev, float sigma, float clip, int64_t row0, int device, void* stream) {
  DeviceGuard guard(device);
  const int64_t tiles = (n + hk_actor::kRows - 1) / hk_actor::kRows;
  const unsigned grid = (unsigned)std::min<int64_t>(tiles, actorSms(device));
  if (noisy && sigma != 0.0f) {
    static bool configured[64] = {false};
    if (int rc = actorConfigure((const void*)hk_actor::k_actor_mlp_noisy, configured, device)) return rc;
    hk_actor::k_actor_mlp_noisy<<<grid, hk_actor::kThreads, hk_actor::kSmemBytes, (cudaStream_t)stream>>>(
        (const unsigned char*)params_dev, obs_dev, act_dev, act_stride, (long long)n, seed, counter_dev, sigma, effectiveClip(clip),
        (long long)row0);
  } else {
    static bool configured[64] = {false};
    if (int rc = actorConfigure((const void*)hk_actor::k_actor_mlp, configured, device)) return rc;
    hk_actor::k_actor_mlp<<<grid, hk_actor::kThreads, hk_actor::kSmemBytes, (cudaStream_t)stream>>>(
        (const unsigned char*)params_dev, obs_dev, act_dev, act_stride, (long long)n);
  }
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_actor_forward(const void* params_dev, const float* obs_dev, float* act_dev, int act_stride, int64_t n, int device, void* stream) {
  const char* who = "hk_actor_forward";
  if (int rc = actorCheck(who, params_dev, obs_dev, act_dev, act_stride, n)) return rc;
  if (int rc = deviceCheck(who, device)) return rc;
  return actorLaunch(params_dev, obs_dev, act_dev, act_stride, n, false, 0, nullptr, 0.0f, 0.0f, 0, device, stream);
}

int hk_actor_forward_noisy(const void* params_dev, const float* obs_dev, float* act_dev, int act_stride, int64_t n, uint64_t seed,
                           const uint64_t* counter_dev, float sigma, float clip, int64_t row0, int device, void* stream) {
  const char* who = "hk_actor_forward_noisy";
  if (int rc = actorCheck(who, params_dev, obs_dev, act_dev, act_stride, n)) return rc;
  if (int rc = noiseCheck(who, counter_dev, sigma, clip, row0)) return rc;
  if (int rc = deviceCheck(who, device)) return rc;
  return actorLaunch(params_dev, obs_dev, act_dev, act_stride, n, true, seed, counter_dev, sigma, clip, row0, device, stream);
}

int64_t hk_actor_pool_scratch_bytes(int64_t n, int k) {
  if (n <= 0 || n > INT32_MAX || k < 1 || k > hk_actor::kPoolMaxK)
    return fail(HK_E_INVALID, "hk_actor_pool_scratch_bytes: n must be in [1, 2^31 - 1] and k in [1, 4096]");
  return 4 * hk_actor::poolScratchWords(n, k);
}

static int poolCheck(const char* who, const void* params_dev, int k, const int32_t* choice_dev, const float* obs_dev, float* act_dev,
                     int act_stride, int64_t n, void* scratch_dev) {
  using namespace hk_actor;
  if (!params_dev || !choice_dev || !obs_dev || !act_dev || !scratch_dev) return fail(HK_E_INVALID, std::string(who) + ": NULL argument");
  if (n <= 0 || n > INT32_MAX || act_stride < kAct)
    return fail(HK_E_INVALID, std::string(who) + ": n must be in [1, 2^31 - 1] and act_stride >= 4");
  if (k < 1 || k > kPoolMaxK) return fail(HK_E_INVALID, std::string(who) + ": k must be in [1, 4096]");
  if ((((uintptr_t)params_dev) & 15u) || (((uintptr_t)obs_dev) & 7u) || (((uintptr_t)choice_dev) & 3u) || (((uintptr_t)scratch_dev) & 15u))
    return fail(HK_E_INVALID, std::string(who) + ": params and scratch need 16-byte, obs 8-byte, choice 4-byte alignment");
  return HK_OK;
}

// The grouping kernels, then the pooled tensor-core kernel; sigma == 0 runs the plain one (bit-identical to
// hk_actor_forward_pool).
static int poolLaunch(const void* params_dev, int k, const int32_t* choice_dev, const float* obs_dev, float* act_dev, int act_stride,
                      int64_t n, void* scratch_dev, bool noisy, uint64_t seed, const uint64_t* counter_dev, float sigma, float clip,
                      int64_t row0, int device, void* stream) {
  using namespace hk_actor;
  DeviceGuard guard(device);
  const bool withNoise = noisy && sigma != 0.0f;
  static bool configured[64] = {false}, configuredNoisy[64] = {false};
  if (int rc = withNoise ? actorConfigure((const void*)k_actor_pool_mlp_noisy, configuredNoisy, device) : actorConfigure((const void*)k_actor_pool_mlp, configured, device))
    return rc;
  const int sms = actorSms(device);
  cudaStream_t st = (cudaStream_t)stream;
  int32_t* scratch = (int32_t*)scratch_dev;
  HK_CUDA(cudaMemsetAsync(scratch, 0, sizeof(int32_t) * (size_t)k, st));  // counts
  const int64_t chunks = (n + kPoolThreads * kPoolItems - 1) / (kPoolThreads * kPoolItems);
  const unsigned histBlocks = (unsigned)std::min<int64_t>(chunks, 4 * (int64_t)sms);
  k_pool_count<<<histBlocks, kPoolThreads, sizeof(int32_t) * (size_t)k, st>>>(choice_dev, (long long)n, k, scratch);
  k_pool_scan<<<1, kScanThreads, 0, st>>>(scratch, k);
  k_pool_scatter<<<histBlocks, kPoolThreads, 2 * sizeof(int32_t) * (size_t)k, st>>>(choice_dev, (long long)n, k, scratch);
  // the tile count is only known on the device: at most ceil(n / 128) + k - 1 tiles (one partial tile per group)
  const int64_t grid = std::min<int64_t>(sms, (n + kRows - 1) / kRows + k);
  if (withNoise)
    k_actor_pool_mlp_noisy<<<(unsigned)grid, kThreads, kSmemBytes, st>>>((const unsigned char*)params_dev, k, scratch, obs_dev, act_dev,
                                                                         act_stride, seed, counter_dev, sigma, effectiveClip(clip), (long long)row0);
  else
    k_actor_pool_mlp<<<(unsigned)grid, kThreads, kSmemBytes, st>>>((const unsigned char*)params_dev, k, scratch, obs_dev, act_dev, act_stride);
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_actor_forward_pool(const void* params_dev, int k, const int32_t* choice_dev, const float* obs_dev, float* act_dev,
                          int act_stride, int64_t n, void* scratch_dev, int device, void* stream) {
  const char* who = "hk_actor_forward_pool";
  if (int rc = poolCheck(who, params_dev, k, choice_dev, obs_dev, act_dev, act_stride, n, scratch_dev)) return rc;
  if (int rc = deviceCheck(who, device)) return rc;
  return poolLaunch(params_dev, k, choice_dev, obs_dev, act_dev, act_stride, n, scratch_dev, false, 0, nullptr, 0.0f, 0.0f, 0, device, stream);
}

int hk_actor_forward_pool_noisy(const void* params_dev, int k, const int32_t* choice_dev, const float* obs_dev, float* act_dev,
                                int act_stride, int64_t n, void* scratch_dev, uint64_t seed, const uint64_t* counter_dev, float sigma,
                                float clip, int64_t row0, int device, void* stream) {
  const char* who = "hk_actor_forward_pool_noisy";
  if (int rc = poolCheck(who, params_dev, k, choice_dev, obs_dev, act_dev, act_stride, n, scratch_dev)) return rc;
  if (int rc = noiseCheck(who, counter_dev, sigma, clip, row0)) return rc;
  if (int rc = deviceCheck(who, device)) return rc;
  return poolLaunch(params_dev, k, choice_dev, obs_dev, act_dev, act_stride, n, scratch_dev, true, seed, counter_dev, sigma, clip, row0,
                    device, stream);
}

int hk_actor_pack(const float* w1, const float* b1, const float* w2, const float* b2, const float* w3, const float* b3, void* params_dev,
                  int device, void* stream) {
  const char* who = "hk_actor_pack";
  if (!w1 || !b1 || !w2 || !b2 || !w3 || !b3 || !params_dev) return fail(HK_E_INVALID, std::string(who) + ": NULL argument");
  if (((uintptr_t)params_dev) & 15u) return fail(HK_E_INVALID, std::string(who) + ": params need 16-byte alignment");
  if ((((uintptr_t)w1) | ((uintptr_t)b1) | ((uintptr_t)w2) | ((uintptr_t)b2) | ((uintptr_t)w3) | ((uintptr_t)b3)) & 3u)
    return fail(HK_E_INVALID, std::string(who) + ": weights and biases need 4-byte alignment");
  if (int rc = deviceCheck(who, device)) return rc;
  DeviceGuard guard(device);
  using namespace hk_actor;
  k_actor_pack<<<(kParamWords + kPackThreads - 1) / kPackThreads, kPackThreads, 0, (cudaStream_t)stream>>>(w1, b1, w2, b2, w3, b3,
                                                                                                          (uint32_t*)params_dev);
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int hk_actor_pack_many(const float* actors_dev, int64_t stride_floats, int k, void* table_dev, int device, void* stream) {
  const char* who = "hk_actor_pack_many";
  if (!actors_dev || !table_dev) return fail(HK_E_INVALID, std::string(who) + ": NULL argument");
  if (k < 1 || k > hk_actor::kPoolMaxK) return fail(HK_E_INVALID, std::string(who) + ": k must be in [1, 4096]");
  if (stride_floats < hk_actor::kActorFloats) return fail(HK_E_INVALID, std::string(who) + ": stride_floats must be >= 71684");
  if (((uintptr_t)table_dev) & 15u) return fail(HK_E_INVALID, std::string(who) + ": table needs 16-byte alignment");
  if (((uintptr_t)actors_dev) & 3u) return fail(HK_E_INVALID, std::string(who) + ": actors need 4-byte alignment");
  if (int rc = deviceCheck(who, device)) return rc;
  DeviceGuard guard(device);
  using namespace hk_actor;
  const dim3 grid((kParamWords + kPackThreads - 1) / kPackThreads, (unsigned)k);
  k_actor_pack_many<<<grid, kPackThreads, 0, (cudaStream_t)stream>>>(actors_dev, (long long)stride_floats, (uint32_t*)table_dev);
  HK_CUDA(cudaGetLastError());
  return HK_OK;
}

int64_t hk_td3_arena_bytes(void) { return 4 * hk_td3::kArenaFloats; }

int64_t hk_td3_scratch_bytes(int batch) {
  if (batch < 1 || batch > hk_td3::kMaxBatch) return fail(HK_E_INVALID, "hk_td3_scratch_bytes: batch must be in [1, 1024]");
  return 4 * hk_td3::carve(nullptr, batch).floats;
}

// The cluster size of k_td3_update on `device`: 16 CTAs (non-portable) when the device can co-schedule such a cluster,
// else the portable 8.  The result does not depend on it (csrc/hk_td3.cuh).  HK_TD3_CLUSTER=n (read once) lowers the
// size to n >= 1, so that the tests can run the update at other sizes; it never raises the probed size.
static int td3Cluster(int device) {
  static int size[64] = {0};
  static const int cap = [] {
    const char* e = getenv("HK_TD3_CLUSTER");
    return e ? atoi(e) : 0;
  }();
  int& s = size[device & 63];
  if (s == 0) {
    const void* k = (const void*)hk_td3::k_td3_update;
    s = 8;
    if (cudaFuncSetAttribute(k, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
      cudaLaunchConfig_t cfg = {};
      cudaLaunchAttribute attr;
      attr.id = cudaLaunchAttributeClusterDimension;
      attr.val.clusterDim.x = hk_td3::kClusterMax;
      attr.val.clusterDim.y = attr.val.clusterDim.z = 1;
      cfg.gridDim = dim3(hk_td3::kClusterMax);
      cfg.blockDim = dim3(hk_td3::kThreads);
      cfg.attrs = &attr;
      cfg.numAttrs = 1;
      int clusters = 0;
      if (cudaOccupancyMaxActiveClusters(&clusters, k, &cfg) == cudaSuccess && clusters >= 1) s = hk_td3::kClusterMax;
    }
    cudaGetLastError();  // a refused probe leaves no sticky error
    if (cap >= 1 && cap < s) s = cap;
  }
  return s;
}

int hk_td3_cluster_size(int device) {
  if (int rc = deviceCheck("hk_td3_cluster_size", device)) return rc;
  DeviceGuard guard(device);
  return td3Cluster(device);
}

static bool finiteNonNeg(float x) { return x >= 0.0f && !std::isinf(x); }

// The ten hyper-parameters; `who` prefixes the message ("hk_td3_update" or "hk_td3_update_population: member m").
static int td3HparamsCheck(const std::string& who, const hk_td3_hparams* hp) {
  const float hv[10] = {hp->gamma, hp->tau_actor, hp->tau_critic, hp->lr_actor, hp->lr_critic, hp->wd_actor, hp->wd_critic,
                        hp->beta, hp->target_noise, hp->target_noise_clip};
  const char* hn[10] = {"gamma", "tau_actor", "tau_critic", "lr_actor", "lr_critic", "wd_actor", "wd_critic", "beta",
                        "target_noise", "target_noise_clip"};
  for (int i = 0; i < 10; ++i)
    if (!finiteNonNeg(hv[i])) return fail(HK_E_INVALID, who + ": " + hn[i] + " must be finite and >= 0");
  return HK_OK;
}

// The kernel arguments of one learner's update; the batch's idx / prio_idx are taken from `batch` as given.
static hk_td3::Args td3Args(void* arena_dev, void* scratch_dev, const hk_td3_batch* batch, int batch_size, const hk_td3_hparams* hp,
                            const float* action_low_dev, const float* action_range_dev, uint64_t seed, int do_actor, float* losses_dev) {
  hk_td3::Args a;
  a.arena = (float*)arena_dev;
  a.scratch = (float*)scratch_dev;
  a.obs = batch->obs;
  a.act = batch->action;
  a.rew = batch->reward;
  a.nobs = batch->next_obs;
  a.done = batch->done;
  a.idx = (const long long*)batch->idx;
  a.pw = batch->prio_weights;
  a.pidx = (const long long*)batch->prio_idx;
  a.pn = (long long)batch->prio_n;
  a.alow = action_low_dev;
  a.arange = action_range_dev;
  a.losses = losses_dev;
  a.seed = seed;
  a.B = batch_size;
  a.doActor = do_actor ? 1 : 0;
  a.gamma = hp->gamma;
  a.tauA = hp->tau_actor;
  a.tauC = hp->tau_critic;
  a.lrA = hp->lr_actor;
  a.lrC = hp->lr_critic;
  a.wdA = hp->wd_actor;
  a.wdC = hp->wd_critic;
  a.beta = hp->beta;
  a.sigma = hp->target_noise;
  a.clip = hp->target_noise_clip;
  return a;
}

static cudaLaunchConfig_t td3LaunchConfig(cudaLaunchAttribute* attr, int cluster, int clusters, void* stream) {
  cudaLaunchConfig_t cfg = {};
  attr->id = cudaLaunchAttributeClusterDimension;
  attr->val.clusterDim.x = (unsigned)cluster;
  attr->val.clusterDim.y = attr->val.clusterDim.z = 1;
  cfg.gridDim = dim3((unsigned)(cluster * clusters));
  cfg.blockDim = dim3(hk_td3::kThreads);
  cfg.stream = (cudaStream_t)stream;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cfg;
}

int hk_td3_update(void* arena_dev, void* scratch_dev, const hk_td3_batch* batch, int batch_size, const hk_td3_hparams* hp,
                  const float* action_low_dev, const float* action_range_dev, uint64_t seed, int do_actor, float* losses_dev,
                  int device, void* stream) {
  const std::string who = "hk_td3_update";
  if (!arena_dev || !scratch_dev || !batch || !hp || !action_low_dev || !action_range_dev || !losses_dev)
    return fail(HK_E_INVALID, who + ": NULL argument");
  if (!batch->obs || !batch->action || !batch->reward || !batch->next_obs || !batch->done || !batch->idx)
    return fail(HK_E_INVALID, who + ": NULL batch array");
  if (batch->prio_weights && !batch->prio_idx) return fail(HK_E_INVALID, who + ": NULL prio_idx with prio_weights");
  if ((((uintptr_t)arena_dev) & 15u) || (((uintptr_t)scratch_dev) & 15u))
    return fail(HK_E_INVALID, who + ": arena and scratch need 16-byte alignment");
  if ((((uintptr_t)batch->idx) & 7u) || (batch->prio_weights && (((uintptr_t)batch->prio_idx) & 7u)))
    return fail(HK_E_INVALID, who + ": idx and prio_idx need 8-byte alignment");
  if ((((uintptr_t)batch->obs) | ((uintptr_t)batch->action) | ((uintptr_t)batch->reward) | ((uintptr_t)batch->next_obs) |
       ((uintptr_t)batch->done) | ((uintptr_t)batch->prio_weights) | ((uintptr_t)action_low_dev) | ((uintptr_t)action_range_dev) |
       ((uintptr_t)losses_dev)) & 3u)
    return fail(HK_E_INVALID, who + ": float arrays need 4-byte alignment");
  if (batch_size < 1 || batch_size > hk_td3::kMaxBatch) return fail(HK_E_INVALID, who + ": batch must be in [1, 1024]");
  if (int rc = td3HparamsCheck(who, hp)) return rc;
  if (batch->prio_weights && batch->prio_n < 1) return fail(HK_E_INVALID, who + ": prio_n must be >= 1");
  if (int rc = deviceCheck(who.c_str(), device)) return rc;
  DeviceGuard guard(device);
  const hk_td3::Args a = td3Args(arena_dev, scratch_dev, batch, batch_size, hp, action_low_dev, action_range_dev, seed, do_actor, losses_dev);
  cudaLaunchAttribute attr;
  const cudaLaunchConfig_t cfg = td3LaunchConfig(&attr, td3Cluster(device), 1, stream);
  HK_CUDA(cudaLaunchKernelEx(&cfg, hk_td3::k_td3_update, a));
  return HK_OK;
}

// How many clusters of 16 and of 8 CTAs of k_td3_update_population the device keeps resident at once (probed once per
// device; 0 where the probe is refused).
static void td3PopulationOccupancy(int device, int* occ16, int* occ8) {
  static int probed[64][2] = {{0}};
  static bool done[64] = {false};
  int* p = probed[device & 63];
  if (!done[device & 63]) {
    const void* k = (const void*)hk_td3::k_td3_update_population;
    const bool nonPortable = cudaFuncSetAttribute(k, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess;
    for (int i = 0; i < 2; ++i) {
      const int size = i == 0 ? 16 : 8;
      if (size > 8 && !nonPortable) continue;
      cudaLaunchAttribute attr;
      const cudaLaunchConfig_t cfg = td3LaunchConfig(&attr, size, 1, nullptr);
      int clusters = 0;
      if (cudaOccupancyMaxActiveClusters(&clusters, k, &cfg) == cudaSuccess) p[i] = clusters;
    }
    cudaGetLastError();  // a refused probe leaves no sticky error
    done[device & 63] = true;
  }
  *occ16 = p[0];
  *occ8 = p[1];
}

// The cluster size of a population launch of k members: the largest of {16, 8} at which all k clusters are resident at
// once, else 16 (the clusters then run in waves, and 16-CTA clusters finish each wave sooner).  The result does not depend
// on it.  HK_TD3_CLUSTER (td3Cluster) caps it, for the tests.
static int td3PopulationCluster(int k, int device) {
  int occ16 = 0, occ8 = 0;
  td3PopulationOccupancy(device, &occ16, &occ8);
  return std::min(occ16 >= k ? 16 : occ8 >= k ? 8 : 16, td3Cluster(device));
}

int hk_td3_population_cluster_size(int k, int device) {
  if (k < 1 || k > hk_td3::kMaxPopulation) return fail(HK_E_INVALID, "hk_td3_population_cluster_size: k must be in [1, 64]");
  if (int rc = deviceCheck("hk_td3_population_cluster_size", device)) return rc;
  DeviceGuard guard(device);
  return td3PopulationCluster(k, device);
}

int hk_td3_update_population(void* arenas_dev, void* scratch_dev, const hk_td3_batch* batch, int batch_size, int k,
                             const hk_td3_hparams* hp, const float* const* action_low, const float* const* action_range,
                             const uint64_t* seeds, const uint8_t* do_actor, float* losses_dev, int device, void* stream) {
  const std::string who = "hk_td3_update_population";
  if (!arenas_dev || !scratch_dev || !batch || !hp || !action_low || !action_range || !seeds || !do_actor || !losses_dev)
    return fail(HK_E_INVALID, who + ": NULL argument");
  if (!batch->obs || !batch->action || !batch->reward || !batch->next_obs || !batch->done || !batch->idx)
    return fail(HK_E_INVALID, who + ": NULL batch array");
  if (batch->prio_weights && !batch->prio_idx) return fail(HK_E_INVALID, who + ": NULL prio_idx with prio_weights");
  if ((((uintptr_t)arenas_dev) & 15u) || (((uintptr_t)scratch_dev) & 15u))
    return fail(HK_E_INVALID, who + ": arenas and scratch need 16-byte alignment");
  if ((((uintptr_t)batch->idx) & 7u) || (batch->prio_weights && (((uintptr_t)batch->prio_idx) & 7u)))
    return fail(HK_E_INVALID, who + ": idx and prio_idx need 8-byte alignment");
  if ((((uintptr_t)batch->obs) | ((uintptr_t)batch->action) | ((uintptr_t)batch->reward) | ((uintptr_t)batch->next_obs) |
       ((uintptr_t)batch->done) | ((uintptr_t)batch->prio_weights) | ((uintptr_t)losses_dev)) & 3u)
    return fail(HK_E_INVALID, who + ": float arrays need 4-byte alignment");
  if (k < 1 || k > hk_td3::kMaxPopulation) return fail(HK_E_INVALID, who + ": k must be in [1, 64]");
  if (batch_size < 1 || batch_size > hk_td3::kMaxBatch) return fail(HK_E_INVALID, who + ": batch must be in [1, 1024]");
  if (batch->prio_weights && batch->prio_n < 1) return fail(HK_E_INVALID, who + ": prio_n must be >= 1");
  for (int m = 0; m < k; ++m) {
    const std::string wm = who + ": member " + std::to_string(m);
    if (!action_low[m] || !action_range[m]) return fail(HK_E_INVALID, wm + ": NULL action_low / action_range");
    if ((((uintptr_t)action_low[m]) | ((uintptr_t)action_range[m])) & 3u)
      return fail(HK_E_INVALID, wm + ": action_low / action_range need 4-byte alignment");
    if (int rc = td3HparamsCheck(wm, hp + m)) return rc;
  }
  if (int rc = deviceCheck(who.c_str(), device)) return rc;
  DeviceGuard guard(device);
  const int64_t arenaFloats = hk_td3::kArenaFloats, scratchFloats = hk_td3::carve(nullptr, batch_size).floats;
  hk_td3::PopulationArgs p;
  memset(&p, 0, sizeof(p));
  for (int m = 0; m < k; ++m) {
    hk_td3_batch bm = *batch;
    bm.idx = batch->idx + (int64_t)m * batch_size;
    if (batch->prio_weights) bm.prio_idx = batch->prio_idx + (int64_t)m * batch_size;
    p.m[m] = td3Args((float*)arenas_dev + m * arenaFloats, (float*)scratch_dev + m * scratchFloats, &bm, batch_size, hp + m,
                     action_low[m], action_range[m], seeds[m], do_actor[m], losses_dev + 2 * m);
  }
  cudaLaunchAttribute attr;
  const cudaLaunchConfig_t cfg = td3LaunchConfig(&attr, td3PopulationCluster(k, device), k, stream);
  HK_CUDA(cudaLaunchKernelEx(&cfg, hk_td3::k_td3_update_population, p));
  return HK_OK;
}

int hk_launches_per_step(const hk_env* h) { return h ? h->launches : 0; }

int hk_kernel_timing(hk_env* h, int enable) {
  if (!h) return fail(HK_E_INVALID, "hk_kernel_timing: NULL handle");
  DeviceGuard guard(h->device);
  const int total = hk_env::kTimedSteps * hk_env::kEventsPerStep;
  if (enable && !h->events) {
    h->events = new cudaEvent_t[total];
    for (int k = 0; k < total; ++k) HK_CUDA(cudaEventCreate(&h->events[k]));
  } else if (!enable && h->events) {
    for (int k = 0; k < total; ++k) cudaEventDestroy(h->events[k]);
    delete[] h->events;
    h->events = nullptr;
  }
  h->timedSteps = 0;
  return HK_OK;
}

int hk_kernel_times(hk_env* h, double* out_ms4, int64_t* steps_out) {
  if (!h || !out_ms4) return fail(HK_E_INVALID, "hk_kernel_times: NULL argument");
  if (!h->events) return fail(HK_E_INVALID, "hk_kernel_times: call hk_kernel_timing(env, 1) first");
  DeviceGuard guard(h->device);
  HK_CUDA(cudaDeviceSynchronize());
  for (int k = 0; k < 4; ++k) out_ms4[k] = 0.0;
  for (int s = 0; s < h->timedSteps; ++s)
    for (int k = 0; k < 4; ++k) {
      float ms = 0.0f;
      HK_CUDA(cudaEventElapsedTime(&ms, h->events[s * hk_env::kEventsPerStep + k], h->events[s * hk_env::kEventsPerStep + k + 1]));
      out_ms4[k] += (double)ms;
    }
  if (steps_out) *steps_out = h->timedSteps;
  h->timedSteps = 0;
  return HK_OK;
}

int hk_stats_device_ptr(hk_env* h, double** out_dev) {
  if (!h || !out_dev) return fail(HK_E_INVALID, "hk_stats_device_ptr: NULL argument");
  DeviceGuard guard(h->device);
  double* sum = h->stats + HK_STATS_DIM * kStatsRows;  // refreshed here (legacy default stream); stable address
  k_sum_stats<<<1, HK_STATS_DIM>>>(h->stats, sum);
  HK_CUDA(cudaGetLastError());
  *out_dev = sum;
  return HK_OK;
}

}  // extern "C"
#endif  // !HK_TU_INLINE (pass 1)
