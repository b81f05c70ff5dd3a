// hk_tick.cuh -- one full env tick as the kernels run it: policy -> step -> info/reward ->
// outputs -> auto-reset.  This is the body of HockeyEnv.step / HockeyEnv_BasicOpponent.step
// (reference hockey_env.py:658-695, :882-886) plus the batched API's auto-reset.
#pragma once
#include "hk_state.cuh"
#include "hk_fast.cuh"

namespace hk {

struct StepIO {
  const float* action;  // [n, stride] or null
  int stride;
  int pol1, pol2, flags;
  const uint8_t* pol2v;  // per-env player-2 policy codes (HK_POLICY_PER_ENV) or null
  const uint8_t* resetModes = nullptr;  // per-env HK_MODE_* of the episode an auto-reset starts (hk_set_reset_modes) or null: keep
  float* obs;        // [n,18]
  float* obs2;       // [n,18] or null
  float* reward;     // [n] or null
  float* reward2;    // [n] or null
  uint8_t* done;     // [n] or null
  float* info;       // [n,4] or null
  float* info2;      // [n,4] or null
  float* final_obs;  // [n,18] or null
  int write;         // 0: suppress all per-tick outputs (inner ticks of hk_rollout)
  float* actBuf;     // [n,8] scratch: clipped actions k_fast computed for the envs it hands to the general tiers
  int stageRows;     // k_fast: write obs / final_obs rows warp-cooperatively (needs 16-byte aligned row tensors)
  const uint32_t* waitFlag;  // general tier (hk_step_host): outputs may be written once *waitFlag == waitValue
  uint32_t waitValue;        //   (the DMA of the fast tier's rows into the same host record has finished)
};

HK_HD int pol2Of(const StepIO& io, size_t i) { return io.pol2v ? (int)io.pol2v[i] : io.pol2; }

struct TickStats {
  int episodes, wins, losses, draws, steps, len, touch1, touch2, velIters, toi, overflow;
  double ret1, ret2, ret1sq;
};
HK_HD void tickStatsZero(TickStats& s) {
  s.episodes = s.wins = s.losses = s.draws = s.steps = s.len = s.touch1 = s.touch2 = s.velIters = s.toi = s.overflow = 0;
  s.ret1 = s.ret2 = s.ret1sq = 0.0;
}

HK_HD void writeRow18(float* dst, const float* o) {
  // rows are 72 B: 8-byte aligned, so 9 float2 stores
  for (int k = 0; k < 9; ++k) {
#if defined(__CUDA_ARCH__)
    __stcs(reinterpret_cast<float2*>(dst) + k, make_float2(o[2 * k], o[2 * k + 1]));  // streaming: outputs are not re-read by the kernels
#else
    dst[2 * k] = o[2 * k];
    dst[2 * k + 1] = o[2 * k + 1];
#endif
  }
}

HK_HD void writeRow4(float* dst, float a, float b, float c, float d) {  // info rows are 16 B: one 128-bit store
#if defined(__CUDA_ARCH__)
  __stcs(reinterpret_cast<float4*>(dst), make_float4(a, b, c, d));
#else
  dst[0] = a; dst[1] = b; dst[2] = c; dst[3] = d;
#endif
}

// A warp's 32 observation rows (32 x 72 B = 2304 contiguous bytes when its envs are consecutive) staged in shared
// memory as [lane][18] floats and written with 128-bit stores that cover the span front to back: 4.5 fully coalesced
// 512-byte warp stores instead of nine 8-byte stores per lane at a 72-byte lane stride.  `mask` = lanes whose rows are
// to be written; a float4 that straddles two rows (18 floats per row) degrades to the valid 8-byte half.  dst must be
// 16-byte aligned (it is the row of a warp's first env: 2304 * k bytes into a 16-byte aligned tensor).
#if defined(__CUDACC__)
__device__ __forceinline__ void warpStoreRows18(float* __restrict__ dst, const float* __restrict__ stage, unsigned mask) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int r = 0; r < 5; ++r) {
    const int j = r * 32 + lane;  // float4 index within the warp's span of 144 float4
    if (j < 144) {
      const bool lo = (mask >> ((4 * j) / 18)) & 1u, hi = (mask >> ((4 * j + 2) / 18)) & 1u;
      const float4 v = reinterpret_cast<const float4*>(stage)[j];
      if (lo && hi) __stcs(reinterpret_cast<float4*>(dst) + j, v);
      else if (lo) __stcs(reinterpret_cast<float2*>(dst) + 2 * j, make_float2(v.x, v.y));
      else if (hi) __stcs(reinterpret_cast<float2*>(dst) + 2 * j + 1, make_float2(v.z, v.w));
    }
  }
}
#endif

// everything after the physics of a tick: info/reward, outputs, statistics, auto-reset
// `write` = false suppresses all per-tick outputs (fused rollout, all but the last tick).
// deferRows != null (k_fast): the caller writes the obs row (and the final_obs row unless this env was reset here)
// warp-cooperatively after the call; *deferRows is set when this call already wrote the env's terminal final_obs row.
HK_NI_FASTA void tickFinish(const Scene& S, const Config& cfg, Env& e, uint64_t env_id, size_t i, const StepIO& io, bool write,
                      TickStats& st, int had1, int had2, bool* deferRows = nullptr) {
  double inf[4], inf2[4];
  getInfo(e, false, inf);
  getInfo(e, true, inf2);
  const double cr = computeReward(e);
  const double r = cr + inf[1];
  const double r2 = -cr + inf2[1];
  e.ret[0] += r;
  e.ret[1] += r2;
  st.steps += 1;
  st.velIters += (int)e.nVelIters;
  st.toi += (int)e.nToiEvents;
  st.overflow += (int)e.nOverflow;
  e.nVelIters = e.nToiEvents = e.nOverflow = 0;
  if (e.has1 == HK_MAX_TIME_KEEP_PUCK && had1 != HK_MAX_TIME_KEEP_PUCK) st.touch1 += 1;
  if (e.has2 == HK_MAX_TIME_KEEP_PUCK && had2 != HK_MAX_TIME_KEEP_PUCK) st.touch2 += 1;
  const bool resetNow = e.done && (io.flags & 1);
  if (deferRows) *deferRows = false;
  if (write) {
    if (io.reward) io.reward[i] = (float)r;
    if (io.reward2) io.reward2[i] = (float)r2;
    if (io.done) io.done[i] = e.done ? 1 : 0;
    if (io.info) writeRow4(io.info + 4 * i, (float)inf[0], (float)inf[1], (float)inf[2], (float)inf[3]);
    if (io.info2) writeRow4(io.info2 + 4 * i, (float)inf2[0], (float)inf2[1], (float)inf2[2], (float)inf2[3]);
    if (io.final_obs && (!deferRows || resetNow)) {
      float o[18];
      getObs(e, o);
      writeRow18(io.final_obs + 18 * i, o);
      if (deferRows) *deferRows = true;
    }
  }
  if (resetNow) {
    st.episodes += 1;
    if (e.winner == 1) st.wins += 1;
    else if (e.winner == -1) st.losses += 1;
    else st.draws += 1;
    st.ret1 += e.ret[0];
    st.ret2 += e.ret[1];
    st.ret1sq += e.ret[0] * e.ret[0];
    st.len += e.time;
    envReset(S, cfg, e, env_id, -1, -1, io.resetModes ? (int)io.resetModes[i] : -1);
  }
  if (write) {
    float o[18];
    if (io.obs && !deferRows) {
      getObs(e, o);
      writeRow18(io.obs + 18 * i, o);
    }
    if (io.obs2) {
      getObs2(e, o);
      writeRow18(io.obs2 + 18 * i, o);
    }
  }
}

// general tick.  sweepBudget / allowToiEvents are the budgets of the calling tier (unlimited: 1<<20, true);
// returns false -- with nothing committed -- if a budget ran out (the next tier redoes the tick from the stored state)
HK_HD bool envTick(const Scene& S, const Config& cfg, const Cache& cache, Env& e, uint64_t env_id, size_t i,
                   const StepIO& io, bool write, TickStats& st, int sweepBudget = 1 << 20, bool allowToiEvents = true) {
  float a[8];
  policyActions(cfg, e, env_id, io.action ? io.action + (size_t)io.stride * i : nullptr, io.pol1, pol2Of(io, i), a);
  const int had1 = e.has1, had2 = e.has2;
  e.sweepBudget = sweepBudget;
  e.allowToiEvents = allowToiEvents;
  e.aborted = false;
  envStep(S, cfg, cache, e, a);
  if (e.aborted) return false;
  tickFinish(S, cfg, e, env_id, i, io, write, st, had1, had2);
  return true;
}

// fast tick: returns false (e unusable, nothing written) if the env needs the general path this tick
HK_HD bool envTickFast(const Scene& S, const Config& cfg, Env& e, uint64_t env_id, size_t i, const StepIO& io,
                       bool write, TickStats& st, bool* deferRows = nullptr) {
  float a[8];
  policyActions(cfg, e, env_id, io.action ? io.action + (size_t)io.stride * i : nullptr, io.pol1, pol2Of(io, i), a);
  const int had1 = e.has1, had2 = e.has2;
  if (!envStepFast(S, cfg, e, a)) {
    if (io.actBuf) {  // the general tier redoes the tick from the stored state; spare it the controllers
      for (int k = 0; k < 8; ++k) io.actBuf[8 * i + k] = a[k];
    }
    return false;
  }
  tickFinish(S, cfg, e, env_id, i, io, write, st, had1, had2, deferRows);
  return true;
}

// touch-tier tick (hk_fast.cuh worldStepTouch).  `pre` = this tick's clipped actions if the fast tier already ran the
// controllers (then only their phase side effect is applied), else null.  Returns false -- nothing committed, e
// unusable -- if the env needs the general path.
HK_HD bool envTickTouch(const Scene& S, const Config& cfg, const Cache& cache, Env& e, uint64_t env_id, size_t i,
                        const StepIO& io, bool write, TickStats& st, const float* pre) {
  float a[8];
  if (pre) {
    for (int k = 0; k < 8; ++k) a[k] = pre[k];
    policyAdvancePhases(cfg, e, env_id, io.pol1, pol2Of(io, i));
  } else {
    policyActions(cfg, e, env_id, io.action ? io.action + (size_t)io.stride * i : nullptr, io.pol1, pol2Of(io, i), a);
  }
  const int had1 = e.has1, had2 = e.has2;
  if (!envStepTouch(S, cfg, cache, e, a)) return false;
  tickFinish(S, cfg, e, env_id, i, io, write, st, had1, had2);
  return true;
}

// HockeyEnv.__init__ for one env (hockey_env.py:91-155): phases of the built-in controllers
// (BasicOpponent.__init__, :785), then reset(one_starting=True)
HK_HD void envCreate(const Scene& S, const Config& cfg, Env& e, uint64_t env_id) {
  e.has1 = e.has2 = 0;
  e.one_starts = true;
  e.mode = cfg.mode;
  e.episode = 0;
  e.tick = 0;
  e.nVelIters = e.nToiEvents = e.nOverflow = 0;
  e.sweepBudget = 1 << 20;
  e.allowToiEvents = true;
  e.aborted = false;
  e.dbgEvalClk = e.dbgEventClk = 0;
  e.toiPreFlag = 0;
  e.enabled = 0xFFFFFFFFu;
  e.nmf = 0;
  U4 r = philox(cfg.seed, env_id, 0, HK_STREAM_PHASE0);
  e.phase[0] = 0.0 + (3.14159265358979323846 - 0.0) * u53(r.x, r.y);
  e.phase[1] = 0.0 + (3.14159265358979323846 - 0.0) * u53(r.z, r.w);
  envReset(S, cfg, e, env_id, 1);
}

}  // namespace hk
