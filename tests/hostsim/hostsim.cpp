// tests/hostsim/hostsim.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// Compiles the product's device headers (hockey_env_b200/csrc/*.cuh) for the HOST so that the
// non-GPU test tier can diff the kernel's per-env arithmetic against the CPU oracle bit-for-bit
// (there is no GPU in the build container).  It is not reachable from the hockey_env_b200 package
// and is never a fallback: the package fails loudly without the CUDA library.
#include <cstdio>
#include <cstring>
#include <vector>
#define HK_FAST_DEBUG 1
namespace hk { long long g_fast_bail[16]; long long g_iter_hist[2][182]; long long g_nvc_hist[16]; long long g_period_hist[16]; long long g_toi_dbg[16]; int g_dbg_left = 0; }
#include "../../include/hockey_b200.h"
#include "../../hockey_env_b200/csrc/hk_tick.cuh"

using namespace hk;

// what one env's last tick did: the WorkRecord of the tier that finished it, then that tier
enum { WORK_WORDS = 9, TIER_FAST = 0, TIER_TOUCH = 1, TIER_GENERAL = 2 };

struct HostBatch {
  Scene S;
  Config cfg;
  int64_t n, env_id_offset;
  std::vector<Env> envs;
  std::vector<uint32_t> cache;  // [27*6][n]
  double stats[HK_STATS_DIM];
  int use_fast = 0;
  long long nFast = 0, nSlow = 0, nLong = 0, nTouch = 0;
  int mid_budget = 24;
  std::vector<int32_t> work;  // [n][WORK_WORDS]: hs_last_work
  Cache cacheOf(int64_t i) { Cache c; c.base = cache.data() + i; c.stride = (size_t)n; return c; }
};

static void addStats(double* s, const TickStats& t) {
  s[0] += t.episodes; s[1] += t.wins; s[2] += t.losses; s[3] += t.draws; s[4] += t.steps;
  s[5] += t.ret1; s[6] += t.ret2; s[7] += t.ret1sq; s[8] += t.len; s[9] += t.touch1; s[10] += t.touch2;
  s[11] += t.velIters; s[12] += t.toi; s[13] += t.overflow;
}

extern "C" {
void* hs_create(int64_t n, int mode, int keep_mode, uint64_t seed, int64_t env_id_offset) {
  HostBatch* b = new HostBatch();
  scene_build::build(&b->S);
  b->cfg.mode = mode; b->cfg.keep_mode = keep_mode; b->cfg.max_timesteps = mode == 0 ? 250 : 80; b->cfg.seed = seed;
  b->n = n; b->env_id_offset = env_id_offset;
  b->envs.resize(n);
  b->cache.assign((size_t)n * 27 * 6, 0);
  b->work.assign((size_t)n * WORK_WORDS, 0);
  std::memset(b->stats, 0, sizeof(b->stats));
  for (int64_t i = 0; i < n; ++i) { std::memset(&b->envs[i], 0, sizeof(Env)); envCreate(b->S, b->cfg, b->envs[i], (uint64_t)(env_id_offset + i)); }
  return b;
}
void hs_destroy(void* h) { delete (HostBatch*)h; }
void hs_reset(void* h, const uint8_t* mask, const int8_t* one_starting, float* obs) {
  HostBatch* b = (HostBatch*)h;
  for (int64_t i = 0; i < b->n; ++i) {
    if (mask && !mask[i]) continue;
    envReset(b->S, b->cfg, b->envs[i], (uint64_t)(b->env_id_offset + i), one_starting ? (int)one_starting[i] : -1);
    if (obs) getObs(b->envs[i], obs + 18 * i);
  }
}
void hs_reset_seeded(void* h, const uint8_t* mask, const int8_t* one_starting, const int64_t* seeds, float* obs) {
  HostBatch* b = (HostBatch*)h;
  for (int64_t i = 0; i < b->n; ++i) {
    if (mask && !mask[i]) continue;
    envReset(b->S, b->cfg, b->envs[i], (uint64_t)(b->env_id_offset + i), one_starting ? (int)one_starting[i] : -1, seeds ? seeds[i] : -1);
    if (obs) getObs(b->envs[i], obs + 18 * i);
  }
}
void hs_step(void* h, const float* action, int stride, int pol1, int pol2, int flags, float* obs, float* obs2, float* reward,
             float* reward2, uint8_t* done, float* info, float* info2, float* final_obs) {
  HostBatch* b = (HostBatch*)h;
  StepIO io; io.action = action; io.stride = stride; io.pol1 = pol1; io.pol2 = pol2; io.pol2v = nullptr; io.flags = flags; io.obs = obs; io.obs2 = obs2;
  io.reward = reward; io.reward2 = reward2; io.done = done; io.info = info; io.info2 = info2; io.final_obs = final_obs; io.write = 1; io.actBuf = nullptr; io.stageRows = 0; io.waitFlag = nullptr; io.waitValue = 0;
  for (int64_t i = 0; i < b->n; ++i) {
    // round-trip through the HBM group layout exactly as the kernel does
    F4 g[CORE_GROUPS];
    envToGroups(b->envs[i], g);
    Env e;
    groupsToEnv(g, e);
    TickStats st; tickStatsZero(st);
    int tier = TIER_GENERAL;
    std::memset(&g_work, 0, sizeof(g_work));  // every attempt starts a fresh record: the one that finishes the tick keeps it
    bool done_fast = false;
    int bail = 15;
    if (b->use_fast) {
      Env w = e;
      TickStats st2; tickStatsZero(st2);
      if (envTickFast(b->S, b->cfg, w, (uint64_t)(b->env_id_offset + i), (size_t)i, io, true, st2)) { e = w; st = st2; done_fast = true; tier = TIER_FAST; }
      else bail = w.bailKind;
    }
    bool done_touch = false;
    if (b->use_fast && !done_fast && bailClass(bail) == 0) {  // the touch tier (k_touch) takes work class 0 first
      Env w = e;
      TickStats st2; tickStatsZero(st2);
      std::memset(&g_work, 0, sizeof(g_work));
      if (envTickTouch(b->S, b->cfg, b->cacheOf(i), w, (uint64_t)(b->env_id_offset + i), (size_t)i, io, true, st2, nullptr)) { e = w; st = st2; done_touch = true; tier = TIER_TOUCH; }
    }
    if (done_fast) b->nFast++;
    else if (done_touch) b->nTouch++;
    else if (b->use_fast) {
      // the kernel cascade: budgeted middle tier, then the unlimited tier, each from the stored state
      Env w = e;
      TickStats st2; tickStatsZero(st2);
      std::memset(&g_work, 0, sizeof(g_work));
      if (envTick(b->S, b->cfg, b->cacheOf(i), w, (uint64_t)(b->env_id_offset + i), (size_t)i, io, true, st2, b->mid_budget, false)) { e = w; st = st2; b->nSlow++; }
      else { b->nLong++; std::memset(&g_work, 0, sizeof(g_work)); envTick(b->S, b->cfg, b->cacheOf(i), e, (uint64_t)(b->env_id_offset + i), (size_t)i, io, true, st); }
    } else { b->nSlow++; envTick(b->S, b->cfg, b->cacheOf(i), e, (uint64_t)(b->env_id_offset + i), (size_t)i, io, true, st); }
    b->envs[i] = e;
    addStats(b->stats, st);
    const int32_t rec[WORK_WORDS] = {g_work.kind, g_work.shape, g_work.sweeps, g_work.toi, g_work.maxSub, g_work.skipAfter, g_work.events, g_work.goal, tier};
    std::memcpy(&b->work[(size_t)i * WORK_WORDS], rec, sizeof(rec));
  }
}
void hs_bail_counts(long long* out) { for (int i = 0; i < 16; ++i) out[i] = hk::g_fast_bail[i]; }
void hs_iter_hist(long long* out) { for (int w = 0; w < 2; ++w) for (int i = 0; i < 182; ++i) out[w * 182 + i] = hk::g_iter_hist[w][i]; for (int i = 0; i < 16; ++i) out[364 + i] = hk::g_period_hist[i]; }
// [n][9] int32 of each env's last tick: island solve kind and shape (contacts | points << 4), sweeps, TOI events, highest sub-step count, TOI evaluations
// skipped after an event, event bodies (1: puck, 2: racket), goal, tier that finished it (0 fast, 1 touch, 2 general)
void hs_last_work(void* h, int32_t* out) { HostBatch* b = (HostBatch*)h; std::memcpy(out, b->work.data(), b->work.size() * sizeof(int32_t)); }
void hs_toi_dbg(long long* out) { for (int i = 0; i < 16; ++i) out[i] = hk::g_toi_dbg[i]; }
void hs_set_fast(void* h, int on) { ((HostBatch*)h)->use_fast = on; }
void hs_fast_counts(void* h, long long* out) { out[0] = ((HostBatch*)h)->nFast; out[1] = ((HostBatch*)h)->nSlow; out[2] = ((HostBatch*)h)->nLong; out[3] = ((HostBatch*)h)->nTouch; }
void hs_set_mid_budget(void* h, int b) { ((HostBatch*)h)->mid_budget = b; }
void hs_get_obs(void* h, float* obs, float* obs2) {
  HostBatch* b = (HostBatch*)h;
  for (int64_t i = 0; i < b->n; ++i) { if (obs) getObs(b->envs[i], obs + 18 * i); if (obs2) getObs2(b->envs[i], obs2 + 18 * i); }
}
void hs_get_state(void* h, uint32_t* rec) {
  HostBatch* b = (HostBatch*)h;
  for (int64_t i = 0; i < b->n; ++i) packRecord(b->envs[i], b->cacheOf(i), rec + (size_t)HK_STATE_WORDS * i);
}
void hs_set_state(void* h, const uint32_t* rec) {
  HostBatch* b = (HostBatch*)h;
  for (int64_t i = 0; i < b->n; ++i) unpackRecord(rec + (size_t)HK_STATE_WORDS * i, b->envs[i], b->cacheOf(i));
}
void hs_set_obs_state(void* h, const float* obs18) {
  HostBatch* b = (HostBatch*)h;
  for (int64_t i = 0; i < b->n; ++i) setObsState(b->S, b->envs[i], obs18 + 18 * i, b->cfg.keep_mode);
}
void hs_get_stats(void* h, double* out) { std::memcpy(out, ((HostBatch*)h)->stats, sizeof(double) * HK_STATS_DIM); }
void hs_clear_stats(void* h) { std::memset(((HostBatch*)h)->stats, 0, sizeof(double) * HK_STATS_DIM); }
void hs_scene(void* h, void* out, int64_t nbytes) { std::memcpy(out, &((HostBatch*)h)->S, (size_t)nbytes < sizeof(Scene) ? (size_t)nbytes : sizeof(Scene)); }
int64_t hs_scene_size() { return (int64_t)sizeof(Scene); }
}
