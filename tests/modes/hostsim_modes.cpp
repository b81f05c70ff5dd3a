// tests/modes/hostsim_modes.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// The host build of the device code (tests/hostsim/hostsim.cpp) with per-env game modes: every reset of env i -- masked
// or automatic -- reads the caller's code table like hk_set_reset_modes, and the state record carries word HK_S_MODE
// as hk_get_state / hk_set_state write and read it.  The tier cascade of a tick is the one hs_step emulates.
#include <unordered_map>
#include "../hostsim/hostsim.cpp"

namespace {
std::unordered_map<const void*, const uint8_t*> g_reset_modes;  // batch -> caller-owned codes (null: keep)
const uint8_t* modesOf(const void* h) {
  auto it = g_reset_modes.find(h);
  return it == g_reset_modes.end() ? nullptr : it->second;
}
}  // namespace

extern "C" {
void hsm_set_reset_modes(void* h, const uint8_t* modes) { g_reset_modes[h] = modes; }
void hsm_destroy(void* h) {
  g_reset_modes.erase(h);
  hs_destroy(h);
}
void hsm_get_modes(void* h, uint8_t* modes) {
  HostBatch* b = (HostBatch*)h;
  for (int64_t i = 0; i < b->n; ++i) modes[i] = (uint8_t)b->envs[i].mode;
}
void hsm_reset_seeded(void* h, const uint8_t* mask, const int8_t* one_starting, const int64_t* seeds, float* obs) {
  HostBatch* b = (HostBatch*)h;
  const uint8_t* modes = modesOf(h);
  for (int64_t i = 0; i < b->n; ++i) {
    if (mask && !mask[i]) continue;
    envReset(b->S, b->cfg, b->envs[i], (uint64_t)(b->env_id_offset + i), one_starting ? (int)one_starting[i] : -1,
             seeds ? seeds[i] : -1, modes ? (int)modes[i] : -1);
    if (obs) getObs(b->envs[i], obs + 18 * i);
  }
}
void hsm_step(void* h, const float* action, int stride, int pol1, int pol2, int flags, float* obs, float* obs2, float* reward,
              float* reward2, uint8_t* done, float* info, float* info2, float* final_obs) {
  HostBatch* b = (HostBatch*)h;
  StepIO io; io.action = action; io.stride = stride; io.pol1 = pol1; io.pol2 = pol2; io.pol2v = nullptr; io.flags = flags; io.obs = obs; io.obs2 = obs2;
  io.reward = reward; io.reward2 = reward2; io.done = done; io.info = info; io.info2 = info2; io.final_obs = final_obs; io.write = 1; io.actBuf = nullptr; io.stageRows = 0; io.waitFlag = nullptr; io.waitValue = 0;
  io.resetModes = modesOf(h);
  for (int64_t i = 0; i < b->n; ++i) {
    const uint64_t id = (uint64_t)(b->env_id_offset + i);
    F4 g[CORE_GROUPS];  // round-trip through the HBM group layout exactly as the kernel does
    envToGroups(b->envs[i], g);
    Env e;
    groupsToEnv(g, e);
    TickStats st; tickStatsZero(st);
    bool done_fast = false, done_touch = false;
    int bail = 15;
    if (b->use_fast) {
      Env w = e;
      TickStats st2; tickStatsZero(st2);
      if (envTickFast(b->S, b->cfg, w, id, (size_t)i, io, true, st2)) { e = w; st = st2; done_fast = true; }
      else bail = w.bailKind;
    }
    if (b->use_fast && !done_fast && bailClass(bail) == 0) {  // the touch tier takes work class 0 first
      Env w = e;
      TickStats st2; tickStatsZero(st2);
      if (envTickTouch(b->S, b->cfg, b->cacheOf(i), w, id, (size_t)i, io, true, st2, nullptr)) { e = w; st = st2; done_touch = true; }
    }
    if (!done_fast && !done_touch) {
      if (b->use_fast) {  // budgeted tier, then the unlimited tier, each from the stored state
        Env w = e;
        TickStats st2; tickStatsZero(st2);
        if (envTick(b->S, b->cfg, b->cacheOf(i), w, id, (size_t)i, io, true, st2, b->mid_budget, false)) { e = w; st = st2; }
        else envTick(b->S, b->cfg, b->cacheOf(i), e, id, (size_t)i, io, true, st);
      } else {
        envTick(b->S, b->cfg, b->cacheOf(i), e, id, (size_t)i, io, true, st);
      }
    }
    b->envs[i] = e;
    addStats(b->stats, st);
  }
}
void hsm_get_state(void* h, uint32_t* rec) {
  HostBatch* b = (HostBatch*)h;
  for (int64_t i = 0; i < b->n; ++i) {
    uint32_t* r = rec + (size_t)HK_STATE_WORDS * i;
    packRecord(b->envs[i], b->cacheOf(i), r);
    r[HK_S_MODE] = modeWord(b->envs[i], b->cfg.mode);
  }
}
void hsm_set_state(void* h, const uint32_t* rec) {
  HostBatch* b = (HostBatch*)h;
  for (int64_t i = 0; i < b->n; ++i) {
    const uint32_t* r = rec + (size_t)HK_STATE_WORDS * i;
    unpackRecord(r, b->envs[i], b->cacheOf(i));
    b->envs[i].mode = modeOfWord(r[HK_S_MODE], b->cfg.mode);
  }
}
}
