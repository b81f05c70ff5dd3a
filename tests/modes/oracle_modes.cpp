// tests/modes/oracle_modes.cpp -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// The CPU oracle (oracle/hockey_oracle.cpp, unchanged) with per-env game modes, the way a user of the reference sets
// them: `env.mode = m` before `env.reset()` (hockey_env.py:754-779, 357-364).  The oracle's own reset already keeps
// mode and max_timesteps per env object; this harness only sets an env's mode from the caller's code table before each
// of its resets (masked or automatic), and adds record word HK_S_MODE under the rule of include/hockey_b200.h.
#include <unordered_map>
#include "../../oracle/hockey_oracle.cpp"

namespace {
struct Modes {
  int create_mode;
  const uint8_t* reset_modes;  // caller-owned, read by every later reset (null: keep)
};
std::unordered_map<const void*, Modes> g_modes;

void chooseMode(const void* h, Env* e, size_t i) {
  const uint8_t* m = g_modes[h].reset_modes;
  if (m) e->mode = m[i];
}
}  // namespace

extern "C" {
void* hkm_create(int64_t n, int mode, int keep_mode, uint64_t seed, int64_t env_id_offset) {
  void* h = hko_create(n, mode, keep_mode, seed, env_id_offset, 1);
  g_modes[h] = Modes{mode, nullptr};
  return h;
}
void hkm_destroy(void* h) {
  g_modes.erase(h);
  hko_destroy(h);
}
void hkm_set_reset_modes(void* h, const uint8_t* modes) { g_modes[h].reset_modes = modes; }
void hkm_get_modes(void* h, uint8_t* modes) {
  Batch* b = (Batch*)h;
  for (size_t i = 0; i < b->envs.size(); ++i) modes[i] = (uint8_t)b->envs[i]->mode;
}
void hkm_reset_seeded(void* h, const uint8_t* mask, const int8_t* one_starting, const int64_t* seeds, float* obs) {
  Batch* b = (Batch*)h;
  for (size_t i = 0; i < b->envs.size(); ++i) {
    if (mask && !mask[i]) continue;
    Env* e = b->envs[i];
    chooseMode(h, e, i);
    e->reset_seed = seeds ? seeds[i] : -1;
    e->reset(one_starting ? (int)one_starting[i] : -1);
    e->reset_seed = -1;
    if (obs) e->getObs(obs + 18 * i);
  }
}
// hko_step (stepRange) with the mode of each auto-reset taken from the code table
void hkm_step(void* h, const float* action, int stride, int pol1, int pol2, int flags, float* obs, float* obs2,
              double* reward, double* reward2, uint8_t* done, double* info, double* info2, float* final_obs) {
  Batch* b = (Batch*)h;
  double* stats = b->stats;
  for (size_t i = 0; i < b->envs.size(); ++i) {
    Env* e = b->envs[i];
    float a[8];
    actionsFor(e, action ? action + (size_t)stride * i : nullptr, stride, pol1, pol2, a);
    double r, inf[4], inf2[4];
    int had1 = e->has1, had2 = e->has2;
    e->step(a, nullptr, &r, inf);
    e->getInfo(inf2, true);
    double r2 = -e->computeReward() + inf2[1];
    e->ret[0] += r;
    e->ret[1] += r2;
    stats[4] += 1;
    if (e->has1 == MAX_TIME_KEEP_PUCK && had1 != MAX_TIME_KEEP_PUCK) stats[9] += 1;
    if (e->has2 == MAX_TIME_KEEP_PUCK && had2 != MAX_TIME_KEEP_PUCK) stats[10] += 1;
    if (reward) reward[i] = r;
    if (reward2) reward2[i] = r2;
    if (done) done[i] = e->done ? 1 : 0;
    if (info) std::memcpy(info + 4 * i, inf, sizeof(inf));
    if (info2) std::memcpy(info2 + 4 * i, inf2, sizeof(inf2));
    if (final_obs) e->getObs(final_obs + 18 * i);
    if (e->done && (flags & HK_STEP_AUTORESET)) {
      stats[0] += 1;
      if (e->winner == 1) stats[1] += 1; else if (e->winner == -1) stats[2] += 1; else stats[3] += 1;
      stats[5] += e->ret[0];
      stats[6] += e->ret[1];
      stats[7] += e->ret[0] * e->ret[0];
      stats[8] += e->time;
      chooseMode(h, e, i);
      e->reset(-1);
    }
    if (obs) e->getObs(obs + 18 * i);
    if (obs2) e->getObs2(obs2 + 18 * i);
  }
}
void hkm_get_state(void* h, uint32_t* rec) {
  Batch* b = (Batch*)h;
  const int create = g_modes[h].create_mode;
  for (size_t i = 0; i < b->envs.size(); ++i) {
    uint32_t* r = rec + (size_t)HK_STATE_WORDS * i;
    packState(b->envs[i], r);
    r[HK_S_MODE] = b->envs[i]->mode == create ? 0u : (uint32_t)b->envs[i]->mode + 1u;
  }
}
void hkm_set_state(void* h, const uint32_t* rec) {
  Batch* b = (Batch*)h;
  const int create = g_modes[h].create_mode;
  for (size_t i = 0; i < b->envs.size(); ++i) {
    const uint32_t* r = rec + (size_t)HK_STATE_WORDS * i;
    unpackState(b->envs[i], r);
    const uint32_t w = r[HK_S_MODE];
    Env* e = b->envs[i];
    e->mode = w >= 1u && w <= 3u ? (int)w - 1 : create;
    e->max_timesteps = e->mode == HK_MODE_NORMAL ? 250 : 80;  // what reset() sets for this mode (hockey_env.py:357-364)
  }
}
}
