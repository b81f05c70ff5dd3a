// hk_env.cuh -- the HockeyEnv game logic around the world step, one env per thread.
// Mirrors the reference's gym-facing semantics (hockey/hockey_env.py; line cites per function),
// including its float32/float64 mix: Box2D-side values are float32, the numpy/Python side is float64
// under NumPy-2 scalar rules.
#pragma once
#include "hk_world.cuh"

namespace hk {

// reference constants (hockey_env.py:17-37)
#define HK_FPS 50
#define HK_SCALE 60.0
#define HK_W (600 / HK_SCALE)
#define HK_H (480 / HK_SCALE)
#define HK_CENTER_X (HK_W / 2)
#define HK_CENTER_Y (HK_H / 2)
#define HK_ZONE (HK_W / 20)
#define HK_MAX_ANGLE (3.14159265358979323846 / 3)
#define HK_MAX_TIME_KEEP_PUCK 15
#define HK_GOAL_SIZE 75.0
#define HK_FORCEMULTIPLIER 6000
#define HK_SHOOTFORCEMULTIPLIER 60
#define HK_TORQUEMULTIPLIER 400
#define HK_MAX_PUCK_SPEED 25.0

// _check_boundaries (hockey_env.py:420-434)
HK_HD void checkBoundaries(double force[2], Body& player, bool is_one) {
  double px = player.p.x, py = player.p.y;
  if ((is_one && px < HK_W / 2 - 210 / HK_SCALE && force[0] < 0) || (!is_one && px > HK_W / 2 + 210 / HK_SCALE && force[0] > 0) ||
      (is_one && px > HK_W / 2 && force[0] > 0) || (!is_one && px < HK_W / 2 && force[0] < 0)) {
    player.v.x = 0;  // `player.linearVelocity[0] = 0` writes through the SWIG reference proxy
    force[0] = -(double)player.v.x;
  }
  if ((py > HK_H - 1.2 && force[1] > 0) || (py < 1.2 && force[1] < 0)) {
    player.v.y = 0;
    force[1] = -(double)player.v.y;
  }
}

// _apply_translation_action_with_max_speed (hockey_env.py:436-470), max_speed = 10
HK_NI_FASTA void applyTranslation(const Scene& S, Body& player, int bi, float a0, float a1, bool is_one) {
  const double timeStep = 1.0 / HK_FPS;
  const double max_speed = 10;
  double vel0 = (double)player.v.x, vel1 = (double)player.v.y;
  double speed = sqrt(vel0 * vel0 + vel1 * vel1);
  float force[2];
  if (is_one) {
    force[0] = a0 * (float)HK_FORCEMULTIPLIER;
    force[1] = a1 * (float)HK_FORCEMULTIPLIER;
  } else {
    force[0] = (-a0) * (float)HK_FORCEMULTIPLIER;
    force[1] = (-a1) * (float)HK_FORCEMULTIPLIER;
  }
  double px = player.p.x, vx = player.v.x, mass = S.mass[bi];
  if ((is_one && px > HK_CENTER_X - HK_ZONE) || (!is_one && px < HK_CENTER_X + HK_ZONE)) {
    force[0] = 0;
    if (is_one) {
      if (vx > 0) force[0] = (float)(-2 * vx * mass / timeStep);
      force[0] += (float)(-1 * (px - HK_CENTER_X) * vx * mass / timeStep);
    } else {
      if (vx < 0) force[0] = (float)(-2 * vx * mass / timeStep);
      force[0] += (float)(1 * (px - HK_CENTER_X) * vx * mass / timeStep);
    }
    player.ldamp = 20.0f;
    double f[2] = {force[0], force[1]};
    checkBoundaries(f, player, is_one);
    applyForceToCenter(player, mk((float)f[0], (float)f[1]));
    return;
  }
  if (speed < max_speed) {
    player.ldamp = 5.0f;
    double f[2] = {force[0], force[1]};
    checkBoundaries(f, player, is_one);
    applyForceToCenter(player, mk((float)f[0], (float)f[1]));
  } else {
    player.ldamp = 20.0f;
    float ts = (float)timeStep, m32 = S.mass[bi];
    float dv0 = (ts * force[0]) / m32, dv1 = (ts * force[1]) / m32;
    double n0 = vel0 + (double)dv0, n1 = vel1 + (double)dv1;
    if (sqrt(n0 * n0 + n1 * n1) < speed) {
      double f[2] = {force[0], force[1]};
      checkBoundaries(f, player, is_one);
      applyForceToCenter(player, mk((float)f[0], (float)f[1]));
    }
  }
}

// _apply_rotation_action_with_max_speed (hockey_env.py:472-483)
HK_NI_FASTA void applyRotation(const Scene& S, Body& player, int bi, float action) {
  const double timeStep = 1.0 / HK_FPS;
  double angle = player.a;
  double torque = (double)(action * (float)HK_TORQUEMULTIPLIER);
  if (fabs(angle) > HK_MAX_ANGLE) {
    torque = 0;
    if (angle * (double)player.w > 0) torque = -0.1 * (double)player.w * (double)S.mass[bi] / timeStep;
    torque += -0.1 * angle * (double)S.mass[bi] / timeStep;
    player.adamp = 10.0f;
  } else {
    player.adamp = 2.0f;
  }
  applyTorque(player, (float)torque);
}

// _keep_puck / _shoot (hockey_env.py:618-633)
HK_HD void keepPuck(const Scene& S, Env& e, const Body& player) {
  setTransformPuck(S, e, player.p);
  setLinearVelocity(e.b[B_PUCK], player.v);
}
HK_NI_RARE void shoot(const Scene& S, Env& e, const Body& player, bool is_one) {
  Body& puck = e.b[B_PUCK];
  double s, c;
  sincos_poly((double)player.a, &s, &c);
  double sgn = is_one ? 1.0 : -1.0;
  V2 f = mk((float)(c * sgn), (float)(s * sgn));
  f = mk(f.x * S.mass[B_PUCK], f.y * S.mass[B_PUCK]);
  float ts = (float)(1.0 / HK_FPS);
  f = mk(f.x / ts, f.y / ts);
  f = mk(f.x * (float)HK_SHOOTFORCEMULTIPLIER, f.y * (float)HK_SHOOTFORCEMULTIPLIER);
  applyForceToCenter(puck, f);
}

// _get_obs / obs_agent_two (hockey_env.py:485-516)
HK_HD void getObs(const Env& e, float* o) {
  const Body &p1 = e.b[B_R1], &p2 = e.b[B_R2], &pk = e.b[B_PUCK];
  const float cx = (float)HK_CENTER_X, cy = (float)HK_CENTER_Y;
  o[0] = p1.p.x - cx; o[1] = p1.p.y - cy; o[2] = p1.a; o[3] = p1.v.x; o[4] = p1.v.y; o[5] = p1.w;
  o[6] = p2.p.x - cx; o[7] = p2.p.y - cy; o[8] = p2.a; o[9] = p2.v.x; o[10] = p2.v.y; o[11] = p2.w;
  o[12] = pk.p.x - cx; o[13] = pk.p.y - cy; o[14] = pk.v.x; o[15] = pk.v.y;
  o[16] = (float)e.has1; o[17] = (float)e.has2;
}
HK_HD void getObs2(const Env& e, float* o) {
  const Body &p1 = e.b[B_R1], &p2 = e.b[B_R2], &pk = e.b[B_PUCK];
  const float cx = (float)HK_CENTER_X, cy = (float)HK_CENTER_Y;
  o[0] = -(p2.p.x - cx); o[1] = -(p2.p.y - cy); o[2] = p2.a; o[3] = -p2.v.x; o[4] = -p2.v.y; o[5] = p2.w;
  o[6] = -(p1.p.x - cx); o[7] = -(p1.p.y - cy); o[8] = p1.a; o[9] = -p1.v.x; o[10] = -p1.v.y; o[11] = p1.w;
  o[12] = -(pk.p.x - cx); o[13] = -(pk.p.y - cy); o[14] = -pk.v.x; o[15] = -pk.v.y;
  o[16] = (float)e.has2; o[17] = (float)e.has1;
}

// _get_info / get_info_agent_two (hockey_env.py:542-591): out = winner, closeness, touch, direction
HK_NI_FASTA void getInfo(const Env& e, bool agent_two, double* out) {
  const Body &p1 = e.b[B_R1], &p2 = e.b[B_R2], &pk = e.b[B_PUCK];
  const int max_timesteps = maxTimesteps(e.mode);
  double closeness = 0;
  bool cond = agent_two ? ((double)pk.p.x > HK_CENTER_X && (double)pk.v.x >= 0) : ((double)pk.p.x < HK_CENTER_X && (double)pk.v.x <= 0);
  if (cond) {
    V2 d = (agent_two ? p2.p : p1.p) - pk.p;
    double dist = sqrt((double)d.x * (double)d.x + (double)d.y * (double)d.y);
    double max_dist = 250. / HK_SCALE;
    double max_reward = -30.;
    double factor = max_reward / (max_dist * max_timesteps / 2);
    closeness += dist * factor;
  }
  double touch = 0.;
  if ((agent_two ? e.has2 : e.has1) == HK_MAX_TIME_KEEP_PUCK) touch = 1.;
  double factor = (agent_two ? -1.0 : 1.0) / (max_timesteps * HK_MAX_PUCK_SPEED);
  out[0] = agent_two ? -e.winner : e.winner;
  out[1] = closeness;
  out[2] = touch;
  out[3] = (double)pk.v.x * factor;
}
HK_HD double computeReward(const Env& e) {  // hockey_env.py:518-528
  double r = 0;
  if (e.done) {
    if (e.winner == 1) r += 10;
    else if (e.winner == -1) r -= 10;
  }
  return r;
}

// BasicOpponent.act (hockey_env.py:787-833) on a float32 observation
HK_NI_POLICY void basicAct(const Config& cfg, const float* obs, bool weak, double* phase_io, double u_inc, float out[4]) {
  double p1[3] = {obs[0], obs[1], obs[2]};
  double v1[3] = {obs[3], obs[4], obs[5]};
  double puck0 = obs[12], puck1 = obs[13], puckv0 = obs[14], puckv1 = obs[15];
  double target[3];
  *phase_io += u_inc;
  const double time_to_break = 0.1;
  double kp = weak ? 0.5 : 10;
  const double kd = 0.5;
  if (puckv0 < 30.0 / HK_SCALE) {
    if (p1[0] < puck0 && fabs(p1[1] - puck1) < 30.0 / HK_SCALE) {
      double dx = p1[0] - puck0, dy = p1[1] - puck1;
      double dist = sqrt(dx * dx + dy * dy);
      target[0] = puck0 + 0.2;
      target[1] = puck1 + puckv1 * dist * 0.1;
    } else {
      target[0] = -210 / HK_SCALE;
      target[1] = puck1;
    }
  } else {
    target[0] = -210 / HK_SCALE;
    target[1] = 0;
  }
  double sp, cdummy;
  sincos_poly(*phase_io, &sp, &cdummy);
  target[2] = HK_MAX_ANGLE * sp;
  double shootv = 0.0;
  if (cfg.keep_mode && obs[16] > 0 && obs[16] < 7) shootv = 1.0;
  const double kps[3] = {kp, kp / 5, kp / 2};
  const double ttb[3] = {time_to_break, time_to_break, time_to_break * 10};
  for (int i = 0; i < 3; ++i) {
    double error = target[i] - p1[i];
    double need_break = fabs(error / (v1[i] + 0.01)) < ttb[i] ? 1.0 : 0.0;
    double a = error * kps[i] - v1[i] * need_break * kd;
    a = a < -1 ? -1 : (a > 1 ? 1 : a);
    out[i] = (float)a;
  }
  out[3] = (float)shootv;
}

// reset (hockey_env.py:345-418): overwrite per-env state; the scene itself is constant
// reset_seed >= 0 (HockeyEnv.reset(seed=...), hockey_env.py:347 `self.seed(seed)`): the draws are a function of that seed
// alone -- the same seed gives the same start state on any env of any batch; otherwise they come from the env's own
// stream (library seed, global env id, episode counter).  The mode never enters a draw's key.
#define HK_SEEDED_RESET_TAG 0x5EEDED5EEDull
HK_HD double resetDraw(const Config& cfg, uint64_t env_id, uint32_t episode, int64_t reset_seed, int idx, double lo, double hi) {
  U4 r = reset_seed >= 0 ? philox((uint64_t)reset_seed, HK_SEEDED_RESET_TAG, 0u, (uint32_t)HK_STREAM_RESET | ((uint32_t)(idx >> 1) << 8))
                         : philox(cfg.seed, env_id, episode, (uint32_t)HK_STREAM_RESET | ((uint32_t)(idx >> 1) << 8));
  double u = (idx & 1) ? u53(r.z, r.w) : u53(r.x, r.y);
  return lo + (hi - lo) * u;
}
HK_HD void createDynamicBody(const Scene& S, Env& e, int bi, double px, double py) {
  Body& b = e.b[bi];
  b.p = mk((float)px, (float)py);
  b.q = rotOf(0.0f);
  b.a = b.a0 = 0.0f;
  b.alpha0 = 0.0f;
  b.c = b.c0 = mul(bodyXf(b), mk(S.lcx[bi], S.lcy[bi]));
  b.v = mk(0.0f, 0.0f);
  b.w = 0.0f;
  b.f = mk(0.0f, 0.0f);
  b.tq = 0.0f;
  b.ldamp = bi == B_PUCK ? 0.05f : 0.0f;
  b.adamp = 0.0f;
  b.sleep = 0.0f;
  b.awake = true;
  b.island = false;
  AABB a = shapeAABB(S, bi, bodyXf(b));
  e.fat[bi].lx = a.lx - HK_AABB_EXTENSION;
  e.fat[bi].ly = a.ly - HK_AABB_EXTENSION;
  e.fat[bi].hx = a.hx + HK_AABB_EXTENSION;
  e.fat[bi].hy = a.hy + HK_AABB_EXTENSION;
}
// next_mode: HK_MODE_* of the episode this reset starts (the reference's `mode` setter / reset(mode=...) takes effect
// here, hockey_env.py:350-364), -1 = keep the env's mode
HK_NI_RARE void envReset(const Scene& S, const Config& cfg, Env& e, uint64_t env_id, int one_starting /* -1 = alternate */,
                             int64_t reset_seed = -1, int next_mode = -1) {
  e.done = false;
  e.winner = 0;
  e.time = 0;
  if (next_mode >= 0) e.mode = next_mode;
  const int mode = e.mode;
  // the reference does not clear player{1,2}_has_puck on reset
  if (mode == 0) {
    if (one_starting >= 0) e.one_starts = one_starting != 0;
    else e.one_starts = !e.one_starts;
  }
  e.clist = 0;
  e.ncontacts = 0;
  e.exist = 0;
  e.touch = 0;
  e.pcount = 0;
  e.moved = 15u;
  createDynamicBody(S, e, B_R1, HK_W / 5, HK_H / 2);
  int draw = 0;
  if (mode != 0) {
    double dx = resetDraw(cfg, env_id, e.episode, reset_seed, draw++, -HK_W / 3, HK_W / 6);
    double dy = resetDraw(cfg, env_id, e.episode, reset_seed, draw++, -HK_H / 4, HK_H / 4);
    createDynamicBody(S, e, B_R2, 4 * HK_W / 5 + dx, HK_H / 2 + dy);
  } else {
    createDynamicBody(S, e, B_R2, 4 * HK_W / 5, HK_H / 2);
  }
  if (mode == 0 || mode == 1) {
    double dx = resetDraw(cfg, env_id, e.episode, reset_seed, draw++, HK_H / 8, HK_H / 4);
    double dy = resetDraw(cfg, env_id, e.episode, reset_seed, draw++, -HK_H / 8, HK_H / 8);
    if (e.one_starts || mode == 1) createDynamicBody(S, e, B_PUCK, HK_W / 2 - dx, HK_H / 2 + dy);
    else createDynamicBody(S, e, B_PUCK, HK_W / 2 + dx, HK_H / 2 + dy);
  } else {
    double dx = resetDraw(cfg, env_id, e.episode, reset_seed, draw++, 0, HK_W / 3);
    double dy = resetDraw(cfg, env_id, e.episode, reset_seed, draw++, -HK_H / 2, HK_H / 2);
    createDynamicBody(S, e, B_PUCK, HK_W / 2 + dx, HK_H / 2 + 0.8 * dy);
    double ay = resetDraw(cfg, env_id, e.episode, reset_seed, draw++, -HK_GOAL_SIZE / HK_SCALE, HK_GOAL_SIZE / HK_SCALE);
    Body& puck = e.b[B_PUCK];
    V2 direction = puck.p - mk(0.0f, (float)(HK_H / 2 + .6 * ay));
    float len = length(direction);
    direction = mk(direction.x / len, direction.y / len);
    V2 force = -direction;
    force = mk(force.x * (float)HK_SHOOTFORCEMULTIPLIER, force.y * (float)HK_SHOOTFORCEMULTIPLIER);
    force = mk(force.x * S.mass[B_PUCK], force.y * S.mass[B_PUCK]);
    float ts = (float)(1.0 / HK_FPS);
    force = mk(force.x / ts, force.y / ts);
    applyForceToCenter(puck, force);
  }
  ++e.episode;
  e.ret[0] = e.ret[1] = 0.0;
}

// actions for this tick from the per-player policy (include/hockey_b200.h HK_POLICY_*)
HK_NI_POLICY void policyActions(const Config& cfg, Env& e, uint64_t env_id, const float* ext /* this env's row or null */,
                         int pol1, int pol2, float a[8]) {
  const int pol[2] = {pol1, pol2};
  U4 ro;
  ro.x = ro.y = ro.z = ro.w = 0;
  if (pol1 == 1 || pol1 == 2 || pol2 == 1 || pol2 == 2) ro = philox(cfg.seed, env_id, e.tick, HK_STREAM_OPP);
  for (int k = 0; k < 2; ++k) {
    float* out = a + 4 * k;
    if (pol[k] == 0) {
      for (int i = 0; i < 4; ++i) {
        float x = ext[k * 4 + i];
        out[i] = x < -1.0f ? -1.0f : (x > 1.0f ? 1.0f : x);
      }
    } else if (pol[k] == 1 || pol[k] == 2) {
      float obs[18];
      if (k == 0) getObs(e, obs); else getObs2(e, obs);
      double u = k == 0 ? u53(ro.x, ro.y) : u53(ro.z, ro.w);
      basicAct(cfg, obs, pol[k] == 1, &e.phase[k], 0.0 + (0.2 - 0.0) * u, out);
    } else if (pol[k] == 3) {
      U4 r = philox(cfg.seed, env_id, e.tick, (uint32_t)HK_STREAM_ACT | ((uint32_t)k << 8));
      out[0] = u_pm1(r.x);
      out[1] = u_pm1(r.y);
      out[2] = u_pm1(r.z);
      out[3] = u_pm1(r.w);
    } else {
      out[0] = out[1] = out[2] = out[3] = 0.0f;
    }
  }
}

// the state side effect of policyActions (BasicOpponent.phase += U(0, 0.2), hockey_env.py:796) without the controller
// arithmetic: used when the actions of this tick were already computed by the fast tier
HK_HD void policyAdvancePhases(const Config& cfg, Env& e, uint64_t env_id, int pol1, int pol2) {
  if (pol1 == 1 || pol1 == 2 || pol2 == 1 || pol2 == 2) {
    U4 ro = philox(cfg.seed, env_id, e.tick, HK_STREAM_OPP);
    if (pol1 == 1 || pol1 == 2) e.phase[0] += 0.0 + (0.2 - 0.0) * u53(ro.x, ro.y);
    if (pol2 == 1 || pol2 == 2) e.phase[1] += 0.0 + (0.2 - 0.0) * u53(ro.z, ro.w);
  }
}

// step (hockey_env.py:658-695) with an already clipped float32 action; everything before world.Step
HK_HD_NOINLINE void envStepActions(const Scene& S, const Config& cfg, Env& e, const float action[8]) {
  Body &p1 = e.b[B_R1], &p2 = e.b[B_R2], &puck = e.b[B_PUCK];
  applyTranslation(S, p1, B_R1, action[0], action[1], true);
  applyRotation(S, p1, B_R1, action[2]);
  applyTranslation(S, p2, B_R2, action[4], action[5], false);
  applyRotation(S, p2, B_R2, action[6]);
  {  // _limit_puck_speed (hockey_env.py:610-616)
    double vx = puck.v.x, vy = puck.v.y;
    double puck_speed = sqrt(vx * vx + vy * vy);
    puck.ldamp = puck_speed > HK_MAX_PUCK_SPEED ? 10.0f : 0.05f;
  }
  if (cfg.keep_mode) {
    if (e.has1 > 1) {
      keepPuck(S, e, p1);
      e.has1 -= 1;
      if (e.has1 == 1 || action[3] > 0.5f) {
        shoot(S, e, p1, true);
        e.has1 = 0;
      }
    }
    if (e.has2 > 1) {
      keepPuck(S, e, p2);
      e.has2 -= 1;
      if (e.has2 == 1 || action[7] > 0.5f) {
        shoot(S, e, p2, false);
        e.has2 = 0;
      }
    }
  }
}
HK_HD void envStepAfterWorld(Env& e) {
  if (e.time >= maxTimesteps(e.mode)) e.done = true;
  e.time += 1;
  ++e.tick;
}
HK_HD_NOINLINE void envStep(const Scene& S, const Config& cfg, const Cache& cache, Env& e, const float action[8]) {
  envStepActions(S, cfg, e, action);
  worldStep(S, cfg, cache, e, (float)(1.0 / HK_FPS), 6 * 30, 2 * 30);
  if (e.aborted) return;
  envStepAfterWorld(e);
}

}  // namespace hk
