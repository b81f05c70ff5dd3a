// hk_state.cuh -- per-env state in HBM and its two external forms.
//
// HBM layout ("core"): structure-of-arrays of 16 float4 groups per env, group g of env i at
// core[g * N + i]; a warp reads/writes each group as one coalesced 512-byte transaction of 128-bit
// accesses.  64 words = 256 B per env.  The warm-start cache (6 words x 27 pairs per env, strided
// [slot][env]) is only touched for pairs that hold manifold points.
//
// The canonical record (include/hockey_b200.h HK_S_*) is the implementation-independent form used
// by hk_get_state/hk_set_state and by the parity tests to move whole states between this library
// and the CPU oracle.
#pragma once
#include "hk_env.cuh"

namespace hk {

enum { CORE_GROUPS = 16 };
struct F4 {
  float x, y, z, w;
};

HK_HD float bitsF(uint32_t u) { return u2f(u); }
HK_HD uint32_t bitsU(float f) { return f2u(f); }

HK_HD void dbl2words(double d, float* lo, float* hi) {
  uint64_t u;
#if defined(__CUDA_ARCH__)
  u = (uint64_t)__double_as_longlong(d);
#else
  memcpy(&u, &d, 8);
#endif
  *lo = u2f((uint32_t)u);
  *hi = u2f((uint32_t)(u >> 32));
}
HK_HD double words2dbl(float lo, float hi) {
  uint64_t u = (uint64_t)f2u(lo) | ((uint64_t)f2u(hi) << 32);
#if defined(__CUDA_ARCH__)
  return __longlong_as_double((long long)u);
#else
  double d;
  memcpy(&d, &u, 8);
  return d;
#endif
}

// g[] = the 16 groups of one env
HK_HD void envToGroups(const Env& e, F4* g) {
  const Body &r1 = e.b[0], &r2 = e.b[1], &pk = e.b[2];
  g[0] = F4{r1.p.x, r1.p.y, r1.q.s, r1.q.c};
  g[1] = F4{r1.c.x, r1.c.y, r1.a, r1.w};
  g[2] = F4{r1.v.x, r1.v.y, r2.v.x, r2.v.y};
  g[3] = F4{r2.p.x, r2.p.y, r2.q.s, r2.q.c};
  g[4] = F4{r2.c.x, r2.c.y, r2.a, r2.w};
  g[5] = F4{pk.c.x, pk.c.y, pk.v.x, pk.v.y};
  g[6] = F4{pk.a, pk.w, pk.f.x, pk.f.y};
  uint32_t flags = (r1.awake ? 1u : 0u) | (r2.awake ? 2u : 0u) | (pk.awake ? 4u : 0u) | (e.done ? 8u : 0u) |
                   (e.one_starts ? 16u : 0u) | ((uint32_t)(e.winner + 1) << 5) | ((e.moved & 15u) << 8) |
                   ((uint32_t)e.ncontacts << 12) | ((uint32_t)e.mode << 16);
  g[7] = F4{r1.sleep, r2.sleep, pk.sleep, u2f(flags)};
  for (int k = 0; k < 3; ++k) g[8 + k] = F4{e.fat[k].lx, e.fat[k].ly, e.fat[k].hx, e.fat[k].hy};
  dbl2words(e.phase[0], &g[11].x, &g[11].y);
  dbl2words(e.phase[1], &g[11].z, &g[11].w);
  dbl2words(e.ret[0], &g[12].x, &g[12].y);
  dbl2words(e.ret[1], &g[12].z, &g[12].w);
  g[13] = F4{u2f((uint32_t)e.clist), u2f((uint32_t)(e.clist >> 32)), u2f((uint32_t)e.pcount), u2f((uint32_t)(e.pcount >> 32))};
  g[14] = F4{u2f(e.exist), u2f(e.touch), u2f((uint32_t)e.time), u2f((uint32_t)e.has1 | ((uint32_t)e.has2 << 8))};
  g[15] = F4{u2f(e.episode), u2f(e.tick), pk.c0.x, pk.c0.y};
}

HK_HD void groupsToEnv(const F4* g, Env& e) {
  Body &r1 = e.b[0], &r2 = e.b[1], &pk = e.b[2];
  r1.p = mk(g[0].x, g[0].y); r1.q.s = g[0].z; r1.q.c = g[0].w;
  r1.c = mk(g[1].x, g[1].y); r1.a = g[1].z; r1.w = g[1].w;
  r1.v = mk(g[2].x, g[2].y); r2.v = mk(g[2].z, g[2].w);
  r2.p = mk(g[3].x, g[3].y); r2.q.s = g[3].z; r2.q.c = g[3].w;
  r2.c = mk(g[4].x, g[4].y); r2.a = g[4].z; r2.w = g[4].w;
  pk.c = mk(g[5].x, g[5].y); pk.v = mk(g[5].z, g[5].w);
  pk.a = g[6].x; pk.w = g[6].y; pk.f = mk(g[6].z, g[6].w);
  pk.p = pk.c;
  pk.q.s = 0.0f;  // the puck's rotation never enters any result (circle centred on the body origin)
  pk.q.c = 1.0f;
  uint32_t flags = f2u(g[7].w);
  r1.sleep = g[7].x; r2.sleep = g[7].y; pk.sleep = g[7].z;
  r1.awake = flags & 1u; r2.awake = (flags & 2u) != 0; pk.awake = (flags & 4u) != 0;
  e.done = (flags & 8u) != 0;
  e.one_starts = (flags & 16u) != 0;
  e.winner = (int)((flags >> 5) & 3u) - 1;
  e.moved = (flags >> 8) & 15u;
  e.ncontacts = (int)((flags >> 12) & 15u);
  e.mode = (int)((flags >> 16) & 3u);
  for (int k = 0; k < 3; ++k) {
    e.fat[k].lx = g[8 + k].x; e.fat[k].ly = g[8 + k].y; e.fat[k].hx = g[8 + k].z; e.fat[k].hy = g[8 + k].w;
  }
  e.phase[0] = words2dbl(g[11].x, g[11].y);
  e.phase[1] = words2dbl(g[11].z, g[11].w);
  e.ret[0] = words2dbl(g[12].x, g[12].y);
  e.ret[1] = words2dbl(g[12].z, g[12].w);
  e.clist = (uint64_t)f2u(g[13].x) | ((uint64_t)f2u(g[13].y) << 32);
  e.pcount = (uint64_t)f2u(g[13].z) | ((uint64_t)f2u(g[13].w) << 32);
  e.exist = f2u(g[14].x);
  e.touch = f2u(g[14].y);
  e.time = (int)f2u(g[14].z);
  uint32_t has = f2u(g[14].w);
  e.has1 = (int)(has & 255u);
  e.has2 = (int)((has >> 8) & 255u);
  e.episode = f2u(g[15].x);
  e.tick = f2u(g[15].y);
  pk.c0 = mk(g[15].z, g[15].w);
  // not state: rebuilt every tick before use
  for (int k = 0; k < 3; ++k) {
    Body& b = e.b[k];
    if (k < 2) {
      b.f = mk(0.0f, 0.0f);
      b.c0 = b.c;
    }
    b.a0 = b.a;
    b.tq = 0.0f;
    b.alpha0 = 0.0f;
    b.ldamp = k == 2 ? 0.05f : 0.0f;
    b.adamp = 0.0f;
    b.island = false;
  }
  e.enabled = 0xFFFFFFFFu;
  e.nmf = 0;
  e.nVelIters = e.nToiEvents = e.nOverflow = 0;
  e.sweepBudget = 1 << 20;
  e.allowToiEvents = true;
  e.aborted = false;
  e.dbgEvalClk = e.dbgEventClk = 0;
  e.toiPreFlag = 0;
}

// ---- canonical record <-> Env ------------------------------------------------------------------
HK_HD void packRecord(const Env& e, const Cache& cache, uint32_t* r) {
  for (int i = 0; i < 64 + 27 * 8; ++i) r[i] = 0;
  for (int k = 0; k < 2; ++k) {
    const Body& b = e.b[k];
    uint32_t* p = r + 8 * k;
    p[0] = f2u(b.p.x); p[1] = f2u(b.p.y); p[2] = f2u(b.c.x); p[3] = f2u(b.c.y);
    p[4] = f2u(b.a); p[5] = f2u(b.v.x); p[6] = f2u(b.v.y); p[7] = f2u(b.w);
  }
  const Body& pk = e.b[2];
  r[16] = f2u(pk.c.x); r[17] = f2u(pk.c.y); r[18] = f2u(pk.a); r[19] = f2u(pk.v.x); r[20] = f2u(pk.v.y); r[21] = f2u(pk.w);
  for (int k = 0; k < 3; ++k) r[22 + k] = f2u(e.b[k].sleep);
  r[25] = (e.b[0].awake ? 1u : 0u) | (e.b[1].awake ? 2u : 0u) | (e.b[2].awake ? 4u : 0u) | (e.done ? 8u : 0u) |
          (e.one_starts ? 16u : 0u) | ((uint32_t)(e.winner + 1) << 5);
  r[26] = (uint32_t)e.time;
  r[27] = (uint32_t)e.has1;
  r[28] = (uint32_t)e.has2;
  r[29] = f2u(pk.f.x);
  r[30] = f2u(pk.f.y);
  for (int k = 0; k < 3; ++k) {
    r[31 + 4 * k] = f2u(e.fat[k].lx); r[32 + 4 * k] = f2u(e.fat[k].ly);
    r[33 + 4 * k] = f2u(e.fat[k].hx); r[34 + 4 * k] = f2u(e.fat[k].hy);
  }
  r[43] = e.moved & 15u;
  float lo, hi;
  dbl2words(e.phase[0], &lo, &hi); r[44] = f2u(lo); r[45] = f2u(hi);
  dbl2words(e.phase[1], &lo, &hi); r[46] = f2u(lo); r[47] = f2u(hi);
  r[48] = e.episode;
  r[49] = e.tick;
  dbl2words(e.ret[0], &lo, &hi); r[50] = f2u(lo); r[51] = f2u(hi);
  dbl2words(e.ret[1], &lo, &hi); r[52] = f2u(lo); r[53] = f2u(hi);
  r[54] = f2u(pk.c0.x);
  r[55] = f2u(pk.c0.y);
  for (int i = 0; i < e.ncontacts; ++i) {
    int pid = clistGet(e.clist, i);
    uint32_t* q = r + 64 + 8 * pid;
    q[0] = 1u | (((e.touch >> pid) & 1u) ? 2u : 0u) | ((uint32_t)i << 8);
    int n = getCount(e, pid);
    q[1] = (uint32_t)n;
    for (int j = 0; j < n; ++j) {
      q[2 + j] = cache.at(pid, j);
      q[4 + 2 * j] = cache.at(pid, 2 + 2 * j);
      q[5 + 2 * j] = cache.at(pid, 3 + 2 * j);
    }
  }
}

HK_HD void unpackRecord(const uint32_t* r, Env& e, const Cache& cache) {
  for (int k = 0; k < 2; ++k) {
    Body& b = e.b[k];
    const uint32_t* p = r + 8 * k;
    b.p = mk(u2f(p[0]), u2f(p[1]));
    b.c = mk(u2f(p[2]), u2f(p[3]));
    b.a = u2f(p[4]);
    b.q = rotOf(b.a);
    b.v = mk(u2f(p[5]), u2f(p[6]));
    b.w = u2f(p[7]);
  }
  Body& pk = e.b[2];
  pk.c = mk(u2f(r[16]), u2f(r[17]));
  pk.p = pk.c;
  pk.a = u2f(r[18]);
  pk.q.s = 0.0f;
  pk.q.c = 1.0f;
  pk.v = mk(u2f(r[19]), u2f(r[20]));
  pk.w = u2f(r[21]);
  for (int k = 0; k < 3; ++k) e.b[k].sleep = u2f(r[22 + k]);
  uint32_t flags = r[25];
  e.b[0].awake = (flags & 1u) != 0;
  e.b[1].awake = (flags & 2u) != 0;
  e.b[2].awake = (flags & 4u) != 0;
  e.done = (flags & 8u) != 0;
  e.one_starts = (flags & 16u) != 0;
  e.winner = (int)((flags >> 5) & 3u) - 1;
  e.time = (int)r[26];
  e.has1 = (int)r[27];
  e.has2 = (int)r[28];
  pk.f = mk(u2f(r[29]), u2f(r[30]));
  for (int k = 0; k < 3; ++k) {
    e.fat[k].lx = u2f(r[31 + 4 * k]); e.fat[k].ly = u2f(r[32 + 4 * k]);
    e.fat[k].hx = u2f(r[33 + 4 * k]); e.fat[k].hy = u2f(r[34 + 4 * k]);
  }
  e.moved = r[43] & 15u;
  if (e.moved & 8u) e.moved = 15u;
  e.phase[0] = words2dbl(u2f(r[44]), u2f(r[45]));
  e.phase[1] = words2dbl(u2f(r[46]), u2f(r[47]));
  e.episode = r[48];
  e.tick = r[49];
  e.ret[0] = words2dbl(u2f(r[50]), u2f(r[51]));
  e.ret[1] = words2dbl(u2f(r[52]), u2f(r[53]));
  pk.c0 = mk(u2f(r[54]), u2f(r[55]));
  // contacts, in recorded list order
  e.clist = 0;
  e.ncontacts = 0;
  e.exist = 0;
  e.touch = 0;
  e.pcount = 0;
  int order[27];
  int n = 0;
  for (int pid = 0; pid < 27; ++pid)
    if (r[64 + 8 * pid] & 1u) order[n++] = pid;
  for (int i = 1; i < n; ++i) {  // sort by recorded position
    int p = order[i];
    uint32_t kp = (r[64 + 8 * p] >> 8) & 255u;
    int j = i - 1;
    while (j >= 0 && ((r[64 + 8 * order[j]] >> 8) & 255u) > kp) {
      order[j + 1] = order[j];
      --j;
    }
    order[j + 1] = p;
  }
  for (int i = n - 1; i >= 0; --i) {  // push oldest first so that position 0 ends at the head
    int pid = order[i];
    const uint32_t* q = r + 64 + 8 * pid;
    if (e.ncontacts == MAX_CLIST) break;
    e.clist = (e.clist << 5) | (uint64_t)pid;
    e.ncontacts++;
    e.exist |= 1u << pid;
    if (q[0] & 2u) e.touch |= 1u << pid;
    int cnt = (int)q[1];
    setCount(e, pid, cnt);
    for (int j = 0; j < cnt; ++j) {
      cache.at(pid, j) = q[2 + j];
      cache.at(pid, 2 + 2 * j) = q[4 + 2 * j];
      cache.at(pid, 3 + 2 * j) = q[5 + 2 * j];
    }
  }
  for (int k = 0; k < 3; ++k) {
    Body& b = e.b[k];
    if (k < 2) {
      b.f = mk(0.0f, 0.0f);
      b.c0 = b.c;
    }
    b.a0 = b.a;
    b.tq = 0.0f;
    b.alpha0 = 0.0f;
    b.ldamp = k == 2 ? 0.05f : 0.0f;
    b.adamp = 0.0f;
    b.island = false;
  }
  e.enabled = 0xFFFFFFFFu;
  e.nmf = 0;
  e.nVelIters = e.nToiEvents = e.nOverflow = 0;
  e.sweepBudget = 1 << 20;
  e.allowToiEvents = true;
  e.aborted = false;
  e.dbgEvalClk = e.dbgEventClk = 0;
  e.toiPreFlag = 0;
}

// record word HK_S_MODE (56).  createMode = the handle's creation mode (Config::mode): the word holds 0 while the env
// plays it, else mode + 1, so that the records of single-mode handles do not depend on it.  On reading, 1..3 = mode
// 0..2; 0 (single-mode records, records of builds without per-env modes) and any other value = createMode.
HK_HD uint32_t modeWord(const Env& e, int createMode) { return e.mode == createMode ? 0u : (uint32_t)e.mode + 1u; }
HK_HD int modeOfWord(uint32_t w, int createMode) { return w >= 1u && w <= 3u ? (int)w - 1 : createMode; }

// HockeyEnv.set_state (hockey_env.py:594-608): 18 visible values; goes through b2Body::SetTransform
// / SetLinearVelocity / SetAngularVelocity semantics like the reference's property setters.
HK_HD void setObsState(const Scene& S, Env& e, const float* s, int keep_mode) {
  for (int k = 0; k < 2; ++k) {
    Body& b = e.b[k];
    const float* q = s + 6 * k;
    for (int pass = 0; pass < 2; ++pass) {
      V2 pos = pass == 0 ? mk((float)((double)q[0] + HK_CENTER_X), (float)((double)q[1] + HK_CENTER_Y)) : b.p;
      float ang = pass == 0 ? b.a : q[2];
      b.q = rotOf(ang);
      b.p = pos;
      b.c = mul(bodyXf(b), mk(S.lcx[k], S.lcy[k]));
      b.a = ang;
      b.c0 = b.c;
      b.a0 = ang;
      AABB a1 = shapeAABB(S, k, bodyXf(b));
      moveProxy(e, k, a1, b.p - b.p);
    }
    setLinearVelocity(b, mk(q[3], q[4]));
    if (q[5] * q[5] > 0.0f) setAwake(b, true);
    b.w = q[5];
  }
  setTransformPuck(S, e, mk((float)((double)s[12] + HK_CENTER_X), (float)((double)s[13] + HK_CENTER_Y)));
  setLinearVelocity(e.b[B_PUCK], mk(s[14], s[15]));
  if (keep_mode) {
    e.has1 = (int)s[16];
    e.has2 = (int)s[17];
  }
}

}  // namespace hk
