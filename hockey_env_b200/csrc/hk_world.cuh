// hk_world.cuh -- one env's world step: Collide -> island solve -> SolveTOI, specialised to the fixed
// HockeyEnv scene (3 dynamic bodies, 10 static fixtures, 27 candidate pairs).
//
// Replaces `self.world.Step(self.timeStep, 6 * 30, 2 * 30)` (reference hockey_env.py:682) and the
// ContactDetector callbacks it fires (hockey_env.py:50-73).  B200-first restructuring relative to
// a general engine:
//   * no dynamic tree / pair hash: the broad phase is three fat AABBs per env tested against a
//     constant table; the set of live contacts is one 64-bit packed list (newest first, the order
//     Box2D's contact list would have) plus 27-bit masks;
//   * no heap, no pointers between bodies: 3 dynamic bodies live in registers / local memory,
//     statics are rows of the constant Scene;
//   * the 180 velocity iterations stop as soon as one full Gauss-Seidel sweep applies only zero
//     impulses -- from then on every later sweep is bit-identical, so the result equals running
//     all 180 (checked against the oracle, which always runs 180);
//   * warm-start impulses live in a lazily touched global cache, not in the per-step state record.
#pragma once
#include "hk_collide.cuh"

namespace hk {

#if defined(HK_FAST_DEBUG) && !defined(__CUDA_ARCH__)
extern long long g_iter_hist[2][182];
extern long long g_nvc_hist[16];
extern long long g_period_hist[16];
extern long long g_toi_dbg[16];
#define HK_TOI_DBG(k) g_toi_dbg[k]++
#define HK_ITER_HIST(w, n) g_iter_hist[w][n]++
#define HK_NVC_HIST(n) g_nvc_hist[n]++
#else
#define HK_ITER_HIST(w, n)
#define HK_NVC_HIST(n)
#define HK_TOI_DBG(k)
#endif

enum { MAX_MANIFOLDS = 8, MAX_CLIST = 12 };

struct Body {
  V2 p;   // m_xf.p (body origin)
  Rot q;  // m_xf.q
  V2 c0, c;
  float a0, a, alpha0;
  V2 v;
  float w;
  V2 f;
  float tq;
  float ldamp, adamp, sleep;
  bool awake, island;
};

// persistent warm-start cache: 6 words per pair (key0,key1,ni0,ti0,ni1,ti1), strided over envs
struct Cache {
  uint32_t* base;  // already offset to this env
  size_t stride;   // in words, between consecutive (pair,word) slots
  HK_HD uint32_t& at(int pid, int k) const { return base[(size_t)(pid * 6 + k) * stride]; }
};
HK_HD float u2f(uint32_t u) {
#if defined(__CUDA_ARCH__)
  return __uint_as_float(u);
#else
  float f;
  memcpy(&f, &u, 4);
  return f;
#endif
}
HK_HD uint32_t f2u(float f) {
#if defined(__CUDA_ARCH__)
  return __float_as_uint(f);
#else
  uint32_t u;
  memcpy(&u, &f, 4);
  return u;
#endif
}

struct Env {
  Body b[3];
  int has1, has2, time, winner;
  bool done, one_starts;
  int mode;  // HK_MODE_* of the running episode (chosen at its reset)
  AABB fat[3];
  uint32_t moved;  // bit0-2: buffered proxy moves (r1, r2, puck); bit3: new fixtures since last step
  double phase[2];
  uint32_t episode, tick;
  double ret[2];
  uint64_t clist;  // packed live-contact list, 5 bits per pair id, entry 0 = newest
  int ncontacts;
  uint32_t exist, touch;  // 27-bit masks
  uint64_t pcount;        // 2 bits per pair: manifold point count held in the cache
  // per-step scratch
  uint32_t enabled;
  uint32_t sepValid;        // pairs whose sepBound / sepNormal were evaluated this tick (one word instead of 27 resets:
                            // every distinct local-memory word a warp touches costs a 128-byte L1 line)
  float sepBound[N_PAIRS];  // per pair: distance lower bound from this tick's Collide (valid if its sepValid bit is set)
  V2 sepNormal[N_PAIRS];    // ... along this world-space face normal of the static polygon
  bool toiEventSeen;
  AABB swept[3];  // tight swept AABB (incl. shape radius) of each body from this tick's island solve
  uint32_t toiPreFlag;      // pairs whose first-pass TOI was computed ahead of solveTOI (block-wide task pass)
  float toiPre[N_PAIRS];
  Manifold mf[MAX_MANIFOLDS];
  int mfPid[MAX_MANIFOLDS];
  int nmf;
  // counters (statistics)
  uint32_t nVelIters, nToiEvents, nOverflow;
  long long dbgEvalClk, dbgEventClk;  // diagnostics: cycles this lane spent in TOI evaluation / event handling
  uint32_t dbgShape;                  // diagnostics: contacts | manifold points << 4 of this tick's island solve
  // budgets of this tier (hk_lib.cu cascade); exceeding one sets `aborted` and the tick is redone, from the
  // stored state, by the next tier.  Nothing is committed before the end of a tick, so aborting is free.
  int sweepBudget;   // max velocity sweeps a solve may need to converge (>= 180: unlimited)
  bool allowToiEvents;
  bool aborted;
  int bailKind;  // why the fast path gave up (hk_fast.cuh)
};

HK_HD bool sepKnown(const Env& e, int pid) { return ((e.sepValid >> pid) & 1u) != 0; }
HK_HD float sepBoundOf(const Env& e, int pid) { return sepKnown(e, pid) ? e.sepBound[pid] : -HK_MAXFLOAT; }
HK_HD void setSep(Env& e, int pid, float bound, V2 normal) {
  e.sepBound[pid] = bound;
  e.sepNormal[pid] = normal;
  e.sepValid |= 1u << pid;
}

struct Config {
  int mode;           // the handle's creation mode: the mode of new envs, and what record word HK_S_MODE = 0 stands for
  int keep_mode;
  int max_timesteps;  // of the creation mode; a tick reads its env's own limit, maxTimesteps(e.mode)
  uint64_t seed;
};
// max_timesteps of an episode in `mode` (hockey_env.py:357-364)
HK_HD int maxTimesteps(int mode) { return mode == 0 ? 250 : 80; }

HK_HD int clistGet(uint64_t l, int i) { return (int)((l >> (5 * i)) & 31u); }
HK_HD int getCount(const Env& e, int pid) { return (int)((e.pcount >> (2 * pid)) & 3u); }
HK_HD void setCount(Env& e, int pid, int n) {
  e.pcount = (e.pcount & ~((uint64_t)3 << (2 * pid))) | ((uint64_t)n << (2 * pid));
}
HK_HD void clistRemoveAt(Env& e, int i) {
  uint64_t lowMask = ((uint64_t)1 << (5 * i)) - 1;
  uint64_t low = e.clist & lowMask;
  uint64_t high = (i + 1 < MAX_CLIST + 1) ? (e.clist >> (5 * (i + 1))) : 0;
  e.clist = low | (high << (5 * i));
  e.ncontacts--;
}
HK_HD void clistPushHead(Env& e, int pid) {
  if (e.ncontacts == MAX_CLIST) {  // cannot happen in this scene (DESIGN.md); counted, never silent
    int last = clistGet(e.clist, MAX_CLIST - 1);
    e.exist &= ~(1u << last);
    e.touch &= ~(1u << last);
    setCount(e, last, 0);
    clistRemoveAt(e, MAX_CLIST - 1);
    e.nOverflow++;
  }
  e.clist = (e.clist << 5) | (uint64_t)pid;
  e.ncontacts++;
}

HK_HD void setAwake(Body& b, bool flag) {
  if (flag) {
    if (!b.awake) {
      b.awake = true;
      b.sleep = 0.0f;
    }
  } else {
    b.awake = false;
    b.sleep = 0.0f;
    b.v = mk(0.0f, 0.0f);
    b.w = 0.0f;
    b.f = mk(0.0f, 0.0f);
    b.tq = 0.0f;
  }
}
HK_HD void applyForceToCenter(Body& b, V2 f) {  // wake = True at every reference call site
  if (!b.awake) setAwake(b, true);
  b.f += f;
}
HK_HD void applyTorque(Body& b, float t) {
  if (!b.awake) setAwake(b, true);
  b.tq += t;
}
HK_HD void setLinearVelocity(Body& b, V2 v) {
  if (dot(v, v) > 0.0f) setAwake(b, true);
  b.v = v;
}
// b2Body::SynchronizeTransform.  The puck is a circle centred on its body origin with localCenter 0: its
// rotation never enters any result, so its q stays the identity and no sin/cos is evaluated for it.
HK_HD Rot rotForBody(int bi, float a) { return bi == B_PUCK ? rotIdentity() : rotOf(a); }
HK_HD void syncTransform(const Scene& S, Body& b, int bi) {
  b.q = rotForBody(bi, b.a);
  b.p = b.c - mul(b.q, mk(S.lcx[bi], S.lcy[bi]));
}
HK_HD Xf bodyXf(const Body& b) {
  Xf x;
  x.p = b.p;
  x.q = b.q;
  return x;
}
HK_HD Xf staticXf(const Scene& S, int f) {
  Xf x;
  x.p = mk(S.spx[f], S.spy[f]);
  x.q.s = 0.0f;
  x.q.c = 1.0f;
  return x;
}
HK_HD Xf fixtureXf(const Scene& S, const Env& e, int f) { return f < N_STATIC_FIX ? staticXf(S, f) : bodyXf(e.b[f - F_R1]); }
HK_HD AABB fixtureFat(const Scene& S, const Env& e, int f) { return f < N_STATIC_FIX ? S.sfat[f] : e.fat[f - F_R1]; }
HK_HD int staticBodyOf(int f) { return f < 6 ? f : (f < 8 ? 6 : 7); }

// ---- fixture AABB / broad-phase proxy (b2Fixture::Synchronize, b2DynamicTree::MoveProxy) ----------
HK_NI_FASTS AABB shapeAABB(const Scene& S, int bi, const Xf& xf) {
  AABB r;
  if (bi == B_PUCK) {
    float rad = S.puckRadius;
    V2 pp = xf.p + mul(xf.q, mk(0.0f, 0.0f));
    r.lx = pp.x - rad;
    r.ly = pp.y - rad;
    r.hx = pp.x + rad;
    r.hy = pp.y + rad;
    return r;
  }
  const Poly& P = S.poly[F_R1 + bi];
  V2 lower = mul(xf, polyV(P, 0)), upper = lower;
  for (int i = 1; i < P.count; ++i) {
    V2 v = mul(xf, polyV(P, i));
    lower = mk(fmin2(lower.x, v.x), fmin2(lower.y, v.y));
    upper = mk(fmax2(upper.x, v.x), fmax2(upper.y, v.y));
  }
  r.lx = lower.x - HK_POLYGON_RADIUS;
  r.ly = lower.y - HK_POLYGON_RADIUS;
  r.hx = upper.x + HK_POLYGON_RADIUS;
  r.hy = upper.y + HK_POLYGON_RADIUS;
  return r;
}
HK_HD void moveProxy(Env& e, int bi, const AABB& aabb, V2 displacement) {
  if (aabbContains(e.fat[bi], aabb)) return;
  AABB b = aabb;
  b.lx = b.lx - HK_AABB_EXTENSION;
  b.ly = b.ly - HK_AABB_EXTENSION;
  b.hx = b.hx + HK_AABB_EXTENSION;
  b.hy = b.hy + HK_AABB_EXTENSION;
  V2 d = HK_AABB_MULTIPLIER * displacement;
  if (d.x < 0.0f) b.lx += d.x; else b.hx += d.x;
  if (d.y < 0.0f) b.ly += d.y; else b.hy += d.y;
  e.fat[bi] = b;
  e.moved |= 1u << bi;
}
HK_HD_NOINLINE void synchronizeFixtures(const Scene& S, Env& e, int bi) {
  Body& b = e.b[bi];
  Xf xf1;
  xf1.q = rotForBody(bi, b.a0);
  xf1.p = b.c0 - mul(xf1.q, mk(S.lcx[bi], S.lcy[bi]));
  AABB a1 = shapeAABB(S, bi, xf1);
  AABB a2 = shapeAABB(S, bi, bodyXf(b));
  AABB comb;
  comb.lx = fmin2(a1.lx, a2.lx);
  comb.ly = fmin2(a1.ly, a2.ly);
  comb.hx = fmax2(a1.hx, a2.hx);
  comb.hy = fmax2(a1.hy, a2.hy);
  moveProxy(e, bi, comb, b.p - xf1.p);
}
// b2Body::SetTransform (puck teleport, hockey_env.py:619)
HK_NI_RARE void setTransformPuck(const Scene& S, Env& e, V2 position) {
  Body& b = e.b[B_PUCK];
  b.q = rotIdentity();
  b.p = position;
  b.c = mul(bodyXf(b), mk(S.lcx[B_PUCK], S.lcy[B_PUCK]));
  b.c0 = b.c;
  b.a0 = b.a;
  AABB a1 = shapeAABB(S, B_PUCK, bodyXf(b));
  AABB comb;
  comb.lx = fmin2(a1.lx, a1.lx);
  comb.ly = fmin2(a1.ly, a1.ly);
  comb.hx = fmax2(a1.hx, a1.hx);
  comb.hy = fmax2(a1.hy, a1.hy);
  moveProxy(e, B_PUCK, comb, b.p - b.p);
}

// Fat-AABB overlap (b2TestOverlap) of all 27 candidate pairs at once, bit pid: straight-line code that is the same for
// every lane (the pair table is known at compile time), instead of a per-lane walk over each lane's own candidates
HK_HD uint32_t pairOverlapBits(const Scene& S, const Env& e) {
  const AABB f0 = e.fat[0], f1 = e.fat[1], f2 = e.fat[2];
  uint32_t ov = 0;
#pragma unroll
  for (int pid = 0; pid < N_PAIRS; ++pid) {
    int fA = 0, fB = 0;
    pairFixtures(pid, &fA, &fB);
    const AABB a = fA < N_STATIC_FIX ? S.sfat[fA] : (fA == F_R1 ? f0 : f1);
    const AABB b = fB == F_R1 ? f0 : (fB == F_R2 ? f1 : f2);
    const bool apart = (b.lx - a.hx > 0.0f) || (b.ly - a.hy > 0.0f) || (a.lx - b.hx > 0.0f) || (a.ly - b.hy > 0.0f);
    ov |= (apart ? 0u : 1u) << pid;
  }
  return ov;
}

// b2ContactManager::FindNewContacts for the buffered proxy moves
HK_NI_FASTS void findNewContacts(const Scene& S, Env& e) {
  uint32_t mv = e.moved & 7u;
  e.moved &= ~7u;
  if (!mv) return;
  uint32_t cand = 0;
  if (mv & 1u) cand |= HK_PAIRS_R1;
  if (mv & 2u) cand |= HK_PAIRS_R2;
  if (mv & 4u) cand |= HK_PAIRS_PUCK;
  cand &= ~e.exist;
  if (!cand) return;
  const uint32_t fresh = pairOverlapBits(S, e) & cand;
  if (!fresh) return;
  for (int k = 0; k < N_PAIRS; ++k) {  // creation order = sorted (proxyA, proxyB); each goes to the list head
    int pid = S.sortedPairs[k];
    if (!((fresh >> pid) & 1u)) continue;
    clistPushHead(e, pid);
    e.exist |= 1u << pid;
    e.touch &= ~(1u << pid);
    e.enabled |= 1u << pid;
    setCount(e, pid, 0);
    if (!((HK_PAIRS_SENSOR >> pid) & 1u)) {
      int bA = fixtureBody(S.pairFA[pid]), bB = fixtureBody(S.pairFB[pid]);
      if (bA >= 0) setAwake(e.b[bA], true);
      if (bB >= 0) setAwake(e.b[bB], true);
    }
  }
}

// ---- ContactDetector.BeginContact (hockey_env.py:50-73) --------------------------------------------
HK_HD void beginContact(const Config& cfg, Env& e, int pid) {
  if (pid == 24) {  // puck x goal_player_2
    e.done = true;
    e.winner = 1;
  } else if (pid == 23) {  // puck x goal_player_1
    e.done = true;
    e.winner = -1;
  } else if (pid == 25) {
    if (cfg.keep_mode && (double)e.b[B_PUCK].v.x < 0.1) {
      if (e.has1 == 0) e.has1 = 15;
    }
  } else if (pid == 26) {
    if (cfg.keep_mode && (double)e.b[B_PUCK].v.x > -0.1) {
      if (e.has2 == 0) e.has2 = 15;
    }
  }
}

HK_HD int findSlot(const Env& e, int pid) {
  for (int i = 0; i < e.nmf; ++i)
    if (e.mfPid[i] == pid) return i;
  return -1;
}

HK_HD AABB staticCoreAABB(const Scene& S, int f) {  // fat box minus extension and skin (exact enough: eps >> rounding)
  AABB r = S.sfat[f];
  const float d = HK_AABB_EXTENSION + HK_POLYGON_RADIUS;
  r.lx += d;
  r.ly += d;
  r.hx -= d;
  r.hy -= d;
  return r;
}
HK_HD float aabbGap(const AABB& a, const AABB& b) {
  float gx = fmax2(a.lx - b.hx, b.lx - a.hx);
  float gy = fmax2(a.ly - b.hy, b.ly - a.hy);
  return fmax2(gx, gy);
}
// Largest separation of the racket's vertices from a face plane of static polygon f (statics have angle 0).  The
// static polygons have four faces; b2FindMaxSeparation's hill climb (2.3.0) starts at the face best aligned with
// the centroid direction, examines it and both neighbours and keeps the largest, and the start face cannot be the
// one opposite a face that separates the shapes -- so whenever this value exceeds totalRadius the climb returns a
// separation above totalRadius as well and b2CollidePolygons produces no manifold points.
HK_HD float polyStaticFaceGap(const Scene& S, int f, const Poly& PB, const Xf& xfB, V2* normal) {
  const Poly& PA = S.poly[f];
  const float ox = S.spx[f], oy = S.spy[f];
  float s0 = HK_MAXFLOAT, s1 = HK_MAXFLOAT, s2 = HK_MAXFLOAT, s3 = HK_MAXFLOAT;
  for (int i = 0; i < PB.count; ++i) {
    V2 v = mul(xfB, polyV(PB, i));
    const float x = v.x - ox, y = v.y - oy;
    s0 = fmin2(s0, PA.nx[0] * (x - PA.vx[0]) + PA.ny[0] * (y - PA.vy[0]));
    s1 = fmin2(s1, PA.nx[1] * (x - PA.vx[1]) + PA.ny[1] * (y - PA.vy[1]));
    s2 = fmin2(s2, PA.nx[2] * (x - PA.vx[2]) + PA.ny[2] * (y - PA.vy[2]));
    s3 = fmin2(s3, PA.nx[3] * (x - PA.vx[3]) + PA.ny[3] * (y - PA.vy[3]));
  }
  int k = 0;
  float best = s0;
  if (s1 > best) { best = s1; k = 1; }
  if (s2 > best) { best = s2; k = 2; }
  if (s3 > best) { best = s3; k = 3; }
  *normal = polyN(PA, k);
  return best;
}

HK_NI_EVALMF void evaluateManifold(const Scene& S, const Env& e, int pid, Manifold* m) {
  int fA = S.pairFA[pid], fB = S.pairFB[pid];
  Xf xfA = fixtureXf(S, e, fA);
  if (fB == F_PUCK) {
    collidePolygonCircle(m, S.poly[fA], xfA, e.b[B_PUCK].p, S.puckRadius);
  } else {
    if (fA < N_STATIC_FIX) {
      // racket against a static polygon: most candidate pairs are nowhere near touching.  A face of the static
      // polygon that clears every racket vertex by more than totalRadius proves the manifold empty (see
      // polyStaticFaceGap) at a fraction of b2CollidePolygons' two max-separation searches.
      V2 nrm;
      const float gap = polyStaticFaceGap(S, fA, S.poly[fB], bodyXf(e.b[fB - F_R1]), &nrm);
      if (gap > 2.0f * HK_POLYGON_RADIUS + 0.0005f) {
        m->count = 0;
        m->sepBound = gap - 0.001f;
        m->sepNormal = nrm;
        return;
      }
    }
    collidePolygons(m, S.poly[fA], xfA, S.poly[fB], bodyXf(e.b[fB - F_R1]));
  }
}

// b2Contact::Update.  Manifold ids and warm-start impulses of the contacts handled this tick live in the
// manifold slots; the global cache is read the first time a pair is updated in a tick and written once, by
// commitCache(), when the tick completes.
HK_NI_NARROW void updateContact(const Scene& S, const Config& cfg, const Cache& cache, Env& e, int pid) {
  const uint32_t bit = 1u << pid;
  e.enabled |= bit;
  const bool wasTouching = (e.touch & bit) != 0;
  bool touching;
  if ((HK_PAIRS_SENSOR >> pid) & 1u) {
    int fA = S.pairFA[pid];
    // the GJK overlap test only when the puck centre is within reach of the goal box (margin >> float rounding)
    AABB core = staticCoreAABB(S, fA);
    V2 c = e.b[B_PUCK].p;
    AABB pb;
    pb.lx = pb.hx = c.x;
    pb.ly = pb.hy = c.y;
    if (aabbGap(core, pb) > S.puckRadius + HK_POLYGON_RADIUS + 0.005f) touching = false;
    else touching = testOverlapPolyPuck(S.poly[fA], staticXf(S, fA), e.b[B_PUCK].p, S.puckRadius);
  } else {
    int slot = findSlot(e, pid);
    Manifold tmp;
    evaluateManifold(S, e, pid, &tmp);
    setSep(e, pid, tmp.sepBound, tmp.sepNormal);  // statics have angle 0: local normal == world normal
    touching = tmp.count > 0;
    int oldCount;
    uint32_t oldKey[2] = {0, 0};
    float oldNi[2] = {0, 0}, oldTi[2] = {0, 0};
    if (slot >= 0) {
      oldCount = e.mf[slot].count;
      for (int j = 0; j < oldCount; ++j) {
        oldKey[j] = e.mf[slot].key[j];
        oldNi[j] = e.mf[slot].ni[j];
        oldTi[j] = e.mf[slot].ti[j];
      }
    } else {
      oldCount = getCount(e, pid);
      for (int j = 0; j < oldCount; ++j) {
        oldKey[j] = cache.at(pid, j);
        oldNi[j] = u2f(cache.at(pid, 2 + 2 * j));
        oldTi[j] = u2f(cache.at(pid, 3 + 2 * j));
      }
    }
    for (int i = 0; i < tmp.count; ++i) {
      tmp.ni[i] = 0.0f;
      tmp.ti[i] = 0.0f;
      for (int j = 0; j < oldCount; ++j) {
        if (oldKey[j] == tmp.key[i]) {
          tmp.ni[i] = oldNi[j];
          tmp.ti[i] = oldTi[j];
          break;
        }
      }
    }
    setCount(e, pid, tmp.count);
    if (touching) {
      if (slot < 0) {
        if (e.nmf < MAX_MANIFOLDS) {
          slot = e.nmf++;
        } else {
          slot = MAX_MANIFOLDS - 1;  // cannot happen in this scene; counted
          e.nOverflow++;
        }
        e.mfPid[slot] = pid;
      }
      e.mf[slot] = tmp;
    } else if (slot >= 0) {
      e.mf[slot].count = 0;
    }
    if (touching != wasTouching) {
      int bA = fixtureBody(S.pairFA[pid]), bB = fixtureBody(S.pairFB[pid]);
      if (bA >= 0) setAwake(e.b[bA], true);
      if (bB >= 0) setAwake(e.b[bB], true);
    }
  }
  if (touching) e.touch |= bit; else e.touch &= ~bit;
  if (!wasTouching && touching) beginContact(cfg, e, pid);
}

// write the ids / impulses of every manifold handled this tick to the persistent cache (end of a completed tick)
HK_HD_NOINLINE void commitCache(const Cache& cache, const Env& e) {
  for (int sIdx = 0; sIdx < e.nmf; ++sIdx) {
    const Manifold& m = e.mf[sIdx];
    const int pid = e.mfPid[sIdx];
    if (!((e.exist >> pid) & 1u)) continue;
    if (getCount(e, pid) != m.count) continue;  // pair was destroyed and re-created within the tick
    for (int j = 0; j < m.count; ++j) {
      cache.at(pid, j) = m.key[j];
      cache.at(pid, 2 + 2 * j) = f2u(m.ni[j]);
      cache.at(pid, 3 + 2 * j) = f2u(m.ti[j]);
    }
  }
}

HK_HD int ctz32(uint32_t m) {
#if defined(__CUDA_ARCH__)
  return __ffs((int)m) - 1;
#else
  return __builtin_ctz(m);
#endif
}
// The geometry half of b2Contact::Update for one non-sensor pair: manifold at the current poses, separation bound, and -- if
// the shapes touch -- a manifold slot holding the new points with the warm-start impulses of the matching old ids.
// No side effect on flags: collideApply() does the rest.  Returns the manifold point count.
HK_NI_NARROW int collideEvaluate(const Scene& S, const Cache& cache, Env& e, int pid) {
  Manifold tmp;
  evaluateManifold(S, e, pid, &tmp);
  setSep(e, pid, tmp.sepBound, tmp.sepNormal);
  if (tmp.count > 0) {
    const int oldCount = getCount(e, pid);
    uint32_t oldKey[2] = {0, 0};
    float oldNi[2] = {0, 0}, oldTi[2] = {0, 0};
    for (int j = 0; j < oldCount; ++j) {
      oldKey[j] = cache.at(pid, j);
      oldNi[j] = u2f(cache.at(pid, 2 + 2 * j));
      oldTi[j] = u2f(cache.at(pid, 3 + 2 * j));
    }
    for (int i = 0; i < tmp.count; ++i) {
      tmp.ni[i] = 0.0f;
      tmp.ti[i] = 0.0f;
      for (int j = 0; j < oldCount; ++j) {
        if (oldKey[j] == tmp.key[i]) {
          tmp.ni[i] = oldNi[j];
          tmp.ti[i] = oldTi[j];
          break;
        }
      }
    }
    int slot;
    if (e.nmf < MAX_MANIFOLDS) {
      slot = e.nmf++;
    } else {
      slot = MAX_MANIFOLDS - 1;  // cannot happen in this scene; counted
      e.nOverflow++;
    }
    e.mfPid[slot] = pid;
    e.mf[slot] = tmp;
  }
  return tmp.count;
}
// The flag half of b2Contact::Update, in contact-list order: manifold point count, touching bit, wake-ups, BeginContact
HK_HD void collideApply(const Scene& S, const Config& cfg, Env& e, int pid, bool touching, int count, bool sensor) {
  const uint32_t bit = 1u << pid;
  e.enabled |= bit;
  const bool wasTouching = (e.touch & bit) != 0;
  if (!sensor) {
    setCount(e, pid, count);
    if (touching != wasTouching) {
      int bA = fixtureBody(S.pairFA[pid]), bB = fixtureBody(S.pairFB[pid]);
      if (bA >= 0) setAwake(e.b[bA], true);
      if (bB >= 0) setAwake(e.b[bB], true);
    }
  }
  if (touching) e.touch |= bit; else e.touch &= ~bit;
  if (!wasTouching && touching) beginContact(cfg, e, pid);
}

// b2ContactManager::Collide.  b2Contact::Update is split: the geometry of every pair that will be updated is evaluated
// first, ONE KIND OF PAIR AT A TIME (racket x static polygon, puck x static polygon, puck x racket, racket x racket, goal
// sensors), so that the lanes of a warp -- whose contact lists hold different kinds in different positions -- run each
// narrow-phase routine together instead of serialising all of them in every step of the list walk; the flags and events
// are then applied in contact-list order, as Box2D does.  The poses do not change during Collide and bodies only ever wake
// up in it, so the geometry does not depend on the order; a pair whose bodies were both asleep when the evaluation ran and
// that a wake-up reaches later is evaluated on the spot (updateContact).  Only at the start of a world step (no manifold
// slot is in use yet): the re-updates inside SolveTOI go through updateContact.
HK_NI_COLLIDE void collide(const Scene& S, const Config& cfg, const Cache& cache, Env& e) {
  const uint32_t ov = e.ncontacts > 0 ? pairOverlapBits(S, e) : 0u;  // proxies do not move during Collide
  // pairs that the list walk below will certainly update: they exist, their fat AABBs overlap, a body of theirs is awake
  uint32_t todo = 0;
  {
    const uint32_t awakeMask = (e.b[0].awake ? HK_PAIRS_R1 : 0u) | (e.b[1].awake ? HK_PAIRS_R2 : 0u) | (e.b[2].awake ? HK_PAIRS_PUCK : 0u);
    todo = e.exist & ov & awakeMask;
  }
  uint64_t counts = 0;      // 2 bits per pair: manifold point count of the evaluated pairs
  uint32_t sensorTouch = 0;
  for (uint32_t m = todo & 0x0000FFFFu; m;) {  // racket x static polygon
    const int pid = ctz32(m);
    m &= m - 1u;
    counts |= (uint64_t)collideEvaluate(S, cache, e, pid) << (2 * pid);
  }
  for (uint32_t m = todo & 0x007E0000u; m;) {  // puck x static polygon
    const int pid = ctz32(m);
    m &= m - 1u;
    counts |= (uint64_t)collideEvaluate(S, cache, e, pid) << (2 * pid);
  }
  for (uint32_t m = todo & 0x06000000u; m;) {  // puck x racket
    const int pid = ctz32(m);
    m &= m - 1u;
    counts |= (uint64_t)collideEvaluate(S, cache, e, pid) << (2 * pid);
  }
  if (todo & 0x00010000u) counts |= (uint64_t)collideEvaluate(S, cache, e, 16) << 32;  // racket x racket
  for (uint32_t m = todo & HK_PAIRS_SENSOR; m;) {  // puck x goal sensor
    const int pid = ctz32(m);
    m &= m - 1u;
    const int fA = S.pairFA[pid];
    // the GJK overlap test only when the puck centre is within reach of the goal box (margin >> float rounding)
    AABB core = staticCoreAABB(S, fA);
    V2 c = e.b[B_PUCK].p;
    AABB pb;
    pb.lx = pb.hx = c.x;
    pb.ly = pb.hy = c.y;
    bool touching;
    if (aabbGap(core, pb) > S.puckRadius + HK_POLYGON_RADIUS + 0.005f) touching = false;
    else touching = testOverlapPolyPuck(S.poly[fA], staticXf(S, fA), e.b[B_PUCK].p, S.puckRadius);
    if (touching) sensorTouch |= 1u << pid;
  }
  int i = 0;
  while (i < e.ncontacts) {
    int pid = clistGet(e.clist, i);
    int bA = fixtureBody(S.pairFA[pid]), bB = fixtureBody(S.pairFB[pid]);
    bool activeA = bA >= 0 && e.b[bA].awake;
    bool activeB = bB >= 0 && e.b[bB].awake;
    if (!activeA && !activeB) {
      ++i;
      continue;
    }
    if (!((ov >> pid) & 1u)) {
      clistRemoveAt(e, i);
      e.exist &= ~(1u << pid);
      e.touch &= ~(1u << pid);
      setCount(e, pid, 0);
      continue;
    }
    if ((todo >> pid) & 1u) {
      const bool sensor = ((HK_PAIRS_SENSOR >> pid) & 1u) != 0;
      const int count = (int)((counts >> (2 * pid)) & 3u);
      collideApply(S, cfg, e, pid, sensor ? ((sensorTouch >> pid) & 1u) != 0 : count > 0, count, sensor);
    } else {
      updateContact(S, cfg, cache, e, pid);  // woken during this walk
    }
    ++i;
  }
}

// ---- contact solver (b2ContactSolver) ---------------------------------------------------------------
struct VCPoint {
  V2 rA, rB;
  float ni, ti, normalMass, tangentMass, bias;
};
struct VC {
  VCPoint pt[2];
  V2 normal;
  float k11, k12, k22;          // K
  float n11, n12, n21, n22;     // normalMass = K^-1  (ex.x, ey.x, ex.y, ey.y)
  float mA, iA, mB, iB, friction, restitution;
  int bA, bB;  // dynamic body index or -1
  int count, slot;
};

HK_HD void worldManifold(const Manifold& m, const Xf& xfA, float radiusA, const Xf& xfB, float radiusB, V2* normal,
                         V2 points[2]) {
  if (m.type == MANIFOLD_FACE_A) {
    *normal = mul(xfA.q, m.localNormal);
    V2 planePoint = mul(xfA, m.localPoint);
    for (int i = 0; i < m.count; ++i) {
      V2 clipPoint = mul(xfB, m.lp[i]);
      V2 cA = clipPoint + (radiusA - dot(clipPoint - planePoint, *normal)) * (*normal);
      V2 cB = clipPoint - radiusB * (*normal);
      points[i] = 0.5f * (cA + cB);
    }
  } else {
    *normal = mul(xfB.q, m.localNormal);
    V2 planePoint = mul(xfB, m.localPoint);
    for (int i = 0; i < m.count; ++i) {
      V2 clipPoint = mul(xfA, m.lp[i]);
      V2 cB = clipPoint + (radiusB - dot(clipPoint - planePoint, *normal)) * (*normal);
      V2 cA = clipPoint - radiusA * (*normal);
      points[i] = 0.5f * (cA + cB);
    }
    *normal = -(*normal);
  }
}

struct BodyRef {  // position/velocity view of one side of a constraint (static => zeros, fixed pose)
  V2 c;
  float a;
  V2 v;
  float w;
  V2 lc;
  bool rot;  // only rackets have a rotation that matters
};
HK_HD Rot rotIf(bool rot, float a) { return rot ? rotOf(a) : rotIdentity(); }
HK_HD BodyRef bodyRef(const Scene& S, const Env& e, int fixture) {
  BodyRef r;
  if (fixture < N_STATIC_FIX) {
    r.c = mk(S.spx[fixture], S.spy[fixture]);
    r.a = 0.0f;
    r.v = mk(0.0f, 0.0f);
    r.w = 0.0f;
    r.lc = mk(0.0f, 0.0f);
    r.rot = false;
  } else {
    int bi = fixture - F_R1;
    r.rot = bi != B_PUCK;
    r.c = e.b[bi].c;
    r.a = e.b[bi].a;
    r.v = e.b[bi].v;
    r.w = e.b[bi].w;
    r.lc = mk(S.lcx[bi], S.lcy[bi]);
  }
  return r;
}
HK_HD float fixtureRadius(const Scene& S, int f) { return f == F_PUCK ? S.puckRadius : HK_POLYGON_RADIUS; }

// b2ContactSolver ctor + InitializeVelocityConstraints for one contact
HK_HD_NOINLINE void initConstraint(const Scene& S, const Env& e, int pid, int slot, bool warmStarting, VC* vc) {
  const Manifold& m = e.mf[slot];
  int fA = S.pairFA[pid], fB = S.pairFB[pid];
  vc->slot = slot;
  vc->bA = fixtureBody(fA);
  vc->bB = fixtureBody(fB);
  vc->mA = vc->bA >= 0 ? S.invMass[vc->bA] : 0.0f;
  vc->iA = vc->bA >= 0 ? S.invI[vc->bA] : 0.0f;
  vc->mB = vc->bB >= 0 ? S.invMass[vc->bB] : 0.0f;
  vc->iB = vc->bB >= 0 ? S.invI[vc->bB] : 0.0f;
  vc->friction = S.friction[pid];
  vc->restitution = S.restitution[pid];
  vc->count = m.count;
  const float dtRatio = 1.0f;
  for (int j = 0; j < m.count; ++j) {
    vc->pt[j].ni = warmStarting ? dtRatio * m.ni[j] : 0.0f;
    vc->pt[j].ti = warmStarting ? dtRatio * m.ti[j] : 0.0f;
  }
  BodyRef A = bodyRef(S, e, fA), B = bodyRef(S, e, fB);
  float mA = vc->mA, mB = vc->mB, iA = vc->iA, iB = vc->iB;
  Xf xfA, xfB;
  xfA.q = rotIf(A.rot, A.a);
  xfB.q = rotIf(B.rot, B.a);
  xfA.p = A.c - mul(xfA.q, A.lc);
  xfB.p = B.c - mul(xfB.q, B.lc);
  V2 points[2];
  worldManifold(m, xfA, fixtureRadius(S, fA), xfB, fixtureRadius(S, fB), &vc->normal, points);
  for (int j = 0; j < vc->count; ++j) {
    VCPoint* p = vc->pt + j;
    p->rA = points[j] - A.c;
    p->rB = points[j] - B.c;
    float rnA = cross(p->rA, vc->normal);
    float rnB = cross(p->rB, vc->normal);
    float kNormal = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
    p->normalMass = kNormal > 0.0f ? 1.0f / kNormal : 0.0f;
    V2 tangent = cross(vc->normal, 1.0f);
    float rtA = cross(p->rA, tangent);
    float rtB = cross(p->rB, tangent);
    float kTangent = mA + mB + iA * rtA * rtA + iB * rtB * rtB;
    p->tangentMass = kTangent > 0.0f ? 1.0f / kTangent : 0.0f;
    p->bias = 0.0f;
    float vRel = dot(vc->normal, B.v + cross(B.w, p->rB) - A.v - cross(A.w, p->rA));
    if (vRel < -HK_VELOCITY_THRESHOLD) p->bias = -vc->restitution * vRel;
  }
  if (vc->count == 2) {
    VCPoint* p1 = vc->pt + 0;
    VCPoint* p2 = vc->pt + 1;
    float rn1A = cross(p1->rA, vc->normal);
    float rn1B = cross(p1->rB, vc->normal);
    float rn2A = cross(p2->rA, vc->normal);
    float rn2B = cross(p2->rB, vc->normal);
    float k11 = mA + mB + iA * rn1A * rn1A + iB * rn1B * rn1B;
    float k22 = mA + mB + iA * rn2A * rn2A + iB * rn2B * rn2B;
    float k12 = mA + mB + iA * rn1A * rn2A + iB * rn1B * rn2B;
    const float k_maxConditionNumber = 1000.0f;
    if (k11 * k11 < k_maxConditionNumber * (k11 * k22 - k12 * k12)) {
      vc->k11 = k11;
      vc->k12 = k12;
      vc->k22 = k22;
      float a = k11, b = k12, c = k12, d = k22;
      float det = a * d - b * c;
      if (det != 0.0f) det = 1.0f / det;
      vc->n11 = det * d;
      vc->n12 = -det * b;
      vc->n21 = -det * c;
      vc->n22 = det * a;
    } else {
      vc->count = 1;
    }
  }
}

struct Vel {
  V2 v;
  float w;
};
HK_HD Vel loadVel(const Env& e, int bi) {
  Vel r;
  if (bi >= 0) {
    r.v = e.b[bi].v;
    r.w = e.b[bi].w;
  } else {
    r.v = mk(0.0f, 0.0f);
    r.w = 0.0f;
  }
  return r;
}
HK_HD void storeVel(Env& e, int bi, const Vel& x) {
  if (bi >= 0) {
    e.b[bi].v = x.v;
    e.b[bi].w = x.w;
  }
}

HK_HD_NOINLINE void warmStartConstraint(Env& e, const VC& vc) {
  Vel A = loadVel(e, vc.bA), B = loadVel(e, vc.bB);
  V2 normal = vc.normal;
  V2 tangent = cross(normal, 1.0f);
  for (int j = 0; j < vc.count; ++j) {
    const VCPoint& p = vc.pt[j];
    V2 P = p.ni * normal + p.ti * tangent;
    A.w -= vc.iA * cross(p.rA, P);
    A.v -= vc.mA * P;
    B.w += vc.iB * cross(p.rB, P);
    B.v += vc.mB * P;
  }
  storeVel(e, vc.bA, A);
  storeVel(e, vc.bB, B);
}

// one Gauss-Seidel pass over one contact; returns true if any applied impulse increment was non-zero
HK_HD bool solveVelocityConstraintCore(VC& vc, Vel& A, Vel& B) {
  bool changed = false;
  const float mA = vc.mA, iA = vc.iA, mB = vc.mB, iB = vc.iB;
  V2 vA = A.v, vB = B.v;
  float wA = A.w, wB = B.w;
  V2 normal = vc.normal;
  V2 tangent = cross(normal, 1.0f);
  float friction = vc.friction;
  for (int j = 0; j < vc.count; ++j) {
    VCPoint* p = vc.pt + j;
    V2 dv = vB + cross(wB, p->rB) - vA - cross(wA, p->rA);
    float vt = dot(dv, tangent) - 0.0f;
    float lambda = p->tangentMass * (-vt);
    float maxFriction = friction * p->ni;
    float newImpulse = fclamp(p->ti + lambda, -maxFriction, maxFriction);
    lambda = newImpulse - p->ti;
    p->ti = newImpulse;
    changed = changed || (lambda != 0.0f);
    V2 P = lambda * tangent;
    vA -= mA * P;
    wA -= iA * cross(p->rA, P);
    vB += mB * P;
    wB += iB * cross(p->rB, P);
  }
  if (vc.count == 1) {
    VCPoint* p = vc.pt + 0;
    V2 dv = vB + cross(wB, p->rB) - vA - cross(wA, p->rA);
    float vn = dot(dv, normal);
    float lambda = -p->normalMass * (vn - p->bias);
    float newImpulse = fmax2(p->ni + lambda, 0.0f);
    lambda = newImpulse - p->ni;
    p->ni = newImpulse;
    changed = changed || (lambda != 0.0f);
    V2 P = lambda * normal;
    vA -= mA * P;
    wA -= iA * cross(p->rA, P);
    vB += mB * P;
    wB += iB * cross(p->rB, P);
  } else {
    VCPoint* cp1 = vc.pt + 0;
    VCPoint* cp2 = vc.pt + 1;
    V2 a = mk(cp1->ni, cp2->ni);
    V2 dv1 = vB + cross(wB, cp1->rB) - vA - cross(wA, cp1->rA);
    V2 dv2 = vB + cross(wB, cp2->rB) - vA - cross(wA, cp2->rA);
    float vn1 = dot(dv1, normal);
    float vn2 = dot(dv2, normal);
    V2 b;
    b.x = vn1 - cp1->bias;
    b.y = vn2 - cp2->bias;
    b -= mk(vc.k11 * a.x + vc.k12 * a.y, vc.k12 * a.x + vc.k22 * a.y);
    V2 x;
    bool found = false;
    // case 1
    x = -mk(vc.n11 * b.x + vc.n12 * b.y, vc.n21 * b.x + vc.n22 * b.y);
    if (x.x >= 0.0f && x.y >= 0.0f) found = true;
    if (!found) {  // case 2
      x.x = -cp1->normalMass * b.x;
      x.y = 0.0f;
      vn2 = vc.k12 * x.x + b.y;
      if (x.x >= 0.0f && vn2 >= 0.0f) found = true;
    }
    if (!found) {  // case 3
      x.x = 0.0f;
      x.y = -cp2->normalMass * b.y;
      vn1 = vc.k12 * x.y + b.x;
      if (x.y >= 0.0f && vn1 >= 0.0f) found = true;
    }
    if (!found) {  // case 4
      x.x = 0.0f;
      x.y = 0.0f;
      vn1 = b.x;
      vn2 = b.y;
      if (vn1 >= 0.0f && vn2 >= 0.0f) found = true;
    }
    if (found) {
      V2 d = x - a;
      V2 P1 = d.x * normal, P2 = d.y * normal;
      vA -= mA * (P1 + P2);
      wA -= iA * (cross(cp1->rA, P1) + cross(cp2->rA, P2));
      vB += mB * (P1 + P2);
      wB += iB * (cross(cp1->rB, P1) + cross(cp2->rB, P2));
      cp1->ni = x.x;
      cp2->ni = x.y;
      changed = changed || (d.x != 0.0f) || (d.y != 0.0f);
    }
  }
  A.v = vA;
  A.w = wA;
  B.v = vB;
  B.w = wB;
  return changed;
}
HK_HD_NOINLINE bool solveVelocityConstraint(Env& e, VC& vc) {
  Vel A = loadVel(e, vc.bA), B = loadVel(e, vc.bB);
  bool changed = solveVelocityConstraintCore(vc, A, B);
  storeVel(e, vc.bA, A);
  storeVel(e, vc.bB, B);
  return changed;
}

// ---- the 180 velocity iterations, cut short exactly ----------------------------------------------------
// One sweep is a deterministic map F of the solver state s = (body velocities, accumulated impulses).
//  * s_k == s_(k-1) (no non-zero impulse increment in sweep k): fixed point, every later sweep is a no-op;
//  * s_k == s_(k-2): the sequence has entered a period-2 cycle (observed in ~20 % of solves: the last bit of
//    an impulse and of a velocity flip back and forth) -- the state after all N sweeps is s_k or s_(k-1)
//    depending on the parity of N - k.
// Either way the result is numerically identical to running all N sweeps, which is what the oracle does.
// Specialised sweep loop for the dominant case -- one contact with one manifold point (95 % of solves): every
// quantity lives in registers, same expression order as solveVelocityConstraint().
struct VC1 {  // what the one-point loop reads of a VC (64 B instead of 148: hk_lib.cu pools these in shared memory)
  V2 rA, rB, normal;
  float ni, ti, normalMass, tangentMass, bias, mA, iA, mB, iB, friction;
};
HK_HD VC1 vc1Of(const VC& vc) {
  VC1 c;
  c.rA = vc.pt[0].rA; c.rB = vc.pt[0].rB; c.normal = vc.normal;
  c.ni = vc.pt[0].ni; c.ti = vc.pt[0].ti;
  c.normalMass = vc.pt[0].normalMass; c.tangentMass = vc.pt[0].tangentMass; c.bias = vc.pt[0].bias;
  c.mA = vc.mA; c.iA = vc.iA; c.mB = vc.mB; c.iB = vc.iB; c.friction = vc.friction;
  return c;
}
// Sweeps [itStart, itStop) of the velIters-sweep solve; HK_SOLVE_UNFINISHED if it neither ended nor reached velIters.
// The solve may be cut into such ranges anywhere (hk_lib.cu re-packs the lanes of its pooled solves between ranges):
// a fixed point stays a fixed point, and a period-2 cycle found later is resolved by the parity of the ABSOLUTE sweep
// index, so the result does not depend on the cuts.
enum { HK_SOLVE_UNFINISHED = -2 };
HK_NI_LOOP int runVelocityIterations1Range(VC1& vc, Vel& A, Vel& B, int budget, int velIters, int itStart, int itStop,
                                               int* sweepsOut) {
  int sweeps = 0;
  const float mA = vc.mA, iA = vc.iA, mB = vc.mB, iB = vc.iB;
  const V2 normal = vc.normal;
  const V2 tangent = cross(normal, 1.0f);
  const float friction = vc.friction;
  const V2 rA = vc.rA, rB = vc.rB;
  const float normalMass = vc.normalMass, tangentMass = vc.tangentMass, bias = vc.bias;
  float ni = vc.ni, ti = vc.ti;
  V2 vA = A.v, vB = B.v;
  float wA = A.w, wB = B.w;
  // states after the previous sweep (1) and the one before (2)
  V2 vA1 = vA, vB1 = vB, vA2 = vA, vB2 = vB;
  float wA1 = wA, wB1 = wB, ni1 = ni, ti1 = ti, wA2 = wA, wB2 = wB, ni2 = ni, ti2 = ti;
  int it = itStart;
  int result = itStop < velIters ? (int)HK_SOLVE_UNFINISHED : 0;
  for (; it < itStop; ++it) {
    bool changed = false;
    {
      V2 dv = vB + cross(wB, rB) - vA - cross(wA, rA);
      float vt = dot(dv, tangent) - 0.0f;
      float lambda = tangentMass * (-vt);
      float maxFriction = friction * ni;
      float newImpulse = fclamp(ti + lambda, -maxFriction, maxFriction);
      lambda = newImpulse - ti;
      ti = newImpulse;
      changed = changed || (lambda != 0.0f);
      V2 P = lambda * tangent;
      vA -= mA * P;
      wA -= iA * cross(rA, P);
      vB += mB * P;
      wB += iB * cross(rB, P);
    }
    {
      V2 dv = vB + cross(wB, rB) - vA - cross(wA, rA);
      float vn = dot(dv, normal);
      float lambda = -normalMass * (vn - bias);
      float newImpulse = fmax2(ni + lambda, 0.0f);
      lambda = newImpulse - ni;
      ni = newImpulse;
      changed = changed || (lambda != 0.0f);
      V2 P = lambda * normal;
      vA -= mA * P;
      wA -= iA * cross(rA, P);
      vB += mB * P;
      wB += iB * cross(rB, P);
    }
    ++sweeps;
    if (!changed) {
      result = it + 1;
      break;
    }
    if (it >= itStart + 2 && vA.x == vA2.x && vA.y == vA2.y && wA == wA2 && vB.x == vB2.x && vB.y == vB2.y && wB == wB2 &&
        ni == ni2 && ti == ti2) {
      // period-2 cycle: state after sweep it+1 == state after sweep it-1
      const int remaining = velIters - 1 - it;
      if (remaining & 1) {
        vA = vA1; vB = vB1; wA = wA1; wB = wB1; ni = ni1; ti = ti1;
      }
      result = it + 1;
      break;
    }
    vA2 = vA1; vB2 = vB1; wA2 = wA1; wB2 = wB1; ni2 = ni1; ti2 = ti1;
    vA1 = vA; vB1 = vB; wA1 = wA; wB1 = wB; ni1 = ni; ti1 = ti;
    if (it + 1 >= budget && it + 1 < velIters) {
      result = -1;
      break;
    }
    if (it + 1 == velIters) result = velIters;
  }
  vc.ni = ni;
  vc.ti = ti;
  A.v = vA; A.w = wA; B.v = vB; B.w = wB;
  *sweepsOut = sweeps;
  return result;
}
HK_HD int runVelocityIterations1Core(VC1& vc, Vel& A, Vel& B, int budget, int velIters, int* sweepsOut) {
  return runVelocityIterations1Range(vc, A, B, budget, velIters, 0, velIters, sweepsOut);
}
HK_HD int runVelocityIterations1(Env& e, VC& vc, int velIters) {
  Vel A = loadVel(e, vc.bA), B = loadVel(e, vc.bB);
  int sweeps = 0;
  VC1 c = vc1Of(vc);
  const int result = runVelocityIterations1Core(c, A, B, e.sweepBudget, velIters, &sweeps);
  vc.pt[0].ni = c.ni;
  vc.pt[0].ti = c.ti;
  storeVel(e, vc.bA, A);
  storeVel(e, vc.bB, B);
  e.nVelIters += (uint32_t)sweeps;
  return result;
}

// Same for one contact with a two-point manifold (racket resting on a wall / goal): tangent rows, then the 2x2
// block solver of b2ContactSolver::SolveVelocityConstraints, all in registers.
HK_NI_LOOP int runVelocityIterations2Core(VC& vc, Vel& A, Vel& B, int budget, int velIters, int* sweepsOut) {
  int sweeps = 0;
  const float mA = vc.mA, iA = vc.iA, mB = vc.mB, iB = vc.iB;
  const V2 normal = vc.normal;
  const V2 tangent = cross(normal, 1.0f);
  const float friction = vc.friction;
  const V2 rA0 = vc.pt[0].rA, rB0 = vc.pt[0].rB, rA1 = vc.pt[1].rA, rB1 = vc.pt[1].rB;
  const float tm0 = vc.pt[0].tangentMass, tm1 = vc.pt[1].tangentMass;
  const float nm0 = vc.pt[0].normalMass, nm1 = vc.pt[1].normalMass;
  const float bias0 = vc.pt[0].bias, bias1 = vc.pt[1].bias;
  const float k11 = vc.k11, k12 = vc.k12, k22 = vc.k22, n11 = vc.n11, n12 = vc.n12, n21 = vc.n21, n22 = vc.n22;
  float ni0 = vc.pt[0].ni, ti0 = vc.pt[0].ti, ni1 = vc.pt[1].ni, ti1 = vc.pt[1].ti;
  V2 vA = A.v, vB = B.v;
  float wA = A.w, wB = B.w;
  // previous (p) and before-previous (q) states
  V2 vAp = vA, vBp = vB, vAq = vA, vBq = vB;
  float wAp = wA, wBp = wB, wAq = wA, wBq = wB;
  float ni0p = ni0, ti0p = ti0, ni1p = ni1, ti1p = ti1, ni0q = ni0, ti0q = ti0, ni1q = ni1, ti1q = ti1;
  int result = 0;
  for (int it = 0; it < velIters; ++it) {
    bool changed = false;
    {  // tangent, point 0
      V2 dv = vB + cross(wB, rB0) - vA - cross(wA, rA0);
      float vt = dot(dv, tangent) - 0.0f;
      float lambda = tm0 * (-vt);
      float maxFriction = friction * ni0;
      float newImpulse = fclamp(ti0 + lambda, -maxFriction, maxFriction);
      lambda = newImpulse - ti0;
      ti0 = newImpulse;
      changed = changed || (lambda != 0.0f);
      V2 P = lambda * tangent;
      vA -= mA * P;
      wA -= iA * cross(rA0, P);
      vB += mB * P;
      wB += iB * cross(rB0, P);
    }
    {  // tangent, point 1
      V2 dv = vB + cross(wB, rB1) - vA - cross(wA, rA1);
      float vt = dot(dv, tangent) - 0.0f;
      float lambda = tm1 * (-vt);
      float maxFriction = friction * ni1;
      float newImpulse = fclamp(ti1 + lambda, -maxFriction, maxFriction);
      lambda = newImpulse - ti1;
      ti1 = newImpulse;
      changed = changed || (lambda != 0.0f);
      V2 P = lambda * tangent;
      vA -= mA * P;
      wA -= iA * cross(rA1, P);
      vB += mB * P;
      wB += iB * cross(rB1, P);
    }
    {  // block solver
      V2 a = mk(ni0, ni1);
      V2 dv1 = vB + cross(wB, rB0) - vA - cross(wA, rA0);
      V2 dv2 = vB + cross(wB, rB1) - vA - cross(wA, rA1);
      float vn1 = dot(dv1, normal);
      float vn2 = dot(dv2, normal);
      V2 b;
      b.x = vn1 - bias0;
      b.y = vn2 - bias1;
      b -= mk(k11 * a.x + k12 * a.y, k12 * a.x + k22 * a.y);
      V2 x;
      bool found = false;
      x = -mk(n11 * b.x + n12 * b.y, n21 * b.x + n22 * b.y);
      if (x.x >= 0.0f && x.y >= 0.0f) found = true;
      if (!found) {
        x.x = -nm0 * b.x;
        x.y = 0.0f;
        vn2 = k12 * x.x + b.y;
        if (x.x >= 0.0f && vn2 >= 0.0f) found = true;
      }
      if (!found) {
        x.x = 0.0f;
        x.y = -nm1 * b.y;
        vn1 = k12 * x.y + b.x;
        if (x.y >= 0.0f && vn1 >= 0.0f) found = true;
      }
      if (!found) {
        x.x = 0.0f;
        x.y = 0.0f;
        vn1 = b.x;
        vn2 = b.y;
        if (vn1 >= 0.0f && vn2 >= 0.0f) found = true;
      }
      if (found) {
        V2 d = x - a;
        V2 P1 = d.x * normal, P2 = d.y * normal;
        vA -= mA * (P1 + P2);
        wA -= iA * (cross(rA0, P1) + cross(rA1, P2));
        vB += mB * (P1 + P2);
        wB += iB * (cross(rB0, P1) + cross(rB1, P2));
        ni0 = x.x;
        ni1 = x.y;
        changed = changed || (d.x != 0.0f) || (d.y != 0.0f);
      }
    }
    ++sweeps;
    result = it + 1;
    if (!changed) break;
    if (it >= 2 && vA.x == vAq.x && vA.y == vAq.y && wA == wAq && vB.x == vBq.x && vB.y == vBq.y && wB == wBq &&
        ni0 == ni0q && ti0 == ti0q && ni1 == ni1q && ti1 == ti1q) {
      const int remaining = velIters - 1 - it;
      if (remaining & 1) {
        vA = vAp; vB = vBp; wA = wAp; wB = wBp; ni0 = ni0p; ti0 = ti0p; ni1 = ni1p; ti1 = ti1p;
      }
      break;
    }
    vAq = vAp; vBq = vBp; wAq = wAp; wBq = wBp; ni0q = ni0p; ti0q = ti0p; ni1q = ni1p; ti1q = ti1p;
    vAp = vA; vBp = vB; wAp = wA; wBp = wB; ni0p = ni0; ti0p = ti0; ni1p = ni1; ti1p = ti1;
    if (it + 1 >= budget && it + 1 < velIters) {
      result = -1;
      break;
    }
  }
  vc.pt[0].ni = ni0;
  vc.pt[0].ti = ti0;
  vc.pt[1].ni = ni1;
  vc.pt[1].ti = ti1;
  A.v = vA; A.w = wA; B.v = vB; B.w = wB;
  *sweepsOut = sweeps;
  return result;
}
HK_HD int runVelocityIterations2(Env& e, VC& vc, int velIters) {
  Vel A = loadVel(e, vc.bA), B = loadVel(e, vc.bB);
  int sweeps = 0;
  const int result = runVelocityIterations2Core(vc, A, B, e.sweepBudget, velIters, &sweeps);
  storeVel(e, vc.bA, A);
  storeVel(e, vc.bB, B);
  e.nVelIters += (uint32_t)sweeps;
  return result;
}

// ---- general loop: any number of contacts ------------------------------------------------------------------
// The constraint being swept lives in registers (VCR); the next one is loaded while the current one is computed
// (its loads do not depend on the arithmetic chain, so their latency hides behind it) and only the accumulated
// impulses go back to memory.  The three bodies' velocities and their values after the previous two sweeps are
// registers as well; the impulse history needed for the period-2 test is a write-only rotating snapshot that is
// read back only when all nine velocity components already repeat.
struct VCR {
  V2 normal;
  float friction, mA, iA, mB, iB;
  int bA, bB, count;
  V2 rA0, rB0, rA1, rB1;
  float nm0, tm0, bias0, ni0, ti0, nm1, tm1, bias1, ni1, ti1;
  float k11, k12, k22, n11, n12, n21, n22;
};
HK_HD void vcrLoad(VCR& r, const VC& m) {
  r.normal = m.normal;
  r.friction = m.friction;
  r.mA = m.mA; r.iA = m.iA; r.mB = m.mB; r.iB = m.iB;
  r.bA = m.bA; r.bB = m.bB; r.count = m.count;
  r.rA0 = m.pt[0].rA; r.rB0 = m.pt[0].rB;
  r.nm0 = m.pt[0].normalMass; r.tm0 = m.pt[0].tangentMass; r.bias0 = m.pt[0].bias;
  r.ni0 = m.pt[0].ni; r.ti0 = m.pt[0].ti;
  if (m.count == 2) {
    r.rA1 = m.pt[1].rA; r.rB1 = m.pt[1].rB;
    r.nm1 = m.pt[1].normalMass; r.tm1 = m.pt[1].tangentMass; r.bias1 = m.pt[1].bias;
    r.ni1 = m.pt[1].ni; r.ti1 = m.pt[1].ti;
    r.k11 = m.k11; r.k12 = m.k12; r.k22 = m.k22;
    r.n11 = m.n11; r.n12 = m.n12; r.n21 = m.n21; r.n22 = m.n22;
  } else {
    r.rA1 = r.rB1 = mk(0.0f, 0.0f);
    r.nm1 = r.tm1 = r.bias1 = r.ni1 = r.ti1 = 0.0f;
    r.k11 = r.k12 = r.k22 = r.n11 = r.n12 = r.n21 = r.n22 = 0.0f;
  }
}
// one Gauss-Seidel pass over one contact held in registers: same expression order as solveVelocityConstraintCore()
template <int COUNT>  // COUNT = 1 / 2: manifold points known at compile time; 0: read c.count
HK_HD bool vcrSweep(VCR& c, Vel& A, Vel& B) {
  bool changed = false;
  const float mA = c.mA, iA = c.iA, mB = c.mB, iB = c.iB;
  V2 vA = A.v, vB = B.v;
  float wA = A.w, wB = B.w;
  const V2 normal = c.normal;
  const V2 tangent = cross(normal, 1.0f);
  {  // tangent, point 0
    V2 dv = vB + cross(wB, c.rB0) - vA - cross(wA, c.rA0);
    float vt = dot(dv, tangent) - 0.0f;
    float lambda = c.tm0 * (-vt);
    float maxFriction = c.friction * c.ni0;
    float newImpulse = fclamp(c.ti0 + lambda, -maxFriction, maxFriction);
    lambda = newImpulse - c.ti0;
    c.ti0 = newImpulse;
    changed = changed || (lambda != 0.0f);
    V2 P = lambda * tangent;
    vA -= mA * P;
    wA -= iA * cross(c.rA0, P);
    vB += mB * P;
    wB += iB * cross(c.rB0, P);
  }
  if (COUNT == 1 || (COUNT == 0 && c.count == 1)) {
    V2 dv = vB + cross(wB, c.rB0) - vA - cross(wA, c.rA0);
    float vn = dot(dv, normal);
    float lambda = -c.nm0 * (vn - c.bias0);
    float newImpulse = fmax2(c.ni0 + lambda, 0.0f);
    lambda = newImpulse - c.ni0;
    c.ni0 = newImpulse;
    changed = changed || (lambda != 0.0f);
    V2 P = lambda * normal;
    vA -= mA * P;
    wA -= iA * cross(c.rA0, P);
    vB += mB * P;
    wB += iB * cross(c.rB0, P);
  } else {
    {  // tangent, point 1
      V2 dv = vB + cross(wB, c.rB1) - vA - cross(wA, c.rA1);
      float vt = dot(dv, tangent) - 0.0f;
      float lambda = c.tm1 * (-vt);
      float maxFriction = c.friction * c.ni1;
      float newImpulse = fclamp(c.ti1 + lambda, -maxFriction, maxFriction);
      lambda = newImpulse - c.ti1;
      c.ti1 = newImpulse;
      changed = changed || (lambda != 0.0f);
      V2 P = lambda * tangent;
      vA -= mA * P;
      wA -= iA * cross(c.rA1, P);
      vB += mB * P;
      wB += iB * cross(c.rB1, P);
    }
    // block solver
    V2 a = mk(c.ni0, c.ni1);
    V2 dv1 = vB + cross(wB, c.rB0) - vA - cross(wA, c.rA0);
    V2 dv2 = vB + cross(wB, c.rB1) - vA - cross(wA, c.rA1);
    float vn1 = dot(dv1, normal);
    float vn2 = dot(dv2, normal);
    V2 b;
    b.x = vn1 - c.bias0;
    b.y = vn2 - c.bias1;
    b -= mk(c.k11 * a.x + c.k12 * a.y, c.k12 * a.x + c.k22 * a.y);
    V2 x;
    bool found = false;
    x = -mk(c.n11 * b.x + c.n12 * b.y, c.n21 * b.x + c.n22 * b.y);
    if (x.x >= 0.0f && x.y >= 0.0f) found = true;
    if (!found) {
      x.x = -c.nm0 * b.x;
      x.y = 0.0f;
      vn2 = c.k12 * x.x + b.y;
      if (x.x >= 0.0f && vn2 >= 0.0f) found = true;
    }
    if (!found) {
      x.x = 0.0f;
      x.y = -c.nm1 * b.y;
      vn1 = c.k12 * x.y + b.x;
      if (x.y >= 0.0f && vn1 >= 0.0f) found = true;
    }
    if (!found) {
      x.x = 0.0f;
      x.y = 0.0f;
      vn1 = b.x;
      vn2 = b.y;
      if (vn1 >= 0.0f && vn2 >= 0.0f) found = true;
    }
    if (found) {
      V2 d = x - a;
      V2 P1 = d.x * normal, P2 = d.y * normal;
      vA -= mA * (P1 + P2);
      wA -= iA * (cross(c.rA0, P1) + cross(c.rA1, P2));
      vB += mB * (P1 + P2);
      wB += iB * (cross(c.rB0, P1) + cross(c.rB1, P2));
      c.ni0 = x.x;
      c.ni1 = x.y;
      changed = changed || (d.x != 0.0f) || (d.y != 0.0f);
    }
  }
  A.v = vA;
  A.w = wA;
  B.v = vB;
  B.w = wB;
  return changed;
}
HK_HD bool velEq(const Vel& a, const Vel& b) { return a.v.x == b.v.x && a.v.y == b.v.y && a.w == b.w; }

// sweep constraint k (held in c) against the register-resident body velocities, write its impulses back
HK_HD bool vcrStep(VCR& c, int k, Vel& v0, Vel& v1, Vel& v2, VC* vcs, float* h) {
  Vel zero;
  zero.v = mk(0.0f, 0.0f);
  zero.w = 0.0f;
  const int bA = c.bA, bB = c.bB;
  Vel A = bA == 0 ? v0 : (bA == 1 ? v1 : (bA == 2 ? v2 : zero));
  Vel B = bB == 0 ? v0 : (bB == 1 ? v1 : (bB == 2 ? v2 : zero));
  const bool changed = vcrSweep<0>(c, A, B);
  if (bA == 0) v0 = A; else if (bA == 1) v1 = A; else if (bA == 2) v2 = A;
  if (bB == 0) v0 = B; else if (bB == 1) v1 = B; else if (bB == 2) v2 = B;
  vcs[k].pt[0].ni = c.ni0;
  vcs[k].pt[0].ti = c.ti0;
  h[4 * k] = c.ni0;
  h[4 * k + 1] = c.ti0;
  if (c.count == 2) {
    vcs[k].pt[1].ni = c.ni1;
    vcs[k].pt[1].ti = c.ti1;
  }
  h[4 * k + 2] = c.ni1;
  h[4 * k + 3] = c.ti1;
  return changed;
}

// ---- fixed shapes: two contacts (point counts C0, C1), everything in registers for the whole loop ------------
// The tick time of a small batch is the time of its slowest env, and the slowest envs are the solves that never
// settle (racket pressed on a bar while it holds the puck: two or three contacts, all 180 sweeps).  For them the
// loop below has no memory traffic at all: both constraints, the three body velocities and the two previous states
// needed for the period-2 test are registers; the point counts are template parameters.
struct VelTriple {
  Vel b0, b1, b2;
};
HK_HD float sel3(bool p0, bool p1, bool p2, float x0, float x1, float x2) { return p0 ? x0 : (p1 ? x1 : (p2 ? x2 : 0.0f)); }
// sweep constraint c against the three register-resident body velocities: the two bodies it couples are picked
// and written back with scalar selects (no branches; bA != bB, and -1 = static reads as zero and is never written)
template <int COUNT>
HK_HD bool vcrStepR(VCR& c, VelTriple& v) {
  const bool a0 = c.bA == 0, a1 = c.bA == 1, a2 = c.bA == 2;
  const bool b0 = c.bB == 0, b1 = c.bB == 1, b2 = c.bB == 2;
  Vel A, B;
  A.v.x = sel3(a0, a1, a2, v.b0.v.x, v.b1.v.x, v.b2.v.x);
  A.v.y = sel3(a0, a1, a2, v.b0.v.y, v.b1.v.y, v.b2.v.y);
  A.w = sel3(a0, a1, a2, v.b0.w, v.b1.w, v.b2.w);
  B.v.x = sel3(b0, b1, b2, v.b0.v.x, v.b1.v.x, v.b2.v.x);
  B.v.y = sel3(b0, b1, b2, v.b0.v.y, v.b1.v.y, v.b2.v.y);
  B.w = sel3(b0, b1, b2, v.b0.w, v.b1.w, v.b2.w);
  const bool changed = vcrSweep<COUNT>(c, A, B);
  v.b0.v.x = a0 ? A.v.x : (b0 ? B.v.x : v.b0.v.x);
  v.b0.v.y = a0 ? A.v.y : (b0 ? B.v.y : v.b0.v.y);
  v.b0.w = a0 ? A.w : (b0 ? B.w : v.b0.w);
  v.b1.v.x = a1 ? A.v.x : (b1 ? B.v.x : v.b1.v.x);
  v.b1.v.y = a1 ? A.v.y : (b1 ? B.v.y : v.b1.v.y);
  v.b1.w = a1 ? A.w : (b1 ? B.w : v.b1.w);
  v.b2.v.x = a2 ? A.v.x : (b2 ? B.v.x : v.b2.v.x);
  v.b2.v.y = a2 ? A.v.y : (b2 ? B.v.y : v.b2.v.y);
  v.b2.w = a2 ? A.w : (b2 ? B.w : v.b2.w);
  return changed;
}
struct Imp4 {
  float ni0, ti0, ni1, ti1;
};
HK_HD Imp4 impOf(const VCR& c) {
  Imp4 r;
  r.ni0 = c.ni0; r.ti0 = c.ti0; r.ni1 = c.ni1; r.ti1 = c.ti1;
  return r;
}
HK_HD void impTo(VCR& c, const Imp4& r) {
  c.ni0 = r.ni0; c.ti0 = r.ti0; c.ni1 = r.ni1; c.ti1 = r.ti1;
}
template <int COUNT>
HK_HD bool impEq(const VCR& c, const Imp4& r) {
  return c.ni0 == r.ni0 && c.ti0 == r.ti0 && (COUNT == 1 || (c.ni1 == r.ni1 && c.ti1 == r.ti1));
}
HK_HD bool velTripleEq(const VelTriple& a, const VelTriple& b) { return velEq(a.b0, b.b0) && velEq(a.b1, b.b1) && velEq(a.b2, b.b2); }
HK_HD void vcrStoreImpulses(const VCR& c, VC& m) {
  m.pt[0].ni = c.ni0;
  m.pt[0].ti = c.ti0;
  if (m.count == 2) {
    m.pt[1].ni = c.ni1;
    m.pt[1].ti = c.ti1;
  }
}
// `vcs` may live anywhere (the caller's local array, or a block-shared task record another lane filled in: hk_lib.cu
// hands the multi-contact solves of a block to warps that each run ONE loop shape)
template <int C0, int C1, int C2>  // C2 == 0: two contacts
HK_NI_LOOP int runVelocityIterationsFixedCore(VC* vcs, VelTriple& vio, int budget, int velIters, int* sweepsOut) {
  int sweeps = 0;
  VelTriple v = vio;  // registers for the whole loop
  VCR a, b, c;
  vcrLoad(a, vcs[0]);
  vcrLoad(b, vcs[1]);
  if (C2 != 0) vcrLoad(c, vcs[2]);
  VelTriple p = v, q = v;  // after the previous sweep, after the one before
  Imp4 pa = impOf(a), pb = impOf(b), pc = impOf(C2 != 0 ? c : a), qa = pa, qb = pb, qc = pc;
  int result = 0;
  for (int it = 0; it < velIters; ++it) {
    bool changed = vcrStepR<C0>(a, v);
    changed = vcrStepR<C1>(b, v) || changed;
    if (C2 != 0) changed = vcrStepR<C2 == 0 ? 1 : C2>(c, v) || changed;
    ++sweeps;
    result = it + 1;
    if (!changed) break;
    if (it >= 2 && velTripleEq(v, q) && impEq<C0>(a, qa) && impEq<C1>(b, qb) && (C2 == 0 || impEq<C2 == 0 ? 1 : C2>(c, qc))) {
      const int remaining = velIters - 1 - it;  // period-2 cycle: state after sweep it == state after sweep it - 2
      if (remaining & 1) {
        v = p;
        impTo(a, pa);
        impTo(b, pb);
        if (C2 != 0) impTo(c, pc);
      }
      break;
    }
    q = p;
    qa = pa; qb = pb;
    p = v;
    pa = impOf(a); pb = impOf(b);
    if (C2 != 0) {
      qc = pc;
      pc = impOf(c);
    }
    if (it + 1 >= budget && it + 1 < velIters) {
      result = -1;
      break;
    }
  }
  vcrStoreImpulses(a, vcs[0]);
  vcrStoreImpulses(b, vcs[1]);
  if (C2 != 0) vcrStoreImpulses(c, vcs[2]);
  vio = v;
  *sweepsOut = sweeps;
  return result;
}
// shape of a multi-contact solve that has a fixed-shape loop: 1..4 = two contacts with (1,1) (1,2) (2,1) (2,2)
// manifold points, 5 = three single-point contacts, 6..8 = three contacts with (1,1,2) (1,2,1) (2,1,1) points, 0 = none
// (anything larger: general loop, ~3,500 cycles per sweep against ~1,400 here; one contact: own loops)
enum { HK_MULTI_KINDS = 8 };
HK_HD int solveKind(const VC* vcs, int nvc) {
  if (nvc == 2) return 1 + (vcs[0].count - 1) * 2 + (vcs[1].count - 1);
  if (nvc == 3) {
    const int c0 = vcs[0].count, c1 = vcs[1].count, c2 = vcs[2].count;
    if (c0 + c1 + c2 == 3) return 5;
    if (c0 + c1 + c2 == 4) return c2 == 2 ? 6 : (c1 == 2 ? 7 : 8);
  }
  return 0;
}
HK_HD int runVelocityIterationsKind(int kind, VC* vcs, VelTriple& v, int budget, int velIters, int* sweepsOut) {
  switch (kind) {
    case 1: return runVelocityIterationsFixedCore<1, 1, 0>(vcs, v, budget, velIters, sweepsOut);
    case 2: return runVelocityIterationsFixedCore<1, 2, 0>(vcs, v, budget, velIters, sweepsOut);
    case 3: return runVelocityIterationsFixedCore<2, 1, 0>(vcs, v, budget, velIters, sweepsOut);
    case 4: return runVelocityIterationsFixedCore<2, 2, 0>(vcs, v, budget, velIters, sweepsOut);
    case 5: return runVelocityIterationsFixedCore<1, 1, 1>(vcs, v, budget, velIters, sweepsOut);
    case 6: return runVelocityIterationsFixedCore<1, 1, 2>(vcs, v, budget, velIters, sweepsOut);
    case 7: return runVelocityIterationsFixedCore<1, 2, 1>(vcs, v, budget, velIters, sweepsOut);
    default: return runVelocityIterationsFixedCore<2, 1, 1>(vcs, v, budget, velIters, sweepsOut);
  }
}

// returns the number of sweeps executed, or -1 if the tier's sweep budget ran out before the state repeated
HK_HD_NOINLINE int runVelocityIterations(Env& e, VC* vcs, int nvc, int velIters) {
  if (nvc == 1 && vcs[0].count == 1) return runVelocityIterations1(e, vcs[0], velIters);
  if (nvc == 1 && vcs[0].count == 2) return runVelocityIterations2(e, vcs[0], velIters);
  if (const int kind = solveKind(vcs, nvc)) {
    VelTriple v;
    v.b0 = loadVel(e, 0);
    v.b1 = loadVel(e, 1);
    v.b2 = loadVel(e, 2);
    int sweeps = 0;
    const int result = runVelocityIterationsKind(kind, vcs, v, e.sweepBudget, velIters, &sweeps);
    storeVel(e, 0, v.b0);
    storeVel(e, 1, v.b1);
    storeVel(e, 2, v.b2);
    e.nVelIters += (uint32_t)sweeps;
    return result;
  }
  const int budget = e.sweepBudget;
  int sweeps = 0;
  float hist[3][MAX_MANIFOLDS * 4];  // [it % 3] = impulses after sweep it
  Vel v0 = loadVel(e, 0), v1 = loadVel(e, 1), v2 = loadVel(e, 2);
  Vel p0 = v0, p1 = v1, p2 = v2, q0 = v0, q1 = v1, q2 = v2;  // after the previous sweep (p) and the one before (q)
  int result = 0;
  // Two register copies alternate (no copy between contacts): while `a` is swept, `b` is loaded with the next
  // constraint, and vice versa.  At the end of a sweep `a` holds constraint 0 again, loaded after its impulses of
  // this sweep were stored (nvc >= 2 here).
  VCR a, b;
  vcrLoad(a, vcs[0]);
  for (int it = 0; it < velIters; ++it) {
    bool changed = false;
    float* h = hist[it % 3];
    for (int k = 0; k < nvc; k += 2) {
      vcrLoad(b, vcs[k + 1 < nvc ? k + 1 : 0]);  // issued ahead of the arithmetic on `a`
      changed = vcrStep(a, k, v0, v1, v2, vcs, h) || changed;
      if (k + 1 < nvc) {
        vcrLoad(a, vcs[k + 2 < nvc ? k + 2 : 0]);
        changed = vcrStep(b, k + 1, v0, v1, v2, vcs, h) || changed;
      } else {
        a = b;  // odd number of contacts: `b` already holds constraint 0 for the next sweep
      }
    }
    ++sweeps;
    result = it + 1;
    if (!changed) break;
    if (it >= 2 && velEq(v0, q0) && velEq(v1, q1) && velEq(v2, q2)) {
      const float* h2 = hist[(it + 1) % 3];  // (it - 2) % 3
      bool same = true;
      for (int i = 0; i < 4 * nvc; ++i) same = same && (h[i] == h2[i]);
      if (same) {  // period-2 cycle: state after sweep it == state after sweep it - 2
        const int remaining = velIters - 1 - it;
        if (remaining & 1) {
          const float* h1 = hist[(it + 2) % 3];  // (it - 1) % 3
          v0 = p0; v1 = p1; v2 = p2;
          for (int k = 0; k < nvc; ++k) {
            vcs[k].pt[0].ni = h1[4 * k];
            vcs[k].pt[0].ti = h1[4 * k + 1];
            if (vcs[k].count > 1) {
              vcs[k].pt[1].ni = h1[4 * k + 2];
              vcs[k].pt[1].ti = h1[4 * k + 3];
            }
          }
        }
        break;
      }
    }
    q0 = p0; q1 = p1; q2 = p2;
    p0 = v0; p1 = v1; p2 = v2;
    if (it + 1 >= budget && it + 1 < velIters) {
      result = -1;
      break;
    }
  }
  storeVel(e, 0, v0);
  storeVel(e, 1, v1);
  storeVel(e, 2, v2);
  e.nVelIters += (uint32_t)sweeps;
  return result;
}

// b2ContactSolver::SolvePositionConstraints / SolveTOIPositionConstraints for one contact.
// In a TOI island every contact is (static A, the TOI dynamic body B), so the TOI mass rule
// ("only the two TOI bodies have mass") reduces to the normal masses.
HK_HD_NOINLINE float solvePositionConstraint(const Scene& S, Env& e, int pid, const Manifold& m, int count, bool toi) {
  float minSeparation = 0.0f;
  int fA = S.pairFA[pid], fB = S.pairFB[pid];
  int bA = fixtureBody(fA), bB = fixtureBody(fB);
  BodyRef A = bodyRef(S, e, fA), B = bodyRef(S, e, fB);
  float mA = bA >= 0 ? S.invMass[bA] : 0.0f, iA = bA >= 0 ? S.invI[bA] : 0.0f;
  float mB = bB >= 0 ? S.invMass[bB] : 0.0f, iB = bB >= 0 ? S.invI[bB] : 0.0f;
  float radiusA = fixtureRadius(S, fA), radiusB = fixtureRadius(S, fB);
  V2 cA = A.c, cB = B.c;
  float aA = A.a, aB = B.a;
  for (int j = 0; j < count; ++j) {
    Xf xfA, xfB;
    xfA.q = rotIf(A.rot, aA);
    xfB.q = rotIf(B.rot, aB);
    xfA.p = cA - mul(xfA.q, A.lc);
    xfB.p = cB - mul(xfB.q, B.lc);
    V2 normal, point;
    float separation;
    if (m.type == MANIFOLD_FACE_A) {
      normal = mul(xfA.q, m.localNormal);
      V2 planePoint = mul(xfA, m.localPoint);
      V2 clipPoint = mul(xfB, m.lp[j]);
      separation = dot(clipPoint - planePoint, normal) - radiusA - radiusB;
      point = clipPoint;
    } else {
      normal = mul(xfB.q, m.localNormal);
      V2 planePoint = mul(xfB, m.localPoint);
      V2 clipPoint = mul(xfA, m.lp[j]);
      separation = dot(clipPoint - planePoint, normal) - radiusA - radiusB;
      point = clipPoint;
      normal = -normal;
    }
    V2 rA = point - cA;
    V2 rB = point - cB;
    minSeparation = fmin2(minSeparation, separation);
    float C = fclamp((toi ? HK_TOI_BAUMGARTE : HK_BAUMGARTE) * (separation + HK_LINEAR_SLOP), -HK_MAX_LINEAR_CORRECTION, 0.0f);
    float rnA = cross(rA, normal);
    float rnB = cross(rB, normal);
    float K = mA + mB + iA * rnA * rnA + iB * rnB * rnB;
    float impulse = K > 0.0f ? -C / K : 0.0f;
    V2 P = impulse * normal;
    cA -= mA * P;
    aA -= iA * cross(rA, P);
    cB += mB * P;
    aB += iB * cross(rB, P);
  }
  if (bA >= 0) {
    e.b[bA].c = cA;
    e.b[bA].a = aA;
  }
  if (bB >= 0) {
    e.b[bB].c = cB;
    e.b[bB].a = aB;
  }
  return minSeparation;
}

HK_HD void integratePosition(Body& b, float h) {
  V2 translation = h * b.v;
  if (dot(translation, translation) > HK_MAX_TRANSLATION * HK_MAX_TRANSLATION) {
    float ratio = HK_MAX_TRANSLATION / length(translation);
    b.v *= ratio;
  }
  float rotation = h * b.w;
  if (rotation * rotation > HK_MAX_ROTATION * HK_MAX_ROTATION) {
    float ratio = HK_MAX_ROTATION / fabs2(rotation);
    b.w *= ratio;
  }
  b.c += h * b.v;
  b.a += h * b.w;
}

// b2World::Solve.  Islands are found by Box2D's DFS from (puck, racket2, racket1); because islands share no
// dynamic body they are solved here in ONE pass -- all velocity constraints in one Gauss-Seidel loop (an island
// that has converged only sees no-op sweeps, so the result equals solving island after island), position
// iterations with a per-island "done" mask (that loop is not a fixed-point iteration, so each island must stop
// exactly where b2Island::Solve would).  One loop per env instead of one per island keeps the lanes of a warp
// in the same loop at the same time.
HK_HD_NOINLINE void synchronizeFixturesQ0(const Scene& S, Env& e, int bi, Rot q0) {
  Body& b = e.b[bi];
  Xf xf1;
  xf1.q = q0;
  xf1.p = b.c0 - mul(xf1.q, mk(S.lcx[bi], S.lcy[bi]));
  AABB a1 = shapeAABB(S, bi, xf1);
  AABB a2 = shapeAABB(S, bi, bodyXf(b));
  AABB comb;
  comb.lx = fmin2(a1.lx, a2.lx);
  comb.ly = fmin2(a1.ly, a2.ly);
  comb.hx = fmax2(a1.hx, a2.hx);
  comb.hy = fmax2(a1.hy, a2.hy);
  e.swept[bi] = comb;
  moveProxy(e, bi, comb, b.p - xf1.p);
}

// what the first half of the island solve (islands, velocity integration, constraint setup, warm start) leaves for
// the velocity iterations and the second half (position iterations, sleeping, proxies)
struct IslandCtx {
  int ic[MAX_MANIFOLDS];  // island contacts in solver order
  unsigned char icIsl[MAX_MANIFOLDS];
  uint32_t islBodies[3];
  int nIsl;
  Rot q0[3];
  int nvc;
  VC vcs[MAX_MANIFOLDS];
};
HK_HD_NOINLINE void solveIslandsBegin(const Scene& S, const Cache& cache, Env& e, float h, IslandCtx& ctx) {
  e.b[0].island = e.b[1].island = e.b[2].island = false;
  uint32_t inIsland = 0;  // contacts
  int* ic = ctx.ic;
  unsigned char* icIsl = ctx.icIsl;
  int nic = 0;
  uint32_t* islBodies = ctx.islBodies;
  int nIsl = 0;
  for (int seed = 2; seed >= 0; --seed) {
    if (e.b[seed].island) continue;
    if (!e.b[seed].awake) continue;
    uint32_t bm = 0;
    int stack[3];
    int sp = 0;
    stack[sp++] = seed;
    e.b[seed].island = true;
    while (sp > 0) {
      int bi = stack[--sp];
      bm |= 1u << bi;
      setAwake(e.b[bi], true);
      uint32_t mine = bi == 0 ? HK_PAIRS_R1 : (bi == 1 ? HK_PAIRS_R2 : HK_PAIRS_PUCK);
      if (!(mine & e.touch & e.enabled & ~HK_PAIRS_SENSOR & ~inIsland)) continue;
      for (int i = 0; i < e.ncontacts; ++i) {
        int pid = clistGet(e.clist, i);
        uint32_t bit = 1u << pid;
        if (!(mine & bit)) continue;
        if (inIsland & bit) continue;
        if (!(e.enabled & bit) || !(e.touch & bit)) continue;
        if (HK_PAIRS_SENSOR & bit) continue;
        if (nic < MAX_MANIFOLDS) {
          ic[nic] = pid;
          icIsl[nic] = (unsigned char)nIsl;
          ++nic;
        } else {
          e.nOverflow++;
        }
        inIsland |= bit;
        int bA = fixtureBody(S.pairFA[pid]), bB = fixtureBody(S.pairFB[pid]);
        int other = (bA == bi) ? bB : bA;
        if (other < 0) continue;  // statics never propagate the island
        if (e.b[other].island) continue;
        stack[sp++] = other;
        e.b[other].island = true;
      }
    }
    islBodies[nIsl++] = bm;
  }
  ctx.nIsl = nIsl;
  // ---- integrate velocities (b2Island::Solve, first loop) ----
  Rot* q0 = ctx.q0;
  for (int bi = 0; bi < 3; ++bi) {
    Body& b = e.b[bi];
    q0[bi] = b.q;
    if (!b.island) continue;
    b.c0 = b.c;
    b.a0 = b.a;
    b.v += h * (1.0f * mk(0.0f, 0.0f) + S.invMass[bi] * b.f);
    b.w += h * S.invI[bi] * b.tq;
    b.v *= fclamp(1.0f - h * b.ldamp, 0.0f, 1.0f);
    b.w *= fclamp(1.0f - h * b.adamp, 0.0f, 1.0f);
  }
  // ---- constraints ----
  VC* vcs = ctx.vcs;
  int nvc = 0;
  for (int k = 0; k < nic; ++k) {
    int pid = ic[k];
    int slot = findSlot(e, pid);
    if (slot < 0) {
      // touching contact whose Collide update was skipped (both bodies were asleep): geometry from the
      // current poses, ids/impulses from the cache
      if (e.nmf >= MAX_MANIFOLDS) {
        e.nOverflow++;
        continue;
      }
      slot = e.nmf++;
      e.mfPid[slot] = pid;
      evaluateManifold(S, e, pid, &e.mf[slot]);
      int oldCount = getCount(e, pid);
      for (int i = 0; i < e.mf[slot].count; ++i) {
        e.mf[slot].ni[i] = 0.0f;
        e.mf[slot].ti[i] = 0.0f;
        for (int j = 0; j < oldCount; ++j)
          if (cache.at(pid, j) == e.mf[slot].key[i]) {
            e.mf[slot].ni[i] = u2f(cache.at(pid, 2 + 2 * j));
            e.mf[slot].ti[i] = u2f(cache.at(pid, 3 + 2 * j));
            break;
          }
      }
    }
    if (e.mf[slot].count == 0) continue;
    ic[nvc] = pid;
    icIsl[nvc] = icIsl[k];
    initConstraint(S, e, pid, slot, true, &vcs[nvc]);
    ++nvc;
  }
  {
    int npts = 0;
    for (int k = 0; k < nvc; ++k) npts += vcs[k].count;
    e.dbgShape = (uint32_t)nvc | ((uint32_t)npts << 4);
  }
  ctx.nvc = nvc;
  for (int k = 0; k < nvc; ++k) warmStartConstraint(e, vcs[k]);
}
// itc = what the velocity iterations over ctx.vcs returned (ignored when there are no constraints)
HK_HD_NOINLINE void solveIslandsEnd(const Scene& S, Env& e, float h, int posIters, IslandCtx& ctx, int itc) {
  const int nvc = ctx.nvc, nIsl = ctx.nIsl;
  VC* vcs = ctx.vcs;
  const int* ic = ctx.ic;
  const unsigned char* icIsl = ctx.icIsl;
  const uint32_t* islBodies = ctx.islBodies;
  const Rot* q0 = ctx.q0;
  if (nvc > 0) {
    if (itc < 0) {
      e.aborted = true;
      return;
    }
    HK_ITER_HIST(0, itc);
    HK_NVC_HIST(nvc);
    // StoreImpulses
    for (int k = 0; k < nvc; ++k) {
      Manifold& m = e.mf[vcs[k].slot];
      for (int j = 0; j < vcs[k].count; ++j) {
        m.ni[j] = vcs[k].pt[j].ni;
        m.ti[j] = vcs[k].pt[j].ti;
      }
    }
  }
  for (int bi = 0; bi < 3; ++bi)
    if (e.b[bi].island) integratePosition(e.b[bi], h);
  // ---- position iterations, each island stops on its own criterion ----
  uint32_t islSolved = 0;  // positionSolved per island
  {
    uint32_t withContacts = 0;
    for (int k = 0; k < nvc; ++k) withContacts |= 1u << icIsl[k];
    islSolved = ~withContacts;  // an island without contacts is solved by the first (empty) iteration
    uint32_t active = withContacts;
    for (int it = 0; it < posIters && active; ++it) {
      float minSep[3] = {0.0f, 0.0f, 0.0f};
      for (int k = 0; k < nvc; ++k) {
        int isl = icIsl[k];
        if (!((active >> isl) & 1u)) continue;
        const Manifold& m = e.mf[vcs[k].slot];
        minSep[isl] = fmin2(minSep[isl], solvePositionConstraint(S, e, ic[k], m, m.count, false));
      }
      for (int isl = 0; isl < nIsl; ++isl) {
        if (!((active >> isl) & 1u)) continue;
        if (minSep[isl] >= -3.0f * HK_LINEAR_SLOP) {
          active &= ~(1u << isl);
          islSolved |= 1u << isl;
        }
      }
    }
  }
  for (int bi = 0; bi < 3; ++bi)
    if (e.b[bi].island) syncTransform(S, e.b[bi], bi);
  // ---- sleep management per island ----
  for (int isl = 0; isl < nIsl; ++isl) {
    const uint32_t bm = islBodies[isl];
    float minSleepTime = HK_MAXFLOAT;
    const float linTolSqr = HK_LINEAR_SLEEP_TOL * HK_LINEAR_SLEEP_TOL;
    const float angTolSqr = HK_ANGULAR_SLEEP_TOL * HK_ANGULAR_SLEEP_TOL;
    for (int bi = 0; bi < 3; ++bi) {
      if (!((bm >> bi) & 1u)) continue;
      Body& b = e.b[bi];
      if (b.w * b.w > angTolSqr || dot(b.v, b.v) > linTolSqr) {
        b.sleep = 0.0f;
        minSleepTime = 0.0f;
      } else {
        b.sleep += h;
        minSleepTime = fmin2(minSleepTime, b.sleep);
      }
    }
    if (minSleepTime >= HK_TIME_TO_SLEEP && ((islSolved >> isl) & 1u)) {
      for (int bi = 0; bi < 3; ++bi)
        if ((bm >> bi) & 1u) setAwake(e.b[bi], false);
    }
  }
  for (int bi = 2; bi >= 0; --bi)
    if (e.b[bi].island) synchronizeFixturesQ0(S, e, bi, q0[bi]);
  findNewContacts(S, e);
}
HK_HD_NOINLINE void solveIslands(const Scene& S, const Config& cfg, const Cache& cache, Env& e, float h, int velIters, int posIters) {
  (void)cfg;
  IslandCtx ctx;
  solveIslandsBegin(S, cache, e, h, ctx);
  const int itc = ctx.nvc > 0 ? runVelocityIterations(e, ctx.vcs, ctx.nvc, velIters) : 0;
  solveIslandsEnd(S, e, h, posIters, ctx, itc);
}

// ---- b2World::SolveTOI: continuous collision of the dynamic bodies against the statics ---------------
HK_HD Sweep bodySweep(const Scene& S, const Body& b, int bi) {
  Sweep s;
  s.lc = mk(S.lcx[bi], S.lcy[bi]);
  s.c0 = b.c0;
  s.c = b.c;
  s.a0 = b.a0;
  s.a = b.a;
  s.alpha0 = b.alpha0;
  s.rot = bi != B_PUCK;
  return s;
}
HK_HD void bodyAdvance(const Scene& S, Body& b, int bi, float alpha) {  // b2Body::Advance
  Sweep s = bodySweep(S, b, bi);
  sweepAdvance(s, alpha);
  b.c0 = s.c0;
  b.a0 = s.a0;
  b.alpha0 = s.alpha0;
  b.c = b.c0;
  b.a = b.a0;
  b.q = rotForBody(bi, b.a);
  b.p = b.c - mul(b.q, s.lc);
}

// separation of an AABB (its corner deepest along -n) from the slanted inner face of a corner trapezoid (f = 2..5)
HK_HD float slantedFaceGap(const Scene& S, int f, const AABB& b) {
  const int k = (f & 1) ? 1 : 3;  // index of the slanted face in the hull order of polygons 2..5 (hk_scene.cuh)
  const Poly& P = S.poly[f];
  const float nx = P.nx[k], ny = P.ny[k];
  const float px = P.vx[k] + S.spx[f], py = P.vy[k] + S.spy[f];
  const float cx = nx > 0.0f ? b.lx : b.hx, cy = ny > 0.0f ? b.ly : b.hy;
  return nx * (cx - px) + ny * (cy - py);
}

// Exact proof that b2TimeOfImpact cannot answer "touching" for static fixture fA vs body bi over this tick's sweep
// (see the comment at its use in solveTOI).  Only valid before any TOI event, with the body's sweep start being the
// pose Collide saw (the body went through this tick's island solve) and alpha0 == 0.
HK_HD bool toiProvablySeparated(const Scene& S, const Env& e, int pid, int fA, int bi, float radiusB) {
  const Body& B = e.b[bi];
  V2 dc = B.c - B.c0;
  const bool known = sepKnown(e, pid);
  const float sepB = known ? e.sepBound[pid] : -HK_MAXFLOAT;
  const V2 sn = known ? e.sepNormal[pid] : mk(0.0f, 0.0f);
  // a zero normal marks a distance bound without a fixed direction: the whole displacement counts
  float toward = (sn.x == 0.0f && sn.y == 0.0f) ? length(dc) : -dot(sn, dc);
  float disp = fmax2(toward, 0.0f) + (bi == B_PUCK ? 0.0f : 0.5f * fabs2(B.a - B.a0));
  float totalRadius = HK_POLYGON_RADIUS + radiusB;
  float target = fmax2(HK_LINEAR_SLOP, totalRadius - 3.0f * HK_LINEAR_SLOP);
  if (sepB - disp > target + 0.25f * HK_LINEAR_SLOP + 0.002f) return true;
  float da = fabs2(B.a - B.a0);
  if (bi != B_PUCK && da > 0.2f) return false;
  float sag = bi == B_PUCK ? 0.0f : 0.0625f * da * da;
  // second proof (rackets): along a fixed face normal n of the static polygon every racket vertex moves on
  // n.p(t) = linear + |r| cos(theta(t) + phi), which stays above the lower of its two end values minus the
  // sagitta |r| da^2 / 8 (|r| <= 0.5 m) -- so the face separation during the sweep is at least
  // min(start, end) - sag.  The start value is sepBound; the end value is evaluated here from the final pose.
  if (bi != B_PUCK && !(sn.x == 0.0f && sn.y == 0.0f) && sepB > 0.0f) {
    const Poly& PA = S.poly[fA];
    int k = -1;
    for (int i = 0; i < PA.count; ++i)
      if (PA.nx[i] == sn.x && PA.ny[i] == sn.y) k = i;
    if (k >= 0) {
      const Poly& PB = S.poly[F_R1 + bi];
      const Xf xfB = bodyXf(B);
      const float px = PA.vx[k] + S.spx[fA], py = PA.vy[k] + S.spy[fA];
      float sEnd = HK_MAXFLOAT;
      for (int i = 0; i < PB.count; ++i) {
        V2 v = mul(xfB, polyV(PB, i));
        sEnd = fmin2(sEnd, sn.x * (v.x - px) + sn.y * (v.y - py));
      }
      if (fmin2(sepB, sEnd) - sag - 0.001f > target + 0.25f * HK_LINEAR_SLOP + 0.002f) return true;
    }
  }
  // third proof (same as the fast tier): the swept core AABB of the body stays clear of the static core AABB
  AABB st = S.sfat[fA];
  const float d = HK_AABB_EXTENSION + HK_POLYGON_RADIUS;
  st.lx += d; st.ly += d; st.hx -= d; st.hy -= d;
  AABB mv = e.swept[bi];
  mv.lx += radiusB; mv.ly += radiusB; mv.hx -= radiusB; mv.hy -= radiusB;
  float gx = fmax2(st.lx - mv.hx, mv.lx - st.hx), gy = fmax2(st.ly - mv.hy, mv.ly - st.hy);
  float gap = fmax2(gx, gy);
  if (fA >= 2 && fA < 6) gap = fmax2(gap, slantedFaceGap(S, fA, mv));
  return gap > target + 0.25f * HK_LINEAR_SLOP + sag + 0.005f;
}

// The same first proof after a TOI event of body bi: every pair of that body that the event re-evaluated
// (b2Contact::Update at the advanced pose) has a fresh separation bound, valid at pose (atC, atA).  The sub-step's
// position correction moved the sweep start away from that pose by at most |dc| + R |da| (R <= 0.5 m), the rest of
// the sweep approaches the static face by at most `disp` as above.
HK_HD bool toiSeparatedAfterEvent(const Scene& S, const Env& e, int pid, int bi, float radiusB, V2 atC, float atA) {
  const Body& B = e.b[bi];
  const bool puck = bi == B_PUCK;
  const V2 dc = B.c - B.c0;
  const V2 sn = e.sepNormal[pid];
  const float toward = (sn.x == 0.0f && sn.y == 0.0f) ? length(dc) : -dot(sn, dc);
  const float disp = fmax2(toward, 0.0f) + (puck ? 0.0f : 0.5f * fabs2(B.a - B.a0));
  const float corr = length(B.c0 - atC) + (puck ? 0.0f : 0.5f * fabs2(B.a0 - atA));
  const float totalRadius = HK_POLYGON_RADIUS + radiusB;
  const float target = fmax2(HK_LINEAR_SLOP, totalRadius - 3.0f * HK_LINEAR_SLOP);
  return sepBoundOf(e, pid) - corr - disp > target + 0.25f * HK_LINEAR_SLOP + 0.004f;
}

// One first-pass TOI evaluation as a self-contained task (hk_lib.cu runs these block-wide, one task per thread,
// so that the lanes of a warp sit in b2TimeOfImpact together instead of one after the other).
struct ToiTask {
  V2 c0, c;
  float a0, a;
  int pid;
};
HK_HD float toiTaskRun(const Scene& S, const ToiTask& t) {
  const int fA = S.pairFA[t.pid], fB = S.pairFB[t.pid];
  const int bi = fB - F_R1;
  Proxy pA, pB;
  pA.poly = &S.poly[fA];
  pA.radius = HK_POLYGON_RADIUS;
  if (fB == F_PUCK) {
    pB.poly = nullptr;
    pB.radius = S.puckRadius;
  } else {
    pB.poly = &S.poly[fB];
    pB.radius = HK_POLYGON_RADIUS;
  }
  Sweep sA;
  sA.lc = mk(0.0f, 0.0f);
  sA.c0 = sA.c = mk(S.spx[fA], S.spy[fA]);
  sA.a0 = sA.a = 0.0f;
  sA.alpha0 = 0.0f;
  sA.rot = false;
  Sweep sB;
  sB.lc = mk(S.lcx[bi], S.lcy[bi]);
  sB.c0 = t.c0;
  sB.c = t.c;
  sB.a0 = t.a0;
  sB.a = t.a;
  sB.alpha0 = 0.0f;
  sB.rot = bi != B_PUCK;
  int state;
  float tt;
  timeOfImpact(&state, &tt, pA, sA, pB, sB, 1.0f);
  const float alpha0 = 0.0f;
  return state == TOI_TOUCHING ? fmin2(alpha0 + (1.0f - alpha0) * tt, 1.0f) : 1.0f;
}
// First pass of b2World::SolveTOI's candidate loop for one env: pairs that the proofs settle get alpha = 1 right
// away, the others become tasks (up to maxTasks; the rest is left to solveTOI itself).  Returns the task count.
HK_HD int toiCollect(const Scene& S, Env& e, ToiTask* tasks, int maxTasks) {
  e.toiPreFlag = 0;
  int nt = 0;
  const uint32_t solvedMask = (e.b[0].island ? 1u : 0u) | (e.b[1].island ? 2u : 0u) | (e.b[2].island ? 4u : 0u);
  for (int i = 0; i < e.ncontacts; ++i) {
    int pid = clistGet(e.clist, i);
    uint32_t bit = 1u << pid;
    if (!(e.enabled & bit) || !(HK_PAIRS_TOI & bit)) continue;
    int fA = S.pairFA[pid], fB = S.pairFB[pid];
    int bi = fB - F_R1;
    const Body& B = e.b[bi];
    if (!B.awake) continue;
    float rB = fB == F_PUCK ? S.puckRadius : HK_POLYGON_RADIUS;
    if (((solvedMask >> bi) & 1u) && toiProvablySeparated(S, e, pid, fA, bi, rB)) {
      e.toiPre[pid] = 1.0f;
      e.toiPreFlag |= bit;
    } else if (nt < maxTasks) {
      ToiTask& t = tasks[nt++];
      t.c0 = B.c0;
      t.c = B.c;
      t.a0 = B.a0;
      t.a = B.a;
      t.pid = pid;
    }
  }
  return nt;
}

HK_HD_NOINLINE void solveTOI(const Scene& S, const Config& cfg, const Cache& cache, Env& e, float dt, int velIters) {
  HK_TOI_DBG(10);
  float salpha[8];  // alpha0 of the 8 static bodies (statics are immovable: only alpha0 advances)
  for (int i = 0; i < 8; ++i) salpha[i] = 0.0f;
  // bodies that went through this tick's island solve: their sweep start (c0, a0) is the pose Collide saw
  const uint32_t solvedMask = (e.b[0].island ? 1u : 0u) | (e.b[1].island ? 2u : 0u) | (e.b[2].island ? 4u : 0u);
  e.b[0].island = e.b[1].island = e.b[2].island = false;
  e.b[0].alpha0 = e.b[1].alpha0 = e.b[2].alpha0 = 0.0f;
  uint32_t toiFlag = e.toiPreFlag;  // first-pass results computed ahead by the block-wide task pass (or 0)
  // cached alphas live in e.toiPre itself (its first-pass contents are only valid under toiFlag and dead after this
  // function); the per-pair sub-step counters are 4-bit fields of two words -- no per-pair local arrays to reset
  float* toi = e.toiPre;
  uint64_t toiCountLo = 0, toiCountHi = 0;  // pairs 0-15 / 16-26
  e.toiPreFlag = 0;
  // pairs whose separation bound the latest event refreshed (see toiSeparatedAfterEvent)
  uint32_t freshMask = 0;
  int freshBody = -1;
  V2 freshC = mk(0.0f, 0.0f);
  float freshA = 0.0f;
  for (;;) {
    int minPid = -1;
    float minAlpha = 1.0f;
    for (int i = 0; i < e.ncontacts; ++i) {
      int pid = clistGet(e.clist, i);
      uint32_t bit = 1u << pid;
      if (!(e.enabled & bit)) continue;
      if ((int)(((pid < 16 ? toiCountLo : toiCountHi) >> (4 * (pid & 15))) & 15u) > HK_MAX_SUBSTEPS) continue;
      float alpha = 1.0f;
      if (toiFlag & bit) {
        alpha = toi[pid];
      } else {
        if (!(HK_PAIRS_TOI & bit)) continue;  // sensors and dynamic-dynamic pairs are skipped
        int fA = S.pairFA[pid], fB = S.pairFB[pid];
        int bi = fB - F_R1;
        Body& B = e.b[bi];
        if (!B.awake) continue;
        int sb = staticBodyOf(fA);
        float alpha0 = salpha[sb];
        if (salpha[sb] < B.alpha0) {
          alpha0 = B.alpha0;
          salpha[sb] = alpha0;
        } else if (B.alpha0 < salpha[sb]) {
          alpha0 = salpha[sb];
          Sweep s = bodySweep(S, B, bi);
          sweepAdvance(s, alpha0);
          B.c0 = s.c0;
          B.a0 = s.a0;
          B.alpha0 = s.alpha0;
        }
        Proxy pA, pB;
        pA.poly = &S.poly[fA];
        pA.radius = HK_POLYGON_RADIUS;
        if (fB == F_PUCK) {
          pB.poly = nullptr;
          pB.radius = S.puckRadius;
        } else {
          pB.poly = &S.poly[fB];
          pB.radius = HK_POLYGON_RADIUS;
        }
        Sweep sA;
        sA.lc = mk(0.0f, 0.0f);
        sA.c0 = sA.c = mk(S.spx[fA], S.spy[fA]);
        sA.a0 = sA.a = 0.0f;
        sA.alpha0 = salpha[sb];
        sA.rot = false;
        Sweep sB = bodySweep(S, B, bi);
        int state;
        float t;
        // Exact skip: b2TimeOfImpact can only answer "touching" if the core shapes come within target + tolerance
        // at some time of the sweep.  sepBound is the separation of the moving shape from a face plane of the
        // static polygon at the sweep start pose (from this tick's Collide), hence a lower bound of the distance;
        // along that face normal n no point of the body approaches the plane by more than max(0, -n.dc) + R |da|
        // (linear centre motion, |r| <= R = 0.5 m from the centre of mass).  If what remains stays above
        // target + tolerance (+ margin) the answer is alpha = 1.
        bool skip = !e.toiEventSeen && alpha0 == 0.0f && ((solvedMask >> bi) & 1u) &&
                    toiProvablySeparated(S, e, pid, fA, bi, pB.radius);
        if (!skip && bi == freshBody && (freshMask & bit) && sepKnown(e, pid))
          skip = toiSeparatedAfterEvent(S, e, pid, bi, pB.radius, freshC, freshA);
        HK_TOI_DBG(bi == B_PUCK ? 0 : 1);
        if (skip) {
          state = TOI_SEPARATED;
          t = 1.0f;
          HK_TOI_DBG(bi == B_PUCK ? 2 : 3);
        } else {
#if defined(__CUDA_ARCH__)
          long long c0_ = clock64();
#endif
          timeOfImpact(&state, &t, pA, sA, pB, sB, 1.0f);
#if defined(__CUDA_ARCH__)
          e.dbgEvalClk += clock64() - c0_;
#endif
          HK_TOI_DBG(bi == B_PUCK ? 4 : 5);
          if (e.toiEventSeen) HK_TOI_DBG(6);
          else if (!(alpha0 == 0.0f && ((solvedMask >> bi) & 1u))) HK_TOI_DBG(7);
          else if (!sepKnown(e, pid)) HK_TOI_DBG(8);
          if (state == TOI_TOUCHING) HK_TOI_DBG(9);
        }
        float beta = t;
        if (state == TOI_TOUCHING) alpha = fmin2(alpha0 + (1.0f - alpha0) * beta, 1.0f);
        else alpha = 1.0f;
        toi[pid] = alpha;
        toiFlag |= bit;
      }
      if (alpha < minAlpha) {
        minPid = pid;
        minAlpha = alpha;
      }
    }
    if (minPid < 0 || 1.0f - 10.0f * HK_EPS < minAlpha) break;
    if (!e.allowToiEvents) {
      e.aborted = true;
      return;
    }
    e.nToiEvents++;
    e.toiEventSeen = true;
#if defined(__CUDA_ARCH__)
    long long ev0_ = clock64();
#endif

    const int fA = S.pairFA[minPid], fB = S.pairFB[minPid];
    const int bi = fB - F_R1;
    const int sbA = staticBodyOf(fA);
    Body& B = e.b[bi];
    const Body backupB = B;
    const float backupSA = salpha[sbA];
    salpha[sbA] = minAlpha;
    bodyAdvance(S, B, bi, minAlpha);
    freshBody = bi;
    freshC = B.c;
    freshA = B.a;
    freshMask = 1u << minPid;
    updateContact(S, cfg, cache, e, minPid);
    toiFlag &= ~(1u << minPid);
    if (minPid < 16) toiCountLo += 1ull << (4 * minPid); else toiCountHi += 1ull << (4 * (minPid - 16));
    if (!(e.enabled & (1u << minPid)) || !(e.touch & (1u << minPid))) {
      e.enabled &= ~(1u << minPid);
      // restore sweeps (awake/sleep changes made by Update persist, as in b2World::SolveTOI)
      salpha[sbA] = backupSA;
      B.c0 = backupB.c0;
      B.c = backupB.c;
      B.a0 = backupB.a0;
      B.a = backupB.a;
      B.alpha0 = backupB.alpha0;
      syncTransform(S, B, bi);
      freshBody = -1;  // the body is back on its old sweep: the refreshed bounds do not describe its start
      continue;
    }
    setAwake(B, true);
    int ic[MAX_MANIFOLDS];
    int nic = 0;
    ic[nic++] = minPid;
    uint32_t inIsland = 1u << minPid;
    uint32_t staticIsland = 1u << sbA;
    const uint32_t mine = bi == 0 ? HK_PAIRS_R1 : (bi == 1 ? HK_PAIRS_R2 : HK_PAIRS_PUCK);
    for (int i = 0; i < e.ncontacts; ++i) {
      int pid = clistGet(e.clist, i);
      uint32_t bit = 1u << pid;
      if (!(mine & bit)) continue;
      if (nic == MAX_MANIFOLDS) break;
      if (inIsland & bit) continue;
      if (!(HK_PAIRS_TOI & bit)) continue;  // other body dynamic, or sensor
      int so = staticBodyOf(S.pairFA[pid]);
      float backup = salpha[so];
      if (!((staticIsland >> so) & 1u)) salpha[so] = minAlpha;
      updateContact(S, cfg, cache, e, pid);
      freshMask |= bit;
      if (!(e.enabled & bit) || !(e.touch & bit)) {
        salpha[so] = backup;
        continue;
      }
      inIsland |= bit;
      ic[nic++] = pid;
      staticIsland |= 1u << so;
    }
    const float subDt = (1.0f - minAlpha) * dt;
    // ---- b2Island::SolveTOI ----
    for (int it = 0; it < 20; ++it) {
      float minSeparation = 0.0f;
      for (int k = 0; k < nic; ++k) {
        int slot = findSlot(e, ic[k]);
        if (slot < 0) continue;
        const Manifold& m = e.mf[slot];
        minSeparation = fmin2(minSeparation, solvePositionConstraint(S, e, ic[k], m, m.count, true));
      }
      if (minSeparation >= -1.5f * HK_LINEAR_SLOP) break;
    }
    B.c0 = B.c;
    B.a0 = B.a;
    VC vcs[MAX_MANIFOLDS];
    int nvc = 0;
    for (int k = 0; k < nic; ++k) {
      int slot = findSlot(e, ic[k]);
      if (slot < 0 || e.mf[slot].count == 0) continue;
      initConstraint(S, e, ic[k], slot, false, &vcs[nvc]);
      ++nvc;
    }
    int itc = runVelocityIterations(e, vcs, nvc, velIters);
    if (itc < 0) {
      e.aborted = true;
      return;
    }
    HK_ITER_HIST(1, itc);
    integratePosition(B, subDt);
    syncTransform(S, B, bi);
    B.island = false;
    synchronizeFixtures(S, e, bi);
    toiFlag &= ~mine;
    findNewContacts(S, e);
#if defined(__CUDA_ARCH__)
    e.dbgEventClk += clock64() - ev0_;
#endif
  }
}

// b2World::Step(dt, velocityIterations, positionIterations), cut into four phases.  The general kernels run
// one phase at a time for the whole thread block (hk_lib.cu) so that the warps of an SM execute the same code
// region together and share instruction-cache lines; worldStep() below is the same sequence in one call.
HK_HD_NOINLINE void worldStepCollide(const Scene& S, const Config& cfg, const Cache& cache, Env& e) {
  e.enabled = 0xFFFFFFFFu;
  e.nmf = 0;
  e.toiEventSeen = false;
  e.toiPreFlag = 0;
  e.sepValid = 0;
  if (e.moved & 8u) {
    e.moved &= ~8u;
    findNewContacts(S, e);
  }
  collide(S, cfg, cache, e);
}
HK_HD void worldStepFinish(const Cache& cache, Env& e) {
  commitCache(cache, e);
  for (int bi = 0; bi < 3; ++bi) {  // ClearForces
    e.b[bi].f = mk(0.0f, 0.0f);
    e.b[bi].tq = 0.0f;
  }
}
HK_HD_NOINLINE void worldStep(const Scene& S, const Config& cfg, const Cache& cache, Env& e, float dt, int velIters, int posIters) {
  worldStepCollide(S, cfg, cache, e);
  solveIslands(S, cfg, cache, e, dt, velIters, posIters);
  if (e.aborted) return;
  if (e.exist & HK_PAIRS_TOI) solveTOI(S, cfg, cache, e, dt, velIters);
  if (e.aborted) return;
  worldStepFinish(cache, e);
}

}  // namespace hk
