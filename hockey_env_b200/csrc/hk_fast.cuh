// hk_fast.cuh -- the contact-free fast path of one world step.
//
// Most env-ticks have nothing to solve: no solid contact touches and no continuous-collision event
// can occur.  worldStepFast() proves that cheaply and then does exactly what the general worldStep()
// would do in that case (integrate, sync proxies, find new contacts, sleep bookkeeping).  If the
// proof fails at any point it returns false WITHOUT side effects that matter: the caller discards
// the working copy and queues the env for the general path (hk_world.cuh), which redoes the tick
// from the stored state.  A fast tick never writes the warm-start cache.
//
// The proofs are conservative bounds with a margin far above float rounding:
//  * polygon-polygon manifold is empty if the incident polygon lies beyond an axis-aligned face of
//    the (axis-aligned or trapezoid) static polygon by more than totalRadius + eps: every static
//    polygon of the scene has +-x face normals and the boxes also +-y, and b2CollidePolygons returns
//    no points as soon as the max face separation exceeds totalRadius;
//  * a sensor does not overlap if the puck centre is farther than r + skin + eps from the goal box;
//  * b2TimeOfImpact can only report "touching" if the core shapes come within target + tolerance at
//    some time of the sweep; if the swept core AABB of the moving shape stays farther than that (plus
//    the chord-to-arc sagitta of the rotation and eps) from the static core AABB, alpha is 1.
#pragma once
#include "hk_world.cuh"

namespace hk {

#define HK_FAST_EPS 0.005f
// bail reason -> work class of the general tier (hk_lib.cu sorts the slow queue by class so that the lanes of a
// warp do the same kind of work): 0 puck against a racket (keep/shoot ticks; these go through the touch tier first),
// 1 racket against statics, 2 puck against statics / sensors, 3 other
#if defined(HK_FAST_DEBUG) && !defined(__CUDA_ARCH__)
extern long long g_fast_bail[16];
#define HK_BAIL(k) do { g_fast_bail[k]++; e.bailKind = (k); return false; } while (0)
#else
#define HK_BAIL(k) do { e.bailKind = (k); return false; } while (0)
#endif
HK_HD int bailClass(int kind) {
  if (kind == 0 || kind == 4) return 0;  // puck against a racket (keep/shoot ticks, plain hits): the touch tier
  if (kind == 6 || kind == 9 || kind == 8) return 1;
  if (kind == 2 || kind == 3 || kind == 10) return 2;
  return 3;
}

// PUCK_RACKET = false: the contact-free fast tier.  PUCK_RACKET = true (touch tier): the puck x racket pairs are
// updated exactly (b2Contact::Update with manifold, warm-start ids, BeginContact) and may touch; every other pair
// must still be provably clear.
template <bool PUCK_RACKET>
HK_NI_FASTW1 bool collideFast(const Scene& S, const Config& cfg, const Cache& cache, Env& e) {
  int i = 0;
  const uint32_t ov = e.ncontacts > 0 ? pairOverlapBits(S, e) : 0u;  // proxies do not move during Collide
  while (i < e.ncontacts) {
    int pid = clistGet(e.clist, i);
    const uint32_t bit = 1u << pid;
    int fA = S.pairFA[pid], fB = S.pairFB[pid];
    int bA = fixtureBody(fA), bB = fixtureBody(fB);
    bool activeA = bA >= 0 && e.b[bA].awake;
    bool activeB = bB >= 0 && e.b[bB].awake;
    if (!activeA && !activeB) {
      // a sleeping pair that still touches would have to be solved if something wakes it: not a fast tick
      if ((e.touch & bit) && !(HK_PAIRS_SENSOR & bit)) HK_BAIL(1);
      ++i;
      continue;
    }
    if (!(ov & bit)) {
      clistRemoveAt(e, i);
      e.exist &= ~bit;
      e.touch &= ~bit;
      setCount(e, pid, 0);
      continue;
    }
    if (PUCK_RACKET && fB == F_PUCK && fA >= F_R1) {
      updateContact(S, cfg, cache, e, pid);
      ++i;
      continue;
    }
    e.enabled |= bit;
    const bool wasTouching = (e.touch & bit) != 0;
    bool touching;
    if (HK_PAIRS_SENSOR & bit) {
      AABB a = staticCoreAABB(S, fA);
      V2 c = e.b[B_PUCK].p;
      AABB pb;
      pb.lx = pb.hx = c.x;
      pb.ly = pb.hy = c.y;
      float gap = aabbGap(a, pb);
      if (gap > S.puckRadius + HK_POLYGON_RADIUS + HK_FAST_EPS) touching = false;
      else HK_BAIL(2);  // needs the GJK test
    } else if (fB == F_PUCK) {
      Manifold m;
      collidePolygonCircle(&m, S.poly[fA], fixtureXf(S, e, fA), e.b[B_PUCK].p, S.puckRadius);
      if (m.count > 0) HK_BAIL(3 + (fA >= F_R1 ? 1 : 0));
      setSep(e, pid, m.sepBound, m.sepNormal);
      touching = false;
    } else {
      if (bA >= 0) HK_BAIL(5);  // racket x racket: general path
      // the face separation doubles as the distance bound of the TOI proof (toiProvablySeparated); 0.001 covers the
      // rounding of this evaluation order against the one a real face separation would have
      V2 nrm;
      const float gap = polyStaticFaceGap(S, fA, S.poly[fB], bodyXf(e.b[bB]), &nrm);
      setSep(e, pid, gap - 0.001f, nrm);
      if (gap > 2.0f * HK_POLYGON_RADIUS + 0.0005f) {
        touching = false;
      } else {
        // corner against corner: a racket face may separate the shapes.  This is b2CollidePolygons' own second
        // search (same function, same arguments): above totalRadius it returns without manifold points.
        int edgeB = 0;
        const float sB = findMaxSeparation(&edgeB, S.poly[fB], bodyXf(e.b[bB]), S.poly[fA], staticXf(S, fA));
        if (!(sB > 2.0f * HK_POLYGON_RADIUS)) HK_BAIL(6);
        touching = false;
        if (sB - 0.001f > e.sepBound[pid]) {  // distance bound without a fixed direction (the racket's face turns with it)
          e.sepBound[pid] = sB - 0.001f;
          e.sepNormal[pid] = mk(0.0f, 0.0f);
        }
      }
    }
    if (!(HK_PAIRS_SENSOR & bit)) {
      setCount(e, pid, 0);
      if (touching != wasTouching) {
        if (bA >= 0) setAwake(e.b[bA], true);
        if (bB >= 0) setAwake(e.b[bB], true);
      }
    }
    if (touching) e.touch |= bit; else e.touch &= ~bit;
    if (!wasTouching && touching) beginContact(cfg, e, pid);
    ++i;
  }
  return true;
}

// synchronizeFixtures that also keeps the tight swept box; q0 = rotation at the sweep start (== b.q before the move)
HK_NI_FASTW2 void synchronizeFixturesKeep(const Scene& S, Env& e, int bi, Rot q0, AABB* keep) {
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
  *keep = comb;
  moveProxy(e, bi, comb, b.p - xf1.p);
}

HK_NI_FASTW bool worldStepFast(const Scene& S, const Config& cfg, Env& e, float h) {
  e.enabled = 0xFFFFFFFFu;
  e.nmf = 0;
  e.sepValid = 0;
  if (e.moved & 8u) {
    e.moved &= ~8u;
    findNewContacts(S, e);
  }
  Cache none;
  none.base = nullptr;
  none.stride = 0;
  if (!collideFast<false>(S, cfg, none, e)) return false;  // bailKind set by collideFast
  // ---- b2World::Solve with no constraints: every awake body is its own island ----
  Rot q0[3];
  for (int bi = 2; bi >= 0; --bi) {
    Body& b = e.b[bi];
    b.island = false;
    if (!b.awake) continue;
    b.island = true;
    q0[bi] = b.q;
    b.c0 = b.c;
    b.a0 = b.a;
    b.v += h * (1.0f * mk(0.0f, 0.0f) + S.invMass[bi] * b.f);
    b.w += h * S.invI[bi] * b.tq;
    b.v *= fclamp(1.0f - h * b.ldamp, 0.0f, 1.0f);
    b.w *= fclamp(1.0f - h * b.adamp, 0.0f, 1.0f);
    integratePosition(b, h);
    syncTransform(S, b, bi);
    const float linTolSqr = HK_LINEAR_SLEEP_TOL * HK_LINEAR_SLEEP_TOL;
    const float angTolSqr = HK_ANGULAR_SLEEP_TOL * HK_ANGULAR_SLEEP_TOL;
    float minSleepTime;
    if (b.w * b.w > angTolSqr || dot(b.v, b.v) > linTolSqr) {
      b.sleep = 0.0f;
      minSleepTime = 0.0f;
    } else {
      b.sleep += h;
      minSleepTime = fmin2(HK_MAXFLOAT, b.sleep);
    }
    if (minSleepTime >= HK_TIME_TO_SLEEP) setAwake(b, false);
  }
  for (int bi = 2; bi >= 0; --bi)
    if (e.b[bi].island) synchronizeFixturesKeep(S, e, bi, q0[bi], &e.swept[bi]);
  findNewContacts(S, e);
  // ---- b2World::SolveTOI: prove alpha == 1 for every candidate ----
  uint32_t cand = e.exist & HK_PAIRS_TOI;
  if (cand) {
    for (int i = 0; i < e.ncontacts; ++i) {
      int pid = clistGet(e.clist, i);
      if (!((cand >> pid) & 1u)) continue;
      int fA = S.pairFA[pid], fB = S.pairFB[pid];
      int bi = fB - F_R1;
      const Body& B = e.b[bi];
      if (!B.awake) continue;
      if (!B.island) HK_BAIL(7);  // woken after the solve (new contact): its sweep is stale, take the general path
      const float r = bi == B_PUCK ? S.puckRadius : HK_POLYGON_RADIUS;
      if (!toiProvablySeparated(S, e, pid, fA, bi, r)) HK_BAIL(9 + (bi == B_PUCK ? 1 : 0));
    }
  }
  for (int bi = 0; bi < 3; ++bi) {
    e.b[bi].f = mk(0.0f, 0.0f);
    e.b[bi].tq = 0.0f;
  }
  return true;
}

// ---- touch tier: ticks whose only touching solid contacts are puck x racket (every keep/shoot tick: the puck is
// teleported into the racket, hockey_env.py:618-620,668-680) and that provably have no continuous-collision event.
// Collide is the fast one plus an exact update of the puck x racket pairs; the island solve is the general one
// (hk_world.cuh: one contact, one manifold point -> the register-resident sweep loop, then the position iterations);
// SolveTOI is replaced by the fast tier's proofs.  Returns false without side effects that matter otherwise.
// The touch step in three pieces (k_touch walks them with block barriers in between; worldStepTouch is their sequence).
HK_HD bool worldStepTouchCollide(const Scene& S, const Config& cfg, const Cache& cache, Env& e) {
  e.enabled = 0xFFFFFFFFu;
  e.nmf = 0;
  e.toiEventSeen = false;
  e.toiPreFlag = 0;
  e.sepValid = 0;
  if (e.moved & 8u) {
    e.moved &= ~8u;
    findNewContacts(S, e);
  }
  return collideFast<true>(S, cfg, cache, e);
}
HK_HD bool worldStepTouchSolve(const Scene& S, const Config& cfg, const Cache& cache, Env& e, float h) {
  solveIslands(S, cfg, cache, e, h, 6 * 30, 2 * 30);
  if (e.aborted) HK_BAIL(11);
  return true;
}
HK_HD bool worldStepTouchFinish(const Scene& S, const Cache& cache, Env& e) {
  uint32_t cand = e.exist & HK_PAIRS_TOI;
  if (cand) {
    for (int i = 0; i < e.ncontacts; ++i) {
      int pid = clistGet(e.clist, i);
      if (!((cand >> pid) & 1u)) continue;
      int fA = S.pairFA[pid], fB = S.pairFB[pid];
      int bi = fB - F_R1;
      const Body& B = e.b[bi];
      if (!B.awake) continue;
      if (!B.island) HK_BAIL(7);
      const float r = bi == B_PUCK ? S.puckRadius : HK_POLYGON_RADIUS;
      if (!toiProvablySeparated(S, e, pid, fA, bi, r)) HK_BAIL(9 + (bi == B_PUCK ? 1 : 0));
    }
  }
  e.b[0].island = e.b[1].island = e.b[2].island = false;
  worldStepFinish(cache, e);
  return true;
}
HK_HD_NOINLINE bool worldStepTouch(const Scene& S, const Config& cfg, const Cache& cache, Env& e, float h) {
  return worldStepTouchCollide(S, cfg, cache, e) && worldStepTouchSolve(S, cfg, cache, e, h) && worldStepTouchFinish(S, cache, e);
}
HK_HD bool envStepTouch(const Scene& S, const Config& cfg, const Cache& cache, Env& e, const float action[8]) {
  envStepActions(S, cfg, e, action);
  e.sweepBudget = 1 << 20;
  e.allowToiEvents = true;
  e.aborted = false;
  if (!worldStepTouch(S, cfg, cache, e, (float)(1.0 / HK_FPS))) return false;
  envStepAfterWorld(e);
  return true;
}

// fast variant of envStep: returns false if the tick needs the general path (e is then garbage)
HK_HD bool envStepFast(const Scene& S, const Config& cfg, Env& e, const float action[8]) {
  Body &p1 = e.b[B_R1], &p2 = e.b[B_R2], &puck = e.b[B_PUCK];
  if (cfg.keep_mode && (e.has1 > 1 || e.has2 > 1)) HK_BAIL(0);  // keep/shoot ticks always have a deep contact
  applyTranslation(S, p1, B_R1, action[0], action[1], true);
  applyRotation(S, p1, B_R1, action[2]);
  applyTranslation(S, p2, B_R2, action[4], action[5], false);
  applyRotation(S, p2, B_R2, action[6]);
  {
    double vx = puck.v.x, vy = puck.v.y;
    double puck_speed = sqrt(vx * vx + vy * vy);
    puck.ldamp = puck_speed > HK_MAX_PUCK_SPEED ? 10.0f : 0.05f;
  }
  if (!worldStepFast(S, cfg, e, (float)(1.0 / HK_FPS))) return false;
  if (e.time >= maxTimesteps(e.mode)) e.done = true;
  e.time += 1;
  ++e.tick;
  return true;
}

}  // namespace hk
