// hk_math.cuh -- scalar float32 vector math, reproducible trig and Philox for the hockey kernels.
//
// Arithmetic contract (DESIGN.md "Numerics"): every float op is a single IEEE-754 binary32
// operation in the order the Box2D 2.3.0 sources evaluate it; the library is compiled with
// -fmad=false (no FMA contraction), sqrt/div are the correctly rounded CUDA defaults.  That makes
// the kernel bit-comparable with an x86-64 SSE build of the engine (which is what box2d-py ships)
// and with the CPU oracle under oracle/.
#pragma once
#include <stdint.h>
#include <float.h>
#include <math.h>

#if defined(__CUDACC__)
#define HK_HD __host__ __device__ __forceinline__
// The large device helpers are functions in pass 1 of hk_lib.cu and inlined in pass 2 (-DHK_INLINE_ALL; see hk_lib.cu,
// namespace hkinl).  They are tagged by group so that a build can keep one group out of line in pass 2 (-DHK_OUT_<G>) or
// inline it in pass 1 (-DHK_IN_<G>): the A/B switches behind profiles/README.md's inlining table.
#define HK_FN_INLINE __host__ __device__ __forceinline__
#define HK_FN_OUTLINE inline __host__ __device__ __noinline__  // `inline`: one (weak) host definition although both passes of hk_lib.cu hold it
#if defined(HK_INLINE_ALL)
#define HK_HD_NOINLINE HK_FN_INLINE
#else
#define HK_HD_NOINLINE HK_FN_OUTLINE
#endif
#if (defined(HK_INLINE_ALL) && !defined(HK_OUT_RARE)) || defined(HK_IN_RARE)
#define HK_NI_RARE HK_FN_INLINE      // reset, controllers, shoot: run by few lanes per tick
#else
#define HK_NI_RARE HK_FN_OUTLINE
#endif
#if (defined(HK_INLINE_ALL) && !defined(HK_OUT_TOI)) || defined(HK_IN_TOI)
#define HK_NI_TOI HK_FN_INLINE       // b2TimeOfImpact, GJK, separation function
#else
#define HK_NI_TOI HK_FN_OUTLINE
#endif
#if (defined(HK_INLINE_ALL) && !defined(HK_OUT_LOOP)) || defined(HK_IN_LOOP)
#define HK_NI_LOOP HK_FN_INLINE      // register-resident velocity-iteration loops
#else
#define HK_NI_LOOP HK_FN_OUTLINE
#endif
#if (defined(HK_INLINE_ALL) && !defined(HK_OUT_NARROW)) || defined(HK_IN_NARROW)
#define HK_NI_NARROW HK_FN_INLINE    // manifold routines and b2Contact::Update
#else
#define HK_NI_NARROW HK_FN_OUTLINE
#endif
#if (defined(HK_INLINE_ALL) && !defined(HK_OUT_MATH)) || defined(HK_IN_MATH)
#define HK_NI_MATH HK_FN_INLINE      // sin/cos polynomial
#else
#define HK_NI_MATH HK_FN_OUTLINE
#endif
#if (defined(HK_INLINE_ALL) && !defined(HK_OUT_FASTW)) || defined(HK_IN_FASTW)
#define HK_NI_FASTW HK_FN_INLINE     // the fast tier's world step
#else
#define HK_NI_FASTW HK_FN_OUTLINE
#endif
#if (defined(HK_INLINE_ALL) && !defined(HK_OUT_COLLIDE)) || defined(HK_IN_COLLIDE)
#define HK_NI_COLLIDE HK_FN_INLINE   // b2ContactManager::Collide (the contact-list walk)
#else
#define HK_NI_COLLIDE HK_FN_OUTLINE
#endif
#if (defined(HK_INLINE_ALL) && !defined(HK_OUT_POLICY)) || defined(HK_IN_POLICY)
#define HK_NI_POLICY HK_FN_INLINE    // in-kernel controllers
#else
#define HK_NI_POLICY HK_FN_OUTLINE
#endif
#if (defined(HK_INLINE_ALL) && !defined(HK_OUT_EVALMF)) || defined(HK_IN_EVALMF)
#define HK_NI_EVALMF HK_FN_INLINE    // evaluateManifold (the manifold routines' common entry: 4 call sites)
#else
#define HK_NI_EVALMF HK_FN_OUTLINE
#endif
#if (defined(HK_INLINE_ALL) && !defined(HK_OUT_TOIFN)) || defined(HK_IN_TOIFN)
#define HK_NI_TOIFN HK_FN_INLINE     // b2TimeOfImpact itself (2 call sites; its internals are group TOI)
#else
#define HK_NI_TOIFN HK_FN_OUTLINE
#endif
#if defined(HK_IN_FASTW1) && !defined(HK_OUT_FASTW1)
#define HK_NI_FASTW1 HK_FN_INLINE
#elif defined(HK_OUT_FASTW1)
#define HK_NI_FASTW1 HK_FN_OUTLINE
#else
#define HK_NI_FASTW1 HK_NI_FASTW
#endif
#if defined(HK_IN_FASTW2)
#define HK_NI_FASTW2 HK_FN_INLINE
#else
#define HK_NI_FASTW2 HK_NI_FASTW
#endif
#if (defined(HK_INLINE_ALL) && !defined(HK_OUT_FASTA)) || defined(HK_IN_FASTA)
#define HK_NI_FASTA HK_FN_INLINE     // force shaping, info, tick epilogue
#else
#define HK_NI_FASTA HK_FN_OUTLINE
#endif
#if (defined(HK_INLINE_ALL) && !defined(HK_OUT_FASTS)) || defined(HK_IN_FASTS)
#define HK_NI_FASTS HK_FN_INLINE     // proxy AABBs and the pair scan
#else
#define HK_NI_FASTS HK_FN_OUTLINE
#endif
#else
#define HK_HD inline
#define HK_HD_NOINLINE inline
#define HK_NI_FASTW inline
#define HK_NI_EVALMF inline
#define HK_NI_TOIFN inline
#define HK_NI_COLLIDE inline
#define HK_NI_POLICY inline
#define HK_NI_FASTW1 inline
#define HK_NI_FASTW2 inline
#define HK_NI_FASTA inline
#define HK_NI_FASTS inline
#define HK_NI_RARE inline
#define HK_NI_TOI inline
#define HK_NI_LOOP inline
#define HK_NI_NARROW inline
#define HK_NI_MATH inline
#endif

namespace hk {

// ---- b2Settings.h (reference engine constants; box2d-py builds with 16 polygon vertices) -------
#define HK_EPS FLT_EPSILON
#define HK_MAXFLOAT FLT_MAX
#define HK_PI 3.14159265359f
#define HK_LINEAR_SLOP 0.005f
#define HK_POLYGON_RADIUS (2.0f * HK_LINEAR_SLOP)
#define HK_MAX_POLY_VERTS 16
#define HK_VELOCITY_THRESHOLD 1.0f
#define HK_MAX_LINEAR_CORRECTION 0.2f
#define HK_MAX_TRANSLATION 2.0f
#define HK_MAX_ROTATION (0.5f * HK_PI)
#define HK_BAUMGARTE 0.2f
#define HK_TOI_BAUMGARTE 0.75f
#define HK_TIME_TO_SLEEP 0.5f
#define HK_LINEAR_SLEEP_TOL 0.01f
#define HK_ANGULAR_SLEEP_TOL (2.0f / 180.0f * HK_PI)
#define HK_AABB_EXTENSION 0.1f
#define HK_AABB_MULTIPLIER 2.0f
#define HK_MAX_SUBSTEPS 8

struct V2 {
  float x, y;
};
HK_HD V2 mk(float x, float y) {
  V2 r;
  r.x = x;
  r.y = y;
  return r;
}
HK_HD V2 operator+(V2 a, V2 b) { return mk(a.x + b.x, a.y + b.y); }
HK_HD V2 operator-(V2 a, V2 b) { return mk(a.x - b.x, a.y - b.y); }
HK_HD V2 operator-(V2 a) { return mk(-a.x, -a.y); }
HK_HD V2 operator*(float s, V2 a) { return mk(s * a.x, s * a.y); }
HK_HD void operator+=(V2& a, V2 b) {
  a.x += b.x;
  a.y += b.y;
}
HK_HD void operator-=(V2& a, V2 b) {
  a.x -= b.x;
  a.y -= b.y;
}
HK_HD void operator*=(V2& a, float s) {
  a.x *= s;
  a.y *= s;
}
HK_HD float dot(V2 a, V2 b) { return a.x * b.x + a.y * b.y; }
HK_HD float cross(V2 a, V2 b) { return a.x * b.y - a.y * b.x; }
HK_HD V2 cross(V2 a, float s) { return mk(s * a.y, -s * a.x); }
HK_HD V2 cross(float s, V2 a) { return mk(-s * a.y, s * a.x); }
HK_HD float length(V2 a) { return sqrtf(a.x * a.x + a.y * a.y); }
HK_HD float lengthSq(V2 a) { return a.x * a.x + a.y * a.y; }
HK_HD float normalize(V2& a) {
  float len = length(a);
  if (len < HK_EPS) return 0.0f;
  float inv = 1.0f / len;
  a.x *= inv;
  a.y *= inv;
  return len;
}
HK_HD float distanceSq(V2 a, V2 b) {
  V2 c = a - b;
  return dot(c, c);
}
// b2Min/b2Max/b2Clamp/b2Abs are ternaries in Box2D -- keep their NaN/zero-sign behaviour.
HK_HD float fmin2(float a, float b) { return a < b ? a : b; }
HK_HD float fmax2(float a, float b) { return a > b ? a : b; }
HK_HD float fclamp(float a, float lo, float hi) { return fmax2(lo, fmin2(a, hi)); }
HK_HD float fabs2(float a) { return a > 0.0f ? a : -a; }

// sin/cos evaluated in double by a fixed polynomial (fdlibm kernel coefficients, Cody-Waite
// reduction) and rounded to float: equals the correctly rounded sinf/cosf for all but ~1e-8 of
// arguments and is bit-identical on host and device (no libm / libdevice dependence).
HK_NI_MATH void sincos_poly(double x, double* s, double* c) {
  const double kd = rint(x * 0.63661977236758134308);
  const long long k = (long long)kd;
  double r = (x - kd * 1.57079632673412561417e+00) - kd * 6.07710050650619224932e-11;
  const double z = r * r;
  const double ps =
      -1.66666666666666324348e-01 +
      z * (8.33333333332248946124e-03 +
           z * (-1.98412698298579493134e-04 +
                z * (2.75573137070700676789e-06 +
                     z * (-2.50507602534068634195e-08 + z * 1.58969099521155010221e-10))));
  const double pc =
      4.16666666666666019037e-02 +
      z * (-1.38888888888741095749e-03 +
           z * (2.48015872894767294178e-05 +
                z * (-2.75573143513906633035e-07 +
                     z * (2.08757232129817482790e-09 + z * -1.13596475577881948265e-11))));
  const double sr = r + (r * z) * ps;
  const double cr = 1.0 - (0.5 * z - (z * z) * pc);
  switch ((int)(k & 3)) {
    case 0: *s = sr; *c = cr; break;
    case 1: *s = cr; *c = -sr; break;
    case 2: *s = -sr; *c = -cr; break;
    default: *s = -cr; *c = sr; break;
  }
}

struct Rot {
  float s, c;
};
HK_HD Rot rotOf(float angle) {
  double sd, cd;
  sincos_poly((double)angle, &sd, &cd);
  Rot q;
  q.s = (float)sd;
  q.c = (float)cd;
  return q;
}
struct Xf {
  V2 p;
  Rot q;
};
HK_HD V2 mul(Rot q, V2 v) { return mk(q.c * v.x - q.s * v.y, q.s * v.x + q.c * v.y); }
HK_HD V2 mulT(Rot q, V2 v) { return mk(q.c * v.x + q.s * v.y, -q.s * v.x + q.c * v.y); }
HK_HD V2 mul(const Xf& T, V2 v) {
  float x = (T.q.c * v.x - T.q.s * v.y) + T.p.x;
  float y = (T.q.s * v.x + T.q.c * v.y) + T.p.y;
  return mk(x, y);
}
HK_HD V2 mulT(const Xf& T, V2 v) {
  float px = v.x - T.p.x;
  float py = v.y - T.p.y;
  return mk(T.q.c * px + T.q.s * py, -T.q.s * px + T.q.c * py);
}

struct Sweep {
  V2 lc, c0, c;
  float a0, a, alpha0;
  bool rot;  // false: static body or the puck -- the rotation never enters a result (angle 0 resp. circle
             // centred on the body origin with localCenter 0), so the sin/cos evaluation is skipped
};
HK_HD Rot rotIdentity() {
  Rot q;
  q.s = 0.0f;
  q.c = 1.0f;
  return q;
}
HK_HD void sweepXf(const Sweep& s, Xf* xf, float beta) {
  xf->p = (1.0f - beta) * s.c0 + beta * s.c;
  float angle = (1.0f - beta) * s.a0 + beta * s.a;
  xf->q = s.rot ? rotOf(angle) : rotIdentity();
  xf->p -= mul(xf->q, s.lc);
}
HK_HD void sweepAdvance(Sweep& s, float alpha) {
  float beta = (alpha - s.alpha0) / (1.0f - s.alpha0);
  s.c0 = (1.0f - beta) * s.c0 + beta * s.c;
  s.a0 = (1.0f - beta) * s.a0 + beta * s.a;
  s.alpha0 = alpha;
}
HK_HD void sweepNormalize(Sweep& s) {
  float twoPi = 2.0f * HK_PI;
  float d = twoPi * floorf(s.a0 / twoPi);
  s.a0 -= d;
  s.a -= d;
}

struct AABB {
  float lx, ly, hx, hy;
};
HK_HD bool aabbContains(const AABB& a, const AABB& o) {
  return a.lx <= o.lx && a.ly <= o.ly && o.hx <= a.hx && o.hy <= a.hy;
}
HK_HD bool aabbOverlap(const AABB& a, const AABB& b) {
  float d1x = b.lx - a.hx, d1y = b.ly - a.hy, d2x = a.lx - b.hx, d2y = a.ly - b.hy;
  if (d1x > 0.0f || d1y > 0.0f) return false;
  if (d2x > 0.0f || d2y > 0.0f) return false;
  return true;
}

// ---- Philox4x32-10, keyed (seed, global env id, counter, stream) -------------------------------
struct U4 {
  uint32_t x, y, z, w;
};
HK_NI_RARE U4 philox(uint64_t seed, uint64_t env, uint32_t c2, uint32_t c3) {
  uint32_t k0 = (uint32_t)seed, k1 = (uint32_t)(seed >> 32);
  uint32_t c0 = (uint32_t)env, c1 = (uint32_t)(env >> 32);
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    uint64_t p0 = (uint64_t)0xD2511F53u * c0;
    uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c0 = n0;
    c1 = n1;
    c2 = n2;
    c3 = n3;
    k0 += 0x9E3779B9u;
    k1 += 0xBB67AE85u;
  }
  U4 r;
  r.x = c0;
  r.y = c1;
  r.z = c2;
  r.w = c3;
  return r;
}
HK_HD double u53(uint32_t hi, uint32_t lo) {
  return ((double)(hi >> 5) * 67108864.0 + (double)(lo >> 6)) * (1.0 / 9007199254740992.0);
}
HK_HD float u_pm1(uint32_t x) { return (float)(x >> 8) * (1.0f / 8388608.0f) - 1.0f; }
enum { HK_STREAM_RESET = 0, HK_STREAM_OPP = 1, HK_STREAM_ACT = 2, HK_STREAM_PHASE0 = 3, HK_STREAM_ACTOR_NOISE = 4, HK_STREAM_TD3_TARGET = 5 };  // 4: hk_actor.cuh NoiseKey; 5: hk_td3.cuh target noise

}  // namespace hk
