// msv_device.cuh -- device-side geometry / contact / TOI primitives of the
// batched masurvival step kernel (sm_100a).
//
// Every routine is the float32 arithmetic of the Box2D v2.3.x function it
// names, specialised to the only body kinds the masurvival step path creates
// (SURVEY.md Appendix A.2): dynamic circles (agents), static oriented boxes
// (boxes at angle 0, the four room walls) and sensor circles (items).  There
// are no body/fixture/contact objects: a static box is 9 scalars, an agent is
// a column of shared memory, a contact is an index into a fixed pair matrix.
// Compiled with -fmad=false so results equal an SSE2 (no-FMA) build.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>

#define DEV __device__ __forceinline__

// b2Settings.h
#define B2_PI 3.14159265359f
#define B2_EPS FLT_EPSILON
#define B2_LINEAR_SLOP 0.005f
#define B2_POLY_RADIUS (2.0f * B2_LINEAR_SLOP)
#define B2_AABB_EXT 0.1f
#define B2_AABB_MULT 2.0f
#define B2_VEL_THRESHOLD 1.0f
#define B2_MAX_LIN_CORR 0.2f
#define B2_MAX_TRANSLATION 2.0f
#define B2_MAX_ROTATION (0.5f * B2_PI)
#define B2_BAUMGARTE 0.2f
#define B2_TOI_BAUMGARTE 0.75f
#define B2_TIME_TO_SLEEP 0.5f
#define B2_LIN_SLEEP_TOL 0.01f
#define B2_ANG_SLEEP_TOL (2.0f / 180.0f * B2_PI)
#define B2_MAX_SUBSTEPS 8

struct f2 { float x, y; };
DEV f2 mk2(float x, float y) { f2 r; r.x = x; r.y = y; return r; }
DEV f2 vadd(f2 a, f2 b) { return mk2(a.x + b.x, a.y + b.y); }
DEV f2 vsub(f2 a, f2 b) { return mk2(a.x - b.x, a.y - b.y); }
DEV f2 vmul(float s, f2 a) { return mk2(s * a.x, s * a.y); }
DEV f2 vneg(f2 a) { return mk2(-a.x, -a.y); }
DEV float vdot(f2 a, f2 b) { return a.x * b.x + a.y * b.y; }
DEV float vcross(f2 a, f2 b) { return a.x * b.y - a.y * b.x; }
DEV f2 cross_vs(f2 a, float s) { return mk2(s * a.y, -s * a.x); }
DEV f2 cross_sv(float s, f2 a) { return mk2(-s * a.y, s * a.x); }
DEV float vlen2(f2 a) { return a.x * a.x + a.y * a.y; }
DEV float vlen(f2 a) { return sqrtf(a.x * a.x + a.y * a.y); }
DEV float vnormalize(f2& a) {
  float length = vlen(a);
  if (length < B2_EPS) return 0.0f;
  float inv = 1.0f / length;
  a.x *= inv; a.y *= inv;
  return length;
}
DEV float fmin_(float a, float b) { return a < b ? a : b; }
DEV float fmax_(float a, float b) { return a > b ? a : b; }
DEV float fclamp_(float a, float lo, float hi) { return fmax_(lo, fmin_(a, hi)); }

// b2Rot::Set: sinf/cosf evaluated in double and rounded (correctly rounded
// float on every platform the oracle runs on).
__device__ __noinline__ f2 rot_sc(float angle) {   // (sin, cos), returned in registers
  double ds, dc;
  sincos((double)angle, &ds, &dc);
  return mk2((float)ds, (float)dc);
}
DEV void rot_set(float angle, float& s, float& c) { f2 r = rot_sc(angle); s = r.x; c = r.y; }
DEV f2 qmul(float s, float c, f2 v) { return mk2(c * v.x - s * v.y, s * v.x + c * v.y); }
DEV f2 qmulT(float s, float c, f2 v) { return mk2(c * v.x + s * v.y, -s * v.x + c * v.y); }

// sim.from_polar (simulation.py:20-23): R.angle = angle; R * b2Vec2(L, 0)
DEV f2 from_polar(float L, float angle) {
  float s, c; rot_set(angle, s, c);
  return mk2(c * L + (-s) * 0.0f, s * L + c * 0.0f);
}

// A static oriented box: position, rotation, half extents, normal scales
// (ax, ay == 1 for b2PolygonShape::SetAsBox; x*(1/x) after ::Set re-hulls it)
// and the vertex-order rotation (0 SetAsBox, 1 re-hulled; SURVEY Q8).
struct SBox { float px, py, qs, qc, hx, hy, ax, ay, ang; int rot; };

DEV f2 sb_vert(const SBox& b, int k) {
  int j = (k + b.rot) & 3;
  return mk2((j == 1 || j == 2) ? b.hx : -b.hx, (j >= 2) ? b.hy : -b.hy);
}
DEV f2 sb_normal(const SBox& b, int k) {
  int j = (k + b.rot) & 3;
  if (j == 0) return mk2(0.0f, -b.ax);
  if (j == 1) return mk2(b.ay, 0.0f);
  if (j == 2) return mk2(0.0f, b.ax);
  return mk2(-b.ay, 0.0f);
}
DEV f2 sb_mul(const SBox& b, f2 v) {   // b2Mul(xf, v)
  return mk2((b.qc * v.x - b.qs * v.y) + b.px, (b.qs * v.x + b.qc * v.y) + b.py);
}
DEV f2 sb_mulT(const SBox& b, f2 v) {  // b2MulT(xf, v)
  float px = v.x - b.px, py = v.y - b.py;
  return mk2(b.qc * px + b.qs * py, -b.qs * px + b.qc * py);
}
// normal scales of a re-hulled box: normalize(cross(edge,1)) componentwise
DEV void sb_set_shape(SBox& b, float hx, float hy, int rehulled) {
  b.hx = hx; b.hy = hy; b.rot = rehulled ? 1 : 0;
  if (rehulled) {
    float ex = hx + hx, ey = hy + hy;  // edge lengths, exact
    b.ax = ex * (1.0f / ex);
    b.ay = ey * (1.0f / ey);
  } else { b.ax = 1.0f; b.ay = 1.0f; }
}
// b2PolygonShape::ComputeAABB + b2DynamicTree::CreateProxy (fat AABB)
DEV void sb_fat(const SBox& b, float out[4]) {
  f2 lo = sb_mul(b, sb_vert(b, 0)), hi = lo;
#pragma unroll
  for (int i = 1; i < 4; ++i) {
    f2 v = sb_mul(b, sb_vert(b, i));
    lo = mk2(fmin_(lo.x, v.x), fmin_(lo.y, v.y));
    hi = mk2(fmax_(hi.x, v.x), fmax_(hi.y, v.y));
  }
  out[0] = (lo.x - B2_POLY_RADIUS) - B2_AABB_EXT; out[1] = (lo.y - B2_POLY_RADIUS) - B2_AABB_EXT;
  out[2] = (hi.x + B2_POLY_RADIUS) + B2_AABB_EXT; out[3] = (hi.y + B2_POLY_RADIUS) + B2_AABB_EXT;
}

DEV bool aabb_overlap(const float* a, const float* b) {  // b2TestOverlap(AABB)
  float d1x = b[0] - a[2], d1y = b[1] - a[3];
  float d2x = a[0] - b[2], d2y = a[1] - b[3];
  if (d1x > 0.0f || d1y > 0.0f) return false;
  if (d2x > 0.0f || d2y > 0.0f) return false;
  return true;
}

// ---------------------------------------------------------------- ray casts
// b2CircleShape::RayCast with maxFraction = 1 (circle centred on its body)
DEV bool ray_circle(f2 center, float radius, f2 p1, f2 p2, float& fraction) {
  f2 s = vsub(p1, center);
  float b = vdot(s, s) - radius * radius;
  f2 r = vsub(p2, p1);
  float c = vdot(s, r);
  float rr = vdot(r, r);
  float sigma = c * c - rr * b;
  if (sigma < 0.0f || rr < B2_EPS) return false;
  float a = -(c + sqrtf(sigma));
  if (0.0f <= a && a <= 1.0f * rr) { fraction = a / rr; return true; }
  return false;
}
// b2PolygonShape::RayCast with maxFraction = 1
// (out-of-line functions take the box BY VALUE: by reference it would be spilled to the stack)
// returns the hit fraction in [0, 1], or -1 for a miss (by value: no stack traffic at the call)
__device__ __noinline__ float ray_box_f(const SBox bx, f2 p1w, f2 p2w) {
  f2 p1 = sb_mulT(bx, p1w), p2 = sb_mulT(bx, p2w);
  f2 d = vsub(p2, p1);
  float lower = 0.0f, upper = 1.0f;
  int index = -1;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f2 n = sb_normal(bx, i);
    float numerator = vdot(n, vsub(sb_vert(bx, i), p1));
    float denominator = vdot(n, d);
    if (denominator == 0.0f) {
      if (numerator < 0.0f) return -1.0f;
    } else {
      if (denominator < 0.0f && numerator < lower * denominator) { lower = numerator / denominator; index = i; }
      else if (denominator > 0.0f && numerator < upper * denominator) { upper = numerator / denominator; }
    }
    if (upper < lower) return -1.0f;
  }
  if (index >= 0) return lower;
  return -1.0f;
}
DEV bool ray_box(const SBox& bx, f2 p1w, f2 p2w, float& fraction) {
  float f = ray_box_f(bx, p1w, p2w);
  if (f < 0.0f) return false;
  fraction = f; return true;
}

// ---------------------------------------------------------------- manifolds
struct Manifold { int type; f2 localNormal, localPoint; };  // type 0 circles, 1 faceA

// b2CollideCircles (both centres at their body origins)
DEV bool collide_circles(f2 cA, f2 cB, float rA, float rB, Manifold& m) {
  f2 d = vsub(cB, cA);
  float distSqr = vdot(d, d);
  float radius = rA + rB;
  if (distSqr > radius * radius) return false;
  m.type = 0; m.localNormal = mk2(0.0f, 0.0f); m.localPoint = mk2(0.0f, 0.0f);
  return true;
}
// b2CollidePolygonAndCircle (polygon = static box A, circle B at cW)
DEV bool collide_box_circle(const SBox& A, f2 cW, float rB, Manifold& m) {
  f2 cLocal = sb_mulT(A, cW);
  int normalIndex = 0;
  float separation = -FLT_MAX;
  float radius = B2_POLY_RADIUS + rB;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float s = vdot(sb_normal(A, i), vsub(cLocal, sb_vert(A, i)));
    if (s > radius) return false;
    if (s > separation) { separation = s; normalIndex = i; }
  }
  int vi1 = normalIndex, vi2 = vi1 + 1 < 4 ? vi1 + 1 : 0;
  f2 v1 = sb_vert(A, vi1), v2 = sb_vert(A, vi2);
  m.type = 1;
  if (separation < B2_EPS) {
    m.localNormal = sb_normal(A, normalIndex);
    m.localPoint = vmul(0.5f, vadd(v1, v2));
    return true;
  }
  float u1 = vdot(vsub(cLocal, v1), vsub(v2, v1));
  float u2 = vdot(vsub(cLocal, v2), vsub(v1, v2));
  if (u1 <= 0.0f) {
    if (vlen2(vsub(cLocal, v1)) > radius * radius) return false;
    m.localNormal = vsub(cLocal, v1); vnormalize(m.localNormal);
    m.localPoint = v1;
  } else if (u2 <= 0.0f) {
    if (vlen2(vsub(cLocal, v2)) > radius * radius) return false;
    m.localNormal = vsub(cLocal, v2); vnormalize(m.localNormal);
    m.localPoint = v2;
  } else {
    f2 faceCenter = vmul(0.5f, vadd(v1, v2));
    float sep = vdot(vsub(cLocal, faceCenter), sb_normal(A, vi1));
    if (sep > radius) return false;
    m.localNormal = sb_normal(A, vi1);
    m.localPoint = faceCenter;
  }
  return true;
}

// ---------------------------------------------------- GJK / time of impact
// proxy A = the 4 vertices of a static box, proxy B = one point (the circle
// centre): every vertex has indexB == 0 and wB == pB.
struct SimplexV { f2 wA, w; float a; int indexA; };
struct SimplexCache { float metric; int count; int indexA[3]; };

DEV int box_support(const SBox& b, f2 d) {  // b2DistanceProxy::GetSupport
  int best = 0; float bestValue = vdot(sb_vert(b, 0), d);
#pragma unroll
  for (int i = 1; i < 4; ++i) {
    float value = vdot(sb_vert(b, i), d);
    if (value > bestValue) { best = i; bestValue = value; }
  }
  return best;
}

DEV float simplex_metric(const SimplexV* v, int count) {
  if (count == 2) return vlen(vsub(v[0].w, v[1].w));
  if (count == 3) return vcross(vsub(v[1].w, v[0].w), vsub(v[2].w, v[0].w));
  return 0.0f;
}

// b2Distance(useRadii = false): returns distance, updates the cache.  The simplex (at most three
// box vertices against the one point) is three named records, every branch of b2Simplex::Solve2 /
// Solve3 addresses them statically, so the whole state stays in registers (an indexed SimplexV[3]
// lived in local memory); the arithmetic and the order of operations are those of b2Distance.
struct SimplexV3 { SimplexV v0, v1, v2; int count; };
DEV float simplex_metric3(const SimplexV3& s) {
  if (s.count == 2) return vlen(vsub(s.v0.w, s.v1.w));
  if (s.count == 3) return vcross(vsub(s.v1.w, s.v0.w), vsub(s.v2.w, s.v0.w));
  return 0.0f;
}
DEV SimplexV simplex_vertex(const SBox& A, f2 pB, int indexA, float a) {
  SimplexV v; v.indexA = indexA; v.wA = sb_mul(A, sb_vert(A, indexA)); v.w = vsub(pB, v.wA); v.a = a;
  return v;
}
DEV float gjk_distance(SimplexCache& cache, const SBox& A, f2 pB) {
  SimplexV3 s; s.count = cache.count;
  s.v0 = simplex_vertex(A, pB, 0, 0.0f); s.v1 = s.v0; s.v2 = s.v0;
  if (s.count > 0) s.v0 = simplex_vertex(A, pB, cache.indexA[0], 0.0f);   // b2Simplex::ReadCache
  if (s.count > 1) s.v1 = simplex_vertex(A, pB, cache.indexA[1], 0.0f);
  if (s.count > 2) s.v2 = simplex_vertex(A, pB, cache.indexA[2], 0.0f);
  if (s.count > 1) {
    float metric1 = cache.metric, metric2 = simplex_metric3(s);
    if (metric2 < 0.5f * metric1 || 2.0f * metric1 < metric2 || metric2 < B2_EPS) s.count = 0;
  }
  if (s.count == 0) { s.v0 = simplex_vertex(A, pB, 0, 1.0f); s.count = 1; }
  int iter = 0;
  while (iter < 20) {
    const int saveCount = s.count;
    const int save0 = s.v0.indexA, save1 = s.v1.indexA, save2 = s.v2.indexA;
    if (s.count == 2) {  // b2Simplex::Solve2
      f2 w1 = s.v0.w, w2 = s.v1.w, e12 = vsub(w2, w1);
      float d12_2 = -vdot(w1, e12);
      if (d12_2 <= 0.0f) { s.v0.a = 1.0f; s.count = 1; }
      else {
        float d12_1 = vdot(w2, e12);
        if (d12_1 <= 0.0f) { s.v1.a = 1.0f; s.count = 1; s.v0 = s.v1; }
        else { float inv = 1.0f / (d12_1 + d12_2); s.v0.a = d12_1 * inv; s.v1.a = d12_2 * inv; }
      }
    } else if (s.count == 3) {  // b2Simplex::Solve3
      f2 w1 = s.v0.w, w2 = s.v1.w, w3 = s.v2.w;
      f2 e12 = vsub(w2, w1);
      float w1e12 = vdot(w1, e12), w2e12 = vdot(w2, e12);
      float d12_1 = w2e12, d12_2 = -w1e12;
      f2 e13 = vsub(w3, w1);
      float w1e13 = vdot(w1, e13), w3e13 = vdot(w3, e13);
      float d13_1 = w3e13, d13_2 = -w1e13;
      f2 e23 = vsub(w3, w2);
      float w2e23 = vdot(w2, e23), w3e23 = vdot(w3, e23);
      float d23_1 = w3e23, d23_2 = -w2e23;
      float n123 = vcross(e12, e13);
      float d123_1 = n123 * vcross(w2, w3);
      float d123_2 = n123 * vcross(w3, w1);
      float d123_3 = n123 * vcross(w1, w2);
      if (d12_2 <= 0.0f && d13_2 <= 0.0f) { s.v0.a = 1.0f; s.count = 1; }
      else if (d12_1 > 0.0f && d12_2 > 0.0f && d123_3 <= 0.0f) {
        float inv = 1.0f / (d12_1 + d12_2); s.v0.a = d12_1 * inv; s.v1.a = d12_2 * inv; s.count = 2;
      } else if (d13_1 > 0.0f && d13_2 > 0.0f && d123_2 <= 0.0f) {
        float inv = 1.0f / (d13_1 + d13_2); s.v0.a = d13_1 * inv; s.v2.a = d13_2 * inv; s.count = 2; s.v1 = s.v2;
      } else if (d12_1 <= 0.0f && d23_2 <= 0.0f) { s.v1.a = 1.0f; s.count = 1; s.v0 = s.v1; }
      else if (d13_1 <= 0.0f && d23_1 <= 0.0f) { s.v2.a = 1.0f; s.count = 1; s.v0 = s.v2; }
      else if (d23_1 > 0.0f && d23_2 > 0.0f && d123_1 <= 0.0f) {
        float inv = 1.0f / (d23_1 + d23_2); s.v1.a = d23_1 * inv; s.v2.a = d23_2 * inv; s.count = 2; s.v0 = s.v2;
      } else {
        float inv = 1.0f / (d123_1 + d123_2 + d123_3);
        s.v0.a = d123_1 * inv; s.v1.a = d123_2 * inv; s.v2.a = d123_3 * inv; s.count = 3;
      }
    }
    if (s.count == 3) break;
    f2 d;  // b2Simplex::GetSearchDirection
    if (s.count == 1) d = vneg(s.v0.w);
    else {
      f2 e12 = vsub(s.v1.w, s.v0.w);
      float sgn = vcross(e12, vneg(s.v0.w));
      d = sgn > 0.0f ? cross_sv(1.0f, e12) : cross_vs(e12, 1.0f);
    }
    if (vlen2(d) < B2_EPS * B2_EPS) break;
    const SimplexV nv = simplex_vertex(A, pB, box_support(A, qmulT(A.qs, A.qc, vneg(d))), 0.0f);   // (its .a is set by the next Solve)
    ++iter;
    bool duplicate = (saveCount > 0 && nv.indexA == save0) || (saveCount > 1 && nv.indexA == save1) || (saveCount > 2 && nv.indexA == save2);
    if (duplicate) break;
    if (s.count == 1) { const float a1 = s.v1.a; s.v1 = nv; s.v1.a = a1; } else { const float a2 = s.v2.a; s.v2 = nv; s.v2.a = a2; }   // vertex[count] keeps its stale weight, as in b2Distance
    ++s.count;
  }
  f2 pointA, pointB;  // b2Simplex::GetWitnessPoints
  if (s.count == 1) { pointA = s.v0.wA; pointB = pB; }
  else if (s.count == 2) {
    pointA = vadd(vmul(s.v0.a, s.v0.wA), vmul(s.v1.a, s.v1.wA));
    pointB = vadd(vmul(s.v0.a, pB), vmul(s.v1.a, pB));
  } else {
    pointA = vadd(vadd(vmul(s.v0.a, s.v0.wA), vmul(s.v1.a, s.v1.wA)), vmul(s.v2.a, s.v2.wA));
    pointB = pointA;
  }
  float distance = vlen(vsub(pointA, pointB));
  cache.metric = simplex_metric3(s);
  cache.count = s.count;
  cache.indexA[0] = s.v0.indexA;
  if (s.count > 1) cache.indexA[1] = s.v1.indexA;
  if (s.count > 2) cache.indexA[2] = s.v2.indexA;
  return distance;
}

// b2Sweep::GetTransform for the static box (c0 == c, a0 == a) and the circle
DEV SBox box_at(const SBox& A, float beta) {
  SBox r = A;
  r.px = (1.0f - beta) * A.px + beta * A.px;
  r.py = (1.0f - beta) * A.py + beta * A.py;
  if (A.ang != 0.0f) {
    float angle = (1.0f - beta) * A.ang + beta * A.ang;
    if (angle != A.ang) rot_set(angle, r.qs, r.qc);
  }
  return r;
}
DEV f2 point_at(f2 c0, f2 c, float beta) { return vadd(vmul(1.0f - beta, c0), vmul(beta, c)); }

#define TOI_FAILED 1
#define TOI_OVERLAPPED 2
#define TOI_TOUCHING 3
#define TOI_SEPARATED 4

// make CHECK=1: every indexed access to the environment's shared-memory column (and the fixed-capacity lists
// behind it) is bounds-checked; violations are counted (msv_debug_check_failures) and the index clamped.
// compute-sanitizer is not available on the GPU pool, so this build is the memory-safety evidence.
#ifdef MSV_CHECK
__device__ unsigned long long g_chk[2];   // [0] violations, [1] line of the last one
#define CHK(cond) do { if (!(cond)) { atomicAdd(&g_chk[0], 1ull); g_chk[1] = __LINE__; } } while (0)
__device__ __forceinline__ int chk_idx_(int i, int n, int line) {
  if ((unsigned)i < (unsigned)n) return i;
  atomicAdd(&g_chk[0], 1ull); g_chk[1] = (unsigned long long)line;
  return 0;
}
#define CHK_IDX(i, n) chk_idx_((i), (n), __LINE__)
#else
#define CHK(cond) do { } while (0)
#define CHK_IDX(i, n) (i)
#endif
#ifdef MSV_PROFILE
__device__ unsigned long long g_dbg[8];
// rare-path census: [2k] number of calls, [2k+1] clock64() cycles spent in them (k: 0 generic island solve,
// 1 TOI event, 2 reset, 3 deaths, 4 pickups, 5 use/give, 6 contact numbering, 7 box removal)
__device__ unsigned long long g_cnt[16];
__device__ unsigned long long g_sub[16];   // sub-phase cycle sums inside toi_event (development)
__device__ unsigned long long g_toi[16];   // the longest solve_toi call since the last read: [0] cycles, [1] loop iterations, [2] events run, [3] not touching, [4] identical repeats, [5] cycles in events, [6] cycles in scans
#define TOIPROF(x) x
#define SUB_BEGIN() long long sub_t_ = clock64()
#define SUB(k) do { long long n_ = clock64(); atomicAdd(&g_sub[k], (unsigned long long)(n_ - sub_t_)); sub_t_ = n_; } while (0)
#define SUBCNT(k, v) atomicAdd(&g_sub[k], (unsigned long long)(v))
// maximum duration (cycles << 8 | tag) of a section
#define SUBMAX(k, tag) atomicMax(&g_sub[k], ((unsigned long long)(clock64() - sub_t_) << 8) | (unsigned long long)((tag) & 255))
#define RARE_BEGIN() long long rare_t0_ = clock64()
#define RARE_END(k) do { atomicAdd(&g_cnt[2 * (k)], 1ull); atomicAdd(&g_cnt[2 * (k) + 1], (unsigned long long)(clock64() - rare_t0_)); } while (0)
#else
#define RARE_BEGIN() do { } while (0)
#define RARE_END(k) do { } while (0)
#define SUB_BEGIN() do { } while (0)
#define SUB(k) do { } while (0)
#define SUBCNT(k, v) do { } while (0)
#define SUBMAX(k, tag) do { } while (0)
#define TOIPROF(x)
#endif
// b2TimeOfImpact(proxyA = box, proxyB = circle centre), tMax = 1
struct ToiOut { int state; float t; };
__device__ __noinline__ ToiOut time_of_impact_v(const SBox A, f2 c0, f2 c, float rB) {
  int state = 0; float tOut = 1.0f;
  const float tMax = 1.0f;
#ifdef MSV_PROFILE
  long long dbg_t0 = clock64(); int dbg_roots = 0, dbg_push = 0;
#endif
  float totalRadius = B2_POLY_RADIUS + rB;
  float target = fmax_(B2_LINEAR_SLOP, totalRadius - 3.0f * B2_LINEAR_SLOP);
  float tolerance = 0.25f * B2_LINEAR_SLOP;
  float t1 = 0.0f;
  int iter = 0;
  {
    // First outer iteration, t1 = 0: the sweep positions are exactly (A, c0) and the
    // function returns e_touching at t = 0 iff the GJK distance is in (0, target + tol).
    // GJK on a 4-vertex polygon against a point is exact to ~1e-6, so when the plain
    // point-to-box distance is inside that interval by a 1e-3 margin the outcome is
    // certain and the simplex iteration can be skipped (a body resting in, or wedged
    // into, contact lands here every substep).
    f2 l = sb_mulT(A, c0);
    float dx = fmax_(fabsf(l.x) - A.hx, 0.0f), dy = fmax_(fabsf(l.y) - A.hy, 0.0f);
    float d = sqrtf(dx * dx + dy * dy);
    if (d > 1e-3f && d < (target + tolerance) - 1e-3f) { ToiOut r0; r0.state = TOI_TOUCHING; r0.t = 0.0f; return r0; }
  }
  SimplexCache cache; cache.count = 0;
  for (;;) {
    // One outer iteration is a pure function of (t1, simplex cache).  When it
    // returns to the same (t1, cache) without finishing -- t1 already at tMax and
    // the separating axis within tolerance of target while the true distance is
    // not -- b2TimeOfImpact repeats it verbatim until iter == 20 and reports
    // e_failed at t1; that fixed point is detected and cut short (same result).
    const float t1_in = t1; const SimplexCache cache_in = cache;
    SBox xfA = box_at(A, t1); f2 pB = point_at(c0, c, t1);
    float distance = gjk_distance(cache, xfA, pB);
    if (distance <= 0.0f) { state = TOI_OVERLAPPED; tOut = 0.0f; break; }
    if (distance < target + tolerance) { state = TOI_TOUCHING; tOut = t1; break; }
    // b2SeparationFunction::Initialize: count==1 -> e_points, count==2 -> e_faceA
    int ftype; f2 axis, localPoint = mk2(0.0f, 0.0f); int ptIndexA = 0;
    if (cache.count == 1) {
      ftype = 0; ptIndexA = cache.indexA[0];
      f2 pointA = sb_mul(xfA, sb_vert(xfA, cache.indexA[0]));
      axis = vsub(pB, pointA); vnormalize(axis);
    } else {
      ftype = 1;
      f2 lA1 = sb_vert(xfA, cache.indexA[0]), lA2 = sb_vert(xfA, cache.indexA[1]);
      axis = cross_vs(vsub(lA2, lA1), 1.0f); vnormalize(axis);
      f2 normal = qmul(xfA.qs, xfA.qc, axis);
      localPoint = vmul(0.5f, vadd(lA1, lA2));
      f2 pointA = sb_mul(xfA, localPoint);
      float s = vdot(vsub(pB, pointA), normal);
      if (s < 0.0f) axis = vneg(axis);
    }
    (void)ptIndexA;
    bool done = false;
    float t2 = tMax;
    int pushBackIter = 0;
    for (;;) {
      // FindMinSeparation(t2)
      int indexA = -1; float s2;
      {
        SBox x2 = box_at(A, t2); f2 p2 = point_at(c0, c, t2);
        if (ftype == 0) {
          indexA = box_support(x2, qmulT(x2.qs, x2.qc, axis));
          f2 pointA = sb_mul(x2, sb_vert(x2, indexA));
          s2 = vdot(vsub(p2, pointA), axis);
        } else {
          f2 normal = qmul(x2.qs, x2.qc, axis);
          f2 pointA = sb_mul(x2, localPoint);
          s2 = vdot(vsub(p2, pointA), normal);
        }
      }
      if (s2 > target + tolerance) { state = TOI_SEPARATED; tOut = tMax; done = true; break; }
      if (s2 > target - tolerance) { t1 = t2; break; }
      // Evaluate(indexA, indexB, t)
      auto evaluate = [&](float t) -> float {
        SBox xt = box_at(A, t); f2 pt = point_at(c0, c, t);
        if (ftype == 0) {
          f2 pointA = sb_mul(xt, sb_vert(xt, indexA));
          return vdot(vsub(pt, pointA), axis);
        }
        f2 normal = qmul(xt.qs, xt.qc, axis);
        f2 pointA = sb_mul(xt, localPoint);
        return vdot(vsub(pt, pointA), normal);
      };
      float s1 = evaluate(t1);
      if (s1 < target - tolerance) { state = TOI_FAILED; tOut = t1; done = true; break; }
      if (s1 <= target + tolerance) { state = TOI_TOUCHING; tOut = t1; done = true; break; }
      int rootIterCount = 0;
      float a1 = t1, a2 = t2;
      for (;;) {
        float t;
        if (rootIterCount & 1) t = a1 + (target - s1) * (a2 - a1) / (s2 - s1);
        else t = 0.5f * (a1 + a2);
        ++rootIterCount;
#ifdef MSV_PROFILE
        ++dbg_roots;
#endif
        float s = evaluate(t);
        if (fabsf(s - target) < tolerance) { t2 = t; break; }
        if (s > target) { a1 = t; s1 = s; } else { a2 = t; s2 = s; }
        if (rootIterCount == 50) break;
      }
      ++pushBackIter;
#ifdef MSV_PROFILE
      ++dbg_push;
#endif
      if (pushBackIter == 8) break;
    }
    ++iter;
    if (done) break;
    if (iter == 20) { state = TOI_FAILED; tOut = t1; break; }
    if (t1 == t1_in && cache.count == cache_in.count && cache.metric == cache_in.metric &&
        cache.indexA[0] == cache_in.indexA[0] && (cache.count < 2 || cache.indexA[1] == cache_in.indexA[1]) &&
        (cache.count < 3 || cache.indexA[2] == cache_in.indexA[2])) {
      state = TOI_FAILED; tOut = t1; break;
    }
  }
#ifdef MSV_PROFILE
  atomicAdd(&g_dbg[0], 1ull); atomicMax(&g_dbg[1], (unsigned long long)iter); atomicMax(&g_dbg[2], (unsigned long long)dbg_roots);
  atomicMax(&g_dbg[3], (unsigned long long)dbg_push); atomicMax(&g_dbg[4], (unsigned long long)(clock64() - dbg_t0));
  atomicAdd(&g_dbg[5], (unsigned long long)(clock64() - dbg_t0));
#endif
  ToiOut r; r.state = state; r.t = tOut;
  return r;
}
DEV int time_of_impact(const SBox& A, f2 c0, f2 c, float rB, float& tOut) {
  ToiOut r = time_of_impact_v(A, c0, c, rB);
  tOut = r.t; return r.state;
}

// ------------------------------------------------------------------ Philox
DEV void philox4x32(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3,
                    uint32_t k0, uint32_t k1, uint32_t out[4]) {
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(0xD2511F53u, c0), lo0 = 0xD2511F53u * c0;
    uint32_t hi1 = __umulhi(0xCD9E8D57u, c2), lo1 = 0xCD9E8D57u * c2;
    uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
    c0 = n0; c1 = n1; c2 = n2; c3 = n3;
    k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
  }
  out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
