// CUDA kernels of the distributed ray-tracing hot path (sm_100a).
//
//   render_wave<R>    : persistent, phase-locked CTAs working through ray pools.  Replaces the
//       sample loop of renderImage (render_final_project.cpp:1062-1212) and the whole recursive
//       rayColor (487-961): camera ray with thin-lens DOF, closest-hit search over the flattened
//       primitives (+ LBVH traversal for triangle meshes), Fresnel refraction, mirror / glossy
//       reflection lobes, per-light shadow rays (point / rectangle / sphere lights),
//       Oren-Nayar / Cook-Torrance / Lambert+Phong shading, nearest-texel texture fetch through
//       CUDA texture objects, emissive shapes, motion-blur re-traces.  Every rayColor invocation
//       only ever ADDS a k-weighted term to the sample's colour, so the order the tree is
//       walked in does not matter.
//   cloud_corners<R>  : skyColor/cloudColor (146-192) + noise.h per PIXEL CORNER.
//       getPerspEyeRay takes int pixel coordinates (helpers.h:320, quirk Q1), so
//       every sample of a pixel that misses the scene asks for the same background
//       colour; it is evaluated once per corner instead of once per sample.
//   resolve           : sample average, clamp, *255, float->u8 truncation, y-flip
//       (render_final_project.cpp:1213-1217 + helpers.h:174-195).
#pragma once
#include "drt_device.cuh"
#include "drt_launch.h"
#include <cstddef>
#ifdef DRT_PASS_STATS
#include <cstdio>
#endif

#ifndef DRT_FORCE_TREE
#define DRT_FORCE_TREE 0   // diagnostic: 1 walks the replayed reference tree for every ray
#endif

namespace drt {


// One pending rayColor invocation: 64 bytes in the reference precision (48 in single), four 16-byte words.  Every ray
// is written to the CTA pool once and stays in its slot until it is finished: TRACE reads it, and when it hit something
// SHADE reads it again through the 16-byte hit record (HitRef) -- the record size is DRAM traffic.
template <typename R>
struct alignas(16) Task {
  Vec<R> org, dir;
  float k;
  uint32_t path;
  float dt;              // time offset of this trace (0 for the primary trace); the y shift of "rectangle" shapes in a
                         // reference-mode blur re-trace is a function of it (blurVal)
  unsigned char depth;   // remaining recursion depth (<= 32)
  unsigned char bits;    // bit0: on the "last invocation" chain that decides in_motion (quirk Q4); bit1: root ray of the primary trace
  unsigned short slot;   // sample slot inside the CTA's batch
};
#define TASK_CHAIN 1
#define TASK_ROOT 2
static_assert(sizeof(Task<double>) == 64 && sizeof(Task<float>) == 48, "ray records are whole 16-byte words");
static_assert(offsetof(Task<double>, depth) >= 48 && offsetof(Task<float>, depth) >= 32, "depth lives in the last word (poolStoreEmpty)");

// The CTA ray pool is stored as planes of 16-byte words: word w of record i lives at plane w, slot i.  Warps pop and push
// runs of neighbouring slots, so every load / store instruction of a warp covers 512 contiguous bytes (whole sectors)
// instead of 32 half-used sectors at a 64-byte stride.  The records bypass the L1, which is better spent on the geom /
// material records and the local-memory frames: stores keep the record in the L2 under the normal policy (it is read back
// within a pass or two), the loads are streaming ones (measured: TRACE's load with the normal policy, so that SHADE's
// second read of a ray that hit finds it in the L2 more often, 740-742 vs 744-746 Msamples/s).
template <typename T, bool STREAM>
__device__ __forceinline__ void poolLoad(T& dst, const uint4* planes, const size_t cap, const int i) {
  uint4* d = reinterpret_cast<uint4*>(&dst);
#pragma unroll
  for (int w = 0; w < (int)(sizeof(T) / 16); w++) d[w] = STREAM ? __ldcs(planes + w * cap + i) : __ldcg(planes + w * cap + i);
}
template <typename T>
__device__ __forceinline__ void poolStore(uint4* planes, const size_t cap, const int i, const T& src) {
  const uint4* q = reinterpret_cast<const uint4*>(&src);
#pragma unroll
  for (int w = 0; w < (int)(sizeof(T) / 16); w++) __stcg(planes + w * cap + i, q[w]);
}
// an empty slot of a partly filled chunk: only the last word (it holds `depth`) is written; depth 0 makes TRACE skip it
template <typename T>
__device__ __forceinline__ void poolStoreEmpty(uint4* planes, const size_t cap, const int i) {
  __stcg(planes + (sizeof(T) / 16 - 1) * cap + i, make_uint4(0u, 0u, 0u, 0u));
}

template <typename R>
struct Moved {           // per-trace displacement state (motion blur)
  float val;             // reference mode: y shift of "rectangle" shapes
  R time;                // velocity mode: time offset
  int velocity_mode;
};

// render_final_project.cpp:1104-1188: shapes named "rectangle" move in y by `val` during a blur re-trace at time
// offset dt, once frame >= frame_prism (below that the reference's `val` is uninitialised, quirk Q16: 0 here).
template <typename R>
__device__ __forceinline__ float blurVal(const Params<R>& P, const float dt) {
  if (dt == 0.0f || P.blur_mode != 0 || P.frame < P.frame_prism) return 0.0f;
  if (P.frame >= P.frame_blur) return (float)((double)(P.move_per_frame * dt) + (double)P.accel_t * ((double)dt * (double)dt * (double)dt));
  return P.move_per_frame * dt;
}

template <typename R, int F>
__device__ __forceinline__ Vec<R> shiftPoint(const Moved<R>& mv, int gflags, const Vec<R>& vel, Vec<R> p) {
  if ((F & FT_VEL) && mv.velocity_mode) return p + vel * mv.time;
  if ((F & FT_REFBLUR) && (gflags & GF_NAME_RECTANGLE)) p.y += (R)mv.val;
  return p;
}

// The displacement state of one trace.  An instantiation without FT_VEL / FT_REFBLUR never re-traces (the host selects it
// when blur_samples == 0 or no primitive carries the motion flag), so every field is a compile-time zero there.
template <typename R, int F>
__device__ __forceinline__ Moved<R> makeMoved(const Params<R>& P, const float dt) {
  Moved<R> mv;
  mv.val = (F & FT_REFBLUR) ? blurVal(P, dt) : 0.0f;
  mv.time = (F & FT_VEL) ? (R)dt : R(0);
  mv.velocity_mode = (F & FT_VEL) ? ((((F & FT_REFBLUR) ? P.blur_mode == 1 : true) && dt != 0.0f) ? 1 : 0) : 0;
  return mv;
}

// ---- rectangle tests: Rectangle::intersect / intersectShadow (geometry.cpp:640-741)
template <typename R>
__device__ inline bool rectHit(const Vec<R>& A, const Vec<R>& nrm, const Vec<R>& e1, const Vec<R>& e2, R rlen1, R rlen2,
                               float eps, const Vec<R>& ray, const Vec<R>& start, float& t, float& c1o, float& c2o) {
  float dn = (float)dot(ray, nrm);
  if (dn == 0.0f) return false;
  float t_final = (float)(dot(A - start, nrm) / (R)dn);   // double / float -> double, then narrowed (geometry.cpp:676)
  if (t_final <= eps) return false;
  Vec<R> point = start + (R)t_final * ray;
  Vec<R> V_hit = point - A;
  float check1 = (float)dot(e1, V_hit);
  float check2 = (float)dot(e2, V_hit);
  // `check1 <= V1.norm()` compares a float with a double
  if (0 <= check1 && (R)check1 <= rlen1 && 0 <= check2 && (R)check2 <= rlen2) {
    t = t_final; c1o = check1; c2o = check2;
    return true;
  }
  return false;
}

// BoundingVolume::intersect (geometry.cpp:2657-2740): slab test on the ray LINE,
// accepted when tmax > 0.  Leaf boxes are widened in y by the motion-blur
// displacement exactly as bumpBVH does (helpers.h:530-552; interior nodes are not).
template <typename R, int F>
__device__ inline bool boxHit(const NodeD<R>& nd, const Vec<R>& ray, const Vec<R>& inv_ray, const Vec<R>& start,
                              const Moved<R>& mv) {
  R loy = nd.lo.y, hiy = nd.hi.y;
  if ((F & FT_REFBLUR) && nd.leaf && !mv.velocity_mode) { loy -= (R)mv.val; hiy += (R)mv.val; }
  float tmin, tmax;
  if (isinf(inv_ray.x)) {
    if (!(start.x >= nd.lo.x && start.x <= nd.hi.x)) return false;
    tmin = FLT_MIN; tmax = FLT_MAX;
  } else if (ray.x < R(0)) { tmin = (float)((nd.hi.x - start.x) * inv_ray.x); tmax = (float)((nd.lo.x - start.x) * inv_ray.x); }
  else { tmin = (float)((nd.lo.x - start.x) * inv_ray.x); tmax = (float)((nd.hi.x - start.x) * inv_ray.x); }
  float tymin, tymax;
  if (isinf(inv_ray.y)) {
    if (!(start.y >= loy && start.y <= hiy)) return false;
    tymin = FLT_MIN; tymax = FLT_MAX;
  } else if (ray.y < R(0)) { tymin = (float)((hiy - start.y) * inv_ray.y); tymax = (float)((loy - start.y) * inv_ray.y); }
  else { tymin = (float)((loy - start.y) * inv_ray.y); tymax = (float)((hiy - start.y) * inv_ray.y); }
  if (tmin > tymax || tymin > tmax) return false;
  if (tymin > tmin) tmin = tymin;
  if (tymax < tmax) tmax = tymax;
  float tzmin, tzmax;
  if (isinf(inv_ray.z)) {
    if (!(start.z >= nd.lo.z && start.z <= nd.hi.z)) return false;
    tzmin = FLT_MIN; tzmax = FLT_MAX;
  } else if (ray.z < R(0)) { tzmin = (float)((nd.hi.z - start.z) * inv_ray.z); tzmax = (float)((nd.lo.z - start.z) * inv_ray.z); }
  else { tzmin = (float)((nd.lo.z - start.z) * inv_ray.z); tzmax = (float)((nd.hi.z - start.z) * inv_ray.z); }
  if (tmin > tzmax || tzmin > tmax) return false;
  if (tzmin > tmin) tmin = tzmin;
  if (tzmax < tmax) tmax = tzmax;
  return tmax > 0;
}


template <typename R>
__device__ inline Vec<R> mulPoint(const R* m, const Vec<R>& p) {  // (M*(p,1)).head<3>(), 4-term sums as (a+b)+(c+d)
  return mk<R>((m[0] * p.x + m[1] * p.y) + (m[2] * p.z + m[3]), (m[4] * p.x + m[5] * p.y) + (m[6] * p.z + m[7]),
               (m[8] * p.x + m[9] * p.y) + (m[10] * p.z + m[11]));
}

// ---- the slab-box prisms: RectPrism / RectPrismWithCylinder / RectPrismWithHoles (geometry.cpp:950-2246) --------------
// Only in instantiations with FT_BOX.  The box is the WORLD AABB of the corners (geometry.cpp:987-988); the three classes
// open with the BoundingVolume-style slab test and differ in how an axis-parallel ray is detected and whether a start point
// ON the bound counts:
//   kind 0 RectPrism::intersect             isinf(1/ray)  lbound <= start <= ubound   :998-1069
//   kind 1 RectPrismWithCylinder::intersect |ray| < eps   lbound <= start <= ubound   :1517-1588
//   kind 2 the intersectShadow of both      |ray| < eps   lbound <  start <  ubound   :1093-1164, 1683-1754
//   kind 3 RectPrismWithHoles (both)        isinf(1/ray)  no start test               :1893-1955, 2062-2118
template <typename R>
__device__ inline bool prismSlabs(const Vec<R>& lb, const Vec<R>& ub, const Vec<R>& ray, const Vec<R>& start, const int kind,
                                  const float eps, float& tmin, float& tmax) {
  const R rr[3] = {ray.x, ray.y, ray.z}, ss[3] = {start.x, start.y, start.z}, lo3[3] = {lb.x, lb.y, lb.z}, hi3[3] = {ub.x, ub.y, ub.z};
#pragma unroll
  for (int a = 0; a < 3; a++) {
    const R inv = R(1) / rr[a];
    const bool parallel = (kind == 0 || kind == 3) ? (bool)isinf(inv) : (fabs(rr[a]) < (R)eps);
    float lo, hi;
    if (parallel) {
      if (kind == 0 || kind == 1) { if (!(ss[a] >= lo3[a] && ss[a] <= hi3[a])) return false; }
      else if (kind == 2) { if (!(ss[a] > lo3[a] && ss[a] < hi3[a])) return false; }
      lo = FLT_MIN; hi = FLT_MAX;
    } else if (rr[a] < R(0)) { lo = (float)((hi3[a] - ss[a]) * inv); hi = (float)((lo3[a] - ss[a]) * inv); }
    else { lo = (float)((lo3[a] - ss[a]) * inv); hi = (float)((hi3[a] - ss[a]) * inv); }
    if (a == 0) { tmin = lo; tmax = hi; }
    else {
      if (tmin > hi || lo > tmax) return false;
      if (lo > tmin) tmin = lo;
      if (hi < tmax) tmax = hi;
    }
  }
  return true;
}
// Sphere::intersect (geometry.cpp:106-140) / Cylinder::intersect (242-295) on a hole
template <typename R>
__device__ inline bool holeIntersect(const HoleD<R>& h, const Vec<R>& ray, const Vec<R>& start, float& t, int& inside) {
  if (h.type == G_SPHERE) {
    const Vec<R> sc = start - h.c1;
    float A = (float)dot(ray, ray);
    float B = (float)(R(2) * dot(ray, sc));
    float C = (float)(dot(sc, sc) - (R)((double)h.radius * (double)h.radius));
    float disc = (float)((double)B * (double)B - (double)(4 * A * C));
    if (disc < 0) return false;
    float sq = sqrtf(disc);
    float t0 = (-B + sq) / (2 * A), t1 = (-B - sq) / (2 * A);
    if (t0 <= 0.001f && t1 <= 0.001f) { inside = 0; return false; }
    else if (t0 <= 0.001f || t1 <= 0.001f) { t = fmaxf(t0, t1); inside = 1; return true; }
    t = fminf(t0, t1); inside = 0; return true;
  }
  const float eps = 1e-3f;
  const Vec<R> axis = h.axis;
  Vec<R> ray_a_proj = ray - dot(ray, axis) * axis;
  Vec<R> sc = start - h.c1;
  Vec<R> constant = sc - dot(sc, axis) * axis;
  float A = (float)dot(ray_a_proj, ray_a_proj);
  float B = (float)(R(2) * dot(ray_a_proj, constant));
  float C = (float)(dot(constant, constant) - (R)((double)h.radius * (double)h.radius));
  float disc = (float)((double)B * (double)B - (double)(4 * A * C));
  if (!(disc >= 0)) return false;
  float sq = sqrtf(disc);
  float t1_body = (-B + sq) / (2 * A), t2_body = (-B - sq) / (2 * A);
  if (t1_body <= eps && t2_body <= eps) { inside = 0; return false; }
  float tc; int ins;
  if (t1_body <= eps || t2_body <= eps) { tc = t1_body; ins = 1; } else { tc = t2_body; ins = 0; }
  Vec<R> pt = start + (R)tc * ray;
  if (dot(axis, pt - h.c1) > R(0) && dot(axis, pt - h.c2) < R(0)) { t = tc; inside = ins; return true; }
  return false;
}
// Cylinder::intersectCap (geometry.cpp:297-324): the two cap PLANES, no radius test
template <typename R>
__device__ inline bool holeIntersectCap(const HoleD<R>& h, const Vec<R>& ray, const Vec<R>& start, float& t, int& inside) {
  const float eps = 1e-3f;
  inside = 0;
  float rdota = (float)dot(ray, h.axis);
  if (rdota == 0.0f) return false;
  float t1 = (float)((dot(h.c1, h.axis) - dot(start, h.axis)) / (R)rdota);
  float t2 = (float)((dot(h.c2, h.axis) - dot(start, h.axis)) / (R)rdota);
  if (t1 < eps && t2 < eps) return false;
  else if (t1 < eps || t2 < eps) { inside = 1; t = fmaxf(t1, t2); return true; }
  t = fminf(t1, t2); return true;
}
// Sphere::intersectMax (geometry.cpp:142-171) / Cylinder::intersectMax (326-366): the far root of a double intersection
template <typename R>
__device__ inline bool holeIntersectMax(const HoleD<R>& h, const Vec<R>& ray, const Vec<R>& start, float& t) {
  if (h.type == G_SPHERE) {
    const Vec<R> sc = start - h.c1;
    float A = (float)dot(ray, ray);
    float B = (float)(R(2) * dot(ray, sc));
    float C = (float)(dot(sc, sc) - (R)((double)h.radius * (double)h.radius));
    float disc = (float)((double)B * (double)B - (double)(4 * A * C));
    if (disc < 0) return false;
    float sq = sqrtf(disc);
    float t0 = (-B + sq) / (2 * A), t1 = (-B - sq) / (2 * A);
    if (t0 <= 0.001f || t1 <= 0.001f) return false;
    t = fmaxf(t0, t1);
    return true;
  }
  const float eps = 1e-3f;
  const Vec<R> axis = h.axis;
  Vec<R> ray_a_proj = ray - dot(ray, axis) * axis;
  Vec<R> sc = start - h.c1;
  Vec<R> constant = sc - dot(sc, axis) * axis;
  float A = (float)dot(ray_a_proj, ray_a_proj);
  float B = (float)(R(2) * dot(ray_a_proj, constant));
  float C = (float)(dot(constant, constant) - (R)((double)h.radius * (double)h.radius));
  float disc = (float)((double)B * (double)B - (double)(4 * A * C));
  if (!(disc >= 0)) return false;
  float sq = sqrtf(disc);
  float t1_body = (-B + sq) / (2 * A), t2_body = (-B - sq) / (2 * A);
  if (t1_body <= eps || t2_body <= eps) return false;
  Vec<R> pt = start + (R)t2_body * ray;
  if (dot(axis, pt - h.c1) > R(0) && dot(axis, pt - h.c2) < R(0)) { t = t1_body; return true; }
  return false;
}
template <typename R>
__device__ inline Vec<R> holeNorm(const HoleD<R>& h, const Vec<R>& point) {   // Sphere / Cylinder::getNorm
  if (h.type == G_SPHERE) { Vec<R> n = point - h.c1; return n / norm(n); }
  Vec<R> pc = point - h.c1;
  return normalized(pc - dot(pc, h.axis) * h.axis);
}
template <typename R>
__device__ inline bool vecApprox(const Vec<R>& a, const Vec<R>& b) {   // Eigen isApprox: |a-b|^2 <= 1e-24 min(|a|^2, |b|^2)
  const Vec<R> d = a - b;
  return dot(d, d) <= R(1e-24) * fmin(dot(a, a), dot(b, b));
}
// RectPrismWithHoles::getNorm (geometry.cpp:2204-2246): the hole's normal when the last intersect() recorded one, else the
// face picked in object coordinates -- only three faces are recognised, anything else throws (`aborted`, quirk Q15)
template <typename R>
__device__ inline Vec<R> prismHolesNorm(const PrimD<R>& pr, const Vec<R>& point, const int last_hit, bool& aborted) {
  if (last_hit >= 0) return holeNorm<R>(pr.holes[last_hit], point);
  const Vec<R> pObj = mulPoint<R>(pr.objM, point);
  const float eps = 1e-3f;
  if (fabs(pObj.y - (R)(pr.height / 2)) <= (R)eps) return (pObj.y < R(0)) ? pr.n0 : -pr.n0;     // -+ (F-E)x(H-E)^ ; n0 = -(F-E)x(H-E)^
  if (fabs(pObj.x - (R)(pr.length / 2)) <= (R)eps) return (pObj.x < R(0)) ? -pr.n1 : pr.n1;
  if (fabs(pObj.z - (R)(pr.width / 2)) <= (R)eps) return (pObj.z < R(0)) ? -pr.n2 : pr.n2;
  aborted = true;
  return mk<R>(R(0), R(0), R(0));
}
// intersect() of the three classes.  `sel`: 0 keeps the prism's colour, 3 + i takes hole i's (and, for RectPrismWithHoles,
// records lastHit = i for getNorm).  The reference WRITES the hole's colour into the prism for good (geometry.cpp:1650,
// 2005, 2044), which makes its picture depend on pixel order; here the colour belongs to the hit (pinned, DESIGN Q19).
template <typename R>
__device__ __noinline__ bool boxIntersect(const PrimD<R>& pr, const Vec<R>& lb, const Vec<R>& ub, const Vec<R>& ray, const Vec<R>& start,
                                          float& t, int& inside, int& sel) {
  float tmin, tmax;
  inside = 0; sel = 0;
  if (pr.type == 8) {                                                    // RectPrism :990-1085
    const float eps = 1e-6f;
    if (!prismSlabs<R>(lb, ub, ray, start, 0, eps, tmin, tmax)) return false;
    const R nr = norm(ray);
    if (tmin < eps && tmax > eps) { t = (float)(((R)tmax * nr) / nr); inside = 1; return true; }
    if (tmax <= eps) return false;
    t = (float)(((R)tmin * nr) / nr);
    return true;
  }
  const float eps = 1e-4f;
  if (pr.type == 9) {                                                    // RectPrismWithCylinder :1509-1657
    if (!prismSlabs<R>(lb, ub, ray, start, 1, eps, tmin, tmax)) return false;
    if (tmax <= eps) return false;
    if (tmin < eps && tmax > eps) inside = 1;
    t = tmin;                                                            // (sic) :1600
    float tcyl = FLT_MAX;
    int inside_cyl = 0, hit_cyl = -1;
    bool hit = false, cap_hit = false;                                   // uninitialised in the reference: pinned false (Q18)
    for (int i = 0; i < pr.n_holes; i++) {
      float t_tmp; int in_tmp = 0;
      if (holeIntersect<R>(pr.holes[i], ray, start, t_tmp, in_tmp)) { hit = true; if (t_tmp <= tcyl) { hit_cyl = i; inside_cyl = in_tmp; tcyl = t_tmp; } }
      if (holeIntersectCap<R>(pr.holes[i], ray, start, t_tmp, in_tmp)) { hit = true; if (t_tmp <= tcyl) { hit_cyl = i; cap_hit = true; inside_cyl = in_tmp; tcyl = t_tmp; } }
    }
    if (hit && tcyl <= t) {
      if (cap_hit) return false;
      inside = inside_cyl; t = tcyl; sel = 3 + hit_cyl;
    }
    return true;
  }
  // RectPrismWithHoles :1883-2053
  if (!prismSlabs<R>(lb, ub, ray, start, 3, eps, tmin, tmax)) return false;
  if (tmin < eps && tmax > eps) { t = tmax; inside = 1; }
  else { if (tmax <= eps) return false; t = tmin; }
  float tmin_tmp = FLT_MAX, t_tmp;
  int last = -1, in_tmp;
  for (int i = 0; i < pr.n_holes; i++) {
    if (inside) { if (holeIntersect<R>(pr.holes[i], ray, start, t_tmp, in_tmp) && t_tmp <= tmin_tmp) { tmin_tmp = t_tmp; last = i; } }
    else if (holeIntersectMax<R>(pr.holes[i], ray, start, t_tmp) && t_tmp < tmin_tmp) { tmin_tmp = t_tmp; last = i; }
  }
  if (last >= 0) {
    // (sic) `ray + t * start`; getNorm answers with the HOLE's normal because lastHit is already set
    const Vec<R> checknorm = holeNorm<R>(pr.holes[last], ray + (R)t * start);
    const Vec<R> shapenorm = holeNorm<R>(pr.holes[last], ray + (R)tmin_tmp * start);
    if (vecApprox<R>(checknorm, shapenorm) || vecApprox<R>(checknorm, -shapenorm)) return false;
    if (inside && tmin_tmp > t) return true;
    sel = 3 + last; t = tmin_tmp;
  }
  return true;
}
// intersectShadow() of the three classes; `aborted`: RectPrismWithHoles::getNorm threw
template <typename R>
__device__ __noinline__ bool boxShadow(const PrimD<R>& pr, const Vec<R>& lb, const Vec<R>& ub, const Vec<R>& ray, const Vec<R>& start,
                                       const float t_max, bool& aborted) {
  float tmin, tmax;
  if (pr.type == 8) {                                                    // :1087-1180
    const float eps = 1e-6f;
    if (!prismSlabs<R>(lb, ub, ray, start, 2, eps, tmin, tmax)) return false;
    if (tmin < eps && tmax > eps) return t_max > tmax;
    if (tmax <= eps) return false;
    return t_max > tmin;
  }
  const float eps = 1e-4f;
  if (pr.type == 9) {                                                    // :1659-1794
    if (!prismSlabs<R>(lb, ub, ray, start, 2, eps, tmin, tmax)) return false;
    if (tmax <= eps) return false;
    if (tmin < eps && tmax > eps) { if (tmax >= t_max) return false; }
    const float t = tmin;                                                // (sic) :1744; tmin is never compared with t_max
    float tcyl = FLT_MAX;
    bool hit = false, cap_hit = false;                                   // uninitialised in the reference: pinned false (Q18)
    for (int i = 0; i < pr.n_holes; i++) {
      float t_tmp = FLT_MIN; int in_tmp = 0;
      if (holeIntersect<R>(pr.holes[i], ray, start, t_tmp, in_tmp) && t_tmp > eps && t_tmp < t_max) { hit = true; if (t_tmp <= tcyl) tcyl = t_tmp; }
      if (holeIntersectCap<R>(pr.holes[i], ray, start, t_tmp, in_tmp) && t_tmp > eps && t_tmp < t_max) { hit = true; if (t_tmp <= tcyl) { cap_hit = true; tcyl = t_tmp; } }
    }
    if (hit && tcyl <= t && tcyl > eps && tcyl < t_max && cap_hit) return false;
    return true;
  }
  // RectPrismWithHoles :2055-2202
  bool inside = false;
  float t;
  if (!prismSlabs<R>(lb, ub, ray, start, 3, eps, tmin, tmax)) return false;
  if (tmin < eps && tmax > eps) { if (tmax >= t_max) return false; t = tmax; inside = true; }
  else { if (tmax <= eps || tmin >= t_max) return false; t = tmin; }
  float tmin_tmp = FLT_MAX, t_tmp;
  int last = -1, in_tmp;
  for (int i = 0; i < pr.n_holes; i++) {
    if (inside) { if (holeIntersect<R>(pr.holes[i], ray, start, t_tmp, in_tmp) && t_tmp <= tmin_tmp) { tmin_tmp = t_tmp; last = i; } }
    else if (holeIntersectMax<R>(pr.holes[i], ray, start, t_tmp) && t_tmp < tmin_tmp) { tmin_tmp = t_tmp; last = i; }
  }
  if (last >= 0) {
    // lastHit stays -1 in intersectShadow, so getNorm picks a prism face in object coordinates -- or throws
    const Vec<R> checknorm = prismHolesNorm<R>(pr, ray + (R)t * start, -1, aborted);
    if (aborted) return false;
    const Vec<R> shapenorm = holeNorm<R>(pr.holes[last], ray + (R)tmin_tmp * start);
    if (vecApprox<R>(checknorm, shapenorm) || vecApprox<R>(checknorm, -shapenorm)) return false;
  }
  return true;
}

struct HitRec {
  float t;
  int geom;
  int inside;
  int checker_sel;  // 0: keep prim colour, 1: color1, 2: color2
};

// render_wave's dynamic shared memory: [ acc: slots x 3 x u64 | flags: slots x u32 | order: hits x u16 | hkey: hits x u8 ]
// (waveDynSmemBytes), then, in FT_RECS instantiations, the scene records [ geoms | prims | lights ] (Params::smem_recs)
extern __shared__ __align__(16) unsigned char s_dyn[];
__host__ __device__ constexpr size_t waveDynSmemBytes() { return (size_t)DRT_CTA_SLOTS * 28 + (size_t)DRT_CTA_HITS * 3; }
static_assert(waveDynSmemBytes() % 16 == 0, "the staged records start on a 16-byte boundary");

// The geom, primitive and light tables: the CTA's copy in shared memory in FT_RECS instantiations (every exact test and
// every shading step starts with loads from them; from global memory half of them missed the L1), else the global tables.
template <typename R, int F>
__device__ __forceinline__ const Geom<R>* geomRecs(const Params<R>& P) {
  return (F & FT_RECS) ? (const Geom<R>*)(s_dyn + waveDynSmemBytes()) : P.geoms;
}
template <typename R, int F>
__device__ __forceinline__ const PrimD<R>* primRecs(const Params<R>& P) {
  return (F & FT_RECS) ? (const PrimD<R>*)(geomRecs<R, F>(P) + P.n_geoms) : P.prims;
}
template <typename R, int F>
__device__ __forceinline__ const LightD<R>* lightRecs(const Params<R>& P) {
  return (F & FT_RECS) ? (const LightD<R>*)(primRecs<R, F>(P) + P.n_prims) : P.lights;
}
// render_wave's staging copy, by the whole CTA; the records are alignas(16), so whole 16-byte words
__device__ __forceinline__ void ctaCopy16(void* dst, const void* src, const int bytes) {
  for (int i = threadIdx.x; i < bytes / 16; i += blockDim.x) ((uint4*)dst)[i] = __ldg((const uint4*)src + i);
}

// One candidate of the closest-hit search: the intersect() of the geom's class.
template <typename R, int F>
__device__ inline bool geomIntersect(const Params<R>& P, const Geom<R>& g, int gi, const int type, const Moved<R>& mv,
                                     const Vec<R>& ray, const Vec<R>& start, float& t_hit, int& inside, int& sel) {
  bool ok = false;
  inside = 0; sel = 0;
    if ((F & FT_BOX) && type == G_BOX) {
      return boxIntersect<R>(primRecs<R, F>(P)[g.owner], shiftPoint<R, F>(mv, 0, g.vel, g.p0), shiftPoint<R, F>(mv, 0, g.vel, g.p1), ray, start, t_hit, inside, sel);
    } else if (type == G_RECT || type == G_CHECKER) {
      Vec<R> A = shiftPoint<R, F>(mv, g.flags, g.vel, g.p0);
      if (type == G_CHECKER) {  // exact-zero edge path pinned to "no hit" (quirk Q17)
        if (dot(g.p1, ray) == R(0)) return false;
      }
      float c1, c2;
      ok = rectHit<R>(A, g.p1, g.p2, g.p3, g.len1, g.len2, g.eps, ray, start, t_hit, c1, c2);
      if (ok && type == G_CHECKER) {
        if (g.flags & GF_HAS_HOLE) {  // CheckerboardWithHole: inner Rectangle cancels the hit (geometry.cpp:2408-2414)
          const Geom<R>& hgeo = geomRecs<R, F>(P)[gi + 1];
          float th, d1, d2;
          if (rectHit<R>(hgeo.p0, hgeo.p1, hgeo.p2, hgeo.p3, hgeo.len1, hgeo.len2, hgeo.eps, ray, start, th, d1, d2))
            ok = false;
        }
        if (ok) {  // checker parity (geometry.cpp:2313-2337)
          int i = (int)(c1 / g.f2);
          int j = (int)(c2 / g.f2);
          int pi = i % 2, pj = j % 2;
          if (pi == 0) { if (pj == 0) sel = 1; if (pj == 1) sel = 2; }
          if (pi == 1) { if (pj == 0) sel = 2; if (pj == 1) sel = 1; }
        }
      }
    } else if (type == G_SPHERE) {  // Sphere::intersect geometry.cpp:106-140
      Vec<R> sc = start - shiftPoint<R, F>(mv, g.flags, g.vel, g.p0);
      float A = (float)dot(ray, ray);
      float B = (float)(R(2) * dot(ray, sc));
      float C = (float)(dot(sc, sc) - (R)((double)g.f0 * (double)g.f0));
      float disc = (float)((double)B * (double)B - (double)(4 * A * C));
      if (disc < 0) return false;
      float sq = sqrtf(disc);
      float t0 = (-B + sq) / (2 * A);
      float t1 = (-B - sq) / (2 * A);
      if (t0 <= 0.001f && t1 <= 0.001f) return false;
      else if (t0 <= 0.001f || t1 <= 0.001f) { t_hit = fmaxf(t0, t1); inside = 1; ok = true; }
      else { t_hit = fminf(t0, t1); inside = 0; ok = true; }
    } else if (type == G_CYL) {  // Cylinder::intersect geometry.cpp:242-295
      const float eps = 1e-3f;
      Vec<R> c1 = shiftPoint<R, F>(mv, g.flags, g.vel, g.p0), c2 = shiftPoint<R, F>(mv, g.flags, g.vel, g.p1);
      Vec<R> axis = g.p2;
      if ((F & FT_VEL) && (g.flags & GF_VERTEX_MOTION) && mv.velocity_mode) {   // two poses: the axis follows the end points
        c2 = g.p1 + g.cylV2() * mv.time;
        axis = normalized(c2 - c1);
      }
      Vec<R> ray_a_proj = ray - dot(ray, axis) * axis;
      Vec<R> sc = start - c1;
      Vec<R> constant = sc - dot(sc, axis) * axis;
      float A = (float)dot(ray_a_proj, ray_a_proj);
      float B = (float)(R(2) * dot(ray_a_proj, constant));
      float C = (float)(dot(constant, constant) - (R)((double)g.f0 * (double)g.f0));
      float disc = (float)((double)B * (double)B - (double)(4 * A * C));
      if (!(disc >= 0)) return false;
      float sq = sqrtf(disc);
      float t1_body = (-B + sq) / (2 * A);
      float t2_body = (-B - sq) / (2 * A);
      if (t1_body <= eps && t2_body <= eps) return false;
      float tc; int ins;
      if (t1_body <= eps || t2_body <= eps) { tc = t1_body; ins = 1; } else { tc = t2_body; ins = 0; }
      Vec<R> pt = start + (R)tc * ray;
      if (dot(axis, pt - c1) > R(0) && dot(axis, pt - c2) < R(0)) { t_hit = tc; inside = ins; ok = true; }
    } else {  // G_TRI: Triangle::intersect geometry.cpp:488-553
      Vec<R> A = shiftPoint<R, F>(mv, g.flags, g.vel, g.p0);
      const Vec<R> r1 = g.p1, r2 = g.p2;
      Vec<R> hh = cross(ray, r2);
      float det = (float)dot(r1, hh);
      float invdet = 1.0f / det;   // == (float)(1.0 / (double)det) up to double rounding on float ties
      if (det >= -0.0001f && det <= 0.0001f) return false;
      Vec<R> A0 = start - A;
      float u = (float)((double)invdet * (double)dot(A0, hh));   // float * double evaluates in double
      if (u < 0 || u > 1) return false;
      Vec<R> DA0 = cross(A0, r1);
      float v = (float)((double)dot(ray, DA0) * (double)invdet);
      if (v < 0 || u + v > 1) return false;
      float t_final = (float)((double)dot(r2, DA0) * (double)invdet);
      if (t_final > 0.0001f) {
        if (g.flags & GF_MESH) { if (dot(ray, g.p3) > R(0)) inside = 1; }
        t_hit = t_final; ok = true;
      }
    }
  return ok;
}

// Conservative single-precision slab test against the geom's padded bounds: a cheap
// filter in front of the exact (double) class test.  Never rejects a true hit: the
// boxes are padded beyond the rounding of the class's exact test (padBounds, drt_box.cuh)
// and the comparison keeps a relative margin, so only the cost -- not the hits -- changes.
__device__ inline bool slabMayHit(const float4 blo, const float4 bhi, const float nox, const float noy, const float noz,
                                  const float ix, const float iy, const float iz, const float t_limit, const float err) {
  // nox = -ox*ix etc. are hoisted per ray: each slab bound is one FFMA.  `err` bounds the
  // cancellation error of b*i - o*i (a few ulps of |o*i|); inf/NaN (axis-parallel rays) make
  // every comparison below false, i.e. never reject.
  float t0 = fmaf(blo.x, ix, nox), t1 = fmaf(bhi.x, ix, nox);
  float tn = fminf(t0, t1), tf = fmaxf(t0, t1);
  t0 = fmaf(blo.y, iy, noy); t1 = fmaf(bhi.y, iy, noy);
  tn = fmaxf(tn, fminf(t0, t1)); tf = fminf(tf, fmaxf(t0, t1));
  t0 = fmaf(blo.z, iz, noz); t1 = fmaf(bhi.z, iz, noz);
  tn = fmaxf(tn, fminf(t0, t1)); tf = fminf(tf, fmaxf(t0, t1));
  return !(tn > tf * 1.0001f + 1e-4f + err) && !(tf < -err) && !(tn > t_limit + err);
}

// ---- packed slab filter over the whole scene -------------------------------------------------
// The per-scene filter table holds the padded boxes as CENTRE / HALF-EXTENT, two geoms per
// record of three float4:  {cx0 cx1 cy0 cy1} {cz0 cz1 hx0 hx1} {hy0 hy1 hz0 hz1}.
// Per axis  t_near = (c*i - o*i) - h*|i|,  t_far = (c*i - o*i) + h*|i|  are three fused
// multiply-adds, and sm_100's packed FFMA2 (fma.rn.f32x2) evaluates them for both geoms of the
// record at once: 9 FFMA2 + 4 FMNMX3 per PAIR instead of 12 FFMA + 12 FMNMX + 4 FMNMX3.
// Holes and the padding entry of an odd count carry h = -1e30 and never pass.
struct SlabRay {
  float2 i[3], no[3], ai[3], nai[3];   // 1/d, -o/d, |1/d|, -|1/d|, each duplicated into both halves
  float2 grow, slack;                  // t_far * 1.0001 + (1e-4 + err)
  float floor_t, lim;                  // t_far >= -err  and  t_near <= t_limit + err, folded into one compare
};
__device__ __forceinline__ SlabRay slabRay(const float ix, const float iy, const float iz, const float nox, const float noy,
                                           const float noz, const float t_limit) {
  SlabRay r;
  const float err = 4e-7f * (fabsf(nox) + fabsf(noy) + fabsf(noz));   // cancellation error of c*i - o*i
  r.i[0] = make_float2(ix, ix); r.i[1] = make_float2(iy, iy); r.i[2] = make_float2(iz, iz);
  r.no[0] = make_float2(nox, nox); r.no[1] = make_float2(noy, noy); r.no[2] = make_float2(noz, noz);
  const float ax = fabsf(ix), ay = fabsf(iy), az = fabsf(iz);
  r.ai[0] = make_float2(ax, ax); r.ai[1] = make_float2(ay, ay); r.ai[2] = make_float2(az, az);
  r.nai[0] = make_float2(-ax, -ax); r.nai[1] = make_float2(-ay, -ay); r.nai[2] = make_float2(-az, -az);
  const float c = 1e-4f + err;
  r.grow = make_float2(1.0001f, 1.0001f); r.slack = make_float2(c, c);
  r.floor_t = fmaf(-1.0002f, err, c);   // t_far' >= floor_t  <=>  t_far >= -err (a hair looser)
  r.lim = t_limit + err;
  return r;
}
__device__ __forceinline__ unsigned int slabAll(const int g0, const int g1) {   // every geom of the group [g0, g1)
  return (g1 - g0 >= 32) ? 0xffffffffu : ((1u << (g1 - g0)) - 1u);
}
// The table is addressed by a byte offset from `tab`: a 32-bit shared-window address when the CTA staged it in shared
// memory (explicit ld.shared.v4 with the record offsets folded into the instruction), a global pointer otherwise.
struct SlabTab {
  const float4* g;      // global table (P.gbounds)
  unsigned s;           // the same table in the CTA's shared memory (shared-window address)
};
template <bool SMEM>
__device__ __forceinline__ float4 slabLoad(const SlabTab tab, const int word) {   // word = index of the float4
  if (SMEM) {
    float4 v;
    // volatile: must not be speculated above the `smem` test
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(tab.s + 16u * (unsigned)word));
    return v;
  }
  return __ldg(tab.g + word);
}
// Bit k of the result: geom g0 + k may be hit.  inf/NaN terms (axis-parallel rays) drop out of
// the min/max chains or make the final compare false, i.e. never reject.
// Two-level form: the table also holds one box per GROUP of 8 consecutive geoms (4 pair records; consecutive geoms are
// neighbours in the reference's BVH order, and a prism's 6 faces are consecutive).  A lane runs a group's records only
// if its ray may hit the group box -- the branch is per lane, so the warp skips the block when no lane needs it, which
// is the common case now that a warp's rays leave from one surface (geom-sorted SHADE, child-index-major pushes).
// The pair records are padded to whole groups (never-passing entries), so a group is always four records.
__host__ __device__ constexpr int slabPairWords(const int n_geoms) { return 3 * 4 * ((n_geoms + 7) / 8); }   // float4 words before the group boxes
__device__ __forceinline__ bool slabGroupMayHit(const float4 G0, const float4 G1, const SlabRay& r) {
  const float mx = fmaf(G0.x, r.i[0].x, r.no[0].x), my = fmaf(G0.y, r.i[1].x, r.no[1].x), mz = fmaf(G0.z, r.i[2].x, r.no[2].x);
  const float tn = fmaxf(fmaxf(fmaf(G0.w, r.nai[0].x, mx), fmaf(G1.x, r.nai[1].x, my)), fmaf(G1.y, r.nai[2].x, mz));
  const float tf = fminf(fminf(fmaf(G0.w, r.ai[0].x, mx), fmaf(G1.x, r.ai[1].x, my)), fmaf(G1.y, r.ai[2].x, mz));
  return !(fmaxf(tn, r.floor_t) > fminf(fmaf(tf, r.grow.x, r.slack.x), r.lim));
}
template <bool SMEM>
__device__ __forceinline__ unsigned int slabMask(const SlabTab tab, const int n_geoms, const int g0, const int g1, const SlabRay& r) {
  unsigned int mask = 0;
  const int gw = slabPairWords(n_geoms);                          // group boxes follow the pair records
  for (int q0 = g0; q0 < g1; q0 += 8) {
    const int grp = q0 >> 3;
    const float4 G0 = slabLoad<SMEM>(tab, gw + 2 * grp), G1 = slabLoad<SMEM>(tab, gw + 2 * grp + 1);
    if (!slabGroupMayHit(G0, G1, r)) continue;
    unsigned int sub = 0;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const int w = 12 * grp + 3 * k;
      const float4 A = slabLoad<SMEM>(tab, w), B = slabLoad<SMEM>(tab, w + 1), C = slabLoad<SMEM>(tab, w + 2);
      const float2 mx = __ffma2_rn(make_float2(A.x, A.y), r.i[0], r.no[0]);
      const float2 my = __ffma2_rn(make_float2(A.z, A.w), r.i[1], r.no[1]);
      const float2 mz = __ffma2_rn(make_float2(B.x, B.y), r.i[2], r.no[2]);
      const float2 hx = make_float2(B.z, B.w), hy = make_float2(C.x, C.y), hz = make_float2(C.z, C.w);
      const float2 nx = __ffma2_rn(hx, r.nai[0], mx), fx = __ffma2_rn(hx, r.ai[0], mx);
      const float2 ny = __ffma2_rn(hy, r.nai[1], my), fy = __ffma2_rn(hy, r.ai[1], my);
      const float2 nz = __ffma2_rn(hz, r.nai[2], mz), fz = __ffma2_rn(hz, r.ai[2], mz);
      const float tn0 = fmaxf(fmaxf(nx.x, ny.x), nz.x), tn1 = fmaxf(fmaxf(nx.y, ny.y), nz.y);
      const float2 tf = __ffma2_rn(make_float2(fminf(fminf(fx.x, fy.x), fz.x), fminf(fminf(fx.y, fy.y), fz.y)), r.grow, r.slack);
      if (!(fmaxf(tn0, r.floor_t) > fminf(tf.x, r.lim))) sub |= 1u << (2 * k);
      if (!(fmaxf(tn1, r.floor_t) > fminf(tf.y, r.lim))) sub |= 2u << (2 * k);
    }
    mask |= sub << (q0 - g0);
  }
  // a ray with an infinite error bound (exactly axis-parallel) passes everything, the padding entries included
  return mask & slabAll(g0, g1);
}

// One pair record of the slab filter (see slabMask) -> pass flags and entry distances of its two boxes.
__device__ __forceinline__ void slabPair(const float4 A, const float4 B, const float4 C, const SlabRay& r, bool& ok0, bool& ok1,
                                         float& tn0, float& tn1) {
  const float2 mx = __ffma2_rn(make_float2(A.x, A.y), r.i[0], r.no[0]);
  const float2 my = __ffma2_rn(make_float2(A.z, A.w), r.i[1], r.no[1]);
  const float2 mz = __ffma2_rn(make_float2(B.x, B.y), r.i[2], r.no[2]);
  const float2 hx = make_float2(B.z, B.w), hy = make_float2(C.x, C.y), hz = make_float2(C.z, C.w);
  const float2 nx = __ffma2_rn(hx, r.nai[0], mx), fx = __ffma2_rn(hx, r.ai[0], mx);
  const float2 ny = __ffma2_rn(hy, r.nai[1], my), fy = __ffma2_rn(hy, r.ai[1], my);
  const float2 nz = __ffma2_rn(hz, r.nai[2], mz), fz = __ffma2_rn(hz, r.ai[2], mz);
  tn0 = fmaxf(fmaxf(nx.x, ny.x), nz.x); tn1 = fmaxf(fmaxf(nx.y, ny.y), nz.y);
  const float2 tf = __ffma2_rn(make_float2(fminf(fminf(fx.x, fy.x), fz.x), fminf(fminf(fx.y, fy.y), fz.y)), r.grow, r.slack);
  ok0 = !(fmaxf(tn0, r.floor_t) > fminf(tf.x, r.lim));
  ok1 = !(fmaxf(tn1, r.floor_t) > fminf(tf.y, r.lim));
}

// ---- 4-wide tree traversal (the mesh LBVH of drt_lbvh.cuh, and the tree over the analytic geoms of big scenes) ------------
// A node visit tests its four child boxes with the packed slab test, descends into the nearest one that passes (CLOSEST)
// and pushes the others with their entry distances; an entry whose distance lies beyond the best hit found meanwhile is
// dropped when popped.  Without CLOSEST (any hit) the order does not matter: the last passing child is next.
#define DRT_MESH_DONE ((int)0x80000000)
template <bool CLOSEST>
__device__ __forceinline__ int bvh4Pop(const int2* stack, int& sp, const float lim) {
  while (sp > 0) {
    const int2 e = stack[--sp];
    if (CLOSEST && __int_as_float(e.y) > lim) continue;
    return e.x;
  }
  return DRT_MESH_DONE;
}
template <bool CLOSEST>
__device__ __forceinline__ int bvh4Visit(const float4* __restrict__ nodes, const int cur, const SlabRay& sr, int2* stack, int& sp, int* overflow) {
  const float4* nd = nodes + 8 * (size_t)cur;
  const float4 A0 = __ldg(nd), B0 = __ldg(nd + 1), C0 = __ldg(nd + 2), A1 = __ldg(nd + 3), B1 = __ldg(nd + 4), C1 = __ldg(nd + 5);
  const float4 K = __ldg(nd + 6);
  bool ok0, ok1, ok2, ok3; float t0, t1, t2, t3;
  slabPair(A0, B0, C0, sr, ok0, ok1, t0, t1);
  slabPair(A1, B1, C1, sr, ok2, ok3, t2, t3);
  const int r0 = __float_as_int(K.x), r1 = __float_as_int(K.y), r2 = __float_as_int(K.z), r3 = __float_as_int(K.w);
  ok2 = ok2 && r2 != DRT_MESH_DONE; ok3 = ok3 && r3 != DRT_MESH_DONE;     // empty slots (NaN slab terms of an axis-parallel ray pass the test)
  if (sp > DRT_NODE_STACK - 4) { *overflow = 1; sp = 0; return DRT_MESH_DONE; }   // degenerate input only: the frame is rejected, not wrong
  if (CLOSEST) {
    // descend into the nearest passing child: order key = entry distance (clamped at 0, low two mantissa bits = slot)
    const int k0 = ok0 ? ((__float_as_int(fmaxf(t0, 0.f)) & ~3) | 0) : 0x7fffffff;
    const int k1 = ok1 ? ((__float_as_int(fmaxf(t1, 0.f)) & ~3) | 1) : 0x7fffffff;
    const int k2 = ok2 ? ((__float_as_int(fmaxf(t2, 0.f)) & ~3) | 2) : 0x7fffffff;
    const int k3 = ok3 ? ((__float_as_int(fmaxf(t3, 0.f)) & ~3) | 3) : 0x7fffffff;
    const int kb = min(min(k0, k1), min(k2, k3));
    if (kb == 0x7fffffff) return bvh4Pop<CLOSEST>(stack, sp, sr.lim);
    if (ok0 && k0 != kb) stack[sp++] = make_int2(r0, __float_as_int(t0));
    if (ok1 && k1 != kb) stack[sp++] = make_int2(r1, __float_as_int(t1));
    if (ok2 && k2 != kb) stack[sp++] = make_int2(r2, __float_as_int(t2));
    if (ok3 && k3 != kb) stack[sp++] = make_int2(r3, __float_as_int(t3));
    const int bk = kb & 3;
    return bk == 0 ? r0 : bk == 1 ? r1 : bk == 2 ? r2 : r3;
  }
  int nxt = DRT_MESH_DONE;
  if (ok0) nxt = r0;
  if (ok1) { if (nxt != DRT_MESH_DONE) stack[sp++] = make_int2(nxt, 0); nxt = r1; }
  if (ok2) { if (nxt != DRT_MESH_DONE) stack[sp++] = make_int2(nxt, 0); nxt = r2; }
  if (ok3) { if (nxt != DRT_MESH_DONE) stack[sp++] = make_int2(nxt, 0); nxt = r3; }
  return (nxt != DRT_MESH_DONE) ? nxt : bvh4Pop<CLOSEST>(stack, sp, sr.lim);
}

// Would the reference's BVH walk along (ray, start) have gathered this geom?  BoundingVolume::intersect on its leaf and
// every ancestor (the walk descends only through nodes whose box test passes, render_final_project.cpp:492-512).
template <typename R, int F, bool COUNT>
__device__ __noinline__ bool gatherReplay(const Params<R>& P, const int leaf, const Vec<R> ray, const Vec<R> start, const Moved<R> mv, Counts& cnt) {   // by value: no addressable copies at the call sites
  const Vec<R> inv_ray = mk<R>(R(1) / ray.x, R(1) / ray.y, R(1) / ray.z);   // ray.cwiseInverse() :499, :813
  for (int ni = leaf; ni >= 0; ni = P.nodes[ni].parent) {
    if (COUNT) cnt.node_tests++;
    if (!boxHit<R, F>(P.nodes[ni], ray, inv_ray, start, mv)) return false;
  }
  return true;
}

// Closest hit over all flattened primitives (the candidate loop of rayColor,
// render_final_project.cpp:522-538, with each class's intersect()).
//
// The reference gathers candidates through its BVH; for these rays the gather walks the
// same ray the tests use and its boxes are padded supersets of the shapes, so culling
// never changes which shape is closest.  The geoms are therefore tested directly, in
// the reference's candidate order (ties of t keep the first, :531), behind the cheap
// slab filter.  Only while "rectangle" shapes are displaced by reference-mode motion
// blur (mv.val != 0) is the reference tree walked node by node: bumpBVH widens leaf
// boxes but not interior ones (quirk Q14), which can cull a moved rectangle.
template <typename R, int F, bool COUNT>
__device__ inline void closestHit(const Params<R>& P, const SlabTab gb, const Moved<R>& mv, const Vec<R>& ray,
                                  const Vec<R>& start, HitRec& h, Counts& cnt) {
  h.t = FLT_MAX; h.geom = -1; h.inside = 0; h.checker_sel = 0;
  if ((!(F & FT_REFBLUR) || mv.val == 0.0f) && !DRT_FORCE_TREE) {
    // Two passes per group of 32 geoms: (1) the slab filter runs over the group in
    // lock-step (warp-uniform loads) and leaves each lane a bit mask of ITS candidates;
    // (2) every lane then walks its own mask, so one loop trip runs one exact test per
    // lane -- whatever geom that is -- instead of one geom for the few lanes that need it.
    const float ix = 1.0f / (float)ray.x, iy = 1.0f / (float)ray.y, iz = 1.0f / (float)ray.z;
    const float ox = -(float)start.x * ix, oy = -(float)start.y * iy, oz = -(float)start.z * iz;   // slabMayHit's hoisted terms
    const float serr = 4e-7f * (fabsf(ox) + fabsf(oy) + fabsf(oz));
    const bool cull = !((F & FT_VEL) && mv.velocity_mode) || P.swept_cull;
    const bool smem = !(F & FT_BIG) || P.n_geoms <= DRT_SMEM_GEOMS;     // CTA-uniform: the table is staged in shared memory
    if ((F & FT_BIG) && cull && P.geom_tree) {
      // more geoms than the filter table in shared memory holds: candidates come from the 4-wide tree over the geoms.  The
      // tree hands them over in its own order, so a tie of t goes to the lower geom index explicitly (:531 keeps the first)
      SlabRay st = slabRay(ix, iy, iz, ox, oy, oz, FLT_MAX);
      int2 stack[DRT_NODE_STACK];
      int sp = 0, cur = 0;
      for (;;) {
        while (cur >= 0) { if (COUNT) cnt.node_tests += 4; cur = bvh4Visit<true>(P.geom_tree, cur, st, stack, sp, P.overflow); }
        if (cur == DRT_MESH_DONE) break;
        const int gi = -cur - 1;
        const Geom<R>& g = geomRecs<R, F>(P)[gi];
        const int type = g.type;
        if (COUNT) cnt.geom_tests[type]++;
        float t_hit; int inside, sel;
        if (geomIntersect<R, F>(P, g, gi, type, mv, ray, start, t_hit, inside, sel) && (t_hit < h.t || (t_hit == h.t && gi < h.geom)) &&
            (!(F & FT_SPILL) || !(g.flags & GF_SPILL) || ((F & FT_VEL) && mv.velocity_mode) || gatherReplay<R, F, COUNT>(P, g.leaf, ray, start, mv, cnt))) {
          h.t = t_hit; h.geom = gi; h.inside = inside; h.checker_sel = sel;
          st.lim = (t_hit * 1.0001f + 1e-4f) + serr;
        }
        cur = bvh4Pop<true>(stack, sp, st.lim);
      }
      return;
    }
    const SlabRay sr = slabRay(ix, iy, iz, ox, oy, oz, FLT_MAX);
    const int n = P.n_geoms;
    for (int g0 = 0; g0 < n; g0 += 32) {
      const int g1 = min(n, g0 + 32);
      unsigned int mask = !cull ? slabAll(g0, g1) : smem ? slabMask<true>(gb, n, g0, g1, sr) : slabMask<false>(gb, n, g0, g1, sr);
      while (mask) {
        const int gi = g0 + __ffs(mask) - 1;      // ascending = the reference's candidate order
        mask &= mask - 1;
        const Geom<R>& g = geomRecs<R, F>(P)[gi];
        const int type = g.type;
        if (type == G_HOLE) continue;
        // a box whose entry lies beyond the best hit cannot hold a closer (or tying) one
        if (cull && h.t < FLT_MAX && !slabMayHit(g.blo, g.bhi, ox, oy, oz, ix, iy, iz, h.t * 1.0001f + 1e-4f, serr)) continue;
        if (COUNT) cnt.geom_tests[type]++;
        float t_hit; int inside, sel;
        // (a hit on a GF_SPILL rectangle counts only if the reference's gather reaches its leaf, see rectGeom in drt_api.cu)
        if (geomIntersect<R, F>(P, g, gi, type, mv, ray, start, t_hit, inside, sel) && t_hit < h.t &&
            (!(F & FT_SPILL) || !(g.flags & GF_SPILL) || ((F & FT_VEL) && mv.velocity_mode) || gatherReplay<R, F, COUNT>(P, g.leaf, ray, start, mv, cnt))) {
          h.t = t_hit; h.geom = gi; h.inside = inside; h.checker_sel = sel;
        }
      }
    }
    return;
  }
  int stack[DRT_NODE_STACK];
  int sp = 0;
  stack[sp++] = 0;
  const Vec<R> inv_ray = mk<R>(R(1) / ray.x, R(1) / ray.y, R(1) / ray.z);   // ray.cwiseInverse() :499
  while (sp > 0) {
    const NodeD<R>& nd = P.nodes[stack[--sp]];
    if (COUNT) cnt.node_tests++;
    if (!boxHit<R, F>(nd, ray, inv_ray, start, mv)) continue;
    if (!nd.leaf) { stack[sp++] = nd.left; stack[sp++] = nd.right; continue; }   // right child is popped first (:497-509)
    const int g_end = nd.first + nd.count;
    for (int gi = nd.first; gi < g_end; gi++) {
      const Geom<R>& g = geomRecs<R, F>(P)[gi];
      const int type = g.type;
      if (type == G_HOLE) continue;
      if (COUNT) cnt.geom_tests[type]++;
      float t_hit; int inside, sel;
      if (geomIntersect<R, F>(P, g, gi, type, mv, ray, start, t_hit, inside, sel) && t_hit < h.t) {
        h.t = t_hit; h.geom = gi; h.inside = inside; h.checker_sel = sel;
      }
    }
  }
}

// One candidate of the shadow test: the intersectShadow() of the geom's class.
// `ray` is normalised, `start` already offset by 1e-3 along it.
template <typename R, int F>
__device__ inline bool geomShadow(const Params<R>& P, const Geom<R>& g, int gi, const int type, const Moved<R>& mv,
                                  const Vec<R>& ray, const Vec<R>& start, const float t_max, float& t_occ, bool& aborted) {
    t_occ = 0.0f;   // on success: a ray parameter at which the ray certainly touches the geom
    if ((F & FT_BOX) && type == G_BOX) {
      // t_occ stays 0: these classes report occlusion without a touch point, so the reference gather is always replayed
      return boxShadow<R>(primRecs<R, F>(P)[g.owner], shiftPoint<R, F>(mv, 0, g.vel, g.p0), shiftPoint<R, F>(mv, 0, g.vel, g.p1), ray, start, t_max, aborted);
    } else if (type == G_RECT || type == G_CHECKER) {
      Vec<R> A = shiftPoint<R, F>(mv, g.flags, g.vel, g.p0);
      // Checkerboard inherits Rectangle::intersectShadow (eps 1e-4); CheckerboardWithHole
      // has its own with eps 1e-3 (geometry.cpp:2446-2498)
      float eps = (type == G_CHECKER && !(g.flags & GF_HAS_HOLE)) ? 1e-4f : g.eps;
      float th, c1, c2;
      if (rectHit<R>(A, g.p1, g.p2, g.p3, g.len1, g.len2, eps, ray, start, th, c1, c2) && th < t_max) {
        if (g.flags & GF_HAS_HOLE) {
          const Geom<R>& hgeo = geomRecs<R, F>(P)[gi + 1];
          float t2, d1, d2;
          if (rectHit<R>(hgeo.p0, hgeo.p1, hgeo.p2, hgeo.p3, hgeo.len1, hgeo.len2, hgeo.eps, ray, start, t2, d1, d2) &&
              t2 < t_max)
            return false;
        }
        t_occ = th;
        return true;
      }
    } else if (type == G_SPHERE) {  // geometry.cpp:173-197
      const float eps = 1e-3f;
      Vec<R> sc = start - shiftPoint<R, F>(mv, g.flags, g.vel, g.p0);
      float A = (float)dot(ray, ray);
      float B = (float)(R(2) * dot(ray, sc));
      float C = (float)(dot(sc, sc) - (R)((double)g.f0 * (double)g.f0));
      float disc = (float)((double)B * (double)B - (double)(4 * A * C));
      if (disc < 0) return false;
      float sq = sqrtf(disc);
      float t0 = (-B + sq) / (2 * A);
      float t1 = (-B - sq) / (2 * A);
      if ((t0 <= eps || t0 >= t_max) && (t1 <= eps || t1 >= t_max)) return false;
      t_occ = (t0 > eps && t0 < t_max) ? t0 : t1;   // t0 is the far root
      return true;
    } else if (type == G_CYL) {  // geometry.cpp:368-417
      const float eps = 1e-3f;
      Vec<R> c1 = shiftPoint<R, F>(mv, g.flags, g.vel, g.p0), c2 = shiftPoint<R, F>(mv, g.flags, g.vel, g.p1);
      Vec<R> axis = g.p2;
      if ((F & FT_VEL) && (g.flags & GF_VERTEX_MOTION) && mv.velocity_mode) {   // two poses: the axis follows the end points
        c2 = g.p1 + g.cylV2() * mv.time;
        axis = normalized(c2 - c1);
      }
      Vec<R> ray_a_proj = ray - dot(ray, axis) * axis;
      Vec<R> sc = start - c1;
      Vec<R> constant = sc - dot(sc, axis) * axis;
      float A = (float)dot(ray_a_proj, ray_a_proj);
      float B = (float)(R(2) * dot(ray_a_proj, constant));
      float C = (float)(dot(constant, constant) - (R)((double)g.f0 * (double)g.f0));
      float disc = (float)((double)B * (double)B - (double)(4 * A * C));
      if (!(disc >= 0)) return false;
      float sq = sqrtf(disc);
      float t1_body = (-B + sq) / (2 * A);
      float t2_body = (-B - sq) / (2 * A);
      if ((t1_body <= eps || t1_body >= t_max) && (t2_body <= eps || t2_body >= t_max)) return false;
      float tc = (t1_body <= eps || t2_body <= eps) ? t1_body : t2_body;
      Vec<R> pt = start + (R)tc * ray;
      if (dot(axis, pt - c1) > R(0) && dot(axis, pt - c2) < R(0) && tc < t_max) { t_occ = tc; return true; }
    } else {  // G_TRI geometry.cpp:555-586
      Vec<R> A = shiftPoint<R, F>(mv, g.flags, g.vel, g.p0);
      const Vec<R> r1 = g.p1, r2 = g.p2;
      Vec<R> hh = cross(ray, r2);
      float det = (float)dot(r1, hh);
      float invdet = 1.0f / det;   // == (float)(1.0 / (double)det) up to double rounding on float ties
      if (det >= -0.0001f && det <= 0.0001f) return false;
      Vec<R> A0 = start - A;
      float u = (float)((double)invdet * (double)dot(A0, hh));
      if (u < 0 || u > 1) return false;
      Vec<R> DA0 = cross(A0, r1);
      float v = (float)((double)dot(ray, DA0) * (double)invdet);
      if (v < 0 || u + v > 1) return false;
      float t_final = (float)((double)dot(r2, DA0) * (double)invdet);
      if (t_final > 0.001f && t_final < t_max) { t_occ = t_final; return true; }
    }
  return false;
}

// Any-hit for shadow rays (render_final_project.cpp:806-851).
//
// The reference gathers candidates along the UNNORMALISED light vector from
// isectP + sray*1e-3 (:814) but tests occlusion along the normalised one from
// isectP + s^*1e-3 (:838): with the sphere-light quirk (sampleRay returns a position,
// |sray| ~ tens of units) occluders within the first centimetres are never gathered.
// That is reproduced exactly, lazily: geoms are tested directly (slab filter + exact
// class test) and only a geom that DOES occlude is checked against the reference
// gather, by running BoundingVolume::intersect on its leaf and every ancestor.
template <typename R, int F, bool COUNT>
__device__ inline bool anyHit(const Params<R>& P, const SlabTab gb, const Moved<R>& mv, const Vec<R>& gather_ray,
                              const Vec<R>& gather_start, const Vec<R>& ray, const Vec<R>& start, float t_max, int skip_owner,
                              Counts& cnt, bool& aborted) {
  if ((!(F & FT_REFBLUR) || mv.val == 0.0f) && !DRT_FORCE_TREE) {
    const float ix = 1.0f / (float)ray.x, iy = 1.0f / (float)ray.y, iz = 1.0f / (float)ray.z;
    const float ox = -(float)start.x * ix, oy = -(float)start.y * iy, oz = -(float)start.z * iz;   // slabMayHit's hoisted terms
    const bool cull = !((F & FT_VEL) && mv.velocity_mode) || P.swept_cull;
    // distance by which the reference's gather origin runs ahead of the test origin
    const float gather_lead = t_max * 1e-3f;
    const int n = P.n_geoms;
    const bool smem = !(F & FT_BIG) || n <= DRT_SMEM_GEOMS;
    const SlabRay sr = slabRay(ix, iy, iz, ox, oy, oz, t_max * 1.0001f + 1e-4f);
    // one candidate: 1 = the ray is occluded, -1 = the reference throws (slab-box prisms), 0 = go on
    auto candidate = [&](const int gi) -> int {
      const Geom<R>& g = geomRecs<R, F>(P)[gi];
      const int type = g.type;
      if (type == G_HOLE || g.owner == skip_owner) return 0;     // an area light never shadows itself (832-837)
      if (COUNT) cnt.geom_tests[type]++;
      float t_occ;
      if (!geomShadow<R, F>(P, g, gi, type, mv, ray, start, t_max, t_occ, aborted)) return ((F & FT_BOX) && aborted) ? -1 : 0;
      if ((F & FT_VEL) && mv.velocity_mode) return 1;            // time-displaced geometry: no reference tree to consult
      // The occluder touches the ray at distance t_occ from the test origin.  If that point
      // lies ahead of the gather origin it is inside the geom's leaf box and every ancestor
      // box (they are padded supersets), so BoundingVolume::intersect returns tmax > 0 for all
      // of them and the reference does gather this geom.  Only nearer occluders need the
      // exact replay of the reference's box tests.
      // (not so for a GF_SPILL rectangle, whose touch point can lie outside its box: always replayed)
      if (t_occ > gather_lead * 1.001f + 2e-3f && !((F & FT_SPILL) && (g.flags & GF_SPILL))) return 1;
      return gatherReplay<R, F, COUNT>(P, g.leaf, gather_ray, gather_start, mv, cnt) ? 1 : 0;   // rare path: three divisions
    };
    if ((F & FT_BIG) && cull && P.geom_tree) {                    // big scenes: candidates from the tree over the geoms (see closestHit)
      int2 stack[DRT_NODE_STACK];
      int sp = 0, cur = 0;
      for (;;) {
        while (cur >= 0) { if (COUNT) cnt.node_tests += 4; cur = bvh4Visit<false>(P.geom_tree, cur, sr, stack, sp, P.overflow); }
        if (cur == DRT_MESH_DONE) break;
        if (candidate(-cur - 1) == 1) return true;
        cur = bvh4Pop<false>(stack, sp, sr.lim);
      }
      return false;
    }
    for (int g0 = 0; g0 < n; g0 += 32) {
      const int g1 = min(n, g0 + 32);
      // lock-step, branch-free slab filter -> per-lane candidate mask
      unsigned int mask = !cull ? slabAll(g0, g1) : smem ? slabMask<true>(gb, n, g0, g1, sr) : slabMask<false>(gb, n, g0, g1, sr);
      while (mask) {                                // each lane walks its own candidates
        const int gi = g0 + __ffs(mask) - 1;
        mask &= mask - 1;
        const int c = candidate(gi);
        if (c == 1) return true;
        if ((F & FT_BOX) && c == -1) return false;
      }
    }
    return false;
  }
  int stack[DRT_NODE_STACK];
  int sp = 0;
  stack[sp++] = 0;
  const Vec<R> inv_ray = mk<R>(R(1) / gather_ray.x, R(1) / gather_ray.y, R(1) / gather_ray.z);   // sray.cwiseInverse() :813
  while (sp > 0) {
    const NodeD<R>& nd = P.nodes[stack[--sp]];
    if (COUNT) cnt.node_tests++;
    if (!boxHit<R, F>(nd, gather_ray, inv_ray, gather_start, mv)) continue;
    if (!nd.leaf) { stack[sp++] = nd.left; stack[sp++] = nd.right; continue; }
    const int g_end = nd.first + nd.count;
    for (int gi = nd.first; gi < g_end; gi++) {
      const Geom<R>& g = geomRecs<R, F>(P)[gi];
      const int type = g.type;
      if (type == G_HOLE) continue;
      if (g.owner == skip_owner) continue;
      if (COUNT) cnt.geom_tests[type]++;
      float t_occ;
      if (geomShadow<R, F>(P, g, gi, type, mv, ray, start, t_max, t_occ, aborted)) return true;
      if ((F & FT_BOX) && aborted) return false;
    }
  }
  return false;
}

// ---- triangle mesh: LBVH traversal (drt_lbvh.cuh) ------------------------------------------
// Triangle::intersect (geometry.cpp:488-553) on a mesh triangle; returns t or a negative value.
template <typename R>
__device__ __forceinline__ float meshTriT(const Vec<R>& tA, const Vec<R>& tB, const Vec<R>& tC, const Vec<R>& ray, const Vec<R>& start) {
  const Vec<R> r1 = tB - tA, r2 = tC - tA;
  const Vec<R> hh = cross(ray, r2);
  const float det = (float)dot(r1, hh);
  const float invdet = 1.0f / det;   // == (float)(1.0 / (double)det) up to double rounding on float ties
  if (det >= -0.0001f && det <= 0.0001f) return -1.f;
  const Vec<R> A0 = start - tA;
  const float u = (float)((double)invdet * (double)dot(A0, hh));
  if (u < 0 || u > 1) return -1.f;
  const Vec<R> DA0 = cross(A0, r1);
  const float v = (float)((double)dot(ray, DA0) * (double)invdet);
  if (v < 0 || u + v > 1) return -1.f;
  return (float)((double)dot(r2, DA0) * (double)invdet);
}

// Traversal of the 4-wide LBVH (drt_lbvh.cuh), "while-while": a lane first descends through internal nodes until the
// next thing it has to do is an exact triangle test (or nothing), and only then -- together with the other lanes of the
// warp that reached a leaf -- runs the reference's Moeller-Trumbore test in the vector precision.  With the test inline in
// the node loop it ran with ~4 of 32 lanes (profiles/r1_ncu_full_band_c5_mesh.txt).  Node visits: bvh4Visit.
// CLOSEST: keeps the nearest hit with t > 1e-4 (strict `<` against the best so far, so analytic primitives -- tested
// first -- win ties).  !CLOSEST: any hit with 1e-3 < t < t_max (Triangle::intersectShadow geometry.cpp:555-586) that the
// reference would also have gathered (its gather origin runs ahead by |sray|*1e-3, :814; a mesh triangle stands in its
// own leaf box: bounds +- 1e-2, geometry.cpp:2653-2654).
template <typename R, int F, bool COUNT, bool CLOSEST>
__device__ bool meshTraverse(const Params<R>& P, const Vec<R>& ray, const Vec<R>& start, float t_limit, HitRec* h,
                             const Vec<R>& gather_ray, const Vec<R>& gather_start, const bool vel_retrace, const R time, Counts& cnt) {
  // A velocity re-trace at time offset `time` displaces the whole mesh by mesh_vel * time.  The tree stays as built and is
  // walked with the ray moved the other way (its boxes are padded far beyond the rounding of that); the exact test runs
  // on the displaced vertices, as the oracle twin's per-triangle walk does.  (Only the time is carried through the walk.)
  const bool disp = (F & FT_VEL) && vel_retrace && (P.mesh_vel.x != R(0) || P.mesh_vel.y != R(0) || P.mesh_vel.z != R(0));
  const float ix = 1.0f / (float)ray.x, iy = 1.0f / (float)ray.y, iz = 1.0f / (float)ray.z;
  float nox = -(float)start.x * ix, noy = -(float)start.y * iy, noz = -(float)start.z * iz;
  if (disp) {
    const Vec<R> shift = P.mesh_vel * time;
    nox = -(float)(start.x - shift.x) * ix; noy = -(float)(start.y - shift.y) * iy; noz = -(float)(start.z - shift.z) * iz;
  }
  const float serr = 4e-7f * (fabsf(nox) + fabsf(noy) + fabsf(noz));           // as in slabRay
  SlabRay sr = slabRay(ix, iy, iz, nox, noy, noz, (t_limit < FLT_MAX) ? t_limit * 1.0001f + 1e-4f : FLT_MAX);
  int2 stack[DRT_NODE_STACK];                                                   // (child reference, entry distance bits)
  int sp = 0;
  int cur = 0;
  bool found = false;
  for (;;) {
    while (cur >= 0) {                                                          // ---- internal nodes
      if (COUNT) cnt.node_tests += 4;
      cur = bvh4Visit<CLOSEST>(P.mesh_nodes, cur, sr, stack, sp, P.overflow);
    }
    if (cur == DRT_MESH_DONE) break;
    {                                                                           // ---- leaf: exact test
      const int tri = -cur - 1;
      if (COUNT) cnt.geom_tests[G_TRI]++;
      const MeshTri<R>& tr = P.mesh_tris[tri];
      float t;
      if (disp) { const Vec<R> shift = P.mesh_vel * time; t = meshTriT<R>(tr.A + shift, tr.B + shift, tr.C + shift, ray, start); }
      else t = meshTriT<R>(tr.A, tr.B, tr.C, ray, start);
      if (CLOSEST) {
        if (t > 0.0001f && t < h->t) {
          h->t = t; h->geom = P.n_geoms + tri; h->inside = 0; h->checker_sel = 0; found = true;
          sr.lim = (t * 1.0001f + 1e-4f) + serr;
        }
      } else if (t > 0.001f && t < t_limit) {
        if ((F & FT_VEL) && vel_retrace) return true;                           // a velocity re-trace has no reference gather: every triangle is a candidate
        if (t > t_limit * 1e-3f * 1.001f + 2e-3f) return true;                  // touch point ahead of the gather origin
        NodeD<R> nd;                                                            // its own leaf box, BoundingVolume semantics
        nd.lo = mk<R>(fmin(fmin(tr.A.x, tr.B.x), tr.C.x) - R(1e-2), fmin(fmin(tr.A.y, tr.B.y), tr.C.y) - R(1e-2),
                      fmin(fmin(tr.A.z, tr.B.z), tr.C.z) - R(1e-2));
        nd.hi = mk<R>(fmax(fmax(fmax(tr.A.x, tr.B.x), tr.C.x), (R)FLT_MIN) + R(1e-2),
                      fmax(fmax(fmax(tr.A.y, tr.B.y), tr.C.y), (R)FLT_MIN) + R(1e-2),
                      fmax(fmax(fmax(tr.A.z, tr.B.z), tr.C.z), (R)FLT_MIN) + R(1e-2));
        nd.leaf = 1;
        Moved<R> still; still.val = 0; still.time = 0; still.velocity_mode = 0;
        const Vec<R> inv = mk<R>(R(1) / gather_ray.x, R(1) / gather_ray.y, R(1) / gather_ray.z);
        if (boxHit<R, F>(nd, gather_ray, inv, gather_start, still)) return true;
      }
    }
    cur = bvh4Pop<CLOSEST>(stack, sp, sr.lim);
  }
  return found;
}

// Rectangle::samplePoint (geometry.cpp:772-782)
template <typename R>
__device__ inline Vec<R> rectSample(const Vec<R>& A, const Vec<R>& B, const Vec<R>& D, uint32_t key, uint32_t dim) {
  float x = rng_u01(key, dim);
  float y = rng_u01(key, dim + 1);
  return A + (R)x * (B - A) + (R)y * (D - A);
}


template <typename R>
__device__ inline Vec<R> eyeRay(const Params<R>& P, int i, int j) {  // getPerspEyeRay helpers.h:320-324
  float su = P.l + (P.r - P.l) * i / P.xRes;
  float sv = P.b + (P.t - P.b) * j / P.yRes;
  return (R)su * P.X + (R)sv * P.Y - (R)P.near_plane * P.Z;
}


// ---- out-of-line helpers ---------------------------------------------------------
// render_wave is fetch-bound when everything is inlined (14k SASS instructions = 225 KB,
// ncu "no_instructions" stalls: profiles/r1_band_wave.txt).  Blocks that are large (double
// precision pow/exp/acos/sin/cos expansions) or rarely taken are kept out of line so the
// trace / shadow / shade loops stay compact in the instruction caches.
static __device__ __noinline__ double drt_pow(double x, double y) { return pow(x, y); }
__device__ __forceinline__ double pow5(double x) { const double x2 = x * x; return x2 * x2 * x; }

// sphereLight::sampleRay (geometry.cpp:2770-2826); returns the sampled POINT (quirk Q10)
template <typename R>
__device__ __noinline__ bool sampleSphereLight(const LightD<R>& L, const Vec<R>& isectP, uint32_t path, int li, Vec<R>& out) {
  // one evaluation site for the sample (the transcendental expansions are a few hundred instructions), sin and cos of an
  // angle from one sincos: the same values as separate calls, one argument reduction instead of two
  Vec<R> tmp;
  const Vec<R> pc = isectP - L.center;
  for (int attempt = 0;; attempt++) {
    const double theta = 2 * DRT_PI * (double)rng_u01(path, rng_dim_light(li, attempt));
    const double phi = acos(1 - 2 * (double)rng_u01(path, rng_dim_light(li, attempt) + 1));
    double st, ct, sp, cp;
    sincos(theta, &st, &ct);
    sincos(phi, &sp, &cp);
    const Vec<R> dirv = mk<R>((R)(sp * ct), (R)(sp * st), (R)cp);
    tmp = (R)L.radius * dirv + L.center;
    const Vec<R> d = tmp - L.center;
    const bool bad = dot(d, pc) < R(0) || (L.use_baxis && dot(d, L.baxis) < R(0));
    if (!bad) break;
    if (20 - attempt < 0) return false;                               // sample_limit ran out: throws geometry.cpp:2785-2789
    const Vec<R> rev = (R)(-L.radius) * dirv + L.center;
    const Vec<R> dr = rev - L.center;
    const bool ok = dot(dr, pc) >= R(0) && (!L.use_baxis || dot(dr, L.baxis) >= R(0));
    if (ok) { tmp = rev; break; }
  }
  out = tmp;
  return true;
}

// BRDF switch of rayColor (render_final_project.cpp:894-948) for one unoccluded light.
template <typename R>
__device__ __noinline__ void evalBRDF(const PrimD<R>& pr, const float* Lcolor, const float* shape_color, const Vec<R>& e,
                                      const Vec<R>& normal, const Vec<R>& sray, const Vec<R>& sdir, float phong, double* ray_color) {
  if (pr.model == 1) {                                              // oren-nayar
    float vn = (float)dot(e, normal);
    float ln = (float)dot(sdir, normal);
    float irradiance = fmaxf(0.0f, ln);
    float vn_theta = acosf(vn);
    float ln_theta = acosf(ln);
    float angleDiff = (float)fmax(0.0, (double)dot(normalized(e - normal * (R)vn), normalized(sray - normal * (R)ln)));
    float alpha = fmaxf(vn_theta, ln_theta);
    float beta = fminf(vn_theta, ln_theta);
    float f = pr.on_A + pr.on_B * angleDiff * sinf(alpha) * tanf(beta);
    for (int c = 0; c < 3; c++) ray_color[c] = (((double)shape_color[c] * (double)Lcolor[c]) * (double)irradiance) * (double)f;
  } else if (pr.model == 2) {                                       // cook-torrance
    Vec<R> H = normalized(e + sray);                                // unnormalised sray (Q9)
    float hn = (float)fmax(0.0, (double)dot(normal, H));
    float vh = (float)dot(e, H);
    float vn = (float)dot(e, normal);
    float ln = (float)dot(sdir, normal);
    float alpha = acosf(hn);
    double r2 = (double)pr.roughness * (double)pr.roughness;
    double ca = (double)cosf(alpha);
    double ta = (double)(tanf(alpha) / pr.roughness);
    float D = (float)(1.0 / (r2 * (ca * ca * ca * ca)) * exp(-(ta * ta)));
    float G1 = (float)(2.0 * hn * vn / vh);
    float G2 = (float)(2.0 * hn * ln / vh);
    float G = fminf(1.0f, fminf(G1, G2));
    float F = (float)((double)(pr.schlick_R0 + (1 - pr.schlick_R0)) + pow5((double)(1 - vn)));   // helpers.h:316, Q8
    float FDG = F * D * G;
    double den = (double)(ln * vn) * DRT_PI;
    float mx = fmaxf(0.0f, ln);
    for (int c = 0; c < 3; c++) {
      double sh = (0.4 * (double)Lcolor[c]) * (double)mx + ((0.8 * (double)Lcolor[c]) * (double)FDG) / den;
      ray_color[c] = (double)shape_color[c] * sh;
    }
  } else if (pr.model == 3) {                                       // raw
    for (int c = 0; c < 3; c++) ray_color[c] = shape_color[c];
  } else {                                                          // Lambert + Phong :943-948
    Vec<R> rr = normalized(R(-1) * sray + (R(2) * dot(normal, sray)) * normal);   // :856
    double lam = fmax(0.0, (double)dot(normal, sdir));
    double base = fmax(0.0, (double)dot(rr, e));
    double spec;
    if (phong == 10.0f) { const double b2 = base * base, b4 = b2 * b2; spec = b4 * b4 * b2; }   // the reference's fixed exponent (:72)
    else spec = drt_pow(base, (double)phong);
    for (int c = 0; c < 3; c++) {
      double sh = (double)Lcolor[c] * lam + (double)Lcolor[c] * spec;
      ray_color[c] = (double)shape_color[c] * sh;
    }
  }
}

// A rayColor invocation (render_final_project.cpp:487-961) is processed in two steps so the
// warp can regroup between them (render_wave): traceRay() finds the closest hit
// (:491-544), shadeHit() does everything after it (:546-960).
//
// Every invocation ADDS exactly one k-weighted term to the sample's colour (emissive
// term or the hits-averaged light sum) and spawns up to brdf_samples+1 child rays; the
// children are returned to the caller, which owns the scheduling.
// What TRACE leaves for SHADE about a ray that hit: 16 bytes.  The ray itself stays in its pool slot.
struct alignas(16) HitRef {
  float t;
  int geom;
  int inside_sel;   // inside | checker_sel << 1
  int slot;         // pool slot of the ray
};

// shading record of mesh triangle `tri`: the mesh's material table follows the analytic primitives
template <typename R>
__device__ __forceinline__ int meshOwner(const Params<R>& P, const int tri) {
  return P.mesh_prim + (P.mesh_mat ? (int)__ldg(P.mesh_mat + tri) : 0);
}

// Returns true when the ray hit something (h filled in).  `motion` is -1 unless this task is
// on the "last invocation" chain that decides in_motion (quirk Q4), else the new flag value.
template <typename R, int F, bool COUNT>
__device__ inline bool traceRay(const Params<R>& P, const SlabTab gb, const Task<R>& T, HitRec& h, int& motion,
                                Counts& cnt) {
  motion = -1;
  if (T.depth == 0) return false;                                       // :489
  if (COUNT) cnt.rays++;
  const Moved<R> mv = makeMoved<R, F>(P, T.dt);
  closestHit<R, F, COUNT>(P, gb, mv, T.dir, T.org, h, cnt);
  if ((F & FT_MESH) && P.n_mesh_tris > 0) {
    meshTraverse<R, F, COUNT, true>(P, T.dir, T.org, h.t, &h, T.dir, T.org, (F & FT_VEL) && mv.velocity_mode, mv.time, cnt);
  }
  // the in_motion chain only matters when a blur re-trace can follow
  if ((F & (FT_VEL | FT_REFBLUR)) && (T.bits & TASK_CHAIN)) motion = 0;             // :519
  if (h.geom < 0) return false;                                         // :541-544
  if ((F & (FT_VEL | FT_REFBLUR)) && (T.bits & TASK_CHAIN)) {
    const int owner = h.geom >= P.n_geoms ? meshOwner(P, h.geom - P.n_geoms) : geomRecs<R, F>(P)[h.geom].owner;
    motion = (primRecs<R, F>(P)[owner].flags & 2) ? 1 : 0;                        // DRT_FLAG_MOTION, :564
  }
  return true;
}

//   stack[0..n_out) : child tasks in the reference's call order
//   add / has_add   : the term to accumulate
//
// Shading one hit is itself split in three so that the shadow rays -- one per (hit, light)
// pair -- can be spread over all lanes of the warp:
//   shadeA     per hit : normal, refraction / reflection / glossy children, emissive term;
//   shadowPair per pair: LightPrimitive::sampleRay + the occlusion test;
//   shadeB     per hit : texture lookup + BRDF for the unoccluded lights, `hits` average.
// The lane that ran shadeA for a hit also runs shadeB for it, so the hit's state stays in
// registers (ShadeState); only the hit point and the pair results go through memory.
template <typename R>
struct ShadeState {
  Vec<R> isectP, normal, e;
  Moved<R> mv;
  float shape_color[3];
  float k;
  uint32_t path;   // the invocation's key in the sample stream (light samples are drawn from it)
  int prim;
  int tri;         // mesh triangle id, or -1
  bool lights;     // the hit is not a light shape: the light loop has to run
  bool aborted, early;
  int hits;
  double tmp[3];
};

template <typename R>
struct PairIn {   // what a shadow pair needs to know about its hit (kept in the hit lane's registers, fetched by shuffle)
  Vec<R> isectP;
  uint32_t path;
  float val, dt;
  int want;
};
// Results of the (hit, light) pairs of one warp pass, index light * 32 + hit.  The visibility flag goes through the warp's
// slice of shared memory.  The light vector `sray` is NOT passed on for point and rectangle lights: the hit lane draws it
// again from the keyed stream (the same expression, so the same bits) -- cheaper than a 24-byte round trip through global
// memory per pair, every byte of which also reached DRAM (28 GB of the 135 GB a bench frame wrote).  Only the sphere
// light, whose sampler is a rejection loop over acos / sin / cos, hands its sample over in global structure-of-arrays
// scratch (the 32 pair lanes of a pass write neighbouring words, the 32 hit lanes read neighbouring words back).
template <typename R>
struct PairOut {
  R* x; R* y; R* z;          // sray of sphere-light pairs (global scratch)
  unsigned char* state;      // shared memory: 0 occluded, 1 visible, 2 the light sampler aborted (reference throws)
};
template <typename R>
__host__ __device__ constexpr size_t pairOutBytes() { return (size_t)32 * DRT_PAIR_LIGHTS * 3 * sizeof(R); }

template <typename R, int F, bool COUNT>
__device__ void shadeA(const Params<R>& P, const Task<R>& T, const HitRec& h, Task<R>* stack, int& n_out, double (&add)[3],
                       bool& has_add, bool& aborted, ShadeState<R>& S, Counts& cnt) {
  int sp = 0;
  n_out = 0; has_add = false;
  add[0] = add[1] = add[2] = 0.0;
  const Moved<R> mv = makeMoved<R, F>(P, T.dt);
  S.lights = false; S.aborted = false; S.early = false; S.hits = 0; S.tmp[0] = S.tmp[1] = S.tmp[2] = 0.0; S.mv = mv;
  do {
    const Vec<R> ray = T.dir, eye = T.org;
    const float k = T.k;
    const int mesh_tri = ((F & FT_MESH) && h.geom >= P.n_geoms) ? h.geom - P.n_geoms : -1;
    const int owner = mesh_tri >= 0 ? meshOwner(P, mesh_tri) : geomRecs<R, F>(P)[h.geom].owner;
    const PrimD<R>& pr = primRecs<R, F>(P)[owner];

    const Vec<R> isectP = eye + (R)h.t * ray;                           // :548
    // ---- getNorm of the hit class ------------------------------------------------
    Vec<R> normal;
    if (pr.type == 0) {                                                 // Sphere geometry.cpp:199-204
      Vec<R> nn = isectP - shiftPoint<R, F>(mv, 0, pr.vel, pr.pA);
      normal = nn / norm(nn);
    } else if (pr.type == 1 || pr.type == 7) {                          // Cylinder geometry.cpp:419-425
      const Vec<R> c1 = shiftPoint<R, F>(mv, 0, pr.vel, pr.pA);
      Vec<R> axis = pr.pG;
      if ((F & FT_VEL) && (pr.flags & 64) && mv.velocity_mode) axis = normalized((pr.n1 + pr.n2 * mv.time) - c1);   // DRT_FLAG_VERTEX_MOTION: n1 = c2, n2 = its velocity
      Vec<R> pc = isectP - c1;
      normal = normalized(pc - dot(pc, axis) * axis);
    } else if ((F & FT_BOX) && pr.type == 9) {                          // RectPrismWithCylinder geometry.cpp:1796-1821 (lastHit is -1 by now)
      const float eps = 1e-3f;
      const Vec<R> pa = isectP - shiftPoint<R, F>(mv, 0, pr.vel, pr.pA);
      if (dot(pa, pr.n0) <= (R)eps) normal = pr.n0;
      else if (dot(pa, pr.n1) <= (R)eps) normal = pr.n1;
      else if (dot(pa, pr.n2) <= (R)eps) normal = pr.n2;
      else { aborted = true; break; }                                   // throws :1819-1820
    } else if ((F & FT_BOX) && pr.type == 10) {                         // RectPrismWithHoles geometry.cpp:2204-2246
      normal = prismHolesNorm<R>(pr, isectP, h.checker_sel >= 3 ? h.checker_sel - 3 : -1, aborted);
      if (aborted) break;
    } else if (pr.type == 4 || ((F & FT_BOX) && pr.type == 8)) {        // RectPrismV2 geometry.cpp:863-920, RectPrism 1279-1379
      const float eps = 1e-3f;
      Vec<R> dA = normalized(isectP - shiftPoint<R, F>(mv, 0, pr.vel, pr.pA));
      Vec<R> dG = normalized(isectP - shiftPoint<R, F>(mv, 0, pr.vel, pr.pG));
      float pa_bot = fabsf((float)dot(dA, pr.n0)), pg_bot = fabsf((float)dot(dG, pr.n0));
      float pa_right = fabsf((float)dot(dA, pr.n1)), pg_right = fabsf((float)dot(dG, pr.n1));
      float pa_front = fabsf((float)dot(dA, pr.n2)), pg_front = fabsf((float)dot(dG, pr.n2));
      if (pa_bot <= eps || pg_bot <= eps) normal = pr.n0;
      else if (pa_right <= eps || pg_right <= eps) normal = pr.n1;
      else if (pa_front <= eps || pg_front <= eps) normal = pr.n2;
      else {
        float min_side = fminf(fminf(fminf(pa_bot, pg_bot), fminf(pa_right, pg_right)), fminf(pa_front, pg_front));
        if (pa_bot == min_side || pg_bot == min_side) normal = pr.n0;
        else if (pa_right == min_side || pg_right == min_side) normal = pr.n1;
        else normal = pr.n2;
      }
    } else if (mesh_tri >= 0) {                                         // Triangle::getNorm geometry.cpp:588-594
      const MeshTri<R>& tr = P.mesh_tris[mesh_tri];
      const Vec<R> tA = shiftPoint<R, F>(mv, 0, P.mesh_vel, tr.A), tB = shiftPoint<R, F>(mv, 0, P.mesh_vel, tr.B), tC = shiftPoint<R, F>(mv, 0, P.mesh_vel, tr.C);
      normal = normalized(cross(tB - tA, tC - tA));
    } else {
      normal = pr.n0;                                                   // Triangle / Rectangle family
    }
    const Vec<R> in = normalized(ray);
    if (dot(in * R(1e4), normal) >= R(0)) normal = normal * R(-1);      // fixNorm geometry.cpp:17-24

    float shape_color[3];
    if (h.checker_sel == 1) { shape_color[0] = pr.color1[0]; shape_color[1] = pr.color1[1]; shape_color[2] = pr.color1[2]; }
    else if (h.checker_sel == 2) { shape_color[0] = pr.color2[0]; shape_color[1] = pr.color2[1]; shape_color[2] = pr.color2[2]; }
    else if ((F & FT_BOX) && h.checker_sel >= 3) {                      // the wall of a prism's hole: the hole's own colour
      const HoleD<R>& hd = pr.holes[h.checker_sel - 3];
      shape_color[0] = hd.color[0]; shape_color[1] = hd.color[1]; shape_color[2] = hd.color[2];
    }
    else { shape_color[0] = pr.color[0]; shape_color[1] = pr.color[1]; shape_color[2] = pr.color[2]; }

    // ---- reflection / refraction children (:574-769) ---------------------------
    if (P.reflect && pr.material != 0) {
      const float eps = 1e-3f;
      const bool glossy = (pr.flags & 8) != 0;                          // DRT_FLAG_GLOSSY
      float k_refl = 1, k_refr = 1;
      int n_children = 0;        // children pushed for this node, in the reference's call order
      int first_child = sp;
      if ((F & FT_GLASS) && pr.material == 1) {                         // glass :592-626
        float cos_theta = (float)dot(normal, -in);
        float sin_theta = (float)sqrt(1.0 - (double)cos_theta * (double)cos_theta);
        float refr_1 = h.inside ? P.refr_glass : P.refr_air;
        float refr_2 = h.inside ? P.refr_air : P.refr_glass;
        double din = (double)dot(in, normal);
        float rr = refr_1 / refr_2;
        float int_refl_check = (float)(1.0 - (double)rr * (double)rr * (1.0 - din * din));   // helpers.h:286
        if (!(int_refl_check < 0)) {
          float s1 = rr * sin_theta;
          float s2 = 1 / sin_theta;
          Vec<R> out = (R)s1 * ((R)s2 * (in + normal * (R)cos_theta)) - (R)sqrtf(int_refl_check) * normal;
          float gg = P.refr_glass / P.refr_air;
          float cos_phi = (float)sqrt(1.0 - (double)gg * (double)gg * (1.0 - din * din));       // :619
          // fresnel helpers.h:297-303
          float rho_par = (P.refr_glass * cos_theta - P.refr_air * cos_phi) / (P.refr_glass * cos_theta + P.refr_air * cos_phi);
          float rho_perp = (P.refr_air * cos_theta - P.refr_glass * cos_phi) / (P.refr_air * cos_theta + P.refr_glass * cos_phi);
          k_refl = (float)(0.5 * ((double)rho_par * (double)rho_par + (double)rho_perp * (double)rho_perp));
          k_refr = 1 - k_refl;
          if (sp < DRT_MAX_CHILDREN) {
            Task<R>& c = stack[sp++];
            c.org = isectP + in * (R)eps; c.dir = out; c.k = k_refr * k; c.path = rng_key_child(T.path, 0);
            c.depth = (unsigned char)(T.depth - 1); c.bits = 0; c.slot = T.slot; c.dt = T.dt; n_children++;
          }
        }
      }
      Vec<R> refl_ray = in - (R(2) * dot(normal, in)) * normal;         // :628
      R rdn = dot(refl_ray, normal);
      if (rdn <= R(0)) { aborted = true; break; }                       // throws :631-638
      if (rdn > (R)eps) {                                               // :641
        if (glossy && !P.nogloss) {                                     // :644-762
          Vec<R> gloss_ray = refl_ray * R(2);
          const float length = 1, width = 0.5f;
          Vec<R> length_vector = normalized(cross(gloss_ray, mk<R>(1, 0, 0)));
          if (isZero(length_vector)) length_vector = cross(gloss_ray, mk<R>(0, 0, 1));
          Vec<R> cc = gloss_ray + isectP;
          Vec<R> p1 = (R)(length / 2) * length_vector + cc;
          Vec<R> width_vector = normalized(cross(-gloss_ray, length_vector));
          Vec<R> A = width_vector * (R)width / R(2) + p1;
          Vec<R> B = A - length_vector * (R)length;
          Vec<R> C = B - width_vector * (R)width;
          Vec<R> D = A - width_vector * (R)width;
          Vec<R> width_adj = width_vector;
          if (dot(width_vector, normal) <= R(0)) width_adj = -width_adj;
          Vec<R> length_adj = length_vector;
          if (dot(length_vector, normal) <= R(0)) length_adj = -length_adj;
          Vec<R> step = width_adj * R(0.1) + length_adj * R(0.1);
          // the reference loops unboundedly (:697-712); 4096 steps of 0.1 bound a hang
          for (int it = 0; it < 4096 && dot(A - isectP, normal) <= R(0); it++) A = A + width_adj * R(0.1) + length_adj * R(0.1);
          for (int it = 0; it < 4096 && dot(B - isectP, normal) <= R(0); it++) B = B + width_adj * R(0.1) + length_adj * R(0.1);
          for (int it = 0; it < 4096 && dot(C - isectP, normal) <= R(0); it++) C = C + width_adj * R(0.1) + length_adj * R(0.1);
          for (int it = 0; it < 4096 && dot(D - isectP, normal) <= R(0); it++) D = D + width_adj * R(0.1) + length_adj * R(0.1);
          (void)step; (void)C;
          for (int i = 0; i < P.brdf_samples; i++) {                    // :715-761
            int attempt = 0;
            Vec<R> sample_refl = rectSample<R>(A, B, D, T.path, rng_dim_gloss(i, attempt)) - isectP;
            int sample_limit = 10;
            while (dot(sample_refl, normal) <= R(0)) {
              if (sample_limit < 0) { aborted = true; break; }          // throws :724-740
              float multiplier = ldexpf(1.0f, 11 - sample_limit);                     // pow(2, 11 - sample_limit)
              gloss_ray = refl_ray * (R)multiplier;
              length_vector = normalized(cross(gloss_ray, mk<R>(1, 0, 0)));
              if (isZero(length_vector)) length_vector = cross(gloss_ray, mk<R>(0, 0, 1));
              cc = gloss_ray + isectP;
              p1 = (R)(length / 2) * length_vector + cc;
              width_vector = normalized(cross(-gloss_ray, length_vector));
              A = width_vector * (R)width / R(2) + p1;
              B = A - length_vector * (R)length;
              D = A - width_vector * (R)width;
              attempt++;
              sample_refl = rectSample<R>(A, B, D, T.path, rng_dim_gloss(i, attempt)) - isectP;
              sample_limit--;
            }
            if (aborted) break;
            if (sp < DRT_MAX_CHILDREN) {
              Task<R>& c = stack[sp++];
              c.org = isectP + sample_refl * (R)eps; c.dir = sample_refl; c.k = k_refl * k / P.brdf_samples;
              c.path = rng_key_child(T.path, 2 + i); c.depth = (unsigned char)(T.depth - 1); c.bits = 0; c.slot = T.slot; c.dt = T.dt; n_children++;
            }
          }
          if (aborted) break;
        } else {                                                        // mirror :765
          if (sp < DRT_MAX_CHILDREN) {
            Task<R>& c = stack[sp++];
            c.org = isectP + refl_ray * (R)eps; c.dir = refl_ray; c.k = k_refl * k; c.path = rng_key_child(T.path, 1);
            c.depth = (unsigned char)(T.depth - 1); c.bits = 0; c.slot = T.slot; c.dt = T.dt; n_children++;
          }
        }
      }
      // the reference's LAST child call continues the in_motion chain (quirk Q4)
      if ((T.bits & TASK_CHAIN) && n_children > 0) stack[first_child + n_children - 1].bits = TASK_CHAIN;
    }

    // ---- local shading (:772-960) ------------------------------------------------
    if (pr.flags & 1) {                                                 // hit a light shape :775-789
      if (pr.name == 2) {                                               // spherelight
        float hitdot = (float)dot(in, normalized(shiftPoint<R, F>(mv, 0, pr.vel, pr.center) - isectP));
        double f = 0.1 * (double)hitdot + 0.05 * pow5((double)hitdot) + 0.9;
        for (int c = 0; c < 3; c++) add[c] += ((double)k * (double)shape_color[c]) * f;
        has_add = true;
      }
      if (pr.name == 3) {                                               // rectanglelight
        float dist = (float)((double)(norm(isectP - pr.eA) + norm(isectP - pr.eB) + norm(isectP - pr.eC) + norm(isectP - pr.eD)) /
                             (double)pr.e_den);
        double f = 0.1 * (double)dist + 0.05 * pow5((double)dist) + 0.9;
        for (int c = 0; c < 3; c++) add[c] += ((double)k * (double)shape_color[c]) * f;
        has_add = true;
      }
      continue;
    }

    S.isectP = isectP; S.normal = normal; S.e = normalized(eye - isectP);   // :795
    S.shape_color[0] = shape_color[0]; S.shape_color[1] = shape_color[1]; S.shape_color[2] = shape_color[2];
    S.k = k; S.path = T.path; S.prim = owner; S.tri = mesh_tri; S.lights = true;
  } while (0);
  n_out = sp;
}

// LightPrimitive::sampleRay (:802) + the shadow test (:806-855) for one (hit, light) pair.
template <typename R, int F, bool COUNT>
__device__ void shadowPair(const Params<R>& P, const SlabTab gb, const PairIn<R>& in, int li, const PairOut<R>& out, const int oi,
                           Counts& cnt) {
  const LightD<R>& L = lightRecs<R, F>(P)[li];
  const Vec<R> isectP = in.isectP;
  Moved<R> mv;                                      // makeMoved, with blurVal(P, dt) as shadeA evaluated it
  mv.val = (F & FT_REFBLUR) ? in.val : 0.0f;
  mv.time = (F & FT_VEL) ? (R)in.dt : R(0);
  mv.velocity_mode = (F & FT_VEL) ? ((((F & FT_REFBLUR) ? P.blur_mode == 1 : true) && in.dt != 0.0f) ? 1 : 0) : 0;
  Vec<R> sray;
  if (L.type == 0) sray = L.center - isectP;                        // pointLight geometry.cpp:2751-2754
  else if (L.type == 2) sray = rectSample<R>(L.A, L.B, L.D, in.path, rng_dim_light(li, 0)) - isectP;   // :2845-2849
  else {
    if (!sampleSphereLight<R>(L, isectP, in.path, li, sray)) { out.state[oi] = 2; return; }   // (returns the POINT, Q10)
    out.x[oi] = sray.x; out.y[oi] = sray.y; out.z[oi] = sray.z;
  }
  const float t_max = (float)norm(sray);                            // :804
  const Vec<R> sdir = normalized(sray);
  if (COUNT) cnt.shadow_rays++;
  // candidates are gathered along the UNNORMALISED sray from isectP + sray*1e-3 (:814),
  // occlusion is tested along the normalised one from isectP + s^*1e-3 (:838)
  bool threw = false;
  bool occluded = anyHit<R, F, COUNT>(P, gb, mv, sray, isectP + sray * R(1e-3), sdir, isectP + sdir * R(1e-3), t_max, L.prim_index, cnt, threw);
  if ((F & FT_BOX) && threw) { out.state[oi] = 2; return; }             // RectPrismWithHoles::getNorm threw inside intersectShadow
  if ((F & FT_MESH) && !occluded && P.n_mesh_tris > 0)
    occluded = meshTraverse<R, F, COUNT, false>(P, sdir, isectP + sdir * R(1e-3), t_max, nullptr, sray, isectP + sray * R(1e-3),
                                                (F & FT_VEL) && mv.velocity_mode, mv.time, cnt);
  out.state[oi] = occluded ? 0 : 1;
}

// The rest of the light loop (:856-959) for lights [l0, l1) of one hit, in order.
template <typename R, int F, bool COUNT>
__device__ void shadeB(const Params<R>& P, ShadeState<R>& S, const PairOut<R>& res, const int hit_lane, int l0, int l1, Counts& cnt) {
  const PrimD<R>& pr = primRecs<R, F>(P)[S.prim];
  for (int li = l0; li < l1 && !S.early && !S.aborted; li++) {
    const int oi = (li - l0) * 32 + hit_lane;                          // light-major: [light][hit]
    const int state = res.state[oi];
    if (state == 2) { S.aborted = true; break; }                     // throws geometry.cpp:2785-2789
    if (state == 0) continue;                                         // shadowed :852-855
    const LightD<R>& L = lightRecs<R, F>(P)[li];
    Vec<R> sray;                                                      // as shadowPair drew it
    if (L.type == 0) sray = L.center - S.isectP;
    else if (L.type == 2) sray = rectSample<R>(L.A, L.B, L.D, S.path, rng_dim_light(li, 0)) - S.isectP;
    else sray = mk<R>(res.x[oi], res.y[oi], res.z[oi]);
    const Vec<R> sdir = normalized(sray);
      // ---- texture (:859-893) ---------------------------------------------------
      if ((F & FT_TEX) && (pr.flags & 4)) {
        float u = 0, v = 0; int type = 0;
        if (pr.type == 3 || pr.type == 5 || pr.type == 4) {            // Rectangle::getUV (prism: top face)
          Vec<R> uA = shiftPoint<R, F>(S.mv, pr.name == 1 ? GF_NAME_RECTANGLE : 0, pr.vel, pr.uvA);
          Vec<R> uD = shiftPoint<R, F>(S.mv, pr.name == 1 ? GF_NAME_RECTANGLE : 0, pr.vel, pr.uvD);
          u = (float)(norm(cross(S.isectP - uA, pr.uv_ad)) / pr.uv_den_u);
          v = (float)(norm(cross(S.isectP - uD, pr.uv_dc)) / pr.uv_den_v);
          type = 1;
        } else if ((F & FT_BOX) && pr.type >= 8 && pr.type <= 10) {     // RectPrism::getUV geometry.cpp:1440-1461
          const Vec<R> uA = shiftPoint<R, F>(S.mv, 0, pr.vel, pr.uvA), uD = shiftPoint<R, F>(S.mv, 0, pr.vel, pr.uvD);
          if (fabs(dot(cross(pr.uv_ad, pr.uv_dc), S.isectP)) <= R(1e-5)) {
            u = (float)(norm(cross(S.isectP - uA, pr.uv_ad)) / pr.uv_den_u);
            v = (float)(norm(cross(S.isectP - uD, pr.uv_dc)) / pr.uv_den_v);
            type = 1;
          } else type = 0;
        } else if (pr.type == 6) {                                      // CheckerboardWithHole::getUV geometry.cpp:2500-2561
          Vec<R> V_hit = S.isectP - pr.rA;
          float check1 = (float)dot(pr.re1, V_hit), check2 = (float)dot(pr.re2, V_hit);
          if (0 <= check1 && (R)check1 <= pr.rlen1 && 0 <= check2 && (R)check2 <= pr.rlen2) {
            // hole->intersectShadow(VEC3(1,1,1), p - VEC3(1,1,1), FLT_MAX)
            float th, d1, d2;
            Vec<R> one = mk<R>(1, 1, 1);
            bool in_hole;
            {
              const Vec<R> ray1 = one, start1 = S.isectP - one;
              float dn = (float)dot(ray1, pr.hn);
              in_hole = false;
              if (dn != 0.0f) {
                float t_final = (float)(dot(pr.hA - start1, pr.hn) / (R)dn);
                if (!(t_final <= 1e-4f)) {
                  Vec<R> point = start1 + (R)t_final * ray1;
                  Vec<R> Vh = point - pr.hA;
                  float k1 = (float)dot(pr.he1, Vh), k2 = (float)dot(pr.he2, Vh);
                  if (0 <= k1 && (R)k1 <= pr.hlen1 && 0 <= k2 && (R)k2 <= pr.hlen2 && t_final < FLT_MAX) in_hole = true;
                }
              }
              (void)th; (void)d1; (void)d2;
            }
            if (in_hole) type = 0;
            else {
              float gu = (float)(norm(cross(S.isectP - pr.uvA, pr.uv_ad)) / pr.uv_den_u);
              float gv = (float)(norm(cross(S.isectP - pr.uvD, pr.uv_dc)) / pr.uv_den_v);
              float miniu_dist = pr.S / pr.length;
              float miniv_dist = pr.S / pr.width;
              float miniu = gu / miniu_dist - (int)(gu / miniu_dist);
              float miniv = gv / miniv_dist - (int)(gv / miniv_dist);
              if (miniu < 0) miniu = 0;
              if (miniv < 0) miniv = 0;
              u = miniu; v = miniv;
              float bw = pr.borderwidth / (2 * pr.S);
              type = ((miniu <= bw || miniu >= 1 - bw) || (miniv <= bw || miniv >= 1 - bw)) ? 2 : 1;
            }
          } else type = 0;
        } else if (pr.type == 2) {                                      // Triangle::getUV geometry.cpp:447-486
          Vec<R> tA = shiftPoint<R, F>(S.mv, 0, pr.vel, pr.tA), tB = shiftPoint<R, F>(S.mv, 0, pr.vel, pr.tB), tC = shiftPoint<R, F>(S.mv, 0, pr.vel, pr.tC);
          const float* tuv = pr.tuv;
          if ((F & FT_MESH) && S.tri >= 0) {
            const MeshTri<R>& tr = P.mesh_tris[S.tri];
            tA = shiftPoint<R, F>(S.mv, 0, P.mesh_vel, tr.A); tB = shiftPoint<R, F>(S.mv, 0, P.mesh_vel, tr.B); tC = shiftPoint<R, F>(S.mv, 0, P.mesh_vel, tr.C);
            tuv = tr.uv;
          }
          Vec<R> nn = cross(tB - tA, tC - tA);
          Vec<R> n_a = cross(tC - tB, S.isectP - tB), n_b = cross(tA - tC, S.isectP - tC);
          float n_sq = (float)dot(nn, nn);
          float alpha = (float)((double)dot(nn, n_a) / (double)n_sq);
          float beta = (float)((double)dot(nn, n_b) / (double)n_sq);
          float gamma = 1 - alpha - beta;
          if (alpha < 0 || alpha > 1 || beta < 0 || beta > 1 || gamma < 0 || gamma > 1) type = 0;
          else if (!(pr.flags & 32)) { S.aborted = true; break; }         // throws geometry.cpp:456-460
          else {
            u = (float)(((double)alpha * tuv[0] + (double)beta * tuv[2]) + (double)gamma * tuv[4]);
            v = (float)(((double)alpha * tuv[1] + (double)beta * tuv[3]) + (double)gamma * tuv[5]);
            // the reference compares the double UV against [0,1] before narrowing; equivalent here
            type = 1;
          }
        } else if (pr.type == 7) {                                      // CheckerCylinder::getUV geometry.cpp:2588-2630
          Vec<R> p_obj = mulPoint<R>(pr.objM, S.isectP);
          float cu = 0;
          if (S.isectP.x != R(0)) cu = (float)((atan2((double)p_obj.y, (double)p_obj.x) + DRT_PI) / (2 * DRT_PI));
          float cv = (float)((double)p_obj.z / (double)pr.axis_norm);
          float miniu_dist = (float)((double)pr.S / (2 * DRT_PI * (double)pr.radius));
          float miniv_dist = (float)((double)pr.S / (double)pr.axis_norm);
          float miniu = cu / miniu_dist - (int)(cu / miniu_dist);
          float miniv = cv / miniv_dist - (int)(cv / miniv_dist);
          if (miniu > 1 || miniu < 0 || miniv > 1 || miniv < 0) { S.aborted = true; break; }   // throws :2610-2614
          u = miniu; v = miniv;
          float bw = pr.borderwidth / (2 * pr.S);
          type = ((miniu <= bw || miniu >= 1 - bw) || (miniv <= bw || miniv >= 1 - bw)) ? 2 : 1;
        } else { S.aborted = true; break; }
        if (type == 0) { S.early = true; break; }                  // quirk Q7 (:866-869)
        if (u < 0 || v < 0 || u > 1 || v > 1) { S.aborted = true; break; }   // throws :870-877
        if (type == 2) { S.shape_color[0] = pr.bordercolor[0]; S.shape_color[1] = pr.bordercolor[1]; S.shape_color[2] = pr.bordercolor[2]; }
        else {
          int2 dims = P.texdims[pr.tex];
          int x_tex = (int)((dims.x - 1) * u);
          int y_tex = (int)((dims.y - 1) * v);
          float4 tx = tex2D<float4>(P.tex[pr.tex], x_tex + 0.5f, y_tex + 0.5f);   // nearest texel, byte/255
          S.shape_color[0] = tx.x; S.shape_color[1] = tx.y; S.shape_color[2] = tx.z;
        }
      }
      if (COUNT) cnt.shade_evals++;
      // ---- BRDF (:894-948) ---------------------------------------------------------
      double ray_color[3];
      evalBRDF<R>(pr, L.color, S.shape_color, S.e, S.normal, sray, sdir, P.phong, ray_color);
      // !ray_color.isApprox(0): exact-zero test; NaN counts as a hit (:950-954, Q6)
      double sq = ray_color[0] * ray_color[0] + (ray_color[1] * ray_color[1] + ray_color[2] * ray_color[2]);
      if (!(sq <= 0.0)) { S.hits++; for (int c = 0; c < 3; c++) S.tmp[c] += (double)S.k * ray_color[c]; }
  }
}

// ---------------------------------------------------------------------------
// render_wave: why the unit of scheduling is the RAY, not the camera sample.
//
// A thread-per-sample walk of the ray tree leaves most lanes idle: tree sizes are heavy-tailed
// (glossy lobes and glass fan out 2-3 rays per bounce to depth 10), so a warp runs as long as
// its largest tree (ncu, profiles/r1_ncu_full_bench_chunk0_thread_per_sample.txt: 7 of 32 lanes
// active in the object-heavy half of the C2 frame).  Here
//   * a persistent CTA repeatedly claims a batch of DRT_CTA_SLOTS consecutive camera samples
//     from a global counter (dynamic load balance, no tail of straggler blocks);
//   * all pending rays of the batch live in the CTA's LIFO pool in global memory; hits wait in
//     a hit buffer; warps grab 32-item chunks of either, one item per lane;
//   * children are compacted back with a warp prefix sum (shuffle scan);
//   * per-sample radiance is accumulated in 64-bit fixed point (2^-32) with shared-memory
//     atomics, so the sum does not depend on the order rays are processed in and the output
//     stays bit-reproducible.

// per-sample state bits (shared memory) -- the low 4 are also the output flag bits
#define SS_HIT 16u
#define SS_MOTION 32u
#define SS_NAN(c) (256u << (c))
#define SS_PINF(c) (2048u << (c))
#define SS_NINF(c) (16384u << (c))

// ---- the per-pixel shuffle of the lens samples (helpers.h:270-279, render_final_project.cpp:1059) -------------------
// The reference draws antialias_samples lens points per pixel (getDOFSamples), shuffles them with
// `for i = size-1 .. 1: j = round(u * i); swap(v[i], v[j])` and hands point i of the shuffled list to camera sample i.
// Here every draw is keyed, so camera sample s only needs to know WHICH lens point ended up at position s: it undoes the
// swaps in reverse order (lensIndexScan in drt_rng.cuh; only steps i >= s can move the element that ends up at s).
template <typename R>
__device__ __forceinline__ uint32_t pixelKeyOf(const Params<R>& P, const int pt) {
  const int x = P.x0 + pt % P.w, y = P.y0 + pt / P.w;
  return rng_key_pixel(P.seed, (uint32_t)(y * P.xRes + x));
}
// lensSwapTargetsFill: the swap targets j_i of every pixel the CTA's batch [g0, g0 + nv) touches, hashed once by all threads
// into `jt` (shared memory, `cap` 16-bit entries, A per pixel); the samples of a pixel then share them.  Returns false
// (CTA-uniform) when they do not fit; primaryRay then hashes per sample (lensIndexScan).  Ends with a barrier.
template <typename R>
__device__ inline bool lensSwapTargetsFill(const Params<R>& P, const long long g0, const int nv, unsigned short* jt, const int cap) {
  if (!(P.aperture > 0) || nv <= 0) return false;
  const int A = P.antialias_samples;
  const int pt0 = (int)(g0 / P.spp), npx = (int)((g0 + nv - 1) / P.spp) - pt0 + 1;
  if ((long long)npx * A > cap || A > 65535) return false;
  for (int e = threadIdx.x; e < npx * A; e += blockDim.x) {
    const int q = e / A, i = e - q * A;
    jt[e] = (unsigned short)(i ? rng_shuffle_j(pixelKeyOf(P, pt0 + q), i) : 0);
  }
  __syncthreads();
  return true;
}
// lensIndexScan (drt_rng.cuh) over a pixel's table of swap targets
__device__ __forceinline__ int lensIndexFromTable(const unsigned short* j, const int s, const int n_lens) {
  int idx = s;
  for (int i = s > 1 ? s : 1; i < n_lens; i++) {
    const int ji = j[i];
    idx = (idx == i) ? ji : ((idx == ji) ? i : idx);
  }
  return idx;
}

// `perm`: lensSwapTargetsFill's table for the batch starting at pixel `perm_pt0`, or nullptr (hash per sample).
// `lens` false: only the pixel / corner outputs are wanted.
template <typename R>
__device__ __noinline__ void primaryRay(const Params<R>& P, long long gidx, const unsigned short* perm, const int perm_pt0, const bool lens,
                                        Vec<R>& org, Vec<R>& dir, uint32_t& skey, int& pi, int& pj, int& px, int& py) {
  const int s = (int)(gidx % P.spp);
  const int pt = (int)(gidx / P.spp);
  px = pt % P.w; py = pt / P.w;
  const int x = P.x0 + px, y = P.y0 + py;
  const uint32_t pixel = (uint32_t)(y * P.xRes + x);
  const uint32_t pkey = rng_key_pixel(P.seed, pixel);
  skey = rng_key_sample(pkey, (uint32_t)s);
  // lens sample (getDOFSamples :195-210): point `li` of the pixel's shuffled list
  Vec<R> eye_sample = P.eye;
  if (lens && P.aperture > 0) {
    const uint32_t li = (uint32_t)(perm ? lensIndexFromTable(perm + (pt - perm_pt0) * P.antialias_samples, s, P.antialias_samples)
                                        : lensIndexScan(pkey, s, P.antialias_samples));
    float r = (float)((double)(P.aperture / 2) * (double)rng_u01(pkey, 4u * li));
    float theta = (float)(2 * DRT_PI * (double)rng_u01(pkey, 4u * li + 1));
    // cos / sin of the float angle, correctly rounded to float through the double-precision functions: the reference calls
    // the host's cosf / sinf, which CUDA's single-precision versions (1 ulp) miss in several percent of the arguments -- a
    // lens point an ulp off is invisible, except where it flips a grazing shadow test (3 pixels of one fuzz scene)
    double snd, csd;
    sincos((double)theta, &snd, &csd);
    const float cs = (float)csd, sn = (float)snd;
    eye_sample = P.eye + (R)(r * cs) * P.X + (R)(r * sn) * P.Y;
  }
  // jitter (:1048-1056): computed, then truncated by getPerspEyeRay(int,int) (Q1)
  const int ii = s / P.n, jj = s % P.n;
  float adj_x = (float)((double)x + ((double)(float)ii + (double)rng_u01(pkey, 4u * s + 2)) / 9.0);
  float adj_y = (float)((double)y + ((double)(float)jj + (double)rng_u01(pkey, 4u * s + 3)) / 9.0);
  pi = (int)(double)adj_x; pj = (int)(double)adj_y;
  const Vec<R> rayDir = eyeRay<R>(P, pi, pj);
  const Vec<R> focalPoint = P.eye + (R)P.focal_length * rayDir;        // :1069
  org = eye_sample;
  dir = focalPoint - eye_sample;
}

// Scratch of one persistent CTA in global memory (L2 resident):
//   [ pool_cap ray slots | DRT_CTA_HITS hit references | per warp: sphere-light samples of 32 x DRT_PAIR_LIGHTS shadow pairs |
//     three u32 tables of pool_cap / 32 chunk ids: stack, free list, in flight ]
// pool_cap (Params::pool_cap, a multiple of 32) is sized per render on the host from brdf_samples / max_depth / blur_samples.
#ifndef DRT_WAVE_CTAS_PER_SM
#define DRT_WAVE_CTAS_PER_SM 1
#endif
#define DRT_HIT_BUCKETS 64     // hits are grouped by min(geom, 63) before SHADE
template <typename R>
__host__ __device__ constexpr size_t waveScratchBytes(int pool_cap) {
  return (size_t)pool_cap * sizeof(Task<R>) + DRT_CTA_HITS * sizeof(HitRef) + DRT_WAVE_WARPS * pairOutBytes<R>() +
         3 * (size_t)(pool_cap / 32) * sizeof(uint32_t);
}

// render_wave -- phase-locked persistent CTA with CTA-wide work pools.
//
// One CTA of DRT_WAVE_WARPS warps per SM.  All warps run the same phase at the same time
// (GEN -> TRACE -> SHADE, separated by __syncthreads), so the SM's instruction cache only has to
// hold one phase's code: with free-running warps the 14k-instruction kernel saturated the GPC
// instruction cache (ncu: gcc__cache_requests_type_instruction 95 % of peak,
// sm__icc_request_hit_rate 62 %, 43 % of stall samples "no_instructions").
// Pending rays of the CTA's current batch (DRT_CTA_SLOTS camera samples) live in ONE pool per CTA; inside a phase every
// warp keeps grabbing the next 32 items through a shared-memory cursor until the phase's work is gone, so all lanes of
// all warps stay busy and a phase ends within one 32-item bite of the last warp (with warp-private pools 27 % of the
// stall samples were barrier waits).
//
// The pool is managed in CHUNKS of 32 slots (one bite of a warp).  A LIFO stack of chunk ids says which chunks hold
// pending rays, a free list which ones are empty.  TRACE pops a chunk and traces its rays; a ray that hit something STAYS
// in its slot and only a 16-byte reference (HitRef) goes to the hit buffer, so a chunk with hits is "in flight" until SHADE
// has consumed them (a chunk without hits is free at once).  SHADE numbers the pass's children through one CTA-wide
// cursor and writes them, 32 to a chunk, into chunks taken in order from the top of the free list, so a pass leaves at
// most one partly filled chunk; when the phase ends the chunks in flight return to the free list.  (Round 1 copied every
// ray that hit into an 80-byte hit record: 64 more bytes written to DRAM per hit, ~45 GB per bench frame.)  The unfilled
// slots of the pass's last chunk are marked empty (depth 0, which TRACE skips like the reference's `depth == 0` return).
template <typename R, int F, bool COUNT>
__global__ void __launch_bounds__(32 * DRT_WAVE_WARPS, DRT_WAVE_CTAS_PER_SM) render_wave(const __grid_constant__ Params<R> P) {
  // dynamic shared memory: see s_dyn
  unsigned long long(*s_acc)[3] = (unsigned long long(*)[3])s_dyn;
  unsigned int* s_flags = (unsigned int*)(s_dyn + (size_t)DRT_CTA_SLOTS * 24);
  unsigned short* s_order = (unsigned short*)(s_dyn + (size_t)DRT_CTA_SLOTS * 28);
  unsigned char* s_hkey = s_dyn + (size_t)DRT_CTA_SLOTS * 28 + (size_t)DRT_CTA_HITS * 2;
  // s_nst: chunks on the stack; s_nfree: chunks on the free list; s_ninfl: chunks in flight; s_kid: children SHADE placed so far;
  // s_count: rays generated by a blur re-trace pass
  __shared__ int s_nst, s_nfree, s_ninfl, s_kid, s_count, s_nhits, s_grab, s_state, s_nvalid;
  __shared__ int s_hist[DRT_HIT_BUCKETS];                 // SHADE order: counting sort of the hit buffer by geom
  __shared__ long long s_idx0, s_unit_next, s_unit_end;
  // slab-filter table of the whole scene, staged once per persistent CTA (48 B per pair of geoms)
  __shared__ float4 s_gb[3 * DRT_SMEM_GEOMS / 2 + 2 * DRT_SMEM_GEOMS / 8];
  SlabTab gb; gb.g = P.gbounds; gb.s = 0u;
  if (!(F & FT_BIG) || P.n_geoms <= DRT_SMEM_GEOMS) {
    for (int i = threadIdx.x; i < slabPairWords(P.n_geoms) + 2 * ((P.n_geoms + 7) / 8); i += blockDim.x) s_gb[i] = P.gbounds[i];
    gb.s = (unsigned)__cvta_generic_to_shared(s_gb);
  }
  if (F & FT_RECS) {                  // the geom, primitive and light records (published by the barrier below)
    ctaCopy16((void*)geomRecs<R, F>(P), P.geoms, P.n_geoms * (int)sizeof(Geom<R>));
    ctaCopy16((void*)primRecs<R, F>(P), P.prims, P.n_prims * (int)sizeof(PrimD<R>));
    ctaCopy16((void*)lightRecs<R, F>(P), P.lights, P.n_lights * (int)sizeof(LightD<R>));
  }
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31, wib = threadIdx.x >> 5, tid = threadIdx.x;
  const size_t cap = (size_t)P.pool_cap;
  const int n_chunks = P.pool_cap >> 5;
  char* cbase = (char*)P.pool_raw + (size_t)blockIdx.x * waveScratchBytes<R>(P.pool_cap);
  uint4* pool = (uint4*)cbase;                                         // planes of 16-byte words, see poolLoad
  uint4* hits = (uint4*)(cbase + cap * sizeof(Task<R>));               // HitRef records
  char* wbase = (char*)(hits + DRT_CTA_HITS) + (size_t)wib * pairOutBytes<R>();
  uint32_t* stk = (uint32_t*)((char*)(hits + DRT_CTA_HITS) + (size_t)DRT_WAVE_WARPS * pairOutBytes<R>());
  uint32_t* fre = stk + n_chunks;
  uint32_t* infl = fre + n_chunks;
  PairOut<R> pairout;
  __shared__ unsigned char s_pstate[DRT_WAVE_WARPS * 32 * DRT_PAIR_LIGHTS];
  pairout.x = (R*)wbase; pairout.y = pairout.x + 32 * DRT_PAIR_LIGHTS; pairout.z = pairout.y + 32 * DRT_PAIR_LIGHTS;
  pairout.state = s_pstate + wib * 32 * DRT_PAIR_LIGHTS;
  unsigned long long(*acc)[3] = s_acc;
  unsigned int* sfl = s_flags;
  const long long n_units = (P.sample_count + P.unit_samples - 1) / P.unit_samples;
#ifdef DRT_PASS_STATS
  // scheduling statistics of a diagnostic build (tools/pass_stats.py sums the lines printed at exit):
  // [0] batches [1] passes [2] slots traced [3] of them empty [4] SHADE bites [5] partly filled chunks pushed
  // [6] rays traced in the current pass [8 + b] TRACE passes whose ray count has bit length b (b = 0: none; 15: >= 16384)
  __shared__ unsigned long long s_ps[24];
  for (int i = tid; i < 24; i += blockDim.x) s_ps[i] = 0ull;
#endif

  Counts cnt;
  if (COUNT) { cnt.samples = 0; cnt.rays = 0; cnt.shadow_rays = 0; cnt.shade_evals = 0; cnt.noise_evals = 0; cnt.node_tests = 0;
               for (int i = 0; i < 7; i++) cnt.geom_tests[i] = 0; }

  // every chunk starts on the free list, lowest id on top
  for (int i = tid; i < n_chunks; i += blockDim.x) __stcg(fre + i, (uint32_t)(n_chunks - 1 - i));
  // s_state: 0 = no batch, 1 = primary trees in flight, 2 = blur re-traces in flight, 3 = all batches done
  if (tid == 0) { s_nst = 0; s_nfree = n_chunks; s_ninfl = 0; s_kid = 0; s_count = 0; s_nhits = 0; s_state = 0; s_nvalid = 0;
                  s_idx0 = 0; s_unit_next = 0; s_unit_end = 0; }
  __syncthreads();

  for (;;) {
    // ================= GEN: batch bookkeeping (rare) =================================
    if (s_nst == 0 && s_nhits == 0) {                                    // CTA-uniform: the current trees are drained
      const int state = s_state;
      const int n_valid = s_nvalid;
      const long long idx0 = s_idx0;
      const int f0 = s_nfree;                                            // every chunk is free here: f0 == n_chunks
      __syncthreads();
      bool finalize = false;
      if ((F & (FT_VEL | FT_REFBLUR)) && state == 1 && P.blur_samples > 0) {
        // motion blur: re-trace the samples whose in_motion flag ended up set
        // (render_final_project.cpp:1095-1210); the extra traces go through the same pool
        int mine = 0;
        for (int s2 = tid; s2 < n_valid; s2 += blockDim.x) mine |= ((sfl[s2] & (SS_MOTION | SF_ABORT)) == SS_MOTION);
        if (__syncthreads_or(mine)) {
          const bool have_perm = lensSwapTargetsFill<R>(P, P.sample_base + idx0, n_valid, s_order, DRT_CTA_HITS);
          const int perm_pt0 = (int)((P.sample_base + idx0) / P.spp);
          for (int s2 = tid; s2 < n_valid; s2 += blockDim.x) {
            if ((sfl[s2] & (SS_MOTION | SF_ABORT)) != SS_MOTION) continue;
            Task<R> T; uint32_t skey; int pi, pj, px, py;
            primaryRay<R>(P, P.sample_base + idx0 + s2, have_perm ? s_order : nullptr, perm_pt0, true, T.org, T.dir, skey, pi, pj, px, py);
            T.k = 1.0f; T.depth = (unsigned char)P.max_depth; T.bits = 0; T.slot = (unsigned short)s2;
            const int at = atomicAdd(&s_count, P.blur_samples);
            for (int m = 0; m < P.blur_samples; m++) {
              float frame_sample = (float)((double)(float)P.frame + (double)rng_u01(skey, (uint32_t)m) * (double)P.frame_range);
              T.dt = frame_sample - (float)P.frame;
              T.path = rng_key_child(skey, 1 + m);
              // ray number at + m goes to lane (at + m) % 32 of the ((at + m) / 32)-th chunk from the top of the free list
              // (<= DRT_CTA_SLOTS * blur_samples rays, within the pool by the host's sizing)
              const int q = at + m;
              poolStore(pool, cap, (int)__ldcg(fre + f0 - 1 - (q >> 5)) * 32 + (q & 31), T);
            }
          }
          __syncthreads();
          const int total = s_count, nch = (total + 31) >> 5;
          for (int q = total + tid; q < nch * 32; q += blockDim.x) poolStoreEmpty<Task<R>>(pool, cap, (int)__ldcg(fre + f0 - 1 - (q >> 5)) * 32 + (q & 31));
          for (int c = tid; c < nch; c += blockDim.x) __stcg(stk + c, __ldcg(fre + f0 - 1 - c));
          if (tid == 0) { s_state = 2; s_nst = nch; s_nfree = f0 - nch; }   // (s_count is reset behind the next barrier: other warps may still be reading it)
        } else finalize = true;
      } else if (state == 1 || state == 2) finalize = true;
      if (finalize) {
        // ---- per-sample results -----------------------------------------------------
        for (int s2 = tid; s2 < n_valid; s2 += blockDim.x) {
          const unsigned int f = sfl[s2];
          double c[3];
          for (int k = 0; k < 3; k++) {
            c[k] = (double)(long long)acc[s2][k] * (1.0 / 4294967296.0);
            const bool pinf = f & SS_PINF(k), ninf = f & SS_NINF(k);
            if ((f & SS_NAN(k)) || (pinf && ninf)) c[k] = __longlong_as_double(0x7ff8000000000000ll);
            else if (pinf) c[k] = __longlong_as_double(0x7ff0000000000000ll);
            else if (ninf) c[k] = __longlong_as_double(0xfff0000000000000ll);
          }
          uint32_t flags = 0;
          if (f & SF_ABORT) flags |= SF_ABORT;
          else if (!(f & SS_HIT)) {                                     // :1074-1094
            c[0] = c[1] = c[2] = 0;                                     // default_col
            if (P.perlin_cloud) {
              Vec<R> o, d; uint32_t skey; int pi, pj, px, py;
              primaryRay<R>(P, P.sample_base + idx0 + s2, nullptr, 0, false, o, d, skey, pi, pj, px, py);
              int cx = min(max(pi - P.x0, 0), P.w), cy = min(max(pj - P.y0, 0), P.h);   // corner in the tile's (w+1)x(h+1) grid
              flags |= SF_MISS | ((uint32_t)((cx - px) | ((cy - py) << 1)) << SF_CORNER_SHIFT);
              if (P.need[cy * (P.w + 1) + cx] == 0) P.need[cy * (P.w + 1) + cx] = 1;   // benign race: all writers store 1
            }
          } else if (f & SS_MOTION) {
            const double inv = (double)(P.blur_samples + 1);
            c[0] /= inv; c[1] /= inv; c[2] /= inv;
          }
          P.samples[idx0 + s2] = make_float4((float)c[0], (float)c[1], (float)c[2], __uint_as_float(flags));
        }
        if (tid == 0) s_state = 0;
      }
      __syncthreads();
      if (s_state == 0) {                                                // claim the next batch of camera samples
        if (tid == 0) {
          long long next = s_unit_next, end = s_unit_end;
          if (next >= end) {                                             // the CTA's unit is used up: claim another one
            const long long u = (long long)(P.steal ? atomicAdd_system(P.batch_counter, 1ull) : atomicAdd(P.batch_counter, 1ull));
            if (u >= n_units) s_state = 3;
            else {
              next = u * P.unit_samples;
              end = min(next + P.unit_samples, P.sample_count);
              s_unit_end = end;
              if (P.owned) P.owned[u] = 1;
            }
          }
          if (next < end) {
            s_idx0 = next;                                               // chunk-local sample index of slot 0
            s_nvalid = (int)min((long long)DRT_CTA_SLOTS, end - next);
            s_unit_next = next + s_nvalid;
            s_state = 1;
#ifdef DRT_PASS_STATS
            s_ps[0]++;
#endif
          }
        }
        __syncthreads();
        if (s_state == 3) break;
        const int nv = s_nvalid;
        const long long i0 = s_idx0;
        for (int s2 = tid; s2 < DRT_CTA_SLOTS; s2 += blockDim.x) { acc[s2][0] = acc[s2][1] = acc[s2][2] = 0ull; sfl[s2] = 0u; }
        // the hit-sort scratch is idle while the pool is empty: it holds the swap targets of the batch's lens-sample shuffles
        const bool have_perm = lensSwapTargetsFill<R>(P, P.sample_base + i0, nv, s_order, DRT_CTA_HITS);
        const int perm_pt0 = (int)((P.sample_base + i0) / P.spp);
        const int nch = (nv + 31) >> 5;                                  // primary rays -> the first nch chunks of the free list
        for (int s2 = tid; s2 < nch * 32; s2 += blockDim.x) {
          const uint32_t id = __ldcg(fre + f0 - 1 - (s2 >> 5));
          if ((s2 & 31) == 0) __stcg(stk + (s2 >> 5), id);
          if (s2 >= nv) { poolStoreEmpty<Task<R>>(pool, cap, (int)id * 32 + (s2 & 31)); continue; }
          Task<R> T; uint32_t skey; int pi, pj, px, py;
          primaryRay<R>(P, P.sample_base + i0 + s2, have_perm ? s_order : nullptr, perm_pt0, true, T.org, T.dir, skey, pi, pj, px, py);
          T.k = 1.0f; T.path = rng_key_child(skey, 0); T.dt = 0.f; T.depth = (unsigned char)P.max_depth;
          T.bits = TASK_CHAIN | TASK_ROOT; T.slot = (unsigned short)s2;
          poolStore(pool, cap, (int)id * 32 + (s2 & 31), T);
          if (COUNT) cnt.samples++;
        }
        if (tid == 0) { s_nst = nch; s_nfree = f0 - nch; }
      }
      __syncthreads();
    }

    // ================= TRACE: closest hits; a ray that hit stays in its slot, its reference goes to the hit buffer ====
    // (rays that miss are finished: they only update the in_motion chain flag)
    const int nst0 = s_nst;
    if (tid == 0) { s_grab = nst0; s_count = 0; }
    __syncthreads();
    for (;;) {
      if (((volatile int*)&s_nhits)[0] >= DRT_TRACE_HITS_TARGET) break;  // enough hits for a full SHADE pass are waiting
      int top = 0;
      uint32_t id = 0;
      if (lane == 0) { top = atomicSub(&s_grab, 1); if (top > 0) id = __ldcg(stk + top - 1); }
      top = __shfl_sync(FULL, top, 0);
      if (top <= 0) break;
      id = __shfl_sync(FULL, id, 0);
      const int slot = (int)id * 32 + lane;
      bool hit = false;
      HitRec h; h.t = 0.f; h.geom = -1; h.inside = 0; h.checker_sel = 0;
      {
        Task<R> T;
        poolLoad<Task<R>, true>(T, pool, cap, slot);
#ifdef DRT_PASS_STATS
        const int n_empty = __popc(__ballot_sync(FULL, T.depth == 0));
        if (lane == 0) { atomicAdd(&s_ps[2], 32ull); atomicAdd(&s_ps[3], (unsigned long long)n_empty);
                         atomicAdd(&s_ps[6], (unsigned long long)(32 - n_empty)); }
#endif
        if (T.depth != 0 && !(((volatile unsigned int*)sfl)[T.slot] & SF_ABORT)) {   // empty slot / an aborted sample spawns no more work (Q15)
          int motion;
          hit = traceRay<R, F, COUNT>(P, gb, T, h, motion, cnt);
          unsigned int orf = 0;
          if ((T.bits & TASK_ROOT) && hit) orf |= SS_HIT;
          if (motion == 1) orf |= SS_MOTION;
          if (orf) atomicOr(&sfl[T.slot], orf);
          if (motion == 0) atomicAnd(&sfl[T.slot], ~SS_MOTION);
        }
      }
      const unsigned int hm = __ballot_sync(FULL, hit);
      int hbase = 0;
      if (lane == 0) {
        if (hm) { hbase = atomicAdd(&s_nhits, __popc(hm)); __stcg(infl + atomicAdd(&s_ninfl, 1), id); }   // in flight until SHADE is done
        else __stcg(fre + atomicAdd(&s_nfree, 1), id);                                                  // nothing left in it
      }
      hbase = __shfl_sync(FULL, hbase, 0);
      if (hit) {
        const int at = hbase + __popc(hm & ((1u << lane) - 1u));
        __stcg(hits + at, make_uint4(__float_as_uint(h.t), (unsigned)h.geom, (unsigned)(h.inside | (h.checker_sel << 1)), (unsigned)slot));
        s_hkey[at] = (unsigned char)min(h.geom, DRT_HIT_BUCKETS - 1);
      }
    }
    __syncthreads();
    const int nh = s_nhits;
    const int nst_base = max(s_grab, 0);                                 // untouched chunks stay at the bottom of the stack
    __syncthreads();
    if (tid == 0) s_grab = nh;
#ifdef DRT_PASS_STATS
    if (tid == 0) { s_ps[1]++; s_ps[8 + min(64 - __clzll((long long)s_ps[6]), 15)]++; s_ps[6] = 0ull; }
#endif
    // ---- counting sort of the waiting hits by geom: the 32 hits a warp shades together then share
    // the material / model / texture branches of shadeA, evalBRDF and shadeB, and their shadow rays
    // leave from the same surface
    for (int i = tid; i < DRT_HIT_BUCKETS; i += blockDim.x) s_hist[i] = 0;
    __syncthreads();
    int rank[(DRT_CTA_HITS + 32 * DRT_WAVE_WARPS - 1) / (32 * DRT_WAVE_WARPS)];
#pragma unroll
    for (int k = 0; k < (DRT_CTA_HITS + 32 * DRT_WAVE_WARPS - 1) / (32 * DRT_WAVE_WARPS); k++) {
      const int i = tid + k * 32 * DRT_WAVE_WARPS;
      rank[k] = (i < nh) ? atomicAdd(&s_hist[s_hkey[i]], 1) : 0;
    }
    __syncthreads();
    if (wib == 0) {                                                      // exclusive scan of the bucket counts
      int run = 0;
      for (int b0 = 0; b0 < DRT_HIT_BUCKETS; b0 += 32) {
        const int c = s_hist[b0 + lane];
        int incl = c;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { int v = __shfl_up_sync(FULL, incl, d); if (lane >= d) incl += v; }
        s_hist[b0 + lane] = run + incl - c;
        run += __shfl_sync(FULL, incl, 31);
      }
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < (DRT_CTA_HITS + 32 * DRT_WAVE_WARPS - 1) / (32 * DRT_WAVE_WARPS); k++) {
      const int i = tid + k * 32 * DRT_WAVE_WARPS;
      if (i < nh) s_order[s_hist[s_hkey[i]] + rank[k]] = (unsigned short)i;
    }
    __syncthreads();

    // ================= SHADE: waiting hits -> radiance terms + child rays ====================
    const int f0 = s_nfree;                                              // the free list holds still while SHADE runs
    for (;;) {
      int end = 0;
      if (lane == 0) end = atomicSub(&s_grab, 32);
      end = __shfl_sync(FULL, end, 0);
      if (end <= 0) break;
#ifdef DRT_PASS_STATS
      if (lane == 0) atomicAdd(&s_ps[4], 1ull);
#endif
      const int begin = max(end - 32, 0);
      const int take = end - begin;
      const bool active = lane < take;
      Task<R> kids[DRT_MAX_CHILDREN];
      int nk = 0;
      ShadeState<R> S; S.lights = false; S.aborted = false;
      double add[3] = {0, 0, 0}; bool has_add = false, aborted = false;
      unsigned short slot = 0;
      // -- step A (lane = hit): normal, children, emissive term
      PairIn<R> pin; pin.want = 0; pin.isectP = mk<R>(R(0), R(0), R(0)); pin.path = 0u; pin.val = 0.f; pin.dt = 0.f;
      if (active) {
        const uint4 hr = __ldcs(hits + (int)s_order[end - 1 - lane]);
        Task<R> T;
        poolLoad<Task<R>, true>(T, pool, cap, (int)hr.w);
        HitRec h; h.t = __uint_as_float(hr.x); h.geom = (int)hr.y; h.inside = (int)(hr.z & 1u); h.checker_sel = (int)(hr.z >> 1);
        slot = T.slot;
        shadeA<R, F, COUNT>(P, T, h, kids, nk, add, has_add, aborted, S, cnt);
        // children of depth 0 return at once (traceRay, :489) without touching the sample's flags: they are not placed,
        // so TRACE's chunks hold only rays it traces
        if (T.depth == 1) nk = 0;
        if (!aborted && S.lights) { pin.isectP = S.isectP; pin.path = T.path; pin.val = S.mv.val; pin.dt = T.dt; pin.want = 1; }
      }
      // -- step B (lane = (hit, light) pair): light sample + shadow ray, DRT_PAIR_LIGHTS lights at a time; a pair lane
      //    fetches its hit's point from the hit lane by shuffle
      for (int l0 = 0; l0 < P.n_lights; l0 += DRT_PAIR_LIGHTS) {
        const int nl = min(DRT_PAIR_LIGHTS, P.n_lights - l0);
        for (int p0 = 0; p0 < take * nl; p0 += 32) {
          const int pid = p0 + lane;
          const bool on = pid < take * nl;
          const int lj = on ? pid / take : 0, hh = on ? pid - lj * take : 0;   // light-major: one pass of the warp heads for one light
          PairIn<R> q;
          q.isectP = mk<R>(__shfl_sync(FULL, pin.isectP.x, hh), __shfl_sync(FULL, pin.isectP.y, hh), __shfl_sync(FULL, pin.isectP.z, hh));
          q.path = __shfl_sync(FULL, pin.path, hh);
          q.val = (F & FT_REFBLUR) ? __shfl_sync(FULL, pin.val, hh) : 0.f;
          q.dt = (F & (FT_VEL | FT_REFBLUR)) ? __shfl_sync(FULL, pin.dt, hh) : 0.f;
          q.want = __shfl_sync(FULL, pin.want, hh);
          if (on && q.want) shadowPair<R, F, COUNT>(P, gb, q, l0 + lj, pairout, lj * 32 + hh, cnt);
        }
        __syncwarp();
        // -- step C (lane = hit again): texture + BRDF of the unoccluded lights, in light order
        if (active && !aborted && S.lights) shadeB<R, F, COUNT>(P, S, pairout, lane, l0, l0 + nl, cnt);
        __syncwarp();
      }
      if (active) {
        if (S.lights && !aborted) {
          if (S.aborted) aborted = true;
          else if (!S.early && S.hits > 0) { for (int c = 0; c < 3; c++) add[c] += S.tmp[c] / S.hits; has_add = true; }   // :956-959
        }
        if (aborted) { atomicOr(&sfl[slot], SF_ABORT); nk = 0; }
        else if (has_add) {
          unsigned int orf = 0;
          for (int c = 0; c < 3; c++) {
            const double v = add[c];
            if (v != v) orf |= SS_NAN(c);
            // beyond the fixed-point range: recorded like an infinity (the output clamps to [0, 1] anyway), never added --
            // two saturated terms would wrap the 64-bit sum
            else if (v > 1073741824.0) orf |= SS_PINF(c);
            else if (v < -1073741824.0) orf |= SS_NINF(c);
            else atomicAdd(&acc[slot][c], (unsigned long long)__double2ll_rn(v * 4294967296.0));
          }
          if (orf) atomicOr(&sfl[slot], orf);
        }
      }
      // the bite's children take the next `total` numbers of the pass's child cursor, child-index-major: the j-th children
      // of the warp's 32 (geom-sorted) hits -- the same kind of ray leaving the same surface -- end up adjacent, so a later
      // TRACE warp works on rays with similar candidates.  Child v goes to lane v & 31 of chunk c = v >> 5, the c-th chunk
      // from the top of the free list, which the bite that writes its lane 0 puts on the stack at nst_base + c.
      const int total = __reduce_add_sync(FULL, nk);
      if (total) {
        int base = 0;
        if (lane == 0) base = atomicAdd(&s_kid, total);
        base = __shfl_sync(FULL, base, 0);
        const int c0 = base >> 5, room = 32 * f0;                         // the bite's first chunk; child slots the free list holds
        if (lane == 0 && base + total > room) *P.overflow = 1;            // cannot happen within the validated bounds
        int myid = 0;                                                     // lane k: id of chunk c0 + k
        if (lane <= ((base + total - 1) >> 5) - c0 && c0 + lane < f0) {
          myid = (int)__ldcg(fre + f0 - 1 - (c0 + lane));
          if (((c0 + lane) << 5) >= base) __stcg(stk + nst_base + c0 + lane, (uint32_t)myid);
        }
#pragma unroll 1
        for (int j = 0; j < DRT_MAX_CHILDREN; j++) {                      // a rolled loop: the bench workload has at most 3 children per hit
          const unsigned int kbj = __ballot_sync(FULL, nk > j);
          if (!kbj) break;
          const int g = base + __popc(kbj & ((1u << lane) - 1u));
          const int cid = __shfl_sync(FULL, myid, (nk > j) ? (g >> 5) - c0 : 0);
          if (nk > j) {
            if (g < room) poolStore(pool, cap, cid * 32 + (g & 31), kids[j]);
            else atomicOr(&sfl[kids[j].slot], SF_ABORT);                  // overflow: the sample is aborted, the frame rejected
          }
          base += __popc(kbj);
        }
      }
    }
    __syncthreads();
    {  // the children's chunks have left the free list (the unused slots of the last one are marked empty), and the chunks
       // in flight are consumed: back to the free list
      const int nkid = s_kid, nch = min((nkid + 31) >> 5, f0), ninfl = s_ninfl;
      if (nkid < nch * 32) {
        const int last = (int)__ldcg(stk + nst_base + nch - 1);
        for (int q = nkid + tid; q < nch * 32; q += blockDim.x) poolStoreEmpty<Task<R>>(pool, cap, last * 32 + (q & 31));
      }
      for (int i = tid; i < ninfl; i += blockDim.x) __stcg(fre + f0 - nch + i, __ldcg(infl + i));
      __syncthreads();
      if (tid == 0) { s_nfree = f0 - nch + ninfl; s_ninfl = 0; s_nst = nst_base + nch; s_kid = 0; s_nhits = 0; }
#ifdef DRT_PASS_STATS
      if (tid == 0 && nkid < nch * 32) s_ps[5]++;
#endif
    }
    __syncthreads();
  }
#ifdef DRT_PASS_STATS
  if (tid == 0)   // one printf per CTA, so that the lines of different CTAs do not interleave
    printf("PASS_STATS %d %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu\n",
           blockIdx.x, s_ps[0], s_ps[1], s_ps[2], s_ps[3], s_ps[4], s_ps[5], s_ps[8], s_ps[9], s_ps[10], s_ps[11], s_ps[12],
           s_ps[13], s_ps[14], s_ps[15], s_ps[16], s_ps[17], s_ps[18], s_ps[19], s_ps[20], s_ps[21], s_ps[22], s_ps[23]);
#endif

  if (COUNT) {
    atomicAdd(&P.counts->samples, cnt.samples); atomicAdd(&P.counts->rays, cnt.rays);
    atomicAdd(&P.counts->shadow_rays, cnt.shadow_rays); atomicAdd(&P.counts->shade_evals, cnt.shade_evals);
    atomicAdd(&P.counts->node_tests, cnt.node_tests);
    for (int i = 0; i < 7; i++) if (cnt.geom_tests[i]) atomicAdd(&P.counts->geom_tests[i], cnt.geom_tests[i]);
  }
}

// ---------------------------------------------------------------------------
// noise.h -- integer-hash value noise.  The 8 Smoothed3D taps of one
// InterpolatedNoise3D call (noise.h:89-96) read a 4x4x4 block of lattice hashes;
// they are hashed once (64 instead of 216 Noise3D calls per octave).
// prime table of noise.h:12-23 (constant bank: a local array would be re-initialised per call)
__constant__ int kNoisePrimes[10][3] = {{995615039, 600173719, 701464987}, {831731269, 162318869, 136250887},
                                        {174329291, 946737083, 245679977}, {362489573, 795918041, 350777237},
                                        {457025711, 880830799, 909678923}, {787070341, 177340217, 593320781},
                                        {405493717, 291031019, 391950901}, {458904767, 676625681, 424452397},
                                        {531736441, 939683957, 810651871}, {997169939, 842027887, 423882827}};

// Noise3D (noise.h:31-39) of one lattice point, int32 wrap-around explicit.  The reference forms the lattice index in
// double (`x + y * 57 + z * pow(57, 2)`) and converts it back to int, converts the hash to double and divides; the
// conversions (I2F / F2I / F2F) all run on the SM's conversion unit, which the first version of this kernel kept 77 % busy
// (profiles: cloud_corners, XU pipe) while the FP64 pipe idled.  Here the index is integer arithmetic -- the same number
// while |x + 57 y + 3249 z| < 2^31, i.e. for every lattice point within ~600 000 units of the origin; beyond that the
// reference's double -> int conversion is undefined behaviour and this wraps --, the hash becomes a double through the 2^52
// trick, and lattice values widen back to double by bit manipulation: exact replacements that leave one conversion per
// lattice point.
__device__ __forceinline__ float noiseLattice(const uint32_t a, const uint32_t b, const uint32_t c, const int n) {
  uint32_t un = (uint32_t)n;
  un = (un << 13) ^ un;
  const int t = (int)((un * (un * un * a + b) + c) & 0x7fffffffu);
  const double td = __hiloint2double(0x43300000, t) - 4503599627370496.0;   // (double)t, exact for 0 <= t < 2^31
  // the reference divides by denom = 1073741823; the product with the reciprocal differs from the
  // correctly rounded quotient by at most an ulp of a value that is then narrowed to float,
  // and spares a software double division per lattice hash (204 800 per background evaluation)
  return (float)(1.0 - td * (1.0 / 1073741823.0));
}
// float -> double for the lattice values (|v| <= 1, never subnormal): exponent rebias + mantissa shift, exact for every
// value but 0.0f, which comes out as 2^-127 -- one hash in 2^31 gives zero, and 6e-39 vanishes in the rounding of the
// first sum it enters
__device__ __forceinline__ double latticeWiden(const float f) {
  const uint32_t u = __float_as_uint(f);
  const uint32_t hi = (u & 0x80000000u) | (((u >> 3) & 0x0fffffffu) + 0x38000000u);
  return __hiloint2double((int)hi, (int)(u << 29));
}
__device__ inline double cosInterp(double a, double b, double x) {     // noise.h:25-29
  double f = (1 - cos(x * DRT_PI)) * 0.5;
  return a * (1 - f) + b * f;
}

__device__ inline double interpolatedNoise3D(int ip, double x, double y, double z) {   // noise.h:81-107
  int iX = (int)x; double fX = x - iX;
  int iY = (int)y; double fY = y - iY;
  int iZ = (int)z; double fZ = z - iZ;
  // lattice block [iX-1, iX+2] x [iY-1, iY+2] x [iZ-1, iZ+2]
  float lat[4][4][4];
  const uint32_t pa = (uint32_t)kNoisePrimes[ip][0], pb = (uint32_t)kNoisePrimes[ip][1], pc = (uint32_t)kNoisePrimes[ip][2];
  const int base = (iX - 1) + (iY - 1) * 57 + (iZ - 1) * 3249;
#pragma unroll
  for (int a = 0; a < 4; a++)
#pragma unroll
    for (int b = 0; b < 4; b++)
#pragma unroll
      for (int c = 0; c < 4; c++)
        lat[a][b][c] = noiseLattice(pa, pb, pc, base + a + 57 * b + 3249 * c);
  const double alpha = 9.0 / 18, beta = 2.0 / (8 * 18), gamma = 4.0 / (6 * 18), delta = 3.0 / (12 * 18);
  double v[2][2][2];
  // Smoothed3D(ip, iX+dx, iY+dy, iZ+dz) (noise.h:51-70) = alpha * centre + beta * (8 corners) + gamma * (6 sides) + delta *
  // (12 edge neighbours) of a 3x3x3 neighbourhood.  The eight taps overlap: per z-column of the block the two outer values
  // of a tap's three are added once (E), the middle one is widened once (C), and every tap sums columns -- 14 additions
  // and no conversions per tap instead of 26 additions and 27 widenings.  (The order of the additions differs from the
  // reference's expression by design: the sums agree to an ulp or two of values that are narrowed to float further on.)
#pragma unroll
  for (int dz = 0; dz < 2; dz++) {
    double E[4][4], C[4][4];
#pragma unroll
    for (int a = 0; a < 4; a++)
#pragma unroll
      for (int b = 0; b < 4; b++) {
        E[a][b] = latticeWiden(lat[a][b][dz]) + latticeWiden(lat[a][b][dz + 2]);
        C[a][b] = latticeWiden(lat[a][b][dz + 1]);
      }
#pragma unroll
    for (int dx = 0; dx < 2; dx++)
#pragma unroll
      for (int dy = 0; dy < 2; dy++) {
        const int x = 1 + dx, y = 1 + dy;
        const double corners = (E[x - 1][y - 1] + E[x - 1][y + 1]) + (E[x + 1][y - 1] + E[x + 1][y + 1]);
        const double sides = ((C[x - 1][y] + C[x + 1][y]) + (C[x][y - 1] + C[x][y + 1])) + E[x][y];
        const double dg = ((C[x - 1][y - 1] + C[x - 1][y + 1]) + (C[x + 1][y - 1] + C[x + 1][y + 1])) +
                          ((E[x - 1][y] + E[x + 1][y]) + (E[x][y - 1] + E[x][y + 1]));
        v[dx][dy][dz] = alpha * C[x][y] + beta * corners + gamma * sides + delta * dg;
      }
  }
  // cosInterpolate (noise.h:25-29): the blend factor depends only on the axis fraction, so it is
  // evaluated once per axis (3 cosines) instead of once per call (7)
  // cospi(f) for the reference's cos(f * M_PI): the same function of f to within an ulp of a value that ends up in a float
  // a few operations later, without the multiplication's rounding and the general-argument reduction (config 3: 198 -> 193 ms)
  const double gx = (1 - cospi(fX)) * 0.5, gy = (1 - cospi(fY)) * 0.5, gz = (1 - cospi(fZ)) * 0.5;
  const double w3 = v[0][0][0] * (1 - gx) + v[1][0][0] * gx, w4 = v[0][1][0] * (1 - gx) + v[1][1][0] * gx;
  const double w1 = v[0][0][1] * (1 - gx) + v[1][0][1] * gx, w2 = v[0][1][1] * (1 - gx) + v[1][1][1] * gx;
  const double i1 = w3 * (1 - gy) + w4 * gy, i2 = w1 * (1 - gy) + w2 * gy;
  return i1 * (1 - gz) + i2 * gz;
}

// skyColor / cloudColor (:146-192) for one pixel corner, evaluated by a QUAD of lanes.
// The reference marches the ray back to front through ~200 steps (z = clouddist, z -= 0.05 in float, while z > 0); each
// step costs one ValueNoise_3D = four octaves of InterpolatedNoise3D (64 lattice hashes each), and the compositing
// `col = (1 - d) col + d cloud` makes the steps sequential.  With a thread per corner that is a ~5 ms serial chain, which
// is what limits a frame shared by several GPUs (the background pass of 10^6 corners is only a couple of such chains
// long per SM, so the last wave runs half empty).  Here lane 4q + o evaluates octave o of corner q's current step; the
// four octaves are summed in the reference's order after a shuffle and all four lanes replay the (cheap) compositing.
// Same arithmetic per step, a 4x shorter chain, 8 corners per warp.  `active` false: the quad only takes part in the
// shuffles.
template <typename R>
__device__ void cloudColorQuad(const Params<R>& P, const bool active, const Vec<R>& ray, float frame, double (&out)[3], int& steps) {
  const unsigned FULL = 0xffffffffu;
  const int lane = threadIdx.x & 31, octave = lane & 3, quad0 = lane & ~3;
  double sky[3] = {0, 0, 0}, col[3] = {0, 0, 0};
  if (active) {
    Vec<R> rnorm = normalized(ray);
    float sundot = clampf((float)dot(rnorm, P.sun));
    double p1 = pow((double)sundot, 1.0), p2 = pow((double)sundot, 2.0), p256 = pow((double)sundot, 256.0), p8 = pow((double)sundot, 8.0);
    for (int c = 0; c < 3; c++) {
      double cc = (0.05 * P.sun_outer[c]) * p1 + (0.1 * P.sun_inner[c]) * p2 + (0.9 * P.sun_core[c]) * p256;
      double sk = P.bluesky[c] * (1 - 1.5 * p8) + (P.redsky[c] * 1.5) * p8;
      sky[c] = cc + sk * (1.0 - 0.8 * (double)rnorm.y);
      col[c] = sky[c];
    }
  }
  // ValueNoise_3D (noise.h:124-136): frequency 8, 4, 2, 1 and amplitude 1/8, 1/4, 1/2, 1 for octaves 0..3
  const double frequency = (double)(8 >> octave), amplitude = 0.125 * (double)(1 << octave);
  steps = 0;
  for (float z = P.clouddist; z > 0; z = (float)((double)z - 0.05)) {      // the same z sequence on every lane
    double v = 0.0;
    const double py = (double)z * (double)ray.y;
    if (active) {
      const double px = (double)z * (double)ray.x, pz = (double)z * (double)ray.z + (double)frame;
      v = interpolatedNoise3D(octave, px * frequency, py * frequency, pz * frequency) * amplitude;
    }
    const double v0 = __shfl_sync(FULL, v, quad0), v1 = __shfl_sync(FULL, v, quad0 + 1);
    const double v2 = __shfl_sync(FULL, v, quad0 + 2), v3 = __shfl_sync(FULL, v, quad0 + 3);
    steps++;
    if (!active) continue;
    double total = 0;
    total += v0; total += v1; total += v2; total += v3;
    float noise = (float)(0.7 * total);
    float clouddistance = (float)((py + (double)noise) + (double)P.cloudhoff);
    if (clouddistance < 0) {
      float density = clampf(fabsf(clouddistance));
      double d4 = (double)density * 0.4;
      double rev[3] = {sky[2], sky[1], sky[0]};
      for (int c = 0; c < 3; c++) {
        double cloudcolor = 1.0 - (double)density * rev[c];
        col[c] = (1 - d4) * col[c] + d4 * cloudcolor;
      }
    }
  }
  for (int c = 0; c < 3; c++) {
    double v = clampf((float)col[c]);
    col[c] = 3 * pow(v, 2.0) - 2 * pow(v, 3.0);
  }
  double s = col[0] + (col[1] + col[2]);
  for (int c = 0; c < 3; c++) out[c] = (double)(1 + P.saturation) * col[c] - (double)P.saturation * (0.33 * s);
}

// One quad of lanes per pixel corner of the tile's (w+1)x(h+1) grid: a CTA of 128 threads takes a block of 32 corners.  A
// block is either the CTA's own (blockIdx) or -- one frame on several GPUs -- claimed from a counter all devices share,
// the marks and colours then living in the gathering device's maps (peer loads / stores).
#define DRT_CLOUD_BLOCK 32
#ifndef DRT_CLOUD_MIN_BLOCKS
#define DRT_CLOUD_MIN_BLOCKS 3   // 142 registers: three CTAs of four warps per SM (1 -> 208 registers, two CTAs: 205 vs 198 ms on config 3)
#endif
template <typename R>
__global__ void __launch_bounds__(128, DRT_CLOUD_MIN_BLOCKS) cloud_corners(const __grid_constant__ Params<R> P) {
  const int gw = P.w + 1, gh = P.h + 1;
  const int n_blocks = (gw * gh + DRT_CLOUD_BLOCK - 1) / DRT_CLOUD_BLOCK;
  __shared__ int s_blk;
  for (int blk = blockIdx.x;; ) {
    if (P.corner_counter) {
      __syncthreads();
      if (threadIdx.x == 0) s_blk = (int)min(atomicAdd_system(P.corner_counter, 1ull), (unsigned long long)n_blocks);
      __syncthreads();
      blk = s_blk;
    }
    if (blk >= n_blocks) return;
    const int idx = blk * DRT_CLOUD_BLOCK + (threadIdx.x >> 2);
    // 0: not wanted, 2: already computed by an earlier row chunk
    const bool wanted = idx < gw * gh && (P.cloud_only || P.need[idx] == 1);
    if (__ballot_sync(0xffffffffu, wanted)) {                          // some corner of this warp's eight is wanted
      Vec<R> point = mk<R>(R(0), R(0), R(0));
      if (wanted) {
        const int cx = idx % gw, cy = idx / gw;
        const int x = P.x0 + cx, y = P.y0 + cy;
        const Vec<R> rayDir = eyeRay<R>(P, x, y);
        if (P.cloud_only) point = mulPoint<R>(P.cloud_mcam, rayDir + P.eye);             // renderImageCloud :1265-1268
        else {
          const Vec<R> focalPoint = P.eye + (R)P.focal_length * rayDir;
          point = (P.frame >= P.frame_cloud) ? mulPoint<R>(P.new_mcam, focalPoint) : mulPoint<R>(P.mcam, focalPoint);   // :1079-1087
        }
      }
      double c[3];
      int steps;
      cloudColorQuad<R>(P, wanted, point, (float)P.frame, c, steps);
      if (wanted && (threadIdx.x & 3) == 0) {
        P.bg[idx] = make_float4((float)c[0], (float)c[1], (float)c[2], 0.f);
        if (!P.cloud_only) P.need[idx] = 2;
        if (P.counts) atomicAdd(&P.counts->noise_evals, (unsigned long long)steps);
      }
    }
    if (!P.corner_counter) return;
  }
}

// drt_render_multi: a device's corner marks of the current row chunk -> the gathering device's map (peer stores).
// `mine` holds 0 / 1 / 2 like the shared map, 2 only where the shared map already has it.
static __global__ void need_push(const unsigned char* __restrict__ mine, unsigned char* shared, const size_t n) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n && mine[i] == 1) shared[i] = 1;
}

// One thread per pixel: (:1213-1217) + writePPM's truncation (helpers.h:178-179).
template <typename R>
__global__ void __launch_bounds__(256) resolve(const __grid_constant__ Params<R> P, int row0, int rows) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= P.w * rows) return;
  const int px = idx % P.w, py = row0 + idx / P.w;
  // one frame on several GPUs: this GPU writes the pixels of the units it claimed (units cover whole pixels)
  if (P.owned && !P.owned[((long long)idx * P.spp) / P.unit_samples]) return;
  double c[3] = {0, 0, 0};
  bool aborted = false;
  if (P.cloud_only) {
    float4 b = P.bg[py * (P.w + 1) + px];
    c[0] = b.x; c[1] = b.y; c[2] = b.z;
  } else {
    const float4* sp = P.samples + ((long long)(py - row0) * P.w + px) * P.spp;
    for (int s = 0; s < P.spp; s++) {
      float4 v = sp[s];
      uint32_t f = __float_as_uint(v.w);
      if (f & SF_ABORT) aborted = true;
      if (f & SF_MISS) {
        uint32_t corner = f >> SF_CORNER_SHIFT;
        float4 b = P.bg[(py + (int)((corner >> 1) & 1)) * (P.w + 1) + px + (int)(corner & 1)];
        v.x = b.x; v.y = b.y; v.z = b.z;
      }
      c[0] += (double)v.x; c[1] += (double)v.y; c[2] += (double)v.z;
    }
    c[0] /= P.spp; c[1] /= P.spp; c[2] /= P.spp;
  }
  float o[3];
  for (int k = 0; k < 3; k++) o[k] = aborted ? 0.0f : clampf((float)c[k]) * 255.0f;
  const size_t orow = (size_t)(P.h - 1 - py);                        // rows flipped :1215
  const size_t oi = (orow * P.w + px) * 3;
  if (P.out_f32) { P.out_f32[oi] = o[0]; P.out_f32[oi + 1] = o[1]; P.out_f32[oi + 2] = o[2]; }
  for (int k = 0; k < 3; k++) {
    // (unsigned char)float on x86-64: cvttss2si then low byte; NaN -> 0x80000000 -> 0
    int iv = (o[k] == o[k]) ? (int)o[k] : 0;
    P.out_u8[oi + k] = (unsigned char)iv;
  }
}

}  // namespace drt
