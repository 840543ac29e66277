// C ABI (include/drt.h) of the CUDA hot path: scene flattening + upload, kernel
// launches, timing, read-back.  Host code only prepares data; every pixel is
// computed by the kernels in drt_kernels.cuh.  There is no CPU fallback.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/drt.h"
#include "drt_box.cuh"
#include "drt_launch.h"
#include "drt_bvh_order.h"
#include "drt_mesh.h"
#include "drt_skeleton.h"

using namespace drt;

namespace {

thread_local std::string g_err;
int fail(int code, const std::string& m) { g_err = m; return code; }

#define CK(call)                                                                                   \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      return fail(DRT_ERR_CUDA, std::string(#call) + " failed: " + cudaGetErrorString(e_));        \
  } while (0)

typedef Vec<double> D3;
D3 V(const double* p) { return mk<double>(p[0], p[1], p[2]); }
template <typename R> Vec<R> cv(const D3& v) { return mk<R>((R)v.x, (R)v.y, (R)v.z); }
void f3(float* o, const double* p) { o[0] = (float)p[0]; o[1] = (float)p[1]; o[2] = (float)p[2]; }

void rows3x4(double* out, const D3& r0, const D3& r1, const D3& r2, const D3& eye);
#define DRT_SWEPT_FRAMES 1   // the slab-filter boxes of moving geoms cover time offsets up to this many frames
struct RectD { D3 A, nrm, e1, e2; double len1, len2; };
RectD makeRect(const D3& A, const D3& B, const D3& C, const D3& D) {
  RectD r;
  r.A = A;
  r.nrm = normalized(normalized(cross(B - A, C - A)));   // getNorm(start).normalized(), geometry.cpp:671,743-749
  r.e1 = normalized(B - A); r.e2 = normalized(D - A);    // V1.normalized(), V2.normalized()
  r.len1 = norm(B - A); r.len2 = norm(D - A);
  return r;
}

// padded single-precision bounds for the slab filter (drt_kernels.cuh slabMayHit); `planar`: see padBounds in drt_box.cuh
template <typename R>
void setBounds(Geom<R>& g, const D3* pts, int n, double extra, bool planar) {
  double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
  for (int i = 0; i < n; i++) {
    const double v[3] = {pts[i].x, pts[i].y, pts[i].z};
    for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], v[a] - extra); hi[a] = std::max(hi[a], v[a] + extra); }
  }
  float fl[3], fh[3];
  for (int a = 0; a < 3; a++) padBounds(lo[a], hi[a], planar, sizeof(R) == sizeof(float), fl[a], fh[a]);
  g.blo = make_float4(fl[0], fl[1], fl[2], 0.f); g.bhi = make_float4(fh[0], fh[1], fh[2], 0.f);
}

template <typename R>
Geom<R> rectGeom(int type, int owner, int flags, float eps, const RectD& r, float S, const D3& vel) {
  Geom<R> g; memset(&g, 0, sizeof(g));
  g.type = type; g.owner = owner; g.flags = flags; g.eps = eps;
  g.p0 = cv<R>(r.A); g.p1 = cv<R>(r.nrm); g.p2 = cv<R>(r.e1); g.p3 = cv<R>(r.e2);
  g.len1 = (R)r.len1; g.len2 = (R)r.len2; g.f0 = (float)r.len1; g.f1 = (float)r.len2; g.f2 = S;
  g.vel = cv<R>(vel);
  const D3 u = r.e1 * r.len1, v = r.e2 * r.len2;
  D3 pts[8] = {r.A, r.A + u, r.A + v, r.A + u + v};
  int n_pts = 4;
  // Rectangle::intersect accepts a point P of the plane when 0 <= e1.(P - A) <= |B - A| and 0 <= e2.(P - A) <= |D - A|
  // (geometry.cpp:681-686).  For orthogonal edges that is the rectangle.  Several of the reference's own builders list
  // the corners of a wall as (a, b, c, d) with d DIAGONALLY opposite a, so that D - A is a diagonal: the accepted region is
  // then a long parallelogram reaching far beyond the vertices.  The filter box has to hold that region (corners: the
  // solutions of the two projections at their bounds), and the reference finds such a hit only when its BVH gather reaches
  // the leaf -- GF_SPILL makes closestHit / anyHit replay that gather for every hit on this geom.
  const double c = dot(r.e1, r.e2);
  bool unbounded = false;
  if (std::fabs(c) > 1e-12 || std::fabs(dot(r.e2, r.nrm)) > 1e-9 || std::fabs(dot(r.e1, r.nrm)) > 1e-9) {
    g.flags |= GF_SPILL;
    const double den = 1.0 - c * c;
    if (den < 1e-9 || std::fabs(dot(r.e2, r.nrm)) > 1e-9 || std::fabs(dot(r.e1, r.nrm)) > 1e-9) unbounded = true;   // (nearly) parallel edges / a corner off the plane
    else
      for (int k = 0; k < 4; k++) {
        const double d1 = (k & 1) ? r.len1 : 0.0, d2 = (k & 2) ? r.len2 : 0.0;
        pts[n_pts++] = r.A + r.e1 * ((d1 - c * d2) / den) + r.e2 * ((d2 - c * d1) / den);
      }
  }
  setBounds(g, pts, n_pts, 0.0, !(g.flags & GF_SPILL));   // a GF_SPILL region is as thin as the angle between its edges
  if (unbounded) { g.blo = make_float4(-1e30f, -1e30f, -1e30f, 0.f); g.bhi = make_float4(1e30f, 1e30f, 1e30f, 0.f); }
  return g;
}

template <typename R>
void objMatrix(R* out, const D3& axis, const D3& c1) {   // buildCOB(axis) * origin(-c1), geometry.cpp:27-40, 2580-2585
  D3 w = normalized(axis);
  D3 u = normalized(cross(mk<double>(1, 0, 0), w));
  if (!(dot(u, u) > 0)) u = normalized(cross(mk<double>(0, 1, 0), w));
  D3 v = normalized(cross(w, u));
  const D3 rows[3] = {u, v, w};
  for (int i = 0; i < 3; i++) {
    out[4 * i + 0] = (R)rows[i].x; out[4 * i + 1] = (R)rows[i].y; out[4 * i + 2] = (R)rows[i].z;
    // (cob*origin)(i,3) = (r0*0 + r1*0) + (r2*0 + ...) -> -(row . c1) in the 4-term (a+b)+(c+d) order
    out[4 * i + 3] = (R)((rows[i].x * -c1.x + rows[i].y * -c1.y) + (rows[i].z * -c1.z + 0.0));
  }
}

// getBounds of each GeoPrimitive class (geometry.cpp:206-210, 427-431, 596-602, 761-770, 922-941)
void primBounds(const drt_prim& p, double lo[3], double hi[3]) {
  auto acc = [&](const double* v, bool first) {
    for (int a = 0; a < 3; a++) { if (first || v[a] < lo[a]) lo[a] = v[a]; if (first || hi[a] < v[a]) hi[a] = v[a]; }
  };
  const float radius = (float)p.radius;
  switch (p.type) {
    case DRT_PRIM_SPHERE:
      for (int a = 0; a < 3; a++) { lo[a] = p.center[a] - radius; hi[a] = p.center[a] + radius; }
      break;
    case DRT_PRIM_CYLINDER: case DRT_PRIM_CHECKER_CYLINDER:
      for (int a = 0; a < 3; a++) {
        lo[a] = std::min(p.c1[a] - radius, p.c2[a] - radius);
        hi[a] = std::max(p.c1[a] + radius, p.c2[a] + radius);
      }
      break;
    case DRT_PRIM_TRIANGLE: acc(p.A, true); acc(p.B, false); acc(p.C, false); break;
    case DRT_PRIM_RECTPRISMV2: case DRT_PRIM_RECTPRISM: case DRT_PRIM_RECTPRISM_CYL: case DRT_PRIM_RECTPRISM_HOLES:
      acc(p.A, true); acc(p.B, false); acc(p.C, false); acc(p.D, false); acc(p.E, false); acc(p.F, false); acc(p.G, false); acc(p.H, false);
      break;
    default: acc(p.A, true); acc(p.B, false); acc(p.C, false); acc(p.D, false); break;
  }
}

// the flattener's replay of the reference's BVH build over the primitives (drt_bvh_order.h)
ReferenceBVH referenceBVH(const drt_prim* prims, int n_prims) {
  std::vector<double> centers(3 * (size_t)n_prims);
  for (int i = 0; i < n_prims; i++) for (int a = 0; a < 3; a++) centers[3 * i + a] = prims[i].center[a];
  ReferenceBVH bvh;
  bvh.build(centers.data(), n_prims, [&](int prim, double lo[3], double hi[3]) { primBounds(prims[prim], lo, hi); });
  return bvh;
}

// Slab-filter table (drt_kernels.cuh: slabMask) over the padded fp32 boxes of the geoms: one pair record (drt_box.cuh) per
// two geoms, padded to whole groups of 8 geoms (slabPairWords), then one box per group {cx cy cz hx} {hy hz - -}.  Holes
// and the padding entries are empty so that they never pass.
template <typename R>
std::vector<float4> slabTable(const std::vector<Geom<R>>& geoms) {
  const size_t n_pairs = 4 * ((geoms.size() + 7) / 8);
  std::vector<float4> t(3 * n_pairs);
  for (size_t p = 0; p < n_pairs; p++) {
    float c[2][3], h[2][3];
    for (int k = 0; k < 2; k++) {
      const size_t gi = 2 * p + k;
      const bool live = gi < geoms.size() && geoms[gi].type != G_HOLE;
      for (int a = 0; a < 3; a++) {
        if (live) centreHalf((&geoms[gi].blo.x)[a], (&geoms[gi].bhi.x)[a], c[k][a], h[k][a]);
        else { c[k][a] = 0.f; h[k][a] = kEmptyHalf; }
      }
    }
    packPair(&t[3 * p], c[0], h[0], c[1], h[1]);
  }
  for (size_t g0 = 0; g0 < geoms.size(); g0 += 8) {
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    bool any = false;
    for (size_t gi = g0; gi < std::min(geoms.size(), g0 + 8); gi++) {
      if (geoms[gi].type == G_HOLE) continue;
      any = true;
      for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], (&geoms[gi].blo.x)[a]); hi[a] = std::max(hi[a], (&geoms[gi].bhi.x)[a]); }
    }
    float c[3], h[3];
    for (int a = 0; a < 3; a++) {
      if (!any) { c[a] = 0.f; h[a] = kEmptyHalf; continue; }
      centreHalf(lo[a], hi[a], c[a], h[a]);
      h[a] = nextafterf(h[a], INFINITY) * 1.000001f;   // also covers the members' own rounded-up half-extents
    }
    t.push_back(make_float4(c[0], c[1], c[2], h[0]));
    t.push_back(make_float4(h[1], h[2], 0.f, 0.f));
  }
  return t;
}

// For scenes with more geoms than the shared-memory table holds: a 4-wide tree (drt_box.cuh) over the geoms, so that
// closestHit / anyHit gather candidates in O(log n) instead of running the filter over all n.  Median splits of the box
// centres along the widest axis, twice per node; leaf = one geom (reference -(geom + 1)); node 0 is the root.  Empty when
// not built: below that size, and when a slab-box prism is present (its intersectShadow can throw, and which pixels then
// abort depends on the reference's candidate ORDER, which only the linear walk keeps).
template <typename R>
std::vector<float4> geomTree(const std::vector<Geom<R>>& geoms) {
  std::vector<float4> tree;
  std::vector<int> items;
  bool any_box = false;
  for (size_t gi = 0; gi < geoms.size(); gi++) {
    if (geoms[gi].type == G_BOX) any_box = true;
    if (geoms[gi].type != G_HOLE) items.push_back((int)gi);
  }
  if ((int)geoms.size() <= DRT_SMEM_GEOMS || any_box || items.size() < 2) return tree;
  auto centre = [&](int gi, int a) { return 0.5f * ((&geoms[gi].blo.x)[a] + (&geoms[gi].bhi.x)[a]); };
  auto halve = [&](int* first, int* last) {            // median split along the widest axis of the box centres
    float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
    for (int* it = first; it != last; ++it) for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], centre(*it, a)); hi[a] = std::max(hi[a], centre(*it, a)); }
    int ax = 0; for (int a = 1; a < 3; a++) if (hi[a] - lo[a] > hi[ax] - lo[ax]) ax = a;
    int* mid = first + (last - first) / 2;
    std::nth_element(first, mid, last, [&](int x, int y) { const float cx = centre(x, ax), cy = centre(y, ax); return cx < cy || (cx == cy && x < y); });
    return mid;
  };
  // iterative build: a work list of (node index, item range)
  struct Work { int node; int* first; int* last; };
  std::vector<Work> work;
  tree.resize(8);
  work.push_back({0, items.data(), items.data() + items.size()});
  while (!work.empty()) {
    const Work w = work.back(); work.pop_back();
    int* cuts[5] = {w.first, nullptr, nullptr, nullptr, w.last};
    cuts[2] = halve(w.first, w.last);
    cuts[1] = (cuts[2] - cuts[0] >= 2) ? halve(cuts[0], cuts[2]) : cuts[0];
    cuts[3] = (cuts[4] - cuts[2] >= 2) ? halve(cuts[2], cuts[4]) : cuts[2];
    float cc[4][3], hh[4][3]; int ref[4]; int m = 0;
    for (int k = 0; k < 4; k++) {
      if (cuts[k + 1] == cuts[k]) continue;
      float lo[3] = {FLT_MAX, FLT_MAX, FLT_MAX}, hi[3] = {-FLT_MAX, -FLT_MAX, -FLT_MAX};
      for (const int* it = cuts[k]; it != cuts[k + 1]; ++it)
        for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], (&geoms[*it].blo.x)[a]); hi[a] = std::max(hi[a], (&geoms[*it].bhi.x)[a]); }
      for (int a = 0; a < 3; a++) centreHalf(lo[a], hi[a], cc[m][a], hh[m][a]);
      if (cuts[k + 1] - cuts[k] == 1) ref[m] = -(*cuts[k] + 1);
      else { ref[m] = (int)(tree.size() / 8); tree.resize(tree.size() + 8); work.push_back({ref[m], cuts[k], cuts[k + 1]}); }
      m++;
    }
    packNode4(tree.data() + 8 * (size_t)w.node, m, cc, hh, ref);
  }
  return tree;
}

template <typename R>
struct HostScene {
  std::vector<NodeD<R>> nodes;
  std::vector<float4> gbounds;
  int geom_tree = -1;       // word offset of the geom tree appended to gbounds, or -1
  std::vector<Geom<R>> geoms;
  std::vector<PrimD<R>> prims;
  std::vector<LightD<R>> lights;
};

template <typename R>
int flatten(const drt_prim* prims, int n_prims, const drt_light* lights, int n_lights, int n_textures, HostScene<R>& hs) {
  hs.geoms.clear(); hs.prims.clear(); hs.lights.clear();
  hs.prims.assign(n_prims, PrimD<R>());
  // geoms are emitted in the reference's candidate order so that ties of t between
  // coplanar shapes resolve to the same shape (see drt_bvh_order.h)
  const ReferenceBVH bvh = referenceBVH(prims, n_prims);
  const std::vector<int>& order = bvh.order;
  std::vector<int> geom_start(n_prims + 1, 0);   // first geom of the oi-th primitive in reference order
  for (int oi = 0; oi < n_prims; oi++) {
    const int i = order[oi];
    geom_start[oi] = (int)hs.geoms.size();
    const drt_prim& p = prims[i];
    if (p.type < 0 || p.type >= DRT_PRIM_TYPE_COUNT)
      return fail(DRT_ERR_UNSUPPORTED, "primitive " + std::to_string(i) + ": unsupported type " + std::to_string(p.type));
    if ((p.flags & DRT_FLAG_VERTEX_MOTION) && p.type != DRT_PRIM_CYLINDER)
      return fail(DRT_ERR_UNSUPPORTED, "primitive " + std::to_string(i) + ": DRT_FLAG_VERTEX_MOTION is for cylinders only");
    if ((p.flags & DRT_FLAG_TEXTURE) && (p.type == DRT_PRIM_SPHERE || p.type == DRT_PRIM_CYLINDER))
      return fail(DRT_ERR_UNSUPPORTED, "textured Sphere/Cylinder: GeoPrimitive::getUV has no body (geometry.h:36)");
    if ((p.flags & DRT_FLAG_TEXTURE) && (p.tex_frame < 0 || p.tex_frame >= n_textures))
      return fail(DRT_ERR_INVALID, "primitive " + std::to_string(i) + ": tex_frame out of range");
    PrimD<R> q; memset(&q, 0, sizeof(q));
    q.type = p.type; q.name = p.name; q.material = p.material; q.model = p.model; q.flags = p.flags; q.tex = p.tex_frame;
    const float rough = (float)p.roughness;
    q.roughness = rough;
    q.on_A = (float)(1.0 - (0.5 * pow((double)rough, 2)) / (pow((double)rough, 2) + 0.33));   // :896
    q.on_B = (float)((0.45 * pow((double)rough, 2)) / (pow((double)rough, 2) + 0.09));         // :897
    q.schlick_R0 = (float)((pow(p.refr[0] - 1, 2) + pow(p.refr[1], 2)) / (pow(p.refr[0] + 1, 2) + pow(p.refr[1], 2)));
    q.radius = (float)p.radius; q.S = (float)p.S; q.borderwidth = (float)p.borderwidth;
    f3(q.color, p.color); f3(q.bordercolor, p.bordercolor); f3(q.color1, p.color1); f3(q.color2, p.color2);
    const D3 A = V(p.A), B = V(p.B), C = V(p.C), D = V(p.D), E = V(p.E), F = V(p.F), G = V(p.G), H = V(p.H);
    const D3 vel = V(p.velocity);
    q.vel = cv<R>(vel);
    q.length = (float)norm(B - A); q.width = (float)norm(D - A);
    q.center = cv<R>(V(p.center));
    const int gflags = (p.name == DRT_NAME_RECTANGLE) ? GF_NAME_RECTANGLE : 0;
    auto setUVRect = [&](const D3& a, const D3& c, const D3& d) {       // Rectangle::getUV geometry.cpp:751-759
      D3 ad = d - a, dc = c - d;
      q.uvA = cv<R>(a); q.uvD = cv<R>(d); q.uv_ad = cv<R>(ad); q.uv_dc = cv<R>(dc);
      q.uv_den_u = (R)(norm(ad) * norm(dc)); q.uv_den_v = (R)(norm(dc) * norm(ad));
    };
    switch (p.type) {
      case DRT_PRIM_SPHERE: {
        q.pA = cv<R>(V(p.center));
        Geom<R> g; memset(&g, 0, sizeof(g));
        g.type = G_SPHERE; g.owner = i; g.flags = 0; g.p0 = cv<R>(V(p.center)); g.f0 = (float)p.radius; g.vel = cv<R>(vel);
        { const D3 pts[1] = {V(p.center)}; setBounds(g, pts, 1, (double)(float)p.radius, false); }
        hs.geoms.push_back(g);
        break; }
      case DRT_PRIM_CYLINDER: case DRT_PRIM_CHECKER_CYLINDER: {
        D3 c1 = V(p.c1), c2 = V(p.c2);
        D3 axis = normalized(c2 - c1);                                   // geometry.cpp:231
        q.pA = cv<R>(c1); q.pG = cv<R>(axis); q.axis_norm = (float)norm(axis);
        if (p.type == DRT_PRIM_CHECKER_CYLINDER) objMatrix<R>(q.objM, axis, c1);
        if (p.flags & DRT_FLAG_VERTEX_MOTION) { q.n1 = cv<R>(c2); q.n2 = cv<R>(V(p.velocity2)); }   // see PrimD::vel
        Geom<R> g; memset(&g, 0, sizeof(g));
        g.type = G_CYL; g.owner = i; g.p0 = cv<R>(c1); g.p1 = cv<R>(c2); g.p2 = cv<R>(axis); g.f0 = (float)p.radius; g.vel = cv<R>(vel);
        if (p.flags & DRT_FLAG_VERTEX_MOTION) {
          g.flags |= GF_VERTEX_MOTION;
          g.len1 = (R)p.velocity2[0]; g.len2 = (R)p.velocity2[1]; g.pad_ = (R)p.velocity2[2];   // Geom::cylV2
        }
        { const D3 pts[2] = {c1, c2}; setBounds(g, pts, 2, (double)(float)p.radius, false); }
        hs.geoms.push_back(g);
        break; }
      case DRT_PRIM_TRIANGLE: {
        q.n0 = cv<R>(normalized(cross(B - A, C - A)));                   // geometry.cpp:588-594
        q.tA = cv<R>(A); q.tB = cv<R>(B); q.tC = cv<R>(C);
        q.tuv[0] = (float)p.uvA[0]; q.tuv[1] = (float)p.uvA[1]; q.tuv[2] = (float)p.uvB[0];
        q.tuv[3] = (float)p.uvB[1]; q.tuv[4] = (float)p.uvC[0]; q.tuv[5] = (float)p.uvC[1];
        Geom<R> g; memset(&g, 0, sizeof(g));
        g.type = G_TRI; g.owner = i; g.flags = (p.flags & DRT_FLAG_MESH) ? GF_MESH : 0;
        g.p0 = cv<R>(A); g.p1 = cv<R>(B - A); g.p2 = cv<R>(C - A); g.p3 = cv<R>(V(p.mesh_normal)); g.vel = cv<R>(vel);
        { const D3 pts[3] = {A, B, C}; setBounds(g, pts, 3, 0.0, true); }
        hs.geoms.push_back(g);
        break; }
      case DRT_PRIM_RECTANGLE: case DRT_PRIM_CHECKERBOARD: case DRT_PRIM_CHECKERBOARD_HOLE: {
        RectD r = makeRect(A, B, C, D);
        q.n0 = cv<R>(normalized(cross(B - A, C - A)));                   // geometry.cpp:743-749
        setUVRect(A, C, D);
        q.eA = cv<R>(A); q.eB = cv<R>(B); q.eC = cv<R>(C); q.eD = cv<R>(D);
        q.e_den = (R)(8 * norm(V(p.center) - A));                        // :786
        if (p.type == DRT_PRIM_RECTANGLE) {
          hs.geoms.push_back(rectGeom<R>(G_RECT, i, gflags, 1e-4f, r, 0.f, vel));
        } else {
          const bool hole = p.type == DRT_PRIM_CHECKERBOARD_HOLE;
          hs.geoms.push_back(rectGeom<R>(G_CHECKER, i, gflags | (hole ? GF_HAS_HOLE : 0), 1e-3f, r, (float)p.S, vel));
          if (hole) {
            RectD hr = makeRect(V(p.hole[0]), V(p.hole[1]), V(p.hole[2]), V(p.hole[3]));
            hs.geoms.push_back(rectGeom<R>(G_HOLE, i, 0, 1e-4f, hr, 0.f, vel));
            q.rA = cv<R>(r.A); q.re1 = cv<R>(r.e1); q.re2 = cv<R>(r.e2); q.rlen1 = (R)r.len1; q.rlen2 = (R)r.len2;
            q.hA = cv<R>(hr.A); q.hn = cv<R>(hr.nrm); q.he1 = cv<R>(hr.e1); q.he2 = cv<R>(hr.e2);
            q.hlen1 = (R)hr.len1; q.hlen2 = (R)hr.len2;
          }
        }
        break; }
      case DRT_PRIM_RECTPRISM: case DRT_PRIM_RECTPRISM_CYL: case DRT_PRIM_RECTPRISM_HOLES: {
        // the slab-box prisms (geometry.cpp:950-2246): ONE geom, the world AABB of the corners (getBounds overwrites the
        // object-space bounds, :987-988); the class, the holes and the normals live in the shading record
        if (p.type != DRT_PRIM_RECTPRISM) {
          if (p.n_holes < 0 || p.n_holes > DRT_MAX_HOLES)
            return fail(DRT_ERR_UNSUPPORTED, "primitive " + std::to_string(i) + ": more than DRT_MAX_HOLES holes");
          for (int k = 0; k < p.n_holes; k++) {
            const int ht = p.holes[k].type;
            if (!(ht == DRT_PRIM_CYLINDER || (ht == DRT_PRIM_SPHERE && p.type == DRT_PRIM_RECTPRISM_HOLES)))
              return fail(DRT_ERR_UNSUPPORTED, "primitive " + std::to_string(i) + ": hole of a class the reference has no intersectCap / intersectMax for");
          }
        }
        q.n0 = cv<R>(-normalized(cross(F - E, H - E)));                  // normbot   geometry.cpp:1325
        q.n1 = cv<R>(normalized(cross(E - A, D - A)));                   // normright
        q.n2 = cv<R>(normalized(cross(B - A, E - A)));                   // normfront
        q.pA = cv<R>(A); q.pG = cv<R>(G);
        setUVRect(A, C, D);                                              // RectPrism::getUV geometry.cpp:1440-1461
        q.height = (float)norm(E - A);
        { double m[12]; rows3x4(m, normalized(B - A), normalized(D - A), normalized(E - A), V(p.center)); for (int k = 0; k < 12; k++) q.objM[k] = (R)m[k]; }   // :975-984
        q.n_holes = p.type == DRT_PRIM_RECTPRISM ? 0 : p.n_holes;
        for (int k = 0; k < q.n_holes; k++) {
          const drt_hole& hh = p.holes[k];
          HoleD<R>& o = q.holes[k];
          o.type = hh.type == DRT_PRIM_SPHERE ? G_SPHERE : G_CYL;
          o.c1 = cv<R>(V(hh.c1)); o.c2 = cv<R>(V(hh.c2)); o.axis = cv<R>(normalized(V(hh.c2) - V(hh.c1)));
          o.radius = (float)hh.radius; f3(o.color, hh.color);
        }
        Geom<R> g; memset(&g, 0, sizeof(g));
        g.type = G_BOX; g.owner = i; g.vel = cv<R>(vel);
        const D3 cs[8] = {A, B, C, D, E, F, G, H};
        D3 lo = A, hi = A;
        for (const D3& c8 : cs) {
          lo = mk<double>(std::min(lo.x, c8.x), std::min(lo.y, c8.y), std::min(lo.z, c8.z));
          hi = mk<double>(std::max(hi.x, c8.x), std::max(hi.y, c8.y), std::max(hi.z, c8.z));
        }
        g.p0 = cv<R>(lo); g.p1 = cv<R>(hi);
        // never culled by the fp32 filter: a hole can stick out of the box (the hit is then nearer than the box), and
        // RectPrismWithCylinder::intersectShadow reports boxes BEYOND the light as occluders (:1744)
        g.blo = make_float4(-1e30f, -1e30f, -1e30f, 0.f); g.bhi = make_float4(1e30f, 1e30f, 1e30f, 0.f);
        hs.geoms.push_back(g);
        break; }
      case DRT_PRIM_RECTPRISMV2: {
        q.n0 = cv<R>(-normalized(cross(F - E, H - E)));                  // normbot   geometry.cpp:866
        q.n1 = cv<R>(normalized(cross(E - A, D - A)));                   // normright geometry.cpp:867
        q.n2 = cv<R>(normalized(cross(B - A, E - A)));                   // normfront geometry.cpp:868
        q.pA = cv<R>(A); q.pG = cv<R>(G);
        setUVRect(A, C, D);                                              // faces[0]  geometry.cpp:943-948
        const D3 f[6][4] = {{A, B, C, D}, {E, F, G, H}, {A, B, F, E}, {D, A, E, H}, {B, C, G, F}, {C, D, H, G}};   // :796-801
        for (int k = 0; k < 6; k++)
          hs.geoms.push_back(rectGeom<R>(G_RECT, i, 0, 1e-4f, makeRect(f[k][0], f[k][1], f[k][2], f[k][3]), 0.f, vel));
        break; }
    }
    hs.prims[i] = q;
  }
  geom_start[n_prims] = (int)hs.geoms.size();
  // DRT_BLUR_VELOCITY: the filter boxes of moving geoms cover their whole path over one frame (time offsets lie in
  // [0, frame_range), frame_range <= DRT_SWEPT_FRAMES) -- every point of a translated shape, and of a cylinder whose end
  // points move linearly, stays inside the union of its boxes at the two ends of the path -- so re-traces keep the filter
  for (Geom<R>& g : hs.geoms) {
    if (g.type == G_BOX) continue;
    const drt_prim& p = prims[g.owner];
    const D3 v1 = V(p.velocity), v2 = (p.flags & DRT_FLAG_VERTEX_MOTION) ? V(p.velocity2) : v1;
    if (!(dot(v1, v1) > 0) && !(dot(v2, v2) > 0)) continue;
    const double T = DRT_SWEPT_FRAMES;
    for (int a = 0; a < 3; a++) {
      const double d1 = (&v1.x)[a] * T, d2 = (&v2.x)[a] * T;
      const double lo = std::min(0.0, std::min(d1, d2)), hi = std::max(0.0, std::max(d1, d2));
      (&g.blo.x)[a] = std::nextafterf((float)((double)(&g.blo.x)[a] + lo * (1 + 1e-6) - 1e-6), -INFINITY);
      (&g.bhi.x)[a] = std::nextafterf((float)((double)(&g.bhi.x)[a] + hi * (1 + 1e-6) + 1e-6), INFINITY);
    }
  }
  hs.nodes.clear();
  for (const RefNode& rn : bvh.nodes) {
    NodeD<R> nd; memset(&nd, 0, sizeof(nd));
    nd.lo = mk<R>((R)rn.lo[0], (R)rn.lo[1], (R)rn.lo[2]); nd.hi = mk<R>((R)rn.hi[0], (R)rn.hi[1], (R)rn.hi[2]);
    nd.leaf = rn.leaf; nd.left = rn.left; nd.right = rn.right;
    nd.parent = -1;
    if (rn.leaf) { nd.first = geom_start[rn.first]; nd.count = geom_start[rn.first + rn.count] - nd.first; }
    hs.nodes.push_back(nd);
  }
  hs.gbounds = slabTable(hs.geoms);
  const std::vector<float4> tree = geomTree(hs.geoms);
  hs.geom_tree = tree.empty() ? -1 : (int)hs.gbounds.size();
  hs.gbounds.insert(hs.gbounds.end(), tree.begin(), tree.end());
  for (size_t k = 0; k < hs.nodes.size(); k++) {
    NodeD<R>& nd = hs.nodes[k];
    if (nd.leaf) { for (int gi = nd.first; gi < nd.first + nd.count; gi++) hs.geoms[gi].leaf = (int)k; }
    else { hs.nodes[nd.left].parent = (int)k; hs.nodes[nd.right].parent = (int)k; }
  }
  {  // traversal stack bound: depth of the deepest leaf
    std::vector<int> depth(bvh.nodes.size(), 0);
    int maxd = 0;
    for (size_t k = 0; k < bvh.nodes.size(); k++) {   // parents precede children in the node array
      const RefNode& rn = bvh.nodes[k];
      if (!rn.leaf) { depth[rn.left] = depth[k] + 1; depth[rn.right] = depth[k] + 1; }
      maxd = std::max(maxd, depth[k]);
    }
    if (maxd + 2 > DRT_NODE_STACK) return fail(DRT_ERR_UNSUPPORTED, "reference BVH deeper than the traversal stack");
  }
  for (int i = 0; i < n_lights; i++) {
    const drt_light& l = lights[i];
    if (l.type < 0 || l.type > DRT_LIGHT_RECT) return fail(DRT_ERR_UNSUPPORTED, "unknown light type");
    if (l.prim_index >= n_prims) return fail(DRT_ERR_INVALID, "light prim_index out of range");
    LightD<R> q; memset(&q, 0, sizeof(q));
    q.type = l.type; q.prim_index = l.prim_index; q.radius = (float)l.radius;
    D3 bax = V(l.baxis);
    q.use_baxis = dot(bax, bax) > 0 ? 1 : 0;                             // !baxis.isApprox(0)
    f3(q.color, l.color);
    q.center = cv<R>(V(l.center)); q.baxis = cv<R>(bax); q.A = cv<R>(V(l.A)); q.B = cv<R>(V(l.B)); q.D = cv<R>(V(l.D));
    hs.lights.push_back(q);
  }
  return DRT_OK;
}

template <typename R>
struct DevScene {
  DevBuf<Geom<R>> geoms; DevBuf<PrimD<R>> prims; DevBuf<LightD<R>> lights; DevBuf<NodeD<R>> nodes;
  DevBuf<float4> gbounds;
  int geom_tree = -1;       // word offset of the 4-wide tree over the geoms inside gbounds, or -1 (HostScene::geom_tree)
  int n_geoms = 0, n_prims = 0, n_lights = 0, n_nodes = 0;
};

// Scene tables go to the device through one pinned staging buffer and cudaMemcpyAsync on the scene's own stream: the
// per-frame update of one scene handle then neither waits for nor stalls another handle's kernel on the same GPU
// (a synchronous cudaMemcpy from pageable memory did), and the render launches that follow are ordered behind the
// copies by the stream.  The caller synchronises the stream before the stage is filled again.
struct PinnedStage {
  char* base = nullptr; size_t cap = 0, used = 0;
  int reserve(size_t bytes) {
    used = 0;
    if (bytes <= cap) return DRT_OK;
    if (base) cudaFreeHost(base);
    base = nullptr; cap = 0;
    CK(cudaMallocHost((void**)&base, bytes));
    cap = bytes;
    return DRT_OK;
  }
  int push(void* dst, const void* src, size_t bytes, cudaStream_t q) {
    if (!bytes) return DRT_OK;
    if (used + bytes > cap) return fail(DRT_ERR_INVALID, "internal: upload stage too small");
    memcpy(base + used, src, bytes);
    CK(cudaMemcpyAsync(dst, base + used, bytes, cudaMemcpyHostToDevice, q));
    used += (bytes + 255) & ~(size_t)255;
    return DRT_OK;
  }
};

template <typename R>
size_t uploadBytes(const HostScene<R>& hs) {
  auto pad = [](size_t b) { return (b + 255) & ~(size_t)255; };
  return pad(sizeof(float4) * hs.gbounds.size()) + pad(sizeof(NodeD<R>) * hs.nodes.size()) + pad(sizeof(Geom<R>) * hs.geoms.size()) +
         pad(sizeof(PrimD<R>) * hs.prims.size()) + pad(sizeof(LightD<R>) * hs.lights.size());
}

template <typename R>
int upload(const HostScene<R>& hs, DevScene<R>& ds, PinnedStage& stage, cudaStream_t q) {
  CK(ds.gbounds.reserve(sizeof(float4) * std::max<size_t>(3, hs.gbounds.size())));
  CK(ds.nodes.reserve(sizeof(NodeD<R>) * std::max<size_t>(1, hs.nodes.size())));
  CK(ds.geoms.reserve(sizeof(Geom<R>) * std::max<size_t>(1, hs.geoms.size())));
  CK(ds.prims.reserve(sizeof(PrimD<R>) * std::max<size_t>(1, hs.prims.size())));
  CK(ds.lights.reserve(sizeof(LightD<R>) * std::max<size_t>(1, hs.lights.size())));
  ds.geom_tree = hs.geom_tree;
  ds.n_nodes = (int)hs.nodes.size(); ds.n_geoms = (int)hs.geoms.size(); ds.n_prims = (int)hs.prims.size(); ds.n_lights = (int)hs.lights.size();
  { int rc = stage.push(ds.gbounds, hs.gbounds.data(), sizeof(float4) * hs.gbounds.size(), q); if (rc) return rc; }
  { int rc = stage.push(ds.nodes, hs.nodes.data(), sizeof(NodeD<R>) * ds.n_nodes, q); if (rc) return rc; }
  { int rc = stage.push(ds.geoms, hs.geoms.data(), sizeof(Geom<R>) * ds.n_geoms, q); if (rc) return rc; }
  { int rc = stage.push(ds.prims, hs.prims.data(), sizeof(PrimD<R>) * ds.n_prims, q); if (rc) return rc; }
  { int rc = stage.push(ds.lights, hs.lights.data(), sizeof(LightD<R>) * ds.n_lights, q); if (rc) return rc; }
  return DRT_OK;
}

}  // namespace

namespace drt {
static const int kWaveFeats[] = DRT_WAVE_FEATS;
const int* waveFeatList(int* n) { *n = (int)(sizeof(kWaveFeats) / sizeof(int)); return kWaveFeats; }
int waveFeatPick(int need) {
  int best = FT_ALL, best_bits = 99;
  for (int f : kWaveFeats) {
    if ((f & need) != need) continue;
    const int bits = __builtin_popcount((unsigned)f);
    if (bits < best_bits) { best = f; best_bits = bits; }
  }
  return best;
}
}  // namespace drt

struct drt_scene {
  int device = 0;
  std::vector<drt_prim> prims; std::vector<drt_light> lights; int n_textures = 0;
  bool any_glass = false, any_tex = false, any_motion = false, any_box = false, any_spill = false;
  DevScene<double> dd; DevScene<float> df;
  std::vector<cudaArray_t> tex_arrays; std::vector<cudaTextureObject_t> tex_objs;
  DevBuf<cudaTextureObject_t> d_tex; DevBuf<int2> d_texdims;
  cudaStream_t stream = nullptr; cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // scratch, grown on demand
  DevBuf<float4> samples;
  DevBuf<unsigned char> need; DevBuf<float4> bg;
  DevBuf<unsigned char> out_u8; DevBuf<float> out_f32;
  DevBuf<Counts> counts;
  DevBuf<char> pool;
  DevBuf<unsigned long long> batch_counter; DevBuf<int> overflow;
  DevBuf<unsigned long long> steal_counters;                    // drt_render_multi: one counter per row chunk, claimed by every device
  DevBuf<unsigned char> owned;                                  // drt_render_multi: units of the current chunk this device rendered
  cudaEvent_t ev_sync = nullptr;                                // cross-device ordering (drt_render_multi)
  int wave_blocks_f64 = 0, wave_blocks_f32 = 0;
  MeshBuffers mesh; bool has_mesh = false;
  std::vector<drt_prim> mesh_materials;   // the mesh's material table (one entry when all triangles share drt_mesh.material)
  PinnedStage stage;
};

namespace {

template <typename R>
int addMeshMaterial(const drt_prim& m, int n_textures, HostScene<R>& hs) {
  // shading record of the mesh's shared material: flatten it as a stand-alone triangle and keep
  // only the PrimD (its Geom/tree entries are dropped: mesh triangles live in the LBVH)
  HostScene<R> tmp;
  drt_prim p = m;
  p.type = DRT_PRIM_TRIANGLE;
  const double A[3] = {0, 0, 0}, B[3] = {1, 0, 0}, C[3] = {0, 1, 0};
  memcpy(p.A, A, sizeof(A)); memcpy(p.B, B, sizeof(B)); memcpy(p.C, C, sizeof(C));
  int rc = flatten<R>(&p, 1, nullptr, 0, n_textures, tmp);
  if (rc) return rc;
  hs.prims.push_back(tmp.prims[0]);
  return DRT_OK;
}

int flattenAndUpload(drt_scene* s) {
  HostScene<double> hd; HostScene<float> hf;
  int rc = flatten<double>(s->prims.data(), (int)s->prims.size(), s->lights.data(), (int)s->lights.size(), s->n_textures, hd);
  if (rc) return rc;
  rc = flatten<float>(s->prims.data(), (int)s->prims.size(), s->lights.data(), (int)s->lights.size(), s->n_textures, hf);
  if (rc) return rc;
  if (s->has_mesh) {
    for (const drt_prim& m : s->mesh_materials) {
      rc = addMeshMaterial<double>(m, s->n_textures, hd); if (rc) return rc;
      rc = addMeshMaterial<float>(m, s->n_textures, hf); if (rc) return rc;
    }
  }
  CK(cudaStreamSynchronize(s->stream));                     // the stage may still feed the previous update's copies
  rc = s->stage.reserve(uploadBytes(hd) + uploadBytes(hf)); if (rc) return rc;
  rc = upload(hd, s->dd, s->stage, s->stream); if (rc) return rc;
  rc = upload(hf, s->df, s->stage, s->stream); if (rc) return rc;
  s->any_glass = s->any_tex = s->any_motion = s->any_box = s->any_spill = false;
  for (const auto& g : hd.geoms) if (g.flags & GF_SPILL) s->any_spill = true;
  auto scan = [&](const drt_prim& p) {
    if (p.type == DRT_PRIM_RECTPRISM || p.type == DRT_PRIM_RECTPRISM_CYL || p.type == DRT_PRIM_RECTPRISM_HOLES) s->any_box = true;
    if (p.material == DRT_MAT_GLASS) s->any_glass = true;
    if (p.flags & DRT_FLAG_TEXTURE) s->any_tex = true;
    if (p.flags & DRT_FLAG_MOTION) s->any_motion = true;
  };
  for (const drt_prim& p : s->prims) scan(p);
  if (s->has_mesh) for (const drt_prim& m : s->mesh_materials) scan(m);
  return DRT_OK;
}

struct CameraD { D3 eye, X, Y, Z; double mcam[12], new_mcam[12], cloud_mcam[12]; float t, b, r, l; };

void rows3x4(double* out, const D3& r0, const D3& r1, const D3& r2, const D3& eye) {   // (cob * origin) rows, :1011-1021
  const D3 rows[3] = {r0, r1, r2};
  for (int i = 0; i < 3; i++) {
    out[4 * i] = rows[i].x; out[4 * i + 1] = rows[i].y; out[4 * i + 2] = rows[i].z;
    out[4 * i + 3] = (rows[i].x * -eye.x + rows[i].y * -eye.y) + (rows[i].z * -eye.z + 0.0);
  }
}

int makeCamera(const drt_settings& st, CameraD& c) {                     // render_final_project.cpp:989-1027
  D3 eye = V(st.eye), look = V(st.lookingAt), up = V(st.up);
  c.eye = eye;
  c.Z = -normalized(look - eye);
  c.X = normalized(cross(up, c.Z));
  if (!(dot(c.X, c.X) > 0)) return fail(DRT_ERR_SCENE, "Gaze direction can't be equal to up vector!!!");
  c.Y = normalized(cross(c.Z, c.X));
  D3 newX = mk<double>(0, 0, 0), newY = newX;
  if (st.frame >= st.frame_cloud) {
    D3 new_up = mk<double>(-1, 0, 0);
    newX = normalized(cross(new_up, c.Z));
    newY = normalized(cross(c.Z, newX));
  }
  rows3x4(c.mcam, c.X, c.Y, c.Z, eye);
  rows3x4(c.new_mcam, newX, newY, c.Z, eye);
  rows3x4(c.cloud_mcam, c.X, c.Y, -c.Z, eye);                           // renderImageCloud :1253-1259
  c.t = (float)(tan((double)st.fov * M_PI / 360.0) * (double)fabsf(st.near_plane));
  c.b = -c.t;
  c.r = st.aspect * c.t;
  c.l = -c.r;
  return DRT_OK;
}

template <typename R>
void fillParams(Params<R>& P, const drt_scene* s, const DevScene<R>& ds, const drt_settings& st, const CameraD& c, const drt_tile& tile) {
  memset(&P, 0, sizeof(P));
  P.eye = cv<R>(c.eye); P.X = cv<R>(c.X); P.Y = cv<R>(c.Y); P.Z = cv<R>(c.Z);
  for (int i = 0; i < 12; i++) { P.mcam[i] = (R)c.mcam[i]; P.new_mcam[i] = (R)c.new_mcam[i]; P.cloud_mcam[i] = (R)c.cloud_mcam[i]; }
  P.t = c.t; P.b = c.b; P.r = c.r; P.l = c.l;
  P.near_plane = st.near_plane; P.focal_length = st.focal_length; P.aperture = st.aperture;
  P.xRes = st.xRes; P.yRes = st.yRes;
  P.n = (int)sqrt((double)st.antialias_samples);                        // :1046
  P.spp = P.n * P.n;                                                    // :1061
  P.antialias_samples = st.antialias_samples;
  P.brdf_samples = st.brdf_samples; P.blur_samples = st.blur_samples; P.frame_range = st.frame_range; P.max_depth = st.max_depth;
  P.reflect = st.reflect; P.nogloss = st.nogloss; P.perlin_cloud = st.perlin_cloud; P.cloud_only = st.cloud_only;
  P.frame = st.frame; P.frame_prism = st.frame_prism; P.frame_blur = st.frame_blur; P.frame_cloud = st.frame_cloud;
  P.move_per_frame = st.move_per_frame; P.accel_t = st.accel_t; P.refr_air = st.refr_air; P.refr_glass = st.refr_glass;
  P.phong = st.phong; P.seed = st.seed; P.blur_mode = st.blur_mode;
  P.swept_cull = (st.blur_mode == DRT_BLUR_VELOCITY && st.frame_range <= DRT_SWEPT_FRAMES) ? 1 : 0;
  P.sun = cv<R>(normalized(V(st.sundir)));
  f3(P.sun_outer, st.sun_outer); f3(P.sun_inner, st.sun_inner); f3(P.sun_core, st.sun_core);
  f3(P.bluesky, st.bluesky); f3(P.redsky, st.redsky);
  P.saturation = st.saturation; P.clouddist = st.clouddist; P.cloudhoff = st.cloudhoff;
  P.x0 = tile.x0; P.y0 = tile.y0; P.w = tile.width; P.h = tile.height;
  P.geoms = ds.geoms; P.n_geoms = ds.n_geoms; P.gbounds = ds.gbounds; P.geom_tree = ds.geom_tree >= 0 ? ds.gbounds + ds.geom_tree : nullptr; P.nodes = ds.nodes; P.n_nodes = ds.n_nodes; P.prims = ds.prims; P.n_prims = ds.n_prims; P.lights = ds.lights; P.n_lights = ds.n_lights;
  // render_wave serves the records from shared memory when they fit; big scenes (FT_BIG) keep them in global memory
  const size_t recs = sizeof(Geom<R>) * ds.n_geoms + sizeof(PrimD<R>) * ds.n_prims + sizeof(LightD<R>) * ds.n_lights;
  P.smem_recs = (ds.n_geoms <= DRT_SMEM_GEOMS && recs <= DRT_SMEM_RECS) ? (int)recs : 0;
  P.tex = s->d_tex; P.texdims = s->d_texdims;
  if (s->has_mesh) {
    P.mesh_nodes = s->mesh.nodes; P.n_mesh_tris = s->mesh.n_tris; P.mesh_prim = (int)s->prims.size();
    if constexpr (sizeof(R) == 8) P.mesh_tris = s->mesh.tris_f64; else P.mesh_tris = s->mesh.tris_f32;
    P.mesh_mat = s->mesh.mat_ids;
    const drt_prim& m0 = s->mesh_materials[0];
    P.mesh_vel = mk<R>((R)m0.velocity[0], (R)m0.velocity[1], (R)m0.velocity[2]);
  } else P.mesh_vel = mk<R>(R(0), R(0), R(0));
}

int ensureScratch(drt_scene* s, size_t n_samples, size_t n_corners, size_t n_out) {
  CK(s->samples.reserve(n_samples * sizeof(float4)));
  CK(s->need.reserve(n_corners));
  CK(s->bg.reserve(n_corners * sizeof(float4)));
  CK(s->out_u8.reserve(n_out));
  CK(s->out_f32.reserve(n_out * sizeof(float)));
  CK(s->counts.reserve(sizeof(Counts)));
  CK(s->batch_counter.reserve(sizeof(unsigned long long)));
  if (!s->overflow) { CK(s->overflow.reserve(sizeof(int))); CK(cudaMemsetAsync(s->overflow, 0, sizeof(int), s->stream)); }
  return DRT_OK;
}

// Samples held in HBM at once: up to 2^29 float4 = 8 GiB of the B200's 180 (the buffer is sized by what a frame needs), so
// that a 1080p 256 spp or 4K 64 spp frame (530.8 M samples) is ONE launch of the persistent kernel -- every extra launch
// pays one more drain (the last batches finish with few warps busy) and ramp, and on several GPUs one more round of
// barriers.  DRT_CHUNK_LOG2 overrides the bound (smaller GPUs / tests of the multi-chunk path).
long long maxChunkSamples() {
  const char* e = getenv("DRT_CHUNK_LOG2");
  int b = e ? atoi(e) : 29;
  b = std::max(12, std::min(30, b));
  return 1ll << b;
}

// One frame on several devices (drt_render_multi): where the shared claim counters and the gathered frame live.
#define DRT_MULTI_MAX_CHUNKS 1024
struct MultiCtx {
  unsigned long long* counters;   // DRT_MULTI_MAX_CHUNKS counters in the gathering device's memory, zeroed
  unsigned char* gather_u8;       // the gathering device's frame buffer: every device's resolve writes its own pixels there
};

// What one render call launches on one scene handle, split into stages so that drt_render_multi can interleave the
// stages of several handles: plan (allocations, kernel parameters) -> per row chunk: render, background, resolve.
template <typename R>
struct LaunchPlan {
  Params<R> P;
  bool collect = false, perlin = false, cloud_only = false;
  int tile_h = 0, rows_per_chunk = 1, n_chunks = 1;
  long long per_row = 0;
  size_t n_corners = 0;
  int feat = 0, wave_blocks = 0, launches = 0, variant = -1;
};

template <typename R> const DevScene<R>& devScene(const drt_scene* s) { if constexpr (sizeof(R) == 8) return s->dd; else return s->df; }

// Camera samples per tile row, and rows per render launch: as many as fit maxChunkSamples(), at least one (the whole tile
// for cloud_only frames, which render no samples)
void chunking(const drt_settings& st, const drt_tile& tile, long long& per_row, int& rows_per_chunk) {
  const int n = (int)sqrt((double)st.antialias_samples);
  per_row = (long long)tile.width * (n * n);
  rows_per_chunk = st.cloud_only ? tile.height : (int)std::max<long long>(1, std::min<long long>(tile.height, maxChunkSamples() / std::max<long long>(1, per_row)));
}

template <typename R>
int planLaunch(drt_scene* s, const drt_settings& st, const CameraD& cam, const drt_tile& tile, int pool_cap, bool want_f32,
               drt_counters* counters, const MultiCtx* mc, LaunchPlan<R>& lp) {
  const DevScene<R>& ds = devScene<R>(s);
  Params<R>& P = lp.P;
  fillParams<R>(P, s, ds, st, cam, tile);
  lp.collect = counters && counters->collect;
  lp.perlin = st.perlin_cloud && !st.cloud_only; lp.cloud_only = st.cloud_only; lp.tile_h = tile.height;
  chunking(st, tile, lp.per_row, lp.rows_per_chunk);
  lp.n_chunks = (tile.height + lp.rows_per_chunk - 1) / lp.rows_per_chunk;
  lp.n_corners = (size_t)(tile.width + 1) * (tile.height + 1);
  int rc = ensureScratch(s, st.cloud_only ? 1 : (size_t)lp.rows_per_chunk * lp.per_row, lp.n_corners, (size_t)tile.width * tile.height * 3);
  if (rc) return rc;
  P.samples = s->samples; P.need = s->need; P.bg = s->bg; P.out_u8 = s->out_u8; P.out_f32 = want_f32 ? s->out_f32.p : nullptr;
  // claim units: one batch on a single device; whole pixels (at least one batch's worth) when devices share the frame
  P.unit_samples = DRT_CTA_SLOTS;
  if (mc) {
    const int unit_pixels = std::max(1, (DRT_CTA_SLOTS + P.spp - 1) / P.spp);
    P.unit_samples = unit_pixels * P.spp;
    const size_t n_units = ((size_t)lp.rows_per_chunk * lp.per_row + P.unit_samples - 1) / P.unit_samples;
    if (lp.n_chunks > DRT_MULTI_MAX_CHUNKS) return fail(DRT_ERR_UNSUPPORTED, "frame cut into too many row chunks");
    CK(s->owned.reserve(n_units));
    P.steal = 1; P.owned = s->owned; P.out_u8 = mc->gather_u8; P.out_f32 = nullptr;
  }
  P.counts = lp.collect ? s->counts.p : nullptr;
  int& wave_blocks = sizeof(R) == 8 ? s->wave_blocks_f64 : s->wave_blocks_f32;
  if (!wave_blocks) wave_blocks = waveGridBlocks<R>();
  lp.wave_blocks = wave_blocks;
  if (!st.cloud_only && s->pool.reserve(wavePoolBytes<R>(wave_blocks, pool_cap)) != cudaSuccess) {
    cudaGetLastError();
    return fail(DRT_ERR_CUDA, "out of device memory for the ray pools (brdf_samples * max_depth too large)");
  }
  P.pool_raw = s->pool; P.pool_cap = pool_cap; P.batch_counter = s->batch_counter; P.overflow = s->overflow;
  // what this call can reach decides the render_wave instantiation (drt_launch.h WaveFeat)
  int feat = 0;
  if (s->has_mesh) feat |= FT_MESH;
  if (st.blur_samples > 0 && s->any_motion) feat |= (st.blur_mode == DRT_BLUR_VELOCITY) ? FT_VEL : FT_REFBLUR;
  if (s->any_glass && st.reflect) feat |= FT_GLASS;
  if (s->any_tex) feat |= FT_TEX;
  if (ds.n_geoms > DRT_SMEM_GEOMS) feat |= FT_BIG;
  if (s->any_box) feat |= FT_BOX;
  if (s->any_spill) feat |= FT_SPILL;
  if (const char* e = getenv("DRT_WAVE_FEAT")) feat |= atoi(e);      // tuning: force a larger instantiation (255 = generic)
  lp.feat = feat;
  return DRT_OK;
}

// first launches of a call: counters, timing start, background map reset
template <typename R>
int stageBegin(drt_scene* s, LaunchPlan<R>& lp) {
  cudaStream_t q = s->stream;
  if (lp.collect) CK(cudaMemsetAsync(s->counts, 0, sizeof(Counts), q));
  CK(cudaEventRecord(s->ev0, q));
  if (lp.perlin) CK(cudaMemsetAsync(s->need, 0, lp.n_corners, q));
  return DRT_OK;
}
template <typename R>
int stageRender(drt_scene* s, LaunchPlan<R>& lp, int chunk, const MultiCtx* mc) {
  Params<R>& P = lp.P;
  cudaStream_t q = s->stream;
  const int row0 = chunk * lp.rows_per_chunk, rows = std::min(lp.rows_per_chunk, lp.tile_h - row0);
  P.sample_base = (long long)row0 * lp.per_row;
  P.sample_count = (long long)rows * lp.per_row;
  if (mc) {
    P.batch_counter = mc->counters + chunk;
    CK(cudaMemsetAsync(s->owned, 0, ((size_t)P.sample_count + P.unit_samples - 1) / P.unit_samples, q));
  } else CK(cudaMemsetAsync(s->batch_counter, 0, sizeof(unsigned long long), q));
  lp.variant = launchRenderSamples<R>(P, lp.collect, lp.feat, lp.wave_blocks, q); lp.launches++;
  return DRT_OK;
}
// background colours of the pixel corners marked so far.  `shared`: the marks and colours live in the gathering device's
// maps and all devices claim blocks of corners from `corner_counter` there (drt_render_multi).
template <typename R>
int stageCloud(drt_scene* s, LaunchPlan<R>& lp, unsigned char* need, float4* bg, unsigned long long* corner_counter) {
  Params<R> P = lp.P;
  P.need = need; P.bg = bg; P.corner_counter = corner_counter;
  launchCloudCorners<R>(P, s->stream); lp.launches++;
  return DRT_OK;
}
template <typename R>
int stageResolve(drt_scene* s, LaunchPlan<R>& lp, int chunk) {
  const int row0 = chunk * lp.rows_per_chunk, rows = std::min(lp.rows_per_chunk, lp.tile_h - row0);
  launchResolve<R>(lp.P, row0, rows, s->stream); lp.launches++;
  return DRT_OK;
}
template <typename R>
int stageEnd(drt_scene* s, LaunchPlan<R>& lp, drt_counters* counters) {
  CK(cudaEventRecord(s->ev1, s->stream));
  CK(cudaGetLastError());
  if (counters) { counters->kernel_launches = lp.launches; counters->kernel_variant = lp.variant; }
  return DRT_OK;
}

template <typename R>
int launchAll(drt_scene* s, const drt_settings& st, const CameraD& cam, const drt_tile& tile, int pool_cap, bool want_f32,
              drt_counters* counters) {
  LaunchPlan<R> lp;
  int rc = planLaunch<R>(s, st, cam, tile, pool_cap, want_f32, counters, nullptr, lp);
  if (rc) return rc;
  if ((rc = stageBegin(s, lp))) return rc;
  if (st.cloud_only) {
    if ((rc = stageCloud(s, lp, s->need, s->bg, nullptr))) return rc;
    if ((rc = stageResolve(s, lp, 0))) return rc;
  } else {
    for (int c = 0; c < lp.n_chunks; c++) {
      if ((rc = stageRender(s, lp, c, nullptr))) return rc;
      if (lp.perlin && (rc = stageCloud(s, lp, s->need, s->bg, nullptr))) return rc;
      if ((rc = stageResolve(s, lp, c))) return rc;
    }
  }
  return stageEnd(s, lp, counters);
}

// Validation shared by every render entry point; sizes the CTA ray pools and builds the camera.
int planRender(drt_scene* s, const drt_settings* st, const drt_tile* tile, int& pool_cap, CameraD& cam) {
  if (!s || !st || !tile) return fail(DRT_ERR_INVALID, "null argument");
  if (st->xRes < 1 || st->yRes < 1 || tile->width < 1 || tile->height < 1 || tile->x0 < 0 || tile->y0 < 0 ||
      tile->x0 + tile->width > st->xRes || tile->y0 + tile->height > st->yRes)
    return fail(DRT_ERR_INVALID, "tile outside the frame");
  if (st->antialias_samples < 1) return fail(DRT_ERR_INVALID, "antialias_samples < 1");
  if (st->sample_mode != DRT_SAMPLES_KEYED) return fail(DRT_ERR_UNSUPPORTED, "unknown sample_mode");
  if (st->precision != DRT_PRECISION_REFERENCE && st->precision != DRT_PRECISION_FP32) return fail(DRT_ERR_INVALID, "unknown precision");
  if (st->max_depth < 0 || st->max_depth > 32) return fail(DRT_ERR_UNSUPPORTED, "max_depth outside [0,32]");
  // the background of a missed sample is looked up at pixel corner (x + (i+u)/9, y + (j+u)/9) truncated (:1052-1053, Q1); the
  // per-sample record encodes that corner as an offset of 0 or 1, which holds while sqrt(antialias_samples) <= 18
  if (st->perlin_cloud && !st->cloud_only && (int)sqrt((double)st->antialias_samples) > 18)
    return fail(DRT_ERR_UNSUPPORTED, "perlin_cloud with more than 18 x 18 samples per pixel");
  {  // CTA ray-pool bound (render_wave): the pool is a LIFO over the trees of one batch of DRT_CTA_SLOTS samples.  A
     // TRACE pass turns at most DRT_HITS_PER_PASS rays into hits, a hit spawns at most `fan` children (lobes [+1 for
     // glass]), and only the rays on top are traced next, so at most per_pass x (fan - 1) rays are left behind per level.
    const int lobes = std::max(1, st->nogloss ? 1 : st->brdf_samples);
    const int fan = lobes + (s->any_glass ? 1 : 0);
    if (st->brdf_samples < 1 || fan > DRT_MAX_CHILDREN) return fail(DRT_ERR_UNSUPPORTED, "brdf_samples outside [1, 5]");
    if (st->blur_samples < 0 || st->blur_samples > 64) return fail(DRT_ERR_UNSUPPORTED, "blur_samples outside [0, 64]");
    const long long need = (long long)DRT_CTA_SLOTS * std::max(1, st->blur_samples) +
                           (long long)DRT_HITS_PER_PASS * (1 + (long long)st->max_depth * (fan - 1));
    if (need > (1ll << 22)) return fail(DRT_ERR_UNSUPPORTED, "brdf_samples * max_depth needs more than 4 M rays per CTA pool");
    // The pool is handed out in chunks of 32 slots.  On top of the chunks the pending rays fill: a chunk TRACE popped stays
    // "in flight" until SHADE has consumed its hits (each holds at least one of the pass's hits), and a SHADE pass leaves at
    // most one partly filled chunk behind, which lives until the LIFO comes back to it (`partial` allows DRT_WAVE_WARPS x 4
    // of them per tree level).
    const long long live = (need + 31) / 32;
    const long long in_flight = std::min<long long>(live, DRT_CTA_HITS);
    const long long partial = (long long)DRT_WAVE_WARPS * 4 * (st->max_depth + 2);
    pool_cap = (int)(32 * (live + in_flight + partial));
  }
  return makeCamera(*st, cam);
}

int launchFor(drt_scene* s, const drt_settings* st, const CameraD& cam, const drt_tile* tile, int pool_cap, bool want_f32,
              drt_counters* counters) {
  if (st->precision == DRT_PRECISION_FP32) return launchAll<float>(s, *st, cam, *tile, pool_cap, want_f32, counters);
  return launchAll<double>(s, *st, cam, *tile, pool_cap, want_f32, counters);
}

// After the scene's stream has been synchronised: overflow flag, timing, event counters (`hc` already copied back).
int finishRender(drt_scene* s, drt_counters* counters, const Counts& hc, int overflowed) {
  if (overflowed) {   // the kernel dropped rays instead of writing past its pool: the frame is not valid
    CK(cudaMemsetAsync(s->overflow, 0, sizeof(int), s->stream));
    CK(cudaStreamSynchronize(s->stream));
    return fail(DRT_ERR_UNSUPPORTED, "a CTA ray pool overflowed (brdf_samples * max_depth beyond the sized bound)");
  }
  if (counters) {
    float ms = 0; CK(cudaEventElapsedTime(&ms, s->ev0, s->ev1));
    counters->kernel_ms = ms;
    if (counters->collect) {
      counters->samples = hc.samples; counters->rays = hc.rays; counters->shadow_rays = hc.shadow_rays;
      counters->shade_evals = hc.shade_evals; counters->noise_evals = hc.noise_evals; counters->node_tests = hc.node_tests;
      for (int i = 0; i < DRT_PRIM_TYPE_COUNT; i++) counters->prim_tests[i] = 0;
      counters->prim_tests[DRT_PRIM_SPHERE] = hc.geom_tests[G_SPHERE];
      counters->prim_tests[DRT_PRIM_CYLINDER] = hc.geom_tests[G_CYL];
      counters->prim_tests[DRT_PRIM_TRIANGLE] = hc.geom_tests[G_TRI];
      counters->prim_tests[DRT_PRIM_RECTANGLE] = hc.geom_tests[G_RECT] + hc.geom_tests[G_CHECKER];   // rectangle tests incl. prism faces
      counters->prim_tests[DRT_PRIM_RECTPRISM] = hc.geom_tests[G_BOX];                              // all three slab-box classes
    }
  }
  return DRT_OK;
}

// End of a render call on one scene handle (its device current): event counters and overflow flag back, wait for the
// scene's stream, finishRender.
int readBack(drt_scene* s, drt_counters* counters, bool check_overflow) {
  Counts hc; memset(&hc, 0, sizeof(hc));
  if (counters && counters->collect) CK(cudaMemcpyAsync(&hc, s->counts, sizeof(Counts), cudaMemcpyDeviceToHost, s->stream));
  int overflowed = 0;
  if (check_overflow) CK(cudaMemcpyAsync(&overflowed, s->overflow, sizeof(int), cudaMemcpyDeviceToHost, s->stream));
  CK(cudaStreamSynchronize(s->stream));
  return finishRender(s, counters, hc, overflowed);
}

int renderCommon(const drt_scene* cs, const drt_settings* st, const drt_tile* tile, float* out_f32, uint8_t* out_u8,
                 drt_counters* counters, bool copy_back) {
  drt_scene* s = const_cast<drt_scene*>(cs);
  int pool_cap = 0;
  CameraD cam;
  int rc = planRender(s, st, tile, pool_cap, cam);
  if (rc) return rc;
  if (tile->device != s->device) return fail(DRT_ERR_INVALID, "tile.device differs from the scene's device");
  CK(cudaSetDevice(s->device));
  const bool want_f32 = out_f32 != nullptr;
  rc = launchFor(s, st, cam, tile, pool_cap, want_f32, counters);
  if (rc) return rc;
  const size_t n_out = (size_t)tile->width * tile->height * 3;
  if (copy_back) {
    if (out_u8) CK(cudaMemcpyAsync(out_u8, s->out_u8, n_out, cudaMemcpyDeviceToHost, s->stream));
    if (out_f32) CK(cudaMemcpyAsync(out_f32, s->out_f32, n_out * sizeof(float), cudaMemcpyDeviceToHost, s->stream));
  }
  return readBack(s, counters, !st->cloud_only);
}

// The stages of drt_render_multi on all n handles, interleaved chunk by chunk.
template <typename R>
int launchMulti(drt_scene* const* scenes, int n, const drt_settings& st, const CameraD& cam, const drt_tile& tile,
                const int* pool_cap, drt_counters* counters, const MultiCtx& mc) {
  drt_scene* g = scenes[0];                                     // the gathering device
  std::vector<LaunchPlan<R>> plans(n);
  for (int i = 0; i < n; i++) {
    drt_scene* s = scenes[i];
    CK(cudaSetDevice(s->device));
    if (i) CK(cudaStreamWaitEvent(s->stream, g->ev_sync, 0));
    drt_tile t = tile; t.device = s->device;
    int rc = planLaunch<R>(s, st, cam, t, pool_cap[i], false, counters ? &counters[i] : nullptr, &mc, plans[i]);
    if (rc) return rc;
    if ((rc = stageBegin(s, plans[i]))) return rc;
    if (i == 0) CK(cudaEventRecord(g->ev_sync, g->stream));    // ... and the shared background map is reset
  }
  // every stream waits for every other stream's work so far (events only: the host does not block)
  auto barrier = [&]() -> int {
    for (int i = 0; i < n; i++) { CK(cudaSetDevice(scenes[i]->device)); CK(cudaEventRecord(scenes[i]->ev_sync, scenes[i]->stream)); }
    for (int i = 0; i < n; i++) {
      CK(cudaSetDevice(scenes[i]->device));
      for (int k = 0; k < n; k++) if (k != i) CK(cudaStreamWaitEvent(scenes[i]->stream, scenes[k]->ev_sync, 0));
    }
    return DRT_OK;
  };
  const LaunchPlan<R>& lp0 = plans[0];
  for (int c = 0; c < lp0.n_chunks; c++) {
    for (int i = 0; i < n; i++) {
      CK(cudaSetDevice(scenes[i]->device));
      int rc = stageRender(scenes[i], plans[i], c, &mc);
      if (rc) return rc;
    }
    if (lp0.perlin) {
      // The background of a missed sample is a 200-step noise march per pixel CORNER, shared by the four pixels around it:
      // with the frame dealt out in small units every device would evaluate the corners of its own pixels, up to 4x the
      // work.  Instead the devices' corner marks are merged in the gathering device's map, all devices claim blocks of
      // marked corners from one counter, write the colours there, and pull the finished map back before resolving.
      int rc;
      for (int i = 1; i < n; i++) {
        CK(cudaSetDevice(scenes[i]->device));
        launchNeedPush(scenes[i]->need, g->need, lp0.n_corners, scenes[i]->stream); plans[i].launches++;
      }
      CK(cudaSetDevice(g->device));
      CK(cudaMemsetAsync(g->steal_counters + DRT_MULTI_MAX_CHUNKS + c, 0, sizeof(unsigned long long), g->stream));
      if ((rc = barrier())) return rc;
      for (int i = 0; i < n; i++) {
        CK(cudaSetDevice(scenes[i]->device));
        if ((rc = stageCloud(scenes[i], plans[i], g->need, g->bg, g->steal_counters + DRT_MULTI_MAX_CHUNKS + c))) return rc;
      }
      if ((rc = barrier())) return rc;
      for (int i = 1; i < n; i++) {
        CK(cudaSetDevice(scenes[i]->device));
        CK(cudaMemcpyAsync(scenes[i]->need, g->need, lp0.n_corners, cudaMemcpyDeviceToDevice, scenes[i]->stream));
        CK(cudaMemcpyAsync(scenes[i]->bg, g->bg, lp0.n_corners * sizeof(float4), cudaMemcpyDeviceToDevice, scenes[i]->stream));
      }
    }
    for (int i = 0; i < n; i++) {
      CK(cudaSetDevice(scenes[i]->device));
      int rc = stageResolve(scenes[i], plans[i], c);
      if (rc) return rc;
    }
    // the next chunk's marks and colours go into the gathering device's maps: its resolve must have read them first
    if (lp0.perlin && c + 1 < lp0.n_chunks) { int rc = barrier(); if (rc) return rc; }
  }
  for (int i = 0; i < n; i++) {
    CK(cudaSetDevice(scenes[i]->device));
    int rc = stageEnd(scenes[i], plans[i], counters ? &counters[i] : nullptr);
    if (rc) return rc;
  }
  return DRT_OK;
}

// One frame on several devices at once (include/drt.h drt_render_multi).
int renderMulti(drt_scene* const* scenes, int n, const drt_settings* st, const drt_tile* tile, uint8_t* out_u8, drt_counters* counters) {
  if (!scenes || n < 1 || !out_u8) return fail(DRT_ERR_INVALID, "null argument");
  if (n > 64) return fail(DRT_ERR_INVALID, "more than 64 scene handles");
  for (int i = 0; i < n; i++) {
    if (!scenes[i]) return fail(DRT_ERR_INVALID, "null scene handle");
    for (int k = 0; k < i; k++) if (scenes[k] == scenes[i]) return fail(DRT_ERR_INVALID, "the same scene handle twice");
  }
  if (st && st->cloud_only) return fail(DRT_ERR_UNSUPPORTED, "cloud_only frames are rendered on one device (drt_render)");
  int pool_cap[64]; CameraD cam;
  for (int i = 0; i < n; i++) { int rc = planRender(scenes[i], st, tile, pool_cap[i], cam); if (rc) return rc; }
  drt_scene* g = scenes[0];                                     // the gathering device
  // every other device claims from, and resolves into, the gathering device's memory
  for (int i = 1; i < n; i++) {
    if (scenes[i]->device == g->device) continue;
    int can = 0;
    CK(cudaDeviceCanAccessPeer(&can, scenes[i]->device, g->device));
    if (!can) return fail(DRT_ERR_UNSUPPORTED, "no peer access between the devices (cut the frame into tiles and use drt_render)");
    CK(cudaSetDevice(scenes[i]->device));
    const cudaError_t e = cudaDeviceEnablePeerAccess(g->device, 0);
    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) return fail(DRT_ERR_CUDA, std::string("cudaDeviceEnablePeerAccess: ") + cudaGetErrorString(e));
    cudaGetLastError();
  }
  CK(cudaSetDevice(g->device));
  const size_t n_out = (size_t)tile->width * tile->height * 3;
  {
    long long per_row; int rows_per_chunk;
    chunking(*st, *tile, per_row, rows_per_chunk);
    int rc = ensureScratch(g, (size_t)rows_per_chunk * per_row, (size_t)(tile->width + 1) * (tile->height + 1), n_out);
    if (rc) return rc;
  }
  // [0, MAX_CHUNKS): unit counters of the row chunks; [MAX_CHUNKS, 2 MAX_CHUNKS): corner-block counters of the background passes
  CK(g->steal_counters.reserve(sizeof(unsigned long long) * 2 * DRT_MULTI_MAX_CHUNKS));
  CK(cudaMemsetAsync(g->steal_counters, 0, sizeof(unsigned long long) * 2 * DRT_MULTI_MAX_CHUNKS, g->stream));
  for (int i = 0; i < n; i++) if (!scenes[i]->ev_sync) { CK(cudaSetDevice(scenes[i]->device)); CK(cudaEventCreateWithFlags(&scenes[i]->ev_sync, cudaEventDisableTiming)); }
  CK(cudaSetDevice(g->device));
  CK(cudaEventRecord(g->ev_sync, g->stream));                  // counters zeroed, frame buffer allocated
  MultiCtx mc; mc.counters = g->steal_counters; mc.gather_u8 = g->out_u8;
  int rc = st->precision == DRT_PRECISION_FP32 ? launchMulti<float>(scenes, n, *st, cam, *tile, pool_cap, counters, mc)
                                               : launchMulti<double>(scenes, n, *st, cam, *tile, pool_cap, counters, mc);
  if (rc) return rc;
  // the gathering stream waits for everyone's pixels, then one copy to the host
  for (int i = 1; i < n; i++) {
    CK(cudaSetDevice(scenes[i]->device));
    CK(cudaEventRecord(scenes[i]->ev_sync, scenes[i]->stream));
  }
  CK(cudaSetDevice(g->device));
  for (int i = 1; i < n; i++) CK(cudaStreamWaitEvent(g->stream, scenes[i]->ev_sync, 0));
  CK(cudaMemcpyAsync(out_u8, g->out_u8, n_out, cudaMemcpyDeviceToHost, g->stream));
  for (int i = n - 1; i >= 0; i--) {                            // the gathering stream (0) last: it waits for the others
    CK(cudaSetDevice(scenes[i]->device));
    const int rc_i = readBack(scenes[i], counters ? &counters[i] : nullptr, true);
    if (rc_i) rc = rc_i;
  }
  return rc;
}

}  // namespace

extern "C" {

const char* drt_last_error(void) { return g_err.c_str(); }

int drt_device_count(void) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
  return n;
}

void drt_settings_default(drt_settings* s) {                            // render_final_project.cpp:48-138
  memset(s, 0, sizeof(*s));
  s->xRes = 1920; s->yRes = 1080;
  s->eye[0] = -6; s->eye[1] = 0.5; s->eye[2] = 1;
  s->lookingAt[0] = 0.5; s->lookingAt[1] = 0.5; s->lookingAt[2] = 1;
  s->up[1] = 1;
  s->aspect = (float)1920 / (float)1080; s->near_plane = 1; s->fov = 45.0f; s->aperture = 0.2f; s->focal_length = 10;
  s->nogloss = 0; s->refr_air = 1; s->refr_glass = 1.5f; s->max_depth = 10; s->phong = 10;
  s->antialias_samples = 10; s->brdf_samples = 2; s->blur_samples = 2; s->frame_range = 1;
  s->frame_prism = 960; s->frame_cloud = 1952; s->frame_blur = 1600;
  s->move_per_frame = (float)(0.1 / 8); s->accel_t = (float)(80 / pow(360, 3));
  s->sundir[1] = 0.1; s->sundir[2] = -1;
  s->perlin_cloud = 0; s->saturation = 0.2f; s->clouddist = 10; s->cloudhoff = 0.2f;
  const double so[3] = {0.9, 0.3, 0.9}, si[3] = {1.0, 0.7, 0.7}, sc[3] = {1, 1, 1}, bs[3] = {0.3, 0.55, 0.8}, rs[3] = {0.8, 0.8, 0.6};
  memcpy(s->sun_outer, so, sizeof(so)); memcpy(s->sun_inner, si, sizeof(si)); memcpy(s->sun_core, sc, sizeof(sc));
  memcpy(s->bluesky, bs, sizeof(bs)); memcpy(s->redsky, rs, sizeof(rs));
  s->reflect = 1;
}

void drt_prim_default(drt_prim* p) {                                    // geometry.h:39-57
  memset(p, 0, sizeof(*p));
  p->tex_frame = -1;
}

int drt_scene_create(const drt_scene_desc* d, int device, drt_scene** out) {
  if (!d || !out) return fail(DRT_ERR_INVALID, "null argument");
  if (d->abi_version != DRT_ABI_VERSION) return fail(DRT_ERR_INVALID, "ABI version mismatch");
  if ((d->n_prims < 1 || !d->prims) && !d->mesh) return fail(DRT_ERR_SCENE, "No shapes to render!");   // render_final_project.cpp:973-977
  int ndev = drt_device_count();
  if (ndev < 1) return fail(DRT_ERR_NO_DEVICE, "no CUDA device: this library has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(DRT_ERR_INVALID, "device ordinal out of range");
  CK(cudaSetDevice(device));
  drt_scene* s = new drt_scene();
  s->device = device;
  if (d->n_prims > 0) s->prims.assign(d->prims, d->prims + d->n_prims);
  if (d->n_lights > 0) s->lights.assign(d->lights, d->lights + d->n_lights);
  s->n_textures = d->n_textures;
  auto bail = [&](int rc) { drt_scene_destroy(s); return rc; };
  if (cudaStreamCreateWithFlags(&s->stream, cudaStreamNonBlocking) != cudaSuccess || cudaEventCreate(&s->ev0) != cudaSuccess ||
      cudaEventCreate(&s->ev1) != cudaSuccess)
    return bail(fail(DRT_ERR_CUDA, "stream/event creation failed"));
  // textures -> CUDA arrays + texture objects (point sampled, byte/255 as float)
  std::vector<int2> dims;
  for (int i = 0; i < d->n_textures; i++) {
    const drt_texture& t = d->textures[i];
    if (t.width < 1 || t.height < 1 || !t.rgb) return bail(fail(DRT_ERR_INVALID, "bad texture"));
    std::vector<uchar4> rgba((size_t)t.width * t.height);
    for (size_t k = 0; k < rgba.size(); k++) rgba[k] = make_uchar4(t.rgb[3 * k], t.rgb[3 * k + 1], t.rgb[3 * k + 2], 255);
    cudaChannelFormatDesc cd = cudaCreateChannelDesc<uchar4>();
    cudaArray_t arr = nullptr;
    if (cudaMallocArray(&arr, &cd, t.width, t.height) != cudaSuccess) return bail(fail(DRT_ERR_CUDA, "cudaMallocArray failed"));
    s->tex_arrays.push_back(arr);
    if (cudaMemcpy2DToArray(arr, 0, 0, rgba.data(), (size_t)t.width * 4, (size_t)t.width * 4, t.height, cudaMemcpyHostToDevice) != cudaSuccess)
      return bail(fail(DRT_ERR_CUDA, "texture upload failed"));
    cudaResourceDesc rd; memset(&rd, 0, sizeof(rd)); rd.resType = cudaResourceTypeArray; rd.res.array.array = arr;
    cudaTextureDesc td; memset(&td, 0, sizeof(td));
    td.addressMode[0] = td.addressMode[1] = cudaAddressModeClamp; td.filterMode = cudaFilterModePoint;
    td.readMode = cudaReadModeNormalizedFloat; td.normalizedCoords = 0;
    cudaTextureObject_t to = 0;
    if (cudaCreateTextureObject(&to, &rd, &td, nullptr) != cudaSuccess) return bail(fail(DRT_ERR_CUDA, "cudaCreateTextureObject failed"));
    s->tex_objs.push_back(to);
    dims.push_back(make_int2(t.width, t.height));
  }
  if (d->n_textures > 0) {
    if (s->d_tex.reserve(sizeof(cudaTextureObject_t) * d->n_textures) != cudaSuccess ||
        s->d_texdims.reserve(sizeof(int2) * d->n_textures) != cudaSuccess ||
        cudaMemcpy(s->d_tex, s->tex_objs.data(), sizeof(cudaTextureObject_t) * d->n_textures, cudaMemcpyHostToDevice) != cudaSuccess ||
        cudaMemcpy(s->d_texdims, dims.data(), sizeof(int2) * d->n_textures, cudaMemcpyHostToDevice) != cudaSuccess)
      return bail(fail(DRT_ERR_CUDA, "texture table upload failed"));
  }
  if (d->mesh) {
    if (d->mesh->n_materials > 0 && d->mesh->materials) s->mesh_materials.assign(d->mesh->materials, d->mesh->materials + d->mesh->n_materials);
    else s->mesh_materials.assign(1, d->mesh->material);
    for (const drt_prim& m : s->mesh_materials) {
      if ((m.flags & DRT_FLAG_TEXTURE) && !d->mesh->texcoords) return bail(fail(DRT_ERR_INVALID, "textured mesh without texcoords"));
      // DRT_BLUR_VELOCITY moves a mesh rigidly: the traversal shifts the ray instead of a million triangles
      for (int a = 0; a < 3; a++)
        if (m.velocity[a] != s->mesh_materials[0].velocity[a]) return bail(fail(DRT_ERR_UNSUPPORTED, "mesh materials with different velocities (a mesh moves as a whole)"));
      if (m.flags & DRT_FLAG_VERTEX_MOTION) return bail(fail(DRT_ERR_UNSUPPORTED, "DRT_FLAG_VERTEX_MOTION on a mesh material"));
    }
    std::string err;
    int mrc = buildMesh(d->mesh, &s->mesh, err);
    if (mrc) return bail(fail(mrc, err));
    s->has_mesh = true;
  }
  int rc = flattenAndUpload(s);
  if (rc) return bail(rc);
  *out = s;
  return DRT_OK;
}

int drt_scene_update_prims(drt_scene* s, const drt_prim* prims, int32_t n_prims) {
  if (!s || !prims) return fail(DRT_ERR_INVALID, "null argument");
  if (n_prims != (int)s->prims.size()) return fail(DRT_ERR_INVALID, "primitive count changed");
  for (int i = 0; i < n_prims; i++)
    if (prims[i].type != s->prims[i].type) return fail(DRT_ERR_INVALID, "primitive type changed");
  CK(cudaSetDevice(s->device));
  CK(cudaStreamSynchronize(s->stream));
  const std::vector<drt_prim> before = s->prims;
  s->prims.assign(prims, prims + n_prims);
  const int rc = flattenAndUpload(s);
  if (rc) s->prims = before;      // the device copy is untouched when validation fails
  return rc;
}

int drt_scene_update_lights(drt_scene* s, const drt_light* lights, int32_t n_lights) {
  if (!s || (n_lights > 0 && !lights) || n_lights < 0) return fail(DRT_ERR_INVALID, "null argument");
  CK(cudaSetDevice(s->device));
  CK(cudaStreamSynchronize(s->stream));
  const std::vector<drt_light> before = s->lights;
  s->lights.assign(lights, lights + n_lights);
  const int rc = flattenAndUpload(s);
  if (rc) s->lights = before;     // the device copy is untouched when validation fails
  return rc;
}

void drt_scene_destroy(drt_scene* s) {
  if (!s) return;
  cudaSetDevice(s->device);
  if (s->stream) cudaStreamSynchronize(s->stream);
  for (auto t : s->tex_objs) cudaDestroyTextureObject(t);
  for (auto a : s->tex_arrays) cudaFreeArray(a);
  if (s->stage.base) cudaFreeHost(s->stage.base);
  if (s->ev0) cudaEventDestroy(s->ev0);
  if (s->ev1) cudaEventDestroy(s->ev1);
  if (s->ev_sync) cudaEventDestroy(s->ev_sync);
  if (s->stream) cudaStreamDestroy(s->stream);
  delete s;                       // frees the scene's device buffers (DevBuf)
}

// ---- mocap skeletons: parse + device forward kinematics live in drt_skeleton.cu ------------
struct drt_skeleton { drt::Skeleton* impl = nullptr; };

int drt_skeleton_create(const char* asf_text, size_t asf_len, const char* amc_text, size_t amc_len, double scale, int device,
                        drt_skeleton** out) {
  if (!out) return fail(DRT_ERR_INVALID, "null argument");
  drt::Skeleton* impl = nullptr;
  const int rc = skeletonCreate(asf_text, asf_len, amc_text, amc_len, scale, device, &impl);
  if (rc) return fail(rc, skeletonError());
  *out = new drt_skeleton();
  (*out)->impl = impl;
  return DRT_OK;
}

int drt_skeleton_load(const char* asf_path, const char* amc_path, double scale, int device, drt_skeleton** out) {
  if (!asf_path || !amc_path) return fail(DRT_ERR_INVALID, "null argument");
  std::string text[2];
  const char* paths[2] = {asf_path, amc_path};
  for (int i = 0; i < 2; i++) {
    FILE* f = fopen(paths[i], "rb");
    if (!f) return fail(DRT_ERR_INVALID, std::string("cannot open ") + paths[i]);   // the reference throws 1 (skeleton.cpp:575-577)
    char buf[65536]; size_t n;
    while ((n = fread(buf, 1, sizeof(buf), f)) > 0) text[i].append(buf, n);
    fclose(f);
  }
  return drt_skeleton_create(text[0].data(), text[0].size(), text[1].data(), text[1].size(), scale, device, out);
}

int drt_skeleton_info(const drt_skeleton* skel, int32_t* n_cylinders, int32_t* n_frames, float* fk_ms) {
  if (!skel || !skel->impl) return fail(DRT_ERR_INVALID, "null skeleton");
  if (n_cylinders) *n_cylinders = skeletonCylinders(skel->impl);
  if (n_frames) *n_frames = skeletonFrames(skel->impl);
  if (fk_ms) *fk_ms = skeletonFkMs(skel->impl);
  return DRT_OK;
}

int drt_skeleton_bones(const drt_skeleton* skel, int32_t frame0, int32_t n_frames, double* out) {
  if (!skel || !skel->impl) return fail(DRT_ERR_INVALID, "null skeleton");
  const int rc = skeletonReadBones(skel->impl, frame0, n_frames, out);
  return rc ? fail(rc, skeletonError()) : DRT_OK;
}

int drt_scene_pose_skeleton(drt_scene* s, const drt_skeleton* skel, int32_t frame, int32_t first_prim, double drop_y,
                            int32_t set_velocity) {
  if (!s || !skel || !skel->impl) return fail(DRT_ERR_INVALID, "null argument");
  if (frame < 0) return fail(DRT_ERR_INVALID, "frameIndex is illegal");                      // scene.h:111-115
  const int nc = skeletonCylinders(skel->impl), nf = skeletonFrames(skel->impl);
  if (first_prim < 0 || first_prim + nc > (int)s->prims.size()) return fail(DRT_ERR_INVALID, "bone cylinders outside the scene's primitives");
  for (int k = 0; k < nc; k++)
    if (s->prims[first_prim + k].type != DRT_PRIM_CYLINDER) return fail(DRT_ERR_INVALID, "primitive to re-pose is not a cylinder");
  const int f0 = std::min(frame, nf - 1), f1 = std::min(f0 + 1, nf - 1);                     // scene.h:117-121
  const double* tab = skeletonHostTable(skel->impl);
  CK(cudaSetDevice(s->device));
  CK(cudaStreamSynchronize(s->stream));
  const std::vector<drt_prim> before = s->prims;
  for (int k = 0; k < nc; k++) {
    drt_prim& p = s->prims[first_prim + k];
    const double* a = tab + ((size_t)f0 * nc + k) * 6;
    const double* b = tab + ((size_t)f1 * nc + k) * 6;
    double c1[3], c2[3], n1[3], n2[3];
    for (int i = 0; i < 3; i++) { c1[i] = a[i]; c2[i] = a[3 + i]; n1[i] = b[i]; n2[i] = b[3 + i]; }
    if (drop_y != 0.0) { c1[1] -= drop_y; c2[1] -= drop_y; n1[1] -= drop_y; n2[1] -= drop_y; }   // scene.h:646-650
    for (int i = 0; i < 3; i++) {
      p.c1[i] = c1[i]; p.c2[i] = c2[i];
      p.center[i] = (c1[i] + c2[i]) / 2;
      if (set_velocity == 2) { p.velocity[i] = n1[i] - c1[i]; p.velocity2[i] = n2[i] - c2[i]; }   // each end point to its own next pose
      else { p.velocity[i] = set_velocity ? ((n1[i] + n2[i]) - (c1[i] + c2[i])) / 2 : 0.0; p.velocity2[i] = 0.0; }
    }
    if (set_velocity) p.flags |= DRT_FLAG_MOTION;
    if (set_velocity == 2) p.flags |= DRT_FLAG_VERTEX_MOTION; else p.flags &= ~DRT_FLAG_VERTEX_MOTION;
  }
  const int rc = flattenAndUpload(s);
  if (rc) s->prims = before;
  return rc;
}

int drt_debug_skeleton_parse(const char* asf_text, size_t asf_len, const char* amc_text, size_t amc_len, double scale,
                             int32_t* n_bones, int32_t* n_frames, int32_t* parents, int32_t* dofs, int32_t cap) {
  const int rc = skeletonParseInfo(asf_text, asf_len, amc_text, amc_len, scale, n_bones, n_frames, parents, dofs, cap);
  return rc ? fail(rc, skeletonError()) : DRT_OK;
}

void drt_skeleton_destroy(drt_skeleton* skel) {
  if (!skel) return;
  skeletonDestroy(skel->impl);
  delete skel;
}

int drt_render(const drt_scene* scene, const drt_settings* settings, const drt_tile* tile, uint8_t* out_rgb, drt_counters* counters) {
  if (!out_rgb) return fail(DRT_ERR_INVALID, "out_rgb is null");
  return renderCommon(scene, settings, tile, nullptr, out_rgb, counters, true);
}

int drt_render_float(const drt_scene* scene, const drt_settings* settings, const drt_tile* tile, float* out_rgb_f32,
                     uint8_t* out_rgb, drt_counters* counters) {
  if (!out_rgb_f32 && !out_rgb) return fail(DRT_ERR_INVALID, "both outputs are null");
  return renderCommon(scene, settings, tile, out_rgb_f32, out_rgb, counters, true);
}

int drt_render_device(const drt_scene* scene, const drt_settings* settings, const drt_tile* tile, drt_counters* counters) {
  return renderCommon(scene, settings, tile, nullptr, nullptr, counters, false);
}

int drt_render_multi(drt_scene* const* scenes, int32_t n_scenes, const drt_settings* settings, const drt_tile* tile, uint8_t* out_rgb,
                     drt_counters* counters) {
  return renderMulti(scenes, n_scenes, settings, tile, out_rgb, counters);
}

int drt_write_ppm(const char* filename, int32_t width, int32_t height, const uint8_t* rgb) {   // helpers.h:174-195
  if (!filename || !rgb || width < 1 || height < 1) return fail(DRT_ERR_INVALID, "bad argument");
  FILE* fp = fopen(filename, "wb");
  if (!fp) return fail(DRT_ERR_INVALID, std::string("Could not open file \"") + filename + "\" for writing.");
  fprintf(fp, "P6\n%d %d\n255\n", width, height);
  fwrite(rgb, 1, (size_t)width * height * 3, fp);
  fclose(fp);
  return DRT_OK;
}

// struct sizes, for the ctypes mirror to verify its layout against
void drt_abi_sizes(int32_t* out6) {
  out6[0] = (int32_t)sizeof(drt_prim); out6[1] = (int32_t)sizeof(drt_light); out6[2] = (int32_t)sizeof(drt_scene_desc);
  out6[3] = (int32_t)sizeof(drt_settings); out6[4] = (int32_t)sizeof(drt_tile); out6[5] = (int32_t)sizeof(drt_counters);
}

// The candidate order the scene flattener derives from its replay of the reference's BVH build
// (drt_bvh_order.h): primitive indices, `cap` entries at most; returns the count.  Host only.
int drt_debug_candidate_order(const drt_prim* prims, int32_t n_prims, int32_t* out, int32_t cap) {
  if (!prims || n_prims < 1 || !out) return 0;
  int n = 0;
  for (int i : referenceBVH(prims, n_prims).order) { if (n < cap) out[n] = i; n++; }
  return n;
}

// Evaluates the device sample stream on the HOST copy of the same inline
// functions (drt_rng.cuh) so tests can compare it with the oracle's copy.
float drt_debug_rng(uint32_t seed, uint32_t pixel, uint32_t sample, uint32_t child, uint32_t dim) {
  uint32_t pk = rng_key_pixel(seed, pixel);
  uint32_t sk = rng_key_sample(pk, sample);
  return rng_u01(rng_key_child(sk, child), dim);
}

// Step i of the keyed lens-sample shuffle of a pixel (j = round(u*i), helpers.h:274), and the lens point that ends up at
// position `sample` of `n_lens`, from the same inline functions the kernels use.
int drt_debug_shuffle_j(uint32_t seed, uint32_t pixel, int32_t i) { return rng_shuffle_j(rng_key_pixel(seed, pixel), i); }
int drt_debug_lens_index(uint32_t seed, uint32_t pixel, int32_t sample, int32_t n_lens) {
  return lensIndexScan(rng_key_pixel(seed, pixel), sample, n_lens);
}

}  // extern "C"
