// The fp32 box format of the slab filter and of the 4-wide trees, and its one writer.  The kernels read it in
// drt_kernels.cuh (slabPair, slabGroupMayHit, bvh4Visit); the host (drt_api.cu, drt_mesh.cu) and the LBVH build
// (drt_lbvh.cuh) write it through the functions below.
//
// A box is stored as CENTRE / HALF-EXTENT, rounded so that [c - h, c + h] contains [lo, hi] (centreHalf).
// PAIR RECORD, 48 bytes, two boxes 0 and 1:  {cx0 cx1 cy0 cy1} {cz0 cz1 hx0 hx1} {hy0 hy1 hz0 hz1}
// 4-WIDE NODE, 128 bytes (float4 x 8, one cache line):
//   [0..2] pair record of children 0, 1
//   [3..5] pair record of children 2, 3
//   [6]    child references as int bits: >= 0 node index; < 0 leaf, item = -ref - 1
//   [7]    padding
// An EMPTY slot has half-extent kEmptyHalf and, in a node, the reference kEmptyRef: it never passes, not even for an
// axis-parallel ray whose slab terms are NaN.
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <string.h>

namespace drt {

constexpr float kEmptyHalf = -1e30f;
constexpr int kEmptyRef = (int)0x80000000;

// ---- padding: exact bounds -> fp32 filter bounds of the analytic geoms (setBounds in drt_api.cu) ---------------
// The filter must pass every geom whose exact test accepts a hit.  It is handed an fp32 box [flo, fhi] and, per ray,
// keeps the slack of slabRay (drt_kernels.cuh): t_near <= t_far * 1.0001 + 1e-4 + err and t_far >= -err, err covering
// the rounding of the slab terms.  So a hit at parameter t passes when a point of the ray at a parameter within a
// relative ~1e-4 of t lies in the box.  Below: u = 2^-24; m = max(|lo|, |hi|) of the axis; D = the distance from the
// ray's origin to the hit's plane.
//
// CURVED (sphere, cylinder, and an unbounded or GF_SPILL rectangle): pad 1e-3 + 1e-5 m.  The quadratics are formed in
// float, so a grazing hit can lie ~sqrt(u) r outside the true surface.  A GF_SPILL rectangle's accepted parallelogram
// can be arbitrarily thin, which magnifies its rounding by 1 / sin of the angle between its edges.  (Slab-box prisms
// are never culled.)
//
// PLANAR (rectangle / checkerboard of orthogonal edges, analytic triangle): pad kPlanarRel m plus a floor,
// kPlanarAbs64 for R = double and kPlanarAbs32 for R = float.  The accepted regions:
//  - Triangle, R = double (G_TRI in geomIntersect / geomShadow): u, v and t are the exact Cramer quotients times one
//    common factor (the fp32 det and its fp32 reciprocal), each with one more fp32 rounding.  So the exact
//    intersection P(t*) of the ray with the plane has barycentrics u*, v* >= 0, u* + v* <= 1 + 4u, and t* lies within
//    3u t of the accepted t.  P(t*) is in the triangle grown by 4u of its edges (<= 8u m per axis), and t* is inside
//    the slack.  This holds at any D.
//  - Rectangle, R = double (rectHit): t is the exact plane quotient with two fp32 roundings, and the in-plane
//    coordinates are taken at the accepted point P' = start + t ray, not at the exact intersection.  P' is within
//    u len1 e1 + u len2 e2 (<= 4u m per axis) of the rectangle in the plane, and within 2u D of the plane along its
//    normal n.  In an axis a with n_a != 0 the off-plane part moves P' out of the box by up to 2u D |n_a|.  The slack
//    covers that as a t error of 2u D |n_a| / |ray_a|, i.e. unless the ray is within ~1e-3 of perpendicular to axis a.
//    Example: n = (1, 1, 0) / sqrt 2, a ray along -y grazing the rectangle's edge of largest x, hit at distance D:
//    x is constant along the ray, and the accepted point may lie u D beyond that edge.
//    The floor holds this part while 2u D <= kPlanarAbs64: D up to ~80.
//  - R = float: vertices and corners are stored in float (u m), and every product and sum of the tests rounds in
//    float.  The backward error of either test is a few u of |start|, |P| and |A|, below ~45u D, with the same
//    axis-perpendicular exception.  kPlanarAbs32 holds it for D up to ~35, and kPlanarRel m (17u m) the parts in the
//    geom's own coordinates.
// ASSUMPTION: ray origins lie within those distances of the planar geoms they hit (cameras within ~35 of the scene in
// float, ~80 in double).  Beyond them a ray within ~1e-3 of perpendicular to an axis that hits within u D of a planar
// geom's edge may be culled.  The old pad 1e-3 + 1e-5 m made the same assumption at 10 (float) and 100 (double)
// times these distances.
// A moving geom's swept box (flatten, DRT_BLUR_VELOCITY) adds the translation to this box with its own relative and
// absolute margin.  The exact tests translate the vertices by the same vector in R, which moves the accepted region
// with them (in float within u of the translated coordinate, inside that margin).
// The analytic candidates are tested in geom order (the geom tree of big scenes breaks ties of t by geom index), so
// these boxes decide which exact tests run, never which hit wins.  Mesh triangles keep the LBVH's own pad
// (lbvh_tri_setup in drt_lbvh.cuh): the mesh walk is nearest-box-first and keeps the first of two hits with equal t,
// so on an edge shared by two triangles the boxes decide which one is shaded, and tighter boxes change pixels.
// lo is rounded down and hi up (nearest, then one ulp outward), so the fp32 box holds the padded double box.
constexpr double kPlanarRel = 1e-6, kPlanarAbs64 = 1e-5, kPlanarAbs32 = 1e-4;
__host__ __device__ inline void padBounds(const double lo, const double hi, const bool planar, const bool single,
                                          float& flo, float& fhi) {
  const double m = fmax(fabs(lo), fabs(hi));
  const double pad = planar ? kPlanarRel * m + (single ? kPlanarAbs32 : kPlanarAbs64) : 1e-3 + 1e-5 * m;
  flo = nextafterf((float)(lo - pad), -INFINITY);
  fhi = nextafterf((float)(hi + pad), INFINITY);
}

// Centre / half-extent of [lo, hi].  The half-extent is rounded up to float, then widened by one more ulp.  The round-up
// is written as a cast to nearest plus one ulp when that fell below `hd`: for every hd >= 0 that is the smallest float
// >= hd, which is what __double2float_ru returns, overflow to infinity included (a value above FLT_MAX rounds to FLT_MAX
// or infinity; FLT_MAX < hd then steps to infinity).  So host and device give the same bits.
__host__ __device__ inline void centreHalf(const float lo, const float hi, float& c, float& h) {
  c = (float)(0.5 * ((double)lo + (double)hi));
  const double hd = fmax((double)hi - (double)c, (double)c - (double)lo);
  h = (float)hd;
  if ((double)h < hd) h = nextafterf(h, INFINITY);
  h = nextafterf(h, INFINITY);
}

// One pair record at `rec` from the centres / half-extents of boxes 0 and 1.
__host__ __device__ inline void packPair(float4* rec, const float c0[3], const float h0[3], const float c1[3], const float h1[3]) {
  rec[0] = make_float4(c0[0], c1[0], c0[1], c1[1]);
  rec[1] = make_float4(c0[2], c1[2], h0[0], h1[0]);
  rec[2] = make_float4(h0[1], h1[1], h0[2], h1[2]);
}

// One 4-wide node at `nd` from its first m children (centre / half-extent, reference); slots m..3 are made empty.
__host__ __device__ inline void packNode4(float4* nd, const int m, float c[4][3], float h[4][3], int ref[4]) {
  for (int k = 0; k < 4; k++) {
    if (k < m) continue;
    ref[k] = kEmptyRef;
    for (int a = 0; a < 3; a++) { c[k][a] = 0.f; h[k][a] = kEmptyHalf; }
  }
  packPair(nd, c[0], h[0], c[1], h[1]);
  packPair(nd + 3, c[2], h[2], c[3], h[3]);
  float r[4];
  memcpy(r, ref, sizeof(r));
  nd[6] = make_float4(r[0], r[1], r[2], r[3]);
  nd[7] = make_float4(0.f, 0.f, 0.f, 0.f);
}

}  // namespace drt
