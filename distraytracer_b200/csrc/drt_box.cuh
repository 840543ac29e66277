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
