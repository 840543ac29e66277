// Device-built LBVH over an indexed triangle mesh (BASELINE config 5: ~1 M triangles).
//
// Replaces, for meshes, the reference's generateBVH (helpers.h:381-472), whose SAH sweep copies
// both index vectors for every candidate split -- O(n^2) per node, infeasible beyond ~10^4
// primitives (SURVEY.md 8a a8).  Build = Morton codes of triangle centroids (63 bit, cubic cells), radix sort
// (cub::DeviceRadixSort -- the one library call, build-time plumbing, never per ray), Karras
// 2012 binary radix tree, bottom-up refit with one atomic counter per internal node, then a
// collapse into 4-WIDE nodes: every binary node at even depth becomes a traversal node whose children are its
// grandchildren (or a child that is a leaf), so a ray takes half as many dependent node fetches.
//
// Traversal node: the 4-wide node of drt_box.cuh, so the LBVH and the slab filter share the packed FFMA2 test.
#pragma once
#include <cuda_runtime.h>
#include <cub/device/device_radix_sort.cuh>
#include <stdint.h>

#include "drt_box.cuh"
#include "drt_device.cuh"

namespace drt {

__device__ __forceinline__ uint64_t expandBits21(uint64_t v) {   // 21 bits -> every third bit
  v &= 0x1fffffull;
  v = (v | (v << 32)) & 0x001f00000000ffffull;
  v = (v | (v << 16)) & 0x001f0000ff0000ffull;
  v = (v | (v << 8)) & 0x100f00f00f00f00full;
  v = (v | (v << 4)) & 0x10c30c30c30c30c3ull;
  v = (v | (v << 2)) & 0x1249249249249249ull;
  return v;
}

// per triangle: fp32 bounds + Morton code of the centroid.  The pad is the curved rule of padBounds (drt_box.cuh),
// 1e-3 + 1e-5 |coordinate|, in float: padBounds says why mesh triangles do not take the planar pad.
// The code cells are CUBES (`sinv` is one scale for all three axes: 1 / the largest extent) of 2^-21 of that extent.
// With a scale per axis a flat mesh -- the terrain of config 5 is 12 x 2 x 12 -- spends every third level of the tree on a
// split by height, whose two halves overlap almost everywhere in x and z (measured on that terrain: 32 % more node visits
// per ray); 10 bits per axis also left both triangles of most grid quads in one cell, split by index instead of position.
__global__ void lbvh_tri_setup(int n, const float* __restrict__ verts, const int* __restrict__ idx, float3 slo, float sinv,
                               float4* __restrict__ tlo, float4* __restrict__ thi, uint64_t* __restrict__ codes,
                               int* __restrict__ ids) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  float lo[3] = {3e38f, 3e38f, 3e38f}, hi[3] = {-3e38f, -3e38f, -3e38f}, c[3] = {0, 0, 0};
  for (int k = 0; k < 3; k++) {
    const int v = idx[3 * i + k];
    for (int a = 0; a < 3; a++) {
      const float x = verts[3 * v + a];
      lo[a] = fminf(lo[a], x); hi[a] = fmaxf(hi[a], x); c[a] += x * (1.0f / 3.0f);
    }
  }
  for (int a = 0; a < 3; a++) {
    const float pad = 1e-3f + 1e-5f * fmaxf(fabsf(lo[a]), fabsf(hi[a]));
    lo[a] -= pad; hi[a] += pad;
  }
  tlo[i] = make_float4(lo[0], lo[1], lo[2], 0.f);
  thi[i] = make_float4(hi[0], hi[1], hi[2], 0.f);
  const double fx = fmin(fmax(((double)c[0] - (double)slo.x) * (double)sinv * 2097152.0, 0.0), 2097151.0);
  const double fy = fmin(fmax(((double)c[1] - (double)slo.y) * (double)sinv * 2097152.0, 0.0), 2097151.0);
  const double fz = fmin(fmax(((double)c[2] - (double)slo.z) * (double)sinv * 2097152.0, 0.0), 2097151.0);
  codes[i] = (expandBits21((uint64_t)fx) << 2) | (expandBits21((uint64_t)fy) << 1) | expandBits21((uint64_t)fz);
  ids[i] = i;
}

// Karras: common-prefix length of keys i and j (ties broken by index)
__device__ __forceinline__ int lbvh_delta(const uint64_t* __restrict__ codes, int n, int i, int j) {
  if (j < 0 || j >= n) return -1;
  const uint64_t a = codes[i], b = codes[j];
  if (a == b) return 64 + __clz((uint32_t)i ^ (uint32_t)j);
  return __clzll((long long)(a ^ b));
}

// one thread per internal node i in [0, n-1): children + parent links
__global__ void lbvh_karras(int n, const uint64_t* __restrict__ codes, int* __restrict__ left, int* __restrict__ right,
                            int* __restrict__ parent_internal, int* __restrict__ parent_leaf) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n - 1) return;
  const int d = (lbvh_delta(codes, n, i, i + 1) - lbvh_delta(codes, n, i, i - 1)) >= 0 ? 1 : -1;
  const int dmin = lbvh_delta(codes, n, i, i - d);
  int lmax = 2;
  while (lbvh_delta(codes, n, i, i + lmax * d) > dmin) lmax *= 2;
  int l = 0;
  for (int t = lmax / 2; t >= 1; t /= 2)
    if (lbvh_delta(codes, n, i, i + (l + t) * d) > dmin) l += t;
  const int j = i + l * d;
  const int dnode = lbvh_delta(codes, n, i, j);
  int s = 0;
  int t = l;
  do {
    t = (t + 1) >> 1;
    if (lbvh_delta(codes, n, i, i + (s + t) * d) > dnode) s += t;
  } while (t > 1);
  const int gamma = i + s * d + min(d, 0);
  const int lo = min(i, j), hi = max(i, j);
  // child encoding: >= 0 internal node, < 0 leaf (sorted position = -c - 1)
  const int lc = (lo == gamma) ? -(gamma + 1) : gamma;
  const int rc = (hi == gamma + 1) ? -(gamma + 2) : gamma + 1;
  left[i] = lc; right[i] = rc;
  if (lc >= 0) parent_internal[lc] = i; else parent_leaf[gamma] = i;
  if (rc >= 0) parent_internal[rc] = i; else parent_leaf[gamma + 1] = i;
}

// one thread per leaf: climb, the second arrival at a node merges its children's boxes
__global__ void lbvh_refit(int n, const int* __restrict__ ids, const float4* __restrict__ tlo, const float4* __restrict__ thi,
                           const int* __restrict__ left, const int* __restrict__ right, const int* __restrict__ parent_internal,
                           const int* __restrict__ parent_leaf, float4* nlo, float4* nhi, int* __restrict__ visits) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  int node = parent_leaf[i];
  while (node >= 0) {
    if (atomicAdd(&visits[node], 1) == 0) return;          // first arrival: the sibling subtree is not done yet
    __threadfence();
    float4 lo[2], hi[2];
    const int ch[2] = {left[node], right[node]};
    for (int k = 0; k < 2; k++) {
      if (ch[k] >= 0) { lo[k] = __ldcg(&nlo[ch[k]]); hi[k] = __ldcg(&nhi[ch[k]]); }   // L2 reads: written by another SM
      else { const int t = ids[-ch[k] - 1]; lo[k] = tlo[t]; hi[k] = thi[t]; }
    }
    nlo[node] = make_float4(fminf(lo[0].x, lo[1].x), fminf(lo[0].y, lo[1].y), fminf(lo[0].z, lo[1].z), 0.f);
    nhi[node] = make_float4(fmaxf(hi[0].x, hi[1].x), fmaxf(hi[0].y, hi[1].y), fmaxf(hi[0].z, hi[1].z), 0.f);
    __threadfence();
    node = (node == 0) ? -1 : parent_internal[node];
  }
}

// collapse into the 128-byte 4-wide traversal nodes: one thread per binary internal node, even depths only
__global__ void lbvh_pack4(int n, const int* __restrict__ ids, const float4* __restrict__ tlo, const float4* __restrict__ thi,
                           const int* __restrict__ left, const int* __restrict__ right, const int* __restrict__ parent_internal,
                           const float4* __restrict__ nlo, const float4* __restrict__ nhi, float4* __restrict__ nodes) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n - 1) return;
  int depth = 0;
  for (int k = i; k != 0; k = parent_internal[k]) depth++;             // node 0 is the root of Karras' tree
  if (depth & 1) return;
  int c[4], m = 0;
  const int side[2] = {left[i], right[i]};
  for (int k = 0; k < 2; k++) {
    if (side[k] < 0) c[m++] = side[k];
    else { c[m++] = left[side[k]]; c[m++] = right[side[k]]; }
  }
  float cc[4][3], hh[4][3]; int ref[4];
  for (int k = 0; k < 4; k++) {
    if (k >= m) continue;
    float4 lo, hi;
    if (c[k] >= 0) { lo = nlo[c[k]]; hi = nhi[c[k]]; ref[k] = c[k]; }
    else { const int t = ids[-c[k] - 1]; lo = tlo[t]; hi = thi[t]; ref[k] = -(t + 1); }
    centreHalf(lo.x, hi.x, cc[k][0], hh[k][0]);
    centreHalf(lo.y, hi.y, cc[k][1], hh[k][1]);
    centreHalf(lo.z, hi.z, cc[k][2], hh[k][2]);
  }
  packNode4(nodes + 8 * (size_t)i, m, cc, hh, ref);
}

// exact-test records: the three vertices in the vector scalar R (the reference recomputes B-A,
// C-A per call, geometry.cpp:516-517), plus per-vertex UVs
template <typename R>
__global__ void lbvh_tri_records(int n, const float* __restrict__ verts, const int* __restrict__ idx, const float* __restrict__ tc,
                                 MeshTri<R>* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  MeshTri<R> t;
  Vec<R>* P[3] = {&t.A, &t.B, &t.C};
  for (int k = 0; k < 3; k++) {
    const int v = idx[3 * i + k];
    *P[k] = mk<R>((R)verts[3 * v], (R)verts[3 * v + 1], (R)verts[3 * v + 2]);
    t.uv[2 * k] = tc ? tc[2 * v] : 0.f; t.uv[2 * k + 1] = tc ? tc[2 * v + 1] : 0.f;
  }
  out[i] = t;
}

}  // namespace drt
