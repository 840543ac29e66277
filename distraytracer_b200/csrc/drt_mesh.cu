// Device LBVH build for drt_mesh (see drt_lbvh.cuh for the kernels).
#include <algorithm>
#include <cmath>
#include <vector>

#include "drt_box.cuh"
#include "drt_lbvh.cuh"
#include "drt_mesh.h"

namespace drt {

#define MCK(call)                                                                           \
  do {                                                                                      \
    cudaError_t e_ = (call);                                                                \
    if (e_ != cudaSuccess) { err = std::string(#call) + " failed: " + cudaGetErrorString(e_); return DRT_ERR_CUDA; } \
  } while (0)

int buildMesh(const drt_mesh* mesh, MeshBuffers* out, std::string& err) {
  const long long nv = mesh->n_vertices, nt = mesh->n_triangles;
  if (nv < 3 || nt < 1 || !mesh->vertices || !mesh->indices) { err = "empty mesh"; return DRT_ERR_INVALID; }
  if (nt > (1ll << 30)) { err = "mesh too large"; return DRT_ERR_UNSUPPORTED; }
  for (long long i = 0; i < 3 * nt; i++)
    if (mesh->indices[i] < 0 || mesh->indices[i] >= nv) { err = "mesh index out of range"; return DRT_ERR_INVALID; }
  if (mesh->n_materials < 0 || mesh->n_materials > 65535) { err = "mesh material table larger than 65535 entries"; return DRT_ERR_UNSUPPORTED; }
  if (mesh->n_materials > 0) {
    if (!mesh->materials || !mesh->material_ids) { err = "mesh material table without ids"; return DRT_ERR_INVALID; }
    for (long long t = 0; t < nt; t++)
      if (mesh->material_ids[t] < 0 || mesh->material_ids[t] >= mesh->n_materials) { err = "mesh material id out of range"; return DRT_ERR_INVALID; }
  }
  const int n = (int)nt;
  // scene bounds of the centroids' support (host: one pass over the vertices)
  float lo[3] = {3e38f, 3e38f, 3e38f}, hi[3] = {-3e38f, -3e38f, -3e38f};
  for (long long v = 0; v < nv; v++)
    for (int a = 0; a < 3; a++) { lo[a] = std::min(lo[a], mesh->vertices[3 * v + a]); hi[a] = std::max(hi[a], mesh->vertices[3 * v + a]); }
  float3 slo = make_float3(lo[0], lo[1], lo[2]);
  const float sinv = 1.0f / std::max(std::max(hi[0] - lo[0], hi[1] - lo[1]), std::max(hi[2] - lo[2], 1e-20f));   // cubic Morton cells

  DevBuf<float> d_verts, d_tc; DevBuf<int> d_idx;
  DevBuf<float4> tlo, thi, nlo, nhi;
  DevBuf<uint64_t> codes, codes2; DevBuf<int> ids, ids2;
  DevBuf<int> left, right, pin, pleaf, visits;
  DevBuf<char> tmp; size_t tmp_bytes = 0;
  MeshBuffers mb;
  mb.n_tris = n;
  const int B = 256, G = (n + B - 1) / B;
  MCK(d_verts.reserve(sizeof(float) * 3 * nv));
  MCK(d_idx.reserve(sizeof(int) * 3 * nt));
  MCK(cudaMemcpy(d_verts, mesh->vertices, sizeof(float) * 3 * nv, cudaMemcpyHostToDevice));
  MCK(cudaMemcpy(d_idx, mesh->indices, sizeof(int) * 3 * nt, cudaMemcpyHostToDevice));
  if (mesh->texcoords) {
    MCK(d_tc.reserve(sizeof(float) * 2 * nv));
    MCK(cudaMemcpy(d_tc, mesh->texcoords, sizeof(float) * 2 * nv, cudaMemcpyHostToDevice));
  }
  MCK(tlo.reserve(sizeof(float4) * n)); MCK(thi.reserve(sizeof(float4) * n));
  MCK(nlo.reserve(sizeof(float4) * std::max(1, n - 1))); MCK(nhi.reserve(sizeof(float4) * std::max(1, n - 1)));
  MCK(codes.reserve(sizeof(uint64_t) * n)); MCK(codes2.reserve(sizeof(uint64_t) * n));
  MCK(ids.reserve(sizeof(int) * n)); MCK(ids2.reserve(sizeof(int) * n));
  MCK(left.reserve(sizeof(int) * std::max(1, n - 1))); MCK(right.reserve(sizeof(int) * std::max(1, n - 1)));
  MCK(pin.reserve(sizeof(int) * std::max(1, n - 1))); MCK(pleaf.reserve(sizeof(int) * n));
  MCK(visits.reserve(sizeof(int) * std::max(1, n - 1)));
  MCK(mb.nodes.reserve(sizeof(float4) * 8 * std::max(1, n - 1)));
  MCK(mb.tris_f64.reserve(sizeof(MeshTri<double>) * n));
  MCK(mb.tris_f32.reserve(sizeof(MeshTri<float>) * n));
  if (mesh->n_materials > 0) {
    std::vector<unsigned short> ids((size_t)n);
    for (int t = 0; t < n; t++) ids[t] = (unsigned short)mesh->material_ids[t];
    MCK(mb.mat_ids.reserve(sizeof(unsigned short) * n));
    MCK(cudaMemcpy(mb.mat_ids, ids.data(), sizeof(unsigned short) * n, cudaMemcpyHostToDevice));
  }
  lbvh_tri_setup<<<G, B>>>(n, d_verts, d_idx, slo, sinv, tlo, thi, codes, ids);
  lbvh_tri_records<double><<<G, B>>>(n, d_verts, d_idx, d_tc, mb.tris_f64);
  lbvh_tri_records<float><<<G, B>>>(n, d_verts, d_idx, d_tc, mb.tris_f32);
  if (n > 1) {
    MCK(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, codes.p, codes2.p, ids.p, ids2.p, n, 0, 63));
    MCK(tmp.reserve(tmp_bytes));
    MCK(cub::DeviceRadixSort::SortPairs(tmp.p, tmp_bytes, codes.p, codes2.p, ids.p, ids2.p, n, 0, 63));
    MCK(cudaMemset(visits, 0, sizeof(int) * (n - 1)));
    lbvh_karras<<<(n - 1 + B - 1) / B, B>>>(n, codes2, left, right, pin, pleaf);
    lbvh_refit<<<G, B>>>(n, ids2, tlo, thi, left, right, pin, pleaf, nlo, nhi, visits);
    lbvh_pack4<<<(n - 1 + B - 1) / B, B>>>(n, ids2, tlo, thi, left, right, pin, nlo, nhi, mb.nodes);
  } else {
    // single triangle: one node whose slots 0 and 1 both hold it (only slots 2 and 3 may be empty); a second test of it
    // changes nothing
    float4 h_lo, h_hi;
    MCK(cudaMemcpy(&h_lo, tlo, sizeof(float4), cudaMemcpyDeviceToHost));
    MCK(cudaMemcpy(&h_hi, thi, sizeof(float4), cudaMemcpyDeviceToHost));
    float c[4][3], h[4][3];
    int ref[4] = {-1, -1};
    for (int a = 0; a < 3; a++) {
      centreHalf((&h_lo.x)[a], (&h_hi.x)[a], c[0][a], h[0][a]);
      c[1][a] = c[0][a]; h[1][a] = h[0][a];
    }
    float4 nd[8];
    packNode4(nd, 2, c, h, ref);
    MCK(cudaMemcpy(mb.nodes, nd, sizeof(nd), cudaMemcpyHostToDevice));
  }
  MCK(cudaDeviceSynchronize());
  MCK(cudaGetLastError());
  *out = std::move(mb);
  return DRT_OK;
}

}  // namespace drt
