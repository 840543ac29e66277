// Host entry points of the device LBVH build (drt_mesh.cu).
#pragma once
#include <string>
#include <cuda_runtime.h>
#include "../../include/drt.h"
#include "drt_device.cuh"

namespace drt {
struct MeshBuffers {
  DevBuf<float4> nodes;              // 4-wide LBVH nodes (drt_box.cuh), 8 float4 per node
  DevBuf<MeshTri<double>> tris_f64;  // [n_tris]
  DevBuf<MeshTri<float>> tris_f32;   // [n_tris]
  DevBuf<unsigned short> mat_ids;    // per-triangle index into the mesh's material table, or empty (one material)
  int n_tris = 0;
};
// Uploads the mesh, builds the LBVH on the current device.  Returns a drt_status.
int buildMesh(const drt_mesh* mesh, MeshBuffers* out, std::string& err);
}  // namespace drt
