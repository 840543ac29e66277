// Device-side data layout and math for the distributed ray-tracing hot path.
//
// Everything is templated on the vector scalar R:
//   R = double : "reference" precision -- double vectors with float scalar
//                temporaries, expression by expression like the reference
//                (SETTINGS.h:13 Real=double; geometry.cpp keeps A,B,C,disc,t in float);
//   R = float  : fp32 variant.
//
// The scene is flattened on the host (drt_api.cu) into
//   Geom<R>  : one intersectable piece (sphere, open cylinder, triangle, rectangle
//              or checker rectangle, plus "hole" records).  RectPrismV2 becomes its
//              six face rectangles in the reference's face order
//              (geometry.cpp:796-801); min-t with strict `<` over consecutive
//              candidates is what RectPrismV2::intersect computes (815-838).
//   PrimD<R> : the per-GeoPrimitive shading record (material, normal, UV, emissive).
//   LightD<R>: the LightPrimitive records.
// Records are 16-byte aligned and whole 16-byte words (render_wave copies them to shared
// memory word by word); every lane of a warp reads the same record in the
// candidate loops, so loads are warp-uniform broadcasts.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <float.h>
#include <math.h>
#include <utility>

#include "drt_rng.cuh"

#define DRT_PI 3.14159265358979323846
#define DRT_NODE_STACK 64  // per-thread BVH traversal stack (node indices)

namespace drt {

template <typename R> struct Vec { R x, y, z; };

template <typename R> __host__ __device__ inline Vec<R> mk(R x, R y, R z) { Vec<R> v; v.x = x; v.y = y; v.z = z; return v; }
template <typename R> __host__ __device__ inline Vec<R> operator+(Vec<R> a, Vec<R> b) { return mk<R>(a.x + b.x, a.y + b.y, a.z + b.z); }
template <typename R> __host__ __device__ inline Vec<R> operator-(Vec<R> a, Vec<R> b) { return mk<R>(a.x - b.x, a.y - b.y, a.z - b.z); }
template <typename R> __host__ __device__ inline Vec<R> operator-(Vec<R> a) { return mk<R>(-a.x, -a.y, -a.z); }
template <typename R> __host__ __device__ inline Vec<R> operator*(Vec<R> a, R s) { return mk<R>(a.x * s, a.y * s, a.z * s); }
template <typename R> __host__ __device__ inline Vec<R> operator*(R s, Vec<R> a) { return mk<R>(s * a.x, s * a.y, s * a.z); }
template <typename R> __host__ __device__ inline Vec<R> operator/(Vec<R> a, R s) { return mk<R>(a.x / s, a.y / s, a.z / s); }
// Eigen's unrolled 3-coefficient reduction: c0 + (c1 + c2)
template <typename R> __host__ __device__ inline R dot(Vec<R> a, Vec<R> b) { return a.x * b.x + (a.y * b.y + a.z * b.z); }
template <typename R> __host__ __device__ inline R norm(Vec<R> a) { return sqrt(dot(a, a)); }
// x / s for three numerators sharing one divisor: one IEEE division for the reciprocal, then
// per numerator q = x*r refined by two fused steps (rem = x - q*s; q += rem*r), which yields
// the correctly rounded quotient -- the same bits as the reference's three divisions -- at a
// third of the cost of three software double divides.
__device__ __forceinline__ double div_shared(double x, double s, double r) {
  const double q = x * r;
  const double rem = fma(-q, s, x);
  return fma(rem, r, q);
}
template <typename R> __host__ __device__ inline Vec<R> normalized(Vec<R> a) {  // Eigen >= 3.3 semantics
  R z = dot(a, a);
  if (z > R(0)) {
#if defined(__CUDA_ARCH__) && !defined(DRT_OLD_NORMALIZE)
    if (sizeof(R) == 8) {
      const double s = sqrt((double)z);
      const double r = 1.0 / s;
      return mk<R>((R)div_shared((double)a.x, s, r), (R)div_shared((double)a.y, s, r), (R)div_shared((double)a.z, s, r));
    }
#endif
    return a / (R)sqrt(z);
  }
  return a;
}
template <typename R> __host__ __device__ inline Vec<R> cross(Vec<R> a, Vec<R> b) {
  return mk<R>(a.y * b.z - a.z * b.y, a.z * b.x - a.x * b.z, a.x * b.y - a.y * b.x);
}
template <typename R> __host__ __device__ inline Vec<R> cmul(Vec<R> a, Vec<R> b) { return mk<R>(a.x * b.x, a.y * b.y, a.z * b.z); }
template <typename R> __host__ __device__ inline bool isZero(Vec<R> a) { return !(dot(a, a) > R(0)) && dot(a, a) == dot(a, a); }

// ---------------------------------------------------------------------------
enum GeomType { G_SPHERE = 0, G_CYL = 1, G_TRI = 2, G_RECT = 3, G_CHECKER = 4, G_HOLE = 5, G_BOX = 6 };
enum GeomFlags {
  GF_NAME_RECTANGLE = 1,  // moves in y during reference-mode motion blur (render_final_project.cpp:1116)
  GF_HAS_HOLE = 2,        // next record is this checkerboard's hole rectangle
  GF_MESH = 4,            // Triangle::mesh (inside test against mesh_normal)
  GF_VERTEX_MOTION = 8,   // cylinder whose end points move independently (DRT_FLAG_VERTEX_MOTION): p1 moves by vel2
  GF_SPILL = 16           // rectangle whose edges B-A, D-A are not orthogonal: Rectangle::intersect accepts points outside the
                          // vertices' bounding box, and whether the reference finds such a hit depends on its BVH gather
};

template <typename R>
struct alignas(16) Geom {
  int type;     // GeomType
  int owner;    // index into prims
  int flags;    // GeomFlags
  float eps;    // rectangle t threshold: 1e-4 (Rectangle) or 1e-3 (Checkerboard*)
  // sphere : p0 center                                   f0 radius
  // cyl    : p0 c1, p1 c2, p2 axis                       f0 radius
  // tri    : p0 A,  p1 B-A, p2 C-A, p3 mesh_normal
  // rect   : p0 A,  p1 unit normal, p2 (B-A)^, p3 (D-A)^ len1 |B-A|, len2 |D-A|, f2 S
  // box    : p0 lbound, p1 ubound (world AABB of the prism's corners); holes and the class live in prims[owner]
  Vec<R> p0, p1, p2, p3;
  float f0, f1, f2, f3;
  Vec<R> vel;   // DRT_BLUR_VELOCITY displacement per unit time
  // rectangles: edge lengths |B-A|, |D-A|.  Cylinders with GF_VERTEX_MOTION keep the displacement of their second end
  // point per unit time in the same three words (cylV2): the record stays 224 bytes.
  R len1, len2, pad_;
  __host__ __device__ Vec<R> cylV2() const { return mk<R>(len1, len2, pad_); }
  float4 blo, bhi;   // padded single-precision bounds for the slab filter
  int leaf;          // reference BVH leaf holding this geom
  int pad2_[3];
};

// One BoundingVolume of the reference's tree (drt_bvh_order.h), 16-byte aligned.
template <typename R>
struct alignas(16) NodeD {
  Vec<R> lo, hi;
  int leaf;          // 1: geoms [first, first+count)
  int first, count;
  int left, right;
  int parent;        // -1 at the root
  int pad_[2];
};

// One hole of RectPrismWithCylinder / RectPrismWithHoles (geometry.h:195, 216)
template <typename R>
struct alignas(16) HoleD {
  Vec<R> c1, c2, axis;   // sphere: c1 = centre
  float radius;
  int type;              // G_SPHERE or G_CYL
  float color[3];
  float pad_;
};

template <typename R>
struct alignas(16) PrimD {
  int type, name, material, model, flags, tex;
  float roughness;
  float on_A, on_B;        // Oren-Nayar A,B (render_final_project.cpp:896-897)
  float schlick_R0;        // helpers.h:315
  float radius, S, borderwidth, length, width, axis_norm;
  float color[3], bordercolor[3], color1[3], color2[3];
  // normals: n0 = rect/tri normal or prism "bot"; n1 prism "right"; n2 prism "front"
  Vec<R> n0, n1, n2;
  Vec<R> pA, pG;           // prism corners A,G; sphere: pA=center; cylinder: pA=c1, pG=axis
  // UV rectangle (Rectangle::getUV geometry.cpp:751-759): A, D, ad, dc, denominators
  Vec<R> uvA, uvD, uv_ad, uv_dc;
  R uv_den_u, uv_den_v;
  // CheckerboardWithHole::getUV: outer rect basis + hole rect
  Vec<R> rA, re1, re2; R rlen1, rlen2;
  Vec<R> hA, hn, he1, he2; R hlen1, hlen2;
  // Triangle::getUV
  Vec<R> tA, tB, tC; float tuv[6];
  // CheckerCylinder::getUV object matrix rows (geometry.cpp:2580-2585)
  R objM[12];
  // emissive (render_final_project.cpp:775-789)
  Vec<R> center, eA, eB, eC, eD; R e_den;
  Vec<R> vel;              // DRT_FLAG_VERTEX_MOTION cylinders keep c2 in n1 and its velocity in n2 (prism normals otherwise)
  // slab-box prisms (types 8-10): objM above holds cob * origin (geometry.cpp:975-984)
  float height; int n_holes;
  HoleD<R> holes[4];
};

// one mesh triangle for the exact test + texture coordinates (drt_lbvh.cuh)
template <typename R>
struct alignas(16) MeshTri {
  Vec<R> A, B, C;
  float uv[6];
};

template <typename R>
struct alignas(16) LightD {
  int type, prim_index;
  float radius;
  int use_baxis;
  float color[3];
  float pad_;
  Vec<R> center, baxis, A, B, D;
};

struct Counts {
  unsigned long long samples, rays, shadow_rays, geom_tests[7], shade_evals, noise_evals, node_tests;
};

template <typename R>
struct Params {
  // camera (render_final_project.cpp:989-1027)
  Vec<R> eye, X, Y, Z;
  R mcam[12], new_mcam[12], cloud_mcam[12];
  float t, b, r, l;
  float near_plane, focal_length, aperture;
  int xRes, yRes;
  int n, spp, antialias_samples;
  int brdf_samples, blur_samples, frame_range, max_depth;
  int reflect, nogloss, perlin_cloud, cloud_only;
  int frame, frame_prism, frame_blur, frame_cloud;
  int swept_cull;           // velocity-mode re-traces may use the slab filter: its boxes cover the motion over frame_range
  float move_per_frame, accel_t, refr_air, refr_glass, phong;
  uint32_t seed;
  int blur_mode;
  // sky (render_final_project.cpp:127-136)
  Vec<R> sun;   // sundir.normalized()
  float sun_outer[3], sun_inner[3], sun_core[3], bluesky[3], redsky[3];
  float saturation, clouddist, cloudhoff;
  // tile
  int x0, y0, w, h;
  // scene
  const Geom<R>* geoms; int n_geoms;
  const float4* gbounds;    // slab-filter table: one pair record per PAIR of geoms (drt_box.cuh, see slabMask)
  const float4* geom_tree;  // 4-wide tree over the geoms (nodes of drt_box.cuh) for scenes beyond DRT_SMEM_GEOMS, or nullptr
  const NodeD<R>* nodes; int n_nodes;
  const PrimD<R>* prims; int n_prims;
  const LightD<R>* lights; int n_lights;
  int smem_recs;            // bytes of geoms + prims + lights when they fit DRT_SMEM_RECS (an FT_RECS render_wave stages them), else 0
  // triangle mesh (optional): LBVH nodes (drt_box.cuh, 8 float4 each), exact-test records, material = prims[mesh_prim]
  const float4* mesh_nodes; const MeshTri<R>* mesh_tris; int n_mesh_tris; int mesh_prim;
  const unsigned short* mesh_mat;   // per-triangle material: prims[mesh_prim + mesh_mat[tri]]; nullptr: prims[mesh_prim]
  Vec<R> mesh_vel;                  // DRT_BLUR_VELOCITY: the mesh moves as a whole by mesh_vel * time (its materials' common velocity)
  const cudaTextureObject_t* tex; const int2* texdims;
  // buffers
  float4* samples;          // [pixel_in_tile * spp + s] : rgb + flag bits
  unsigned char* need;      // (w+1)*(h+1) pixel-corner "background wanted" map
  float4* bg;               // (w+1)*(h+1) background colours
  float* out_f32;           // w*h*3 (PPM row order) or nullptr
  unsigned char* out_u8;    // w*h*3 (PPM row order)
  Counts* counts;           // nullptr unless collecting
  long long sample_base;    // first (pixel*spp+s) index handled by this launch (row chunking)
  long long sample_count;
  void* pool_raw;           // per-CTA scratch: ray pool, hit buffer, shadow-pair buffers (waveScratchBytes)
  int pool_cap;             // ray tasks per CTA pool
  // work distribution: persistent CTAs claim UNITS of `unit_samples` consecutive camera samples of the launch from
  // `batch_counter` and work through a unit in batches of DRT_CTA_SLOTS.  One GPU: unit = one batch, the counter is local.
  // One frame on several GPUs (drt_render_multi): every GPU's kernel claims from the SAME counter in the gathering GPU's
  // memory (system-scope atomics over NVLink), units cover whole pixels, and `owned` (local, one byte per unit) records
  // which units this GPU rendered so that its resolve pass writes exactly those pixels.
  unsigned long long* batch_counter;
  int unit_samples;
  int steal;                // 1: batch_counter is shared between devices
  unsigned char* owned;     // nullptr unless stealing
  unsigned long long* corner_counter;   // cloud_corners: nullptr, or the counter all devices claim blocks of corners from
  int* overflow;
};

// sample flag bits stored in samples[].w
#define SF_ABORT 1u
#define SF_MISS 2u
#define SF_CORNER_SHIFT 2

__host__ __device__ inline float clampf(float v) {  // helpers.h:230-235
  if (v < 0.0f) return 0.0f;
  else if (v > 1.0f) return 1.0f;
  return v;
}

// Host side: device memory that frees itself.  Grow-only, move-only; reads as a T* wherever one is expected.
template <typename T>
struct DevBuf {
  T* p = nullptr;
  size_t cap = 0;   // bytes
  DevBuf() = default;
  DevBuf(const DevBuf&) = delete;
  DevBuf& operator=(const DevBuf&) = delete;
  DevBuf(DevBuf&& o) noexcept : p(o.p), cap(o.cap) { o.p = nullptr; o.cap = 0; }
  DevBuf& operator=(DevBuf&& o) noexcept { std::swap(p, o.p); std::swap(cap, o.cap); return *this; }
  ~DevBuf() { if (p) cudaFree(p); }
  // at least `bytes`; a buffer that is already large enough is kept, a smaller one is replaced (contents lost)
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) cudaFree(p);
    p = nullptr; cap = 0;
    const cudaError_t e = cudaMalloc(&p, bytes);
    if (e == cudaSuccess) cap = bytes; else p = nullptr;
    return e;
  }
  operator T*() const { return p; }
};

}  // namespace drt
