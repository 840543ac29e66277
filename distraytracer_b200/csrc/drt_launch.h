// Launch wrappers.  The kernels are instantiated in two translation units so the
// two precisions can be compiled with different floating-point contraction:
//   drt_kernels_f64.cu  (R = double, "reference" precision)  -fmad=false
//       The reference ran on x86-64 without FMA; several of its own scenes put
//       area-light panels IN the ceiling plane, where shadow-ray plane tests
//       divide two rounding residues (~1e-17) and the image is decided by the
//       last bit.  With contraction off, CUDA's double +,-,*,/ and sqrt are the
//       same IEEE operations in the same order, so those decisions match.
//   drt_kernels_f32.cu  (R = float)                            default (FMA on)
#pragma once
#include "drt_device.cuh"

// ---- shape of one persistent render_wave CTA (shared by the kernels and the host-side pool sizing)
#ifndef DRT_WAVE_WARPS
#define DRT_WAVE_WARPS 16
#endif
#ifndef DRT_BATCH
#define DRT_BATCH 64          // camera samples per warp in a CTA batch
#endif
#define DRT_CTA_SLOTS (DRT_WAVE_WARPS * DRT_BATCH)   // camera samples per CTA batch
// TRACE stops feeding the hit buffer at this many hits.  Larger = fewer phase switches, more 32-hit bites
// per warp and pass (shorter barrier tails) and bigger geom buckets in the SHADE sort; costs a deeper ray pool.
#ifndef DRT_TRACE_HITS_TARGET
#define DRT_TRACE_HITS_TARGET 8192
#endif
#define DRT_HITS_PER_PASS (DRT_TRACE_HITS_TARGET + 32 * DRT_WAVE_WARPS)   // a TRACE pass can overshoot by one bite per warp
#define DRT_CTA_HITS (DRT_HITS_PER_PASS + 64)
#define DRT_MAX_CHILDREN 6    // refraction + max(brdf_samples, 1)
#ifndef DRT_PAIR_LIGHTS
#define DRT_PAIR_LIGHTS 8      // lights whose shadow rays are spread over the warp per pass
#endif
#define DRT_SMEM_GEOMS 256     // slab-filter entries staged in shared memory per CTA
// Bytes of geom + primitive + light records staged in shared memory per CTA (FT_RECS); a scene with more reads them from
// global memory.  With the CTA's other 65.0 KB of shared memory (11.3 KB static + 53.7 KB waveDynSmemBytes) and the 1 KB
// reserved per block this stays within a 100 KB shared-memory carve-out: one CTA of 16 warps per SM, 156 KB of L1 left.
#define DRT_SMEM_RECS (32 * 1024)

// ---- feature mask of a render_wave instantiation ------------------------------------------------------------------
// render_wave is compiled once per feature set and the host picks the smallest instantiation that covers the scene and
// settings of a render call: code a scene cannot reach (mesh traversal, time-displaced geometry, the replayed reference
// tree of reference-mode blur, glass, textures) costs registers and instruction-cache space even when it never runs
// (ncu round 1: 11.9 % of the stall samples "no_instructions" at 16 k SASS instructions, 0.5 G spill instructions per band).
enum WaveFeat {
  FT_MESH = 1,      // a triangle mesh (LBVH traversal, drt_lbvh.cuh) is present
  FT_VEL = 2,       // blur re-traces with per-primitive velocities (DRT_BLUR_VELOCITY) can occur
  FT_REFBLUR = 4,   // reference-mode blur re-traces can occur: "rectangle" shapes move, the reference tree is walked
  FT_GLASS = 8,     // some primitive is glass (refraction children)
  FT_TEX = 16,      // some primitive is textured
  FT_BIG = 32,      // more geoms than the shared-memory slab table holds (DRT_SMEM_GEOMS)
  FT_BOX = 64,      // slab-box prisms (RectPrism / RectPrismWithCylinder / RectPrismWithHoles) are present
  FT_SPILL = 128,   // a rectangle whose edges B-A, D-A are not orthogonal is present (GF_SPILL: hits need the reference's gather replayed)
  FT_ALL = 255,
  // Not a scene feature: the instantiation reads the geom, primitive and light records from a copy in shared memory, which
  // the launcher picks when the scene's records fit (Params::smem_recs).  A compile-time choice: with the table picked at
  // run time, the pointer select held registers and turned ld.shared into generic loads (the bench instantiation: 56-92
  // bytes of spill stores instead of 20).  Every mask of DRT_WAVE_FEATS but FT_ALL is also instantiated with it.
  FT_RECS = 256
};

// the instantiated masks (drt_launch_impl.cuh must hold one DRT_WAVE_CASE per entry); FT_ALL last
#define DRT_WAVE_FEATS {FT_GLASS | FT_TEX, 0, FT_TEX, FT_VEL, FT_MESH | FT_TEX, FT_MESH | FT_VEL | FT_TEX, FT_REFBLUR | FT_GLASS | FT_TEX, FT_ALL}

namespace drt {
// feature masks this precision's translation units instantiate, `n` of them; the last one is FT_ALL
const int* waveFeatList(int* n);
// smallest instantiated superset of `need`
int waveFeatPick(int need);
// persistent grid of render_wave: blocks that are co-resident on the current device
template <typename R> int waveGridBlocks();
// bytes of scratch (ray pools of `pool_cap` tasks, hit buffers, shadow-pair buffers) a grid of `blocks` CTAs needs
template <typename R> size_t wavePoolBytes(int blocks, int pool_cap);
// `feat`: what the call needs (any mask; the launcher maps it to an instantiation, adding FT_RECS when P.smem_recs).
// Returns the mask launched.
template <typename R> int launchRenderSamples(const Params<R>& P, bool collect, int feat, int blocks, cudaStream_t q);
// one translation unit per (precision, group) instantiates part of the list: kernel of mask `feat`, or nullptr
template <typename R> using WaveFnT = void (*)(Params<R>);
template <typename R, int GROUP> WaveFnT<R> waveKernelOfGroup(int feat, bool collect);
template <typename R> void launchCloudCorners(const Params<R>& P, cudaStream_t q);
template <typename R> void launchResolve(const Params<R>& P, int row0, int rows, cudaStream_t q);
void launchNeedPush(const unsigned char* mine, unsigned char* shared, size_t n, cudaStream_t q);
}  // namespace drt
