// Included by drt_kernels_{f64,f32}_g{0,1,2}.cu with DRT_REAL and DRT_GROUP defined.  The render_wave instantiations of
// one precision are spread over three translation units (they compile in parallel); group 0 also holds the launchers and
// the two small kernels.
#include <algorithm>
#include "drt_kernels.cuh"
#include "drt_launch.h"

namespace drt {
typedef WaveFnT<DRT_REAL> WaveFn;
// each mask with and without FT_RECS (records in shared memory)
#define DRT_WAVE_CASE(mask)                                                                                              \
  if ((feat & ~FT_RECS) == (mask) && !collect)                                                                           \
    return (feat & FT_RECS) ? render_wave<DRT_REAL, (mask) | FT_RECS, false> : render_wave<DRT_REAL, (mask), false>
#if DRT_GROUP == 0
// static scenes: the bench workload (glass + textures), plain and textured analytic scenes
template <> WaveFn waveKernelOfGroup<DRT_REAL, 0>(int feat, bool collect) {
  DRT_WAVE_CASE(FT_GLASS | FT_TEX);
  DRT_WAVE_CASE(0);
  DRT_WAVE_CASE(FT_TEX);
  return nullptr;
}
#elif DRT_GROUP == 1
// velocity-mode motion blur (mocap bones) and triangle meshes
template <> WaveFn waveKernelOfGroup<DRT_REAL, 1>(int feat, bool collect) {
  DRT_WAVE_CASE(FT_VEL);
  DRT_WAVE_CASE(FT_MESH | FT_TEX);
  DRT_WAVE_CASE(FT_MESH | FT_VEL | FT_TEX);
  return nullptr;
}
#else
// reference-mode motion blur, and the instantiation that can do everything (also the counting build)
template <> WaveFn waveKernelOfGroup<DRT_REAL, 2>(int feat, bool collect) {
  DRT_WAVE_CASE(FT_REFBLUR | FT_GLASS | FT_TEX);
  if (feat == FT_ALL) return collect ? render_wave<DRT_REAL, FT_ALL, true> : render_wave<DRT_REAL, FT_ALL, false>;   // global records
  return nullptr;
}
#endif

#if DRT_GROUP == 0
static WaveFn waveKernel(int feat, bool collect) {
  WaveFn f = waveKernelOfGroup<DRT_REAL, 0>(feat, collect);
  if (!f) f = waveKernelOfGroup<DRT_REAL, 1>(feat, collect);
  if (!f) f = waveKernelOfGroup<DRT_REAL, 2>(feat, collect);
  return f;
}
template <> int waveGridBlocks<DRT_REAL>() {
  int dev = 0, sms = 0, per_sm = 1 << 30, n = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  const int* list = waveFeatList(&n);
  auto fit = [&](WaveFn f, const size_t smem) {
    int k = 0;
    cudaFuncSetAttribute((const void*)f, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&k, (const void*)f, 32 * DRT_WAVE_WARPS, smem);
    per_sm = k < per_sm ? k : per_sm;
  };
  // every instantiation (FT_RECS: with a full record table) + the counting build; the grid fits the hungriest one
  for (int i = 0; i < n; i++) {
    fit(waveKernel(list[i], false), waveDynSmemBytes());
    if (list[i] != FT_ALL) fit(waveKernel(list[i] | FT_RECS, false), waveDynSmemBytes() + DRT_SMEM_RECS);
  }
  fit(waveKernel(FT_ALL, true), waveDynSmemBytes());
  if (per_sm < 1) per_sm = 1;
  return sms * per_sm;   // a whole multiple of the SM count: every SM holds the same number of persistent CTAs
}
template <> size_t wavePoolBytes<DRT_REAL>(int blocks, int pool_cap) { return (size_t)blocks * waveScratchBytes<DRT_REAL>(pool_cap); }
template <> int launchRenderSamples<DRT_REAL>(const Params<DRT_REAL>& P, bool collect, int feat, int blocks, cudaStream_t q) {
  int pick = collect ? FT_ALL : waveFeatPick(feat);
  if (pick != FT_ALL && P.smem_recs) pick |= FT_RECS;
  waveKernel(pick, collect)<<<blocks, 32 * DRT_WAVE_WARPS, waveDynSmemBytes() + ((pick & FT_RECS) ? P.smem_recs : 0), q>>>(P);
  return pick;
}
template <> void launchCloudCorners<DRT_REAL>(const Params<DRT_REAL>& P, cudaStream_t q) {
  const int n = (P.w + 1) * (P.h + 1);
  int blocks = (n + DRT_CLOUD_BLOCK - 1) / DRT_CLOUD_BLOCK;
  if (P.corner_counter) {             // blocks of corners are claimed from a shared counter: a resident grid is enough
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    blocks = std::min(blocks, sms * 16);
  }
  cloud_corners<DRT_REAL><<<blocks, 128, 0, q>>>(P);
}
#ifdef DRT_DEFINE_SHARED_LAUNCHERS
void launchNeedPush(const unsigned char* mine, unsigned char* shared, size_t n, cudaStream_t q) {
  need_push<<<(unsigned)((n + 255) / 256), 256, 0, q>>>(mine, shared, n);
}
#endif
template <> void launchResolve<DRT_REAL>(const Params<DRT_REAL>& P, int row0, int rows, cudaStream_t q) {
  resolve<DRT_REAL><<<(P.w * rows + 255) / 256, 256, 0, q>>>(P, row0, rows);
}
#endif
}  // namespace drt
