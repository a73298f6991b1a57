// common.cuh — error plumbing and small device helpers shared by all kernels.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <atomic>

#include "../../include/iswm_b200.h"

namespace iswm {

void set_error(const char* fmt, ...);
extern std::atomic<int64_t> g_launches;
// measurement aid (iswm_debug_set_skip): entry points of a masked kernel family return 0 without launching, so that a
// whole step can be timed with and without that family (its marginal cost inside the real launch pipeline)
extern std::atomic<int> g_skip_mask;
inline bool debug_skip(int family_bit) { return (g_skip_mask.load(std::memory_order_relaxed) & family_bit) != 0; }

inline int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s: %s", what, cudaGetErrorString(e));
    return 1;
  }
  g_launches.fetch_add(1, std::memory_order_relaxed);
  return 0;
}

#define ISWM_REQUIRE(cond, ...)            \
  do {                                     \
    if (!(cond)) {                         \
      ::iswm::set_error(__VA_ARGS__);      \
      return 2;                            \
    }                                      \
  } while (0)

// ---- programmatic dependent launch (PDL) -------------------------------------------------------------------
// Kernels launched through launch_k() carry cudaLaunchAttributeProgrammaticStreamSerialization: the next kernel
// of the stream may be scheduled (and run its prologue: barrier init, TMEM allocation, index setup) while this
// one drains. Every such kernel calls pdl_wait() before its first access to global memory (it returns once the
// preceding grid has completed and its writes are visible) and then pdl_launch() to let ITS successor queue up.
// ISWM_PDL=0 in the environment turns the attribute off (plain stream order; the device calls become no-ops).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
bool pdl_enabled();

template <typename... KArgs, typename... Args>
inline void launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl_enabled() ? 1 : 0;
  cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);   // errors surface in check_launch()
}

inline int num_sms() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// Largest grid of a grid-stride kernel that is resident all at once: SMs x the occupancy the compiled kernel really
// gets (register count decides it, e.g. 44 registers x 256 threads = 5 blocks per SM, not the 8 a 32-register kernel
// would have). A grid above this runs as 1.x waves and the partial last wave is a pure tail. Cached per kernel.
template <typename K>
inline int resident_grid(K kernel, int block, size_t smem = 0) {
  struct Slot { const void* fn; int blocks; };
  static thread_local Slot cache[64];
  static thread_local int n_cached = 0;
  const void* key = reinterpret_cast<const void*>(kernel);
  for (int i = 0; i < n_cached; i++)
    if (cache[i].fn == key) return cache[i].blocks * num_sms();
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, block, smem) != cudaSuccess || occ <= 0) {
    cudaGetLastError();
    occ = 4;
  }
  if (n_cached < 64) cache[n_cached++] = Slot{key, occ};
  return occ * num_sms();
}

__device__ __forceinline__ float bf16_bits_to_float(uint32_t bits16) {
  return __uint_as_float(bits16 << 16);
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ void unpack_bf16x2(uint32_t v, float& lo, float& hi) {
  lo = __uint_as_float(v << 16);
  hi = __uint_as_float(v & 0xffff0000u);
}

// streaming 16-byte load that does not pollute L1 (guide: Guideline 13)
__device__ __forceinline__ int4 ld_stream16(const void* p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream16(void* p, const int4& v) {
  asm volatile("st.global.L1::no_allocate.v4.s32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x),
               "r"(v.y), "r"(v.z), "r"(v.w)
               : "memory");
}

// bilinear source coordinates of output index o (align_corners=False, as F.interpolate at network/utils.py:22)
__device__ __forceinline__ void bil_src(int o, float scale, int in, int& i0, int& i1, float& l1) {
  float src = ((float)o + 0.5f) * scale - 0.5f;
  src = src < 0.f ? 0.f : src;
  i0 = (int)src;
  if (i0 > in - 1) i0 = in - 1;
  i1 = i0 + ((i0 < in - 1) ? 1 : 0);
  l1 = src - (float)i0;
}
// the four-tap mix with a FIXED contraction (explicit fma chain): every kernel that interpolates logits produces the
// same bits, so the fused predict epilogue equals upsample-then-threshold exactly
__device__ __forceinline__ float bil_mix(float w00, float v00, float w01, float v01, float w10, float v10, float w11, float v11) {
  return fmaf(w11, v11, fmaf(w10, v10, fmaf(w01, v01, w00 * v00)));
}

// counter-based dropout keep decision shared by forward and backward
__device__ __forceinline__ bool drop_keep(uint64_t seed, uint64_t idx, float p) {
  uint64_t z = idx + seed * 0x9E3779B97F4A7C15ull + 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  z = z ^ (z >> 31);
  float u = (float)(uint32_t)(z >> 40) * (1.0f / 16777216.0f);
  return u >= p;
}

}  // namespace iswm
