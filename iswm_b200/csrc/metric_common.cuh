// metric_common.cuh - packed vector loads / stores and the block counter flush shared by the HBM-bound metric kernels
// (loss_metric.cu, tta.cu).
#pragma once
#include "common.cuh"

namespace iswm {

// ---------------------------------------------------------------------------
// packed loads
template <int BYTES> struct Pack;
template <> struct __align__(1) Pack<1> { uint8_t v; };
template <> struct __align__(2) Pack<2> { uint16_t v; };
template <> struct __align__(4) Pack<4> { uint32_t v; };
template <> struct __align__(8) Pack<8> { uint2 v; };
template <> struct __align__(16) Pack<16> { uint4 v; };
template <> struct __align__(16) Pack<32> { uint4 v[2]; };
template <> struct __align__(16) Pack<64> { uint4 v[4]; };
template <> struct __align__(16) Pack<128> { uint4 v[8]; };

template <typename T, int N>
struct Vec {
  union {
    Pack<sizeof(T) * N> p;
    T e[N];
  };
  __device__ __forceinline__ Vec() {}
};

template <typename T, int N>
__device__ __forceinline__ void vload(Vec<T, N>& dst, const T* src) {
  constexpr int BYTES = sizeof(T) * N;
  if constexpr (BYTES >= 16) {
    const uint4* s = reinterpret_cast<const uint4*>(src);
#pragma unroll
    for (int i = 0; i < BYTES / 16; i++) {
      uint4 t = __ldcs(s + i);
      reinterpret_cast<uint4*>(&dst.p)[i] = t;
    }
  } else {
    dst.p = *reinterpret_cast<const Pack<BYTES>*>(src);
  }
}
template <typename T, int N>
__device__ __forceinline__ void vstore(T* dst, const Vec<T, N>& src) {
  constexpr int BYTES = sizeof(T) * N;
  if constexpr (BYTES >= 16) {
    uint4* d = reinterpret_cast<uint4*>(dst);
#pragma unroll
    for (int i = 0; i < BYTES / 16; i++) __stcs(d + i, reinterpret_cast<const uint4*>(&src.p)[i]);
  } else {
    *reinterpret_cast<Pack<BYTES>*>(dst) = src.p;
  }
}

__device__ __forceinline__ unsigned warp_sum_u32(unsigned v) { return __reduce_add_sync(0xffffffffu, v); }

constexpr int kThreads = 256;
constexpr int kWarps = kThreads / 32;

// block-level flush of NREG per-thread counters into int64 global counters
template <int NREG>
__device__ __forceinline__ void flush_counters(unsigned (&cnt)[NREG], int n_valid,
                                               unsigned long long* g_out) {
  __shared__ unsigned s_part[kWarps][NREG];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
#pragma unroll
  for (int k = 0; k < NREG; k++) {
    unsigned s = warp_sum_u32(cnt[k]);
    if (lane == 0) s_part[warp][k] = s;
  }
  __syncthreads();
  if (threadIdx.x < NREG && (int)threadIdx.x < n_valid) {
    unsigned long long t = 0;
#pragma unroll
    for (int w = 0; w < kWarps; w++) t += s_part[w][threadIdx.x];
    if (t) atomicAdd(g_out + threadIdx.x, t);
  }
}

}  // namespace iswm
