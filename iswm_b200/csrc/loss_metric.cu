// loss_metric.cu — the HBM-bound trio of the ISWM hot path, as single-pass
// vectorised kernels with register counters and warp-aggregated atomics:
//   class histogram          (reference: train.py:388-410, calculate_class_weights)
//   weighted softmax-CE f+b  (reference: train.py:454-459 criterion, :1046-1048)
//   confusion matrix         (reference: metrics/stream_metrics.py:24-31, :122)
//   argmax/threshold + cm    (reference: train.py:644,659; predict.py:264-275)
// Integer outputs are exact (int64 counters); float math is fp32 with a
// double-precision loss numerator.
#include "metric_common.cuh"

namespace iswm {

__device__ __forceinline__ float to_f32(float v) { return v; }
__device__ __forceinline__ float to_f32(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_f32(float v);
template <> __device__ __forceinline__ float from_f32<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_f32<__nv_bfloat16>(float v) {
  return __float2bfloat16_rn(v);
}

__device__ __forceinline__ float warp_sum_f32(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---------------------------------------------------------------------------
// class histogram
template <typename T>
__global__ void __launch_bounds__(kThreads)
class_hist_small_kernel(const T* __restrict__ labels, int64_t n, int n_classes,
                        unsigned long long* __restrict__ hist) {
  pdl_wait();
  pdl_launch();
  constexpr int VEC = 16 / sizeof(T);  // elements per 16-byte load
#ifndef ISWM_HIST_UNROLL
#define ISWM_HIST_UNROLL 4
#endif
  constexpr int UNROLL = ISWM_HIST_UNROLL;
  unsigned cnt[4] = {0, 0, 0, 0};
  const int64_t nvec = n / VEC;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  int64_t v = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  for (; v + (UNROLL - 1) * stride < nvec; v += UNROLL * stride) {
    Vec<T, VEC> x[UNROLL];
#pragma unroll
    for (int u = 0; u < UNROLL; u++) vload(x[u], labels + (v + u * stride) * VEC);
#pragma unroll
    for (int u = 0; u < UNROLL; u++)
#pragma unroll
      for (int i = 0; i < VEC; i++) {
        const long long y = (long long)x[u].e[i];
#pragma unroll
        for (int k = 0; k < 4; k++) cnt[k] += (y == k);
      }
  }
  for (; v < nvec; v += stride) {
    Vec<T, VEC> x;
    vload(x, labels + v * VEC);
#pragma unroll
    for (int i = 0; i < VEC; i++) {
      const long long y = (long long)x.e[i];
#pragma unroll
      for (int k = 0; k < 4; k++) cnt[k] += (y == k);
    }
  }
  // scalar tail
  if (blockIdx.x == 0) {
    for (int64_t i = nvec * VEC + threadIdx.x; i < n; i += kThreads) {
      const long long y = (long long)labels[i];
#pragma unroll
      for (int k = 0; k < 4; k++) cnt[k] += (y == k);
    }
  }
  flush_counters<4>(cnt, n_classes, hist);
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
class_hist_generic_kernel(const T* __restrict__ labels, int64_t n, int n_classes,
                          unsigned long long* __restrict__ hist) {
  pdl_wait();
  pdl_launch();
  extern __shared__ unsigned s_hist[];
  for (int i = threadIdx.x; i < n_classes; i += kThreads) s_hist[i] = 0;
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += stride) {
    const long long y = (long long)labels[i];
    const bool ok = (y >= 0 && y < n_classes);
    // warp-aggregated: lanes holding the same class elect one leader
    const unsigned active = __ballot_sync(__activemask(), ok);
    if (ok) {
      const unsigned peers = __match_any_sync(active, (int)y);
      const int leader = __ffs(peers) - 1;
      if ((int)(threadIdx.x & 31) == leader) atomicAdd(&s_hist[y], (unsigned)__popc(peers));
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < n_classes; i += kThreads)
    if (s_hist[i]) atomicAdd(hist + i, (unsigned long long)s_hist[i]);
}

template <typename T>
static int launch_class_hist(const void* labels, int64_t n, int n_classes, int64_t* hist,
                             cudaStream_t st) {
  const T* p = static_cast<const T*>(labels);
  auto* h = reinterpret_cast<unsigned long long*>(hist);
  const bool aligned = (reinterpret_cast<uintptr_t>(p) & 15) == 0;
  if (n_classes <= 4 && aligned) {
    constexpr int VEC = 16 / sizeof(T);
    int64_t want = (n / VEC + kThreads * ISWM_HIST_UNROLL - 1) / (kThreads * ISWM_HIST_UNROLL);
    int grid = (int)std::min<int64_t>(std::max<int64_t>(want, 1), (int64_t)resident_grid(class_hist_small_kernel<T>, kThreads));
    launch_k(class_hist_small_kernel<T>, dim3(grid), dim3(kThreads), 0, st, p, n, n_classes, h);
  } else {
    int64_t want = (n + kThreads * 8 - 1) / (kThreads * 8);
    int grid = (int)std::min<int64_t>(std::max<int64_t>(want, 1), (int64_t)resident_grid(class_hist_generic_kernel<T>, kThreads, n_classes * sizeof(unsigned)));
    launch_k(class_hist_generic_kernel<T>, dim3(grid), dim3(kThreads), n_classes * sizeof(unsigned), st, p, n, n_classes, h);
  }
  return check_launch("class_hist");
}

// ---------------------------------------------------------------------------
// weighted softmax cross-entropy, forward + backward in one pass

struct WceParams {
  int64_t B, HW;
  int C, ignore_index;
  float grad_scale;
};

__device__ __forceinline__ double wce_denominator(const float* w, const int64_t* hist, int C,
                                                  int ignore_index) {
  double D = 0.0;
  for (int c = 0; c < C; c++) {
    if (c == ignore_index) continue;
    D += (double)(w ? w[c] : 1.0f) * (double)hist[c];
  }
  return D;
}

__device__ __forceinline__ void block_add_double(float partial, double* g_out) {
  __shared__ float s_red[kWarps];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  float s = warp_sum_f32(partial);
  if (lane == 0) s_red[warp] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < kWarps; w++) t += (double)s_red[w];
    atomicAdd(g_out, t);
  }
}

// two-class fast path: VEC pixels per thread per step, both channel planes read
// with 16-byte loads, gradient planes written with 16-byte stores.
template <typename LT, typename YT, bool HAS_GRAD>
__global__ void __launch_bounds__(kThreads)
wce2_kernel(const LT* __restrict__ logits, const YT* __restrict__ labels,
            const float* __restrict__ weight, const int64_t* __restrict__ hist, WceParams p,
            LT* __restrict__ grad, double* __restrict__ loss_num) {
  pdl_wait();
  pdl_launch();
  constexpr int VEC = 16 / sizeof(LT);
  __shared__ float s_gs;
  if (threadIdx.x == 0) {
    const double D = wce_denominator(weight, hist, 2, p.ignore_index);
    s_gs = (float)((double)p.grad_scale / D);  // inf when D == 0; only multiplies valid pixels
  }
  __syncthreads();
  const float gs = s_gs;
  const float w0 = weight ? weight[0] : 1.0f, w1 = weight ? weight[1] : 1.0f;
  const int64_t vec_per_img = p.HW / VEC;
  const int64_t nvec = p.B * vec_per_img;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  float acc = 0.0f;
  for (int64_t v = (int64_t)blockIdx.x * kThreads + threadIdx.x; v < nvec; v += stride) {
    const int64_t b = v / vec_per_img;
    const int64_t i = (v - b * vec_per_img) * VEC;
    const LT* x0p = logits + (b * 2) * p.HW + i;
    Vec<LT, VEC> x0, x1;
    Vec<YT, VEC> y;
    vload(x0, x0p);
    vload(x1, x0p + p.HW);
    vload(y, labels + b * p.HW + i);
    Vec<LT, VEC> g0, g1;
#pragma unroll
    for (int k = 0; k < VEC; k++) {
      const long long yy = (long long)y.e[k];
      const bool valid = (yy == 0 || yy == 1) && yy != p.ignore_index;
      const float a0 = to_f32(x0.e[k]), a1 = to_f32(x1.e[k]);
      // d = x_other - x_target ; nll = softplus(d) ; p_other = sigmoid(d)
      const float d = (yy == 1) ? (a0 - a1) : (a1 - a0);
      const float e = expf(-fabsf(d));
      const float nll = fmaxf(d, 0.0f) + log1pf(e);
      const float inv = 1.0f / (1.0f + e);
      const float p_other = (d >= 0.0f) ? inv : e * inv;
      const float w = (yy == 1) ? w1 : w0;
      if (valid) acc += w * nll;
      if constexpr (HAS_GRAD) {
        const float gt = valid ? (w * p_other) * gs : 0.0f;  // +on other class, -on target
        g0.e[k] = from_f32<LT>((yy == 1) ? gt : -gt);
        g1.e[k] = from_f32<LT>((yy == 1) ? -gt : gt);
      }
    }
    if constexpr (HAS_GRAD) {
      LT* g0p = grad + (b * 2) * p.HW + i;
      vstore(g0p, g0);
      vstore(g0p + p.HW, g1);
    }
  }
  block_add_double(acc, loss_num);
}

// generic path: any C, any HW; one pixel per thread step, two sweeps over channels
template <typename LT, typename YT, bool HAS_GRAD>
__global__ void __launch_bounds__(kThreads)
wce_generic_kernel(const LT* __restrict__ logits, const YT* __restrict__ labels,
                   const float* __restrict__ weight, const int64_t* __restrict__ hist,
                   WceParams p, LT* __restrict__ grad, double* __restrict__ loss_num) {
  pdl_wait();
  pdl_launch();
  __shared__ float s_gs;
  if (threadIdx.x == 0) {
    const double D = wce_denominator(weight, hist, p.C, p.ignore_index);
    s_gs = (float)((double)p.grad_scale / D);
  }
  __syncthreads();
  const float gs = s_gs;
  const int64_t n = p.B * p.HW;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  float acc = 0.0f;
  for (int64_t idx = (int64_t)blockIdx.x * kThreads + threadIdx.x; idx < n; idx += stride) {
    const int64_t b = idx / p.HW, i = idx - b * p.HW;
    const LT* xp = logits + b * p.C * p.HW + i;
    const long long yy = (long long)labels[idx];
    const bool valid = (yy >= 0 && yy < p.C && yy != p.ignore_index);
    float m = -INFINITY;
    for (int c = 0; c < p.C; c++) m = fmaxf(m, to_f32(xp[(int64_t)c * p.HW]));
    float s = 0.0f;
    for (int c = 0; c < p.C; c++) s += expf(to_f32(xp[(int64_t)c * p.HW]) - m);
    const float lse = m + logf(s);
    float w = 0.0f;
    if (valid) {
      w = weight ? weight[yy] : 1.0f;
      acc += w * (lse - to_f32(xp[yy * p.HW]));
    }
    if constexpr (HAS_GRAD) {
      LT* gp = grad + b * p.C * p.HW + i;
      for (int c = 0; c < p.C; c++) {
        float g = 0.0f;
        if (valid) {
          const float pc = expf(to_f32(xp[(int64_t)c * p.HW]) - lse);
          g = w * (pc - (c == yy ? 1.0f : 0.0f)) * gs;
        }
        gp[(int64_t)c * p.HW] = from_f32<LT>(g);
      }
    }
  }
  block_add_double(acc, loss_num);
}

__global__ void wce_finalize_kernel(const double* loss_num, const float* weight,
                                    const int64_t* hist, int C, int ignore_index, float* loss) {
  pdl_wait();
  pdl_launch();
  const double D = wce_denominator(weight, hist, C, ignore_index);
  *loss = (float)(*loss_num / D);  // 0/0 -> nan, as PyTorch for an all-ignored batch
}

template <typename LT, typename YT>
static int launch_wce(const void* logits, const void* labels, const float* weight,
                      const int64_t* hist, const WceParams& p, void* grad, double* loss_num,
                      cudaStream_t st) {
  const LT* x = static_cast<const LT*>(logits);
  const YT* y = static_cast<const YT*>(labels);
  LT* g = static_cast<LT*>(grad);
  constexpr int VEC = 16 / sizeof(LT);
  const bool vec_ok = p.C == 2 && (p.HW % VEC == 0) &&
                      ((reinterpret_cast<uintptr_t>(x) & 15) == 0) &&
                      ((reinterpret_cast<uintptr_t>(y) % (sizeof(YT) * VEC >= 16 ? 16 : sizeof(YT) * VEC)) == 0) &&
                      (g == nullptr || (reinterpret_cast<uintptr_t>(g) & 15) == 0);
  if (vec_ok) {
    const int64_t nvec = p.B * (p.HW / VEC);
    const int cap = g ? resident_grid(wce2_kernel<LT, YT, true>, kThreads) : resident_grid(wce2_kernel<LT, YT, false>, kThreads);
    int grid = (int)std::min<int64_t>(std::max<int64_t>((nvec + kThreads - 1) / kThreads, 1), (int64_t)cap);
    if (g) launch_k(wce2_kernel<LT, YT, true>, dim3(grid), dim3(kThreads), 0, st, x, y, weight, hist, p, g, loss_num);
    else   launch_k(wce2_kernel<LT, YT, false>, dim3(grid), dim3(kThreads), 0, st, x, y, weight, hist, p, g, loss_num);
  } else {
    const int64_t n = p.B * p.HW;
    const int cap = g ? resident_grid(wce_generic_kernel<LT, YT, true>, kThreads) : resident_grid(wce_generic_kernel<LT, YT, false>, kThreads);
    int grid = (int)std::min<int64_t>(std::max<int64_t>((n + kThreads - 1) / kThreads, 1), (int64_t)cap);
    if (g) launch_k(wce_generic_kernel<LT, YT, true>, dim3(grid), dim3(kThreads), 0, st, x, y, weight, hist, p, g, loss_num);
    else   launch_k(wce_generic_kernel<LT, YT, false>, dim3(grid), dim3(kThreads), 0, st, x, y, weight, hist, p, g, loss_num);
  }
  return check_launch("wce_fwd_bwd");
}

// ---------------------------------------------------------------------------
// confusion matrix

template <typename TT, typename PT>
__global__ void __launch_bounds__(kThreads)
confusion2_kernel(const TT* __restrict__ tru, const PT* __restrict__ prd, int64_t n,
                  unsigned long long* __restrict__ cm) {
  pdl_wait();
  pdl_launch();
  // n_classes == 2: 4 cells + 1 "pred out of range" slot kept in registers
  constexpr int VEC = (sizeof(TT) >= sizeof(PT)) ? 16 / sizeof(TT) : 16 / sizeof(PT);
  unsigned cnt[5] = {0, 0, 0, 0, 0};
  const int64_t nvec = n / VEC;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  auto tally = [&](long long t, long long q) {
    const bool tv = (t == 0 || t == 1);
    const bool pv = (q == 0 || q == 1);
    const int cell = (int)(t * 2 + q);
#pragma unroll
    for (int k = 0; k < 4; k++) cnt[k] += (tv && pv && cell == k);
    cnt[4] += (tv && !pv);
  };
  int64_t v = (int64_t)blockIdx.x * kThreads + threadIdx.x;
  for (; v + stride < nvec; v += 2 * stride) {
    Vec<TT, VEC> t0, t1;
    Vec<PT, VEC> p0, p1;
    vload(t0, tru + v * VEC);
    vload(p0, prd + v * VEC);
    vload(t1, tru + (v + stride) * VEC);
    vload(p1, prd + (v + stride) * VEC);
#pragma unroll
    for (int i = 0; i < VEC; i++) tally((long long)t0.e[i], (long long)p0.e[i]);
#pragma unroll
    for (int i = 0; i < VEC; i++) tally((long long)t1.e[i], (long long)p1.e[i]);
  }
  for (; v < nvec; v += stride) {
    Vec<TT, VEC> t0;
    Vec<PT, VEC> p0;
    vload(t0, tru + v * VEC);
    vload(p0, prd + v * VEC);
#pragma unroll
    for (int i = 0; i < VEC; i++) tally((long long)t0.e[i], (long long)p0.e[i]);
  }
  if (blockIdx.x == 0)
    for (int64_t i = nvec * VEC + threadIdx.x; i < n; i += kThreads)
      tally((long long)tru[i], (long long)prd[i]);
  flush_counters<5>(cnt, 5, cm);
}

template <typename TT, typename PT>
__global__ void __launch_bounds__(kThreads)
confusion_generic_kernel(const TT* __restrict__ tru, const PT* __restrict__ prd, int64_t n,
                         int nc, unsigned long long* __restrict__ cm) {
  pdl_wait();
  pdl_launch();
  extern __shared__ unsigned s_cm[];
  const int cells = nc * nc + 1;
  for (int i = threadIdx.x; i < cells; i += kThreads) s_cm[i] = 0;
  __syncthreads();
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  for (int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x; i < n; i += stride) {
    const long long t = (long long)tru[i], q = (long long)prd[i];
    const bool tv = (t >= 0 && t < nc);
    const unsigned active = __ballot_sync(__activemask(), tv);
    if (tv) {
      const int cell = (q >= 0 && q < nc) ? (int)(t * nc + q) : nc * nc;
      const unsigned peers = __match_any_sync(active, cell);
      if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&s_cm[cell], (unsigned)__popc(peers));
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < cells; i += kThreads)
    if (s_cm[i]) atomicAdd(cm + i, (unsigned long long)s_cm[i]);
}

template <typename TT, typename PT>
static int launch_confusion(const void* tru, const void* prd, int64_t n, int nc, int64_t* cm,
                            cudaStream_t st) {
  const TT* t = static_cast<const TT*>(tru);
  const PT* q = static_cast<const PT*>(prd);
  auto* c = reinterpret_cast<unsigned long long*>(cm);
  constexpr int VEC = (sizeof(TT) >= sizeof(PT)) ? 16 / sizeof(TT) : 16 / sizeof(PT);
  const bool aligned = (reinterpret_cast<uintptr_t>(t) % (sizeof(TT) * VEC) == 0) &&
                       (reinterpret_cast<uintptr_t>(q) % (sizeof(PT) * VEC) == 0);
  if (nc == 2 && aligned) {
    int64_t want = (n / VEC + kThreads * 2 - 1) / (kThreads * 2);
    int grid = (int)std::min<int64_t>(std::max<int64_t>(want, 1), (int64_t)resident_grid(confusion2_kernel<TT, PT>, kThreads));
    launch_k(confusion2_kernel<TT, PT>, dim3(grid), dim3(kThreads), 0, st, t, q, n, c);
  } else {
    int64_t want = (n + kThreads * 8 - 1) / (kThreads * 8);
    int grid = (int)std::min<int64_t>(std::max<int64_t>(want, 1), (int64_t)resident_grid(confusion_generic_kernel<TT, PT>, kThreads, (nc * nc + 1) * sizeof(unsigned)));
    launch_k(confusion_generic_kernel<TT, PT>, dim3(grid), dim3(kThreads), (nc * nc + 1) * sizeof(unsigned), st, t, q, n, nc, c);
  }
  return check_launch("confusion");
}

// ---------------------------------------------------------------------------
// argmax / threshold fused with confusion matrix

template <typename LT, typename TT>
__global__ void __launch_bounds__(kThreads)
argmax_confusion_kernel(const LT* __restrict__ logits, const TT* __restrict__ tru, int64_t B,
                        int C, int64_t HW, int mode, float threshold,
                        uint8_t* __restrict__ pred_out, uint8_t* __restrict__ conf_out,
                        unsigned long long* __restrict__ cm) {
  pdl_wait();
  pdl_launch();
  extern __shared__ unsigned s_cm[];
  const int cells = C * C + 1;
  if (cm) {
    for (int i = threadIdx.x; i < cells; i += kThreads) s_cm[i] = 0;
    __syncthreads();
  }
  const int64_t n = B * HW;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  for (int64_t idx = (int64_t)blockIdx.x * kThreads + threadIdx.x; idx < n; idx += stride) {
    const int64_t b = idx / HW, i = idx - b * HW;
    const LT* xp = logits + b * C * HW + i;
    int pred = 0;
    float p1 = 0.0f;
    if (mode == 0) {
      float best = to_f32(xp[0]);
      for (int c = 1; c < C; c++) {
        const float v = to_f32(xp[(int64_t)c * HW]);
        if (v > best) { best = v; pred = c; }  // strict: first maximum wins (torch.max)
      }
    } else {
      float m = -INFINITY;
      for (int c = 0; c < C; c++) m = fmaxf(m, to_f32(xp[(int64_t)c * HW]));
      float s = 0.0f;
      for (int c = 0; c < C; c++) s += expf(to_f32(xp[(int64_t)c * HW]) - m);
      p1 = expf(to_f32(xp[HW]) - m) / s;
      pred = (p1 > threshold) ? 1 : 0;
    }
    if (pred_out) pred_out[idx] = (uint8_t)pred;
    if (conf_out) conf_out[idx] = (uint8_t)(p1 * 255.0f);  // truncation, as ndarray.astype(uint8)
    if (cm) {
      const long long t = (long long)tru[idx];
      const bool tv = (t >= 0 && t < C);
      const unsigned active = __ballot_sync(__activemask(), tv);
      if (tv) {
        const int cell = (int)(t * C + pred);
        const unsigned peers = __match_any_sync(active, cell);
        if ((int)(threadIdx.x & 31) == __ffs(peers) - 1) atomicAdd(&s_cm[cell], (unsigned)__popc(peers));
      }
    }
  }
  if (cm) {
    __syncthreads();
    for (int i = threadIdx.x; i < cells; i += kThreads)
      if (s_cm[i]) atomicAdd(cm + i, (unsigned long long)s_cm[i]);
  }
}

// two-class vectorised path: 16-byte loads on both logit planes, register counters
template <typename LT, typename TT, bool HAS_CM>
__global__ void __launch_bounds__(kThreads)
argmax_confusion2_kernel(const LT* __restrict__ logits, const TT* __restrict__ tru, int64_t B,
                         int64_t HW, int mode, float threshold, uint8_t* __restrict__ pred_out,
                         uint8_t* __restrict__ conf_out, unsigned long long* __restrict__ cm) {
  pdl_wait();
  pdl_launch();
  constexpr int VEC = 16 / sizeof(LT);
  unsigned cnt[4] = {0, 0, 0, 0};
  const int64_t vec_per_img = HW / VEC;
  const int64_t nvec = B * vec_per_img;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  for (int64_t v = (int64_t)blockIdx.x * kThreads + threadIdx.x; v < nvec; v += stride) {
    const int64_t b = v / vec_per_img;
    const int64_t i = (v - b * vec_per_img) * VEC;
    const LT* x0p = logits + (b * 2) * HW + i;
    Vec<LT, VEC> x0, x1;
    vload(x0, x0p);
    vload(x1, x0p + HW);
    Vec<TT, VEC> t;
    if constexpr (HAS_CM) vload(t, tru + b * HW + i);
    Vec<uint8_t, VEC> po, co;
#pragma unroll
    for (int k = 0; k < VEC; k++) {
      const float a0 = to_f32(x0.e[k]), a1 = to_f32(x1.e[k]);
      int pred;
      float p1 = 0.0f;
      if (mode == 0) {
        pred = (a1 > a0) ? 1 : 0;
      } else {
        const float m = fmaxf(a0, a1);
        const float e0 = expf(a0 - m), e1 = expf(a1 - m);
        p1 = e1 / (e0 + e1);
        pred = (p1 > threshold) ? 1 : 0;
      }
      po.e[k] = (uint8_t)pred;
      co.e[k] = (uint8_t)(p1 * 255.0f);
      if constexpr (HAS_CM) {
        const long long tt = (long long)t.e[k];
        const bool tv = (tt == 0 || tt == 1);
        const int cell = (int)(tt * 2 + pred);
#pragma unroll
        for (int c = 0; c < 4; c++) cnt[c] += (tv && cell == c);
      }
    }
    if (pred_out) vstore(pred_out + b * HW + i, po);
    if (conf_out) vstore(conf_out + b * HW + i, co);
  }
  if constexpr (HAS_CM) flush_counters<4>(cnt, 4, cm);
}

template <typename LT, typename TT>
static int launch_argmax_confusion(const void* logits, const void* tru, int64_t B, int C,
                                   int64_t HW, int mode, float threshold, uint8_t* pred_out,
                                   uint8_t* conf_out, int64_t* cm, cudaStream_t st) {
  const LT* x = static_cast<const LT*>(logits);
  const TT* t = static_cast<const TT*>(tru);
  auto* c = reinterpret_cast<unsigned long long*>(cm);
  constexpr int VEC = 16 / sizeof(LT);
  const bool has_cm = (cm != nullptr && tru != nullptr);
  const bool vec_ok = C == 2 && (HW % VEC == 0) && ((reinterpret_cast<uintptr_t>(x) & 15) == 0) &&
                      (!has_cm || (reinterpret_cast<uintptr_t>(t) % (sizeof(TT) * VEC >= 16 ? 16 : sizeof(TT) * VEC)) == 0) &&
                      (pred_out == nullptr || (reinterpret_cast<uintptr_t>(pred_out) % VEC) == 0) &&
                      (conf_out == nullptr || (reinterpret_cast<uintptr_t>(conf_out) % VEC) == 0);
  if (vec_ok) {
    const int64_t nvec = B * (HW / VEC);
    const int cap = has_cm ? resident_grid(argmax_confusion2_kernel<LT, TT, true>, kThreads) : resident_grid(argmax_confusion2_kernel<LT, TT, false>, kThreads);
    int grid = (int)std::min<int64_t>(std::max<int64_t>((nvec + kThreads - 1) / kThreads, 1), (int64_t)cap);
    if (has_cm)
      launch_k(argmax_confusion2_kernel<LT, TT, true>, dim3(grid), dim3(kThreads), 0, st, x, t, B, HW, mode, threshold, pred_out, conf_out, c);
    else
      launch_k(argmax_confusion2_kernel<LT, TT, false>, dim3(grid), dim3(kThreads), 0, st, x, t, B, HW, mode, threshold, pred_out, conf_out, c);
  } else {
    const int64_t n = B * HW;
    int grid = (int)std::min<int64_t>(std::max<int64_t>((n + kThreads - 1) / kThreads, 1),
                                      (int64_t)resident_grid(argmax_confusion_kernel<LT, TT>, kThreads, (C * C + 1) * sizeof(unsigned)));
    launch_k(argmax_confusion_kernel<LT, TT>, dim3(grid), dim3(kThreads), (C * C + 1) * sizeof(unsigned), st, 
        x, t, B, C, HW, mode, threshold, pred_out, conf_out, has_cm ? c : nullptr);
  }
  return check_launch("argmax_confusion");
}


// ---------------------------------------------------------------------------
// predict epilogue (SURVEY 8f rank 3): final bilinear x4 upsample of the low-resolution logits (network/utils.py:22)
// + 2-class softmax + threshold + uint8 confidence map (predict.py:262-290) + optional confusion matrix
// (evaluate_quantization.py:265-270) in ONE pass that writes uint8 maps only: the full-resolution fp32 logits
// (268 MB at 8 x 2 x 2048^2) are never materialised. Same arithmetic as logits_up_fwd followed by
// argmax_confusion2 (bil_mix / expf / divide in the same order), so the maps and counts are bit-identical.
// One grid row per output image row; a thread produces 4 consecutive pixels (one 32-bit store per map).
template <typename TT, bool HAS_CM>
__global__ void __launch_bounds__(kThreads)
predict_epilogue2_kernel(const float* __restrict__ lo, int Hi, int Wi, int Ho, int Wo, int mode, float threshold,
                         const TT* __restrict__ tru, uint8_t* __restrict__ pred_out,
                         uint8_t* __restrict__ conf_out, unsigned long long* __restrict__ cm) {
  pdl_wait();
  pdl_launch();
  const float sh = (float)Hi / (float)Ho, sw = (float)Wi / (float)Wo;
  const int ho = blockIdx.x % Ho, b = blockIdx.x / Ho;
  int y0, y1;
  float ly;
  bil_src(ho, sh, Hi, y0, y1, ly);
  const float2* r0 = reinterpret_cast<const float2*>(lo) + ((int64_t)b * Hi + y0) * Wi;   // NHWC, C == 2
  const float2* r1 = reinterpret_cast<const float2*>(lo) + ((int64_t)b * Hi + y1) * Wi;
  const int64_t row_off = ((int64_t)b * Ho + ho) * Wo;
  unsigned cnt[4] = {0, 0, 0, 0};
  const int nquad = Wo >> 2;                      // Wo % 4 == 0 (checked by the launcher)
  for (int qd = blockIdx.y * kThreads + threadIdx.x; qd < nquad; qd += gridDim.y * kThreads) {
    const int wo0 = qd << 2;
    Vec<TT, 4> t;
    if constexpr (HAS_CM) vload(t, tru + row_off + wo0);
    Vec<uint8_t, 4> po, co;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      int x0, x1;
      float lx;
      bil_src(wo0 + k, sw, Wi, x0, x1, lx);
      const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
      const float2 v00 = __ldg(r0 + x0), v01 = __ldg(r0 + x1), v10 = __ldg(r1 + x0), v11 = __ldg(r1 + x1);
      const float a0 = bil_mix(w00, v00.x, w01, v01.x, w10, v10.x, w11, v11.x);
      const float a1 = bil_mix(w00, v00.y, w01, v01.y, w10, v10.y, w11, v11.y);
      int pred;
      float p1 = 0.0f;
      if (mode == 0) {
        pred = (a1 > a0) ? 1 : 0;
      } else {
        const float m = fmaxf(a0, a1);
        const float e0 = expf(a0 - m), e1 = expf(a1 - m);
        p1 = e1 / (e0 + e1);
        pred = (p1 > threshold) ? 1 : 0;
      }
      po.e[k] = (uint8_t)pred;
      co.e[k] = (uint8_t)(p1 * 255.0f);
      if constexpr (HAS_CM) {
        const long long tt = (long long)t.e[k];
        const bool tv = (tt == 0 || tt == 1);
        const int cell = (int)(tt * 2 + pred);
#pragma unroll
        for (int c = 0; c < 4; c++) cnt[c] += (tv && cell == c);
      }
    }
    if (pred_out) vstore(pred_out + row_off + wo0, po);
    if (conf_out) vstore(conf_out + row_off + wo0, co);
  }
  if constexpr (HAS_CM) flush_counters<4>(cnt, 4, cm);
}

template <typename TT>
static int launch_predict_epilogue(const float* lo, const void* tru, int B, int Hi, int Wi, int Ho, int Wo, int mode,
                                   float threshold, uint8_t* pred_out, uint8_t* conf_out, int64_t* cm, cudaStream_t st) {
  const TT* t = static_cast<const TT*>(tru);
  auto* c = reinterpret_cast<unsigned long long*>(cm);
  const bool has_cm = (cm != nullptr && tru != nullptr);
  dim3 grid((unsigned)(B * Ho), (unsigned)std::max(1, std::min(8, (Wo / 4 + kThreads - 1) / kThreads)));
  if (has_cm)
    launch_k(predict_epilogue2_kernel<TT, true>, grid, dim3(kThreads), 0, st, lo, Hi, Wi, Ho, Wo, mode, threshold, t, pred_out, conf_out, c);
  else
    launch_k(predict_epilogue2_kernel<TT, false>, grid, dim3(kThreads), 0, st, lo, Hi, Wi, Ho, Wo, mode, threshold, t, pred_out, conf_out, c);
  return check_launch("predict_epilogue");
}

// ---------------------------------------------------------------------------
// focal loss (utils/loss.py:14-35), forward + backward in one pass, any C:
//   ce_i = w[y_i] * nll_i (0 where ignored);  pt = exp(-ce_i);  focal_i = alpha * (1 - pt)^gamma * ce_i
//   loss = sum_i focal_i * (size_average ? 1/N : 1) with N = ALL pixels (ignored ones included, as `.mean()` does)
//   d focal / d ce = alpha * ((1 - pt)^gamma + gamma * ce * (1 - pt)^(gamma - 1) * pt)
template <typename LT, typename YT, bool HAS_GRAD>
__global__ void __launch_bounds__(kThreads)
focal_kernel(const LT* __restrict__ logits, const YT* __restrict__ labels, const float* __restrict__ weight,
             WceParams p, float alpha, float gamma, float out_scale, LT* __restrict__ grad,
             double* __restrict__ loss_num) {
  pdl_wait();
  pdl_launch();
  const int64_t n = p.B * p.HW;
  const int64_t stride = (int64_t)gridDim.x * kThreads;
  float acc = 0.0f;
  for (int64_t idx = (int64_t)blockIdx.x * kThreads + threadIdx.x; idx < n; idx += stride) {
    const int64_t b = idx / p.HW, i = idx - b * p.HW;
    const LT* xp = logits + b * p.C * p.HW + i;
    const long long yy = (long long)labels[idx];
    const bool valid = (yy >= 0 && yy < p.C && yy != p.ignore_index);
    float m = -INFINITY;
    for (int c = 0; c < p.C; c++) m = fmaxf(m, to_f32(xp[(int64_t)c * p.HW]));
    float s = 0.0f;
    for (int c = 0; c < p.C; c++) s += expf(to_f32(xp[(int64_t)c * p.HW]) - m);
    const float lse = m + logf(s);
    float w = 0.0f, dfdce = 0.0f;
    if (valid) {
      w = weight ? weight[yy] : 1.0f;
      const float ce = w * (lse - to_f32(xp[yy * p.HW]));
      const float pt = expf(-ce);
      const float om = 1.0f - pt;
      const float mod = (gamma == 0.0f) ? 1.0f : powf(om, gamma);
      acc += alpha * mod * ce;
      // gamma * ce * om^(gamma-1) * pt, written as gamma * ce * pt * mod / om (om > 0 whenever ce > 0)
      dfdce = alpha * (mod + ((gamma == 0.0f || om <= 0.0f) ? 0.0f : gamma * ce * pt * mod / om));
    }
    if constexpr (HAS_GRAD) {
      LT* gp = grad + b * p.C * p.HW + i;
      for (int c = 0; c < p.C; c++) {
        float g = 0.0f;
        if (valid) {
          const float pc = expf(to_f32(xp[(int64_t)c * p.HW]) - lse);
          g = dfdce * w * (pc - (c == yy ? 1.0f : 0.0f)) * out_scale;
        }
        gp[(int64_t)c * p.HW] = from_f32<LT>(g);
      }
    }
  }
  block_add_double(acc, loss_num);
}

__global__ void focal_finalize_kernel(const double* loss_num, float out_scale, float* loss) {
  pdl_wait();
  pdl_launch();
  *loss = (float)(*loss_num * (double)out_scale);
}

template <typename LT, typename YT>
static int launch_focal(const void* logits, const void* labels, const float* weight, const WceParams& p, float alpha,
                        float gamma, float out_scale, void* grad, double* loss_num, cudaStream_t st) {
  const LT* x = static_cast<const LT*>(logits);
  const YT* y = static_cast<const YT*>(labels);
  LT* g = static_cast<LT*>(grad);
  const int64_t n = p.B * p.HW;
  const int cap = g ? resident_grid(focal_kernel<LT, YT, true>, kThreads) : resident_grid(focal_kernel<LT, YT, false>, kThreads);
  int grid = (int)std::min<int64_t>(std::max<int64_t>((n + kThreads - 1) / kThreads, 1), (int64_t)cap);
  if (g) launch_k(focal_kernel<LT, YT, true>, dim3(grid), dim3(kThreads), 0, st, x, y, weight, p, alpha, gamma, out_scale, g, loss_num);
  else   launch_k(focal_kernel<LT, YT, false>, dim3(grid), dim3(kThreads), 0, st, x, y, weight, p, alpha, gamma, out_scale, g, loss_num);
  return check_launch("focal_fwd_bwd");
}

}  // namespace iswm

// ---------------------------------------------------------------------------
// C ABI
using namespace iswm;

#define DISPATCH_LABEL(dt, FN, ...)                                    \
  switch (dt) {                                                        \
    case ISWM_U8:  return FN<uint8_t>(__VA_ARGS__);                    \
    case ISWM_I32: return FN<int32_t>(__VA_ARGS__);                    \
    case ISWM_I64: return FN<int64_t>(__VA_ARGS__);                    \
    default: set_error("bad label dtype %d", dt); return 2;            \
  }

extern "C" int iswm_class_hist(const void* d_labels, int label_dtype, int64_t n, int n_classes,
                               int64_t* d_hist, void* stream) {
  ISWM_REQUIRE(n >= 0 && n_classes >= 1 && n_classes <= 8192, "class_hist: bad sizes n=%lld C=%d", (long long)n, n_classes);
  ISWM_REQUIRE(d_hist != nullptr, "class_hist: null hist");
  if (n == 0) return 0;
  ISWM_REQUIRE(d_labels != nullptr, "class_hist: null labels");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  DISPATCH_LABEL(label_dtype, launch_class_hist, d_labels, n, n_classes, d_hist, st);
}

template <typename LT>
static int wce_dispatch_label(int label_dtype, const void* logits, const void* labels,
                              const float* weight, const int64_t* hist, const WceParams& p,
                              void* grad, double* loss_num, cudaStream_t st) {
  switch (label_dtype) {
    case ISWM_U8:  return launch_wce<LT, uint8_t>(logits, labels, weight, hist, p, grad, loss_num, st);
    case ISWM_I32: return launch_wce<LT, int32_t>(logits, labels, weight, hist, p, grad, loss_num, st);
    case ISWM_I64: return launch_wce<LT, int64_t>(logits, labels, weight, hist, p, grad, loss_num, st);
    default: set_error("bad label dtype %d", label_dtype); return 2;
  }
}

extern "C" int iswm_wce_fwd_bwd(const void* d_logits, int logit_dtype, const void* d_labels,
                                int label_dtype, const float* d_weight, const int64_t* d_hist,
                                int64_t B, int C, int64_t HW, int ignore_index, float grad_scale,
                                void* d_grad, double* d_loss_num, float* d_loss, void* stream) {
  ISWM_REQUIRE(B >= 0 && HW >= 0 && C >= 1 && C <= 8192, "wce: bad sizes");
  ISWM_REQUIRE(d_hist && d_loss_num, "wce: null hist / loss_num");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  WceParams p{B, HW, C, ignore_index, grad_scale};
  if (B * HW > 0) {
    ISWM_REQUIRE(d_logits && d_labels, "wce: null logits / labels");
    int rc;
    if (logit_dtype == ISWM_F32)
      rc = wce_dispatch_label<float>(label_dtype, d_logits, d_labels, d_weight, d_hist, p, d_grad, d_loss_num, st);
    else if (logit_dtype == ISWM_BF16)
      rc = wce_dispatch_label<__nv_bfloat16>(label_dtype, d_logits, d_labels, d_weight, d_hist, p, d_grad, d_loss_num, st);
    else { set_error("bad logit dtype %d", logit_dtype); return 2; }
    if (rc) return rc;
  }
  if (d_loss) {
    launch_k(wce_finalize_kernel, dim3(1), dim3(1), 0, st, d_loss_num, d_weight, d_hist, C, ignore_index, d_loss);
    return check_launch("wce_finalize");
  }
  return 0;
}

template <typename TT>
static int confusion_dispatch_pred(int pred_dtype, const void* t, const void* q, int64_t n, int nc,
                                   int64_t* cm, cudaStream_t st) {
  switch (pred_dtype) {
    case ISWM_U8:  return launch_confusion<TT, uint8_t>(t, q, n, nc, cm, st);
    case ISWM_I32: return launch_confusion<TT, int32_t>(t, q, n, nc, cm, st);
    case ISWM_I64: return launch_confusion<TT, int64_t>(t, q, n, nc, cm, st);
    default: set_error("bad pred dtype %d", pred_dtype); return 2;
  }
}

extern "C" int iswm_confusion(const void* d_true, int true_dtype, const void* d_pred,
                              int pred_dtype, int64_t n, int n_classes, int64_t* d_cm,
                              void* stream) {
  ISWM_REQUIRE(n >= 0 && n_classes >= 1 && n_classes <= 100, "confusion: bad sizes");
  ISWM_REQUIRE(d_cm, "confusion: null cm");
  if (n == 0) return 0;
  ISWM_REQUIRE(d_true && d_pred, "confusion: null inputs");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (true_dtype) {
    case ISWM_U8:  return confusion_dispatch_pred<uint8_t>(pred_dtype, d_true, d_pred, n, n_classes, d_cm, st);
    case ISWM_I32: return confusion_dispatch_pred<int32_t>(pred_dtype, d_true, d_pred, n, n_classes, d_cm, st);
    case ISWM_I64: return confusion_dispatch_pred<int64_t>(pred_dtype, d_true, d_pred, n, n_classes, d_cm, st);
    default: set_error("bad true dtype %d", true_dtype); return 2;
  }
}

template <typename LT>
static int amc_dispatch(int true_dtype, const void* logits, const void* tru, int64_t B, int C,
                        int64_t HW, int mode, float thr, uint8_t* po, uint8_t* co, int64_t* cm,
                        cudaStream_t st) {
  switch (true_dtype) {
    case ISWM_U8:  return launch_argmax_confusion<LT, uint8_t>(logits, tru, B, C, HW, mode, thr, po, co, cm, st);
    case ISWM_I32: return launch_argmax_confusion<LT, int32_t>(logits, tru, B, C, HW, mode, thr, po, co, cm, st);
    case ISWM_I64: return launch_argmax_confusion<LT, int64_t>(logits, tru, B, C, HW, mode, thr, po, co, cm, st);
    default: set_error("bad true dtype %d", true_dtype); return 2;
  }
}

extern "C" int iswm_argmax_confusion(const void* d_logits, int logit_dtype, const void* d_true,
                                     int true_dtype, int64_t B, int C, int64_t HW, int mode,
                                     float threshold, uint8_t* d_pred_out, uint8_t* d_conf_out,
                                     int64_t* d_cm, void* stream) {
  ISWM_REQUIRE(B >= 0 && HW >= 0 && C >= 1 && C <= 100, "argmax_confusion: bad sizes");
  ISWM_REQUIRE(mode == 0 || (mode == 1 && C >= 2), "argmax_confusion: bad mode %d for C=%d", mode, C);
  if (B * HW == 0) return 0;
  ISWM_REQUIRE(d_logits, "argmax_confusion: null logits");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (logit_dtype == ISWM_F32)
    return amc_dispatch<float>(true_dtype, d_logits, d_true, B, C, HW, mode, threshold, d_pred_out, d_conf_out, d_cm, st);
  if (logit_dtype == ISWM_BF16)
    return amc_dispatch<__nv_bfloat16>(true_dtype, d_logits, d_true, B, C, HW, mode, threshold, d_pred_out, d_conf_out, d_cm, st);
  set_error("bad logit dtype %d", logit_dtype);
  return 2;
}

extern "C" int iswm_predict_epilogue(const float* d_lo, int B, int Hi, int Wi, int C, int Ho, int Wo, int mode,
                                     float threshold, const void* d_true, int true_dtype, uint8_t* d_pred_out,
                                     uint8_t* d_conf_out, int64_t* d_cm, void* stream) {
  ISWM_REQUIRE(d_lo && B >= 0 && Hi >= 1 && Wi >= 1 && Ho >= 1 && Wo >= 1, "predict_epilogue: bad sizes");
  ISWM_REQUIRE(C == 2, "predict_epilogue: the fused path is the reference's two-class case (C=%d); use logits_up_fwd + argmax_confusion", C);
  ISWM_REQUIRE(mode == 0 || mode == 1, "predict_epilogue: bad mode %d", mode);
  ISWM_REQUIRE((Wo & 3) == 0, "predict_epilogue: output width %d must be a multiple of 4", Wo);
  ISWM_REQUIRE((reinterpret_cast<uintptr_t>(d_lo) & 7) == 0, "predict_epilogue: logits must be 8-byte aligned");
  ISWM_REQUIRE(!d_pred_out || (reinterpret_cast<uintptr_t>(d_pred_out) & 3) == 0, "predict_epilogue: pred map must be 4-byte aligned");
  ISWM_REQUIRE(!d_conf_out || (reinterpret_cast<uintptr_t>(d_conf_out) & 3) == 0, "predict_epilogue: confidence map must be 4-byte aligned");
  ISWM_REQUIRE((int64_t)B * Ho < (1ll << 31), "predict_epilogue: too many rows");
  if (B == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (d_true && d_cm) {
    const size_t esz = true_dtype == ISWM_U8 ? 1 : (true_dtype == ISWM_I32 ? 4 : 8);
    ISWM_REQUIRE((reinterpret_cast<uintptr_t>(d_true) % (esz * 4 >= 16 ? 16 : esz * 4)) == 0, "predict_epilogue: labels must be aligned to 4 elements");
  }
  switch (true_dtype) {
    case ISWM_U8:  return launch_predict_epilogue<uint8_t>(d_lo, d_true, B, Hi, Wi, Ho, Wo, mode, threshold, d_pred_out, d_conf_out, d_cm, st);
    case ISWM_I32: return launch_predict_epilogue<int32_t>(d_lo, d_true, B, Hi, Wi, Ho, Wo, mode, threshold, d_pred_out, d_conf_out, d_cm, st);
    case ISWM_I64: return launch_predict_epilogue<int64_t>(d_lo, d_true, B, Hi, Wi, Ho, Wo, mode, threshold, d_pred_out, d_conf_out, d_cm, st);
    default: set_error("bad true dtype %d", true_dtype); return 2;
  }
}

template <typename LT>
static int focal_dispatch_label(int label_dtype, const void* logits, const void* labels, const float* weight,
                                const WceParams& p, float alpha, float gamma, float out_scale, void* grad,
                                double* loss_num, cudaStream_t st) {
  switch (label_dtype) {
    case ISWM_U8:  return launch_focal<LT, uint8_t>(logits, labels, weight, p, alpha, gamma, out_scale, grad, loss_num, st);
    case ISWM_I32: return launch_focal<LT, int32_t>(logits, labels, weight, p, alpha, gamma, out_scale, grad, loss_num, st);
    case ISWM_I64: return launch_focal<LT, int64_t>(logits, labels, weight, p, alpha, gamma, out_scale, grad, loss_num, st);
    default: set_error("bad label dtype %d", label_dtype); return 2;
  }
}

extern "C" int iswm_focal_fwd_bwd(const void* d_logits, int logit_dtype, const void* d_labels, int label_dtype,
                                  const float* d_weight, int64_t B, int C, int64_t HW, int ignore_index,
                                  float alpha, float gamma, int size_average, void* d_grad, double* d_loss_num,
                                  float* d_loss, void* stream) {
  ISWM_REQUIRE(B >= 0 && HW >= 0 && C >= 1 && C <= 8192, "focal: bad sizes");
  ISWM_REQUIRE(d_loss_num, "focal: null loss_num");
  ISWM_REQUIRE(gamma >= 0.f, "focal: gamma=%f must be >= 0", (double)gamma);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  WceParams p{B, HW, C, ignore_index, 1.0f};
  const int64_t n = B * HW;
  // mean over ALL pixels: an empty input is 0/0 = nan, as torch's .mean() of an empty tensor
  const float out_scale = size_average ? (float)(1.0 / (double)n) : 1.0f;
  if (n > 0) {
    ISWM_REQUIRE(d_logits && d_labels, "focal: null logits / labels");
    int rc;
    if (logit_dtype == ISWM_F32)
      rc = focal_dispatch_label<float>(label_dtype, d_logits, d_labels, d_weight, p, alpha, gamma, out_scale, d_grad, d_loss_num, st);
    else if (logit_dtype == ISWM_BF16)
      rc = focal_dispatch_label<__nv_bfloat16>(label_dtype, d_logits, d_labels, d_weight, p, alpha, gamma, out_scale, d_grad, d_loss_num, st);
    else { set_error("bad logit dtype %d", logit_dtype); return 2; }
    if (rc) return rc;
  }
  if (d_loss) {
    launch_k(focal_finalize_kernel, dim3(1), dim3(1), 0, st, d_loss_num, n > 0 ? out_scale : NAN, d_loss);
    return check_launch("focal_finalize");
  }
  return 0;
}
