// stem_pool.cu — BatchNorm + ReLU + 3x3/s2 max pooling of the ResNet stem as ONE forward pass
// (network/backbone/resnet.py:145-147: bn1 -> relu -> maxpool after the 7x7 convolution).
//
// Unfused, the 64-channel half-resolution stem activation (134 MB at cfg2) is written by the BatchNorm pass and read by the
// pooling pass. Here the forward reads the pre-BN convolution output (each element up to 4 times, from L1/L2), normalises +
// ReLUs on the fly, writes the pooled tensor and the per-channel argmax code (which of the 9 window positions won: first
// maximum in window order, the rule of maxpool_fwd_kernel): the activation never exists. Same arithmetic as bn_train_apply
// and maxpool_fwd run one after the other (the pooled values and codes are bit-identical). The backward runs maxpool_bwd,
// bn_bwd_reduce and bn_bwd_apply on the argmax codes.
#include "common.cuh"
#include "ew_common.cuh"
#include <math.h>

namespace iswm {

constexpr int kC = 64;          // stem width (8 channel groups of 8)

struct StemBn {
  const double* stats;          // sum x, sum x^2 over the M stem pixels, `stats_rep` copies
  int stats_rep;
  const float* gamma;
  const float* beta;
  float* running_mean;
  float* running_var;
  long long* nbt;
  float* save_mean;             // written for the backward's BatchNorm kernels
  float* save_invstd;
};

__device__ __forceinline__ float bn_relu_bf16(float x, float sc, float sh) {
  // what bn_train_apply stores: relu(fma(x, sc, sh)) rounded to bf16
  return __bfloat162float(__float2bfloat16_rn(fmaxf(fmaf(x, sc, sh), 0.f)));
}

// GCNT (synchronised BatchNorm): bn.stats holds the sums over every rank's pixels (one copy) followed by the global pixel
// count at [2C]; M only describes this rank's tensor
template <bool GCNT>
__global__ void __launch_bounds__(kT)
stem_pool_fwd_kernel(const __nv_bfloat16* __restrict__ raw, StemBn bn, int B, int H, int W, int Ho, int Wo, int64_t M,
                     float eps, float momentum, __nv_bfloat16* __restrict__ out, uint8_t* __restrict__ idx) {
  pdl_wait();
  pdl_launch();
  __shared__ double s_stat[2 * kC];
  for (int i = threadIdx.x; i < 2 * kC; i += kT) {
    double a = bn.stats[i];
    for (int r = 1; r < bn.stats_rep; r++) a += bn.stats[(size_t)r * 2 * kC + i];
    s_stat[i] = a;
  }
  __syncthreads();
  const int cg = threadIdx.x & 7;                       // kT and the grid stride are multiples of 8: a thread keeps its channels
  const int c0 = cg << 3;
  const double cnt = GCNT ? bn.stats[2 * kC] : 0.0;
  const double invM = GCNT ? 1.0 / cnt : 1.0 / (double)M;
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const int c = c0 + j;
    const double mean_d = s_stat[c] * invM;
    const float mean = (float)mean_d;
    const float var = fmaxf((float)(s_stat[kC + c] * invM - mean_d * mean_d), 0.f);
    const float invstd = rsqrtf(var + eps);
    sc[j] = bn.gamma[c] * invstd;
    sh[j] = fmaf(-mean, sc[j], bn.beta[c]);
    if (blockIdx.x == 0 && threadIdx.x < 8) {
      bn.save_mean[c] = mean;
      bn.save_invstd[c] = invstd;
      if (bn.running_mean) {
        float unbiased;
        if (GCNT) unbiased = (cnt > 1.0) ? var * ((float)cnt / (float)(cnt - 1.0)) : var;
        else unbiased = (M > 1) ? var * ((float)M / (float)(M - 1)) : var;
        bn.running_mean[c] = (1.f - momentum) * bn.running_mean[c] + momentum * mean;
        bn.running_var[c] = (1.f - momentum) * bn.running_var[c] + momentum * unbiased;
      }
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && bn.nbt) *bn.nbt += 1;
  const int64_t total = (int64_t)B * Ho * Wo * 8;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int64_t m = i >> 3;
    const int wo = (int)(m % Wo), ho = (int)((m / Wo) % Ho), b = (int)(m / ((int64_t)Wo * Ho));
    const __nv_bfloat16* img = raw + (int64_t)b * H * W * kC + c0;
    uint4 ld[9];
    bool ok[9];
#pragma unroll
    for (int r = 0; r < 3; r++) {
      const int hi = 2 * ho + r - 1;
      const int hc = min(max(hi, 0), H - 1);
#pragma unroll
      for (int s2 = 0; s2 < 3; s2++) {
        const int wi = 2 * wo + s2 - 1;
        const int wc = min(max(wi, 0), W - 1);
        ok[r * 3 + s2] = (hi >= 0 && hi < H && wi >= 0 && wi < W);
        ld[r * 3 + s2] = load_raw(img + ((int64_t)hc * W + wc) * kC);
      }
    }
    float best[8];
    int arg[8];
#pragma unroll
    for (int j = 0; j < 8; j++) { best[j] = -INFINITY; arg[j] = 0; }
#pragma unroll
    for (int t = 0; t < 9; t++) {
      if (!ok[t]) continue;
      const F8 v = unpack8(ld[t]);
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const float y = bn_relu_bf16(v.v[j], sc[j], sh[j]);
        if (y > best[j]) { best[j] = y; arg[j] = t; }
      }
    }
    F8 o;
#pragma unroll
    for (int j = 0; j < 8; j++) o.v[j] = best[j];
    store8(out + m * kC + c0, o);
    uint2 pk;
    pk.x = arg[0] | (arg[1] << 8) | (arg[2] << 16) | (arg[3] << 24);
    pk.y = arg[4] | (arg[5] << 8) | (arg[6] << 16) | (arg[7] << 24);
    *reinterpret_cast<uint2*>(idx + m * kC + c0) = pk;
  }
}

}  // namespace iswm

using namespace iswm;

#define ST(s) static_cast<cudaStream_t>(s)
#define BF(p) static_cast<const __nv_bfloat16*>(p)
#define BFW(p) static_cast<__nv_bfloat16*>(p)

static int stem_grid(int64_t work_items) {
  // grid-stride over (pixel, channel group) items; a multiple of 8 threads per block keeps a thread on its channel group
  const int64_t g = (work_items + kT - 1) / kT;
  return (int)std::max<int64_t>(1, std::min<int64_t>(g, (int64_t)num_sms() * 8));
}

static int stem_pool_fwd_impl(bool global, const void* d_raw, const iswm_bn_side* bn, int B, int H, int W, int C, int Ho, int Wo,
                              float eps, float momentum, void* d_out, uint8_t* d_idx, void* stream) {
  if (debug_skip(ISWM_SKIP_BN)) return 0;
  ISWM_REQUIRE(d_raw && bn && d_out && d_idx && bn->stats && bn->gamma && bn->beta && bn->save_mean && bn->save_invstd, "stem_pool_fwd: null argument");
  ISWM_REQUIRE(C == kC, "stem_pool_fwd: C=%d (the stem has %d channels)", C, kC);
  ISWM_REQUIRE(Ho == (H - 1) / 2 + 1 && Wo == (W - 1) / 2 + 1 && B >= 1, "stem_pool_fwd: 3x3 / stride 2 / pad 1 geometry expected");
  ISWM_REQUIRE(!global || bn->stats_replicas <= 1, "stem_pool_fwd_global: the global sums are one copy (stats_replicas=%d)", bn->stats_replicas);
  const StemBn sb{bn->stats, bn->stats_replicas > 1 ? bn->stats_replicas : 1, bn->gamma, bn->beta, bn->running_mean, bn->running_var,
                  reinterpret_cast<long long*>(bn->num_batches_tracked), bn->save_mean, bn->save_invstd};
  if (global)
    launch_k(stem_pool_fwd_kernel<true>, dim3(stem_grid((int64_t)B * Ho * Wo * 8)), dim3(kT), 0, ST(stream), BF(d_raw), sb, B, H, W, Ho, Wo,
             (int64_t)B * H * W, eps, momentum, BFW(d_out), d_idx);
  else
    launch_k(stem_pool_fwd_kernel<false>, dim3(stem_grid((int64_t)B * Ho * Wo * 8)), dim3(kT), 0, ST(stream), BF(d_raw), sb, B, H, W, Ho, Wo,
             (int64_t)B * H * W, eps, momentum, BFW(d_out), d_idx);
  return check_launch("stem_pool_fwd");
}

extern "C" int iswm_stem_pool_fwd(const void* d_raw, const iswm_bn_side* bn, int B, int H, int W, int C, int Ho, int Wo,
                                  float eps, float momentum, void* d_out, uint8_t* d_idx, void* stream) {
  return stem_pool_fwd_impl(false, d_raw, bn, B, H, W, C, Ho, Wo, eps, momentum, d_out, d_idx, stream);
}

extern "C" int iswm_stem_pool_fwd_global(const void* d_raw, const iswm_bn_side* bn, int B, int H, int W, int C, int Ho, int Wo,
                                         float eps, float momentum, void* d_out, uint8_t* d_idx, void* stream) {
  return stem_pool_fwd_impl(true, d_raw, bn, B, H, W, C, Ho, Wo, eps, momentum, d_out, d_idx, stream);
}
