// quant.cu — the FP8 (e4m3) inference path's kernels besides the convolution itself (iswm_b200/quant.py): per-output-channel
// weight quantisation into the packed operand of conv_igemm_f8_kernel, and the glue kernels at the boundaries between
// e4m3 activations and the parts of the network that stay bf16 (the stem, the pooled ASPP branch, the ASPP projection).
//
// An e4m3 activation q stands for q * s with one fp32 scale s per tensor. Every conversion to e4m3 here is
// cvt.rn.satfinite(x / s) with an IEEE fp32 division, so a host restatement (torch: (x / s).clamp(-448, 448) rounded to
// float8_e4m3fn) reproduces it bit for bit.
#include "common.cuh"
#include "ew_common.cuh"
#include <cuda_fp8.h>

namespace iswm {

__device__ __forceinline__ uint8_t to_e4m3(float x) {
  return (uint8_t)(__nv_cvt_float2_to_fp8x2(make_float2(x, 0.f), __NV_SATFINITE, __NV_E4M3) & 0xffu);
}
__device__ __forceinline__ float from_e4m3(uint8_t v) {
  const __half_raw h = __nv_cvt_fp8_to_halfraw((__nv_fp8_storage_t)v, __NV_E4M3);
  return __half2float(__half(h));
}
// 8 fp32 values / s -> 8 e4m3 bytes (one 8-byte store)
__device__ __forceinline__ uint2 quant8(const float* v, float s) {
  uint32_t w[2] = {0u, 0u};
#pragma unroll
  for (int j = 0; j < 8; j++) w[j >> 2] |= (uint32_t)to_e4m3(__fdiv_rn(v[j], s)) << (8 * (j & 3));
  return make_uint2(w[0], w[1]);
}

// one block per output channel: s_w[o] = amax_o / 448 (1 where the channel is all zero), then
// out[o][t][c] = e4m3(w[o][c][t] / s_w[o]) for c < Cin, 0 in the padding channels up to cin_pad
__global__ void __launch_bounds__(kT)
pack_weight_f8_kernel(const float* __restrict__ w, int Cin, int RS, int cin_pad, uint8_t* __restrict__ out, float* __restrict__ s_w) {
  pdl_wait();
  pdl_launch();
  const int o = blockIdx.x;
  const int n = Cin * RS;
  const float* wo = w + (int64_t)o * n;
  float m = 0.f;
  for (int i = threadIdx.x; i < n; i += kT) m = fmaxf(m, fabsf(wo[i]));
  __shared__ float red[kT / 32];
#pragma unroll
  for (int k = 16; k > 0; k >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, k));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = m;
  __syncthreads();
  m = red[0];
#pragma unroll
  for (int k = 1; k < kT / 32; k++) m = fmaxf(m, red[k]);
  const float s = (m > 0.f) ? __fdiv_rn(m, 448.f) : 1.f;
  if (threadIdx.x == 0) s_w[o] = s;
  uint8_t* dst = out + (int64_t)o * RS * cin_pad;
  for (int i = threadIdx.x; i < RS * cin_pad; i += kT) {
    const int t = i / cin_pad, c = i - t * cin_pad;
    dst[i] = (c < Cin) ? to_e4m3(__fdiv_rn(wo[c * RS + t], s)) : (uint8_t)0;
  }
}

// MaxPool2d(3, 2, 1) of the bf16 stem output straight into e4m3 (the first backbone activation); max commutes with the
// monotone rounding, so this equals rounding the bf16 maxpool's output
__global__ void __launch_bounds__(kT)
maxpool_fwd_f8_kernel(const __nv_bfloat16* __restrict__ x, int B, int H, int W, int C, int Ho, int Wo, float s, uint8_t* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int nvec = C >> 3;
  const int64_t total = (int64_t)B * Ho * Wo * nvec;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int cg = (int)(i % nvec);
    const int64_t m = i / nvec;
    const int wo = (int)(m % Wo), ho = (int)((m / Wo) % Ho), b = (int)(m / ((int64_t)Wo * Ho));
    float best[8];
#pragma unroll
    for (int j = 0; j < 8; j++) best[j] = -INFINITY;
    const __nv_bfloat16* img = x + (int64_t)b * H * W * C + cg * 8;
    for (int r = 0; r < 3; r++) {
      const int hi = 2 * ho + r - 1;
      if (hi < 0 || hi >= H) continue;
      for (int s2 = 0; s2 < 3; s2++) {
        const int wi = 2 * wo + s2 - 1;
        if (wi < 0 || wi >= W) continue;
        const F8 v = load8(img + ((int64_t)hi * W + wi) * C);
#pragma unroll
        for (int j = 0; j < 8; j++) best[j] = fmaxf(best[j], v.v[j]);
      }
    }
    *reinterpret_cast<uint2*>(out + m * C + cg * 8) = quant8(best, s);
  }
}

// AdaptiveAvgPool2d(1) of an e4m3 activation (scale s) -> bf16 [B, C]: out = bf16((sum_hw q) / HW * s). Block = (64-channel
// slice, image); 8 channel groups x 32 pixel rows per block, fixed-order tree over the rows.
__global__ void __launch_bounds__(kT)
gap_fwd_f8_kernel(const uint8_t* __restrict__ x, int x_ld, int64_t HW, int C, float s, __nv_bfloat16* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int g = threadIdx.x & 7, r = threadIdx.x >> 3;
  const int c0 = blockIdx.x * 64 + g * 8;
  const int b = blockIdx.y;
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; j++) acc[j] = 0.f;
  if (c0 < C) {
    for (int64_t p = r; p < HW; p += 32) {
      const uint2 v = *reinterpret_cast<const uint2*>(x + ((int64_t)b * HW + p) * x_ld + c0);
#pragma unroll
      for (int j = 0; j < 8; j++) acc[j] += from_e4m3((uint8_t)(((j < 4 ? v.x : v.y) >> (8 * (j & 3))) & 0xffu));
    }
  }
  __shared__ float red[32][65];
#pragma unroll
  for (int j = 0; j < 8; j++) red[r][g * 8 + j] = acc[j];
  __syncthreads();
  for (int h = 16; h > 0; h >>= 1) {
    if (r < h)
#pragma unroll
      for (int j = 0; j < 8; j++) red[r][g * 8 + j] += red[r + h][g * 8 + j];
    __syncthreads();
  }
  if (r == 0 && c0 < C)
#pragma unroll
    for (int j = 0; j < 8; j++) out[(int64_t)b * C + c0 + j] = __float2bfloat16_rn(red[0][g * 8 + j] / (float)HW * s);
}

// bf16 [B, C] broadcast over HW into an e4m3 channel slice (scale s): the pooled ASPP branch into the ASPP concat
__global__ void __launch_bounds__(kT)
broadcast_hw_f8_kernel(const __nv_bfloat16* __restrict__ x, int B, int64_t HW, int C, float s, uint8_t* __restrict__ out, int out_ld) {
  pdl_wait();
  pdl_launch();
  const int nvec = C >> 3;
  const int64_t total = (int64_t)B * HW * nvec;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int cg = (int)(i % nvec);
    const int64_t m = i / nvec;
    const int b = (int)(m / HW);
    const F8 v = load8(x + (int64_t)b * C + cg * 8);
    *reinterpret_cast<uint2*>(out + m * out_ld + cg * 8) = quant8(v.v, s);
  }
}

// F.interpolate(bilinear, align_corners=False) of a bf16 NHWC tensor into an e4m3 channel slice (scale s): the ASPP output
// into the decoder concat. Same source taps and expression as bilinear_fwd_kernel, then / s.
__global__ void __launch_bounds__(kT)
bilinear_fwd_f8_kernel(const __nv_bfloat16* __restrict__ x, int x_ld, int B, int Hi, int Wi, int C, int Ho, int Wo, float s,
                       uint8_t* __restrict__ out, int out_ld) {
  pdl_wait();
  pdl_launch();
  const int nvec = C >> 3;
  const float sh = (float)Hi / (float)Ho, sw = (float)Wi / (float)Wo;
  const int ho = blockIdx.x % Ho, b = blockIdx.x / Ho;
  int y0, y1;
  float ly;
  bil_src(ho, sh, Hi, y0, y1, ly);
  const __nv_bfloat16* r0 = x + ((int64_t)b * Hi + y0) * Wi * x_ld;
  const __nv_bfloat16* r1 = x + ((int64_t)b * Hi + y1) * Wi * x_ld;
  uint8_t* orow = out + ((int64_t)b * Ho + ho) * Wo * out_ld;
  const int total = Wo * nvec;
  for (int i = blockIdx.y * kT + threadIdx.x; i < total; i += gridDim.y * kT) {
    const int wo = i / nvec, c8 = (i - wo * nvec) << 3;
    int x0, x1;
    float lx;
    bil_src(wo, sw, Wi, x0, x1, lx);
    const F8 v00 = load8(r0 + (int64_t)x0 * x_ld + c8);
    const F8 v01 = load8(r0 + (int64_t)x1 * x_ld + c8);
    const F8 v10 = load8(r1 + (int64_t)x0 * x_ld + c8);
    const F8 v11 = load8(r1 + (int64_t)x1 * x_ld + c8);
    const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; j++) o[j] = w00 * v00.v[j] + w01 * v01.v[j] + w10 * v10.v[j] + w11 * v11.v[j];
    *reinterpret_cast<uint2*>(orow + (int64_t)wo * out_ld + c8) = quant8(o, s);
  }
}

// stride-2 helpers over one-byte elements, 16 channels per access: phase split (phases = 4: out[(p*2+q)][b][i][j] =
// x[b][2i+p][2j+q], zero beyond the image) and subsampling (phases = 1: out[b][i][j] = x[b][2i][2j])
__global__ void __launch_bounds__(kT)
phase_split_b8_kernel(const uint8_t* __restrict__ x, int x_ld, int B, int H, int W, int C, int Hp, int Wp, int phases,
                      uint8_t* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int nvec = C >> 4;
  const int64_t total = (int64_t)phases * B * Hp * Wp * nvec;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int cg = (int)(i % nvec);
    int64_t m = i / nvec;
    const int j = (int)(m % Wp); m /= Wp;
    const int ii = (int)(m % Hp); m /= Hp;
    const int b = (int)(m % B);
    const int ph = (int)(m / B);
    const int h = 2 * ii + (ph >> 1), w = 2 * j + (ph & 1);
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (h < H && w < W) v = *reinterpret_cast<const uint4*>(x + (((int64_t)b * H + h) * W + w) * x_ld + cg * 16);
    *reinterpret_cast<uint4*>(out + (i / nvec) * C + cg * 16) = v;
  }
}

}  // namespace iswm

using namespace iswm;

static inline int grid_of(int64_t work, int waves = 8) {
  const int64_t g = (work + kT - 1) / kT;
  return (int)std::max<int64_t>(1, std::min<int64_t>(g, (int64_t)num_sms() * waves));
}
#define ST(s) static_cast<cudaStream_t>(s)
#define BF(p) static_cast<const __nv_bfloat16*>(p)
#define REQ_SCALE(s, what) ISWM_REQUIRE((s) > 0.f && (s) < INFINITY, what ": scale %g must be positive and finite", (double)(s))

extern "C" int iswm_pack_weight_f8(const float* d_w, int Cout, int Cin, int RS, int cin_pad, void* d_out, float* d_sw, void* stream) {
  ISWM_REQUIRE(d_w && d_out && d_sw && Cout >= 1 && Cin >= 1 && RS >= 1, "pack_weight_f8: bad arguments");
  ISWM_REQUIRE(cin_pad >= Cin && (cin_pad % 128) == 0, "pack_weight_f8: cin_pad=%d must be a multiple of 128 and >= Cin=%d", cin_pad, Cin);
  launch_k(pack_weight_f8_kernel, dim3(Cout), dim3(kT), 0, ST(stream), d_w, Cin, RS, cin_pad, static_cast<uint8_t*>(d_out), d_sw);
  return check_launch("pack_weight_f8");
}
extern "C" int iswm_maxpool_fwd_f8(const void* d_x, int B, int H, int W, int C, int Ho, int Wo, float s, void* d_out, void* stream) {
  ISWM_REQUIRE(d_x && d_out && C > 0 && (C % 8) == 0, "maxpool_fwd_f8: null argument or C=%d not a multiple of 8", C);
  REQ_SCALE(s, "maxpool_fwd_f8");
  launch_k(maxpool_fwd_f8_kernel, dim3(grid_of((int64_t)B * Ho * Wo * (C / 8))), dim3(kT), 0, ST(stream), BF(d_x), B, H, W, C, Ho, Wo, s,
           static_cast<uint8_t*>(d_out));
  return check_launch("maxpool_fwd_f8");
}
extern "C" int iswm_gap_fwd_f8(const void* d_x, int x_ld, int B, int64_t HW, int C, float s, void* d_out, void* stream) {
  ISWM_REQUIRE(d_x && d_out && HW > 0 && C > 0 && (C % 8) == 0 && (x_ld % 8) == 0 && x_ld >= C, "gap_fwd_f8: bad arguments (C=%d x_ld=%d)", C, x_ld);
  REQ_SCALE(s, "gap_fwd_f8");
  launch_k(gap_fwd_f8_kernel, dim3((C + 63) / 64, B), dim3(kT), 0, ST(stream), static_cast<const uint8_t*>(d_x), x_ld, HW, C, s,
           static_cast<__nv_bfloat16*>(d_out));
  return check_launch("gap_fwd_f8");
}
extern "C" int iswm_broadcast_hw_f8(const void* d_x, int B, int64_t HW, int C, float s, void* d_out, int out_ld, void* stream) {
  ISWM_REQUIRE(d_x && d_out && C > 0 && (C % 8) == 0 && (out_ld % 8) == 0, "broadcast_hw_f8: bad arguments (C=%d out_ld=%d)", C, out_ld);
  REQ_SCALE(s, "broadcast_hw_f8");
  launch_k(broadcast_hw_f8_kernel, dim3(grid_of((int64_t)B * HW * (C / 8))), dim3(kT), 0, ST(stream), BF(d_x), B, HW, C, s,
           static_cast<uint8_t*>(d_out), out_ld);
  return check_launch("broadcast_hw_f8");
}
extern "C" int iswm_bilinear_fwd_f8(const void* d_x, int x_ld, int B, int Hi, int Wi, int C, int Ho, int Wo, float s, void* d_out,
                                    int out_ld, void* stream) {
  ISWM_REQUIRE(d_x && d_out && C > 0 && (C % 8) == 0 && (x_ld % 8) == 0 && (out_ld % 8) == 0, "bilinear_fwd_f8: bad arguments");
  REQ_SCALE(s, "bilinear_fwd_f8");
  launch_k(bilinear_fwd_f8_kernel, dim3((unsigned)(B * Ho), (unsigned)std::min(8, (Wo * (C / 8) + kT - 1) / kT)), dim3(kT), 0, ST(stream),
           BF(d_x), x_ld, B, Hi, Wi, C, Ho, Wo, s, static_cast<uint8_t*>(d_out), out_ld);
  return check_launch("bilinear_fwd_f8");
}
extern "C" int iswm_phase_split_b8(const void* d_x, int x_ld, int B, int H, int W, int C, void* d_out, void* stream) {
  ISWM_REQUIRE(d_x && d_out && C > 0 && (C % 16) == 0 && (x_ld % 16) == 0, "phase_split_b8: C=%d and x_ld=%d must be multiples of 16", C, x_ld);
  const int Hp = (H + 1) / 2, Wp = (W + 1) / 2;
  launch_k(phase_split_b8_kernel, dim3(grid_of((int64_t)4 * B * Hp * Wp * (C / 16))), dim3(kT), 0, ST(stream), static_cast<const uint8_t*>(d_x),
           x_ld, B, H, W, C, Hp, Wp, 4, static_cast<uint8_t*>(d_out));
  return check_launch("phase_split_b8");
}
extern "C" int iswm_subsample2_b8(const void* d_x, int x_ld, int B, int H, int W, int C, void* d_out, void* stream) {
  ISWM_REQUIRE(d_x && d_out && C > 0 && (C % 16) == 0 && (x_ld % 16) == 0, "subsample2_b8: C=%d and x_ld=%d must be multiples of 16", C, x_ld);
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2;
  launch_k(phase_split_b8_kernel, dim3(grid_of((int64_t)B * Ho * Wo * (C / 16))), dim3(kT), 0, ST(stream), static_cast<const uint8_t*>(d_x),
           x_ld, B, H, W, C, Ho, Wo, 1, static_cast<uint8_t*>(d_out));
  return check_launch("subsample2_b8");
}
