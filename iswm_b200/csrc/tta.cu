// tta.cu — multi-scale + horizontal-flip test-time augmentation for the predict step (DeepLabV3+ "MS + Flip"
// evaluation): the input resize / mirror that builds each view, and ONE epilogue over the low-resolution logits of
// every view that writes the uint8 maps (and confusion counts) of the averaged probabilities. Neither the views'
// full-resolution logits nor the output-resolution logits are ever written.
#include "metric_common.cuh"

#include <algorithm>

namespace iswm {

// ---------------------------------------------------------------------------
// resize + mirror of the fp32 NCHW input: F.interpolate(bilinear, align_corners=False) then .flip(-1).
// One grid row per (image, channel, output row); consecutive threads write consecutive output columns.
__global__ void __launch_bounds__(kThreads)
resize_flip_f32_kernel(const float* __restrict__ x, int Hi, int Wi, int Ho, int Wo, int flip, float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int64_t row = blockIdx.x;                     // (b * C + c) * Ho + ho
  const int ho = (int)(row % Ho);
  const float* plane = x + (row / Ho) * Hi * Wi;
  float* dst = out + row * Wo;
  if (Hi == Ho && Wi == Wo) {                         // scale 1: an exact copy, as the reference skips the resize
    const float* s = plane + (int64_t)ho * Wi;
    for (int wo = blockIdx.y * kThreads + threadIdx.x; wo < Wo; wo += gridDim.y * kThreads)
      dst[wo] = __ldg(s + (flip ? Wo - 1 - wo : wo));
    return;
  }
  const float sh = (float)Hi / (float)Ho, sw = (float)Wi / (float)Wo;
  int y0, y1;
  float ly;
  bil_src(ho, sh, Hi, y0, y1, ly);
  const float* r0 = plane + (int64_t)y0 * Wi;
  const float* r1 = plane + (int64_t)y1 * Wi;
  for (int wo = blockIdx.y * kThreads + threadIdx.x; wo < Wo; wo += gridDim.y * kThreads) {
    int x0, x1;
    float lx;
    bil_src(flip ? Wo - 1 - wo : wo, sw, Wi, x0, x1, lx);
    // separable, in the association of torch's CUDA upsample_bilinear2d (rows mixed first, then the two rows, each sum
    // as an fma onto the second product), not bil_mix: the views' inputs then carry torch's rounding, which a bf16
    // network would otherwise amplify into p1 differences of up to ~6e-3 against the torch composition
    const float a = fmaf(1.f - lx, __ldg(r0 + x0), lx * __ldg(r0 + x1));
    const float b = fmaf(1.f - lx, __ldg(r1 + x0), lx * __ldg(r1 + x1));
    dst[wo] = fmaf(1.f - ly, a, ly * b);
  }
}

// ---------------------------------------------------------------------------
// multi-view predict epilogue
struct TtaViews {
  IswmTtaView v[ISWM_TTA_MAX_VIEWS];
};

// One grid row per output image row; a thread produces 4 consecutive pixels, looping over the views for each of them
// (the views' low-resolution logits are small and stay in L1 / L2, so the taps cost latency, not HBM traffic).
template <typename TT, bool HAS_CM, bool VEC4>
__global__ void __launch_bounds__(kThreads, 4)
predict_tta_epilogue_kernel(const __grid_constant__ TtaViews views, int n_views, int Ho, int Wo, int mode, float threshold,
                            const TT* __restrict__ tru, uint8_t* __restrict__ pred_out, uint8_t* __restrict__ conf_out,
                            unsigned long long* __restrict__ cm) {
  pdl_wait();
  pdl_launch();
  const int ho = blockIdx.x % Ho, b = blockIdx.x / Ho;
  const int64_t row_off = ((int64_t)b * Ho + ho) * Wo;
  unsigned cnt[4] = {0, 0, 0, 0};
  const int nquad = (Wo + 3) >> 2;
  for (int qd = blockIdx.y * kThreads + threadIdx.x; qd < nquad; qd += gridDim.y * kThreads) {
    const int wo0 = qd << 2;
    float s0[4] = {0.f, 0.f, 0.f, 0.f}, s1[4] = {0.f, 0.f, 0.f, 0.f}, margin[4] = {0.f, 0.f, 0.f, 0.f};
    for (int vi = 0; vi < n_views; vi++) {
      const IswmTtaView& v = views.v[vi];
      const float2* lo = reinterpret_cast<const float2*>(v.lo) + (int64_t)b * v.Hi * v.Wi;   // NHWC, C == 2
      const float ish = (float)v.Hi / (float)v.Hv, isw = (float)v.Wi / (float)v.Wv;
      const bool direct = (v.Hv == Ho && v.Wv == Wo);
      // the view-grid rows this output row reads (one row with weight 0 on the second when direct), and for each the
      // low-resolution row pair of the first resize
      int u0 = ho, u1 = ho;
      float lu = 0.f;
      if (!direct) bil_src(ho, (float)v.Hv / (float)Ho, v.Hv, u0, u1, lu);
      int y0, y1;
      float ly0, ly1;
      bil_src(u0, ish, v.Hi, y0, y1, ly0);
      const float2* r00 = lo + (int64_t)y0 * v.Wi;
      const float2* r01 = lo + (int64_t)y1 * v.Wi;
      bil_src(u1, ish, v.Hi, y0, y1, ly1);
      const float2* r10 = lo + (int64_t)y0 * v.Wi;
      const float2* r11 = lo + (int64_t)y1 * v.Wi;
      const float osw = (float)v.Wv / (float)Wo;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const int wo = wo0 + k;
        if (!VEC4 && wo >= Wo) break;
        const int c = v.flip ? Wo - 1 - wo : wo;       // the column before the mirror
        float a0, a1;
        if (direct) {
          const float2 a = lo_tap(r00, r01, ly0, c, isw, v.Wi);
          a0 = a.x;
          a1 = a.y;
        } else {
          int t0, t1;
          float lt;
          bil_src(c, osw, v.Wv, t0, t1, lt);
          const float w00 = (1.f - lu) * (1.f - lt), w01 = (1.f - lu) * lt, w10 = lu * (1.f - lt), w11 = lu * lt;
          const float2 q00 = lo_tap(r00, r01, ly0, t0, isw, v.Wi), q01 = lo_tap(r00, r01, ly0, t1, isw, v.Wi);
          const float2 q10 = lo_tap(r10, r11, ly1, t0, isw, v.Wi), q11 = lo_tap(r10, r11, ly1, t1, isw, v.Wi);
          a0 = bil_mix(w00, q00.x, w01, q01.x, w10, q10.x, w11, q11.x);
          a1 = bil_mix(w00, q00.y, w01, q01.y, w10, q10.y, w11, q11.y);
        }
        // the 2-class softmax in predict_epilogue2's order
        const float m = fmaxf(a0, a1);
        const float e0 = expf(a0 - m), e1 = expf(a1 - m);
        s1[k] += e1 / (e0 + e1);
        if (mode == 0) {
          s0[k] += e0 / (e0 + e1);
          margin[k] += a1 - a0;
        }
      }
    }
    Vec<TT, 4> t;
    if constexpr (HAS_CM && VEC4) vload(t, tru + row_off + wo0);
    Vec<uint8_t, 4> po, co;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const float p1 = s1[k] / (float)n_views;
      int pred;
      if (mode == 0) {
        const float p0 = s0[k] / (float)n_views;
        pred = (p1 > p0 || (p1 == p0 && margin[k] > 0.f)) ? 1 : 0;   // one view: exactly a1 > a0
      } else {
        pred = (p1 > threshold) ? 1 : 0;
      }
      po.e[k] = (uint8_t)pred;
      co.e[k] = mode == 0 ? (uint8_t)0 : (uint8_t)(p1 * 255.0f);      // truncation, as ndarray.astype(uint8)
      if constexpr (HAS_CM) {
        if (VEC4 || wo0 + k < Wo) {
          const long long tt = VEC4 ? (long long)t.e[k] : (long long)tru[row_off + wo0 + k];
          const bool tv = (tt == 0 || tt == 1);
          const int cell = (int)(tt * 2 + pred);
#pragma unroll
          for (int cc = 0; cc < 4; cc++) cnt[cc] += (tv && cell == cc);
        }
      }
    }
    if constexpr (VEC4) {
      if (pred_out) vstore(pred_out + row_off + wo0, po);
      if (conf_out) vstore(conf_out + row_off + wo0, co);
    } else {
#pragma unroll
      for (int k = 0; k < 4; k++) {
        if (wo0 + k >= Wo) break;
        if (pred_out) pred_out[row_off + wo0 + k] = po.e[k];
        if (conf_out) conf_out[row_off + wo0 + k] = co.e[k];
      }
    }
  }
  if constexpr (HAS_CM) flush_counters<4>(cnt, 4, cm);
}

template <typename TT, bool HAS_CM>
static void launch_tta_vec(bool vec4, dim3 grid, const TtaViews& v, int n, int Ho, int Wo, int mode, float thr, const TT* t,
                           uint8_t* pred, uint8_t* conf, unsigned long long* c, cudaStream_t st) {
  if (vec4)
    launch_k(predict_tta_epilogue_kernel<TT, HAS_CM, true>, grid, dim3(kThreads), 0, st, v, n, Ho, Wo, mode, thr, t, pred, conf, c);
  else
    launch_k(predict_tta_epilogue_kernel<TT, HAS_CM, false>, grid, dim3(kThreads), 0, st, v, n, Ho, Wo, mode, thr, t, pred, conf, c);
}

template <typename TT>
static int launch_predict_tta(const TtaViews& v, int n, const void* tru, int B, int Ho, int Wo, int mode, float thr,
                              uint8_t* pred, uint8_t* conf, int64_t* cm, cudaStream_t st) {
  const TT* t = static_cast<const TT*>(tru);
  auto* c = reinterpret_cast<unsigned long long*>(cm);
  const bool vec4 = (Wo & 3) == 0;
  dim3 grid((unsigned)(B * Ho), (unsigned)std::max(1, std::min(8, ((Wo + 3) / 4 + kThreads - 1) / kThreads)));
  if (cm != nullptr && tru != nullptr)
    launch_tta_vec<TT, true>(vec4, grid, v, n, Ho, Wo, mode, thr, t, pred, conf, c, st);
  else
    launch_tta_vec<TT, false>(vec4, grid, v, n, Ho, Wo, mode, thr, t, pred, conf, c, st);
  return check_launch("predict_tta_epilogue");
}

}  // namespace iswm

using namespace iswm;

extern "C" int iswm_resize_flip_f32(const float* d_x, int B, int C, int Hi, int Wi, int Ho, int Wo, int flip, float* d_out,
                                    void* stream) {
  ISWM_REQUIRE(B >= 0 && C >= 1 && Hi >= 1 && Wi >= 1 && Ho >= 1 && Wo >= 1, "resize_flip_f32: bad sizes");
  ISWM_REQUIRE((int64_t)B * C * Ho < (1ll << 31), "resize_flip_f32: too many rows");
  if (B == 0) return 0;
  ISWM_REQUIRE(d_x && d_out, "resize_flip_f32: null pointer");
  dim3 grid((unsigned)((int64_t)B * C * Ho), (unsigned)std::max(1, std::min(8, (Wo + kThreads - 1) / kThreads)));
  launch_k(resize_flip_f32_kernel, grid, dim3(kThreads), 0, static_cast<cudaStream_t>(stream), d_x, Hi, Wi, Ho, Wo,
           flip ? 1 : 0, d_out);
  return check_launch("resize_flip_f32");
}

extern "C" int iswm_predict_tta_epilogue(const IswmTtaView* h_views, int n_views, int B, int C, int Ho, int Wo, int mode,
                                         float threshold, const void* d_true, int true_dtype, uint8_t* d_pred_out,
                                         uint8_t* d_conf_out, int64_t* d_cm, void* stream) {
  ISWM_REQUIRE(h_views && n_views >= 1 && n_views <= ISWM_TTA_MAX_VIEWS, "predict_tta_epilogue: %d views (1..%d)", n_views,
               ISWM_TTA_MAX_VIEWS);
  ISWM_REQUIRE(C == 2, "predict_tta_epilogue: test-time augmentation is the two-class case (C=%d)", C);
  ISWM_REQUIRE(B >= 0 && Ho >= 1 && Wo >= 1, "predict_tta_epilogue: bad sizes");
  ISWM_REQUIRE(mode == 0 || mode == 1, "predict_tta_epilogue: bad mode %d", mode);
  ISWM_REQUIRE((int64_t)B * Ho < (1ll << 31), "predict_tta_epilogue: too many rows");
  TtaViews v = {};
  for (int i = 0; i < n_views; i++) {
    const IswmTtaView& s = h_views[i];
    ISWM_REQUIRE(s.lo && s.Hi >= 1 && s.Wi >= 1 && s.Hv >= 1 && s.Wv >= 1, "predict_tta_epilogue: view %d has bad sizes", i);
    ISWM_REQUIRE((reinterpret_cast<uintptr_t>(s.lo) & 7) == 0, "predict_tta_epilogue: view %d logits must be 8-byte aligned", i);
    v.v[i] = s;
    v.v[i].flip = s.flip ? 1 : 0;
  }
  if ((Wo & 3) == 0) {        // 32-bit map stores and 4-element label loads
    ISWM_REQUIRE(!d_pred_out || (reinterpret_cast<uintptr_t>(d_pred_out) & 3) == 0, "predict_tta_epilogue: pred map must be 4-byte aligned");
    ISWM_REQUIRE(!d_conf_out || (reinterpret_cast<uintptr_t>(d_conf_out) & 3) == 0, "predict_tta_epilogue: confidence map must be 4-byte aligned");
    if (d_true && d_cm) {
      const size_t esz = true_dtype == ISWM_U8 ? 1 : (true_dtype == ISWM_I32 ? 4 : 8);
      ISWM_REQUIRE((reinterpret_cast<uintptr_t>(d_true) % (esz * 4 >= 16 ? 16 : esz * 4)) == 0, "predict_tta_epilogue: labels must be aligned to 4 elements");
    }
  }
  if (B == 0) return 0;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (true_dtype) {
    case ISWM_U8:  return launch_predict_tta<uint8_t>(v, n_views, d_true, B, Ho, Wo, mode, threshold, d_pred_out, d_conf_out, d_cm, st);
    case ISWM_I32: return launch_predict_tta<int32_t>(v, n_views, d_true, B, Ho, Wo, mode, threshold, d_pred_out, d_conf_out, d_cm, st);
    case ISWM_I64: return launch_predict_tta<int64_t>(v, n_views, d_true, B, Ho, Wo, mode, threshold, d_pred_out, d_conf_out, d_cm, st);
    default: set_error("bad true dtype %d", true_dtype); return 2;
  }
}
