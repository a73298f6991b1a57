// window.cu — sliding-window inference for the predict step (mmseg's mode='slide'): the gather that cuts windows of the
// fp32 NCHW scene straight into the batch of the next forward, and ONE epilogue over the low-resolution logits of every
// window that writes the uint8 maps (and confusion counts) of the overlap-averaged probabilities. Neither the windows'
// full-resolution logits nor the scene-sized probability sums are ever written.
#include "metric_common.cuh"

#include <algorithm>

namespace iswm {

// ---------------------------------------------------------------------------
// The placement rule along one axis of length L (shared by both kernels and the host checks): the window side is
// w = min(window, L), there are n = ceil((L - w) / s) + 1 windows at offsets o_i = min(i * s, L - w) (only the last one
// can be snapped to the border), and the windows covering pixel p are a contiguous index range [lo, hi].
struct WinAxis {
  int L, w, s, n;
  __host__ __device__ WinAxis(int L_, int window, int s_)
      : L(L_), w(window < L_ ? window : L_), s(s_), n((L_ - (window < L_ ? window : L_) + s_ - 1) / s_ + 1) {}
  __host__ __device__ int off(int i) const { return i * s < L - w ? i * s : L - w; }
  __host__ __device__ void cover(int p, int& lo, int& hi) const {
    lo = p < w ? 0 : (p - w) / s + 1;       // the first i with i * s + w > p; past the unsnapped windows only the last
    if (lo > n - 1) lo = n - 1;
    hi = p >= L - w ? n - 1 : p / s;        // the last i with o_i <= p
  }
};

// ---------------------------------------------------------------------------
// windows [first, first + n) of the flat list (image-major, then row-major over (iy, ix)) of fp32 NCHW [B,C,H,W] into
// [n,C,wh,ww]. One grid row per (window, channel, window row); consecutive threads copy consecutive columns.
__global__ void __launch_bounds__(kThreads)
window_gather_f32_kernel(const float* __restrict__ x, int C, int H, int W, WinAxis ay, WinAxis ax, int first,
                         float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int64_t row = blockIdx.x;                      // (k * C + c) * wh + y
  const int y = (int)(row % ay.w);
  const int64_t kc = row / ay.w;
  const int c = (int)(kc % C);
  const int64_t g = first + kc / C;                   // the window's index in the flat list
  const int per_img = ay.n * ax.n;
  const int64_t b = g / per_img;
  const int r = (int)(g % per_img);
  const float* src = x + (((b * C + c) * H) + ay.off(r / ax.n) + y) * (int64_t)W + ax.off(r % ax.n);
  float* dst = out + row * ax.w;
  for (int j = blockIdx.y * kThreads + threadIdx.x; j < ax.w; j += gridDim.y * kThreads) dst[j] = __ldg(src + j);
}

// ---------------------------------------------------------------------------
// Overlap-averaging predict epilogue. One grid row per scene row; a thread produces 4 consecutive pixels. The block
// finds the window rows covering its scene row once; per pixel the covering window columns are looped over in
// ascending (iy, ix) order, each window's logits taken at the window-local coordinate with logits_up_fwd's arithmetic
// (lo_tap), then the 2-class softmax in predict_epilogue2's order. No loop is capped: at most ceil(w/s)+1 windows
// cover a pixel per axis. The windows' low-resolution logits are small and stay in L1 / L2.
template <typename TT, bool HAS_CM, bool VEC4>
__global__ void __launch_bounds__(kThreads, 4)
predict_window_epilogue_kernel(const float2* __restrict__ lo, int H, int W, WinAxis ay, WinAxis ax, int hi, int wi,
                               float threshold, const TT* __restrict__ tru, uint8_t* __restrict__ pred_out,
                               uint8_t* __restrict__ conf_out, unsigned long long* __restrict__ cm) {
  pdl_wait();
  pdl_launch();
  const int h = blockIdx.x % H, b = blockIdx.x / H;
  const int64_t row_off = ((int64_t)b * H + h) * W;
  const float ish = (float)hi / (float)ay.w, isw = (float)wi / (float)ax.w;
  const int64_t win_sz = (int64_t)hi * wi;
  int iy0, iy1;
  ay.cover(h, iy0, iy1);
  unsigned cnt[4] = {0, 0, 0, 0};
  const int nquad = (W + 3) >> 2;
  for (int qd = blockIdx.y * kThreads + threadIdx.x; qd < nquad; qd += gridDim.y * kThreads) {
    const int w0 = qd << 2;
    float s1[4] = {0.f, 0.f, 0.f, 0.f};
    int nc[4] = {0, 0, 0, 0};
    for (int iy = iy0; iy <= iy1; iy++) {
      int y0, y1;
      float ly;
      bil_src(h - ay.off(iy), ish, hi, y0, y1, ly);
      const float2* wrow = lo + ((int64_t)b * ay.n + iy) * ax.n * win_sz;     // window (b, iy, 0)
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const int w = w0 + k;
        if (!VEC4 && w >= W) break;
        int ix0, ix1;
        ax.cover(w, ix0, ix1);
        for (int ix = ix0; ix <= ix1; ix++) {
          const float2* lw = wrow + ix * win_sz;
          const float2 a = lo_tap(lw + (int64_t)y0 * wi, lw + (int64_t)y1 * wi, ly, w - ax.off(ix), isw, wi);
          const float m = fmaxf(a.x, a.y);
          const float e0 = expf(a.x - m), e1 = expf(a.y - m);
          s1[k] += e1 / (e0 + e1);
        }
        nc[k] += ix1 - ix0 + 1;
      }
    }
    Vec<TT, 4> t;
    if constexpr (HAS_CM && VEC4) vload(t, tru + row_off + w0);
    Vec<uint8_t, 4> po, co;
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const float p1 = s1[k] / (float)nc[k];
      const int pred = (p1 > threshold) ? 1 : 0;
      po.e[k] = (uint8_t)pred;
      co.e[k] = (uint8_t)(p1 * 255.0f);                              // truncation, as ndarray.astype(uint8)
      if constexpr (HAS_CM) {
        if (VEC4 || w0 + k < W) {
          const long long tt = VEC4 ? (long long)t.e[k] : (long long)tru[row_off + w0 + k];
          const bool tv = (tt == 0 || tt == 1);
          const int cell = (int)(tt * 2 + pred);
#pragma unroll
          for (int cc = 0; cc < 4; cc++) cnt[cc] += (tv && cell == cc);
        }
      }
    }
    if constexpr (VEC4) {
      if (pred_out) vstore(pred_out + row_off + w0, po);
      if (conf_out) vstore(conf_out + row_off + w0, co);
    } else {
#pragma unroll
      for (int k = 0; k < 4; k++) {
        if (w0 + k >= W) break;
        if (pred_out) pred_out[row_off + w0 + k] = po.e[k];
        if (conf_out) conf_out[row_off + w0 + k] = co.e[k];
      }
    }
  }
  if constexpr (HAS_CM) flush_counters<4>(cnt, 4, cm);
}

template <typename TT, bool HAS_CM>
static void launch_window_vec(bool vec4, dim3 grid, const float2* lo, int H, int W, const WinAxis& ay, const WinAxis& ax,
                              int hi, int wi, float thr, const TT* t, uint8_t* pred, uint8_t* conf, unsigned long long* c,
                              cudaStream_t st) {
  if (vec4)
    launch_k(predict_window_epilogue_kernel<TT, HAS_CM, true>, grid, dim3(kThreads), 0, st, lo, H, W, ay, ax, hi, wi, thr, t, pred, conf, c);
  else
    launch_k(predict_window_epilogue_kernel<TT, HAS_CM, false>, grid, dim3(kThreads), 0, st, lo, H, W, ay, ax, hi, wi, thr, t, pred, conf, c);
}

template <typename TT>
static int launch_predict_window(const float2* lo, int B, int H, int W, const WinAxis& ay, const WinAxis& ax, int hi, int wi,
                                 float thr, const void* tru, uint8_t* pred, uint8_t* conf, int64_t* cm, cudaStream_t st) {
  const TT* t = static_cast<const TT*>(tru);
  auto* c = reinterpret_cast<unsigned long long*>(cm);
  const bool vec4 = (W & 3) == 0;
  dim3 grid((unsigned)(B * H), (unsigned)std::max(1, std::min(8, ((W + 3) / 4 + kThreads - 1) / kThreads)));
  if (cm != nullptr && tru != nullptr)
    launch_window_vec<TT, true>(vec4, grid, lo, H, W, ay, ax, hi, wi, thr, t, pred, conf, c, st);
  else
    launch_window_vec<TT, false>(vec4, grid, lo, H, W, ay, ax, hi, wi, thr, t, pred, conf, c, st);
  return check_launch("predict_window_epilogue");
}

}  // namespace iswm

using namespace iswm;

extern "C" int iswm_window_gather_f32(const float* d_x, int B, int C, int H, int W, int wh, int ww, int sh, int sw, int first,
                                      int n, float* d_out, void* stream) {
  ISWM_REQUIRE(B >= 0 && C >= 1 && H >= 1 && W >= 1, "window_gather_f32: bad sizes");
  ISWM_REQUIRE(wh >= 1 && ww >= 1 && sh >= 1 && sw >= 1 && sh <= wh && sw <= ww,
               "window_gather_f32: window %dx%d, stride %dx%d (need 1 <= stride <= window)", wh, ww, sh, sw);
  const WinAxis ay(H, wh, sh), ax(W, ww, sw);
  const int64_t total = (int64_t)B * ay.n * ax.n;
  ISWM_REQUIRE(first >= 0 && n >= 0 && first + (int64_t)n <= total, "window_gather_f32: windows [%d, %d) outside the %lld of the batch",
               first, first + n, (long long)total);
  ISWM_REQUIRE((int64_t)n * C * ay.w < (1ll << 31), "window_gather_f32: too many rows");
  if (n == 0) return 0;
  ISWM_REQUIRE(d_x && d_out, "window_gather_f32: null pointer");
  dim3 grid((unsigned)((int64_t)n * C * ay.w), (unsigned)std::max(1, std::min(8, (ax.w + kThreads - 1) / kThreads)));
  launch_k(window_gather_f32_kernel, grid, dim3(kThreads), 0, static_cast<cudaStream_t>(stream), d_x, C, H, W, ay, ax, first, d_out);
  return check_launch("window_gather_f32");
}

extern "C" int iswm_predict_window_epilogue(const float* d_lo, int B, int H, int W, int wh, int ww, int sh, int sw, int hi,
                                            int wi, int C, float threshold, const void* d_true, int true_dtype,
                                            uint8_t* d_pred_out, uint8_t* d_conf_out, int64_t* d_cm, void* stream) {
  ISWM_REQUIRE(C == 2, "predict_window_epilogue: sliding-window inference is the two-class case (C=%d)", C);
  ISWM_REQUIRE(B >= 0 && H >= 1 && W >= 1 && hi >= 1 && wi >= 1, "predict_window_epilogue: bad sizes");
  ISWM_REQUIRE(wh >= 1 && ww >= 1 && sh >= 1 && sw >= 1 && sh <= wh && sw <= ww,
               "predict_window_epilogue: window %dx%d, stride %dx%d (need 1 <= stride <= window)", wh, ww, sh, sw);
  ISWM_REQUIRE((int64_t)B * H < (1ll << 31), "predict_window_epilogue: too many rows");
  ISWM_REQUIRE(!d_lo || (reinterpret_cast<uintptr_t>(d_lo) & 7) == 0, "predict_window_epilogue: logits must be 8-byte aligned");
  if ((W & 3) == 0) {        // 32-bit map stores and 4-element label loads
    ISWM_REQUIRE(!d_pred_out || (reinterpret_cast<uintptr_t>(d_pred_out) & 3) == 0, "predict_window_epilogue: pred map must be 4-byte aligned");
    ISWM_REQUIRE(!d_conf_out || (reinterpret_cast<uintptr_t>(d_conf_out) & 3) == 0, "predict_window_epilogue: confidence map must be 4-byte aligned");
    if (d_true && d_cm) {
      const size_t esz = true_dtype == ISWM_U8 ? 1 : (true_dtype == ISWM_I32 ? 4 : 8);
      ISWM_REQUIRE((reinterpret_cast<uintptr_t>(d_true) % (esz * 4 >= 16 ? 16 : esz * 4)) == 0, "predict_window_epilogue: labels must be aligned to 4 elements");
    }
  }
  if (B == 0) return 0;
  ISWM_REQUIRE(d_lo, "predict_window_epilogue: null logits");
  const WinAxis ay(H, wh, sh), ax(W, ww, sw);
  const float2* lo = reinterpret_cast<const float2*>(d_lo);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  switch (true_dtype) {
    case ISWM_U8:  return launch_predict_window<uint8_t>(lo, B, H, W, ay, ax, hi, wi, threshold, d_true, d_pred_out, d_conf_out, d_cm, st);
    case ISWM_I32: return launch_predict_window<int32_t>(lo, B, H, W, ay, ax, hi, wi, threshold, d_true, d_pred_out, d_conf_out, d_cm, st);
    case ISWM_I64: return launch_predict_window<int64_t>(lo, B, H, W, ay, ax, hi, wi, threshold, d_true, d_pred_out, d_conf_out, d_cm, st);
    default: set_error("bad true dtype %d", true_dtype); return 2;
  }
}
