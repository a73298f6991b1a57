// bn_dual.cu — the closing BatchNorm of a bottleneck block WITH a downsample branch, both branches in one pass.
//
//   out = relu( bn3(conv3(...)) + bn_ds(conv_ds(x)) )          network/backbone/resnet.py:99-120 with `downsample` set (:176-186)
//
// The block's two BatchNorms normalise tensors of the same [M][C] geometry and meet in one add + ReLU. Running them as
// separate kernels costs a round trip of the normalised shortcut (written by the downsample BatchNorm, read back by the
// closing one) and, in backward, a second read of the block-output gradient and its ReLU sign bits by the downsample
// BatchNorm's two passes. Here each pass handles both branches:
//   forward   reads raw3, raw_ds                      writes out (+ sign bits)      [was: +2 B written and +2 B read per element]
//   reduce    reads dout, bits, raw3, raw_ds          -> sum dz, sum dz.xhat3, sum dz.xhat_ds
//   apply     reads dout, bits, raw3, raw_ds          writes dy3, dy_ds
// dz = dout where the block's ReLU was active (the packed sign bits the forward pass wrote). Same thread layout and
// arithmetic as the single-branch kernels of elementwise.cu (per-channel constants in registers, 16-byte row accesses,
// fp32 partial sums in a fixed order inside a block, fp64 atomics across blocks).
#include "common.cuh"
#include "ew_common.cuh"
#include <stdlib.h>

namespace iswm {

struct BnSide {                      // one BatchNorm's per-channel vectors
  const double* stats;               // forward: sum x, sum x^2 (from the convolution epilogue)
  const float* gamma;
  const float* beta;
  float* running_mean;
  float* running_var;
  long long* nbt;
  float* save_mean;                  // forward: written; backward: read
  float* save_invstd;
  int stats_rep;                     // copies of the statistics vector to sum
};

// ------------------------------------------------------------------------------------------------------------- forward
// GCNT (synchronised BatchNorm): each side's `stats` holds the sums over every rank's rows (one copy) followed by the global
// row count at [2C]; M only bounds this rank's row walk
template <bool GCNT>
__global__ void __launch_bounds__(kT, 2)
bn_dual_train_apply_kernel(const __nv_bfloat16* __restrict__ xa, int xa_ld, const __nv_bfloat16* __restrict__ xb, int xb_ld,
                           BnSide A, BnSide Bs, int64_t M, int C, float eps, float momentum,
                           __nv_bfloat16* __restrict__ out, int out_ld, uint8_t* __restrict__ relu_bits,
                           int nx, int ny, int rows_per_block) {
  pdl_wait();
  pdl_launch();
  const int tx = threadIdx.x % nx, ty = threadIdx.x / nx;
  if (ty >= ny) return;
  const int c0 = tx << 3;
  constexpr int U = 4;
  const RowWalk w = row_walk(M, rows_per_block, ty, ny);
  const __nv_bfloat16* pa = xa + w.first * xa_ld + c0;
  const __nv_bfloat16* pb = xb + w.first * xb_ld + c0;
  const int64_t sa = (int64_t)ny * xa_ld, sb = (int64_t)ny * xb_ld;
  uint4 ra[U], rb[U];
  if (w.n >= U) {
#pragma unroll
    for (int u = 0; u < U; u++) {
      ra[u] = load_raw(pa + u * sa);
      rb[u] = load_raw(pb + u * sb);
    }
  }
  const double cnt = GCNT ? A.stats[2 * C] : 0.0;
  const double invM = GCNT ? 1.0 / cnt : 1.0 / (double)M;
  float sc[8], sc2[8], sh[8];         // out = relu(x*sc + y*sc2 + sh), sh = both shifts
  auto side = [&](const BnSide& S, float* scv, float* shv) {
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const int c = c0 + j;
      double s1 = S.stats[c], s2 = S.stats[C + c];
      for (int r = 1; r < S.stats_rep; r++) {
        s1 += S.stats[(size_t)r * 2 * C + c];
        s2 += S.stats[(size_t)r * 2 * C + C + c];
      }
      const double mean_d = s1 * invM;
      const float mean = (float)mean_d;
      const float var = fmaxf((float)(s2 * invM - mean_d * mean_d), 0.f);
      const float invstd = rsqrtf(var + eps);
      scv[j] = S.gamma[c] * invstd;
      shv[j] = fmaf(-mean, scv[j], S.beta[c]);
      if (blockIdx.x == 0 && ty == 0) {
        S.save_mean[c] = mean;
        S.save_invstd[c] = invstd;
        if (S.running_mean) {
          float unbiased;
          if (GCNT) unbiased = (cnt > 1.0) ? var * ((float)cnt / (float)(cnt - 1.0)) : var;
          else unbiased = (M > 1) ? var * ((float)M / (float)(M - 1)) : var;
          S.running_mean[c] = (1.f - momentum) * S.running_mean[c] + momentum * mean;
          S.running_var[c] = (1.f - momentum) * S.running_var[c] + momentum * unbiased;
        }
      }
    }
  };
  float shb[8];
  side(A, sc, sh);
  side(Bs, sc2, shb);
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    if (A.nbt) *A.nbt += 1;
    if (Bs.nbt) *Bs.nbt += 1;
  }
  __nv_bfloat16* po = out + w.first * out_ld + c0;
  const int64_t so = (int64_t)ny * out_ld;
  uint8_t* pbit = relu_bits ? relu_bits + w.first * (C >> 3) + tx : nullptr;
  const int64_t sbit = (int64_t)ny * (C >> 3);
  auto one = [&](const uint4& a4, const uint4& b4, __nv_bfloat16* o, uint8_t* ob) {
    const F8 a = unpack8(a4), b = unpack8(b4);
    F8 f;
    unsigned bits = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      // main branch first, then the shortcut added in fp32 (the single-branch pair rounds the shortcut to bf16 in between)
      const float v = fmaf(a.v[j], sc[j], sh[j]) + fmaf(b.v[j], sc2[j], shb[j]);
      bits |= (v > 0.f) ? (1u << j) : 0u;
      f.v[j] = fmaxf(v, 0.f);
    }
    if (ob) *ob = (uint8_t)bits;
    store8(o, f);
  };
  int i = 0;
  for (; i + U <= w.n; i += U) {
    if (i > 0) {
#pragma unroll
      for (int u = 0; u < U; u++) {
        ra[u] = load_raw(pa + u * sa);
        rb[u] = load_raw(pb + u * sb);
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) one(ra[u], rb[u], po + u * so, pbit ? pbit + u * sbit : nullptr);
    pa += U * sa; pb += U * sb; po += U * so;
    if (pbit) pbit += U * sbit;
  }
  for (; i < w.n; i++) {
    one(load_raw(pa), load_raw(pb), po, pbit);
    pa += sa; pb += sb; po += so;
    if (pbit) pbit += sbit;
  }
}

// ------------------------------------------------------------------------------------------------------------- backward, pass 1
__global__ void __launch_bounds__(kT, 2)
bn_dual_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ dout, int dout_ld, const uint8_t* __restrict__ bits,
                          const __nv_bfloat16* __restrict__ xa, int xa_ld, const __nv_bfloat16* __restrict__ xb, int xb_ld,
                          int64_t M, int C, const float* __restrict__ mean_a, const float* __restrict__ invstd_a,
                          const float* __restrict__ mean_b, const float* __restrict__ invstd_b,
                          double* __restrict__ sums_a, double* __restrict__ sums_b, int nx, int ny, int rows_per_block) {
  pdl_wait();
  pdl_launch();
  __shared__ float s_red[kT * 24];
  const int tx = threadIdx.x % nx, ty = threadIdx.x / nx;
  const int cbase = blockIdx.y * (nx << 3);
  const int c0 = cbase + (tx << 3);
  constexpr int U = 4;
  const bool live = (ty < ny) && (c0 < C);
  const RowWalk w = live ? row_walk(M, rows_per_block, ty, ny) : RowWalk{0, 0};
  const __nv_bfloat16* pg = dout + w.first * dout_ld + c0;
  const __nv_bfloat16* pa = xa + w.first * xa_ld + c0;
  const __nv_bfloat16* pb = xb + w.first * xb_ld + c0;
  const uint8_t* pm = bits + w.first * (C >> 3) + (c0 >> 3);
  const int64_t sg = (int64_t)ny * dout_ld, sa = (int64_t)ny * xa_ld, sb = (int64_t)ny * xb_ld, sm_ = (int64_t)ny * (C >> 3);
  float a[8], ba[8], bb[8];
#pragma unroll
  for (int j = 0; j < 8; j++) { a[j] = 0.f; ba[j] = 0.f; bb[j] = 0.f; }
  if (live) {
    auto one = [&](const uint4& g4, const uint4& a4, const uint4& b4, unsigned mbits) {
      F8 g = unpack8(g4);
      const F8 xv = unpack8(a4), yv = unpack8(b4);
#pragma unroll
      for (int j = 0; j < 8; j++) {
        const float gz = ((mbits >> j) & 1u) ? g.v[j] : 0.f;
        a[j] += gz;
        ba[j] = fmaf(gz, xv.v[j], ba[j]);
        bb[j] = fmaf(gz, yv.v[j], bb[j]);
      }
    };
    int i = 0;
    for (; i + U <= w.n; i += U) {
      uint4 gr[U], ar[U], br[U];
      unsigned mb[U];
#pragma unroll
      for (int u = 0; u < U; u++) {
        gr[u] = load_raw(pg + u * sg);
        ar[u] = load_raw(pa + u * sa);
        br[u] = load_raw(pb + u * sb);
        mb[u] = pm[u * sm_];
      }
#pragma unroll
      for (int u = 0; u < U; u++) one(gr[u], ar[u], br[u], mb[u]);
      pg += U * sg; pa += U * sa; pb += U * sb; pm += U * sm_;
    }
    for (; i < w.n; i++) {
      one(load_raw(pg), load_raw(pa), load_raw(pb), *pm);
      pg += sg; pa += sa; pb += sb; pm += sm_;
    }
  }
#pragma unroll
  for (int j = 0; j < 8; j++) {
    s_red[threadIdx.x * 24 + j] = a[j];
    s_red[threadIdx.x * 24 + 8 + j] = ba[j];
    s_red[threadIdx.x * 24 + 16 + j] = bb[j];
  }
  __syncthreads();
  for (int o = threadIdx.x; o < nx * 8; o += kT) {
    const int gx = o >> 3, j = o & 7;
    float ta = 0.f, tba = 0.f, tbb = 0.f;
    for (int y = 0; y < ny; y++) {
      ta += s_red[(y * nx + gx) * 24 + j];
      tba += s_red[(y * nx + gx) * 24 + 8 + j];
      tbb += s_red[(y * nx + gx) * 24 + 16 + j];
    }
    const int c = cbase + (gx << 3) + j;
    if (c < C) {
      atomicAdd(sums_a + c, (double)ta);
      atomicAdd(sums_a + C + c, (double)invstd_a[c] * ((double)tba - (double)mean_a[c] * (double)ta));
      atomicAdd(sums_b + c, (double)ta);
      atomicAdd(sums_b + C + c, (double)invstd_b[c] * ((double)tbb - (double)mean_b[c] * (double)ta));
    }
  }
}

// ------------------------------------------------------------------------------------------------------------- backward, pass 2
struct BnBwdSide {
  const float* gamma;
  const float* mean;
  const float* invstd;
  const double* sums;
  float* dgamma;
  float* dbeta;
};

// GCNT (synchronised BatchNorm): the sides' `sums` are the sums over every rank's rows with the global row count at [2C];
// dgamma / dbeta accumulate this rank's own sums (lsums_a / lsums_b)
template <bool GCNT>
__global__ void __launch_bounds__(kT, 2)
bn_dual_bwd_apply_kernel(const __nv_bfloat16* __restrict__ dout, int dout_ld, const uint8_t* __restrict__ bits,
                         const __nv_bfloat16* __restrict__ xa, int xa_ld, const __nv_bfloat16* __restrict__ xb, int xb_ld,
                         int64_t M, int C, BnBwdSide A, BnBwdSide Bs,
                         __nv_bfloat16* __restrict__ dxa, int dxa_ld, __nv_bfloat16* __restrict__ dxb, int dxb_ld,
                         int nx, int ny, int rows_per_block, const double* __restrict__ lsums_a, const double* __restrict__ lsums_b) {
  pdl_wait();
  pdl_launch();
  const int tx = threadIdx.x % nx, ty = threadIdx.x / nx;
  if (ty >= ny) return;
  const int c0 = tx << 3;
  constexpr int U = 3;          // 4 rows of three tensors in flight next to 48 per-channel constants spill at 128 registers
  const RowWalk w = row_walk(M, rows_per_block, ty, ny);
  const __nv_bfloat16* pg = dout + w.first * dout_ld + c0;
  const __nv_bfloat16* pa = xa + w.first * xa_ld + c0;
  const __nv_bfloat16* pb = xb + w.first * xb_ld + c0;
  const uint8_t* pm = bits + w.first * (C >> 3) + tx;
  const int64_t sg = (int64_t)ny * dout_ld, sa = (int64_t)ny * xa_ld, sb = (int64_t)ny * xb_ld, sm_ = (int64_t)ny * (C >> 3);
  uint4 gr[U], ar[U], br[U];
  unsigned mb[U];
  if (w.n >= U) {
#pragma unroll
    for (int u = 0; u < U; u++) {
      gr[u] = load_raw(pg + u * sg);
      ar[u] = load_raw(pa + u * sa);
      br[u] = load_raw(pb + u * sb);
      mb[u] = pm[u * sm_];
    }
  }
  const float invM = GCNT ? 1.0f / (float)A.sums[2 * C] : 1.0f / (float)M;
  // dx = k*dz + p*x + q  with  k = gamma*invstd, p = -k*invstd*mean(dz*xhat), q = -k*mean(dz) - p*mu   (per branch)
  float ka[8], pa_[8], qa[8], kb[8], pb_[8], qb[8];
  auto side = [&](const BnBwdSide& S, const double* ls, float* kk, float* pp, float* qq) {
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const int c = c0 + j;
      const float is = S.invstd[c], mu = S.mean[c];
      const float k = S.gamma[c] * is;
      const float s0 = (float)S.sums[c], s1 = (float)S.sums[C + c];
      kk[j] = k;
      pp[j] = -k * is * (s1 * invM);
      qq[j] = -k * (s0 * invM) - pp[j] * mu;
      if (blockIdx.x == 0 && ty == 0) {
        if (S.dbeta) S.dbeta[c] += GCNT ? (float)ls[c] : s0;
        if (S.dgamma) S.dgamma[c] += GCNT ? (float)ls[C + c] : s1;
      }
    }
  };
  side(A, lsums_a, ka, pa_, qa);
  side(Bs, lsums_b, kb, pb_, qb);
  __nv_bfloat16* oa = dxa + w.first * dxa_ld + c0;
  __nv_bfloat16* ob = dxb + w.first * dxb_ld + c0;
  const int64_t soa = (int64_t)ny * dxa_ld, sob = (int64_t)ny * dxb_ld;
  auto one = [&](const uint4& g4, const uint4& a4, const uint4& b4, unsigned mbits, __nv_bfloat16* da, __nv_bfloat16* db) {
    const F8 g = unpack8(g4), xv = unpack8(a4), yv = unpack8(b4);
    F8 ra, rb;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      const float gz = ((mbits >> j) & 1u) ? g.v[j] : 0.f;
      ra.v[j] = fmaf(ka[j], gz, fmaf(pa_[j], xv.v[j], qa[j]));
      rb.v[j] = fmaf(kb[j], gz, fmaf(pb_[j], yv.v[j], qb[j]));
    }
    store8(da, ra);
    store8(db, rb);
  };
  int i = 0;
  for (; i + U <= w.n; i += U) {
    if (i > 0) {
#pragma unroll
      for (int u = 0; u < U; u++) {
        gr[u] = load_raw(pg + u * sg);
        ar[u] = load_raw(pa + u * sa);
        br[u] = load_raw(pb + u * sb);
        mb[u] = pm[u * sm_];
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) one(gr[u], ar[u], br[u], mb[u], oa + u * soa, ob + u * sob);
    pg += U * sg; pa += U * sa; pb += U * sb; pm += U * sm_; oa += U * soa; ob += U * sob;
  }
  for (; i < w.n; i++) {
    one(load_raw(pg), load_raw(pa), load_raw(pb), *pm, oa, ob);
    pg += sg; pa += sa; pb += sb; pm += sm_; oa += soa; ob += sob;
  }
}

}  // namespace iswm

using namespace iswm;

#define ST(s) static_cast<cudaStream_t>(s)
#define BF(p) static_cast<const __nv_bfloat16*>(p)
#define BFW(p) static_cast<__nv_bfloat16*>(p)

static int check_dual(const char* what, int64_t M, int C, int ld0, int ld1, int ld2) {
  ISWM_REQUIRE(M > 0 && C > 0 && (C % 8) == 0 && C <= 2048, "%s: C=%d must be a multiple of 8, at most 2048 (M=%lld)", what, C, (long long)M);
  ISWM_REQUIRE((ld0 % 8) == 0 && (ld1 % 8) == 0 && (ld2 % 8) == 0, "%s: row pitches must be multiples of 8", what);
  return 0;
}

static int bn_dual_train_apply_impl(bool global, const void* d_x, int x_ld, const iswm_bn_side* main_bn,
                                   const void* d_x_ds, int x_ds_ld, const iswm_bn_side* ds_bn,
                                   int64_t M, int C, float eps, float momentum,
                                   void* d_out, int out_ld, uint8_t* d_relu_bits, void* stream) {
  if (debug_skip(ISWM_SKIP_BN)) return 0;
  ISWM_REQUIRE(d_x && d_x_ds && main_bn && ds_bn && d_out, "bn_dual_train_apply: null argument");
  if (int rc = check_dual("bn_dual_train_apply", M, C, x_ld, x_ds_ld, out_ld)) return rc;
  for (const iswm_bn_side* s : {main_bn, ds_bn}) {
    ISWM_REQUIRE(s->stats && s->gamma && s->beta && s->save_mean && s->save_invstd, "bn_dual_train_apply: a BatchNorm side lacks stats / gamma / beta / save slots");
    ISWM_REQUIRE(!global || s->stats_replicas <= 1, "bn_dual_train_apply_global: the global sums are one copy (stats_replicas=%d)", s->stats_replicas);
  }
  int nx, ny, rpb, blocks;
  bn_row_grid(C, M, 4, nx, ny, rpb, blocks, 2);          // 2 resident blocks per SM (launch bounds): one wave
  auto mk = [](const iswm_bn_side* s) {
    return BnSide{s->stats, s->gamma, s->beta, s->running_mean, s->running_var, reinterpret_cast<long long*>(s->num_batches_tracked), s->save_mean, s->save_invstd, s->stats_replicas > 1 ? s->stats_replicas : 1};
  };
  if (global)
    launch_k(bn_dual_train_apply_kernel<true>, dim3(blocks), dim3(kT), 0, ST(stream), BF(d_x), x_ld, BF(d_x_ds), x_ds_ld, mk(main_bn), mk(ds_bn),
             M, C, eps, momentum, BFW(d_out), out_ld, d_relu_bits, nx, ny, rpb);
  else
    launch_k(bn_dual_train_apply_kernel<false>, dim3(blocks), dim3(kT), 0, ST(stream), BF(d_x), x_ld, BF(d_x_ds), x_ds_ld, mk(main_bn), mk(ds_bn),
             M, C, eps, momentum, BFW(d_out), out_ld, d_relu_bits, nx, ny, rpb);
  return check_launch("bn_dual_train_apply");
}
extern "C" int iswm_bn_dual_train_apply(const void* d_x, int x_ld, const iswm_bn_side* main_bn,
                                        const void* d_x_ds, int x_ds_ld, const iswm_bn_side* ds_bn,
                                        int64_t M, int C, float eps, float momentum,
                                        void* d_out, int out_ld, uint8_t* d_relu_bits, void* stream) {
  return bn_dual_train_apply_impl(false, d_x, x_ld, main_bn, d_x_ds, x_ds_ld, ds_bn, M, C, eps, momentum, d_out, out_ld, d_relu_bits, stream);
}
extern "C" int iswm_bn_dual_train_apply_global(const void* d_x, int x_ld, const iswm_bn_side* main_bn,
                                               const void* d_x_ds, int x_ds_ld, const iswm_bn_side* ds_bn,
                                               int64_t M, int C, float eps, float momentum,
                                               void* d_out, int out_ld, uint8_t* d_relu_bits, void* stream) {
  return bn_dual_train_apply_impl(true, d_x, x_ld, main_bn, d_x_ds, x_ds_ld, ds_bn, M, C, eps, momentum, d_out, out_ld, d_relu_bits, stream);
}

extern "C" int iswm_bn_dual_bwd_reduce(const void* d_dout, int dout_ld, const uint8_t* d_relu_bits,
                                       const void* d_x, int x_ld, const iswm_bn_side* main_bn,
                                       const void* d_x_ds, int x_ds_ld, const iswm_bn_side* ds_bn,
                                       int64_t M, int C, double* d_sums, double* d_sums_ds, void* stream) {
  if (debug_skip(ISWM_SKIP_BN)) return 0;
  ISWM_REQUIRE(d_dout && d_relu_bits && d_x && d_x_ds && main_bn && ds_bn && d_sums && d_sums_ds, "bn_dual_bwd_reduce: null argument");
  if (int rc = check_dual("bn_dual_bwd_reduce", M, C, dout_ld, x_ld, x_ds_ld)) return rc;
  for (const iswm_bn_side* s : {main_bn, ds_bn})
    ISWM_REQUIRE(s->save_mean && s->save_invstd, "bn_dual_bwd_reduce: a BatchNorm side lacks its saved mean / invstd");
  int nx, ny, rows_per_block, blocks, groups = 1;
  if (C > 256) {            // channel groups of 256 x row blocks, one resident wave in all (see iswm_bn_bwd_reduce)
    nx = 32; ny = kT / nx;
    groups = (C / 8 + nx - 1) / nx;
    int64_t want = (M + (int64_t)ny * 8 - 1) / ((int64_t)ny * 8);
    want = std::max<int64_t>(1, std::min<int64_t>(want, std::max(1, num_sms() * 2 / groups)));
    rows_per_block = (int)((M + want - 1) / want);
    blocks = (int)((M + rows_per_block - 1) / rows_per_block);
  } else {
    bn_row_grid(C, M, 8, nx, ny, rows_per_block, blocks, 2);
  }
  launch_k(bn_dual_bwd_reduce_kernel, dim3(blocks, groups), dim3(kT), 0, ST(stream), BF(d_dout), dout_ld, d_relu_bits, BF(d_x), x_ld,
           BF(d_x_ds), x_ds_ld, M, C, (const float*)main_bn->save_mean, (const float*)main_bn->save_invstd,
           (const float*)ds_bn->save_mean, (const float*)ds_bn->save_invstd, d_sums, d_sums_ds, nx, ny, rows_per_block);
  return check_launch("bn_dual_bwd_reduce");
}

static int bn_dual_bwd_apply_impl(const double* d_lsums, const double* d_lsums_ds, const void* d_dout, int dout_ld, const uint8_t* d_relu_bits,
                                  const void* d_x, int x_ld, const iswm_bn_side* main_bn, const double* d_sums,
                                  const void* d_x_ds, int x_ds_ld, const iswm_bn_side* ds_bn, const double* d_sums_ds,
                                  int64_t M, int C, void* d_dx, int dx_ld, void* d_dx_ds, int dx_ds_ld,
                                  float* d_dgamma, float* d_dbeta, float* d_dgamma_ds, float* d_dbeta_ds, void* stream) {
  if (debug_skip(ISWM_SKIP_BN)) return 0;
  ISWM_REQUIRE(d_dout && d_relu_bits && d_x && d_x_ds && main_bn && ds_bn && d_sums && d_sums_ds && d_dx && d_dx_ds, "bn_dual_bwd_apply: null argument");
  if (int rc = check_dual("bn_dual_bwd_apply", M, C, dout_ld, x_ld, x_ds_ld)) return rc;
  ISWM_REQUIRE((dx_ld % 8) == 0 && (dx_ds_ld % 8) == 0, "bn_dual_bwd_apply: gradient row pitches must be multiples of 8");
  for (const iswm_bn_side* s : {main_bn, ds_bn})
    ISWM_REQUIRE(s->gamma && s->save_mean && s->save_invstd, "bn_dual_bwd_apply: a BatchNorm side lacks gamma / saved mean / invstd");
  int nx, ny, rpb, blocks;
  bn_row_grid(C, M, 4, nx, ny, rpb, blocks, 2);
  const BnBwdSide A{main_bn->gamma, main_bn->save_mean, main_bn->save_invstd, d_sums, d_dgamma, d_dbeta};
  const BnBwdSide Bs{ds_bn->gamma, ds_bn->save_mean, ds_bn->save_invstd, d_sums_ds, d_dgamma_ds, d_dbeta_ds};
  if (d_lsums)
    launch_k(bn_dual_bwd_apply_kernel<true>, dim3(blocks), dim3(kT), 0, ST(stream), BF(d_dout), dout_ld, d_relu_bits, BF(d_x), x_ld, BF(d_x_ds), x_ds_ld,
             M, C, A, Bs, BFW(d_dx), dx_ld, BFW(d_dx_ds), dx_ds_ld, nx, ny, rpb, d_lsums, d_lsums_ds);
  else
    launch_k(bn_dual_bwd_apply_kernel<false>, dim3(blocks), dim3(kT), 0, ST(stream), BF(d_dout), dout_ld, d_relu_bits, BF(d_x), x_ld, BF(d_x_ds), x_ds_ld,
             M, C, A, Bs, BFW(d_dx), dx_ld, BFW(d_dx_ds), dx_ds_ld, nx, ny, rpb, (const double*)nullptr, (const double*)nullptr);
  return check_launch("bn_dual_bwd_apply");
}

extern "C" int iswm_bn_dual_bwd_apply(const void* d_dout, int dout_ld, const uint8_t* d_relu_bits,
                                      const void* d_x, int x_ld, const iswm_bn_side* main_bn, const double* d_sums,
                                      const void* d_x_ds, int x_ds_ld, const iswm_bn_side* ds_bn, const double* d_sums_ds,
                                      int64_t M, int C, void* d_dx, int dx_ld, void* d_dx_ds, int dx_ds_ld,
                                      float* d_dgamma, float* d_dbeta, float* d_dgamma_ds, float* d_dbeta_ds, void* stream) {
  return bn_dual_bwd_apply_impl(nullptr, nullptr, d_dout, dout_ld, d_relu_bits, d_x, x_ld, main_bn, d_sums, d_x_ds, x_ds_ld, ds_bn, d_sums_ds,
                                M, C, d_dx, dx_ld, d_dx_ds, dx_ds_ld, d_dgamma, d_dbeta, d_dgamma_ds, d_dbeta_ds, stream);
}

extern "C" int iswm_bn_dual_bwd_apply_global(const void* d_dout, int dout_ld, const uint8_t* d_relu_bits,
                                             const void* d_x, int x_ld, const iswm_bn_side* main_bn, const double* d_gsums, const double* d_local_sums,
                                             const void* d_x_ds, int x_ds_ld, const iswm_bn_side* ds_bn, const double* d_gsums_ds,
                                             const double* d_local_sums_ds, int64_t M, int C, void* d_dx, int dx_ld, void* d_dx_ds, int dx_ds_ld,
                                             float* d_dgamma, float* d_dbeta, float* d_dgamma_ds, float* d_dbeta_ds, void* stream) {
  ISWM_REQUIRE(d_local_sums && d_local_sums_ds, "bn_dual_bwd_apply_global: null local sums");
  return bn_dual_bwd_apply_impl(d_local_sums, d_local_sums_ds, d_dout, dout_ld, d_relu_bits, d_x, x_ld, main_bn, d_gsums, d_x_ds, x_ds_ld, ds_bn,
                                d_gsums_ds, M, C, d_dx, dx_ld, d_dx_ds, dx_ds_ld, d_dgamma, d_dbeta, d_dgamma_ds, d_dbeta_ds, stream);
}
