// elementwise.cu — the HBM-bound glue between the tensor-core convolutions: BatchNorm
// (training statistics -> normalise, backward), pooling, bilinear resampling, layout and
// stride helpers, weight packing, optimiser step. Activations are NHWC bf16 and every
// kernel moves 16 bytes (8 channels) per thread access, rows addressed through an explicit
// pitch (ld) so that channel slices of a concat buffer are read and written in place —
// torch.cat (network/_deeplab.py:59, :171) never materialises.
#include "common.cuh"
#include "ew_common.cuh"
#include <algorithm>
#include <stdlib.h>

namespace iswm {

static inline int grid_for(int64_t work, int per_block = kT, int waves = 8) {
  int64_t g = (work + per_block - 1) / per_block;
  return (int)std::max<int64_t>(1, std::min<int64_t>(g, (int64_t)num_sms() * waves));
}

// ---------------------------------------------------------------------------
// weight packing
__global__ void pack_weight_fwd_kernel(const float* __restrict__ w, int Cout, int Cin, int RS,
                                       int cin_pad, int row_ld, __nv_bfloat16* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int64_t total = (int64_t)Cout * row_ld;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int o = (int)(i / row_ld), k = (int)(i % row_ld);
    const int t = k / cin_pad, c = k % cin_pad;
    float v = 0.f;
    if (t < RS && c < Cin) v = w[((int64_t)o * Cin + c) * RS + t];
    out[i] = __float2bfloat16_rn(v);
  }
}
__global__ void pack_weight_dgrad_kernel(const float* __restrict__ w, int Cout, int Cin, int RS,
                                         int cout_pad, __nv_bfloat16* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int64_t total = (int64_t)Cin * RS * cout_pad;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int o = (int)(i % cout_pad);
    const int t = (int)((i / cout_pad) % RS);
    const int c = (int)(i / ((int64_t)cout_pad * RS));
    float v = 0.f;
    if (o < Cout) v = w[((int64_t)o * Cin + c) * RS + t];
    out[i] = __float2bfloat16_rn(v);
  }
}
__global__ void unpack_wgrad_kernel(const float* __restrict__ dw, int Cout, int Cin, int RS,
                                    int cin_stride, int row_ld, float beta, float* __restrict__ g) {
  pdl_wait();
  pdl_launch();
  const int64_t total = (int64_t)Cout * Cin * RS;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int t = (int)(i % RS);
    const int c = (int)((i / RS) % Cin);
    const int o = (int)(i / ((int64_t)RS * Cin));
    const float v = dw[(int64_t)o * row_ld + (int64_t)t * cin_stride + c];
    g[i] = (beta == 0.f) ? v : fmaf(beta, g[i], v);
  }
}

// k x k case (RS <= 9, dense rows): for one output channel both layouts are ONE contiguous block of RS*Cin floats, so a
// block stages a [RS][512-channel] slab in shared memory with coalesced reads and writes it back permuted, coalesced too
// (the generic kernel above reads with a stride of Cin floats: 8x sector overfetch, 22 launches = 0.29 ms per step).
constexpr int kUnpackChunk = 512;
__global__ void __launch_bounds__(kT)
unpack_wgrad_tiled_kernel(const float* __restrict__ dw, int Cin, int RS, float beta, float* __restrict__ g) {
  pdl_wait();
  pdl_launch();
  __shared__ float s_t[9][kUnpackChunk + 1];
  const int o = blockIdx.x;
  const int cb = blockIdx.y * kUnpackChunk;
  const int nc = min(kUnpackChunk, Cin - cb);
  const float* src = dw + (int64_t)o * RS * Cin + cb;
  for (int t = 0; t < RS; t++)
    for (int c = threadIdx.x; c < nc; c += kT) s_t[t][c] = src[(int64_t)t * Cin + c];
  __syncthreads();
  float* dst = g + ((int64_t)o * Cin + cb) * RS;
  const int n = nc * RS;
  for (int i = threadIdx.x; i < n; i += kT) {
    const int c = i / RS, t = i - c * RS;
    const float v = s_t[t][c];
    dst[i] = (beta == 0.f) ? v : fmaf(beta, dst[i], v);
  }
}

// every k x k convolution's weight-gradient accumulator unpacked in ONE launch at the end of the backward sweep (22
// per-layer launches were mostly launch boundaries on the weight-gradient stream); blocks find their job by binary search
struct UnpackJob {
  const float* src;
  float* dst;
  int Cout, Cin, RS, chunks;
  int blk_begin, pad_;
};
__global__ void __launch_bounds__(kT)
unpack_wgrad_batched_kernel(const UnpackJob* __restrict__ jobs, int n_jobs) {
  pdl_wait();
  pdl_launch();
  __shared__ float s_t[9][kUnpackChunk + 1];
  int lo = 0, hi = n_jobs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].blk_begin <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const UnpackJob jb = jobs[lo];
  const int local = blockIdx.x - jb.blk_begin;
  const int o = local / jb.chunks, cb = (local - o * jb.chunks) * kUnpackChunk;
  if (o >= jb.Cout) return;
  const int nc = min(kUnpackChunk, jb.Cin - cb);
  const float* src = jb.src + (int64_t)o * jb.RS * jb.Cin + cb;
  for (int t = 0; t < jb.RS; t++)
    for (int c = threadIdx.x; c < nc; c += kT) s_t[t][c] = src[(int64_t)t * jb.Cin + c];
  __syncthreads();
  float* dst = jb.dst + ((int64_t)o * jb.Cin + cb) * jb.RS;
  const int n = nc * jb.RS;
  for (int i = threadIdx.x; i < n; i += kT) {
    const int c = i / jb.RS, t = i - c * jb.RS;
    dst[i] += s_t[t][c];                 // gradients ACCUMULATE into .grad (zeroed by the sweep when it is fresh)
  }
}

// all convolutions' weights packed in ONE launch. Blocks are dealt to jobs in proportion to their size
// (blk_begin / blk_count, filled in by the host); a block finds its job by binary search.
struct PackJob {
  const float* w;
  __nv_bfloat16* dst;
  int Cout, Cin, RS, pad, row_ld, mode;   // mode 0: forward operand (pad = cin_pad), 1: dgrad operand (pad = cout_pad), 2: stem row taps
  int blk_begin, blk_count;               // this job owns blocks [blk_begin, blk_begin + blk_count)
};
__global__ void __launch_bounds__(kT)
pack_weights_batched_kernel(const PackJob* __restrict__ jobs, int n_jobs) {
  pdl_wait();
  pdl_launch();
  // Both packings are transposes of small matrices, staged through shared memory so that the fp32 reads AND the
  // bf16 writes are coalesced (the source is [Cout][Cin][RS] with RS innermost).
  __shared__ float tile[64 * 65];
  int lo = 0, hi = n_jobs - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (jobs[mid].blk_begin <= (int)blockIdx.x) lo = mid; else hi = mid - 1;
  }
  const PackJob j = jobs[lo];
  const int lb = (int)blockIdx.x - j.blk_begin, nb = j.blk_count;
  if (lb >= nb) return;
  const int tid = threadIdx.x;
  if (j.mode == 0 && j.RS == 1 && (j.Cin & 7) == 0) {
    // 1x1 forward operand: dst[o][c] = w[o][c], zero padded to `pad` channels: 8 elements per thread
    const int vec_per_row = j.pad >> 3;
    const int64_t total = (int64_t)j.Cout * vec_per_row;
    for (int64_t i = (int64_t)lb * kT + tid; i < total; i += (int64_t)nb * kT) {
      const int o = (int)(i / vec_per_row), c = (int)(i - (int64_t)o * vec_per_row) << 3;
      F8 f;
      if (c < j.Cin) {
        const float4 a = *reinterpret_cast<const float4*>(j.w + (int64_t)o * j.Cin + c);
        const float4 b2 = *reinterpret_cast<const float4*>(j.w + (int64_t)o * j.Cin + c + 4);
        f.v[0] = a.x; f.v[1] = a.y; f.v[2] = a.z; f.v[3] = a.w; f.v[4] = b2.x; f.v[5] = b2.y; f.v[6] = b2.z; f.v[7] = b2.w;
      } else {
#pragma unroll
        for (int k = 0; k < 8; k++) f.v[k] = 0.f;
      }
      store8(j.dst + (int64_t)o * j.row_ld + c, f);
    }
  } else if (j.mode == 0 && j.pad >= 64 && j.RS <= 16) {
    // k x k forward operand: dst[o][t][c] <- w[o][c][t]. unit = (o, 256-channel chunk): RS*256 contiguous floats in
    // (every thread has RS independent loads in flight), RS rows of 256 bf16 out, 8 channels per store.
    const int RS = j.RS;
    const int cchunks = (j.pad + 255) >> 8;
    const int units = j.Cout * cchunks;
    for (int u = lb; u < units; u += nb) {
      const int o = u / cchunks, c0 = (u - o * cchunks) << 8;
      const int ncp = min(256, j.pad - c0);               // padded channels of this chunk (multiple of 64)
      const int nc = max(0, min(256, j.Cin - c0));        // valid channels
      const float* src = j.w + ((int64_t)o * j.Cin + c0) * RS;
      __syncthreads();
      for (int i = tid; i < nc * RS; i += kT) tile[i] = src[i];          // tile[c*RS + t]
      __syncthreads();
      const int vecs = ncp >> 3;
      for (int i = tid; i < RS * vecs; i += kT) {
        const int t = i / vecs, c = (i - t * vecs) << 3;
        F8 f;
#pragma unroll
        for (int k = 0; k < 8; k++) f.v[k] = (c + k < nc) ? tile[(c + k) * RS + t] : 0.f;
        store8(j.dst + (int64_t)o * j.row_ld + (int64_t)t * j.pad + c0 + c, f);
      }
    }
  } else if (j.mode == 2) {
    // stem, row-tap form: dst[o][r][q] with q = s*Cin + c (kernel column s, input channel c), zero padded to `pad` per kernel
    // row r: the operand of the 7-tap convolution over the x-unrolled image rows (stem_rows_kernel)
    int ks = 1;
    while (ks * ks < j.RS) ks++;
    const int64_t total = (int64_t)j.Cout * j.row_ld;
    for (int64_t i = (int64_t)lb * kT + tid; i < total; i += (int64_t)nb * kT) {
      const int o = (int)(i / j.row_ld), k = (int)(i % j.row_ld);
      const int r = k / j.pad, q = k % j.pad;
      const int sx = q / j.Cin, c = q % j.Cin;
      float v = 0.f;
      if (r < ks && sx < ks) v = j.w[((int64_t)o * j.Cin + c) * j.RS + r * ks + sx];
      j.dst[i] = __float2bfloat16_rn(v);
    }
  } else if (j.mode == 0) {
    // anything else (the stem's im2col form: pad = Cin = 3, RS = 49): element-wise
    const int64_t total = (int64_t)j.Cout * j.row_ld;
    for (int64_t i = (int64_t)lb * kT + tid; i < total; i += (int64_t)nb * kT) {
      const int o = (int)(i / j.row_ld), k = (int)(i % j.row_ld);
      const int t = k / j.pad, c = k % j.pad;
      float v = 0.f;
      if (t < j.RS && c < j.Cin) v = j.w[((int64_t)o * j.Cin + c) * j.RS + t];
      j.dst[i] = __float2bfloat16_rn(v);
    }
  } else {
    // dgrad operand: dst[f][o] (f = c*RS + t, o padded to `pad`) <- w[o][f]: a [Cout x F] -> [F x pad] transpose,
    // 64 x 64 tiles; writes are 8 output channels (16 bytes) per thread
    const int F = j.Cin * j.RS;
    const int ftiles = (F + 63) >> 6, otiles = j.pad >> 6;
    const int units = ftiles * otiles;
    for (int u = lb; u < units; u += nb) {
      const int ot = u / ftiles, ft = u - ot * ftiles;
      const int o0 = ot << 6, f0 = ft << 6;
      __syncthreads();
#pragma unroll 4
      for (int i = tid; i < 64 * 64; i += kT) {
        const int o = i >> 6, f = i & 63;
        tile[o * 65 + f] = (o0 + o < j.Cout && f0 + f < F) ? j.w[(int64_t)(o0 + o) * F + f0 + f] : 0.f;
      }
      __syncthreads();
      for (int i = tid; i < 64 * 8; i += kT) {
        const int f = i >> 3, o = (i & 7) << 3;
        if (f0 + f < F) {
          F8 v;
#pragma unroll
          for (int k = 0; k < 8; k++) v.v[k] = tile[(o + k) * 65 + f];
          // row_ld > 0: this tensor's RS taps are a slice of a K-CONCATENATED row of row_ld taps (dst points at the slice's
          // first tap): row (c, t) lands at c * row_ld + t instead of c * RS + t
          const int64_t rowi = j.row_ld > 0 ? (int64_t)((f0 + f) / j.RS) * j.row_ld + (f0 + f) % j.RS : (int64_t)(f0 + f);
          store8(j.dst + rowi * j.pad + o0 + o, v);
        }
      }
    }
  }
}

// ---------------------------------------------------------------------------
// BatchNorm kernels share one thread layout: blockDim = 256 = nx * ny (+ idle), tx = channel group
// (8 channels = 16 bytes), ty = row lane. Per-channel constants live in registers; a block walks
// its row range with several rows in flight per thread, so there is no per-element index math.

// Row walk shared by the three kernels: thread (tx, ty) owns channels [8tx, 8tx+8) of rows r0+ty, r0+ty+ny, ...
// of its block; pointers advance by a fixed stride (no per-row 64-bit multiplies) and the main loop handles U rows
// per trip without bounds checks (U independent 16-byte loads per tensor in flight), a scalar tail the rest.
// dropout seed of one launch: a by-value part plus an optional per-step counter read from DEVICE memory, so that a train
// step captured in a CUDA graph draws a fresh mask on every replay (effective seed = seed + 1000003 * *step, 48 bits)
struct DropSeed {
  uint64_t seed;
  const long long* step;
  __device__ __forceinline__ uint64_t resolve() const {
    return (seed + (step ? (uint64_t)(*step) * 1000003ull : 0ull)) & 0xFFFFFFFFFFFFull;
  }
};

// BatchNorm training forward: stats -> normalise (+residual, ReLU, dropout)
// GCNT (synchronised BatchNorm): `stats` holds the sums over every rank's rows (one copy) followed by the global row count at
// [2C]; the count normalises and sets the running-variance factor, M only bounds this rank's row walk
template <bool RES, bool RELU, bool DROP, bool GCNT = false>
__global__ void __launch_bounds__(kT, 3)
bn_train_apply_kernel(const __nv_bfloat16* __restrict__ x, int x_ld, const double* __restrict__ stats, int stats_rep,
                      int64_t M, int C, const float* __restrict__ gamma, const float* __restrict__ beta,
                      float eps, float momentum, float* running_mean, float* running_var,
                      long long* nbt, float* save_mean, float* save_invstd,
                      const __nv_bfloat16* __restrict__ res, int res_ld, float drop_p,
                      DropSeed drop_seed_in, __nv_bfloat16* __restrict__ out, int out_ld, int nx, int ny,
                      int rows_per_block, uint8_t* __restrict__ relu_bits) {
  pdl_wait();
  pdl_launch();
  const uint64_t drop_seed = DROP ? drop_seed_in.resolve() : 0ull;
  const int tx = threadIdx.x % nx, ty = threadIdx.x / nx;
  // statistics spread over several copies (narrow convolutions, iswm_conv_desc.stats_replicas; C <= 128 there): the block folds
  // them once into shared memory - one value per thread - instead of every thread summing the copies of its 8 channels
  __shared__ double s_stat[256];
  const bool folded = stats_rep > 1 && 2 * C <= 256;
  if (folded) {
    for (int i = threadIdx.x; i < 2 * C; i += kT) {
      double a = stats[i];
      for (int r = 1; r < stats_rep; r++) a += stats[(size_t)r * 2 * C + i];
      s_stat[i] = a;
    }
    __syncthreads();
  }
  if (ty >= ny) return;
  const int c0 = tx << 3;
  // the first U rows are requested BEFORE the per-channel constants (a chain of dependent global loads and fp64
  // math): the two latencies overlap, which is most of a thread's life on small tensors
  constexpr int U = 4;
  const RowWalk w = row_walk(M, rows_per_block, ty, ny);
  const __nv_bfloat16* px = x + w.first * x_ld + c0;
  const __nv_bfloat16* pr = RES ? res + w.first * res_ld + c0 : nullptr;
  const int64_t sx = (int64_t)ny * x_ld, sr = (int64_t)ny * res_ld;
  uint4 fr[U], rr[U];
  const bool pre = w.n >= U;
  if (pre) {
#pragma unroll
    for (int u = 0; u < U; u++) {
      fr[u] = load_raw(px + u * sx);
      if (RES) rr[u] = load_raw(pr + u * sr);
    }
  }
  const double cnt = GCNT ? stats[2 * C] : 0.0;
  const double invM = GCNT ? 1.0 / cnt : 1.0 / (double)M;
  float sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const int c = c0 + j;
    // fp64 sums (see conv_igemm.cu): E[x^2] - mean^2 without cancellation trouble, rounded to fp32 once
    double s1, s2;
    if (folded) {
      s1 = s_stat[c]; s2 = s_stat[C + c];
    } else {
      s1 = stats[c]; s2 = stats[C + c];
      for (int r = 1; r < stats_rep; r++) {       // copies filled by different CTAs of the convolution (fixed order; fp64)
        s1 += stats[(size_t)r * 2 * C + c];
        s2 += stats[(size_t)r * 2 * C + C + c];
      }
    }
    const double mean_d = s1 * invM;
    const float mean = (float)mean_d;
    const float var = fmaxf((float)(s2 * invM - mean_d * mean_d), 0.f);
    const float invstd = rsqrtf(var + eps);
    sc[j] = gamma[c] * invstd;
    sh[j] = fmaf(-mean, sc[j], beta[c]);          // same expression in the backward kernels (mask recomputation)
    if (blockIdx.x == 0 && ty == 0) {
      if (save_mean) save_mean[c] = mean;
      if (save_invstd) save_invstd[c] = invstd;
      if (running_mean) {
        float unbiased;
        if (GCNT) unbiased = (cnt > 1.0) ? var * ((float)cnt / (float)(cnt - 1.0)) : var;
        else unbiased = (M > 1) ? var * ((float)M / (float)(M - 1)) : var;
        running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * mean;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * unbiased;
      }
    }
  }
  if (blockIdx.x == 0 && threadIdx.x == 0 && nbt) *nbt += 1;
  const float keep_scale = DROP ? 1.f / (1.f - drop_p) : 1.f;
  __nv_bfloat16* po = out + w.first * out_ld + c0;
  const int64_t so = (int64_t)ny * out_ld;
  uint64_t didx = (uint64_t)w.first * C + c0;                 // dropout counter of this thread's first element
  const uint64_t sd = (uint64_t)ny * C;
  // ReLU sign bits of this thread's 8 channels, one byte per (row, channel group): the backward kernels of residual
  // units read it instead of the 16-byte activation (the mask cannot be recomputed from x alone there)
  uint8_t* pb = relu_bits ? relu_bits + w.first * (C >> 3) + tx : nullptr;
  const int64_t sb = (int64_t)ny * (C >> 3);
  auto one = [&](const uint4& f4, const uint4& r4, __nv_bfloat16* o, uint64_t di, uint8_t* ob) {
    F8 f = unpack8(f4);
#pragma unroll
    for (int j = 0; j < 8; j++) f.v[j] = fmaf(f.v[j], sc[j], sh[j]);
    if (RES) {
      const F8 r = unpack8(r4);
#pragma unroll
      for (int j = 0; j < 8; j++) f.v[j] += r.v[j];
    }
    if (RELU) {
      if (ob) {
        unsigned bits = 0;
#pragma unroll
        for (int j = 0; j < 8; j++) bits |= (f.v[j] > 0.f) ? (1u << j) : 0u;
        *ob = (uint8_t)bits;
      }
#pragma unroll
      for (int j = 0; j < 8; j++) f.v[j] = fmaxf(f.v[j], 0.f);
    }
    if (DROP) {
#pragma unroll
      for (int j = 0; j < 8; j++) f.v[j] = drop_keep(drop_seed, di + j, drop_p) ? f.v[j] * keep_scale : 0.f;
    }
    store8(o, f);
  };
  int i = 0;
  for (; i + U <= w.n; i += U) {
    if (i > 0) {
#pragma unroll
      for (int u = 0; u < U; u++) {
        fr[u] = load_raw(px + u * sx);
        if (RES) rr[u] = load_raw(pr + u * sr);
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) one(fr[u], rr[u], po + u * so, didx + u * sd, pb ? pb + u * sb : nullptr);
    px += U * sx; po += U * so; didx += U * sd;
    if (RES) pr += U * sr;
    if (pb) pb += U * sb;
  }
  for (; i < w.n; i++) {
    const uint4 f4 = load_raw(px);
    uint4 r4 = f4;
    if (RES) r4 = load_raw(pr);
    one(f4, r4, po, didx, pb);
    px += sx; po += so; didx += sd;
    if (RES) pr += sr;
    if (pb) pb += sb;
  }
}

__global__ void bn_fold_kernel(const float* gamma, const float* beta, const float* mean,
                               const float* var, float eps, int C, float* scale, float* shift) {
  pdl_wait();
  pdl_launch();
  const int c = blockIdx.x * kT + threadIdx.x;
  if (c < C) {
    const float sc = gamma[c] / sqrtf(var[c] + eps);
    scale[c] = sc;
    shift[c] = beta[c] - mean[c] * sc;
  }
}

// BatchNorm backward pass 1: per-channel sum(dz), sum(dz * xhat). MASK: 0 none, 1 from the stored activation
// (residual units), 2 recomputed from x with the forward kernel's own scale/shift arithmetic (one tensor read less).
// The loop accumulates sum(dz) and sum(dz * x); sum(dz * xhat) = invstd * (sum(dz*x) - mean * sum(dz)) is formed once
// per block in fp64.
template <int MASK, bool DROP>
__global__ void __launch_bounds__(kT, 3)
bn_bwd_reduce_kernel(const __nv_bfloat16* __restrict__ dout, int dout_ld,
                     const __nv_bfloat16* __restrict__ x, int x_ld,
                     const __nv_bfloat16* __restrict__ act, int act_ld, int64_t M, int C,
                     const float* __restrict__ mean, const float* __restrict__ invstd,
                     const float* __restrict__ gamma, const float* __restrict__ beta,
                     float drop_p, DropSeed drop_seed_in, double* __restrict__ sums, int nx, int ny,
                     int rows_per_block) {
  pdl_wait();
  pdl_launch();
  const uint64_t drop_seed = DROP ? drop_seed_in.resolve() : 0ull;
  __shared__ float s_red[kT * 16];
  const int tx = threadIdx.x % nx, ty = threadIdx.x / nx;
  const float keep_scale = DROP ? 1.f / (1.f - drop_p) : 1.f;
  // blockIdx.y = channel group of nx*8 channels: wide layers are cut into 256-channel groups so that a block ends with
  // 2*256 fp64 atomics instead of 2*C (C = 2048: 1.8 M same-address-heavy atomics per launch were a 10-20 us tail)
  const int cbase = blockIdx.y * (nx << 3);
  const int c0 = cbase + (tx << 3);
  constexpr int U = 4;
  // first batch of rows requested before the per-channel constants are loaded (overlapping latencies)
  const bool live = (ty < ny) && (c0 < C);
  const RowWalk w = live ? row_walk(M, rows_per_block, ty, ny) : RowWalk{0, 0};
  const __nv_bfloat16* pg = dout + w.first * dout_ld + c0;
  const __nv_bfloat16* px = x + w.first * x_ld + c0;
  const __nv_bfloat16* pa = (MASK == 1) ? act + w.first * act_ld + c0 : nullptr;
  const uint8_t* pm = (MASK == 3) ? reinterpret_cast<const uint8_t*>(act) + w.first * (C >> 3) + (c0 >> 3) : nullptr;
  const int64_t sm_ = (int64_t)ny * (C >> 3);
  const int64_t sg = (int64_t)ny * dout_ld, sx = (int64_t)ny * x_ld, sa = (int64_t)ny * act_ld;
  uint4 gr[U], xr[U], orr[U];
  if (w.n >= U) {
#pragma unroll
    for (int u = 0; u < U; u++) {
      gr[u] = load_raw(pg + u * sg);
      xr[u] = load_raw(px + u * sx);
      if (MASK == 1) orr[u] = load_raw(pa + u * sa); else if (MASK == 3) { orr[u] = gr[u]; orr[u].x = pm[u * sm_]; } else orr[u] = gr[u];
    }
  }
  float a[8], b[8], sc[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; j++) {
    a[j] = 0.f; b[j] = 0.f;
    if (MASK == 2 && live) {
      sc[j] = gamma[c0 + j] * invstd[c0 + j];
      sh[j] = fmaf(-mean[c0 + j], sc[j], beta[c0 + j]);
    } else {
      sc[j] = 0.f; sh[j] = 0.f;
    }
  }
  if (live) {
    uint64_t didx = (uint64_t)w.first * C + c0;
    const uint64_t sd = (uint64_t)ny * C;
    auto one = [&](const uint4& gr, const uint4& xr, const uint4& orr, uint64_t di) {
      F8 g = unpack8(gr);
      const F8 xv = unpack8(xr);
      if (MASK == 1) {
        const F8 o = unpack8(orr);
#pragma unroll
        for (int j = 0; j < 8; j++) g.v[j] = (o.v[j] > 0.f) ? g.v[j] : 0.f;
      } else if (MASK == 3) {
        const unsigned bits = orr.x;
#pragma unroll
        for (int j = 0; j < 8; j++) g.v[j] = ((bits >> j) & 1u) ? g.v[j] : 0.f;
      } else if (MASK == 2) {
#pragma unroll
        for (int j = 0; j < 8; j++) g.v[j] = (fmaf(xv.v[j], sc[j], sh[j]) > 0.f) ? g.v[j] : 0.f;
      }
      if (DROP) {
#pragma unroll
        for (int j = 0; j < 8; j++) g.v[j] = drop_keep(drop_seed, di + j, drop_p) ? g.v[j] * keep_scale : 0.f;
      }
#pragma unroll
      for (int j = 0; j < 8; j++) {
        a[j] += g.v[j];
        b[j] = fmaf(g.v[j], xv.v[j], b[j]);
      }
    };
    int i = 0;
    for (; i + U <= w.n; i += U) {
      if (i > 0) {
#pragma unroll
        for (int u = 0; u < U; u++) {
          gr[u] = load_raw(pg + u * sg);
          xr[u] = load_raw(px + u * sx);
          if (MASK == 1) orr[u] = load_raw(pa + u * sa); else if (MASK == 3) { orr[u] = gr[u]; orr[u].x = pm[u * sm_]; } else orr[u] = gr[u];
        }
      }
#pragma unroll
      for (int u = 0; u < U; u++) one(gr[u], xr[u], orr[u], didx + u * sd);
      pg += U * sg; px += U * sx; didx += U * sd;
      if (MASK == 1) pa += U * sa;
      if (MASK == 3) pm += U * sm_;
    }
    for (; i < w.n; i++) {
      const uint4 g1 = load_raw(pg), x1 = load_raw(px);
      uint4 o1 = g1;
      if (MASK == 1) o1 = load_raw(pa);
      if (MASK == 3) o1.x = *pm;
      one(g1, x1, o1, didx);
      pg += sg; px += sx; didx += sd;
      if (MASK == 1) pa += sa;
      if (MASK == 3) pm += sm_;
    }
  }
#pragma unroll
  for (int j = 0; j < 8; j++) {
    s_red[threadIdx.x * 16 + j] = a[j];
    s_red[threadIdx.x * 16 + 8 + j] = b[j];
  }
  __syncthreads();
  // one thread per channel of the block's channel range: fixed-order sum over ty, xhat fix-up in fp64, two atomics
  for (int o = threadIdx.x; o < nx * 8; o += kT) {
    const int gx = o >> 3, j = o & 7;
    float ta = 0.f, tb = 0.f;
    for (int y = 0; y < ny; y++) {
      ta += s_red[(y * nx + gx) * 16 + j];
      tb += s_red[(y * nx + gx) * 16 + 8 + j];
    }
    const int c = cbase + (gx << 3) + j;
    if (c < C) {
      atomicAdd(sums + c, (double)ta);
      atomicAdd(sums + C + c, (double)invstd[c] * ((double)tb - (double)mean[c] * (double)ta));
    }
  }
}

// BatchNorm backward pass 2
// GCNT (synchronised BatchNorm): `sums` are the sums over every rank's rows with the global row count at [2C], and
// dgamma / dbeta accumulate this rank's own sums `lsums` (the gradient all-reduce adds the other ranks')
template <int MASK, bool DROP, bool DZ, bool GCNT = false>
__global__ void __launch_bounds__(kT, 3)
bn_bwd_apply_kernel(const __nv_bfloat16* __restrict__ dout, int dout_ld,
                    const __nv_bfloat16* __restrict__ x, int x_ld,
                    const __nv_bfloat16* __restrict__ act, int act_ld, int64_t M, int C,
                    const float* __restrict__ gamma, const float* __restrict__ beta, const float* __restrict__ mean,
                    const float* __restrict__ invstd, const double* __restrict__ sums,
                    float drop_p, DropSeed drop_seed_in, __nv_bfloat16* __restrict__ dx, int dx_ld,
                    __nv_bfloat16* __restrict__ dz, int dz_ld, float* dgamma, float* dbeta, int nx,
                    int ny, int rows_per_block, const double* __restrict__ lsums) {
  pdl_wait();
  pdl_launch();
  const uint64_t drop_seed = DROP ? drop_seed_in.resolve() : 0ull;
  const int tx = threadIdx.x % nx, ty = threadIdx.x / nx;
  if (ty >= ny) return;
  const int c0 = tx << 3;
  constexpr int U = 4;
  // first batch of rows requested before the per-channel constants are loaded (overlapping latencies)
  const RowWalk w = row_walk(M, rows_per_block, ty, ny);
  const __nv_bfloat16* pg = dout + w.first * dout_ld + c0;
  const __nv_bfloat16* px = x + w.first * x_ld + c0;
  const __nv_bfloat16* pa = (MASK == 1) ? act + w.first * act_ld + c0 : nullptr;
  const uint8_t* pm = (MASK == 3) ? reinterpret_cast<const uint8_t*>(act) + w.first * (C >> 3) + tx : nullptr;
  const int64_t sm_ = (int64_t)ny * (C >> 3);
  const int64_t sg = (int64_t)ny * dout_ld, sx = (int64_t)ny * x_ld, sa_ = (int64_t)ny * act_ld;
  uint4 gr[U], xr[U], orr[U];
  if (w.n >= U) {
#pragma unroll
    for (int u = 0; u < U; u++) {
      gr[u] = load_raw(pg + u * sg);
      xr[u] = load_raw(px + u * sx);
      if (MASK == 1) orr[u] = load_raw(pa + u * sa_); else if (MASK == 3) { orr[u] = gr[u]; orr[u].x = pm[u * sm_]; } else orr[u] = gr[u];
    }
  }
  const float invM = GCNT ? 1.0f / (float)sums[2 * C] : 1.0f / (float)M;
  // dx = k*dz + p*x + q  with  k = gamma*invstd, p = -k*invstd*mean(dz*xhat), q = -k*mean(dz) - p*mu
  float kk[8], pp[8], qq[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; j++) {
    const int c = c0 + j;
    const float is = invstd[c], mu = mean[c];
    const float k = gamma[c] * is;
    sh[j] = (MASK == 2) ? fmaf(-mu, k, beta[c]) : 0.f;
    const float sa = (float)sums[c], sb = (float)sums[C + c];
    const float ma = sa * invM, mb = sb * invM;
    kk[j] = k;
    pp[j] = -k * is * mb;
    qq[j] = -k * ma - pp[j] * mu;
    if (blockIdx.x == 0 && ty == 0) {
      if (dbeta) dbeta[c] += GCNT ? (float)lsums[c] : sa;
      if (dgamma) dgamma[c] += GCNT ? (float)lsums[C + c] : sb;
    }
  }
  const float keep_scale = DROP ? 1.f / (1.f - drop_p) : 1.f;
  __nv_bfloat16* pdx = dx + w.first * dx_ld + c0;
  __nv_bfloat16* pdz = DZ ? dz + w.first * dz_ld + c0 : nullptr;
  const int64_t sdx = (int64_t)ny * dx_ld, sdz = (int64_t)ny * dz_ld;
  uint64_t didx = (uint64_t)w.first * C + c0;
  const uint64_t sd = (uint64_t)ny * C;
  auto one = [&](const uint4& gr, const uint4& xr, const uint4& orr, __nv_bfloat16* odx, __nv_bfloat16* odz, uint64_t di) {
    F8 g = unpack8(gr);
    const F8 xv = unpack8(xr);
    if (MASK == 1) {
      const F8 o = unpack8(orr);
#pragma unroll
      for (int j = 0; j < 8; j++) g.v[j] = (o.v[j] > 0.f) ? g.v[j] : 0.f;
    } else if (MASK == 3) {
      const unsigned bits = orr.x;
#pragma unroll
      for (int j = 0; j < 8; j++) g.v[j] = ((bits >> j) & 1u) ? g.v[j] : 0.f;
    } else if (MASK == 2) {
#pragma unroll
      for (int j = 0; j < 8; j++) g.v[j] = (fmaf(xv.v[j], kk[j], sh[j]) > 0.f) ? g.v[j] : 0.f;
    }
    if (DROP) {
#pragma unroll
      for (int j = 0; j < 8; j++) g.v[j] = drop_keep(drop_seed, di + j, drop_p) ? g.v[j] * keep_scale : 0.f;
    }
    if (DZ) store8(odz, g);
    F8 r;
#pragma unroll
    for (int j = 0; j < 8; j++) r.v[j] = fmaf(kk[j], g.v[j], fmaf(pp[j], xv.v[j], qq[j]));
    store8(odx, r);
  };
  int i = 0;
  for (; i + U <= w.n; i += U) {
    if (i > 0) {
#pragma unroll
      for (int u = 0; u < U; u++) {
        gr[u] = load_raw(pg + u * sg);
        xr[u] = load_raw(px + u * sx);
        if (MASK == 1) orr[u] = load_raw(pa + u * sa_); else if (MASK == 3) { orr[u] = gr[u]; orr[u].x = pm[u * sm_]; } else orr[u] = gr[u];
      }
    }
#pragma unroll
    for (int u = 0; u < U; u++) one(gr[u], xr[u], orr[u], pdx + u * sdx, DZ ? pdz + u * sdz : nullptr, didx + u * sd);
    pg += U * sg; px += U * sx; pdx += U * sdx; didx += U * sd;
    if (MASK == 1) pa += U * sa_;
    if (MASK == 3) pm += U * sm_;
    if (DZ) pdz += U * sdz;
  }
  for (; i < w.n; i++) {
    const uint4 g1 = load_raw(pg), x1 = load_raw(px);
    uint4 o1 = g1;
    if (MASK == 1) o1 = load_raw(pa);
      if (MASK == 3) o1.x = *pm;
    one(g1, x1, o1, pdx, pdz, didx);
    pg += sg; px += sx; pdx += sdx; didx += sd;
    if (MASK == 1) pa += sa_;
    if (MASK == 3) pm += sm_;
    if (DZ) pdz += sdz;
  }
}

// ---------------------------------------------------------------------------
// stem im2col: NCHW fp32 image -> [B*Ho*Wo][Kpad] bf16, col = (r*7+s)*Cin + c.
// One block per (image, output row, 64-pixel strip): the 7-row input patch is staged in shared memory with
// coalesced reads along W, then every thread emits 16-byte chunks of consecutive output rows.
constexpr int kStemStrip = 64;
constexpr int kStemPatchW = 2 * kStemStrip + 5;           // 133 input columns feed 64 stride-2 outputs
// Stem, row-tap form (network/backbone/resnet.py:144: 7x7 / stride 2 / pad 3 on a 3-channel image). The image is unrolled
// along x ONLY: out[p][b][hh][wo][s*Cin + c] = img[b][c][2*hh + p][2*wo + s - 3] (zero outside the image, kpitch - 7*Cin
// zero channels of padding), p = row parity. The 7 kernel ROWS then run as 7 taps of the ordinary implicit GEMM over the two
// parity phases (tap r reads phase (r+1)&1 at row offset (r-3-p)/2), so the matrix the GEMM reads is 48 bytes per output
// pixel and row instead of the 320-byte rows of a full 7x7 im2col: 100 MB instead of 335 MB at cfg2, and the fill is a plain
// streaming kernel. One thread = one (p, b, hh, wo) pixel = kpitch bf16.
template <int CIN>
__global__ void __launch_bounds__(kT)
stem_rows_kernel(const float* __restrict__ img, int B, int H, int W, int Hh, int Wo, int kpitch,
                 __nv_bfloat16* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int64_t total = 2ll * B * Hh * Wo;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int wo = (int)(i % Wo);
    int64_t r = i / Wo;
    const int hh = (int)(r % Hh);
    r /= Hh;
    const int b = (int)(r % B), p = (int)(r / B);
    const int h = 2 * hh + p;
    float v[24];
#pragma unroll
    for (int k = 0; k < 24; k++) v[k] = 0.f;
    if (h < H) {
#pragma unroll
      for (int c = 0; c < CIN; c++) {
        const float* row = img + (((int64_t)b * CIN + c) * H + h) * W;
#pragma unroll
        for (int sx = 0; sx < 7; sx++) {
          const int w = 2 * wo + sx - 3;
          v[sx * CIN + c] = (w >= 0 && w < W) ? __ldg(row + w) : 0.f;
        }
      }
    }
    __nv_bfloat16* o = out + i * kpitch;
#pragma unroll
    for (int k = 0; k < 24; k += 8) {
      F8 f;
#pragma unroll
      for (int e = 0; e < 8; e++) f.v[e] = v[k + e];
      store8(o + k, f);
    }
    for (int k = 24; k < kpitch; k += 8) {
      F8 f;
#pragma unroll
      for (int e = 0; e < 8; e++) f.v[e] = 0.f;
      store8(o + k, f);
    }
  }
}
// weight-gradient accumulator of the row-tap stem [Cout][ks][kpitch] (q = s*Cin + c) -> fp32 OIHW gradient
__global__ void unpack_wgrad_stem_kernel(const float* __restrict__ dw, int Cout, int Cin, int ks, int kpitch, float beta,
                                         float* __restrict__ g) {
  pdl_wait();
  pdl_launch();
  const int total = Cout * Cin * ks * ks;
  for (int i = blockIdx.x * kT + threadIdx.x; i < total; i += gridDim.x * kT) {
    const int sx = i % ks, r = (i / ks) % ks, c = (i / (ks * ks)) % Cin, o = i / (ks * ks * Cin);
    const float v = dw[((int64_t)o * ks + r) * kpitch + sx * Cin + c];
    g[i] = (beta == 0.f) ? v : fmaf(beta, g[i], v);
  }
}

__global__ void __launch_bounds__(kT)
stem_im2col_kernel(const float* __restrict__ img, int B, int Cin, int H, int W, int Ho, int Wo,
                   int Kpad, __nv_bfloat16* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  extern __shared__ float patch[];                          // [Cin][7][kStemPatchW + 1]
  constexpr int PW = kStemPatchW + 1;
  const int strips = (Wo + kStemStrip - 1) / kStemStrip;
  const int wo0 = (blockIdx.x % strips) * kStemStrip;
  const int ho = (blockIdx.x / strips) % Ho;
  const int b = blockIdx.x / (strips * Ho);
  const int wi0 = 2 * wo0 - 3, hi0 = 2 * ho - 3;
  for (int i = threadIdx.x; i < Cin * 7 * kStemPatchW; i += kT) {
    const int col = i % kStemPatchW, rc = i / kStemPatchW;
    const int r = rc % 7, c = rc / 7;
    const int hi = hi0 + r, wi = wi0 + col;
    float v = 0.f;
    if (hi >= 0 && hi < H && wi >= 0 && wi < W) v = __ldg(img + (((int64_t)b * Cin + c) * H + hi) * W + wi);
    patch[(c * 7 + r) * PW + col] = v;
  }
  // column k of the im2col row -> offset of its tap inside the patch (-1: zero padding of K up to Kpad)
  __shared__ int koff[256];
  const int K = 49 * Cin;
  for (int k = threadIdx.x; k < Kpad; k += kT) {
    int off = -1;
    if (k < K) {
      const int t = k / Cin, c = k - t * Cin;
      const int r = t / 7, sx = t - r * 7;
      off = (c * 7 + r) * PW + sx;
    }
    koff[k] = off;
  }
  __syncthreads();
  const int koct = Kpad >> 3;
  const int npx = min(kStemStrip, Wo - wo0);
  const int64_t m0 = ((int64_t)b * Ho + ho) * Wo + wo0;
  // thread -> one 16-byte chunk position ko of the im2col row (its 8 patch offsets live in registers) and a pixel lane:
  // consecutive threads write consecutive chunks of one row (coalesced), and the inner loop is 8 shared-memory loads per
  // 16-byte store instead of 16 (the offset table is not re-read per pixel)
  const int ko = threadIdx.x % koct, pl = threadIdx.x / koct, npl = kT / koct;
  if (pl < npl) {
    int offs[8];
#pragma unroll
    for (int jj = 0; jj < 8; jj++) offs[jj] = koff[ko * 8 + jj];
    for (int px = pl; px < npx; px += npl) {
      const float* pp = patch + 2 * px;
      F8 f;
#pragma unroll
      for (int jj = 0; jj < 8; jj++) f.v[jj] = offs[jj] >= 0 ? pp[offs[jj]] : 0.f;
      store8(out + (m0 + px) * Kpad + ko * 8, f);
    }
  }
}

// ---------------------------------------------------------------------------
// MaxPool2d(3, 2, 1)
__global__ void __launch_bounds__(kT)
maxpool_fwd_kernel(const __nv_bfloat16* __restrict__ x, int B, int H, int W, int C, int Ho, int Wo,
                   __nv_bfloat16* __restrict__ out, uint8_t* __restrict__ idx) {
  pdl_wait();
  pdl_launch();
  const int nvec = C >> 3;
  const int64_t total = (int64_t)B * Ho * Wo * nvec;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int cg = (int)(i % nvec);
    const int64_t m = i / nvec;
    const int wo = (int)(m % Wo), ho = (int)((m / Wo) % Ho), b = (int)(m / ((int64_t)Wo * Ho));
    float best[8];
    int arg[8];
#pragma unroll
    for (int j = 0; j < 8; j++) { best[j] = -INFINITY; arg[j] = 0; }
    // all nine 16-byte loads are issued first (from clamped, always valid addresses), then compared in window order:
    // nine independent loads in flight instead of a load -> compare chain
    const __nv_bfloat16* img = x + (int64_t)b * H * W * C + cg * 8;
    uint4 raw[9];
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
        raw[r * 3 + s2] = load_raw(img + ((int64_t)hc * W + wc) * C);
      }
    }
#pragma unroll
    for (int t = 0; t < 9; t++) {
      if (!ok[t]) continue;
      const F8 v = unpack8(raw[t]);
#pragma unroll
      for (int j = 0; j < 8; j++)
        if (v.v[j] > best[j]) { best[j] = v.v[j]; arg[j] = t; }
    }
    F8 o;
#pragma unroll
    for (int j = 0; j < 8; j++) o.v[j] = best[j];
    store8(out + m * C + cg * 8, o);
    if (idx) {
      uint2 pk;
      pk.x = arg[0] | (arg[1] << 8) | (arg[2] << 16) | (arg[3] << 24);
      pk.y = arg[4] | (arg[5] << 8) | (arg[6] << 16) | (arg[7] << 24);
      *reinterpret_cast<uint2*>(idx + m * C + cg * 8) = pk;
    }
  }
}
// Each thread owns a 2x2 block of input pixels (8 channels): the only windows that can have selected them are
// (ho, wo) in {i, i+1} x {j, j+1}, loaded once each (row 2i belongs to window row i as r=1, row 2i+1 to window
// row i as r=2 and to window row i+1 as r=0; columns alike).
__global__ void __launch_bounds__(kT)
maxpool_bwd_kernel(const __nv_bfloat16* __restrict__ dout, const uint8_t* __restrict__ idx, int B,
                   int H, int W, int C, int Ho, int Wo, __nv_bfloat16* __restrict__ dx) {
  pdl_wait();
  pdl_launch();
  const int nvec = C >> 3;
  const int Hb = (H + 1) >> 1, Wb = (W + 1) >> 1;
  const int64_t total = (int64_t)B * Hb * Wb * nvec;
  for (int64_t it = (int64_t)blockIdx.x * kT + threadIdx.x; it < total; it += (int64_t)gridDim.x * kT) {
    const int cg = (int)(it % nvec);
    const int64_t m = it / nvec;
    const int j = (int)(m % Wb), i = (int)((m / Wb) % Hb), b = (int)(m / ((int64_t)Wb * Hb));
    float acc[2][2][8];
#pragma unroll
    for (int a = 0; a < 2; a++)
#pragma unroll
      for (int c = 0; c < 2; c++)
#pragma unroll
        for (int k = 0; k < 8; k++) acc[a][c][k] = 0.f;
#pragma unroll
    for (int dho = 0; dho < 2; dho++) {
      const int ho = i + dho;
      if (ho >= Ho) continue;
#pragma unroll
      for (int dwo = 0; dwo < 2; dwo++) {
        const int wo = j + dwo;
        if (wo >= Wo) continue;
        const int64_t om = ((int64_t)b * Ho + ho) * Wo + wo;
        const uint2 pk = *reinterpret_cast<const uint2*>(idx + om * C + cg * 8);
        const F8 g = load8(dout + om * C + cg * 8);
#pragma unroll
        for (int dy = dho; dy < 2; dy++) {                 // window row i+1 reaches only block row 1 (as r = 0)
          const int r = dho ? 0 : 1 + dy;
#pragma unroll
          for (int dxx = dwo; dxx < 2; dxx++) {
            const int sx = dwo ? 0 : 1 + dxx;
            const int code = r * 3 + sx;
#pragma unroll
            for (int k = 0; k < 8; k++) {
              const int a = ((k < 4 ? pk.x : pk.y) >> (8 * (k & 3))) & 0xff;
              if (a == code) acc[dy][dxx][k] += g.v[k];
            }
          }
        }
      }
    }
#pragma unroll
    for (int dy = 0; dy < 2; dy++) {
      const int hi = 2 * i + dy;
      if (hi >= H) continue;
#pragma unroll
      for (int dxx = 0; dxx < 2; dxx++) {
        const int wi = 2 * j + dxx;
        if (wi >= W) continue;
        F8 o;
#pragma unroll
        for (int k = 0; k < 8; k++) o.v[k] = acc[dy][dxx][k];
        store8(dx + (((int64_t)b * H + hi) * W + wi) * C + cg * 8, o);
      }
    }
  }
}

// ---------------------------------------------------------------------------
// reductions / broadcasts over the spatial axis: [B, HW, C] <-> [B, C]
__global__ void __launch_bounds__(kT)
reduce_hw_kernel(const __nv_bfloat16* __restrict__ x, int x_ld, int64_t HW, int C, float scale,
                 __nv_bfloat16* __restrict__ out, int nx, int ny) {
  pdl_wait();
  pdl_launch();
  __shared__ float s_red[kT * 8];
  const int b = blockIdx.y;
  const int tx = threadIdx.x % nx, ty = threadIdx.x / nx;
  const int cg = blockIdx.x * nx + tx;
  const int nvec = C >> 3;
  float a[8];
#pragma unroll
  for (int j = 0; j < 8; j++) a[j] = 0.f;
  if (cg < nvec && ty < ny) {
    const __nv_bfloat16* xp = x + (int64_t)b * HW * x_ld + cg * 8;
    int64_t r = ty;
    for (; r + 3 * ny < HW; r += 4 * ny) {        // four independent 16-byte loads in flight (was a load -> add chain)
      uint4 q[4];
#pragma unroll
      for (int u = 0; u < 4; u++) q[u] = load_raw(xp + (r + (int64_t)u * ny) * x_ld);
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const F8 v = unpack8(q[u]);
#pragma unroll
        for (int j = 0; j < 8; j++) a[j] += v.v[j];
      }
    }
    for (; r < HW; r += ny) {
      const F8 v = load8(xp + r * x_ld);
#pragma unroll
      for (int j = 0; j < 8; j++) a[j] += v.v[j];
    }
  }
#pragma unroll
  for (int j = 0; j < 8; j++) s_red[threadIdx.x * 8 + j] = a[j];
  __syncthreads();
  if (ty == 0 && cg < nvec) {
    F8 o;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      float t = 0.f;
      for (int y = 0; y < ny; y++) t += s_red[(y * nx + tx) * 8 + j];
      o.v[j] = t * scale;
    }
    store8(out + (int64_t)b * C + cg * 8, o);
  }
}
__global__ void __launch_bounds__(kT)
broadcast_hw_kernel(const __nv_bfloat16* __restrict__ x, int B, int64_t HW, int C,
                    __nv_bfloat16* __restrict__ out, int out_ld, float scale, int accumulate) {
  pdl_wait();
  pdl_launch();
  const int nvec = C >> 3;
  const int64_t total = (int64_t)B * HW * nvec;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int cg = (int)(i % nvec);
    const int64_t m = i / nvec;
    const int b = (int)(m / HW);
    F8 v = load8(x + (int64_t)b * C + cg * 8);
    __nv_bfloat16* op = out + m * out_ld + cg * 8;
    if (accumulate) {
      const F8 o = load8(op);
#pragma unroll
      for (int j = 0; j < 8; j++) v.v[j] = fmaf(v.v[j], scale, o.v[j]);
    } else if (scale != 1.f) {
#pragma unroll
      for (int j = 0; j < 8; j++) v.v[j] *= scale;
    }
    store8(op, v);
  }
}

// ---------------------------------------------------------------------------
// bilinear, align_corners=False (ATen upsample_bilinear2d index rule)
// One grid row (blockIdx.x, up to 2^31-1 of them) per output image row: the vertical source rows / weight are block constants and the
// remaining index math is 32-bit.
__global__ void __launch_bounds__(kT)
bilinear_fwd_kernel(const __nv_bfloat16* __restrict__ x, int x_ld, int B, int Hi, int Wi, int C,
                    int Ho, int Wo, __nv_bfloat16* __restrict__ out, int out_ld) {
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
  __nv_bfloat16* orow = out + ((int64_t)b * Ho + ho) * Wo * out_ld;
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
    F8 o;
#pragma unroll
    for (int j = 0; j < 8; j++) o.v[j] = w00 * v00.v[j] + w01 * v01.v[j] + w10 * v10.v[j] + w11 * v11.v[j];
    store8(orow + (int64_t)wo * out_ld + c8, o);
  }
}

// candidate output range that can touch input index i
__device__ __forceinline__ void bil_range(int i, float rscale, int out, int& lo, int& hi) {
  lo = (int)floorf(((float)i - 0.5f) * rscale - 0.5f) - 1;
  hi = (int)ceilf(((float)i + 1.5f) * rscale - 0.5f) + 1;
  lo = lo < 0 ? 0 : lo;
  hi = hi > out - 1 ? out - 1 : hi;
}

// adjoint, separable: a block owns one INPUT row yi of one image and a 64-channel chunk. Pass 1 folds the <= ~12
// output rows that touch yi into ONE row v[ox][c] in shared memory (coalesced 16-byte loads, each output element is
// read by the 2 input rows it feeds instead of the 4 pixels of the gather form); pass 2 folds v along x. The gather
// form spent its time recomputing source coordinates inside a ~100-iteration loop (109 us at cfg2).
constexpr int kBilChunk = 64;
constexpr int kBilRows = 64;                                 // capacity of the per-block row list (scale ratios up to ~14)
// rows oy in [lo, hi] with weight wy(oy -> yi) != 0 (or owned for the bias sum): built once per block by thread 0, so the
// row loops below are short, branch-free and can keep several loads in flight
__device__ __forceinline__ void bil_row_list(int yi, int lo, int hi, float sh, int Hi, int own_lo, int own_hi,
                                             int* s_oy, float* s_wy, int* s_n) {
  if (threadIdx.x == 0) {
    int n = 0;
    for (int oy = lo; oy <= hi && n < kBilRows; oy++) {
      int y0, y1; float ly;
      bil_src(oy, sh, Hi, y0, y1, ly);
      const float wy = (y0 == yi ? 1.f - ly : 0.f) + (y1 == yi ? ly : 0.f);
      const bool mine = oy >= own_lo && oy < own_hi;
      if (wy != 0.f || mine) { s_oy[n] = mine ? (oy | 0x40000000) : oy; s_wy[n] = wy; n++; }
    }
    *s_n = n;
  }
  __syncthreads();
}
__global__ void __launch_bounds__(kT)
bilinear_bwd_kernel(const __nv_bfloat16* __restrict__ dout, int dout_ld, int B, int Hi, int Wi,
                    int C, int Ho, int Wo, __nv_bfloat16* __restrict__ dx, int dx_ld) {
  pdl_wait();
  pdl_launch();
  extern __shared__ float s_v[];                              // [Wo][kBilChunk]
  const float sh = (float)Hi / (float)Ho, sw = (float)Wi / (float)Wo;
  const float rh = (float)Ho / (float)Hi, rw = (float)Wo / (float)Wi;
  const int yi = blockIdx.x % Hi, b = blockIdx.x / Hi;
  const int cb = blockIdx.y * kBilChunk;
  const int nvec = min(kBilChunk, C - cb) >> 3;
  int ylo, yhi;
  bil_range(yi, rh, Ho, ylo, yhi);
  __shared__ int s_oy[kBilRows];
  __shared__ float s_wy[kBilRows];
  __shared__ int s_n;
  bil_row_list(yi, ylo, yhi, sh, Hi, 0, 0, s_oy, s_wy, &s_n);
  const int nrows = s_n;
  const __nv_bfloat16* base = dout + (int64_t)b * Ho * Wo * dout_ld + cb;
  for (int i = threadIdx.x; i < Wo * nvec; i += kT) {
    const int ox = i / nvec, c8 = (i - ox * nvec) << 3;
    const __nv_bfloat16* col = base + (int64_t)ox * dout_ld + c8;
    const int64_t rs = (int64_t)Wo * dout_ld;
    F8 acc;
#pragma unroll
    for (int j = 0; j < 8; j++) acc.v[j] = 0.f;
    int r = 0;
    for (; r + 4 <= nrows; r += 4) {                          // four independent 16-byte loads in flight
      uint4 g[4];
#pragma unroll
      for (int u = 0; u < 4; u++) g[u] = load_raw(col + s_oy[r + u] * rs);
#pragma unroll
      for (int u = 0; u < 4; u++) {
        const F8 f = unpack8(g[u]);
        const float wy = s_wy[r + u];
#pragma unroll
        for (int j = 0; j < 8; j++) acc.v[j] = fmaf(wy, f.v[j], acc.v[j]);
      }
    }
    for (; r < nrows; r++) {
      const F8 f = load8(col + s_oy[r] * rs);
      const float wy = s_wy[r];
#pragma unroll
      for (int j = 0; j < 8; j++) acc.v[j] = fmaf(wy, f.v[j], acc.v[j]);
    }
    float4* d = reinterpret_cast<float4*>(s_v + ox * kBilChunk + c8);
    d[0] = make_float4(acc.v[0], acc.v[1], acc.v[2], acc.v[3]);
    d[1] = make_float4(acc.v[4], acc.v[5], acc.v[6], acc.v[7]);
  }
  __syncthreads();
  __nv_bfloat16* orow = dx + ((int64_t)b * Hi + yi) * Wi * dx_ld + cb;
  for (int i = threadIdx.x; i < Wi * nvec; i += kT) {
    const int xi = i / nvec, c8 = (i - xi * nvec) << 3;
    int xlo, xhi;
    bil_range(xi, rw, Wo, xlo, xhi);
    F8 acc;
#pragma unroll
    for (int j = 0; j < 8; j++) acc.v[j] = 0.f;
    for (int ox = xlo; ox <= xhi; ox++) {
      int x0, x1; float lx;
      bil_src(ox, sw, Wi, x0, x1, lx);
      const float wx = (x0 == xi ? 1.f - lx : 0.f) + (x1 == xi ? lx : 0.f);
      if (wx == 0.f) continue;
      const float4* v = reinterpret_cast<const float4*>(s_v + ox * kBilChunk + c8);
      const float4 a = v[0], c = v[1];
      acc.v[0] = fmaf(wx, a.x, acc.v[0]); acc.v[1] = fmaf(wx, a.y, acc.v[1]); acc.v[2] = fmaf(wx, a.z, acc.v[2]); acc.v[3] = fmaf(wx, a.w, acc.v[3]);
      acc.v[4] = fmaf(wx, c.x, acc.v[4]); acc.v[5] = fmaf(wx, c.y, acc.v[5]); acc.v[6] = fmaf(wx, c.z, acc.v[6]); acc.v[7] = fmaf(wx, c.w, acc.v[7]);
    }
    store8(orow + (int64_t)xi * dx_ld + c8, acc);
  }
}

// final logits upsample: NHWC fp32 [B,h,w,C] -> NCHW fp32 [B,C,H,W]; grid row = (image, output row)
__global__ void __launch_bounds__(kT)
logits_up_fwd_kernel(const float* __restrict__ x, int B, int Hi, int Wi, int C, int Ho, int Wo,
                     float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const float sh = (float)Hi / (float)Ho, sw = (float)Wi / (float)Wo;
  const int ho = blockIdx.x % Ho, b = blockIdx.x / Ho;
  int y0, y1;
  float ly;
  bil_src(ho, sh, Hi, y0, y1, ly);
  const float* r0 = x + ((int64_t)b * Hi + y0) * Wi * C;
  const float* r1 = x + ((int64_t)b * Hi + y1) * Wi * C;
  for (int wo = blockIdx.y * kT + threadIdx.x; wo < Wo; wo += gridDim.y * kT) {
    int x0, x1;
    float lx;
    bil_src(wo, sw, Wi, x0, x1, lx);
    const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
    const float* p00 = r0 + (int64_t)x0 * C;
    const float* p01 = r0 + (int64_t)x1 * C;
    const float* p10 = r1 + (int64_t)x0 * C;
    const float* p11 = r1 + (int64_t)x1 * C;
    for (int c = 0; c < C; c++) {
      const float v = bil_mix(w00, __ldg(p00 + c), w01, __ldg(p01 + c), w10, __ldg(p10 + c), w11, __ldg(p11 + c));
      out[(((int64_t)b * C + c) * Ho + ho) * Wo + wo] = v;
    }
  }
}
// adjoint: NCHW fp32 dlogits -> NHWC bf16 [B,h,w,dx_ld] (channels >= C zero-filled); a block owns one INPUT row yi of one
// image: pass 1 folds the output rows that touch yi into v[c][ox] in shared memory (coalesced reads along W), pass 2
// folds v along x. Optionally the same pass accumulates the classifier bias gradient sum_{b,y,x} dlogits[b,c,y,x]
// (each output row counted by the ONE input row floor(oy*Hi/Ho) that owns it), replacing a second sweep over dlogits.
__global__ void __launch_bounds__(kT)
logits_up_bwd_kernel(const float* __restrict__ dout, int B, int Hi, int Wi, int C, int Ho, int Wo,
                     __nv_bfloat16* __restrict__ dx, int dx_ld, float* __restrict__ bias_grad) {
  pdl_wait();
  pdl_launch();
  extern __shared__ float s_v[];                              // [C][Wo], then [C] bias partials
  float* s_bias = s_v + C * Wo;
  const float sh = (float)Hi / (float)Ho, sw = (float)Wi / (float)Wo;
  const float rh = (float)Ho / (float)Hi, rw = (float)Wo / (float)Wi;
  const int yi = blockIdx.x % Hi, b = blockIdx.x / Hi;
  int ylo, yhi;
  bil_range(yi, rh, Ho, ylo, yhi);
  if (bias_grad) {
    for (int c = threadIdx.x; c < C; c += kT) s_bias[c] = 0.f;
    __syncthreads();
  }
  // rows [own_lo, own_hi) of the output belong to this input row for the bias sum (a partition of [0, Ho))
  const int own_lo = (int)(((int64_t)yi * Ho + Hi - 1) / Hi), own_hi = (int)(((int64_t)(yi + 1) * Ho + Hi - 1) / Hi);
  __shared__ int s_oy[kBilRows];
  __shared__ float s_wy[kBilRows];
  __shared__ int s_n;
  bil_row_list(yi, min(ylo, own_lo), max(yhi, own_hi - 1), sh, Hi, bias_grad ? own_lo : 0, bias_grad ? own_hi : 0, s_oy, s_wy, &s_n);
  const int nrows = s_n;
  for (int i0 = 0; i0 < C * Wo; i0 += kT) {                 // uniform trip count: the warp shuffles below need all lanes
    const int i = i0 + threadIdx.x;
    const bool in = i < C * Wo;
    const int c = in ? i / Wo : -1, ox = in ? i - c * Wo : 0;
    float acc = 0.f, own = 0.f;
    if (in) {
      const float* col = dout + ((int64_t)b * C + c) * Ho * Wo + ox;
      int r = 0;
      for (; r + 4 <= nrows; r += 4) {
        float g[4];
#pragma unroll
        for (int u = 0; u < 4; u++) g[u] = __ldg(col + (int64_t)(s_oy[r + u] & 0x3fffffff) * Wo);
#pragma unroll
        for (int u = 0; u < 4; u++) {
          acc = fmaf(s_wy[r + u], g[u], acc);
          if (s_oy[r + u] & 0x40000000) own += g[u];
        }
      }
      for (; r < nrows; r++) {
        const float g = __ldg(col + (int64_t)(s_oy[r] & 0x3fffffff) * Wo);
        acc = fmaf(s_wy[r], g, acc);
        if (s_oy[r] & 0x40000000) own += g;
      }
      s_v[i] = acc;
    }
    if (bias_grad) {
      // segmented warp sum: lanes hold consecutive i, so c is non-decreasing across the warp; the first lane of every
      // run of equal c ends up with the run's total and adds it to the block's per-class partial
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const float other = __shfl_down_sync(0xffffffffu, own, o);
        const int oc = __shfl_down_sync(0xffffffffu, c, o);
        if ((int)(threadIdx.x & 31) + o < 32 && oc == c) own += other;
      }
      const int pc = __shfl_up_sync(0xffffffffu, c, 1);
      if (in && ((threadIdx.x & 31) == 0 || pc != c)) atomicAdd(s_bias + c, own);
    }
  }
  __syncthreads();
  if (bias_grad)
    for (int c = threadIdx.x; c < C; c += kT) atomicAdd(bias_grad + c, s_bias[c]);
  for (int i = threadIdx.x; i < Wi * C; i += kT) {
    const int xi = i / C, c = i - xi * C;
    int xlo, xhi;
    bil_range(xi, rw, Wo, xlo, xhi);
    const float* v = s_v + c * Wo;
    float acc = 0.f;
    for (int ox = xlo; ox <= xhi; ox++) {
      int x0, x1; float lx;
      bil_src(ox, sw, Wi, x0, x1, lx);
      const float wx = (x0 == xi ? 1.f - lx : 0.f) + (x1 == xi ? lx : 0.f);
      if (wx != 0.f) acc = fmaf(wx, v[ox], acc);
    }
    const int64_t m = ((int64_t)b * Hi + yi) * Wi + xi;
    dx[m * dx_ld + c] = __float2bfloat16_rn(acc);
    if (c == C - 1)
      for (int cc = C; cc < dx_ld; cc++) dx[m * dx_ld + cc] = __float2bfloat16_rn(0.f);
  }
}

// ---------------------------------------------------------------------------
// stride-2 helpers
// phase split: out[(p*2+q)][b][i][j][c] = x[b][2i+p][2j+q][c]  (zero beyond the image)
__global__ void __launch_bounds__(kT)
phase_split_kernel(const __nv_bfloat16* __restrict__ x, int x_ld, int B, int H, int W, int C,
                   int Hp, int Wp, __nv_bfloat16* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int nvec = C >> 3;
  const int64_t total = (int64_t)4 * B * Hp * Wp * nvec;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int cg = (int)(i % nvec);
    int64_t m = i / nvec;
    const int j = (int)(m % Wp); m /= Wp;
    const int ii = (int)(m % Hp); m /= Hp;
    const int b = (int)(m % B);
    const int ph = (int)(m / B);
    const int h = 2 * ii + (ph >> 1), w = 2 * j + (ph & 1);
    F8 v;
    if (h < H && w < W) v = load8(x + (((int64_t)b * H + h) * W + w) * x_ld + cg * 8);
    else {
#pragma unroll
      for (int k = 0; k < 8; k++) v.v[k] = 0.f;
    }
    store8(out + (i / nvec) * C + cg * 8, v);
  }
}
// subsample: out[b][i][j] = x[b][2i][2j]
__global__ void __launch_bounds__(kT)
subsample2_kernel(const __nv_bfloat16* __restrict__ x, int x_ld, int B, int H, int W, int C,
                  int Ho, int Wo, __nv_bfloat16* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int nvec = C >> 3;
  const int64_t total = (int64_t)B * Ho * Wo * nvec;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int cg = (int)(i % nvec);
    const int64_t m = i / nvec;
    const int j = (int)(m % Wo), ii = (int)((m / Wo) % Ho), b = (int)(m / ((int64_t)Wo * Ho));
    const F8 v = load8(x + (((int64_t)b * H + 2 * ii) * W + 2 * j) * x_ld + cg * 8);
    store8(out + m * C + cg * 8, v);
  }
}
// zero stuff: out[b][h][w] = (h,w even and in range) ? x[b][h/2][w/2] : 0 ; mode 1: out += at even sites
__global__ void __launch_bounds__(kT)
stuff2_kernel(const __nv_bfloat16* __restrict__ x, int B, int Ho, int Wo, int C, int H, int W,
              __nv_bfloat16* __restrict__ out, int accumulate) {
  pdl_wait();
  pdl_launch();
  const int nvec = C >> 3;
  if (accumulate) {
    const int64_t total = (int64_t)B * Ho * Wo * nvec;
    for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
      const int cg = (int)(i % nvec);
      const int64_t m = i / nvec;
      const int j = (int)(m % Wo), ii = (int)((m / Wo) % Ho), b = (int)(m / ((int64_t)Wo * Ho));
      if (2 * ii >= H || 2 * j >= W) continue;
      __nv_bfloat16* op = out + (((int64_t)b * H + 2 * ii) * W + 2 * j) * C + cg * 8;
      F8 o = load8(op);
      const F8 v = load8(x + m * C + cg * 8);
#pragma unroll
      for (int k = 0; k < 8; k++) o.v[k] += v.v[k];
      store8(op, o);
    }
  } else {
    const int64_t total = (int64_t)B * H * W * nvec;
    for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
      const int cg = (int)(i % nvec);
      const int64_t m = i / nvec;
      const int w = (int)(m % W), h = (int)((m / W) % H), b = (int)(m / ((int64_t)W * H));
      F8 v;
      if (!(h & 1) && !(w & 1) && (h >> 1) < Ho && (w >> 1) < Wo)
        v = load8(x + (((int64_t)b * Ho + (h >> 1)) * Wo + (w >> 1)) * C + cg * 8);
      else {
#pragma unroll
        for (int k = 0; k < 8; k++) v.v[k] = 0.f;
      }
      store8(out + m * C + cg * 8, v);
    }
  }
}

__global__ void __launch_bounds__(kT)
add_bf16_kernel(const __nv_bfloat16* __restrict__ a, const __nv_bfloat16* __restrict__ b, int64_t nvec8,
                __nv_bfloat16* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < nvec8; i += (int64_t)gridDim.x * kT) {
    F8 x = load8(a + i * 8);
    const F8 y = load8(b + i * 8);
#pragma unroll
    for (int k = 0; k < 8; k++) x.v[k] += y.v[k];
    store8(out + i * 8, x);
  }
}

// layout converters (API boundary / tests)
__global__ void __launch_bounds__(kT)
nhwc_to_nchw_f32_kernel(const __nv_bfloat16* __restrict__ x, int x_ld, int B, int64_t HW, int C,
                        float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int64_t total = (int64_t)B * C * HW;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int64_t p = i % HW;
    const int c = (int)((i / HW) % C);
    const int64_t b = i / (HW * C);
    out[i] = __bfloat162float(x[(b * HW + p) * x_ld + c]);
  }
}
__global__ void __launch_bounds__(kT)
nchw_f32_to_nhwc_kernel(const float* __restrict__ x, int B, int64_t HW, int C,
                        __nv_bfloat16* __restrict__ out, int out_ld) {
  pdl_wait();
  pdl_launch();
  const int64_t total = (int64_t)B * HW * C;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int c = (int)(i % C);
    const int64_t p = (i / C) % HW;
    const int64_t b = i / ((int64_t)C * HW);
    out[(b * HW + p) * out_ld + c] = __float2bfloat16_rn(x[(b * C + c) * HW + p]);
  }
}

// fused SGD(momentum, nesterov, weight decay) over a flat fp32 buffer (torch.optim.SGD rule)
__global__ void __launch_bounds__(kT)
sgd_step_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ mom, int64_t n,
                float lr, float momentum, float wd, int nesterov, int first, const float* __restrict__ d_lr) {
  pdl_wait();
  pdl_launch();
  if (d_lr) lr = *d_lr;                  // learning rate from device memory (CUDA-graph replays follow the scheduler)
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < n; i += (int64_t)gridDim.x * kT) {
    float grad = g[i];
    const float w = p[i];
    if (wd != 0.f) grad = fmaf(wd, w, grad);
    if (momentum != 0.f) {
      const float buf = first ? grad : fmaf(momentum, mom[i], grad);
      mom[i] = buf;
      grad = nesterov ? fmaf(momentum, buf, grad) : buf;
    }
    p[i] = fmaf(-lr, grad, w);
  }
}


// fused Adam / AdamW over a flat fp32 buffer (torch.optim.Adam / AdamW single-tensor rule, train.py:432-441):
//   Adam : g += wd * p            AdamW: p *= 1 - lr * wd
//   m = m + (g - m) * (1 - b1);   v = b2 * v + (1 - b2) * g * g
//   p -= (lr / (1 - b1^t)) * m / (sqrt(v) / sqrt(1 - b2^t) + eps)
__global__ void __launch_bounds__(kT)
adam_step_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                 int64_t n, float lr, float b1, float b2, float eps, float wd, int adamw, float step_size,
                 float inv_sqrt_bc2, const float* __restrict__ d_lr, const long long* __restrict__ d_step) {
  pdl_wait();
  pdl_launch();
  if (d_lr || d_step) {                  // device-resident schedule state (CUDA-graph replays): redo the host's scalar math
    const double lr_host = (double)lr;
    const double lr_d = d_lr ? (double)*d_lr : lr_host;
    if (d_step) {
      const double t = (double)*d_step;
      step_size = (float)(lr_d / (1.0 - pow((double)b1, t)));
      inv_sqrt_bc2 = (float)(1.0 / sqrt(1.0 - pow((double)b2, t)));
    } else {
      step_size = (float)((double)step_size * (lr_d / lr_host));
    }
    lr = (float)lr_d;
  }
  auto one = [&](float& w, float grad, float& mm, float& vv) {
    if (adamw) w = w * (1.f - lr * wd);
    else if (wd != 0.f) grad = fmaf(wd, w, grad);
    mm = fmaf(grad - mm, 1.f - b1, mm);
    vv = fmaf(vv, b2, (1.f - b2) * grad * grad);
    const float denom = sqrtf(vv) * inv_sqrt_bc2 + eps;
    w = fmaf(-step_size, mm / denom, w);
  };
  const int64_t n4 = n >> 2;
  const int64_t stride = (int64_t)gridDim.x * kT;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < n4; i += stride) {
    float4 w4 = reinterpret_cast<float4*>(p)[i];
    const float4 g4 = reinterpret_cast<const float4*>(g)[i];
    float4 m4 = reinterpret_cast<float4*>(m)[i], v4 = reinterpret_cast<float4*>(v)[i];
    one(w4.x, g4.x, m4.x, v4.x); one(w4.y, g4.y, m4.y, v4.y); one(w4.z, g4.z, m4.z, v4.z); one(w4.w, g4.w, m4.w, v4.w);
    reinterpret_cast<float4*>(p)[i] = w4;
    reinterpret_cast<float4*>(m)[i] = m4;
    reinterpret_cast<float4*>(v)[i] = v4;
  }
  for (int64_t i = (n4 << 2) + (int64_t)blockIdx.x * kT + threadIdx.x; i < n; i += stride) one(p[i], g[i], m[i], v[i]);
}

// ---------------------------------------------------------------------------
// device input pipeline (SURVEY 8f rank 2): ExtRandomCrop (window origin per image) + ExtRandomHorizontalFlip +
// ExtToTensor + ExtNormalize (utils/ext_transforms.py:94-111, :273-324, :327-393) on uint8 HWC tiles, one pass:
//   out[b,c,y,x] = ((float(src[b, y0+y, x0 + (flip ? W-1-x : x), c]) / 255) - mean[c]) / std[c]
// (IEEE divisions: bit-identical to F.to_tensor + F.normalize). A thread makes 4 consecutive output pixels.
__global__ void __launch_bounds__(kT)
u8_to_f32_norm_kernel(const uint8_t* __restrict__ src, int Hs, int Ws, int C, const int* __restrict__ org_xy,
                      const uint8_t* __restrict__ flip, float3 mean, float3 stdv, float mean3, float std3,
                      int H, int W, float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int y = blockIdx.x % H, b = blockIdx.x / H;
  const int x0 = org_xy ? org_xy[2 * b] : 0, y0 = org_xy ? org_xy[2 * b + 1] : 0;
  const bool fl = flip ? flip[b] != 0 : false;
  const uint8_t* row = src + (((int64_t)b * Hs + (y0 + y)) * Ws + x0) * C;
  const float mu[4] = {mean.x, mean.y, mean.z, mean3}, sd[4] = {stdv.x, stdv.y, stdv.z, std3};
  const int64_t plane = (int64_t)H * W;
  float* obase = out + (int64_t)b * C * plane + (int64_t)y * W;
  const int nquad = (W + 3) >> 2;
  for (int qd = blockIdx.y * kT + threadIdx.x; qd < nquad; qd += gridDim.y * kT) {
    const int xo = qd << 2;
    const int nval = min(4, W - xo);
    float v[4][4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
      if (k < nval) {
        const int xs = fl ? (W - 1 - (xo + k)) : (xo + k);
#pragma unroll
        for (int c = 0; c < 4; c++)
          if (c < C) v[c][k] = __fdiv_rn(__fsub_rn(__fdiv_rn((float)row[(int64_t)xs * C + c], 255.f), mu[c]), sd[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < 4; c++) {
      if (c >= C) break;
      float* o = obase + (int64_t)c * plane + xo;
      if (nval == 4 && ((reinterpret_cast<uintptr_t>(o) & 15) == 0)) {
        *reinterpret_cast<float4*>(o) = make_float4(v[c][0], v[c][1], v[c][2], v[c][3]);
      } else {
        for (int k = 0; k < nval; k++) o[k] = v[c][k];
      }
    }
  }
}

// the label tile of the same crop / flip: uint8 [B,Hs,Ws] -> uint8 [B,H,W]
__global__ void __launch_bounds__(kT)
crop_flip_u8_kernel(const uint8_t* __restrict__ src, int Hs, int Ws, const int* __restrict__ org_xy,
                    const uint8_t* __restrict__ flip, int H, int W, uint8_t* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  const int y = blockIdx.x % H, b = blockIdx.x / H;
  const int x0 = org_xy ? org_xy[2 * b] : 0, y0 = org_xy ? org_xy[2 * b + 1] : 0;
  const bool fl = flip ? flip[b] != 0 : false;
  const uint8_t* row = src + ((int64_t)b * Hs + (y0 + y)) * Ws + x0;
  uint8_t* orow = out + ((int64_t)b * H + y) * W;
  for (int x = blockIdx.y * kT + threadIdx.x; x < W; x += gridDim.y * kT) orow[x] = row[fl ? (W - 1 - x) : x];
}

// per-channel sum of an NCHW fp32 tensor (classifier bias gradient): out[c] += sum_{b,p} d[b,c,p]
__global__ void __launch_bounds__(kT)
bias_grad_nchw_kernel(const float* __restrict__ d, int B, int C, int64_t HW, float* __restrict__ out) {
  pdl_wait();
  pdl_launch();
  __shared__ float s_red[kT / 32];
  const int c = blockIdx.y;
  float acc = 0.f;
  const int64_t total = (int64_t)B * HW;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int64_t b = i / HW, p = i - b * HW;
    acc += __ldg(d + (b * C + c) * HW + p);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int w = 0; w < kT / 32; w++) t += s_red[w];
    atomicAdd(out + c, t);
  }
}

// x *= *scalar, skipped entirely when the device scalar is exactly 1 (the loss.backward() case)
template <typename T>
__global__ void __launch_bounds__(kT)
scale_by_device_scalar_kernel(T* __restrict__ x, int64_t n, const float* __restrict__ scalar) {
  pdl_wait();
  pdl_launch();
  const float s = *scalar;
  if (s == 1.0f) return;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < n; i += (int64_t)gridDim.x * kT)
    x[i] = (T)((float)x[i] * s);
}

}  // namespace iswm

// ---------------------------------------------------------------------------
using namespace iswm;
#define ST(s) static_cast<cudaStream_t>(s)
#define BF(p) static_cast<const __nv_bfloat16*>(p)
#define BFW(p) static_cast<__nv_bfloat16*>(p)
#define REQ_C8(C, what) ISWM_REQUIRE(((C) % 8) == 0 && (C) > 0, what ": channel count %d must be a positive multiple of 8", (int)(C))
#define REQ_LD8(ld, what) ISWM_REQUIRE(((ld) % 8) == 0, what ": row pitch %d must be a multiple of 8", (int)(ld))

extern "C" int iswm_pack_weight_fwd(const float* d_w, int Cout, int Cin, int RS, int cin_pad,
                                    int row_ld, void* d_out, void* stream) {
  ISWM_REQUIRE(d_w && d_out && cin_pad >= Cin && row_ld >= RS * cin_pad, "pack_weight_fwd: bad args");
  launch_k(pack_weight_fwd_kernel, dim3(grid_for((int64_t)Cout * row_ld)), dim3(kT), 0, ST(stream), d_w, Cout, Cin, RS, cin_pad, row_ld, BFW(d_out));
  return check_launch("pack_weight_fwd");
}
extern "C" int iswm_pack_weight_dgrad(const float* d_w, int Cout, int Cin, int RS, int cout_pad,
                                      void* d_out, void* stream) {
  ISWM_REQUIRE(d_w && d_out && cout_pad >= Cout, "pack_weight_dgrad: bad args");
  launch_k(pack_weight_dgrad_kernel, dim3(grid_for((int64_t)Cin * RS * cout_pad)), dim3(kT), 0, ST(stream), d_w, Cout, Cin, RS, cout_pad, BFW(d_out));
  return check_launch("pack_weight_dgrad");
}
extern "C" int iswm_unpack_wgrad(const float* d_dw, int Cout, int Cin, int RS, int cin_stride,
                                 int row_ld, float beta, float* d_grad_oihw, void* stream) {
  ISWM_REQUIRE(d_dw && d_grad_oihw, "unpack_wgrad: null");
  if (RS <= 9 && RS > 1 && cin_stride == Cin && row_ld == RS * Cin && Cout <= 65535 * 32) {
    launch_k(unpack_wgrad_tiled_kernel, dim3((unsigned)Cout, (unsigned)((Cin + kUnpackChunk - 1) / kUnpackChunk)), dim3(kT), 0, ST(stream), d_dw, Cin, RS, beta, d_grad_oihw);
    return check_launch("unpack_wgrad");
  }
  launch_k(unpack_wgrad_kernel, dim3(grid_for((int64_t)Cout * Cin * RS)), dim3(kT), 0, ST(stream), d_dw, Cout, Cin, RS, cin_stride, row_ld, beta, d_grad_oihw);
  return check_launch("unpack_wgrad");
}

static int bn_train_apply_impl(bool global, const void* d_x, int x_ld, const double* d_stats, int stats_replicas, int64_t M, int C,
                               const float* d_gamma, const float* d_beta, float eps, float momentum,
                               float* d_running_mean, float* d_running_var, int64_t* d_nbt,
                               float* d_save_mean, float* d_save_invstd, const void* d_res, int res_ld,
                               int relu, float drop_p, uint64_t drop_seed, const int64_t* d_drop_step, void* d_out, int out_ld,
                               uint8_t* d_relu_bits, void* stream) {
  if (debug_skip(ISWM_SKIP_BN)) return 0;
  REQ_C8(C, "bn_train_apply"); REQ_LD8(x_ld, "bn_train_apply"); REQ_LD8(out_ld, "bn_train_apply");
  ISWM_REQUIRE(d_x && d_stats && d_gamma && d_beta && d_out && M > 0, "bn_train_apply: null/empty");
  ISWM_REQUIRE(!d_res || (res_ld % 8) == 0, "bn_train_apply: res_ld");
  ISWM_REQUIRE(C <= 2048, "bn_train_apply: C=%d > 2048 not supported", C);
  ISWM_REQUIRE(!global || stats_replicas <= 1, "bn_train_apply_global: the global sums are one copy (stats_replicas=%d)", stats_replicas);
  int nx, ny, rpb, blocks;
  // blocks per SM the row range is cut for: 3 = exactly the resident blocks (80 registers x 256 threads), ONE wave.
  // Measured on B200 against 6 (two waves): 33.6 MB tensor 17.1 -> 12.3 us, 67 MB 30.0 -> 24.9 us, cfg2 1074 -> 1088
  // img/s: a second wave is mostly a tail (each thread's life is one or two batches of loads).
  bn_row_grid(C, M, 4, nx, ny, rpb, blocks, 3);
  const bool has_res = d_res != nullptr, has_drop = drop_p > 0.f;
#define ISWM_BN_APPLY_G(R, L, D, G)                                                                                \
  launch_k(bn_train_apply_kernel<R, L, D, G>, dim3(blocks), dim3(kT), 0, ST(stream), BF(d_x), x_ld, d_stats, std::max(1, stats_replicas), M, C, \
           d_gamma, d_beta, eps, momentum, d_running_mean, d_running_var, reinterpret_cast<long long*>(d_nbt),      \
           d_save_mean, d_save_invstd, BF(d_res), res_ld, drop_p, DropSeed{drop_seed, reinterpret_cast<const long long*>(d_drop_step)}, BFW(d_out), out_ld, nx, ny, rpb, relu ? d_relu_bits : nullptr)
#define ISWM_BN_APPLY(R, L, D) do { if (global) ISWM_BN_APPLY_G(R, L, D, true); else ISWM_BN_APPLY_G(R, L, D, false); } while (0)
  if (has_drop) {
    if (has_res) { if (relu) ISWM_BN_APPLY(true, true, true); else ISWM_BN_APPLY(true, false, true); }
    else         { if (relu) ISWM_BN_APPLY(false, true, true); else ISWM_BN_APPLY(false, false, true); }
  } else {
    if (has_res) { if (relu) ISWM_BN_APPLY(true, true, false); else ISWM_BN_APPLY(true, false, false); }
    else         { if (relu) ISWM_BN_APPLY(false, true, false); else ISWM_BN_APPLY(false, false, false); }
  }
#undef ISWM_BN_APPLY
#undef ISWM_BN_APPLY_G
  return check_launch("bn_train_apply");
}
extern "C" int iswm_bn_train_apply(const void* d_x, int x_ld, const double* d_stats, int stats_replicas, int64_t M, int C,
                                   const float* d_gamma, const float* d_beta, float eps, float momentum,
                                   float* d_running_mean, float* d_running_var, int64_t* d_nbt,
                                   float* d_save_mean, float* d_save_invstd, const void* d_res, int res_ld,
                                   int relu, float drop_p, uint64_t drop_seed, const int64_t* d_drop_step, void* d_out, int out_ld,
                                   uint8_t* d_relu_bits, void* stream) {
  return bn_train_apply_impl(false, d_x, x_ld, d_stats, stats_replicas, M, C, d_gamma, d_beta, eps, momentum, d_running_mean, d_running_var,
                             d_nbt, d_save_mean, d_save_invstd, d_res, res_ld, relu, drop_p, drop_seed, d_drop_step, d_out, out_ld, d_relu_bits, stream);
}
extern "C" int iswm_bn_train_apply_global(const void* d_x, int x_ld, const double* d_gstats, int64_t M, int C,
                                          const float* d_gamma, const float* d_beta, float eps, float momentum,
                                          float* d_running_mean, float* d_running_var, int64_t* d_nbt,
                                          float* d_save_mean, float* d_save_invstd, const void* d_res, int res_ld,
                                          int relu, float drop_p, uint64_t drop_seed, const int64_t* d_drop_step, void* d_out, int out_ld,
                                          uint8_t* d_relu_bits, void* stream) {
  return bn_train_apply_impl(true, d_x, x_ld, d_gstats, 1, M, C, d_gamma, d_beta, eps, momentum, d_running_mean, d_running_var,
                             d_nbt, d_save_mean, d_save_invstd, d_res, res_ld, relu, drop_p, drop_seed, d_drop_step, d_out, out_ld, d_relu_bits, stream);
}
extern "C" int iswm_bn_fold(const float* d_gamma, const float* d_beta, const float* d_mean,
                            const float* d_var, float eps, int C, float* d_scale, float* d_shift,
                            void* stream) {
  ISWM_REQUIRE(d_gamma && d_beta && d_mean && d_var && d_scale && d_shift && C > 0, "bn_fold: null");
  launch_k(bn_fold_kernel, dim3((C + kT - 1) / kT), dim3(kT), 0, ST(stream), d_gamma, d_beta, d_mean, d_var, eps, C, d_scale, d_shift);
  return check_launch("bn_fold");
}

extern "C" int iswm_bn_bwd_reduce(const void* d_dout, int dout_ld, const void* d_x, int x_ld,
                                  const void* d_out_act, int act_ld, int64_t M, int C,
                                  const float* d_save_mean, const float* d_save_invstd,
                                  const float* d_gamma, const float* d_beta, int relu,
                                  float drop_p, uint64_t drop_seed, const int64_t* d_drop_step, double* d_sums, void* stream) {
  if (debug_skip(ISWM_SKIP_BN)) return 0;
  REQ_C8(C, "bn_bwd_reduce"); REQ_LD8(dout_ld, "bn_bwd_reduce"); REQ_LD8(x_ld, "bn_bwd_reduce");
  ISWM_REQUIRE(d_dout && d_x && d_save_mean && d_save_invstd && d_sums && M > 0, "bn_bwd_reduce: null/empty");
  ISWM_REQUIRE(relu >= 0 && relu <= 2, "bn_bwd_reduce: relu mode %d", relu);
  ISWM_REQUIRE(relu != 1 || (d_out_act && (act_ld % 8) == 0) || (!d_out_act && d_gamma && d_beta),
               "bn_bwd_reduce: relu needs the activation (or gamma and beta to recompute the mask)");
  ISWM_REQUIRE(relu != 2 || d_out_act, "bn_bwd_reduce: relu mode 2 needs the packed sign bits in d_out_act");
  ISWM_REQUIRE(C <= 2048, "bn_bwd_reduce: C=%d > 2048 not supported", C);
  int nx, ny, rows_per_block, blocks, groups = 1;
  if (C > 256) {
    // channel groups of 256 (32 threads x 8 channels, 512 contiguous bytes per row) x row blocks, one resident wave in all
    nx = 32; ny = kT / nx;
    groups = (C / 8 + nx - 1) / nx;
    int64_t want = (M + (int64_t)ny * 8 - 1) / ((int64_t)ny * 8);
    want = std::max<int64_t>(1, std::min<int64_t>(want, std::max(1, num_sms() * 3 / groups)));
    rows_per_block = (int)((M + want - 1) / want);
    blocks = (int)((M + rows_per_block - 1) / rows_per_block);
  } else {
    bn_row_grid(C, M, 8, nx, ny, rows_per_block, blocks, 3);   // one wave: every block ends with fp64 atomics on the same 2C addresses
  }
  const int mask = !relu ? 0 : (relu == 2 ? 3 : (d_out_act ? 1 : 2));
  const bool has_drop = drop_p > 0.f;
#define ISWM_BN_RED(MK, D)                                                                                          \
  launch_k(bn_bwd_reduce_kernel<MK, D>, dim3(blocks, groups), dim3(kT), 0, ST(stream), BF(d_dout), dout_ld, BF(d_x), x_ld,   \
           BF(d_out_act), act_ld, M, C, d_save_mean, d_save_invstd, d_gamma, d_beta, drop_p, DropSeed{drop_seed, reinterpret_cast<const long long*>(d_drop_step)}, d_sums, nx, \
           ny, rows_per_block)
  if (has_drop) { if (mask == 0) ISWM_BN_RED(0, true); else if (mask == 1) ISWM_BN_RED(1, true); else if (mask == 2) ISWM_BN_RED(2, true); else ISWM_BN_RED(3, true); }
  else          { if (mask == 0) ISWM_BN_RED(0, false); else if (mask == 1) ISWM_BN_RED(1, false); else if (mask == 2) ISWM_BN_RED(2, false); else ISWM_BN_RED(3, false); }
#undef ISWM_BN_RED
  return check_launch("bn_bwd_reduce");
}
static int bn_bwd_apply_impl(const double* d_lsums, const void* d_dout, int dout_ld, const void* d_x, int x_ld,
                             const void* d_out_act, int act_ld, int64_t M, int C,
                             const float* d_gamma, const float* d_beta, const float* d_save_mean,
                             const float* d_save_invstd, const double* d_sums, int relu, float drop_p, uint64_t drop_seed, const int64_t* d_drop_step,
                             void* d_dx, int dx_ld, void* d_dz, int dz_ld, float* d_dgamma,
                             float* d_dbeta, void* stream) {
  if (debug_skip(ISWM_SKIP_BN)) return 0;
  REQ_C8(C, "bn_bwd_apply"); REQ_LD8(dout_ld, "bn_bwd_apply"); REQ_LD8(x_ld, "bn_bwd_apply"); REQ_LD8(dx_ld, "bn_bwd_apply");
  ISWM_REQUIRE(d_dout && d_x && d_gamma && d_save_mean && d_save_invstd && d_sums && d_dx && M > 0, "bn_bwd_apply: null/empty");
  ISWM_REQUIRE(relu >= 0 && relu <= 2, "bn_bwd_apply: relu mode %d", relu);
  ISWM_REQUIRE(relu != 1 || (d_out_act && (act_ld % 8) == 0) || (!d_out_act && d_beta),
               "bn_bwd_apply: relu needs the activation (or beta to recompute the mask)");
  ISWM_REQUIRE(relu != 2 || d_out_act, "bn_bwd_apply: relu mode 2 needs the packed sign bits in d_out_act");
  ISWM_REQUIRE(!d_dz || (dz_ld % 8) == 0, "bn_bwd_apply: dz_ld");
  ISWM_REQUIRE(C <= 2048, "bn_bwd_apply: C=%d > 2048 not supported", C);
  int nx, ny, rpb, blocks;
  bn_row_grid(C, M, 4, nx, ny, rpb, blocks, 3);   // one wave, see iswm_bn_train_apply
  const int mask = !relu ? 0 : (relu == 2 ? 3 : (d_out_act ? 1 : 2));
  const bool has_drop = drop_p > 0.f, has_dz = d_dz != nullptr;
#define ISWM_BN_BAP_G(MK, D, Z, G)                                                                                     \
  launch_k(bn_bwd_apply_kernel<MK, D, Z, G>, dim3(blocks), dim3(kT), 0, ST(stream), BF(d_dout), dout_ld, BF(d_x), x_ld, \
           BF(d_out_act), act_ld, M, C, d_gamma, d_beta, d_save_mean, d_save_invstd, d_sums, drop_p, DropSeed{drop_seed, reinterpret_cast<const long long*>(d_drop_step)},        \
           BFW(d_dx), dx_ld, BFW(d_dz), dz_ld, d_dgamma, d_dbeta, nx, ny, rpb, d_lsums)
#define ISWM_BN_BAP(MK, D, Z) do { if (d_lsums) ISWM_BN_BAP_G(MK, D, Z, true); else ISWM_BN_BAP_G(MK, D, Z, false); } while (0)
#define ISWM_BN_BAP_M(D, Z) \
  do { if (mask == 0) ISWM_BN_BAP(0, D, Z); else if (mask == 1) ISWM_BN_BAP(1, D, Z); else if (mask == 2) ISWM_BN_BAP(2, D, Z); else ISWM_BN_BAP(3, D, Z); } while (0)
  if (has_drop) { if (has_dz) ISWM_BN_BAP_M(true, true); else ISWM_BN_BAP_M(true, false); }
  else          { if (has_dz) ISWM_BN_BAP_M(false, true); else ISWM_BN_BAP_M(false, false); }
#undef ISWM_BN_BAP_M
#undef ISWM_BN_BAP
#undef ISWM_BN_BAP_G
  return check_launch("bn_bwd_apply");
}
extern "C" int iswm_bn_bwd_apply(const void* d_dout, int dout_ld, const void* d_x, int x_ld,
                                 const void* d_out_act, int act_ld, int64_t M, int C,
                                 const float* d_gamma, const float* d_beta, const float* d_save_mean,
                                 const float* d_save_invstd, const double* d_sums, int relu, float drop_p, uint64_t drop_seed, const int64_t* d_drop_step,
                                 void* d_dx, int dx_ld, void* d_dz, int dz_ld, float* d_dgamma,
                                 float* d_dbeta, void* stream) {
  return bn_bwd_apply_impl(nullptr, d_dout, dout_ld, d_x, x_ld, d_out_act, act_ld, M, C, d_gamma, d_beta, d_save_mean, d_save_invstd, d_sums,
                           relu, drop_p, drop_seed, d_drop_step, d_dx, dx_ld, d_dz, dz_ld, d_dgamma, d_dbeta, stream);
}
extern "C" int iswm_bn_bwd_apply_global(const void* d_dout, int dout_ld, const void* d_x, int x_ld,
                                        const void* d_out_act, int act_ld, int64_t M, int C,
                                        const float* d_gamma, const float* d_beta, const float* d_save_mean,
                                        const float* d_save_invstd, const double* d_gsums, const double* d_local_sums, int relu, float drop_p,
                                        uint64_t drop_seed, const int64_t* d_drop_step, void* d_dx, int dx_ld, void* d_dz, int dz_ld,
                                        float* d_dgamma, float* d_dbeta, void* stream) {
  ISWM_REQUIRE(d_local_sums, "bn_bwd_apply_global: null local sums");
  return bn_bwd_apply_impl(d_local_sums, d_dout, dout_ld, d_x, x_ld, d_out_act, act_ld, M, C, d_gamma, d_beta, d_save_mean, d_save_invstd, d_gsums,
                           relu, drop_p, drop_seed, d_drop_step, d_dx, dx_ld, d_dz, dz_ld, d_dgamma, d_dbeta, stream);
}

extern "C" int iswm_stem_im2col(const float* d_img, int B, int Cin, int H, int W, int Ho, int Wo,
                                int Kpad, void* d_out, void* stream) {
  ISWM_REQUIRE(d_img && d_out && (Kpad % 8) == 0 && Kpad >= 49 * Cin && Kpad <= 256, "stem_im2col: bad args (Kpad %% 8 == 0, 49*Cin <= Kpad <= 256)");
  ISWM_REQUIRE(Cin >= 1 && Cin <= 5, "stem_im2col: Cin=%d (1..5 supported)", Cin);
  const int strips = (Wo + kStemStrip - 1) / kStemStrip;
  const int64_t blocks = (int64_t)B * Ho * strips;
  ISWM_REQUIRE(blocks < (1ll << 31), "stem_im2col: too many blocks");
  const size_t smem = (size_t)Cin * 7 * (kStemPatchW + 1) * sizeof(float);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(stem_im2col_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    ISWM_REQUIRE(e == cudaSuccess, "stem_im2col: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  }
  launch_k(stem_im2col_kernel, dim3((unsigned)blocks), dim3(kT), smem, ST(stream), d_img, B, Cin, H, W, Ho, Wo, Kpad, BFW(d_out));
  return check_launch("stem_im2col");
}
extern "C" int iswm_stem_rows(const float* d_img, int B, int Cin, int H, int W, int Hh, int Wo, int kpitch, void* d_out, void* stream) {
  ISWM_REQUIRE(d_img && d_out && B >= 1 && H >= 1 && W >= 1, "stem_rows: null/empty");
  ISWM_REQUIRE(Cin >= 1 && Cin <= 3 && 7 * Cin <= 24 && kpitch >= 24 && (kpitch % 8) == 0 && kpitch <= 64,
               "stem_rows: Cin=%d (1..3), kpitch=%d (a multiple of 8 in 24..64)", Cin, kpitch);
  ISWM_REQUIRE(Hh == (H + 1) / 2 && Wo == (W + 1) / 2, "stem_rows: Hh / Wo must be ceil(H/2) / ceil(W/2)");
  const int64_t total = 2ll * B * Hh * Wo;
  const int grid = grid_for(total, kT, 16);
  if (Cin == 3) launch_k(stem_rows_kernel<3>, dim3(grid), dim3(kT), 0, ST(stream), d_img, B, H, W, Hh, Wo, kpitch, BFW(d_out));
  else if (Cin == 2) launch_k(stem_rows_kernel<2>, dim3(grid), dim3(kT), 0, ST(stream), d_img, B, H, W, Hh, Wo, kpitch, BFW(d_out));
  else launch_k(stem_rows_kernel<1>, dim3(grid), dim3(kT), 0, ST(stream), d_img, B, H, W, Hh, Wo, kpitch, BFW(d_out));
  return check_launch("stem_rows");
}
extern "C" int iswm_unpack_wgrad_stem(const float* d_dw, int Cout, int Cin, int ks, int kpitch, float beta, float* d_grad, void* stream) {
  ISWM_REQUIRE(d_dw && d_grad && Cout >= 1 && Cin >= 1 && ks >= 1 && ks * Cin <= kpitch, "unpack_wgrad_stem: bad arguments");
  launch_k(unpack_wgrad_stem_kernel, dim3(grid_for((int64_t)Cout * Cin * ks * ks)), dim3(kT), 0, ST(stream), d_dw, Cout, Cin, ks, kpitch, beta, d_grad);
  return check_launch("unpack_wgrad_stem");
}
extern "C" int iswm_maxpool_fwd(const void* d_x, int B, int H, int W, int C, int Ho, int Wo,
                                void* d_out, uint8_t* d_idx, void* stream) {
  REQ_C8(C, "maxpool_fwd");
  ISWM_REQUIRE(d_x && d_out, "maxpool_fwd: null");
  launch_k(maxpool_fwd_kernel, dim3(grid_for((int64_t)B * Ho * Wo * (C / 8))), dim3(kT), 0, ST(stream), BF(d_x), B, H, W, C, Ho, Wo, BFW(d_out), d_idx);
  return check_launch("maxpool_fwd");
}
extern "C" int iswm_maxpool_bwd(const void* d_dout, const uint8_t* d_idx, int B, int H, int W, int C,
                                int Ho, int Wo, void* d_dx, void* stream) {
  REQ_C8(C, "maxpool_bwd");
  ISWM_REQUIRE(d_dout && d_idx && d_dx, "maxpool_bwd: null");
  launch_k(maxpool_bwd_kernel, dim3(grid_for((int64_t)B * ((H + 1) / 2) * ((W + 1) / 2) * (C / 8), kT, 16)), dim3(kT), 0, ST(stream), BF(d_dout), d_idx, B, H, W, C, Ho, Wo, BFW(d_dx));
  return check_launch("maxpool_bwd");
}

static int launch_reduce_hw(const void* d_x, int x_ld, int B, int64_t HW, int C, float scale, void* d_out, void* stream) {
  const int nvec = C / 8;
  const int nx = std::min(nvec, 16);
  const int ny = kT / nx;
  dim3 grid((nvec + nx - 1) / nx, B);
  launch_k(reduce_hw_kernel, dim3(grid), dim3(kT), 0, ST(stream), BF(d_x), x_ld, HW, C, scale, BFW(d_out), nx, ny);
  return check_launch("reduce_hw");
}
extern "C" int iswm_gap_fwd(const void* d_x, int x_ld, int B, int64_t HW, int C, void* d_out, void* stream) {
  REQ_C8(C, "gap_fwd"); REQ_LD8(x_ld, "gap_fwd");
  ISWM_REQUIRE(d_x && d_out && HW > 0, "gap_fwd: null/empty");
  return launch_reduce_hw(d_x, x_ld, B, HW, C, 1.0f / (float)HW, d_out, stream);
}
extern "C" int iswm_sum_hw(const void* d_x, int x_ld, int B, int64_t HW, int C, void* d_out, void* stream) {
  REQ_C8(C, "sum_hw"); REQ_LD8(x_ld, "sum_hw");
  ISWM_REQUIRE(d_x && d_out && HW > 0, "sum_hw: null/empty");
  return launch_reduce_hw(d_x, x_ld, B, HW, C, 1.0f, d_out, stream);
}
extern "C" int iswm_broadcast_hw(const void* d_x, int B, int64_t HW, int C, void* d_out, int out_ld, void* stream) {
  REQ_C8(C, "broadcast_hw"); REQ_LD8(out_ld, "broadcast_hw");
  ISWM_REQUIRE(d_x && d_out, "broadcast_hw: null");
  launch_k(broadcast_hw_kernel, dim3(grid_for((int64_t)B * HW * (C / 8))), dim3(kT), 0, ST(stream), BF(d_x), B, HW, C, BFW(d_out), out_ld, 1.f, 0);
  return check_launch("broadcast_hw");
}
extern "C" int iswm_gap_bwd_add(const void* d_dpool, int B, int64_t HW, int C, void* d_dx, int dx_ld, void* stream) {
  REQ_C8(C, "gap_bwd_add"); REQ_LD8(dx_ld, "gap_bwd_add");
  ISWM_REQUIRE(d_dpool && d_dx && HW > 0, "gap_bwd_add: null/empty");
  launch_k(broadcast_hw_kernel, dim3(grid_for((int64_t)B * HW * (C / 8))), dim3(kT), 0, ST(stream), BF(d_dpool), B, HW, C, BFW(d_dx), dx_ld, 1.0f / (float)HW, 1);
  return check_launch("gap_bwd_add");
}
namespace iswm {
// x4 upsampling (the decoder's interpolate of the ASPP output, network/_deeplab.py:58, and every size the model is used at):
// a thread owns a 4 x 4 block of output pixels of one 8-channel group. Output rows 4r, 4r+1 share their two source rows, so do
// 4r+2, 4r+3 (only the weights differ) - borders included, because bil_src clamps both the same way - and likewise for columns:
// per row pair 2 x 4 source pixels are loaded for 2 x 4 outputs, 16 loads per 16 stores instead of the generic kernel's 64 (it is
// bound by L2 reads: 4 x 16 B per 16 B written, 11 TB/s of L2 traffic at cfg2). Same weights (bil_src per output) and the
// same expression as the generic kernel: bit-identical results; all register indices are static.
__global__ void __launch_bounds__(kT, 2)
bilinear_up4_fwd_kernel(const __nv_bfloat16* __restrict__ x, int x_ld, int B, int Hi, int Wi, int C,
                        __nv_bfloat16* __restrict__ out, int out_ld) {
  pdl_wait();
  pdl_launch();
  const int nvec = C >> 3;
  const int Ho = 4 * Hi, Wo = 4 * Wi;
  const int64_t total = (int64_t)B * Hi * Wi * nvec;
  for (int64_t i = (int64_t)blockIdx.x * kT + threadIdx.x; i < total; i += (int64_t)gridDim.x * kT) {
    const int c8 = (int)(i % nvec) << 3;
    int64_t m = i / nvec;
    const int k = (int)(m % Wi), r = (int)((m / Wi) % Hi), b = (int)(m / ((int64_t)Wi * Hi));
    int xc[4];                                           // source columns of output columns {4k, 4k+1} and {4k+2, 4k+3}
    float lxs[4];
    {
      float t;
      bil_src(4 * k, 0.25f, Wi, xc[0], xc[1], t);
      bil_src(4 * k + 2, 0.25f, Wi, xc[2], xc[3], t);
#pragma unroll
      for (int dx = 0; dx < 4; dx++) {
        int a0, a1;
        bil_src(4 * k + dx, 0.25f, Wi, a0, a1, lxs[dx]);
      }
    }
#pragma unroll
    for (int g = 0; g < 2; g++) {                        // row pair {4r + 2g, 4r + 2g + 1}
      int y0, y1;
      float t;
      bil_src(4 * r + 2 * g, 0.25f, Hi, y0, y1, t);
      F8 v[2][4];
      const __nv_bfloat16* r0 = x + ((int64_t)b * Hi + y0) * Wi * x_ld + c8;
      const __nv_bfloat16* r1 = x + ((int64_t)b * Hi + y1) * Wi * x_ld + c8;
#pragma unroll
      for (int c = 0; c < 4; c++) {
        v[0][c] = load8(r0 + (int64_t)xc[c] * x_ld);
        v[1][c] = load8(r1 + (int64_t)xc[c] * x_ld);
      }
#pragma unroll
      for (int dy = 0; dy < 2; dy++) {
        const int ho = 4 * r + 2 * g + dy;
        int a0, a1;
        float ly;
        bil_src(ho, 0.25f, Hi, a0, a1, ly);
#pragma unroll
        for (int dx = 0; dx < 4; dx++) {
          const float lx = lxs[dx];
          const float w00 = (1.f - ly) * (1.f - lx), w01 = (1.f - ly) * lx, w10 = ly * (1.f - lx), w11 = ly * lx;
          const int c0 = (dx < 2) ? 0 : 2;               // static after unrolling
          F8 o;
#pragma unroll
          for (int j = 0; j < 8; j++)
            o.v[j] = w00 * v[0][c0].v[j] + w01 * v[0][c0 + 1].v[j] + w10 * v[1][c0].v[j] + w11 * v[1][c0 + 1].v[j];
          store8(out + (((int64_t)b * Ho + ho) * Wo + 4 * k + dx) * out_ld + c8, o);
        }
      }
    }
  }
}
}  // namespace iswm

extern "C" int iswm_bilinear_fwd(const void* d_x, int x_ld, int B, int Hi, int Wi, int C, int Ho, int Wo,
                                 void* d_out, int out_ld, void* stream) {
  REQ_C8(C, "bilinear_fwd"); REQ_LD8(x_ld, "bilinear_fwd"); REQ_LD8(out_ld, "bilinear_fwd");
  ISWM_REQUIRE(d_x && d_out, "bilinear_fwd: null");
  if (Ho == 4 * Hi && Wo == 4 * Wi) {
    const char* e = getenv("ISWM_BILINEAR_UP4");         // "0": the generic kernel (tests compare the two bit for bit)
    if (!(e && e[0] == '0')) {
      launch_k(bilinear_up4_fwd_kernel, dim3(grid_for((int64_t)B * Hi * Wi * (C / 8), kT, 16)), dim3(kT), 0, ST(stream), BF(d_x), x_ld, B, Hi, Wi, C, BFW(d_out), out_ld);
      return check_launch("bilinear_fwd (x4)");
    }
  }
  launch_k(bilinear_fwd_kernel, dim3((unsigned)(B * Ho), (unsigned)std::min(8, (Wo * (C / 8) + kT - 1) / kT)), dim3(kT), 0, ST(stream), BF(d_x), x_ld, B, Hi, Wi, C, Ho, Wo, BFW(d_out), out_ld);
  return check_launch("bilinear_fwd");
}
extern "C" int iswm_bilinear_bwd(const void* d_dout, int dout_ld, int B, int Hi, int Wi, int C, int Ho, int Wo,
                                 void* d_dx, int dx_ld, void* stream) {
  REQ_C8(C, "bilinear_bwd"); REQ_LD8(dout_ld, "bilinear_bwd"); REQ_LD8(dx_ld, "bilinear_bwd");
  ISWM_REQUIRE(d_dout && d_dx, "bilinear_bwd: null");
  ISWM_REQUIRE(Ho <= 14 * Hi, "bilinear_bwd: scale ratio %d/%d above the row-list capacity", Ho, Hi);
  const size_t smem = (size_t)Wo * kBilChunk * sizeof(float);
  ISWM_REQUIRE(smem <= 200 * 1024, "bilinear_bwd: output width %d too large for the shared-memory row", Wo);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(bilinear_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    ISWM_REQUIRE(e == cudaSuccess, "bilinear_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  }
  launch_k(bilinear_bwd_kernel, dim3((unsigned)(B * Hi), (unsigned)((C + kBilChunk - 1) / kBilChunk)), dim3(kT), smem, ST(stream), BF(d_dout), dout_ld, B, Hi, Wi, C, Ho, Wo, BFW(d_dx), dx_ld);
  return check_launch("bilinear_bwd");
}
extern "C" int iswm_logits_up_fwd(const float* d_x, int B, int Hi, int Wi, int C, int Ho, int Wo, float* d_out, void* stream) {
  ISWM_REQUIRE(d_x && d_out && C >= 1, "logits_up_fwd: null");
  launch_k(logits_up_fwd_kernel, dim3((unsigned)(B * Ho), (unsigned)std::min(8, (Wo + kT - 1) / kT)), dim3(kT), 0, ST(stream), d_x, B, Hi, Wi, C, Ho, Wo, d_out);
  return check_launch("logits_up_fwd");
}
extern "C" int iswm_logits_up_bwd(const float* d_dout, int B, int Hi, int Wi, int C, int Ho, int Wo, void* d_dx, int dx_ld,
                                  float* d_bias_grad, void* stream) {
  ISWM_REQUIRE(d_dout && d_dx && C >= 1 && dx_ld >= C, "logits_up_bwd: bad args");
  ISWM_REQUIRE(Ho <= 14 * Hi, "logits_up_bwd: scale ratio %d/%d above the row-list capacity", Ho, Hi);
  const size_t smem = ((size_t)C * Wo + C) * sizeof(float);
  ISWM_REQUIRE(smem <= 200 * 1024, "logits_up_bwd: C * output width = %d x %d too large for the shared-memory row", C, Wo);
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(logits_up_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    ISWM_REQUIRE(e == cudaSuccess, "logits_up_bwd: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
  }
  launch_k(logits_up_bwd_kernel, dim3((unsigned)(B * Hi)), dim3(kT), smem, ST(stream), d_dout, B, Hi, Wi, C, Ho, Wo, BFW(d_dx), dx_ld, d_bias_grad);
  return check_launch("logits_up_bwd");
}
extern "C" int iswm_phase_split(const void* d_x, int x_ld, int B, int H, int W, int C, void* d_out, void* stream) {
  REQ_C8(C, "phase_split"); REQ_LD8(x_ld, "phase_split");
  ISWM_REQUIRE(d_x && d_out, "phase_split: null");
  const int Hp = (H + 1) / 2, Wp = (W + 1) / 2;
  launch_k(phase_split_kernel, dim3(grid_for((int64_t)4 * B * Hp * Wp * (C / 8))), dim3(kT), 0, ST(stream), BF(d_x), x_ld, B, H, W, C, Hp, Wp, BFW(d_out));
  return check_launch("phase_split");
}
extern "C" int iswm_subsample2(const void* d_x, int x_ld, int B, int H, int W, int C, void* d_out, void* stream) {
  REQ_C8(C, "subsample2"); REQ_LD8(x_ld, "subsample2");
  ISWM_REQUIRE(d_x && d_out, "subsample2: null");
  const int Ho = (H + 1) / 2, Wo = (W + 1) / 2;
  launch_k(subsample2_kernel, dim3(grid_for((int64_t)B * Ho * Wo * (C / 8))), dim3(kT), 0, ST(stream), BF(d_x), x_ld, B, H, W, C, Ho, Wo, BFW(d_out));
  return check_launch("subsample2");
}
extern "C" int iswm_zero_stuff2(const void* d_x, int B, int Ho, int Wo, int C, int H, int W, void* d_out, void* stream) {
  REQ_C8(C, "zero_stuff2");
  ISWM_REQUIRE(d_x && d_out, "zero_stuff2: null");
  launch_k(stuff2_kernel, dim3(grid_for((int64_t)B * H * W * (C / 8))), dim3(kT), 0, ST(stream), BF(d_x), B, Ho, Wo, C, H, W, BFW(d_out), 0);
  return check_launch("zero_stuff2");
}
extern "C" int iswm_scatter2_add(const void* d_x, int B, int Ho, int Wo, int C, int H, int W, void* d_inout, void* stream) {
  REQ_C8(C, "scatter2_add");
  ISWM_REQUIRE(d_x && d_inout, "scatter2_add: null");
  launch_k(stuff2_kernel, dim3(grid_for((int64_t)B * Ho * Wo * (C / 8))), dim3(kT), 0, ST(stream), BF(d_x), B, Ho, Wo, C, H, W, BFW(d_inout), 1);
  return check_launch("scatter2_add");
}
extern "C" int iswm_add_bf16(const void* d_a, const void* d_b, int64_t n, void* d_out, void* stream) {
  ISWM_REQUIRE(d_a && d_b && d_out && (n % 8) == 0, "add_bf16: n must be a multiple of 8");
  if (n == 0) return 0;
  launch_k(add_bf16_kernel, dim3(grid_for(n / 8)), dim3(kT), 0, ST(stream), BF(d_a), BF(d_b), n / 8, BFW(d_out));
  return check_launch("add_bf16");
}
extern "C" int iswm_nhwc_to_nchw_f32(const void* d_x, int x_ld, int B, int64_t HW, int C, float* d_out, void* stream) {
  ISWM_REQUIRE(d_x && d_out, "nhwc_to_nchw_f32: null");
  launch_k(nhwc_to_nchw_f32_kernel, dim3(grid_for((int64_t)B * HW * C)), dim3(kT), 0, ST(stream), BF(d_x), x_ld, B, HW, C, d_out);
  return check_launch("nhwc_to_nchw_f32");
}
extern "C" int iswm_nchw_f32_to_nhwc(const float* d_x, int B, int64_t HW, int C, void* d_out, int out_ld, void* stream) {
  ISWM_REQUIRE(d_x && d_out, "nchw_f32_to_nhwc: null");
  launch_k(nchw_f32_to_nhwc_kernel, dim3(grid_for((int64_t)B * HW * C)), dim3(kT), 0, ST(stream), d_x, B, HW, C, BFW(d_out), out_ld);
  return check_launch("nchw_f32_to_nhwc");
}
extern "C" int iswm_sgd_step(float* d_param, const float* d_grad, float* d_mom, int64_t n, float lr,
                             float momentum, float weight_decay, int nesterov, int first_step, const float* d_lr, void* stream) {
  ISWM_REQUIRE(d_param && d_grad && (momentum == 0.f || d_mom), "sgd_step: null");
  if (n == 0) return 0;
  launch_k(sgd_step_kernel, dim3(grid_for(n)), dim3(kT), 0, ST(stream), d_param, d_grad, d_mom, n, lr, momentum, weight_decay, nesterov, first_step, d_lr);
  return check_launch("sgd_step");
}

extern "C" int iswm_bias_grad_nchw(const float* d_dout, int B, int C, int64_t HW, float* d_out, void* stream) {
  ISWM_REQUIRE(d_dout && d_out && C >= 1, "bias_grad_nchw: null");
  if ((int64_t)B * HW == 0) return 0;
  dim3 grid(grid_for((int64_t)B * HW, kT * 8, 2), C);
  launch_k(bias_grad_nchw_kernel, dim3(grid), dim3(kT), 0, ST(stream), d_dout, B, C, HW, d_out);
  return check_launch("bias_grad_nchw");
}
extern "C" int iswm_scale_by_device_scalar(void* d_x, int dtype, int64_t n, const float* d_scalar, void* stream) {
  ISWM_REQUIRE(d_x && d_scalar, "scale_by_device_scalar: null");
  if (n == 0) return 0;
  if (dtype == ISWM_F32)
    launch_k(scale_by_device_scalar_kernel<float>, dim3(grid_for(n)), dim3(kT), 0, ST(stream), static_cast<float*>(d_x), n, d_scalar);
  else if (dtype == ISWM_BF16)
    launch_k(scale_by_device_scalar_kernel<__nv_bfloat16>, dim3(grid_for(n)), dim3(kT), 0, ST(stream), BFW(d_x), n, d_scalar);
  else { set_error("scale_by_device_scalar: bad dtype %d", dtype); return 2; }
  return check_launch("scale_by_device_scalar");
}

extern "C" int iswm_pack_weights_batched(const void* d_jobs, int n_jobs, int total_blocks, void* stream) {
  static_assert(sizeof(PackJob) == 48, "PackJob layout is part of the C ABI (iswm_pack_job)");
  ISWM_REQUIRE(d_jobs && n_jobs >= 1 && total_blocks >= 1, "pack_weights_batched: bad args");
  launch_k(pack_weights_batched_kernel, dim3(total_blocks), dim3(kT), 0, ST(stream), static_cast<const PackJob*>(d_jobs), n_jobs);
  return check_launch("pack_weights_batched");
}

extern "C" int iswm_adam_step(float* d_param, const float* d_grad, float* d_exp_avg, float* d_exp_avg_sq, int64_t n,
                              float lr, float beta1, float beta2, float eps, float weight_decay, int adamw,
                              int64_t step, const float* d_lr, const int64_t* d_step, void* stream) {
  ISWM_REQUIRE(d_param && d_grad && d_exp_avg && d_exp_avg_sq, "adam_step: null");
  ISWM_REQUIRE(step >= 1 || d_step, "adam_step: step=%lld must be >= 1 (1 on the first update)", (long long)step);
  if (step < 1) step = 1;
  ISWM_REQUIRE(((reinterpret_cast<uintptr_t>(d_param) | reinterpret_cast<uintptr_t>(d_grad) | reinterpret_cast<uintptr_t>(d_exp_avg) |
                 reinterpret_cast<uintptr_t>(d_exp_avg_sq)) & 15) == 0, "adam_step: buffers must be 16-byte aligned");
  if (n == 0) return 0;
  // bias corrections on the host in double, as torch computes them from a Python float step
  const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
  const float step_size = (float)((double)lr / bc1);
  const float inv_sqrt_bc2 = (float)(1.0 / sqrt(bc2));
  launch_k(adam_step_kernel, dim3(grid_for(n, kT * 4)), dim3(kT), 0, ST(stream), d_param, d_grad, d_exp_avg, d_exp_avg_sq, n, lr, beta1, beta2,
           eps, weight_decay, adamw, step_size, inv_sqrt_bc2, d_lr, reinterpret_cast<const long long*>(d_step));
  return check_launch("adam_step");
}

extern "C" int iswm_u8_to_f32_norm(const uint8_t* d_src, int B, int Hs, int Ws, int C, const int32_t* d_origin_xy,
                                   const uint8_t* d_flip, const float* mean, const float* stdv, int H, int W,
                                   float* d_out, void* stream) {
  ISWM_REQUIRE(d_src && d_out && mean && stdv, "u8_to_f32_norm: null");
  ISWM_REQUIRE(C >= 1 && C <= 4, "u8_to_f32_norm: C=%d (1..4 channels)", C);
  ISWM_REQUIRE(B >= 0 && H >= 1 && W >= 1 && H <= Hs && W <= Ws, "u8_to_f32_norm: window %dx%d does not fit the %dx%d source", H, W, Hs, Ws);
  ISWM_REQUIRE((int64_t)B * H < (1ll << 31), "u8_to_f32_norm: too many rows");
  if (B == 0) return 0;
  float mu[4] = {0, 0, 0, 0}, sd[4] = {1, 1, 1, 1};
  for (int c = 0; c < C; c++) { mu[c] = mean[c]; sd[c] = stdv[c]; }       // host arrays (3 floats), passed by value
  dim3 grid((unsigned)(B * H), (unsigned)std::max(1, std::min(8, ((W + 3) / 4 + kT - 1) / kT)));
  launch_k(u8_to_f32_norm_kernel, grid, dim3(kT), 0, ST(stream), d_src, Hs, Ws, C, d_origin_xy, d_flip, make_float3(mu[0], mu[1], mu[2]),
           make_float3(sd[0], sd[1], sd[2]), mu[3], sd[3], H, W, d_out);
  return check_launch("u8_to_f32_norm");
}

extern "C" int iswm_crop_flip_u8(const uint8_t* d_src, int B, int Hs, int Ws, const int32_t* d_origin_xy,
                                 const uint8_t* d_flip, int H, int W, uint8_t* d_out, void* stream) {
  ISWM_REQUIRE(d_src && d_out, "crop_flip_u8: null");
  ISWM_REQUIRE(B >= 0 && H >= 1 && W >= 1 && H <= Hs && W <= Ws, "crop_flip_u8: window %dx%d does not fit the %dx%d source", H, W, Hs, Ws);
  ISWM_REQUIRE((int64_t)B * H < (1ll << 31), "crop_flip_u8: too many rows");
  if (B == 0) return 0;
  dim3 grid((unsigned)(B * H), (unsigned)std::max(1, std::min(8, (W + kT - 1) / kT)));
  launch_k(crop_flip_u8_kernel, grid, dim3(kT), 0, ST(stream), d_src, Hs, Ws, d_origin_xy, d_flip, H, W, d_out);
  return check_launch("crop_flip_u8");
}

extern "C" int iswm_unpack_wgrad_batched(const void* d_jobs, int n_jobs, int total_blocks, void* stream) {
  ISWM_REQUIRE(d_jobs && n_jobs >= 1 && total_blocks >= 1, "unpack_wgrad_batched: empty job list");
  static_assert(sizeof(UnpackJob) == 40, "iswm_unpack_job layout");
  launch_k(unpack_wgrad_batched_kernel, dim3((unsigned)total_blocks), dim3(kT), 0, ST(stream), static_cast<const UnpackJob*>(d_jobs), n_jobs);
  return check_launch("unpack_wgrad_batched");
}
