// conv_wgrad.cu — weight gradient of a convolution on tcgen05 tensor cores.
//
//   dW[cout, tap, cin] = sum_pixels dy[pixel, cout] * x[pixel + offset(tap), cin]
//
// GEMM view: M = cout (128 per tile), N = (tap, cin) columns, K = pixels. Both
// operands are NHWC, i.e. the contraction index (pixel) is the slow one, so both are fed
// to the MMA as MN-major 128B-swizzled tiles: a TMA box of {64 channels, 64 pixels} lands
// as 64 rows (K) of 128 bytes (64 channels of M or N). The tap shift and the zero padding
// come from the TMA coordinates exactly as in conv_igemm.cu. The pixel range is split
// across CTAs (split-K) and partial tiles are reduced with fp32 atomics into dW.
//
// The N side of a tile is a run of up to 6 "column chunks" of the linearised (tap, 64-channel slice) axis, each loaded
// with its own tap shift: narrow layers put several taps side by side behind ONE dy tile (3x3 64->64: three taps per
// tile, N = 192, instead of nine N = 64 tiles that each re-read dy), and Cin = 304 runs as one 5-chunk tile per tap
// (N = 192 + 112 as two MMAs into 320 TMEM columns) instead of two 160-column tiles. Tiles wider than 256 columns use a
// single accumulator (each CTA owns one tile in split mode, so there is nothing to double-buffer against).
//
// Replaces the autograd weight gradients of every nn.Conv2d on the hot path
// (network/backbone/resnet.py:27-35, network/_deeplab.py:37-51,124,134,149,162)
// produced by loss.backward() at train.py:1048.
#include "tc_common.cuh"
#include <algorithm>
#include <array>
#include <cmath>
#include <vector>

namespace iswm {

constexpr int kWStages = 8;
constexpr int kWTileM = 128;
constexpr int kPixBlock = 64;               // pixels per k-block
constexpr int kChunkBytes = 64 * 128;       // one {64 ch x 64 px} box = 8 KiB
constexpr int kWTmemCols = 512;
constexpr int kWSmemBudget = 232448 - 1024 - 256;   // opt-in limit minus alignment slack and barriers
constexpr int kMaxG = 6;                            // column chunks per tile

struct WgradKParams {
  int Cout, Cin, ntaps;
  int lgBW, lgBH;                 // pixel box: BW*BH*BB == 64
  int tiles_w, tiles_h, tiles_b;  // pixel blocks
  int pix_blocks;
  int tiles_m, tiles_n, stages;
  int G, cchunks, T;              // chunks per tile, 64-channel slices per tap, total chunks = ntaps * cchunks
  int tail_cols;                  // valid columns of a tap's last slice rounded up to 16 (64 when Cin % 64 == 0)
  int acc_cols, nacc;             // TMEM columns per accumulator, accumulators (2 while 2 * 64 * G <= 512)
  int n_tiles;                    // output tiles = tiles_m * tiles_n
  long long total_kblocks;        // n_tiles * pix_blocks
  long long kblocks_per_cta;      // stream-K mode: equal contiguous ranges of the linearised (tile, pixel block) space
  int splits, split_len;          // split mode (splits > 0): CTA = (tile, split); same-split CTAs walk the same pixels
  int vec_red;
  int nprod;                      // producer warps (1 or 2) taking alternate pixel blocks
  int n_img_per_phase;
  int phase_view, pv_ld;          // x read as the four parity phases of a dense tensor through a 5-D tensor map
  int8_t dh[ISWM_MAX_TAPS], dw[ISWM_MAX_TAPS], phase[ISWM_MAX_TAPS];
  float* dwgt;
  int* abort_flag;
};

__global__ void __launch_bounds__(256, 1)
conv_wgrad_kernel(const __grid_constant__ CUtensorMap tmap_dy,
                  const __grid_constant__ CUtensorMap tmap_x, const WgradKParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = tc::smem_u32(smem_raw);
  const uint32_t ring = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (ring - raw_addr);
  const uint32_t a_bytes = 2 * kChunkBytes;
  const uint32_t stage_bytes = a_bytes + (uint32_t)p.G * kChunkBytes;
  uint8_t* tail = smem + (size_t)p.stages * stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kWStages + 4);

  const uint32_t bar_full = tc::smem_u32(bars);
  const uint32_t bar_empty = bar_full + 8 * kWStages;
  const uint32_t bar_tfull = bar_empty + 8 * kWStages;
  const uint32_t bar_tempty = bar_tfull + 16;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 0 && lane == 0) {
    tc::tma_prefetch_desc(&tmap_dy);
    tc::tma_prefetch_desc(&tmap_x);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.stages; s++) {
      tc::mbar_init(bar_full + 8 * s, 1);
      tc::mbar_init(bar_empty + 8 * s, 1);
    }
    for (int s = 0; s < 2; s++) {
      tc::mbar_init(bar_tfull + 8 * s, 1);
      tc::mbar_init(bar_tempty + 8 * s, 4);
    }
    tc::fence_barrier_init();
  }
  if (warp == 2) {
    tc::tmem_alloc(tc::smem_u32(tmem_slot), kWTmemCols);
    tc::tmem_relinquish();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  // prologue done (barriers, TMEM, descriptor prefetch touch no global data): wait for the producer grid, then let
  // the next kernel of the stream start its own prologue under our main loop
  pdl_wait();
  pdl_launch();

  const int BW = 1 << p.lgBW, BH = 1 << p.lgBH;
  const int BB = kPixBlock >> (p.lgBW + p.lgBH);

  // Stream-K: the (output tile, pixel block) space is linearised and cut into equal contiguous
  // ranges, one per CTA; a CTA flushes its partial tile with fp32 reductions whenever its range
  // crosses a tile boundary. tile -> (m tile, tap, n tile), n fastest (neighbours share dy in L2).
  auto decode = [&](int tile, int& mt, int& nt) {
    nt = tile % p.tiles_n;
    mt = tile / p.tiles_n;
  };
  // columns of n-tile nt: gc chunks starting at chunk g0 of the (tap, slice) axis; the MMA covers ncols of them (a trailing
  // partial slice is trimmed to 16; partial slices in the middle of a tile run as zero columns)
  auto tile_cols = [&](int nt, int& g0, int& gc, int& ncols) {
    g0 = nt * p.G;
    gc = min(p.G, p.T - g0);
    const int last = g0 + gc - 1;
    const bool tail = (last % p.cchunks) == p.cchunks - 1;
    ncols = 64 * (gc - 1) + (tail ? p.tail_cols : 64);
  };
  long long range_lo, range_hi;
  if (p.splits > 0) {
    // every CTA of one split index reads the SAME pixel blocks at the same time (different output tiles), so dy / x
    // stream from HBM once and are shared through L2; partial tiles are reduced with fp32 atomics at the end
    const int t = (int)(blockIdx.x % (unsigned)p.n_tiles), sp = (int)(blockIdx.x / (unsigned)p.n_tiles);
    range_lo = (long long)t * p.pix_blocks + (long long)sp * p.split_len;
    range_hi = min(range_lo + p.split_len, (long long)(t + 1) * p.pix_blocks);
  } else {
    range_lo = (long long)blockIdx.x * p.kblocks_per_cta;
    range_hi = min(range_lo + p.kblocks_per_cta, p.total_kblocks);
  }

  // producer / MMA roles: ONE elected thread runs the whole schedule (see conv_igemm.cu); producer warps 0 and 3 take
  // alternate k-blocks (pixel blocks) of the CTA's range; pixel-block coordinates advance incrementally (no divisions
  // inside the k loop)
  if (warp == 0 || (warp == 3 && p.nprod == 2)) {
    if (tc::elect_one()) {
      const int me = (warp == 0) ? 0 : 1;
      const int np = p.nprod;
      int stage = me % p.stages;
      uint32_t phase = 0;
      long long q0 = 0;                         // k-blocks of this CTA issued before the current segment
      bool ok = true;
      for (long long cur = range_lo; cur < range_hi && ok;) {
        const int tile = (int)(cur / p.pix_blocks);
        const int pb0 = (int)(cur - (long long)tile * p.pix_blocks);
        const int pb1 = (int)min((long long)p.pix_blocks, pb0 + (range_hi - cur));
        int mt, nt, g0, gc, ncols;
        decode(tile, mt, nt);
        tile_cols(nt, g0, gc, ncols);
        const int m0 = mt * kWTileM;
        // per-chunk tap shift and channel origin of this tile (registers; the k loop below only adds the pixel-block origin)
        int c_dw[kMaxG], c_dh[kMaxG], c_db[kMaxG], c_ch[kMaxG];
        {
          int tap = g0 / p.cchunks, cc = g0 - tap * p.cchunks;
#pragma unroll
          for (int j = 0; j < kMaxG; j++) {
            const int t_ = min(tap, p.ntaps - 1);
            c_dw[j] = p.dw[t_]; c_dh[j] = p.dh[t_]; c_ch[j] = cc * 64;
            if (p.phase_view) { c_db[j] = p.phase[t_] >> 1; c_ch[j] += (p.phase[t_] & 1) * p.pv_ld; }   // row parity; column parity in the channel coordinate
            else c_db[j] = p.phase[t_] * p.n_img_per_phase;
            if (++cc == p.cchunks) { cc = 0; tap++; }
          }
        }
        const uint32_t tx_bytes = a_bytes + (uint32_t)gc * kChunkBytes;
        int off = me - (int)(q0 % np);
        if (off < 0) off += np;
        int pb = pb0 + off;
        int tw = pb % p.tiles_w, th = (pb / p.tiles_w) % p.tiles_h, tb = pb / (p.tiles_w * p.tiles_h);
        for (; pb < pb1; pb += np) {
          const int w0 = tw * BW, h0 = th * BH, b0 = tb * BB;
          ok = tc::mbar_wait(bar_empty + 8 * stage, phase ^ 1, p.abort_flag, 11);
          if (!ok) break;
          const uint32_t dst = ring + stage * stage_bytes;
          const uint32_t bar = bar_full + 8 * stage;
          tc::mbar_expect_tx(bar, tx_bytes);
          tc::tma_load_4d(dst, &tmap_dy, bar, m0, w0, h0, b0);
          tc::tma_load_4d(dst + kChunkBytes, &tmap_dy, bar, m0 + 64, w0, h0, b0);
#pragma unroll
          for (int j = 0; j < kMaxG; j++)
            if (j < gc) {
              if (p.phase_view) tc::tma_load_5d(dst + a_bytes + j * kChunkBytes, &tmap_x, bar, c_ch[j], w0 + c_dw[j], c_db[j], h0 + c_dh[j], b0);
              else tc::tma_load_4d(dst + a_bytes + j * kChunkBytes, &tmap_x, bar, c_ch[j], w0 + c_dw[j], h0 + c_dh[j], b0 + c_db[j]);
            }
          stage += np;
          if (stage >= p.stages) { stage -= p.stages; phase ^= 1; }
          tw += np;
          while (tw >= p.tiles_w) { tw -= p.tiles_w; th++; }
          while (th >= p.tiles_h) { th -= p.tiles_h; tb++; }
        }
        q0 += pb1 - pb0;
        cur += pb1 - pb0;
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (tc::elect_one()) {
      int stage = 0, as = 0;
      uint32_t phase = 0, aphase = 0;
      bool ok = true;
      for (long long cur = range_lo; cur < range_hi && ok;) {
        const int tile = (int)(cur / p.pix_blocks);
        const int pb0 = (int)(cur - (long long)tile * p.pix_blocks);
        const int pb1 = (int)min((long long)p.pix_blocks, pb0 + (range_hi - cur));
        int mt, nt, g0, gc, ncols;
        decode(tile, mt, nt);
        tile_cols(nt, g0, gc, ncols);
        // up to 256 columns per MMA: wider tiles run as two MMAs over the first h1 chunks and the rest
        const int h1 = (ncols <= 256) ? gc : (gc + 1) / 2;
        const int n1 = (ncols <= 256) ? ncols : 64 * h1, n2 = ncols - n1;
        const uint32_t idesc1 = tc::make_idesc_bf16(kWTileM, n1, 1, 1);   // both operands MN-major
        const uint32_t idesc2 = tc::make_idesc_bf16(kWTileM, n2 > 0 ? n2 : 16, 1, 1);
        ok = tc::mbar_wait(bar_tempty + 8 * as, aphase ^ 1, p.abort_flag, 12);
        if (!ok) break;
        tc::tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * p.acc_cols);
        for (int pb = pb0; pb < pb1; pb++) {
          ok = tc::mbar_wait(bar_full + 8 * stage, phase, p.abort_flag, 13);
          if (!ok) break;
          tc::tc_fence_after();
          const uint32_t a_addr = ring + stage * stage_bytes;
          // MN-major SW128: LBO = byte stride between 64-channel chunks, SBO = 8 pixel rows
          const uint64_t da = tc::make_smem_desc_sw128(a_addr, kChunkBytes, 1024);
          const uint64_t db = tc::make_smem_desc_sw128(a_addr + a_bytes, kChunkBytes, 1024);
          const uint32_t first = (pb > pb0) ? 1u : 0u;
#pragma unroll
          for (int k = 0; k < kPixBlock / 16; k++)     // 16 pixel rows = 2048 bytes per MMA
            tc::umma_bf16(d_tmem, da + 128 * k, db + 128 * k, idesc1, first | (uint32_t)(k > 0));
          if (n2 > 0) {
            const uint64_t db2 = tc::make_smem_desc_sw128(a_addr + a_bytes + (uint32_t)h1 * kChunkBytes, kChunkBytes, 1024);
#pragma unroll
            for (int k = 0; k < kPixBlock / 16; k++)
              tc::umma_bf16(d_tmem + (uint32_t)n1, da + 128 * k, db2 + 128 * k, idesc2, first | (uint32_t)(k > 0));
          }
          tc::umma_commit(bar_empty + 8 * stage);
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
        if (!ok) break;
        tc::umma_commit(bar_tfull + 8 * as);
        if (++as == p.nacc) { as = 0; aphase ^= 1; }
        cur += pb1 - pb0;
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    const int ew = warp - 4;
    const int row = ew * 32 + lane;
    int as = 0;
    uint32_t aphase = 0;
    for (long long cur = range_lo; cur < range_hi;) {
      const int tile = (int)(cur / p.pix_blocks);
      const int pb0 = (int)(cur - (long long)tile * p.pix_blocks);
      const int pb1 = (int)min((long long)p.pix_blocks, pb0 + (range_hi - cur));
      int mt, nt, g0, gc, ncols;
      decode(tile, mt, nt);
      tile_cols(nt, g0, gc, ncols);
      const int m = mt * kWTileM + row;
      if (!tc::mbar_wait(bar_tfull + 8 * as, aphase, p.abort_flag, 14)) break;
      tc::tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(as * p.acc_cols);
      int tap = g0 / p.cchunks, cc = g0 - tap * p.cchunks;
      for (int j = 0; j < gc; j++) {                     // one 64-channel slice of one tap per chunk
        float* orow = p.dwgt + ((size_t)m * p.ntaps + tap) * p.Cin + cc * 64;
        const int nvalid = min(64, p.Cin - cc * 64);     // channels of this slice that exist
        const int ccols = min(64, ncols - 64 * j);       // columns of it the MMA produced
        for (int c = 0; c < ccols; c += 16) {
          uint32_t v[16];
          tc::tmem_ld16(t_row + 64 * j + c, v);
          tc::tmem_ld_wait();
          if (m < p.Cout) {
            if (p.vec_red && c + 16 <= nvalid) {
#pragma unroll
              for (int i = 0; i < 16; i += 4)
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(orow + c + i),
                             "f"(__uint_as_float(v[i])), "f"(__uint_as_float(v[i + 1])),
                             "f"(__uint_as_float(v[i + 2])), "f"(__uint_as_float(v[i + 3]))
                             : "memory");
            } else {
#pragma unroll
              for (int i = 0; i < 16; i++)
                if (c + i < nvalid) atomicAdd(orow + c + i, __uint_as_float(v[i]));
            }
          }
        }
        if (++cc == p.cchunks) { cc = 0; tap++; }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(bar_tempty + 8 * as);
      if (++as == p.nacc) { as = 0; aphase ^= 1; }
      cur += pb1 - pb0;
    }
  }

  tc::tc_fence_before();
  __syncthreads();
  if (warp == 2) tc::tmem_dealloc(tmem_base, kWTmemCols);
}

// ---------------------------------------------------------------------------------------------------------------------
// Grouped launch: the weight gradients of SEVERAL convolutions (one ResNet layer's worth) in one kernel. A small GEMM
// launched alone has to be cut into many pixel-range splits to occupy 148 SMs, and every split ends by adding its whole
// partial tile into dW with fp32 reductions - for a 1x1 layer at 32x32 that flush is most of the launch. With 10-20 layers
// side by side there are enough output tiles to go round: units of work = (job, output tile, pixel-block range), few splits
// per tile, dealt to the CTAs by the host (longest first onto the least loaded CTA); a CTA walks its list with the TMA ring,
// the accumulator pair and the barriers running straight through the unit boundaries.
constexpr int kMaxJobs = 24;
struct WJob {
  CUtensorMap tmap_dy, tmap_x;
  WgradKParams p;
};
struct WGroupParams {
  int n_jobs, max_units, stages, G, nprod;
  const int4* units;                 // [grid][max_units]: {job, tile, first pixel block, end pixel block}; job < 0 ends a CTA's list
  int* abort_flag;
  WJob jobs[kMaxJobs];
};

__global__ void __launch_bounds__(256, 1)
conv_wgrad_grouped_kernel(const __grid_constant__ WGroupParams P) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = tc::smem_u32(smem_raw);
  const uint32_t ring = (raw_addr + 1023u) & ~1023u;
  uint8_t* smem = smem_raw + (ring - raw_addr);
  const uint32_t a_bytes = 2 * kChunkBytes;
  const uint32_t stage_bytes = a_bytes + (uint32_t)P.G * kChunkBytes;
  uint8_t* tail = smem + (size_t)P.stages * stage_bytes;
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail);
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kWStages + 4);
  const uint32_t bar_full = tc::smem_u32(bars);
  const uint32_t bar_empty = bar_full + 8 * kWStages;
  const uint32_t bar_tfull = bar_empty + 8 * kWStages;
  const uint32_t bar_tempty = bar_tfull + 16;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < P.stages; s++) {
      tc::mbar_init(bar_full + 8 * s, 1);
      tc::mbar_init(bar_empty + 8 * s, 1);
    }
    for (int s = 0; s < 2; s++) {
      tc::mbar_init(bar_tfull + 8 * s, 1);
      tc::mbar_init(bar_tempty + 8 * s, 4);
    }
    tc::fence_barrier_init();
  }
  if (warp == 2) {
    tc::tmem_alloc(tc::smem_u32(tmem_slot), kWTmemCols);
    tc::tmem_relinquish();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_wait();
  pdl_launch();
  const int4* my_units = P.units + (size_t)blockIdx.x * P.max_units;
  constexpr uint32_t kAccStride = 256;                    // two accumulators of up to 256 columns (jobs run <= 4 chunks per tile)

  auto tile_cols = [](const WgradKParams& p, int nt, int& g0, int& gc, int& ncols) {
    g0 = nt * p.G;
    gc = min(p.G, p.T - g0);
    const int last = g0 + gc - 1;
    const bool tl = (last % p.cchunks) == p.cchunks - 1;
    ncols = 64 * (gc - 1) + (tl ? p.tail_cols : 64);
  };

  if (warp == 0 || (warp == 3 && P.nprod == 2)) {
    if (tc::elect_one()) {
      const int me = (warp == 0) ? 0 : 1;
      const int np = P.nprod;
      int stage = me % P.stages;
      uint32_t phase = 0;
      long long q0 = 0;
      bool ok = true;
      for (int ui = 0; ui < P.max_units && ok; ui++) {
        const int4 u = my_units[ui];
        if (u.x < 0) break;
        const WgradKParams& p = P.jobs[u.x].p;
        const CUtensorMap* tm_dy = &P.jobs[u.x].tmap_dy;
        const CUtensorMap* tm_x = &P.jobs[u.x].tmap_x;
        const int BW = 1 << p.lgBW, BH = 1 << p.lgBH, BB = kPixBlock >> (p.lgBW + p.lgBH);
        const int nt = u.y % p.tiles_n, mt = u.y / p.tiles_n;
        int g0, gc, ncols;
        tile_cols(p, nt, g0, gc, ncols);
        const int m0 = mt * kWTileM;
        int c_dw[4], c_dh[4], c_db[4], c_ch[4];
        {
          int tap = g0 / p.cchunks, cc = g0 - tap * p.cchunks;
#pragma unroll
          for (int j = 0; j < 4; j++) {
            const int t_ = min(tap, p.ntaps - 1);
            c_dw[j] = p.dw[t_]; c_dh[j] = p.dh[t_]; c_ch[j] = cc * 64;
            if (p.phase_view) { c_db[j] = p.phase[t_] >> 1; c_ch[j] += (p.phase[t_] & 1) * p.pv_ld; }
            else c_db[j] = p.phase[t_] * p.n_img_per_phase;
            if (++cc == p.cchunks) { cc = 0; tap++; }
          }
        }
        const uint32_t tx_bytes = a_bytes + (uint32_t)gc * kChunkBytes;
        int off = me - (int)(q0 % np);
        if (off < 0) off += np;
        int pb = u.z + off;
        int tw = pb % p.tiles_w, th = (pb / p.tiles_w) % p.tiles_h, tb = pb / (p.tiles_w * p.tiles_h);
        for (; pb < u.w; pb += np) {
          const int w0 = tw * BW, h0 = th * BH, b0 = tb * BB;
          ok = tc::mbar_wait(bar_empty + 8 * stage, phase ^ 1, P.abort_flag, 41);
          if (!ok) break;
          const uint32_t dst = ring + stage * stage_bytes;
          const uint32_t bar = bar_full + 8 * stage;
          tc::mbar_expect_tx(bar, tx_bytes);
          tc::tma_load_4d(dst, tm_dy, bar, m0, w0, h0, b0);
          tc::tma_load_4d(dst + kChunkBytes, tm_dy, bar, m0 + 64, w0, h0, b0);
#pragma unroll
          for (int j = 0; j < 4; j++)
            if (j < gc) {
              if (p.phase_view) tc::tma_load_5d(dst + a_bytes + j * kChunkBytes, tm_x, bar, c_ch[j], w0 + c_dw[j], c_db[j], h0 + c_dh[j], b0);
              else tc::tma_load_4d(dst + a_bytes + j * kChunkBytes, tm_x, bar, c_ch[j], w0 + c_dw[j], h0 + c_dh[j], b0 + c_db[j]);
            }
          stage += np;
          if (stage >= P.stages) { stage -= P.stages; phase ^= 1; }
          tw += np;
          while (tw >= p.tiles_w) { tw -= p.tiles_w; th++; }
          while (th >= p.tiles_h) { th -= p.tiles_h; tb++; }
        }
        q0 += u.w - u.z;
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (tc::elect_one()) {
      int stage = 0, as = 0;
      uint32_t phase = 0, aphase = 0;
      bool ok = true;
      for (int ui = 0; ui < P.max_units && ok; ui++) {
        const int4 u = my_units[ui];
        if (u.x < 0) break;
        const WgradKParams& p = P.jobs[u.x].p;
        int g0, gc, ncols;
        tile_cols(p, u.y % p.tiles_n, g0, gc, ncols);
        const uint32_t idesc = tc::make_idesc_bf16(kWTileM, ncols, 1, 1);
        ok = tc::mbar_wait(bar_tempty + 8 * as, aphase ^ 1, P.abort_flag, 42);
        if (!ok) break;
        tc::tc_fence_after();
        const uint32_t d_tmem = tmem_base + (uint32_t)as * kAccStride;
        for (int pb = u.z; pb < u.w; pb++) {
          ok = tc::mbar_wait(bar_full + 8 * stage, phase, P.abort_flag, 43);
          if (!ok) break;
          tc::tc_fence_after();
          const uint32_t a_addr = ring + stage * stage_bytes;
          const uint64_t da = tc::make_smem_desc_sw128(a_addr, kChunkBytes, 1024);
          const uint64_t db = tc::make_smem_desc_sw128(a_addr + a_bytes, kChunkBytes, 1024);
          const uint32_t first = (pb > u.z) ? 1u : 0u;
#pragma unroll
          for (int k = 0; k < kPixBlock / 16; k++)
            tc::umma_bf16(d_tmem, da + 128 * k, db + 128 * k, idesc, first | (uint32_t)(k > 0));
          tc::umma_commit(bar_empty + 8 * stage);
          if (++stage == P.stages) { stage = 0; phase ^= 1; }
        }
        if (!ok) break;
        tc::umma_commit(bar_tfull + 8 * as);
        as ^= 1;
        if (as == 0) aphase ^= 1;
      }
    }
    __syncwarp();
  } else if (warp >= 4) {
    const int ew = warp - 4;
    const int row = ew * 32 + lane;
    int as = 0;
    uint32_t aphase = 0;
    for (int ui = 0; ui < P.max_units; ui++) {
      const int4 u = my_units[ui];
      if (u.x < 0) break;
      const WgradKParams& p = P.jobs[u.x].p;
      const int nt = u.y % p.tiles_n, mt = u.y / p.tiles_n;
      int g0, gc, ncols;
      tile_cols(p, nt, g0, gc, ncols);
      const int m = mt * kWTileM + row;
      if (!tc::mbar_wait(bar_tfull + 8 * as, aphase, P.abort_flag, 44)) break;
      tc::tc_fence_after();
      const uint32_t t_row = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)as * kAccStride;
      int tap = g0 / p.cchunks, cc = g0 - tap * p.cchunks;
      for (int j = 0; j < gc; j++) {
        float* orow = p.dwgt + ((size_t)m * p.ntaps + tap) * p.Cin + cc * 64;
        const int nvalid = min(64, p.Cin - cc * 64);
        const int ccols = min(64, ncols - 64 * j);
        for (int c = 0; c < ccols; c += 16) {
          uint32_t v[16];
          tc::tmem_ld16(t_row + 64 * j + c, v);
          tc::tmem_ld_wait();
          if (m < p.Cout) {
            if (p.vec_red && c + 16 <= nvalid) {
#pragma unroll
              for (int i = 0; i < 16; i += 4)
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(orow + c + i),
                             "f"(__uint_as_float(v[i])), "f"(__uint_as_float(v[i + 1])),
                             "f"(__uint_as_float(v[i + 2])), "f"(__uint_as_float(v[i + 3]))
                             : "memory");
            } else {
#pragma unroll
              for (int i = 0; i < 16; i++)
                if (c + i < nvalid) atomicAdd(orow + c + i, __uint_as_float(v[i]));
            }
          }
        }
        if (++cc == p.cchunks) { cc = 0; tap++; }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(bar_tempty + 8 * as);
      as ^= 1;
      if (as == 0) aphase ^= 1;
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 2) tc::tmem_dealloc(tmem_base, kWTmemCols);
}

static int ilog2_ceil_w(int v) {
  int l = 0;
  while ((1 << l) < v) l++;
  return l;
}

}  // namespace iswm

using namespace iswm;

extern "C" int iswm_conv_wgrad(const iswm_conv_desc* d, const void* d_in, const void* d_dy,
                               float* d_dw, void* stream) {
  return iswm_conv_wgrad_ex(d, d_in, d_dy, d_dw, 0, stream);
}

extern "C" int iswm_conv_wgrad_ex(const iswm_conv_desc* d, const void* d_in, const void* d_dy,
                                  float* d_dw, int max_ctas, void* stream) {
  if (debug_skip(ISWM_SKIP_CONV_WGRAD)) return 0;
  ISWM_REQUIRE(d && d_in && d_dy && d_dw, "conv_wgrad: null argument");
  ISWM_REQUIRE(d->ntaps >= 1 && d->ntaps <= ISWM_MAX_TAPS, "conv_wgrad: ntaps=%d", d->ntaps);
  ISWM_REQUIRE((d->in_ld % 8) == 0 && (d->out_ld % 8) == 0, "conv_wgrad: row pitches must be multiples of 8 (in_ld=%d out_ld=%d)", d->in_ld, d->out_ld);
  ISWM_REQUIRE((reinterpret_cast<uintptr_t>(d_in) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_dy) & 15) == 0, "conv_wgrad: operands must be 16-byte aligned");
  int* abort_flag = abort_flag_ptr();
  ISWM_REQUIRE(abort_flag, "conv_wgrad: cannot allocate abort flag");

  WgradKParams p;
  memset(&p, 0, sizeof(p));
  int B = d->B, Hi = d->Hi, Wi = d->Wi, Ho = d->Ho, Wo = d->Wo, n_img = d->n_img;
  const bool phase_view = d->in_phase_view != 0;
  ISWM_REQUIRE(!phase_view || ((d->Cin % 64) == 0 && n_img == B), "conv_wgrad: in_phase_view needs Cin %% 64 == 0 and n_img == B");
  bool pointwise = (d->ntaps == 1 && d->dh[0] == 0 && d->dw[0] == 0 && d->phase[0] == 0 &&
                    Hi == Ho && Wi == Wo && n_img == B && !phase_view);
  if (pointwise) {
    const int64_t M = (int64_t)B * Ho * Wo;
    if (M < (1ll << 31)) {
      Wo = Wi = (int)M;
      Ho = Hi = 1;
      B = n_img = 1;
    }
  }
  p.Cout = d->Cout; p.Cin = d->Cin; p.ntaps = d->ntaps;
  p.lgBW = std::min(6, ilog2_ceil_w(Wo));
  p.lgBH = std::min(6 - p.lgBW, ilog2_ceil_w(Ho));
  const int BW = 1 << p.lgBW, BH = 1 << p.lgBH, BB = kPixBlock / (BW * BH);
  p.tiles_w = (Wo + BW - 1) / BW;
  p.tiles_h = (Ho + BH - 1) / BH;
  p.tiles_b = (B + BB - 1) / BB;
  const int64_t pbs = (int64_t)p.tiles_w * p.tiles_h * p.tiles_b;
  ISWM_REQUIRE(pbs < (1ll << 31), "conv_wgrad: too many pixel blocks");
  p.pix_blocks = (int)pbs;
  p.tiles_m = (d->Cout + kWTileM - 1) / kWTileM;
  // the SMs this launch plans for: all of them, or a share when several small weight gradients are launched next to each other
  // on different streams (every split adds a whole partial-tile reduction: a small GEMM spread over 148 SMs is mostly that)
  const int sms = (max_ctas > 0) ? std::max(1, std::min(num_sms(), max_ctas)) : num_sms();
  p.cchunks = (d->Cin + 63) / 64;
  p.T = d->ntaps * p.cchunks;
  p.tail_cols = (d->Cin % 64) ? (((d->Cin % 64) + 15) / 16) * 16 : 64;
  {
    // chunks per tile, by a small cost model fitted to the sweep recorded in DESIGN.md: a CTA streams its share of the pixel blocks at
    // max(MMA time, operand bytes at ~100 B/clk of L2 -> SM ingest) per block, then adds its partial tile into dW with
    // red.global (~2 TB/s device-wide, and EVERY split flushes the whole tile): wide tiles re-read dy less but need more
    // splits to fill the SMs, i.e. more reduction traffic - 1x1 and small 3x3 layers end up at 2 chunks, the decoder at 4-5.
    int G = 1;
    double best = 1e30;
    for (int g = 1; g <= std::min(kMaxG, p.T); g++) {
      const int64_t tiles = (int64_t)p.tiles_m * ((p.T + g - 1) / g);
      double kb, flush_tiles;
      if (tiles <= sms) {
        const int64_t sp = std::max<int64_t>(1, std::min<int64_t>(pbs, sms / tiles));
        kb = (double)((pbs + sp - 1) / sp);
        flush_tiles = (double)(tiles * sp);
      } else {
        kb = (double)((tiles * pbs + sms - 1) / sms);
        flush_tiles = (double)sms * (1.0 + kb / (double)pbs);
      }
      const double mma = 2.0 * 64 * g, load = 82.0 * (2 + g);                     // cycles per 64-pixel block
      const double t_stream = kb * std::max(mma, load) / 1700.0;                  // us at ~1.7 GHz
      const double t_flush = flush_tiles * std::min(128, d->Cout) * 64.0 * g * 4.0 / 2.0e6;
      const double cost = t_stream + t_flush + ((p.T % g) ? 0.03 * t_stream : 0.0);
      if (cost < best) { best = cost; G = g; }
    }
    p.G = G;
  }
  p.tiles_n = (p.T + p.G - 1) / p.G;
  p.acc_cols = 64 * p.G;
  p.nacc = (2 * p.acc_cols <= kWTmemCols) ? 2 : 1;
  const int64_t n_tiles = (int64_t)p.tiles_m * p.tiles_n;
  ISWM_REQUIRE(n_tiles < (1ll << 31), "conv_wgrad: too many output tiles");
  p.n_tiles = (int)n_tiles;
  p.total_kblocks = n_tiles * pbs;
  int grid;
  if (n_tiles <= sms) {
    // split mode, ONE resident wave: as many splits as fit on the SMs next to each other. More CTAs than SMs (the former
    // "best fill of whole waves" rule picked e.g. 37 splits x 8 tiles = 2 waves) doubles the fp32 reduction traffic - every
    // CTA ends by adding its whole 128 x BN partial tile into dW with red.global, ~2 TB/s device-wide - for no gain in
    // parallelism; measured sweep (recorded in DESIGN.md): 1024->256 at 32x32 32.8 -> 22.5 us, 2048->256 55.3 -> 31.6,
    // 1024->2048 86.0 -> 66.6
    const int best = (int)std::max<int64_t>(1, std::min<int64_t>(pbs, sms / n_tiles));
    p.split_len = (int)((pbs + best - 1) / best);
    p.splits = (int)((pbs + p.split_len - 1) / p.split_len);
    grid = (int)(n_tiles * p.splits);
  } else {
    // stream-K: equal k-block ranges per CTA; at least ~4 k-blocks each so a flush is amortised
    grid = (int)std::max<int64_t>(1, std::min<int64_t>(sms, p.total_kblocks / 4));
    p.kblocks_per_cta = (p.total_kblocks + grid - 1) / grid;
    grid = (int)((p.total_kblocks + p.kblocks_per_cta - 1) / p.kblocks_per_cta);
  }
  p.vec_red = ((reinterpret_cast<uintptr_t>(d_dw) & 15) == 0 && (d->Cin % 4) == 0) ? 1 : 0;
  const int stage_bytes = (2 + p.G) * kChunkBytes;
  p.stages = std::max(2, std::min(kWStages, kWSmemBudget / stage_bytes));
  p.n_img_per_phase = B;
  p.nprod = p.stages >= 4 ? 2 : 1;
  for (int t = 0; t < d->ntaps; t++) {
    p.dh[t] = d->dh[t]; p.dw[t] = d->dw[t]; p.phase[t] = d->phase[t];
    ISWM_REQUIRE(d->coff[t] == 0, "conv_wgrad: per-tap channel offsets are a forward / data-gradient feature");
  }
  p.dwgt = d_dw;
  p.abort_flag = abort_flag;

  CUtensorMap tmap_dy, tmap_x;
  {
    const uint64_t dims[4] = {(uint64_t)d->Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)B};
    const uint64_t str[4] = {1, (uint64_t)d->out_ld, (uint64_t)Wo * d->out_ld, (uint64_t)Ho * Wo * d->out_ld};
    const uint32_t box[4] = {64u, (uint32_t)BW, (uint32_t)BH, (uint32_t)BB};
    if (int rc = encode_tmap_bf16(&tmap_dy, d_dy, 4, dims, str, box)) return rc;
  }
  if (phase_view) {
    const uint64_t ld = (uint64_t)d->in_ld, Wf = 2ull * Wi, Hf = 2ull * Hi;
    const uint64_t dims[5] = {ld + (uint64_t)d->Cin, (uint64_t)Wi, 2, (uint64_t)Hi, (uint64_t)B};
    const uint64_t str[5] = {1, 2 * ld, Wf * ld, 2 * Wf * ld, Hf * Wf * ld};
    const uint32_t box[5] = {64u, (uint32_t)BW, 1, (uint32_t)BH, (uint32_t)BB};
    if (int rc = encode_tmap_bf16(&tmap_x, d_in, 5, dims, str, box)) return rc;
    p.phase_view = 1;
    p.pv_ld = d->in_ld;
  } else {
    const uint64_t dims[4] = {(uint64_t)d->Cin, (uint64_t)Wi, (uint64_t)Hi, (uint64_t)n_img};
    const uint64_t str[4] = {1, (uint64_t)d->in_ld, (uint64_t)Wi * d->in_ld, (uint64_t)Hi * Wi * d->in_ld};
    const uint32_t box[4] = {64u, (uint32_t)BW, (uint32_t)BH, (uint32_t)BB};
    if (int rc = encode_tmap_bf16(&tmap_x, d_in, 4, dims, str, box)) return rc;
  }
  const int smem_bytes = p.stages * stage_bytes + 1024 + 256;
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_wgrad_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    ISWM_REQUIRE(e == cudaSuccess, "conv_wgrad: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set = true;
  }
  launch_k(conv_wgrad_kernel, dim3(grid), dim3(256), smem_bytes, static_cast<cudaStream_t>(stream), tmap_dy, tmap_x, p);
  return check_launch("conv_wgrad");
}

// ---- grouped launch: host side -------------------------------------------------------------------------------------
namespace {

struct GroupPlan {                 // depends on the jobs' SHAPES only: cached, the unit table lives in device memory
  std::vector<long long> sig;
  int4* d_units = nullptr;
  int grid = 0, max_units = 0, G = 1, stages = 2, nprod = 1;
  std::vector<WgradKParams> jp;    // per-job geometry (pointers filled per call)
};

// geometry of one job for the grouped kernel (the part of iswm_conv_wgrad_ex's set-up that does not depend on the launch width)
int group_job_geometry(const iswm_conv_desc* d, WgradKParams& p, int& Wo_, int& Ho_, int& B_, int& Wi_, int& Hi_, int& n_img_) {
  memset(&p, 0, sizeof(p));
  int B = d->B, Hi = d->Hi, Wi = d->Wi, Ho = d->Ho, Wo = d->Wo, n_img = d->n_img;
  const bool phase_view = d->in_phase_view != 0;
  ISWM_REQUIRE(!phase_view || ((d->Cin % 64) == 0 && n_img == B), "conv_wgrad_grouped: in_phase_view needs Cin %% 64 == 0 and n_img == B");
  const bool pointwise = (d->ntaps == 1 && d->dh[0] == 0 && d->dw[0] == 0 && d->phase[0] == 0 && Hi == Ho && Wi == Wo && n_img == B && !phase_view);
  if (pointwise) {
    const int64_t M = (int64_t)B * Ho * Wo;
    if (M < (1ll << 31)) { Wo = Wi = (int)M; Ho = Hi = 1; B = n_img = 1; }
  }
  p.Cout = d->Cout; p.Cin = d->Cin; p.ntaps = d->ntaps;
  p.lgBW = std::min(6, ilog2_ceil_w(Wo));
  p.lgBH = std::min(6 - p.lgBW, ilog2_ceil_w(Ho));
  const int BW = 1 << p.lgBW, BH = 1 << p.lgBH, BB = kPixBlock / (BW * BH);
  p.tiles_w = (Wo + BW - 1) / BW;
  p.tiles_h = (Ho + BH - 1) / BH;
  p.tiles_b = (B + BB - 1) / BB;
  const int64_t pbs = (int64_t)p.tiles_w * p.tiles_h * p.tiles_b;
  ISWM_REQUIRE(pbs < (1ll << 31), "conv_wgrad_grouped: too many pixel blocks");
  p.pix_blocks = (int)pbs;
  p.tiles_m = (d->Cout + kWTileM - 1) / kWTileM;
  p.cchunks = (d->Cin + 63) / 64;
  p.T = d->ntaps * p.cchunks;
  p.tail_cols = (d->Cin % 64) ? (((d->Cin % 64) + 15) / 16) * 16 : 64;
  // widest tile of <= 4 chunks that divides the chunk axis evenly (4 chunks otherwise): few splits are needed here, so the
  // reduction traffic that favours narrow tiles in a lone launch does not apply
  int G = std::min(4, p.T);
  for (int g = std::min(4, p.T); g >= 2; g--)
    if (p.T % g == 0) { G = g; break; }
  p.G = G;
  p.tiles_n = (p.T + G - 1) / G;
  p.acc_cols = 64 * G;
  p.nacc = 2;
  const int64_t n_tiles = (int64_t)p.tiles_m * p.tiles_n;
  ISWM_REQUIRE(n_tiles < (1ll << 24), "conv_wgrad_grouped: too many output tiles");
  p.n_tiles = (int)n_tiles;
  p.n_img_per_phase = B;
  for (int t = 0; t < d->ntaps; t++) {
    p.dh[t] = d->dh[t]; p.dw[t] = d->dw[t]; p.phase[t] = d->phase[t];
    ISWM_REQUIRE(d->coff[t] == 0, "conv_wgrad_grouped: per-tap channel offsets are a forward / data-gradient feature");
  }
  if (phase_view) { p.phase_view = 1; p.pv_ld = d->in_ld; }
  Wo_ = Wo; Ho_ = Ho; B_ = B; Wi_ = Wi; Hi_ = Hi; n_img_ = n_img;
  return 0;
}

std::vector<GroupPlan>& plan_cache() {
  static std::vector<GroupPlan> c;
  return c;
}

}  // namespace

extern "C" int iswm_conv_wgrad_grouped(const iswm_conv_desc* descs, const void* const* d_in, const void* const* d_dy,
                                       float* const* d_dw, int n_jobs, void* stream) {
  if (debug_skip(ISWM_SKIP_CONV_WGRAD)) return 0;
  ISWM_REQUIRE(descs && d_in && d_dy && d_dw && n_jobs >= 1, "conv_wgrad_grouped: null / empty");
  int* abort_flag = abort_flag_ptr();
  ISWM_REQUIRE(abort_flag, "conv_wgrad_grouped: cannot allocate abort flag");
  static bool attr_set = false;
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(conv_wgrad_grouped_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    ISWM_REQUIRE(e == cudaSuccess, "conv_wgrad_grouped: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    attr_set = true;
  }
  for (int j0 = 0; j0 < n_jobs; j0 += kMaxJobs) {
    const int nj = std::min(kMaxJobs, n_jobs - j0);
    // ---- plan (cached on the shapes)
    std::vector<long long> sig;
    for (int j = 0; j < nj; j++) {
      const iswm_conv_desc& d = descs[j0 + j];
      ISWM_REQUIRE(d.ntaps >= 1 && d.ntaps <= ISWM_MAX_TAPS && (d.in_ld % 8) == 0 && (d.out_ld % 8) == 0, "conv_wgrad_grouped: job %d: bad descriptor", j0 + j);
      const long long f[] = {d.B, d.Hi, d.Wi, d.Cin, d.in_ld, d.n_img, d.Ho, d.Wo, d.Cout, d.out_ld, d.ntaps, d.in_phase_view};
      sig.insert(sig.end(), f, f + 12);
      for (int t = 0; t < d.ntaps; t++) sig.push_back(((long long)(uint8_t)d.dh[t] << 16) | ((long long)(uint8_t)d.dw[t] << 8) | (uint8_t)d.phase[t]);
    }
    GroupPlan* plan = nullptr;
    for (auto& c : plan_cache())
      if (c.sig == sig) { plan = &c; break; }
    std::vector<std::array<int, 6>> geo(nj);             // Wo, Ho, B, Wi, Hi, n_img as the kernel sees them (1x1 layers flattened)
    if (!plan) {
      GroupPlan np;
      np.sig = sig;
      np.jp.resize(nj);
      const int sms = num_sms();
      struct Unit { int job, tile, pb0, pb1; double cost; };
      std::vector<Unit> units;
      double total = 0.0;
      std::vector<double> kcost(nj);
      for (int j = 0; j < nj; j++) {
        int a, b, c, e, f2, g2;
        if (int rc = group_job_geometry(&descs[j0 + j], np.jp[j], a, b, c, e, f2, g2)) return rc;
        const WgradKParams& p = np.jp[j];
        kcost[j] = std::max(2.0 * 64 * p.G, 82.0 * (2 + p.G)) + 40.0;          // cycles per pixel block (+ issue overhead)
        total += kcost[j] * p.pix_blocks * p.n_tiles + 3000.0 * p.n_tiles;
        np.G = std::max(np.G, p.G);
      }
      const double target = total / sms;
      for (int j = 0; j < nj; j++) {
        const WgradKParams& p = np.jp[j];
        const double t_tile = kcost[j] * p.pix_blocks;
        int sp = (int)std::ceil(t_tile / std::max(1.0, 0.5 * target));
        sp = std::max(1, std::min(sp, std::max(1, p.pix_blocks / 8)));
        const int len = (p.pix_blocks + sp - 1) / sp;
        for (int t = 0; t < p.n_tiles; t++)
          for (int pb = 0; pb < p.pix_blocks; pb += len)
            units.push_back({j, t, pb, std::min(p.pix_blocks, pb + len), kcost[j] * (std::min(p.pix_blocks, pb + len) - pb) + 3000.0});
      }
      // longest unit first onto the least loaded CTA
      std::stable_sort(units.begin(), units.end(), [](const Unit& x, const Unit& y) { return x.cost > y.cost; });
      np.grid = (int)std::min<size_t>(sms, units.size());
      std::vector<std::vector<Unit>> per(np.grid);
      std::vector<double> load(np.grid, 0.0);
      for (const Unit& u : units) {
        int best = 0;
        for (int c = 1; c < np.grid; c++)
          if (load[c] < load[best]) best = c;
        per[best].push_back(u);
        load[best] += u.cost;
      }
      np.max_units = 0;
      for (auto& v : per) np.max_units = std::max<int>(np.max_units, (int)v.size() + 1);
      std::vector<int4> table((size_t)np.grid * np.max_units, make_int4(-1, 0, 0, 0));
      for (int c = 0; c < np.grid; c++) {
        // same job / tile next to each other: the operands of neighbouring units stay in L2
        std::stable_sort(per[c].begin(), per[c].end(), [](const Unit& x, const Unit& y) { return x.job != y.job ? x.job < y.job : (x.tile != y.tile ? x.tile < y.tile : x.pb0 < y.pb0); });
        for (size_t i = 0; i < per[c].size(); i++) table[(size_t)c * np.max_units + i] = make_int4(per[c][i].job, per[c][i].tile, per[c][i].pb0, per[c][i].pb1);
      }
      const int stage_bytes = (2 + np.G) * kChunkBytes;
      np.stages = std::max(2, std::min(kWStages, kWSmemBudget / stage_bytes));
      np.nprod = np.stages >= 4 ? 2 : 1;
      cudaError_t e = cudaMalloc(&np.d_units, table.size() * sizeof(int4));
      ISWM_REQUIRE(e == cudaSuccess, "conv_wgrad_grouped: cudaMalloc of the unit table: %s (the first call of a shape set must not happen inside a stream capture)", cudaGetErrorString(e));
      e = cudaMemcpy(np.d_units, table.data(), table.size() * sizeof(int4), cudaMemcpyHostToDevice);
      ISWM_REQUIRE(e == cudaSuccess, "conv_wgrad_grouped: unit table upload: %s", cudaGetErrorString(e));
      plan_cache().push_back(std::move(np));
      plan = &plan_cache().back();
    }
    // ---- parameters of this call: pointers and tensor maps
    static thread_local WGroupParams P;                    // 12 KB: not on the stack
    memset(&P, 0, sizeof(int) * 8);
    P.n_jobs = nj; P.max_units = plan->max_units; P.stages = plan->stages; P.G = plan->G; P.nprod = plan->nprod;
    P.units = plan->d_units;
    P.abort_flag = abort_flag;
    for (int j = 0; j < nj; j++) {
      const iswm_conv_desc* d = &descs[j0 + j];
      ISWM_REQUIRE(d_in[j0 + j] && d_dy[j0 + j] && d_dw[j0 + j], "conv_wgrad_grouped: job %d: null pointer", j0 + j);
      ISWM_REQUIRE((reinterpret_cast<uintptr_t>(d_in[j0 + j]) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_dy[j0 + j]) & 15) == 0, "conv_wgrad_grouped: operands must be 16-byte aligned");
      WJob& J = P.jobs[j];
      J.p = plan->jp[j];
      J.p.dwgt = d_dw[j0 + j];
      J.p.abort_flag = abort_flag;
      J.p.vec_red = ((reinterpret_cast<uintptr_t>(d_dw[j0 + j]) & 15) == 0 && (d->Cin % 4) == 0) ? 1 : 0;
      // geometry as the kernel sees it (1x1 layers are flattened to one row of B*H*W pixels)
      int B = d->B, Hi = d->Hi, Wi = d->Wi, Ho = d->Ho, Wo = d->Wo, n_img = d->n_img;
      const bool phase_view = d->in_phase_view != 0;
      const bool pointwise = (d->ntaps == 1 && d->dh[0] == 0 && d->dw[0] == 0 && d->phase[0] == 0 && Hi == Ho && Wi == Wo && n_img == B && !phase_view);
      if (pointwise && (int64_t)B * Ho * Wo < (1ll << 31)) { Wo = Wi = B * Ho * Wo; Ho = Hi = 1; B = n_img = 1; }
      const int BW = 1 << J.p.lgBW, BH = 1 << J.p.lgBH, BB = kPixBlock / (BW * BH);
      {
        const uint64_t dims[4] = {(uint64_t)d->Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)B};
        const uint64_t str[4] = {1, (uint64_t)d->out_ld, (uint64_t)Wo * d->out_ld, (uint64_t)Ho * Wo * d->out_ld};
        const uint32_t box[4] = {64u, (uint32_t)BW, (uint32_t)BH, (uint32_t)BB};
        if (int rc = encode_tmap_bf16(&J.tmap_dy, d_dy[j0 + j], 4, dims, str, box)) return rc;
      }
      if (phase_view) {
        const uint64_t ld = (uint64_t)d->in_ld, Wf = 2ull * Wi, Hf = 2ull * Hi;
        const uint64_t dims[5] = {ld + (uint64_t)d->Cin, (uint64_t)Wi, 2, (uint64_t)Hi, (uint64_t)B};
        const uint64_t str[5] = {1, 2 * ld, Wf * ld, 2 * Wf * ld, Hf * Wf * ld};
        const uint32_t box[5] = {64u, (uint32_t)BW, 1, (uint32_t)BH, (uint32_t)BB};
        if (int rc = encode_tmap_bf16(&J.tmap_x, d_in[j0 + j], 5, dims, str, box)) return rc;
      } else {
        const uint64_t dims[4] = {(uint64_t)d->Cin, (uint64_t)Wi, (uint64_t)Hi, (uint64_t)n_img};
        const uint64_t str[4] = {1, (uint64_t)d->in_ld, (uint64_t)Wi * d->in_ld, (uint64_t)Hi * Wi * d->in_ld};
        const uint32_t box[4] = {64u, (uint32_t)BW, (uint32_t)BH, (uint32_t)BB};
        if (int rc = encode_tmap_bf16(&J.tmap_x, d_in[j0 + j], 4, dims, str, box)) return rc;
      }
    }
    const int smem_bytes = plan->stages * (2 + plan->G) * kChunkBytes + 1024 + 256;
    launch_k(conv_wgrad_grouped_kernel, dim3(plan->grid), dim3(256), smem_bytes, static_cast<cudaStream_t>(stream), P);
    if (int rc = check_launch("conv_wgrad_grouped")) return rc;
  }
  return 0;
}
