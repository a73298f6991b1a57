// conv_igemm.cu — convolution as an implicit GEMM on the 5th-gen tensor cores.
//
//   D[pixel, cout] = sum_tap sum_cin  A_tap[pixel, cin] * W[cout, tap, cin]
//
// One persistent CTA per SM, warp-specialised:
//   warp 0   TMA producer: per (tap, 64-channel slice) one 4-D box load of the NHWC
//            activations shifted by the tap offset (out-of-image elements arrive as
//            zeros = the convolution padding, so no im2col buffer exists anywhere)
//            plus one 2-D box of the packed weights, into a multi-stage smem ring;
//   warp 1   one thread issues tcgen05.mma (128 x BN x 16, bf16 -> fp32) into a
//            double-buffered TMEM accumulator and commits stage/accumulator barriers;
//   warp 2   TMEM allocator;
//   warps 4-11 epilogue, two warpgroups that take alternate 64-channel chunks of the
//            accumulator: one tcgen05.ld of 64 columns per thread (= one output pixel), then
//            any of: per-channel affine (folded eval BatchNorm / bias), residual add (the
//            thread's 128 contiguous bytes, loaded under the TMEM read), ReLU; bf16 results are
//            staged in 128B-swizzled smem and written with TMA tensor stores (coalesced, edge
//            clipping by the hardware). Training BatchNorm statistics (per-channel sum and
//            sum of squares of the bf16 values BatchNorm will read back) are column sums of the
//            staged tile, kept in registers across the CTA's tiles and flushed with one fp32
//            atomic per channel per CTA. fp32 / unaligned outputs use direct stores.
//
// Forward convs of network/backbone/resnet.py:27-35 (conv3x3 / conv1x1, all dilations)
// and network/_deeplab.py:37-51,124,134,149,162; their data gradients run through the
// same kernel with transposed packed weights and negated tap offsets.
//
// conv_igemm_f8_kernel is the same body over e4m3 operands (tcgen05.mma kind::f8f6f4, E4M3 x E4M3 -> fp32) for the
// post-training-quantised inference path (iswm_b200/quant.py): a k-block is still one 128-byte swizzle row, now 128
// channels, and each of its four MMAs still advances the operand descriptors by 32 bytes (K = 32 instead of 16). Its
// epilogue reads an e4m3 residual scaled by a per-call factor and writes e4m3 / bf16 / fp32 with direct stores.
#include "tc_common.cuh"
#include <algorithm>
#include <cuda_fp8.h>

namespace iswm {

constexpr int kMaxStages = 8;
constexpr int kTileM = 128;
constexpr int kKBlock = 64;                 // bf16 elements per k-block = one 128-byte swizzle row
constexpr int kABytes = kTileM * 128;       // 16 KiB
constexpr int kTmemCols = 512;
constexpr int kSmemMax = 232448;            // 227 KiB dynamic smem per CTA
constexpr int kStageBuf = 128 * 128;        // one 128-row x 64-channel bf16 staging tile

struct ConvKParams {
  int B, Ho, Wo, Cout;
  int lgBW, lgBH;                // log2 of the pixel-tile box (BW*BH*BB == 128)
  int tiles_w, tiles_h, tiles_b, tiles_n, total_tiles;
  int BN, kchunks, cin_pad, ntaps, stages, flags;
  int n_img_per_phase;
  int step, s_nt, s_tw, s_th, s_tb;   // grid size and its mixed-radix digits over (tiles_n, tiles_w, tiles_h, tiles_b): tile decode without divisions
  int nprod;                     // producer warps (1 or 2) taking alternate k-blocks of the CTA's schedule
  int out_ld, res_ld;
  int use_tma_out;               // bf16 output through smem staging + TMA store
  int res_prefetch;              // residual rows prefetched into shared memory one chunk ahead (short-K convolutions)
  int phase_view, pv_ld;         // input read as the four parity phases of a dense tensor through a 5-D tensor map (pv_ld = its pixel pitch)
  int narrow_tail;               // BN is not a multiple of 64: a tile's last chunk is written with plain stores, not the TMA box
  int8_t dh[ISWM_MAX_TAPS], dw[ISWM_MAX_TAPS], phase[ISWM_MAX_TAPS];
  int16_t coff[ISWM_MAX_TAPS];   // per-tap channel offset into the input buffer (K-concatenated convolutions)
  int8_t wtap[ISWM_MAX_TAPS];    // weight tap each tap reads (a subset of a packed tensor's taps)
  long long o_ws, o_hs, o_bs;    // output element strides along w / h / image (dense or a strided view)
  long long r_ws, r_hs, r_bs;    // residual, same geometry
  void* out;
  const float* scale;
  const float* shift;
  const __nv_bfloat16* res;
  const uint8_t* mask;           // ISWM_EPI_RES_MASK: ReLU sign bits [pixels][Cout/8] gating the residual (dz = dout . mask)
  double* stats;                 // fp64 accumulators: cross-CTA summation order no longer shows up in fp32 results
  int stats_rep;                 // copies of the accumulator vector; this CTA adds into copy blockIdx.x % stats_rep
  int* abort_flag;
  float res_scale;               // e4m3 kernel: the residual is added as res_scale * residual
  int out_f8;                    // e4m3 kernel: write e4m3 (satfinite) instead of bf16 / fp32
};

// four fp32 values -> four e4m3 bytes (round to nearest even, saturating to +-448), first value in the lowest byte
__device__ __forceinline__ uint32_t pack_e4m3x4(float a, float b, float c, float d) {
  const uint32_t lo = __nv_cvt_float2_to_fp8x2(make_float2(a, b), __NV_SATFINITE, __NV_E4M3);
  const uint32_t hi = __nv_cvt_float2_to_fp8x2(make_float2(c, d), __NV_SATFINITE, __NV_E4M3);
  return lo | (hi << 16);
}
__device__ __forceinline__ void unpack_e4m3x2(uint32_t v, float& lo, float& hi) {
  const __half2_raw h = __nv_cvt_fp8x2_to_halfraw2((__nv_fp8x2_storage_t)(v & 0xffffu), __NV_E4M3);
  const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&h));
  lo = f.x;
  hi = f.y;
}

// A CTA's tile schedule (tile = blockIdx.x, += gridDim.x ...) decoded into (n tile, w / h / image tile) coordinates. The decode
// of the first tile uses integer divisions once; every later tile adds the precomputed mixed-radix digits of the grid size with
// carries (each digit < its radix, so one conditional subtraction per digit) - the per-tile divisions used to cost each of
// the three roles ~100 issue slots per tile, which showed on the short-K convolutions (1-9 k-blocks per tile).
struct TileIter {
  int tile, nt, tw, th, tb;
  __device__ __forceinline__ void init(const ConvKParams& p, int t0) {
    tile = t0;
    const int mt = t0 / p.tiles_n;
    nt = t0 - mt * p.tiles_n;
    tw = mt % p.tiles_w;
    const int r = mt / p.tiles_w;
    th = r % p.tiles_h;
    tb = r / p.tiles_h;
  }
  __device__ __forceinline__ void next(const ConvKParams& p) {
    tile += p.step;
    nt += p.s_nt;
    int c = nt >= p.tiles_n ? 1 : 0;
    nt -= c ? p.tiles_n : 0;
    tw += p.s_tw + c;
    c = tw >= p.tiles_w ? 1 : 0;
    tw -= c ? p.tiles_w : 0;
    th += p.s_th + c;
    c = th >= p.tiles_h ? 1 : 0;
    th -= c ? p.tiles_h : 0;
    tb += p.s_tb + c;
  }
};

// Epilogue warpgroups: two (384 threads, up to 168 registers each). A third one for short-K (epilogue-bound) convolutions
// was measured and lost (cfg2 16.05 vs 15.64 ms/step, cfg4 27.1 vs 26.5): it costs a ring stage and 40 registers per
// thread, and the epilogue is paced by TMEM-read and barrier latency rather than by warp count (DESIGN.md).
constexpr int kEpiWG = 2;
constexpr int kConvThreads = 128 * (kEpiWG + 1);

// F8 = false: bf16 operands, 64 channels per k-block; true: e4m3 operands, 128 channels per k-block (no statistics,
// residual mask, strided output or TMA store: the host rejects or disables them)
template <bool F8>
__device__ __forceinline__ void conv_igemm_body(const CUtensorMap& tmap_a, const CUtensorMap& tmap_b,
                                                const CUtensorMap& tmap_out, const ConvKParams& p) {
  constexpr int KB = F8 ? 128 : kKBlock;      // elements per k-block
  extern __shared__ uint8_t smem_raw[];
#ifdef ISWM_EPI_TIMING
  unsigned long long gt_entry, gt_prol = 0, gt_dep = 0;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt_entry));
#endif
  const uint32_t raw_addr = tc::smem_u32(smem_raw);
  const uint32_t ring = (raw_addr + 1023u) & ~1023u;     // swizzle-128B tiles need 1 KiB alignment
  uint8_t* smem = smem_raw + (ring - raw_addr);
  const uint32_t b_bytes = (uint32_t)p.BN * 128u;
  const uint32_t stage_bytes = kABytes + b_bytes;
  // [ring stages][out staging: one 16K tile per epilogue warpgroup, if TMA out][residual prefetch: same][barriers][scale, shift]
  const bool tma_out = !F8 && p.use_tma_out != 0;
  uint32_t off = (uint32_t)p.stages * stage_bytes;
  const uint32_t obuf = ring + off;
  if (tma_out) off += kEpiWG * kStageBuf;
  const uint32_t rbuf = ring + off;                        // residual prefetch tile, one per epilogue warpgroup
  if (!F8 && p.res_prefetch) off += kEpiWG * kStageBuf;
  uint8_t* tail = smem + off;
  uint64_t* bars = reinterpret_cast<uint64_t*>(tail);      // full[8] empty[8] tfull[2] tempty[2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kMaxStages + 6);
  float* s_scale = reinterpret_cast<float*>(tail + 256);
  float* s_shift = s_scale + 256;

  const uint32_t bar_full = tc::smem_u32(bars);
  const uint32_t bar_empty = bar_full + 8 * kMaxStages;
  const uint32_t bar_tfull = bar_empty + 8 * kMaxStages;
  const uint32_t bar_tempty = bar_tfull + 16;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  if (warp == 0 && lane == 0) {
    tc::tma_prefetch_desc(&tmap_a);
    tc::tma_prefetch_desc(&tmap_b);
    if (tma_out) tc::tma_prefetch_desc(&tmap_out);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < p.stages; s++) {
      tc::mbar_init(bar_full + 8 * s, 1);
      tc::mbar_init(bar_empty + 8 * s, 1);
    }
    for (int s = 0; s < 2; s++) {
      tc::mbar_init(bar_tfull + 8 * s, 1);
      tc::mbar_init(bar_tempty + 8 * s, 4 * kEpiWG);   // one arrival per epilogue warp
    }
    tc::fence_barrier_init();
  }
  if (warp == 2) {
    tc::tmem_alloc(tc::smem_u32(tmem_slot), kTmemCols);
    tc::tmem_relinquish();
  }
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
#ifdef ISWM_EPI_TIMING
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt_prol));
#endif
  // prologue done (barriers, TMEM, descriptor prefetch touch no global data): wait for the producer grid, then let
  // the next kernel of the stream start its own prologue under our main loop
  pdl_wait();
  pdl_launch();
#ifdef ISWM_EPI_TIMING
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt_dep));
#endif

  const int kblocks = p.ntaps * p.kchunks;
  const int BW = 1 << p.lgBW, BH = 1 << p.lgBH;
  const int BB = kTileM >> (p.lgBW + p.lgBH);

  // Producer and MMA roles: ONE elected thread runs the whole schedule (elect.sync: the compiler sees a single active
  // thread, so TMA / MMA operands move to uniform registers with plain R2UR - no waterfall loop, and no per-iteration
  // vote / shuffle / reconvergence as in the earlier all-lanes-walk-elect-to-issue form, whose ~80-instruction serial loop
  // body cost ~700-900 cycles per k-block: 5x the MMA time of a 128x64x64 block, ncu profiles/r2a). Two producer warps
  // (0 and 3) take alternate k-blocks of the CTA's linear (tile, tap, channel slice) schedule, which halves the issue
  // latency per k-block again for the short-K convolutions.
  if (warp == 0 || (warp == 3 && p.nprod == 2)) {
    // ===================== TMA producers =====================
    if (tc::elect_one()) {
      const int me = (warp == 0) ? 0 : 1;
      const int np = p.nprod;
      int g = 0;                                  // global k-block counter at the start of the current tile
      int stage = me % p.stages;
      uint32_t phase = (uint32_t)((me / p.stages) & 1);
      bool ok = true;
#ifdef ISWM_EPI_TIMING
      long long pw = 0, pt0 = clock64();
      int pn = 0;
#endif
      TileIter ti;
      ti.init(p, blockIdx.x);
      for (; ti.tile < p.total_tiles && ok; ti.next(p)) {
        const int w0 = ti.tw * BW, h0 = ti.th * BH, b0 = ti.tb * BB, n0 = ti.nt * p.BN;
        // first k-block of this tile that is mine: (g + kb) % np == me
        int kb = me - (g % np);
        if (kb < 0) kb += np;
        int t = kb / p.kchunks, kc = kb - t * p.kchunks;
        for (; kb < kblocks; kb += np) {
#ifdef ISWM_EPI_TIMING
          const long long w0c = clock64();
#endif
          ok = tc::mbar_wait(bar_empty + 8 * stage, phase ^ 1, p.abort_flag, 1);
          if (!ok) break;
#ifdef ISWM_EPI_TIMING
          pw += clock64() - w0c; pn++;
#endif
          const int cw = w0 + p.dw[t], ch = h0 + p.dh[t], cb = p.phase[t] * p.n_img_per_phase + b0;
          const uint32_t a_dst = ring + stage * stage_bytes;
          tc::mbar_expect_tx(bar_full + 8 * stage, stage_bytes);
          if (p.phase_view)
            tc::tma_load_5d(a_dst, &tmap_a, bar_full + 8 * stage, (p.phase[t] & 1) * p.pv_ld + p.coff[t] + kc * KB, cw, p.phase[t] >> 1, ch, b0);
          else
            tc::tma_load_4d(a_dst, &tmap_a, bar_full + 8 * stage, p.coff[t] + kc * KB, cw, ch, cb);
          tc::tma_load_2d(a_dst + kABytes, &tmap_b, bar_full + 8 * stage, p.wtap[t] * p.cin_pad + kc * KB, n0);
          stage += np;
          if (stage >= p.stages) { stage -= p.stages; phase ^= 1; }
          kc += np;
          while (kc >= p.kchunks) { kc -= p.kchunks; t++; }
        }
        g += kblocks;
      }
#ifdef ISWM_EPI_TIMING
      if (blockIdx.x == 0) printf("producer %d: total %lld  waiting for a free stage %lld  k-blocks issued %d (stages %d, kblocks/tile %d, nprod %d)\n", me, clock64() - pt0, pw, pn, p.stages, kblocks, np);
#endif
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    if (tc::elect_one()) {
      const uint32_t idesc = F8 ? tc::make_idesc_e4m3(kTileM, p.BN) : tc::make_idesc_bf16(kTileM, p.BN, 0, 0);
      int stage = 0, as = 0;
      uint32_t phase = 0, aphase = 0;
      bool ok = true;
#ifdef ISWM_EPI_TIMING
      long long mw_acc = 0, mw_full = 0, mt0 = clock64(), c0;
      int ntl = 0;
#endif
      for (int tile = blockIdx.x; tile < p.total_tiles && ok; tile += p.step) {
#ifdef ISWM_EPI_TIMING
        c0 = clock64(); ntl++;
#endif
        ok = tc::mbar_wait(bar_tempty + 8 * as, aphase ^ 1, p.abort_flag, 2);
        if (!ok) break;
        tc::tc_fence_after();
#ifdef ISWM_EPI_TIMING
        mw_acc += clock64() - c0;
#endif
        const uint32_t d_tmem = tmem_base + (uint32_t)(as * p.BN);
        for (int kb = 0; kb < kblocks; kb++) {
#ifdef ISWM_EPI_TIMING
          c0 = clock64();
#endif
          ok = tc::mbar_wait(bar_full + 8 * stage, phase, p.abort_flag, 3);
          if (!ok) break;
          tc::tc_fence_after();
#ifdef ISWM_EPI_TIMING
          mw_full += clock64() - c0;
#endif
          const uint32_t a_addr = ring + stage * stage_bytes;
          const uint64_t da = tc::make_smem_desc_sw128(a_addr, 16, 1024);
          const uint64_t db = tc::make_smem_desc_sw128(a_addr + kABytes, 16, 1024);
#pragma unroll
          for (int k = 0; k < 4; k++) {                // 32 bytes of K per MMA: 16 bf16 or 32 e4m3 channels
            if constexpr (F8) tc::umma_f8(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
            else tc::umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
          }
          tc::umma_commit(bar_empty + 8 * stage);     // frees this smem stage when the MMAs retire
          if (++stage == p.stages) { stage = 0; phase ^= 1; }
        }
        if (!ok) break;
        tc::umma_commit(bar_tfull + 8 * as);          // accumulator complete -> epilogue
        as ^= 1;
        if (as == 0) aphase ^= 1;
      }
#ifdef ISWM_EPI_TIMING
      if (blockIdx.x == 0) printf("mma: total %lld  waiting for operands %lld  waiting for a free accumulator %lld  (tiles %d)\n", clock64() - mt0, mw_full, mw_acc, ntl);
#endif
    }
    __syncwarp();
  } else if (warp >= 4) {
    // ===================== epilogue: two warpgroups, 64-channel chunks alternate between them =====================
    const int nchunk64 = (p.BN + 63) >> 6;
    const int wg = (warp - 4) >> 2;                     // warpgroup 0 or 1
    constexpr int NSLOT = 2;                            // statistics slots per thread (chunk positions it can own)
    // which warpgroup owns 64-channel chunk c of this CTA's it-th tile: the two warpgroups take alternate chunks
    // (alternate tiles when a tile is a single chunk)
    auto owner_of = [&](int it_, int c_) -> int { return ((nchunk64 == 1) ? it_ : c_) & 1; };
    const int q = warp & 3;                             // TMEM lane quadrant of this warp (warp % 4)
    const int row = q * 32 + lane;                      // accumulator row = thread index inside the warpgroup
    const int bb = row >> (p.lgBW + p.lgBH);
    const int hh = (row >> p.lgBW) & (BH - 1);
    const int ww = row & (BW - 1);
    const bool f_aff = p.flags & ISWM_EPI_AFFINE, f_relu = p.flags & ISWM_EPI_RELU, f_res = p.flags & ISWM_EPI_RESIDUAL,
               f_stats = !F8 && (p.flags & ISWM_EPI_STATS), f_mask = !F8 && (p.flags & ISWM_EPI_RES_MASK), f_f32 = p.flags & ISWM_EPI_OUT_F32;
    // Each epilogue WARP is independent between channel-tile changes: it stages its own 32 rows (a 4 KiB, 1 KiB-aligned
    // slice of the warpgroup's staging tile), issues its own TMA store (a 32-pixel sub-box of the tile) and sums its own
    // rows for the statistics - __syncwarp() instead of three 128-thread named barriers per chunk, so the eight warps
    // drift apart and hide each other's TMEM-load / shared-memory latencies (the epilogue bounds every short-K convolution).
    const bool issuer = (lane == 0);                    // issues this warp's TMA stores
    const int srow = q * 32;                            // first tile row of this warp: its sub-box origin inside the tile
    const int sub_b = srow >> (p.lgBW + p.lgBH), sub_h = (srow >> p.lgBW) & (BH - 1), sub_w = srow & (BW - 1);
    const uint32_t ob = obuf + (uint32_t)wg * kStageBuf; // this warpgroup's 128 x 64 bf16 staging tile
    const uint32_t row_off = (uint32_t)row * 128u;
    const uint32_t sw = (uint32_t)(row & 7);            // 128B swizzle: 16-byte chunk index ^= row % 8
    const int bar_wg = 4 + wg;                          // named barrier of this warpgroup (3 = all epilogue warps)
    // BatchNorm statistics: thread (q, lane) owns channel pair `lane` of rows [32q, 32q+32) of each staged
    // chunk; partial sums stay in registers across this CTA's tiles while the channel tile is unchanged.
    float st[NSLOT][4];
#pragma unroll
    for (int i = 0; i < NSLOT; i++)
#pragma unroll
      for (int j = 0; j < 4; j++) st[i][j] = 0.f;
    // flush: the four quadrant warps of a warpgroup combine their partial sums through the (idle) staging tile in a
    // fixed order, then ONE fp64 atomic per channel and component leaves the CTA (fp64: the order in which CTAs
    // arrive does not show up in the fp32 mean / variance, so a training step is reproducible bit for bit)
    double* const stats_mine = p.stats + (size_t)(blockIdx.x % (unsigned)p.stats_rep) * (size_t)(2 * p.Cout);
    auto flush_stats = [&](int n0f) {
      if (issuer) tc::tma_store_wait_read<0>();        // every warp's stores have left the staging tile
      asm volatile("bar.sync %0, 128;" ::"r"(bar_wg) : "memory");
#pragma unroll
      for (int slot = 0; slot < NSLOT; slot++)
#pragma unroll
        for (int j = 0; j < 4; j++) {
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(ob + (uint32_t)((((q * NSLOT + slot) * 4 + j) * 32 + lane) * 4)), "f"(st[slot][j]) : "memory");
          st[slot][j] = 0.f;
        }
      asm volatile("bar.sync %0, 128;" ::"r"(bar_wg) : "memory");
      if (q == 0) {
#pragma unroll
        for (int slot = 0; slot < NSLOT; slot++) {
          const int c64 = (nchunk64 == 1) ? 0 : 2 * slot + wg;
          if (c64 >= nchunk64) continue;
          float t[4];
#pragma unroll
          for (int j = 0; j < 4; j++) {
            t[j] = 0.f;
#pragma unroll
            for (int qq = 0; qq < 4; qq++) {
              float v;
              asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(ob + (uint32_t)((((qq * NSLOT + slot) * 4 + j) * 32 + lane) * 4)));
              t[j] += v;
            }
          }
          const int col = n0f + c64 * 64 + 2 * lane;
          if (col < p.Cout) {
            atomicAdd(stats_mine + col, (double)t[0]);
            atomicAdd(stats_mine + p.Cout + col, (double)t[2]);
          }
          if (col + 1 < p.Cout) {
            atomicAdd(stats_mine + col + 1, (double)t[1]);
            atomicAdd(stats_mine + p.Cout + col + 1, (double)t[3]);
          }
        }
      }
      asm volatile("bar.sync %0, 128;" ::"r"(bar_wg) : "memory");   // the staging tile is free for the next chunk
    };
    // Residual operand (eval-mode shortcut add, gradient accumulation): this thread's 128-byte row of the NEXT chunk
    // is prefetched with cp.async into the warpgroup's residual tile while the current chunk is processed; only the
    // issuing thread reads it back, so no barrier is involved.
    const uint32_t rb_row = rbuf + (uint32_t)wg * kStageBuf + row_off;
    const bool res_pf_ok = !F8 && f_res && p.res_prefetch != 0;
    auto chunk_owner_ok = [&](const TileIter& ti_, int it_, int c_) -> bool {
      if (owner_of(it_, c_) != wg) return false;
      return ti_.nt * p.BN + c_ * 64 < p.Cout;
    };
    // advance (ti_, it_, c_) to the next chunk this warpgroup owns; false when the CTA's schedule is exhausted
    auto next_chunk = [&](TileIter& ti_, int& it_, int& c_) -> bool {
      c_++;
      while (ti_.tile < p.total_tiles) {
        for (; c_ < nchunk64; c_++)
          if (chunk_owner_ok(ti_, it_, c_)) return true;
        ti_.next(p); it_++; c_ = 0;
      }
      return false;
    };
    // issue the prefetch of chunk (ti_, c_); returns whether the vector path applies to it for this thread
    auto prefetch_res = [&](const TileIter& ti_, int c_) -> bool {
      const int w_ = ti_.tw * BW + ww, h_ = ti_.th * BH + hh, b_ = ti_.tb * BB + bb;
      const int nc_ = ti_.nt * p.BN + c_ * 64;
      const bool ok_ = (b_ < p.B) && (h_ < p.Ho) && (w_ < p.Wo) && min(p.BN - c_ * 64, p.Cout - nc_) >= 64;
      if (ok_) {
        const __nv_bfloat16* rp = p.res + ((long long)b_ * p.r_bs + (long long)h_ * p.r_hs + (long long)w_ * p.r_ws) + nc_;
#pragma unroll
        for (int j = 0; j < 8; j++)
          asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(rb_row + ((((uint32_t)j) ^ sw) << 4)), "l"(rp + 8 * j) : "memory");
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
      return ok_;
    };
    TileIter pf_ti;
    pf_ti.init(p, blockIdx.x);
    int pf_it = 0, pf_c = -1;
    bool pf_more = false, pf_vec = false;
    if (res_pf_ok) {
      pf_more = next_chunk(pf_ti, pf_it, pf_c);
      if (pf_more) pf_vec = prefetch_res(pf_ti, pf_c);
    }
    int as = 0, it = 0, cur_n0 = -1;
    uint32_t aphase = 0;
#ifdef ISWM_EPI_TIMING
    long long tm[6] = {0, 0, 0, 0, 0, 0};
    long long tprev = clock64();
#define TMARK(i) { const long long tn = clock64(); tm[i] += tn - tprev; tprev = tn; }
#else
#define TMARK(i)
#endif
    TileIter ti;
    ti.init(p, blockIdx.x);
    for (; ti.tile < p.total_tiles; ti.next(p), it++) {
      const int w0 = ti.tw * BW, h0 = ti.th * BH, b0 = ti.tb * BB, n0 = ti.nt * p.BN;
      const int w = w0 + ww, h = h0 + hh, b = b0 + bb;
      const bool valid = (b < p.B) && (h < p.Ho) && (w < p.Wo);
      const long long opix = (long long)b * p.o_bs + (long long)h * p.o_hs + (long long)w * p.o_ws;   // element offsets
      const long long rpix = (long long)b * p.r_bs + (long long)h * p.r_hs + (long long)w * p.r_ws;
      if (n0 != cur_n0) {
        if (f_stats && cur_n0 >= 0) flush_stats(cur_n0);
        if (f_aff) {
          asm volatile("bar.sync 3, %0;" ::"n"(128 * kEpiWG) : "memory");   // every reader of the previous channel tile is done
          for (int i = threadIdx.x - 128; i < p.BN; i += 128 * kEpiWG) {
            const int n = n0 + i;
            s_scale[i] = (n < p.Cout) ? p.scale[n] : 0.f;
            s_shift[i] = (n < p.Cout) ? p.shift[n] : 0.f;
          }
          asm volatile("bar.sync 3, %0;" ::"n"(128 * kEpiWG) : "memory");
        }
        cur_n0 = n0;
      }
      TMARK(0)
      if (!tc::mbar_wait(bar_tfull + 8 * as, aphase, p.abort_flag, 4)) break;
      tc::tc_fence_after();
      TMARK(1)
      const uint32_t t_row = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(as * p.BN);
      for (int c64 = 0; c64 < nchunk64; c64++) {
        if (owner_of(it, c64) != wg) continue;
        const int nc = n0 + c64 * 64;                   // first output channel of this chunk
        if (nc >= p.Cout) continue;
        const int ncols = min(64, min(p.BN - c64 * 64, p.Cout - nc));
        uint32_t v[64];
        tc::tmem_ld64(t_row + c64 * 64, v);
        // residual: this thread's row of the chunk (128 contiguous bytes) was prefetched into shared memory
        uint4 rr[8];
        const bool res_vec = res_pf_ok ? pf_vec : (f_res && valid && ncols == 64 && (p.res_ld & (F8 ? 15 : 7)) == 0);
        if (f_res && !res_pf_ok && res_vec) {             // long-K convolution: direct loads, issued under the TMEM read
          if constexpr (F8) {
            const uint4* rp = reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(p.res) + rpix + nc);
#pragma unroll
            for (int j = 0; j < 4; j++) rr[j] = rp[j];
          } else {
            const uint4* rp = reinterpret_cast<const uint4*>(p.res + rpix + nc);
#pragma unroll
            for (int j = 0; j < 8; j++) rr[j] = rp[j];
          }
        }
        if (res_pf_ok) {                                   // (pf_ti.tile, pf_c) == (ti.tile, c64) by construction
          asm volatile("cp.async.wait_group 0;" ::: "memory");
          if (res_vec) {
#pragma unroll
            for (int j = 0; j < 8; j++)
              asm volatile("ld.shared.v4.u32 {%0,%1,%2,%3}, [%4];" : "=r"(rr[j].x), "=r"(rr[j].y), "=r"(rr[j].z), "=r"(rr[j].w)
                           : "r"(rb_row + ((((uint32_t)j) ^ sw) << 4)));
          }
          pf_more = next_chunk(pf_ti, pf_it, pf_c);        // the row is in registers: refill the tile for the next chunk
          if (pf_more) pf_vec = prefetch_res(pf_ti, pf_c);
        }
        unsigned long long mbits = ~0ull;                 // residual gate: bit j = channel nc + j of this pixel
        if (f_mask && valid && ncols == 64)
          mbits = *reinterpret_cast<const unsigned long long*>(p.mask + (((size_t)b * p.Ho + h) * p.Wo + w) * (size_t)(p.Cout >> 3) + (nc >> 3));
        tc::tmem_ld_wait();
        TMARK(2)
        float f[64];
#pragma unroll
        for (int j = 0; j < 64; j++) f[j] = __uint_as_float(v[j]);
        if (f_aff) {
          const float4* sc4 = reinterpret_cast<const float4*>(s_scale + c64 * 64);
          const float4* sh4 = reinterpret_cast<const float4*>(s_shift + c64 * 64);
#pragma unroll
          for (int j = 0; j < 16; j++) {
            const float4 a = sc4[j], c = sh4[j];
            f[4 * j] = fmaf(f[4 * j], a.x, c.x);
            f[4 * j + 1] = fmaf(f[4 * j + 1], a.y, c.y);
            f[4 * j + 2] = fmaf(f[4 * j + 2], a.z, c.z);
            f[4 * j + 3] = fmaf(f[4 * j + 3], a.w, c.w);
          }
        }
        if (F8 && f_res) {                                 // f += res_scale * residual (e4m3)
          if (res_vec) {
#pragma unroll
            for (int j = 0; j < 4; j++) {
              const uint32_t r4[4] = {rr[j].x, rr[j].y, rr[j].z, rr[j].w};
#pragma unroll
              for (int k = 0; k < 4; k++) {
                float a0, a1, a2, a3;
                unpack_e4m3x2(r4[k], a0, a1);
                unpack_e4m3x2(r4[k] >> 16, a2, a3);
                f[16 * j + 4 * k] = fmaf(a0, p.res_scale, f[16 * j + 4 * k]);
                f[16 * j + 4 * k + 1] = fmaf(a1, p.res_scale, f[16 * j + 4 * k + 1]);
                f[16 * j + 4 * k + 2] = fmaf(a2, p.res_scale, f[16 * j + 4 * k + 2]);
                f[16 * j + 4 * k + 3] = fmaf(a3, p.res_scale, f[16 * j + 4 * k + 3]);
              }
            }
          } else if (valid) {
            const uint8_t* rp = reinterpret_cast<const uint8_t*>(p.res) + rpix + nc;
#pragma unroll
            for (int j = 0; j < 64; j += 2)
              if (j < ncols) {
                float a0, a1;
                unpack_e4m3x2(rp[j] | ((j + 1 < ncols ? (uint32_t)rp[j + 1] : 0u) << 8), a0, a1);
                f[j] = fmaf(a0, p.res_scale, f[j]);
                if (j + 1 < ncols) f[j + 1] = fmaf(a1, p.res_scale, f[j + 1]);
              }
          }
        } else if (f_res) {
          if (res_vec) {
#pragma unroll
            for (int j = 0; j < 8; j++) {
              const uint32_t r4[4] = {rr[j].x, rr[j].y, rr[j].z, rr[j].w};
#pragma unroll
              for (int k = 0; k < 4; k++) {
                float lo, hi;
                unpack_bf16x2(r4[k], lo, hi);
                if (f_mask) {
                  lo = ((mbits >> (8 * j + 2 * k)) & 1ull) ? lo : 0.f;
                  hi = ((mbits >> (8 * j + 2 * k + 1)) & 1ull) ? hi : 0.f;
                }
                f[8 * j + 2 * k] += lo;
                f[8 * j + 2 * k + 1] += hi;
              }
            }
          } else if (valid) {
            const __nv_bfloat16* rp = p.res + rpix + nc;
#pragma unroll
            for (int j = 0; j < 64; j++)
              if (j < ncols && ((mbits >> j) & 1ull)) f[j] += __bfloat162float(rp[j]);
          }
        }
        if (f_relu) {
#pragma unroll
          for (int j = 0; j < 64; j++) f[j] = fmaxf(f[j], 0.f);
        }
        if (tma_out && !(p.narrow_tail && p.BN - c64 * 64 < 64)) {
          uint32_t pk[32];
#pragma unroll
          for (int j = 0; j < 32; j++) pk[j] = pack_bf16x2(f[2 * j], f[2 * j + 1]);
          if (!valid) {                                    // rows outside the image: clipped by the store, zero for the statistics
#pragma unroll
            for (int j = 0; j < 32; j++) pk[j] = 0u;
          }
          // the previous store of this warpgroup has finished reading the staging tile (and so have the
          // statistics readers, who arrive at this barrier after their loop)
          TMARK(0)
          if (issuer) tc::tma_store_wait_read<0>();
          __syncwarp();
          TMARK(3)
#pragma unroll
          for (int j = 0; j < 8; j++)
            asm volatile("st.shared.v4.u32 [%0], {%1,%2,%3,%4};" ::"r"(ob + row_off + ((((uint32_t)j) ^ sw) << 4)),
                         "r"(pk[4 * j]), "r"(pk[4 * j + 1]), "r"(pk[4 * j + 2]), "r"(pk[4 * j + 3]) : "memory");
          tc::fence_proxy_async();                        // staging writes -> visible to the TMA engine
          __syncwarp();
          if (issuer) {
            tc::tma_store_4d(&tmap_out, ob + (uint32_t)srow * 128u, nc, w0 + sub_w, h0 + sub_h, b0 + sub_b);
            tc::tma_store_commit();
          }
          TMARK(4)
          if (f_stats) {
            const int slot = c64 >> 1;
            // plain shared-memory loads (ordered after the barrier above by its memory clobber): 8 rows in flight,
            // then their sums, so the loads are not serialised behind the dependent adds
            const uint8_t* sbase = smem + (ob - ring) + (uint32_t)(q * 32) * 128u + (uint32_t)((lane & 3) << 2);
            const uint32_t ch = (uint32_t)(lane >> 2);
            float s0 = 0.f, s1 = 0.f, q0 = 0.f, q1 = 0.f;
#pragma unroll
            for (int r0 = 0; r0 < 32; r0 += 8) {
              uint32_t wv[8];
#pragma unroll
              for (int r = 0; r < 8; r++)
                wv[r] = *reinterpret_cast<const uint32_t*>(sbase + (uint32_t)(r0 + r) * 128u + ((ch ^ (uint32_t)r) << 4));
#pragma unroll
              for (int r = 0; r < 8; r++) {
                float lo, hi;
                unpack_bf16x2(wv[r], lo, hi);
                s0 += lo; s1 += hi;
                q0 = fmaf(lo, lo, q0); q1 = fmaf(hi, hi, q1);
              }
            }
            // predicated adds on statically indexed registers (a runtime index put the array in local memory)
#pragma unroll
            for (int sl = 0; sl < NSLOT; sl++) {
              const bool mine = (sl == slot);
              st[sl][0] += mine ? s0 : 0.f; st[sl][1] += mine ? s1 : 0.f; st[sl][2] += mine ? q0 : 0.f; st[sl][3] += mine ? q1 : 0.f;
            }
            TMARK(5)
          }
        } else if (valid) {
          if (f_f32) {
            float* op = reinterpret_cast<float*>(p.out) + opix + nc;
            if (ncols == 64 && (p.out_ld & 3) == 0) {
#pragma unroll
              for (int j = 0; j < 16; j++)
                *reinterpret_cast<float4*>(op + 4 * j) = make_float4(f[4 * j], f[4 * j + 1], f[4 * j + 2], f[4 * j + 3]);
            } else {
#pragma unroll
              for (int j = 0; j < 64; j++)
                if (j < ncols) op[j] = f[j];
            }
          } else if (F8 && p.out_f8) {
            uint8_t* op = reinterpret_cast<uint8_t*>(p.out) + opix + nc;
            if ((ncols & 15) == 0 && (p.out_ld & 15) == 0 && (nc & 15) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0) {
              // 16-byte stores; a narrow chunk (the 48-channel slice of the decoder concat) writes its first ncols bytes
#pragma unroll
              for (int j = 0; j < 4; j++)
                if (16 * j < ncols)
                  *reinterpret_cast<uint4*>(op + 16 * j) = make_uint4(pack_e4m3x4(f[16 * j], f[16 * j + 1], f[16 * j + 2], f[16 * j + 3]),
                                                                      pack_e4m3x4(f[16 * j + 4], f[16 * j + 5], f[16 * j + 6], f[16 * j + 7]),
                                                                      pack_e4m3x4(f[16 * j + 8], f[16 * j + 9], f[16 * j + 10], f[16 * j + 11]),
                                                                      pack_e4m3x4(f[16 * j + 12], f[16 * j + 13], f[16 * j + 14], f[16 * j + 15]));
            } else {
#pragma unroll
              for (int j = 0; j < 64; j++)
                if (j < ncols) op[j] = (uint8_t)(pack_e4m3x4(f[j], 0.f, 0.f, 0.f) & 0xffu);
            }
          } else {
            __nv_bfloat16* op = reinterpret_cast<__nv_bfloat16*>(p.out) + opix + nc;
            if ((ncols & 7) == 0 && (p.out_ld & 7) == 0 && (nc & 7) == 0 && (reinterpret_cast<uintptr_t>(p.out) & 15) == 0) {
              // narrow last chunk of a channel tile that is not a multiple of 64 wide (304 = 2 x 160): 16-byte stores
#pragma unroll
              for (int j = 0; j < 8; j++)
                if (8 * j < ncols)
                  *reinterpret_cast<uint4*>(op + 8 * j) = make_uint4(pack_bf16x2(f[8 * j], f[8 * j + 1]), pack_bf16x2(f[8 * j + 2], f[8 * j + 3]),
                                                                     pack_bf16x2(f[8 * j + 4], f[8 * j + 5]), pack_bf16x2(f[8 * j + 6], f[8 * j + 7]));
            } else {
#pragma unroll
              for (int j = 0; j < 64; j++)
                if (j < ncols) op[j] = __float2bfloat16_rn(f[j]);
            }
          }
        }
      }
      tc::tc_fence_before();
      __syncwarp();
      if (lane == 0) tc::mbar_arrive(bar_tempty + 8 * as);   // this warp has drained its part of the accumulator
      as ^= 1;
      if (as == 0) aphase ^= 1;
    }
    if (f_stats && cur_n0 >= 0) flush_stats(cur_n0);
#ifdef ISWM_EPI_TIMING
    // debug build only: [math+other, tfull wait, tmem load, staging free wait, stage+store, stats] cycles of thread 0/32 of each warpgroup
    if (blockIdx.x == 0 && (row == 0 || row == 32)) {
      printf("epi timing wg%d row%d: other %lld  tfull %lld  tmem %lld  stfree %lld  stage %lld  stats %lld  (tiles %d)\n", wg, row,
             tm[0], tm[1], tm[2], tm[3], tm[4], tm[5], it);
    }
#endif
    if (tma_out && issuer) tc::tma_store_wait_all();         // staging smem must outlive the last store
  }

  tc::tc_fence_before();
  __syncthreads();
  if (warp == 2) tc::tmem_dealloc(tmem_base, kTmemCols);
#ifdef ISWM_EPI_TIMING
  if (threadIdx.x == 0) {
    unsigned long long gt_end;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(gt_end));
    printf("CTA %d entry %llu prologue +%llu dep +%llu end +%llu\n", blockIdx.x, gt_entry, gt_prol - gt_entry, gt_dep - gt_entry, gt_end - gt_entry);
  }
#endif
}

__global__ void __launch_bounds__(kConvThreads, 1)
conv_igemm_kernel(const __grid_constant__ CUtensorMap tmap_a,
                  const __grid_constant__ CUtensorMap tmap_b,
                  const __grid_constant__ CUtensorMap tmap_out, const ConvKParams p) {
  conv_igemm_body<false>(tmap_a, tmap_b, tmap_out, p);
}

__global__ void __launch_bounds__(kConvThreads, 1)
conv_igemm_f8_kernel(const __grid_constant__ CUtensorMap tmap_a,
                     const __grid_constant__ CUtensorMap tmap_b,
                     const __grid_constant__ CUtensorMap tmap_out, const ConvKParams p) {
  conv_igemm_body<true>(tmap_a, tmap_b, tmap_out, p);
}

static int ilog2_ceil(int v) {
  int l = 0;
  while ((1 << l) < v) l++;
  return l;
}

}  // namespace iswm

using namespace iswm;

extern "C" int iswm_conv_igemm(const iswm_conv_desc* d, const void* d_in, const void* d_wgt,
                               void* d_out, const float* d_scale, const float* d_shift,
                               const void* d_res, double* d_stats, void* stream) {
  return iswm_conv_igemm_ex(d, d_in, d_wgt, d_out, d_scale, d_shift, d_res, d_stats, nullptr, stream);
}

// f8: e4m3 operands / residual (conv_igemm_f8_kernel), output type out_type (ISWM_E4M3 / ISWM_BF16 / ISWM_F32)
static int conv_igemm_launch(const iswm_conv_desc* d, const void* d_in, const void* d_wgt, void* d_out, const float* d_scale,
                             const float* d_shift, const void* d_res, double* d_stats, const uint8_t* d_res_mask, bool f8,
                             float res_scale, int out_type, void* stream) {
  const int KB = f8 ? 128 : kKBlock;                       // channels per k-block
  if (f8) {
    ISWM_REQUIRE(d && (d->flags & ~(ISWM_EPI_AFFINE | ISWM_EPI_RELU | ISWM_EPI_RESIDUAL)) == 0,
                 "conv_igemm_f8: only AFFINE, RELU and RESIDUAL (statistics, residual masks and fp32 output flags are training-side)");
    ISWM_REQUIRE(d->out_ws == 0 && d->out_hs == 0 && d->out_bs == 0, "conv_igemm_f8: strided outputs are not supported");
    ISWM_REQUIRE(out_type == ISWM_E4M3 || out_type == ISWM_BF16 || out_type == ISWM_F32, "conv_igemm_f8: out_type %d", out_type);
    ISWM_REQUIRE((d->in_ld % 16) == 0, "conv_igemm_f8: in_ld=%d must be a multiple of 16 (tensor-map row pitch in bytes)", d->in_ld);
  }
  ISWM_REQUIRE(!(d && (d->flags & ISWM_EPI_RES_MASK)) || (d_res_mask && (d->flags & ISWM_EPI_RESIDUAL) && (d->Cout % 64) == 0 &&
                                                          d->out_ws == 0 && d->out_hs == 0 && d->out_bs == 0),
               "conv_igemm: RES_MASK needs RESIDUAL, the bit tensor, Cout %% 64 == 0 and a dense output");
  ISWM_REQUIRE(d && d_in && d_wgt && d_out, "conv_igemm: null argument");
  ISWM_REQUIRE((d->flags & ~63) == 0, "conv_igemm: unknown epilogue flags (flags=%d)", d->flags);
  ISWM_REQUIRE(d->ntaps >= 1 && d->ntaps <= ISWM_MAX_TAPS, "conv_igemm: ntaps=%d", d->ntaps);
  ISWM_REQUIRE(d->Cin >= 1 && d->Cout >= 1 && d->B >= 1 && d->Ho >= 1 && d->Wo >= 1, "conv_igemm: bad dims");
  ISWM_REQUIRE((d->in_ld % 8) == 0 && d->in_ld >= d->Cin, "conv_igemm: in_ld=%d must be a multiple of 8 and >= Cin=%d", d->in_ld, d->Cin);
  ISWM_REQUIRE((reinterpret_cast<uintptr_t>(d_in) & 15) == 0 && (reinterpret_cast<uintptr_t>(d_wgt) & 15) == 0, "conv_igemm: operands must be 16-byte aligned");
  ISWM_REQUIRE(!(d->flags & ISWM_EPI_AFFINE) || (d_scale && d_shift), "conv_igemm: AFFINE needs scale/shift");
  ISWM_REQUIRE(!(d->flags & ISWM_EPI_RESIDUAL) || d_res, "conv_igemm: RESIDUAL needs d_res");
  ISWM_REQUIRE(!(d->flags & ISWM_EPI_STATS) || d_stats, "conv_igemm: STATS needs d_stats");
  int* abort_flag = abort_flag_ptr();
  ISWM_REQUIRE(abort_flag, "conv_igemm: cannot allocate abort flag");

  ConvKParams p;
  memset(&p, 0, sizeof(p));
  int B = d->B, Hi = d->Hi, Wi = d->Wi, Ho = d->Ho, Wo = d->Wo, n_img = d->n_img;
  const bool strided_out = d->out_ws != 0 || d->out_hs != 0 || d->out_bs != 0;
  const bool phase_view = d->in_phase_view != 0;
  ISWM_REQUIRE(!phase_view || ((d->Cin % KB) == 0 && n_img == B), "conv_igemm: in_phase_view needs Cin %% %d == 0 and n_img == B (Cin=%d n_img=%d B=%d)", KB, d->Cin, n_img, B);
  bool pointwise = (d->ntaps == 1 && d->dh[0] == 0 && d->dw[0] == 0 && d->phase[0] == 0 &&
                    Hi == Ho && Wi == Wo && n_img == B && !strided_out && !phase_view);
  if (pointwise) {  // a 1x1 convolution is a plain GEMM over all pixels: no tile-edge waste
    const int64_t M = (int64_t)B * Ho * Wo;
    if (M < (1ll << 31)) {
      Wo = Wi = (int)M;
      Ho = Hi = 1;
      B = n_img = 1;
    }
  }
  p.lgBW = std::min(7, ilog2_ceil(Wo));
  p.lgBH = std::min(7 - p.lgBW, ilog2_ceil(Ho));
  const int BW = 1 << p.lgBW, BH = 1 << p.lgBH, BB = kTileM / (BW * BH);
  p.B = B; p.Ho = Ho; p.Wo = Wo; p.Cout = d->Cout;
  p.tiles_w = (Wo + BW - 1) / BW;
  p.tiles_h = (Ho + BH - 1) / BH;
  p.tiles_b = (B + BB - 1) / BB;
  // N tile: one tile of ceil16(Cout) columns up to 256; above that equal tiles rounded up to the 64-channel store
  // chunk (304 output channels -> 2 x 192 instead of 256 + 48-in-256: a quarter less MMA work)
  int BN;
  if (d->Cout <= 256) {
    BN = ((d->Cout + 15) / 16) * 16;
  } else {
    const int nt = (d->Cout + 255) / 256;
    BN = std::min(256, (((d->Cout + nt - 1) / nt + 63) / 64) * 64);
    // without statistics / residual the tile's last 64-channel chunk may be narrow (written with plain 16-byte stores instead of
    // the TMA box): 304 channels run as 2 x 160 columns instead of 2 x 192 - a sixth less MMA work on the decoder's data gradient
    if (!(d->flags & (ISWM_EPI_STATS | ISWM_EPI_RESIDUAL)) && (d->Cout % 8) == 0)
      BN = std::min(BN, (((d->Cout + nt - 1) / nt + 31) / 32) * 32);
    p.narrow_tail = (BN % 64) != 0 ? 1 : 0;
  }
  p.BN = BN;
  p.tiles_n = (d->Cout + BN - 1) / BN;
  const int64_t total = (int64_t)p.tiles_w * p.tiles_h * p.tiles_b * p.tiles_n;
  ISWM_REQUIRE(total < (1ll << 31), "conv_igemm: too many tiles");
  p.total_tiles = (int)total;
  p.kchunks = (d->Cin + KB - 1) / KB;
  p.cin_pad = p.kchunks * KB;
  p.ntaps = d->ntaps;
  const int stage_bytes = kABytes + BN * 128;
  p.use_tma_out = (!f8 && !(d->flags & ISWM_EPI_OUT_F32) && (d->out_ld % 8) == 0 &&
                   (reinterpret_cast<uintptr_t>(d_out) & 15) == 0) ? 1 : 0;
  ISWM_REQUIRE(!(d->flags & ISWM_EPI_RESIDUAL) || (reinterpret_cast<uintptr_t>(d_res) & 15) == 0 || (d->res_ld & 7) != 0,
               "conv_igemm: a residual with res_ld %% 8 == 0 must be 16-byte aligned");
  ISWM_REQUIRE(!(d->flags & ISWM_EPI_STATS) || p.use_tma_out, "conv_igemm: STATS needs a bf16 output with out_ld %% 8 == 0 and a 16-byte aligned base");
  int fixed = 1024 /*align*/ + 256 /*barriers*/ + ((d->flags & ISWM_EPI_AFFINE) ? 2048 : 0);
  if (p.use_tma_out) fixed += kEpiWG * kStageBuf;
  // epilogue-bound (short-K) convolutions hide the residual read behind a shared-memory prefetch; long-K ones keep
  // the ring stage instead and load the residual directly under the TMEM read
  p.res_prefetch = (!f8 && (d->flags & ISWM_EPI_RESIDUAL) && (d->res_ld % 8) == 0 && d->ntaps * p.kchunks <= 16) ? 1 : 0;
  if (p.res_prefetch) fixed += kEpiWG * kStageBuf;
  p.stages = std::max(2, std::min(kMaxStages, (kSmemMax - fixed) / stage_bytes));
  p.flags = d->flags | ((f8 && out_type == ISWM_F32) ? ISWM_EPI_OUT_F32 : 0);
  p.res_scale = res_scale;
  p.out_f8 = (f8 && out_type == ISWM_E4M3) ? 1 : 0;
  p.n_img_per_phase = B;
  p.out_ld = d->out_ld;
  p.res_ld = d->res_ld;
  ISWM_REQUIRE(!strided_out || (d->out_ws >= d->out_ld && d->out_hs > 0 && d->out_bs > 0 && (d->out_ws % 8) == 0 && (d->out_hs % 8) == 0 && (d->out_bs % 8) == 0),
               "conv_igemm: strided output needs positive strides that are multiples of 8 elements (ws=%d hs=%d bs=%lld)", d->out_ws, d->out_hs, (long long)d->out_bs);
  ISWM_REQUIRE(!strided_out || p.use_tma_out, "conv_igemm: a strided output view needs the bf16 TMA output path");
  ISWM_REQUIRE(!strided_out || !(d->flags & ISWM_EPI_RESIDUAL) || d->res_ld == d->out_ld, "conv_igemm: strided residual must share the output geometry");
  if (strided_out) {
    p.o_ws = d->out_ws; p.o_hs = d->out_hs; p.o_bs = d->out_bs;
    p.r_ws = p.o_ws; p.r_hs = p.o_hs; p.r_bs = p.o_bs;
  } else {
    p.o_ws = d->out_ld; p.o_hs = (long long)Wo * d->out_ld; p.o_bs = (long long)Ho * Wo * d->out_ld;
    p.r_ws = d->res_ld; p.r_hs = (long long)Wo * d->res_ld; p.r_bs = (long long)Ho * Wo * d->res_ld;
  }
  int in_c = d->Cin;                                       // channels the input tensor map must span
  for (int t = 0; t < d->ntaps; t++) {
    p.dh[t] = d->dh[t]; p.dw[t] = d->dw[t]; p.phase[t] = d->phase[t]; p.coff[t] = d->coff[t];
    p.wtap[t] = d->wtap[t] > 0 ? (int8_t)(d->wtap[t] - 1) : (int8_t)t;
    ISWM_REQUIRE(d->coff[t] >= 0 && (d->coff[t] % 8) == 0 && d->coff[t] + d->Cin <= d->in_ld,
                 "conv_igemm: tap %d channel offset %d (must be a multiple of 8 with offset + Cin <= in_ld)", t, (int)d->coff[t]);
    ISWM_REQUIRE(d->coff[t] == 0 || (d->Cin % KB) == 0, "conv_igemm: channel-offset taps need Cin %% %d == 0 (the K tail is zero-filled by the tensor map's edge)", KB);
    in_c = std::max(in_c, d->coff[t] + d->Cin);
  }
  p.out = d_out; p.scale = d_scale; p.shift = d_shift;
  p.res = static_cast<const __nv_bfloat16*>(d_res);
  p.mask = d_res_mask;
  p.stats = d_stats;
  p.stats_rep = ((d->flags & ISWM_EPI_STATS) && d->stats_replicas > 1) ? d->stats_replicas : 1;
  ISWM_REQUIRE(p.stats_rep <= 64, "conv_igemm: stats_replicas=%d (at most 64)", d->stats_replicas);
  p.abort_flag = abort_flag;

  auto encode = f8 ? encode_tmap_u8 : encode_tmap_bf16;
  CUtensorMap tmap_a, tmap_b;
  if (phase_view) {
    // dense [B, 2Hi, 2Wi, ld] read as four parity phases: {column parity * ld + channel, w, row parity, h, image}
    const uint64_t ld = (uint64_t)d->in_ld, Wf = 2ull * Wi, Hf = 2ull * Hi;
    const uint64_t dims[5] = {ld + (uint64_t)in_c, (uint64_t)Wi, 2, (uint64_t)Hi, (uint64_t)B};
    const uint64_t str[5] = {1, 2 * ld, Wf * ld, 2 * Wf * ld, Hf * Wf * ld};
    const uint32_t box[5] = {(uint32_t)KB, (uint32_t)BW, 1, (uint32_t)BH, (uint32_t)BB};
    if (int rc = encode(&tmap_a, d_in, 5, dims, str, box)) return rc;
    p.phase_view = 1;
    p.pv_ld = d->in_ld;
  } else {
    const uint64_t dims[4] = {(uint64_t)in_c, (uint64_t)Wi, (uint64_t)Hi, (uint64_t)n_img};
    const uint64_t str[4] = {1, (uint64_t)d->in_ld, (uint64_t)Wi * d->in_ld, (uint64_t)Hi * Wi * d->in_ld};
    const uint32_t box[4] = {(uint32_t)KB, (uint32_t)BW, (uint32_t)BH, (uint32_t)BB};
    if (int rc = encode(&tmap_a, d_in, 4, dims, str, box)) return rc;
  }
  {
    const int w_ntaps = d->w_ntaps > 0 ? d->w_ntaps : d->ntaps;
    for (int t = 0; t < d->ntaps; t++)
      ISWM_REQUIRE(p.wtap[t] >= 0 && p.wtap[t] < w_ntaps, "conv_igemm: tap %d reads weight tap %d of %d", t, (int)p.wtap[t], w_ntaps);
    const uint64_t ktot = (uint64_t)w_ntaps * p.cin_pad;
    const uint64_t dims[2] = {ktot, (uint64_t)d->Cout};
    const uint64_t str[2] = {1, ktot};
    const uint32_t box[2] = {(uint32_t)KB, (uint32_t)BN};
    if (int rc = encode(&tmap_b, d_wgt, 2, dims, str, box)) return rc;
  }
  CUtensorMap tmap_out = tmap_a;                         // placeholder when unused
  if (p.use_tma_out) {
    const uint64_t dims[4] = {(uint64_t)d->Cout, (uint64_t)Wo, (uint64_t)Ho, (uint64_t)B};
    // one store per epilogue warp: the 32 consecutive tile rows of a warp are a sub-box of the 128-pixel tile
    const int sBW = std::min(BW, 32), sBH = std::min(BH, 32 / sBW), sBB = 32 / (sBW * sBH);
    const uint32_t box[4] = {(uint32_t)kKBlock, (uint32_t)sBW, (uint32_t)sBH, (uint32_t)sBB};
    const uint64_t str[4] = {1, (uint64_t)p.o_ws, (uint64_t)p.o_hs, (uint64_t)p.o_bs};
    if (int rc = encode_tmap_bf16(&tmap_out, d_out, 4, dims, str, box)) return rc;
  }
  const int smem_bytes = p.stages * stage_bytes + fixed;
  auto kernel = f8 ? conv_igemm_f8_kernel : conv_igemm_kernel;
  static bool attr_set[2] = {false, false};
  if (!attr_set[f8]) {
    const cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 232448);
    ISWM_REQUIRE(e == cudaSuccess, "conv_igemm: cudaFuncSetAttribute: %s", cudaGetErrorString(e));
    static_assert(kSmemMax == 232448, "opt-in shared memory limit of sm_100");
    attr_set[f8] = true;
  }
  const int grid = std::min(p.total_tiles, num_sms());
  {
    // mixed-radix digits of the grid size over (tiles_n, tiles_w, tiles_h, tiles_b) for TileIter::next
    int r = grid;
    p.step = grid;
    p.s_nt = r % p.tiles_n; r /= p.tiles_n;
    p.s_tw = r % p.tiles_w; r /= p.tiles_w;
    p.s_th = r % p.tiles_h; r /= p.tiles_h;
    p.s_tb = r;
  }
  // second producer warp: pays off when a k-block's MMA time (128 x BN x 64) is short against the ~300-cycle issue path of
  // one producer thread, i.e. for narrow N tiles
  p.nprod = (BN <= 128 && p.stages >= 4) ? 2 : 1;
  launch_k(kernel, dim3(grid), dim3(kConvThreads), smem_bytes, static_cast<cudaStream_t>(stream), tmap_a, tmap_b, tmap_out, p);
  return check_launch(f8 ? "conv_igemm_f8" : "conv_igemm");
}

extern "C" int iswm_conv_igemm_ex(const iswm_conv_desc* d, const void* d_in, const void* d_wgt,
                                  void* d_out, const float* d_scale, const float* d_shift,
                                  const void* d_res, double* d_stats, const uint8_t* d_res_mask, void* stream) {
  if (debug_skip(ISWM_SKIP_CONV_IGEMM)) return 0;
  return conv_igemm_launch(d, d_in, d_wgt, d_out, d_scale, d_shift, d_res, d_stats, d_res_mask, false, 1.f, ISWM_BF16, stream);
}

extern "C" int iswm_conv_igemm_f8(const iswm_conv_desc* d, const void* d_in, const void* d_wgt, void* d_out,
                                  const float* d_scale, const float* d_shift, const void* d_res, float res_scale,
                                  int out_type, void* stream) {
  return conv_igemm_launch(d, d_in, d_wgt, d_out, d_scale, d_shift, d_res, nullptr, nullptr, true, res_scale, out_type, stream);
}

extern "C" int iswm_aspp_bwd(const void* d_dycat, int dy_ld, const void* d_wcat, int B, int H, int W, int Cb, int Cfeat,
                             const int* rates, void* d_dfeat, int dfeat_ld, int accumulate, void* stream) {
  ISWM_REQUIRE(d_dycat && d_wcat && d_dfeat && rates, "aspp_bwd: null argument");
  ISWM_REQUIRE(Cb >= 64 && (Cb % 64) == 0 && 4 * Cb <= dy_ld, "aspp_bwd: Cb=%d must be a multiple of 64 with 4*Cb <= dy_ld=%d", Cb, dy_ld);
  iswm_conv_desc d;
  memset(&d, 0, sizeof(d));
  d.B = B; d.Hi = H; d.Wi = W; d.Cin = Cb; d.in_ld = dy_ld; d.n_img = B;
  d.Ho = H; d.Wo = W; d.Cout = Cfeat; d.out_ld = dfeat_ld; d.res_ld = dfeat_ld;
  int t = 0;
  d.dh[t] = 0; d.dw[t] = 0; d.phase[t] = 0; d.coff[t] = 0; t++;            // branch 0: 1x1
  for (int i = 0; i < 3; i++) {
    const int r = rates[i];
    ISWM_REQUIRE(r >= 1 && r <= 127, "aspp_bwd: rate %d out of range", r);
    for (int a = -1; a <= 1; a++)
      for (int b = -1; b <= 1; b++) {                                          // data gradient: negated forward taps, forward tap ORDER
        d.dh[t] = (int8_t)(-a * r); d.dw[t] = (int8_t)(-b * r); d.phase[t] = 0; d.coff[t] = (int16_t)((i + 1) * Cb); t++;
      }
  }
  d.ntaps = t;
  d.flags = accumulate ? ISWM_EPI_RESIDUAL : 0;
  return iswm_conv_igemm(&d, d_dycat, d_wcat, d_dfeat, nullptr, nullptr, accumulate ? d_dfeat : nullptr, nullptr, stream);
}
