/*
 * iswm_b200.h — C ABI of libiswm_b200.so (sm_100a only).
 *
 * Drop-in boundary for the ONE hot path of Alanlee0323/ISWM: the DeepLabV3+
 * train / predict step, its weighted cross-entropy and its confusion matrix.
 * The reference has no FFI of its own (pure Python, SURVEY.md §8b); each entry
 * point below names the reference Python call site it replaces (file:line
 * relative to the reference tree).
 *
 * Conventions (all entry points):
 *   - plain pointers and sizes only; no torch types;
 *   - every pointer named d_* is a DEVICE pointer owned by the caller; the
 *     library never frees or retains it (tensor-map caches key on the address);
 *   - every call enqueues on `stream` (a cudaStream_t passed as void*) and
 *     never synchronises;
 *   - return 0 on success, non-zero on error; iswm_last_error() gives a
 *     thread-local message; no C++ exception crosses the boundary;
 *   - activations are NHWC bf16 unless stated, parameters handed over in the
 *     reference's own layout (fp32 OIHW) and packed by iswm_pack_*.
 */
#ifndef ISWM_B200_H
#define ISWM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- library ---------------------------------------------------------- */
const char* iswm_last_error(void);
int iswm_version(void);
/* number of kernels this library has launched in this process (bench.py's
 * gpu_launches claim is read from here). */
int64_t iswm_launch_count(void);
void iswm_reset_launch_count(void);
/* synchronising health check (tests / debug): code recorded by a tensor-core kernel whose
 * bounded mbarrier wait timed out (0 = healthy); clears it. */
int iswm_debug_abort_code(void);
/* Measurement aid: entry points of the masked kernel families return 0 WITHOUT launching (outputs stay unwritten).
 * bench.py times whole steps with and without a family to get its marginal cost inside the real launch pipeline
 * (per-launch CUDA events add ~7 us of drain per kernel and break the programmatic-dependent-launch overlap). */
enum { ISWM_SKIP_CONV_IGEMM = 1, ISWM_SKIP_CONV_WGRAD = 2, ISWM_SKIP_BN = 4 };
void iswm_debug_set_skip(int mask);

/* element type codes for label / prediction buffers */
enum { ISWM_U8 = 0, ISWM_I32 = 1, ISWM_I64 = 2 };
/* element type codes for floating tensors */
enum { ISWM_F32 = 0, ISWM_BF16 = 1, ISWM_E4M3 = 2 };

/* ---- loss / histogram / metric (HBM-bound) ----------------------------- */

/* Per-class pixel counts: d_hist[c] += #{i : labels[i] == c}, 0 <= c < n_classes.
 * Values outside [0,n_classes) (e.g. ignore 255) are counted nowhere.
 * Replaces: train.py:401-402 `(labels == 0).sum()`, `(labels == 1).sum()` in
 * calculate_class_weights, and the implicit per-class counts behind
 * nn.CrossEntropyLoss's weighted-mean denominator (train.py:457-459).
 * d_hist: int64[n_classes], ACCUMULATED into (zero it first for a fresh count). */
int iswm_class_hist(const void* d_labels, int label_dtype, int64_t n,
                    int n_classes, int64_t* d_hist, void* stream);

/* Fused weighted softmax cross-entropy forward + backward, one HBM pass.
 * Semantics = nn.CrossEntropyLoss(weight=w, ignore_index, reduction='mean')
 * (train.py:454-459) called at train.py:1046 and differentiated at :1048.
 *   d_logits : [B, C, HW] (NCHW), fp32 or bf16 (logit_dtype)
 *   d_labels : [B, HW]
 *   d_weight : float[C] or NULL (all ones)
 *   d_hist   : int64[C] per-class counts of THIS loss's batch (global batch
 *              when data-parallel), from iswm_class_hist; gives the
 *              denominator D = sum_c w_c * hist[c] (c != ignore_index)
 *   d_grad   : same shape/dtype as logits, = grad_scale * dL/dlogits, or NULL
 *   d_loss_num: double[1], ACCUMULATES sum_i w[y_i] * nll_i (zero it first)
 *   d_loss   : float[1] or NULL; if non-NULL a last-block epilogue writes
 *              loss = loss_num / D
 */
int iswm_wce_fwd_bwd(const void* d_logits, int logit_dtype, const void* d_labels,
                     int label_dtype, const float* d_weight, const int64_t* d_hist,
                     int64_t B, int C, int64_t HW, int ignore_index,
                     float grad_scale, void* d_grad, double* d_loss_num,
                     float* d_loss, void* stream);

/* Confusion matrix: cm[t*n + p] += 1 for every i with 0 <= t=true[i] < n
 * (pred p outside [0,n) is dropped and counted in d_cm[n*n], one extra slot).
 * Replaces: metrics/stream_metrics.py:24-31 `_fast_hist` + :122 accumulation.
 * d_cm: int64[n*n + 1], ACCUMULATED into. */
int iswm_confusion(const void* d_true, int true_dtype, const void* d_pred,
                   int pred_dtype, int64_t n, int n_classes, int64_t* d_cm,
                   void* stream);

/* argmax / threshold fused with the confusion matrix.
 * Replaces: train.py:644,659 `logits.max(1)[1]` (mode 0: first maximum wins,
 * ties -> lowest class) and predict.py:264-275 / evaluate_quantization.py:265-269
 * `softmax(logits,1)[:,1] > threshold` (mode 1, C must be >= 2), followed by
 * `_fast_hist`.
 *   d_pred_out: optional uint8[B*HW] class map (NULL to skip)
 *   d_conf_out: optional uint8[B*HW] `uint8(prob1*255)` map, mode 1 only
 *               (predict.py:285-288), NULL to skip
 *   d_true may be NULL (no confusion matrix, predictions only). */
int iswm_argmax_confusion(const void* d_logits, int logit_dtype, const void* d_true,
                          int true_dtype, int64_t B, int C, int64_t HW, int mode,
                          float threshold, uint8_t* d_pred_out, uint8_t* d_conf_out,
                          int64_t* d_cm, void* stream);

/* ---- the step after the hot path: fused predict epilogue (SURVEY 8f rank 3) ---------------- */
/* Final bilinear upsample (network/utils.py:22, align_corners=False) of the LOW-resolution two-class logits fused with
 * softmax + threshold + confidence map (predict.py:262-290) and, optionally, the confusion matrix
 * (evaluate_quantization.py:265-270): writes uint8 maps only, the full-resolution fp32 logits never exist.
 *   d_lo        float32 NHWC [B,Hi,Wi,2] (what the classifier 1x1 conv writes)
 *   mode        0: pred = argmax (ties -> 0); 1: pred = softmax[:,1] > threshold
 *   d_true      labels [B,Ho,Wo] or NULL; d_cm int64[5] accumulated into (layout of iswm_confusion) or NULL
 *   d_pred_out  uint8 [B,Ho,Wo] or NULL; d_conf_out uint8 [B,Ho,Wo] = uint8(prob1*255) (mode 1) or NULL
 * Bit-identical to iswm_logits_up_fwd followed by iswm_argmax_confusion. Requires C == 2 and Wo % 4 == 0. */
int iswm_predict_epilogue(const float* d_lo, int B, int Hi, int Wi, int C, int Ho, int Wo, int mode,
                          float threshold, const void* d_true, int true_dtype, uint8_t* d_pred_out,
                          uint8_t* d_conf_out, int64_t* d_cm, void* stream);

/* ---- test-time augmentation (multi-scale + horizontal flip) for the predict step --------------------- */
/* Bilinear resize (align_corners=False, no antialias) of fp32 NCHW [B,C,Hi,Wi] to [B,C,Ho,Wo], then an optional
 * horizontal mirror: F.interpolate(x, size=(Ho,Wo), mode="bilinear") followed by .flip(-1), with the four taps mixed in
 * torch's association. With (Ho,Wo) == (Hi,Wi) it is an exact copy (mirrored when flip). d_out may be a batch slice of a
 * larger buffer. */
int iswm_resize_flip_f32(const float* d_x, int B, int C, int Hi, int Wi, int Ho, int Wo, int flip, float* d_out,
                         void* stream);

/* One view of iswm_predict_tta_epilogue: the low-resolution logits of the network run on the view's input. */
typedef struct {
  const float* lo; /* device, float32 NHWC [B,Hi,Wi,2] (forward_lowres output, or a batch slice of it) */
  int Hi, Wi;      /* low-resolution size */
  int Hv, Wv;      /* the view's full-resolution size (the size of the input the network ran on) */
  int flip;        /* 1: the view's input was mirrored horizontally */
} IswmTtaView;
#define ISWM_TTA_MAX_VIEWS 8

/* Multi-view predict epilogue: for every output pixel and view v, logits bilinear (Hi,Wi) -> (Hv,Wv) -> (Ho,Wo)
 * (the second resize skipped when (Hv,Wv) == (Ho,Wo)), un-mirrored when flip, then the 2-class softmax; the
 * probabilities are summed in view order and divided by n_views. mode 1: pred = p1 > threshold; mode 0: pred = p1 > p0
 * (a tie goes to the sign of the summed logit margin, which makes one view equal the logit argmax).
 * d_conf_out = uint8(p1*255) in mode 1, zeros in mode 0. d_true / d_cm / d_pred_out / d_conf_out as in
 * iswm_predict_epilogue. h_views is a HOST array of n_views (1..ISWM_TTA_MAX_VIEWS) records passed to the kernel by
 * value (graph-capturable). C == 2 only; any Wo >= 1. A single unflipped view with (Hv,Wv) == (Ho,Wo) is
 * bit-identical to iswm_predict_epilogue. */
int iswm_predict_tta_epilogue(const IswmTtaView* h_views, int n_views, int B, int C, int Ho, int Wo, int mode,
                              float threshold, const void* d_true, int true_dtype, uint8_t* d_pred_out,
                              uint8_t* d_conf_out, int64_t* d_cm, void* stream);

/* Focal loss forward + backward in one pass (utils/loss.py:14-35 FocalLoss, exported through create_loss :37-39):
 *   ce_i = w[y_i] * nll_i (0 where y_i == ignore_index or outside [0,C)); pt = exp(-ce_i)
 *   loss = sum_i alpha * (1 - pt)^gamma * ce_i, divided by the number of ALL pixels when size_average
 *   d_grad (same shape / dtype as logits, or NULL) = dloss/dlogits; d_loss_num double[1] ACCUMULATES the sum;
 *   d_loss float[1] or NULL receives the final scalar. */
int iswm_focal_fwd_bwd(const void* d_logits, int logit_dtype, const void* d_labels, int label_dtype,
                       const float* d_weight, int64_t B, int C, int64_t HW, int ignore_index,
                       float alpha, float gamma, int size_average, void* d_grad, double* d_loss_num,
                       float* d_loss, void* stream);

/* ---- convolution as implicit GEMM on tcgen05 / TMEM / TMA -------------- */

#define ISWM_MAX_TAPS 32

/* epilogue flags */
enum {
  ISWM_EPI_AFFINE   = 1,  /* y = acc * scale[c] + shift[c] (eval BN folded / bias) */
  ISWM_EPI_RELU     = 2,
  ISWM_EPI_RESIDUAL = 4,  /* y += residual (bf16, same geometry, own ld)      */
  ISWM_EPI_STATS    = 8,  /* accumulate per-channel fp32 sum / sum^2 of the STORED bf16 outputs (needs bf16 out, out_ld % 8 == 0) */
  ISWM_EPI_OUT_F32  = 16, /* write fp32 instead of bf16                       */
  ISWM_EPI_RES_MASK = 32  /* the residual is gated by packed ReLU sign bits (iswm_conv_igemm_ex): y += res * bit  */
};

/* Geometry of one implicit-GEMM convolution over NHWC bf16 activations.
 * out[b,ho,wo,n] = sum_t sum_c in[img(t,b), ho + dh[t], wo + dw[t], coff[t] + c] * wgt[n, t, c]
 * with zero fill outside [0,Hi)x[0,Wi). coff[t] (a multiple of 8, 0 for an ordinary convolution) selects a channel slice
 * of a wider input buffer per tap: several convolutions that read different slices of one buffer and sum into the same
 * output run as ONE K-concatenated GEMM (the four ASPP branches' input gradients, iswm_aspp_bwd). Strided convolutions are expressed
 * over the 4 parity phases of the input (phase-major [4][B][Hi][Wi][C]),
 * img(t,b) = phase[t]*B + b.
 * Replaces nn.Conv2d at network/backbone/resnet.py:27-35 (conv3x3/conv1x1),
 * network/_deeplab.py:37,45,48,51,124,134,149,162 and, with transposed packed
 * weights and negated taps, their input gradients. */
typedef struct {
  int32_t B, Hi, Wi, Cin;     /* input images (per phase), spatial, channels  */
  int32_t in_ld;              /* input row pitch in elements (>= Cin)          */
  int32_t n_img;              /* images in the input tensor (B * n_phases)     */
  int32_t Ho, Wo, Cout;
  int32_t out_ld;             /* output row pitch in elements                  */
  int32_t res_ld;             /* residual row pitch in elements                */
  int32_t ntaps;
  int8_t  dh[ISWM_MAX_TAPS], dw[ISWM_MAX_TAPS], phase[ISWM_MAX_TAPS];
  int16_t coff[ISWM_MAX_TAPS]; /* per-tap channel offset into the input buffer (elements)  */
  int8_t  wtap[ISWM_MAX_TAPS]; /* 0: tap t reads weight tap t; k > 0: weight tap k - 1 (a SUBSET of a packed tensor's taps:
                                  the per-phase data gradients of a stride-2 convolution)   */
  int32_t flags;
  /* strided output (all 0 = dense [B,Ho,Wo] rows of out_ld): element strides between consecutive output pixels along w, h and
   * images, e.g. 2*ld, 2*W*ld, H*W*ld writes one parity phase of a [B,H,W] tensor. The residual, when present, has the
   * same geometry (its strides are these scaled by res_ld / out_ld; res_ld == out_ld in strided mode). bf16 TMA output only. */
  int32_t out_ws, out_hs;
  int64_t out_bs;
  int32_t w_ntaps;            /* taps per row of the packed weight tensor when wtap[] selects a subset (0 = ntaps) */
  int32_t stats_replicas;     /* ISWM_EPI_STATS: d_stats holds this many copies of double[2*Cout] (0 / 1 = one); CTA i adds into copy
                                 i % replicas and the consumer (iswm_bn_train_apply) sums the copies. With one copy every CTA of a
                                 narrow layer ends on the same 2*Cout addresses: 296 same-address fp64 atomics per channel cost a
                                 64-channel 3x3 convolution 14 of its 51 us (tools/prof_conv.py) */
  int32_t in_phase_view;      /* != 0: d_in is a DENSE bf16 [B, 2*Hi, 2*Wi, in_ld] tensor and the convolution reads its four stride-2 parity
                                 phases in place (phase[t] = 2*row parity + column parity, as for the phase-major copy, but n_img = B):
                                 the stride-2 3x3 / 1x1 convolutions of resnet.py:104,183 without iswm_phase_split / iswm_subsample2
                                 copies. The tensor map is 5-D {(column parity, channel), w, row parity, h, image}. Needs Cin %% 64 == 0. */
  int32_t reserved2_;
} iswm_conv_desc;

/* d_in: bf16 activations; d_wgt: packed bf16 [Cout][ntaps][Cin_pad] (Cin_pad =
 * Cin rounded up to 64, zero padded) from iswm_pack_weight*; d_out bf16/fp32;
 * d_scale/d_shift float[Cout] (AFFINE); d_res bf16 (RESIDUAL); d_stats
 * double[2*Cout] accumulated (STATS): per-CTA partial sums are fp32 in a fixed order, the cross-CTA
 * accumulation is fp64 atomics, so the fp32 mean / variance derived from them do not depend on CTA order. */
int iswm_conv_igemm(const iswm_conv_desc* desc, const void* d_in, const void* d_wgt,
                    void* d_out, const float* d_scale, const float* d_shift,
                    const void* d_res, double* d_stats, void* stream);
/* Same, plus d_res_mask for ISWM_EPI_RES_MASK: uint8 [B*Ho*Wo][Cout/8] ReLU sign bits as written by iswm_bn_train_apply; the
 * residual element of channel c is added only where bit c is set. Used by the backward of a bottleneck block: the block
 * input's gradient = conv1's data gradient + (block output gradient where the block's ReLU was active), so the identity
 * path's gradient (resnet.py:112-118) is never written out as a tensor of its own. */
int iswm_conv_igemm_ex(const iswm_conv_desc* desc, const void* d_in, const void* d_wgt,
                       void* d_out, const float* d_scale, const float* d_shift,
                       const void* d_res, double* d_stats, const uint8_t* d_res_mask, void* stream);

/* FP8 (e4m3) inference form of iswm_conv_igemm (iswm_b200/quant.py): d_in e4m3 NHWC activations (in_ld %% 16 == 0), d_wgt
 * e4m3 [Cout][ntaps][Cin_pad] with Cin_pad = Cin rounded up to 128 (iswm_pack_weight_f8), tcgen05 kind::f8f6f4 with fp32
 * accumulation. Epilogue, in this order: y = acc * scale[c] + shift[c] (AFFINE), y += res_scale * res (RESIDUAL, d_res e4m3 of
 * the output geometry, pitch res_ld), ReLU (RELU), then the store as out_type: ISWM_E4M3 (round to nearest even, saturating
 * to +-448), ISWM_BF16 or ISWM_F32. Statistics, residual masks, ISWM_EPI_OUT_F32 and strided outputs are rejected; a
 * stride-2 convolution's in_phase_view needs Cin %% 128 == 0. */
int iswm_conv_igemm_f8(const iswm_conv_desc* desc, const void* d_in, const void* d_wgt, void* d_out,
                       const float* d_scale, const float* d_shift, const void* d_res, float res_scale,
                       int out_type, void* stream);

/* ASPP backward, data-gradient half (network/_deeplab.py:143-172: the 1x1 branch and the three dilated 3x3 branches all
 * read the SAME 2048-channel feature map): ONE K-concatenated implicit GEMM
 *   dfeat[b,h,w,c] (+)= sum_{branch i} sum_{tap t of i} dy_i[b, h - dh_t, w - dw_t, :] . W_i[:, c, t]
 * over K = (1 + 9 + 9 + 9) taps x Cb channels instead of four data-gradient launches with three read-modify-write passes over
 * the feature gradient. d_dycat: bf16 [B,H,W,dy_ld], branch i's BatchNorm-backward output in channels [i*Cb, (i+1)*Cb);
 * d_wcat: bf16 [Cfeat][28][Cb] = the branches' dgrad operands concatenated along the tap axis (iswm_pack_weights_batched,
 * mode 1, row_ld = 28); rates[3] = the dilations of branches 1..3; d_dfeat bf16 [B,H,W,dfeat_ld]; accumulate != 0 adds to
 * what d_dfeat holds (e.g. the pooled branch's gradient). Cb %% 64 == 0. */
int iswm_aspp_bwd(const void* d_dycat, int dy_ld, const void* d_wcat, int B, int H, int W, int Cb, int Cfeat,
                  const int* rates, void* d_dfeat, int dfeat_ld, int accumulate, void* stream);

/* ---- data-parallel exchanges over NVLink / NVSwitch PEER MEMORY (csrc/peer_allreduce.cu) --------------------------------
 * Replaces nn.DataParallel's gradient reduce-add (train.py:970) and the small per-step reductions of SURVEY 8e. All pointer
 * arrays are HOST arrays of `world` device pointers: rank q's buffer as mapped into THIS rank's address space (symmetric
 * memory; q == rank is the local buffer). Plain stream-ordered kernels, no host synchronisation: capturable in a CUDA graph.
 * iswm_peer_barrier: all ranks have reached this point of their streams and everything they wrote before it is visible
 *   (flag_ptrs[q]: uint32[8] zero-initialised symmetric flags of rank q; d_epoch: this rank's private uint32 barrier count).
 * iswm_peer_allreduce_f32: buf[offset, offset+n) = sum over ranks, identical bits on every rank (fixed rank order); rank r
 *   reduces slice r (pull) and stores it to every rank (push). Callers bracket it with two barriers (data ready / stores landed).
 * iswm_peer_small_publish / _sum: all-reduce of up to 64 int64 or double values through per-rank symmetric slots
 *   (publish -> barrier -> sum); slot_off (8-byte elements) selects the slot region of a call site. */
int iswm_peer_barrier(const void* const* flag_ptrs, int rank, int world, uint32_t* d_epoch, void* stream);
int iswm_peer_allreduce_f32(const void* const* buf_ptrs, int rank, int world, int64_t offset, int64_t n, int max_blocks, void* stream);
int iswm_peer_small_publish(const void* const* slot_ptrs, int rank, int world, const void* d_src, int n, int slot_off, int is_f64, void* stream);
int iswm_peer_small_sum(const void* const* slot_ptrs, int world, void* d_dst, int n, int slot_off, int is_f64, void* stream);

/* Synchronised BatchNorm statistics exchange (one launch, one block). The fp64 vectors live in a symmetric arena that every
 * rank carves at the same offsets: job j reads n values x `replicas` copies (iswm_conv_desc.stats_replicas layout: n = 2*C
 * forward, replicas 1 backward) at arena_ptrs[q] + src_off on every rank q. The kernel writes `count` (this rank's rows) into
 * the word after job 0's copies, passes a barrier on flag_ptrs / d_epoch (as iswm_peer_barrier), then stores
 * dst[i] = sum over ranks 0..world-1 in that order of (sum of the copies in order) - identical bits on every rank - and
 * dst[n] = the sum of the ranks' counts. flag_ptrs NULL (world = 1 only): no barrier - folds the copies and writes the count
 * (what a torch.distributed transport then all-reduces). At most 4 jobs per call, all with the same row count. */
typedef struct {
  int64_t src_off;              /* fp64 elements from the arena base */
  double* dst;                  /* local: double[n + 1] */
  int32_t n;
  int32_t replicas;
} iswm_syncbn_job;
int iswm_syncbn_exchange(const iswm_syncbn_job* jobs, int n_jobs, const void* const* arena_ptrs, const void* const* flag_ptrs,
                         int rank, int world, double count, uint32_t* d_epoch, void* stream);

/* Weight gradient: dW[n, t, c] += sum_{b,ho,wo} dy[b,ho,wo,n] * in[img(t,b), ho+dh[t], wo+dw[t], c]
 * desc as for the forward conv (Cout = channels of dy). d_dw: float [Cout][ntaps][Cin],
 * ACCUMULATED into with fp32 reductions (zero it first). dy row pitch = out_ld. */
int iswm_conv_wgrad(const iswm_conv_desc* desc, const void* d_in, const void* d_dy,
                    float* d_dw, void* stream);
/* The weight gradients of SEVERAL convolutions in ONE launch (csrc/conv_wgrad.cu, grouped kernel): descs[n_jobs] with the
 * per-job device pointers d_in[j] / d_dy[j] / d_dw[j] (host arrays). Work units (job, output tile, pixel-block range) are
 * dealt to the CTAs on the host - a layer's worth of small GEMMs has enough tiles to fill the SMs with few pixel-range splits,
 * so almost no partial-tile reductions remain. Results as n_jobs calls of iswm_conv_wgrad (accumulated into d_dw[j]). The
 * plan is cached per set of shapes; the first call of a shape set allocates device memory (not inside a stream capture). */
int iswm_conv_wgrad_grouped(const iswm_conv_desc* descs, const void* const* d_in, const void* const* d_dy,
                            float* const* d_dw, int n_jobs, void* stream);
/* Same with a CTA budget: the launch plans its tiles x splits for max_ctas SMs instead of all of them (0 = all), so that several
 * small weight gradients launched on different streams run next to each other, each with few splits - a split costs a whole
 * partial-tile fp32 reduction, and a 1x1 layer at 32x32 spread over 148 SMs is mostly that. */
int iswm_conv_wgrad_ex(const iswm_conv_desc* desc, const void* d_in, const void* d_dy,
                       float* d_dw, int max_ctas, void* stream);

/* fp32 OIHW [Cout][Cin][R*S] -> bf16 rows of row_ld elements, element (t*cin_pad + c) = w[o][c][t],
 * zero elsewhere. Forward operand: cin_pad = Cin rounded up to 64, row_ld = R*S*cin_pad.
 * Stem (7x7 over the im2col matrix): cin_pad = Cin, row_ld = 49*Cin rounded up to 64. */
int iswm_pack_weight_fwd(const float* d_w, int Cout, int Cin, int RS, int cin_pad, int row_ld,
                         void* d_out, void* stream);
/* fp32 OIHW -> bf16 [Cin][R*S][cout_pad] (dgrad operand, taps kept in forward order) */
int iswm_pack_weight_dgrad(const float* d_w, int Cout, int Cin, int RS, int cout_pad, void* d_out,
                           void* stream);
/* One launch for many weight tensors (after an optimiser step): d_jobs is a DEVICE array of n_jobs
 * records; mode 0 = forward operand (as iswm_pack_weight_fwd, pad = cin_pad), mode 1 = dgrad operand
 * (as iswm_pack_weight_dgrad, pad = cout_pad; row_ld = 0, or the number of taps of a K-CONCATENATED row of which this
 * tensor's R*S taps are a slice starting at dst: row (c, t) is written at c * row_ld + t, the layout iswm_aspp_bwd
 * reads). The caller deals thread blocks to jobs in
 * proportion to their size: job i owns blocks [blk_begin, blk_begin + blk_count), blk_begin ascending and
 * contiguous from 0; total_blocks = sum of blk_count. */
typedef struct {
  const float* w;      /* fp32 OIHW source (device) */
  void* dst;           /* bf16 destination (device) */
  int32_t Cout, Cin, RS, pad, row_ld, mode;
  int32_t blk_begin, blk_count;
} iswm_pack_job;
int iswm_pack_weights_batched(const void* d_jobs, int n_jobs, int total_blocks, void* stream);

/* Optimiser step + operand repack in ONE pass (csrc/sgd_pack.cu; train.py:421-431 torch.optim.SGD and :1049 optimizer.step()):
 * the job table covers the flat parameter buffer - convolution weights (mode 1: update, then both packed bf16 layouts from the
 * same shared-memory tile; mode 2: the stem, update + row-tap forward operand) and the ranges between them (mode 0: update only).
 * Same arithmetic as iswm_sgd_step followed by iswm_pack_weights_batched: bit-identical weights, momentum and operands.
 * Padding elements of the packed buffers (Cin / Cout rounded up to 64) are NOT written: pack once with
 * iswm_pack_weights_batched before the first fused step. Job j owns thread blocks [blk_begin, blk_begin + blk_count). */
typedef struct {
  float* w; const float* g; float* m;          /* fp32 master weights / gradient / momentum (m NULL: no momentum) */
  void* dst_f; void* dst_d;                    /* packed bf16 forward / data-gradient operands (NULL: none) */
  int64_t n;                                   /* element count (modes 0 and 2) */
  int32_t Cout, Cin, RS;
  int32_t pad_f, row_ld_f;                     /* forward: channels per tap, elements per output channel */
  int32_t pad_d, row_ld_d;                     /* dgrad: Cout padded to 64; taps per row of a K-concatenated operand (0 = RS) */
  int32_t mode;                                /* 0 plain, 1 convolution, 2 stem */
  int32_t TC;                                  /* input channels per tile (mode 1): a multiple of 8 with 16 * TC * RS <= 2304 */
  int32_t blk_begin, blk_count;
} iswm_sgd_pack_job;
int iswm_sgd_pack_batched(const void* d_jobs, int n_jobs, int total_blocks, float lr, float momentum, float weight_decay,
                          int nesterov, int first_step, const float* d_lr, void* stream);

/* wgrad accumulator (fp32 rows of row_ld, element t*cin_stride + c) -> fp32 OIHW grad,
 * dst = beta*dst + src. Normal: cin_stride = Cin, row_ld = R*S*Cin. */
int iswm_unpack_wgrad(const float* d_dw, int Cout, int Cin, int RS, int cin_stride, int row_ld,
                      float beta, float* d_grad_oihw, void* stream);

/* All k x k (2 <= RS <= 9, dense rows) accumulators of a step in ONE launch (dst += src permuted): the
 * caller lists its jobs in a device array and deals blocks to them, job j owning blocks
 * [blk_begin, blk_begin + Cout * chunks) with chunks = ceil(Cin / 512). */
typedef struct {
  const float* src;           /* [Cout][RS][Cin] accumulator */
  float* dst;                 /* [Cout][Cin][RS] = OIHW gradient */
  int32_t Cout, Cin, RS, chunks;
  int32_t blk_begin, pad_;
} iswm_unpack_job;
int iswm_unpack_wgrad_batched(const void* d_jobs, int n_jobs, int total_blocks, void* stream);

/* ---- HBM-bound glue kernels (see src for reference citations) ---------- */

/* BatchNorm2d training forward, second half (network/backbone/resnet.py:92-110 bn1..bn3,
 * network/_deeplab.py:38,46,49,125,135,150,163): from per-channel sum/sum^2
 * (conv epilogue STATS) compute batch mean / biased var, write
 * out = [relu]( gamma*(x-mean)*invstd + beta [+ residual] ) with optional dropout,
 * save mean/invstd for backward, update running stats (momentum, unbiased var).
 * Dropout (network/_deeplab.py:165 nn.Dropout(0.1)) is counter-based: element i is kept iff hash(seed_eff, i) >= p with
 * seed_eff = (drop_seed + 1000003 * *d_drop_step) mod 2^48; d_drop_step (int64 on the DEVICE, or NULL = 0) lets a
 * train step captured in a CUDA graph draw a fresh mask on every replay. The backward kernels take the same pair.
 * d_relu_bits (optional, with relu): uint8 [M, C/8], bit j of byte (row, g) = output channel 8g+j is positive. The
 * backward kernels of residual units read these bits (relu mode 2, passed in d_out_act) instead of the 16-byte
 * activation row: the mask of relu(bn(x) + residual) cannot be recomputed from x alone. */
int iswm_bn_train_apply(const void* d_x, int x_ld, const double* d_stats, int stats_replicas, int64_t M, int C,
                        const float* d_gamma, const float* d_beta, float eps, float momentum,
                        float* d_running_mean, float* d_running_var, int64_t* d_num_batches_tracked,
                        float* d_save_mean, float* d_save_invstd, const void* d_res, int res_ld, int relu,
                        float drop_p, uint64_t drop_seed, const int64_t* d_drop_step, void* d_out, int out_ld,
                        uint8_t* d_relu_bits, void* stream);
/* Synchronised BatchNorm (iswm_syncbn_exchange): d_gstats = double[2*C + 1], the sums over every rank's rows (one copy) and the
 * global row count; mean, variance and the running variance's unbiased factor use that count, M is this rank's rows. With
 * the local sums and count = M it computes exactly what iswm_bn_train_apply does. */
int iswm_bn_train_apply_global(const void* d_x, int x_ld, const double* d_gstats, int64_t M, int C,
                               const float* d_gamma, const float* d_beta, float eps, float momentum,
                               float* d_running_mean, float* d_running_var, int64_t* d_num_batches_tracked,
                               float* d_save_mean, float* d_save_invstd, const void* d_res, int res_ld, int relu,
                               float drop_p, uint64_t drop_seed, const int64_t* d_drop_step, void* d_out, int out_ld,
                               uint8_t* d_relu_bits, void* stream);

/* eval-mode BN folding: scale = gamma / sqrt(running_var + eps), shift = beta - mean*scale */
int iswm_bn_fold(const float* d_gamma, const float* d_beta, const float* d_mean, const float* d_var,
                 float eps, int C, float* d_scale, float* d_shift, void* stream);

/* BatchNorm backward, pass 1: dz = dout * [out>0 if relu] * dropmask;
 * sums[c] = sum dz, sums[C+c] = sum dz * xhat. d_out_act = post-activation output (for the ReLU mask);
 * pass NULL for a unit WITHOUT a residual add and the mask is recomputed from d_x with the forward
 * kernel's own arithmetic, gamma*invstd*x + (beta - mean*gamma*invstd) > 0 (one tensor read less).
 * relu: 0 = no mask, 1 = as above, 2 = d_out_act points at the packed sign bits written by iswm_bn_train_apply
 * (uint8 [M, C/8], act_ld ignored): 1 byte instead of 16 per 8 channels on residual units. Same in iswm_bn_bwd_apply. */
int iswm_bn_bwd_reduce(const void* d_dout, int dout_ld, const void* d_x, int x_ld,
                       const void* d_out_act, int act_ld, int64_t M, int C,
                       const float* d_save_mean, const float* d_save_invstd,
                       const float* d_gamma, const float* d_beta, int relu,
                       float drop_p, uint64_t drop_seed, const int64_t* d_drop_step, double* d_sums, void* stream);
/* pass 2: dx = gamma*invstd*(dz - sum_dz/M - xhat*sum_dzxhat/M); dgamma += , dbeta += ;
 * optionally writes dz (the pre-activation gradient, used by the residual identity path). */
int iswm_bn_bwd_apply(const void* d_dout, int dout_ld, const void* d_x, int x_ld,
                      const void* d_out_act, int act_ld, int64_t M, int C,
                      const float* d_gamma, const float* d_beta, const float* d_save_mean,
                      const float* d_save_invstd, const double* d_sums, int relu, float drop_p, uint64_t drop_seed, const int64_t* d_drop_step,
                      void* d_dx, int dx_ld, void* d_dz, int dz_ld,
                      float* d_dgamma, float* d_dbeta, void* stream);
/* Synchronised BatchNorm: d_gsums = double[2*C + 1], the exchanged sums of iswm_bn_bwd_reduce over every rank and the global
 * row count (the normaliser); dgamma / dbeta accumulate THIS rank's sums d_local_sums, so that a SUM all-reduce of the
 * parameter gradients yields the global values. */
int iswm_bn_bwd_apply_global(const void* d_dout, int dout_ld, const void* d_x, int x_ld,
                             const void* d_out_act, int act_ld, int64_t M, int C,
                             const float* d_gamma, const float* d_beta, const float* d_save_mean,
                             const float* d_save_invstd, const double* d_gsums, const double* d_local_sums, int relu, float drop_p,
                             uint64_t drop_seed, const int64_t* d_drop_step, void* d_dx, int dx_ld, void* d_dz, int dz_ld,
                             float* d_dgamma, float* d_dbeta, void* stream);

/* ---- the closing BatchNorm of a bottleneck block WITH a downsample branch, both branches per pass (csrc/bn_dual.cu) ----
 *   out = relu( bn3(raw) + bn_ds(raw_ds) )        network/backbone/resnet.py:110-118 with `downsample` (:176-186)
 * raw / raw_ds: bf16 [M][C] pre-BatchNorm outputs of conv3 and of the downsample convolution (iswm_conv_igemm with
 * ISWM_EPI_STATS). The normalised shortcut is never written out, and in backward the block-output gradient and its
 * ReLU sign bits are read once per pass for both BatchNorms instead of once per BatchNorm. One iswm_bn_side per BatchNorm:
 * forward reads stats / gamma / beta, updates running_mean / running_var / num_batches_tracked (NULL = skip) and writes
 * save_mean / save_invstd; the backward passes read gamma / save_mean / save_invstd. */
typedef struct {
  const double* stats;          /* double[2*C]: sum x, sum x^2 over the M rows (forward only) */
  const float*  gamma;
  const float*  beta;
  float*        running_mean;
  float*        running_var;
  int64_t*      num_batches_tracked;
  float*        save_mean;      /* float[C] */
  float*        save_invstd;    /* float[C] */
  int32_t       stats_replicas; /* copies of double[2*C] in `stats` to sum (0 / 1 = one; see iswm_conv_desc.stats_replicas) */
} iswm_bn_side;
/* d_relu_bits (uint8 [M][C/8], may be NULL): sign bits of the block output, as iswm_bn_train_apply writes them. */
int iswm_bn_dual_train_apply(const void* d_x, int x_ld, const iswm_bn_side* main_bn,
                             const void* d_x_ds, int x_ds_ld, const iswm_bn_side* ds_bn,
                             int64_t M, int C, float eps, float momentum,
                             void* d_out, int out_ld, uint8_t* d_relu_bits, void* stream);
/* pass 1: dz = dout where the bit is set; d_sums[c] += sum dz, d_sums[C+c] += sum dz.xhat (main), d_sums_ds likewise with
 * the downsample branch's xhat (its first half equals d_sums'). double[2*C] each, zeroed by the caller. */
int iswm_bn_dual_bwd_reduce(const void* d_dout, int dout_ld, const uint8_t* d_relu_bits,
                            const void* d_x, int x_ld, const iswm_bn_side* main_bn,
                            const void* d_x_ds, int x_ds_ld, const iswm_bn_side* ds_bn,
                            int64_t M, int C, double* d_sums, double* d_sums_ds, void* stream);
/* pass 2: d_dx = gradient w.r.t. raw, d_dx_ds = gradient w.r.t. raw_ds (bf16, own pitches); dgamma / dbeta ACCUMULATE. */
int iswm_bn_dual_bwd_apply(const void* d_dout, int dout_ld, const uint8_t* d_relu_bits,
                           const void* d_x, int x_ld, const iswm_bn_side* main_bn, const double* d_sums,
                           const void* d_x_ds, int x_ds_ld, const iswm_bn_side* ds_bn, const double* d_sums_ds,
                           int64_t M, int C, void* d_dx, int dx_ld, void* d_dx_ds, int dx_ds_ld,
                           float* d_dgamma, float* d_dbeta, float* d_dgamma_ds, float* d_dbeta_ds, void* stream);
/* Synchronised BatchNorm forms: the sides' stats (forward) and d_gsums / d_gsums_ds (backward) are double[2*C + 1] exchanged
 * sums with the global row count (iswm_syncbn_exchange; one copy); the backward adds the local sums into dgamma / dbeta. */
int iswm_bn_dual_train_apply_global(const void* d_x, int x_ld, const iswm_bn_side* main_bn,
                                    const void* d_x_ds, int x_ds_ld, const iswm_bn_side* ds_bn,
                                    int64_t M, int C, float eps, float momentum,
                                    void* d_out, int out_ld, uint8_t* d_relu_bits, void* stream);
int iswm_bn_dual_bwd_apply_global(const void* d_dout, int dout_ld, const uint8_t* d_relu_bits,
                                  const void* d_x, int x_ld, const iswm_bn_side* main_bn, const double* d_gsums, const double* d_local_sums,
                                  const void* d_x_ds, int x_ds_ld, const iswm_bn_side* ds_bn, const double* d_gsums_ds,
                                  const double* d_local_sums_ds, int64_t M, int C, void* d_dx, int dx_ld, void* d_dx_ds, int dx_ds_ld,
                                  float* d_dgamma, float* d_dbeta, float* d_dgamma_ds, float* d_dbeta_ds, void* stream);

/* ---- stem tail: BatchNorm + ReLU + 3x3/s2/p1 max pooling in ONE pass (csrc/stem_pool.cu; network/backbone/resnet.py:145-147) ----
 * d_raw bf16 [B,H,W,64] = the stem convolution's pre-BN output (with its statistics in bn->stats); writes the pooled
 * bf16 [B,Ho,Wo,64] tensor and, per pooled element, which of the 9 window positions won (uint8 [B,Ho,Wo,64], first maximum in
 * window order) - the normalised half-resolution activation is never written. bn: stats / gamma / beta read, running statistics
 * updated, save_mean / save_invstd written. */
int iswm_stem_pool_fwd(const void* d_raw, const iswm_bn_side* bn, int B, int H, int W, int C, int Ho, int Wo,
                       float eps, float momentum, void* d_out, uint8_t* d_idx, void* stream);
/* Synchronised BatchNorm form: bn->stats = double[2*64 + 1] exchanged sums with the global pixel count (one copy). */
int iswm_stem_pool_fwd_global(const void* d_raw, const iswm_bn_side* bn, int B, int H, int W, int C, int Ho, int Wo,
                              float eps, float momentum, void* d_out, uint8_t* d_idx, void* stream);

/* Stem 7x7 / stride 2 / pad 3 (network/backbone/resnet.py:144), ROW-TAP form - what the engine runs. The fp32 NCHW image is
 * unrolled along x only: d_out bf16 [2][B][Hh][Wo][kpitch], element [p][b][hh][wo][s*Cin + c] = img[b][c][2*hh + p][2*wo + s - 3]
 * (zero outside the image and in the kpitch - 7*Cin padding channels), p = row parity, Hh = ceil(H/2), Wo = ceil(W/2). The
 * convolution is then iswm_conv_igemm over that tensor with Cin = kpitch, n_img = 2*B and 7 taps r = 0..6 =
 * (dh = (r - 3 - p)/2, dw = 0, phase p = (r + 1) & 1), weights packed by iswm_pack_weights_batched mode 2 ([Cout][7][64]);
 * its weight gradient is iswm_conv_wgrad with the same descriptor ([Cout][7][kpitch] fp32) unpacked by iswm_unpack_wgrad_stem. */
int iswm_stem_rows(const float* d_img, int B, int Cin, int H, int W, int Hh, int Wo, int kpitch, void* d_out, void* stream);
int iswm_unpack_wgrad_stem(const float* d_dw, int Cout, int Cin, int ks, int kpitch, float beta, float* d_grad, void* stream);

/* NCHW fp32 image -> stem im2col matrix bf16 [B*Ho*Wo][Kpad] for the 7x7/s2/p3 conv
 * (network/backbone/resnet.py:144); column = (r*7+s)*Cin + c, zero padded to Kpad. */
int iswm_stem_im2col(const float* d_img, int B, int Cin, int H, int W, int Ho, int Wo,
                     int Kpad, void* d_out, void* stream);
/* MaxPool2d(3,2,1) (resnet.py:148), NHWC bf16; d_idx uint8 window argmax (first max wins) */
int iswm_maxpool_fwd(const void* d_x, int B, int H, int W, int C, int Ho, int Wo,
                     void* d_out, uint8_t* d_idx, void* stream);
int iswm_maxpool_bwd(const void* d_dout, const uint8_t* d_idx, int B, int H, int W, int C,
                     int Ho, int Wo, void* d_dx, void* stream);
/* AdaptiveAvgPool2d(1) (network/_deeplab.py:133): [B,HW,C] bf16 -> [B,C] bf16 */
int iswm_gap_fwd(const void* d_x, int x_ld, int B, int64_t HW, int C, void* d_out, void* stream);
/* broadcast [B,C] over HW into a channel slice (the bilinear upsample of a 1x1 map, _deeplab.py:141) */
int iswm_broadcast_hw(const void* d_x, int B, int64_t HW, int C, void* d_out, int out_ld, void* stream);
/* adjoint of broadcast (sum over HW) and of GAP (scale 1/HW, broadcast add) */
int iswm_sum_hw(const void* d_x, int x_ld, int B, int64_t HW, int C, void* d_out, void* stream);
int iswm_gap_bwd_add(const void* d_dpool, int B, int64_t HW, int C, void* d_dx, int dx_ld, void* stream);
/* F.interpolate(bilinear, align_corners=False) on NHWC bf16 (network/_deeplab.py:58) and its adjoint */
int iswm_bilinear_fwd(const void* d_x, int x_ld, int B, int Hi, int Wi, int C, int Ho, int Wo,
                      void* d_out, int out_ld, void* stream);
int iswm_bilinear_bwd(const void* d_dout, int dout_ld, int B, int Hi, int Wi, int C, int Ho, int Wo,
                      void* d_dx, int dx_ld, void* stream);
/* final upsample (network/utils.py:22): NHWC fp32 [B,h,w,C] logits -> NCHW fp32 [B,C,H,W]; and adjoint
 * NCHW fp32 dlogits -> NHWC bf16 [B,h,w,dx_ld] (channels C..dx_ld-1 zero-filled) */
int iswm_logits_up_fwd(const float* d_x, int B, int Hi, int Wi, int C, int Ho, int Wo, float* d_out, void* stream);
/* d_bias_grad (optional, float[C], ACCUMULATED into): the classifier bias gradient sum_{b,y,x} dlogits[b,c,y,x]
 * (network/_deeplab.py:51 Conv2d(256, C, 1) bias) from the same sweep over dlogits */
int iswm_logits_up_bwd(const float* d_dout, int B, int Hi, int Wi, int C, int Ho, int Wo, void* d_dx, int dx_ld,
                       float* d_bias_grad, void* stream);
/* ---- FP8 (e4m3) inference path (csrc/quant.cu, iswm_b200/quant.py) ----------------------------------------------------
 * An e4m3 activation q stands for q * s with one fp32 scale s per tensor; every conversion to e4m3 is
 * cvt.rn.satfinite(x / s) with an IEEE fp32 division.
 * iswm_pack_weight_f8: fp32 OIHW -> d_sw[o] = max_i |w[o,i]| / 448 (1 for an all-zero channel) and e4m3
 *   d_out [Cout][RS][cin_pad] = e4m3(w[o][c][t] / d_sw[o]), zero for c >= Cin; cin_pad a multiple of 128.
 * iswm_maxpool_fwd_f8: MaxPool2d(3,2,1) of bf16 NHWC [B,H,W,C] -> e4m3 [B,Ho,Wo,C] with scale s.
 * iswm_gap_fwd_f8: e4m3 [B,HW,x_ld] (scale s) -> bf16 [B,C] = (sum over HW) / HW * s.
 * iswm_broadcast_hw_f8: bf16 [B,C] -> e4m3 channel slice [B,HW,out_ld] with scale s.
 * iswm_bilinear_fwd_f8: as iswm_bilinear_fwd (generic kernel), bf16 in, e4m3 channel slice out with scale s.
 * iswm_phase_split_b8 / iswm_subsample2_b8: iswm_phase_split / iswm_subsample2 over one-byte elements (C, x_ld multiples of 16). */
int iswm_pack_weight_f8(const float* d_w, int Cout, int Cin, int RS, int cin_pad, void* d_out, float* d_sw, void* stream);
int iswm_maxpool_fwd_f8(const void* d_x, int B, int H, int W, int C, int Ho, int Wo, float s, void* d_out, void* stream);
int iswm_gap_fwd_f8(const void* d_x, int x_ld, int B, int64_t HW, int C, float s, void* d_out, void* stream);
int iswm_broadcast_hw_f8(const void* d_x, int B, int64_t HW, int C, float s, void* d_out, int out_ld, void* stream);
int iswm_bilinear_fwd_f8(const void* d_x, int x_ld, int B, int Hi, int Wi, int C, int Ho, int Wo, float s, void* d_out,
                         int out_ld, void* stream);
int iswm_phase_split_b8(const void* d_x, int x_ld, int B, int H, int W, int C, void* d_out, void* stream);
int iswm_subsample2_b8(const void* d_x, int x_ld, int B, int H, int W, int C, void* d_out, void* stream);

/* strided helpers for stride-2 convolutions */
int iswm_phase_split(const void* d_x, int x_ld, int B, int H, int W, int C, void* d_out, void* stream);   /* -> [4][B][ceil(H/2)][ceil(W/2)][C], phase = (h&1)*2 + (w&1) */
int iswm_subsample2(const void* d_x, int x_ld, int B, int H, int W, int C, void* d_out, void* stream);    /* -> [B][ceil(H/2)][ceil(W/2)][C] */
int iswm_zero_stuff2(const void* d_x, int B, int Ho, int Wo, int C, int H, int W, void* d_out, void* stream); /* out[b,2i,2j]=x[b,i,j], else 0 */
int iswm_scatter2_add(const void* d_x, int B, int Ho, int Wo, int C, int H, int W, void* d_inout, void* stream); /* inout[b,2i,2j]+=x */
/* elementwise bf16: out = a + b */
int iswm_add_bf16(const void* d_a, const void* d_b, int64_t n, void* d_out, void* stream);
/* NHWC bf16 -> NCHW fp32 (feature export for tests / API) and back */
int iswm_nhwc_to_nchw_f32(const void* d_x, int x_ld, int B, int64_t HW, int C, float* d_out, void* stream);
int iswm_nchw_f32_to_nhwc(const float* d_x, int B, int64_t HW, int C, void* d_out, int out_ld, void* stream);

/* classifier bias gradient (network/_deeplab.py:51 Conv2d(256, C, 1) bias): out[c] += sum_{b,p} d[b,c,p], NCHW fp32 */
int iswm_bias_grad_nchw(const float* d_dout, int B, int C, int64_t HW, float* d_out, void* stream);
/* x *= *d_scalar in place; a no-op pass when the device scalar is exactly 1.0 (criterion backward
 * under the implicit grad_output of loss.backward(), train.py:1048) */
int iswm_scale_by_device_scalar(void* d_x, int dtype, int64_t n, const float* d_scalar, void* stream);

/* fused multi-tensor SGD(momentum, nesterov, weight decay) step (train.py:421-431, :1049) on a flat fp32 buffer */
/* d_lr: optional DEVICE float overriding `lr` (a step replayed from a CUDA graph follows the LR schedule through it) */
int iswm_sgd_step(float* d_param, const float* d_grad, float* d_mom, int64_t n, float lr, float momentum,
                  float weight_decay, int nesterov, int first_step, const float* d_lr, void* stream);

/* fused Adam / AdamW step on a flat fp32 buffer: torch.optim.Adam(weight_decay) and torch.optim.AdamW(weight_decay)
 * as train.py:432-441 builds them (torch defaults lr 1e-3, betas (0.9, 0.999), eps 1e-8), stepped at train.py:1049.
 * adamw = 0: L2 decay added to the gradient; 1: decoupled decay. step = 1 on the first update (bias correction).
 * d_lr / d_step: optional DEVICE float / int64 overriding `lr` / `step` (CUDA-graph replays). */
int iswm_adam_step(float* d_param, const float* d_grad, float* d_exp_avg, float* d_exp_avg_sq, int64_t n,
                   float lr, float beta1, float beta2, float eps, float weight_decay, int adamw,
                   int64_t step, const float* d_lr, const int64_t* d_step, void* stream);

/* ---- the step before the hot path: device input pipeline (SURVEY 8f rank 2) ---------------- */
/* ExtRandomCrop (window origin per image, no padding) + ExtRandomHorizontalFlip + ExtToTensor + ExtNormalize
 * (utils/ext_transforms.py:327-393, :94-111, :273-293, :298-324; composed at train.py:355-368) on uint8 HWC tiles:
 *   d_src        uint8 [B,Hs,Ws,C] (C = 1..4), device
 *   d_origin_xy  int32 [B,2] = (x0, y0) of each image's H x W window, device, or NULL (0,0)
 *   d_flip       uint8 [B], non-zero = mirror the window horizontally, device, or NULL
 *   mean, stdv   HOST float[C]
 *   d_out        float32 NCHW [B,C,H,W] = ((src/255) - mean) / std, IEEE arithmetic (bit-identical to torchvision)
 * iswm_crop_flip_u8 applies the same window / flip to the uint8 label tile [B,Hs,Ws] -> [B,H,W]. */
int iswm_u8_to_f32_norm(const uint8_t* d_src, int B, int Hs, int Ws, int C, const int32_t* d_origin_xy,
                        const uint8_t* d_flip, const float* mean, const float* stdv, int H, int W,
                        float* d_out, void* stream);
int iswm_crop_flip_u8(const uint8_t* d_src, int B, int Hs, int Ws, const int32_t* d_origin_xy,
                      const uint8_t* d_flip, int H, int W, uint8_t* d_out, void* stream);

/* The reference's whole TRAIN transform (train.py:355-362) on uint8 tiles, one call:
 *   ExtRandomScale (utils/ext_transforms.py:94-111: F.resize to (int(h*s), int(w*s)), bilinear for the image, nearest for the label)
 *   -> ExtRandomCrop(pad_if_needed=True) (:366-393: zero padding on all four sides when the scaled tile is smaller than the crop, then
 *   F.crop) -> ExtRandomHorizontalFlip (:94-111 of the flip class) -> ExtToTensor -> ExtNormalize (:273-324).
 * The resampling arithmetic is Pillow's (Resample.c two-pass 8 bpc fixed point; Geometry.c ImagingScaleAffine), restated in
 * iswm_b200/csrc/scale_math.h: images and labels are BIT-IDENTICAL to the PIL pipeline for the same random draws.
 *   d_img      uint8 [B,Hs,Ws,C] (C = 1..4), device;  d_lbl uint8 [B,Hs,Ws] or NULL (then d_lbl_out NULL too)
 *   d_geom     int32 [B,8] device, one record per sample, written by the host that drew the random numbers:
 *              {sh, sw = scaled size; pad = zero padding per side; y0, x0 = crop origin in the padded tile; flip; 0; 0}
 *   kmax       taps per coefficient row, >= ceil(max(Hs/sh, Ws/sw, 1)) * 2 + 1 over the batch (3..16)
 *   tab_w/h    table capacity: >= max sw / max sh over the batch
 *   d_tables   int32 workspace, B * iswm_random_scale_table_words(tab_w, tab_h, kmax) words (coefficient rows + index tables)
 *   mean, stdv HOST float[C];  d_out float32 NCHW [B,C,H,W];  d_lbl_out uint8 [B,H,W] (padding = 0, like F.pad's default fill)
 * Three launches (plan, image, label) on `stream`. */
int64_t iswm_random_scale_table_words(int tab_w, int tab_h, int kmax);
int iswm_random_scale_crop(const uint8_t* d_img, const uint8_t* d_lbl, int B, int Hs, int Ws, int C, const int32_t* d_geom,
                           int kmax, int tab_w, int tab_h, int32_t* d_tables, const float* mean, const float* stdv,
                           int H, int W, float* d_out, uint8_t* d_lbl_out, void* stream);

/* ---- the per-frame evaluators beside the confusion matrix (SURVEY 8f rank 4): image-processing half on the device ---------
 * Integer / byte work, bit-exact against OpenCV / SciPy as the reference calls them; the float64 scalar arithmetic on top
 * (a few hundred numbers per frame) runs on the host in iswm_b200/metrics/shape_metrics.py in the reference's operation order.
 * Masks are [N,H,W] device arrays of `dtype` (ISWM_U8 / ISWM_I32 / ISWM_I64), foreground = value > 0 (mask_utils.py:14).
 * d_work: iswm_mask_work_bytes(N, H, W) bytes of device scratch. */
int64_t iswm_mask_work_bytes(int N, int H, int W);
/* MaskUtils.preprocess_mask (metrics/utils/mask_utils.py:7-52) + find_front_positions' row scan (:66-74):
 *   3x3 close, 3x3 open (cv2.morphologyEx, default border), 8-connected components with areas
 *   (cv2.connectedComponentsWithStats), largest component among those with area >= min_valid_area (the caller passes
 *   H*W*0.001 as the reference computes it), area ties to the first label in OpenCV's numbering.
 *   d_support uint8 [N,H,W]  the chosen component (all zero when there is none)
 *   d_front   int32 [N,H]    its leftmost column per row, -1 = row empty
 *   d_info    int32 [N,8]    {components, valid components, area of the chosen one, support pixels, its root pixel index, 0, 0, 0}
 * The reference's return value is support * weight with weight = 1 for <= 1 valid component, else max(0.4, 1 - 0.2 (valid - 1)). */
int iswm_mask_preprocess(const void* d_mask, int dtype, int N, int H, int W, double min_valid_area, uint8_t* d_support,
                         int32_t* d_front, int32_t* d_info, void* d_work, void* stream);
/* RegionMetrics.calculate_region_metrics (metrics/region_metrics.py:6-12 repair_small_gaps = dilate x3, erode x2 with a 3x3 box;
 * :74-92 intersection / union with the ground truth; :44-61 scipy.ndimage.label with the 8-connected structure, areas >= min_area):
 *   d_counts int32 [N,8]   {sum(pred > 0), sum(gt > 0), |repaired & gt|, |repaired | gt|, regions with area >= min_area, components, 0, 0}
 *   d_areas  int32 [N,cap] the areas of those regions, unordered (at most cap are stored; counts[4] still counts all) */
int iswm_region_components(const void* d_pred, int pred_dtype, const void* d_gt, int gt_dtype, int N, int H, int W, int min_area,
                           int cap, int32_t* d_counts, int32_t* d_areas, void* d_work, void* stream);
/* FrontTrackingMetrics.calculate_error's two nearest-point loops (metrics/front_tracking_metrics.py:48-63, :72-85): for every row i
 * with a front point (i, a[i]) the FIRST closest point (j, b[j]) in row order: d2 = squared distance (-1 = no point in this row or B is
 * empty), dx = |a[i] - b[j]|. d_front_a / d_front_b / d_d2 / d_dx int32 [N,H]. */
int iswm_front_nearest(const int32_t* d_front_a, const int32_t* d_front_b, int N, int H, int32_t* d_d2, int32_t* d_dx, void* stream);
/* MaskUtils.calculate_stability's row loop (metrics/utils/mask_utils.py:117-133): |front - x| of the first set pixel x of `d_other`
 * (uint8 [N,H,W]) inside [front - window, front + window) clipped to the row; -1 = no front in this row or nothing in the window. */
int iswm_front_window_diff(const int32_t* d_front, const uint8_t* d_other, int N, int H, int W, int window, int32_t* d_diff, void* stream);

/* ---- the train-mode tail without its full-resolution tensors (SURVEY kernels K11 + K12 + K13) ------------------------------
 * network/utils.py:22 (F.interpolate of the classifier output to the input size) + train.py:1046 (weighted CE, ignore_index,
 * mean) + train.py:1048 (their backward down to the classifier output), for 2 classes and an exact x4 upsample:
 *   iswm_tail_fwd   d_lo fp32 NHWC [B,h,w,2] low-res logits, labels [B,4h,4w] of `label_dtype` ->
 *                   d_dlo_acc fp32 [B,h,w,2] = adjoint of the upsample applied to w_y (softmax - onehot), NOT yet divided by
 *                   the normaliser; d_hist int64[2] += class counts; d_loss_num double += sum_i w_{y_i} nll_i
 *                   (the caller zeroes hist and loss_num; a data-parallel caller all-reduces d_hist before the next two calls)
 *   iswm_tail_loss  d_loss = loss_num / sum_c w_c hist_c (nan for an all-ignored batch, like torch)
 *   iswm_tail_bwd   d_dlo bf16 [B,h,w,dx_ld] = dlo_acc * (*d_gscale or 1) / sum_c w_c hist_c, channels >= 2 zero;
 *                   d_bias_grad[0] += sum, [1] -= sum (classifier bias gradient; may be NULL); d_scratch: 8200 bytes of device
 *                   memory, zero before the first call, owned by the caller (per-block partials + a self-resetting counter)
 * Same per-pixel arithmetic as iswm_logits_up_fwd + iswm_wce_fwd_bwd (identical logits and nll); the gradient differs from the
 * unfused chain only in where the 1/normaliser is applied (after the adjoint instead of before): fp32 rounding, below bf16. */
int iswm_tail_fwd(const float* d_lo, int B, int h, int w, const void* d_labels, int label_dtype, int H, int W, const float* d_weight,
                  int ignore_index, float* d_dlo_acc, int64_t* d_hist, double* d_loss_num, void* stream);
int iswm_tail_loss(const double* d_loss_num, const float* d_weight, const int64_t* d_hist, int ignore_index, float* d_loss, void* stream);
int iswm_tail_bwd(const float* d_dlo_acc, int B, int h, int w, const float* d_weight, const int64_t* d_hist, int ignore_index,
                  const float* d_gscale, void* d_dlo, int dx_ld, float* d_bias_grad, void* d_scratch, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* ISWM_B200_H */
