"""Tensor-level wrappers over the C ABI (include/iswm_b200.h).

Each function takes CUDA torch tensors, passes raw device pointers + sizes + the current
CUDA stream to libiswm_b200.so, and raises on any error. PyTorch is used for memory and
streams only. There is no fallback path: a CPU tensor or a missing library is an error.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import ConvDesc, check

_LABEL_CODE = {torch.uint8: _lib.U8, torch.int32: _lib.I32, torch.int64: _lib.I64}
_FLOAT_CODE = {torch.float32: _lib.F32, torch.bfloat16: _lib.BF16}


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("iswm_b200 ops need CUDA tensors (no CPU fallback exists)")
    return t.data_ptr()


def _label_code(t: torch.Tensor) -> int:
    try:
        return _LABEL_CODE[t.dtype]
    except KeyError:
        raise TypeError(f"label dtype {t.dtype} not supported (uint8/int32/int64)") from None


# ----------------------------------------------------------------------------- loss / metric

def class_hist(labels: torch.Tensor, n_classes: int, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """int64[n_classes] pixel counts; accumulates into `out` when given (train.py:401-402)."""
    labels = labels.contiguous()
    if out is None:
        out = torch.zeros(n_classes, dtype=torch.int64, device=labels.device)
    check(_lib.lib().iswm_class_hist(_ptr(labels), _label_code(labels), labels.numel(), n_classes,
                                     _ptr(out), _stream()), "class_hist")
    return out


def wce_fwd_bwd(logits: torch.Tensor, labels: torch.Tensor, weight: Optional[torch.Tensor],
                hist: torch.Tensor, ignore_index: int = 255, grad_scale: float = 1.0,
                want_grad: bool = True) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """Fused weighted CE forward(+backward). Returns (loss[0-dim fp32], dlogits or None)."""
    assert logits.dim() >= 2
    logits = logits.contiguous()
    labels = labels.contiguous()
    B, Cc = logits.shape[0], logits.shape[1]
    HW = logits.numel() // max(1, B * Cc)
    if labels.numel() != B * HW:
        raise ValueError(f"labels {tuple(labels.shape)} do not match logits {tuple(logits.shape)}")
    grad = torch.empty_like(logits) if want_grad else None
    num = torch.zeros(1, dtype=torch.float64, device=logits.device)
    loss = torch.empty((), dtype=torch.float32, device=logits.device)
    w = None if weight is None else weight.to(device=logits.device, dtype=torch.float32).contiguous()
    check(_lib.lib().iswm_wce_fwd_bwd(_ptr(logits), _FLOAT_CODE[logits.dtype], _ptr(labels),
                                      _label_code(labels), _ptr(w), _ptr(hist), B, Cc, HW,
                                      ignore_index, grad_scale, _ptr(grad), _ptr(num), _ptr(loss),
                                      _stream()), "wce_fwd_bwd")
    return loss, grad


def confusion(true: torch.Tensor, pred: torch.Tensor, n_classes: int,
              out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """int64[n*n+1] confusion counts (last slot: predictions outside [0,n))."""
    true = true.contiguous()
    pred = pred.contiguous()
    if true.numel() != pred.numel():
        raise ValueError("true / pred size mismatch")
    if out is None:
        out = torch.zeros(n_classes * n_classes + 1, dtype=torch.int64, device=true.device)
    check(_lib.lib().iswm_confusion(_ptr(true), _label_code(true), _ptr(pred), _label_code(pred),
                                    true.numel(), n_classes, _ptr(out), _stream()), "confusion")
    return out


def argmax_confusion(logits: torch.Tensor, true: Optional[torch.Tensor], mode: int = 0,
                     threshold: float = 0.5, want_pred: bool = False, want_conf: bool = False,
                     out: Optional[torch.Tensor] = None):
    logits = logits.contiguous()
    B, Cc = logits.shape[0], logits.shape[1]
    HW = logits.numel() // max(1, B * Cc)
    dev = logits.device
    pred = torch.empty((B,) + tuple(logits.shape[2:]), dtype=torch.uint8, device=dev) if want_pred else None
    conf = torch.empty((B,) + tuple(logits.shape[2:]), dtype=torch.uint8, device=dev) if want_conf else None
    if true is not None:
        true = true.contiguous()
        if out is None:
            out = torch.zeros(Cc * Cc + 1, dtype=torch.int64, device=dev)
    check(_lib.lib().iswm_argmax_confusion(_ptr(logits), _FLOAT_CODE[logits.dtype], _ptr(true),
                                           _label_code(true) if true is not None else _lib.I64,
                                           B, Cc, HW, mode, threshold, _ptr(pred), _ptr(conf),
                                           _ptr(out) if true is not None else None, _stream()),
          "argmax_confusion")
    return out, pred, conf


def predict_epilogue(lo: torch.Tensor, H: int, W: int, true: Optional[torch.Tensor] = None, mode: int = 1,
                     threshold: float = 0.5, want_pred: bool = True, want_conf: bool = True,
                     out: Optional[torch.Tensor] = None):
    """Fused final upsample + softmax/threshold + uint8 maps (+ confusion counts) from the LOW-resolution fp32 NHWC
    logits [B,h,w,2] (network/utils.py:22 + predict.py:262-290). Returns (cm or None, pred, conf)."""
    if lo.dtype != torch.float32 or lo.dim() != 4:
        raise TypeError("predict_epilogue wants fp32 NHWC [B,h,w,C] low-resolution logits")
    lo = lo.contiguous()
    B, Hi, Wi, Cc = lo.shape
    dev = lo.device
    pred = torch.empty((B, H, W), dtype=torch.uint8, device=dev) if want_pred else None
    conf = torch.empty((B, H, W), dtype=torch.uint8, device=dev) if want_conf else None
    if true is not None:
        true = true.contiguous()
        if true.numel() != B * H * W:
            raise ValueError(f"labels {tuple(true.shape)} do not match the {B}x{H}x{W} output")
        if out is None:
            out = torch.zeros(Cc * Cc + 1, dtype=torch.int64, device=dev)
    check(_lib.lib().iswm_predict_epilogue(_ptr(lo), B, Hi, Wi, Cc, H, W, mode, threshold, _ptr(true),
                                           _label_code(true) if true is not None else _lib.I64, _ptr(pred), _ptr(conf),
                                           _ptr(out) if true is not None else None, _stream()), "predict_epilogue")
    return (out if true is not None else None), pred, conf


def resize_flip_f32(x: torch.Tensor, size: Tuple[int, int], flip: bool = False, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """fp32 NCHW [B,C,H,W] -> [B,C,*size]: F.interpolate(bilinear, align_corners=False) then .flip(-1) when `flip`; an exact
    (mirrored) copy when `size` is the input's. `out` may be a contiguous batch slice of a larger buffer."""
    if x.dtype != torch.float32 or x.dim() != 4:
        raise TypeError("resize_flip_f32 wants fp32 NCHW [B,C,H,W]")
    x = x.contiguous()
    B, Cc, Hi, Wi = x.shape
    Ho, Wo = size
    if out is None:
        out = torch.empty((B, Cc, Ho, Wo), dtype=torch.float32, device=x.device)
    if tuple(out.shape) != (B, Cc, Ho, Wo) or out.dtype != torch.float32 or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous fp32 [{B},{Cc},{Ho},{Wo}] tensor")
    check(_lib.lib().iswm_resize_flip_f32(_ptr(x), B, Cc, Hi, Wi, Ho, Wo, 1 if flip else 0, _ptr(out), _stream()), "resize_flip_f32")
    return out


def predict_tta_epilogue(views: Sequence[Tuple[torch.Tensor, Tuple[int, int], bool]], H: int, W: int,
                         true: Optional[torch.Tensor] = None, mode: int = 1, threshold: float = 0.5,
                         out: Optional[torch.Tensor] = None, pred: Optional[torch.Tensor] = None,
                         conf: Optional[torch.Tensor] = None):
    """Multi-view form of predict_epilogue (test-time augmentation): `views` lists (lo, (Hv, Wv), flip) with lo the fp32
    NHWC [B,h,w,2] low-resolution logits of the network run on a view of full-resolution size (Hv, Wv), mirrored when
    `flip`. Writes the uint8 maps of the view-averaged softmax at [B,H,W] (into `pred` / `conf` when given, e.g. batch
    slices of larger maps) and accumulates the confusion counts into `out`. Returns (cm or None, pred, conf)."""
    if not views:
        raise ValueError("predict_tta_epilogue needs at least one view")
    arr = (_lib.TtaView * len(views))()
    keep = []
    B = Cc = None
    for i, (lo, (Hv, Wv), flip) in enumerate(views):
        if lo.dtype != torch.float32 or lo.dim() != 4:
            raise TypeError("predict_tta_epilogue wants fp32 NHWC [B,h,w,C] low-resolution logits")
        lo = lo.contiguous()
        keep.append(lo)
        if B is None:
            B, Cc = lo.shape[0], lo.shape[3]
        elif (lo.shape[0], lo.shape[3]) != (B, Cc):
            raise ValueError("every view needs the same batch and class count")
        arr[i].lo, arr[i].Hi, arr[i].Wi, arr[i].Hv, arr[i].Wv, arr[i].flip = _ptr(lo), lo.shape[1], lo.shape[2], Hv, Wv, int(bool(flip))
    dev = keep[0].device
    for name, t in (("pred", pred), ("conf", conf)):
        if t is not None and (tuple(t.shape) != (B, H, W) or t.dtype != torch.uint8 or not t.is_contiguous()):
            raise ValueError(f"{name} must be a contiguous uint8 [{B},{H},{W}] tensor")
    pred = torch.empty((B, H, W), dtype=torch.uint8, device=dev) if pred is None else pred
    conf = torch.empty((B, H, W), dtype=torch.uint8, device=dev) if conf is None else conf
    if true is not None:
        true = true.contiguous()
        if true.numel() != B * H * W:
            raise ValueError(f"labels {tuple(true.shape)} do not match the {B}x{H}x{W} output")
        if out is None:
            out = torch.zeros(Cc * Cc + 1, dtype=torch.int64, device=dev)
    check(_lib.lib().iswm_predict_tta_epilogue(arr, len(views), B, Cc, H, W, mode, threshold, _ptr(true),
                                               _label_code(true) if true is not None else _lib.I64, _ptr(pred), _ptr(conf),
                                               _ptr(out) if true is not None else None, _stream()), "predict_tta_epilogue")
    return (out if true is not None else None), pred, conf


def window_offsets(L: int, window: int, stride: int) -> Tuple[int, List[int]]:
    """Window placement along an axis of length L (the rule of csrc/window.cu's WinAxis): the side w = min(window, L)
    and the offsets min(i * stride, L - w) of the ceil((L - w) / stride) + 1 windows, the last one snapped to the border.
    A stride above the window would leave pixels uncovered."""
    if window < 1 or not 1 <= stride <= window:
        raise ValueError(f"window {window}, stride {stride}: need 1 <= stride <= window")
    w = min(window, L)
    return w, [min(i * stride, L - w) for i in range((L - w + stride - 1) // stride + 1)]


def window_gather_f32(x: torch.Tensor, window: Tuple[int, int], stride: Tuple[int, int], first: int = 0,
                      n: Optional[int] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """fp32 NCHW [B,C,H,W] -> windows [first, first+n) of the batch's window list (image-major, then row-major over the
    window grid) as [n,C,wh,ww], copied exactly; (wh, ww) is `window` clamped to the scene. `out` may be a contiguous
    batch slice of a larger buffer."""
    if x.dtype != torch.float32 or x.dim() != 4:
        raise TypeError("window_gather_f32 wants fp32 NCHW [B,C,H,W]")
    x = x.contiguous()
    B, Cc, H, W = x.shape
    (wh, ys), (ww, xs) = window_offsets(H, window[0], stride[0]), window_offsets(W, window[1], stride[1])
    total = B * len(ys) * len(xs)
    n = total - first if n is None else n
    if first < 0 or n < 0 or first + n > total:
        raise ValueError(f"windows [{first}, {first + n}) outside the {total} windows of the batch")
    if out is None:
        out = torch.empty((n, Cc, wh, ww), dtype=torch.float32, device=x.device)
    if tuple(out.shape) != (n, Cc, wh, ww) or out.dtype != torch.float32 or not out.is_contiguous():
        raise ValueError(f"out must be a contiguous fp32 [{n},{Cc},{wh},{ww}] tensor")
    check(_lib.lib().iswm_window_gather_f32(_ptr(x), B, Cc, H, W, window[0], window[1], stride[0], stride[1], first, n,
                                            _ptr(out), _stream()), "window_gather_f32")
    return out


def predict_window_epilogue(lo: torch.Tensor, H: int, W: int, window: Tuple[int, int], stride: Tuple[int, int],
                            true: Optional[torch.Tensor] = None, threshold: float = 0.5, out: Optional[torch.Tensor] = None,
                            pred: Optional[torch.Tensor] = None, conf: Optional[torch.Tensor] = None):
    """Sliding-window form of predict_epilogue: `lo` is fp32 NHWC [B*ny*nx,h,w,2], the low-resolution logits of every
    window of B scenes of [H,W] in window_gather_f32's order. Writes the uint8 maps of the softmax averaged over the
    windows covering each pixel at [B,H,W] (threshold mode; into `pred` / `conf` when given) and accumulates the
    confusion counts into `out`. Returns (cm or None, pred, conf)."""
    if lo.dtype != torch.float32 or lo.dim() != 4:
        raise TypeError("predict_window_epilogue wants fp32 NHWC [N,h,w,C] low-resolution logits")
    lo = lo.contiguous()
    N, hi, wi, Cc = lo.shape
    per_img = len(window_offsets(H, window[0], stride[0])[1]) * len(window_offsets(W, window[1], stride[1])[1])
    if N % per_img:
        raise ValueError(f"{N} windows of logits are not a whole number of {H}x{W} scenes of {per_img} windows")
    B = N // per_img
    dev = lo.device
    for name, t in (("pred", pred), ("conf", conf)):
        if t is not None and (tuple(t.shape) != (B, H, W) or t.dtype != torch.uint8 or not t.is_contiguous()):
            raise ValueError(f"{name} must be a contiguous uint8 [{B},{H},{W}] tensor")
    pred = torch.empty((B, H, W), dtype=torch.uint8, device=dev) if pred is None else pred
    conf = torch.empty((B, H, W), dtype=torch.uint8, device=dev) if conf is None else conf
    if true is not None:
        true = true.contiguous()
        if true.numel() != B * H * W:
            raise ValueError(f"labels {tuple(true.shape)} do not match the {B}x{H}x{W} output")
        if out is None:
            out = torch.zeros(Cc * Cc + 1, dtype=torch.int64, device=dev)
    check(_lib.lib().iswm_predict_window_epilogue(_ptr(lo), B, H, W, window[0], window[1], stride[0], stride[1], hi, wi, Cc,
                                                  threshold, _ptr(true), _label_code(true) if true is not None else _lib.I64,
                                                  _ptr(pred), _ptr(conf), _ptr(out) if true is not None else None, _stream()),
          "predict_window_epilogue")
    return (out if true is not None else None), pred, conf


def focal_fwd_bwd(logits: torch.Tensor, labels: torch.Tensor, weight: Optional[torch.Tensor], alpha: float = 1.0,
                  gamma: float = 0.0, size_average: bool = True, ignore_index: int = 255,
                  want_grad: bool = True) -> Tuple[torch.Tensor, Optional[torch.Tensor]]:
    """Fused focal loss forward(+backward) (utils/loss.py:14-35). Returns (loss[0-dim fp32], dlogits or None)."""
    logits = logits.contiguous()
    labels = labels.contiguous()
    B, Cc = logits.shape[0], logits.shape[1]
    HW = logits.numel() // max(1, B * Cc)
    if labels.numel() != B * HW:
        raise ValueError(f"labels {tuple(labels.shape)} do not match logits {tuple(logits.shape)}")
    grad = torch.empty_like(logits) if want_grad else None
    num = torch.zeros(1, dtype=torch.float64, device=logits.device)
    loss = torch.empty((), dtype=torch.float32, device=logits.device)
    w = None if weight is None else weight.to(device=logits.device, dtype=torch.float32).contiguous()
    check(_lib.lib().iswm_focal_fwd_bwd(_ptr(logits), _FLOAT_CODE[logits.dtype], _ptr(labels), _label_code(labels), _ptr(w),
                                        B, Cc, HW, ignore_index, float(alpha), float(gamma), 1 if size_average else 0,
                                        _ptr(grad), _ptr(num), _ptr(loss), _stream()), "focal_fwd_bwd")
    return loss, grad


def u8_to_f32_norm(src: torch.Tensor, mean: Sequence[float], std: Sequence[float], size: Optional[Tuple[int, int]] = None,
                   origin_xy: Optional[torch.Tensor] = None, flip: Optional[torch.Tensor] = None,
                   out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 [B,Hs,Ws,C] tiles -> float32 NCHW [B,C,H,W] = ((src/255) - mean) / std over an optional per-image
    window (origin_xy int32 [B,2]) and horizontal flip (uint8 [B]) (utils/ext_transforms.py:94-111, :273-393)."""
    if src.dtype != torch.uint8 or src.dim() != 4:
        raise TypeError("u8_to_f32_norm wants uint8 [B,H,W,C] tiles")
    src = src.contiguous()
    B, Hs, Ws, Cc = src.shape
    H, W = size if size is not None else (Hs, Ws)
    if len(mean) != Cc or len(std) != Cc:
        raise ValueError("mean / std need one value per channel")
    if out is None:
        out = torch.empty((B, Cc, H, W), dtype=torch.float32, device=src.device)
    mu = (C.c_float * Cc)(*[float(v) for v in mean])
    sd = (C.c_float * Cc)(*[float(v) for v in std])
    check(_lib.lib().iswm_u8_to_f32_norm(_ptr(src), B, Hs, Ws, Cc, _ptr(origin_xy), _ptr(flip), mu, sd, H, W, _ptr(out),
                                         _stream()), "u8_to_f32_norm")
    return out


def crop_flip_u8(src: torch.Tensor, size: Optional[Tuple[int, int]] = None, origin_xy: Optional[torch.Tensor] = None,
                 flip: Optional[torch.Tensor] = None, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """uint8 label tiles [B,Hs,Ws] -> [B,H,W] under the same window / flip as u8_to_f32_norm."""
    if src.dtype != torch.uint8 or src.dim() != 3:
        raise TypeError("crop_flip_u8 wants uint8 [B,H,W] label tiles")
    src = src.contiguous()
    B, Hs, Ws = src.shape
    H, W = size if size is not None else (Hs, Ws)
    if out is None:
        out = torch.empty((B, H, W), dtype=torch.uint8, device=src.device)
    check(_lib.lib().iswm_crop_flip_u8(_ptr(src), B, Hs, Ws, _ptr(origin_xy), _ptr(flip), H, W, _ptr(out), _stream()), "crop_flip_u8")
    return out


def random_scale_kmax(Hs: int, Ws: int, geom) -> int:
    """Taps per coefficient row iswm_random_scale_crop needs for a batch of geometry records (host int array [B,8]):
    Pillow's ksize = ceil(max(in / out, 1)) * 2 + 1, the largest over both axes and all samples."""
    k = 3
    for g in geom:
        sh, sw = int(g[0]), int(g[1])
        if sh < 1 or sw < 1:
            raise ValueError(f"scaled size {sh}x{sw}: the scale collapses the tile")
        for n_in, n_out in ((Hs, sh), (Ws, sw)):
            fs = max(float(n_in) / n_out, 1.0)
            c = int(fs)
            k = max(k, (c + (1 if c < fs else 0)) * 2 + 1)
    return k


def random_scale_crop(img: torch.Tensor, lbl: Optional[torch.Tensor], geom: torch.Tensor, size: Tuple[int, int],
                      mean: Sequence[float], std: Sequence[float], kmax: int, tab_hw: Tuple[int, int],
                      tables: Optional[torch.Tensor] = None):
    """ExtRandomScale -> ExtRandomCrop(pad_if_needed) -> ExtRandomHorizontalFlip -> ExtToTensor -> ExtNormalize
    (train.py:355-362) on uint8 tiles [B,Hs,Ws,C] (+ uint8 labels [B,Hs,Ws]): float32 [B,C,H,W] and uint8 [B,H,W],
    bit-identical to the PIL pipeline for the draws in `geom` (int32 [B,8] on the device, see include/iswm_b200.h)."""
    if img.dtype != torch.uint8 or img.dim() != 4:
        raise TypeError("random_scale_crop wants uint8 [B,H,W,C] tiles")
    if lbl is not None and (lbl.dtype != torch.uint8 or lbl.dim() != 3 or lbl.shape != img.shape[:3]):
        raise TypeError("random_scale_crop wants uint8 [B,H,W] labels of the image's size")
    if geom.dtype != torch.int32 or geom.dim() != 2 or geom.shape[1] != 8 or geom.shape[0] != img.shape[0] or not geom.is_cuda:
        raise TypeError("random_scale_crop wants an int32 [B,8] device geometry tensor")
    img = img.contiguous()
    lbl = None if lbl is None else lbl.contiguous()
    geom = geom.contiguous()
    B, Hs, Ws, Cc = img.shape
    H, W = size
    if len(mean) != Cc or len(std) != Cc:
        raise ValueError("mean / std need one value per channel")
    tab_h, tab_w = tab_hw
    words = int(_lib.lib().iswm_random_scale_table_words(tab_w, tab_h, kmax)) * max(B, 1)
    if tables is None or tables.numel() < words:
        tables = torch.empty(words, dtype=torch.int32, device=img.device)
    out = torch.empty((B, Cc, H, W), dtype=torch.float32, device=img.device)
    lout = None if lbl is None else torch.empty((B, H, W), dtype=torch.uint8, device=img.device)
    mu = (C.c_float * Cc)(*[float(v) for v in mean])
    sd = (C.c_float * Cc)(*[float(v) for v in std])
    check(_lib.lib().iswm_random_scale_crop(_ptr(img), _ptr(lbl), B, Hs, Ws, Cc, _ptr(geom), kmax, tab_w, tab_h, _ptr(tables), mu, sd,
                                            H, W, _ptr(out), _ptr(lout), _stream()), "random_scale_crop")
    return out, lout, tables


# ----------------------------------------------------------------------------- shape / front evaluators (SURVEY 8f rank 4)

_MASK_DTYPES = {torch.uint8: _lib.U8, torch.int32: _lib.I32, torch.int64: _lib.I64}


def _mask3(m: torch.Tensor) -> torch.Tensor:
    if m.dtype not in _MASK_DTYPES:
        raise TypeError(f"mask dtype {m.dtype}: uint8, int32 or int64")
    if m.dim() == 2:
        m = m.unsqueeze(0)
    if m.dim() != 3:
        raise TypeError("masks are [H,W] or [N,H,W]")
    return m.contiguous()


def _mask_work(N: int, H: int, W: int, device) -> torch.Tensor:
    return torch.empty(int(_lib.lib().iswm_mask_work_bytes(N, H, W)), dtype=torch.uint8, device=device)


def mask_preprocess(mask: torch.Tensor, min_valid_area: Optional[float] = None):
    """MaskUtils.preprocess_mask + the front scan (metrics/utils/mask_utils.py:7-76) for [N,H,W] masks: returns
    (support uint8 [N,H,W], front int32 [N,H], info int32 [N,8]) on the device, see include/iswm_b200.h."""
    m = _mask3(mask)
    N, H, W = m.shape
    support = torch.empty((N, H, W), dtype=torch.uint8, device=m.device)
    front = torch.empty((N, H), dtype=torch.int32, device=m.device)
    info = torch.empty((N, 8), dtype=torch.int32, device=m.device)
    thr = (H * W) * 0.001 if min_valid_area is None else float(min_valid_area)
    check(_lib.lib().iswm_mask_preprocess(_ptr(m), _MASK_DTYPES[m.dtype], N, H, W, thr, _ptr(support), _ptr(front), _ptr(info),
                                          _ptr(_mask_work(N, H, W, m.device)), _stream()), "mask_preprocess")
    return support, front, info


def region_components(pred: torch.Tensor, gt: torch.Tensor, min_area: int = 50, cap: int = 1024):
    """RegionMetrics' image half (metrics/region_metrics.py:6-12, :44-61, :74-92): (counts int32 [N,8], areas int32 [N,cap])."""
    p, g = _mask3(pred), _mask3(gt)
    if p.shape != g.shape:
        raise ValueError("prediction and ground truth differ in shape")
    if g.dtype != p.dtype:
        g = g.to(p.dtype)
    N, H, W = p.shape
    counts = torch.empty((N, 8), dtype=torch.int32, device=p.device)
    areas = torch.zeros((N, cap), dtype=torch.int32, device=p.device)
    check(_lib.lib().iswm_region_components(_ptr(p), _MASK_DTYPES[p.dtype], _ptr(g), _MASK_DTYPES[g.dtype], N, H, W, int(min_area), cap,
                                            _ptr(counts), _ptr(areas), _ptr(_mask_work(N, H, W, p.device)), _stream()), "region_components")
    return counts, areas


def front_nearest(front_a: torch.Tensor, front_b: torch.Tensor):
    """First closest front point of B for every front point of A (metrics/front_tracking_metrics.py:48-63): (d2, dx) int32 [N,H]."""
    a, b = front_a.contiguous(), front_b.contiguous()
    if a.dtype != torch.int32 or b.dtype != torch.int32 or a.shape != b.shape or a.dim() != 2:
        raise TypeError("front_nearest wants two int32 [N,H] front tables")
    d2, dx = torch.empty_like(a), torch.empty_like(a)
    check(_lib.lib().iswm_front_nearest(_ptr(a), _ptr(b), a.shape[0], a.shape[1], _ptr(d2), _ptr(dx), _stream()), "front_nearest")
    return d2, dx


def front_window_diff(front: torch.Tensor, other: torch.Tensor, window: int) -> torch.Tensor:
    """Row loop of MaskUtils.calculate_stability (metrics/utils/mask_utils.py:117-133): int32 [N,H], -1 = no score for the row."""
    f, o = front.contiguous(), other.contiguous()
    if f.dtype != torch.int32 or o.dtype != torch.uint8 or o.dim() != 3 or f.shape != o.shape[:2]:
        raise TypeError("front_window_diff wants int32 [N,H] fronts and uint8 [N,H,W] masks")
    diff = torch.empty_like(f)
    check(_lib.lib().iswm_front_window_diff(_ptr(f), _ptr(o), o.shape[0], o.shape[1], o.shape[2], int(window), _ptr(diff), _stream()),
          "front_window_diff")
    return diff


# ----------------------------------------------------------------------------- fused train tail (K11 + K12 + K13)

def tail_fwd(lo: torch.Tensor, labels: torch.Tensor, weight: Optional[torch.Tensor], ignore_index: int = 255):
    """Upsample x4 + weighted CE + adjoint of the upsample from the classifier's fp32 NHWC [B,h,w,2] output (network/utils.py:22,
    train.py:1046-1048): returns (dlo_acc fp32 [B,h,w,2] - unnormalised -, hist int64 [2], loss_num float64 [1])."""
    if lo.dtype != torch.float32 or lo.dim() != 4 or lo.shape[3] != 2:
        raise TypeError("tail_fwd wants fp32 NHWC [B,h,w,2] low-resolution logits")
    B, h, w, _ = lo.shape
    if labels.dim() != 3 or tuple(labels.shape) != (B, 4 * h, 4 * w):
        raise ValueError(f"tail_fwd: labels {tuple(labels.shape)} are not the x4 grid of {tuple(lo.shape)}")
    lo, labels = lo.contiguous(), labels.contiguous()
    dlo_acc = torch.empty_like(lo)
    hist = torch.zeros(2, dtype=torch.int64, device=lo.device)
    num = torch.zeros(1, dtype=torch.float64, device=lo.device)
    check(_lib.lib().iswm_tail_fwd(_ptr(lo), B, h, w, _ptr(labels), _label_code(labels), 4 * h, 4 * w, _ptr(weight), int(ignore_index),
                                   _ptr(dlo_acc), _ptr(hist), _ptr(num), _stream()), "tail_fwd")
    return dlo_acc, hist, num


def tail_loss(loss_num: torch.Tensor, weight: Optional[torch.Tensor], hist: torch.Tensor, ignore_index: int = 255) -> torch.Tensor:
    loss = torch.empty((), dtype=torch.float32, device=hist.device)
    check(_lib.lib().iswm_tail_loss(_ptr(loss_num), _ptr(weight), _ptr(hist), int(ignore_index), _ptr(loss), _stream()), "tail_loss")
    return loss


def tail_bwd(dlo_acc: torch.Tensor, weight: Optional[torch.Tensor], hist: torch.Tensor, ignore_index: int, gscale: Optional[torch.Tensor],
             dlo: torch.Tensor, bias_grad: Optional[torch.Tensor], scratch: torch.Tensor) -> None:
    """dlo (bf16 [B,h,w,ldp]) = dlo_acc * gscale / sum_c w_c hist_c, bias_grad[0] += sum, [1] -= sum; `scratch`: >= 8200 zeroed bytes."""
    B, h, w, _ = dlo_acc.shape
    if dlo.dtype != torch.bfloat16 or tuple(dlo.shape[:3]) != (B, h, w) or not dlo.is_contiguous() or scratch.numel() * scratch.element_size() < 8200:
        raise TypeError("tail_bwd: bad dlo / scratch")
    check(_lib.lib().iswm_tail_bwd(_ptr(dlo_acc), B, h, w, _ptr(weight), _ptr(hist), int(ignore_index), _ptr(gscale), _ptr(dlo), dlo.shape[3],
                                   _ptr(bias_grad), _ptr(scratch), _stream()), "tail_bwd")


# ----------------------------------------------------------------------------- convolution

def make_conv_desc(B: int, Hi: int, Wi: int, Cin: int, in_ld: int, n_img: int, Ho: int, Wo: int,
                   Cout: int, out_ld: int, taps: Sequence[Tuple[int, int, int]], flags: int = 0,
                   res_ld: int = 0, wtaps: Optional[Sequence[int]] = None,
                   out_strides: Optional[Tuple[int, int, int]] = None, w_ntaps: int = 0, phase_view: bool = False) -> ConvDesc:
    d = ConvDesc()
    d.B, d.Hi, d.Wi, d.Cin, d.in_ld, d.n_img = B, Hi, Wi, Cin, in_ld, n_img
    d.Ho, d.Wo, d.Cout, d.out_ld, d.res_ld = Ho, Wo, Cout, out_ld, res_ld
    d.ntaps = len(taps)
    if d.ntaps > _lib.MAX_TAPS:
        raise ValueError("too many taps")
    for i, tap in enumerate(taps):                    # (dh, dw, phase) or (dh, dw, phase, channel offset)
        d.dh[i], d.dw[i], d.phase[i] = tap[0], tap[1], tap[2]
        d.coff[i] = tap[3] if len(tap) > 3 else 0
        d.wtap[i] = 0 if wtaps is None else wtaps[i] + 1
    d.flags = flags
    d.w_ntaps = w_ntaps
    d.in_phase_view = 1 if phase_view else 0         # x is the dense [B, 2Hi, 2Wi, ld] tensor, read as its four parity phases in place
    if out_strides is not None:                      # (w, h, image) element strides of a strided output view
        d.out_ws, d.out_hs, d.out_bs = out_strides
    return d


def conv_igemm(desc: ConvDesc, x: torch.Tensor, wgt: torch.Tensor, out: torch.Tensor,
               scale: Optional[torch.Tensor] = None, shift: Optional[torch.Tensor] = None,
               res: Optional[torch.Tensor] = None, stats: Optional[torch.Tensor] = None) -> None:
    check(_lib.lib().iswm_conv_igemm(C.byref(desc), _ptr(x), _ptr(wgt), _ptr(out), _ptr(scale),
                                     _ptr(shift), _ptr(res), _ptr(stats), _stream()), "conv_igemm")


def aspp_bwd(dycat: torch.Tensor, wcat: torch.Tensor, rates: Sequence[int], dfeat: torch.Tensor, accumulate: bool = False) -> None:
    """K-concatenated data gradient of the four ASPP conv branches (iswm_aspp_bwd): dycat bf16 [B,H,W,4*Cb], wcat the concatenated
    dgrad operand [Cfeat][28][Cb], dfeat bf16 [B,H,W,Cfeat] written (or accumulated into)."""
    B, H, W, C4 = dycat.shape
    r = (C.c_int * 3)(*[int(v) for v in rates])
    check(_lib.lib().iswm_aspp_bwd(_ptr(dycat), dycat.stride(2), _ptr(wcat), B, H, W, C4 // 4, dfeat.shape[-1], r, _ptr(dfeat),
                                   dfeat.stride(2), 1 if accumulate else 0, _stream()), "aspp_bwd")


def conv_wgrad_grouped(jobs, stream: Optional[int] = None) -> None:
    """jobs: sequence of (ConvDesc, x, dy, dw) - the weight gradients of several convolutions in ONE launch (iswm_conv_wgrad_grouped)."""
    n = len(jobs)
    descs = (ConvDesc * n)(*[j[0] for j in jobs])
    P = C.c_void_p * n
    xin, dys, dws = P(*[j[1].data_ptr() for j in jobs]), P(*[j[2].data_ptr() for j in jobs]), P(*[j[3].data_ptr() for j in jobs])
    check(_lib.lib().iswm_conv_wgrad_grouped(descs, xin, dys, dws, n, _stream() if stream is None else stream), "conv_wgrad_grouped")


def conv_wgrad(desc: ConvDesc, x: torch.Tensor, dy: torch.Tensor, dw: torch.Tensor) -> None:
    check(_lib.lib().iswm_conv_wgrad(C.byref(desc), _ptr(x), _ptr(dy), _ptr(dw), _stream()), "conv_wgrad")


def pack_weight_fwd(w: torch.Tensor, out: Optional[torch.Tensor] = None, stem: bool = False) -> torch.Tensor:
    """fp32 OIHW -> packed bf16 forward operand [Cout][R*S][cin_pad] (or the stem's [Cout][K192])."""
    w = w.contiguous()
    Cout, Cin, R, S = w.shape
    RS = R * S
    if stem:
        cin_pad, row_ld = Cin, ((RS * Cin + 63) // 64) * 64
    else:
        cin_pad = ((Cin + 63) // 64) * 64
        row_ld = RS * cin_pad
    if out is None:
        out = torch.empty(Cout * row_ld, dtype=torch.bfloat16, device=w.device)
    check(_lib.lib().iswm_pack_weight_fwd(_ptr(w), Cout, Cin, RS, cin_pad, row_ld, _ptr(out), _stream()),
          "pack_weight_fwd")
    return out


def pack_weight_dgrad(w: torch.Tensor, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """fp32 OIHW -> packed bf16 dgrad operand [Cin][R*S][cout_pad]."""
    w = w.contiguous()
    Cout, Cin, R, S = w.shape
    cout_pad = ((Cout + 63) // 64) * 64
    if out is None:
        out = torch.empty(Cin * R * S * cout_pad, dtype=torch.bfloat16, device=w.device)
    check(_lib.lib().iswm_pack_weight_dgrad(_ptr(w), Cout, Cin, R * S, cout_pad, _ptr(out), _stream()),
          "pack_weight_dgrad")
    return out


def unpack_wgrad(dw: torch.Tensor, grad_oihw: torch.Tensor, beta: float = 0.0, stem_row_ld: int = 0) -> None:
    Cout, Cin, R, S = grad_oihw.shape
    RS = R * S
    if stem_row_ld:
        cin_stride, row_ld = Cin, stem_row_ld
    else:
        cin_stride, row_ld = Cin, RS * Cin
    check(_lib.lib().iswm_unpack_wgrad(_ptr(dw), Cout, Cin, RS, cin_stride, row_ld, beta,
                                       _ptr(grad_oihw), _stream()), "unpack_wgrad")


def conv_taps(k: int, dilation: int) -> list:
    """Tap offsets of a stride-1 k x k convolution with padding = dilation*(k//2)."""
    h = k // 2
    return [((r - h) * dilation, (s - h) * dilation, 0) for r in range(k) for s in range(k)]


def conv_taps_s2_3x3() -> list:
    """Taps of a 3x3 / stride 2 / pad 1 convolution over the 4 parity phases of its input."""
    def split(r):  # input row 2i + r - 1 -> (phase parity, offset in the phase image)
        return (1, -1) if r == 0 else ((0, 0) if r == 1 else (1, 0))
    taps = []
    for r in range(3):
        p, dh = split(r)
        for s in range(3):
            q, dw = split(s)
            taps.append((dh, dw, p * 2 + q))
    return taps


def abort_code() -> int:
    return int(_lib.lib().iswm_debug_abort_code())
