"""Inference step of the hot path (reference: predict.py:258-290 `predict_mask`, batched).

    logits = model(x); prob = softmax(logits, 1); pred = prob[:, 1] > threshold; confidence = uint8(prob[:, 1] * 255)

For the reference's two-class models the final bilinear upsample, softmax, threshold and confidence map run as ONE
pass over the LOW-resolution logits (`iswm_predict_epilogue`) writing uint8 maps only - the full-resolution fp32
logits (268 MB at 8 x 2 x 2048^2) are never written or read; other class counts take `iswm_argmax_confusion` on the
upsampled logits. With `labels` given the same pass also accumulates the confusion matrix the way
evaluate_quantization.py:265-270 feeds `StreamMetrics`.

Test-time augmentation (`scales`, `flip`: DeepLabV3+'s multi-scale + flip evaluation) averages the softmax over the
views (s, f), s in scales, f in (False, True) when flip:

    xv = flip_f(resize(x, (int(H*s+0.5), int(W*s+0.5))));  p += softmax(flip_f(resize(model(xv), (H, W))), 1);  p /= V

The fused path builds each scale's views with `iswm_resize_flip_f32` into one input (unflipped and flipped halves run
as one forward: eval-mode BatchNorm is per sample), keeps every view's low-resolution logits, and runs ONE
`iswm_predict_tta_epilogue` over all of them; no view's full-resolution logits are written.
"""
from __future__ import annotations

import math
from typing import List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

from . import _lib, ops

# B x H x W of the largest single forward the test-time augmentation issues: that of the largest predict geometry the
# engine is benchmarked at (8 x 2048^2). Beyond it the engine's 32-bit element counts are untested (at s = 2 on 2048^2
# inputs, 8 images of layer1 activations hold exactly 2^31 elements), so larger batches run in chunks.
MAX_FORWARD_PIXELS = 8 * 2048 * 2048


def _tta_views(scales: Sequence[float], flip: bool, H: int, W: int) -> List[Tuple[float, Tuple[int, int], bool]]:
    """[(s, (Hs, Ws), f)] in view order, validated."""
    scales = [float(s) for s in scales]
    if not scales:
        raise ValueError("scales must name at least one scale")
    views = []
    for s in scales:
        if not math.isfinite(s) or s <= 0:
            raise ValueError(f"scale {s} must be finite and > 0")
        size = (H, W) if s == 1.0 else (int(H * s + 0.5), int(W * s + 0.5))
        if min(size) < 16:
            raise ValueError(f"scale {s} makes a {size[0]}x{size[1]} view; views need at least 16x16 pixels")
        views += [(s, size, f) for f in ((False, True) if flip else (False,))]
    if len(views) > _lib.TTA_MAX_VIEWS:
        raise ValueError(f"{len(views)} views requested; test-time augmentation takes at most {_lib.TTA_MAX_VIEWS}")
    return views


@torch.no_grad()
def predict_mask(model, images: torch.Tensor, threshold: float = 0.5, labels: Optional[torch.Tensor] = None,
                 metrics=None, fused: bool = True, scales: Sequence[float] = (1.0,),
                 flip: bool = False) -> Tuple[torch.Tensor, torch.Tensor]:
    """images: float32 [B,3,H,W] on CUDA (already normalised, predict.py:259-260). Returns (pred uint8 [B,H,W] in
    {0,1}, confidence uint8 [B,H,W]); `metrics` (a StreamMetrics) receives the confusion counts when labels are given.
    `scales` / `flip` request test-time augmentation (two-class models; at most 8 views); the defaults run one view."""
    if not images.is_cuda:
        raise RuntimeError("iswm_b200.predict runs on CUDA only (no CPU fallback)")
    net = getattr(model, "module", model)
    cm = metrics._cm() if (metrics is not None and labels is not None) else None
    H, W = images.shape[-2:]
    n_classes = net.engine().cls.cout
    if n_classes < 2:
        raise ValueError("predict_mask needs at least 2 classes (foreground = class 1)")
    if flip or [float(s) for s in scales] != [1.0]:
        views = _tta_views(scales, flip, H, W)
        if n_classes != 2:
            raise ValueError(f"test-time augmentation (scales / flip) needs a two-class model, this one has {n_classes}")
        if fused:
            return _predict_tta(net, images, views, flip, threshold, labels if cm is not None else None, cm)
        return _predict_tta_unfused(model, images, views, threshold, labels if cm is not None else None, cm)
    if fused and n_classes == 2 and W % 4 == 0:
        # the reference's binary case: upsample + softmax + threshold + uint8 maps (+ confusion counts) in ONE kernel
        # over the low-resolution logits; bit-identical to the unfused path below
        lo = net.forward_lowres(images)
        _, pred, conf = ops.predict_epilogue(lo, H, W, labels if cm is not None else None, mode=1, threshold=threshold, out=cm)
        return pred, conf
    was_training = model.training
    model.eval()
    try:
        logits = model(images)
    finally:
        if was_training:
            model.train()
    _, pred, conf = ops.argmax_confusion(logits, labels if cm is not None else None, mode=1, threshold=threshold,
                                         want_pred=True, want_conf=True, out=cm)
    return pred, conf


def _predict_tta(net, images, views, flip, threshold, labels, cm):
    """Fused test-time augmentation: per batch chunk, one forward per scale (two when its flipped and unflipped halves
    together would exceed MAX_FORWARD_PIXELS), then one epilogue over every view's low-resolution logits that writes the
    chunk's slice of the maps."""
    x = images.contiguous()
    B, C, H, W = x.shape
    pred = torch.empty((B, H, W), dtype=torch.uint8, device=x.device)
    conf = torch.empty((B, H, W), dtype=torch.uint8, device=x.device)
    per_image = max(Hs * Ws for _, (Hs, Ws), _ in views)
    chunk = max(1, min(B, MAX_FORWARD_PIXELS // per_image))
    nf = 2 if flip else 1
    for b0 in range(0, B, chunk):
        xb = x[b0:b0 + chunk]
        n = xb.shape[0]
        lows = []
        for g in range(0, len(views), nf):
            _, (Hs, Ws), _ = views[g]
            flips = [f for _, _, f in views[g:g + nf]]
            if flips == [False] and (Hs, Ws) == (H, W):
                lows.append((net.forward_lowres(xb), (H, W), False))        # the plain view needs no copy
            elif nf * n * Hs * Ws <= MAX_FORWARD_PIXELS:
                buf = torch.empty((nf * n, C, Hs, Ws), dtype=torch.float32, device=x.device)
                for i, f in enumerate(flips):
                    ops.resize_flip_f32(xb, (Hs, Ws), f, out=buf[i * n:(i + 1) * n])
                lo = net.forward_lowres(buf)
                lows += [(lo[i * n:(i + 1) * n], (Hs, Ws), f) for i, f in enumerate(flips)]
            else:
                lows += [(net.forward_lowres(ops.resize_flip_f32(xb, (Hs, Ws), f)), (Hs, Ws), f) for f in flips]
        ops.predict_tta_epilogue(lows, H, W, None if labels is None else labels[b0:b0 + n], mode=1, threshold=threshold,
                                 out=cm, pred=pred[b0:b0 + n], conf=conf[b0:b0 + n])
    return pred, conf


def _predict_tta_unfused(model, images, views, threshold, labels, cm):
    """The torch composition of test-time augmentation through the public forward: the reference the fused path is
    tested against."""
    H, W = images.shape[-2:]
    was_training = model.training
    model.eval()
    try:
        p = None
        for s, (Hs, Ws), f in views:
            xv = images if s == 1.0 else F.interpolate(images, size=(Hs, Ws), mode="bilinear", align_corners=False)
            lv = model(xv.flip(-1) if f else xv)
            if (Hs, Ws) != (H, W):
                lv = F.interpolate(lv, size=(H, W), mode="bilinear", align_corners=False)
            sm = torch.softmax(lv.flip(-1) if f else lv, 1)
            p = sm if p is None else p + sm
    finally:
        if was_training:
            model.train()
    p1 = p[:, 1] / len(views)
    pred = (p1 > threshold).to(torch.uint8)
    conf = (p1 * 255).to(torch.uint8)
    if cm is not None:
        ops.confusion(labels, pred, 2, out=cm)
    return pred, conf
