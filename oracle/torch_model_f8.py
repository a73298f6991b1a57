"""FP8 precision-matched oracle — TEST INFRASTRUCTURE ONLY.

The eval graph of oracle/torch_model_q.py with an e4m3 rounding at exactly the points where iswm_b200/quant.py stores
e4m3 activations, the engine's own activation scales and e4m3 weights (QuantizedModel.export()), and its epilogue
formula (BatchNorm folded into fp32 scale / shift constants, iswm_b200.quant.epilogue_constants). The stem and the
pooled-ASPP 1x1 stay bf16, as in the engine. Products of two e4m3 values are exact in fp32, so against this oracle the
engine differs only by summation order and the roundings that order moves.
"""
from __future__ import annotations

import torch
import torch.nn.functional as F

from oracle.torch_model_q import BN_EPS, q

E4M3_MAX = 448.0


def e4m3(t: torch.Tensor) -> torch.Tensor:
    """Round to e4m3 (nearest even) with the hardware's satfinite: torch's own cast turns |x| >= 480 into NaN."""
    return t.clamp(-E4M3_MAX, E4M3_MAX).to(torch.float8_e4m3fn).float()


def quantize_weight(w: torch.Tensor):
    """Per-output-channel weight quantisation: s_w[c] = amax_c / 448 (1 for an all-zero channel), q = e4m3(w / s_w[c])."""
    w = w.detach().float()
    amax = w.abs().flatten(1).amax(1)
    s_w = torch.where(amax > 0, amax / torch.tensor(E4M3_MAX), torch.ones_like(amax))
    return e4m3(w / s_w[:, None, None, None]), s_w


def epilogue_constants(s_in, s_w, bn_scale, bn_shift, s_out):
    f = lambda v: torch.tensor(v, dtype=torch.float32)
    return ((f(s_in) * s_w) * bn_scale) / f(s_out), bn_shift / f(s_out)


def _fold(bn):
    scale = bn.weight / torch.sqrt(bn.running_var + BN_EPS)
    return scale, bn.bias - bn.running_mean * scale


def unit_f8(xq, wq, s_w, conv, bn, s_in, s_out, relu=True, res=None, s_res=None, out="e4m3"):
    """One e4m3 convolution of the engine: e4m3 input values xq (scale s_in), e4m3 weight values wq with per-channel scales
    s_w, BatchNorm `bn` (None: the classifier's bias) folded into the epilogue constants, optional e4m3 residual res (scale
    s_res), ReLU, then the output format ('e4m3' values for scale s_out, 'bf16' or 'f32')."""
    acc = F.conv2d(xq, wq, None, conv.stride, conv.padding, conv.dilation)
    bs, bsh = _fold(bn) if bn is not None else (torch.ones_like(s_w), conv.bias.detach().float())
    scale, shift = epilogue_constants(s_in, s_w, bs, bsh, s_out)
    z = acc * scale[None, :, None, None] + shift[None, :, None, None]
    if res is not None:
        z = z + res * (torch.tensor(s_res, dtype=torch.float32) / torch.tensor(s_out, dtype=torch.float32))
    if relu:
        z = F.relu(z)
    return e4m3(z) if out == "e4m3" else (q(z) if out == "bf16" else z)


def forward_f8(model, x: torch.Tensor, export: dict, taps: dict = None) -> torch.Tensor:
    """model: oracle.torch_model.OracleDeepLabV3Plus with the quantised model's source weights; export:
    QuantizedModel.export(). Returns fp32 logits [B,C,H,W]. `taps` (a dict, optional) receives every stored tensor under the
    name the engine's debug taps use: the producing convolution's name, 'pool' for the maxpool output."""
    S, W = export["scales"], export["weights"]
    bb, head = model.backbone, model.classifier

    def unit(xq, name, conv, bn, s_in, s_out, relu=True, res=None, s_res=None, out="e4m3"):
        r = unit_f8(xq, W[name][0], W[name][1], conv, bn, s_in, s_out, relu, res, s_res, out)
        if taps is not None:
            taps[name] = r
        return r

    def bf16_unit(xb, conv, bn):
        scale, shift = _fold(bn)
        y = F.conv2d(xb, q(conv.weight.detach()), None, conv.stride, conv.padding, conv.dilation)
        return q(F.relu(y * scale[None, :, None, None] + shift[None, :, None, None]))

    size = x.shape[-2:]
    stem = bf16_unit(q(x), bb["conv1"], bb["bn1"])
    a, s_a = e4m3(F.max_pool2d(stem, 3, 2, 1) / torch.tensor(S["pool"])), S["pool"]
    if taps is not None:
        taps["pool"] = a
    low = s_low = None
    for lname in ("layer1", "layer2", "layer3", "layer4"):
        for bi, blk in enumerate(bb[lname]):
            p = f"backbone.{lname}.{bi}"
            if blk.downsample is None:
                idt, s_idt = a, s_a
            else:
                idt, s_idt = unit(a, p + ".downsample.0", blk.downsample[0], blk.downsample[1], s_a, S[p + ".downsample.0"], relu=False), S[p + ".downsample.0"]
            y = unit(a, p + ".conv1", blk.conv1, blk.bn1, s_a, S[p + ".conv1"])
            y = unit(y, p + ".conv2", blk.conv2, blk.bn2, S[p + ".conv1"], S[p + ".conv2"])
            a = unit(y, p + ".conv3", blk.conv3, blk.bn3, S[p + ".conv2"], S[p + ".conv3"], res=idt, s_res=s_idt)
            s_a = S[p + ".conv3"]
        if lname == "layer1":
            low, s_low = a, s_a
    feat = a
    c1, c2 = S["cat1"], S["cat2"]
    lowp = unit(low, "classifier.project.0", head.project[0], head.project[1], s_low, c2)
    aspp = head.aspp
    outs = [unit(feat, f"classifier.aspp.convs.{i}.0", aspp.convs[i][0], aspp.convs[i][1], s_a, c1) for i in range(4)]
    pooled = q((feat * torch.tensor(s_a)).mean((2, 3), keepdim=True))
    pv = bf16_unit(pooled, aspp.convs[4][1], aspp.convs[4][2])
    outs.append(e4m3(pv / torch.tensor(c1)).expand(-1, -1, feat.shape[2], feat.shape[3]))
    ao = unit(torch.cat(outs, 1), "classifier.aspp.project.0", aspp.project[0], aspp.project[1], c1, 1.0, out="bf16")
    up = e4m3(F.interpolate(ao, size=lowp.shape[2:], mode="bilinear", align_corners=False) / torch.tensor(c2))
    cl = head.classifier
    y = unit(torch.cat([lowp, up], 1), "classifier.classifier.0", cl[0], cl[1], c2, S["classifier.classifier.0"])
    y = unit(y, "classifier.classifier.3", cl[3], cl[4], S["classifier.classifier.0"], S["classifier.classifier.3"])
    lo = unit(y, "classifier.classifier.6", cl[6], None, S["classifier.classifier.3"], 1.0, relu=False, out="f32")
    return F.interpolate(lo, size=size, mode="bilinear", align_corners=False)
