"""FP8 (e4m3) post-training-quantised inference of the DeepLabV3+ engine.

    qmodel = quantize_fp8(model, calibration)       # calibration: CUDA fp32 [B,3,H,W] tensor or an iterable of them
    logits = qmodel(images)                          # fp32 [B,C,H,W], like model.eval()(images)
    pred, conf = predict_mask(qmodel, images, 0.5, labels, metrics)

The FP8 counterpart of the reference's fbgemm-INT8 post-training quantisation (evaluate_quantization.py). `quantize_fp8`
reads the weights and BatchNorm running statistics ONCE: the returned model owns every tensor its forward reads, so later
training of `model` does not change it, and `model` itself is left as it was. Inference only.

Numerics (oracle/torch_model_f8.py restates them on the host):
  * An e4m3 activation q stands for q * s, one fp32 scale s per stored tensor: s = amax / 448 (1 where amax is 0), amax the
    largest |x| the bf16 eval forward produced for that tensor over the calibration batches. The ASPP concat (1280
    channels) and the decoder concat (304) are one tensor each with one scale shared by all their producers.
  * Weights, per output channel: s_w[c] = amax_c / 448, q = e4m3_rn_satfinite(w / s_w[c]) (iswm_pack_weight_f8).
  * BatchNorm is folded into each convolution's epilogue, not into its weights (fp32, in this order):
        scale'[c] = ((s_in * s_w[c]) * bn_scale[c]) / s_out,   shift'[c] = bn_shift[c] / s_out,   residual factor s_res / s_out
    and the epilogue computes relu(fma(res, factor, fma(acc, scale', shift'))) before rounding to the output format.
  * Every convolution whose input is a stored activation runs e4m3 x e4m3 -> fp32 (iswm_conv_igemm_f8); its output is
    e4m3 when another e4m3 convolution reads it, bf16 when a glue kernel does (the ASPP projection, read by the bilinear
    upsample), fp32 for the classifier. The stem (it reads the image) and the pooled-ASPP 1x1 (a B x 1 x 1 vector) stay
    bf16, with weights and folded BatchNorm copied into the snapshot.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, Iterable, Union

import torch

from . import _lib, ops
from ._lib import check
from .engine import STEM_KPITCH, Act, Engine, _st, _StreamScope

E4M3_MAX = 448.0


def scale_of(amax: torch.Tensor) -> float:
    """Per-tensor scale of an e4m3 activation: fp32 amax / 448, 1 for an all-zero tensor."""
    a = amax.detach().float().cpu().reshape(())
    return 1.0 if float(a) == 0.0 else float(a / torch.tensor(E4M3_MAX, dtype=torch.float32))


def epilogue_constants(s_in: float, s_w: torch.Tensor, bn_scale: torch.Tensor, bn_shift: torch.Tensor, s_out: float):
    """fp32 epilogue constants of an e4m3 convolution: scale' = ((s_in * s_w) * bn_scale) / s_out, shift' = bn_shift / s_out."""
    f = lambda v: torch.tensor(v, dtype=torch.float32, device=s_w.device)
    return ((f(s_in) * s_w) * bn_scale) / f(s_out), bn_shift / f(s_out)


def residual_factor(s_res: float, s_out: float) -> float:
    return float(torch.tensor(s_res, dtype=torch.float32) / torch.tensor(s_out, dtype=torch.float32))


def _new8(B, H, W, Cc, dev) -> Act:
    return Act(torch.empty((B, H, W, Cc), dtype=torch.float8_e4m3fn, device=dev), B, H, W, Cc, Cc)


class _QConv:
    """Snapshot of one e4m3 convolution: packed e4m3 weights, per-channel weight scales, the folded BatchNorm and,
    once the activation scales are known, the epilogue constants."""

    def __init__(self, eng: Engine, s):
        self.spec = s
        w = s.conv.weight.detach().float().contiguous()
        Cout, Cin, R, S_ = w.shape
        self.cin_pad = (Cin + 127) // 128 * 128
        self.w = torch.empty(Cout * R * S_ * self.cin_pad, dtype=torch.uint8, device=w.device)
        self.s_w = torch.empty(Cout, dtype=torch.float32, device=w.device)
        check(_lib.lib().iswm_pack_weight_f8(w.data_ptr(), Cout, Cin, R * S_, self.cin_pad, self.w.data_ptr(), self.s_w.data_ptr(), _st()),
              "pack_weight_f8 " + s.name)
        if s.bn is not None:
            eng._fold(s)
            self.bn_scale, self.bn_shift = s.fold_scale.clone(), s.fold_shift.clone()
        else:                                       # the classifier: bias only
            self.bn_scale = torch.ones(Cout, dtype=torch.float32, device=w.device)
            self.bn_shift = s.conv.bias.detach().float().clone()
        self.scale = self.shift = None

    def set_scales(self, s_in: float, s_out: float):
        self.s_in, self.s_out = s_in, s_out
        self.scale, self.shift = epilogue_constants(s_in, self.s_w, self.bn_scale, self.bn_shift, s_out)


class QuantizedModel(torch.nn.Module):
    """The FP8 inference model `quantize_fp8` returns. Eval-only: train(True) raises."""

    def __init__(self, eng: Engine, qconv: Dict[str, _QConv], bf16: Dict[str, tuple], scales: Dict[str, float]):
        super().__init__()
        self._eng, self.qconv, self.bf16, self.scales = eng, qconv, bf16, scales
        self.training = False

    def train(self, mode: bool = True):
        if mode:
            raise RuntimeError("a model quantised by quantize_fp8 is inference-only")
        return self

    def engine(self) -> Engine:
        return self._eng

    def forward(self, images: torch.Tensor) -> torch.Tensor:
        return self._run(images, lowres=False)

    def forward_lowres(self, images: torch.Tensor) -> torch.Tensor:
        """The classifier's fp32 NHWC [B,H/4,W/4,C] logits before the final upsample (what predict_mask's fused epilogue reads)."""
        return self._run(images, lowres=True)

    def export(self) -> dict:
        """Host copies of what the FP8 forward reads, for oracle/torch_model_f8.py: activation scales by producing convolution
        ('pool' = the maxpool output, 'cat1' / 'cat2' = the ASPP and decoder concats) and each e4m3 convolution's weights as
        e4m3 values [Cout,Cin,R,S] with their per-channel scales."""
        w = {}
        for name, q in self.qconv.items():
            Cout, Cin, R, S_ = q.spec.conv.weight.shape
            v = q.w.view(torch.float8_e4m3fn).float().view(Cout, R * S_, q.cin_pad)[:, :, :Cin]
            w[name] = (v.permute(0, 2, 1).reshape(Cout, Cin, R, S_).cpu(), q.s_w.cpu())
        return dict(scales=dict(self.scales), weights=w)

    # ------------------------------------------------------------------ the FP8 walk
    def _run(self, x: torch.Tensor, lowres: bool) -> torch.Tensor:
        if not x.is_cuda:
            raise RuntimeError("iswm_b200 runs on CUDA only: move the model and the input to a B200 (no CPU fallback)")
        if torch.is_grad_enabled() and x.requires_grad:
            raise RuntimeError("a model quantised by quantize_fp8 is inference-only: run it under torch.no_grad()")
        eng = self._eng
        with _StreamScope():
            eng._check_device(x)
            if x.dim() != 4 or x.shape[1] != eng.stem.cin:
                raise ValueError(f"expected [B,{eng.stem.cin},H,W] input, got {tuple(x.shape)}")
            return self._walk(x.contiguous().float(), lowres)

    def _prep(self, s, x: Act):
        """stride 2: the parity phases of the dense e4m3 input in place, or (odd sizes) a phase-split / subsampled copy"""
        if s.stride == 1:
            return x, ops.conv_taps(s.k, s.dilation), x.B, x.H, x.W
        L, dev = _lib.lib(), x.t.device
        Ho, Wo = (x.H + 1) // 2, (x.W + 1) // 2
        if x.H % 2 == 0 and x.W % 2 == 0 and x.C % 128 == 0 and x.ld % 16 == 0:
            xv = Act(x.t, x.B, Ho, Wo, x.C, x.ld)
            xv.phase_view = True
            return xv, (ops.conv_taps(1, 1) if s.k == 1 else ops.conv_taps_s2_3x3()), x.B, Ho, Wo
        if s.k == 1:
            xs = _new8(x.B, Ho, Wo, x.C, dev)
            check(L.iswm_subsample2_b8(x.ptr, x.ld, x.B, x.H, x.W, x.C, xs.ptr, _st()), "subsample2_b8")
            return xs, ops.conv_taps(1, 1), x.B, Ho, Wo
        ph = torch.empty((4 * x.B, Ho, Wo, x.C), dtype=torch.float8_e4m3fn, device=dev)
        check(L.iswm_phase_split_b8(x.ptr, x.ld, x.B, x.H, x.W, x.C, ph.data_ptr(), _st()), "phase_split_b8")
        return Act(ph, x.B, Ho, Wo, x.C, x.C), ops.conv_taps_s2_3x3(), 4 * x.B, Ho, Wo

    def _unit(self, name: str, x: Act, out: Act = None, relu: bool = True, res: Act = None, res_factor: float = 0.0,
              out_type: int = _lib.E4M3) -> Act:
        q = self.qconv[name]
        s = q.spec
        xin, taps, n_img, Ho, Wo = self._prep(s, x)
        if out is None:
            out = _new8(x.B, Ho, Wo, s.cout, x.t.device) if out_type == _lib.E4M3 else Act.new(x.B, Ho, Wo, s.cout, x.t.device)
        flags = _lib.EPI_AFFINE | (_lib.EPI_RELU if relu else 0) | (_lib.EPI_RESIDUAL if res is not None else 0)
        d = ops.make_conv_desc(xin.B, xin.H, xin.W, xin.C, xin.ld, n_img, Ho, Wo, s.cout, out.ld, taps, flags,
                               0 if res is None else res.ld, phase_view=xin.phase_view)
        eng = self._eng
        ev = eng._prof_begin()
        check(_lib.lib().iswm_conv_igemm_f8(C.byref(d), xin.ptr, q.w.data_ptr(), out.ptr, q.scale.data_ptr(), q.shift.data_ptr(),
                                            None if res is None else res.ptr, res_factor, out_type, _st()), "conv_igemm_f8 " + name)
        eng._prof_end(ev, "conv_igemm_f8", 2.0 * x.B * Ho * Wo * s.cout * s.cin * len(taps), "fwd " + name)
        eng._tap(name, out)
        return out

    def _walk(self, x: torch.Tensor, lowres: bool) -> torch.Tensor:
        eng, L, S = self._eng, _lib.lib(), self.scales
        B, _, H, W = x.shape
        dev = x.device
        # ---- stem (bf16) -> maxpool into e4m3
        H1, W1 = (H + 1) // 2, (W + 1) // 2
        rows = torch.empty((2 * B, H1, W1, STEM_KPITCH), dtype=torch.bfloat16, device=dev)
        check(L.iswm_stem_rows(x.data_ptr(), B, eng.stem.cin, H, W, H1, W1, STEM_KPITCH, rows.data_ptr(), _st()), "stem_rows")
        colA = Act(rows, B, H1, W1, STEM_KPITCH, STEM_KPITCH)
        stem_taps = [((r - 3 - ((r + 1) & 1)) // 2, 0, (r + 1) & 1) for r in range(7)]
        stem_out = Act.new(B, H1, W1, 64, dev)
        wst, sst, hst = self.bf16[eng.stem.name]
        eng._conv(eng.stem, colA, stem_out.t, 64, H1, W1, stem_taps, 2 * B, _lib.EPI_AFFINE | _lib.EPI_RELU, sst, hst,
                  cin=colA.C, Hi=H1, Wi=W1, B=B, wgt=wst)
        H2, W2 = (H1 + 1) // 2, (W1 + 1) // 2
        a = _new8(B, H2, W2, 64, dev)
        check(L.iswm_maxpool_fwd_f8(stem_out.ptr, B, H1, W1, 64, H2, W2, S["pool"], a.ptr, _st()), "maxpool_fwd_f8")
        eng._tap("pool", a)
        s_a = S["pool"]
        # ---- residual layers
        cat2 = low = None
        for li, blocks in enumerate(eng.layers):
            for (c1, c2, c3, ds) in blocks:
                if ds is None:
                    idt, s_idt = a, s_a
                else:
                    idt, s_idt = self._unit(ds.name, a, relu=False), S[ds.name]
                y = self._unit(c1.name, a)
                y = self._unit(c2.name, y)
                a = self._unit(c3.name, y, res=idt, res_factor=residual_factor(s_idt, S[c3.name]))
                s_a = S[c3.name]
            if li == 0:
                low = a
                cat2 = _new8(B, a.H, a.W, 304, dev)
                with eng._fwd_fork():
                    self._unit(eng.low_proj.name, low, out=cat2.slice(0, 48))
        feat = a
        hf, wf, h4, w4 = feat.H, feat.W, low.H, low.W
        # ---- ASPP: four e4m3 branches and the bf16 pooled branch into one e4m3 concat
        cat1 = _new8(B, hf, wf, 1280, dev)
        with eng._fwd_fork():
            pooled = Act.new(B, 1, 1, feat.C, dev)
            check(L.iswm_gap_fwd_f8(feat.ptr, feat.ld, B, hf * wf, feat.C, s_a, pooled.ptr, _st()), "gap_fwd_f8")
            v = Act.new(B, 1, 1, 256, dev)
            wp, sp, hp = self.bf16[eng.aspp_pool.name]
            eng._conv(eng.aspp_pool, pooled, v.t, 256, 1, 1, ops.conv_taps(1, 1), B, _lib.EPI_AFFINE | _lib.EPI_RELU, sp, hp, wgt=wp)
            dst = cat1.slice(1024, 256)
            check(L.iswm_broadcast_hw_f8(v.ptr, B, hf * wf, 256, S["cat1"], dst.ptr, dst.ld, _st()), "broadcast_hw_f8")
            eng._fwd_keep.extend((pooled.t, v.t))
        for i, s in enumerate(eng.aspp_branches):
            self._unit(s.name, feat, out=cat1.slice(256 * i, 256))
        eng._fwd_join()
        aspp_out = self._unit(eng.aspp_proj.name, cat1, out_type=_lib.BF16)
        up = cat2.slice(48, 256)
        check(L.iswm_bilinear_fwd_f8(aspp_out.ptr, aspp_out.ld, B, hf, wf, 256, h4, w4, S["cat2"], up.ptr, up.ld, _st()), "bilinear_fwd_f8")
        y = self._unit(eng.dec1.name, cat2)
        y = self._unit(eng.dec2.name, y)
        ncls = eng.cls.cout
        lo = torch.empty((B, h4, w4, ncls), dtype=torch.float32, device=dev)
        self._unit(eng.cls.name, y, out=Act(lo, B, h4, w4, ncls, ncls), relu=False, out_type=_lib.F32)
        if lowres:
            return lo
        logits = torch.empty((B, ncls, H, W), dtype=torch.float32, device=dev)
        check(L.iswm_logits_up_fwd(lo.data_ptr(), B, h4, w4, ncls, H, W, logits.data_ptr(), _st()), "logits_up_fwd")
        return logits


def _calibrate(eng: Engine, batches) -> Dict[str, torch.Tensor]:
    """The bf16 eval forward (Engine's own units) over the calibration batches, recording max |x| of exactly the tensors the
    FP8 forward stores in e4m3, keyed by the convolution that produces them ('pool', 'cat1', 'cat2' for the rest)."""
    L = _lib.lib()
    amax: Dict[str, torch.Tensor] = {}

    def rec(key, a: Act):
        m = a.t.abs().amax().float()
        amax[key] = m if key not in amax else torch.maximum(amax[key], m)

    n = 0
    for x in batches:
        n += 1
        if not isinstance(x, torch.Tensor) or not x.is_cuda:
            raise RuntimeError("quantize_fp8: calibration batches must be CUDA fp32 [B,3,H,W] tensors")
        with _StreamScope():
            eng._check_device(x)
            if x.dim() != 4 or x.shape[1] != eng.stem.cin:
                raise ValueError(f"expected [B,{eng.stem.cin},H,W] calibration input, got {tuple(x.shape)}")
            x = x.contiguous().float()
            B, _, H, W = x.shape
            dev = x.device
            H1, W1 = (H + 1) // 2, (W + 1) // 2
            rows = torch.empty((2 * B, H1, W1, STEM_KPITCH), dtype=torch.bfloat16, device=dev)
            check(L.iswm_stem_rows(x.data_ptr(), B, eng.stem.cin, H, W, H1, W1, STEM_KPITCH, rows.data_ptr(), _st()), "stem_rows")
            stem_taps = [((r - 3 - ((r + 1) & 1)) // 2, 0, (r + 1) & 1) for r in range(7)]
            stem_out = eng._stem_unit(Act(rows, B, H1, W1, STEM_KPITCH, STEM_KPITCH), B, H1, W1, False, stem_taps, 2 * B)
            H2, W2 = (H1 + 1) // 2, (W1 + 1) // 2
            a = Act.new(B, H2, W2, 64, dev)
            check(L.iswm_maxpool_fwd(stem_out.ptr, B, H1, W1, 64, H2, W2, a.ptr, None, _st()), "maxpool_fwd")
            rec("pool", a)
            cat2 = None
            for li, blocks in enumerate(eng.layers):
                for (c1, c2, c3, ds) in blocks:
                    idt = a
                    if ds is not None:
                        idt = eng._unit_eval(ds, a, relu=False)
                        rec(ds.name, idt)
                    y = eng._unit_eval(c1, a)
                    rec(c1.name, y)
                    y = eng._unit_eval(c2, y)
                    rec(c2.name, y)
                    a = eng._unit_eval(c3, y, relu=True, residual=idt)
                    rec(c3.name, a)
                if li == 0:
                    cat2 = Act.new(B, a.H, a.W, 304, dev)
                    eng._unit_eval(eng.low_proj, a, out=cat2.slice(0, 48))
            feat = a
            cat1 = Act.new(B, feat.H, feat.W, 1280, dev)
            eng._aspp_pool(feat, cat1.slice(1024, 256), False)
            eng._fwd_keep = []
            for i, s in enumerate(eng.aspp_branches):
                eng._unit_eval(s, feat, out=cat1.slice(256 * i, 256))
            rec("cat1", cat1)
            ao = eng._unit_eval(eng.aspp_proj, cat1)
            up = cat2.slice(48, 256)
            check(L.iswm_bilinear_fwd(ao.ptr, ao.ld, B, feat.H, feat.W, 256, cat2.H, cat2.W, up.ptr, up.ld, _st()), "bilinear_fwd")
            rec("cat2", cat2)
            y = eng._unit_eval(eng.dec1, cat2)
            rec(eng.dec1.name, y)
            rec(eng.dec2.name, eng._unit_eval(eng.dec2, y))
    if n == 0:
        raise ValueError("quantize_fp8: no calibration batches")
    return amax


@torch.no_grad()
def quantize_fp8(model, calibration: Union[torch.Tensor, Iterable[torch.Tensor]]) -> QuantizedModel:
    """Post-training FP8 quantisation of a DeepLabV3+ (ResNet-50 / ResNet-101, output stride 8 or 16, any number of classes).
    `calibration`: a CUDA fp32 [B,3,H,W] tensor or an iterable of them, normalised like the model's inputs. Returns an
    inference-only model with its own copy of every weight it reads; `model` is not modified."""
    net = getattr(model, "module", model)
    eng: Engine = net.engine()
    if not eng.stem_rows:
        raise ValueError("quantize_fp8 supports models with at most 3 input channels (the row-tap stem)")
    batches = [calibration] if isinstance(calibration, torch.Tensor) else calibration
    amax = _calibrate(eng, batches)
    dev = eng.device
    S = {k: scale_of(v) for k, v in amax.items()}
    # bf16 snapshot: the stem and the pooled-ASPP 1x1 (packed operand + folded BatchNorm)
    bf16 = {}
    for s in (eng.stem, eng.aspp_pool):
        eng._pack(s, False)
        eng._fold(s)
        bf16[s.name] = (s.packed_fwd.clone(), s.fold_scale.clone(), s.fold_shift.clone())
    qconv: Dict[str, _QConv] = {}

    def q(s, s_in, s_out):
        qconv[s.name] = _QConv(eng, s)
        qconv[s.name].set_scales(s_in, s_out)

    s_a = S["pool"]
    for li, blocks in enumerate(eng.layers):
        for (c1, c2, c3, ds) in blocks:
            if ds is not None:
                q(ds, s_a, S[ds.name])
            q(c1, s_a, S[c1.name])
            q(c2, S[c1.name], S[c2.name])
            q(c3, S[c2.name], S[c3.name])
            s_a = S[c3.name]
        if li == 0:
            q(eng.low_proj, s_a, S["cat2"])
    for s in eng.aspp_branches:
        q(s, s_a, S["cat1"])
    q(eng.aspp_proj, S["cat1"], 1.0)
    q(eng.dec1, S["cat2"], S[eng.dec1.name])
    q(eng.dec2, S[eng.dec1.name], S[eng.dec2.name])
    q(eng.cls, S[eng.dec2.name], 1.0)
    torch.cuda.current_stream(dev).synchronize()
    return QuantizedModel(eng, qconv, bf16, S)
