"""Whole-network executor for the DeepLabV3+ (ResNet-50/101) hot path.

The nn.Module tree (iswm_b200/network) only OWNS parameters under the reference's state_dict
names; this module RUNS them: it walks the known graph (network/utils.py:16-25 forward,
network/backbone/resnet.py:99-120 bottleneck, network/_deeplab.py:55-61, :167-172 head/ASPP),
launching libiswm_b200.so kernels on the current CUDA stream through raw pointers. Activations
are NHWC bf16; concat buffers are written in place through channel slices. In training mode each
op records a closure on a tape and `backward()` replays it in reverse — a hand-written reverse
sweep, not torch.autograd — writing fp32 OIHW parameter gradients into one flat buffer that the
data-parallel layer all-reduces in buckets.

No op here has a PyTorch / cuDNN fallback: torch is used for allocation, memsets and streams.
"""
from __future__ import annotations

import ctypes as C
from typing import Callable, List, Optional

import torch

from . import _lib, ops
from ._lib import check

BN_EPS = 1e-5
BN_MOMENTUM = 0.1
# channels per pixel of the x-unrolled stem rows (21 used): 32 = 64-byte pixels; 24 (48-byte, sector-straddling pixels) makes the
# TMA loads of the 7-tap convolution 2.3x slower (tools/prof_stem.py: 231 vs 99 us)
STEM_KPITCH = 32
# weight gradients of these backbone layers are collected while the layer's backward runs and launched as ONE grouped kernel
# when it ends (iswm_conv_wgrad_grouped: a layer's 13-19 small GEMMs side by side need almost no pixel-range splits, i.e.
# almost no partial-tile reductions; layer3 325 -> 192 us, layer2 282 -> 230 us, tools/prof_wgrad_group.py). layer1
# (operands far larger than L2: every tile would stream them from HBM again: 319 -> 374 us) keeps one launch per
# convolution. conv_wgrad 2.63 -> 2.28 ms/step, step 12.50 -> 12.42.
GROUP_WGRAD_LAYERS = ("layer2", "layer3", "layer4")


class _StreamCache:
    """Raw handle of the CUDA stream the engine is launching on. torch.cuda.current_stream() costs a few microseconds
    per call and the engine makes ~550 launches per step, so forward() / backward() look it up once and the
    weight-gradient context swaps it explicitly."""
    handle = None


def _st() -> int:
    h = _StreamCache.handle
    return torch.cuda.current_stream().cuda_stream if h is None else h


class _StreamScope:
    """with _StreamScope(): ... pins _st() to the stream that is current on entry."""

    def __enter__(self):
        self.prev = _StreamCache.handle
        _StreamCache.handle = torch.cuda.current_stream().cuda_stream
        return self

    def __exit__(self, *a):
        _StreamCache.handle = self.prev
        return False


class Act:
    """NHWC bf16 activation: `t` is a [B,H,W,C] view whose row pitch is `ld` elements."""

    __slots__ = ("t", "B", "H", "W", "C", "ld", "grad", "pending", "masked_ok", "phase_view")

    def __init__(self, t: torch.Tensor, B: int, H: int, W: int, Cc: int, ld: int):
        self.t, self.B, self.H, self.W, self.C, self.ld = t, B, H, W, Cc, ld
        self.grad: Optional["Act"] = None             # gradient w.r.t. this activation (same geometry)
        # identity-path gradient of a bottleneck block that has NOT been written out: (block-output gradient, ReLU sign bits);
        # the block's conv1 data gradient adds it, gated by the bits, in its epilogue (ISWM_EPI_RES_MASK)
        self.pending = None
        self.masked_ok = False                        # set on block inputs whose only other consumer is that conv1
        self.phase_view = False                       # (H, W) are per-phase dims of a dense [B, 2H, 2W, ld] tensor read in place (stride-2 convs)

    @property
    def M(self) -> int:
        return self.B * self.H * self.W

    @property
    def ptr(self) -> int:
        return self.t.data_ptr()

    @staticmethod
    def new(B, H, W, Cc, device) -> "Act":
        return Act(torch.empty((B, H, W, Cc), dtype=torch.bfloat16, device=device), B, H, W, Cc, Cc)

    def slice(self, off: int, Cc: int) -> "Act":
        return Act(self.t[..., off:off + Cc], self.B, self.H, self.W, Cc, self.ld)

    def new_grad(self) -> "Act":
        """Allocate a dense gradient buffer of this activation's geometry and attach it."""
        self.grad = Act.new(self.B, self.H, self.W, self.C, self.t.device)
        return self.grad


class ConvSpec:
    """Static description of one convolution + its packed-weight cache."""

    def __init__(self, name, conv, bn, k, stride, dilation):
        self.name, self.conv, self.bn = name, conv, bn
        self.k, self.stride, self.dilation = k, stride, dilation
        self.cout, self.cin = conv.weight.shape[0], conv.weight.shape[1]
        self.packed_fwd = None
        self.packed_dgrad = None
        self.version = -1
        self.fold_scale = None
        self.fold_shift = None
        self.fold_version = None
        self.is_stem = False


class Engine:
    def __init__(self, model):
        self.model = model
        self.device = None
        self.specs: List[ConvSpec] = []
        self._build_specs()
        self.tape: List[Callable[[], None]] = []
        self.step = 0
        self.generation = 0           # train-mode forwards issued so far (a backward must belong to the latest one)
        self.flat_g = None            # fp32 flat gradient buffer (all parameters, registration order)
        self.ext_flat_g = None        # set by iswm_b200.parallel: a symmetric-memory allocation to use as flat_g
        self.grad_views = {}
        self.wacc = None              # fp32 scratch for k>1 weight gradients
        self.grad_ready_hook: Optional[Callable[[torch.nn.Parameter], None]] = None
        self.dropout_p = 0.1
        self.seed = 0x5EED
        self._saved = None
        self.weights_epoch = 0        # bumped by optimisers that update parameters behind autograd's back
        self.flat_w = None            # fp32 flat master weights (parameters become views of it)
        self.batched_pack = True      # repack all weights in one launch when any changed
        # The attributes below select between two implementations of one step; tests and the benchmark set them to time or
        # compare the other form. All default to the faster one.
        # weight gradients feed nothing inside the backward sweep: they run on a second stream so that their
        # (tensor-core) kernels overlap the HBM-bound BatchNorm kernels and the launch / fill / drain gaps of the
        # data-gradient chain; False puts them back in line
        self.async_wgrad = True
        # forward branches nothing on the main chain consumes for a while run on that second stream too (_fwd_fork)
        self.fwd_overlap = True
        # k x k weight gradients are unpacked in one launch at the end of the sweep (_unpack_all)
        self.batch_unpack = True
        # ASPP backward: one K-concatenated data-gradient GEMM over the four conv branches (iswm_aspp_bwd) instead of four
        # launches with three read-modify-write passes over the 2048-channel feature gradient
        self.aspp_fused_bwd = True
        # identity-path gradient of non-first bottleneck blocks folded into the block's conv1 data-gradient epilogue
        # (ISWM_EPI_RES_MASK) instead of a tensor written by bn_bwd_apply and read back
        self.masked_identity = True
        # blocks with a downsample branch: the closing BatchNorm and the downsample BatchNorm run as ONE kernel per pass
        # (csrc/bn_dual.cu; the normalised shortcut is never written, backward reads dout / sign bits once per pass for both)
        self.dual_bn = True
        # stem tail (train): BatchNorm + ReLU + maxpool as one forward pass (csrc/stem_pool.cu: the half-resolution activation is
        # never written); False: separate kernels
        self.stem_pool = True
        self._wq, self._wq_layer = [], None
        self._fwd_keep = []
        self._wstream = None
        self._wgrad_keep = []
        self.profile = None           # list of (kernel, algorithmic_flops, start_event, end_event) when profiling
        self.debug_taps = None        # dict name -> NCHW fp32 copy of each unit's output (tools/layer_diff.py)
        self.debug_units = None       # list of per-unit records of the engine's own tensors (tests/test_unit_replay_gpu.py)
        # synchronised BatchNorm (set by iswm_b200.parallel.DataParallel(sync_bn=True)): bn_sync(srcs, dsts, n, rows, stream) turns
        # this rank's fp64 statistics slots `srcs` [(slot, replicas)] of n = 2C values into the sums over every rank plus the
        # global row count, dsts[i][:n + 1]; called between each train-mode BatchNorm's producer and its consumer, on the stream
        # the unit runs on. None: every rank normalises with its own shard's statistics (nn.DataParallel)
        self.bn_sync: Optional[Callable] = None
        self.ext_scratch64 = None     # set with bn_sync on the peer transport: a symmetric allocation to carve the fp64 slots from

    # ------------------------------------------------------------------ graph description
    def _build_specs(self):
        m = self.model
        bb, head = m.backbone, m.classifier
        S = self._spec
        self.stem = S("backbone.conv1", bb.conv1, bb.bn1, 7, 2, 1)
        self.stem.is_stem = True
        self.layers = []
        for lname in ("layer1", "layer2", "layer3", "layer4"):
            blocks = []
            for bi, blk in enumerate(getattr(bb, lname)):
                p = f"backbone.{lname}.{bi}"
                c1 = S(p + ".conv1", blk.conv1, blk.bn1, 1, 1, 1)
                c2 = S(p + ".conv2", blk.conv2, blk.bn2, 3, blk.stride, blk.dilation)
                c3 = S(p + ".conv3", blk.conv3, blk.bn3, 1, 1, 1)
                ds = None
                if blk.downsample is not None:
                    ds = S(p + ".downsample.0", blk.downsample[0], blk.downsample[1], 1, blk.stride, 1)
                blocks.append((c1, c2, c3, ds))
            self.layers.append(blocks)
        self.low_proj = S("classifier.project.0", head.project[0], head.project[1], 1, 1, 1)
        aspp = head.aspp
        self.aspp_branches = [S("classifier.aspp.convs.0.0", aspp.convs[0][0], aspp.convs[0][1], 1, 1, 1)]
        for i, r in enumerate(aspp.rates):
            self.aspp_branches.append(S(f"classifier.aspp.convs.{i + 1}.0", aspp.convs[i + 1][0], aspp.convs[i + 1][1], 3, 1, r))
        self.aspp_pool = S("classifier.aspp.convs.4.1", aspp.convs[4][1], aspp.convs[4][2], 1, 1, 1)
        self.aspp_proj = S("classifier.aspp.project.0", aspp.project[0], aspp.project[1], 1, 1, 1)
        cl = head.classifier
        self.dec1 = S("classifier.classifier.0", cl[0], cl[1], 3, 1, 1)
        self.dec2 = S("classifier.classifier.3", cl[3], cl[4], 3, 1, 1)
        self.cls = S("classifier.classifier.6", cl[6], None, 1, 1, 1)

    @property
    def stem_rows(self) -> bool:
        """The stem 7x7/s2 runs on the image unrolled along x only (iswm_stem_rows, 48 B per pixel row) with the 7 kernel rows
        as 7 taps of the implicit GEMM over the two row-parity phases, instead of a full im2col matrix (320 B per pixel) + one
        GEMM; the im2col form serves inputs of more than 3 channels."""
        return self.stem.cin <= 3

    def _spec(self, name, conv, bn, k, stride, dilation) -> ConvSpec:
        s = ConvSpec(name, conv, bn, k, stride, dilation)
        self.specs.append(s)
        return s

    # ------------------------------------------------------------------ parameters / packing
    def _param_list(self):
        """model.parameters() walks the whole module tree (~25k Python calls); the tree is static, so walk it once."""
        pl = getattr(self, "_params_cache", None)
        if pl is None:
            pl = self._params_cache = list(self.model.parameters())
        return pl

    def _check_device(self, x: torch.Tensor):
        if not x.is_cuda:
            raise RuntimeError("iswm_b200 runs on CUDA only: move the model and the input to a B200 (no CPU fallback)")
        for p in self._param_list():
            if p.device != x.device:
                raise RuntimeError(f"parameter on {p.device} but input on {x.device}: call model.to(device) first")
            break
        self.device = x.device

    def pack_all(self, need_dgrad: bool = True):
        """Repack every convolution's weights (both operand layouts) in ONE kernel launch; called when the
        parameters changed (optimiser step, load_state_dict) instead of 2 small launches per layer."""
        import numpy as np
        sig = tuple((s.conv.weight.data_ptr(), tuple(s.conv.weight.shape)) for s in self.specs) + (need_dgrad, str(self.device), self.stem_rows)
        if getattr(self, "_pack_sig", None) != sig:
            jobs = []
            for s in self.specs:
                w = s.conv.weight
                Cout, Cin, R, S = w.shape
                RS = R * S
                if s.is_stem and self.stem_rows:
                    cin_pad, row_ld = 64, 7 * 64              # [Cout][7 kernel rows][64]: (kernel column, channel) pairs inside a row
                elif s.is_stem:
                    cin_pad, row_ld = Cin, ((RS * Cin + 63) // 64) * 64
                else:
                    cin_pad = ((Cin + 63) // 64) * 64
                    row_ld = RS * cin_pad
                if s.packed_fwd is None or s.packed_fwd.numel() != Cout * row_ld or s.packed_fwd.device != w.device:
                    s.packed_fwd = torch.empty(Cout * row_ld, dtype=torch.bfloat16, device=w.device)
                jobs.append((w.data_ptr(), s.packed_fwd.data_ptr(), Cout, Cin, RS, cin_pad, row_ld, 2 if (s.is_stem and self.stem_rows) else 0))
                if need_dgrad and s.name in self._aspp_cat_slot():
                    # the four ASPP conv branches share ONE K-concatenated dgrad operand [Cfeat][28 taps][256]
                    # (iswm_aspp_bwd): each branch's taps are a slice of the concatenated row
                    tap_off, taps_total = self._aspp_cat_slot()[s.name]
                    cout_pad = ((Cout + 63) // 64) * 64
                    n = Cin * taps_total * cout_pad
                    if getattr(self, "aspp_wcat", None) is None or self.aspp_wcat.numel() != n or self.aspp_wcat.device != w.device:
                        self.aspp_wcat = torch.empty(n, dtype=torch.bfloat16, device=w.device)
                    jobs.append((w.data_ptr(), self.aspp_wcat.data_ptr() + 2 * tap_off * cout_pad, Cout, Cin, RS, cout_pad, taps_total, 1))
                elif need_dgrad and not s.is_stem:
                    cout_pad = ((Cout + 63) // 64) * 64
                    n = Cin * RS * cout_pad
                    if s.packed_dgrad is None or s.packed_dgrad.numel() != n or s.packed_dgrad.device != w.device:
                        s.packed_dgrad = torch.empty(n, dtype=torch.bfloat16, device=w.device)
                    jobs.append((w.data_ptr(), s.packed_dgrad.data_ptr(), Cout, Cin, RS, cout_pad, 0, 1))
            arr, self._pack_blocks = _lib.fill_pack_jobs(jobs)
            host = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).clone()
            self._pack_jobs = host.to(self.device)
            self._pack_njobs = len(jobs)
            self._pack_sig = sig
        check(_lib.lib().iswm_pack_weights_batched(self._pack_jobs.data_ptr(), self._pack_njobs, self._pack_blocks, _st()), "pack_weights_batched")
        for s in self.specs:
            w = s.conv.weight
            s.version = (w._version, self.weights_epoch, w.data_ptr())
            s.has_dgrad = need_dgrad and not s.is_stem

    # ------------------------------------------------------------------ optimiser step fused with the repack
    def packed_is_fresh(self) -> bool:
        """True when every convolution's packed bf16 operands (both layouts) match the current master weights."""
        for s in self.specs:
            w = s.conv.weight
            if s.packed_fwd is None or s.version != (w._version, self.weights_epoch, w.data_ptr()) or not (s.is_stem or getattr(s, "has_dgrad", False)):
                return False
        return True

    def mark_packed_fresh(self):
        """The packed operands were just rewritten from the master weights by a kernel (iswm_sgd_pack_batched): advance the
        weights epoch (BatchNorm folds etc. refresh) and record that no repack is due."""
        self.weights_epoch += 1
        for s in self.specs:
            w = s.conv.weight
            s.version = (w._version, self.weights_epoch, w.data_ptr())

    def sgd_pack_jobs(self, flat_w: torch.Tensor, flat_g: torch.Tensor, mom: Optional[torch.Tensor]):
        """Job table of iswm_sgd_pack_batched over the flat parameter buffer, or None when the fused step does not apply
        (operands not packed yet, per-layer packing, im2col stem). Cached on the buffers' addresses."""
        if not (self.batched_pack and self.stem_rows) or not self.packed_is_fresh():
            return None
        params = self._param_list()
        sig = (flat_w.data_ptr(), flat_g.data_ptr(), 0 if mom is None else mom.data_ptr(), getattr(self, "_pack_sig", None),
               tuple(s.packed_fwd.data_ptr() for s in self.specs))
        if getattr(self, "_sgd_pack_sig", None) == sig:
            return self._sgd_pack_cache
        spec_of = {id(s.conv.weight): s for s in self.specs}
        slots = self._aspp_cat_slot()
        rows, off, run = [], 0, None                       # run = [start, end) of consecutive non-convolution parameters
        def flush():
            nonlocal run
            if run is not None:
                rows.append(dict(mode=0, off=run[0], n=run[1] - run[0]))
                run = None
        for p in params:
            n = p.numel()
            if p.data_ptr() != flat_w.data_ptr() + 4 * off:
                return None                                # parameters are not views of the flat buffer (flatten_parameters first)
            s = spec_of.get(id(p))
            if s is None:
                run = [off, off + n] if run is None else [run[0], off + n]
            else:
                flush()
                Cout, Cin, R, S_ = p.shape
                RS = R * S_
                if s.is_stem:
                    rows.append(dict(mode=2, off=off, n=n, Cout=Cout, Cin=Cin, RS=RS, dst_f=s.packed_fwd.data_ptr(), dst_d=0, pad_f=64, row_ld_f=7 * 64,
                                     pad_d=0, row_ld_d=0, TC=0))
                else:
                    cin_pad, cout_pad = ((Cin + 63) // 64) * 64, ((Cout + 63) // 64) * 64
                    if s.name in slots:
                        tap_off, taps_total = slots[s.name]
                        dst_d, row_ld_d = self.aspp_wcat.data_ptr() + 2 * tap_off * cout_pad, taps_total
                    else:
                        if s.packed_dgrad is None:
                            return None
                        dst_d, row_ld_d = s.packed_dgrad.data_ptr(), 0
                    TC = 128 if RS == 1 else max(8, (144 // RS) // 8 * 8)
                    rows.append(dict(mode=1, off=off, n=n, Cout=Cout, Cin=Cin, RS=RS, dst_f=s.packed_fwd.data_ptr(), dst_d=dst_d, pad_f=cin_pad,
                                     row_ld_f=RS * cin_pad, pad_d=cout_pad, row_ld_d=row_ld_d, TC=TC))
            off += n
        flush()
        arr = (_lib.SgdPackJob * len(rows))()
        begin = 0
        for i, r in enumerate(rows):
            j = arr[i]
            j.w, j.g = flat_w.data_ptr() + 4 * r["off"], flat_g.data_ptr() + 4 * r["off"]
            j.m = None if mom is None else mom.data_ptr() + 4 * r["off"]
            j.n, j.mode = r["n"], r["mode"]
            if r["mode"] == 0:
                j.blk_count = max(1, min(64, (r["n"] + 4095) // 4096))
            else:
                j.dst_f, j.dst_d = r["dst_f"], r["dst_d"] or None
                j.Cout, j.Cin, j.RS, j.pad_f, j.row_ld_f, j.pad_d, j.row_ld_d, j.TC = (r["Cout"], r["Cin"], r["RS"], r["pad_f"], r["row_ld_f"],
                                                                                          r["pad_d"], r["row_ld_d"], r["TC"])
                if r["mode"] == 2:
                    j.blk_count = max(1, min(64, (r["n"] + 1023) // 1024))
                else:
                    tiles = ((r["Cout"] + 15) // 16) * ((r["Cin"] + r["TC"] - 1) // r["TC"])
                    j.blk_count = max(1, min(512, tiles // 2))
            j.blk_begin = begin
            begin += j.blk_count
        dev_jobs = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).clone().to(flat_w.device)
        self._sgd_pack_sig, self._sgd_pack_cache = sig, (dev_jobs, len(rows), begin)
        return self._sgd_pack_cache

    def _aspp_cat_slot(self):
        """name -> (first tap, total taps) of the ASPP conv branches inside the concatenated dgrad operand; empty when the
        fused ASPP backward is off (aspp_fused_bwd = False) or the branch widths do not allow it."""
        d = getattr(self, "_aspp_slots", None)
        if d is None:
            d = {}
            br = self.aspp_branches
            ok = self.aspp_fused_bwd and self.batched_pack and len(br) == 4 and all(b.cout == br[0].cout and b.cin == br[0].cin for b in br) \
                and br[0].cout % 64 == 0 and br[0].k == 1 and all(b.k == 3 for b in br[1:])
            if ok:
                total = sum(b.k * b.k for b in br)
                off = 0
                for b in br:
                    d[b.name] = (off, total)
                    off += b.k * b.k
            self._aspp_slots = d
        return d

    def _pack(self, s: ConvSpec, need_dgrad: bool):
        w = s.conv.weight
        v = (w._version, self.weights_epoch, w.data_ptr())
        if self.batched_pack and (s.packed_fwd is None or s.version != v or (need_dgrad and not s.is_stem and not getattr(s, "has_dgrad", False))):
            self.pack_all(need_dgrad or self.model.training)
            return
        if s.is_stem and self.stem_rows:
            if s.packed_fwd is None or s.version != v or s.packed_fwd.device != w.device or s.packed_fwd.numel() != s.cout * 448:
                s.packed_fwd = torch.empty(s.cout * 448, dtype=torch.bfloat16, device=w.device)
                arr, nblk = _lib.fill_pack_jobs([(w.data_ptr(), s.packed_fwd.data_ptr(), s.cout, s.cin, 49, 64, 448, 2)])
                jobs = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).clone().to(w.device)
                check(_lib.lib().iswm_pack_weights_batched(jobs.data_ptr(), 1, nblk, _st()), "pack stem")
                self._stem_job_keep = jobs
                s.version = v
            return
        if s.packed_fwd is None or s.version != v or s.packed_fwd.device != w.device:
            s.packed_fwd = ops.pack_weight_fwd(w.detach(), out=s.packed_fwd if (s.packed_fwd is not None and s.packed_fwd.device == w.device) else None, stem=s.is_stem)
            s.packed_dgrad = None
            s.has_dgrad = False
            s.version = v
        if need_dgrad and (s.packed_dgrad is None or not getattr(s, "has_dgrad", False)) and not s.is_stem:
            s.packed_dgrad = ops.pack_weight_dgrad(w.detach())
            s.has_dgrad = True

    def flatten_parameters(self):
        """Re-point every parameter at a view of ONE flat fp32 buffer (same registration order as the flat
        gradient buffer) so the optimiser step and the gradient all-reduce are single passes over
        contiguous memory. Parameter objects keep their identity; state_dict / checkpoints are unchanged."""
        params = self._param_list()
        total = sum(p.numel() for p in params)
        dev = params[0].device
        if self.flat_w is not None and self.flat_w.device == dev and self.flat_w.numel() == total:
            off = 0
            ok = True
            for p in params:
                if p.data_ptr() != self.flat_w.data_ptr() + 4 * off:
                    ok = False
                    break
                off += p.numel()
            if ok:
                return self.flat_w
        flat = torch.empty(total, dtype=torch.float32, device=dev)
        off = 0
        with torch.no_grad():
            for p in params:
                v = flat[off:off + p.numel()].view_as(p)
                v.copy_(p.data)
                p.data = v
                off += p.numel()
        self.flat_w = flat
        self.weights_epoch += 1
        return flat

    def invalidate_packed(self):
        self.weights_epoch += 1

    def _ensure_grad_buffers(self):
        params = self._param_list()
        total = sum(p.numel() for p in params)
        ext = self.ext_flat_g
        if ext is not None and (self.flat_g is None or self.flat_g.data_ptr() != ext.data_ptr()):
            if ext.numel() < total or ext.device != self.device or ext.dtype != torch.float32:
                raise RuntimeError("external gradient buffer does not fit the model")
            self.flat_g = None
        if self.flat_g is None or self.flat_g.numel() != total or self.flat_g.device != self.device:
            self.flat_g = ext[:total] if ext is not None else torch.zeros(total, dtype=torch.float32, device=self.device)
            self.grad_views = {}
            off = 0
            for p in params:
                self.grad_views[id(p)] = self.flat_g[off:off + p.numel()].view_as(p)
                off += p.numel()
            wsz = 0
            self.wacc_off = {}
            for s in self.specs:
                if s.k > 1:
                    n = s.cout * (7 * STEM_KPITCH if s.is_stem else s.k * s.k * s.cin)   # stem: [Cout][7][kpitch] (row taps) or [Cout][160] (im2col)
                    self.wacc_off[s.name] = (wsz, n)
                    wsz += n
            self.wacc = torch.zeros(wsz, dtype=torch.float32, device=self.device)

    # ------------------------------------------------------------------ low-level launches
    def _conv(self, s: ConvSpec, x: Act, out_t: torch.Tensor, out_ld: int, Ho: int, Wo: int, taps, n_img: int,
              flags: int = 0, scale=None, shift=None, res: Optional[torch.Tensor] = None, res_ld: int = 0,
              stats=None, wgt=None, cin=None, cout=None, Hi=None, Wi=None, B=None):
        d = ops.make_conv_desc(B if B is not None else x.B, Hi if Hi is not None else x.H, Wi if Wi is not None else x.W,
                               cin if cin is not None else x.C, x.ld, n_img, Ho, Wo,
                               cout if cout is not None else s.cout, out_ld, taps, flags, res_ld, phase_view=x.phase_view)
        if stats is not None:
            d.stats_replicas = stats.numel() // (2 * d.Cout)
        ev = self._prof_begin()
        check(_lib.lib().iswm_conv_igemm(C.byref(d), x.ptr, (wgt if wgt is not None else s.packed_fwd).data_ptr(),
                                         out_t.data_ptr(), None if scale is None else scale.data_ptr(),
                                         None if shift is None else shift.data_ptr(),
                                         None if res is None else res.data_ptr(),
                                         None if stats is None else stats.data_ptr(), _st()), "conv_igemm " + s.name)
        self._prof_end(ev, "conv_igemm", 2.0 * d.B * Ho * Wo * d.Cout * (147 if s.is_stem else d.Cin * d.ntaps), "fwd " + s.name)

    def _prep_input(self, s: ConvSpec, x: Act):
        """Returns (conv input Act, taps, n_img, Ho, Wo) handling stride 2 by phase split / subsampling."""
        L = _lib.lib()
        if s.stride == 1:
            return x, ops.conv_taps(s.k, s.dilation), x.B, x.H, x.W
        assert s.stride == 2 and s.dilation == 1
        Ho, Wo = (x.H + 1) // 2, (x.W + 1) // 2
        # stride-2 convolutions read the parity phases of their dense input in place through a 5-D tensor map
        # (iswm_conv_desc.in_phase_view); odd sizes and misaligned channels go through phase_split / subsample2 copies
        if x.H % 2 == 0 and x.W % 2 == 0 and x.C % 64 == 0 and x.ld % 8 == 0:
            xv = Act(x.t, x.B, Ho, Wo, x.C, x.ld)
            xv.phase_view = True
            return xv, (ops.conv_taps(1, 1) if s.k == 1 else ops.conv_taps_s2_3x3()), x.B, Ho, Wo
        if s.k == 1:
            xs = Act.new(x.B, Ho, Wo, x.C, self.device)
            check(L.iswm_subsample2(x.ptr, x.ld, x.B, x.H, x.W, x.C, xs.ptr, _st()), "subsample2")
            return xs, ops.conv_taps(1, 1), x.B, Ho, Wo
        ph = torch.empty((4 * x.B, Ho, Wo, x.C), dtype=torch.bfloat16, device=self.device)
        check(L.iswm_phase_split(x.ptr, x.ld, x.B, x.H, x.W, x.C, ph.data_ptr(), _st()), "phase_split")
        xa = Act(ph, x.B, Ho, Wo, x.C, x.C)
        return xa, ops.conv_taps_s2_3x3(), 4 * x.B, Ho, Wo

    # ------------------------------------------------------------------ eval-mode unit: conv + folded BN (+res, relu)
    def _fold(self, s: ConvSpec):
        bn = s.bn
        # running statistics are updated by kernels through raw pointers and the affine through the flat master buffer
        # (fused optimisers, graph replays): neither bumps a tensor version, so the key also carries the engine's own
        # counters - `step` moves with every train-mode forward / graph replay, `weights_epoch` with every fused step
        key = (bn.weight._version, bn.bias._version, bn.running_mean._version, bn.running_var._version,
               self.weights_epoch, self.step)
        if s.fold_scale is None or s.fold_version != key or s.fold_scale.device != self.device:
            s.fold_scale = torch.empty(s.cout, dtype=torch.float32, device=self.device)
            s.fold_shift = torch.empty(s.cout, dtype=torch.float32, device=self.device)
            check(_lib.lib().iswm_bn_fold(bn.weight.data_ptr(), bn.bias.data_ptr(), bn.running_mean.data_ptr(),
                                          bn.running_var.data_ptr(), BN_EPS, s.cout, s.fold_scale.data_ptr(),
                                          s.fold_shift.data_ptr(), _st()), "bn_fold")
            s.fold_version = key

    def _unit_eval(self, s: ConvSpec, x: Act, relu=True, residual: Optional[Act] = None, out: Optional[Act] = None) -> Act:
        self._pack(s, False)
        self._fold(s)
        xin, taps, n_img, Ho, Wo = self._prep_input(s, x)
        if out is None:
            out = Act.new(x.B, Ho, Wo, s.cout, self.device)
        flags = _lib.EPI_AFFINE | (_lib.EPI_RELU if relu else 0) | (_lib.EPI_RESIDUAL if residual is not None else 0)
        self._conv(s, xin, out.t, out.ld, Ho, Wo, taps, n_img, flags, s.fold_scale, s.fold_shift,
                   None if residual is None else residual.t, 0 if residual is None else residual.ld)
        self._tap(s.name, out)
        return out

    # ------------------------------------------------------------------ train-mode unit: conv(+stats) -> BN apply, taped
    def _unit_train(self, s: ConvSpec, x: Act, relu=True, residual: Optional[Act] = None, out: Optional[Act] = None,
                    drop_p: float = 0.0, need_dx: bool = True, dy_into: Optional[Callable[[], torch.Tensor]] = None) -> Act:
        """`dy_into`: called in backward, returns the [B,Ho,Wo,Cout] (possibly channel-sliced) view the BatchNorm backward
        writes this unit's pre-activation gradient into instead of a private buffer (ASPP: slices of one concatenated buffer)."""
        L = _lib.lib()
        self._pack(s, need_dx)
        xin, taps, n_img, Ho, Wo = self._prep_input(s, x)
        B = x.B
        M = B * Ho * Wo
        Cout = s.cout
        raw = torch.empty((B, Ho, Wo, Cout), dtype=torch.bfloat16, device=self.device)
        rep = self._stats_rep(Cout)
        sync = self.bn_sync is not None
        stats = self._stats_slot(2 * Cout * rep + (1 if sync else 0))     # synchronised: + this rank's row count
        self._conv(s, xin, raw, Cout, Ho, Wo, taps, n_img, _lib.EPI_STATS, stats=stats)
        if sync:
            stats, rep = self._bn_exchange([(stats, rep)], 2 * Cout, M)[0], 1
        if out is None:
            out = Act.new(B, Ho, Wo, Cout, self.device)
        save = self._save_slot(2 * Cout)
        bn = s.bn
        # dropout seed = by-value part (unit position) + 1000003 * the DEVICE step counter: identical masks in forward and
        # backward of one step, a fresh one every step, and valid inside a replayed CUDA graph (iswm_b200.graphs)
        seed = (self.seed + len(self.tape)) & 0xFFFFFFFFFFFF
        step_ptr = self._step_dev.data_ptr() if drop_p > 0.0 else None
        # residual units: the ReLU sign bits go out as one byte per 8 channels, read back by the backward kernels
        # instead of the block output
        bits = torch.empty((M, Cout // 8), dtype=torch.uint8, device=self.device) if (relu and residual is not None) else None
        ev = self._prof_begin()
        apply_args = (bn.weight.data_ptr(), bn.bias.data_ptr(), BN_EPS, BN_MOMENTUM, bn.running_mean.data_ptr(), bn.running_var.data_ptr(),
                      bn.num_batches_tracked.data_ptr(), save.data_ptr(), save[Cout:].data_ptr(),
                      None if residual is None else residual.ptr, 0 if residual is None else residual.ld,
                      1 if relu else 0, drop_p, seed, step_ptr, out.ptr, out.ld, None if bits is None else bits.data_ptr(), _st())
        if sync:
            check(L.iswm_bn_train_apply_global(raw.data_ptr(), Cout, stats.data_ptr(), M, Cout, *apply_args), "bn_train_apply_global " + s.name)
        else:
            check(L.iswm_bn_train_apply(raw.data_ptr(), Cout, stats.data_ptr(), rep, M, Cout, *apply_args), "bn_train_apply " + s.name)
        # HBM-bound kernels are recorded with their algorithmic BYTES in the flops slot (kernel name prefixed "hbm:")
        self._prof_end(ev, "hbm:bn_train_apply", 2.0 * M * Cout * (3 if residual is not None else 2) + (M * Cout / 8 if bits is not None else 0), "bn_apply " + s.name)
        self._tap(s.name, out)
        if self.debug_taps is not None:
            self.debug_taps[s.name + ":raw"] = raw.float().permute(0, 3, 1, 2).cpu()

        def backward():
            dout = out.grad
            pend_bits = None
            if dout is None and out.pending is not None:
                # this unit's output was the identity operand of a block-closing add + ReLU (downsample branch): its gradient is
                # the block-output gradient gated by the block's ReLU sign bits, which the kernels apply on the fly (mode 2)
                dout, pend_bits = out.pending
                out.pending = None
            assert dout is not None, f"no gradient reached {s.name}"
            rec = None
            if self.debug_units is not None:
                rec = dict(name=s.name, k=s.k, stride=s.stride, dilation=s.dilation, relu=relu, x=x.t.clone(), raw=raw.clone(),
                           out=out.t.clone(), dout=dout.t.clone(), mean=save[:Cout].clone(), invstd=save[Cout:2 * Cout].clone(),
                           gamma=bn.weight.detach().clone(), beta=bn.bias.detach().clone(), w=s.conv.weight.detach().clone(),
                           residual=None if residual is None else residual.t.clone(),
                           xgrad_before=None if x.grad is None else x.grad.t.clone(),
                           resgrad_before=None if (residual is None or residual.grad is None) else residual.grad.t.clone())
            sums = self._stats_slot(2 * Cout + 2)
            # the ReLU mask comes from the sign bits where a residual was added (post add + ReLU); otherwise the kernel
            # recomputes it from raw (one tensor read less in each pass)
            act_ptr, relu_mode = None, (1 if relu else 0)
            if bits is not None:
                act_ptr, relu_mode = bits.data_ptr(), 2
            if pend_bits is not None:
                assert not relu and bits is None
                act_ptr, relu_mode = pend_bits.data_ptr(), 2
            dy = dy_into() if dy_into is not None else torch.empty((B, Ho, Wo, Cout), dtype=torch.bfloat16, device=self.device)
            dy_ld = dy.stride(2)
            dz_ptr, dz_ld, dz_tmp = None, 0, None
            defer_dz = (residual is not None and residual.grad is None and residual.masked_ok and bits is not None and drop_p == 0.0
                        and self.masked_identity and self.debug_units is None and residual.ld == residual.C and dout.ld == Cout and Cout % 64 == 0)
            if defer_dz:
                # the identity path's gradient dz = dout . relu_mask is NOT written: the block's conv1 data gradient (the only
                # other contribution to the block input's gradient) reads dout and the sign bits in its epilogue instead
                residual.pending = (dout, bits)
            elif residual is not None:
                if residual.grad is None:
                    residual.new_grad()
                    dz_ptr, dz_ld = residual.grad.ptr, residual.C
                else:
                    assert residual.grad.ld == residual.C
                    dz_tmp = torch.empty_like(residual.grad.t)
                    dz_ptr, dz_ld = dz_tmp.data_ptr(), residual.C
            nmask = (1.0 / 16 if bits is not None else 1) if act_ptr is not None else 0
            ev = self._prof_begin()
            check(L.iswm_bn_bwd_reduce(dout.ptr, dout.ld, raw.data_ptr(), Cout, act_ptr, out.ld, M, Cout,
                                       save.data_ptr(), save[Cout:].data_ptr(), bn.weight.data_ptr(), bn.bias.data_ptr(),
                                       relu_mode, drop_p, seed, step_ptr, sums.data_ptr(), _st()), "bn_bwd_reduce " + s.name)
            self._prof_end(ev, "hbm:bn_bwd_reduce", 2.0 * M * Cout * (2 + nmask), "bn_bwd_reduce " + s.name)
            ev = self._prof_begin()
            head = (dout.ptr, dout.ld, raw.data_ptr(), Cout, act_ptr, out.ld, M, Cout,
                    bn.weight.data_ptr(), bn.bias.data_ptr(), save.data_ptr(), save[Cout:].data_ptr())
            tail = (relu_mode, drop_p, seed, step_ptr, dy.data_ptr(), dy_ld, dz_ptr, dz_ld,
                    self.grad_views[id(bn.weight)].data_ptr(), self.grad_views[id(bn.bias)].data_ptr(), _st())
            if sync:
                gsums = self._bn_exchange([(sums, 1)], 2 * Cout, M)[0]
                check(L.iswm_bn_bwd_apply_global(*head, gsums.data_ptr(), sums.data_ptr(), *tail), "bn_bwd_apply_global " + s.name)
            else:
                check(L.iswm_bn_bwd_apply(*head, sums.data_ptr(), *tail), "bn_bwd_apply " + s.name)
            self._prof_end(ev, "hbm:bn_bwd_apply", 2.0 * M * Cout * (3 + nmask + (1 if dz_ptr is not None else 0)), "bn_bwd_apply " + s.name)
            if dz_tmp is not None:
                check(L.iswm_add_bf16(residual.grad.ptr, dz_tmp.data_ptr(), dz_tmp.numel(), residual.grad.ptr, _st()), "add_bf16")
            out.grad = None
            self._conv_backward(s, x, xin, taps, n_img, Ho, Wo, dy, need_dx)
            if rec is not None:
                rec.update(dy=dy.clone(), dW=self.grad_views[id(s.conv.weight)].clone(), dgamma=self.grad_views[id(bn.weight)].clone(),
                           dbeta=self.grad_views[id(bn.bias)].clone(), xgrad_after=None if x.grad is None else x.grad.t.clone(),
                           resgrad_after=None if residual is None else residual.grad.t.clone())
                self.debug_units.append(rec)

        self.tape.append(backward)
        return out

    def _conv_raw(self, s: ConvSpec, x: Act):
        """Train-mode convolution alone: raw (pre-BN) bf16 output + its per-channel statistics; the BatchNorm comes later."""
        self._pack(s, True)
        xin, taps, n_img, Ho, Wo = self._prep_input(s, x)
        raw = torch.empty((x.B, Ho, Wo, s.cout), dtype=torch.bfloat16, device=self.device)
        stats = self._stats_slot(2 * s.cout * self._stats_rep(s.cout) + (1 if self.bn_sync is not None else 0))
        self._conv(s, xin, raw, s.cout, Ho, Wo, taps, n_img, _lib.EPI_STATS, stats=stats)
        return raw, stats, xin, taps, n_img, Ho, Wo

    def _bn_side(self, bn, stats, save, Cc, train_fwd: bool, rep=None):
        return _lib.BnSide(stats.data_ptr() if stats is not None else None, bn.weight.data_ptr(), bn.bias.data_ptr(),
                           bn.running_mean.data_ptr() if train_fwd else None, bn.running_var.data_ptr() if train_fwd else None,
                           bn.num_batches_tracked.data_ptr() if train_fwd else None, save.data_ptr(), save[Cc:].data_ptr(),
                           rep if rep is not None else (1 if stats is None else stats.numel() // (2 * Cc)))

    def _bn_exchange(self, srcs, n: int, rows: int):
        """Synchronised BatchNorm: fp64 slots holding the sums over every rank of the vectors `srcs` [(slot, replicas)] of n
        values, followed by the global row count (this rank contributes `rows`), from the same slots of every rank's arena."""
        dsts = [self._stats_slot(n + 1) for _ in srcs]
        self.bn_sync(srcs, dsts, n, rows, _st())
        return dsts

    def _unit_train_dual(self, s: ConvSpec, x: Act, sds: ConvSpec, dsc) -> Act:
        """Closing unit of a bottleneck block with a downsample branch (resnet.py:110-118): out = relu(bn3(conv3(x)) +
        bn_ds(conv_ds(block input))), both BatchNorms in one kernel per pass (csrc/bn_dual.cu). `dsc` = _conv_raw(sds, block input)
        + (list that receives the downsample branch's dy for its taped backward,)."""
        L = _lib.lib()
        raw, stats, xin, taps, n_img, Ho, Wo = self._conv_raw(s, x)
        raw_ds, stats_ds, _, _, _, Ho_ds, Wo_ds, ds_dy = dsc
        assert (Ho, Wo) == (Ho_ds, Wo_ds) and s.cout == sds.cout
        B, Cout = x.B, s.cout
        M = B * Ho * Wo
        out = Act.new(B, Ho, Wo, Cout, self.device)
        save, save_ds = self._save_slot(2 * Cout), self._save_slot(2 * Cout)
        bits = torch.empty((M, Cout // 8), dtype=torch.uint8, device=self.device)
        sync = self.bn_sync is not None
        if sync:
            # both BatchNorms' statistics are ready here: ONE exchange carries the two vectors
            rep = self._stats_rep(Cout)
            stats, stats_ds = self._bn_exchange([(stats, rep), (stats_ds, rep)], 2 * Cout, M)
        a_side = self._bn_side(s.bn, stats, save, Cout, True, 1 if sync else None)
        d_side = self._bn_side(sds.bn, stats_ds, save_ds, Cout, True, 1 if sync else None)
        ev = self._prof_begin()
        fwd = L.iswm_bn_dual_train_apply_global if sync else L.iswm_bn_dual_train_apply
        check(fwd(raw.data_ptr(), Cout, C.byref(a_side), raw_ds.data_ptr(), Cout, C.byref(d_side), M, Cout,
                  BN_EPS, BN_MOMENTUM, out.ptr, out.ld, bits.data_ptr(), _st()), "bn_dual_train_apply " + s.name)
        self._prof_end(ev, "hbm:bn_train_apply", 2.0 * M * Cout * 3 + M * Cout / 8, "bn_apply " + s.name + "+ds")

        def backward():
            dout = out.grad
            assert dout is not None and dout.ld == Cout, f"no dense gradient reached {s.name}"
            sums, sums_ds = self._stats_slot(2 * Cout + 2), self._stats_slot(2 * Cout + 2)
            a_b, d_b = self._bn_side(s.bn, None, save, Cout, False), self._bn_side(sds.bn, None, save_ds, Cout, False)
            dy = torch.empty((B, Ho, Wo, Cout), dtype=torch.bfloat16, device=self.device)
            dy_ds = torch.empty((B, Ho, Wo, Cout), dtype=torch.bfloat16, device=self.device)
            ev = self._prof_begin()
            check(L.iswm_bn_dual_bwd_reduce(dout.ptr, Cout, bits.data_ptr(), raw.data_ptr(), Cout, C.byref(a_b), raw_ds.data_ptr(), Cout,
                                            C.byref(d_b), M, Cout, sums.data_ptr(), sums_ds.data_ptr(), _st()), "bn_dual_bwd_reduce " + s.name)
            self._prof_end(ev, "hbm:bn_bwd_reduce", 2.0 * M * Cout * 3 + M * Cout / 8, "bn_bwd_reduce " + s.name + "+ds")
            gv = self.grad_views
            ev = self._prof_begin()
            tail = (M, Cout, dy.data_ptr(), Cout, dy_ds.data_ptr(), Cout, gv[id(s.bn.weight)].data_ptr(), gv[id(s.bn.bias)].data_ptr(),
                    gv[id(sds.bn.weight)].data_ptr(), gv[id(sds.bn.bias)].data_ptr(), _st())
            if sync:
                g, g_ds = self._bn_exchange([(sums, 1), (sums_ds, 1)], 2 * Cout, M)
                check(L.iswm_bn_dual_bwd_apply_global(dout.ptr, Cout, bits.data_ptr(), raw.data_ptr(), Cout, C.byref(a_b), g.data_ptr(), sums.data_ptr(),
                                                      raw_ds.data_ptr(), Cout, C.byref(d_b), g_ds.data_ptr(), sums_ds.data_ptr(), *tail),
                      "bn_dual_bwd_apply_global " + s.name)
            else:
                check(L.iswm_bn_dual_bwd_apply(dout.ptr, Cout, bits.data_ptr(), raw.data_ptr(), Cout, C.byref(a_b), sums.data_ptr(),
                                               raw_ds.data_ptr(), Cout, C.byref(d_b), sums_ds.data_ptr(), *tail), "bn_dual_bwd_apply " + s.name)
            self._prof_end(ev, "hbm:bn_bwd_apply", 2.0 * M * Cout * 5 + M * Cout / 8, "bn_bwd_apply " + s.name + "+ds")
            out.grad = None
            self._conv_backward(s, x, xin, taps, n_img, Ho, Wo, dy, True)
            ds_dy.append(dy_ds)                       # the downsample convolution's backward runs after conv1's (taped in forward())

        self.tape.append(backward)
        return out

    def _conv_backward(self, s: ConvSpec, x: Act, xin: Act, taps, n_img, Ho, Wo, dy: torch.Tensor, need_dx: bool):
        """Weight gradient into the flat fp32 buffer and data gradient into x.grad (assign or accumulate)."""
        L = _lib.lib()
        B, Cout = x.B, s.cout
        dy_ld = dy.stride(-2) if dy.dim() >= 2 else dy.shape[-1]          # a channel slice of a wider buffer keeps that buffer's pitch
        gview = self.grad_views[id(s.conv.weight)]
        d = ops.make_conv_desc(B, xin.H, xin.W, xin.C, xin.ld, n_img, Ho, Wo, Cout, dy_ld, taps, phase_view=xin.phase_view)
        dst = gview if s.k == 1 else self.wacc[self.wacc_off[s.name][0]:self.wacc_off[s.name][0] + self.wacc_off[s.name][1]]
        flops = 2.0 * B * Ho * Wo * Cout * s.cin * s.k * s.k
        layer = s.name.split(".")[1] if s.name.startswith("backbone.layer") else None
        if layer in GROUP_WGRAD_LAYERS and self.debug_units is None:
            if self._wq and self._wq_layer != layer:
                self._flush_wgrad_group()
            self._wq_layer = layer
            self._wq.append((d, xin.t, dy, dst, s, flops, gview))
            return self._conv_backward_dx(s, x, dy, dy_ld, taps, Ho, Wo, need_dx)
        if self._wq:
            self._flush_wgrad_group()
        with self._wgrad_ctx(dy, xin.t):
            ev = self._prof_begin()
            check(L.iswm_conv_wgrad(C.byref(d), xin.ptr, dy.data_ptr(), dst.data_ptr(), _st()), "conv_wgrad " + s.name)
            self._prof_end(ev, "conv_wgrad", flops, "wgrad " + s.name)
            if s.k != 1:
                if not self._batched_unpack():
                    check(L.iswm_unpack_wgrad(dst.data_ptr(), Cout, s.cin, s.k * s.k, s.cin, s.k * s.k * s.cin, 1.0, gview.data_ptr(), _st()), "unpack_wgrad")
            # notifications are issued in the same context: a bucket all-reduce launched from here orders itself after
            # this stream, which has seen everything the main stream produced up to this unit (BatchNorm gradients too)
            self._notify(s.conv.weight)
            if s.bn is not None:
                self._notify(s.bn.weight)
                self._notify(s.bn.bias)
        self._conv_backward_dx(s, x, dy, dy_ld, taps, Ho, Wo, need_dx)

    def _flush_wgrad_group(self):
        """One grouped launch for the queued weight gradients of a layer (side stream, after everything the main stream has
        produced so far), then their unpack / gradient-ready notifications."""
        q, self._wq, self._wq_layer = self._wq, [], None
        if not q:
            return
        L = _lib.lib()
        keep = [t for job in q for t in (job[1], job[2])]
        with self._wgrad_ctx(*keep):
            ev = self._prof_begin()
            ops.conv_wgrad_grouped([(d, xt, dy, dst) for (d, xt, dy, dst, _, _, _) in q], _st())
            self._prof_end(ev, "conv_wgrad", sum(job[5] for job in q), "wgrad group " + q[0][4].name.split(".")[1])
            for (d, xt, dy, dst, s, _, gview) in q:
                if s.k != 1 and not self._batched_unpack():
                    check(L.iswm_unpack_wgrad(dst.data_ptr(), s.cout, s.cin, s.k * s.k, s.cin, s.k * s.k * s.cin, 1.0, gview.data_ptr(), _st()), "unpack_wgrad")
                self._notify(s.conv.weight)
                if s.bn is not None:
                    self._notify(s.bn.weight)
                    self._notify(s.bn.bias)

    def _conv_backward_dx(self, s: ConvSpec, x: Act, dy: torch.Tensor, dy_ld: int, taps, Ho, Wo, need_dx: bool):
        """Data gradient into x.grad (assign or accumulate)."""
        L = _lib.lib()
        B, Cout = x.B, s.cout
        if not need_dx:
            return
        Cin = s.cin
        if s.stride == 1:
            dtaps = [(-a, -b, 0) for (a, b, _) in taps]
            self._dgrad_into(s, x, dy, dy_ld, x.H, x.W, dtaps, x.H, x.W)
        elif s.k == 3:
            # stride-2 3x3: each of the four PARITY PHASES of dx is its own small convolution over dy with a subset of the taps
            # (dx[2a+pu, 2b+pv] = sum over taps r = pu+1 (mod 2), s = pv+1 (mod 2) of dy[a + (r==0), b + (s==0)] . w[r,s]):
            # 1 + 2 + 2 + 4 taps instead of 9 taps over a zero-stuffed tensor (4x dead MACs and a helper pass)
            fresh = x.grad is None
            if fresh:
                x.new_grad()
            g = x.grad
            H, W = x.H, x.W
            flags, res_ld = (0, 0) if fresh else (_lib.EPI_RESIDUAL, g.ld)
            for pu in (0, 1):
                rs = [(1, 0)] if pu == 0 else [(0, 1), (2, 0)]            # (forward tap row r, dy row offset)
                for pv in (0, 1):
                    ss = [(1, 0)] if pv == 0 else [(0, 1), (2, 0)]
                    Hp, Wp = (H - pu + 1) // 2, (W - pv + 1) // 2
                    if Hp <= 0 or Wp <= 0:
                        continue
                    ptaps = [(di, dj, 0) for (r, di) in rs for (sx, dj) in ss]
                    wt = [r * 3 + sx for (r, di) in rs for (sx, dj) in ss]
                    dd = ops.make_conv_desc(B, Ho, Wo, Cout, dy_ld, B, Hp, Wp, Cin, g.ld, ptaps, flags, res_ld, wtaps=wt,
                                            out_strides=(2 * g.ld, 2 * W * g.ld, H * W * g.ld), w_ntaps=9)
                    base = g.ptr + 2 * (pu * W + pv) * g.ld
                    ev = self._prof_begin()
                    check(L.iswm_conv_igemm(C.byref(dd), dy.data_ptr(), s.packed_dgrad.data_ptr(), base, None, None,
                                            None if fresh else base, None, _st()), "dgrad (phase) " + s.name)
                    # algorithmic FLOPs of the whole data gradient = those of the forward conv; booked on the last phase
                    self._prof_end(ev, "conv_igemm", 2.0 * B * Ho * Wo * Cout * Cin * 9 if (pu, pv) == (1, 1) else 0.0, "dgrad " + s.name)
        else:
            # stride-2 1x1 (downsample branch): the data gradient lives on the even-even phase of x only
            fresh = x.grad is None
            if fresh:
                x.new_grad()
                x.grad.t.zero_()
            g = x.grad
            H, W = x.H, x.W
            dd = ops.make_conv_desc(B, Ho, Wo, Cout, dy_ld, B, Ho, Wo, Cin, g.ld, [(0, 0, 0)], _lib.EPI_RESIDUAL, g.ld,
                                    out_strides=(2 * g.ld, 2 * W * g.ld, H * W * g.ld))
            ev = self._prof_begin()
            check(L.iswm_conv_igemm(C.byref(dd), dy.data_ptr(), s.packed_dgrad.data_ptr(), g.ptr, None, None, g.ptr, None, _st()), "dgrad " + s.name)
            self._prof_end(ev, "conv_igemm", 2.0 * B * Ho * Wo * Cout * Cin, "dgrad " + s.name)

    def _batched_unpack(self) -> bool:
        """k x k weight gradients leave their [Cout][tap][Cin] accumulators in ONE launch at the end of the sweep -
        unless somebody consumes gradients tensor by tensor (data-parallel bucket hooks, the unit-replay recorder)."""
        return self.batch_unpack and self.grad_ready_hook is None and self.debug_units is None

    def _unpack_all(self):
        sig = (self.wacc.data_ptr(), self.flat_g.data_ptr())
        if getattr(self, "_unpack_sig", None) != sig:
            jobs = []
            for s in self.specs:
                if s.k > 1 and not s.is_stem:
                    off, n = self.wacc_off[s.name]
                    jobs.append((self.wacc.data_ptr() + 4 * off, self.grad_views[id(s.conv.weight)].data_ptr(), s.cout, s.cin, s.k * s.k))
            arr, self._unpack_blocks = _lib.fill_unpack_jobs(jobs)
            self._unpack_jobs = torch.frombuffer(bytearray(bytes(arr)), dtype=torch.uint8).clone().to(self.device)
            self._unpack_njobs = len(jobs)
            self._unpack_sig = sig
        check(_lib.lib().iswm_unpack_wgrad_batched(self._unpack_jobs.data_ptr(), self._unpack_njobs, self._unpack_blocks, _st()), "unpack_wgrad_batched")

    def _dgrad_into(self, s: ConvSpec, x: Act, dy: torch.Tensor, dy_ld: int, Hi, Wi, dtaps, Ho, Wo):
        L = _lib.lib()
        B, Cin, Cout = x.B, s.cin, s.cout
        flags, res, mask = 0, None, None
        if x.grad is None:
            x.new_grad()
            if x.pending is not None:              # + (block-output gradient where the block's ReLU was active)
                res, mbits = x.pending
                x.pending = None
                flags, mask = _lib.EPI_RESIDUAL | _lib.EPI_RES_MASK, mbits
        else:
            assert x.pending is None
            flags, res = _lib.EPI_RESIDUAL, x.grad
        g = x.grad
        dd = ops.make_conv_desc(B, Hi, Wi, Cout, dy_ld, B, Ho, Wo, Cin, g.ld, dtaps, flags, g.ld if res is None else res.ld)
        ev = self._prof_begin()
        check(L.iswm_conv_igemm_ex(C.byref(dd), dy.data_ptr(), s.packed_dgrad.data_ptr(), g.ptr, None, None,
                                   None if res is None else res.ptr, None, None if mask is None else mask.data_ptr(), _st()), "dgrad " + s.name)
        # algorithmic FLOPs of a data gradient = those of the forward conv it differentiates (no credit
        # for the zero-stuffed positions of the stride-2 case)
        fwd_pix = B * (Ho // s.stride if s.stride > 1 else Ho) * (Wo // s.stride if s.stride > 1 else Wo)
        self._prof_end(ev, "conv_igemm", 2.0 * fwd_pix * Cout * Cin * len(dtaps), "dgrad " + s.name)

    # ------------------------------------------------------------------ weight-gradient stream
    class _NullCtx:
        def __enter__(self): return None
        def __exit__(self, *a): return False

    class _SideCtx:
        def __init__(self, stream):
            self.ctx = torch.cuda.stream(stream)
            self.handle = stream.cuda_stream

        def __enter__(self):
            self.ctx.__enter__()
            self.prev = _StreamCache.handle
            _StreamCache.handle = self.handle
            return self

        def __exit__(self, *a):
            _StreamCache.handle = self.prev
            return self.ctx.__exit__(*a)

    def _wgrad_ctx(self, *keep_alive: torch.Tensor):
        """Context in which weight-gradient kernels (and the gradient-ready notifications that depend on them) are
        issued: the side stream, after everything enqueued so far on the main stream. `keep_alive` tensors are read
        there, so the caching allocator must not recycle them before the side stream is done with them."""
        if not self.async_wgrad or self.debug_units is not None:      # the unit-replay recorder reads dW right away
            return Engine._NullCtx()
        if self._wstream is None or self._wstream.device != self.device:
            self._wstream = torch.cuda.Stream(self.device)
        main = torch.cuda.current_stream(self.device)
        self._wstream.wait_event(main.record_event())
        # held until the join below: their memory returns to the (main-stream) allocator pool only after the main
        # stream has waited for the side stream, so no record_stream() bookkeeping (which makes the allocator grow
        # and stall when the host runs far ahead) is needed
        self._wgrad_keep.extend(keep_alive)
        return Engine._SideCtx(self._wstream)

    class _HandleCtx:
        """Launch the library kernels issued inside on `stream` WITHOUT changing torch's current stream: tensors are still
        allocated from (and returned to) the main stream's pool, so they must stay referenced until the join."""

        def __init__(self, stream):
            self.handle = stream.cuda_stream

        def __enter__(self):
            self.prev = _StreamCache.handle
            _StreamCache.handle = self.handle
            return self

        def __exit__(self, *a):
            _StreamCache.handle = self.prev
            return False

    def _fwd_fork(self):
        """Context for a forward branch nothing on the main chain consumes for a while (low-level projection, pooled ASPP
        branch): its launches go to the side stream after everything enqueued so far, and run under the main chain's
        convolutions (which leave 20 of the 148 SMs idle at 128 tiles). `_fwd_join()` makes the main stream wait."""
        if not (self.async_wgrad and self.fwd_overlap) or self.profile is not None or self.debug_units is not None or self.debug_taps is not None:
            return Engine._NullCtx()
        if self._wstream is None or self._wstream.device != self.device:
            self._wstream = torch.cuda.Stream(self.device)
        self._wstream.wait_event(torch.cuda.current_stream(self.device).record_event())
        self._fwd_forked = True
        return Engine._HandleCtx(self._wstream)

    def _fwd_join(self):
        if getattr(self, "_fwd_forked", False):
            torch.cuda.current_stream(self.device).wait_stream(self._wstream)
            self._fwd_forked = False
        self._fwd_keep = []

    def _wgrad_join(self):
        if self.async_wgrad and self._wstream is not None:
            torch.cuda.current_stream(self.device).wait_stream(self._wstream)
        self._wgrad_keep = []

    def _prof_begin(self):
        if self.profile is None:
            return None
        ev = torch.cuda.Event(enable_timing=True)
        ev.record()
        return ev

    def _prof_end(self, ev0, kernel: str, flops: float, tag: str = ""):
        if ev0 is None:
            return
        ev1 = torch.cuda.Event(enable_timing=True)
        ev1.record()
        self.profile.append((kernel, flops, ev0, ev1, tag))

    def _tap(self, name: str, a: Act):
        if self.debug_taps is not None:
            self.debug_taps[name] = a.t.float().permute(0, 3, 1, 2).cpu()

    def _notify(self, p):
        if self.grad_ready_hook is not None:
            self.grad_ready_hook(p)

    # per-step scratch carved from two zeroed buffers: fp64 accumulators (conv-epilogue statistics, BN-backward sums)
    # and fp32 saved mean / invstd
    def scratch_need(self, sync: bool) -> int:
        """fp64 elements of the per-step scratch arena; depends on the model's channel counts only (not on the batch)."""
        need = 0
        for s in self.specs:
            if s.bn is not None:
                need += 2 * s.cout * (self._stats_rep(s.cout) + 1) + 192    # fwd stats (x copies) + bwd sums and barrier counter (fp64); covers mean/invstd (fp32) too
                if sync:
                    need += 4 * s.cout + 192                                  # + row counts, global forward and backward sums (+ counts)
        return need + 4096

    def _begin_scratch(self):
        need = self.scratch_need(self.bn_sync is not None)
        ext = self.ext_scratch64
        if ext is not None and (getattr(self, "_scratch64", None) is None or self._scratch64.data_ptr() != ext.data_ptr()):
            if ext.numel() < need or ext.device != self.device or ext.dtype != torch.float64:
                raise RuntimeError("external statistics arena does not fit the model")
            self._scratch64 = ext
            self._scratch32 = torch.empty(need, dtype=torch.float32, device=self.device)
        if getattr(self, "_scratch64", None) is None or self._scratch64.numel() < need or self._scratch64.device != self.device:
            self._scratch64 = torch.empty(need, dtype=torch.float64, device=self.device)
            self._scratch32 = torch.empty(need, dtype=torch.float32, device=self.device)
        self._scratch64.zero_()
        self._scratch64_off = 0
        self._scratch32_off = 0

    @staticmethod
    def _stats_rep(cout: int) -> int:
        """Copies of a convolution's statistics accumulator (iswm_conv_desc.stats_replicas): narrow layers end every CTA on the
        same 2*Cout addresses, so their fp64 atomics are spread over 4 copies that the BatchNorm kernel folds (cfg2 same-box: 12.87 -> 12.65 ms/step; 8 copies: 12.73)."""
        return 4 if cout <= 128 else 1

    def _stats_slot(self, n: int) -> torch.Tensor:
        """zeroed fp64 accumulator slot"""
        n_al = (n + 63) // 64 * 64
        t = self._scratch64[self._scratch64_off:self._scratch64_off + n]
        self._scratch64_off += n_al
        assert self._scratch64_off <= self._scratch64.numel(), "scratch exhausted"
        return t

    def _save_slot(self, n: int) -> torch.Tensor:
        """fp32 slot (fully overwritten by its producer)"""
        n_al = (n + 63) // 64 * 64
        t = self._scratch32[self._scratch32_off:self._scratch32_off + n]
        self._scratch32_off += n_al
        assert self._scratch32_off <= self._scratch32.numel(), "scratch exhausted"
        return t

    # ------------------------------------------------------------------ forward
    def forward(self, x: torch.Tensor, train: bool, lowres: bool = False, fused_tail: bool = False) -> torch.Tensor:
        """x: fp32 NCHW [B,3,H,W] on CUDA -> fp32 NCHW logits [B,num_classes,H,W]; with `lowres` the classifier's fp32 NHWC
        [B,H/4,W/4,num_classes] output, for consumers that fuse the final upsample: ops.predict_epilogue in eval mode, and in
        train mode (`fused_tail=True`, then backward_tail() instead of backward()) the fused upsample + criterion + adjoint."""
        if not x.is_cuda:                    # before any CUDA call: the message must be ours, not the driver's
            raise RuntimeError("iswm_b200 runs on CUDA only: move the model and the input to a B200 (no CPU fallback)")
        with _StreamScope():
            return self._forward(x, train, lowres, fused_tail)

    def _forward(self, x: torch.Tensor, train: bool, lowres: bool = False, fused_tail: bool = False) -> torch.Tensor:
        self._check_device(x)
        if x.dim() != 4 or x.shape[1] != self.stem.cin:
            raise ValueError(f"expected [B,{self.stem.cin},H,W] input, got {tuple(x.shape)}")
        x = x.contiguous().float()
        self._image = x if self.debug_units is not None else None
        L = _lib.lib()
        if train:
            # an eval / predict forward between a train forward and its backward leaves the pending tape, the BatchNorm
            # accumulators and the saved head tensors alone; a second TRAIN forward supersedes the first (generation
            # counter: the stale autograd node raises instead of sweeping the wrong tape)
            self.tape = []
            self.generation += 1
            self._begin_scratch()
            self._ensure_grad_buffers()
            self.step += 1
            if getattr(self, "_step_dev", None) is None or self._step_dev.device != self.device:
                self._step_dev = torch.full((1,), self.step - 1, dtype=torch.int64, device=self.device)
            self._step_dev.add_(1)          # on the stream (and in the graph, when captured): == self.step in eager mode
        unit = self._unit_train if train else self._unit_eval
        B, _, H, W = x.shape
        dev = self.device

        # ---- stem: 7x7/s2 conv as im2col GEMM -> BN -> ReLU -> maxpool 3x3/s2 (resnet.py:144-148)
        H1, W1 = (H + 1) // 2, (W + 1) // 2
        if self.stem_rows:
            # x-unrolled rows, phase-major over the row parity: [2][B][H1][W1][kpitch]; the 7 kernel rows are the convolution's taps
            rows = torch.empty((2 * B, H1, W1, STEM_KPITCH), dtype=torch.bfloat16, device=dev)
            ev = self._prof_begin()
            check(L.iswm_stem_rows(x.data_ptr(), B, self.stem.cin, H, W, H1, W1, STEM_KPITCH, rows.data_ptr(), _st()), "stem_rows")
            self._prof_end(ev, "hbm:stem_rows", 4.0 * x.numel() + 2.0 * rows.numel(), "stem_rows")
            colA = Act(rows, B, H1, W1, STEM_KPITCH, STEM_KPITCH)
            stem_taps = [((r - 3 - ((r + 1) & 1)) // 2, 0, (r + 1) & 1) for r in range(7)]
            stem_out = self._stem_unit(colA, B, H1, W1, train, stem_taps, 2 * B)
        else:
            Kp = 160
            col = torch.empty((B * H1 * W1, Kp), dtype=torch.bfloat16, device=dev)
            check(L.iswm_stem_im2col(x.data_ptr(), B, 3, H, W, H1, W1, Kp, col.data_ptr(), _st()), "stem_im2col")
            colA = Act(col.view(1, 1, B * H1 * W1, Kp), 1, 1, B * H1 * W1, Kp, Kp)
            stem_out = self._stem_unit(colA, B, H1, W1, train)
        H2, W2 = (H1 + 1) // 2, (W1 + 1) // 2
        if isinstance(stem_out, tuple):                  # fused stem tail: (pooled activation) came out of _stem_unit directly
            pooled = stem_out[0]
            stem_out = None
        else:
            pooled = Act.new(B, H2, W2, 64, dev)
            idx = torch.empty((B, H2, W2, 64), dtype=torch.uint8, device=dev) if train else None
            check(L.iswm_maxpool_fwd(stem_out.ptr, B, H1, W1, 64, H2, W2, pooled.ptr, None if idx is None else idx.data_ptr(), _st()), "maxpool_fwd")
        if train and stem_out is not None:
            def pool_bwd():
                g = pooled.grad
                assert g.ld == 64
                stem_out.new_grad()
                check(L.iswm_maxpool_bwd(g.ptr, idx.data_ptr(), B, H1, W1, 64, H2, W2, stem_out.grad.ptr, _st()), "maxpool_bwd")
                pooled.grad = None
            self.tape.append(pool_bwd)

        # ---- residual layers (resnet.py:99-120, :176-198)
        a = pooled
        low_level = None
        cat2 = low_slice = None
        for li, blocks in enumerate(self.layers):
            for (c1, c2, c3, ds) in blocks:
                if ds is None and c1.k == 1 and c1.stride == 1:
                    a.masked_ok = True            # consumers of this block input: conv1 and the identity add, nothing else
                if (ds is not None and train and self.dual_bn and self.debug_units is None and self.debug_taps is None
                        and c3.cout % 8 == 0):
                    dsc = self._conv_raw(ds, a)   # downsample convolution now; its BatchNorm rides on the block's closing one
                    # its backward is taped HERE, i.e. it runs after conv1's: conv1's data gradient then writes the block input's
                    # gradient fresh and the (strided, for stride 2) downsample gradient accumulates into a quarter of it - the other
                    # order needs a zero fill of the whole tensor and a full read-modify-write by conv1
                    ds_dy = []
                    self.tape.append(lambda ds=ds, a=a, dsc=dsc, ds_dy=ds_dy: ds_dy and self._conv_backward(ds, a, dsc[2], dsc[3], dsc[4], dsc[5], dsc[6], ds_dy.pop(), True))
                    dsc = dsc + (ds_dy,)
                    y = unit(c1, a)
                    y = unit(c2, y)
                    a = self._unit_train_dual(c3, y, ds, dsc)
                    continue
                idt = a if ds is None else unit(ds, a, relu=False)
                if ds is not None:
                    idt.masked_ok = True          # the downsample output feeds the block-closing add only
                y = unit(c1, a)
                y = unit(c2, y)
                a = unit(c3, y, relu=True, residual=idt)
            if li == 0:
                low_level = a
                # head, part 1 (_deeplab.py:56): the low-level projection only needs layer1's output; it is issued now,
                # on the side stream, and runs under layers 2-4 (its consumer is the decoder, ~40 launches later)
                h4, w4 = low_level.H, low_level.W
                cat2 = Act.new(B, h4, w4, 304, dev)
                low_slice = cat2.slice(0, 48)
                with self._fwd_fork():
                    unit(self.low_proj, low_level, out=low_slice)
        feat = a

        # ---- head (_deeplab.py:55-61): ASPP branches write straight into the concat buffer
        hf, wf = feat.H, feat.W
        cat1 = Act.new(B, hf, wf, 1280, dev)
        br_slices = [cat1.slice(256 * i, 256) for i in range(5)]
        with self._fwd_fork():                               # four tiny latency-bound launches under the big branch convs
            self._aspp_pool(feat, br_slices[4], train)
        fused_aspp_bwd = train and bool(self._aspp_cat_slot()) and self.debug_units is None   # the unit-replay recorder wants per-unit dx
        if fused_aspp_bwd:
            cb = self.aspp_branches[0].cout
            dycat = [None]

            def dy_slice(i):
                def get():
                    if dycat[0] is None:
                        dycat[0] = torch.empty((B, hf, wf, 4 * cb), dtype=torch.bfloat16, device=dev)
                    return dycat[0][..., i * cb:(i + 1) * cb]
                return get

            def aspp_dgrad():
                # runs after the four branch closures (reverse tape order): every slice of dycat is written
                first = feat.grad is None
                if first:
                    feat.new_grad()
                g = feat.grad
                rates = (C.c_int * 3)(*[b.dilation for b in self.aspp_branches[1:]])
                ev = self._prof_begin()
                check(L.iswm_aspp_bwd(dycat[0].data_ptr(), 4 * cb, self.aspp_wcat.data_ptr(), B, hf, wf, cb, feat.C, rates,
                                      g.ptr, g.ld, 0 if first else 1, _st()), "aspp_bwd")
                self._prof_end(ev, "conv_igemm", 2.0 * B * hf * wf * feat.C * cb * 28, "dgrad classifier.aspp.convs.0-3(fused)")
                dycat[0] = None
            self.tape.append(aspp_dgrad)
            for i, s in enumerate(self.aspp_branches):
                self._unit_train(s, feat, out=br_slices[i], need_dx=False, dy_into=dy_slice(i))
        else:
            for i, s in enumerate(self.aspp_branches):
                unit(s, feat, out=br_slices[i])
        self._fwd_join()
        if train:
            self._slice_grad_split(cat1, [(br_slices[i], 256 * i) for i in range(5)])
            aspp_out = self._unit_train(self.aspp_proj, cat1, drop_p=self.dropout_p)
        else:
            aspp_out = self._unit_eval(self.aspp_proj, cat1)
        up = cat2.slice(48, 256)
        check(L.iswm_bilinear_fwd(aspp_out.ptr, aspp_out.ld, B, hf, wf, 256, h4, w4, up.ptr, up.ld, _st()), "bilinear_fwd")
        if train:
            def up_bwd():
                g = up.grad
                aspp_out.new_grad()
                check(L.iswm_bilinear_bwd(g.ptr, g.ld, B, hf, wf, 256, h4, w4, aspp_out.grad.ptr, 256, _st()), "bilinear_bwd")
                up.grad = None
            self.tape.append(up_bwd)
            self._slice_grad_split(cat2, [(low_slice, 0), (up, 48)])
        y = unit(self.dec1, cat2)
        y = unit(self.dec2, y)

        # ---- classifier 1x1 (+bias) -> fp32 NHWC low-res logits -> bilinear to input size (utils.py:22)
        ncls = self.cls.cout
        self._pack(self.cls, train)
        bias = self.cls.conv.bias
        ones = self._ones(ncls)
        lo = torch.empty((B, h4, w4, ncls), dtype=torch.float32, device=dev)
        self._conv(self.cls, y, lo, ncls, h4, w4, ops.conv_taps(1, 1), B, _lib.EPI_AFFINE | _lib.EPI_OUT_F32, ones, bias.detach())
        if lowres:
            if train and not fused_tail:
                raise RuntimeError("low-resolution logits are an inference-only output (or the fused train tail's: fused_tail=True)")
            if train:
                self._saved = (y, B, h4, w4, H, W, ncls)
            return lo
        logits = torch.empty((B, ncls, H, W), dtype=torch.float32, device=dev)
        check(L.iswm_logits_up_fwd(lo.data_ptr(), B, h4, w4, ncls, H, W, logits.data_ptr(), _st()), "logits_up_fwd")
        if train:
            self._saved = (y, B, h4, w4, H, W, ncls)
        return logits

    def _ones(self, n):
        t = getattr(self, "_ones_t", None)
        if t is None or t.numel() < n or t.device != self.device:
            t = torch.ones(max(n, 64), dtype=torch.float32, device=self.device)
            self._ones_t = t
        return t

    def _stem_unit(self, colA: Act, B, H1, W1, train, row_taps=None, n_img=1) -> Act:
        """The stem conv: `row_taps` given = 7 row taps over the x-unrolled image rows (colA = [2B,H1,W1,24] phase-major);
        else a 1-tap GEMM over the im2col matrix. Output [B,H1,W1,64]."""
        L = _lib.lib()
        s = self.stem
        self._pack(s, False)
        M = B * H1 * W1
        dev = self.device
        out = Act.new(B, H1, W1, 64, dev)
        if row_taps is not None:
            taps, geo = row_taps, dict(Hi=H1, Wi=W1, B=B)
            Ho_, Wo_ = H1, W1
        else:
            taps, geo = [(0, 0, 0)], {}
            Ho_, Wo_ = 1, M
        if not train:
            self._fold(s)
            self._conv(s, colA, out.t, 64, Ho_, Wo_, taps, n_img, _lib.EPI_AFFINE | _lib.EPI_RELU, s.fold_scale, s.fold_shift, cin=colA.C, **geo)
            self._tap(s.name, out)
            return out
        raw = torch.empty((M, 64), dtype=torch.bfloat16, device=dev)
        rep = self._stats_rep(64)
        sync = self.bn_sync is not None
        stats = self._stats_slot(128 * rep + (1 if sync else 0))
        self._conv(s, colA, raw, 64, Ho_, Wo_, taps, n_img, _lib.EPI_STATS, stats=stats, cin=colA.C, **geo)
        if sync:
            stats, rep = self._bn_exchange([(stats, rep)], 128, M)[0], 1
        save = self._save_slot(128)
        bn = s.bn
        fused_tail = self.stem_pool and self.debug_units is None and self.debug_taps is None
        if fused_tail:
            H2, W2 = (H1 + 1) // 2, (W1 + 1) // 2
            pooled = Act.new(B, H2, W2, 64, dev)
            idx = torch.empty((B, H2, W2, 64), dtype=torch.uint8, device=dev)
            side = self._bn_side(bn, stats, save, 64, True, rep)
            ev = self._prof_begin()
            fwd = L.iswm_stem_pool_fwd_global if sync else L.iswm_stem_pool_fwd
            check(fwd(raw.data_ptr(), C.byref(side), B, H1, W1, 64, H2, W2, BN_EPS, BN_MOMENTUM, pooled.ptr, idx.data_ptr(), _st()), "stem_pool_fwd")
            self._prof_end(ev, "hbm:stem_pool_fwd", 2.0 * M * 64 + 3.0 * B * H2 * W2 * 64, "stem_pool_fwd")

            def backward_fused():
                g = pooled.grad
                assert g is not None and g.ld == 64
                sums = self._stats_slot(130)
                dy = torch.empty((M, 64), dtype=torch.bfloat16, device=dev)
                dact = torch.empty((M, 64), dtype=torch.bfloat16, device=dev)
                check(L.iswm_maxpool_bwd(g.ptr, idx.data_ptr(), B, H1, W1, 64, H2, W2, dact.data_ptr(), _st()), "maxpool_bwd")
                check(L.iswm_bn_bwd_reduce(dact.data_ptr(), 64, raw.data_ptr(), 64, None, 64, M, 64, save.data_ptr(), save[64:].data_ptr(),
                                           bn.weight.data_ptr(), bn.bias.data_ptr(), 1, 0.0, 0, None, sums.data_ptr(), _st()), "bn_bwd_reduce stem")
                self._stem_bwd_apply(bn, dact.data_ptr(), 64, raw, save, sums, dy, M)
                pooled.grad = None
                self._stem_wgrad(s, bn, colA, dy, B, H1, W1, M, taps, row_taps, n_img)

            self.tape.append(backward_fused)
            return (pooled,)
        apply_args = (bn.weight.data_ptr(), bn.bias.data_ptr(), BN_EPS, BN_MOMENTUM, bn.running_mean.data_ptr(), bn.running_var.data_ptr(),
                      bn.num_batches_tracked.data_ptr(), save.data_ptr(), save[64:].data_ptr(), None, 0, 1, 0.0, 0, None, out.ptr, 64, None, _st())
        if sync:
            check(L.iswm_bn_train_apply_global(raw.data_ptr(), 64, stats.data_ptr(), M, 64, *apply_args), "bn_train_apply_global stem")
        else:
            check(L.iswm_bn_train_apply(raw.data_ptr(), 64, stats.data_ptr(), rep, M, 64, *apply_args), "bn_train_apply stem")
        self._tap(s.name, out)

        def backward():
            dout = out.grad
            sums = self._stats_slot(130)
            dy = torch.empty((M, 64), dtype=torch.bfloat16, device=dev)
            check(L.iswm_bn_bwd_reduce(dout.ptr, dout.ld, raw.data_ptr(), 64, None, 64, M, 64, save.data_ptr(), save[64:].data_ptr(),
                                       bn.weight.data_ptr(), bn.bias.data_ptr(), 1, 0.0, 0, None, sums.data_ptr(), _st()), "bn_bwd_reduce stem")
            self._stem_bwd_apply(bn, dout.ptr, dout.ld, raw, save, sums, dy, M)
            out.grad = None
            gview = self.grad_views[id(s.conv.weight)]
            self._stem_wgrad(s, bn, colA, dy, B, H1, W1, M, taps, row_taps, n_img)
            if self.debug_units is not None:
                self.debug_units.append(dict(name=s.name, k=7, stride=2, dilation=1, relu=True, x=None, image=self._image, raw=raw.view(B, H1, W1, 64).clone(),
                                             out=out.t.clone(), dout=dout.t.clone(), mean=save[:64].clone(), invstd=save[64:128].clone(),
                                             gamma=bn.weight.detach().clone(), beta=bn.bias.detach().clone(), w=s.conv.weight.detach().clone(),
                                             residual=None, xgrad_before=None, resgrad_before=None, dy=dy.view(B, H1, W1, 64).clone(),
                                             dW=gview.clone(), dgamma=self.grad_views[id(bn.weight)].clone(), dbeta=self.grad_views[id(bn.bias)].clone(),
                                             xgrad_after=None, resgrad_after=None))

        self.tape.append(backward)
        return out

    def _stem_bwd_apply(self, bn, dout_ptr, dout_ld, raw, save, sums, dy, M):
        """The stem BatchNorm's backward pass 2 (after iswm_bn_bwd_reduce into `sums`), synchronised or not."""
        L = _lib.lib()
        head = (dout_ptr, dout_ld, raw.data_ptr(), 64, None, 64, M, 64, bn.weight.data_ptr(), bn.bias.data_ptr(), save.data_ptr(), save[64:].data_ptr())
        tail = (1, 0.0, 0, None, dy.data_ptr(), 64, None, 0, self.grad_views[id(bn.weight)].data_ptr(), self.grad_views[id(bn.bias)].data_ptr(), _st())
        if self.bn_sync is not None:
            gsums = self._bn_exchange([(sums, 1)], 128, M)[0]
            check(L.iswm_bn_bwd_apply_global(*head, gsums.data_ptr(), sums.data_ptr(), *tail), "bn_bwd_apply_global stem")
        else:
            check(L.iswm_bn_bwd_apply(*head, sums.data_ptr(), *tail), "bn_bwd_apply stem")

    def _stem_wgrad(self, s, bn, colA: Act, dy: torch.Tensor, B, H1, W1, M, taps, row_taps, n_img):
        """Weight gradient of the stem convolution from dy (gradient of its pre-BN output) on the weight-gradient stream."""
        L = _lib.lib()
        off, n = self.wacc_off[s.name]
        acc = self.wacc[off:off + n]
        if row_taps is not None:
            d = ops.make_conv_desc(B, H1, W1, colA.C, colA.ld, n_img, H1, W1, 64, 64, taps)
        else:
            d = ops.make_conv_desc(1, 1, M, colA.C, colA.ld, 1, 1, M, 64, 64, taps)
        gview = self.grad_views[id(s.conv.weight)]
        with self._wgrad_ctx(dy, colA.t):
            ev = self._prof_begin()
            check(L.iswm_conv_wgrad(C.byref(d), colA.ptr, dy.data_ptr(), acc.data_ptr(), _st()), "conv_wgrad stem")
            self._prof_end(ev, "conv_wgrad", 2.0 * M * 64 * 147, "wgrad " + s.name)
            if row_taps is not None:
                check(L.iswm_unpack_wgrad_stem(acc.data_ptr(), 64, s.cin, 7, colA.C, 1.0, gview.data_ptr(), _st()), "unpack_wgrad_stem")
            else:
                check(L.iswm_unpack_wgrad(acc.data_ptr(), 64, s.cin, 49, s.cin, colA.C, 1.0, gview.data_ptr(), _st()), "unpack_wgrad stem")
            self._notify(s.conv.weight)
            self._notify(bn.weight)
            self._notify(bn.bias)

    def _aspp_pool(self, feat: Act, dst: Act, train: bool):
        """ASPPPooling (_deeplab.py:130-141): GAP -> 1x1 -> BN -> ReLU -> broadcast (bilinear from 1x1)."""
        L = _lib.lib()
        B, HW, dev = feat.B, feat.H * feat.W, self.device
        pooled = Act.new(B, 1, 1, feat.C, dev)
        check(L.iswm_gap_fwd(feat.ptr, feat.ld, B, HW, feat.C, pooled.ptr, _st()), "gap_fwd")
        if train:
            def gap_bwd():
                g = pooled.grad
                assert g.ld == feat.C
                if feat.grad is None:
                    feat.new_grad()
                    feat.grad.t.zero_()
                check(L.iswm_gap_bwd_add(g.ptr, B, HW, feat.C, feat.grad.ptr, feat.grad.ld, _st()), "gap_bwd_add")
                pooled.grad = None
            self.tape.append(gap_bwd)
            v = self._unit_train(self.aspp_pool, pooled)
        else:
            v = self._unit_eval(self.aspp_pool, pooled)
        check(L.iswm_broadcast_hw(v.ptr, B, HW, 256, dst.ptr, dst.ld, _st()), "broadcast_hw")
        self._fwd_keep.extend((pooled.t, v.t))               # may be running on the side stream: alive until the join
        if train:
            def bc_bwd():
                g = dst.grad
                v.new_grad()
                check(L.iswm_sum_hw(g.ptr, g.ld, B, HW, 256, v.grad.ptr, _st()), "sum_hw")
                dst.grad = None
            self.tape.append(bc_bwd)

    def _slice_grad_split(self, cat: Act, parts):
        """After the consumer of a concat buffer produced cat.grad, hand each producer its channel slice
        (a strided view of cat.grad: no copy)."""
        def split():
            g = cat.grad
            for act, off in parts:
                act.grad = g.slice(off, act.C)
            cat.grad = None
        self.tape.append(split)

    # ------------------------------------------------------------------ backward
    def backward(self, dlogits: torch.Tensor):
        """dlogits: fp32 NCHW gradient of the loss w.r.t. the logits returned by forward(train=True)."""
        with _StreamScope():
            self._backward(dlogits)

    def backward_tail(self, fill_dlo):
        """Backward of a forward(train=True, lowres=True, fused_tail=True): `fill_dlo(dlo bf16 [B,h,w,ldp], bias_grad fp32 [ncls])`
        writes the gradient w.r.t. the classifier's output (all ldp channels) and ADDS the classifier bias gradient - the fused
        tail's iswm_tail_bwd - in place of the adjoint of the full-resolution upsample."""
        with _StreamScope():
            self._backward(None, fill_dlo)

    def _backward(self, dlogits, fill_dlo=None):
        L = _lib.lib()
        y, B, h4, w4, H, W, ncls = self._saved
        dev = self.device
        if fill_dlo is None:
            dlogits = dlogits.contiguous().float()
        params = self._param_list()
        fresh = all(p.grad is None for p in params)
        if fresh:
            self.flat_g.zero_()
            for p in params:
                p.grad = self.grad_views[id(p)]
        else:
            for p in params:
                if p.grad is None:
                    self.grad_views[id(p)].zero_()
                    p.grad = self.grad_views[id(p)]
                elif p.grad.data_ptr() != self.grad_views[id(p)].data_ptr():
                    raise RuntimeError("parameter .grad was replaced by a foreign tensor; call optimizer.zero_grad(set_to_none=True)")
        self.wacc.zero_()
        self._wq, self._wq_layer = [], None
        # classifier: bias grad, low-res logits gradient, weight grad, data grad
        cls = self.cls
        ldp = 8 * ((ncls + 7) // 8)
        dlo = torch.empty((B, h4, w4, ldp), dtype=torch.bfloat16, device=dev)
        if fill_dlo is not None:
            fill_dlo(dlo, self.grad_views[id(cls.conv.bias)])
        else:
            # adjoint of the final upsample; the classifier bias gradient (sum of dlogits per class) rides on the same sweep
            check(L.iswm_logits_up_bwd(dlogits.data_ptr(), B, h4, w4, ncls, H, W, dlo.data_ptr(), ldp,
                                       self.grad_views[id(cls.conv.bias)].data_ptr(), _st()), "logits_up_bwd")
        d = ops.make_conv_desc(B, h4, w4, y.C, y.ld, B, h4, w4, ncls, ldp, [(0, 0, 0)])
        with self._wgrad_ctx(dlo, y.t):
            check(L.iswm_conv_wgrad(C.byref(d), y.ptr, dlo.data_ptr(), self.grad_views[id(cls.conv.weight)].data_ptr(), _st()), "conv_wgrad cls")
            self._notify(cls.conv.bias)
            self._notify(cls.conv.weight)
        self._dgrad_into(cls, y, dlo, ldp, h4, w4, [(0, 0, 0)], h4, w4)
        if self.debug_units is not None:
            self.debug_units.append(dict(name=cls.name, kind="cls", x=y.t.clone(), dlogits=None if dlogits is None else dlogits.clone(), dlo=dlo.clone(),
                                         w=cls.conv.weight.detach().clone(), dW=self.grad_views[id(cls.conv.weight)].clone(),
                                         dbias=self.grad_views[id(cls.conv.bias)].clone(), xgrad_after=y.grad.t.clone()))
        # reverse sweep
        for fn in reversed(self.tape):
            fn()
        if self._wq:
            self._flush_wgrad_group()
        if self._batched_unpack():
            with self._wgrad_ctx():              # after every weight-gradient kernel of the sweep, on their stream
                self._unpack_all()
        self._wgrad_join()                       # the optimiser / all-reduce tail sees every weight gradient
        self.tape = []
        self._saved = None
