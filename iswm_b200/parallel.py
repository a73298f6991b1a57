"""Data parallelism for the hot path: one process per GPU, NCCL over NVLink 5 / NVSwitch.

The reference is single-process nn.DataParallel (train.py:970): parameters replicated, the batch
scattered along dim 0, PER-REPLICA BatchNorm statistics (the default here too; `sync_bn=True` for statistics over the global
batch, below), logits gathered to GPU 0 where the criterion
normalises over the WHOLE batch (train.py:1045-1046), gradients reduce-added to GPU 0. The same
semantics here, without the GPU-0 bottleneck:
  * each rank runs forward/backward on its shard with its own BN statistics;
  * the per-class pixel histogram is all-reduced (SUM, C int64) before the fused CE kernel, so every
    rank divides by the GLOBAL denominator sum_c w_c n_c; gradients are then all-reduced with SUM
    (a DDP-style mean of per-rank means would differ whenever class mixes differ across ranks);
  * gradient all-reduce is bucketed over the engine's flat fp32 gradient buffer and launched from the
    backward sweep as soon as the last tensor of a bucket has been produced (reverse registration
    order: head first, stem last), overlapping the exchange with the remaining backward kernels.

Two transports. "peer" (the default on GPUs): the flat gradient buffer lives in symmetric memory and every exchange of the
step - histogram, gradient buckets, loss - is a plain kernel over NVLink peer memory (iswm_b200.peer / csrc/peer_allreduce.cu)
on a communication stream ordered by events, with sums that are bit-identical on every rank. No host synchronisation and no
library call, so the data-parallel step is captured in ONE CUDA graph (GraphedTrainStep(dp=...)). "nccl": torch.distributed
collectives (async_op on the bucket all-reduces); also what the gloo CPU tests drive.

Synchronised BatchNorm (`sync_bn=True`, torch.nn.SyncBatchNorm semantics; convert_sync_batchnorm does not apply to this model,
whose BatchNorms are parameter holders the engine runs itself): every train-mode BatchNorm normalises with the mean and biased
variance over ALL ranks' rows, the running variance uses the unbiased factor of the global row count, and the input gradient
uses the globally reduced sum(dz), sum(dz.xhat) and count. The gamma / beta gradients each rank writes are its OWN
contributions, which the gradient all-reduce (SUM) completes. Each BatchNorm's per-channel fp64 sums (convolution epilogue
forward, iswm_bn_bwd_reduce backward) and its row count are exchanged between producer and consumer (Engine.bn_sync):
  * peer: the engine's fp64 scratch arena is a symmetric allocation carved at the same offsets on every rank, and one
    iswm_syncbn_exchange launch per exchange reads the peers' slots in place after a barrier, summing in rank order (same bits
    on every rank); capturable, so GraphedTrainStep(dp=...) still replays ONE graph per step;
  * nccl: the same kernel folds this rank's copies and count into a slot that dist.all_reduce (SUM) completes, eagerly.
Counts are exchanged, not assumed: shards of different sizes are normalised over the true global batch.
"""
from __future__ import annotations

import os
from typing import List, Optional

import torch
import torch.distributed as dist


class GradBucketer:
    """Splits a flat gradient buffer into ~bucket_bytes contiguous buckets aligned to tensor
    boundaries and all-reduces each one when all of its tensors have been marked ready.
    Pure torch.distributed logic (works with gloo on CPU for tests, NCCL on GPUs)."""

    def __init__(self, flat: torch.Tensor, sizes: List[int], bucket_bytes: int = 25 << 20, group=None, align: int = 1,
                 launch=None, finish=None):
        """`align`: bucket boundaries fall on multiples of `align` elements (the peer-memory kernel moves float4);
        `launch(start, end)` / `finish()` replace the torch.distributed transport."""
        self.flat, self.group = flat, group
        self._launch_fn, self._finish_fn = launch, finish
        self.bounds = []                 # (start, end) element ranges, in registration order
        self.tensor_bucket = []
        elems = max(1, bucket_bytes // flat.element_size())
        # build from the END (backward produces the last-registered parameters first)
        cuts, acc, off = [], 0, sum(sizes)
        ends = []
        o = 0
        for n in sizes:
            o += n
            ends.append(o)
        start_of = [e - n for e, n in zip(ends, sizes)]
        bucket_end = off
        for i in range(len(sizes) - 1, -1, -1):
            acc += sizes[i]
            if (acc >= elems and start_of[i] % align == 0) or i == 0:
                cuts.append((start_of[i], bucket_end))
                bucket_end = start_of[i]
                acc = 0
        self.bounds = cuts               # cuts[0] is the LAST range of the buffer (first to be ready)
        self.tensor_bucket = [0] * len(sizes)
        for b, (s, e) in enumerate(self.bounds):
            for i in range(len(sizes)):
                if start_of[i] >= s and ends[i] <= e:
                    self.tensor_bucket[i] = b
        self.need = [0] * len(self.bounds)
        for b in self.tensor_bucket:
            self.need[b] += 1
        self.reset()

    def reset(self):
        self.pending = list(self.need)
        self.works = []
        self.launched = [False] * len(self.bounds)

    def mark_ready(self, tensor_index: int):
        b = self.tensor_bucket[tensor_index]
        self.pending[b] -= 1
        if self.pending[b] == 0 and not self.launched[b]:
            self._launch(b)

    def _launch(self, b: int):
        s, e = self.bounds[b]
        self.launched[b] = True
        if self._launch_fn is not None:
            self._launch_fn(s, e)
        else:
            self.works.append(dist.all_reduce(self.flat[s:e], op=dist.ReduceOp.SUM, group=self.group, async_op=True))

    def finish(self):
        for b in range(len(self.bounds)):
            if not self.launched[b]:
                self._launch(b)
        for w in self.works:
            w.wait()
        if self._finish_fn is not None:
            self._finish_fn()
        self.reset()


class DataParallel:
    """Wraps an iswm_b200 DeepLabV3 model + criterion for multi-rank training (see module docstring)."""

    def __init__(self, model, criterion, bucket_bytes: int = 25 << 20, group=None, metrics=None, comm: str = "auto",
                 sync_bn: bool = False):
        if not dist.is_initialized():
            raise RuntimeError("torch.distributed must be initialised (backend 'nccl', one process per GPU)")
        self.model, self.criterion, self.group = model, criterion, group
        self.engine = model.engine()
        self.world = dist.get_world_size(group)
        self.bucket_bytes = int(os.environ.get("ISWM_DP_BUCKET_MB", "0")) << 20 or bucket_bytes   # experiment knob
        self.bucketer: Optional[GradBucketer] = None
        self.comm_mode, self.peer = "nccl", None
        p0 = next(iter(model.parameters()))
        want = os.environ.get("ISWM_DP_COMM", comm)
        if want not in ("auto", "peer", "nccl"):
            raise ValueError("comm must be 'auto', 'peer' or 'nccl'")
        if want != "nccl" and p0.is_cuda and self.world <= 8:
            try:
                self._setup_peer(p0.device)
            except Exception as e:                         # no symmetric memory on this system: torch.distributed transport
                if want == "peer":
                    raise
                import warnings
                warnings.warn(f"iswm_b200.parallel: peer-memory transport unavailable ({e!r}); using torch.distributed collectives")
                self.comm_mode, self.peer = "nccl", None
        # every rank must have taken the same decision
        flag = torch.tensor([1 if self.comm_mode == "peer" else 0], device=p0.device)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
        if int(flag) == 0 and self.comm_mode == "peer":
            self.comm_mode, self.peer = "nccl", None
            self.engine.ext_flat_g = None
        # identical replicas: rank 0's parameters AND buffers are canonical (DataParallel's replica 0)
        with torch.no_grad():
            for t in list(model.parameters()) + list(model.buffers()):
                dist.broadcast(t.data, 0, group=group)
        self.sync_bn = bool(sync_bn)
        if self.sync_bn:
            self._setup_sync_bn(p0.device)
        criterion.hist_hook = self._allreduce_hist_peer if self.comm_mode == "peer" else self._allreduce_hist
        self.engine.grad_ready_hook = self._grad_ready
        self._index = {id(p): i for i, p in enumerate(model.parameters())}
        if metrics is not None:
            self.attach_metrics(metrics)

    def attach_metrics(self, metrics):
        """Validation under data parallelism (SURVEY 8e "Metric"): every rank accumulates the confusion counts of ITS shard on
        the device; `metrics.get_results()` / `.confusion_matrix` then all-reduce (SUM) the n*n int64 counters once, so every
        rank reports the whole validation set's numbers - bit-exact by construction (metrics/stream_metrics.py:122)."""
        metrics.process_group = self.group if self.group is not None else dist.group.WORLD
        return metrics

    # ---- peer-memory transport ---------------------------------------------------------------------------------
    def _setup_peer(self, device):
        from .peer import PeerComm
        self.peer = PeerComm(device, self.group)
        total = sum(p.numel() for p in self.model.parameters())
        padded = (total + 3) // 4 * 4
        flat, ptrs = self.peer.alloc(padded, torch.float32)
        flat.zero_()
        self._flat_ptrs = self.peer._ptr_array(ptrs)
        self._flat_padded = padded
        self.engine.ext_flat_g = flat                      # the engine's flat gradient buffer IS the symmetric allocation
        self.comm_stream = torch.cuda.Stream(device)
        # a bucket's kernel only runs in the gaps the (register-file-filling) convolution CTAs leave: a modest grid is enough
        self._ar_blocks = int(os.environ.get("ISWM_DP_AR_BLOCKS", "64"))
        self.comm_mode = "peer"

    # ---- synchronised BatchNorm ------------------------------------------------------------------------------------
    def _setup_sync_bn(self, device):
        eng = self.engine
        if self.comm_mode == "peer":
            # size depends on the model's channel counts only: every rank allocates (collectively) the same arena, and the
            # engine carves it in the same order, so a BatchNorm's slot sits at the same offset on every rank
            arena, ptrs = self.peer.alloc(eng.scratch_need(True), torch.float64)
            arena.zero_()
            self._arena = arena
            self._arena_ptrs = self.peer._ptr_array(ptrs)
            eng.ext_scratch64 = arena
            eng.bn_sync = self._bn_exchange_peer
        else:
            eng.bn_sync = self._bn_exchange_nccl

    def _bn_jobs(self, srcs, dsts, n: int, base: int, size: int):
        from . import _lib
        jobs = (_lib.SyncBnJob * len(srcs))()
        for j, ((src, rep), dst) in enumerate(zip(srcs, dsts)):
            off = src.data_ptr() - base
            if off < 0 or off + 8 * (n * rep + 1) > 8 * size:
                raise RuntimeError("synchronised BatchNorm: a statistics slot lies outside the engine's arena")
            jobs[j].src_off, jobs[j].dst, jobs[j].n, jobs[j].replicas = off // 8, dst.data_ptr(), n, rep
        return jobs

    def _bn_exchange_peer(self, srcs, dsts, n: int, rows: int, stream: int):
        # Barrier ordering: exchanges on the main stream share channel 0 with the histogram and loss reductions (all issued in
        # program order on one stream, the same on every rank). The low-level projection and the pooled ASPP branch run on the
        # engine's side stream during the forward (Engine._fwd_fork), where they interleave with the main stream's exchanges in
        # an order that differs from rank to rank: they use their own channel 2, whose barriers are in program order on that stream.
        # Arena reuse: a peer reads this rank's step-i slots only inside step i's exchanges. This rank zeroes its arena for step
        # i+1 (Engine._begin_scratch) after the loss reduction of step i (train_step: channel-0 barrier after the backward),
        # which no peer passes before its stream has finished every exchange of step i - the backward's last (the stem's) on
        # the main stream, the side-stream ones before the forward's join - so no peer can still be reading.
        ws = self.engine._wstream
        channel = 2 if (ws is not None and stream == ws.cuda_stream) else 0
        jobs = self._bn_jobs(srcs, dsts, n, self._arena.data_ptr(), self._arena.numel())
        self.peer.bn_exchange(self._arena_ptrs, jobs, len(srcs), rows, channel, stream)

    def _bn_exchange_nccl(self, srcs, dsts, n: int, rows: int, stream: int):
        from . import _lib
        from ._lib import check
        import ctypes as C
        arena = self.engine._scratch64
        jobs = self._bn_jobs(srcs, dsts, n, arena.data_ptr(), arena.numel())
        local = (C.c_void_p * 1)(arena.data_ptr())
        check(_lib.lib().iswm_syncbn_exchange(jobs, len(srcs), local, None, 0, 1, float(rows), None, stream), "syncbn_exchange (fold)")
        cur = torch.cuda.current_stream()
        ctx = torch.cuda.stream(torch.cuda.ExternalStream(stream)) if cur.cuda_stream != stream else None
        if ctx is not None:
            ctx.__enter__()
        try:
            for d in dsts:
                dist.all_reduce(d, op=dist.ReduceOp.SUM, group=self.group)
        finally:
            if ctx is not None:
                ctx.__exit__(None, None, None)

    def _launch_peer(self, s: int, e: int):
        cur = torch.cuda.current_stream()                  # the stream that produced the bucket (weight-gradient stream)
        self.comm_stream.wait_event(cur.record_event())
        e4 = min(self._flat_padded, (e + 3) // 4 * 4)      # only the LAST bucket ends off a multiple of 4: the zero padding rides along
        self.peer.allreduce_f32(self._flat_ptrs, s, e4 - s, self.comm_stream.cuda_stream, self._ar_blocks)

    def _finish_peer(self):
        torch.cuda.current_stream().wait_stream(self.comm_stream)

    def _allreduce_hist_peer(self, hist: torch.Tensor):
        self.peer.small_allreduce_(hist, 0, torch.cuda.current_stream().cuda_stream)

    def _allreduce_hist(self, hist: torch.Tensor):
        dist.all_reduce(hist, op=dist.ReduceOp.SUM, group=self.group)

    def _grad_ready(self, p):
        if self.bucketer is None:
            sizes = [q.numel() for q in self.model.parameters()]
            if self.comm_mode == "peer":
                self.bucketer = GradBucketer(self.engine.flat_g, sizes, self.bucket_bytes, self.group, align=4,
                                             launch=self._launch_peer, finish=self._finish_peer)
            else:
                self.bucketer = GradBucketer(self.engine.flat_g, sizes, self.bucket_bytes, self.group)
        self.bucketer.mark_ready(self._index[id(p)])

    def train_step(self, images, labels, optimizer=None):
        """forward -> global-batch weighted CE -> backward with overlapped bucketed all-reduce -> step.
        Returns the GLOBAL loss (sum over ranks of local numerators / global denominator)."""
        if getattr(self, "fused_tail", False):
            loss = getattr(self.model, "module", self.model).forward_loss(images, labels, self.criterion)
        else:
            logits = self.model(images)
            loss = self.criterion(logits, labels)
        if optimizer is not None:
            optimizer.zero_grad()
        loss.backward()
        if self.bucketer is not None:
            self.bucketer.finish()
        if self.comm_mode == "peer":
            # loss_r = numerator_r / D with the GLOBAL denominator: the global loss is their sum (fp64 slots, fixed order)
            if getattr(self, "_gl64", None) is None:
                self._gl64 = torch.zeros(1, dtype=torch.float64, device=loss.device)
                self._gl32 = torch.zeros((), dtype=torch.float32, device=loss.device)
            self._gl64.copy_(loss.detach().reshape(1))
            self.peer.small_allreduce_(self._gl64, 1, torch.cuda.current_stream().cuda_stream)
            self._gl32.copy_(self._gl64[0])
            gl = self._gl32
        else:
            gl = loss.detach().clone()
            dist.all_reduce(gl, op=dist.ReduceOp.SUM, group=self.group)
        if optimizer is not None:
            optimizer.step()
        return gl
