"""A whole train step as ONE CUDA graph launch.

The eager step (`logits = model(x); loss = criterion(logits, y); optimizer.zero_grad(); loss.backward();
optimizer.step()`, train.py:1039-1049) enqueues ~430 kernels through Python/ctypes: about 10.5 ms of host work per step
at cfg2 against 14.8 ms of GPU work - the host keeps up, but only just, and it has no time left for the data loader.
`GraphedTrainStep` captures that exact sequence once (both streams: the weight-gradient side stream forks and joins
inside the capture) and replays it with one `cudaGraphLaunch` per step: 11 us of host time, and the GPU runs the
kernels back to back without enqueue jitter (cfg2 on B200: 15.04 -> 14.80 ms/step).

What makes the replay a TRAINING step rather than a recording of one:
  * inputs are copied into static device buffers (`.images`, `.labels`) - or written there directly by the loader;
  * the Dropout mask depends on a step counter in device memory that the captured forward increments (engine.py),
    BatchNorm's num_batches_tracked is incremented by the kernel itself;
  * the learning rate (and Adam's step count) are read by the optimiser kernel from device memory
    (`optimizer.enable_device_state()`), refreshed from `param_groups[0]['lr']` before each replay, so
    `CosineAnnealingLR.step()` (train.py:1103) keeps working;
  * the packed bf16 weights are refreshed at the START of the captured step (weights changed at the end of the
    previous one); after a replay the engine is told so, and an eager eval forward repacks.
The returned loss is a static 0-dim device tensor, overwritten by the next call (copy it, or use DeferredLoss).
Data parallel: `GraphedTrainStep(model, criterion, optimizer, dp=DataParallel(...))` captures the multi-GPU step too - on
the peer-memory transport every exchange (class histogram, gradient buckets, loss) is a plain kernel over NVLink peer memory
on an event-ordered communication stream (iswm_b200.peer), so there is nothing un-capturable in it. (Capturing the
torch.distributed / NCCL all-reduces issued with async_op from the backward hooks hung at the first replay on 2 B200s in
round 1; that transport stays eager and is refused here.)
"""
from __future__ import annotations

import torch


def _fused_tail_default() -> bool:
    import os
    return os.environ.get("ISWM_FUSED_TAIL", "1") != "0"


class GraphedTrainStep:
    def __init__(self, model, criterion, optimizer, warmup_steps: int = 2, dp=None, fused_tail=None):
        """`dp`: an iswm_b200.parallel.DataParallel on the peer-memory transport - its step (histogram / gradient-bucket /
        loss exchanges are plain kernels on event-ordered streams) is captured like the single-GPU one; the returned loss is
        then the GLOBAL loss. Every rank must construct and call the stepper in lockstep."""
        self.model = getattr(model, "module", model)
        self.criterion, self.optimizer = criterion, optimizer
        self.engine = self.model.engine()
        self.warmup_steps = max(1, warmup_steps)
        self.graph = None
        self._fused_pack = False
        self.images = self.labels = self.loss = None
        self.dp = dp
        # fused train tail (model.forward_loss: upsample + criterion + their backward without full-resolution tensors);
        # None = the ISWM_FUSED_TAIL environment switch
        self.fused_tail = _fused_tail_default() if fused_tail is None else bool(fused_tail)
        if dp is not None:
            dp.fused_tail = self.fused_tail
        if dp is not None and getattr(dp, "comm_mode", "nccl") != "peer":
            raise RuntimeError("GraphedTrainStep(dp=...) needs the peer-memory transport (torch.distributed collectives issued from "
                               "Python hooks are not captured); construct DataParallel(..., comm='peer')")
        if dp is None and self.engine.grad_ready_hook is not None:
            raise RuntimeError("this model is wrapped by iswm_b200.parallel.DataParallel: pass it as GraphedTrainStep(..., dp=dp)")

    def _eager(self, x, y):
        if self.dp is not None:
            return self.dp.train_step(x, y, self.optimizer).detach()
        if self.fused_tail:
            loss = self.model.forward_loss(x, y, self.criterion)
        else:
            logits = self.model(x)
            loss = self.criterion(logits, y)
        self.optimizer.zero_grad()
        loss.backward()
        self.optimizer.step()
        return loss.detach()

    def _capture(self, x, y):
        if not self.model.training:
            raise RuntimeError("GraphedTrainStep captures a TRAINING step: call model.train() first")
        self.optimizer.enable_device_state()
        self.optimizer.sync_device_state()
        self.images = torch.empty_like(x)
        self.labels = torch.empty_like(y)
        self.images.copy_(x)
        self.labels.copy_(y)
        # allocations, weight flattening, lazy buffers happen in eager warm-up steps outside the capture, on a side
        # stream (torch's capture recipe); the training state they advance is put back afterwards, so the first call
        # of this object is ONE step like every other
        snap = self._snapshot()
        s = torch.cuda.Stream(x.device)
        s.wait_stream(torch.cuda.current_stream(x.device))
        with torch.cuda.stream(s):
            for _ in range(self.warmup_steps):
                self._eager(self.images, self.labels)
        torch.cuda.current_stream(x.device).wait_stream(s)
        from . import _lib
        n0 = _lib.launch_count()
        self.graph = torch.cuda.CUDAGraph()
        # Stream priorities were measured and do NOT help (cfg2, same box): capturing on a high-priority stream (weight-gradient
        # stream lowest) 12.60 -> 13.09 ms/step, the reverse 12.61 -> 12.77; long weight gradients cut into batch slices on top
        # of either: no better. Both streams keep the default priority.
        with torch.cuda.graph(self.graph):
            self.loss = self._eager(self.images, self.labels)
        self.launches_per_replay = _lib.launch_count() - n0      # library kernels recorded in the graph
        # did the captured optimiser step repack the operands itself (FusedSGD with iswm_sgd_pack_batched)? then the graph holds no
        # pack launch at its start and __call__ keeps the bookkeeping
        self._fused_pack = self.engine.packed_is_fresh()
        self._restore(snap)
        self.engine.invalidate_packed()

    def _snapshot(self):
        eng, opt = self.engine, self.optimizer
        flat_w = eng.flatten_parameters()
        return {"w": flat_w.clone(), "buffers": [b.detach().clone() for b in self.model.buffers()], "step": eng.step,
                "opt_steps": opt._steps, "opt_state": {k: (None if getattr(opt, k, None) is None else getattr(opt, k).clone())
                                                       for k in ("_mom", "_m", "_v") if hasattr(opt, k)}}

    def _restore(self, snap):
        eng, opt = self.engine, self.optimizer
        with torch.no_grad():
            eng.flat_w.copy_(snap["w"])
            for b, v in zip(self.model.buffers(), snap["buffers"]):
                b.copy_(v)
            for k, v in snap["opt_state"].items():
                cur = getattr(opt, k)
                if cur is not None:
                    cur.zero_() if v is None else cur.copy_(v)
        eng.step = snap["step"]
        if getattr(eng, "_step_dev", None) is not None:
            eng._step_dev.fill_(snap["step"])
        opt._steps = snap["opt_steps"]
        if opt.step_dev is not None:
            opt.step_dev.fill_(snap["opt_steps"])

    def __call__(self, images: torch.Tensor, labels: torch.Tensor) -> torch.Tensor:
        if self.graph is None:
            self._capture(images, labels)                # the capture itself does not execute: fall through and replay
        elif images.shape != self.images.shape or labels.shape != self.labels.shape:
            raise ValueError("GraphedTrainStep was captured for a fixed batch geometry; build another one for this shape")
        elif labels.dtype != self.labels.dtype and (labels.is_floating_point() or labels.dtype == torch.bool):
            raise ValueError(f"labels of dtype {labels.dtype}: integer class indices expected")
        # integer labels of another width (the reference's loader yields uint8, train.py:1040 widens them with .to(device, dtype=torch.long))
        # are widened / narrowed by the copy into the captured step's label buffer
        if images.data_ptr() != self.images.data_ptr():
            self.images.copy_(images, non_blocking=True)
        if labels.data_ptr() != self.labels.data_ptr():
            self.labels.copy_(labels, non_blocking=True)
        self.optimizer.sync_device_state()
        if self._fused_pack and not self.engine.packed_is_fresh():
            # the captured step does not repack at its start (its optimiser kernel leaves the operands fresh): weights changed from
            # outside since the last replay (snapshot restore after the capture, load_state_dict, manual edits) are packed here
            self.engine.pack_all(True)
        self.graph.replay()
        if self._fused_pack:
            self.engine.mark_packed_fresh()              # weights AND packed operands moved together inside the replay
        else:
            self.engine.invalidate_packed()              # the replay changed the weights behind Python's back
        self.optimizer._steps += 1
        self.engine.step += 1
        return self.loss
