"""Fused optimiser step for the hot path's tail (reference: train.py:421-444 builds
torch.optim.SGD(momentum=0.9, nesterov=True, weight_decay), Adam or AdamW at torch's default lr 1e-3 — `--lr`
never reaches them — and train.py:1049 steps it every iteration).

`FusedSGD` / `FusedAdam` / `FusedAdamW` have the torch.optim update rules but run as ONE kernel over the engine's
flat fp32 master-weight / gradient / state buffers instead of a multi-tensor foreach sweep."""
from __future__ import annotations

import torch

from . import _lib


class FusedSGD:
    def __init__(self, model, lr: float = 1e-3, momentum: float = 0.9, weight_decay: float = 0.0, nesterov: bool = True):
        if nesterov and momentum <= 0:
            raise ValueError("Nesterov momentum requires a momentum and zero dampening")
        self.model = getattr(model, "module", model)
        self.engine = self.model.engine()
        self.lr, self.momentum, self.weight_decay, self.nesterov = lr, momentum, weight_decay, nesterov
        self.param_groups = [{"lr": lr, "momentum": momentum, "weight_decay": weight_decay, "nesterov": nesterov}]
        self._mom = None
        self._steps = 0
        # the step also rewrites the packed bf16 convolution operands (one pass over the weights instead of two; False:
        # iswm_sgd_step, and the next forward repacks)
        self.fuse_pack = True
        self.lr_dev = None                 # device copy of the learning rate (enable_device_state: CUDA-graph replays)
        self.step_dev = None

    def enable_device_state(self):
        """Keep the schedule state the kernels read (learning rate, step count) in DEVICE memory, so that an optimiser
        step captured in a CUDA graph (iswm_b200.graphs.GraphedTrainStep) follows `param_groups[0]['lr']` and counts
        its own replays. `sync_device_state()` pushes the current host-side learning rate (one 4-byte async copy)."""
        dev = next(iter(self.engine._param_list())).device
        if self.lr_dev is None or self.lr_dev.device != dev:
            self.lr_dev = torch.tensor([self.param_groups[0]["lr"]], dtype=torch.float32, device=dev)
            self.step_dev = torch.tensor([self._steps], dtype=torch.int64, device=dev)
            self._lr_host = torch.empty(1, dtype=torch.float32).pin_memory()
            self._lr_pushed = None

    def sync_device_state(self):
        lr = float(self.param_groups[0]["lr"])
        if self.lr_dev is not None and lr != self._lr_pushed:
            self._lr_host[0] = lr
            self.lr_dev.copy_(self._lr_host, non_blocking=True)
            self._lr_pushed = lr

    def zero_grad(self, set_to_none: bool = True):
        for p in self.engine._param_list():
            if set_to_none:
                p.grad = None
            elif p.grad is not None:
                p.grad.zero_()

    def step(self):
        eng = self.engine
        flat_w = eng.flatten_parameters()
        flat_g = eng.flat_g
        if flat_g is None:
            raise RuntimeError("FusedSGD.step() before any backward pass")
        if self._mom is None or self._mom.numel() != flat_w.numel() or self._mom.device != flat_w.device:
            self._mom = torch.zeros_like(flat_w)
            self._steps = 0
        lr = self.param_groups[0]["lr"]
        jobs = eng.sgd_pack_jobs(flat_w, flat_g, self._mom) if self.fuse_pack else None
        if jobs is not None:
            # update + both bf16 operand packings of every convolution in ONE pass over the weights (csrc/sgd_pack.cu); the next
            # forward finds its operands fresh
            dev_jobs, n_jobs, n_blocks = jobs
            _lib.check(_lib.lib().iswm_sgd_pack_batched(dev_jobs.data_ptr(), n_jobs, n_blocks, lr, self.momentum, self.weight_decay,
                                                        1 if self.nesterov else 0, 1 if self._steps == 0 else 0,
                                                        None if self.lr_dev is None else self.lr_dev.data_ptr(),
                                                        torch.cuda.current_stream().cuda_stream), "sgd_pack_batched")
            self._steps += 1
            eng.mark_packed_fresh()
            return
        _lib.check(_lib.lib().iswm_sgd_step(flat_w.data_ptr(), flat_g.data_ptr(), self._mom.data_ptr(), flat_w.numel(),
                                            lr, self.momentum, self.weight_decay, 1 if self.nesterov else 0,
                                            1 if self._steps == 0 else 0, None if self.lr_dev is None else self.lr_dev.data_ptr(),
                                            torch.cuda.current_stream().cuda_stream), "sgd_step")
        self._steps += 1
        eng.invalidate_packed()

    def state_dict(self):
        """Flat layout (ONE momentum buffer over the engine's flat parameter buffer). A checkpoint's `optimizer_state`
        written by the reference's torch.optim objects (per-parameter `state` dict, train.py:569) is NOT loadable here
        and vice versa; model / scheduler states are interchangeable."""
        return {"momentum_buffer": self._mom, "steps": self._steps, "param_groups": self.param_groups}

    def _adopt(self, name: str, t):
        """validate a loaded flat state buffer against the engine's flat parameter buffer"""
        if t is None:
            return None
        flat_w = self.engine.flatten_parameters()
        if not isinstance(t, torch.Tensor) or t.numel() != flat_w.numel():
            raise ValueError(f"{type(self).__name__}.load_state_dict: '{name}' does not match the model's {flat_w.numel()} "
                             "parameters (a reference torch.optim state_dict is not loadable, see state_dict())")
        return t.detach().to(device=flat_w.device, dtype=torch.float32).contiguous().clone()

    def _resync_device_state(self):
        if self.lr_dev is not None:
            self.step_dev.fill_(self._steps)
            self._lr_pushed = None
            self.sync_device_state()

    def load_state_dict(self, sd):
        self._mom, self._steps = self._adopt("momentum_buffer", sd["momentum_buffer"]), int(sd["steps"])
        self.param_groups = [dict(g) for g in sd["param_groups"]]
        self._resync_device_state()


class FusedAdam:
    """torch.optim.Adam(params, weight_decay=wd) as train.py:432-436 builds it (torch defaults lr 1e-3,
    betas (0.9, 0.999), eps 1e-8; L2 decay added to the gradient) as ONE kernel over the engine's flat buffers."""

    decoupled = False

    def __init__(self, model, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 0.0):
        self.model = getattr(model, "module", model)
        self.engine = self.model.engine()
        self.param_groups = [{"lr": lr, "betas": tuple(betas), "eps": eps, "weight_decay": weight_decay}]
        self._m = self._v = None
        self._steps = 0
        self.lr_dev = None
        self.step_dev = None

    zero_grad = FusedSGD.zero_grad
    _adopt = FusedSGD._adopt
    _resync_device_state = FusedSGD._resync_device_state
    enable_device_state = FusedSGD.enable_device_state
    sync_device_state = FusedSGD.sync_device_state

    def step(self):
        eng = self.engine
        flat_w = eng.flatten_parameters()
        flat_g = eng.flat_g
        if flat_g is None:
            raise RuntimeError(f"{type(self).__name__}.step() before any backward pass")
        if self._m is None or self._m.numel() != flat_w.numel() or self._m.device != flat_w.device:
            self._m, self._v = torch.zeros_like(flat_w), torch.zeros_like(flat_w)
            self._steps = 0
        self._steps += 1
        g = self.param_groups[0]
        if self.step_dev is not None:
            self.step_dev.add_(1)          # counted on the stream: a replayed graph advances the bias correction itself
        _lib.check(_lib.lib().iswm_adam_step(flat_w.data_ptr(), flat_g.data_ptr(), self._m.data_ptr(), self._v.data_ptr(),
                                             flat_w.numel(), g["lr"], g["betas"][0], g["betas"][1], g["eps"], g["weight_decay"],
                                             1 if self.decoupled else 0, self._steps,
                                             None if self.lr_dev is None else self.lr_dev.data_ptr(),
                                             None if self.step_dev is None else self.step_dev.data_ptr(),
                                             torch.cuda.current_stream().cuda_stream), "adam_step")
        eng.invalidate_packed()

    def state_dict(self):
        return {"exp_avg": self._m, "exp_avg_sq": self._v, "steps": self._steps, "param_groups": self.param_groups}

    def load_state_dict(self, sd):
        self._m, self._v = self._adopt("exp_avg", sd["exp_avg"]), self._adopt("exp_avg_sq", sd["exp_avg_sq"])
        self._steps = int(sd["steps"])
        self.param_groups = [dict(g) for g in sd["param_groups"]]
        self._resync_device_state()


class FusedAdamW(FusedAdam):
    """torch.optim.AdamW(params, weight_decay=wd) (train.py:437-441): decoupled decay p *= 1 - lr * wd."""

    decoupled = True

    def __init__(self, model, lr: float = 1e-3, betas=(0.9, 0.999), eps: float = 1e-8, weight_decay: float = 1e-2):
        super().__init__(model, lr, betas, eps, weight_decay)


def setup_optimizer(model, opts):
    """train.py:421-444: opts.optimizer in {'sgd', 'adam', 'adamw'}, opts.weight_decay; the learning rate is torch's
    default 1e-3 for all three (`--lr` only reaches the scheduler's eta_min, train.py:446-452)."""
    if opts.optimizer == "sgd":
        return FusedSGD(model, momentum=0.9, weight_decay=opts.weight_decay, nesterov=True)
    elif opts.optimizer == "adam":
        return FusedAdam(model, weight_decay=opts.weight_decay)
    elif opts.optimizer == "adamw":
        return FusedAdamW(model, weight_decay=opts.weight_decay)
    raise ValueError(f"Unsupported optimizer: {opts.optimizer}")


def setup_scheduler(optimizer, opts):
    """train.py:446-452."""
    return CosineAnnealingLR(optimizer, T_max=opts.total_itrs, eta_min=opts.lr * 0.01)


class CosineAnnealingLR:
    """torch.optim.lr_scheduler.CosineAnnealingLR(T_max=total_itrs, eta_min=lr*0.01) as set up at
    train.py:446-452 and stepped every iteration (train.py:1103); closed form."""

    def __init__(self, optimizer, T_max: int, eta_min: float = 0.0):
        import math
        self._math = math
        self.opt, self.T_max, self.eta_min = optimizer, T_max, eta_min
        self.base_lr = optimizer.param_groups[0]["lr"]
        self.last_epoch = 0

    def step(self):
        self.last_epoch += 1
        m = self._math
        lr = self.eta_min + (self.base_lr - self.eta_min) * (1 + m.cos(m.pi * self.last_epoch / self.T_max)) / 2
        self.opt.param_groups[0]["lr"] = lr

    def get_last_lr(self):
        return [self.opt.param_groups[0]["lr"]]

    def state_dict(self):
        """Same keys torch's scheduler saves (train.py:570 stores it in every checkpoint, :1016 restores it)."""
        return {"T_max": self.T_max, "eta_min": self.eta_min, "base_lrs": [self.base_lr], "last_epoch": self.last_epoch,
                "_step_count": self.last_epoch + 1, "_last_lr": self.get_last_lr()}

    def load_state_dict(self, sd):
        self.T_max, self.eta_min = sd["T_max"], sd["eta_min"]
        self.base_lr = sd["base_lrs"][0] if "base_lrs" in sd else sd["base_lr"]
        self.last_epoch = sd["last_epoch"]
        if "_last_lr" in sd:
            self.opt.param_groups[0]["lr"] = sd["_last_lr"][0]
