"""Peer-memory communicator: the data-parallel exchanges of a train step as plain CUDA kernels over NVLink 5 / NVSwitch.

One process per GPU. Buffers that ranks exchange live in SYMMETRIC memory (torch.distributed._symmetric_memory: same size on
every GPU, every rank's copy mapped into every other rank's address space); the kernels of csrc/peer_allreduce.cu read and
write the peers' copies directly. Nothing here synchronises with the host and nothing calls into a communication library
after set-up, so the whole data-parallel step - gradient all-reduce included - is captured in ONE CUDA graph.

Three independent barrier CHANNELS (own flags, own epoch counter): 0 for the main stream's exchanges (class histogram before
the loss kernel, loss numerators after it, and with synchronised BatchNorm the statistics of every BatchNorm the main stream
runs), 1 for the gradient buckets on the communication stream, 2 for the synchronised-BatchNorm statistics of the forward
branches the engine runs on its side stream (low-level projection, pooled ASPP branch). Barriers of one channel are issued in
the same order on every rank; barriers of different channels may interleave differently per rank.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.distributed as dist

from . import _lib
from ._lib import check

_FLAGS_BYTES = 64            # per channel: 8 x uint32 (+ padding)
_N_CHANNELS = 3
_SLOT_REGION = 64            # 8-byte slots per region
_N_REGIONS = 4
_CTL_BYTES = _N_CHANNELS * _FLAGS_BYTES + _N_REGIONS * _SLOT_REGION * 8


class PeerComm:
    def __init__(self, device: torch.device, group=None):
        import torch.distributed._symmetric_memory as symm
        if not dist.is_initialized():
            raise RuntimeError("torch.distributed must be initialised first")
        self._symm = symm
        self.group = group if group is not None else dist.group.WORLD
        self.rank, self.world = dist.get_rank(self.group), dist.get_world_size(self.group)
        if self.world > 8:
            raise RuntimeError("PeerComm covers the GPUs of ONE NVSwitch domain (<= 8 ranks)")
        self.device = device
        self.ctl, self.ctl_ptrs = self.alloc(_CTL_BYTES, torch.uint8)
        self.ctl.zero_()
        torch.cuda.synchronize(device)
        dist.barrier(self.group)                                     # every rank's flags are zero before anyone signals
        self._flag_ptrs = [self._ptr_array([p + ch * _FLAGS_BYTES for p in self.ctl_ptrs]) for ch in range(_N_CHANNELS)]
        base = _N_CHANNELS * _FLAGS_BYTES
        self._slot_ptrs = self._ptr_array([p + base for p in self.ctl_ptrs])
        self.epochs = torch.zeros(_N_CHANNELS, dtype=torch.int32, device=device)

    def _ptr_array(self, ptrs):
        return (C.c_void_p * self.world)(*[int(p) for p in ptrs])

    def alloc(self, numel: int, dtype: torch.dtype):
        """(tensor, [peer pointers]) of a symmetric allocation; collective (every rank calls it with the same size)."""
        t = self._symm.empty(numel, dtype=dtype, device=self.device)
        hdl = self._symm.rendezvous(t, self.group)
        ptrs = [int(p) for p in hdl.buffer_ptrs]
        if ptrs[self.rank] != t.data_ptr():
            raise RuntimeError("symmetric memory: the local mapping differs from the tensor's pointer")
        keep = getattr(self, "_handles", None)
        if keep is None:
            keep = self._handles = []
        keep.append((t, hdl))
        return t, ptrs

    def barrier(self, channel: int, stream: int):
        check(_lib.lib().iswm_peer_barrier(self._flag_ptrs[channel], self.rank, self.world, self.epochs[channel:].data_ptr(), stream), "peer_barrier")

    def allreduce_f32(self, ptr_array, offset: int, n: int, stream: int, max_blocks: int = 0, channel: int = 1):
        """buf[offset:offset+n] = sum over ranks (bit-identical on every rank), bracketed by the two barriers it needs."""
        L = _lib.lib()
        self.barrier(channel, stream)
        check(L.iswm_peer_allreduce_f32(ptr_array, self.rank, self.world, offset, n, max_blocks, stream), "peer_allreduce_f32")
        self.barrier(channel, stream)

    def bn_exchange(self, arena_ptrs, jobs, n_jobs: int, rows: int, channel: int, stream: int):
        """Synchronised BatchNorm statistics (iswm_syncbn_exchange): `jobs` (ctypes iswm_syncbn_job array) name slots of the
        symmetric arena whose peer mappings are `arena_ptrs`; this rank contributes `rows` rows to the global count."""
        check(_lib.lib().iswm_syncbn_exchange(jobs, n_jobs, arena_ptrs, self._flag_ptrs[channel], self.rank, self.world, float(rows),
                                              self.epochs[channel:].data_ptr(), stream), "syncbn_exchange")

    def small_allreduce_(self, t: torch.Tensor, region: int, stream: int, channel: int = 0) -> torch.Tensor:
        """In-place SUM over ranks of a small int64 / float64 device vector (<= 64 values); `region` names the call site."""
        if t.dtype not in (torch.int64, torch.float64) or t.numel() > _SLOT_REGION or not t.is_contiguous():
            raise ValueError("small_allreduce_: contiguous int64 / float64 vector of at most 64 values")
        if not 0 <= region < _N_REGIONS:
            raise ValueError("small_allreduce_: region out of range")
        L = _lib.lib()
        f64 = 1 if t.dtype == torch.float64 else 0
        off = region * _SLOT_REGION
        check(L.iswm_peer_small_publish(self._slot_ptrs, self.rank, self.world, t.data_ptr(), t.numel(), off, f64, stream), "peer_small_publish")
        self.barrier(channel, stream)
        check(L.iswm_peer_small_sum(self._slot_ptrs, self.world, t.data_ptr(), t.numel(), off, f64, stream), "peer_small_sum")
        return t
