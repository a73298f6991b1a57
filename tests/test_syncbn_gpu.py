"""Synchronised BatchNorm (DataParallel(..., sync_bn=True)).

One GPU: with one rank's statistics as the "global" sums (folded by iswm_syncbn_exchange itself, count = M), every
*_global BatchNorm kernel is bit-identical to the kernel it extends, for every variant the engine launches.
One rank of torch.distributed: the whole synchronised step - symmetric arena, exchange launches with their barriers, every
BatchNorm site, graph capture - computes what the unsynchronised step computes (global = local statistics).
Two GPUs (skipped below 2): a synchronised data-parallel step matches one GPU taking the whole batch, on both transports,
with equal and unequal shards, graphed and eager; the unsynchronised step visibly does not."""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import sys

import pytest
import torch

from iswm_b200 import _lib
from iswm_b200._lib import check

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DEV = torch.device("cuda", 0)


def _st():
    return torch.cuda.current_stream().cuda_stream


def _bf16(*shape, seed):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * 1.5 + 0.3).to(torch.bfloat16).to(DEV)


def _fold(vecs, n, rows):
    """The exchange kernel at one rank: [(tensor of n*rep fp64, rep)] -> slots of n sums + the row count."""
    L = _lib.lib()
    total = sum(((n * rep + 1 + 63) // 64) * 64 for _, rep in vecs) + len(vecs) * (((n + 1 + 63) // 64) * 64)
    arena = torch.zeros(total, dtype=torch.float64, device=DEV)
    jobs = (_lib.SyncBnJob * len(vecs))()
    off, dsts = 0, []
    for j, (v, rep) in enumerate(vecs):
        arena[off:off + n * rep].copy_(v)
        jobs[j].src_off, jobs[j].n, jobs[j].replicas = off, n, rep
        off += ((n * rep + 1 + 63) // 64) * 64
    for j in range(len(vecs)):
        d = arena[off:off + n + 1]
        jobs[j].dst = d.data_ptr()
        dsts.append(d)
        off += ((n + 1 + 63) // 64) * 64
    local = (C.c_void_p * 1)(arena.data_ptr())
    check(L.iswm_syncbn_exchange(jobs, len(vecs), local, None, 0, 1, float(rows), None, _st()), "syncbn_exchange")
    return dsts


def _stats_of(raw, rep):
    """fp64 per-channel (sum, sum of squares) spread over `rep` copies the way the convolution epilogue may leave them."""
    x = raw.double().reshape(-1, raw.shape[-1])
    s = torch.cat([x.sum(0), (x * x).sum(0)])
    if rep == 1:
        return s
    parts = [s * (0.5 ** (r + 1)) for r in range(rep - 1)]
    return torch.cat(parts + [s - sum(parts)])


def _bn_state(C_, seed):
    g = torch.Generator().manual_seed(seed)
    return dict(gamma=(torch.rand(C_, generator=g) + 0.5).to(DEV), beta=(torch.randn(C_, generator=g) * 0.1).to(DEV),
                rm=(torch.randn(C_, generator=g) * 0.1).to(DEV), rv=(torch.rand(C_, generator=g) + 0.5).to(DEV),
                nbt=torch.zeros(1, dtype=torch.int64, device=DEV))


def _clone_state(st):
    return {k: v.clone() for k, v in st.items()}


@pytest.mark.parametrize("rep", [1, 4])
@pytest.mark.parametrize("res", [False, True])
@pytest.mark.parametrize("relu", [0, 1])
@pytest.mark.parametrize("drop", [0.0, 0.1])
def test_bn_train_apply_global_is_bit_identical_at_one_rank(rep, res, relu, drop):
    L = _lib.lib()
    M, C_ = 1000, 64 if rep > 1 else 256
    x = _bf16(M, C_, seed=1)
    r = _bf16(M, C_, seed=2) if res else None
    stats = _stats_of(x, rep)
    gstats = _fold([(stats, rep)], 2 * C_, M)[0]
    step = torch.full((1,), 3, dtype=torch.int64, device=DEV)
    outs = []
    for glob in (False, True):
        st = _bn_state(C_, 3)
        save = torch.empty(2 * C_, dtype=torch.float32, device=DEV)
        out = torch.empty(M, C_, dtype=torch.bfloat16, device=DEV)
        bits = torch.zeros(M, C_ // 8, dtype=torch.uint8, device=DEV) if (relu and res) else None
        tail = (st["gamma"].data_ptr(), st["beta"].data_ptr(), 1e-5, 0.1, st["rm"].data_ptr(), st["rv"].data_ptr(), st["nbt"].data_ptr(),
                save.data_ptr(), save[C_:].data_ptr(), None if r is None else r.data_ptr(), C_, relu, drop, 77, step.data_ptr(),
                out.data_ptr(), C_, None if bits is None else bits.data_ptr(), _st())
        if glob:
            check(L.iswm_bn_train_apply_global(x.data_ptr(), C_, gstats.data_ptr(), M, C_, *tail))
        else:
            check(L.iswm_bn_train_apply(x.data_ptr(), C_, stats.data_ptr(), rep, M, C_, *tail))
        outs.append([out, save, st["rm"], st["rv"], st["nbt"]] + ([bits] if bits is not None else []))
    torch.cuda.synchronize()
    for a, b in zip(*outs):
        assert torch.equal(a, b)


@pytest.mark.parametrize("mode", ["none", "recompute", "act", "bits"])
@pytest.mark.parametrize("drop", [0.0, 0.1])
@pytest.mark.parametrize("dz", [False, True])
def test_bn_bwd_apply_global_is_bit_identical_at_one_rank(mode, drop, dz):
    L = _lib.lib()
    M, C_ = 1000, 128
    dout, x = _bf16(M, C_, seed=4), _bf16(M, C_, seed=5)
    st = _bn_state(C_, 6)
    xd = x.double()
    mean, var = xd.mean(0), xd.var(0, unbiased=False)
    save = torch.cat([mean.float(), torch.rsqrt(var.float() + 1e-5)])
    act, relu, act_ld = None, 0, C_
    if mode == "recompute":
        relu = 1
    elif mode == "act":
        act, relu = _bf16(M, C_, seed=7), 1
    elif mode == "bits":
        act, relu = torch.randint(0, 256, (M, C_ // 8), dtype=torch.uint8, device=DEV), 2
    step = torch.full((1,), 5, dtype=torch.int64, device=DEV)
    sums = torch.zeros(2 * C_ + 2, dtype=torch.float64, device=DEV)
    check(L.iswm_bn_bwd_reduce(dout.data_ptr(), C_, x.data_ptr(), C_, None if act is None else act.data_ptr(), act_ld, M, C_,
                               save.data_ptr(), save[C_:].data_ptr(), st["gamma"].data_ptr(), st["beta"].data_ptr(), relu, drop, 9,
                               step.data_ptr(), sums.data_ptr(), _st()))
    gsums = _fold([(sums[:2 * C_], 1)], 2 * C_, M)[0]
    outs = []
    for glob in (False, True):
        dx = torch.empty(M, C_, dtype=torch.bfloat16, device=DEV)
        dzt = torch.empty(M, C_, dtype=torch.bfloat16, device=DEV) if dz else None
        dg, db = torch.full((C_,), 0.25, device=DEV), torch.full((C_,), -0.5, device=DEV)
        head = (dout.data_ptr(), C_, x.data_ptr(), C_, None if act is None else act.data_ptr(), act_ld, M, C_,
                st["gamma"].data_ptr(), st["beta"].data_ptr(), save.data_ptr(), save[C_:].data_ptr())
        tail = (relu, drop, 9, step.data_ptr(), dx.data_ptr(), C_, None if dzt is None else dzt.data_ptr(), C_, dg.data_ptr(), db.data_ptr(), _st())
        if glob:
            check(L.iswm_bn_bwd_apply_global(*head, gsums.data_ptr(), sums.data_ptr(), *tail))
        else:
            check(L.iswm_bn_bwd_apply(*head, sums.data_ptr(), *tail))
        outs.append([dx, dg, db] + ([dzt] if dz else []))
    torch.cuda.synchronize()
    for a, b in zip(*outs):
        assert torch.equal(a, b)


def _side(st, stats, save, rep, fwd=True):
    return _lib.BnSide(None if stats is None else stats.data_ptr(), st["gamma"].data_ptr(), st["beta"].data_ptr(),
                       st["rm"].data_ptr() if fwd else None, st["rv"].data_ptr() if fwd else None, st["nbt"].data_ptr() if fwd else None,
                       save.data_ptr(), save[save.numel() // 2:].data_ptr(), rep)


@pytest.mark.parametrize("rep", [1, 4])
def test_bn_dual_global_is_bit_identical_at_one_rank(rep):
    L = _lib.lib()
    M, C_ = 777, 128 if rep > 1 else 512
    xa, xb, dout = _bf16(M, C_, seed=10), _bf16(M, C_, seed=11), _bf16(M, C_, seed=12)
    sa, sb = _stats_of(xa, rep), _stats_of(xb, rep)
    ga, gb = _fold([(sa, rep), (sb, rep)], 2 * C_, M)
    res = []
    for glob in (False, True):
        A, Bs = _bn_state(C_, 13), _bn_state(C_, 14)
        save_a, save_b = torch.empty(2 * C_, device=DEV), torch.empty(2 * C_, device=DEV)
        out = torch.empty(M, C_, dtype=torch.bfloat16, device=DEV)
        bits = torch.empty(M, C_ // 8, dtype=torch.uint8, device=DEV)
        a_side = _side(A, ga if glob else sa, save_a, 1 if glob else rep)
        b_side = _side(Bs, gb if glob else sb, save_b, 1 if glob else rep)
        fwd = L.iswm_bn_dual_train_apply_global if glob else L.iswm_bn_dual_train_apply
        check(fwd(xa.data_ptr(), C_, C.byref(a_side), xb.data_ptr(), C_, C.byref(b_side), M, C_, 1e-5, 0.1, out.data_ptr(), C_, bits.data_ptr(), _st()))
        sums_a = torch.zeros(2 * C_ + 2, dtype=torch.float64, device=DEV)
        sums_b = torch.zeros(2 * C_ + 2, dtype=torch.float64, device=DEV)
        a_b, b_b = _side(A, None, save_a, 1, False), _side(Bs, None, save_b, 1, False)
        check(L.iswm_bn_dual_bwd_reduce(dout.data_ptr(), C_, bits.data_ptr(), xa.data_ptr(), C_, C.byref(a_b), xb.data_ptr(), C_, C.byref(b_b),
                                        M, C_, sums_a.data_ptr(), sums_b.data_ptr(), _st()))
        dxa, dxb = torch.empty(M, C_, dtype=torch.bfloat16, device=DEV), torch.empty(M, C_, dtype=torch.bfloat16, device=DEV)
        grads = [torch.full((C_,), v, device=DEV) for v in (0.1, 0.2, 0.3, 0.4)]
        tail = (M, C_, dxa.data_ptr(), C_, dxb.data_ptr(), C_) + tuple(g.data_ptr() for g in grads) + (_st(),)
        if glob:
            gsa, gsb = _fold([(sums_a[:2 * C_], 1), (sums_b[:2 * C_], 1)], 2 * C_, M)
            check(L.iswm_bn_dual_bwd_apply_global(dout.data_ptr(), C_, bits.data_ptr(), xa.data_ptr(), C_, C.byref(a_b), gsa.data_ptr(), sums_a.data_ptr(),
                                                  xb.data_ptr(), C_, C.byref(b_b), gsb.data_ptr(), sums_b.data_ptr(), *tail))
        else:
            check(L.iswm_bn_dual_bwd_apply(dout.data_ptr(), C_, bits.data_ptr(), xa.data_ptr(), C_, C.byref(a_b), sums_a.data_ptr(),
                                           xb.data_ptr(), C_, C.byref(b_b), sums_b.data_ptr(), *tail))
        res.append([out, bits, save_a, save_b, A["rm"], A["rv"], A["nbt"], Bs["rm"], Bs["rv"], Bs["nbt"], dxa, dxb] + grads)
    torch.cuda.synchronize()
    for a, b in zip(*res):
        assert torch.equal(a, b)


@pytest.mark.parametrize("rep", [1, 4])
def test_stem_pool_fwd_global_is_bit_identical_at_one_rank(rep):
    L = _lib.lib()
    B, H, W = 2, 37, 50
    Ho, Wo = (H + 1) // 2, (W + 1) // 2
    raw = _bf16(B, H, W, 64, seed=20)
    stats = _stats_of(raw, rep)
    g = _fold([(stats, rep)], 128, B * H * W)[0]
    res = []
    for glob in (False, True):
        st = _bn_state(64, 21)
        save = torch.empty(128, device=DEV)
        out = torch.empty(B, Ho, Wo, 64, dtype=torch.bfloat16, device=DEV)
        idx = torch.empty(B, Ho, Wo, 64, dtype=torch.uint8, device=DEV)
        side = _side(st, g if glob else stats, save, 1 if glob else rep)
        fwd = L.iswm_stem_pool_fwd_global if glob else L.iswm_stem_pool_fwd
        check(fwd(raw.data_ptr(), C.byref(side), B, H, W, 64, Ho, Wo, 1e-5, 0.1, out.data_ptr(), idx.data_ptr(), _st()))
        res.append([out, idx, save, st["rm"], st["rv"], st["nbt"]])
    torch.cuda.synchronize()
    for a, b in zip(*res):
        assert torch.equal(a, b)


def test_exchange_fold_sums_copies_in_order_and_writes_the_count():
    n, rep = 256, 4
    g = torch.Generator().manual_seed(30)
    v = torch.randn(n * rep, generator=g, dtype=torch.float64).to(DEV)
    d = _fold([(v, rep)], n, 1234)[0]
    ref = v[:n].clone()
    for r in range(1, rep):
        ref = ref + v[r * n:(r + 1) * n]
    torch.cuda.synchronize()
    assert torch.equal(d[:n], ref) and float(d[n]) == 1234.0


WORKER = r'''
import os, sys, datetime
sys.path.insert(0, os.environ["ISWM_ROOT"])
import torch, torch.distributed as dist
from iswm_b200.network import modeling
from iswm_b200.utils.loss import CrossEntropyLoss
from iswm_b200.parallel import DataParallel
from oracle.gen_golden import seeded_state_dict, synth_labels

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
assert world == 2
torch.cuda.set_device(rank)
dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=120))

def build():
    m = modeling.deeplabv3plus_resnet50(num_classes=2, output_stride=16, pretrained_backbone=False)
    m.load_state_dict(seeded_state_dict(m.state_dict(), 5))
    m.to(dev).train()
    m.engine().dropout_p = 0.0
    return m

def bn_stats(m):
    return [b for name, b in m.named_buffers() if name.endswith("running_mean") or name.endswith("running_var")]

def rel_stats(a, b):
    return max(float((x - y).norm() / y.norm()) for x, y in zip(bn_stats(a), bn_stats(b)))

B, H, W = 8, 64, 64
g = torch.Generator().manual_seed(11)
x = torch.randn((B, 3, H, W), generator=g)
x[:4] = x[:4] * 1.7 + 0.4                                    # shards with visibly different statistics
y = synth_labels((B, H, W), seed=12, fg=0.3)
y[:4] = synth_labels((4, H, W), seed=13, fg=0.85)
w = torch.tensor([1.0, 4.0])

# one GPU, whole batch (every rank computes it: the reference is local)
ref = build()
rc = CrossEntropyLoss(weight=w).to(dev)
ref_loss = rc(ref(x.to(dev)), y.to(dev))
ref_loss.backward()
torch.cuda.synchronize()
ref_g = ref.engine().flat_g.clone()
ref_loss = float(ref_loss)

def dp_step(comm, sync, split):
    m = build()
    c = CrossEntropyLoss(weight=w).to(dev)
    d = DataParallel(m, c, bucket_bytes=4 << 20, comm=comm, sync_bn=sync)
    assert d.comm_mode == comm, d.comm_mode
    lo = sum(split[:rank])
    xs, ys = x[lo:lo + split[rank]].to(dev), y[lo:lo + split[rank]].to(dev)
    loss = float(d.train_step(xs, ys, optimizer=None))
    torch.cuda.synchronize()
    flat = m.engine().flat_g[:ref_g.numel()].clone()
    m.engine().grad_ready_hook = None
    return m, loss, flat

def cross_rank_equal(t):
    lst = [torch.zeros_like(t) for _ in range(world)]
    dist.all_gather(lst, t.contiguous())
    return all(torch.equal(a, lst[0]) for a in lst)

for comm in ("peer", "nccl"):
    for split in ((4, 4), (3, 5)):
        m, loss, flat = dp_step(comm, True, split)
        rl = abs(loss - ref_loss) / abs(ref_loss)
        rg = float((flat - ref_g).norm() / ref_g.norm())
        rs = rel_stats(m, ref)
        same = cross_rank_equal(torch.cat([b.flatten() for b in bn_stats(m)]))
        tag = f"{comm} {split[0]}+{split[1]}"
        if rank == 0:
            print(f"RESULT sync_bn=True {tag}: loss_rel={rl:.2e} grad_rel={rg:.2e} running_stats_rel={rs:.2e} ranks_bit_equal={same}", flush=True)
        assert rl <= 1e-5 and rg <= 1e-4 and rs <= 1e-6 and same, (tag, rl, rg, rs, same)
        if split == (4, 4):
            # after a synchronised step every rank evaluates with the same running statistics: identical logits
            m.eval()
            with torch.no_grad():
                logits = m(x[:2].to(dev))
            torch.cuda.synchronize()
            assert cross_rank_equal(logits), "eval logits differ across ranks"
        dist.barrier()
    m, loss, flat = dp_step(comm, False, (4, 4))
    rs_off = rel_stats(m, ref)
    if rank == 0:
        print(f"RESULT sync_bn=False {comm} 4+4: running_stats_rel={rs_off:.2e} (per-shard statistics)", flush=True)
    assert rs_off > 1e-4, rs_off              # per-shard statistics miss the 1e-6 bar by orders of magnitude
    dist.barrier()

# the synchronised data-parallel step replayed from ONE CUDA graph against the same steps launched eagerly, from the same state
from iswm_b200.graphs import GraphedTrainStep
from iswm_b200.optim import FusedSGD
xs, ys = x.chunk(world)[rank].to(dev), y.chunk(world)[rank].to(dev)
res = []
for graphed in (False, True):
    m = build()
    c = CrossEntropyLoss(weight=w).to(dev)
    d = DataParallel(m, c, bucket_bytes=4 << 20, comm="peer", sync_bn=True)
    opt = FusedSGD(m, lr=1e-2, momentum=0.9, weight_decay=1e-4)
    stepper = GraphedTrainStep(m, c, opt, dp=d) if graphed else None
    losses = []
    for _ in range(2):
        l = stepper(xs, ys) if graphed else d.train_step(xs, ys, opt)
        losses.append(float(l))
    torch.cuda.synchronize()
    res.append((losses, m.engine().flat_w.clone(), torch.cat([b.flatten() for b in bn_stats(m)])))
    if graphed:
        assert stepper.launches_per_replay > 0
    m.engine().grad_ready_hook = None
    dist.barrier()
(le, we, se), (lg, wg, sg) = res
relw = float((wg - we).norm() / we.norm())
rels = float((sg - se).norm() / se.norm())
if rank == 0:
    print(f"RESULT graphed sync_bn: losses eager={le} graph={lg} rel_w={relw:.3e} rel_running_stats={rels:.3e}", flush=True)
assert abs(le[0] - lg[0]) <= 1e-6 * abs(le[0]), (le, lg)
assert relw <= 1e-5, relw
assert cross_rank_equal(sg)
dist.barrier()
dist.destroy_process_group()
'''


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_sync_bn_two_ranks_match_one_gpu_on_the_whole_batch(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(WORKER)
    env = dict(os.environ, ISWM_ROOT=ROOT)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr", "127.0.0.1",
                        "--master-port", "29547", str(script)], capture_output=True, text=True, env=env, timeout=900)
    print(r.stdout[-4000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("RESULT") == 7


WORKER_ONE = r"""
import os, sys, datetime
sys.path.insert(0, os.environ["ISWM_ROOT"])
import torch, torch.distributed as dist
from iswm_b200.network import modeling
from iswm_b200.utils.loss import CrossEntropyLoss
from iswm_b200.parallel import DataParallel
from iswm_b200.graphs import GraphedTrainStep
from iswm_b200.optim import FusedSGD
from oracle.gen_golden import seeded_state_dict, synth_labels

dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=120))

def build():
    m = modeling.deeplabv3plus_resnet50(num_classes=2, output_stride=16, pretrained_backbone=False)
    m.load_state_dict(seeded_state_dict(m.state_dict(), 5))
    m.to(dev).train()
    m.engine().dropout_p = 0.0
    return m

def stats(m):
    return torch.cat([b.flatten() for n, b in m.named_buffers() if n.endswith("running_mean") or n.endswith("running_var")])

B, H, W = 5, 64, 64
g = torch.Generator().manual_seed(11)
x = torch.randn((B, 3, H, W), generator=g).to(dev)
y = synth_labels((B, H, W), seed=12, fg=0.3).to(dev)
w = torch.tensor([1.0, 4.0])
for comm in ("peer", "nccl"):
    out = {}
    for sync in (False, True):
        m = build()
        c = CrossEntropyLoss(weight=w).to(dev)
        d = DataParallel(m, c, bucket_bytes=4 << 20, comm=comm, sync_bn=sync)
        assert d.comm_mode == comm
        loss = float(d.train_step(x, y, optimizer=None))
        torch.cuda.synchronize()
        n = sum(p.numel() for p in m.parameters())
        out[sync] = (loss, m.engine().flat_g[:n].clone(), stats(m))
        m.engine().grad_ready_hook = None
    (l0, g0, s0), (l1, g1, s1) = out[False], out[True]
    rl, rg, rs = abs(l1 - l0) / abs(l0), float((g1 - g0).norm() / g0.norm()), float((s1 - s0).norm() / s0.norm())
    print(f"RESULT one rank {comm}: sync vs per-rank loss_rel={rl:.2e} grad_rel={rg:.2e} running_stats_rel={rs:.2e}", flush=True)
    assert rl <= 1e-6 and rg <= 1e-4 and rs <= 1e-7, (comm, rl, rg, rs)
res = []
for graphed in (False, True):
    m = build()
    c = CrossEntropyLoss(weight=w).to(dev)
    d = DataParallel(m, c, bucket_bytes=4 << 20, comm="peer", sync_bn=True)
    opt = FusedSGD(m, lr=1e-2, momentum=0.9, weight_decay=1e-4)
    stepper = GraphedTrainStep(m, c, opt, dp=d) if graphed else None
    losses = [float(stepper(x, y) if graphed else d.train_step(x, y, opt)) for _ in range(2)]
    torch.cuda.synchronize()
    res.append((losses, m.engine().flat_w.clone(), stats(m)))
    m.engine().grad_ready_hook = None
(le, we, se), (lg, wg, sg) = res
relw, rels = float((wg - we).norm() / we.norm()), float((sg - se).norm() / se.norm())
print(f"RESULT one rank graphed sync_bn: losses eager={le} graph={lg} rel_w={relw:.3e} rel_running_stats={rels:.3e}", flush=True)
assert abs(le[0] - lg[0]) <= 1e-6 * abs(le[0]) and relw <= 1e-5 and rels <= 1e-6, (le, lg, relw, rels)
dist.destroy_process_group()
"""


def test_sync_bn_one_rank_matches_per_rank_statistics(tmp_path):
    script = tmp_path / "worker_one.py"
    script.write_text(WORKER_ONE)
    env = dict(os.environ, ISWM_ROOT=ROOT)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "1", "--master-addr", "127.0.0.1",
                        "--master-port", "29549", str(script)], capture_output=True, text=True, env=env, timeout=900)
    print(r.stdout[-3000:])
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-3000:]
    assert r.stdout.count("RESULT") == 3
