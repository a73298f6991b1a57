#!/usr/bin/env python
"""bench.py — headline benchmark of the ISWM hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload train|predict|lossmetric] [--dump-outputs DIR]

Metric (BASELINE.json): train img/s of DeepLabV3+ ResNet-50 OS16, synthetic 512x512 tiles, batch 16
per GPU (cfg2), one step = forward + adaptive weighted CE + backward + SGD step. For N > 1 launch
under torch.distributed.run (one rank per GPU, NCCL); every rank keeps batch 16 (weak scaling).
Prints ONE JSON line (rank 0). `--impl reference` times the reference algorithm's CPU path (the
fp32 torch oracle, a restatement of the reference modules — /root/reference does not exist on the
GPU box) on the host cores.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

TRAIN_GFLOP_PER_IMG = {("resnet50", 16, 512): 413.64, ("resnet50", 16, 1024): 1654.52,
                       ("resnet101", 8, 1024): 6236.69}   # BASELINE.md §3: 3*fwd - stem fwd
FWD_GFLOP_PER_IMG = {("resnet50", 16, 512): 138.29, ("resnet50", 16, 1024): 553.15, ("resnet50", 16, 2048): 2212.58,
                     ("resnet101", 8, 1024): 2080.54}
PEAKS_FALLBACK = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        d["_source"] = "measured"
        return d
    d = dict(PEAKS_FALLBACK)
    d["_source"] = "fallback"
    return d


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.gpu)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def wait_first_sample(self, timeout):
        t0 = time.time()
        while self.proc is not None and not self.lines and time.time() - t0 < timeout:
            time.sleep(0.05)

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=10)                  # nvidia-smi must be gone before anything else is timed
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = float(f[2])
            except ValueError:
                continue
            for n, v in zip(names, f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


def synth_batch(B, H, W, seed, device=None, pinned=False):
    """SURVEY §8(d) synthetic inputs: randn images, 2 % foreground, 1 % ignore(255)."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((B, 3, H, W), generator=g)
    u = torch.rand((B, H, W), generator=g)
    y = (u < 0.02).long()
    y[torch.rand((B, H, W), generator=g) < 0.01] = 255
    if pinned:
        x, y = x.pin_memory(), y.pin_memory()
    if device is not None:
        x, y = x.to(device), y.to(device)
    return x, y


DUMP_SAMPLE = 1 << 22      # elements kept of a larger output: 16 MB of float32, so that no workload dumps more than 64 MB


def dump_sample(t):
    """`t` flattened; above DUMP_SAMPLE elements, a fixed seeded choice of DUMP_SAMPLE of them (in index order), the same
    on every run and for every output of that size."""
    flat = t.detach().reshape(-1)
    if flat.numel() <= DUMP_SAMPLE:
        return flat
    idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_SAMPLE].sort().values
    return flat[idx.to(flat.device)]


def dump_outputs(out_dir, arrays):
    """--dump-outputs: every array as <out_dir>/<name>.npy, int64 counts as float64 (exact), everything else as float32."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.detach().cpu()
        np.save(os.path.join(out_dir, name + ".npy"), (t.double() if t.dtype == torch.int64 else t.float()).numpy())


# ----------------------------------------------------------------------------- CPU arms
def cpu_train_step_rate(B, H, W, steps, warmup, threads=None, backbone="resnet50", output_stride=16):
    """The reference algorithm on the host: fp32 torch oracle (oracle/torch_model.py), zero_grad ->
    forward -> weighted CE -> backward -> SGD step (train.py:1045-1049), all host threads."""
    from oracle import torch_model as TM
    n = threads or os.cpu_count() or 1
    torch.set_num_threads(n)
    torch.manual_seed(0)
    model = TM.oracle_model(backbone, 2, output_stride).train()
    opt = torch.optim.SGD(model.parameters(), momentum=0.9, weight_decay=1e-4, nesterov=True)   # lr: torch default, as train.py:424-431
    crit = torch.nn.CrossEntropyLoss(weight=torch.tensor([1.0, 7.0]), ignore_index=255, reduction="mean")
    x, y = synth_batch(B, H, W, 0)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        logits = model(x)
        loss = crit(logits, y)
        opt.zero_grad()
        loss.backward()
        opt.step()
        float(loss.detach())
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    per = sum(times) / len(times)
    return B / per, per, n


def train_workload_name(backbone, output_stride, H, W, B):
    cfgname = "cfg2" if (backbone, output_stride, H, B) == ("resnet50", 16, 512, 16) else ("cfg3" if backbone == "resnet101" else "custom")
    bbname = {"resnet50": "ResNet-50", "resnet101": "ResNet-101"}[backbone]
    return (f"{cfgname}: DeepLabV3+ {bbname} OS{output_stride}, 2 classes, synthetic {H}x{W}, batch {B} per GPU, one step = forward + "
            "adaptive weighted CE + backward + fused SGD(momentum 0.9, nesterov, wd 1e-4)")


def run_reference(args):
    """CPU arm: the reference algorithm (fp32 torch oracle = restatement of the reference modules, pinned to the
    reference's own outputs by tests/golden; /root/reference does not exist on the GPU box) on all host threads,
    on a BOUNDED sample of our arm's workload (batch 2 per step instead of 16: img/s is per image)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    H = W = args.size
    steps, warmup = args.steps, 1
    if args.workload == "predict":
        Hs = min(H, 1024)
        rate, per, n = cpu_predict_rate(1, Hs, Hs, steps, warmup)
        metric = f"predict img/s DeepLabV3+ R50 {H}^2"
        workload = f"cfg4: predict.py path, DeepLabV3+ ResNet-50 OS16 eval forward on synthetic {H}x{W} tiles, batch {args.batch} per GPU, softmax[:,1] > 0.5 fused with the confusion matrix, mIoU read per step (e2e)"
        sample = f"{warmup} warm-up + {steps} timed steps of batch 1 at {Hs}x{Hs} (img/s scaled by area {Hs * Hs}/{H * W} is NOT applied), fp32"
        if Hs != H:
            rate = rate * (Hs * Hs) / (H * W)
            sample = f"{warmup} warm-up + {steps} timed steps of batch 1 at {Hs}x{Hs}, img/s scaled to {H}x{W} by pixel count (convolutions are linear in pixels), fp32"
    else:
        B = 2
        rate, per, n = cpu_train_step_rate(B, min(H, 512), min(W, 512), steps, warmup, backbone=args.backbone, output_stride=args.output_stride)
        if H > 512:
            rate = rate * (512 * 512) / (H * W)
        metric = f"train img/s DeepLabV3+ {'R50' if args.backbone == 'resnet50' else 'R101'} {H}^2"
        workload = train_workload_name(args.backbone, args.output_stride, H, W, args.batch)
        sample = (f"{warmup} warm-up + {steps} timed steps, batch {B} (of the workload's {args.batch}), {min(H, 512)}x{min(W, 512)}"
                  + (f" scaled to {H}x{W} by pixel count" if H > 512 else "") + f", {args.backbone}-OS{args.output_stride} fwd+CE+bwd+SGD, fp32, torch {torch.__version__}")
    line = {
        "impl": "reference", "metric": metric, "value": rate, "unit": "img/s",
        "n_gpus": args.gpus, "steps": steps, "warmup": warmup, "ms_per_step": per * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": workload,
                   "note": "CPU arm: fp32 torch oracle (restatement of the reference modules; /root/reference is absent on the GPU box) on the host cores, bounded sample"},
        "cpu_baseline": {"value": rate, "unit": "img/s", "cores": n, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "img/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


def traffic_from_profiles(kernel: str):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel`, from the committed ncu --set full
    capture summary (profiles/traffic.json, written by tools/ncu_summary.py); None when no capture exists."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(p):
        return None
    try:
        with open(p) as f:
            return json.load(f).get(kernel, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


def host_head_start(ms: float = 30.0):
    """Park the current stream on a spin kernel so that the host can enqueue an event-instrumented step AHEAD of the
    GPU. CUDA events around single launches measure e0->e1 on the device; when the host is the slower side (event
    creation + two records + ctypes per launch, ~25 us) the stream runs dry after e0 and the wait for the launch to
    arrive is billed to the kernel (measured: every launch read >= 11 us, a 3.5 us kernel included)."""
    torch.cuda._sleep(int(ms * 1e-3 * 1.9e9))


def profile_by_entry(fn, path):
    """One instrumented call of `fn`: CUDA events around EVERY library launch, grouped by C-ABI entry point
    (in-situ times: warm L2, pipelined launches - unlike ncu's serialised cold-cache list)."""
    from iswm_b200 import _lib
    _lib.lib()
    real = _lib._lib
    rec = []

    class _Prof:
        def __getattr__(self, name):
            f = getattr(real, name)
            if not name.startswith("iswm_") or name in ("iswm_last_error", "iswm_launch_count"):
                return f

            def wrapped(*a):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                r = f(*a)
                e1.record()
                rec.append((name, e0, e1))
                return r
            return wrapped
    _lib._lib = _Prof()
    try:
        host_head_start()
        fn()
        torch.cuda.synchronize()
    finally:
        _lib._lib = real
    by = {}
    for name, e0, e1 in rec:
        t, n = by.get(name, (0.0, 0))
        by[name] = (t + e0.elapsed_time(e1), n + 1)
    with open(path, "w") as f:
        tot = sum(t for t, n in by.values())
        for name, (t, n) in sorted(by.items(), key=lambda kv: -kv[1][0]):
            f.write(f"{name:34s} {n:4d} launches {t * 1e3:9.1f} us {100 * t / tot:5.1f}%\n")
        f.write(f"{'total':34s} {len(rec):4d} launches {tot * 1e3:9.1f} us\n")


def _time_region(fn, steps, barrier):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    w0 = time.time()
    e0.record()
    out = None
    for _ in range(steps):
        out = fn()
    e1.record()
    barrier()
    return e0.elapsed_time(e1), w0, time.time(), out


def _max_over_ranks(vals, dev, world):
    if world == 1:
        return vals
    import torch.distributed as dist
    t = torch.tensor(vals, device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return [float(v) for v in t]


def cpu_predict_rate(B, H, W, steps, warmup, threads=None):
    """predict.py:262-278 + evaluate_quantization.py:265-270 on the host: no_grad forward, softmax[:,1] > 0.5,
    StreamMetrics._fast_hist (numpy oracle), fp32 torch oracle network."""
    from oracle import oracle_np as O
    from oracle import torch_model as TM
    n = threads or os.cpu_count() or 1
    torch.set_num_threads(n)
    torch.manual_seed(0)
    model = TM.oracle_model("resnet50", 2, 16).eval()
    x, y = synth_batch(B, H, W, 0)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        with torch.no_grad():
            prob = torch.softmax(model(x), dim=1)
        pred = (prob[:, 1] > 0.5).long().numpy()
        O.fast_hist(y.numpy().reshape(-1), pred.reshape(-1), 2)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    per = sum(times) / len(times)
    return B / per, per, n


def run_predict(args, dev, world, rank, local):
    """cfg4: predict.py's forward -> softmax[:,1] > 0.5 -> StreamMetrics confusion matrix -> mIoU, batched."""
    import torch.distributed as dist
    from iswm_b200 import _lib
    from iswm_b200.metrics import StreamMetrics
    from iswm_b200.network import modeling
    B, H, W = args.batch, args.size, args.size
    torch.manual_seed(0)
    model = modeling.deeplabv3plus_resnet50(num_classes=2, output_stride=16, pretrained_backbone=False).to(dev).eval()
    metrics = StreamMetrics(2, device=dev)
    x_dev, y_dev = synth_batch(B, H, W, rank, device=dev)
    x_host, y_host = synth_batch(B, H, W, rank, pinned=True)
    y_host = y_host.to(torch.uint8).pin_memory()        # the loader's label format (ExtToTensor(target_type='uint8'), utils/ext_transforms.py:273-293)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    from iswm_b200.predict import predict_mask
    fused = os.environ.get("ISWM_PREDICT_FUSED", "1") != "0"

    def step(x, y):
        # predict.py:258-290 batched: forward -> (fused: final upsample +) softmax[:,1] > 0.5 -> uint8 mask and
        # confidence map -> confusion counts (evaluate_quantization.py:265-270)
        return predict_mask(model, x, 0.5, y, metrics, fused=fused)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    for _ in range(args.warmup):
        step(x_dev, y_dev)
    barrier()
    if rank == 0:
        sampler.wait_first_sample(5.0)
    launches0 = _lib.launch_count()
    ms, w0, w1, (pred, conf) = _time_region(lambda: step(x_dev, y_dev), args.steps, barrier)
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop(w0, w1) if rank == 0 else None
    if args.dump_outputs and rank == 0:                 # this rank's counters: the metric's all-reduce needs every rank
        dump_outputs(args.dump_outputs, {"pred": dump_sample(pred), "conf": dump_sample(conf), "confusion": metrics._cm()})
    metrics.reset()

    from iswm_b200.data import HostBatchPrefetcher
    pf = HostBatchPrefetcher([(x_host, y_host)] * 2, dev)
    for xs, ys in pf:                                   # untimed warm-up of the staging path
        step(xs, ys)
    metrics.reset()
    pf.loader = ((x_host, y_host) for _ in range(args.steps))
    pre = iter(pf)

    def e2e_step():
        xs, ys = next(pre)                              # host -> device copy of the NEXT batch overlaps this step
        step(xs, ys)
        return metrics.get_results()["MIoU"]            # device -> host read of the int64 counters every step

    ms_e2e, _, _, miou = _time_region(e2e_step, args.steps, barrier)
    ms, ms_e2e = _max_over_ranks([ms, ms_e2e], dev, world)
    roof = None
    if rank == 0:
        eng = model.engine()
        eng.profile = []
        host_head_start()
        step(x_dev, y_dev)
        torch.cuda.synchronize()
        t_ms = sum(a.elapsed_time(b) for k, fl, a, b, tag in eng.profile if k == "conv_igemm")
        fl = sum(fl for k, fl, a, b, tag in eng.profile if k == "conv_igemm")
        n = sum(1 for k, *_ in eng.profile if k == "conv_igemm")
        if args.profile_detail:
            with open(args.profile_detail, "w") as f:
                for k, fl_, a, b, tag in eng.profile:
                    dt = a.elapsed_time(b)
                    f.write(f"{tag:55s} {fl_ / 1e9:10.2f} GF {dt * 1e3:9.1f} us {fl_ / (dt * 1e-3) / 1e12:8.1f} TF/s\n")
        eng.profile = None
        if args.profile_detail:
            profile_by_entry(lambda: step(x_dev, y_dev), args.profile_detail + ".by_entry")
        pk = peaks()
        peak_tf = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
        ach = fl / (t_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "conv_igemm_kernel (forward implicit GEMMs, BN folded into the epilogue)", "achieved": ach,
                "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf, "traffic": traffic_from_profiles("conv_igemm_kernel"),
                "launches_per_step": n, "kernel_ms_per_step": t_ms, "peak_source": pk["_source"] + " bf16_tflops_sustained"}
    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return
    imgs = B * world * args.steps
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        rate, per, n = cpu_predict_rate(1, min(H, 1024), min(W, 1024), 1, 1)
        cpu = {"value": rate, "unit": "img/s", "cores": n, "kind": "port",
               "sample": f"1 warm-up + 1 timed forward+threshold+fast_hist of batch 1 at {min(H, 1024)}x{min(W, 1024)}, fp32 torch oracle on the host"}
    print(json.dumps({
        "metric": f"predict img/s DeepLabV3+ R50 {H}^2", "value": imgs / (ms * 1e-3), "unit": "img/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": f"cfg4: predict.py path, DeepLabV3+ ResNet-50 OS16 eval forward on synthetic {H}x{W} tiles, batch {B} per GPU, softmax[:,1] > 0.5 fused with the confusion matrix, mIoU read per step (e2e)",
                   "parallelism": f"dp{world}", "global_batch": B * world, "l2": "inputs and activations >> 126 MB L2", "miou": miou},
        "clocks": clocks,
        "e2e": {"value": imgs / (ms_e2e * 1e-3), "unit": "img/s", "h2d_bytes_per_step": (x_host.numel() * 4 + y_host.numel() * y_host.element_size()) * world,
                "d2h_bytes_per_step": 8 * 5 * world, "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches), "roofline": roof, "cpu_baseline": cpu}))


def run_lossmetric(args, dev, world, rank, local):
    """cfg5: class histogram, fused weighted CE fwd+bwd and argmax+confusion matrix on [B,2,S,S] logits."""
    from iswm_b200 import _lib, ops
    B, H, W = args.batch, args.size, args.size
    g = torch.Generator().manual_seed(rank)
    logits = torch.randn((B, 2, H, W), generator=g).to(dev)
    u = torch.rand((B, H, W), generator=g)
    labels = (u < 0.02).long()
    labels[torch.rand((B, H, W), generator=g) < 0.01] = 255
    labels = labels.to(dev)
    w = torch.tensor([1.0, 7.0], device=dev)
    N = B * H * W
    algo = {"class_hist": N * 8, "wce_fwd_bwd": 2 * N * 2 * 4 + N * 8, "argmax_confusion": N * 2 * 4 + N * 8}
    hist = ops.class_hist(labels, 2)
    cm = torch.zeros(5, dtype=torch.int64, device=dev)
    fns = {"class_hist": lambda: ops.class_hist(labels, 2, out=hist),
           "wce_fwd_bwd": lambda: ops.wce_fwd_bwd(logits, labels, w, hist),
           "argmax_confusion": lambda: ops.argmax_confusion(logits, labels, mode=1, threshold=0.5, out=cm)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)       # > 126 MB L2
    res, last = {}, {}
    sampler = ClockSampler(local)
    sampler.start()
    sampler.wait_first_sample(5.0)
    w0 = time.time()
    launches0 = _lib.launch_count()
    for name, fn in fns.items():
        for _ in range(args.warmup):
            fn()
        ts = []
        for _ in range(args.steps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            last[name] = fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        res[name] = {"us": ts[len(ts) // 2] * 1e3, "algorithmic_bytes": algo[name]}
    launches = _lib.launch_count() - launches0
    clocks = sampler.stop(w0, time.time())
    if args.dump_outputs and rank == 0:
        loss, grad = last["wce_fwd_bwd"]
        dump_outputs(args.dump_outputs, {"class_hist": last["class_hist"], "wce_loss": loss, "wce_grad": dump_sample(grad),
                                         "confusion": last["argmax_confusion"][0]})
    pk = peaks()
    for name, r in res.items():
        r["GB/s"] = r["algorithmic_bytes"] / (r["us"] * 1e-6) / 1e9
        r["frac_of_hbm_peak"] = r["GB/s"] / pk["hbm_gbs"]
    # e2e: host logits + labels -> loss scalar on the host, through the criterion API
    from iswm_b200.utils.loss import CrossEntropyLoss
    crit = CrossEntropyLoss(weight=w).to(dev)
    lh, yh = logits.cpu().pin_memory(), labels.cpu().pin_memory()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        v = float(crit(lh.to(dev, non_blocking=True), yh.to(dev, non_blocking=True)))
    e2e_s = (time.perf_counter() - t0) / args.steps
    total_us = sum(r["us"] for r in res.values())
    k = "wce_fwd_bwd"
    cpu = None
    if not args.no_cpu_baseline:
        from oracle import oracle_np as O
        ln, yn, wn = logits[:2].cpu().numpy(), labels[:2].cpu().numpy(), w.cpu().numpy()
        t0 = time.perf_counter()
        O.class_hist(yn, 2)
        O.weighted_ce(ln, yn, wn)
        O.fast_hist(yn.reshape(-1), O.threshold_pred(ln)[0].reshape(-1), 2)
        dt = time.perf_counter() - t0
        cpu = {"value": 2 * H * W / dt / 1e6, "unit": "Mpx/s", "cores": 1, "kind": "port", "sample": f"numpy oracle, histogram + weighted CE fwd/bwd + threshold + fast_hist on 2 of the {B} images"}
    print(json.dumps({
        "metric": "loss+metric Mpx/s (class histogram + weighted CE fwd/bwd + argmax confusion matrix)", "value": N / (total_us * 1e-6) / 1e6, "unit": "Mpx/s",
        "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_us * 1e-3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"cfg5: loss+metrics microbench on {B}x2x{H}x{W} fp32 logits, int64 labels (2 % foreground, 1 % ignore)", "l2": "256 MB flush write between timed launches",
                   "kernels": res, "loss": v},
        "clocks": clocks,
        "e2e": {"value": N / e2e_s / 1e6, "unit": "Mpx/s", "h2d_bytes_per_step": lh.numel() * 4 + yh.numel() * 8, "d2h_bytes_per_step": 4, "ms_per_step": e2e_s * 1e3},
        "gpu_launches": int(launches),
        "roofline": {"bound": "hbm", "kernel": "wce2_kernel (fused weighted softmax-CE forward + backward)", "achieved": res[k]["GB/s"], "peak": pk["hbm_gbs"],
                     "unit": "GB/s", "frac": res[k]["frac_of_hbm_peak"], "traffic": traffic_from_profiles("cfg5:wce_fwd_bwd"), "peak_source": pk["_source"] + " hbm_gbs"},
        "cpu_baseline": cpu}))


def dp_parity_check(dev, world, rank):
    """Multi-rank parity INSIDE the driver's own run (every --gpus N > 1 call, before the timed region): one train step of
    DeepLabV3+ R50-OS16 on a fixed global batch sharded over the ranks (6 images of 128x128 per rank, very different class
    mixes per shard, Dropout off) through iswm_b200.parallel.DataParallel, against rank 0's single-GPU restatement of
    nn.DataParallel's semantics (train.py:970, :1045-1048; SURVEY 8e): per-shard forward / backward with per-shard
    BatchNorm, loss normalised by the GLOBAL class histogram, gradients SUMMED. Also the data-parallel confusion matrix:
    every rank updates StreamMetrics with its shard, the all-reduced matrix must equal the one computed over the whole
    batch bit for bit. Returns {"rel_grad", "rel_loss", "cm_equal", ...} on rank 0 (None elsewhere)."""
    import torch.distributed as dist
    from iswm_b200 import ops
    from iswm_b200.metrics import StreamMetrics
    from iswm_b200.network import modeling
    from iswm_b200.parallel import DataParallel
    from iswm_b200.utils.loss import CrossEntropyLoss
    Bs, H, W = 6, 128, 128
    g = torch.Generator().manual_seed(4242)
    x = torch.randn((world * Bs, 3, H, W), generator=g)
    y = torch.empty((world * Bs, H, W), dtype=torch.int64)
    for r in range(world):                               # foreground fraction 5 % .. 85 % across the shards
        fg = 0.05 + 0.8 * r / max(1, world - 1)
        yy = (torch.rand((Bs, H, W), generator=g) < fg).long()
        yy[torch.rand((Bs, H, W), generator=g) < 0.02] = 255
        y[r * Bs:(r + 1) * Bs] = yy
    w = torch.tensor([1.0, 4.0])

    def build():
        torch.manual_seed(1)
        m = modeling.deeplabv3plus_resnet50(num_classes=2, output_stride=16, pretrained_backbone=False).to(dev).train()
        m.engine().dropout_p = 0.0
        return m

    model = build()
    crit = CrossEntropyLoss(weight=w, ignore_index=255).to(dev)
    sm = StreamMetrics(2, device=dev)
    dp = DataParallel(model, crit, bucket_bytes=8 << 20, metrics=sm)
    xs, ys = x[rank * Bs:(rank + 1) * Bs].to(dev), y[rank * Bs:(rank + 1) * Bs].to(dev)
    loss = dp.train_step(xs, ys, optimizer=None)
    torch.cuda.synchronize()
    flat = model.engine().flat_g.clone()
    model.eval()
    with torch.no_grad():
        sm.update_cuda(ys, model(xs))                    # argmax predictions of this rank's shard
    cm = sm.confusion_matrix                             # all-reduce(SUM) of the int64 counters: every rank calls it
    out = None
    if rank == 0:
        hist = torch.zeros(2, dtype=torch.int64, device=dev)
        ops.class_hist(y.to(dev), 2, out=hist)
        ref_grad, num = None, 0.0
        ref_cm = StreamMetrics(2, device=dev)
        m2 = build()
        sd0 = {k: v.clone() for k, v in m2.state_dict().items()}
        for r in range(world):
            m2.load_state_dict(sd0)                      # every replica starts from the same parameters AND buffers
            m2.train()
            for p in m2.parameters():
                p.grad = None
            c2 = CrossEntropyLoss(weight=w, ignore_index=255).to(dev)
            c2.hist_hook = lambda h: h.copy_(hist)       # the global (all-reduced) histogram
            xr, yr = x[r * Bs:(r + 1) * Bs].to(dev), y[r * Bs:(r + 1) * Bs].to(dev)
            l2 = c2(m2(xr), yr)
            l2.backward()
            torch.cuda.synchronize()
            gr = m2.engine().flat_g.clone()
            ref_grad = gr if ref_grad is None else ref_grad + gr
            num += float(l2)
            m2.eval()
            with torch.no_grad():
                ref_cm.update_cuda(yr, m2(xr))
        rel = float((flat - ref_grad).norm() / ref_grad.norm())
        out = {"rel_grad": rel, "rel_loss": abs(float(loss) - num) / abs(num), "loss": float(loss), "ref_loss": num,
               "cm_equal": bool((cm == ref_cm.confusion_matrix).all()), "cm_total": float(cm.sum()),
               "buckets": len(dp.bucketer.bounds), "case": f"R50-OS16, {Bs} x {H}x{W} per rank, {world} ranks, fg 5-85 % per shard"}
    model.engine().grad_ready_hook = None
    dist.barrier()
    del dp, model
    torch.cuda.empty_cache()
    return out


def run_extras(dev):
    """Compact cfg5 / cfg4 results measured in the SAME process as the headline (so that the driver's own run times
    them): the three loss / metric kernels at 16x2x1024x1024 (median of 10 launches, L2 flushed between them) and the predict
    path at 8 x 2048x2048 (3 steps after 3 warm-ups)."""
    from iswm_b200 import ops
    from iswm_b200.metrics import StreamMetrics
    from iswm_b200.network import modeling
    from iswm_b200.predict import predict_mask
    pk = peaks()
    extra = {}
    B, H, W = 16, 1024, 1024
    g = torch.Generator().manual_seed(0)
    logits = torch.randn((B, 2, H, W), generator=g).to(dev)
    labels = (torch.rand((B, H, W), generator=g) < 0.02).long()
    labels[torch.rand((B, H, W), generator=g) < 0.01] = 255
    labels = labels.to(dev)
    wts = torch.tensor([1.0, 7.0], device=dev)
    N = B * H * W
    hist = ops.class_hist(labels, 2)
    cm = torch.zeros(5, dtype=torch.int64, device=dev)
    fns = {"class_hist": (lambda: ops.class_hist(labels, 2, out=hist), N * 8),
           "wce_fwd_bwd": (lambda: ops.wce_fwd_bwd(logits, labels, wts, hist), 2 * N * 2 * 4 + N * 8),
           "argmax_confusion": (lambda: ops.argmax_confusion(logits, labels, mode=1, threshold=0.5, out=cm), N * 2 * 4 + N * 8)}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    k5 = {}
    for name, (fn, nbytes) in fns.items():
        for _ in range(3):
            fn()
        ts = []
        for _ in range(10):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        us = ts[len(ts) // 2] * 1e3
        k5[name] = {"us": us, "algorithmic_bytes": nbytes, "frac_of_hbm_peak": nbytes / (us * 1e-6) / 1e9 / pk["hbm_gbs"],
                    "traffic": traffic_from_profiles("cfg5:" + name)}
    extra["cfg5"] = {"workload": "16x2x1024x1024 fp32 logits, int64 labels; median of 10 launches, 256 MB L2 flush between", "kernels": k5}
    del logits, labels, flush
    torch.cuda.empty_cache()
    torch.manual_seed(0)
    model = modeling.deeplabv3plus_resnet50(num_classes=2, output_stride=16, pretrained_backbone=False).to(dev).eval()
    metrics = StreamMetrics(2, device=dev)
    x, y = synth_batch(8, 2048, 2048, 0, device=dev)
    for _ in range(3):
        predict_mask(model, x, 0.5, y, metrics, fused=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        predict_mask(model, x, 0.5, y, metrics, fused=True)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 3
    extra["cfg4"] = {"workload": "predict path, R50-OS16 eval, 8 x 2048x2048, fused upsample+softmax+threshold+confusion; 3 steps after 3 warm-ups",
                     "img_per_s": 8 / (ms * 1e-3), "ms_per_step": ms,
                     "whole_step_tensor_frac": FWD_GFLOP_PER_IMG[("resnet50", 16, 2048)] * 8e9 / (ms * 1e-3) / 1e12 / pk.get("bf16_tflops_sustained", 1400.0)}
    del model, x, y
    torch.cuda.empty_cache()
    extra["next_rows"] = run_next_rows(dev, pk)
    return extra


def run_e2e_u8(model, crit, opt, dev, B, H, W, steps):
    """The same train step fed the way SURVEY 8f rank 2 intends: the host ships uint8 HWC tiles and uint8 labels from pinned memory
    (1/4 and 1/8 of the fp32 / int64 bytes of the headline e2e), `DeviceTransform` (flip + ToTensor + Normalize on the device, straight
    into the captured step's input buffer) precedes one graph replay per step, every step's loss is read back on the host."""
    from iswm_b200.data import DeviceTransform, HostBatchPrefetcher
    from iswm_b200.graphs import GraphedTrainStep
    from iswm_b200.train_utils import DeferredLoss
    from iswm_b200 import ops
    g = torch.Generator().manual_seed(123)
    tiles = torch.randint(0, 256, (B, H, W, 3), generator=g, dtype=torch.uint8).pin_memory()
    lab = (torch.rand((B, H, W), generator=g) < 0.02).to(torch.uint8)
    lab[torch.rand((B, H, W), generator=g) < 0.01] = 255
    lab = lab.pin_memory()
    tf = DeviceTransform(crop_size=(H, W), hflip=True, generator=torch.Generator().manual_seed(5))
    stepper = GraphedTrainStep(model, crit, opt)
    x0, y0 = tf(tiles.to(dev), lab.to(dev))
    stepper(x0, y0)                                      # capture for uint8 labels
    torch.cuda.synchronize()

    def run(n):
        pre = HostBatchPrefetcher(((tiles, lab) for _ in range(n)), dev, image_dtype=torch.uint8)
        dl = DeferredLoss()
        for xs, ys in pre:
            org, flip = tf.draw(B, H, W)
            flip_d = flip.to(dev, non_blocking=True)
            ops.u8_to_f32_norm(xs, tf.mean, tf.std, (H, W), None, flip_d, out=stepper.images)     # no staging copy: the graph reads this buffer
            ops.crop_flip_u8(ys, (H, W), None, flip_d, out=stepper.labels)
            dl.push(stepper(stepper.images, stepper.labels))
        return dl.flush()

    run(3)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    last = run(steps)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    del stepper
    return {"workload": "cfg2 train step from uint8 HWC tiles + uint8 labels in pinned host memory: H2D, flip + ToTensor + Normalize on the device (DeviceTransform kernels writing the captured step's input buffers), one graph replay, loss read back",
            "value": B * steps / (ms * 1e-3), "unit": "img/s", "ms_per_step": ms / steps, "h2d_bytes_per_step": tiles.numel() + lab.numel(), "d2h_bytes_per_step": 4,
            "loss": float(last)}


def run_next_rows(dev, pk):
    """The rows either side of the hot path (SURVEY 8f), timed in the driver's own run at cfg2's geometry: the device train
    transform (uint8 tiles -> scaled / cropped / flipped / normalised fp32 batch), the fused train tail against the unfused kernel
    chain, and the image half of the per-frame evaluators. Median of 10 launches, L2 flushed between them."""
    from iswm_b200 import _lib, ops
    from iswm_b200.data import DeviceTransform
    out = {}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def med_us(fn, reps=10):
        for _ in range(2):
            fn()
        ts = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts.sort()
        return ts[len(ts) // 2] * 1e3

    g = torch.Generator().manual_seed(0)
    B, S = 16, 512
    tiles = torch.randint(0, 256, (B, S, S, 3), generator=g, dtype=torch.uint8).to(dev)
    lbl8 = (torch.rand((B, S, S), generator=g) < 0.05).to(torch.uint8).to(dev)
    tf = DeviceTransform(crop_size=S, hflip=True, scale_range=(0.5, 2.0), pad_if_needed=True, generator=torch.Generator().manual_seed(1))
    geom = tf.draw_scaled(B, S, S)
    us = med_us(lambda: tf(tiles, lbl8, params=geom))
    nbytes = B * S * S * (3 * 4 + 1)                      # fp32 image + uint8 label written; the uint8 taps come through L1 / L2
    out["device_transform"] = {"workload": f"ExtRandomScale(0.5-2) + RandomCrop(pad) + flip + ToTensor + Normalize, {B} x {S}x{S} uint8 tiles, 3 launches",
                               "us": us, "img_per_s": B / (us * 1e-6), "written_GB/s": nbytes / (us * 1e-6) / 1e9}
    # fused tail vs the unfused chain (cfg2: 16 x 128x128 low-res logits, int64 labels)
    h = S // 4
    lo = torch.randn((B, h, h, 2), generator=g).to(dev)
    y = (torch.rand((B, S, S), generator=g) < 0.05).long().to(dev)
    wts = torch.tensor([1.0, 7.0], device=dev)
    L = _lib.lib()
    st = lambda: torch.cuda.current_stream().cuda_stream   # noqa: E731
    logits = torch.empty((B, 2, S, S), dtype=torch.float32, device=dev)
    dlo = torch.empty((B, h, h, 8), dtype=torch.bfloat16, device=dev)
    bias = torch.zeros(2, dtype=torch.float32, device=dev)
    scratch = torch.zeros(8200, dtype=torch.uint8, device=dev)

    def unfused():
        _lib.check(L.iswm_logits_up_fwd(lo.data_ptr(), B, h, h, 2, S, S, logits.data_ptr(), st()))
        hist = ops.class_hist(y, 2)
        _, grad = ops.wce_fwd_bwd(logits, y, wts, hist, 255, 1.0, True)
        _lib.check(L.iswm_logits_up_bwd(grad.data_ptr(), B, h, h, 2, S, S, dlo.data_ptr(), 8, bias.data_ptr(), st()))

    def fused():
        acc, hist, num = ops.tail_fwd(lo, y, wts, 255)
        ops.tail_loss(num, wts, hist, 255)
        ops.tail_bwd(acc, wts, hist, 255, None, dlo, bias, scratch)

    uu, fu = med_us(unfused), med_us(fused)
    alg = B * S * S * 8 + 3 * B * h * h * 8 + B * h * h * 16
    out["train_tail"] = {"workload": f"x4 upsample + weighted CE + backward to the classifier output, {B} x {S}x{S}, int64 labels",
                         "unfused_us": uu, "fused_us": fu, "fused_algorithmic_bytes": alg,
                         "fused_frac_of_hbm_peak": alg / (fu * 1e-6) / 1e9 / pk["hbm_gbs"]}
    masks = (torch.rand((8, S, S), generator=g) < 0.02).to(torch.uint8)
    masks[:, 100:400, 200:260] = 1
    masks = masks.to(dev)
    out["shape_metrics"] = {"workload": f"MaskUtils.preprocess_mask image half (close, open, 8-connected components, largest region, fronts), 8 x {S}x{S} masks, 8 launches",
                            "us": med_us(lambda: ops.mask_preprocess(masks)),
                            "region_us": med_us(lambda: ops.region_components(masks, masks))}
    del flush
    torch.cuda.empty_cache()
    return out


# ----------------------------------------------------------------------------- GPU arm
def run_ours(args):
    import torch.distributed as dist
    from iswm_b200 import _lib
    from iswm_b200.network import modeling
    from iswm_b200.optim import FusedSGD
    from iswm_b200.utils.loss import CrossEntropyLoss

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: iswm_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=180))
    if args.workload == "predict":
        return run_predict(args, dev, world, rank, local)
    if args.workload == "lossmetric":
        return run_lossmetric(args, dev, world, rank, local)
    B, H, W = args.batch, args.size, args.size
    dp_parity = dp_parity_check(dev, world, rank) if (world > 1 and not args.no_dp_parity) else None
    torch.manual_seed(0)
    ctor = modeling.deeplabv3plus_resnet50 if args.backbone == "resnet50" else modeling.deeplabv3plus_resnet101
    model = ctor(num_classes=2, output_stride=args.output_stride, pretrained_backbone=False).to(dev).train()
    crit = CrossEntropyLoss(weight=torch.tensor([1.0, 7.0]), ignore_index=255).to(dev)      # [1, sqrt(0.98/0.02)]
    opt = FusedSGD(model, lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)
    dp = None
    if world > 1:
        from iswm_b200.parallel import DataParallel
        dp = DataParallel(model, crit)
    x_dev, y_dev = synth_batch(B, H, W, rank, device=dev)
    x_host, y_host = synth_batch(B, H, W, rank, pinned=True)
    # host labels in the form the reference's loader yields them: uint8 (ExtToTensor(target_type='uint8'), utils/ext_transforms.py:273-293);
    # train.py:1040 widens them with labels.to(device, dtype=torch.long) - here the widening happens on the device, in the copy into the
    # captured step's int64 label buffer
    y_host = y_host.to(torch.uint8).pin_memory()

    def dump_step(loss):
        # --dump-outputs: what the run's SECOND step returned (the loss) and left in the model: parameters after the update, their
        # gradients, the BatchNorm buffers. It is a steady-state step (in graph mode a plain replay: operands packed by the previous
        # step's optimiser kernel, momentum carried over) and still reproducible: weight gradients are summed with fp32 atomics in no
        # fixed order, and from the third step on BatchNorm amplifies those last bits far beyond rounding, so the run's last
        # step is not (DESIGN.md, "A multi-step RUN"; measured at cfg2 by tools/steps_divergence_probe.py).
        if args.dump_outputs and rank == 0:
            params = list(model.parameters())
            dump_outputs(args.dump_outputs, {
                "loss": loss, "params": dump_sample(torch.cat([p.detach().reshape(-1) for p in params])),
                "grads": dump_sample(torch.cat([p.grad.reshape(-1) for p in params])),
                "buffers": torch.cat([b.reshape(-1).float() for b in model.buffers()])})

    # the step is captured once and replayed as ONE CUDA graph launch (iswm_b200.graphs.GraphedTrainStep, the recommended
    # API; ISWM_BENCH_GRAPH=0 times the eager ~430-launch step instead). Data-parallel steps are captured too when the
    # peer-memory transport is up (every exchange is a plain kernel); on the torch.distributed transport they stay eager.
    use_graph = os.environ.get("ISWM_BENCH_GRAPH", "1") != "0" and (world == 1 or dp.comm_mode == "peer")
    stepper = None
    if use_graph:
        from iswm_b200.graphs import GraphedTrainStep
        try:
            stepper = GraphedTrainStep(model, crit, opt, dp=dp)
            stepper(x_dev, y_dev)           # capture now (its warm-up state is restored; then one real step)
            torch.cuda.synchronize()
        except Exception as e:              # never lose the measurement to the launch mode: fall back to eager launches
            print(f"[bench] CUDA graph capture failed ({e!r}); timing the eager step instead", file=sys.stderr)
            stepper = None
        if world > 1:                       # every rank must take the same path (a rank replaying against ranks launching eagerly would deadlock)
            okf = torch.tensor([1 if stepper is not None else 0], device=dev)
            dist.all_reduce(okf, op=dist.ReduceOp.MIN)
            if int(okf) == 0:
                stepper = None
    if stepper is not None:
        # device-resident inputs live in the graph's own static input buffers (what a loader that writes its batches there does,
        # iswm_b200.graphs): the timed region of "value" holds no device-to-device staging copy; "e2e" below still stages every
        # batch host -> prefetch buffer -> static buffer
        x_dev, y_dev = stepper.images, stepper.labels
    eager_only = [False]
    from iswm_b200.graphs import _fused_tail_default
    fused_tail = _fused_tail_default()

    def step(x, y):
        if stepper is not None and not eager_only[0]:
            return stepper(x, y)
        if dp is not None:
            return dp.train_step(x, y, opt)
        if fused_tail:                      # the same tail kernels as the captured step (model.forward_loss)
            loss = model.forward_loss(x, y, crit)
        else:
            logits = model(x)
            loss = crit(logits, y)
        opt.zero_grad()
        loss.backward()
        opt.step()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # nvidia-smi takes a while to attach: start it before the warm-up so that it is sampling (every 100 ms) by the
    # time the timed region begins; it is stopped and reaped before the e2e region
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    done = 0 if stepper is None else 1      # the capture call above ran the first step (capture-time warm-up state restored)
    for _ in range(args.warmup):            # at least 3
        loss = step(x_dev, y_dev)
        done += 1
        if done == 2:
            dump_step(loss)
    barrier()
    if rank == 0:
        sampler.wait_first_sample(5.0)
    # ---- timed region 1: device-resident inputs ("value")
    launches0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    w0 = time.time()
    e0.record()
    for _ in range(args.steps):
        loss = step(x_dev, y_dev)
    e1.record()
    barrier()
    w1 = time.time()
    launches = _lib.launch_count() - launches0
    if stepper is not None:
        launches += args.steps * stepper.launches_per_replay      # kernels inside the replayed graph (counted at capture)
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop(w0, w1) if rank == 0 else None
    # ---- timed region 2: end to end through the public API with HOST buffers ("e2e"): every step's images and
    # labels come from pinned host memory (staged by iswm_b200.data.HostBatchPrefetcher: the copy of batch i+1
    # runs on a side stream under step i) and every step's loss is read back to the host before the next step
    from iswm_b200.data import HostBatchPrefetcher
    pre = HostBatchPrefetcher([(x_host, y_host)] * 2, dev)
    for xs, ys in pre:                                  # untimed warm-up of the staging path (allocates its two buffers)
        step(xs, ys)
    pre.loader = ((x_host, y_host) for _ in range(args.steps))
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    last = 0.0
    from iswm_b200.train_utils import DeferredLoss
    dl = DeferredLoss()                                 # every step's loss is copied device -> host (pinned, async) and
    for xs, ys in pre:                                  # read on the host while the NEXT step is already enqueued
        v = dl.push(step(xs, ys))
        if v is not None:
            last = v
    last = dl.flush()                                   # the final step's loss: inside the timed region
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    if world > 1:
        t = torch.tensor([ms, ms_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_e2e = float(t[0]), float(t[1])
    # ---- roofline of the dominant kernel: one extra instrumented step (CUDA events around every launch)
    roof = None
    # EVERY rank runs the instrumented step (it contains the data-parallel collectives); only rank 0 records events
    eng = model.engine()
    if rank == 0:
        eng.profile = []
    # per-kernel durations are taken with the weight-gradient stream folded back in line: when wgrad kernels share
    # the SMs with the kernel being timed, its CUDA events measure the contention, not the kernel
    async_wgrad = eng.async_wgrad
    eng.async_wgrad = False
    eager_only[0] = True                    # per-kernel events need the eager launch path
    if stepper is not None:
        step(x_dev, y_dev)                  # untimed: the eager path's activations come from cudaMalloc the first time
        barrier()
        if rank == 0:
            eng.profile = []                # drop that step's records
    host_head_start()
    step(x_dev, y_dev)
    barrier()
    eng.async_wgrad = async_wgrad
    if rank == 0 and world == 1 and args.profile_detail:     # (single process only: the extra step has no partner ranks)
        saved = eng.profile
        eng.profile = None
        eng.async_wgrad = False
        profile_by_entry(lambda: step(x_dev, y_dev), args.profile_detail + ".by_entry")
        eng.async_wgrad = async_wgrad
        eng.profile = saved
    if rank == 0:
        agg = {}
        detail = []
        for k, fl, a, b, tag in eng.profile:
            t_, f_, n_ = agg.get(k, (0.0, 0.0, 0))
            dt = a.elapsed_time(b)
            agg[k] = (t_ + dt, f_ + fl, n_ + 1)
            detail.append((tag, fl, dt))
        if args.profile_detail:
            with open(args.profile_detail, "w") as f:
                for tag, fl, dt in detail:
                    if tag.startswith("bn_"):      # HBM-bound entries carry algorithmic bytes
                        f.write(f"{tag:55s} {fl / 1e6:10.2f} MB {dt * 1e3:9.1f} us {fl / (dt * 1e-3) / 1e9:8.1f} GB/s\n")
                    else:
                        f.write(f"{tag:55s} {fl / 1e9:10.2f} GF {dt * 1e3:9.1f} us {fl / (dt * 1e-3) / 1e12:8.1f} TF/s\n")
        eng.profile = None
        pk = peaks()
        peak_tf = pk.get("bf16_tflops_sustained", pk["bf16_tflops"])
        k = "conv_igemm"
        t_ms, fl, n = agg[k]
        ach = fl / (t_ms * 1e-3) / 1e12
        roof = {"bound": "tensor", "kernel": "conv_igemm_kernel (forward + data-gradient implicit GEMMs)",
                "achieved": ach, "peak": peak_tf, "unit": "TFLOP/s", "frac": ach / peak_tf, "traffic": traffic_from_profiles("conv_igemm_kernel"),
                "launches_per_step": n, "kernel_ms_per_step": t_ms, "peak_source": pk["_source"] + " bf16_tflops_sustained (kernel timed inside a long step; the instrumented step runs the weight-gradient stream in line so that events time the kernel alone)",
                "other_kernels": {kk: ({"ms_per_step": v[0], "GB/s": v[1] / (v[0] * 1e-3) / 1e9, "frac_of_hbm_peak": v[1] / (v[0] * 1e-3) / 1e9 / pk["hbm_gbs"], "launches": v[2]}
                                       if kk.startswith("hbm:") else
                                       {"ms_per_step": v[0], "TFLOP/s": v[1] / (v[0] * 1e-3) / 1e12, "launches": v[2]}) for kk, v in agg.items() if kk != k}}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    imgs = B * world * args.steps
    value = imgs / (ms * 1e-3)
    e2e_value = imgs / (ms_e2e * 1e-3)
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        rate, per, n = cpu_train_step_rate(2, min(H, 512), min(W, 512), 2, 1)
        cpu = {"value": rate, "unit": "img/s", "cores": n, "kind": "port",
               "sample": f"1 warm-up + 2 timed steps of batch 2, {H}x{W}, R50-OS16 fwd+CE+bwd+SGD, fp32 torch oracle on the host"}
    gflop = TRAIN_GFLOP_PER_IMG.get((args.backbone, args.output_stride, H))
    extra = None
    launch_mode = "one CUDA graph replay per step (GraphedTrainStep)" if stepper is not None else "eager launches"
    if world == 1 and not args.no_extras and (args.backbone, args.output_stride, H, B) == ("resnet50", 16, 512, 16):
        e2e_u8 = None
        try:
            e2e_u8 = run_e2e_u8(model, crit, opt, dev, B, H, W, args.steps)
        except Exception as e:
            e2e_u8 = {"error": repr(e)}
        del model, opt, stepper, x_dev, y_dev
        torch.cuda.empty_cache()
        try:
            extra = run_extras(dev)
        except Exception as e:                           # the headline must survive a failure of the side measurements
            extra = {"error": repr(e)}
        extra["e2e_u8"] = e2e_u8
    line = {
        "metric": f"train img/s DeepLabV3+ {'R50' if args.backbone == 'resnet50' else 'R101'} {H}^2", "value": value, "unit": "img/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "bf16", "data": "synthetic",
        "config": {"workload": train_workload_name(args.backbone, args.output_stride, H, W, B),
                   "parallelism": f"dp{world}", "global_batch": B * world,
                   "launch": launch_mode,
                   "comm": None if dp is None else ("peer-memory kernels over NVLink (iswm_b200.peer): histogram / gradient buckets / loss, captured in the graph"
                                                    if dp.comm_mode == "peer" else "torch.distributed NCCL collectives"),
                   "l2": "no explicit flush: each step streams > 2 GB of activations (>> 126 MB L2)",
                   "e2e_note": "per step: fp32 images + uint8 labels (what the reference's loader yields; widened to int64 on the device as train.py:1040 does) H2D from pinned memory (HostBatchPrefetcher, copy of batch i+1 under step i) and the loss D2H (DeferredLoss: read on the host one step later, last one before the timer stops)",
                   "whole_step_tensor_frac": (gflop * 1e9 * B * world * args.steps / (ms * 1e-3) / 1e12 / world / peaks().get("bf16_tflops_sustained", 1400.0)) if gflop else None,
                   "loss": last, "dp_parity": dp_parity, "extra": extra},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "img/s", "h2d_bytes_per_step": (x_host.numel() * 4 + y_host.numel() * y_host.element_size()) * world, "d2h_bytes_per_step": 4 * world,
                "ms_per_step": ms_e2e / args.steps},
        "gpu_launches": int(launches),
        "roofline": roof,
        "cpu_baseline": cpu,
    }
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def main():
    sys.dont_write_bytecode = True      # the package is imported below this point: a run leaves no __pycache__ in the tree
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="train", choices=["train", "predict", "lossmetric"],
                    help="train = cfg2 (the headline; cfg3 with --backbone resnet101 --output-stride 8 --size 1024 --batch 4); "
                         "predict = cfg4 (R50 eval forward + threshold + confusion matrix); lossmetric = cfg5 microbench")
    ap.add_argument("--backbone", default="resnet50", choices=["resnet50", "resnet101"])
    ap.add_argument("--output-stride", type=int, default=16, choices=[8, 16])
    ap.add_argument("--batch", type=int, default=0, help="per-GPU batch (default: 16 train, 8 predict, 16 lossmetric)")
    ap.add_argument("--size", type=int, default=0, help="tile edge (default: 512 train, 2048 predict, 1024 lossmetric)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="N=1 cfg2 only: skip the compact cfg5 / cfg4 side measurements (config.extra)")
    ap.add_argument("--no-dp-parity", action="store_true", help="N>1 only: skip the multi-rank parity step before the timed region (config.dp_parity)")
    ap.add_argument("--profile-detail", default="", help="write the per-launch table of the instrumented step here")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write what the timed step function computed as DIR/<name>.npy (float32 / float64, a fixed seeded sample of any "
                         "output over 4 Mi elements): train, its second step from the seeded weights; predict and lossmetric, the last "
                         "timed step. Inputs are seeded, so two runs or two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs dumps the CUDA path (--impl ours)")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    args.batch = args.batch or {"train": 16, "predict": 8, "lossmetric": 16}[args.workload]
    args.size = args.size or {"train": 512, "predict": 2048, "lossmetric": 1024}[args.workload]
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
