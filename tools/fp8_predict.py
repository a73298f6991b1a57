"""bf16 against FP8 (iswm_b200.quant) predict step at cfg4 (R50-OS16, 8 x 2048^2, predict_mask fused with the confusion
counts), alternating in one process, device-event timed after warm-up. Also: per-convolution kernel times of both paths
(per-launch events), the FP8 convolutions' achieved TFLOP/s against the data-sheet dense FP8 figure and against a large-GEMM
ceiling measured here with the same kernel, and the card's name and power limit.

    python tools/fp8_predict.py [--batch 8 --size 2048 --rounds 3 --steps 10] [--out FILE.json]
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from iswm_b200 import _lib, ops  # noqa: E402
from iswm_b200.metrics.stream_metrics import StreamMetrics  # noqa: E402
from iswm_b200.network import modeling  # noqa: E402
from iswm_b200.predict import predict_mask  # noqa: E402
from iswm_b200.quant import quantize_fp8  # noqa: E402
from oracle.gen_golden import seeded_state_dict  # noqa: E402

DATASHEET_FP8_DENSE_TFLOPS = 4500.0       # NVIDIA HGX B200 data sheet, one GPU, dense, 1000 W (a data-sheet number, not a measurement)


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:            # noqa: BLE001
        return f"unknown ({e})"


def timed(fn, steps):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / steps


def per_conv(eng, fn):
    eng.profile = []
    fn()
    torch.cuda.synchronize()
    rows = {}
    for kernel, flops, e0, e1, tag in eng.profile:
        if kernel.startswith("conv_igemm"):
            r = rows.setdefault(tag, [kernel, 0.0, 0.0])
            r[1] += e0.elapsed_time(e1)
            r[2] += flops
    eng.profile = None
    return rows


def gemm_ceiling(f8: bool, M=128 * 148 * 4, K=1024, N=256, reps=50):
    """One 1x1 convolution as a plain GEMM (operands in L2): the kernel's own compute ceiling."""
    dt = torch.float8_e4m3fn if f8 else torch.bfloat16
    x = torch.randn(M, K, device="cuda").to(dt)
    kp = K if not f8 else (K + 127) // 128 * 128
    w = torch.randn(N * kp, device="cuda").to(dt)
    out = torch.empty(M, N, dtype=dt, device="cuda")
    sc, sh = torch.ones(N, device="cuda"), torch.zeros(N, device="cuda")
    d = ops.make_conv_desc(1, 1, M, K, K, 1, 1, M, N, N, ops.conv_taps(1, 1), _lib.EPI_AFFINE)
    st = torch.cuda.current_stream().cuda_stream
    L = _lib.lib()
    if f8:
        fn = lambda: _lib.check(L.iswm_conv_igemm_f8(C.byref(d), x.data_ptr(), w.data_ptr(), out.data_ptr(), sc.data_ptr(), sh.data_ptr(), None, 1.0, _lib.E4M3, st))
    else:
        fn = lambda: _lib.check(L.iswm_conv_igemm(C.byref(d), x.data_ptr(), w.data_ptr(), out.data_ptr(), sc.data_ptr(), sh.data_ptr(), None, None, st))
    for _ in range(5):
        fn()
    ms = timed(fn, reps)
    return 2.0 * M * K * N / (ms * 1e-3) / 1e12


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--size", type=int, default=2048)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fp8_predict.py measures on a GPU; none is available")
    dev = torch.device("cuda:0")
    m = modeling.deeplabv3plus_resnet50(num_classes=2, output_stride=16, pretrained_backbone=False)
    m.load_state_dict(seeded_state_dict(m.state_dict(), 1234))
    m.to(dev).eval()
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(a.batch, 3, a.size, a.size, device=dev, generator=g)
    y = (torch.rand(a.batch, a.size, a.size, device=dev, generator=g) < 0.1).long()
    qm = quantize_fp8(m, x)
    met = StreamMetrics(2, device=dev, shape_metrics=False)
    paths = {"bf16": m, "fp8": qm}
    fns = {k: (lambda net=v: predict_mask(net, x, 0.5, y, met)) for k, v in paths.items()}
    res = {"card (name, power limit, max SM clock)": card(), "batch": a.batch, "size": a.size, "steps": a.steps, "rounds": {}}
    with torch.no_grad():
        for k in fns:
            for _ in range(a.warmup):
                fns[k]()
        torch.cuda.synchronize()
        for r in range(a.rounds):
            for k in fns:
                ms = timed(fns[k], a.steps)
                res["rounds"].setdefault(k, []).append({"ms_per_step": ms, "img_per_s": a.batch * 1e3 / ms})
        best = {k: max(v["img_per_s"] for v in res["rounds"][k]) for k in fns}
        res["img_per_s_best"] = best
        res["fp8_over_bf16"] = best["fp8"] / best["bf16"]
        eng = m.engine()
        rb = per_conv(eng, lambda: m.forward_lowres(x))
        rf = per_conv(eng, lambda: qm.forward_lowres(x))
    shapes = []
    for tag in rf:
        kb, msb, flb = rb.get(tag, ["-", float("nan"), 0.0])
        _, msf, flf = rf[tag]
        shapes.append({"conv": tag, "bf16_ms": msb, "fp8_ms": msf, "fp8_tflops": flf / (msf * 1e-3) / 1e12})
    res["per_conv"] = shapes
    tot_f, tot_ms = sum(v[2] for v in rf.values()), sum(v[1] for v in rf.values())
    res["fp8_convs_total_ms"] = tot_ms
    res["bf16_convs_total_ms"] = sum(v[1] for v in rb.values())
    res["fp8_convs_tflops"] = tot_f / (tot_ms * 1e-3) / 1e12
    res["gemm_ceiling_tflops"] = {"fp8": gemm_ceiling(True), "bf16": gemm_ceiling(False)}
    res["fp8_convs_share_of_datasheet_fp8"] = res["fp8_convs_tflops"] / DATASHEET_FP8_DENSE_TFLOPS
    res["fp8_convs_share_of_measured_ceiling"] = res["fp8_convs_tflops"] / res["gemm_ceiling_tflops"]["fp8"]
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt)


if __name__ == "__main__":
    main()
