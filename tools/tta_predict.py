"""Test-time augmentation cost of the predict step at cfg4 (R50-OS16, 8 x 2048^2, predict_mask fused with the confusion
counts), in bf16 and FP8 (iswm_b200.quant), for the view sets {1.0}, {1.0} x flip and {0.75, 1.0, 1.25} x flip.

- img/s per view set: device events around whole predict_mask calls after warm-up, the paths alternating in rounds.
- The share of the step outside the network forwards: the same step with the resize launches and the epilogue replaced
  by no-ops (the forwards then read unwritten inputs; their cost does not depend on the values), timed in the same
  rounds; share = (full - forwards only) / full. Also the sum of those kernels' own times, replayed in isolation.
- The multi-view epilogue's kernel time over many launches for all 8 images at once, and the bytes it must move
  (every view's low-resolution logits, the int64 labels, the two uint8 maps) over that time, against the 7.7 TB/s of
  the data sheet. The low-resolution logits (about 26 MB per view at s = 1.25) may be served from L2.
- The card's name and power limit, read in the same run.

    python tools/tta_predict.py [--batch 8 --size 2048 --rounds 3 --steps 5] [--out FILE.json]
"""
import argparse
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from iswm_b200 import ops, predict  # noqa: E402
from iswm_b200.metrics.stream_metrics import StreamMetrics  # noqa: E402
from iswm_b200.network import modeling  # noqa: E402
from iswm_b200.quant import quantize_fp8  # noqa: E402
from oracle.gen_golden import seeded_state_dict  # noqa: E402

DATASHEET_HBM_TBPS = 7.7          # NVIDIA HGX B200 data sheet, one GPU (a data-sheet number, not a measurement)
VIEW_SETS = {"1.0": ((1.0,), False), "1.0xflip": ((1.0,), True), "0.75,1.0,1.25xflip": ((0.75, 1.0, 1.25), True)}


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


class Recorder:
    """Replaces the TTA kernels' wrappers for one call: records their arguments, and runs them only when `run`."""

    def __init__(self, run):
        self.run, self.calls = run, []
        self.real = (ops.resize_flip_f32, ops.predict_tta_epilogue)

    def resize(self, x, size, flip=False, out=None):
        if out is None:
            out = torch.empty((x.shape[0], x.shape[1]) + tuple(size), dtype=torch.float32, device=x.device)
        self.calls.append(("resize", (x, size, flip, out)))
        return self.real[0](x, size, flip, out=out) if self.run else out

    def epilogue(self, views, H, W, true=None, **kw):
        self.calls.append(("epilogue", (views, H, W, true, kw)))
        if self.run:
            return self.real[1](views, H, W, true, **kw)
        return kw.get("out"), kw.get("pred"), kw.get("conf")

    def __enter__(self):
        ops.resize_flip_f32, ops.predict_tta_epilogue = self.resize, self.epilogue
        return self

    def __exit__(self, *exc):
        ops.resize_flip_f32, ops.predict_tta_epilogue = self.real


def replay_ms(calls, reps):
    """Summed kernel time of the recorded resize / epilogue calls, each replayed `reps` times in isolation."""
    total = 0.0
    for kind, args in calls:
        if kind == "resize":
            x, size, flip, out = args
            fn = lambda: ops.resize_flip_f32(x, size, flip, out=out)
        else:
            views, H, W, true, kw = args
            kw = dict(kw, out=torch.zeros(5, dtype=torch.int64, device=true.device))
            fn = lambda: ops.predict_tta_epilogue(views, H, W, true, **kw)
        fn()
        total += timed(fn, reps)
    return total


def epilogue_rate(B, H, W, y, reps):
    """All views of the three-scale flip set at once, on random low-resolution logits of the engine's shapes."""
    views = []
    for s in VIEW_SETS["0.75,1.0,1.25xflip"][0]:
        Hs, Ws = (H, W) if s == 1.0 else (int(H * s + 0.5), int(W * s + 0.5))
        h, w = ((Hs + 1) // 2 + 1) // 2, ((Ws + 1) // 2 + 1) // 2
        lo = torch.randn((B, h, w, 2), device=y.device)
        views += [(lo, (Hs, Ws), False), (lo, (Hs, Ws), True)]
    pred = torch.empty((B, H, W), dtype=torch.uint8, device=y.device)
    conf = torch.empty_like(pred)
    cm = torch.zeros(5, dtype=torch.int64, device=y.device)
    fn = lambda: ops.predict_tta_epilogue(views, H, W, y, mode=1, threshold=0.5, out=cm, pred=pred, conf=conf)
    for _ in range(3):
        fn()
    ms = timed(fn, reps)
    nbytes = sum(v[0].numel() * 4 for v in views) + y.numel() * y.element_size() + 2 * pred.numel()
    return {"views": len(views), "ms": ms, "bytes": nbytes, "tb_per_s": nbytes / (ms * 1e-3) / 1e12,
            "share_of_datasheet_hbm": nbytes / (ms * 1e-3) / 1e12 / DATASHEET_HBM_TBPS}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--size", type=int, default=2048)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("tta_predict.py measures on a GPU; none is available")
    dev = torch.device("cuda:0")
    m = modeling.deeplabv3plus_resnet50(num_classes=2, output_stride=16, pretrained_backbone=False)
    m.load_state_dict(seeded_state_dict(m.state_dict(), 1234))
    m.to(dev).eval()
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(a.batch, 3, a.size, a.size, device=dev, generator=g)
    y = (torch.rand(a.batch, a.size, a.size, device=dev, generator=g) < 0.1).long()
    qm = quantize_fp8(m, x)
    met = StreamMetrics(2, device=dev, shape_metrics=False)
    res = {"card (name, power limit, max SM clock)": card(), "batch": a.batch, "size": a.size, "steps": a.steps,
           "max_forward_pixels": predict.MAX_FORWARD_PIXELS, "rounds": {}}
    fns = {}
    for pname, net in (("bf16", m), ("fp8", qm)):
        for vname, (scales, flip) in VIEW_SETS.items():
            fns[f"{pname} {vname}"] = (lambda net=net, scales=scales, flip=flip:
                                       predict.predict_mask(net, x, 0.5, y, met, scales=scales, flip=flip))
    with torch.no_grad():
        for k, fn in fns.items():
            for _ in range(a.warmup):
                fn()
            if "flip" in k:
                with Recorder(run=False):
                    fn()
        torch.cuda.synchronize()
        for _ in range(a.rounds):
            for k, fn in fns.items():
                ms = timed(fn, a.steps)
                row = {"ms_per_step": ms, "img_per_s": a.batch * 1e3 / ms}
                if "flip" in k:
                    with Recorder(run=False):
                        row["forwards_only_ms"] = timed(fn, a.steps)
                res["rounds"].setdefault(k, []).append(row)
        summary = {}
        for k, fn in fns.items():
            rows = res["rounds"][k]
            best = min(rows, key=lambda r: r["ms_per_step"])
            s = {"img_per_s_best": best["img_per_s"], "ms_per_step_best": best["ms_per_step"]}
            if "flip" in k:
                fwd = min(r["forwards_only_ms"] for r in rows)
                s["forwards_only_ms_best"] = fwd
                s["non_forward_share_of_step"] = (best["ms_per_step"] - fwd) / best["ms_per_step"]
                with Recorder(run=True) as rec:
                    fn()
                s["resize_launches"] = sum(1 for c in rec.calls if c[0] == "resize")
                s["epilogue_launches"] = sum(1 for c in rec.calls if c[0] == "epilogue")
                s["resize_plus_epilogue_kernel_ms"] = replay_ms(rec.calls, a.reps)
                s["resize_plus_epilogue_kernel_share"] = s["resize_plus_epilogue_kernel_ms"] / best["ms_per_step"]
            summary[k] = s
        res["summary"] = summary
        res["epilogue_three_scales_flip"] = epilogue_rate(a.batch, a.size, a.size, y, a.reps)
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt)


if __name__ == "__main__":
    main()
