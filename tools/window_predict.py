"""Sliding-window cost of the predict step at cfg4 (R50-OS16, 8 x 2048^2, predict_mask fused with the confusion counts), in
bf16 and FP8 (iswm_b200.quant), for the whole image and windows 512 / stride 384 and 256 / stride 192; one large scene;
and, with --usefulness, whole-image against windowed prediction on a short-trained synthetic task.

- img/s and ms per batch: device events around whole predict_mask calls after warm-up, the paths alternating in rounds.
- The share of the step outside the network forwards (gather + logit copies + epilogue): the step time minus that of
  the same sequence of forward_lowres calls on windows gathered beforehand, timed in the same rounds; share =
  (full - forwards only) / full. Also the sum of those kernels' own times, replayed in isolation.
- The epilogue's kernel time over many launches for all 8 images at once, and the bytes it must move (the
  low-resolution logits of every window, which already carry the overlap factor; the int64 labels; the two uint8 maps)
  over that time, against the 7.7 TB/s of the data sheet.
- ms per scene for one --big x --big scene with windows 512 / 384 (bf16 and FP8, with int64 labels' counts).
- --usefulness N: N training runs of R50-OS16 on 256^2 tiles of the synthetic band task of tests/test_tta_gpu.py
  (150 steps each), each evaluated on 1024^2 scenes of the same task as one forward and in windows 256 / 192.
- The card's name, power limit and max SM clock, read in the same run.

    python tools/window_predict.py [--batch 8 --size 2048 --rounds 3 --steps 3 --big 11000 --usefulness 3] [--out FILE.json]
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
CONFIGS = {"whole": (None, None), "512/384": (512, 384), "256/192": (256, 192)}


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


class Plan:
    """The chunks _predict_window issues for one batch, with every window gathered beforehand, so the forwards, the
    gathers, the logit copies and the epilogue can each be timed on their own."""

    def __init__(self, net, x, y, window, stride):
        B, _, H, W = x.shape
        self.net, self.x, self.y, self.H, self.W = net, x, y, H, W
        self.win = predict._windows(H, W, window, stride)
        wh, ww = self.win.size
        n_win = B * len(self.win.ys) * len(self.win.xs)
        chunk = max(1, min(n_win, predict.MAX_FORWARD_PIXELS // (wh * ww)))
        self.chunks = [(g0, min(chunk, n_win - g0)) for g0 in range(0, n_win, chunk)]
        self.xw = ops.window_gather_f32(x, self.win.size, self.win.stride)
        self.buf = torch.empty((chunk, x.shape[1], wh, ww), dtype=torch.float32, device=x.device)
        lo = net.forward_lowres(self.xw[:1])
        self.lows = torch.empty((n_win,) + tuple(lo.shape[1:]), dtype=torch.float32, device=x.device)
        self.lo_chunk = torch.randn((chunk,) + tuple(lo.shape[1:]), device=x.device)
        self.cm = torch.zeros(5, dtype=torch.int64, device=x.device)
        self.pred = torch.empty((B, H, W), dtype=torch.uint8, device=x.device)
        self.conf = torch.empty_like(self.pred)

    def forwards(self):
        for g0, n in self.chunks:
            self.net.forward_lowres(self.xw[g0:g0 + n])

    def gathers(self):
        for g0, n in self.chunks:
            ops.window_gather_f32(self.x, self.win.size, self.win.stride, g0, n, out=self.buf[:n])

    def copies(self):
        for g0, n in self.chunks:
            self.lows[g0:g0 + n].copy_(self.lo_chunk[:n])

    def epilogue(self):
        ops.predict_window_epilogue(self.lows, self.H, self.W, self.win.size, self.win.stride, self.y, threshold=0.5,
                                    out=self.cm, pred=self.pred, conf=self.conf)

    def epilogue_bytes(self):
        return self.lows.numel() * 4 + self.y.numel() * self.y.element_size() + 2 * self.pred.numel()


def cfg4(a, dev, res):
    m = modeling.deeplabv3plus_resnet50(num_classes=2, output_stride=16, pretrained_backbone=False)
    m.load_state_dict(seeded_state_dict(m.state_dict(), 1234))
    m.to(dev).eval()
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(a.batch, 3, a.size, a.size, device=dev, generator=g)
    y = (torch.rand(a.batch, a.size, a.size, device=dev, generator=g) < 0.1).long()
    qm = quantize_fp8(m, x)
    met = StreamMetrics(2, device=dev, shape_metrics=False)
    fns, plans = {}, {}
    for pname, net in (("bf16", m), ("fp8", qm)):
        for cname, (w, s) in CONFIGS.items():
            fns[f"{pname} {cname}"] = lambda net=net, w=w, s=s: predict.predict_mask(net, x, 0.5, y, met, window=w, stride=s)
            if w is not None:
                plans[f"{pname} {cname}"] = Plan(net, x, y, w, s)
    for k, fn in fns.items():
        for _ in range(a.warmup):
            fn()
            if k in plans:
                plans[k].forwards()
    torch.cuda.synchronize()
    for _ in range(a.rounds):
        for k, fn in fns.items():
            ms = timed(fn, a.steps)
            row = {"ms_per_batch": ms, "img_per_s": a.batch * 1e3 / ms}
            if k in plans:
                row["forwards_only_ms"] = timed(plans[k].forwards, a.steps)
            res["rounds"].setdefault(k, []).append(row)
    summary = {}
    for k in fns:
        rows = res["rounds"][k]
        best = min(rows, key=lambda r: r["ms_per_batch"])
        s = {"img_per_s_best": best["img_per_s"], "ms_per_batch_best": best["ms_per_batch"]}
        whole = min(r["ms_per_batch"] for r in res["rounds"][k.split()[0] + " whole"])
        s["cost_vs_whole_image"] = best["ms_per_batch"] / whole
        if k in plans:
            p = plans[k]
            fwd = min(r["forwards_only_ms"] for r in rows)
            s.update(windows=p.lows.shape[0], forwards=len(p.chunks), windows_per_forward=p.chunks[0][1],
                     forwards_only_ms_best=fwd, non_forward_share_of_step=(best["ms_per_batch"] - fwd) / best["ms_per_batch"])
            for name, f in (("gather", p.gathers), ("copies", p.copies), ("epilogue", p.epilogue)):
                f()
                s[f"{name}_kernel_ms"] = timed(f, a.reps)
            s["gather_copies_epilogue_kernel_share"] = (s["gather_kernel_ms"] + s["copies_kernel_ms"] + s["epilogue_kernel_ms"]) / best["ms_per_batch"]
            nbytes = p.epilogue_bytes()
            s["epilogue_bytes"] = nbytes
            s["epilogue_tb_per_s"] = nbytes / (s["epilogue_kernel_ms"] * 1e-3) / 1e12
            s["epilogue_share_of_datasheet_hbm"] = s["epilogue_tb_per_s"] / DATASHEET_HBM_TBPS
        summary[k] = s
    res["summary"] = summary
    return m, qm


def big_scene(a, dev, m, qm, res):
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.randn(1, 3, a.big, a.big, device=dev, generator=g)
    y = (torch.rand(1, a.big, a.big, device=dev, generator=g) < 0.1).long()
    met = StreamMetrics(2, device=dev, shape_metrics=False)
    out = {"size": a.big, "window": 512, "stride": 384, "windows": len(predict._windows(a.big, a.big, 512, 384).ys) ** 2}
    for pname, net in (("bf16", m), ("fp8", qm)):
        fn = lambda net=net: predict.predict_mask(net, x, 0.5, y, met, window=512, stride=384)
        fn()
        out[f"{pname}_ms_per_scene"] = min(timed(fn, 1) for _ in range(a.rounds))
    res["big_scene"] = out


def usefulness(a, dev, res):
    from iswm_b200.graphs import GraphedTrainStep
    from iswm_b200.optim import FusedSGD
    from iswm_b200.utils.loss import CrossEntropyLoss
    from tests.test_model_gpu import build
    from tests.test_tta_gpu import _band_tiles
    xs, ys = (t.to(dev) for t in _band_tiles(64, 256, 1))
    xt, yt = (t.to(dev) for t in _band_tiles(8, 1024, 2))
    runs = []
    for r in range(a.usefulness):
        torch.manual_seed(r)
        m, _ = build("resnet50", 16, seed=7 + r)
        m.to(dev).train()
        crit = CrossEntropyLoss(weight=torch.tensor([1.0, 4.0])).to(dev)
        step = GraphedTrainStep(m, crit, FusedSGD(m, lr=0.02, momentum=0.9, weight_decay=1e-4))
        for i in range(a.train_steps):
            j = (i * 8) % 64
            loss = step(xs[j:j + 8], ys[j:j + 8])
        m.eval()
        row = {"seed": 7 + r, "final_loss": float(loss)}
        for name, kw in (("whole", {}), ("window_256_192", dict(window=256, stride=192))):
            mt = StreamMetrics(2, device=dev, shape_metrics=False)
            predict.predict_mask(m, xt, 0.5, yt, mt, **kw)
            rr = mt.get_results()
            row[f"fg_iou_{name}"], row[f"miou_{name}"] = float(rr["Foreground IoU"]), float(rr["MIoU"])
        runs.append(row)
        print(json.dumps(row), flush=True)
    res["usefulness"] = {"task": "synthetic bands of tests/test_tta_gpu.py; trained on 64 tiles of 256^2, evaluated on 8 scenes of 1024^2",
                         "train_steps": a.train_steps, "runs": runs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--size", type=int, default=2048)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--big", type=int, default=11000, help="edge of the single large scene (0: skip)")
    ap.add_argument("--usefulness", type=int, default=0, help="training runs of the usefulness comparison (0: skip)")
    ap.add_argument("--train-steps", type=int, default=150)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("window_predict.py measures on a GPU; none is available")
    dev = torch.device("cuda:0")
    res = {"card (name, power limit, max SM clock)": card(), "batch": a.batch, "size": a.size, "steps": a.steps,
           "max_forward_pixels": predict.MAX_FORWARD_PIXELS, "rounds": {}}
    with torch.no_grad():
        m, qm = cfg4(a, dev, res)
        torch.cuda.empty_cache()
        if a.big:
            big_scene(a, dev, m, qm, res)
    del m, qm
    torch.cuda.empty_cache()
    if a.usefulness:
        usefulness(a, dev, res)
    txt = json.dumps(res, indent=1)
    print(txt)
    if a.out:
        os.makedirs(os.path.dirname(a.out) or ".", exist_ok=True)
        with open(a.out, "w") as f:
            f.write(txt)


if __name__ == "__main__":
    main()
