"""Train cfg2 (DeepLabV3+ R50-OS16, batch 16 at 512x512, bench.py's seeded inputs and weights) twice from the same seeded state
and print how far the two runs are apart after every step: loss, and parameters / gradients / BatchNorm buffers at a few steps.
Weight gradients are summed with fp32 atomics in no fixed order, so this shows at which step that last-bit noise stops being
rounding (bench.py --dump-outputs dumps the last step before it)."""
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench  # noqa: E402
from iswm_b200.graphs import GraphedTrainStep  # noqa: E402
from iswm_b200.network import modeling  # noqa: E402
from iswm_b200.optim import FusedSGD  # noqa: E402
from iswm_b200.utils.loss import CrossEntropyLoss  # noqa: E402

dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
x, y = bench.synth_batch(16, 512, 512, 0, device=dev)
N, SNAP = 14, (1, 2, 4, 8, 14)
runs = []
for r in range(2):
    torch.manual_seed(0)
    m = modeling.deeplabv3plus_resnet50(num_classes=2, output_stride=16, pretrained_backbone=False).to(dev).train()
    crit = CrossEntropyLoss(weight=torch.tensor([1.0, 7.0]), ignore_index=255).to(dev)
    opt = FusedSGD(m, lr=1e-3, momentum=0.9, weight_decay=1e-4, nesterov=True)
    st = GraphedTrainStep(m, crit, opt)
    losses, snaps = [], {}
    for i in range(1, N + 1):
        losses.append(float(st(x, y)))
        if i in SNAP:
            ps = list(m.parameters())
            snaps[i] = (torch.cat([p.detach().reshape(-1) for p in ps]).clone(), torch.cat([p.grad.reshape(-1) for p in ps]).clone(),
                        torch.cat([b.reshape(-1).float() for b in m.buffers()]).clone())
    runs.append((losses, snaps))
    del st, m, opt
    torch.cuda.empty_cache()
(la, sa), (lb, sb) = runs
for i in range(N):
    print(f"step {i + 1:2d} loss {la[i]:.9f} {lb[i]:.9f} rel {abs(la[i] - lb[i]) / abs(lb[i]):.3e}")
rel = lambda a, b: float((a - b).norm() / b.norm())
for i in SNAP:
    (wa, ga, ba), (wb, gb, bb) = sa[i], sb[i]
    print(f"after step {i:2d}: params relL2 {rel(wa, wb):.3e} maxabs {float((wa - wb).abs().max()):.3e} | grads relL2 {rel(ga, gb):.3e} "
          f"maxabs {float((ga - gb).abs().max()):.3e} | buffers relL2 {rel(ba, bb):.3e}")
