"""Repeat the same two train steps from identical state several times WITHOUT any synchronisation in between; a race in
the launch pipeline shows up as run-to-run differences far above the ~1e-7 of the weight-gradient atomics."""
import os, sys
sys.path.insert(0, os.getcwd()); sys.path.insert(0, "tests")
import torch
from test_graphs_gpu import _batches, _model, DEV
from iswm_b200.optim import FusedSGD
from iswm_b200.utils.loss import CrossEntropyLoss
reps = int(sys.argv[1]) if len(sys.argv) > 1 else 6
B, S = (int(sys.argv[2]), int(sys.argv[3])) if len(sys.argv) > 3 else (2, 96)
bs = _batches(3, B, S)
crit = CrossEntropyLoss(weight=torch.tensor([1.0, 3.0])).to(DEV)
rows = []
for r in range(reps):
    m = _model(); m.engine().dropout_p = float(os.environ.get("PDROP", "0.1"))
    opt = FusedSGD(m, lr=1e-2, momentum=0.9, weight_decay=1e-4)
    losses = []
    for x, y in bs:
        loss = crit(m(x), y); opt.zero_grad(); loss.backward(); opt.step(); losses.append(loss.detach())
    torch.cuda.synchronize()
    rows.append(([float(l) for l in losses], m.engine().flat_w.clone()))
ref = rows[0]
print({k: os.environ.get(k) for k in ("ISWM_PDL", "PDROP") if os.environ.get(k) is not None})
for i, (l, w) in enumerate(rows):
    print(f"  rep {i}: losses {' '.join(f'{v:.6f}' for v in l)}  w vs rep0 {float((w - ref[1]).norm() / ref[1].norm()):.2e}")
