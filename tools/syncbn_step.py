"""Cost of synchronised BatchNorm: GraphedTrainStep(dp=DataParallel(..., sync_bn=False / True)) on the peer-memory transport,
the two settings alternating in one call, device-event timed after warm-up. Run under torch.distributed.run, one process per GPU:

    python -m torch.distributed.run --nproc-per-node N tools/syncbn_step.py --config cfg2 [--steps 20 --rounds 3] [--out FILE.json]

cfg2 = R50-OS16, 16 x 512^2 per GPU; cfg3 = R101-OS8, 4 x 1024^2 per GPU. Rank 0 prints (and with --out, appends to FILE) one JSON
line: ms/step and img/s (all GPUs) per setting and round, the card's name and power limit.
"""
import argparse
import datetime
import json
import os
import subprocess
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from iswm_b200.graphs import GraphedTrainStep  # noqa: E402
from iswm_b200.network import modeling  # noqa: E402
from iswm_b200.optim import FusedSGD  # noqa: E402
from iswm_b200.parallel import DataParallel  # noqa: E402
from iswm_b200.utils.loss import CrossEntropyLoss  # noqa: E402
from oracle.gen_golden import seeded_state_dict, synth_labels  # noqa: E402

CONFIGS = {"cfg2": ("resnet50", 16, 512, 16), "cfg3": ("resnet101", 8, 1024, 4)}


def card():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:            # noqa: BLE001
        return f"unknown ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--config", choices=sorted(CONFIGS), default="cfg2")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
    dev = torch.device("cuda", torch.cuda.current_device())
    dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=300))
    backbone, os_, size, batch = CONFIGS[a.config]
    g = torch.Generator().manual_seed(100 + rank)
    x = torch.randn((batch, 3, size, size), generator=g).to(dev)
    y = synth_labels((batch, size, size), seed=200 + rank, fg=0.3).to(dev)
    steppers = {}
    for sync in (False, True):
        m = getattr(modeling, f"deeplabv3plus_{backbone}")(num_classes=2, output_stride=os_, pretrained_backbone=False)
        m.load_state_dict(seeded_state_dict(m.state_dict(), 5))
        m.to(dev).train()
        c = CrossEntropyLoss(weight=torch.tensor([1.0, 4.0])).to(dev)
        d = DataParallel(m, c, comm="peer", sync_bn=sync)
        opt = FusedSGD(m, lr=1e-3, momentum=0.9, weight_decay=1e-4)
        st = GraphedTrainStep(m, c, opt, dp=d)
        for _ in range(a.warmup):
            st(x, y)
        torch.cuda.synchronize()
        steppers[sync] = st
    rows = {False: [], True: []}
    for _ in range(a.rounds):
        for sync in (False, True):
            st = steppers[sync]
            dist.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(a.steps):
                st(x, y)
            e1.record()
            e1.synchronize()
            rows[sync].append(e0.elapsed_time(e1) / a.steps)
    # the slowest rank sets the pace of a synchronous step
    t = torch.tensor([rows[False], rows[True]], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    off, on = t[0].tolist(), t[1].tolist()
    if rank == 0:
        res = {"tool": "syncbn_step", "config": a.config, "model": f"{backbone}-OS{os_}", "per_gpu_batch": batch, "size": size,
               "n_gpus": world, "steps": a.steps, "rounds": a.rounds, "card": card(),
               "ms_per_step_sync_off": off, "ms_per_step_sync_on": on,
               "img_s_sync_off": [world * batch * 1000.0 / v for v in off], "img_s_sync_on": [world * batch * 1000.0 / v for v in on],
               "overhead_ms_min": min(on) - min(off), "launches_per_replay": {str(k): v.launches_per_replay for k, v in steppers.items()}}
        line = json.dumps(res)
        print(line, flush=True)
        if a.out:
            with open(a.out, "a") as f:
                f.write(line + "\n")
    for st in steppers.values():
        st.dp.model.engine().grad_ready_hook = None
    dist.barrier()
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
