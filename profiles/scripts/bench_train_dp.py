"""Data-parallel survival training through the public driver, main.train_survival(group=...), on G GPUs of one machine.
Workload: the configs[1] shape (bench.WORKLOADS["cfg2"]: 2x128x128x64 + 20 clinical, blend, batch 16 per GPU, dropout
0.2), synthetic micro-batches resident on the device as fp16 volumes (the stem reads fp16 as it is), round-robin
sharded with distributed.shard_batches.  64 / 16 = 4 micro-batches per optimiser step, so G is 1, 2 or 4.

    torchrun --nproc-per-node G profiles/scripts/bench_train_dp.py [--microbatches 64] [--epochs 2] [--out FILE]

Rank 0 prints one JSON line:
  * epoch_volumes_per_s: training patients of an epoch over the time from the epoch's start to the start of its
    epoch-end phase (forward, backward, gradient reduction, running-statistics bookkeeping and merge, optimiser steps);
  * epoch_end_ms: the epoch-end phase (gathers of the rows and losses, C-indices, validation forward and gathers,
    blending-weight update), ending when train_survival logs the epoch;
  * bn_bookkeeping_us_per_microbatch: RunningStatsMerger.before_forward + after_forward alone, timed with CUDA events
    over 200 repetitions on the trained model, and bn_merge_us_per_step: merge() (one all-reduce, G > 1 only).
Every boundary is a device synchronise on every rank followed by a barrier, so each time is the slowest rank's.  The
first train_survival call (1 epoch of 2 optimiser steps) is warm-up and is not timed."""
import argparse
import json
import os
import sys
import time
from types import SimpleNamespace

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from mmnn_sts_b200 import distributed as D  # noqa: E402
from mmnn_sts_b200 import main as M  # noqa: E402
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_inference_dp import gpu_info  # noqa: E402


def make_batches(wl, ids, dev):
    """Global micro-batches `ids`, each generated from its own seed on the device (the same data for any G)."""
    out = []
    for i in ids:
        g = torch.Generator(device=dev).manual_seed(1000 + i)
        B = wl["batch"]
        im = torch.rand((B, wl["cin"]) + tuple(wl["spatial"]), device=dev, generator=g).half()
        cl = torch.cat([torch.randn((B, 10), device=dev, generator=g), torch.randint(0, 5, (B, 10), device=dev, generator=g).float()], 1)
        ev = torch.randint(0, 2, (B, 2), device=dev, generator=g)
        du = torch.stack([torch.randperm(3650, device=dev, generator=g)[:B] + 1 for _ in range(2)], 1)
        out.append(({"image": im, "clinical": cl}, ev, du))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--microbatches", type=int, default=64, help="global training micro-batches per epoch")
    ap.add_argument("--val-microbatches", type=int, default=4)
    ap.add_argument("--epochs", type=int, default=2)
    ap.add_argument("--out", help="also write the JSON line to this file (rank 0)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    rank, world, dev = D.init_from_env()
    group = dist.group.WORLD if world > 1 else None
    wl = bench.WORKLOADS["cfg2"]
    model = bench.build_model(wl, dev)
    nb, bs = a.microbatches, wl["batch"]
    train = make_batches(wl, D.shard_batches(list(range(nb)), rank, world), dev)
    val = make_batches(wl, D.shard_batches(list(range(nb, nb + a.val_microbatches)), rank, world), dev)

    def args(epochs, n):
        return SimpleNamespace(lr=5e-4, momentum=0.9, weight_decay=1e-4, epochs=epochs, batch_size=bs, blend=True,
                               blend_update_interval=1, num_train=n * bs)

    def settle():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return time.perf_counter()

    # the epoch-end phase starts with the first gather of the rows (G > 1) or the first C-index (one process)
    marks = []                                           # (what, time) at every phase boundary of the timed call
    marker = "_gather_rows" if world > 1 else "getCIndices"
    first_of_epoch_end = getattr(M, marker)
    epoch_end_started = [False]

    def timed_marker(*p, **k):
        if not epoch_end_started[0]:
            epoch_end_started[0] = True
            marks.append(("train_end", settle()))
        return first_of_epoch_end(*p, **k)

    def log(_msg):
        epoch_end_started[0] = False
        marks.append(("epoch_end", settle()))

    M.train_survival(model, train[:8 // world], val, args(1, 8), dev, group=group)       # warm-up: two optimiser steps
    setattr(M, marker, timed_marker)
    marks.append(("epoch_end", settle()))
    M.train_survival(model, train, val, args(a.epochs, nb), dev, group=group, log=log)
    setattr(M, marker, first_of_epoch_end)
    train_s = [marks[i + 1][1] - marks[i][1] for i in range(0, len(marks) - 1, 2)]
    end_s = [marks[i + 2][1] - marks[i + 1][1] for i in range(0, len(marks) - 2, 2)]

    merger = D.RunningStatsMerger(model, group)
    merger.begin(4)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 200
    settle()
    ev0.record()
    for k in range(reps):
        merger.before_forward()
        merger.after_forward(k % 4)
    ev1.record()
    settle()
    book_us = ev0.elapsed_time(ev1) * 1e3 / reps
    merge_us = None
    if world > 1:
        settle()
        ev0.record()
        for _ in range(20):
            merger.merge()
        ev1.record()
        settle()
        merge_us = ev0.elapsed_time(ev1) * 1e3 / 20
    if rank == 0:
        line = {"mode": "train_survival, data parallel", "n_gpus": world, "micro_batch": bs,
                "train_patients_per_epoch": nb * bs, "val_patients": a.val_microbatches * bs, "epochs": a.epochs,
                "epoch_volumes_per_s": [round(nb * bs / s, 1) for s in train_s],
                "epoch_train_ms": [round(s * 1e3, 1) for s in train_s], "epoch_end_ms": [round(s * 1e3, 1) for s in end_s],
                "bn_bookkeeping_us_per_microbatch": round(book_us, 1),
                "bn_merge_us_per_step": round(merge_us, 1) if merge_us is not None else None,
                "workload": wl["name"] + ", dropout 0.2", "gpu": gpu_info(), "torch": torch.__version__,
                "backend": dist.get_backend() if world > 1 else None,
                "note": "phase boundaries are a device synchronise on every rank plus a barrier; volumes resident on the "
                        "device as fp16; first train_survival call (2 steps) untimed warm-up"}
        print(json.dumps(line), flush=True)
        if a.out:
            os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
            with open(a.out, "w") as f:
                f.write(json.dumps(line) + "\n")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
