"""Data-parallel survival inference (BASELINE configs[4], the workload of bench.inference_measure) on G GPUs of one
machine: 10 000 patients of 2x128x128x64 volumes in batches of 16, eval forward of every patient once, then a
1000-resample bootstrap C-index.  Each rank generates its contiguous share (distributed.split_rows) of the patients on
its own device from a seed, inside the timed region, as bench.inference_measure does.

    torchrun --nproc-per-node G profiles/scripts/bench_inference_dp.py [--gradcam] [--out FILE]

Rank 0 prints one JSON line.  Phases are timed one after the other, each ending with a device synchronise on every rank
and a barrier (so each is the slowest rank's time): the rank-local forward (predict_risks), the gather of the risks
(one allgather_varlen of 10 000 rows), and the bootstrap (rank 0 draws the [R, N] resample matrix, broadcast, each rank
counts its share of the resamples, all-gather of the counts, summary).  `patients_per_s_end_to_end` comes from a
separate, complete inference_survival(group=...) call on the same patients, whose C-indices must equal the phased run's.
With --gradcam every batch also goes through the map kernel, and a callback reduces each batch's maps to a checksum."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from mmnn_sts_b200 import distributed as D  # noqa: E402
from mmnn_sts_b200 import main as M  # noqa: E402


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable: " + r.stderr.strip()[:200]


def batches(wl, lo, hi, bs, dev, seed):
    """Patients lo..hi-1 in batches of bs, generated on `dev` (the same generator law as bench.inference_measure)."""
    g = torch.Generator(device=dev).manual_seed(seed)
    for i in range(lo, hi, bs):
        b = min(bs, hi - i)
        inputs = {"image": torch.rand((b, wl["cin"]) + tuple(wl["spatial"]), device=dev, generator=g),
                  "clinical": torch.randn(b, 20, device=dev, generator=g)}
        yield inputs, torch.randint(0, 2, (b, 2), device=dev, generator=g), torch.randint(1, 3651, (b, 2), device=dev, generator=g)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--patients", type=int, default=10000)
    ap.add_argument("--resamples", type=int, default=1000)
    ap.add_argument("--gradcam", action="store_true")
    ap.add_argument("--out", help="also write the JSON line to this file (rank 0)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    rank, world, dev = D.init_from_env()
    group = dist.group.WORLD if world > 1 else None
    wl = bench.WORKLOADS["cfg2"]
    bs, n, R = wl["batch"], args.patients, args.resamples
    model = bench.build_model(wl, dev).eval()
    lo, hi = D.split_rows(n, rank, world)
    ids = torch.arange(lo, hi)
    checksum = torch.zeros((), dtype=torch.float64, device=dev)

    def reduce_maps(i, maps):
        checksum.add_(maps.sum(dtype=torch.float64))

    cb = reduce_maps if args.gradcam else None

    def settle():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        return time.perf_counter()

    # warm-up: module loads, the NCCL communicators, every collective of the path
    M.inference_survival(model, batches(wl, 0, 2 * bs, bs, dev, 5), dev, num_resamples=4, seed=1, gradcam=cb, group=group)
    checksum.zero_()

    t0 = settle()
    preds, ev, du = M.predict_risks(model, batches(wl, lo, hi, bs, dev, 7 + rank), dev, gradcam=cb)
    t1 = settle()
    if world > 1:
        preds, ev, du = M._gather_patients([preds], [ev], [du], ids, group, dev)
    t2 = settle()
    if world > 1:
        c, mean, std = M._bootstrap_split(preds, ev, du, R, 42, group)
    else:                                                # the one-process path of inference_survival
        idx = M._draw_resamples(n, R, 42)
        c, mean, std, _ = M.bootstrap_cindices(preds, ev, du, torch.as_tensor(idx, device=dev))
    t3 = settle()
    full = M.inference_survival(model, batches(wl, lo, hi, bs, dev, 7 + rank), dev, num_resamples=R, seed=42, gradcam=cb,
                                group=group, patient_ids=ids if world > 1 else None)
    t4 = settle()
    assert np.array_equal(full.mean, mean) and np.array_equal(full.per_resample, c, equal_nan=True)
    if world > 1:
        dist.all_reduce(checksum)
    if rank == 0:
        d0 = time.perf_counter()
        M._draw_resamples(n, R, 42)
        draw_ms = (time.perf_counter() - d0) * 1e3
        line = {"mode": "inference+bootstrap, data parallel", "n_gpus": world, "patients": n, "resamples": R, "batch": bs,
                "gradcam": args.gradcam, "forward_volumes_per_s": round(n / (t1 - t0), 1), "forward_ms": round((t1 - t0) * 1e3, 1),
                "gather_ms": round((t2 - t1) * 1e3, 2), "bootstrap_ms": round((t3 - t2) * 1e3, 2),
                "bootstrap_draw_ms_rank0": round(draw_ms, 2),
                "patients_per_s_end_to_end": round(n / (t4 - t3), 1), "end_to_end_ms": round((t4 - t3) * 1e3, 1),
                "cindex_mean": [float(v) for v in mean], "gradcam_checksum": float(checksum) if args.gradcam else None,
                "workload": wl["name"], "gpu": gpu_info(), "torch": torch.__version__,
                "note": "phases timed in sequence, each ending with a device synchronise on every rank and a barrier; "
                        "volumes generated on the device inside the forward and end-to-end regions; bootstrap_ms includes "
                        "rank 0 drawing the resample matrix on the host (bootstrap_draw_ms_rank0 alone)"}
        print(json.dumps(line), flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                f.write(json.dumps(line) + "\n")
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
