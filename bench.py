#!/usr/bin/env python
"""Headline benchmark: multimodal survival TRAINING throughput (volumes/s) on B200.

    python bench.py --gpus N --steps K --warmup W            # this build (sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K --warmup W   # reference's algorithm on the host CPU cores

Workload (BASELINE.json configs[1]): T1+T2 2x128x128x64 volumes + 20 clinical variables, batch 16 per GPU,
3-D DenseNet-121 + clinical MLP + fusion heads, --blend (GradientBlender over 3 heads), Cox loss as the reference calls
it, dropout 0.2 (config.yaml default), backward, SGD(nesterov, momentum 0.9, wd 1e-4) step EVERY batch.
A "step" = one such batch.  Synthetic data (oracle/synth.py distributions), reference-law random weights.

One JSON line on stdout (rank 0).  `value` = device-resident inputs; `e2e` = same step through the public API with the
batch in pinned HOST memory (H2D copy inside the timed region) and the loss read back to the host every step.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    "cfg2": dict(name="configs[1]: T1+T2 2x128x128x64 + 20 clinical, blend, batch 16/GPU", cin=2, spatial=(128, 128, 64), batch=16),
    "cfg1": dict(name="configs[0]: T1 1x64x64x32 + 20 clinical, blend, batch 4/GPU (debug size)", cin=1, spatial=(64, 64, 32), batch=4),
    "cfg4": dict(name="configs[3]: image-only classification, 3-D ResNet (r3d_18) on 1x256x256x64 volumes, batch 8/GPU "
                      "(1 channel: the reference's stem is Conv3d(1, 64), SURVEY.md section 0)", cin=1, spatial=(256, 256, 64), batch=8),
}
BLOCKS = (6, 12, 24, 16)


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf_sust=d.get("bf16_tflops_sustained", d["bf16_tflops"]), src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf_sust=1400.0, src="fallback")


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 50 ms while the timed region runs."""
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index, enabled=True):
        self.index, self.lines, self.proc = index, [], None
        self.t0 = self.t1 = None
        self.enabled = enabled     # only rank 0 samples: N concurrent nvidia-smi pollers contend for the driver on a shared host

    def __enter__(self):
        if not self.enabled:
            return self
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=lambda: [self.lines.append((time.time(), l)) for l in self.proc.stdout], daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def wait_first_sample(self, timeout=5.0):
        """nvidia-smi needs a few hundred ms to start: do not begin the timed region before it delivers."""
        t = time.time()
        while self.proc is not None and not self.lines and time.time() - t < timeout:
            time.sleep(0.02)

    def mark_start(self):
        self.t0 = time.time()

    def mark_end(self):
        self.t1 = time.time()

    def __exit__(self, *a):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        """Median SM clock and the union of throttle reasons over the samples taken between mark_start and mark_end (the
        device-resident and end-to-end timed regions, both under the same load)."""
        sm, mx, reasons = [], 0, set()
        for ts, l in self.lines:
            if self.t0 is not None and (ts < self.t0 or (self.t1 is not None and ts > self.t1 + 0.05)):
                continue
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def conv_flops(wl):
    """Algorithmic FLOPs per batch of each GEMM-shaped kernel class (2*M*N*K, no credit for padding / recompute)."""
    B = wl["batch"]; X, Y, Z = wl["spatial"]; cin = wl["cin"]
    d0 = [(v - 1) // 2 + 1 for v in (X, Y, Z)]
    d = [(v - 1) // 2 + 1 for v in d0]
    M0 = B * d0[0] * d0[1] * d0[2]
    fl = {"stem": 2.0 * M0 * 64 * 343 * cin, "conv1": 0.0, "conv2": 0.0, "trans": 0.0}
    per_layer = {"conv1": [], "conv2": []}
    c = 64
    for b, nl in enumerate(BLOCKS):
        M = B * d[0] * d[1] * d[2]
        for l in range(nl):
            fl["conv1"] += 2.0 * M * 128 * (c + 32 * l)
            fl["conv2"] += 2.0 * M * 32 * 128 * 27
        c += 32 * nl
        if b < len(BLOCKS) - 1:
            fl["trans"] += 2.0 * M * c * (c // 2)
            c //= 2
            d = [v // 2 for v in d]
    return fl


def mem_bytes(wl):
    """Algorithmic bytes per batch of the memory-bound kernel classes (each logical tensor read once + written once in
    its storage dtype: fp16 activations, bf16 gradients, fp32 gradient accumulator; DESIGN.md section 3.2)."""
    B = wl["batch"]; X, Y, Z = wl["spatial"]
    d0 = [(v - 1) // 2 + 1 for v in (X, Y, Z)]
    d = [(v - 1) // 2 + 1 for v in d0]
    M0 = B * d0[0] * d0[1] * d0[2]
    by = {"bn_apply": M0 * 64 * 6.0, "maxpool": M0 * 64 * 2.0, "maxpool_bwd": M0 * 64 * 4.0, "extract": 0.0, "avgpool_bwd": 0.0,
          "trans_pool": 0.0, "s2d": B * wl["cin"] * X * Y * Z * 4.0 + B * (d0[0] + 3) * (d0[1] + 3) * (d0[2] + 3) * 32.0,
          # the 1x1x1 convolutions sit BELOW the ridge of the machine (arithmetic intensity 128 K / (K + 128) <= 113 FLOP/B against
          # 1400.9 TF/s / 6547.5 GB/s = 214 FLOP/B): their roofline is HBM.  16-bit tensors, each read / written once:
          "conv1_fprop": 0.0,    # read M x cin, write M x 128
          "conv1_dgrad": 0.0,    # read dBott M x 128 and the gating activations M x cin, write M x cin
          "conv1_wgrad": 0.0}    # read M x cin and M x 128
    c = 64
    for b, nl in enumerate(BLOCKS):
        M = B * d[0] * d[1] * d[2]
        if b == 0:
            by["maxpool"] += M * 64 * 3.0
            by["maxpool_bwd"] += M * 64 * 5.0
            by["extract"] += M * 64 * 10.0                          # finalize of block 1's input channels in place (read G + x, write G)
        for l in range(nl):
            cin = c + 32 * l
            last = b == len(BLOCKS) - 1
            by["bn_apply"] += M * 128 * 6.0                        # BN2 backward in place on dBott (bf16): read dA2 + bott, write dA2
            by["extract"] += M * 32 * (8.0 + (4.0 if last else 0.0))   # grad_finalize of the layer's slice: read G (fp32) + x, write bf16 (+ fp32 in the last block)
            by["conv1_fprop"] += M * (cin + 128) * 2.0
            by["conv1_dgrad"] += M * 128 * 2.0 + M * cin * (2.0 + 8.0)   # read dBott and the gating activations, read-modify-write the fp32 accumulator
            by["conv1_wgrad"] += M * (cin + 128) * 2.0
        c += 32 * nl
        if b < len(BLOCKS) - 1:
            Mo = B * (d[0] // 2) * (d[1] // 2) * (d[2] // 2)
            by["trans_pool"] += M * c * 2.0 + Mo * c * 2.0
            by["avgpool_bwd"] += M * c * 2.0 + Mo * c * 2.0 + M * c * 4.0     # ONE pass: read x + dpooled, write gamma*v (fp32)
            by["extract"] += Mo * (c // 2) * (8.0 + (4.0 if b + 1 == len(BLOCKS) - 1 else 0.0))   # finalize of the next block's input channels
            c //= 2
            d = [v // 2 for v in d]
        else:
            by["bn_apply"] += M * c * 10.0
    return by


def build_model(wl, device, seed=42):
    from mmnn_sts_b200.models.densenet import DenseNet121
    from mmnn_sts_b200.models.multimodal import MultiModalModel
    torch.manual_seed(seed)
    m = MultiModalModel(DenseNet121(spatial_dims=3, in_channels=wl["cin"], out_channels=2, feature_channels=12, dropout_prob=0.2),
                        ["x"] * 20, 2, 12, blend=True)
    return m.to(device).train()


def make_batches(wl, n, pinned=False, device=None, seed=1234, image_dtype=None):
    """Synthetic batches with the distributions of SURVEY.md section 8d (image U[0,1), 10 N(0,1) + 10 categorical
    clinical columns, Bernoulli events, tie-free integer-day durations)."""
    out = []
    for i in range(n):
        g = torch.Generator().manual_seed(seed + i)
        B = wl["batch"]
        im = torch.rand((B, wl["cin"]) + tuple(wl["spatial"]), generator=g)
        cl = torch.cat([torch.randn((B, 10), generator=g), torch.randint(0, 5, (B, 10), generator=g).float()], 1)
        ev = torch.randint(0, 2, (B, 2), generator=g)
        du = torch.stack([torch.randperm(3650, generator=g)[:B] + 1 for _ in range(2)], 1)
        if image_dtype is not None:
            im = im.to(image_dtype)
        t = [im, cl, ev, du]
        if pinned:
            t = [x.pin_memory() for x in t]
        elif device is not None:
            t = [x.to(device) for x in t]
        out.append(t)
    return out


def dump_outputs(out_dir, tensors):
    """Writes each tensor as out_dir/<name>.npy (float64 stays float64, everything else becomes float32)."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in tensors.items():
        t = t.detach().cpu()
        np.save(os.path.join(out_dir, name + ".npy"), (t if t.dtype == torch.float64 else t.float()).numpy())


def run_ours(args):
    from mmnn_sts_b200 import _lib as L, distributed as D
    from mmnn_sts_b200.losses.GradientBlender import GradientBlender
    from mmnn_sts_b200.losses.losses import CoxPH
    from mmnn_sts_b200.optim import SGD
    from mmnn_sts_b200.utils.utils import surv_criterion
    import torch.distributed as dist
    rank, world, device = D.init_from_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    wl = WORKLOADS[args.workload]
    L.lib()
    model = build_model(wl, device)
    opt = SGD(model.parameters(), 5e-4, momentum=0.9, nesterov=True, weight_decay=1e-4,
              capturable=bool(getattr(args, 'graph', False)))   # one-launch torch.optim.SGD subclass
    blender = GradientBlender(CoxPH, survival=True, surv_criterion=surv_criterion)
    sync = D.GradientAllReducer(model.parameters(), model=model)
    dev_batches = make_batches(wl, 2, device=device, seed=1234 + 100 * rank)
    # e2e arm: the loader hands over 16-bit volumes (the stem rounds the image to fp16 first thing, so this changes no result bit
    # and halves the host->device bytes; --e2e-fp32 ships the reference collate's fp32 tensors instead)
    e2e_dtype = None if args.e2e_fp32 else torch.float16
    host_batches = make_batches(wl, 2, pinned=True, seed=1234 + 100 * rank, image_dtype=e2e_dtype)
    last = {} if args.dump_outputs else None     # --dump-outputs: what the latest step handed back to its caller

    def step(im, cl, ev, du):
        out = model({"image": im, "clinical": cl})
        loss, _ = blender.computeLoss(out, ev, du)
        sync.arm()                               # step every batch: the trunk's gradient groups are all-reduced during backward
        loss.backward()
        sync()
        opt.step()
        opt.zero_grad(set_to_none=True)
        if last is not None:
            last["preds"], last["loss"] = out.detach(), loss.detach()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    copy_stream = torch.cuda.Stream(device=device)
    loss_host = torch.zeros(2, dtype=torch.float32).pin_memory()
    stage = [[torch.empty_like(t, device=device) for t in hb] for hb in host_batches]   # static device staging sets (double buffer)
    slot_free = [None, None]

    def timed(nsteps, e2e):
        """e2e: every step's batch comes from pinned HOST memory (copy of batch i+1 into a static double-buffered device
        staging set is prefetched on a copy stream while step i computes, as an input pipeline would) and every step's loss
        is read back to the host (asynchronously into pinned memory, consumed one step later so the launch queue never
        drains)."""
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ev0.record()
        if not e2e:
            # free-running: the host enqueues ahead.  (Bounding the run-ahead to two steps with blocking event waits was tried for the
            # 8-GPU run-to-run spread of this number -- 10.3-11.2 k volumes/s while the end-to-end loop repeats to 0.2 % -- and did
            # not change it: 11.1 / 10.7 k.)
            for i in range(nsteps):
                step(*dev_batches[i % 2])
        else:
            cur = torch.cuda.current_stream()
            def fetch(i):
                # batch i goes into the static device staging set i % 2 once the step that last read that set (i - 2) is done
                with torch.cuda.stream(copy_stream):
                    if slot_free[i % 2] is not None:
                        copy_stream.wait_event(slot_free[i % 2])
                    for d, h in zip(stage[i % 2], host_batches[i % 2]):
                        d.copy_(h, non_blocking=True)
                    e = torch.cuda.Event(); e.record(copy_stream)
                return stage[i % 2], e
            nxt = fetch(0)
            loss_ev, seen = None, 0.0
            for i in range(nsteps):
                b, e = nxt
                cur.wait_event(e)
                if i + 1 < nsteps:
                    nxt = fetch(i + 1)
                loss = step(*b)
                slot_free[i % 2] = torch.cuda.Event(); slot_free[i % 2].record(cur)
                if loss_ev is not None:
                    loss_ev.synchronize(); seen += float(loss_host[(i - 1) % 2])   # previous step's loss is on the host
                loss_host[i % 2].copy_(loss.detach(), non_blocking=True)
                loss_ev = torch.cuda.Event(); loss_ev.record(cur)
            loss_ev.synchronize(); seen += float(loss_host[(nsteps - 1) % 2])
        ev1.record()
        barrier()
        ms = torch.tensor([ev0.elapsed_time(ev1)], device=device)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms)

    for i in range(args.warmup):
        step(*dev_batches[i % 2])
    eager_step = step
    if args.graph and world == 1:
        from mmnn_sts_b200.graph import GraphedTrainStep
        graphed = GraphedTrainStep(lambda *b: eager_step(*b).detach(), dev_batches[0], warmup=2)
        step = lambda *b: graphed(*b)
    launches0 = L.lib().mmnn_launch_count()
    with ClockSampler(device.index or 0, enabled=(rank == 0)) as cs:
        cs.wait_first_sample()
        timed(2, e2e=True)                       # settle the e2e pipeline (staging buffers, events) before anything is timed
        # ... and the device-resident loop (untimed).  The first ~0.3 s of steps on a fresh box run slower (1 GPU: 8 steps after 3
        # warm-up steps read 1408 volumes/s, 20 after 5: 1435; on 8 GPUs the device-resident region, timed FIRST, spread 10.3-11.2 k
        # run to run while the end-to-end region timed after it repeated to 0.2 %), so the loop runs for about that long before
        # anything is timed
        timed(30, e2e=False)
        launches0 = L.lib().mmnn_launch_count()
        cs.mark_start()
        ms = timed(args.steps, e2e=False)
        launches = (L.lib().mmnn_launch_count() - launches0) // max(1, args.steps)
        ms_e2e = timed(args.steps, e2e=True)
        if last is not None:                     # the last timed step's outputs, before the untimed steps below move the weights
            dumped = {k: v.clone() for k, v in last.items()}
            dumped["state_dict"] = torch.cat([t.detach().reshape(-1).float() for t in model.state_dict().values() if t.is_floating_point()])
        if ms + ms_e2e < 400.0:                  # short runs: keep the same load going until a few 50 ms samples exist
            timed(int((400.0 - ms - ms_e2e) / max(ms / args.steps, 0.1)) + 1, e2e=False)   # (ms is the max over ranks: same count everywhere)
        cs.mark_end()
    if args.graph and world == 1:                # a replayed graph launches the captured kernels without passing the counter
        l0 = L.lib().mmnn_launch_count(); eager_step(*dev_batches[0]); launches = L.lib().mmnn_launch_count() - l0
    clocks = cs.summary()
    h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); h0.record()
    for _ in range(3):
        stage[0][0].copy_(host_batches[0][0], non_blocking=True)
    h1.record(); torch.cuda.synchronize()
    h2d_gbps = 3 * host_batches[0][0].numel() * host_batches[0][0].element_size() / (h0.elapsed_time(h1) / 1e3) / 1e9   # bare pinned-host -> device rate of this box
    vols = wl["batch"] * world * args.steps
    value, value_e2e = vols / (ms / 1e3), vols / (ms_e2e / 1e3)

    # ---- live per-kernel-class timing (CUDA events on the launch stream) for the roofline block
    peaks = load_peaks()
    L.lib().mmnn_profile_enable(1)
    nprof = 2
    for i in range(nprof):
        eager_step(*dev_batches[i % 2])          # per-kernel timing always runs eagerly on one stream
    torch.cuda.synchronize()
    prof = L.profile_collect()
    L.lib().mmnn_profile_enable(0)
    fl = conv_flops(wl)
    gemm_classes = {"stem_fprop": fl["stem"], "stem_wgrad": fl["stem"], "conv1_fprop": fl["conv1"], "conv1_dgrad": fl["conv1"],
                    "conv1_wgrad": fl["conv1"], "conv2_fprop": fl["conv2"], "conv2_dgrad": fl["conv2"], "conv2_wgrad": fl["conv2"],
                    "trans_fprop": fl["trans"], "trans_dgrad": fl["trans"], "trans_wgrad": fl["trans"]}
    mbytes = mem_bytes(wl)
    kernels, total_ms = {}, sum(v[0] for v in prof.values()) / nprof
    for k, (t, n) in prof.items():
        if n == 0:
            continue
        e = {"ms_per_step": round(t / nprof, 4), "launches_per_step": n // nprof, "share": round(t / nprof / total_ms, 4)}
        if k in gemm_classes:
            e["tflops"] = round(gemm_classes[k] / (t / nprof / 1e3) / 1e12, 1)
            e["frac_of_sustained_peak"] = round(e["tflops"] / peaks["tf_sust"], 4)
        if k in mbytes:
            e["gbps"] = round(mbytes[k] / (t / nprof / 1e3) / 1e9, 1)
            e["frac_of_hbm_peak"] = round(e["gbps"] / peaks["hbm"], 4)
        kernels[k] = e
    # `roofline` = the kernel class that takes the most time of the step, whatever bounds it; `roofline_gemm` = the largest
    # tensor-core class; `roofline_step` = the whole step's algorithmic FLOPs against the sustained tensor peak.
    def class_roofline(k):
        e = kernels[k]
        hbm_bound = "gbps" in e and (k not in gemm_classes or k.startswith("conv1_"))
        r = {"kernel": k, "ms_per_step": e["ms_per_step"], "launches_per_step": e["launches_per_step"], "traffic": None}
        if hbm_bound:
            r.update({"bound": "hbm", "achieved": e["gbps"], "peak": peaks["hbm"], "unit": "GB/s", "frac": e["frac_of_hbm_peak"],
                      "peak_source": f"MEASURED_PEAKS.json hbm_gbs ({peaks['src']})",
                      "bytes_per_launch": mbytes[k] / max(1, e["launches_per_step"])})
        else:
            r.update({"bound": "tensor", "achieved": e["tflops"], "peak": peaks["tf_sust"], "unit": "TFLOP/s", "frac": e["frac_of_sustained_peak"],
                      "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peaks['src']})",
                      "flops_per_launch": gemm_classes[k] / max(1, e["launches_per_step"])})
        r["avg_launch_ms"] = round(e["ms_per_step"] / max(1, e["launches_per_step"]), 5)
        return r
    rated = [k for k in kernels if "gbps" in kernels[k] or "tflops" in kernels[k]]
    dom = max(rated, key=lambda k: kernels[k]["ms_per_step"])
    dom_gemm = max((k for k in kernels if k in gemm_classes and not k.startswith("conv1_")), key=lambda k: kernels[k]["ms_per_step"])
    roofline, roofline_gemm = class_roofline(dom), class_roofline(dom_gemm)
    step_flops = 3.0 * (fl["stem"] + fl["conv1"] + fl["conv2"] + fl["trans"]) - fl["stem"]      # fprop + dgrad + wgrad, no stem dgrad
    roofline_step = {"bound": "tensor", "achieved": round(step_flops / (ms / args.steps / 1e3) / 1e12, 1), "peak": peaks["tf_sust"], "unit": "TFLOP/s",
                     "frac": round(step_flops / (ms / args.steps / 1e3) / 1e12 / peaks["tf_sust"], 4),
                     "algorithmic_gflop_per_step_per_gpu": round(step_flops / 1e9, 1),
                     "note": "per GPU; the executed transition GEMMs run on the pooled tensor (8x fewer FLOPs), credited at the un-pooled count"}
    for tag in ("r02", "r01"):
        tpath = os.path.join(ROOT, "profiles", f"{tag}_ncu_traffic.json")
        if os.path.isfile(tpath):
            tj = json.load(open(tpath))
            for r in (roofline, roofline_gemm):
                if r["traffic"] is None and r["kernel"] in tj:   # DRAM bytes of the class's largest launch (ncu --set full), next to that launch's algorithmic bytes
                    r["traffic"] = tj[r["kernel"]]["traffic_bytes"]
                    r["traffic_note"] = {k: tj[r["kernel"]][k] for k in ("launch", "algorithmic_bytes", "duration_us")}
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_reference_arm(wl, steps=1, warmup=1, sample_batch=wl["batch"])      # the SAME batch of 16 the GPU arm steps on
    if rank == 0:
        in_bytes = sum(t.numel() * t.element_size() for t in host_batches[0])
        line = {"metric": "train volumes/sec", "value": round(value, 2), "unit": "volumes/s", "n_gpus": world, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": round(ms / args.steps, 3), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                "dtype_detail": "16-bit tensor-core operands (activations/forward weights fp16, gradients bf16), fp32 accumulate (DESIGN.md 5)",
                "config": {"workload": wl["name"], "global_batch": wl["batch"] * world, "volume": list(wl["spatial"]),
                           "in_channels": wl["cin"], "parallelism": f"dp{world}", "optimizer_step": "every batch", "cuda_graph": bool(args.graph and world == 1),
                           "l2": "inputs (134 MB/batch fp32) and activations (>1 GB) exceed the 126 MB L2; two batches alternate"},
                "e2e": {"value": round(value_e2e, 2), "unit": "volumes/s", "h2d_bytes_per_step": in_bytes, "d2h_bytes_per_step": 4,
                        "ms_per_step": round(ms_e2e / args.steps, 3), "h2d_gbps_alone": round(h2d_gbps, 1),
                        "image_dtype": "float32" if args.e2e_fp32 else "float16 (rounded by the stem to fp16 anyway: bit-identical results)"},
                "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "roofline_gemm": roofline_gemm,
                "roofline_step": roofline_step, "kernels": kernels}
        if cpu is not None:
            line["cpu_baseline"] = cpu
    # ---- the other BASELINE configs, measured in the same invocation so the driver's record carries them:
    # configs[3] (3-D ResNet classification step, N GPUs) and configs[4] (10 000-patient eval forward + 1000-resample bootstrap)
    extra = {}
    if not args.no_extras and args.workload == "cfg2":
        torch.cuda.empty_cache()
        try:
            r = resnet_measure(args, rank, world, device, cpu_baseline=False)
            if r is not None:
                extra["resnet_cfg4"] = {k: r[k] for k in ("metric", "value", "unit", "n_gpus", "ms_per_step", "e2e", "gpu_launches", "roofline", "config", "clocks")}
        except Exception as ex:    # an extra must never take the headline line down
            extra["resnet_cfg4"] = {"error": repr(ex)[:200]}
        torch.cuda.empty_cache()
        if rank == 0:
            try:
                extra["inference_cfg5"] = inference_measure(args, device)
            except Exception as ex:
                extra["inference_cfg5"] = {"error": repr(ex)[:200]}
    if rank == 0:
        if extra:
            line["extra"] = extra
        print(json.dumps(line), flush=True)
        if last is not None:
            dump_outputs(args.dump_outputs, dumped)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_inference(args):
    print(json.dumps(inference_measure(args, torch.device("cuda", 0))), flush=True)


def inference_measure(args, dev):
    """BASELINE.json configs[4]: --inference --bootstrap --no_gradcam on synthetic patients: every patient is forwarded
    ONCE in eval mode (batched), then 1000 bootstrap resamples of the per-class C-index are counted on the GPU
    (/root/reference/main.py:750-887 re-forwards every patient per resample)."""
    import numpy as np
    from mmnn_sts_b200 import main as M
    wl = WORKLOADS["cfg2" if args.workload == "cfg4" else args.workload]
    model = build_model(wl, dev).eval()
    n, bs, R = args.patients, wl["batch"], args.resamples
    g = torch.Generator(device=dev).manual_seed(7)
    preds, ev, du = [], [], []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with torch.no_grad():
        for w in range(2):   # warm-up
            model({"image": torch.rand((bs, wl["cin"]) + tuple(wl["spatial"]), device=dev, generator=g), "clinical": torch.randn(bs, 20, device=dev, generator=g)})
        torch.cuda.synchronize(); e0.record()
        for i in range(0, n, bs):
            b = min(bs, n - i)
            out = model({"image": torch.rand((b, wl["cin"]) + tuple(wl["spatial"]), device=dev, generator=g), "clinical": torch.randn(b, 20, device=dev, generator=g)})
            preds.append(out[0])
        e1.record(); torch.cuda.synchronize()
    fwd_ms = e0.elapsed_time(e1)
    preds = torch.cat(preds)
    events = torch.randint(0, 2, (n, 2), device=dev, generator=g)
    durations = torch.randint(1, 3651, (n, 2), device=dev, generator=g)
    idx = torch.as_tensor(np.stack([np.random.RandomState(42 + r).randint(0, n, n) for r in range(R)]), device=dev)
    M.bootstrap_cindices(preds, events, durations, idx[:2])      # warm-up (module load, attribute set)
    torch.cuda.synchronize(); e0.record()
    c, mean, std, _ = M.bootstrap_cindices(preds, events, durations, idx)
    e1.record(); torch.cuda.synchronize()
    boot_ms = e0.elapsed_time(e1)
    return {"mode": "inference+bootstrap", "patients": n, "resamples": R, "forward_volumes_per_s": round(n / (fwd_ms / 1e3), 1),
            "forward_ms": round(fwd_ms, 1), "bootstrap_ms": round(boot_ms, 2),
            "patients_per_s_end_to_end": round(n / ((fwd_ms + boot_ms) / 1e3), 1), "cindex_mean": [float(v) for v in mean],
            "cindex_std": [float(v) for v in std], "workload": wl["name"], "n_gpus": 1,
            "note": "eval-mode forward of every patient once (batch 16, random volumes generated on the device per batch, inside the timed region), "
                    "then all resamples counted by one cindex_bootstrap launch per class (exact int64 pair counts)"}


def run_preprocess(args):
    """SURVEY.md section 8f rank 1 (extra mode, prints its own JSON line): Normalize -> ScaleIntensity -> Resize of raw
    2-channel volumes to the bench workload's input shape on the GPU, next to the oracle on the host cores."""
    import numpy as np
    from mmnn_sts_b200 import _lib as L
    from mmnn_sts_b200.data.transforms import ValTransformsGPU, IMAGE_DATA_MEAN, IMAGE_DATA_STDDEV
    from oracle import preprocess as op
    dev = torch.device("cuda", 0)
    wl = WORKLOADS[args.workload]
    B, C = wl["batch"], wl["cin"]
    rawdims = tuple(int(v * 1.5) for v in wl["spatial"])          # raw scans are larger than the network input
    g = torch.Generator(device=dev).manual_seed(5)
    raws = [torch.rand((B, C) + rawdims, device=dev, generator=g) * 2000.0 for _ in range(2)]    # 2 x 0.85 GB > L2
    tf = ValTransformsGPU(IMAGE_DATA_MEAN, IMAGE_DATA_STDDEV, wl["spatial"])
    for i in range(3):
        tf(raws[i % 2])
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    for i in range(args.steps):
        out = tf(raws[i % 2])
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    raw_bytes = raws[0].numel() * 4
    alg = 2 * raw_bytes + out.numel() * 4
    peaks = load_peaks()
    one = raws[0][0].cpu().numpy()
    t0 = time.perf_counter(); ref = op.val_transforms(one, IMAGE_DATA_MEAN, IMAGE_DATA_STDDEV, wl["spatial"]); cpu_s = time.perf_counter() - t0
    err = float(np.abs(tf(raws[0])[0].cpu().numpy() - ref).max())
    print(json.dumps({"mode": "preprocess", "metric": "volumes/sec", "value": round(B / (ms / 1e3), 1), "ms_per_batch": round(ms, 3),
                      "batch": B, "raw_shape": [C] + list(rawdims), "out_shape": [C] + list(wl["spatial"]),
                      "roofline": {"bound": "hbm", "achieved": round(alg / (ms / 1e3) / 1e9, 1), "peak": peaks["hbm"], "unit": "GB/s",
                                   "frac": round(alg / (ms / 1e3) / 1e9 / peaks["hbm"], 4), "algorithmic_bytes": alg},
                      "cpu_baseline": {"value": round(1.0 / cpu_s, 2), "unit": "volumes/s", "kind": "port", "cores": os.cpu_count(),
                                       "sample": "1 volume, numpy/torch oracle"},
                      "max_abs_err_vs_oracle": err}), flush=True)


def resnet_cpu_arm(wl, steps, warmup, sample_batch, num_classes=2):
    """The reference's r3d_18 classification train step (oracle/resnet.py restatement, pinned to the unchanged reference
    module by tests/golden/resnet_*.npz) on the host cores: forward, BCE-with-logits 'sum' on the sigmoid output as
    /root/reference/main.py:208 applies it, backward, SGD step; `sample_batch` volumes per step."""
    from oracle import resnet as orn
    ncores = os.cpu_count() or 1
    torch.set_num_threads(ncores)
    sd = orn.make_state_dict(42, num_classes, perturb_bn=False)
    params = {k: (v.clone().requires_grad_(True) if v.dtype.is_floating_point and "running" not in k else v.clone()) for k, v in sd.items()}
    opt = torch.optim.SGD([p for p in params.values() if p.requires_grad], 5e-4, momentum=0.9, nesterov=True, weight_decay=1e-4)
    image, labels = orn.make_batch(77, sample_batch, wl["spatial"], num_classes)
    g = torch.Generator().manual_seed(78)
    masks = [(torch.rand(s, generator=g) >= 0.2).float() for s in orn.stage_shapes(sample_batch, wl["spatial"])]
    pw = torch.tensor([1.5, 2.0])[:num_classes]
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = orn.resnet_forward(params, image, True, 0.2, masks)
        loss = orn.train_step_loss(out, labels, pw)
        loss.backward()
        opt.step(); opt.zero_grad()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    return {"value": round(sample_batch / t, 3), "unit": "volumes/s", "cores": ncores, "kind": "port",
            "sample": f"{steps} timed step(s) of {sample_batch} volumes of 1x{'x'.join(map(str, wl['spatial']))} (same model/loss/optimizer), {warmup} warm-up",
            "sec_per_step": round(t, 3)}


def run_resnet(args):
    import torch.distributed as dist
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    line = resnet_measure(args, rank, world, dev, cpu_baseline=not args.no_cpu_baseline)
    if line is not None:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def resnet_measure(args, rank, world, dev, cpu_baseline=True):
    """SURVEY.md section 8f rank 3 / BASELINE configs[3]: image-only classification training step of the 3-D ResNet encoder --
    forward, BCEWithLogitsLoss(pos_weight, 'sum') on the sigmoid output (the reference's own call, main.py:208), backward,
    SGD(nesterov) step -- batch 8 per GPU of 1x256x256x64 volumes.  Needs an initialised process group when world > 1.
    Returns the JSON line (rank 0) or None."""
    import torch.distributed as dist
    from mmnn_sts_b200 import _lib as L
    from mmnn_sts_b200 import ops
    from mmnn_sts_b200.models.resnet import algorithmic_cost, r3d_18
    from mmnn_sts_b200.optim import SGD
    local = dev.index or 0
    wl = WORKLOADS["cfg4"]
    B, K = wl["batch"], 2
    torch.manual_seed(42)
    m = r3d_18(K).to(dev).train()
    opt = SGD(m.parameters(), 5e-4, momentum=0.9, nesterov=True, weight_decay=1e-4)
    params = [q for q in m.parameters()]
    g = torch.Generator().manual_seed(1234 + rank)
    host = [(torch.rand((B, 1) + wl["spatial"], generator=g).pin_memory(), (torch.rand((B, K), generator=g) < 0.4).float().pin_memory()) for _ in range(2)]
    devb = [(a.to(dev), b.to(dev)) for a, b in host]           # two batches alternate: 2 x 134 MB of input, activations >> L2
    pw = torch.tensor([1.5, 2.0], device=dev)
    stage = [(torch.empty_like(devb[0][0]), torch.empty_like(devb[0][1])) for _ in range(2)]

    def step(im, lab):
        out = m(im)
        loss = ops.bce_with_logits(out, lab, pw).sum()
        loss.backward()
        if world > 1:
            flat = torch.cat([q.grad.reshape(-1) for q in params])
            dist.all_reduce(flat)                               # SUM, as the reference accumulates micro-batches
            off = 0
            for q in params:
                q.grad.copy_(flat[off:off + q.numel()].view_as(q.grad)); off += q.numel()
        opt.step(); opt.zero_grad(set_to_none=True)
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event(), torch.cuda.Event()]
    done = [torch.cuda.Event(), torch.cuda.Event()]

    def fetch(i):
        """H2D copy of batch i from pinned memory into staging set i % 2 on the copy stream (overlaps the previous step)."""
        k = i % 2
        copy_stream.wait_event(done[k])                         # the step that last read this staging set has finished
        with torch.cuda.stream(copy_stream):
            stage[k][0].copy_(host[k][0], non_blocking=True); stage[k][1].copy_(host[k][1], non_blocking=True)
            ready[k].record(copy_stream)

    def timed(n, e2e):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        main = torch.cuda.current_stream()
        for k in range(2):
            done[k].record(main)
        barrier(); e0.record()
        if e2e:
            fetch(0)
        for i in range(n):
            if e2e:
                k = i % 2
                if i + 1 < n:
                    fetch(i + 1)
                main.wait_event(ready[k])
                loss = step(stage[k][0], stage[k][1])
                done[k].record(main)
                loss.item()
            else:
                step(*devb[i % 2])
        e1.record(); barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()) / n

    with ClockSampler(local, enabled=(rank == 0)) as clk:
        for i in range(max(3, args.warmup)):
            step(*devb[i % 2])
        clk.wait_first_sample()
        lc0 = L.lib().mmnn_launch_count()
        clk.mark_start()
        ms = timed(args.steps, False)
        launches = (L.lib().mmnn_launch_count() - lc0) // args.steps
        timed(1, True)
        ms_e2e = timed(args.steps, True)
        clk.mark_end()
        clocks = clk.summary()
    L.lib().mmnn_profile_enable(1)
    step(*devb[0])
    prof = L.profile_collect()
    L.lib().mmnn_profile_enable(0)
    if rank != 0:
        return None
    peaks = load_peaks()
    cost = algorithmic_cost(m, B, wl["spatial"])
    kernels = {}
    for k, (kms, cnt) in prof.items():
        if cnt and kms > 0:
            kernels[k] = {"ms_per_step": round(kms, 3), "launches_per_step": cnt}
            if k in cost:
                kernels[k]["gbps"] = round(cost[k]["bytes"] / kms / 1e6, 1)
                kernels[k]["frac_of_hbm_peak"] = round(cost[k]["bytes"] / kms / 1e6 / peaks["hbm"], 4)
                if cost[k]["flops"]:
                    kernels[k]["tflops"] = round(cost[k]["flops"] / kms / 1e9, 2)
    top = max((k for k in kernels if k in cost), key=lambda k: kernels[k]["ms_per_step"])
    line = {"mode": "resnet", "metric": "train volumes/sec", "value": round(B * world / (ms / 1e3), 2), "unit": "volumes/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": round(ms, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "dtype_detail": "fp16 activations / bf16 gradients, fp32 accumulate: mma.sync m16n8k16 for the 8/16/64-channel 3x3x3 and 1x1x1 convolutions "
                            "(forward 64->8 and 8->8, data gradient 8->64 and 8->8, every weight gradient), fp32 FMA for the stem and the strided / 16-channel "
                            "forward and data-gradient launches (DESIGN.md 3.4)",
            "config": {"workload": wl["name"], "global_batch": B * world, "volume": list(wl["spatial"]), "in_channels": 1,
                       "parallelism": f"dp{world}", "optimizer_step": "every batch",
                       "l2": "two input batches alternate; every activation tensor of layer1 (135 MB - 1.08 GB) exceeds the 126 MB L2"},
            "e2e": {"value": round(B * world / (ms_e2e / 1e3), 2), "unit": "volumes/s", "h2d_bytes_per_step": host[0][0].numel() * 4 + host[0][1].numel() * 4,
                    "d2h_bytes_per_step": 4, "ms_per_step": round(ms_e2e, 3)},
            "gpu_launches": int(launches), "clocks": clocks,
            "roofline": {"kernel": top, "bound": "hbm", "achieved": kernels[top]["gbps"], "peak": peaks["hbm"], "unit": "GB/s",
                         "frac": kernels[top]["frac_of_hbm_peak"], "traffic": None, "peak_source": "MEASURED_PEAKS.json hbm_gbs (" + peaks["src"] + ")",
                         "algorithmic_bytes_per_step": cost[top]["bytes"]},
            "kernels": kernels}
    if cpu_baseline:
        line["cpu_baseline"] = resnet_cpu_arm(wl, steps=1, warmup=1, sample_batch=1)
    return line


def cpu_reference_arm(wl, steps, warmup, sample_batch):
    """The reference's algorithm for one training step on the host cores: fp32 torch CPU forward of the oracle
    restatement (bit-exact to the unchanged reference files, tests/golden), GradientBlender/Cox loss as the reference
    calls it, backward, SGD step.  A bounded sample: `sample_batch` volumes of the workload's shape per step."""
    from oracle import model as om, synth
    from oracle.blender import GradientBlenderOracle
    ncores = os.cpu_count() or 1
    torch.set_num_threads(ncores)
    sd = synth.make_state_dict(42, in_channels=wl["cin"], perturb_bn=False)
    params = {k: (v.clone().requires_grad_(True) if v.dtype.is_floating_point and "running" not in k else v.clone()) for k, v in sd.items()}
    opt = torch.optim.SGD([p for p in params.values() if p.requires_grad], 5e-4, momentum=0.9, nesterov=True, weight_decay=1e-4)
    gb = GradientBlenderOracle()
    im, cl, ev, du = synth.make_batch(77, sample_batch, wl["cin"], wl["spatial"])
    masks = synth.make_masks(78, sample_batch)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        out = om.multimodal_forward(params, im, cl, True, True, masks)
        loss, _ = gb.computeLoss(out, ev, du)
        loss.backward()
        opt.step(); opt.zero_grad()
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    t = sum(times) / len(times)
    return {"value": round(sample_batch / t, 3), "unit": "volumes/s", "cores": ncores, "kind": "port",
            "sample": f"{steps} timed step(s) of {sample_batch} volumes of {wl['cin']}x{'x'.join(map(str, wl['spatial']))} (same model/loss/optimizer), {warmup} warm-up",
            "sec_per_step": round(t, 3)}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    wl = WORKLOADS[args.workload]
    steps, warmup = args.steps, max(1, min(args.warmup, 1))
    cpu = cpu_reference_arm(wl, steps=steps, warmup=warmup, sample_batch=wl["batch"])    # the whole batch of 16: same step as the GPU arm
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    line = {"impl": "reference", "metric": "train volumes/sec", "value": cpu["value"], "unit": "volumes/s", "n_gpus": world,
            "steps": steps, "warmup": warmup, "ms_per_step": round(cpu["sec_per_step"] * 1e3, 1), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["name"], "global_batch": wl["batch"], "volume": list(wl["spatial"]), "in_channels": wl["cin"], "optimizer_step": "every batch",
                       "note": "the reference's algorithm on the host CPU cores (fp32 torch CPU, all host threads): one step = the same batch of "
                               "16 volumes the GPU arm steps on; under torchrun only rank 0 runs it (it does not scale with N)"},
            "cpu_baseline": cpu, "e2e": {"value": cpu["value"], "unit": "volumes/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--e2e-fp32", action="store_true", help="end-to-end arm ships fp32 volumes (default: fp16, same results, half the H2D bytes)")
    ap.add_argument("--no-extras", action="store_true", help="skip the configs[3] / configs[4] side measurements of the default run")
    ap.add_argument("--mode", default="train", choices=["train", "inference", "preprocess", "resnet"])
    ap.add_argument("--graph", action="store_true", help="replay the device-resident step as one CUDA graph (static shapes)")
    ap.add_argument("--patients", type=int, default=10000)
    ap.add_argument("--resamples", type=int, default=1000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps of the training run, write what its last timed step returned to DIR as .npy: preds "
                         "(the [3, B, 2] blended heads), loss, and state_dict (every floating-point tensor of the updated model's "
                         "state_dict, flattened in key order; 45 MB)")
    a = ap.parse_args()
    if a.dump_outputs and (a.mode != "train" or a.impl != "ours"):
        ap.error("--dump-outputs applies to the training run of this build (--mode train --impl ours)")
    if a.warmup < 3 and a.impl == "ours":
        a.warmup = 3
    if a.mode == "inference":
        run_inference(a)
    elif a.mode == "preprocess":
        run_preprocess(a)
    elif a.mode == "resnet":
        run_resnet(a)
    elif a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
