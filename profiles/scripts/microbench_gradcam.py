"""Batched GradCAM maps on one GPU, all in one run: (1) the map kernel alone at the bench shape (B 16, 2 classes,
2x128x128x64 volumes, 4x4x2 trunk), CUDA events over many launches; (2) configs[4]-shaped inference (eval forward of
every patient, batch 16) with and without a discarding `gradcam` callback; (3) the backward-based MultiModalGradCAM at
batch size 1.  Records the card name, power limit and max SM clock in the same run.

    python profiles/scripts/microbench_gradcam.py --out profiles/gradcam_microbench.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
from mmnn_sts_b200 import _lib as L  # noqa: E402
from mmnn_sts_b200.main import predict_risks  # noqa: E402
from mmnn_sts_b200.ops import gradcam_args  # noqa: E402
from mmnn_sts_b200.utils.utils import attention_maps  # noqa: E402

MEASURED_HBM_GBS = 6547.5      # DESIGN.md section 7: measured copy bandwidth of this B200


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip().splitlines()[0] if r.returncode == 0 and r.stdout.strip() else "unavailable: " + r.stderr.strip()[:200]


def batches(wl, n, bs, dev, seed):
    g = torch.Generator(device=dev).manual_seed(seed)
    for i in range(0, n, bs):
        b = min(bs, n - i)
        inputs = {"image": torch.rand((b, wl["cin"]) + tuple(wl["spatial"]), device=dev, generator=g),
                  "clinical": torch.randn(b, 20, device=dev, generator=g)}
        yield inputs, torch.randint(0, 2, (b, 2), device=dev, generator=g), torch.randint(1, 3651, (b, 2), device=dev, generator=g)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--launches", type=int, default=400)
    ap.add_argument("--patients", type=int, default=1024)
    ap.add_argument("--old-patients", type=int, default=32)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    res = {"gpu": gpu_info(), "torch": torch.__version__}
    wl = bench.WORKLOADS["cfg2"]
    model = bench.build_model(wl, dev).eval()

    # (1) kernel alone on the inputs of one bench-shape forward
    x = next(batches(wl, wl["batch"], wl["batch"], dev, 3))[0]
    _, maps_ref = attention_maps(model, x)
    bb = model.gradcam_layer
    ws, xshape, dims, y = bb._last_forward
    act, _ = bb.block_buffer_views(ws, xshape, len(bb._cfg[1]) - 1)
    feats = model.image_model.model.features.feature_layer
    a, maps, keep = gradcam_args(act, y, dims, bb.norm5.weight, bb.norm5.running_var, bb.norm5.eps, feats.weight,
                                 model.output_head.weight, xshape[2:])
    lib, stream = L.lib(), torch.cuda.current_stream().cuda_stream
    ctas = int(lib.mmnn_gradcam_ctas(C.byref(a)))
    for _ in range(20):
        L.check(lib.mmnn_gradcam_maps(C.byref(a), stream), "mmnn_gradcam_maps")
    torch.cuda.synchronize()
    assert torch.equal(maps, maps_ref)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = []
    for _ in range(3):
        e0.record()
        for _ in range(args.launches):
            lib.mmnn_gradcam_maps(C.byref(a), stream)
        e1.record(); torch.cuda.synchronize()
        reps.append(e0.elapsed_time(e1) * 1e3 / args.launches)
    V = dims[0] * dims[1] * dims[2]
    write_b = maps.numel() * 4
    read_b = ctas * V * 32 * (act.element_size() + 4)
    us = min(reps)
    res["kernel"] = {"shape": {"B": xshape[0], "C": a.C, "maps": list(xshape[2:]), "trunk": list(dims)}, "ctas": ctas,
                     "launches_per_rep": args.launches, "us_per_launch_reps": [round(v, 2) for v in reps], "us_per_launch": round(us, 2),
                     "maps_bytes": write_b, "prologue_read_bytes": read_b,
                     "GBps": round((write_b + read_b) / (us * 1e-6) / 1e9, 1),
                     "fraction_of_measured_hbm": round((write_b + read_b) / (us * 1e-6) / 1e9 / MEASURED_HBM_GBS, 3),
                     "note": "back-to-back launches on one stream writing the same 134 MB buffer (larger than the 126 MB L2)"}
    del maps, keep, maps_ref

    # (2) configs[4]-shaped inference with and without a discarding gradcam callback (alternated, best of 2)
    def infer(cb):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        predict_risks(model, batches(wl, args.patients, wl["batch"], dev, 11), dev, gradcam=cb)
        torch.cuda.synchronize()
        return time.perf_counter() - t0

    drop = lambda i, m: None  # noqa: E731
    infer(None); infer(drop)                                   # warm-up
    t_plain, t_maps = [], []
    for _ in range(2):
        t_plain.append(infer(None)); t_maps.append(infer(drop))
    res["inference"] = {"patients": args.patients, "batch": wl["batch"], "workload": wl["name"],
                        "patients_per_s_no_gradcam": round(args.patients / min(t_plain), 1),
                        "patients_per_s_gradcam": round(args.patients / min(t_maps), 1),
                        "seconds_no_gradcam": [round(t, 3) for t in t_plain], "seconds_gradcam": [round(t, 3) for t in t_maps],
                        "note": "predict_risks (eval forward, batch 16, volumes generated on the device per batch inside the timed "
                                "region); gradcam = utils.attention_maps per batch, maps handed to a callback that drops them"}

    # (3) the backward-based MultiModalGradCAM at batch size 1 (it needs a non-blended model: same weights)
    from mmnn_sts_b200.models.densenet import DenseNet121
    from mmnn_sts_b200.models.multimodal import MultiModalModel
    plain = MultiModalModel(DenseNet121(spatial_dims=3, in_channels=wl["cin"], out_channels=2, feature_channels=12, dropout_prob=0.2),
                            ["x"] * 20, 2, 12, blend=False)
    plain.load_state_dict(model.state_dict())
    model = plain.to(dev).eval()
    cam = model.add_gradcam(".")
    one = list(batches(wl, args.old_patients + 2, 1, dev, 13))
    for inputs, _, _ in one[:2]:
        cam(inputs)
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for inputs, _, _ in one[2:]:
        _, m = cam(inputs)
        model.zero_grad(set_to_none=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    res["old_path"] = {"patients": args.old_patients, "patients_per_s": round(args.old_patients / dt, 2),
                       "note": "MultiModalGradCAM (autograd forward + one trunk backward per class), batch size 1, same model"}
    res["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
