"""GPU parity of the 3-D ResNet path (SURVEY.md 8f-3, BASELINE configs[3]) through the C-ABI: per-kernel checks of the
direct convolution (forward / data gradient / weight gradient) for every geometry the network uses, and the whole
network (eval, train without dropout against the reference's golden outputs, train with injected dropout masks against
the oracle).  Tolerances: fp16 storage of every activation and bf16 storage of every gradient tensor against the fp32 oracle."""
import ctypes as C
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import resnet as orn

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
NUM_CLASSES, SPATIAL, BATCH = 5, (12, 32, 24), 3


def _rel(a, b):
    a, b = a.double().cpu(), b.double().cpu()
    return float((a - b).norm() / (b.norm() + 1e-30))


# (Cin, Cout, kernel, stride, pad, input dims): every conv geometry of r3d_18
GEOMS = [
    (1, 64, (1, 7, 7), (1, 2, 2), (1, 3, 3), (5, 20, 18)),
    (64, 8, (3, 3, 3), (1, 1, 1), (1, 1, 1), (6, 9, 10)),
    (64, 8, (1, 1, 1), (1, 1, 1), (0, 0, 0), (6, 9, 10)),
    (8, 8, (3, 3, 3), (1, 1, 1), (1, 1, 1), (7, 8, 9)),
    (8, 8, (3, 3, 3), (1, 1, 1), (1, 1, 1), (3, 7, 37)),
    (64, 8, (3, 3, 3), (1, 1, 1), (1, 1, 1), (3, 5, 35)),
    (8, 16, (3, 3, 3), (2, 2, 2), (1, 1, 1), (7, 8, 9)),
    (8, 16, (1, 1, 1), (2, 2, 2), (0, 0, 0), (7, 8, 9)),
    (16, 16, (3, 3, 3), (1, 1, 1), (1, 1, 1), (4, 5, 6)),
    (16, 16, (3, 3, 3), (1, 1, 1), (1, 1, 1), (3, 11, 21)),
    (16, 8, (3, 3, 3), (2, 2, 2), (1, 1, 1), (6, 5, 8)),
    (16, 8, (1, 1, 1), (2, 2, 2), (0, 0, 0), (6, 5, 8)),
]


@pytest.mark.parametrize("cin,cout,k,s,p,dims", GEOMS)
def test_conv_kernels_match_torch(cin, cout, k, s, p, dims):
    from mmnn_sts_b200 import _lib as L
    lib = L.lib()
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(cin * 100 + cout + k[1])
    N = 2
    x = torch.randn((N, cin) + dims, generator=g)
    w = torch.randn((cout, cin) + k, generator=g) * 0.2
    f32 = cin == 1
    xq = x if f32 else x.half().float()                       # what the kernel reads
    y_ref = F.conv3d(xq, w, None, s, p)
    Do, Ho, Wo = y_ref.shape[2:]
    geom = L.RnConvGeom(N, dims[0], dims[1], dims[2], cin, Do, Ho, Wo, cout, *k, *s, *p)
    x_cl = xq.permute(0, 2, 3, 4, 1).contiguous().to(dev)
    x_dev = x_cl if f32 else x_cl.half()
    w_dev = w.to(dev)
    y = torch.empty((N, Do, Ho, Wo, cout), dtype=torch.float16, device=dev)
    stats = torch.zeros(2 * cout, dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    assert lib.mmnn_rn_conv(C.byref(geom), 0, int(f32), x_dev.data_ptr(), w_dev.data_ptr(), y.data_ptr(), None, stats.data_ptr(), st) == 0
    y_cf = y.float().permute(0, 4, 1, 2, 3).cpu()
    assert (y_cf - y_ref).abs().max() <= 2e-3 * y_ref.abs().max()          # one fp16 rounding of the output
    yr = y.double()
    torch.testing.assert_close(stats[:cout], yr.sum(dim=(0, 1, 2, 3)), rtol=1e-5, atol=1e-4)
    torch.testing.assert_close(stats[cout:], (yr * yr).sum(dim=(0, 1, 2, 3)), rtol=1e-5, atol=1e-4)
    # data gradient (+ fused add) and weight gradient against autograd of the same convolution
    dy = torch.randn(y_ref.shape, generator=g).bfloat16().float()
    xa = xq.clone().requires_grad_(True)
    wa = w.clone().requires_grad_(True)
    F.conv3d(xa, wa, None, s, p).backward(dy)
    dy_dev = dy.permute(0, 2, 3, 4, 1).contiguous().to(dev).bfloat16()
    dw = torch.zeros_like(w_dev)
    assert lib.mmnn_rn_conv_wgrad(C.byref(geom), int(f32), x_dev.data_ptr(), dy_dev.data_ptr(), dw.data_ptr(), st) == 0
    if True:
        # mma.sync wants one operand type: the stem's weight gradient reads the image as bf16 (dy is bf16), the others keep the
        # fp16 activations and rescale dy by a power of two into fp16 (exact) -> one of the two references matches to 1e-4
        xb = xq.bfloat16().float().requires_grad_(False)
        wb_ = w.clone().requires_grad_(True)
        F.conv3d(xb, wb_, None, s, p).backward(dy)
        assert min(_rel(dw, wb_.grad), _rel(dw, wa.grad)) < 1e-4
        assert _rel(dw, wa.grad) < 5e-3
    if not f32:
        add = torch.randn((N,) + dims + (cin,), generator=g).bfloat16()
        dx = torch.empty((N,) + dims + (cin,), dtype=torch.bfloat16, device=dev)
        assert lib.mmnn_rn_conv(C.byref(geom), 1, 0, dy_dev.data_ptr(), w_dev.data_ptr(), dx.data_ptr(), add.to(dev).data_ptr(), None, st) == 0
        ref = xa.grad.permute(0, 2, 3, 4, 1) + add.float()
        assert (dx.float().cpu() - ref).abs().max() <= 1e-2 * ref.abs().max()
        dx.fill_(7.0)                                              # without the fused add (the HMMA 8 -> 64 path takes this form)
        assert lib.mmnn_rn_conv(C.byref(geom), 1, 0, dy_dev.data_ptr(), w_dev.data_ptr(), dx.data_ptr(), None, None, st) == 0
        ref = xa.grad.permute(0, 2, 3, 4, 1)
        assert (dx.float().cpu() - ref).abs().max() <= 1e-2 * ref.abs().max()
        dx.copy_(add)                                              # the add aliasing the output: what the model's strided
        assert lib.mmnn_rn_conv(C.byref(geom), 1, 0, dy_dev.data_ptr(), w_dev.data_ptr(), dx.data_ptr(), dx.data_ptr(), None, st) == 0
        ref = xa.grad.permute(0, 2, 3, 4, 1) + add.float()        # down-sample blocks do, _dgrad(ud, drawd, dx, out=dx)
        assert (dx.float().cpu() - ref).abs().max() <= 1e-2 * ref.abs().max()
    torch.cuda.synchronize()


def test_fused_downsample_pair_matches_separate_calls():
    """mmnn_rn_conv_fwd_ds / mmnn_rn_conv_dgrad_ds (layer1.0: conv1 64 -> 8 3x3x3 + 1x1x1 down-sample on the same input) against
    torch.  Under MMNN_RN_MMA=0 there is no fused kernel: both return -9, and the two separate mmnn_rn_conv calls the model
    then issues (the data gradient's second one in place) are compared with torch instead."""
    from mmnn_sts_b200 import _lib as L
    lib = L.lib()
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(3)
    N, dims = 2, (5, 7, 37)
    x = torch.randn((N, 64) + dims, generator=g).half().float()
    w1 = torch.randn((8, 64, 3, 3, 3), generator=g) * 0.1
    wd = torch.randn((8, 64, 1, 1, 1), generator=g) * 0.3
    geom = L.RnConvGeom(N, *dims, 64, *dims, 8, 3, 3, 3, 1, 1, 1, 1, 1, 1)
    x_dev = x.permute(0, 2, 3, 4, 1).contiguous().to(dev).half()
    y1 = torch.empty((N,) + dims + (8,), dtype=torch.float16, device=dev)
    yd = torch.empty_like(y1)
    s1 = torch.zeros(16, dtype=torch.float64, device=dev)
    sd_ = torch.zeros(16, dtype=torch.float64, device=dev)
    st = torch.cuda.current_stream().cuda_stream
    w1d, wdd = w1.to(dev), wd.to(dev)
    mma = os.environ.get("MMNN_RN_MMA", "1")[:1] != "0"           # csrc/resnet.cu rn_mma_enabled()
    geom_ds = L.RnConvGeom(N, *dims, 64, *dims, 8, 1, 1, 1, 1, 1, 1, 0, 0, 0)
    rc = lib.mmnn_rn_conv_fwd_ds(C.byref(geom), x_dev.data_ptr(), w1d.data_ptr(), wdd.data_ptr(), y1.data_ptr(), yd.data_ptr(),
                                 s1.data_ptr(), sd_.data_ptr(), st)
    assert rc == (0 if mma else -9)
    if not mma:
        assert lib.mmnn_rn_conv(C.byref(geom), 0, 0, x_dev.data_ptr(), w1d.data_ptr(), y1.data_ptr(), None, s1.data_ptr(), st) == 0
        assert lib.mmnn_rn_conv(C.byref(geom_ds), 0, 0, x_dev.data_ptr(), wdd.data_ptr(), yd.data_ptr(), None, sd_.data_ptr(), st) == 0
    r1 = F.conv3d(x, w1, None, 1, 1).permute(0, 2, 3, 4, 1)
    rd = F.conv3d(x, wd, None, 1, 0).permute(0, 2, 3, 4, 1)
    assert (y1.float().cpu() - r1).abs().max() <= 2e-3 * r1.abs().max()
    assert (yd.float().cpu() - rd).abs().max() <= 2e-3 * rd.abs().max()
    torch.testing.assert_close(sd_[:8], yd.double().sum(dim=(0, 1, 2, 3)), rtol=1e-5, atol=1e-4)
    torch.testing.assert_close(sd_[8:], (yd.double() ** 2).sum(dim=(0, 1, 2, 3)), rtol=1e-5, atol=1e-4)
    torch.testing.assert_close(s1[:8], y1.double().sum(dim=(0, 1, 2, 3)), rtol=1e-5, atol=1e-4)
    # data gradient of the pair
    dy1 = torch.randn((N, 8) + dims, generator=g).bfloat16().float()
    dyd = torch.randn((N, 8) + dims, generator=g).bfloat16().float()
    xa = x.clone().requires_grad_(True)
    (F.conv3d(xa, w1.bfloat16().float(), None, 1, 1) * dy1).sum().backward()
    (F.conv3d(xa, wd.bfloat16().float(), None, 1, 0) * dyd).sum().backward()
    dx = torch.empty((N,) + dims + (64,), dtype=torch.bfloat16, device=dev)
    to_cl = lambda t: t.permute(0, 2, 3, 4, 1).contiguous().to(dev).bfloat16()
    dy1_dev, dyd_dev = to_cl(dy1), to_cl(dyd)
    rc = lib.mmnn_rn_conv_dgrad_ds(C.byref(geom), dy1_dev.data_ptr(), w1d.data_ptr(), dyd_dev.data_ptr(), wdd.data_ptr(), dx.data_ptr(), st)
    assert rc == (0 if mma else -9)
    if not mma:
        assert lib.mmnn_rn_conv(C.byref(geom), 1, 0, dy1_dev.data_ptr(), w1d.data_ptr(), dx.data_ptr(), None, None, st) == 0
        assert lib.mmnn_rn_conv(C.byref(geom_ds), 1, 0, dyd_dev.data_ptr(), wdd.data_ptr(), dx.data_ptr(), dx.data_ptr(), None, st) == 0
    ref = xa.grad.permute(0, 2, 3, 4, 1)
    assert (dx.float().cpu() - ref).abs().max() <= 1e-2 * ref.abs().max()
    bad = L.RnConvGeom(N, *dims, 64, *dims, 8, 3, 3, 3, 1, 1, 1, 0, 1, 1)
    assert lib.mmnn_rn_conv_dgrad_ds(C.byref(bad), None, None, None, None, None, st) == -9      # not that pair: caller falls back
    torch.cuda.synchronize()


def _model(dev, sd):
    from mmnn_sts_b200.models.resnet import r3d_18
    m = r3d_18(NUM_CLASSES)
    m.load_state_dict(sd)
    return m.to(dev)


def test_eval_forward_matches_reference_golden():
    dev = torch.device("cuda", 0)
    sd = orn.make_state_dict(7, NUM_CLASSES)
    image, _ = orn.make_batch(11, BATCH, SPATIAL, NUM_CLASSES)
    m = _model(dev, sd).eval()
    with torch.no_grad():
        out = m(image.to(dev)).cpu()
    gold = np.load(os.path.join(GOLD, "resnet_eval.npz"))["out"]
    assert np.abs(out.numpy() - gold).max() < 5e-3                        # sigmoid scores, fp16 activations
    assert int(m.stem[1].num_batches_tracked) == 0


def _train_compare(masks_ncdhw, dropout, batch=BATCH, spatial=SPATIAL, grad_tol=0.2, cos_tol=0.985, training=True):
    """Tolerances: sigmoid scores 5e-3 abs, loss 1e-3 rel (BASELINE north star), gradients by norm-wise relative error and
    cosine against the fp32 oracle.  The default case (3 x 12x32x24) ends in 2x2x2 voxels per sample: BatchNorm over 24 values
    and a gradient that is constant per sample before it make the backward ill-conditioned, which amplifies the bf16
    rounding of the gradient tensors (measured 0.3 % at fc, 6 % at layer4, 8-16 % below, cosine >= 0.99; a larger volume
    measures the same, so it is the bf16 gradient storage, not the tiny BatchNorm populations).  training=False: the model in
    .eval() (running statistics, no dropout) against the oracle's eval forward, backward included."""
    dev = torch.device("cuda", 0)
    sd = orn.make_state_dict(7, NUM_CLASSES)
    image, labels = orn.make_batch(11, batch, spatial, NUM_CLASSES)
    pos_weight = torch.linspace(0.5, 3.0, NUM_CLASSES)
    m = _model(dev, sd).train(training)
    m.dropout.p = 0.2 if dropout else 0.0
    if dropout:
        m.injected_masks = [k.permute(0, 2, 3, 4, 1).contiguous().to(torch.uint8) for k in masks_ncdhw]
    out = m(image.to(dev))
    loss = F.binary_cross_entropy_with_logits(out, labels.to(dev), pos_weight=pos_weight.to(dev), reduction="sum")
    loss.backward()
    p = {k: (v.clone().requires_grad_(True) if v.is_floating_point() and "running" not in k else v.clone()) for k, v in sd.items()}
    ref = orn.resnet_forward(p, image, training=training, masks=masks_ncdhw if dropout else None)
    ref_loss = orn.train_step_loss(ref, labels, pos_weight)
    ref_loss.backward()
    assert (out.detach().cpu() - ref.detach()).abs().max() < 5e-3
    assert abs(loss.item() - ref_loss.item()) < 1e-3 * abs(ref_loss.item())
    named = dict(m.named_parameters())
    worst, worst_cos = 0.0, 1.0
    for k, q in named.items():
        assert q.grad is not None, k
        r = _rel(q.grad, p[k].grad)
        gd, rd = q.grad.double().cpu(), p[k].grad.double()
        cos = float((gd * rd).sum() / (gd.norm() * rd.norm() + 1e-30))
        if q.dim() == 1 and float(rd.norm()) < 0.2:
            # BatchNorm gamma / beta gradients are 8-16 numbers, each a cancelling sum over the whole tensor: the smallest
            # ones (|ref| ~ 0.08 here) sit at the bf16 noise floor of ~0.02 absolute, which also varies run to run with the
            # order of the fp32 atomics through flipped fp16 roundings -> absolute floor instead of a relative bound
            assert float((gd - rd).norm()) < 0.05, (k, r, cos)
            continue
        worst, worst_cos = max(worst, r), min(worst_cos, cos)
        assert r < grad_tol and cos > cos_tol, (k, r, cos)
    msd = m.state_dict()
    if training:
        for k in ("stem.1.running_mean", "stem.1.running_var", "layer2.0.downsample.1.running_var", "layer4.1.conv2.1.running_mean"):
            torch.testing.assert_close(msd[k].cpu(), p[k], rtol=2e-2, atol=2e-3)
        assert int(msd["layer3.0.conv1.1.num_batches_tracked"]) == 1
    else:
        for k in msd:
            if "running" in k:
                assert torch.equal(msd[k].cpu(), sd[k]), k
            elif k.endswith("num_batches_tracked"):
                assert int(msd[k]) == 0, k
    print(f"[resnet {tuple(spatial)} training={training} dropout={dropout}] worst gradient rel-L2 {worst:.3f}, worst cosine {worst_cos:.4f}")
    return out.detach().cpu(), loss.item(), named, worst


def test_train_step_matches_reference_golden_and_oracle():
    # 2x2x2 voxels per sample in layer4: one flipped ReLU there moves every gradient below it -> loose gradient bounds here,
    # the well-conditioned bounds are asserted by test_train_step_larger_volume
    out, loss, named, worst = _train_compare(None, False, grad_tol=0.2, cos_tol=0.975)
    gold = np.load(os.path.join(GOLD, "resnet_train.npz"))
    assert np.abs(out.numpy() - gold["out"]).max() < 5e-3
    assert abs(loss - float(gold["loss"])) < 1e-3 * abs(float(gold["loss"]))
    for k in gold.files:
        if k.startswith("grad:"):
            assert _rel(named[k[5:]].grad, torch.from_numpy(gold[k])) < 0.5 or np.linalg.norm(gold[k]) < 0.2, k
    print(f"worst relative gradient error {worst:.3e}")


def test_train_step_larger_volume():
    g = torch.Generator().manual_seed(6)
    masks = [(torch.rand(s, generator=g) >= 0.2).float() for s in orn.stage_shapes(4, (20, 96, 64))]
    # Round 1 had to allow 0.45 / cosine 0.9 here because the worst tensor moved by 0.10-0.25 BETWEEN RUNS of the same input: the
    # BatchNorm statistics were summed with shared-memory atomics, a last-bit difference flipped an fp16 rounding, that flipped a
    # ReLU, and the bf16 gradient chain amplified it.  The statistics are now summed in a fixed order (RN_WARP_ORDERED, resnet.cu):
    # the forward pass is bit-reproducible and this case measures 0.181 every run -> bound 0.25 / cosine 0.96.
    *_, worst = _train_compare(masks, True, batch=4, spatial=(20, 96, 64), grad_tol=0.25, cos_tol=0.96)
    print(f"worst relative gradient error {worst:.3e}")


def test_eval_backward_matches_oracle():
    # .eval(): BatchNorm from the running statistics (mmnn_rn_bn_bwd_apply eval_mode 1), no dropout, nothing updated
    _train_compare(None, False, training=False)


def test_train_step_with_injected_dropout_masks():
    g = torch.Generator().manual_seed(5)
    masks = [(torch.rand(s, generator=g) >= 0.2).float() for s in orn.stage_shapes(BATCH, SPATIAL)]
    _train_compare(masks, True, grad_tol=0.3, cos_tol=0.95)


def test_hashed_dropout_statistics():
    from mmnn_sts_b200 import _lib as L
    dev = torch.device("cuda", 0)
    n, Cc = 1 << 20, 8
    raw = torch.ones((n, Cc), dtype=torch.float16, device=dev)
    coef = torch.tensor([[1.0] * Cc, [0.0] * Cc, [0.0] * Cc, [1.0] * Cc], device=dev)
    y = torch.empty_like(raw)
    st = torch.cuda.current_stream().cuda_stream
    assert L.lib().mmnn_rn_bn_act(raw.data_ptr(), coef.data_ptr(), 0, None, None, y.data_ptr(), raw.numel(), Cc, 1, 0.2, 12345, None, st) == 0
    kept = (y > 0).float().mean().item()
    assert abs(kept - 0.8) < 2e-3
    assert abs(float(y.float().max()) - 1.25) < 1e-2
    y2 = torch.empty_like(raw)
    assert L.lib().mmnn_rn_bn_act(raw.data_ptr(), coef.data_ptr(), 0, None, None, y2.data_ptr(), raw.numel(), Cc, 1, 0.2, 54321, None, st) == 0
    assert 0.6 < ((y > 0) == (y2 > 0)).float().mean().item() < 0.76      # independent masks agree on 0.68 of the elements


def test_train_classification_driver_with_resnet():
    """mmnn_sts_b200.main.train_classification (mirror of /root/reference/main.py:125-327) around r3d_18: image-only, no blend,
    optimiser step every batch, F1 from the thresholded sigmoid of the outputs; the parameters move, the loss stays finite."""
    from types import SimpleNamespace
    from mmnn_sts_b200.main import train_classification
    from mmnn_sts_b200.models.resnet import r3d_18
    dev = torch.device("cuda", 0)
    torch.manual_seed(3)
    m = r3d_18(3)
    before = {k: v.clone() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(9)
    mk = lambda n: [(torch.rand((4, 1, 8, 32, 32), generator=g), (torch.rand((4, 3), generator=g) < 0.4).float()) for _ in range(n)]
    args = SimpleNamespace(lr=1e-2, momentum=0.9, weight_decay=1e-4, epochs=2, batch_size=4, blend=False, blend_update_interval=5,
                           class_freqs=[0.3, 0.4, 0.5], num_train=12, multimodal=False)
    hist = train_classification(m, mk(3), mk(2), args, dev)
    assert len(hist.train_loss) == 2 and all(np.isfinite(hist.train_loss)) and all(np.isfinite(hist.val_loss))
    assert len(hist.val_f1) == 2 and 0.0 <= hist.best_metric <= 1.0 and hist.best_state is not None
    after = m.state_dict()
    assert any(not torch.equal(before[k].to(dev), after[k]) for k in before if k.endswith("0.weight"))
    assert int(after["stem.1.num_batches_tracked"]) == 6


def test_forward_is_bit_reproducible_and_gradients_stable():
    """Two runs of the same training step: sigmoid scores, loss, running statistics and every BatchNorm-parameter gradient are
    bit-identical (fixed-order statistics); the convolution weight gradients -- still accumulated across thread blocks with fp32
    atomics on this path -- agree to 1e-5 of their norm (no feedback into the step: only their own last bits move)."""
    dev = torch.device("cuda", 0)
    sd = orn.make_state_dict(7, NUM_CLASSES)
    image, labels = orn.make_batch(13, 4, (20, 96, 64), NUM_CLASSES)
    g = torch.Generator().manual_seed(6)
    masks = [(torch.rand(s, generator=g) >= 0.2).float() for s in orn.stage_shapes(4, (20, 96, 64))]
    runs = []
    for _ in range(2):
        m = _model(dev, sd).train()
        m.dropout.p = 0.2
        m.injected_masks = [k.permute(0, 2, 3, 4, 1).contiguous().to(torch.uint8) for k in masks]
        out = m(image.to(dev))
        loss = F.binary_cross_entropy_with_logits(out, labels.to(dev), reduction="sum")
        loss.backward()
        torch.cuda.synchronize()
        runs.append((out.detach().clone(), loss.detach().clone(), {k: q.grad.clone() for k, q in m.named_parameters()},
                     {k: v.clone() for k, v in m.state_dict().items() if "running" in k}))
    a, b = runs
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    for k in a[3]:
        assert torch.equal(a[3][k], b[3][k]), k
    for k in a[2]:
        if a[2][k].dim() == 1:
            assert torch.equal(a[2][k], b[2][k]), k                       # BatchNorm gamma / beta, fc bias
        else:
            assert float((a[2][k] - b[2][k]).norm()) <= 1e-5 * float(a[2][k].norm()) + 1e-12, k
