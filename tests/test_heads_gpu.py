"""GPU parity of the small kernels (clinical MLP + fusion heads, Cox loss, concordance index, GradientBlender)
through the reference-shaped Python API against the CPU oracle and the committed golden vectors.  fp32 kernels:
tolerance 1e-5 relative (summation order); integer work (C-index pair counts) bit-exact."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _golden(name):
    return np.load(os.path.join(os.path.dirname(__file__), "golden", name + ".npz"))


def _close(a, b, rtol=2e-5, atol=2e-6):
    a = torch.as_tensor(a).double().cpu(); b = torch.as_tensor(b).double().cpu()
    assert torch.allclose(a, b, rtol=rtol, atol=atol), f"max abs diff {float((a - b).abs().max())}, ref max {float(b.abs().max())}"


@pytest.mark.parametrize("training,blend,batch", [(True, True, 4), (True, False, 16), (False, True, 5), (True, True, 64)])
def test_mlp_heads_vs_oracle(training, blend, batch):
    from mmnn_sts_b200.models.densenet import DenseNet121
    from mmnn_sts_b200.models.multimodal import MultiModalModel
    from mmnn_sts_b200.ops import MLPHeads
    from oracle import model as om, synth
    import torch.nn.functional as F
    sd = synth.make_state_dict(11)
    _, clinical, _, _ = synth.make_batch(5, batch, 1, (1, 1, 1))
    g = torch.Generator().manual_seed(3)
    img_f = torch.randn(batch, 12, generator=g)
    gw = torch.randn(3 if blend else 1, batch, 2, generator=g)
    masks = synth.make_masks(9, batch) if training else None
    # oracle
    p = {k: (v.clone().requires_grad_(True) if v.dtype.is_floating_point and "running" not in k else v.clone()) for k, v in sd.items()}
    imf = img_f.clone().requires_grad_(True)
    cf = om.mlp_features(p, clinical, training, masks, "clinical_model.model.")
    feats = torch.cat([imf, cf], 1)
    out = F.linear(feats, p["output_head.weight"], p["output_head.bias"])
    if blend:
        out = torch.stack((out, F.linear(imf, p["image_output_head.weight"], p["image_output_head.bias"]),
                           F.linear(cf, p["clinical_output_head.weight"], p["clinical_output_head.bias"])), 0)
    else:
        out = out[None]
    (out * gw).sum().backward()
    # build
    m = MultiModalModel(DenseNet121(spatial_dims=3, in_channels=2, out_channels=2, feature_channels=12), ["x"] * 20, 2, 12, blend=blend)
    m.load_state_dict(sd)
    m = m.cuda().train(training)
    mlp = m.clinical_model.model
    if training:
        mlp.injected_masks = torch.stack(masks["mlp"])
    params, buffers = mlp.kernel_params()
    heads = [m.output_head.weight, m.output_head.bias, m.image_output_head.weight, m.image_output_head.bias,
             m.clinical_output_head.weight, m.clinical_output_head.bias]
    imf_g = img_f.cuda().requires_grad_(True)
    preds = MLPHeads.apply(clinical.cuda(), imf_g, mlp.sample_masks(batch, "cuda"), (training, blend, 2), buffers, *params, *heads)
    (preds * gw.cuda()).sum().backward()
    _close(preds, out.detach(), 1e-4, 1e-5)
    _close(imf_g.grad, imf.grad, 1e-3, 1e-5)
    for k, q in m.named_parameters():
        if k.startswith("image_model") or "dense6" in k:
            continue
        ref = p[k].grad
        if ref is None:
            assert q.grad is None, k
        else:
            _close(q.grad, ref, 2e-3, 2e-5)
    if training:
        for k in ["clinical_model.model.backbone.bn0", "clinical_model.model.features.bn5"]:
            _close(m.state_dict()[k + ".running_mean"], p[k + ".running_mean"], 1e-5, 1e-6)
            _close(m.state_dict()[k + ".running_var"], p[k + ".running_var"], 1e-4, 1e-6)
            assert int(m.state_dict()[k + ".num_batches_tracked"]) == 1


def test_mlp_batch_of_one_raises_like_torch():
    from mmnn_sts_b200.models.densenet import DenseNet121
    from mmnn_sts_b200.models.multimodal import MultiModalModel
    m = MultiModalModel(DenseNet121(spatial_dims=3, in_channels=1, out_channels=2, feature_channels=12), ["x"] * 20, 2, 12).cuda().train()
    with pytest.raises(ValueError, match="Expected more than 1 value per channel"):
        m({"image": torch.rand(1, 1, 32, 32, 32, device="cuda"), "clinical": torch.rand(1, 20, device="cuda")})


def test_cox_kats_and_golden():
    from mmnn_sts_b200.losses.losses import CoxPH, CoxPH_intended
    from oracle import cox
    k = _golden("kats")
    l = CoxPH_intended(torch.tensor([0.5, -1, 2, 0.], device="cuda"), torch.tensor([1, 0, 1, 1], device="cuda"), torch.tensor([4, 3, 2, 1], device="cuda"))
    assert abs(l.item() - 0.86122042) < 5e-7                       # KAT-A
    l = CoxPH(torch.tensor([0.3, -0.7], device="cuda"), torch.tensor([0, 1], device="cuda"), torch.tensor([10, 20], device="cuda"))
    assert abs(l.item() - 0.10442076809345666) < 5e-7               # KAT-B (as written)
    for n in (2, 4, 16, 64, 1000):
        h = torch.tensor(k[f"cox{n}_h"], device="cuda", requires_grad=True)
        e = torch.tensor(k[f"cox{n}_e"], device="cuda"); d = torch.tensor(k[f"cox{n}_d"], device="cuda")
        l = CoxPH_intended(h, e, d); l.backward()                   # tie-free: equals the stored reference-side run
        assert abs(l.item() - float(k[f"cox{n}_intended_loss"])) < 2e-5 * max(1, abs(l.item()))
        assert np.abs(h.grad.cpu().numpy() - k[f"cox{n}_intended_grad"]).max() < 2e-5
        # as written (binary sort key): stable tie order == oracle restatement with stable sort
        h2 = torch.tensor(k[f"cox{n}_h"], device="cuda", requires_grad=True)
        l2 = CoxPH(h2, e, d); l2.backward()
        ln, gn = cox.cox_np(k[f"cox{n}_h"], k[f"cox{n}_e"], k[f"cox{n}_d"])
        assert abs(l2.item() - ln) < 3e-5 * max(1, abs(ln))
        assert np.abs(h2.grad.cpu().numpy() - gn).max() < 3e-5


@pytest.mark.parametrize("n,ties", [(1, False), (3, True), (257, True), (4096, False), (10000, True)])
def test_cox_random_vs_oracle(n, ties):
    from mmnn_sts_b200.ops import cox_ph_segments
    from oracle import cox
    rng = np.random.RandomState(n)
    S = 3
    h = rng.randn(S, n).astype(np.float32)
    key = rng.randint(1, 50 if ties else 10 ** 6, (S, n)) if ties else np.stack([rng.permutation(10 ** 6)[:n] for _ in range(S)])
    w = rng.randint(0, 2, (S, n)); w[:, 0] = 1
    ht = torch.tensor(h, device="cuda", requires_grad=True)
    loss = cox_ph_segments(ht, torch.tensor(key, device="cuda"), torch.tensor(w, device="cuda"))
    loss.sum().backward()
    for s in range(S):
        ln, gn = cox.cox_np(h[s], key[s], w[s])
        assert abs(loss[s].item() - ln) < 1e-4 * max(1, abs(ln)), (s, loss[s].item(), ln)
        assert np.abs(ht.grad[s].cpu().numpy() - gn).max() < 1e-4 * max(1e-3, np.abs(gn).max()) + 1e-6


def test_cox_no_event_is_nan_like_pycox():
    from mmnn_sts_b200.losses.losses import CoxPH_intended
    l = CoxPH_intended(torch.randn(5, device="cuda"), torch.zeros(5, device="cuda"), torch.arange(5, device="cuda"))
    assert torch.isnan(l)


def test_surv_criterion_and_blender_match_oracle():
    from mmnn_sts_b200.losses.GradientBlender import GradientBlender
    from mmnn_sts_b200.losses.losses import CoxPH
    from mmnn_sts_b200.utils.utils import surv_criterion
    from oracle import cox
    from oracle.blender import GradientBlenderOracle
    k = _golden("kats")
    rng = np.random.RandomState(0)
    preds = torch.tensor(rng.randn(3, 16, 2), dtype=torch.float32)
    ev = torch.tensor(rng.randint(0, 2, (16, 2))); du = torch.tensor(np.stack([rng.permutation(3650)[:16] + 1 for _ in range(2)], 1))
    ref = cox.surv_criterion(cox.CoxPH, preds[0], ev, du)
    got = surv_criterion(CoxPH, preds[0].cuda(), ev.cuda(), du.cuda(), "cuda")
    assert abs(got.item() - ref.item()) < 2e-5 * abs(ref.item())
    gb, go = GradientBlender(CoxPH, survival=True, surv_criterion=surv_criterion), GradientBlenderOracle()
    pc = preds.cuda().requires_grad_(True); po = preds.clone().requires_grad_(True)
    l, h0 = gb.computeLoss(pc, ev.cuda(), du.cuda()); lo, h0o = go.computeLoss(po, ev, du)
    assert np.allclose(gb.weights.cpu().numpy(), [1 / 3] * 3)
    assert abs(l.item() - lo.item()) < 2e-5 * abs(lo.item()) and abs(h0.item() - h0o.item()) < 2e-5 * abs(h0o.item())
    l.backward(); lo.backward()
    assert (pc.grad.cpu() - po.grad).abs().max() < 1e-5
    for it in range(3):   # KAT-E sequence: uniform, uniform, softmax(dG/dO^2)
        a = [torch.tensor(k[f"gb{it}_{s}"]) for s in ("tp", "te", "td", "vp", "ve", "vd")]
        gb.updateWeights(*[t.cuda() for t in a]); go.updateWeights(*a)
        assert np.allclose(gb.weights.cpu().numpy(), go.weights.numpy(), rtol=2e-3, atol=1e-5), (it, gb.weights, go.weights)
    assert np.allclose(gb.history[0], [1 / 3] * 3)


def test_cindex_counts_bit_exact():
    from mmnn_sts_b200.ops import concordance_counts
    from oracle import cindex
    k = _golden("kats")
    for n in (6, 64, 500):
        t, p, e = k[f"ci{n}_t"], k[f"ci{n}_p"], k[f"ci{n}_e"]
        c = concordance_counts(torch.tensor(t, device="cuda"), torch.tensor(p, device="cuda"), torch.tensor(e, device="cuda"))
        assert tuple(int(v) for v in c[0].cpu()) == tuple(int(v) for v in k[f"ci{n}_counts"])
    rng = np.random.RandomState(5)
    n = 3000
    t = rng.randint(1, 400, n); p = np.round(rng.randn(n), 2).astype(np.float32); e = rng.randint(0, 2, n)
    idx = rng.randint(0, n, (7, n))
    c = concordance_counts(torch.tensor(t, device="cuda"), torch.tensor(p, device="cuda"), torch.tensor(e, device="cuda"), torch.tensor(idx, device="cuda")).cpu().numpy()
    for r in range(7):
        assert tuple(c[r]) == cindex.concordance_counts(t[idx[r]], p[idx[r]], e[idx[r]]), r
    # all censored -> no admissible pair
    c = concordance_counts(torch.tensor(t, device="cuda"), torch.tensor(p, device="cuda"), torch.zeros(n, device="cuda"))
    assert int(c[0, 2]) == 0


@pytest.mark.gpu
def test_fused_sgd_matches_torch_sgd():
    """mmnn_sts_b200.optim.SGD (one launch) against torch.optim.SGD (the reference's optimiser, main.py:410-414) over
    three steps with OneCycleLR cycling lr and momentum, odd sizes and unaligned gradient views."""
    from mmnn_sts_b200.optim import SGD
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(5)
    shapes = [(128, 64, 1, 1, 1), (64,), (32, 128, 3, 3, 3), (3,), (17, 5), (100003,), (12,)]
    pa = [torch.randn(s, device=dev, generator=g).requires_grad_(True) for s in shapes]
    pb = [p.detach().clone().requires_grad_(True) for p in pa]
    oa = torch.optim.SGD(pa, 5e-2, momentum=0.9, nesterov=True, weight_decay=1e-2)
    ob = SGD(pb, 5e-2, momentum=0.9, nesterov=True, weight_decay=1e-2)
    sa = torch.optim.lr_scheduler.OneCycleLR(oa, max_lr=5e-2, total_steps=4)
    sb = torch.optim.lr_scheduler.OneCycleLR(ob, max_lr=5e-2, total_steps=4)
    for step in range(3):
        total = sum(p.numel() for p in pa)
        flat = torch.randn(total + 1, device=dev, generator=g)[1:]        # 4-byte aligned only: scalar path for every view
        off = 0
        for a, b in zip(pa, pb):
            gr = flat[off:off + a.numel()].view(a.shape) if step == 1 else torch.randn(a.shape, device=dev, generator=g)
            off += a.numel()
            if a is pa[3] and step == 0:
                a.grad = None; b.grad = None                                 # a parameter without gradient is skipped
                continue
            a.grad = gr.clone(); b.grad = gr if step == 1 else gr.clone()
        oa.step(); ob.step(); sa.step(); sb.step()
        for a, b in zip(pa, pb):
            torch.testing.assert_close(b, a, rtol=2e-6, atol=2e-6)
    for a, b in zip(pa, pb):
        if "momentum_buffer" in oa.state[a]:
            torch.testing.assert_close(ob.state[b]["momentum_buffer"], oa.state[a]["momentum_buffer"], rtol=2e-6, atol=2e-6)
    assert set(ob.state_dict()["param_groups"][0].keys()) == set(oa.state_dict()["param_groups"][0].keys())


@pytest.mark.gpu
def test_fused_sgd_survives_state_dict_round_trip_and_moved_tensors():
    """step -> optimizer.load_state_dict(optimizer.state_dict()) (replaces every momentum tensor) -> `p.data = ...` (moves a
    parameter without changing id(p)) -> step: the cached pointer tables must follow (they are keyed on the addresses)."""
    from mmnn_sts_b200.optim import SGD
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(9)
    shapes = [(64, 32), (7,), (4097,)]
    pa = [torch.randn(s, device=dev, generator=g).requires_grad_(True) for s in shapes]
    pb = [p.detach().clone().requires_grad_(True) for p in pa]
    oa = torch.optim.SGD(pa, 1e-1, momentum=0.9, nesterov=True, weight_decay=1e-3)
    ob = SGD(pb, 1e-1, momentum=0.9, nesterov=True, weight_decay=1e-3)

    def one_step():
        for a, b in zip(pa, pb):
            a.grad = torch.randn(a.shape, device=dev, generator=g); b.grad = a.grad.clone()
        oa.step(); ob.step()
        for a, b in zip(pa, pb):
            torch.testing.assert_close(b, a, rtol=2e-6, atol=2e-6)

    one_step()
    import copy
    oa.load_state_dict(copy.deepcopy(oa.state_dict())); ob.load_state_dict(copy.deepcopy(ob.state_dict()))
    one_step()
    for b in pb:
        b.data = b.data.clone()            # new storage, same Parameter object
    one_step()
    for a, b in zip(pa, pb):
        torch.testing.assert_close(ob.state[b]["momentum_buffer"], oa.state[a]["momentum_buffer"], rtol=2e-6, atol=2e-6)


@pytest.mark.gpu
def test_captured_sgd_follows_the_scheduler_and_scalar_capture_is_refused():
    """A CUDA-graph replay of SGD(capturable=True).step() reads lr / momentum / weight decay from device memory: with OneCycleLR
    stepped between replays it matches the eager torch optimiser; a non-capturable SGD refuses to be captured."""
    from mmnn_sts_b200.optim import SGD
    dev = torch.device("cuda", 0)
    g = torch.Generator(device=dev).manual_seed(11)
    pa = [torch.randn(s, device=dev, generator=g).requires_grad_(True) for s in [(33, 5), (1000,)]]
    pb = [p.detach().clone().requires_grad_(True) for p in pa]
    grads = [torch.zeros_like(p) for p in pb]
    for b, gr in zip(pb, grads):
        b.grad = gr
    oa = torch.optim.SGD(pa, 5e-2, momentum=0.9, nesterov=True, weight_decay=1e-2)
    ob = SGD(pb, 5e-2, momentum=0.9, nesterov=True, weight_decay=1e-2, capturable=True)
    sa = torch.optim.lr_scheduler.OneCycleLR(oa, max_lr=5e-2, total_steps=8)
    sb = torch.optim.lr_scheduler.OneCycleLR(ob, max_lr=5e-2, total_steps=8)
    fresh = [torch.randn(p.shape, device=dev, generator=g) for p in pa]
    for a, b, gr, f in zip(pa, pb, grads, fresh):
        a.grad = f.clone(); gr.copy_(f)
    oa.step(); ob.step(); sa.step(); sb.step()          # eager warm-up step (allocates momentum + device hyper-parameters)
    side = torch.cuda.Stream(); side.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(side):
        with torch.cuda.graph(graph, stream=side):
            ob.step()
    # the capture itself does not execute: parameters still equal
    for step in range(4):
        fresh = [torch.randn(p.shape, device=dev, generator=g) for p in pa]
        for a, gr, f in zip(pa, grads, fresh):
            a.grad = f.clone(); gr.copy_(f)
        oa.step(); sa.step()
        ob.refresh_hyper(); graph.replay(); sb.step()
        torch.cuda.synchronize()
        for a, b in zip(pa, pb):
            torch.testing.assert_close(b, a, rtol=3e-6, atol=3e-6)
    oc = SGD([torch.randn(8, device=dev).requires_grad_(True)], 1e-2, momentum=0.9)
    oc.param_groups[0]["params"][0].grad = torch.ones(8, device=dev)
    oc.step()
    g2 = torch.cuda.CUDAGraph()
    with pytest.raises(RuntimeError, match="capturable"):
        with torch.cuda.stream(side):
            with torch.cuda.graph(g2, stream=side):
                oc.step()


@pytest.mark.gpu
@pytest.mark.parametrize("training", [True, False])
def test_clinical_only_mlp_forward(training):
    """MLP.forward of the reference (/root/reference/models/mlp.py:57-63): output_head(features(backbone(x))), forward and
    gradients against the oracle's restatement of the same layers (dropout masks injected)."""
    import torch.nn.functional as F
    from mmnn_sts_b200.models.mlp import MLP
    from oracle import model as om, synth
    sd = synth.make_state_dict(42, in_channels=1)
    pfx = "clinical_model.model."
    sub = {k[len(pfx):]: v for k, v in sd.items() if k.startswith(pfx)}
    m = MLP(20, 2, 12).cuda().train(training)
    m.load_state_dict(sub)
    _, clinical, _, _ = synth.make_batch(21, 16, 1, (8, 8, 8))
    masks = synth.make_masks(5, 16)
    m.injected_masks = torch.stack(masks["mlp"])
    out = m(clinical.cuda())
    p = {k: (v.clone().requires_grad_(True) if v.dtype.is_floating_point and "running" not in k else v.clone()) for k, v in sd.items()}
    f = om.mlp_features(p, clinical, training, masks if training else None, pfx)
    ref = F.linear(f, p[pfx + "output_head.dense6.weight"], p[pfx + "output_head.dense6.bias"])
    assert out.shape == ref.shape == (16, 2)
    torch.testing.assert_close(out.detach().cpu(), ref.detach(), rtol=2e-5, atol=2e-5)
    if training:
        gw = torch.randn(16, 2, generator=torch.Generator().manual_seed(3))
        (out * gw.cuda()).sum().backward(); (ref * gw).sum().backward()
        for k, q in m.named_parameters():
            torch.testing.assert_close(q.grad.cpu(), p[pfx + k].grad, rtol=2e-4, atol=2e-5)


def _within(got, ref, tol, what):
    err = (got.double().cpu() - ref).abs()
    assert bool((err <= tol).all()), f"{what}: worst excess {float((err - tol).max()):.3e}, max |ref| {float(ref.abs().max()):.3e}"


@pytest.mark.parametrize("masked", [False, True])
@pytest.mark.parametrize("B,Cc,V,F", [(1, 1024, 8, 12), (3, 70, 1, 40), (17, 1024, 27, 12), (2, 64, 4096, 3)])
def test_gap_linear_vs_float64(B, Cc, V, F, masked):
    """DenseNet feature head (ops.GapLinearDropout: ReLU -> mean over the volume -> Linear -> dropout mask) against float64
    autograd of Linear(mean_v relu(x)) * mask: the forward and the gradients of x, W and b at 1e-5 of the sum of the absolute
    terms (fp32 kernels), the ReLU mask of dx exact.  C = 70 is not a multiple of the 32-lane stride, F = 40 is more features
    than the block's 8 warps."""
    from mmnn_sts_b200.ops import GapLinearDropout
    import torch.nn.functional as Fn
    g = torch.Generator().manual_seed(B * 1000 + V + F)
    side = {1: (1, 1, 1), 8: (2, 2, 2), 27: (3, 3, 3), 4096: (16, 16, 16)}[V]
    x = torch.randn((B, Cc) + side, generator=g)
    W = torch.randn((F, Cc), generator=g) * 0.05
    b = torch.randn(F, generator=g) * 0.1
    mask = (torch.rand((B, F), generator=g) >= 0.3).float() / 0.7 if masked else None
    if masked:
        mask[0, 0] = 0.0                                 # at least one zero
    gout = torch.randn((B, F), generator=g)
    xd, Wd, bd = (t.cuda().requires_grad_(True) for t in (x, W, b))
    out = GapLinearDropout.apply(xd, Wd, bd, mask.cuda() if masked else None)
    (out * gout.cuda()).sum().backward()
    x64, W64, b64 = (t.double().requires_grad_(True) for t in (x, W, b))
    m64 = mask.double() if masked else torch.ones((B, F), dtype=torch.float64)
    pooled = x64.clamp_min(0.0).mean(dim=(2, 3, 4))
    ref = Fn.linear(pooled, W64, b64) * m64
    (ref * gout.double()).sum().backward()
    pooled, m64, g64 = pooled.detach(), m64, gout.double()
    gm = g64 * m64
    _within(out.detach(), ref.detach(), 1e-5 * (pooled.abs() @ W64.detach().abs().T + b64.detach().abs()) * m64.abs(), "out")
    # dx = [x > 0] * (g * mask) W / V: exactly zero where x <= 0
    dxk = xd.grad.cpu()
    assert bool((dxk[x <= 0] == 0).all())
    dx_abs = (gm.abs() @ W64.detach().abs() / V)[:, :, None, None, None].expand_as(x64)
    pos = x > 0
    _within(dxk[pos], x64.grad[pos], 1e-5 * dx_abs[pos], "dx")
    _within(Wd.grad, W64.grad, 1e-5 * (gm.abs().T @ pooled.abs()), "dW")
    _within(bd.grad, b64.grad, 1e-5 * gm.abs().sum(0), "db")
