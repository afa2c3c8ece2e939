"""Batched GradCAM maps on the GPU (utils.attention_maps -> mmnn_gradcam_maps): the kernel against the float64
restatement oracle/gradcam.py on the kernel's own inputs (read back from the trunk workspace), against the golden maps
of the unchanged reference class, against this package's backward-based MultiModalGradCAM run one sample at a time,
and through inference_survival(gradcam=...)."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden", "gradcam.npz")
TINY_BLOCKS = (6, 12, 4)


def _model(sd, arch="densenet121", cin=1, blend=False):
    from mmnn_sts_b200.models.densenet import DenseNet121, TinyDensenet
    from mmnn_sts_b200.models.multimodal import MultiModalModel
    net = DenseNet121 if arch == "densenet121" else TinyDensenet
    m = MultiModalModel(net(spatial_dims=3, in_channels=cin, out_channels=2, feature_channels=12, dropout_prob=0.0),
                        ["x"] * 20, 2, 12, blend=blend)
    m.load_state_dict(sd)
    return m.cuda().eval()


def _state_dict(seed, arch="densenet121", cin=1):
    from oracle import synth
    if arch == "densenet121":
        return synth.make_state_dict(seed, in_channels=cin)
    return synth.make_state_dict(seed, in_channels=cin, block_config=TINY_BLOCKS)


def _inputs(seed, batch, cin, spatial):
    from oracle import synth
    image, clinical, _, _ = synth.make_batch(seed, batch, cin, spatial)
    return {"image": image.cuda(), "clinical": clinical.cuda()}


def _oracle_on_workspace(m, size):
    """oracle/gradcam.py applied to the activations and trunk output the kernel just read."""
    from oracle import gradcam as og
    bb = m.gradcam_layer
    ws, xshape, (d, h, w), y = bb._last_forward
    act, _ = bb.block_buffer_views(ws, xshape, len(bb._cfg[1]) - 1)
    B, ctot = xshape[0], act.shape[1]
    act = act[:, ctot - 32:].double().reshape(B, d, h, w, 32).permute(0, 4, 1, 2, 3)
    y = y.reshape(B, d, h, w, ctot).permute(0, 4, 1, 2, 3)
    return og.attention_maps(act, y, m.state_dict(), size)


@pytest.mark.parametrize("cin,batch,spatial,trunk", [
    (1, 3, (64, 64, 64), (2, 2, 2)),
    (1, 2, (64, 48, 34), (2, 1, 1)),           # unit trunk dims, Z % 4 != 0 (scalar stores)
    (2, 16, (128, 128, 64), (4, 4, 2)),        # the bench shape
])
def test_kernel_matches_oracle(cin, batch, spatial, trunk):
    from mmnn_sts_b200.utils.utils import attention_maps
    m = _model(_state_dict(61, cin=cin), cin=cin)
    x = _inputs(62, batch, cin, spatial)
    out, maps = attention_maps(m, x)
    assert tuple(m.gradcam_layer._last_forward[2]) == trunk
    assert tuple(maps.shape) == (batch, 2) + spatial and maps.dtype == torch.float32
    ref = _oracle_on_workspace(m, spatial)
    err = float((maps.double() - ref).abs().max())
    print("kernel vs oracle max abs", err, spatial)
    assert err <= 1e-5, err


def test_golden_batch_one():
    """B = 1 on the golden case of the unchanged reference class, with the bounds of the backward-based test."""
    g = np.load(GOLD)
    from mmnn_sts_b200.utils.utils import attention_maps
    from oracle import synth
    sd = synth.make_state_dict(int(g["state_seed"]), in_channels=1)
    image, clinical, _, _ = synth.make_batch(int(g["batch_seed"]), 1, 1, (64, 64, 64))
    m = _model(sd)
    outputs, maps = attention_maps(m, {"image": image.cuda(), "clinical": clinical.cuda()})
    ref_logits = torch.from_numpy(g["logits"])
    assert float((outputs.cpu() - ref_logits).abs().max()) < 2e-2 * float(ref_logits.abs().max()) + 5e-3
    maps = maps[0].cpu()
    ref = torch.from_numpy(g["maps_sub4"])
    sub = maps[:, ::4, ::4, ::4]
    err = float((sub - ref).abs().max())
    print("batched gradcam vs golden max abs", err)
    assert err < 0.05, err
    for c in range(2):
        assert int(sub[c].argmax()) == int(ref[c].argmax())
    np.testing.assert_allclose(maps.mean(dim=(1, 2, 3)).numpy(), g["maps_mean"], atol=0.03)


@pytest.mark.parametrize("arch,spatial", [("densenet121", (64, 64, 64)), ("tiny", (32, 32, 48))])
def test_matches_backward_gradcam_per_sample(arch, spatial):
    """A batch of 3 against MultiModalGradCAM (trunk backward per class) on each sample alone at batch size 1."""
    from mmnn_sts_b200.utils.utils import attention_maps
    m = _model(_state_dict(71, arch), arch)
    x = _inputs(72, 3, 1, spatial)
    _, maps = attention_maps(m, x)
    assert min(m.gradcam_layer._last_forward[2]) >= 2
    cam = m.add_gradcam(".")
    worst = 0.0
    for i in range(3):
        _, ref = cam({"image": x["image"][i:i + 1], "clinical": x["clinical"][i:i + 1]})
        for c in range(2):
            got, want = maps[i, c], ref[c].detach()
            worst = max(worst, float((got - want).abs().max()))
            assert int(got.argmax()) == int(want.argmax()), (i, c)
        m.zero_grad(set_to_none=True)
    print(arch, "batched vs backward GradCAM max abs", worst)
    assert worst <= 1e-2, worst


def test_blended_model_gives_the_multimodal_head_maps():
    from mmnn_sts_b200.utils.utils import attention_maps
    sd = _state_dict(81)
    x = _inputs(82, 2, 1, (64, 64, 64))
    out_b, maps_b = attention_maps(_model(sd, blend=True), x)
    out_p, maps_p = attention_maps(_model(sd), x)
    assert tuple(out_b.shape) == (3, 2, 2) and torch.equal(out_b[0], out_p)
    assert torch.equal(maps_b, maps_p)


def test_inference_survival_with_gradcam_callback():
    from mmnn_sts_b200.main import inference_survival
    from oracle import synth
    m = _model(_state_dict(91))
    batches = []
    for k, bsz in enumerate((4, 4, 3)):
        image, clinical, events, durations = synth.make_batch(92 + k, bsz, 1, (64, 64, 32))
        batches.append(({"image": image, "clinical": clinical}, events, durations))
    seen = []

    def cb(i, maps):
        seen.append((i, tuple(maps.shape), bool(torch.isfinite(maps).all()), float(maps.min()), float(maps.max())))

    dev = torch.device("cuda", 0)
    plain = inference_survival(m, batches, dev, seed=5)
    with_maps = inference_survival(m, batches, dev, seed=5, gradcam=cb)
    assert torch.equal(plain.preds, with_maps.preds)
    np.testing.assert_array_equal(plain.per_resample, with_maps.per_resample)
    np.testing.assert_array_equal(plain.mean, with_maps.mean)
    np.testing.assert_array_equal(plain.std, with_maps.std)
    c_plain, p_plain = inference_survival(m, batches, dev, bootstrap=False)
    c_maps, p_maps = inference_survival(m, batches, dev, bootstrap=False, gradcam=lambda i, maps: None)
    assert c_plain == c_maps and torch.equal(p_plain, p_maps)
    assert [s[0] for s in seen] == [0, 1, 2]
    assert [s[1] for s in seen] == [(4, 2, 64, 64, 32), (4, 2, 64, 64, 32), (3, 2, 64, 64, 32)]
    assert all(s[2] and s[3] >= 0.0 and s[4] <= 1.0 for s in seen), seen


def test_deterministic_and_errors():
    from mmnn_sts_b200 import _lib as L
    from mmnn_sts_b200.ops import gradcam_maps
    from mmnn_sts_b200.utils.utils import attention_maps
    m = _model(_state_dict(101))
    x = _inputs(102, 2, 1, (64, 64, 64))
    _, a = attention_maps(m, x)
    _, b = attention_maps(m, x)
    assert torch.equal(a, b)
    m.train()
    with pytest.raises(ValueError):
        attention_maps(m, x)
    m.eval()
    with pytest.raises(L.MMNNLibraryError):
        attention_maps(m, {k: v.cpu() for k, v in x.items()})
    # C x V cams beyond the kernel's shared memory: 2 classes x 32^3 trunk voxels
    ctot, nf, dims = 64, 12, (32, 32, 32)
    V = dims[0] * dims[1] * dims[2]
    dev = torch.device("cuda", 0)
    adt = torch.float16 if L.lib().mmnn_act_is_fp16() else torch.bfloat16
    with pytest.raises(ValueError, match="shared memory"):
        gradcam_maps(torch.zeros((V, ctot), dtype=adt, device=dev), torch.zeros((V, ctot), device=dev), dims,
                     torch.ones(ctot, device=dev), torch.ones(ctot, device=dev), 1e-5, torch.ones((nf, ctot), device=dev),
                     torch.ones((2, 2 * nf), device=dev), (64, 64, 64))
