"""CPU pins of the batched GradCAM restatement (oracle/gradcam.py) that the GPU tests compare the map kernel with:
its closed-form pooled gradient against autograd through the fp32 oracle network, its maps against the golden maps of
the UNCHANGED reference class (tests/golden/gradcam.npz), and the GradcamArgs ctypes mirror against the library."""
import ctypes
import os

import numpy as np
import pytest
import torch

GOLD = os.path.join(os.path.dirname(__file__), "golden", "gradcam.npz")
NORM5 = "image_model.model.backbone.norm5"


def _trunk_output(block4, sd):
    from oracle import model as om
    return om._bn(block4, dict(sd), NORM5, False)


def test_pooled_gradient_matches_autograd():
    """alpha of oracle.gradcam == the voxel mean of autograd's gradient of output[:, c] w.r.t. block4's last 32
    channels, for B = 2 and both classes; a sample's output has no gradient on the other sample."""
    from oracle import gradcam as og, model as om, synth
    sd = synth.make_state_dict(51, in_channels=1)
    image, clinical, _, _ = synth.make_batch(52, 2, 1, (64, 64, 32))
    col = {}
    out = om.multimodal_forward(dict(sd), image.requires_grad_(True), clinical, False, False, collect=col)
    block4 = col["block4"]
    block4.retain_grad()
    alpha = og.pooled_gradients(_trunk_output(block4, sd).detach(), sd)            # [2, 2, 32] float64
    for c in range(out.shape[1]):
        g, = torch.autograd.grad(out[:, c].sum(), block4, retain_graph=True)
        ref = g[:, -32:].double().mean(dim=(2, 3, 4))                               # [B, 32]
        rel = float((alpha[:, c] - ref).abs().max() / ref.abs().max())
        print("class", c, "pooled-gradient rel err", rel)
        assert rel <= 1e-6, (c, rel)
        g0, = torch.autograd.grad(out[0, c], block4, retain_graph=True)
        assert float(g0[1].abs().max()) == 0.0


def test_oracle_maps_match_reference_golden():
    """The restatement reproduces the maps of the unchanged reference MultiModalGradCAM on its golden case."""
    from oracle import gradcam as og, model as om, synth
    g = np.load(GOLD)
    sd = synth.make_state_dict(int(g["state_seed"]), in_channels=1)
    image, clinical, _, _ = synth.make_batch(int(g["batch_seed"]), 1, 1, (64, 64, 64))
    col = {}
    with torch.no_grad():
        out = om.multimodal_forward(dict(sd), image, clinical, False, False, collect=col)
        y = _trunk_output(col["block4"], sd)
        maps = og.attention_maps(col["block4"][:, -32:], y, sd, (64, 64, 64))[0]
    assert float((out - torch.from_numpy(g["logits"])).abs().max()) <= 1e-6
    assert tuple(maps.shape) == (2, 64, 64, 64)
    err = float((maps[:, ::4, ::4, ::4] - torch.from_numpy(g["maps_sub4"]).double()).abs().max())
    print("oracle maps vs golden max abs err", err)
    assert err <= 1e-6, err


@pytest.fixture(scope="module")
def lib():
    import __graft_entry__ as g
    g.build()
    from mmnn_sts_b200 import _lib
    return _lib.lib()


def test_gradcam_args_size_matches(lib):
    from mmnn_sts_b200 import _lib as L
    assert lib.mmnn_sizeof_gradcam_args() == ctypes.sizeof(L.GradcamArgs)
