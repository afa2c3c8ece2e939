"""Torch restatement (float64 by default) of the batched GradCAM attention maps, from what one eval-mode forward leaves.

TEST INFRASTRUCTURE.  Restates MultiModalGradCAM of the reference (/root/reference/utils/utils.py:253-344) for a whole
batch without its per-class trunk backward:
  * pooled gradient of the hooked conv (last conv2 of the last dense block = the last `growth` channels k' of the
    block's output) in closed form, since that output reaches the logits only through norm5 (eval: fixed affine map)
    -> ReLU -> global average pool -> feature_layer -> output_head (image features first):
        alpha[b][c][k] = (sum_f W_out[c][f] W_feat[f][k']) * gamma5[k'] / sqrt(running_var5[k'] + eps)
                         * count_v(y[b][v][k'] > 0) / V^2
  * the reference's map arithmetic: the activations are re-weighted IN PLACE class after class (class c sees
    alpha[0] * .. * alpha[c]), cam = channel mean, cam -= min, cam /= max, F.interpolate(mode='trilinear',
    align_corners=False) to the volume size -- per sample, with no .squeeze() (a unit trunk dimension works).
Pinned on the CPU against autograd through oracle/model.py and against tests/golden/gradcam.npz
(tests/test_gradcam_batched.py); the GPU tests apply it to the kernel's own inputs.
"""
import torch
import torch.nn.functional as F

PREFIX = "image_model.model."


def pooled_gradients(y, sd, growth=32, eps=1e-5, dtype=torch.float64):
    """alpha [B, C, growth]: d output[b, c] / d block[b, Ctot - growth + k], averaged over the trunk voxels.
    y: the trunk output (norm5 output) NCDHW [B, Ctot, d, h, w]."""
    ctot = y.shape[1]
    ks = slice(ctot - growth, ctot)
    w_feat = sd[PREFIX + "features.feature_layer.weight"].to(dtype)
    nf = w_feat.shape[0]
    w_out = sd["output_head.weight"].to(dtype)[:, :nf]
    head = w_out @ w_feat[:, ks]                                                    # [C, growth]
    bn = PREFIX + "backbone.norm5."
    scale = sd[bn + "weight"].to(dtype)[ks] / torch.sqrt(sd[bn + "running_var"].to(dtype)[ks] + eps)
    V = y[0, 0].numel()
    count = (y[:, ks] > 0).flatten(2).sum(-1).to(dtype)                             # [B, growth]
    return head[None] * scale[None, None] * count[:, None, :] / float(V * V)


def maps_from_alpha(act, alpha, size):
    """act: the hooked conv's output NCDHW [B, growth, d, h, w]; alpha [B, C, growth]; size (X, Y, Z).
    Returns [B, C, X, Y, Z] in alpha's dtype."""
    weighted = act.to(alpha.dtype)
    maps = []
    for c in range(alpha.shape[1]):
        weighted = weighted * alpha[:, c, :, None, None, None]                     # cumulative, as the reference
        cam = weighted.mean(dim=1, keepdim=True)
        cam = cam - cam.amin(dim=(2, 3, 4), keepdim=True)
        cam = cam / cam.amax(dim=(2, 3, 4), keepdim=True)
        maps.append(F.interpolate(cam, size=tuple(size), mode="trilinear")[:, 0])
    return torch.stack(maps, 1)


def attention_maps(act, y, sd, size, growth=32, eps=1e-5, dtype=torch.float64):
    """Batched maps [B, C, X, Y, Z] from (act, y, state_dict): pooled_gradients then maps_from_alpha."""
    return maps_from_alpha(act, pooled_gradients(y, sd, growth, eps, dtype), size)
