"""Hot-path helpers with the reference's names and argument meaning (/root/reference/utils/utils.py:20-29,238-251)."""
import torch
import torch.nn as nn
import torch.nn.functional as F


def criterion(loss_func, preds, labels, device):
    return loss_func(preds, labels).to(device)


def surv_criterion(loss_func, preds, events, durations, device):
    """SUM over classes of loss_func(preds[:, i], events[:, i], durations[:, i]) (/root/reference/utils/utils.py:24-29).
    When loss_func is this package's CoxPH all classes go to the GPU in ONE launch (one segment per class)."""
    from ..losses.losses import CoxPH, _coxph_columns
    if loss_func is CoxPH and preds.is_cuda:
        return _coxph_columns(preds, events, durations).sum().to(device)
    losses = 0
    for i in range(preds.shape[1]):
        losses += loss_func(preds[:, i], events[:, i], durations[:, i]).to(device)
    return losses


class BackpropagatableFeatureExtractor(nn.Module):
    """features(backbone(x)) of a model split into `backbone` and `features` (/root/reference/utils/utils.py:238-251)."""

    def __init__(self, model):
        super().__init__()
        self.model = model

    def forward(self, x):
        x = self.model.backbone(x)
        return self.model.features(x)


def remap_bhb_checkpoint(checkpoint):
    """State-dict keys of the BHB-10K yAware-contrastive DenseNet121 checkpoint renamed to this package's (= the
    reference's MONAI-style) layout.  Same mapping as /root/reference/utils/utils.py:373-382: the DataParallel prefix
    `module.` goes away, and the dense layers of that checkpoint (`features.denseblockB.denselayerL.<leaf>`) gain the
    `layers` container level (`features.denseblockB.denselayerL.layers.<leaf>`).  `checkpoint` is the loaded file, a
    dict whose 'model' entry is the state_dict."""
    def rename(key):
        parts = key.replace('module.', '').split('.')
        in_dense_block = len(parts) > 1 and parts[0] == 'features' and parts[1].startswith('dense')
        if in_dense_block:
            parts = parts[:3] + ['layers'] + parts[3:]
        return '.'.join(parts)

    return {rename(key): tensor for key, tensor in checkpoint['model'].items()}


def loadWeights(model, path, device):
    """`loadWeights` of the reference (/root/reference/utils/utils.py:357-390) without the S3 branch (storage is out of
    scope, DESIGN.md section 9): a plain state_dict loads strictly; the BHB pretrained backbone is remapped and loaded
    with strict=False (it has no classification head).  Works because the parameter containers of
    mmnn_sts_b200.models keep the reference's state_dict keys and shapes."""
    try:
        checkpoint = torch.load(path, map_location=device)
        model.load_state_dict(checkpoint)
    except Exception as e1:
        if str(path).endswith('DenseNet121_BHB-10K_yAwareContrastive.pth'):
            checkpoint = torch.load(path, map_location=device)
            model.load_state_dict(remap_bhb_checkpoint(checkpoint), strict=False)
        else:
            raise e1
    return model


class MultiModalGradCAM(nn.Module):
    """GradCAM of the reference (/root/reference/utils/utils.py:253-344) on the fused trunk (SURVEY.md section 8f rank 4).

    The reference hooks the LAST nn.Conv3d of `model.gradcam_layer` (= denseblock4.denselayer16.layers.conv2) for its
    output and the gradient of that output.  Here the trunk is one fused call, so both are read from its workspace: the
    conv's output is the last 32 channels of the final dense block's buffer, its gradient the same channels of that
    block's fp32 gradient accumulator after a backward pass (mmnn_encoder_debug_offsets).  Everything else follows the
    reference line by line -- including that the activations are scaled IN PLACE class after class (:306-307), so the
    map of class c carries the pooled gradients of classes 0..c -- and that only batch size 1 is accepted (:330).
    The model must be in eval mode (the reference calls it from inference_survival) on a CUDA device."""

    def __init__(self, model):
        super().__init__()
        self.model = model
        self.input_shape = None

    def forward(self, x):
        outputs = self.model(x)
        self.input_shape = x['image'].shape
        att_maps = self.attentionMaps(outputs)
        return outputs, att_maps

    def _last_conv_views(self):
        bb = self.model.gradcam_layer
        ws, xshape = getattr(bb, "_last_ws", None), getattr(bb, "_last_xshape", None)
        if ws is None:
            raise RuntimeError("GradCAM needs a forward pass with autograd enabled (do not wrap it in torch.no_grad())")
        nb = len(bb._cfg[1])
        act, grad = bb.block_buffer_views(ws, xshape, nb - 1)
        d, h, w = bb._last_out_dims
        B, growth = xshape[0], bb._cfg[3]

        def to_ncdhw(t):
            return t[:, t.shape[1] - growth:].float().reshape(B, d, h, w, growth).permute(0, 4, 1, 2, 3).contiguous()
        return act, grad, to_ncdhw

    def attentionMaps(self, outputs):
        """One trilinearly up-sampled, [0, 1]-normalised map per output class (/root/reference/utils/utils.py:293-344).
        Reference behaviours kept on purpose: the activation tensor is re-weighted cumulatively (class c sees the pooled
        gradients of classes 0..c multiplied together) and a batch of more than one volume is rejected."""
        act, grad, to_ncdhw = self._last_conv_views()
        weighted = to_ncdhw(act)                                     # [1, growth, d, h, w], re-weighted in place below
        volume_shape = tuple(self.input_shape[2:])
        maps = []
        for class_index in range(outputs.shape[1]):
            outputs[0, class_index].backward(retain_graph=True)      # fills the block's gradient accumulator
            channel_weight = to_ncdhw(grad).mean(dim=(0, 2, 3, 4))    # GradCAM alpha: gradient pooled over voxels
            weighted.mul_(channel_weight.view(1, -1, 1, 1, 1))
            cam = weighted.mean(dim=1).squeeze()
            cam = cam - cam.min()
            cam = cam / cam.max()
            if cam.ndim != 3:
                raise AssertionError('attention maps are computed one volume at a time: call with batch size 1')
            maps.append(F.interpolate(cam[None, None], volume_shape, mode='trilinear').squeeze())
        return maps


def attention_maps(model, x):
    """GradCAM attention maps of a whole batch: (outputs, maps [B, num_classes, X, Y, Z]) on the device.

    Batched replacement of the reference's per-patient GradCAM (/root/reference/utils/utils.py:253-344, called per patient
    from /root/reference/main.py:750-887): the same maps as MultiModalGradCAM.attentionMaps, for any batch size and
    without a trunk backward.  The pooled gradient of the hooked conv (last conv2 of the last dense block) has a closed
    form in eval mode -- its output reaches the logits only through norm5 (a fixed affine map), ReLU, the average pool,
    feature_layer and output_head -- so ONE kernel launch (mmnn_gradcam_maps) rebuilds every sample's cams from the
    forward's workspace and writes the up-sampled maps.

    `model` is a MultiModalModel (DenseNet121 or TinyDensenet trunk) in eval mode; `x` the {'image', 'clinical'} dict on
    its CUDA device.  One forward runs under torch.no_grad(), then the kernel is enqueued on the same stream: that order is
    what keeps the next forward from overwriting the workspace the kernel reads.  The reference's semantics are kept: class
    c is weighted by the pooled gradients of classes 0..c multiplied together, cam = (cam - min) / max (a constant cam
    gives NaN), trilinear up-sampling with align_corners=False.  Deliberate differences: a trunk dimension of size 1 works
    (the reference's .squeeze() breaks on it), and a blended model gives the maps of the multimodal head outputs[0] (the
    head predict_risks reports; the reference's class raises on it because outputs[0, c] is not a scalar there).
    Raises ValueError in train mode (batch statistics and dropout break the closed form) and MMNNLibraryError for CPU
    tensors."""
    from .. import _lib as L
    from ..models.densenet import Backbone
    from ..ops import GRADCAM_CHANNELS, gradcam_maps
    if model.training:
        raise ValueError("attention_maps needs an eval-mode model (call model.eval()): batch statistics and dropout "
                         "break the closed-form pooled gradient")
    image = x["image"]
    if not image.is_cuda:
        raise L.MMNNLibraryError("attention_maps: mmnn_sts_b200 has no CPU path (got a CPU image tensor)")
    bb = model.gradcam_layer
    if not isinstance(bb, Backbone) or bb._cfg[3] != GRADCAM_CHANNELS:
        raise ValueError("attention_maps needs a DenseNet trunk with growth rate %d" % GRADCAM_CHANNELS)
    with torch.no_grad():
        outputs = model(x)
    ws, xshape, dims, y = bb._last_forward
    act, _ = bb.block_buffer_views(ws, xshape, len(bb._cfg[1]) - 1)
    feats = model.image_model.model.features.feature_layer
    maps = gradcam_maps(act, y, dims, bb.norm5.weight, bb.norm5.running_var, bb.norm5.eps, feats.weight,
                        model.output_head.weight, xshape[2:])
    return outputs, maps
