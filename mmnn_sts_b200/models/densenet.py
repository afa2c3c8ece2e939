"""3-D DenseNet encoder with the reference's constructor signatures and state_dict layout, running on the sm_100a
kernels of libmmnn_b200.so.

Mirrors the interface of /root/reference/models/densenet.py: `DenseNet(spatial_dims, in_channels, out_channels,
feature_channels, init_features=64, growth_rate=32, block_config=(6,12,24,16), bn_size=4, act, norm, dropout_prob)`
(:173-186), `DenseNet121` (:309-324), `TinyDensenet` (:333-356);  sub-modules `backbone` / `features` /
`class_layers` keep the reference's names so `state_dict()` has the identical 779-key layout and
`BackpropagatableFeatureExtractor` (features(backbone(x)), /root/reference/utils/utils.py:238-251) works unchanged.
The torch.nn leaf modules below are parameter CONTAINERS only (names, shapes, initialisation law of :258-265);
the arithmetic is done by one C-ABI call per direction (mmnn_encoder_forward / mmnn_encoder_backward).
No CPU path: CPU tensors raise.
"""
import ctypes as C
from collections import OrderedDict
from typing import Sequence

import torch
import torch.nn as nn

from .. import _lib as L
from ..ops import GapLinearDropout


def _dense_layer(in_channels, growth_rate, bn_size, dropout_prob):
    layer = nn.Module()
    seq = nn.Sequential()
    mid = bn_size * growth_rate
    seq.add_module("norm1", nn.BatchNorm3d(in_channels))
    seq.add_module("relu1", nn.ReLU(inplace=True))
    seq.add_module("conv1", nn.Conv3d(in_channels, mid, kernel_size=1, bias=False))
    seq.add_module("norm2", nn.BatchNorm3d(mid))
    seq.add_module("relu2", nn.ReLU(inplace=True))
    seq.add_module("conv2", nn.Conv3d(mid, growth_rate, kernel_size=3, padding=1, bias=False))
    if dropout_prob > 0:
        seq.add_module("dropout", nn.Dropout3d(dropout_prob))
    layer.add_module("layers", seq)
    return layer


MAX_LIVE_WORKSPACES = 4     # forward passes under autograd that may be outstanding per input shape (each pins ~2 GB at configs[1])


class _Workspace:
    __slots__ = ("tensor", "busy", "gen")

    def __init__(self, nbytes, device):
        self.tensor = torch.empty(nbytes, dtype=torch.uint8, device=device)
        self.busy = False
        self.gen = 0            # bumped every time the workspace is handed to a forward pass


class _BackboneFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, bb, x, *params):
        out, ws, mask = bb._run_forward(x, params, track=True)   # (autograd is disabled inside Function.forward: say it explicitly)
        ctx.bb, ctx.ws, ctx.mask, ctx.shape = bb, ws, mask, tuple(x.shape)
        ctx.gen, ctx.training = ws.gen, bb.training
        ctx.params = params
        return out

    @staticmethod
    def backward(ctx, grad_out):
        bb = ctx.bb
        if ctx.ws.gen != ctx.gen:
            raise RuntimeError(
                "mmnn_sts_b200: the activations of this forward pass are gone -- its workspace was handed to a later forward "
                f"because more than {MAX_LIVE_WORKSPACES} forward passes under autograd were outstanding for this input shape. "
                "Run backward (or drop the graph under torch.no_grad()) before starting that many new forwards.")
        grads = bb._run_backward(ctx.shape, ctx.params, ctx.ws, ctx.mask, grad_out, ctx.training)
        if ctx.training:
            ctx.ws.busy = False            # (an eval-mode graph may be differentiated again: one GradCAM pass per class)
        return (None, None) + tuple(grads)


class Backbone(nn.Sequential):
    """`backbone` of the reference (/root/reference/models/densenet.py:196-231): conv0 .. norm5, one fused call."""

    def __init__(self, in_channels, init_features, growth_rate, block_config, bn_size, dropout_prob):
        super().__init__()
        self.add_module("conv0", nn.Conv3d(in_channels, init_features, kernel_size=7, stride=2, padding=3, bias=False))
        self.add_module("norm0", nn.BatchNorm3d(init_features))
        self.add_module("relu0", nn.ReLU(inplace=True))
        self.add_module("pool0", nn.MaxPool3d(kernel_size=3, stride=2, padding=1))
        c = init_features
        for i, n in enumerate(block_config):
            block = nn.Sequential()
            for j in range(n):
                block.add_module("denselayer%d" % (j + 1), _dense_layer(c, growth_rate, bn_size, dropout_prob))
                c += growth_rate
            self.add_module(f"denseblock{i + 1}", block)
            if i == len(block_config) - 1:
                self.add_module("norm5", nn.BatchNorm3d(c))
            else:
                t = nn.Sequential()
                t.add_module("norm", nn.BatchNorm3d(c))
                t.add_module("relu", nn.ReLU(inplace=True))
                t.add_module("conv", nn.Conv3d(c, c // 2, kernel_size=1, bias=False))
                t.add_module("pool", nn.AvgPool3d(kernel_size=2, stride=2))
                self.add_module(f"transition{i + 1}", t)
                c //= 2
        self.out_channels = c
        self._cfg = (in_channels, tuple(block_config), init_features, growth_rate, bn_size)
        self.dropout_prob = float(dropout_prob)
        self._plan = None
        self._workspaces = {}
        self.injected_dropmask = None  # tests: [num_layers, B, growth] keep-mask / (1-p)
        self.grad_group_hook = None    # data parallel: callable(backbone, flat_grad) run right after backward is enqueued
        self._last_forward = None

    # ---- C-ABI plumbing
    def _get_plan(self):
        if self._plan is None:
            cin, cfg, init_f, growth, bn_size = self._cfg
            arr = (C.c_int * len(cfg))(*cfg)
            h = L.lib().mmnn_encoder_create(cin, arr, len(cfg), init_f, growth, bn_size)
            if not h:
                raise L.MMNNLibraryError(f"unsupported DenseNet configuration for the sm_100a kernels: {self._cfg}")
            self._plan = C.c_void_p(h)
            n_params = sum(1 for _ in self.parameters())
            n_bufs = sum(1 for _ in self.buffers())
            assert L.lib().mmnn_encoder_num_params(self._plan) == n_params, "parameter table mismatch"
            assert L.lib().mmnn_encoder_num_buffers(self._plan) == n_bufs, "buffer table mismatch"
            self._numel = [L.lib().mmnn_encoder_param_numel(self._plan, i) for i in range(n_params)]
            assert self._numel == [p.numel() for p in self.parameters()], "parameter order mismatch"
            self._num_layers = L.lib().mmnn_encoder_num_layers(self._plan)
        return self._plan

    def __del__(self):
        try:
            if self._plan is not None:
                L.lib().mmnn_encoder_destroy(self._plan)
        except Exception:
            pass

    def _acquire_ws(self, key, nbytes, device):
        pool = self._workspaces.setdefault(key, [])
        for w in pool:
            if not w.busy:
                w.gen += 1
                return w
        if len(pool) >= MAX_LIVE_WORKSPACES:
            # forwards under autograd whose backward never ran: reuse the oldest instead of growing without bound.  Its
            # generation changes, so differentiating that stale graph later RAISES (see _BackboneFn.backward) instead of
            # reading another forward's activations.
            w = pool.pop(0)
            pool.append(w)
            w.gen += 1
            return w
        w = _Workspace(nbytes, device)
        pool.append(w)
        return w

    @staticmethod
    def _ptr_array(tensors):
        return (C.c_void_p * len(tensors))(*[t.data_ptr() for t in tensors])

    def _run_forward(self, x, params, track=False):
        if not x.is_cuda:
            raise L.MMNNLibraryError("mmnn_sts_b200 has no CPU path: move the model and inputs to a CUDA device")
        plan = self._get_plan()
        # fp16 volumes are consumed as they are (the stem packs the image into the fp16 activation format first thing, so a loader
        # that ships 16-bit volumes halves the host->device bytes without changing a bit of the result); anything else -> fp32
        half_in = x.dtype == torch.float16 and bool(L.lib().mmnn_act_is_fp16())
        x = x.contiguous() if half_in else x.contiguous().float()
        B, cin, X, Y, Z = x.shape
        assert cin == self._cfg[0], f"expected {self._cfg[0]} input channels, got {cin}"
        lib = L.lib()
        nbytes = lib.mmnn_encoder_workspace_bytes(plan, B, X, Y, Z)
        if nbytes < 0:
            raise ValueError(f"input volume {X}x{Y}x{Z} is too small for this network")
        ws = self._acquire_ws((B, X, Y, Z, x.device.index), nbytes, x.device)
        dims = (C.c_int * 3)()
        lib.mmnn_encoder_out_dims(plan, B, X, Y, Z, dims)
        out = torch.empty((B, dims[0], dims[1], dims[2], self.out_channels), dtype=torch.float32, device=x.device)
        mask = None
        if self.training:
            if self.injected_dropmask is not None:
                mask = self.injected_dropmask.to(device=x.device, dtype=torch.float32).contiguous()
            elif self.dropout_prob > 0:
                keep = 1.0 - self.dropout_prob
                mask = torch.bernoulli(torch.full((self._num_layers, B, 32), keep, device=x.device)) / keep
        bufs = list(self.buffers())
        with torch.cuda.device(x.device):
            stream = torch.cuda.current_stream().cuda_stream
            fwd = lib.mmnn_encoder_forward_f16 if half_in else lib.mmnn_encoder_forward
            rc = fwd(plan, B, X, Y, Z, x.data_ptr(), self._ptr_array(params), self._ptr_array(bufs),
                                          mask.data_ptr() if mask is not None else None, ws.tensor.data_ptr(),
                                          out.data_ptr(), int(self.training), stream)
        L.check(rc, "mmnn_encoder_forward")
        # (workspace, input shape, trunk dims, fp32 output) of the most recent forward in ANY autograd mode: the batched
        # attention maps (utils.attention_maps) read it right after a no-grad forward, on the same stream
        self._last_forward = (ws, (B, cin, X, Y, Z), (dims[0], dims[1], dims[2]), out)
        ws.busy = bool(track)                  # a backward pass will read this workspace
        if ws.busy:
            self._last_ws, self._last_xshape, self._last_out_dims = ws, (B, cin, X, Y, Z), (dims[0], dims[1], dims[2])
        if ws.busy and not self.training:
            # eval-mode forward under autograd (GradCAM, frozen-BN fine-tuning): keep the workspace for its backward, but
            # only the most recent one -- an eval forward that is never differentiated must not pin 2 GB per call
            prev = getattr(self, "_eval_ws", None)
            if prev is not None and prev is not ws:
                prev.busy = False
            self._eval_ws = ws
        return out.permute(0, 4, 1, 2, 3), ws, mask

    def _run_backward(self, xshape, params, ws, mask, grad_out, training=True):
        B, cin, X, Y, Z = xshape
        lib = L.lib()
        g = grad_out.permute(0, 2, 3, 4, 1).contiguous().float()
        flat = torch.zeros(sum(self._numel), dtype=torch.float32, device=g.device)
        grads, off = [], 0
        for p, n in zip(params, self._numel):
            grads.append(flat[off:off + n].view(p.shape))
            off += n
        bufs = list(self.buffers())
        with torch.cuda.device(g.device):
            stream = torch.cuda.current_stream().cuda_stream
            rc = lib.mmnn_encoder_backward(self._plan, B, X, Y, Z, self._ptr_array(params), self._ptr_array(bufs),
                                           self._ptr_array(grads), mask.data_ptr() if mask is not None else None,
                                           ws.tensor.data_ptr(), g.data_ptr(), int(bool(training)), stream)
        L.check(rc, "mmnn_encoder_backward")
        self._flat_grad = flat
        if self.grad_group_hook is not None:
            # everything is only ENQUEUED at this point: the hook can queue per-group all-reduces that start as soon as
            # the group's gradient-ready event fires, i.e. while the earlier blocks are still in backward
            self.grad_group_hook(self, flat)
        return grads

    def grad_groups(self):
        """[(lo, hi)] element ranges of the flat gradient buffer in the order backward finalises them."""
        plan = self._get_plan()
        out = []
        for k in range(L.lib().mmnn_encoder_num_grad_groups(plan)):
            lo, hi = C.c_longlong(), C.c_longlong()
            L.check(L.lib().mmnn_encoder_grad_group_range(plan, k, C.byref(lo), C.byref(hi)), "mmnn_encoder_grad_group_range")
            out.append((lo.value, hi.value))
        return out

    def wait_grad_group(self, k, stream):
        L.check(L.lib().mmnn_encoder_wait_grad_group(self._get_plan(), k, stream.cuda_stream), "mmnn_encoder_wait_grad_group")

    def block_buffer_views(self, ws, xshape, block):
        """(activations [M, Ctot] in the storage dtype, gradient accumulator [M, Ctot] fp32) of dense block `block` inside
        workspace `ws`, plus the block's spatial dims: what GradCAM reads for the last convolution's output channels."""
        B, cin, X, Y, Z = xshape
        nb = len(self._cfg[1])
        offs = (C.c_longlong * (3 + 3 * nb + 2))()
        dims = (C.c_longlong * (4 + 4 * nb + 1))()
        L.check(L.lib().mmnn_encoder_debug_offsets(self._get_plan(), B, X, Y, Z, offs, dims), "mmnn_encoder_debug_offsets")
        M, ctot = int(dims[4 + 4 * block]), int(dims[4 + 4 * block + 1])
        adt = torch.float16 if L.lib().mmnn_act_is_fp16() else torch.bfloat16
        base = ws.tensor
        act = base[int(offs[3 + block]):int(offs[3 + block]) + M * ctot * 2].view(adt).view(M, ctot)
        grad = base[int(offs[3 + 2 * nb + block]):int(offs[3 + 2 * nb + block]) + M * ctot * 4].view(torch.float32).view(M, ctot)
        return act, grad

    def flat_grad_buffer(self):
        """The single contiguous fp32 buffer holding every trunk gradient, if the parameters' .grad tensors are still the
        views handed to autograd by the last backward (autograd adopts them on the first accumulation and adds in place
        afterwards).  Lets the data-parallel reducer all-reduce 11.2 M values with ONE collective and no packing copies."""
        flat = getattr(self, "_flat_grad", None)
        if flat is None:
            return None
        off, base, es = 0, flat.data_ptr(), flat.element_size()
        for p, n in zip(self.parameters(), self._numel):
            if p.grad is None or p.grad.data_ptr() != base + off * es or not p.grad.is_contiguous():
                return None
            off += n
        return flat

    def pack_flat_grad(self):
        """Make flat_grad_buffer() return a buffer: if it does not, every parameter's .grad becomes a view of one fresh
        fp32 buffer holding its current gradient (zeros where it has none).  A data-parallel rank that did no backward
        in an accumulation round then reduces the trunk with the same single collective as the other ranks."""
        flat = self.flat_grad_buffer()
        if flat is not None:
            return flat
        self._get_plan()
        params = list(self.parameters())
        flat = torch.zeros(sum(self._numel), dtype=torch.float32, device=params[0].device)
        off = 0
        for p, n in zip(params, self._numel):
            v = flat[off:off + n].view(p.shape)
            if p.grad is not None:
                v.copy_(p.grad)
            p.grad = v
            off += n
        self._flat_grad = flat
        return flat

    def forward(self, x):
        params = tuple(self.parameters())
        if torch.is_grad_enabled() and any(p.requires_grad for p in params):
            return _BackboneFn.apply(self, x, *params)
        out, ws, _ = self._run_forward(x, params, track=False)
        return out


class _Features(nn.Sequential):
    """`features` head of the reference (:234-247): ReLU -> AdaptiveAvgPool3d(1) -> Flatten -> Linear -> Dropout."""

    def __init__(self, in_channels, feature_channels, dropout_prob):
        super().__init__(OrderedDict([
            ("relu", nn.ReLU(inplace=True)),
            ("pool", nn.AdaptiveAvgPool3d(1)),
            ("flatten", nn.Flatten(1)),
            ("feature_layer", nn.Linear(in_channels, feature_channels)),
            ("dropout", nn.Dropout(dropout_prob)),
        ]))
        self.injected_mask = None  # tests: [B, F] keep-mask / (1-p)

    def forward(self, x):
        p = self.dropout.p if self.training else 0.0
        return GapLinearDropout.run(x, self.feature_layer.weight, self.feature_layer.bias, p, self.injected_mask if self.training else None)


class DenseNet(nn.Module):
    def __init__(self, spatial_dims: int, in_channels: int, out_channels: int, feature_channels: int,
                 init_features: int = 64, growth_rate: int = 32, block_config: Sequence[int] = (6, 12, 24, 16),
                 bn_size: int = 4, act=("relu", {"inplace": True}), norm="batch", dropout_prob: float = 0.0) -> None:
        super().__init__()
        if spatial_dims != 3:
            raise NotImplementedError("the sm_100a build implements the 3-D network only")
        self.backbone = Backbone(in_channels, init_features, growth_rate, block_config, bn_size, dropout_prob)
        self.features = _Features(self.backbone.out_channels, feature_channels, dropout_prob)
        self.class_layers = nn.Sequential(OrderedDict([("out", nn.Linear(feature_channels, out_channels))]))
        for m in self.modules():
            if isinstance(m, nn.Conv3d):
                nn.init.kaiming_normal_(m.weight)
            elif isinstance(m, nn.BatchNorm3d):
                nn.init.constant_(m.weight, 1)
                nn.init.constant_(m.bias, 0)
            elif isinstance(m, nn.Linear):
                nn.init.constant_(m.bias, 0)

    def forward(self, x):
        return self.class_layers(self.features(self.backbone(x)))


class DenseNet121(DenseNet):
    def __init__(self, init_features: int = 64, growth_rate: int = 32, block_config: Sequence[int] = (6, 12, 24, 16),
                 pretrained: bool = False, progress: bool = True, **kwargs) -> None:
        super().__init__(init_features=init_features, growth_rate=growth_rate, block_config=block_config, **kwargs)
        if pretrained:
            raise NotImplementedError("PyTorch Hub provides no pretrained 3-D DenseNet (same as the reference)")


class TinyDensenet(DenseNet):
    def __init__(self, init_features: int = 64, growth_rate: int = 32, block_config: Sequence[int] = (6, 12, 4),
                 pretrained: bool = False, progress: bool = True, **kwargs) -> None:
        super().__init__(init_features=init_features, growth_rate=growth_rate, block_config=block_config, **kwargs)


Densenet = densenet = DenseNet
Densenet121 = densenet121 = DenseNet121
