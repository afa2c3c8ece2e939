"""torch.autograd wrappers around the small C-ABI kernels (feature head, clinical MLP + fusion heads, Cox loss).
Thin by design: tensors in, raw pointers + the current CUDA stream out.  No CPU path."""
import ctypes as C

import torch

from . import _lib as L


def _stream():
    return torch.cuda.current_stream().cuda_stream


def _p(t):
    return t.data_ptr() if t is not None else None


def _require_cuda(t, what):
    if not t.is_cuda:
        raise L.MMNNLibraryError(f"{what}: mmnn_sts_b200 has no CPU path (got a {t.device} tensor)")


class GapLinearDropout(torch.autograd.Function):
    """ReLU -> AdaptiveAvgPool3d(1) -> Flatten -> Linear -> Dropout  (/root/reference/models/densenet.py:234-247)."""

    @staticmethod
    def run(x, weight, bias, p, injected_mask=None):
        mask = None
        if injected_mask is not None:
            mask = injected_mask.to(device=x.device, dtype=torch.float32).contiguous()
        elif p > 0:
            mask = torch.bernoulli(torch.full((x.shape[0], weight.shape[0]), 1.0 - p, device=x.device)) / (1.0 - p)
        return GapLinearDropout.apply(x, weight, bias, mask)

    @staticmethod
    def forward(ctx, x, weight, bias, mask):
        _require_cuda(x, "features")
        B, Cc = x.shape[0], x.shape[1]
        y = x.permute(0, 2, 3, 4, 1).contiguous().float()       # NDHWC; a no-op for the backbone's own output
        V = y.numel() // (B * Cc)
        F = weight.shape[0]
        w = weight.contiguous().float()
        pooled = torch.empty((B, Cc), dtype=torch.float32, device=x.device)
        out = torch.empty((B, F), dtype=torch.float32, device=x.device)
        with torch.cuda.device(x.device):
            L.check(L.lib().mmnn_gap_linear_fwd(_p(y), B, V, Cc, _p(w), _p(bias), _p(mask), F, _p(pooled), _p(out), _stream()),
                    "mmnn_gap_linear_fwd")
        ctx.save_for_backward(y, pooled, w, mask)
        ctx.dims = (B, V, Cc, F, tuple(x.shape))
        return out

    @staticmethod
    def backward(ctx, dout):
        y, pooled, w, mask = ctx.saved_tensors
        B, V, Cc, F, xshape = ctx.dims
        dout = dout.contiguous().float()
        dy = torch.empty_like(y)
        dW = torch.empty_like(w)
        db = torch.empty((F,), dtype=torch.float32, device=y.device)
        with torch.cuda.device(y.device):
            L.check(L.lib().mmnn_gap_linear_bwd(_p(y), _p(pooled), B, V, Cc, _p(w), _p(dout), _p(mask), F, _p(dy), _p(dW),
                                                _p(db), _stream()), "mmnn_gap_linear_bwd")
        return dy.permute(0, 4, 1, 2, 3), dW, db, None


# ------------------------------------------------------------------------------------------------ clinical MLP + heads
class MLPHeads(torch.autograd.Function):
    """6 x (Linear -> BatchNorm1d -> ReLU/Dropout1d) on the clinical vector, then the fusion heads
    (/root/reference/models/mlp.py:19-51, /root/reference/models/multimodal.py:61-77) in ONE kernel.

    forward(x [B,F0], img_f [B,F], mask [6,B] | None, flags, buffers, *params) -> preds [H,B,C] (H = 3 if blend else 1)
    params order: for i in 0..5: W_i, b_i, gamma_i, beta_i ; then Wo, bo, Wi, bi, Wc, bc.
    buffers: list of 6 (running_mean, running_var, num_batches_tracked) triples (updated in place when training).
    """

    @staticmethod
    def _fill(args, x, img_f, mask, flags, buffers, params, saved):
        training, blend, C_ = flags
        for i in range(6):
            args.W[i], args.b[i], args.gamma[i], args.beta[i] = (_p(t) for t in params[4 * i:4 * i + 4])
            args.rmean[i], args.rvar[i], args.nbt[i] = (_p(t) for t in buffers[i])
            args.width[i + 1] = params[4 * i].shape[0]
        args.width[0] = params[0].shape[1]
        args.Wo, args.bo, args.Wi, args.bi, args.Wc, args.bc = (_p(t) for t in params[24:30])
        args.B, args.C, args.blend, args.training = x.shape[0], C_, int(blend), int(training)
        args.x, args.img_f, args.mask = _p(x), _p(img_f), _p(mask)
        args.z, args.a, args.stat = (_p(t) for t in saved)

    @staticmethod
    def forward(ctx, x, img_f, mask, flags, buffers, *params):
        _require_cuda(x, "clinical MLP")
        training, blend, C_ = flags
        B = x.shape[0]
        if training and B == 1:
            raise ValueError(f"Expected more than 1 value per channel when training, got input size {list(x.shape)}")
        x = x.contiguous().float()
        img_f = img_f.contiguous().float()
        params = tuple(p.contiguous() for p in params)
        tot = sum(p.shape[0] for p in params[0:24:4])
        z = torch.empty(B * tot, dtype=torch.float32, device=x.device)
        a = torch.empty_like(z)
        stat = torch.empty(6 * 2 * 32, dtype=torch.float32, device=x.device)
        H = 3 if blend else 1
        preds = torch.empty((H, B, C_), dtype=torch.float32, device=x.device)
        args = L.MlpArgs()
        MLPHeads._fill(args, x, img_f, mask, flags, buffers, params, (z, a, stat))
        args.preds = _p(preds)
        with torch.cuda.device(x.device):
            L.check(L.lib().mmnn_mlp_heads(C.byref(args), 0, _stream()), "mmnn_mlp_heads(fwd)")
        ctx.save_for_backward(x, img_f, mask, z, a, stat, *params)
        ctx.flags, ctx.buffers = flags, buffers
        return preds

    @staticmethod
    def backward(ctx, dpreds):
        x, img_f, mask, z, a, stat = ctx.saved_tensors[:6]
        params = ctx.saved_tensors[6:]
        dpreds = dpreds.contiguous().float()
        B = x.shape[0]
        # one zero fill for all 30 gradient tensors (views of a flat buffer, 16-byte aligned) instead of 30 fill launches
        offs, tot = [], 0
        for p in params:
            offs.append(tot)
            tot += (p.numel() + 3) & ~3
        flat = torch.zeros(tot, dtype=torch.float32, device=x.device)
        grads = [flat[o:o + p.numel()].view(p.shape) for o, p in zip(offs, params)]
        d_img = torch.empty_like(img_f)
        scratch = torch.empty(2 * B * 32, dtype=torch.float32, device=x.device)
        args = L.MlpArgs()
        MLPHeads._fill(args, x, img_f, mask, ctx.flags, ctx.buffers, params, (z, a, stat))
        args.dpreds = _p(dpreds)
        for i in range(6):
            args.dW[i], args.db[i], args.dgamma[i], args.dbeta[i] = (_p(t) for t in grads[4 * i:4 * i + 4])
        args.dWo, args.dbo, args.dWi, args.dbi, args.dWc, args.dbc = (_p(t) for t in grads[24:30])
        args.d_img_f, args.scratch = _p(d_img), _p(scratch)
        with torch.cuda.device(x.device):
            L.check(L.lib().mmnn_mlp_heads(C.byref(args), 1, _stream()), "mmnn_mlp_heads(bwd)")
        blend = ctx.flags[1]
        if not blend:   # modality heads unused: the reference leaves their .grad as None
            grads[26] = grads[27] = grads[28] = grads[29] = None
        return (None, d_img, None, None, None) + tuple(grads)


# ------------------------------------------------------------------------------------------------ Cox loss
class CoxSegments(torch.autograd.Function):
    """Negative log partial likelihood of S independent segments in one launch.
    h [S,N] fp32 log-hazards, key [S,N] (rows ordered by key DEscending, stable), weight [S,N] -> loss [S].
    Semantics: pycox cox_ph_loss (oracle/cox.py) with key := pycox `durations` slot, weight := `events` slot."""

    SORT_MAX = 4096

    @staticmethod
    def forward(ctx, h, key, weight):
        _require_cuda(h, "CoxPH")
        S, N = h.shape
        h = h.contiguous().float()
        key = key.to(torch.float64).contiguous()
        weight = weight.to(torch.float64).contiguous()
        perm = None
        if N > CoxSegments.SORT_MAX:
            perm = torch.sort(key, dim=1, descending=True, stable=True)[1].to(torch.int32).contiguous()
        loss = torch.empty(S, dtype=torch.float32, device=h.device)
        grad = torch.empty((S, N), dtype=torch.float32, device=h.device)
        a = L.CoxArgs(_p(h), N, 1, _p(key), N, 1, _p(weight), N, 1, _p(perm), N, S, 1e-7, _p(loss), _p(grad))
        with torch.cuda.device(h.device):
            L.check(L.lib().mmnn_cox_nll(C.byref(a), _stream()), "mmnn_cox_nll")
        ctx.save_for_backward(grad)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        (grad,) = ctx.saved_tensors
        return grad * dloss[:, None], None, None


def cox_ph_segments(log_h, sort_key, weight):
    return CoxSegments.apply(log_h, sort_key, weight)


# ------------------------------------------------------------------------------------------------ BCE with logits
class BCEWithLogitsElementwise(torch.autograd.Function):
    """Elementwise nn.BCEWithLogitsLoss(pos_weight, reduction='none') of logits [..., N, C] against targets [N, C]
    (the same targets for every leading "head" index) in one launch; saves dloss/dlogit for backward."""

    @staticmethod
    def forward(ctx, logits, targets, pos_weight, threshold, counts):
        _require_cuda(logits, "BCEWithLogitsLoss")
        x = logits.contiguous().float()
        y = targets.contiguous().float()
        Cc = x.shape[-1]
        if y.numel() == 0 or x.numel() % y.numel() != 0 or y.shape[-1] != Cc:
            raise ValueError(f"targets {tuple(targets.shape)} do not tile logits {tuple(logits.shape)}")
        pw = pos_weight.contiguous().float() if pos_weight is not None else None
        loss = torch.empty_like(x)
        grad = torch.empty_like(x)
        nc = y.numel() if counts is not None else 0
        with torch.cuda.device(x.device):
            L.check(L.lib().mmnn_bce_logits(_p(x), _p(y), _p(pw), x.numel(), Cc, y.numel(), _p(loss), _p(grad), float(threshold), nc,
                                            _p(counts), _stream()), "mmnn_bce_logits")
        ctx.save_for_backward(grad)
        return loss

    @staticmethod
    def backward(ctx, dloss):
        (grad,) = ctx.saved_tensors
        return grad * dloss, None, None, None, None


def bce_with_logits(logits, targets, pos_weight=None, threshold=0.5, counts=None):
    return BCEWithLogitsElementwise.apply(logits, targets, pos_weight, threshold, counts)


# ------------------------------------------------------------------------------------------------ concordance index
def concordance_counts(event_times, predicted_scores, event_observed, resample_indices=None):
    """lifelines.utils.concordance_index pair counts (oracle/cindex.py) on the GPU, exact in integers.
    All inputs 1-D CUDA tensors of N patients; resample_indices [R,N] int (bootstrap multisets of patient indices) or
    None for the identity.  Returns int64 [R,3] = (correct, tied, pairs)."""
    _require_cuda(predicted_scores, "concordance_index")
    dev = predicted_scores.device
    t = event_times.to(torch.float64).flatten()
    s = predicted_scores.to(torch.float64).flatten()
    e = (event_observed.to(torch.float64).flatten() != 0)
    N = t.numel()
    if bool(torch.isnan(t).any()) or bool(torch.isnan(s).any()):
        raise ValueError("NaNs detected in inputs, please correct or drop.")
    # order: time ascending, deaths before censored at equal times (two stable sorts)
    o1 = torch.sort((~e).to(torch.int8), stable=True)[1]
    o2 = torch.sort(t[o1], stable=True)[1]
    order = o1[o2]
    ts = t[order]
    uniq, inv = torch.unique(s, return_inverse=True)
    rank = inv[order].to(torch.int32).contiguous()
    is_death = e[order].to(torch.int32).contiguous()
    _, cnt = torch.unique_consecutive(ts, return_counts=True)
    ends = torch.cumsum(cnt, 0)
    group_end = torch.repeat_interleave(ends, cnt).to(torch.int32).contiguous()
    orig = order.to(torch.int32).contiguous()
    if resample_indices is None:
        resample_indices = torch.arange(N, device=dev, dtype=torch.int32)[None]
    res = resample_indices.to(device=dev, dtype=torch.int32).contiguous()
    R = res.shape[0]
    counts = torch.empty((R, 3), dtype=torch.int64, device=dev)
    a = L.CindexArgs(_p(rank), _p(is_death), _p(group_end), _p(orig), _p(res), N, R, int(uniq.numel()), _p(counts))
    with torch.cuda.device(dev):
        L.check(L.lib().mmnn_cindex_bootstrap(C.byref(a), _stream()), "mmnn_cindex_bootstrap")
    return counts


GRADCAM_CHANNELS = 32     # output channels of the hooked conv (the dense layers' growth rate)


def gradcam_args(act, y, trunk_dims, norm5_weight, norm5_running_var, eps, feature_weight, head_weight, size):
    """(GradcamArgs, maps, tensors the struct points to) for mmnn_gradcam_maps; see gradcam_maps."""
    for t, what in ((act, "gradcam activations"), (y, "gradcam trunk output")):
        _require_cuda(t, what)
    d, h, w = (int(v) for v in trunk_dims)
    X, Y, Z = (int(v) for v in size)
    M, ctot = act.shape
    V = d * h * w
    Fn, Cn = feature_weight.shape[0], head_weight.shape[0]
    if (M % V or y.numel() != M * ctot or y.dtype != torch.float32 or not y.is_contiguous() or act.stride(1) != 1
            or act.stride(0) != ctot or tuple(feature_weight.shape) != (Fn, ctot) or tuple(head_weight.shape) != (Cn, 2 * Fn)
            or norm5_weight.numel() != ctot or norm5_running_var.numel() != ctot or ctot < GRADCAM_CHANNELS):
        raise ValueError("gradcam_maps: inconsistent shapes")
    act_dtype = torch.float16 if L.lib().mmnn_act_is_fp16() else torch.bfloat16
    if act.dtype != act_dtype:
        raise ValueError(f"gradcam_maps: activations must be in the library's storage dtype {act_dtype}, got {act.dtype}")
    B = M // V
    dev = y.device
    f32 = [t.detach().to(device=dev, dtype=torch.float32).contiguous()
           for t in (norm5_weight, norm5_running_var, feature_weight, head_weight)]
    maps = torch.empty((B, Cn, X, Y, Z), dtype=torch.float32, device=dev)
    a = L.GradcamArgs(_p(act), _p(y), _p(f32[0]), _p(f32[1]), _p(f32[2]), _p(f32[3]), _p(maps), float(eps),
                      ctot, ctot - GRADCAM_CHANNELS, B, Cn, Fn, d, h, w, X, Y, Z)
    return a, maps, (act, y, f32)


def gradcam_maps(act, y, trunk_dims, norm5_weight, norm5_running_var, eps, feature_weight, head_weight, size):
    """Batched GradCAM maps of the last dense layer's conv2 in ONE launch (mmnn_gradcam_maps, csrc/heads.cu).
    act: the last dense block's buffer [B*V, Ctot] in the activation storage dtype (its last 32 channels are the conv's
    output); y: the trunk's fp32 output (norm5 output, NDHWC) with B*V*Ctot elements; trunk_dims (d, h, w);
    feature_weight [F, Ctot]; head_weight [C, 2F] (image features first); size (X, Y, Z).
    Returns fp32 maps [B, C, X, Y, Z].  ValueError when the shapes disagree or the cams do not fit shared memory."""
    a, maps, _ = gradcam_args(act, y, trunk_dims, norm5_weight, norm5_running_var, eps, feature_weight, head_weight, size)
    with torch.cuda.device(y.device):
        rc = L.lib().mmnn_gradcam_maps(C.byref(a), _stream())
    if rc == -3:
        raise ValueError(f"gradcam_maps: {a.C} classes x {a.d * a.h * a.w} trunk voxels of cams do not fit the kernel's "
                         "shared memory")
    if rc == -2:
        raise ValueError("gradcam_maps: unsupported sizes")
    L.check(rc, "mmnn_gradcam_maps")
    return maps
