"""Train / inference drivers mirroring the hot-path bodies of the reference's main.py (which cannot itself be imported:
/root/reference/main.py:1 imports a non-existent CLASS_FREQUENCIES, SURVEY.md section 0):

  getCIndices          /root/reference/main.py:106-123   (lifelines concordance_index per class)
  train_survival       /root/reference/main.py:385-601   (SGD nesterov + OneCycleLR, gradient accumulation to 64 samples,
                                                          GradientBlender, per-epoch C-index, validation, weight update)
  train_classification /root/reference/main.py:125-327   (BCE-with-logits 'sum' loss with pos_weight, SGD nesterov + OneCycleLR stepped
                                                          every batch, tp / fp / fn -> per-class F1, validation, best-F1 state)
  inference_survival   /root/reference/main.py:750-887   (forward + bootstrap C-index; idiomatic form: every patient is
                                                          forwarded ONCE, resamples are index multisets; GradCAM maps
                                                          batched, utils/utils.py:253-344 -> utils.attention_maps)
Data arrives as an iterable of batches `({'image': ..., 'clinical': ...}, events, durations)` -- what the reference's
multimodal_collate_fn_surv yields -- so the file/S3 datasets of the reference stay out of scope.
"""
import math
from types import SimpleNamespace

import numpy as np
import torch

from .losses.GradientBlender import GradientBlender
from .losses.losses import CoxPH
from .ops import concordance_counts
from .optim import SGD
from .utils.utils import attention_maps, surv_criterion

NUM_CLASSES = 2                 # /root/reference/data/constants.py:95
NUM_BOOTSTRAP_ITERATIONS = 50   # /root/reference/main.py:61
SUPER_BATCH_SIZE = 64           # /root/reference/main.py:62


CLASSIFICATION_THRESHOLD = 0.5   # /root/reference/main.py (threshold applied to sigmoid outputs, :226)


def getF1Score(tps, fps, fns):
    """/root/reference/main.py:98-104: per-class F1 = tp / (tp + 0.5 (fn + fp)) as Python floats."""
    f1s = []
    for idx in range(len(tps)):
        f1 = tps[idx] / (tps[idx] + 0.5 * (fns[idx] + fps[idx]))
        f1s.append(f1.item())
    return f1s


def classification_pos_weights(class_freqs):
    """/root/reference/main.py:148: pos_weight = (1 - f) / f."""
    return (torch.ones_like(class_freqs) - class_freqs) / class_freqs


def _cindex_from_counts(correct, tied, pairs):
    if pairs == 0:
        raise ZeroDivisionError("No admissable pairs in the dataset.")
    return (correct + tied / 2) / pairs


def getCIndices(preds, events, durations, num_classes=NUM_CLASSES):
    """List of per-class Harrell C-indices, `concordance_index(durations[:, i], preds[:, i], events[:, i])`.
    Accepts CUDA tensors (counted on the GPU, exact in int64) ; numpy / CPU tensors are moved to the current device."""
    dev = preds.device if torch.is_tensor(preds) and preds.is_cuda else torch.device("cuda", torch.cuda.current_device())
    preds, events, durations = (torch.as_tensor(np.asarray(t) if not torch.is_tensor(t) else t).to(dev) for t in (preds, events, durations))
    out = []
    for i in range(num_classes):
        c, t, p = (int(v) for v in concordance_counts(durations[:, i], preds[:, i], events[:, i])[0].cpu())
        out.append(_cindex_from_counts(c, t, p))
    return out


def bootstrap_cindices(preds, events, durations, resample_indices, num_classes=NUM_CLASSES):
    """Per-resample, per-class C-index [R, C] (NaN where a resample has no admissible pair: the reference skips it,
    /root/reference/main.py:856-858), plus mean and std (ddof 0) over the kept resamples (:883-887)."""
    counts = torch.stack([concordance_counts(durations[:, i], preds[:, i], events[:, i], resample_indices)
                          for i in range(num_classes)], dim=1).cpu().numpy()      # [R, C, 3] int64
    correct, tied, pairs = counts[..., 0], counts[..., 1], counts[..., 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        c = (correct + tied / 2) / pairs
    c[pairs == 0] = np.nan
    ok = ~np.isnan(c).any(axis=1)
    return c, c[ok].mean(axis=0), c[ok].std(axis=0), counts


def _with_last_flag(iterable):
    """(item, is_last) pairs of one pass over `iterable` without materialising it: a DataLoader with shuffle=True is
    re-iterated (and reshuffled) every epoch, and an epoch of 3-D volumes is never held in host memory at once."""
    it = iter(iterable)
    try:
        prev = next(it)
    except StopIteration:
        return
    for cur in it:
        yield prev, False
        prev = cur
    yield prev, True


def _to_device(batch, device):
    inputs, events, durations = batch
    inputs = {k: v.to(device, non_blocking=True) for k, v in inputs.items()}
    return inputs, events.to(device, non_blocking=True), durations.to(device, non_blocking=True)


def train_survival(model, train_batches, val_batches, args, device, grad_sync=None, log=None):
    """args: lr, momentum, weight_decay, epochs, batch_size, blend, blend_update_interval, num_train (patients).
    grad_sync: optional callable(model) run right before each optimizer.step (data-parallel gradient all-reduce)."""
    model = model.to(device)
    n_train = args.num_train
    super_batch_interval = SUPER_BATCH_SIZE / args.batch_size
    steps_per_epoch = n_train // SUPER_BATCH_SIZE if n_train % SUPER_BATCH_SIZE == 0 else 1 + n_train // SUPER_BATCH_SIZE
    optimizer = SGD(model.parameters(), args.lr, momentum=args.momentum, nesterov=True, weight_decay=args.weight_decay)
    scheduler = torch.optim.lr_scheduler.OneCycleLR(optimizer, max_lr=args.lr, steps_per_epoch=steps_per_epoch, epochs=args.epochs)
    blender = GradientBlender(CoxPH, survival=True, surv_criterion=surv_criterion) if args.blend else None
    hist = SimpleNamespace(train_loss=[], val_loss=[], train_c=[], val_c=[], best_loss=math.inf, best_state=None, blender=blender,
                           step_at=[], lr_trace=[], momentum_trace=[], optimizer=optimizer, scheduler=scheduler)
    for epoch in range(args.epochs):
        model.train()
        losses, c_pred, c_events, c_durations = [], [], [], []
        for i, (batch, is_last) in enumerate(_with_last_flag(train_batches)):
            inputs, events, durations = _to_device(batch, device)
            outputs = model(inputs)
            if args.blend:
                loss, _ = blender.computeLoss(outputs, events, durations)
            else:
                loss = surv_criterion(CoxPH, outputs, events, durations, device)
            if grad_sync is not None and super_batch_interval == 1 and hasattr(grad_sync, "arm"):
                grad_sync.arm()                     # no accumulation: the trunk's gradient groups are all-reduced during backward
            loss.backward()
            losses.append(loss.detach())            # no per-step .item(): one sync per epoch instead of one per step
            if (i + 1) % super_batch_interval == 0 or is_last:
                if grad_sync is not None:
                    grad_sync(model)
                optimizer.step()
                scheduler.step()
                optimizer.zero_grad(set_to_none=True)
                hist.step_at.append((epoch, i))
                hist.lr_trace.append(optimizer.param_groups[0]["lr"]); hist.momentum_trace.append(optimizer.param_groups[0]["momentum"])
            c_pred.append(outputs.detach()); c_events.append(events); c_durations.append(durations)
        if not c_pred:
            raise ValueError("train_batches yielded no batch in epoch %d: pass a re-iterable (list, DataLoader), not a one-shot generator" % (epoch + 1))
        c_pred = torch.cat(c_pred, dim=1 if args.blend else 0)
        c_events, c_durations = torch.cat(c_events), torch.cat(c_durations)
        hist.train_c.append(getCIndices(c_pred[0] if args.blend else c_pred, c_events, c_durations))
        hist.train_loss.append(float(torch.stack(losses).sum()) / n_train)
        if val_batches is not None:
            model.eval()
            with torch.no_grad():
                y_pred, y_events, y_durations, vloss, sel = [], [], [], 0.0, None
                for batch in val_batches:
                    inputs, events, durations = _to_device(batch, device)
                    preds = model(inputs)
                    if args.blend:
                        loss, sel = blender.computeLoss(preds, events, durations)
                    else:
                        loss = sel = surv_criterion(CoxPH, preds, events, durations, device)
                    vloss += float(loss)
                    y_pred.append(preds); y_events.append(events); y_durations.append(durations)
                if not y_pred:
                    raise ValueError("val_batches yielded no batch in epoch %d: pass a re-iterable (list, DataLoader), not a one-shot generator" % (epoch + 1))
                y_pred = torch.cat(y_pred, dim=1 if args.blend else 0)
                y_events, y_durations = torch.cat(y_events), torch.cat(y_durations)
                hist.val_c.append(getCIndices(y_pred[0] if args.blend else y_pred, y_events, y_durations))
                hist.val_loss.append(vloss / max(1, y_events.shape[0]))
                if float(sel) < hist.best_loss:
                    hist.best_loss = float(sel)
                    hist.best_state = {k: v.detach().clone() for k, v in model.state_dict().items()}
            if args.blend and (epoch + 1) % args.blend_update_interval == 0:
                blender.updateWeights(c_pred, c_events, c_durations, y_pred, y_events, y_durations)
        if log is not None:
            log(f"epoch {epoch + 1}: train loss {hist.train_loss[-1]:.4f} train C {hist.train_c[-1]}")
    return hist


def train_classification(model, train_batches, val_batches, args, device, grad_sync=None, log=None):
    """Loop body of /root/reference/main.py:125-327 over iterables of collated batches `(inputs, labels)` -- `inputs` is the image
    tensor [B, C, D, H, W] (image-only models such as r3d_18, `args.multimodal` False) or the {'image', 'clinical'} dict.
    args: lr, momentum, weight_decay, epochs, batch_size, blend, blend_update_interval, class_freqs, num_train, multimodal.
    As in the reference the loss is `BCEWithLogitsLoss(pos_weight=(1 - f) / f)` applied to whatever the model returns (:208 --
    for r3d_18 that is already a sigmoid score, the reference's own quirk), reduction 'sum' for training and 'none' for
    validation, the optimiser steps EVERY batch (:210) and the F1 counters threshold `sigmoid(outputs)` (:216-229)."""
    from .losses.losses import BCEWithLogitsLoss
    from .utils.utils import criterion
    model = model.to(device)
    n_train = args.num_train
    steps_per_epoch = n_train // args.batch_size if n_train % args.batch_size == 0 else 1 + n_train // args.batch_size
    pos_weights = classification_pos_weights(torch.as_tensor(args.class_freqs, dtype=torch.float32)).to(device)
    train_loss_function = BCEWithLogitsLoss(pos_weight=pos_weights, reduction="sum").to(device)
    loss_function = BCEWithLogitsLoss(pos_weight=pos_weights, reduction="none").to(device)
    optimizer = SGD(model.parameters(), args.lr, momentum=args.momentum, nesterov=True, weight_decay=args.weight_decay)
    scheduler = torch.optim.lr_scheduler.OneCycleLR(optimizer, max_lr=args.lr, steps_per_epoch=steps_per_epoch, epochs=args.epochs)
    blender = GradientBlender(loss_function, device=device) if args.blend else None
    hist = SimpleNamespace(train_loss=[], val_loss=[], train_f1=[], val_f1=[], best_metric=-1.0, best_epoch=-1, best_f1s=None,
                           best_state=None, blender=blender)

    def to_dev(batch):
        inputs, labels = batch
        inputs = {k: v.to(device, non_blocking=True) for k, v in inputs.items()} if isinstance(inputs, dict) else inputs.to(device, non_blocking=True)
        return inputs, labels.to(device, non_blocking=True)

    def counts(preds01, labels):
        return torch.stack([((preds01 == 1) & (labels == 1)).sum(0), ((preds01 == 1) & (labels == 0)).sum(0),
                            ((preds01 == 0) & (labels == 1)).sum(0)])

    for epoch in range(args.epochs):
        model.train()
        losses, cnt, tr_preds, tr_gt = [], 0, [], []
        for batch in train_batches:
            inputs, labels = to_dev(batch)
            optimizer.zero_grad(set_to_none=True)
            outputs = model(inputs)
            loss = blender.computeLoss(outputs, labels) if args.blend else criterion(train_loss_function, outputs, labels, device)
            loss.backward()
            if grad_sync is not None:
                grad_sync(model)
            optimizer.step()
            scheduler.step()
            losses.append(loss.detach())                       # no per-step .item(): one host sync per epoch
            probs = torch.sigmoid(outputs.detach())
            if args.blend:
                tr_preds.append(probs); tr_gt.append(labels)
                probs = probs[0]
            cnt = cnt + counts((probs > CLASSIFICATION_THRESHOLD).long(), labels.long())
        hist.train_f1.append(float(np.mean(getF1Score(cnt[0].cpu(), cnt[1].cpu(), cnt[2].cpu()))))
        hist.train_loss.append(float(torch.stack(losses).sum()) / n_train)
        if val_batches is not None:
            model.eval()
            with torch.no_grad():
                vcnt, vloss, nval, va_preds, va_gt = 0, 0.0, 0, [], []
                for batch in val_batches:
                    inputs, labels = to_dev(batch)
                    preds = model(inputs)
                    loss = blender.computeLoss(preds, labels, no_reduce=True) if args.blend else criterion(loss_function, preds, labels, device)
                    vloss += float(loss.sum())
                    p01 = (torch.sigmoid(preds) > CLASSIFICATION_THRESHOLD).long()
                    if args.blend:
                        va_preds.append(p01.float()); va_gt.append(labels)
                        p01 = p01[0]
                    vcnt = vcnt + counts(p01, labels.long())
                    nval += labels.shape[0]
                f1s = np.array(getF1Score(vcnt[0].cpu(), vcnt[1].cpu(), vcnt[2].cpu()))
                hist.val_f1.append(float(np.mean(f1s)))
                hist.val_loss.append(vloss / max(1, nval))
                if hist.val_f1[-1] > hist.best_metric:
                    hist.best_metric, hist.best_f1s, hist.best_epoch = hist.val_f1[-1], f1s, epoch + 1
                    hist.best_state = {k: v.detach().clone() for k, v in model.state_dict().items()}
            if args.blend and (epoch + 1) % args.blend_update_interval == 0:
                blender.updateWeights(torch.cat(tr_preds, dim=1), torch.cat(tr_gt), torch.cat(va_preds, dim=1), torch.cat(va_gt))
        if log is not None:
            log(f"epoch {epoch + 1}: train loss {hist.train_loss[-1]:.4f} train F1 {hist.train_f1[-1]:.4f}")
    return hist


@torch.no_grad()
def predict_risks(model, batches, device, gradcam=None):
    """Eval-mode forward of every patient once (batched). Returns (preds [N,C], events [N,C], durations [N,C]).
    gradcam: optional callable(batch_index, maps).  Each batch then goes through utils.attention_maps (the same forward
    plus ONE map kernel) and the callable receives that batch's maps [B, C, X, Y, Z] on the device -- the batched form of
    the reference's per-patient GradCAM loop (/root/reference/main.py:750-887).  Maps are not kept here (at 10 000
    patients of 128x128x64 they would be 80 GB): the callable writes or reduces them.  The predictions are the same
    bits either way."""
    model = model.to(device).eval()
    preds, ev, du = [], [], []
    for i, batch in enumerate(batches):
        inputs, events, durations = _to_device(batch, device)
        if gradcam is None:
            out = model(inputs)
        else:
            out, maps = attention_maps(model, inputs)
            gradcam(i, maps)
        preds.append(out[0] if out.dim() == 3 else out); ev.append(events); du.append(durations)
    return torch.cat(preds), torch.cat(ev), torch.cat(du)


def inference_survival(model, batches, device, bootstrap=True, num_resamples=NUM_BOOTSTRAP_ITERATIONS, seed=None, gradcam=None):
    """Risks of every patient, then the C-indices (bootstrap: per-resample, mean, std).  gradcam: see predict_risks."""
    preds, events, durations = predict_risks(model, batches, device, gradcam=gradcam)
    n = preds.shape[0]
    if not bootstrap:
        return getCIndices(preds, events, durations), preds
    # sklearn.utils.resample(uids) == uids[RandomState.randint(0, n, n)]  (SURVEY.md appendix B.3)
    rng = np.random.RandomState(seed) if seed is not None else np.random
    idx = np.stack([rng.randint(0, n, n) for _ in range(num_resamples)])
    c, mean, std, _ = bootstrap_cindices(preds, events, durations, torch.as_tensor(idx, device=preds.device))
    return SimpleNamespace(per_resample=c, mean=mean, std=std, preds=preds)
