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
import torch.distributed as dist

from . import distributed as D
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


def _resample_counts(preds, events, durations, resample_indices, num_classes=NUM_CLASSES):
    """int64 [R, C, 3] (correct, tied, pairs) of every resample and class, on the predictions' device."""
    return torch.stack([concordance_counts(durations[:, i], preds[:, i], events[:, i], resample_indices)
                        for i in range(num_classes)], dim=1)


def bootstrap_from_counts(counts):
    """Per-resample, per-class C-index [R, C] of int64 counts [R, C, 3] (NaN where a resample has no admissible pair: the
    reference skips it, /root/reference/main.py:856-858), plus mean and std (ddof 0) over the kept resamples (:883-887)."""
    correct, tied, pairs = counts[..., 0], counts[..., 1], counts[..., 2]
    with np.errstate(divide="ignore", invalid="ignore"):
        c = (correct + tied / 2) / pairs
    c[pairs == 0] = np.nan
    ok = ~np.isnan(c).any(axis=1)
    return c, c[ok].mean(axis=0), c[ok].std(axis=0)


def bootstrap_cindices(preds, events, durations, resample_indices, num_classes=NUM_CLASSES):
    """bootstrap_from_counts of the resamples' counts: (per-resample [R, C], mean, std, counts [R, C, 3])."""
    counts = _resample_counts(preds, events, durations, resample_indices, num_classes).cpu().numpy()
    return bootstrap_from_counts(counts) + (counts,)


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


def _survival_setup(model, args):
    """Optimiser, OneCycleLR schedule (ceil(num_train / 64) steps per epoch), blender and the empty history."""
    n_train = args.num_train
    steps_per_epoch = n_train // SUPER_BATCH_SIZE if n_train % SUPER_BATCH_SIZE == 0 else 1 + n_train // SUPER_BATCH_SIZE
    optimizer = SGD(model.parameters(), args.lr, momentum=args.momentum, nesterov=True, weight_decay=args.weight_decay)
    scheduler = torch.optim.lr_scheduler.OneCycleLR(optimizer, max_lr=args.lr, steps_per_epoch=steps_per_epoch, epochs=args.epochs)
    blender = GradientBlender(CoxPH, survival=True, surv_criterion=surv_criterion) if args.blend else None
    hist = SimpleNamespace(train_loss=[], val_loss=[], train_c=[], val_c=[], best_loss=math.inf, best_state=None, blender=blender,
                           step_at=[], lr_trace=[], momentum_trace=[], optimizer=optimizer, scheduler=scheduler)
    return optimizer, scheduler, blender, hist


def train_survival(model, train_batches, val_batches, args, device, grad_sync=None, log=None, group=None):
    """args: lr, momentum, weight_decay, epochs, batch_size, blend, blend_update_interval, num_train (patients).
    grad_sync: optional callable(model) run right before each optimizer.step (data-parallel gradient all-reduce).

    group: a torch.distributed group of more than one rank trains data-parallel as one process would on all ranks'
    micro-batches (DESIGN.md section 8).  `train_batches` / `val_batches` are then this rank's round-robin shards
    (distributed.shard_batches: local micro-batch i of rank r is global micro-batch i * G + r) and must support len();
    args.num_train is the GLOBAL patient count; 64 / batch_size must be a multiple of G.  train_survival reduces the
    gradients itself (passing grad_sync too raises ValueError), steps after every 64 global patients and after the last
    micro-batch, merges the BatchNorm running statistics at every step, and computes the epoch's losses, C-indices,
    best state and blending-weight update from all ranks' rows in global order, so every rank returns the same hist.
    group=None, or a group of one rank, is the one-process loop."""
    if _world(group) > 1:
        if grad_sync is not None:
            raise ValueError("train_survival: with a group of several ranks train_survival reduces the gradients itself; "
                             "do not pass grad_sync")
        return _train_survival_dp(model, train_batches, val_batches, args, device, log, group)
    model = model.to(device)
    n_train = args.num_train
    super_batch_interval = SUPER_BATCH_SIZE / args.batch_size
    optimizer, scheduler, blender, hist = _survival_setup(model, args)
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


def _len_or_flag(batches):
    """len(batches); -1 when it has none, -2 for None (exchanged, so that every rank raises on a bad input)."""
    if batches is None:
        return -2
    return len(batches) if hasattr(batches, "__len__") else -1


def _keyed_rows(g, preds, events, durations):
    """float64 rows [g, row, H, preds (H x C), events (C), durations (C)] of one micro-batch (H = 1 for [B, C] preds):
    exact for fp32 predictions and integer targets below 2**53, and self-describing, so that a rank without rows can
    still decode what the others gathered."""
    p = preds.detach()
    H = p.shape[0] if p.dim() == 3 else 1
    p = p.permute(1, 0, 2).reshape(p.shape[-2], -1) if p.dim() == 3 else p
    B = p.shape[0]
    dev = p.device
    keys = torch.stack([torch.full((B,), float(g), dtype=torch.float64, device=dev),
                        torch.arange(B, dtype=torch.float64, device=dev),
                        torch.full((B,), float(H), dtype=torch.float64, device=dev)], 1)
    return torch.cat([keys, p.to(torch.float64), events.to(torch.float64).reshape(B, -1),
                      durations.to(torch.float64).reshape(B, -1)], 1)


def _gather_rows(rows, stacked, group, device):
    """All ranks' _keyed_rows in global order: (preds [H, N, C] if stacked else [N, C] float32, events, durations
    float64 [N, C])."""
    rows = torch.cat(rows) if rows else torch.empty((0, 0), dtype=torch.float64, device=device)
    rows = D.allgather_ordered(rows, group)
    N = rows.shape[0]
    if N == 0:
        raise ValueError("train_survival: no rank has a micro-batch")
    H = int(rows[0, 0])
    C = (rows.shape[1] - 1) // (H + 2)
    preds = rows[:, 1:1 + H * C].to(torch.float32)
    preds = preds.reshape(N, H, C).permute(1, 0, 2).contiguous() if stacked else preds
    return preds, rows[:, 1 + H * C:1 + (H + 1) * C], rows[:, 1 + (H + 1) * C:]


def _gather_scalars(rows, width, group, device):
    """All ranks' per-micro-batch scalar rows [g, 0, value...] in global micro-batch order: float64 [N_b, width]."""
    rows = torch.stack(rows) if rows else torch.empty((0, 0), dtype=torch.float64, device=device)
    return D.allgather_ordered(rows, group).reshape(-1, width)


def _train_survival_dp(model, train_batches, val_batches, args, device, log, group):
    """train_survival over the ranks of `group` (see there).  The collectives a rank enters depend only on what every
    rank agrees on (args, the world size and the exchanged per-rank batch counts), never on its own data."""
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    interval = D.check_interval(SUPER_BATCH_SIZE / args.batch_size, world)       # raises before any collective
    model = model.to(device)
    n_train = args.num_train
    optimizer, scheduler, blender, hist = _survival_setup(model, args)
    merger = D.RunningStatsMerger(model, group)
    hooks = [(m, m.grad_group_hook) for m in model.modules() if hasattr(m, "grad_group_hook")]   # restored on return
    reducer = D.GradientAllReducer(model.parameters(), group=group, model=model)

    def loss_of(outputs, events, durations):
        if args.blend:
            return blender.computeLoss(outputs, events, durations)
        loss = surv_criterion(CoxPH, outputs, events, durations, device)
        return loss, loss

    try:
        for epoch in range(args.epochs):
            counts = D.allgather_counts([_len_or_flag(train_batches), _len_or_flag(val_batches)], device, group)
            if any(c[0] == -1 or c[1] == -1 for c in counts):
                raise TypeError("train_survival: under a group every rank's train_batches and val_batches must support "
                                "len() (a list, a DataLoader): the ranks agree on the step schedule before the epoch")
            if any(c[0] < 0 for c in counts) or len({c[1] == -2 for c in counts}) > 1:
                raise ValueError("train_survival: every rank passes train_batches, and either every rank or none val_batches")
            rounds = D.accumulation_rounds([c[0] for c in counts], interval)
            has_val = counts[0][1] != -2
            n_val_batches = D.check_round_robin([c[1] for c in counts], "validation micro-batches") if has_val else 0
            if not rounds:
                raise ValueError("train_batches has no batch in epoch %d" % (epoch + 1))
            model.train()
            it = iter(train_batches)
            losses, rows = [], []
            for lo, hi in rounds:
                merger.begin(hi - lo)
                for g in range(lo + rank, hi, world):
                    inputs, events, durations = _to_device(next(it), device)
                    merger.before_forward()
                    outputs = model(inputs)
                    merger.after_forward(g - lo)
                    loss, _ = loss_of(outputs, events, durations)
                    if hi - lo == world:
                        reducer.arm()       # every rank has exactly this one micro-batch: reduce during backward
                    loss.backward()
                    losses.append(torch.stack([torch.full_like(loss.detach(), g, dtype=torch.float64),
                                               torch.zeros((), dtype=torch.float64, device=loss.device), loss.detach().double()]))
                    rows.append(_keyed_rows(g, outputs, events, durations))
                D.fill_missing_grads(reducer)
                reducer(model)
                merger.merge()
                optimizer.step()
                scheduler.step()
                optimizer.zero_grad(set_to_none=True)
                hist.step_at.append((epoch, hi - 1))
                hist.lr_trace.append(optimizer.param_groups[0]["lr"]); hist.momentum_trace.append(optimizer.param_groups[0]["momentum"])
            c_pred, c_events, c_durations = _gather_rows(rows, args.blend, group, device)
            if c_events.shape[0] != n_train:
                raise ValueError("train_survival: the ranks trained %d patients in epoch %d, args.num_train is %d (the "
                                 "global count)" % (c_events.shape[0], epoch + 1, n_train))
            train_losses = _gather_scalars(losses, 1, group, device)[:, 0].to(torch.float32)
            hist.train_c.append(getCIndices(c_pred[0] if args.blend else c_pred, c_events, c_durations))
            hist.train_loss.append(float(train_losses.sum()) / n_train)
            if has_val:
                if n_val_batches == 0:
                    raise ValueError("val_batches has no batch in epoch %d" % (epoch + 1))
                model.eval()
                with torch.no_grad():
                    vrows, vlosses, i = [], [], -1
                    for i, batch in enumerate(val_batches):
                        g = i * world + rank
                        inputs, events, durations = _to_device(batch, device)
                        preds = model(inputs)
                        loss, sel = loss_of(preds, events, durations)
                        vlosses.append(torch.stack([torch.full_like(loss, g, dtype=torch.float64),
                                                    torch.zeros((), dtype=torch.float64, device=loss.device),
                                                    loss.double(), sel.double()]))
                        vrows.append(_keyed_rows(g, preds, events, durations))
                    if i + 1 != counts[rank][1]:
                        raise ValueError("val_batches yielded %d batches, len() said %d" % (i + 1, counts[rank][1]))
                    y_pred, y_events, y_durations = _gather_rows(vrows, args.blend, group, device)
                    vl = _gather_scalars(vlosses, 2, group, device).tolist()
                    vloss = 0.0
                    for loss, _ in vl:
                        vloss += loss                      # fp32 values as Python floats, summed in global order
                    sel = vl[-1][1]                        # the globally last validation micro-batch
                    hist.val_c.append(getCIndices(y_pred[0] if args.blend else y_pred, y_events, y_durations))
                    hist.val_loss.append(vloss / max(1, y_events.shape[0]))
                    if sel < hist.best_loss:
                        hist.best_loss = sel
                        hist.best_state = {k: v.detach().clone() for k, v in model.state_dict().items()}
                if args.blend and (epoch + 1) % args.blend_update_interval == 0:
                    blender.updateWeights(c_pred, c_events, c_durations, y_pred, y_events, y_durations)
            if log is not None:
                log(f"epoch {epoch + 1}: train loss {hist.train_loss[-1]:.4f} train C {hist.train_c[-1]}")
    finally:
        for m, h in hooks:
            m.grad_group_hook = h
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


def _world(group):
    return 1 if group is None else dist.get_world_size(group)


def _gather_patients(preds, events, durations, patient_ids, group, device):
    """All ranks' rows of (preds, events, durations) in patient order (rank-major without patient_ids).

    One allgather_varlen of float64 rows [preds | events | durations | id]: exact for fp32 predictions and for integer
    events, durations and ids below 2**53, and a rank without patients needs to know neither C nor the dtypes.  The
    predictions come back as float32 (the model's output dtype), events and durations as float64 (concordance_counts
    counts in float64 anyway)."""
    if preds:
        cols = [torch.cat(t).to(torch.float64) for t in (preds, events, durations)]
        if patient_ids is not None:
            ids = torch.as_tensor(patient_ids).to(device=device, dtype=torch.float64).flatten()
            if ids.numel() != cols[0].shape[0]:
                ids = torch.full((cols[0].shape[0],), -1.0, dtype=torch.float64, device=device)   # fails the check below
            cols.append(ids[:, None])
        rows = torch.cat(cols, 1)
    else:
        rows = torch.empty((0, 0), dtype=torch.float64, device=device)
    rows = D.allgather_varlen(rows, group)
    if rows.shape[0] == 0:
        raise ValueError("inference: no rank forwarded any patient")
    C = rows.shape[1] // 3
    if rows.shape[1] % 3:                                         # the id column: some rank passed patient_ids
        ids = rows[:, 3 * C]
        order = torch.argsort(ids, stable=True)
        if not torch.equal(ids[order], torch.arange(rows.shape[0], dtype=torch.float64, device=rows.device)):
            raise ValueError("inference: the gathered patient_ids are not a permutation of 0..N-1 (N = %d); every rank "
                             "passes one global patient index per row it forwards" % rows.shape[0])
        rows = rows[order]
    return rows[:, :C].to(torch.float32), rows[:, C:2 * C], rows[:, 2 * C:3 * C]


@torch.no_grad()
def predict_risks(model, batches, device, gradcam=None, group=None, patient_ids=None):
    """Eval-mode forward of every patient once (batched). Returns (preds [N,C], events [N,C], durations [N,C]).
    gradcam: optional callable(batch_index, maps).  Each batch then goes through utils.attention_maps (the same forward
    plus ONE map kernel) and the callable receives that batch's maps [B, C, X, Y, Z] on the device -- the batched form of
    the reference's per-patient GradCAM loop (/root/reference/main.py:750-887).  Maps are not kept here (at 10 000
    patients of 128x128x64 they would be 80 GB): the callable writes or reduces them.  The predictions are the same
    bits either way.

    Data parallel (a torch.distributed `group` of more than one rank; group=None is one process): `batches` is this
    rank's shard, and each rank forwards only its own patients.  The rows of all ranks are then gathered, so every rank
    returns the same global tensors: in global patient order when `patient_ids` is given (1-D int64, the global index
    of each of this rank's rows in iteration order, e.g. distributed.shard_patients(N, rank, world); ValueError unless
    the gathered ids are a permutation of 0..N-1), otherwise rank-major.  Events and durations come back as float64.
    A rank may have no batches.  GradCAM maps stay on the rank that computed them: `batch_index` counts this rank's
    batches, so batch k holds the global patients patient_ids[s:s + B_k], s being the rows of batches 0..k-1."""
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
    if _world(group) > 1:
        return _gather_patients(preds, ev, du, patient_ids, group, device)
    return torch.cat(preds), torch.cat(ev), torch.cat(du)


def _draw_resamples(n, num_resamples, seed):
    """[R, N] bootstrap resamples of patient indices from RandomState(seed), or the global np.random when seed is None.
    sklearn.utils.resample(uids) == uids[RandomState.randint(0, n, n)]  (SURVEY.md appendix B.3)."""
    rng = np.random.RandomState(seed) if seed is not None else np.random
    return np.stack([rng.randint(0, n, n) for _ in range(num_resamples)])


def _broadcast_resamples(n, num_resamples, seed, group, device):
    """int32 [R, N] bootstrap resample matrix on `device`, the same on every rank: rank 0 draws it (_draw_resamples, as
    the one-process path of inference_survival does) and broadcasts it."""
    dev = D.comm_device(device, group)
    if dist.get_rank(group) == 0:
        idx = torch.as_tensor(_draw_resamples(n, num_resamples, seed)).to(device=dev, dtype=torch.int32)
    else:
        idx = torch.empty((num_resamples, n), dtype=torch.int32, device=dev)
    dist.broadcast(idx, group_src=0, group=group)
    return idx.to(device)


def _bootstrap_split(preds, events, durations, num_resamples, seed, group):
    """bootstrap_cindices over the ranks of `group`: each rank counts its split_rows(R) rows of the broadcast resample
    matrix, and the int64 counts are all-gathered, so every rank summarises the same [R, C, 3] counts as one process."""
    idx = _broadcast_resamples(preds.shape[0], num_resamples, seed, group, preds.device)
    lo, hi = D.split_rows(num_resamples, dist.get_rank(group), dist.get_world_size(group))
    if hi > lo:
        counts = _resample_counts(preds, events, durations, idx[lo:hi])
    else:
        counts = torch.empty((0, NUM_CLASSES, 3), dtype=torch.int64, device=preds.device)
    return bootstrap_from_counts(D.allgather_varlen(counts, group).cpu().numpy())


def inference_survival(model, batches, device, bootstrap=True, num_resamples=NUM_BOOTSTRAP_ITERATIONS, seed=None, gradcam=None,
                       group=None, patient_ids=None):
    """Risks of every patient, then the C-indices (bootstrap: per-resample, mean, std).  gradcam, group, patient_ids: see
    predict_risks.  Under a group of more than one rank every rank returns the same result: the gathered predictions of
    all patients, and the C-indices one process computes from those predictions.  Rank 0 draws the resamples
    (RandomState(seed), or the global np.random when seed is None; the other ranks' np.random is not advanced) and the
    ranks split the counting.  A prediction depends slightly on its batch mates (up to ~1e-4 between batches of 4 and
    11), so it matches a one-process run over other batches to within rounding, not bit for bit (DESIGN.md section 8)."""
    preds, events, durations = predict_risks(model, batches, device, gradcam=gradcam, group=group, patient_ids=patient_ids)
    n = preds.shape[0]
    if not bootstrap:
        return getCIndices(preds, events, durations), preds
    if _world(group) > 1:
        c, mean, std = _bootstrap_split(preds, events, durations, num_resamples, seed, group)
        return SimpleNamespace(per_resample=c, mean=mean, std=std, preds=preds)
    idx = _draw_resamples(n, num_resamples, seed)
    c, mean, std, _ = bootstrap_cindices(preds, events, durations, torch.as_tensor(idx, device=preds.device))
    return SimpleNamespace(per_resample=c, mean=mean, std=std, preds=preds)
