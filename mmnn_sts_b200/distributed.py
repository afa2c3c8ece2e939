"""Data-parallel plumbing: one process per GPU, patients sharded by rank, gradients all-reduced with NCCL.

The reference has no distributed code (SURVEY.md section 2a).  Semantics chosen so that "B patients per GPU on G GPUs"
equals the reference accumulating G micro-batches of B patients before one optimizer step (/root/reference/main.py:
469,478-481): the batch statistics of a forward and the Cox risk set stay within the micro-batch, gradients are SUMMED
(not averaged).  Within a step the only data-path exchange is the gradient all-reduce (payload 11.3 M fp32 = 45 MB).
main.train_survival with a group steps on the global micro-batch count (accumulation_rounds), gives a rank without a
micro-batch in a round zero gradients (fill_missing_grads), merges the BatchNorm running statistics at every step
(RunningStatsMerger) and gathers the epoch's rows in global order (allgather_ordered).
Inference (main.inference_survival with a group) gathers the per-rank risks with allgather_varlen and splits the
bootstrap resamples with split_rows."""
import os

import torch
import torch.distributed as dist
from torch.nn.modules.batchnorm import _BatchNorm


def init_from_env(backend=None):
    """Reads RANK / LOCAL_RANK / WORLD_SIZE / MASTER_ADDR / MASTER_PORT (torchrun). Returns (rank, world, device)."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    use_cuda = torch.cuda.is_available()
    device = torch.device("cuda", local) if use_cuda else torch.device("cpu")
    if use_cuda:
        torch.cuda.set_device(device)
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group(backend or ("nccl" if use_cuda else "gloo"), rank=rank, world_size=world)
    return rank, world, device


def shard_patients(num_patients, rank, world, permutation=None):
    """Rank r takes patients perm[r::world] (SURVEY.md section 8e)."""
    perm = permutation if permutation is not None else torch.arange(num_patients)
    return perm[rank::world]


def shard_batches(batches, rank, world):
    """Rank r's round-robin share batches[r::world] of a sequence of micro-batches: local micro-batch i of rank r is
    global micro-batch i * world + r, the split main.train_survival expects under a group."""
    return batches[rank::world]


def check_interval(interval, world):
    """ValueError unless `interval` (micro-batches per optimiser step) is a positive integer multiple of `world`: only
    then does every round of `interval` global micro-batches give each rank the same number of them."""
    if interval != int(interval) or int(interval) < 1 or int(interval) % world:
        raise ValueError("data-parallel training needs 64 / batch_size = %s micro-batches per optimiser step to be an "
                         "integer multiple of the %d ranks" % (interval, world))
    return int(interval)


def check_round_robin(counts, what="micro-batches"):
    """ValueError unless `counts` (one per rank) are the sizes of a round-robin split of their sum, as shard_batches
    makes them."""
    n, world = sum(counts), len(counts)
    want = [len(range(r, n, world)) for r in range(world)]
    if list(counts) != want:
        raise ValueError("per-rank %s counts %s are not a round-robin split of %d (expected %s): shard with "
                         "distributed.shard_batches" % (what, list(counts), n, want))
    return n


def accumulation_rounds(counts, interval):
    """[(lo, hi)]: the global micro-batch ranges of one epoch's optimiser steps, given every rank's local micro-batch
    count (round-robin shards) and `interval` micro-batches per step.  One process steps after micro-batches
    hi - 1 of these ranges: every `interval`-th one and the last."""
    interval = check_interval(interval, len(counts))
    n = check_round_robin(counts)
    return [(lo, min(lo + interval, n)) for lo in range(0, n, interval)]


def allgather_counts(counts, device, group=None):
    """Every rank's list of integer counts (same length on every rank): [[rank 0's], [rank 1's], ...]."""
    dev = comm_device(device, group)
    t = torch.tensor(counts, dtype=torch.int64, device=dev)
    out = [torch.empty_like(t) for _ in range(dist.get_world_size(group))]
    dist.all_gather(out, t, group=group)
    return [o.tolist() for o in out]


def fill_missing_grads(reducer):
    """Before `reducer(model)` in a round where some rank may have done no backward: every parameter that has a
    gradient on SOME rank gets one on this rank too, zeros where it has none, so that every rank enters the same
    collectives in GradientAllReducer.  Costs one all-reduce of a per-parameter int32 flag.

    A module with a flat gradient buffer (the DenseNet trunk) gets its zeros from `pack_flat_grad()`, which backs every
    parameter's .grad with views of one buffer, so that flat_grad_buffer() is not None on any rank and all of them
    reduce that module with one collective."""
    params, group = reducer.params, reducer.group
    if not params:
        return
    has = torch.tensor([p.grad is not None for p in params], dtype=torch.int32, device=comm_device(params[0].device, group))
    dist.all_reduce(has, op=dist.ReduceOp.MAX, group=group)
    need = {id(p) for p, h in zip(params, has.tolist()) if h}
    for m in reducer.flat_modules:
        if any(id(p) in need for p in m.parameters()):
            m.pack_flat_grad()
    for p in params:
        if p.grad is None and id(p) in need:
            p.grad = torch.zeros_like(p)


class RunningStatsMerger:
    """BatchNorm running statistics over the ranks of `group` equal to one process forwarding the same global
    micro-batches in order, with no kernel change.

    A training forward applies r <- a r + m x (a = 1 - m) to each running buffer.  Over a round of n global
    micro-batches one process ends with r_end = a^n r_start + sum_k m a^(n-1-k) x_k.  Each rank snapshots the buffers
    before each of its forwards (`before_forward`), recovers d_k = u_after - a u_before = m x_k after it
    (`after_forward(k)`, k = the micro-batch's position in the round), and accumulates S += a^(n-1-k) d_k in float64 on
    the device.  `merge()` all-reduces S together with the num_batches_tracked increments and sets r = a^n r_start + S
    and num_batches_tracked = its value at `begin` + the summed increments.  Between `begin` and `merge` a rank's
    buffers hold its own local EMA.  Tracks every _BatchNorm with running statistics; `momentum=None` (cumulative
    average) is refused with ValueError, and `momentum` must be what the module's forward applies."""

    def __init__(self, model, group=None):
        self.group = group
        mods = [m for m in model.modules() if isinstance(m, _BatchNorm) and m.track_running_stats]
        for m in mods:
            if m.momentum is None:
                raise ValueError("RunningStatsMerger: a BatchNorm with momentum=None (cumulative moving average) cannot "
                                 "be merged over ranks")
        self.stats = [t for m in mods for t in (m.running_mean, m.running_var)]
        self.counts = [m.num_batches_tracked for m in mods]
        if not mods:
            return
        dev = self.stats[0].device
        self._numel = sum(t.numel() for t in self.stats)
        self._decay = torch.cat([torch.full((t.numel(),), 1.0 - m.momentum, dtype=torch.float64)
                                 for m in mods for t in (m.running_mean, m.running_var)]).to(dev)
        # fp32 snapshots as views of flat buffers, built once: the copies are single multi-tensor launches (same dtype)
        # and the float64 arithmetic runs on the flat buffers, so a micro-batch costs a handful of launches
        self._start, self._before, self._after = (torch.empty(self._numel, dtype=torch.float32, device=dev) for _ in range(3))
        self._start_v, self._before_v, self._after_v = (self._views(f) for f in (self._start, self._before, self._after))
        self._acc = torch.zeros(self._numel + len(self.counts), dtype=torch.float64, device=dev)   # [S | increments]
        self._count_start = torch.empty(len(self.counts), dtype=torch.int64, device=dev)
        self._n = 0

    def _views(self, flat):
        out, off = [], 0
        for t in self.stats:
            out.append(flat[off:off + t.numel()].view(t.shape))
            off += t.numel()
        return out

    def begin(self, n):
        """Start a round of `n` global micro-batches (every rank calls it, with the same n)."""
        self._n = n
        if not self.counts:
            return
        torch._foreach_copy_(self._start_v, self.stats)
        torch.stack(self.counts, out=self._count_start)
        self._acc.zero_()

    def before_forward(self):
        if self.counts:
            torch._foreach_copy_(self._before_v, self.stats)

    def after_forward(self, k):
        """After the training forward of the round's k-th global micro-batch (0-based)."""
        if not self.counts:
            return
        torch._foreach_copy_(self._after_v, self.stats)
        d = self._after.double().addcmul_(self._decay, self._before.double(), value=-1.0)     # d_k = m x_k
        self._acc[:self._numel].addcmul_(self._decay.pow(self._n - 1 - k), d)

    def merge(self):
        """Set every rank's buffers to the one-process values at the end of the round (a collective)."""
        if not self.counts:
            return
        self._acc[self._numel:] = torch.stack(self.counts) - self._count_start
        dev = comm_device(self._acc.device, self.group)
        acc = self._acc.to(dev)
        dist.all_reduce(acc, op=dist.ReduceOp.SUM, group=self.group)
        acc = acc.to(self._acc.device)
        self._after.copy_(self._decay.pow(self._n) * self._start.double() + acc[:self._numel])
        torch._foreach_copy_(self.stats, self._after_v)
        torch._foreach_copy_(self.counts, list((self._count_start + acc[self._numel:].to(torch.int64)).unbind()))


class GradientAllReducer:
    """Gradient all-reduce (SUM by default).  Parameters that never receive a gradient (the reference's unused
    class_layers.out / dense6 / modality heads, SURVEY.md section 7 hard part 9) are skipped.

    The DenseNet trunk keeps all its gradients in ONE flat buffer and finalises them block by block (last block first).
    With `overlap=True` (default) the reducer hooks the trunk: right after backward has been ENQUEUED it queues one
    all-reduce per gradient group on a communication stream that waits for the group's gradient-ready event
    (`mmnn_encoder_wait_grad_group`), so the reduction of blocks 4, 3, 2 runs while blocks 3, 2, 1 and the stem are still
    in backward; `__call__` (before `optimizer.step()`) then only waits for those collectives and reduces the few small
    head / MLP tensors in one extra bucket.  The overlap must be requested per backward with `arm()` -- only a backward
    that starts from empty gradients and is followed directly by the optimiser step may be reduced early (with gradient
    accumulation the earlier micro-batches must not be reduced on their own).  MMNN_DP_OVERLAP=0, or never calling
    `arm()`, falls back to one all-reduce of the flat buffer after backward."""

    def __init__(self, params, bucket_bytes=64 << 20, average=False, group=None, model=None, overlap=True):
        self.params = [p for p in params if p.requires_grad]
        self.bucket_bytes = bucket_bytes
        self.average = average
        self.group = group
        # modules that keep their gradients in one flat buffer (the DenseNet trunk) are reduced in place, without packing
        self.flat_modules = [m for m in model.modules() if hasattr(m, "flat_grad_buffer")] if model is not None else []
        self._inflight = {}
        self._comm_stream = None
        self._armed = False
        if overlap and os.environ.get("MMNN_DP_OVERLAP", "1") != "0":
            for m in self.flat_modules:
                if hasattr(m, "grad_groups"):
                    m.grad_group_hook = self._on_trunk_backward

    def arm(self):
        """Call right before the `loss.backward()` whose gradients go straight to `optimizer.step()` (no accumulation)."""
        self._armed = True

    def _on_trunk_backward(self, backbone, flat):
        armed, self._armed = self._armed, False
        if not armed or not dist.is_initialized() or dist.get_world_size(self.group) == 1 or not flat.is_cuda:
            return
        if any(p.grad is not None for p in backbone.parameters()):
            return                                   # accumulating into existing gradients: reduce after backward instead
        if self._comm_stream is None:
            self._comm_stream = torch.cuda.Stream(device=flat.device)
        comm = self._comm_stream
        flat.record_stream(comm)
        works = []
        for k, (lo, hi) in enumerate(backbone.grad_groups()):
            backbone.wait_grad_group(k, comm)
            with torch.cuda.stream(comm):
                works.append(dist.all_reduce(flat[lo:hi], op=dist.ReduceOp.SUM, group=self.group, async_op=True))
        self._inflight[id(backbone)] = (works, flat)

    def __call__(self, *_):
        if not dist.is_initialized() or dist.get_world_size(self.group) == 1:
            return
        world = dist.get_world_size(self.group)
        pending_flat, covered = [], set()
        for m in self.flat_modules:
            flat = m.flat_grad_buffer()
            started = self._inflight.pop(id(m), None)
            if flat is not None and started is not None and started[1] is flat:
                for w in started[0]:                      # per-group collectives queued during backward
                    pending_flat.append((w, None))
                if self.average:
                    pending_flat.append((None, flat))
                covered.update(id(p) for p in m.parameters())
            elif flat is not None:
                if started is not None:
                    for w in started[0]:
                        w.wait()
                pending_flat.append((dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True), flat))
                covered.update(id(p) for p in m.parameters())
        grads = [p.grad for p in reversed(self.params) if p.grad is not None and id(p) not in covered]
        buckets, cur, size = [], [], 0
        for g in grads:
            cur.append(g); size += g.numel() * g.element_size()
            if size >= self.bucket_bytes:
                buckets.append(cur); cur, size = [], 0
        if cur:
            buckets.append(cur)
        pending = []
        for b in buckets:
            flat = torch.cat([g.reshape(-1) for g in b])
            work = dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=self.group, async_op=True)
            pending.append((work, flat, b))
        for work, flat in pending_flat:
            if work is not None:
                work.wait()
            if self.average and flat is not None:
                flat.div_(world)
        for work, flat, b in pending:
            work.wait()
            if self.average:
                flat.div_(world)
            off = 0
            for g in b:
                n = g.numel()
                g.copy_(flat[off:off + n].view_as(g))
                off += n


def allgather_rows(t, group=None):
    """All-gather of per-rank row blocks (predictions / targets for the per-epoch C-index and updateWeights)."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return t
    out = [torch.empty_like(t) for _ in range(dist.get_world_size(group))]
    dist.all_gather(out, t.contiguous(), group=group)
    return torch.cat(out, dim=0)


def comm_device(device, group=None):
    """Device on which a collective of `group` takes tensors that live on `device`: that device under NCCL, the host
    under any other backend (gloo exchanges host memory)."""
    return torch.device(device) if dist.get_backend(group) == dist.Backend.NCCL else torch.device("cpu")


def split_rows(n, rank, world):
    """[lo, hi): the contiguous share of `n` rows that `rank` of `world` takes.  Every row goes to exactly one rank; the
    first n % world ranks take one row more, and when n < world the last ranks take none."""
    q, r = divmod(n, world)
    lo = rank * q + min(rank, r)
    return lo, lo + q + (1 if rank < r else 0)


def allgather_varlen(t, group=None):
    """All-gather of per-rank row blocks whose row counts differ (zero included), concatenated in rank order.

    The ranks first exchange their shapes [rows, *row_shape], then every block is padded to the largest row count,
    gathered and trimmed.  All ranks pass the same dtype and number of dimensions; the non-empty blocks must agree on the
    row shape, and a rank with no rows may pass any row shape (it cannot know the others'), e.g. torch.empty(0, 0).
    A mismatch raises ValueError on every rank.  Under NCCL `t` is a CUDA tensor; under gloo the exchange goes through
    host memory and the result is moved back to `t`'s device."""
    if not dist.is_initialized() or dist.get_world_size(group) == 1:
        return t
    world = dist.get_world_size(group)
    dev = comm_device(t.device, group)
    head = torch.tensor(t.shape, dtype=torch.int64, device=dev)
    heads = [torch.empty_like(head) for _ in range(world)]
    dist.all_gather(heads, head, group=group)
    heads = [h.tolist() for h in heads]
    counts = [h[0] for h in heads]
    row_shapes = {tuple(h[1:]) for h in heads if h[0] > 0}
    if len(row_shapes) > 1:
        raise ValueError("allgather_varlen: ranks disagree on the row shape: %s" % sorted(row_shapes))
    m = max(counts)
    if m == 0:
        return t
    row_shape = row_shapes.pop()
    block = torch.zeros((m,) + row_shape, dtype=t.dtype, device=dev)
    if counts[dist.get_rank(group)]:
        block[:t.shape[0]] = t
    out = [torch.empty_like(block) for _ in range(world)]
    dist.all_gather(out, block, group=group)
    return torch.cat([o[:c] for o, c in zip(out, counts)]).to(t.device)


def allgather_ordered(rows, group=None):
    """allgather_varlen of float64 rows [n, 2 + w] whose first two columns are integer keys (global micro-batch index,
    row index within it), returned sorted by (micro-batch, row) without the key columns: the rows of round-robin
    shards in the order one process sees them.  A rank without rows passes torch.empty(0, 0)."""
    rows = allgather_varlen(rows, group)
    if rows.shape[0] == 0:
        return rows
    rows = rows[torch.argsort(rows[:, 1], stable=True)]
    rows = rows[torch.argsort(rows[:, 0], stable=True)]
    return rows[:, 2:]
