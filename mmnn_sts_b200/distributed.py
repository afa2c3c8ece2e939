"""Data-parallel plumbing: one process per GPU, patients sharded by rank, gradients all-reduced with NCCL.

The reference has no distributed code (SURVEY.md section 2a).  Semantics chosen so that "B patients per GPU on G GPUs"
equals the reference accumulating G micro-batches of B patients before one optimizer step (/root/reference/main.py:
469,478-481): BatchNorm statistics and the Cox risk set stay rank-local, gradients are SUMMED (not averaged).
There is no data-path collective in training: the only exchange is the gradient all-reduce (payload 11.3 M fp32 = 45 MB).
Inference (main.inference_survival with a group) gathers the per-rank risks with allgather_varlen and splits the
bootstrap resamples with split_rows."""
import os

import torch
import torch.distributed as dist


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
