"""Data-parallel survival training host logic on the CPU (gloo ranks started with mp.spawn): the global step schedule,
the merge of BatchNorm running statistics over ranks, a round in which one rank has no micro-batch, and the ordered
gather of the epoch's rows.  A mistake in the collective logic shows up as a hang, so every multi-rank case runs under
spawn_ranks' deadline."""
import os
from types import SimpleNamespace

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.dp_helpers import spawn_ranks


def _one_process_steps(nb, interval):
    """Where one process steps: after every `interval`-th micro-batch and after the last (mmnn_sts_b200.main)."""
    return [i for i in range(nb) if (i + 1) % interval == 0 or i == nb - 1]


@pytest.mark.parametrize("nb,interval,world", [(9, 8, 2), (9, 8, 4), (72, 4, 4), (8, 4, 2), (3, 4, 4), (1, 2, 2), (17, 2, 2),
                                               (5, 1, 1), (12, 6, 3)])
def test_rounds_step_where_one_process_steps(nb, interval, world):
    from mmnn_sts_b200.distributed import accumulation_rounds, shard_batches
    counts = [len(shard_batches(list(range(nb)), r, world)) for r in range(world)]
    rounds = accumulation_rounds(counts, interval)
    assert [hi - 1 for _, hi in rounds] == _one_process_steps(nb, interval)
    assert rounds[0][0] == 0 and all(a[1] == b[0] for a, b in zip(rounds, rounds[1:])) and rounds[-1][1] == nb
    # every rank's local micro-batches of a round are the global ones it holds
    for r in range(world):
        mine = shard_batches(list(range(nb)), r, world)
        assert sum((list(range(lo + r, hi, world)) for lo, hi in rounds), []) == mine


@pytest.mark.parametrize("interval,world", [(8, 3), (4, 8), (2.5, 1), (6, 4), (0, 1)])
def test_rounds_refuse_an_interval_that_is_not_a_multiple_of_the_world(interval, world):
    from mmnn_sts_b200.distributed import accumulation_rounds
    with pytest.raises(ValueError, match="multiple"):
        accumulation_rounds([1] * world, interval)


@pytest.mark.parametrize("counts", [[1, 2], [3, 1], [2, 2, 0], [1, 0, 1]])
def test_rounds_refuse_counts_that_are_not_round_robin(counts):
    from mmnn_sts_b200.distributed import accumulation_rounds
    with pytest.raises(ValueError, match="round-robin"):
        accumulation_rounds(counts, 4 if len(counts) == 2 else 3)


# ---------------------------------------------------------------------------------------------------- gloo scenarios
def _schedule(rank, world):
    """Counts exchanged over the group: the good split gives every rank the same rounds, and a bad interval or a
    split that is not round-robin raises on EVERY rank -- also through train_survival itself."""
    from mmnn_sts_b200 import distributed as D
    from mmnn_sts_b200.main import train_survival
    cpu, g = torch.device("cpu"), dist.group.WORLD
    counts = D.allgather_counts([len(range(rank, 9, world)), 0], cpu, g)
    assert D.accumulation_rounds([c[0] for c in counts], 8) == [(0, 8), (8, 9)]
    counts = D.allgather_counts([2 if rank == 0 else 4, 0], cpu, g)
    with pytest.raises(ValueError, match="round-robin"):
        D.accumulation_rounds([c[0] for c in counts], 8)
    model = torch.nn.Linear(3, 2)
    batch = ({"clinical": torch.zeros(4, 3)}, torch.zeros(4, 2), torch.ones(4, 2))
    args = SimpleNamespace(lr=1e-3, momentum=0.9, weight_decay=0.0, epochs=1, batch_size=8, blend=False, blend_update_interval=1,
                           num_train=8 * 9)
    with pytest.raises(ValueError, match="multiple"):           # 64 / 24 micro-batches per step: before any collective
        train_survival(model, [batch], None, SimpleNamespace(**{**vars(args), "batch_size": 24}), cpu, group=g)
    with pytest.raises(ValueError, match="round-robin"):        # rank 0: 2 micro-batches, rank 1: 3
        train_survival(model, [batch] * (2 + rank), None, args, cpu, group=g)
    with pytest.raises(TypeError, match="len"):                 # rank 1 passes a one-shot generator
        train_survival(model, [batch] if rank == 0 else (b for b in [batch]), None, args, cpu, group=g)
    with pytest.raises(ValueError, match="grad_sync"):
        train_survival(model, [batch], None, args, cpu, grad_sync=lambda m: None, group=g)
    dist.barrier()


class _BNNet(torch.nn.Module):
    """BatchNorm1d (default momentum) and BatchNorm3d (momentum 0.3) on the CPU, as torch runs them."""

    def __init__(self, momentum=0.3):
        super().__init__()
        self.bn1 = torch.nn.BatchNorm1d(5)
        self.body = torch.nn.Sequential(torch.nn.Identity(), torch.nn.BatchNorm3d(3, momentum=momentum))

    def forward(self, x):
        return self.bn1(x["flat"]).sum() + self.body(x["vol"]).sum()


def _bn_batch(g):
    gen = torch.Generator().manual_seed(1000 + g)
    return {"flat": torch.randn(6, 5, generator=gen) * (1 + g) + g, "vol": torch.rand(4, 3, 2, 3, 2, generator=gen) * (2 + g) - g}


def _bn_merge(rank, world):
    """2 or 4 ranks forward alternating micro-batches of 2 rounds (interval 4, 6 micro-batches, so the last round is
    partial); after every merge the buffers equal one process's sequential fp32 EMA over the same micro-batches."""
    from mmnn_sts_b200 import distributed as D
    nb, interval = 6, 4
    torch.manual_seed(0)
    ref = _BNNet().train()
    net = _BNNet().train()
    net.load_state_dict(ref.state_dict())
    merger = D.RunningStatsMerger(net, dist.group.WORLD)
    for lo, hi in D.accumulation_rounds([len(range(r, nb, world)) for r in range(world)], interval):
        merger.begin(hi - lo)
        for g in range(lo + rank, hi, world):
            merger.before_forward()
            net(_bn_batch(g))
            merger.after_forward(g - lo)
        merger.merge()
        for g in range(lo, hi):
            ref(_bn_batch(g))
        for (k, a), b in zip(net.named_buffers(), ref.buffers()):
            if k.endswith("num_batches_tracked"):
                assert int(a) == int(b) == hi, (k, int(a), int(b))
            else:
                rel = float((a - b).abs().max() / b.abs().max())
                assert rel <= 1e-5, (k, hi, rel)
    with pytest.raises(ValueError, match="momentum=None"):
        D.RunningStatsMerger(torch.nn.Sequential(torch.nn.BatchNorm1d(2, momentum=None)), dist.group.WORLD)


class _FlatTrunk(torch.nn.Module):
    """Test stand-in for the DenseNet trunk's gradient layout: backward hands autograd its parameter gradients as views
    of one flat buffer, and flat_grad_buffer / grad_groups / pack_flat_grad behave as the trunk's do."""

    def __init__(self):
        super().__init__()
        self.w = torch.nn.Parameter(torch.randn(4, 3, generator=torch.Generator().manual_seed(7)))
        self.b = torch.nn.Parameter(torch.randn(4, generator=torch.Generator().manual_seed(8)))
        self._flat = None
        self.grad_group_hook = None

    def forward(self, x):
        return _FlatFn.apply(self, x, self.w, self.b)

    def grad_groups(self):
        return [(0, 16)]

    def flat_grad_buffer(self):
        f = self._flat
        if f is None or self.w.grad is None or self.b.grad is None:
            return None
        if self.w.grad.data_ptr() != f.data_ptr() or self.b.grad.data_ptr() != f[12:].data_ptr():
            return None
        return f

    def pack_flat_grad(self):
        f = self.flat_grad_buffer()
        if f is not None:
            return f
        f = torch.zeros(16)
        for p, (lo, hi) in zip((self.w, self.b), ((0, 12), (12, 16))):
            v = f[lo:hi].view(p.shape)
            if p.grad is not None:
                v.copy_(p.grad)
            p.grad = v
        self._flat = f
        return f


class _FlatFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, trunk, x, w, b):
        ctx.trunk = trunk
        ctx.save_for_backward(x, w)
        return x @ w.t() + b

    @staticmethod
    def backward(ctx, gy):
        x, w = ctx.saved_tensors
        flat = torch.zeros(16)
        flat[:12].view(4, 3).copy_(gy.t() @ x)
        flat[12:].copy_(gy.sum(0))
        ctx.trunk._flat = flat
        return None, gy @ w, flat[:12].view(4, 3), flat[12:]


class _Net(torch.nn.Module):
    def __init__(self):
        super().__init__()
        self.trunk = _FlatTrunk()
        self.head = torch.nn.Linear(4, 2)
        self.unused = torch.nn.Linear(2, 2)            # never receives a gradient (like the unused reference heads)
        torch.nn.init.constant_(self.head.weight, 0.1)

    def forward(self, x):
        return self.head(torch.tanh(self.trunk(x)))


def _mb(g):
    gen = torch.Generator().manual_seed(50 + g)
    return torch.randn(5, 3, generator=gen), torch.randn(5, 2, generator=gen)


def _empty_rank(rank, world, log):
    """3 ranks, 2 micro-batches in one round (interval 3): rank 2 does no backward.  After fill_missing_grads and the
    reducer every rank holds one process's accumulated gradients, and every rank entered the same collectives."""
    from mmnn_sts_b200 import distributed as D
    calls = []
    for name in ("all_reduce", "all_gather", "broadcast"):
        orig = getattr(dist, name)

        def logged(t, *a, _orig=orig, _name=name, **k):
            first = t[0] if isinstance(t, list) else t
            calls.append((_name, tuple(first.shape) if isinstance(t, torch.Tensor) else len(t), str(first.dtype)))
            return _orig(t, *a, **k)
        setattr(dist, name, logged)
    torch.manual_seed(0)
    net = _Net()
    reducer = D.GradientAllReducer(net.parameters(), group=dist.group.WORLD, model=net, bucket_bytes=16)
    assert reducer.flat_modules == [net.trunk]
    (lo, hi), = D.accumulation_rounds([len(range(r, 2, world)) for r in range(world)], 3)
    for g in range(lo + rank, hi, world):
        x, y = _mb(g)
        ((net(x) - y) ** 2).sum().backward()
    assert (net.trunk.w.grad is None) == (rank == 2)
    D.fill_missing_grads(reducer)
    assert net.trunk.flat_grad_buffer() is not None
    reducer(net)
    torch.manual_seed(0)
    ref = _Net()
    for g in range(2):
        x, y = _mb(g)
        ((ref(x) - y) ** 2).sum().backward()
    for (k, p), q in zip(net.named_parameters(), ref.parameters()):
        if k.startswith("unused"):
            assert p.grad is None and q.grad is None, k
        else:
            assert torch.allclose(p.grad, q.grad, atol=1e-6), (k, p.grad, q.grad)
    log[rank] = calls


def _ordered_gather(rank, world):
    """Round-robin shards of 5 micro-batches over 3 ranks, with a ragged last one: the rows come back in global
    micro-batch order, and main._gather_rows decodes [3, B, C] predictions (also on a rank without rows)."""
    from mmnn_sts_b200 import distributed as D
    from mmnn_sts_b200.main import _gather_rows, _keyed_rows
    cpu, g = torch.device("cpu"), dist.group.WORLD
    sizes = [4, 4, 4, 4, 2]
    ids = torch.arange(sum(sizes)).split(sizes)

    def mb(j):
        p = ids[j].double()
        preds = torch.stack([torch.stack([p + 0.25 * h, -p - 0.25 * h], 1) for h in range(3)]).float()
        return preds, torch.stack([p.long() % 2] * 2, 1), torch.stack([100 + p.long()] * 2, 1)

    for nb in (5, 2):                                   # nb = 2: rank 2 has no micro-batch
        mine = D.shard_batches(list(range(nb)), rank, world)
        rows = [_keyed_rows(j, *mb(j)) for j in mine]
        preds, ev, du = _gather_rows(rows, True, g, cpu)
        n = sum(sizes[:nb])
        want = torch.cat([mb(j)[0] for j in range(nb)], 1)
        assert preds.shape == (3, n, 2) and torch.equal(preds, want), (preds, want)
        assert ev[:, 0].tolist() == [p % 2 for p in range(n)] and du[:, 1].tolist() == [100 + p for p in range(n)]
        flat = D.allgather_ordered(torch.stack([torch.tensor([j, 0, 10.0 * j], dtype=torch.float64) for j in mine])
                                   if mine else torch.empty((0, 0), dtype=torch.float64), g)
        assert flat[:, 0].tolist() == [10.0 * j for j in range(nb)]


SCENARIOS = {"schedule": _schedule, "bn_merge": _bn_merge, "empty_rank": _empty_rank, "ordered_gather": _ordered_gather}


def _worker(rank, world, port, scenario, ret, log):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      CUDA_VISIBLE_DEVICES="")
    from mmnn_sts_b200 import distributed as D
    D.init_from_env(backend="gloo")
    try:
        if scenario == "empty_rank":
            _empty_rank(rank, world, log)
        else:
            SCENARIOS[scenario](rank, world)
        ret[rank] = "ok"
    except BaseException as ex:                          # reported by the parent: an assertion here only ends the child
        ret[rank] = repr(ex)[:2000]
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("scenario,world", [("schedule", 2), ("bn_merge", 2), ("bn_merge", 4), ("empty_rank", 3),
                                            ("ordered_gather", 3)])
def test_dp_train_gloo(scenario, world):
    with mp.Manager() as mgr:
        ret, log = mgr.dict(), mgr.dict()
        spawn_ranks(_worker, world, (scenario, ret, log), timeout=120)
        assert dict(ret) == {r: "ok" for r in range(world)}, dict(ret)
        log = dict(log)
    if scenario == "empty_rank":
        print("collectives of rank 0:", log[0])
        assert all(log[r] == log[0] for r in range(world)), log
