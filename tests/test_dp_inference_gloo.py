"""Data-parallel inference host logic on the CPU (gloo ranks started with mp.spawn): allgather_varlen with uneven and
empty row blocks, split_rows, predict_risks putting the gathered rows in global patient order (and rejecting ids that
are not a permutation), and the broadcast bootstrap resample matrix being the one a single process draws."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from tests.dp_helpers import spawn_ranks


class _Echo(torch.nn.Module):
    """Stand-in model: the 'risk' of a patient is its first two clinical columns."""

    def forward(self, x):
        return x["clinical"][:, :2] * 1.0


def _patient_batches(ids, batch):
    """Batches of the given global patient ids: clinical [p, p + 0.5], event p % 2, duration 100 + p (per class)."""
    out = []
    for s in range(0, len(ids), batch):
        p = torch.as_tensor(ids[s:s + batch], dtype=torch.float32)
        clinical = torch.stack([p, p + 0.5], 1)
        out.append(({"clinical": clinical}, torch.stack([p.long() % 2] * 2, 1), torch.stack([100 + p.long()] * 2, 1)))
    return out


def _allgather(rank, world):
    from mmnn_sts_b200 import distributed as D
    counts = (5, 0, 3) if world == 3 else (0, 0)
    n = counts[rank]
    t = torch.arange(n * 4, dtype=torch.float64).reshape(n, 4) + 100 * rank if n else torch.empty((0, 0), dtype=torch.float64)
    got = D.allgather_varlen(t)
    if sum(counts) == 0:
        assert got.shape[0] == 0
    else:
        want = torch.cat([torch.arange(c * 4, dtype=torch.float64).reshape(c, 4) + 100 * r for r, c in enumerate(counts) if c])
        assert torch.equal(got, want), (got, want)
    ints = D.allgather_varlen(torch.full((n, 2, 3), rank, dtype=torch.int64))
    assert ints.dtype == torch.int64 and ints.shape == (sum(counts), 2, 3)
    assert ints[:, 0, 0].tolist() == sum(([r] * c for r, c in enumerate(counts)), [])
    with pytest.raises(ValueError, match="row shape"):
        D.allgather_varlen(torch.zeros((1, 3 + rank)))


def _order(rank, world):
    from mmnn_sts_b200 import distributed as D
    from mmnn_sts_b200.main import predict_risks
    g = dist.group.WORLD
    cpu = torch.device("cpu")
    for n in (7, 2):                                     # N = 2: the third rank has no patients
        ids = D.shard_patients(n, rank, world)
        preds, ev, du = predict_risks(_Echo(), _patient_batches(ids.tolist(), 2), cpu, group=g, patient_ids=ids)
        assert preds.dtype == torch.float32 and preds.shape == (n, 2)
        assert preds[:, 0].tolist() == list(range(n)) and preds[:, 1].tolist() == [p + 0.5 for p in range(n)]
        assert ev[:, 0].tolist() == [p % 2 for p in range(n)] and du[:, 1].tolist() == [100 + p for p in range(n)]
        # without ids: rank-major
        preds, _, _ = predict_risks(_Echo(), _patient_batches(ids.tolist(), 2), cpu, group=g)
        assert preds[:, 0].tolist() == sum((D.shard_patients(n, r, world).tolist() for r in range(world)), [])
    ids = D.shard_patients(7, rank, world)
    bad = {"duplicate": torch.where(ids == 6, 0, ids), "missing": ids + 1, "too few": ids[:1]}
    for what, b in bad.items():
        with pytest.raises(ValueError, match="permutation"):
            predict_risks(_Echo(), _patient_batches(ids.tolist(), 2), cpu, group=g, patient_ids=b)
    # one process: group=None ignores the other ranks and the ids
    preds, _, _ = predict_risks(_Echo(), _patient_batches(ids.tolist(), 2), cpu, patient_ids=ids)
    assert preds[:, 0].tolist() == ids.tolist()


def _resamples(rank, world):
    from mmnn_sts_b200.main import _broadcast_resamples
    g, cpu = dist.group.WORLD, torch.device("cpu")
    n, R = 11, 9
    got = _broadcast_resamples(n, R, 5, g, cpu)
    rng = np.random.RandomState(5)
    want = np.stack([rng.randint(0, n, n) for _ in range(R)])
    assert got.dtype == torch.int32 and np.array_equal(got.numpy(), want)
    np.random.seed(123 + rank)                           # only rank 0's global generator may be drawn from
    got = _broadcast_resamples(n, R, None, g, cpu)
    np.random.seed(123)
    want = np.stack([np.random.randint(0, n, n) for _ in range(R)])
    assert np.array_equal(got.numpy(), want)


SCENARIOS = {"allgather": _allgather, "order": _order, "resamples": _resamples}


def _worker(rank, world, port, scenario, ret):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      CUDA_VISIBLE_DEVICES="")
    from mmnn_sts_b200 import distributed as D
    D.init_from_env(backend="gloo")
    try:
        SCENARIOS[scenario](rank, world)
        ret[rank] = "ok"
    except BaseException as ex:                          # reported by the parent: an assertion here only ends the child
        ret[rank] = repr(ex)[:2000]
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("scenario,world", [("allgather", 2), ("allgather", 3), ("order", 3), ("resamples", 2)])
def test_dp_inference_gloo(scenario, world):
    with mp.Manager() as mgr:
        ret = mgr.dict()
        spawn_ranks(_worker, world, (scenario, ret))
        assert dict(ret) == {r: "ok" for r in range(world)}, dict(ret)


@pytest.mark.parametrize("n,world", [(3, 5), (4, 4), (10, 4), (1000, 8), (0, 3)])
def test_split_rows_covers_every_row_once(n, world):
    from mmnn_sts_b200.distributed import split_rows
    shares = [split_rows(n, r, world) for r in range(world)]
    assert shares[0][0] == 0 and shares[-1][1] == n
    assert all(a[1] == b[0] for a, b in zip(shares, shares[1:]))
    sizes = [hi - lo for lo, hi in shares]
    assert min(sizes) >= 0 and max(sizes) - min(sizes) <= 1 and sum(sizes) == n
