"""Data-parallel host logic on CPU with world_size 2 (gloo): patient sharding, SUM gradient all-reduce == gradient
accumulation over the same micro-batches (the reference's semantics, /root/reference/main.py:469,478-481), skipping of
parameters that never get a gradient, all-gather of per-rank predictions."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p


def _worker(rank, world, port, ret):
    # no CUDA in the workers: the host logic runs on the CPU even on a machine with fewer GPUs than ranks
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank),
                      CUDA_VISIBLE_DEVICES="")
    from mmnn_sts_b200 import distributed as D
    r, w, dev = D.init_from_env(backend="gloo")
    assert (r, w) == (rank, world) and dev.type == "cpu"
    torch.manual_seed(0)
    model = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.ReLU(), torch.nn.Linear(5, 2))
    unused = torch.nn.Linear(3, 3)                       # never receives a gradient (like class_layers.out / dense6)
    params = list(model.parameters()) + list(unused.parameters())
    x = torch.randn(8, 6, generator=torch.Generator().manual_seed(1)); y = torch.randn(8, 2, generator=torch.Generator().manual_seed(2))
    shard = D.shard_patients(8, rank, world)
    assert shard.tolist() == list(range(rank, 8, world))
    loss = ((model(x[shard]) - y[shard]) ** 2).sum()
    loss.backward()
    D.GradientAllReducer(params, bucket_bytes=64)(model)    # tiny buckets: exercises multi-bucket path
    # single-process reference: accumulate both micro-batches
    torch.manual_seed(0)
    ref = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.ReLU(), torch.nn.Linear(5, 2))
    for rr in range(world):
        s = D.shard_patients(8, rr, world)
        ((ref(x[s]) - y[s]) ** 2).sum().backward()
    ok = all(torch.allclose(p.grad, q.grad, atol=1e-6) for p, q in zip(model.parameters(), ref.parameters()))
    ok = ok and all(p.grad is None for p in unused.parameters())
    gathered = D.allgather_rows(torch.full((2, 3), float(rank)))
    ok = ok and gathered.shape == (2 * world, 3) and gathered[:2].eq(0).all() and gathered[2:].eq(1).all()
    ret[rank] = bool(ok)
    dist.barrier()
    dist.destroy_process_group()


def test_gradient_allreduce_equals_accumulation_world2():
    port = _free_port()
    with mp.Manager() as mgr:
        ret = mgr.dict()
        mp.spawn(_worker, args=(2, port, ret), nprocs=2, join=True)
        assert ret.get(0) is True and ret.get(1) is True, dict(ret)
