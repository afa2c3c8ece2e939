"""Starting torch.distributed ranks from a test with mp.spawn, with a deadline."""
import socket
import time

import pytest
import torch.multiprocessing as mp


def spawn_ranks(fn, world, args, timeout=300):
    """mp.spawn(fn, args=(world, port) + args) joined with a deadline: ranks still running after `timeout` seconds are
    killed and the test fails, so no rank outlives the test."""
    ctx = mp.spawn(fn, args=(world, _free_port()) + tuple(args), nprocs=world, join=False)
    deadline = time.monotonic() + timeout
    while not ctx.join(timeout=5):
        if time.monotonic() > deadline:
            for p in ctx.processes:
                p.kill()
            for p in ctx.processes:
                p.join()
            pytest.fail("ranks still running after %d s" % timeout)


def _free_port():
    s = socket.socket(); s.bind(("127.0.0.1", 0)); p = s.getsockname()[1]; s.close()
    return p
