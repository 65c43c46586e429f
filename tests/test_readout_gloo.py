"""mrphy.parallel.allreduce_signal on CPU with the gloo backend, world_size 2: the readout of a spin shard is a partial sum."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank, world, port, ret):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, 'mrphy.py_b200'))
    from mrphy import parallel
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        # each rank's partial signal depends on its own leaf; the loss on the full signal is the same on every rank
        x = torch.arange(12, dtype=torch.float64).reshape(1, 2, 6).mul(rank + 1).requires_grad_(True)
        S = parallel.allreduce_signal(x * 2.0)
        tot = sum(r + 1 for r in range(world))
        ok = torch.equal(S.detach(), torch.arange(12, dtype=torch.float64).reshape(1, 2, 6) * 2.0 * tot)
        w = torch.linspace(-1, 1, 12, dtype=torch.float64).reshape(1, 2, 6)
        (S * w).sum().backward()
        ok &= torch.equal(x.grad, 2.0 * w)                        # backward: the identity on dL/dS
        ret[rank] = bool(ok)
    finally:
        dist.destroy_process_group()


def test_allreduce_signal_world2():
    world, port = 2, _free_port()
    with mp.Manager() as m:
        ret = m.dict()
        mp.spawn(_worker, args=(world, port, ret), nprocs=world, join=True)
        assert dict(ret) == {0: True, 1: True}


def test_allreduce_signal_without_process_group_is_identity():
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    sys.path.insert(0, os.path.join(root, 'mrphy.py_b200'))
    from mrphy import parallel
    S = torch.ones(2, 2, 3)
    assert parallel.allreduce_signal(S) is S
