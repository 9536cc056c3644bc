"""CPU tests of parallel.gather_slices, the exchange between the phases of ops.ShardedLosses: every rank's send slice
lands in the gathered buffer in rank order, byte for byte, on every rank (world_size-3 gloo group), and without a
process group the buffer is the rank's own slice."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _slice(rank, n):
    return (torch.arange(n, dtype=torch.int64) * 7 + 31 * rank + 1).remainder(256).to(torch.uint8)


def _worker(rank, world_size, port, n, ret):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world_size)
    try:
        from team_b200 import parallel
        send = _slice(rank, n)
        gathered = torch.full((world_size * n,), 255, dtype=torch.uint8)
        parallel.gather_slices(send, gathered)
        ret[rank] = gathered.tolist()
    finally:
        dist.destroy_process_group()


def test_gather_slices_is_rank_major_on_every_rank():
    world, n = 3, 1000
    ret = mp.Manager().dict()
    mp.spawn(_worker, args=(world, _free_port(), n, ret), nprocs=world, join=True)
    want = torch.cat([_slice(r, n) for r in range(world)]).tolist()
    for r in range(world):
        assert ret[r] == want, r


def test_gather_slices_without_a_process_group_copies_the_slice():
    from team_b200 import parallel
    send = _slice(0, 96)
    gathered = torch.zeros(96, dtype=torch.uint8)
    parallel.gather_slices(send, gathered)
    assert torch.equal(gathered, send)
