"""N > 1 host logic on CPU: world_size-2 gloo processes exercise the sharding, the weight replication and the one
all_gather of code maps (SURVEY.md 8e).  No kernels run here."""
import os
import socket
import sys
from unittest import mock

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    for p in (ROOT, os.path.join(ROOT, "rq-vae-transformer_b200")):
        if p not in sys.path:
            sys.path.insert(0, p)
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    from rqvae.utils import dist as rdist
    from tests.test_host_cpu import make_ar

    class A:
        dist_backend, timeout = "gloo", 60

    env = rdist.initialize(A())
    assert env.world_size == world and env.world_rank == rank and env.master == (rank == 0)
    # different init per rank -> identical after the flat broadcast
    torch.manual_seed(100 + rank)
    model = make_ar("tiny")
    box = rdist.dataparallel_and_sync(env, model)
    ref = [torch.zeros_like(p) for p in model.state_dict().values()]
    chk = torch.stack([p.double().sum() for p in box.module.state_dict().values()])
    gathered = [torch.zeros_like(chk) for _ in range(world)]
    dist.all_gather(gathered, chk)
    assert all(torch.equal(g, gathered[0]) for g in gathered)
    # independent images: shard a global batch, "sample" codes locally (seed + rank), all_gather the code maps
    lo, hi = rdist.shard_batch(env, 10)
    g = torch.Generator().manual_seed(1234 + rank)
    local = torch.randint(0, 512, (5, 4, 4, 4), generator=g)[: hi - lo]
    codes = rdist.all_gather_cat(env, local)
    assert codes.shape == (10, 4, 4, 4) and codes.dtype == torch.int64
    exp = torch.cat([torch.randint(0, 512, (5, 4, 4, 4), generator=torch.Generator().manual_seed(1234 + r)) for r in range(world)])
    assert torch.equal(codes, exp)
    dist.barrier()
    dist.destroy_process_group()
    q.put((rank, lo, hi))


def test_two_rank_gloo_sharding_and_gather():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    # CPU-only ranks: with a GPU visible, rank r would claim cuda:r, which a one-GPU machine does not have
    with mock.patch.dict(os.environ, {"CUDA_VISIBLE_DEVICES": ""}):
        for p in procs:
            p.start()
    for p in procs:
        p.join(120)
        assert p.exitcode == 0
    got = sorted(q.get() for _ in range(2))
    assert got == [(0, 0, 5), (1, 5, 10)]
