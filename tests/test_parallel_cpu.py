"""CPU, world_size 2 over gloo: the scene-sharding host logic used by bench.py / multi-GPU sampling."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from diffuscene_b200.parallel import allreduce_gradients, gather_scenes, max_over_ranks, shard_range


def test_shard_range_partitions_exactly():
    for total in (1, 7, 8, 4096, 4097):
        for world in (1, 2, 3, 8):
            seen = []
            for r in range(world):
                off, cnt = shard_range(total, r, world)
                seen += list(range(off, off + cnt))
            assert seen == list(range(total))


def _run_two_ranks(target):
    """Start `target(rank, 2, port, q)` in two spawned processes and return what each put on q.  The port is one the
    OS just handed out, so that concurrent runs of the suite do not meet at the same rendezvous; a rank still alive
    when the test ends (its peer failed) is terminated rather than left waiting for the rendezvous."""
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=target, args=(r, 2, port, q)) for r in range(2)]
    try:
        for p in procs:
            p.start()
        res = [q.get(timeout=120) for _ in procs]
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
        return res
    finally:
        for p in procs:
            if p.is_alive():
                p.terminate()
                p.join()


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    total = 7
    off, cnt = shard_range(total, rank, world)
    local = torch.arange(off, off + cnt, dtype=torch.float32).reshape(cnt, 1, 1).expand(cnt, 2, 3).contiguous()
    full = gather_scenes(local, total)
    ms = max_over_ranks(10.0 + rank, torch.device("cpu"))
    q.put((rank, full[:, 0, 0].tolist(), ms))
    dist.destroy_process_group()


def test_two_rank_gather_and_timing_reduce():
    res = _run_two_ranks(_worker)
    for rank, scenes, ms in res:
        assert scenes == [float(i) for i in range(7)]       # global scene order, every scene exactly once
        assert ms == 11.0                                    # max over ranks


def _make_model():
    torch.manual_seed(3)
    return torch.nn.Sequential(torch.nn.Linear(6, 16), torch.nn.SiLU(), torch.nn.Linear(16, 4))


def _dp_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    model = _make_model()
    g = torch.Generator().manual_seed(11)
    x, y = torch.randn(8, 6, generator=g), torch.randn(8, 4, generator=g)
    xs, ys = x[rank * 4:(rank + 1) * 4], y[rank * 4:(rank + 1) * 4]          # equal per-rank batches
    ((model(xs) - ys) ** 2).mean().backward()
    n_coll = allreduce_gradients(model.parameters(), bucket_bytes=300)      # tiny buckets: several collectives
    q.put((rank, n_coll, [p.grad.tolist() for p in model.parameters()]))     # plain lists: no shared-memory handles
    dist.destroy_process_group()


def test_two_rank_gradient_mean_equals_full_batch_gradient():
    """Data-parallel training (SURVEY 8e): the bucketed all-reduce mean of per-rank gradients on equal shards is
    the gradient of the full-batch mean loss."""
    res = _run_two_ranks(_dp_worker)
    model = _make_model()
    g = torch.Generator().manual_seed(11)
    x, y = torch.randn(8, 6, generator=g), torch.randn(8, 4, generator=g)
    with torch.enable_grad():          # other test modules may leave autograd disabled in this process
        ((model(x) - y) ** 2).mean().backward()
    want = [p.grad for p in model.parameters()]
    for rank, n_coll, grads in res:
        assert n_coll >= 2
        for a, b in zip(grads, want):
            assert torch.allclose(torch.tensor(a), b, rtol=1e-5, atol=1e-7)
    assert allreduce_gradients(model.parameters()) == 0      # outside a process group: no-op
