"""CPU, world_size 3, gloo: the host-side pieces of data-parallel IPR-CycleGAN / IPR-SRGAN training -- the image-pool
query on the gathered global batch (``dist.pool_query``) and the metrics reduction (``dist.reduce_metrics``) -- against
one pool fed the whole batch, as the reference's ``nn.DataParallel`` keeps it."""
import os
import socket

import torch
import torch.multiprocessing as mp

WORLD, PER_RANK, STEPS, POOL = 3, 2, 40, 50          # the pool fills at step ceil(50 / 6) = 9


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def _batches():
    g = torch.Generator().manual_seed(11)
    return [torch.rand(WORLD * PER_RANK, 3, 4, 4, generator=g) * 2 - 1 for _ in range(STEPS)]


def _worker(rank, world, port, out):
    import torch.distributed as dist
    os.environ["MASTER_ADDR"], os.environ["MASTER_PORT"] = "127.0.0.1", str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        import ipr_gan_b200
        ipr_gan_b200.enable_dropin()
        from ipr_gan_b200 import dist as ipr_dist
        from models.cyclegan import ImagePool
        batches = _batches()
        torch.manual_seed(5)                               # every rank seeded alike: the pool's draws in lockstep
        pool = ImagePool(POOL)
        gathered = torch.zeros(WORLD * PER_RANK, 3, 4, 4)
        got, filled_at = [], None
        for i, b in enumerate(batches):
            got.append(ipr_dist.pool_query(pool, ipr_dist.shard(b), gathered).clone())
            if filled_at is None and float(pool.counts) >= POOL:
                filled_at = i + 1
        assert filled_at == 9, filled_at
        # identical pool buffers on every rank
        for buf in (pool.images, pool.counts.reshape(1)):
            every = [torch.empty_like(buf) for _ in range(world)]
            dist.all_gather(every, buf)
            assert all(torch.equal(every[0], e) for e in every)
        # one pool fed the concatenated batches, with the same host RNG stream
        torch.manual_seed(5)
        ref = ImagePool(POOL)
        for b, mine in zip(batches, got):
            assert torch.equal(mine, torch.chunk(ref(b), world)[rank])
        assert torch.equal(ref.images, pool.images) and torch.equal(ref.counts, pool.counts)

        # metrics: the mean over ranks; keys equal on every rank keep their exact value
        assert (0.1 + 0.1 + 0.1) / 3 != 0.1                 # what a sum-then-divide reduction would return
        m = ipr_dist.reduce_metrics({"LR": 2e-4, "P/SignLoss": 0.1, "G/A": float(rank), "D/x": 0.1 * (rank + 1)})
        assert m["LR"] == 2e-4 and m["P/SignLoss"] == 0.1 and m["G/A"] == 1.0
        assert abs(m["D/x"] - 0.2) <= 1e-15
        every = [None] * world
        dist.all_gather_object(every, m)
        assert all(e == m for e in every)
        out[rank] = 1
    finally:
        dist.destroy_process_group()


def test_pool_on_gathered_batch_and_metric_reduction_gloo():
    port = _free_port()
    mgr = mp.Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(WORLD, port, out), nprocs=WORLD, join=True)
    assert dict(out) == {r: 1 for r in range(WORLD)}


def test_single_process_pool_query_is_the_plain_pool():
    """world 1: the same call, the same host RNG draws and the same result as querying the pool directly."""
    from ipr_gan_b200 import dist as ipr_dist
    from models.cyclegan import ImagePool
    batches = _batches()
    outs = []
    for query in (lambda p, b: p(b), ipr_dist.pool_query):
        torch.manual_seed(5)
        pool = ImagePool(POOL)
        outs.append(([query(pool, b).clone() for b in batches], pool.images.clone(), torch.rand(3)))
    (a, ia, ra), (b, ib, rb) = outs
    assert all(torch.equal(x, y) for x, y in zip(a, b)) and torch.equal(ia, ib) and torch.equal(ra, rb)


def test_uneven_shards_are_refused():
    import pytest
    from ipr_gan_b200 import dist as ipr_dist
    with pytest.raises(ValueError):
        ipr_dist.shard(torch.zeros(5, 3), 0, 2)
    assert ipr_dist.shard(torch.arange(6), 2, 3).tolist() == [4, 5]
