"""Data parallelism for the protected step: one process per GPU, ``torch.distributed`` over NCCL/NVLink.

The reference scales with ``nn.DataParallel`` (experiments/base.py:24-39, models/dcgan.py:16-17): the global
batch is scattered in equal chunks, every replica keeps its own BatchNorm statistics, gradients are summed on
device 0 and parameters re-broadcast before every forward.  Here each rank owns ``torch.chunk(batch, world)[rank]``
(the same partition), BatchNorm stays per rank, and the only exchange is ONE all-reduce per network per optimizer
step on the flat gradient arena (mean over ranks == gradient of the global-batch mean loss); replicas stay
bit-identical because they apply identical reduced gradients, so no parameter broadcast is ever needed.
"""
import math

import torch
import torch.distributed as dist


def world():
    return dist.get_world_size() if dist.is_available() and dist.is_initialized() else 1


def rank():
    return dist.get_rank() if dist.is_available() and dist.is_initialized() else 0


def shard(batch, rank_=None, world_=None):
    """This rank's slice of a global batch: the partition nn.DataParallel's scatter makes.  The batch must split into
    equal shards: the mean over ranks of per-shard means is the global mean only then, so uneven shards are refused
    rather than silently weighted."""
    r = rank() if rank_ is None else rank_
    w = world() if world_ is None else world_
    if batch.size(0) % w:
        raise ValueError("a global batch of %d does not split into %d equal shards" % (batch.size(0), w))
    return torch.chunk(batch, w, dim=0)[r]


def allreduce_mean_(flat_tensor):
    """In-place mean over ranks of a flat buffer (gradient arena, or a vector of per-rank loss sums)."""
    w = world()
    if w > 1:
        dist.all_reduce(flat_tensor)
        flat_tensor.mul_(1.0 / w)
    return flat_tensor


def allreduce_sum_(flat_tensor):
    """In-place SUM over ranks (the 1/world factor is folded into the consumer: ``ipr_adam_flat_f32(grad_scale)``
    for gradients, the host-side division in ``get_metrics`` for the loss slots).  No-op for a single process."""
    if world() > 1:
        dist.all_reduce(flat_tensor)
    return flat_tensor


def reduce_metrics(metrics):
    """Average a metrics dict over ranks (per-rank means of equal-size shards) with one small all-gather; every rank
    returns the same dict.  A value that is the same on every rank (the learning rate, the sign loss of the replicated
    weights) comes back exactly: a sum of w copies divided by w need not (0.1 at w = 3).  No-op for a single process."""
    w = world()
    if w == 1:
        return metrics
    keys = sorted(metrics)
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    mine = torch.tensor([metrics[k] for k in keys], dtype=torch.float64, device=dev)
    every = torch.empty(w * len(keys), dtype=torch.float64, device=dev)
    dist.all_gather_into_tensor(every, mine)
    cols = every.view(w, len(keys)).t().tolist()
    return {k: c[0] if all(v == c[0] for v in c) else math.fsum(c) / w for k, c in zip(keys, cols)}


def pool_query(pool, images, gathered=None):
    """This rank's shard of ``pool(global batch)`` for a history pool that draws from the host RNG (CycleGAN's
    ``ImagePool``).  The reference keeps ONE pool and queries it with the batch ``nn.DataParallel`` gathered from all
    replicas; here every rank gathers the shards in rank order (``torch.chunk``'s order) into ``gathered``
    (``(world * n, ...)``, allocated when not given) and queries its own copy of the pool with it.  With every rank
    seeded alike and the pool the step's only host RNG consumer, the draws and so the pool contents stay identical
    on all ranks.  A single process queries the pool with ``images`` directly."""
    w = world()
    if w == 1:
        return pool(images)
    images = images.detach().contiguous()
    if gathered is None:
        gathered = images.new_empty((w * images.size(0),) + tuple(images.shape[1:]))
    dist.all_gather_into_tensor(gathered, images)
    return shard(pool(gathered), rank(), w)
