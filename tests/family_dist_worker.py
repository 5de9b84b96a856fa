"""Worker of tests/test_gpu_dist_families.py: a few protected IPR-SRGAN / IPR-CycleGAN steps through the trainers
(ipr_gan_b200/trainer.py), either data-parallel (launched by torch.distributed.run, one process per rank) or as the
single-process reference the data-parallel run must reproduce.

    family_dist_worker.py KIND MODE BACKEND OUT
      KIND     srgan_same  every rank trains the SAME 4-sample shard; reference: one trainer on that shard
               srgan_diff  global batch 8 split in 2 shards; reference: one replica per shard in one process, gradients
                           averaged before each FlatAdam step (oracle.ShardedStepOracle's recipe)
               cyclegan    global batch 2 at 64 x 64, pool_size 4; reference: one trainer at batch 2
      MODE     eager | graph
      BACKEND  nccl (one GPU per rank) | gloo (every rank on cuda:0, eager only) -- ignored by the reference run
      OUT      torch.save file written by rank 0 (or by the reference process)
"""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

WORLD = 2
STEPS = 2                      # after one warm-up step (capture(warmup=1)) on the first batch


def _batches(kind):
    g = torch.Generator().manual_seed(21)
    if kind.startswith("srgan"):
        n = 4 if kind == "srgan_same" else 4 * WORLD
        return [(torch.rand(n, 3, 24, 24, generator=g), torch.rand(n, 3, 96, 96, generator=g)) for _ in range(STEPS + 1)]
    return [(torch.rand(WORLD, 3, 64, 64, generator=g) * 2 - 1, torch.rand(WORLD, 3, 64, 64, generator=g) * 2 - 1)
            for _ in range(STEPS + 1)]


def _trainer(kind, dev, use_graph, batch):
    from ipr_gan_b200 import trainer as T
    if kind.startswith("srgan"):
        return T.ProtectedSRGANTrainer(batch, dev, use_graph=use_graph)
    tr = T.ProtectedCycleGANTrainer(dev, 64, use_graph=use_graph, batch=batch)
    tr.inner.poolA.pool_size = tr.inner.poolB.pool_size = 4      # full after the second step of global batch 2
    return tr


def _static(tr):
    return (tr.low_res, tr.high_res) if hasattr(tr, "low_res") else (tr.real_A, tr.real_B)


def _nets(tr):
    m = tr.model
    return (m.G, m.D) if hasattr(tr, "low_res") else (m.GA, m.GB, m.DA, m.DB)


def _flat_params(tr):
    return torch.cat([p.detach().reshape(-1) for n in _nets(tr) for p in n.parameters()])


def _run(tr, batches, pick):
    """capture(warmup=1) on the first batch, then one step_from_host per later batch -> metrics of those steps"""
    for dst, src in zip(_static(tr), pick(batches[0])):
        dst.copy_(src)
    tr.capture(warmup=1)
    return [tr.step_from_host(*pick(b)) for b in batches[1:]]


def _result(tr, metrics):
    torch.cuda.synchronize()
    out = {"metrics": metrics, "params": _flat_params(tr).cpu(), "launches": tr.launches_per_step}
    if hasattr(tr, "inner"):
        out["pool"] = [(p.counts.cpu().clone(), p.images.cpu().clone()) for p in (tr.inner.poolA, tr.inner.poolB)]
    return out


def _sharded_srgan_reference(batches, dev):
    """Two native SRGAN replicas in one process, each on its shard; before each FlatAdam step the replicas' gradient
    arenas are replaced by their mean, which is what the summing all-reduce and the 1/world Adam factor compute."""
    reps = [_trainer("srgan_diff", dev, False, 4) for _ in range(WORLD)]

    def deferred(opts, run):
        for o in opts:
            o.step = lambda closure=None: None                 # the real step runs below, on averaged gradients
        try:
            run()
        finally:
            for o in opts:
                del o.step
        mean = (opts[0].arena.grad + opts[1].arena.grad) * 0.5
        for o in opts:
            o.arena.grad.copy_(mean)
            o.step()

    metrics = []
    for i, b in enumerate(batches):                                 # the warm-up step, then the measured ones
        for r, (lo, hi) in zip(reps, zip(*(torch.chunk(t, WORLD) for t in b))):
            r.low_res.copy_(lo), r.high_res.copy_(hi)
        deferred([r.model.optG for r in reps], lambda: [r.model.update_g({"low_res": r.low_res, "high_res": r.high_res,
                                                                          "pretrain": False}) for r in reps])
        deferred([r.model.optD for r in reps], lambda: [r.model.update_d({"high_res": r.model.high_res,
                                                                          "super_res": r.model.super_res}) for r in reps])
        ms = [r.model.get_metrics() for r in reps]
        if i >= 1:
            metrics.append({k: sum(m[k] for m in ms) / WORLD for k in ms[0]})
    for r in reps:
        r.launches_per_step = None
    return _result(reps[0], metrics)


def reference(kind, use_graph, out):
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    batches = _batches(kind)
    if kind == "srgan_diff":
        res = _sharded_srgan_reference(batches, dev)
    else:
        tr = _trainer(kind, dev, use_graph, batches[0][0].size(0))
        res = _result(tr, _run(tr, batches, lambda b: b))
    torch.save(res, out)


def distributed(kind, use_graph, backend, out):
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    assert world == WORLD
    dev = torch.device("cuda", local if backend == "nccl" else 0)
    torch.cuda.set_device(dev)
    if backend == "nccl":
        dist.init_process_group("nccl", device_id=dev)
    else:
        assert not use_graph, "gloo collectives are host calls: they cannot be captured"
        dist.init_process_group("gloo")
    from ipr_gan_b200 import dist as idist
    batches = _batches(kind)
    if kind == "srgan_same":
        tr = _trainer(kind, dev, use_graph, 4)
        got = _run(tr, batches, lambda b: b)
    else:
        tr = _trainer(kind, dev, use_graph, batches[0][0].size(0) // world)
        got = _run(tr, batches, lambda b: tuple(idist.shard(t) for t in b))
    every = [None] * world
    dist.all_gather_object(every, got)                              # what step_from_host returned on each rank
    flat = _flat_params(tr)
    others = [torch.empty_like(flat) for _ in range(world)]
    dist.all_gather(others, flat)
    res = _result(tr, got)
    res.update(rank_metrics=every, replicas_identical=all(torch.equal(others[0], o) for o in others), world=world)
    if hasattr(tr, "inner"):
        pools = [torch.cat([p.counts.reshape(1).to(dev), p.images.reshape(-1)]) for p in (tr.inner.poolA, tr.inner.poolB)]
        mine = torch.cat(pools)
        allp = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allp, mine)
        res["pools_identical"] = all(torch.equal(allp[0], p) for p in allp)
    if rank == 0:
        torch.save(res, out)
    sys.stdout.flush()
    # no process-group teardown: collectives captured in a CUDA graph must not be destroyed under it (bench.py)
    torch.cuda.synchronize()
    os._exit(0)


def main():
    kind, mode, backend, out = sys.argv[1:5]
    torch.backends.cudnn.deterministic = True        # SRGAN's frozen VGG (cuDNN): the same algorithms in every process
    if "RANK" in os.environ:
        distributed(kind, mode == "graph", backend, out)
    else:
        reference(kind, mode == "graph", out)
        sys.stdout.flush()
        torch.cuda.synchronize()
        os._exit(0)


if __name__ == "__main__":
    main()
