"""Weak scaling of the data-parallel IPR-SRGAN / IPR-CycleGAN steps over the GPUs of one box: SRGAN at 16 samples per
GPU (24 -> 96), CycleGAN at 1 per GPU (128 x 128), one process per GPU.

    python scripts/family_scale.py --workload srgan                                   # 1 GPU
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \\
        scripts/family_scale.py --workload cyclegan [--out FILE]

Timing as ``bench.py --workload srgan|cyclegan`` (run_family): CUDA events; ``value`` = back-to-back step replays on
inputs already in HBM, ``e2e`` = per step a pinned host batch in and the metrics dict out (here the global-batch
metrics: the all-gather of ``dist.reduce_metrics`` is inside the window), a 256 MB buffer cleared between e2e steps.
Every rank times its own loop; the slowest rank's time is reported.  Rank 0 prints one JSON line (and appends it to
``--out``) with the card's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

PER_GPU = {"srgan": 16, "cyclegan": 1}


def _card(index):
    q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "nvidia-smi unavailable: " + torch.cuda.get_device_name(index)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workload", choices=sorted(PER_GPU), required=True)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    world, rank = int(os.environ.get("WORLD_SIZE", "1")), int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "family_scale.py needs CUDA"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from ipr_gan_b200 import trainer as T
    n = PER_GPU[args.workload]
    gen = torch.Generator().manual_seed(1234 + rank)           # this rank's shard of a synthetic global batch
    if args.workload == "srgan":
        tr = T.ProtectedSRGANTrainer(n, dev)
        host = (torch.rand(n, 3, 24, 24, generator=gen).pin_memory(), torch.rand(n, 3, 96, 96, generator=gen).pin_memory())
        static = (tr.low_res, tr.high_res)
    else:
        tr = T.ProtectedCycleGANTrainer(dev, 128, batch=n)
        host = ((torch.rand(n, 3, 128, 128, generator=gen) * 2 - 1).pin_memory(),
                (torch.rand(n, 3, 128, 128, generator=gen) * 2 - 1).pin_memory())
        static = (tr.real_A, tr.real_B)
    for dst, src in zip(static, host):
        dst.copy_(src)
    tr.capture(max(3, args.warmup))
    for _ in range(max(3, args.warmup)):
        last = tr.step_from_host(*host)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e2e = 0.0
    for _ in range(args.steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        last = tr.step_from_host(*host)
        b.record()
        torch.cuda.synchronize()
        e2e += a.elapsed_time(b)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps):
        tr.step()
    b.record()
    torch.cuda.synchronize()
    mine = (a.elapsed_time(b) / args.steps, e2e / args.steps, _card(local))
    every = [mine]
    if world > 1:
        every = [None] * world
        dist.all_gather_object(every, mine)
    if rank == 0:
        ms, ms_e2e = max(e[0] for e in every), max(e[1] for e in every)
        line = json.dumps({
            "workload": args.workload, "n_gpus": world, "per_gpu_batch": n, "global_batch": n * world,
            "scaling": "weak", "steps": args.steps, "cuda_graph": tr.use_graph,
            "ms_per_step": ms, "steps_per_s": 1e3 / ms, "samples_per_s": 1e3 / ms * n * world,
            "e2e": {"ms_per_step": ms_e2e, "steps_per_s": 1e3 / ms_e2e, "samples_per_s": 1e3 / ms_e2e * n * world},
            "per_rank_ms": [e[0] for e in every], "gpu_launches_per_step": tr.launches_per_step,
            "cards": sorted(set(e[2] for e in every)), "last_metrics": last})
        print(line)
        if args.out:
            with open(args.out, "a") as f:
                f.write(line + "\n")
    sys.stdout.flush()
    # collectives live in the captured graphs: synchronise and leave without tearing the process group down
    torch.cuda.synchronize()
    os._exit(0)


if __name__ == "__main__":
    main()
