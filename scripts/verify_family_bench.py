"""Throughput of the image-to-image verification sweep (ipr_gan_b200.verify.image_verification_sweep) for the protected
SRGAN generator (config 3: 24 -> 96) or CycleGAN's GB (config 4 eval size: 256 x 256).  Prints one JSON line.

    python scripts/verify_family_bench.py --family srgan --samples 4096 --batch 64 [--eager]
    python -m torch.distributed.run --nproc-per-node 8 scripts/verify_family_bench.py --family cyclegan ...

Inputs are seeded (SRGAN: rand in [0, 1]; CycleGAN: rand * 2 - 1); every rank sweeps its contiguous slice.  Each
timed window repeats whole sweeps (graph capture, staging and the final read-back included) for at least
``--window`` seconds, timed with device events after one warm-up sweep.  With ``--eager`` the eager sweep is timed
as well, its windows alternating with the graph's."""
import argparse
import json
import os
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import ipr_gan_b200  # noqa: E402

ipr_gan_b200.enable_dropin()
import models  # noqa: E402
from configs import presets  # noqa: E402
from ipr_gan_b200 import _lib, dist, verify  # noqa: E402


def power_limit_w(index):
    """The card's enforced power limit in W (read-only query), or None where nvidia-smi cannot say."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader,nounits", "-i", str(index)],
                             capture_output=True, text=True, timeout=30)
        return float(out.stdout.strip().splitlines()[0])
    except (OSError, ValueError, IndexError, subprocess.SubprocessError):
        return None


def build(family, dev):
    torch.manual_seed(1234)
    if family == "srgan":
        os.environ.setdefault("IPR_VGG_RANDOM_INIT", "1")          # the VGG content loss is not part of the sweep
        m = models.SRGAN(presets.srgan_model(), device=[dev])
        m = models.WhiteBoxWrapper(models.BlackBoxWrapper(m, presets.srgan_blackbox()), presets.whitebox("G"))
        return m, m.G
    m = models.CycleGAN(presets.cyclegan_model(), device=[dev])
    m = models.WhiteBoxWrapper(models.BlackBoxWrapper(m, presets.cyclegan_blackbox()), presets.whitebox("GB"))
    return m, m.GB


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--family", choices=("srgan", "cyclegan"), required=True)
    ap.add_argument("--samples", type=int, default=None, help="N inputs over all ranks (srgan 4096, cyclegan 256)")
    ap.add_argument("--batch", type=int, default=None, help="per-rank batch (srgan 64, cyclegan 1)")
    ap.add_argument("--eager", action="store_true", help="also time the eager sweep, alternating with the graph")
    ap.add_argument("--window", type=float, default=1.0, help="seconds of sweeps per timed window")
    ap.add_argument("--rounds", type=int, default=3, help="timed windows per arm")
    a = ap.parse_args()
    n = a.samples or (4096 if a.family == "srgan" else 256)
    batch = a.batch or (64 if a.family == "srgan" else 1)
    if n < 1 or batch < 1 or a.rounds < 1:
        ap.error("--samples, --batch and --rounds must be positive")

    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        sys.exit("verify_family_bench.py needs a CUDA device")
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    if world > 1:
        torch.distributed.init_process_group("nccl", device_id=dev)
    model, G = build(a.family, dev)
    gen = torch.Generator().manual_seed(4321)
    if a.family == "srgan":
        inputs = torch.rand(n, 3, 24, 24, generator=gen)
    else:
        inputs = torch.rand(n, 3, 256, 256, generator=gen) * 2 - 1

    def sweep(eager, x=inputs):
        return verify.image_verification_sweep(G, model.fn_inp, model.fn_out, x, batch=batch, eager=eager)

    # library launches of one batch body: an eager sweep in which every rank evaluates exactly one full batch
    before = _lib.launch_count()
    sweep(True, inputs[:batch * world] if n >= batch * world else inputs)
    launches = _lib.launch_count() - before

    arms = [False, True] if a.eager else [False]
    for eager in arms:                                             # warm-up: plans, workspaces, pinned staging
        res = sweep(eager)
    times = {e: [] for e in arms}
    for _ in range(a.rounds):
        for eager in arms:
            if world > 1:
                torch.distributed.barrier()
            start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            start.record()
            sweeps = 0
            while True:
                sweep(eager)                                       # ends in a host read-back of the sums
                sweeps += 1
                end.record()
                end.synchronize()
                if start.elapsed_time(end) >= a.window * 1e3:
                    break
            ms = torch.tensor([start.elapsed_time(end) / sweeps], dtype=torch.float64, device=dev)
            if world > 1:
                torch.distributed.all_reduce(ms, op=torch.distributed.ReduceOp.MAX)   # the slowest rank ends the sweep
            times[eager].append(float(ms))

    lo, hi = verify.rank_slice(n, 0, world)
    batches = -(-(hi - lo) // batch)                               # the busiest rank's batches per sweep
    runs = []
    for eager in arms:
        ms = sorted(times[eager])[len(times[eager]) // 2]
        runs.append({"graph": not eager, "samples_per_s": n / (ms / 1e3), "ms_per_sweep": ms,
                     "ms_per_batch": ms / batches, "windows_ms_per_sweep": times[eager]})
    if dist.rank() == 0:
        print(json.dumps({
            "workload": "image verification sweep: %s, %d inputs %s, G fwd x2 + triggers + crops + SSIM + pHash p"
                        % (a.family, n, "x".join(map(str, inputs.shape[1:]))),
            "family": a.family, "samples": n, "batch": batch, "world_size": world, "launches_per_batch": launches,
            "runs": runs, "result": {k: res[k] for k in ("Q_WM", "P", "MATCH", "N")},
            "device_name": torch.cuda.get_device_name(dev), "power_limit_w": power_limit_w(local)}))
    sys.stdout.flush()
    if world > 1:
        torch.distributed.barrier()
        os._exit(0)


if __name__ == "__main__":
    main()
