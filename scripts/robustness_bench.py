"""Cost of the robustness attacks on one GPU (ipr_gan_b200.robustness):

1. ``prune_`` (global magnitude pruning, csrc/prune.cu) per generator arena -- G32, G64, SRResNet, Resnet9 GB in a
   GA+GB arena -- against ``torch.nn.utils.prune.global_unstructured`` (L1Unstructured) on GPU copies of the same
   weights, CUDA events around each whole call (host work included), median of ``--reps`` calls at amount 0.5.  The
   arenas (6 to 91 MB) fit in the 126 MB L2 and are restored by a device copy before every call; nothing is flushed,
   so both arms read mostly from L2.
2. A 9-level DCGAN prune sweep (amounts 0.1 .. 0.9, ``--samples`` latents per level) against nine plain
   ``verify.verification_sweep`` calls of the unpruned model, in alternating windows: the perturbation overhead.

Prints the card name and power limit, then one JSON line per measurement (also written to ``--out`` if given).

    python scripts/robustness_bench.py [--reps 20] [--samples 10000] [--windows 3] [--out DIR]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.nn as nn  # noqa: E402
import torch.nn.utils.prune as tprune  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:              # the measurement stands without it, but say so
        q = "nvidia-smi unavailable (%s)" % e
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def _nets(dev):
    import networks
    from ipr_gan_b200 import flat
    torch.manual_seed(0)
    out = {}
    for name, f in (("G32", networks.ConvGenerator32), ("G64", networks.ConvGenerator64), ("SRResNet", networks.SRResNet)):
        net = f().to(dev)
        out[name] = (net, flat.module_arena(net))
    ga, gb = networks.Resnet9Blocks().to(dev), networks.Resnet9Blocks().to(dev)
    out["Resnet9 GB"] = (gb, flat.arena_for(list(ga.parameters()) + list(gb.parameters())))
    return out


def time_prune(reps, amount=0.5):
    from ipr_gan_b200 import robustness
    dev = torch.device("cuda", 0)
    rows = []
    for name, (net, arena) in _nets(dev).items():
        base = arena.param.clone()
        weights = [m.weight for m in net.modules() if isinstance(m, (nn.Conv2d, nn.ConvTranspose2d, nn.Linear))]
        n = sum(w.numel() for w in weights)
        ours, theirs = [], []
        for i in range(reps + 2):                       # the first two calls of each arm are warm-up
            arena.param.copy_(base)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            k = robustness.prune_(net, amount)
            b.record()
            clones = []
            for w in weights:
                c = nn.Module()
                c.weight = nn.Parameter(w.detach().clone())
                clones.append(c)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            tprune.global_unstructured([(c, "weight") for c in clones], pruning_method=tprune.L1Unstructured,
                                       amount=amount)
            c1.record()
            torch.cuda.synchronize()
            if i >= 2:
                ours.append(a.elapsed_time(b) * 1e3)
                theirs.append(c0.elapsed_time(c1) * 1e3)
        arena.param.copy_(base)
        rows.append({"what": "prune", "arena": name, "entries": n, "arena_MB": arena.numel * 4 / 1e6, "k": k,
                     "prune__us_median": statistics.median(ours), "prune__us_min": min(ours),
                     "torch_global_unstructured_us_median": statistics.median(theirs),
                     "torch_global_unstructured_us_min": min(theirs), "reps": reps})
    return rows


def time_sweep(samples, windows):
    import models
    from configs import presets
    from ipr_gan_b200 import robustness, verify
    dev = torch.device("cuda", 0)
    torch.manual_seed(3)
    m = models.DCGAN(presets.dcgan_model(), device=[dev])
    m = models.BlackBoxWrapper(m, presets.dcgan_blackbox())
    m = models.WhiteBoxWrapper(m, presets.dcgan_whitebox())
    amounts = tuple(i / 10 for i in range(1, 10))

    def plain():
        for _ in amounts:
            verify.verification_sweep(m.G, m.fn_inp, m.fn_out, n_samples=samples, sign_model=m.loss_model)

    def swept():
        robustness.prune_sweep(m, amounts, n_samples=samples)

    plain(), swept()                                    # warm-up of every shape
    times = {"plain": [], "prune_sweep": []}
    for _ in range(windows):
        for key, fn in (("plain", plain), ("prune_sweep", swept)):
            torch.cuda.synchronize()
            t = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            times[key].append(time.perf_counter() - t)
    return [{"what": "dcgan_prune_sweep", "levels": len(amounts), "samples_per_level": samples, "windows": windows,
             "plain_s": times["plain"], "prune_sweep_s": times["prune_sweep"],
             "plain_s_median": statistics.median(times["plain"]),
             "prune_sweep_s_median": statistics.median(times["prune_sweep"])}]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--samples", type=int, default=10000)
    ap.add_argument("--windows", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("robustness_bench.py measures on a CUDA device; none is available")
    import ipr_gan_b200
    ipr_gan_b200.enable_dropin()
    rows = [dict(what="card", **card())] + time_prune(args.reps) + time_sweep(args.samples, args.windows)
    lines = [json.dumps(r) for r in rows]
    print("\n".join(lines))
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "robustness_bench.jsonl"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
