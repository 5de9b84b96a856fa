"""A/B of the 64 x 64 protected IPR-DCGAN step (the CUB-200 configs: ConvGenerator64 / SNDiscriminator64, 32 x 32
watermark) with the banded one-launch 3-channel fold against the tap GEMM + col2im3 path (IPR_NO_TAPFOLD=1).

    python scripts/dcgan64_bench.py [--batches 64,512] [--windows 5] [--seconds 0.5] [--out DIR]

One process, one GPU.  Prints the card's name, power limit and maximum SM clock, then per batch builds one captured
trainer per arm (the switch is read while the step is captured), warms both graphs up and times alternating windows
of graph replays with CUDA events, each window at least --seconds long.  Reports median, min and max steps/s and
ms/step per arm and the library launches per step.  With --out it writes the JSON result lines, a summary.txt, and
runs scripts/kernel_times.py (torch.profiler, one process per arm) into that directory.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ipr_gan_b200.trainer import ProtectedDCGANTrainer  # noqa: E402

SIZE, WM = 64, 32
ARMS = (("band", "0"), ("two_launch", "1"))        # (name, IPR_NO_TAPFOLD)


def card():
    name = torch.cuda.get_device_name(0)
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                             capture_output=True, text=True, timeout=60).stdout.strip()
    except (OSError, subprocess.SubprocessError) as e:
        smi = "nvidia-smi unavailable: %s" % e
    return name, smi


def build(batch, no_tapfold):
    os.environ["IPR_NO_TAPFOLD"] = no_tapfold
    dev = torch.device("cuda", 0)
    tr = ProtectedDCGANTrainer(batch, dev, use_graph=True, size=SIZE, wm_size=WM)
    g = torch.Generator().manual_seed(1234)
    tr.set_inputs(torch.randn(batch, 3, SIZE, SIZE, generator=g).clamp(-1, 1), torch.randn(batch, 128, generator=g))
    tr.capture(warmup=3)
    return tr


def replay_ms(tr, n):
    """Device time per step of n back-to-back replays (CUDA events, ending in a synchronise)."""
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(n):
        tr.graph.replay()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / n


def run_batch(batch, windows, seconds):
    trainers = {name: build(batch, flag) for name, flag in ARMS}
    os.environ.pop("IPR_NO_TAPFOLD", None)
    reps = {}
    for name, tr in trainers.items():                # warm-up; size the windows from it
        replay_ms(tr, 10)
        ms = replay_ms(tr, 20)
        reps[name] = max(20, int(seconds * 1e3 / ms) + 1)
    ms = {name: [] for name in trainers}
    for w in range(windows):                          # alternate the arms, and which arm goes first
        order = list(trainers) if w % 2 == 0 else list(trainers)[::-1]
        for name in order:
            ms[name].append(replay_ms(trainers[name], reps[name]))
    out = []
    for name, flag in ARMS:
        vals = ms[name]
        sps = [1e3 / v for v in vals]
        out.append({"batch": batch, "size": SIZE, "wm_size": WM, "arm": name, "IPR_NO_TAPFOLD": flag,
                    "steps_per_s_median": statistics.median(sps), "steps_per_s_min": min(sps),
                    "steps_per_s_max": max(sps), "ms_per_step_median": statistics.median(vals),
                    "ms_per_step_min": min(vals), "ms_per_step_max": max(vals),
                    "replays_per_window": reps[name], "windows": windows,
                    "launches_per_step": trainers[name].launches_per_step})
    del trainers
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--batches", default="64,512")
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--seconds", type=float, default=0.5)
    ap.add_argument("--out", default=None, help="directory for the result lines, summary.txt and kernel tables")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("dcgan64_bench.py needs a CUDA device")
    name, smi = card()
    lines = ["%s; nvidia-smi: %s" % (name, " | ".join(smi.splitlines())),
             "64x64 protected step (wm_size 32), captured graph, CUDA events; %d alternating windows per arm, "
             ">= %.1f s of replays each" % (args.windows, args.seconds)]
    results = []
    for b in (int(x) for x in args.batches.split(",")):
        for r in run_batch(b, args.windows, args.seconds):
            results.append(r)
            print(json.dumps(r), flush=True)
            lines.append("b%-4d %-10s steps/s median %8.2f  min %8.2f  max %8.2f   ms/step median %.4f  "
                         "(min %.4f, max %.4f)   launches/step %d"
                         % (b, r["arm"], r["steps_per_s_median"], r["steps_per_s_min"], r["steps_per_s_max"],
                            r["ms_per_step_median"], r["ms_per_step_min"], r["ms_per_step_max"],
                            r["launches_per_step"]))
    text = "\n".join(lines) + "\n"
    sys.stdout.write(text)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "results.jsonl"), "w") as f:
            f.write("".join(json.dumps(r) + "\n" for r in results))
        with open(os.path.join(args.out, "summary.txt"), "w") as f:
            f.write(text)
        with open(os.path.join(args.out, "card.csv"), "w") as f:
            f.write(smi + "\n")
        for b in (int(x) for x in args.batches.split(",")):
            for arm, flag in ARMS:
                env = dict(os.environ, IPR_NO_TAPFOLD=flag)
                dst = os.path.join(args.out, "kernels_b%d_%s.txt" % (b, arm))
                subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "kernel_times.py"), str(b), dst,
                                str(SIZE)], env=env, check=True, stdout=subprocess.DEVNULL)


if __name__ == "__main__":
    main()
