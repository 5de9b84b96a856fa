"""Cost of the re-training attacks on one GPU (ipr_gan_b200.robustness.finetune_attack), per family at its BASELINE
shape (DCGAN 32x32 batch 64, SRGAN 24 -> 96 batch 16, CycleGAN 128x128 batch 1):

1. attack steps per second -- ``step_from_host`` with a host batch in and the metrics out, after ``finetune_attack``
   with ``steps=0`` switched the trainer to the inhibited step at lr x 0.1 -- captured replays against the eager
   reference-API loop (``use_graph=False``, the same inhibit flags), in alternating windows of at least ``--window``
   seconds after a warm-up; every window's rate is reported.
2. the verification sweep of the same model at a realistic size (DCGAN: 10 000 latents; SRGAN: 256 images of 24 x 24;
   CycleGAN: 64 images of 128 x 128), median of ``--sweeps`` calls, and the share of wall time the sweeps take in a
   schedule of ``--steps`` captured steps verified every ``--every`` steps (at step 0, every ``--every`` and the last),
   computed from the measured step and sweep times.

Prints the card name and power limit, then one JSON line per measurement (also written to ``--out`` if given).

    python scripts/attack_bench.py [--window 0.5] [--windows 5] [--sweeps 3] [--steps 2000] [--every 500] [--out DIR]
"""
import argparse
import gc
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:              # the measurement stands without it, but say so
        q = "nvidia-smi unavailable (%s)" % e
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def _family(kind):
    """-> (trainer factory, host batches, sweep arguments) at the BASELINE shape."""
    from ipr_gan_b200 import trainer as T
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(17)
    if kind == "dcgan":
        make = lambda graph: T.ProtectedDCGANTrainer(64, dev, use_graph=graph)
        batches = [(torch.randn(64, 3, 32, 32, generator=g).clamp(-1, 1), torch.randn(64, 128, generator=g))
                   for _ in range(8)]
        sweep = {"n_samples": 10000}
    elif kind == "srgan":
        make = lambda graph: T.ProtectedSRGANTrainer(16, dev, use_graph=graph)
        batches = [(torch.rand(16, 3, 24, 24, generator=g), torch.rand(16, 3, 96, 96, generator=g)) for _ in range(8)]
        sweep = {"inputs": torch.rand(256, 3, 24, 24, generator=g), "batch": 16}
    else:
        make = lambda graph: T.ProtectedCycleGANTrainer(dev, 128, use_graph=graph)
        batches = [(torch.rand(1, 3, 128, 128, generator=g) * 2 - 1, torch.rand(1, 3, 128, 128, generator=g) * 2 - 1)
                   for _ in range(8)]
        sweep = {"inputs": torch.rand(64, 3, 128, 128, generator=g) * 2 - 1, "batch": 16}
    return make, batches, sweep


def _attacking(make, graph, batches, sweep):
    from ipr_gan_b200 import robustness
    tr = make(graph)
    tr.capture(warmup=2)                                 # untimed protected steps, then the capture
    robustness.finetune_attack(tr, lambda i: batches[i % len(batches)], 0, 1, **sweep)     # lr x 0.1, inhibited step
    for i in range(5):                                   # warm-up: the re-capture for the new rate and flags
        tr.step_from_host(*batches[i % len(batches)])
    torch.cuda.synchronize()
    return tr


def _window(tr, batches, seconds):
    n, i = 0, 0
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    while True:
        for _ in range(10):
            tr.step_from_host(*batches[i % len(batches)])
            i += 1
        n += 10
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if dt >= seconds:
            return n / dt


def measure(kind, args):
    from ipr_gan_b200 import robustness
    make, batches, sweep = _family(kind)
    arms = {"graph": _attacking(make, True, batches, sweep), "eager": _attacking(make, False, batches, sweep)}
    rates = {k: [] for k in arms}
    for _ in range(args.windows):
        for k, tr in arms.items():
            rates[k].append(_window(tr, batches, args.window))
    tr = arms["graph"]
    times = []
    for _ in range(args.sweeps + 1):                     # the first call is warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        with torch.no_grad():
            robustness._sweep(tr.model, sweep)
        torch.cuda.synchronize()
        times.append(time.perf_counter() - t0)
    t_sweep = statistics.median(times[1:])
    step_s = 1.0 / statistics.median(rates["graph"])
    n_sweeps = len(robustness.attack_schedule(args.steps, args.every))
    total = args.steps * step_s + n_sweeps * t_sweep
    n_sweep = sweep.get("n_samples") or sweep["inputs"].shape[0]
    out = [{"what": "attack_steps_per_s", "family": kind, "batch": batches[0][0].shape[0],
            "shape": list(batches[0][0].shape[1:]), "window_s_min": args.window,
            "graph_steps_per_s": rates["graph"], "eager_steps_per_s": rates["eager"],
            "graph_median": statistics.median(rates["graph"]), "eager_median": statistics.median(rates["eager"]),
            "speedup_median": statistics.median(rates["graph"]) / statistics.median(rates["eager"])},
           {"what": "attack_sweep_share", "family": kind, "sweep_samples": n_sweep, "sweep_s": times[1:],
            "sweep_s_median": t_sweep, "schedule_steps": args.steps, "eval_every": args.every, "sweeps": n_sweeps,
            "step_ms_graph_median": step_s * 1e3, "schedule_s": total,
            "sweep_share": n_sweeps * t_sweep / total, "derived": "schedule_s and sweep_share from the medians"}]
    del arms, tr
    gc.collect()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--window", type=float, default=0.5)
    ap.add_argument("--windows", type=int, default=5)
    ap.add_argument("--sweeps", type=int, default=3)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--every", type=int, default=500)
    ap.add_argument("--families", default="dcgan,srgan,cyclegan")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("attack_bench.py measures on a CUDA device; none is available")
    import ipr_gan_b200
    ipr_gan_b200.enable_dropin()
    lines = [json.dumps(dict(what="card", **card()))]
    print(lines[0], flush=True)
    for kind in args.families.split(","):
        for row in measure(kind, args):
            lines.append(json.dumps(row))
            print(lines[-1], flush=True)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "attack_bench.jsonl"), "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
