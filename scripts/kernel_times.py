"""Per-kernel device time of one eager protected IPR-DCGAN step, from torch.profiler (CUDA activities).

    python scripts/kernel_times.py [batch] [out.txt] [size]

size is the image side: 32 (default, the CIFAR configs) or 64 (the CUB-200 configs, with a 32 x 32 watermark).

Three eager steps warm up every shape, then two profiled steps; the table lists each kernel's launches and summed
device time per step, longest first.  Run it in a process of its own: tracing slows the host, so step times taken
with the profiler on are not end-to-end numbers.
"""
import os
import sys
from collections import defaultdict

import torch
from torch.profiler import ProfilerActivity, profile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ipr_gan_b200.trainer import ProtectedDCGANTrainer  # noqa: E402

B = int(sys.argv[1]) if len(sys.argv) > 1 else 512
OUT = sys.argv[2] if len(sys.argv) > 2 and sys.argv[2] else None
SIZE = int(sys.argv[3]) if len(sys.argv) > 3 else 32
STEPS = 2
dev = torch.device("cuda", 0)
tr = ProtectedDCGANTrainer(B, dev, use_graph=False, size=SIZE, wm_size=SIZE // 2)
g = torch.Generator().manual_seed(1234)
tr.set_inputs(torch.randn(B, 3, SIZE, SIZE, generator=g).clamp(-1, 1), torch.randn(B, 128, generator=g))
for _ in range(3):
    tr._step()
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(STEPS):
        tr._step()
    torch.cuda.synchronize()

n, us = defaultdict(int), defaultdict(float)
for e in prof.events():
    if e.device_type == torch.autograd.DeviceType.CUDA:
        name = e.name.replace("(anonymous namespace)::", "").split("(")[0]
        n[name] += 1
        us[name] += e.device_time
lines = ["# batch %d, %dx%d, %s, per step (mean of %d eager steps), IPR_NO_TAPFOLD=%s" %
         (B, SIZE, SIZE, torch.cuda.get_device_name(dev), STEPS, os.environ.get("IPR_NO_TAPFOLD", "0"))]
total = sum(us.values()) / STEPS
lines.append("%-100s %6s %10s" % ("kernel", "n", "us"))
for name in sorted(us, key=lambda k: -us[k]):
    lines.append("%-100s %6d %10.1f" % (name[:100], n[name] // STEPS, us[name] / STEPS))
lines.append("%-100s %6d %10.1f" % ("total", sum(n.values()) // STEPS, total))
text = "\n".join(lines) + "\n"
sys.stdout.write(text)
if OUT:
    os.makedirs(os.path.dirname(os.path.abspath(OUT)), exist_ok=True)
    open(OUT, "w").write(text)
