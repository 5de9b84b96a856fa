#!/bin/bash
# A/B of the one-launch 3-channel layers (csrc/tapfold.cu) against the tap GEMM + col2im3 path (IPR_NO_TAPFOLD=1):
# card and power limit, outputs of bench.py --dump-outputs compared array for array, REPS alternating bench runs per
# arm at batch 512 and 64, and a torch.profiler kernel table per arm.
#   usage: scripts/ab_tapfold.sh [REPS] [OUT_DIR]    (OUT_DIR defaults to a directory under $TMPDIR or /tmp)
REPS=${1:-5}
OUT=${2:-${TMPDIR:-/tmp}/ab_tapfold}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/card.csv"
for v in on off; do
  unset IPR_NO_TAPFOLD; [ $v = off ] && export IPR_NO_TAPFOLD=1
  python bench.py --skip-cpu-baseline --skip-eager-baseline --steps 5 --dump-outputs "$OUT/dump_$v" > /dev/null 2>&1
done
unset IPR_NO_TAPFOLD
python - "$OUT" <<'P'
import glob, os, sys
import numpy as np
out = sys.argv[1]
names = sorted(os.path.basename(f) for f in glob.glob(os.path.join(out, "dump_on", "*.npy")))
bad = [n for n in names if not np.array_equal(np.load(os.path.join(out, "dump_on", n)), np.load(os.path.join(out, "dump_off", n)))]
print("dump-outputs: %d arrays, %d differ %s" % (len(names), len(bad), bad[:5]))
P
for r in $(seq 1 "$REPS"); do
  for v in off on; do
    unset IPR_NO_TAPFOLD; [ $v = off ] && export IPR_NO_TAPFOLD=1
    python bench.py --skip-cpu-baseline --skip-eager-baseline > "$OUT/b512_${v}_$r.json" 2>/dev/null
    python bench.py --batch 64 --skip-cpu-baseline --skip-eager-baseline > "$OUT/b64_${v}_$r.json" 2>/dev/null
  done
done
unset IPR_NO_TAPFOLD
python scripts/kernel_times.py 512 "$OUT/kernels_b512_on.txt" > /dev/null
IPR_NO_TAPFOLD=1 python scripts/kernel_times.py 512 "$OUT/kernels_b512_off.txt" > /dev/null
python - "$OUT" "$REPS" <<'P'
import json, statistics, sys
out, reps = sys.argv[1], int(sys.argv[2])
for b in ("b512", "b64"):
    for v in ("off", "on"):
        vals, gemm = [], []
        for r in range(1, reps + 1):
            d = json.loads(open("%s/%s_%s_%d.json" % (out, b, v, r)).read().strip().splitlines()[-1])
            vals.append(d["value"]); gemm.append(d["roofline"]["gemm_ms_per_step"])
        print("%s %-3s value median %.2f  min %.2f  max %.2f  spread %.2f   gemm_ms_per_step median %.3f   %s"
              % (b, v, statistics.median(vals), min(vals), max(vals), max(vals) - min(vals), statistics.median(gemm),
                 " ".join("%.2f" % x for x in vals)))
P
