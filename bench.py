"""bench.py -- IPR-DCGAN 32x32 protected training steps/sec on N B200s (BASELINE.json metric, configs[1]).

    python bench.py --gpus N --steps K --warmup W                      # this repo (sm_100a kernels)
    python bench.py --impl reference --gpus N --steps K --warmup W      # the reference's CPU path (oracle port)
    python bench.py --gpus N --steps K --warmup W --dump-outputs DIR   # + the last timed step's outputs, DIR/<name>.npy

A "step" is one full protected training step (experiments/image_generation.py:86-101): update_d + update_g
with the black-box trigger / SSIM watermark loss and the white-box sign loss, global batch 512 split evenly over
the ranks (strong scaling), synthetic CIFAR-shaped data, random-init weights.  One JSON line on rank 0.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "IPR-DCGAN 32x32 protected train steps/sec (global batch 512)"
WORKLOAD = ("IPR-DCGAN 32x32 (ConvGenerator32 + SNDiscriminator32) protected step: TransformDist trigger, 16x16 opaque "
            "watermark, SSIM loss lambda=1, sign loss gamma0=0.1 'EXAMPLE A'")
GLOBAL_BATCH = 512
FLOP_PER_SAMPLE = 2.970e9          # SURVEY.md 8d: necessary work of one protected step


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=GLOBAL_BATCH, help="global batch (default: the metric's 512)")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--no-pinned-inputs", action="store_true",
                    help="e2e: copy the batch in front of the graph replay instead of inside the graph")
    ap.add_argument("--skip-cpu-baseline", action="store_true")
    ap.add_argument("--skip-eager-baseline", action="store_true")
    ap.add_argument("--device-latents", action="store_true", help="draw latents on the device instead of copying them")
    ap.add_argument("--workload", default="step", choices=["step", "verify", "srgan", "cyclegan"],
                    help="step: the protected training step (the metric); verify: BASELINE config 5, the watermark / "
                         "signature verification sweep over 10 000 trigger samples, sharded over the ranks; srgan / "
                         "cyclegan: BASELINE configs 3 / 4, one protected step of IPR-SRGAN (batch 16, 24 -> 96) / "
                         "IPR-CycleGAN (batch 1, 128 x 128) on the native networks (single GPU)")
    ap.add_argument("--samples", type=int, default=10000, help="--workload verify: trigger samples in the sweep")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (its metrics, the generated batch, "
                         "the generator / discriminator state) as DIR/<name>.npy, float32 / float64, at most 64 MB: "
                         "two builds run with the same arguments can then be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "b200" or args.workload != "step"):
        ap.error("--dump-outputs is implemented for the protected training step (--impl b200 --workload step)")
    return args


def peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))), "measured"
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback"


# ------------------------------------------------------------------------------------------------ clocks
class ClockSampler(object):
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = sorted(float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit())
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            if len(r) >= 9:
                for name, val in zip(names, r[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ------------------------------------------------------------------------------------------------ CPU arm
def cpu_reference_steps_per_sec(steps, warmup, sample_batch=GLOBAL_BATCH):
    """The reference's CPU implementation of the step (oracle port of models/dcgan.py + models/wrappers.py,
    pinned to the unmodified reference by tests/golden/dcgan_step.npz), all host threads, on a bounded sample:
    a few steps at the metric's own global batch (small batches are far less efficient on the CPU -- scaling a
    batch-64 step by 64/512 under-reports the CPU by 3-4x)."""
    import torch
    from oracle import ipr_oracle as orc
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(1234)
    G, D = orc.make_generator(), orc.make_discriminator()
    mark = os.path.join(ROOT, "ipr_gan_b200", "assets", "watermark_a.png")
    fg, bg = orc.load_watermark(mark, 16, True, True)
    ref = orc.DCGANStepOracle(G, D, orc.transform_dist, lambda y: orc.paste_patch(y, fg, bg, "tl", 16))
    real, z = orc.synth_step_inputs(sample_batch)
    for _ in range(warmup):
        ref.step(real, z)
    t0 = time.perf_counter()
    for _ in range(steps):
        ref.step(real, z)
    dt = time.perf_counter() - t0
    return steps / dt, dt, torch.get_num_threads()


def torch_eager_steps_per_sec(device, batch, steps=10, warmup=3):
    """The SAME oracle step (reference semantics, plain PyTorch operators) run eagerly on the GPU through
    cuDNN / cuBLAS -- what the reference itself would do on this box (SURVEY.md 8d: "the honest thing to beat").
    -> {"fp32": steps/s with TF32 off, "tf32": steps/s with TF32 on}"""
    import torch
    from oracle import ipr_oracle as orc
    mark = os.path.join(ROOT, "ipr_gan_b200", "assets", "watermark_a.png")
    fg, bg = orc.load_watermark(mark, 16, True, True)
    fg, bg = fg.to(device), bg.to(device)
    real, z = orc.synth_step_inputs(batch)
    real_h, z_h = real.pin_memory(), z.pin_memory()
    out = {}
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    try:
        for name, tf32 in (("fp32", False), ("tf32", True)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            torch.backends.cudnn.benchmark = True                      # train.py:43-44
            torch.manual_seed(1234)
            G, D = orc.make_generator().to(device), orc.make_discriminator().to(device)
            ref = orc.DCGANStepOracle(G, D, orc.transform_dist, lambda y: orc.paste_patch(y, fg, bg, "tl", 16))

            def one():
                ref.step(real_h.to(device, non_blocking=True), z_h.to(device, non_blocking=True))
                return ref.metrics()                                   # the reference reads its metrics every step
            for _ in range(warmup):
                one()
            torch.cuda.synchronize(device)
            t0 = time.perf_counter()
            for _ in range(steps):
                one()
            torch.cuda.synchronize(device)
            out[name] = steps / (time.perf_counter() - t0)
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = saved
    return out


def step_traffic():
    """DRAM traffic of the tensor-core GEMM launches of one batch-512 step, from the committed ncu launch list
    (profiles/r2_step_traffic.json, written by scripts/summarize_launches.py from the ncu CSV of the same command)."""
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "r2_step_traffic.json")))
    except Exception:
        return None


DUMP_BYTES = 64 * 10 ** 6


def dump_step_outputs(out_dir, tr, metrics):
    """What the last timed step left a caller, as out_dir/<name>.npy: every metric (float64), the generator and
    discriminator state a checkpoint holds (float32; integer counters as float64) and the generated batch G(z)
    (float32).  When the batch would take the total over DUMP_BYTES, a fixed seeded sample of its rows is written."""
    import numpy as np
    import torch
    torch.cuda.synchronize()
    arrays = {"metric." + k.replace("/", "."): np.float64(v) for k, v in metrics.items()}
    for net in ("G", "D"):
        for k, v in getattr(tr.model, net).state_dict().items():
            v = v.detach().cpu()
            arrays[net + "." + k] = v.numpy().astype(np.float32 if v.is_floating_point() else np.float64)
    fake = tr.model.fake_sample.detach().float().cpu().numpy()
    room = DUMP_BYTES - sum(a.nbytes + 1024 for a in arrays.values()) - 1024     # 1 KiB per .npy header, generously
    if fake.nbytes > room:
        keep = np.random.default_rng(0).choice(len(fake), room // fake[0].nbytes, replace=False)
        fake = fake[np.sort(keep)]
    arrays["fake_sample"] = fake
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warmup = args.steps, max(1, min(args.warmup, 3))
    sample = args.batch
    sps, dt, cores = cpu_reference_steps_per_sec(steps, warmup, sample)
    value = sps * sample / args.batch
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": 1e3 / value, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "fp32", "data": "synthetic",
        # same workload string and batch keys as the b200 arm (the driver compares the two configs)
        "config": {"workload": WORKLOAD, "global_batch": args.batch, "per_gpu_batch": args.batch, "parallelism": "cpu",
                   "note": "reference CPU path (PyTorch CPU, oracle port pinned to the reference), every step a full "
                           "global-batch step"},
        "cpu_baseline": {"value": value, "unit": "steps/s", "cores": cores, "kind": "port",
                         "sample": "%d steps at batch %d (the metric's global batch) in %.1f s after %d warm-up"
                                   % (steps, sample, dt, warmup)},
        "e2e": {"value": value, "unit": "steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


# ------------------------------------------------------------------------------------------------ B200 arm
def _dbg(msg):
    if os.environ.get("IPR_BENCH_DEBUG"):
        sys.stderr.write("[rank %s] %s\n" % (os.environ.get("RANK", "0"), msg))
        sys.stderr.flush()


def run_b200(args):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs CUDA (no CPU fallback)"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        # NCCL may print its version banner on stdout at communicator creation: keep stdout clean for the JSON line
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    assert args.batch % world == 0
    local_batch = args.batch // world

    from ipr_gan_b200 import dense
    from ipr_gan_b200.trainer import ProtectedDCGANTrainer
    tr = ProtectedDCGANTrainer(local_batch, device, use_graph=not args.no_graph, device_latents=args.device_latents,
                               pinned_inputs=not args.no_pinned_inputs)
    gen = torch.Generator().manual_seed(1234 + rank)
    # the batch lives in the trainer's own pinned buffers, where a data loader would put it; every e2e step copies it
    # host -> device again (graph memcpy nodes when pinned_inputs, cudaMemcpyAsync in front of the replay otherwise)
    real_h, z_h = tr.real_host, tr.latent_host
    real_h.copy_(torch.randn(local_batch, 3, 32, 32, generator=gen).clamp(-1, 1))
    z_h.copy_(torch.randn(local_batch, 128, generator=gen))
    _dbg('trainer built')
    tr.set_inputs(real_h, z_h)
    tr.capture()
    _dbg('captured')
    flush = torch.empty(256 * 1024 * 1024 // 4, device=device)       # 256 MiB > 126 MB of L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """sum of per-step device times (CUDA events around each step, L2 flushed in between), max over ranks"""
        barrier()
        evs = []
        for _ in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            evs.append((a, b))
        barrier()
        total = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([total], device=device, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(max(3, args.warmup)):
        tr.step()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    _dbg('warm')
    total_ms = timed(tr.step, args.steps)
    _dbg('timed')
    # end to end through the public call: pinned host batch in, metrics dict out, every step
    metrics_box = {}

    def e2e_step():
        metrics_box["m"] = tr.step_from_host(real_h, None if args.device_latents else z_h)
    for _ in range(3):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    e2e_ms = timed(e2e_step, args.steps)
    wall_e2e = time.perf_counter() - t0
    _dbg('e2e done')
    if args.dump_outputs and rank == 0:
        dump_step_outputs(args.dump_outputs, tr, metrics_box["m"])   # before the profiling step below moves the weights
    clocks = sampler.stop() if rank == 0 else None

    # live tensor-roofline measurement: one eager step with CUDA events around every GEMM launch
    tr._step()                                   # eager warm-up (allocator, lazy attributes)
    torch.cuda.synchronize()
    torch.cuda._sleep(200_000_000)               # ~0.1 s GPU spin: the host enqueues the whole step behind it, so the
    dense.PROFILE = []                           # event pairs below time back-to-back kernels, not launch gaps
    dense.PROFILE_L2 = []                        # bytes each launch's TMA loads pull through L2 (the operand stream)
    from ipr_gan_b200 import engine as _engine
    _side, _engine._USE_SIDE = _engine._USE_SIDE, False     # one stream: every GEMM is timed alone, not overlapped
    tr._step()
    torch.cuda.synchronize()
    _engine._USE_SIDE = _side
    gemm_ms = sum(a.elapsed_time(b) for _, _, a, b in dense.PROFILE)
    gemm_flops = sum(f for _, f, _, _ in dense.PROFILE)
    n_gemm = len(dense.PROFILE)
    by_kind = {}
    for kind, f, a, b in dense.PROFILE:
        e = by_kind.setdefault(kind, [0.0, 0.0, 0])
        e[0] += f
        e[1] += a.elapsed_time(b)
        e[2] += 1
    l2_bytes = sum(b for _, b in dense.PROFILE_L2)
    dense.PROFILE = None
    dense.PROFILE_L2 = None
    l2_cap = 6300.0 * 1965.0e6                   # B/clk chip-wide (B300_MICROARCH.md, LTS cap) x SM clock

    # HBM-roofline figure of the SSIM loss kernel at this rank's training shape and at a large batch
    from ipr_gan_b200 import ops
    pk, pk_src = peaks()

    def ssim_gbs(B):
        x = torch.rand(B, 3, 32, 32, device=device)
        y = torch.rand(B, 3, 32, 32, device=device)
        for _ in range(3):
            ops.ssim_loss_fwd_bwd(x, y, True)
        ts = []
        for _ in range(10):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            ops.ssim_loss_fwd_bwd(x, y, True)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        return 36.0 * B * 32 * 32 / (ts[len(ts) // 2] * 1e-3) / 1e9
    _dbg('profiled gemms')
    ssim_small, ssim_big = ssim_gbs(local_batch), ssim_gbs(16384)
    _dbg('ssim done')

    if rank != 0:
        _finish(world)
        return
    traffic = step_traffic()
    ms = total_ms / args.steps
    value = 1e3 / ms
    e2e_value = 1e3 / (e2e_ms / args.steps)
    achieved = gemm_flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
    peak_tf = pk.get("bf16_tflops_sustained", 1400.0)
    line = {
        "metric": METRIC, "value": value, "unit": "steps/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": {"workload": WORKLOAD,
                   "global_batch": args.batch, "per_gpu_batch": local_batch, "parallelism": "dp%d" % world,
                   "cuda_graph": not args.no_graph, "l2": "flushed (256 MiB memset) between timed steps",
                   "timing": "sum of per-step CUDA-event times, max over ranks"},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "steps/s",
                "h2d_bytes_per_step": int(real_h.numel() * 4 + (0 if args.device_latents else z_h.numel() * 4)) * world,
                "d2h_bytes_per_step": 8 * 4 * world, "wall_s": wall_e2e,
                "input_copies": "inside the step graph, image copy overlapped with G(z)" if tr.graph_pinned is not None else "cudaMemcpyAsync in front of the graph replay",
                "call": "ProtectedDCGANTrainer.step_from_host(real_cpu, latent_cpu) -> metrics dict (one 32-byte "
                        "board copy per rank; the values are already reduced over the ranks on the device)",
                "latents": "device (Philox)" if args.device_latents else "host randn, copied every step"},
        "gpu_launches": int(tr.launches_per_step or 0) * args.steps,
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak_tf, "unit": "TFLOP/s",
                     "frac": achieved / peak_tf,
                     "traffic": (traffic["gemm_dram_bytes_per_step"] / max(1, traffic["gemm_launches"])) if traffic else None,
                     "traffic_note": ("mean DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) per GEMM launch over the "
                                      "%d tapgemm/wgrad launches of one batch-%d step = %.1f MB per step, against %.1f MB of "
                                      "algorithmic operand/result bytes (%s)" % (
                                          traffic["gemm_launches"], traffic["batch"], traffic["gemm_dram_bytes_per_step"] / 1e6,
                                          traffic["gemm_algorithmic_bytes_per_step"] / 1e6, traffic["source"]))
                     if traffic else "profiles/r2_step_traffic.json not present",
                     "kernel": "tapgemm_kernel + wgrad_kernel (tcgen05 implicit GEMM), %d launches/step" % n_gemm,
                     "peak_source": pk_src + " bf16_tflops_sustained",
                     "gemm_ms_per_step": gemm_ms, "gemm_share_of_step": gemm_ms / ms,
                     "step_model_flops_tflops": FLOP_PER_SAMPLE * args.batch / world / (ms * 1e-3) / 1e12,
                     # What bounds these kernels: every 128 x BLOCK_N tile re-reads its A box per tap and its B block per
                     # k-block through L2 (128*BLOCK_N/(128+BLOCK_N) flop per byte), and the L2 -> SM path saturates at
                     # ~6300 B/clk chip-wide (B300_MICROARCH.md, LTS throughput cap; taken as is for B200).
                     "l2_operand_stream": {"bytes_per_step": l2_bytes, "achieved_tb_s": l2_bytes / (gemm_ms * 1e-3) / 1e12,
                                           "cap_tb_s": l2_cap / 1e12, "frac": l2_bytes / (gemm_ms * 1e-3) / l2_cap,
                                           "note": "TMA bytes of the GEMM launches (A boxes per tap + B blocks per k-block, "
                                                   "counted from the tile plans) over their summed duration"},
                     "by_kind": {k: {"tflops": v[0] / (v[1] * 1e-3) / 1e12 if v[1] > 0 else 0.0, "ms": v[1], "launches": v[2]}
                                 for k, v in sorted(by_kind.items())}},
        # BASELINE.json's second metric, stated as such: the SSIM (+ sign-loss) path against the HBM roofline.  The
        # sign loss adds no HBM pass of its own (value: one 448-gamma launch; gradient: inside the BatchNorm backward).
        "secondary_metric": {"metric": "SSIM+sign-loss path HBM GB/s vs peak (SSIM fwd+bwd, 36*B*H*W algorithmic bytes)",
                             "value": ssim_big, "unit": "GB/s", "higher_is_better": True,
                             "frac_of_peak": ssim_big / pk.get("hbm_gbs", 6650.0), "target_frac": 0.70,
                             "peak": pk.get("hbm_gbs"), "peak_source": pk_src, "batch": 16384,
                             "at_step_batch": {"batch": local_batch, "value": ssim_small},
                             "roofline": {"bound": "fp32 FMA pipe (not HBM)", "traffic": 549.2e6,
                                          "traffic_note": "ncu dram read+write of one launch at B=16384 (profiles/"
                                          "r1_ssim32_warp_kernel_full.txt); algorithmic 604 MB, 55 MB of dX still in L2"},
                             "note": "the 70 % target needs more arithmetic than the chip has at fp32 accuracy: see "
                                     "DESIGN.md section 5 (FMA-pipe ceiling 3.2 TB/s; split-bf16 tensor-core variant "
                                     "needs >= 1.1 PFLOP/s at HBM speed)"},
        "last_metrics": metrics_box.get("m"),
    }
    if not args.skip_cpu_baseline and world == 1:
        sps, dt, cores = cpu_reference_steps_per_sec(6, 1, args.batch)
        line["cpu_baseline"] = {"value": sps, "unit": "steps/s", "cores": cores, "kind": "port",
                                "sample": "6 steps at batch %d (the metric's global batch) in %.1f s after 1 warm-up"
                                          % (args.batch, dt)}
    else:
        line["cpu_baseline"] = None
    if not args.skip_eager_baseline and world == 1:
        try:
            eager = torch_eager_steps_per_sec(device, args.batch)
            line["torch_eager_baseline"] = {
                "unit": "steps/s", "fp32": eager["fp32"], "tf32": eager["tf32"],
                "speedup_vs_fp32": e2e_value / eager["fp32"], "speedup_vs_tf32": e2e_value / eager["tf32"],
                "what": "the oracle's step (reference semantics, plain PyTorch ops) run eagerly on this GPU through "
                        "cuDNN/cuBLAS, pinned host batch in, metrics out every step (as train.py does); compared "
                        "with this repo's e2e value"}
        except Exception as e:                       # a baseline leg never takes the measurement down
            line["torch_eager_baseline"] = {"error": repr(e)[:200]}
    print(json.dumps(line))
    _finish(world)


def run_verify(args):
    """BASELINE config 5: watermark / signature verification sweep (experiments/image_generation.py:185-223 and
    sign_flip.py:59-77) over --samples trigger samples, sharded over the ranks, one all-reduce of four sums."""
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        sys.stdout.flush()
        saved = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=device)
            dist.barrier()
        finally:
            sys.stdout.flush()
            os.dup2(saved, 1)
            os.close(saved)
    import ipr_gan_b200
    ipr_gan_b200.enable_dropin()
    import networks
    import tools
    from configs import presets
    from ipr_gan_b200 import _lib, verify
    torch.manual_seed(1234)
    G = networks.ConvGenerator32().to(device)
    bb = presets.dcgan_blackbox()
    fn_inp = tools.TransformDist(bb.fn_inp).to(device)
    fn_out = tools.PasteWatermark(bb.fn_out, normalized=True).to(device)
    sign = tools.SignLossModel(G, presets.dcgan_whitebox()).to(device)

    def sweep():
        return verify.verification_sweep(G, fn_inp, fn_out, args.samples, batch=2500, sign_model=sign)
    for _ in range(max(3, args.warmup)):
        sweep()
    flush = torch.empty(256 * 1024 * 1024 // 4, device=device)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    total, before = 0.0, _lib.launch_count()
    for _ in range(args.steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        res = sweep()
        b.record()
        torch.cuda.synchronize()
        total += a.elapsed_time(b)
    launches = _lib.launch_count() - before
    t = torch.tensor([total], device=device, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    clocks = sampler.stop() if rank == 0 else None
    if rank == 0:
        ms = float(t.item()) / args.steps
        line = {"metric": "watermark verification sweep, trigger samples/sec (G fwd x2, paste, crop, SSIM, pHash p-value, BER)",
                "value": args.samples / (ms * 1e-3), "unit": "samples/s", "n_gpus": world, "steps": args.steps,
                "warmup": max(3, args.warmup), "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
                "vs_baseline": None, "dtype": "bf16 generator, fp32 SSIM, integer hash", "data": "synthetic",
                "config": {"workload": "verification sweep, %d trigger samples (BASELINE config 5)" % args.samples,
                           "per_gpu_samples": (args.samples + world - 1) // world, "l2": "flushed between sweeps",
                           "timing": "CUDA events around each sweep (includes its one host read-back), max over ranks"},
                "clocks": clocks, "gpu_launches": int(launches), "result": {k: v for k, v in res.items() if k != "per_sample"}}
        print(json.dumps(line))
    _finish(world)


def build_family(workload, use_graph=True):
    """-> (trainer, workload name, pinned host inputs) of BASELINE config 3 (srgan) / 4 (cyclegan)."""
    import torch
    from ipr_gan_b200 import trainer as T
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    gen = torch.Generator().manual_seed(1234)
    if workload == "srgan":
        tr = T.ProtectedSRGANTrainer(16, dev, use_graph=use_graph)
        host = (torch.rand(16, 3, 24, 24, generator=gen).pin_memory(), torch.rand(16, 3, 96, 96, generator=gen).pin_memory())
        name = "IPR-SRGAN 24->96 protected step, batch 16 (SRResNet + Discriminator96 + VGG content loss)"
    else:
        tr = T.ProtectedCycleGANTrainer(dev, 128, use_graph=use_graph)
        host = ((torch.rand(1, 3, 128, 128, generator=gen) * 2 - 1).pin_memory(),
                (torch.rand(1, 3, 128, 128, generator=gen) * 2 - 1).pin_memory())
        name = "IPR-CycleGAN 128x128 protected step, batch 1 (Resnet9Blocks x2 + PatchGAN x2, InstanceNorm sign loss)"
    for dst, src in zip((tr.low_res, tr.high_res) if workload == "srgan" else (tr.real_A, tr.real_B), host):
        dst.copy_(src)
    return tr, name, host


def run_family(args):
    """BASELINE configs 3 / 4: one protected training step of IPR-SRGAN (experiments/image_super_resolution.py:84-113) or
    IPR-CycleGAN (experiments/image_translation.py:90-112) through the drop-in models, networks on the native engine;
    the step replays as CUDA graph(s) (ipr_gan_b200/trainer.py), host batch in / metrics out inside the timed region."""
    import torch
    from ipr_gan_b200 import _lib
    tr, name, host = build_family(args.workload, use_graph=not args.no_graph)
    dev = tr.device
    tr.capture(max(3, args.warmup))
    for _ in range(max(3, args.warmup)):
        last = tr.step_from_host(*host)
    flush = torch.empty(256 * 1024 * 1024 // 4, device=dev)
    sampler = ClockSampler(0)
    sampler.start()
    torch.cuda.synchronize()
    total, dev_total = 0.0, 0.0
    for _ in range(args.steps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        last = tr.step_from_host(*host)
        b.record()
        torch.cuda.synchronize()
        total += a.elapsed_time(b)
    # device-resident variant: inputs already in HBM, no read-back inside the timed region
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps):
        tr.step()
    b.record()
    torch.cuda.synchronize()
    dev_ms = a.elapsed_time(b) / args.steps
    launches = (tr.launches_per_step or 0) * args.steps
    ms = total / args.steps
    h2d = sum(t.numel() * 4 for t in host)
    print(json.dumps({"metric": name + ", steps/sec", "value": 1e3 / dev_ms, "unit": "steps/s", "n_gpus": 1, "steps": args.steps,
                      "warmup": max(3, args.warmup), "ms_per_step": dev_ms, "higher_is_better": True, "scaling": "weak",
                      "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
                      "config": {"workload": name, "cuda_graph": tr.use_graph, "l2": "e2e: flushed between steps; value: back-to-back "
                                 "replays (activations of one step exceed L2)",
                                 "timing": "CUDA events; value = inputs resident, e2e = pinned host batch in / metrics out per step"},
                      "clocks": sampler.stop(), "gpu_launches": int(launches),
                      "e2e": {"value": 1e3 / ms, "unit": "steps/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": 64,
                              "ms_per_step": ms},
                      "last_metrics": last}))


def _finish(world):
    """Leave without tearing NCCL down: destroying a process group whose collectives live inside a captured CUDA
    graph can block at exit; the ranks just synchronise and exit."""
    import torch
    sys.stdout.flush()
    sys.stderr.flush()
    if world > 1:
        torch.cuda.synchronize()
        os._exit(0)


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    elif a.workload == "verify":
        run_verify(a)
    elif a.workload in ("srgan", "cyclegan"):
        run_family(a)
    else:
        run_b200(a)
