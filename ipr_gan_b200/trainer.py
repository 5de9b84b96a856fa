"""Protected IPR-DCGAN training step as a user of the drop-in API would run it
(``models.DCGAN`` -> ``BlackBoxWrapper`` -> ``WhiteBoxWrapper``, the stack built by
experiments/image_generation.py:38-84), plus the two B200-specific pieces around it:

* the whole step (update_d + update_g: 2 generator forwards, 3 discriminator forwards, all backwards,
  SSIM + sign loss, both Adam updates) is captured ONCE into a CUDA graph and replayed -- at 64-512
  samples per GPU the step is a few hundred short kernels, so launch latency would otherwise dominate;
* data parallelism is one process per GPU: gradients are all-reduced over NCCL inside
  ``optimizer.step()`` (``dist.AllReduceOptimizer``), BatchNorm statistics stay per rank exactly like the
  reference's ``nn.DataParallel`` replicas (experiments/base.py:36-39).
"""
import contextlib

import torch

import ipr_gan_b200

ipr_gan_b200.enable_dropin()


@contextlib.contextmanager
def _nvtx(name):
    """NVTX range around a step (SURVEY.md section 5: tracing) -- shows up in nsys / ncu timelines; ~1 us."""
    torch.cuda.nvtx.range_push(name)
    try:
        yield
    finally:
        torch.cuda.nvtx.range_pop()

import models  # noqa: E402
from configs import presets  # noqa: E402
from ipr_gan_b200 import _lib, dist, engine  # noqa: E402


class ProtectedDCGANTrainer(object):
    def __init__(self, batch, device, seed=1234, fn_inp="TransformDist", use_graph=True, size=32,
                 device_latents=False, pinned_inputs=False, wm_size=16):
        # size / wm_size: 32 / 16 for the CIFAR configs, 64 / 32 for the CUB-200 ones (SURVEY.md section 8a, A4)
        self.batch, self.device, self.use_graph = batch, device, use_graph
        self.device_latents = device_latents
        # pinned_inputs: a second graph whose first nodes are the host->device copies of the step's batch out of the
        # trainer's own pinned buffers (``real_host`` / ``latent_host``, which a data loader fills in place): the image
        # copy runs on a copy stream that only D(real) waits for, so it overlaps G(z) instead of preceding the step
        self.pinned_inputs = bool(pinned_inputs and use_graph)
        self.graph_pinned = None
        self._copy_stream = torch.cuda.Stream(device=device) if self.pinned_inputs else None
        torch.manual_seed(seed)                      # identical initial replicas on every rank
        mcfg = presets.dcgan_model(size)
        if use_graph:
            mcfg.opt_param["capturable"] = True
        model = models.DCGAN(mcfg, device=[device])
        model = models.BlackBoxWrapper(model, presets.dcgan_blackbox(fn_inp=fn_inp, wm_size=wm_size))
        model = models.WhiteBoxWrapper(model, presets.dcgan_whitebox())
        self.model = model
        self.real = torch.zeros(batch, 3, size, size, device=device)
        self.latent = torch.zeros(batch, 128, device=device)
        self.real_host = torch.zeros(batch, 3, size, size).pin_memory()
        self.latent_host = torch.zeros(batch, 128).pin_memory()
        self.graph = None
        self.launches_per_step = None
        # latents drawn on the device (Philox, position kept in device memory): no host randn + H2D copy per step
        # (experiments/image_generation.py:93-96); one stream per rank
        from ipr_gan_b200 import dist, ops
        self.normal = ops.DeviceNormal(device, seed * 7919 + dist.rank()) if device_latents else None

    # one reference-API step on whatever is in the static device buffers
    def _step(self):
        if self.normal is not None:
            self.normal.fill_(self.latent)
        self.model.update_d({"real_sample": self.real, "latent": self.latent})
        self.model.update_g({"fake_sample": self.model.fake_sample})

    def _step_from_pinned(self):
        """The step preceded by its own input copies (captured as the ``graph_pinned`` variant)."""
        dev = self.device
        main, cs = torch.cuda.current_stream(dev), self._copy_stream
        cs.wait_stream(main)
        with torch.cuda.stream(cs):
            self.real.copy_(self.real_host, non_blocking=True)
        if self.normal is None:
            self.latent.copy_(self.latent_host, non_blocking=True)      # G(z) needs it first: main stream
        if engine.concurrent_passes():
            engine.aux_stream(dev).wait_stream(cs)   # D(real) runs there (models/dcgan.py forward_d): only it waits
        else:
            main.wait_stream(cs)
        self._step()
        main.wait_stream(cs)                         # every forked stream rejoins before the capture ends

    def set_inputs(self, real, latent):
        """Stage a host (or device) batch into the static device buffers (async when the source is pinned)."""
        self.real.copy_(real, non_blocking=True)
        if latent is not None:
            self.latent.copy_(latent, non_blocking=True)

    def capture(self, warmup=3):
        """Warm up eagerly on a side stream, then capture the step into a CUDA graph."""
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            for _ in range(warmup):
                before = _lib.launch_count()
                self._step()
                self.launches_per_step = _lib.launch_count() - before
        torch.cuda.current_stream(self.device).wait_stream(s)
        torch.cuda.synchronize(self.device)
        if not self.use_graph:
            return
        engine.reset_caches()                       # weight packing must be part of the captured step
        self.graph = torch.cuda.CUDAGraph()
        # thread_local: NCCL's watchdog thread may query events while this thread captures (multi-GPU runs)
        with torch.cuda.graph(self.graph, stream=s, capture_error_mode="thread_local"):
            before = _lib.launch_count()
            self._step()
            self.launches_per_step = _lib.launch_count() - before
        torch.cuda.synchronize(self.device)
        if self.pinned_inputs:
            engine.reset_caches()
            self.graph_pinned = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_pinned, stream=s, capture_error_mode="thread_local"):
                self._step_from_pinned()
            torch.cuda.synchronize(self.device)

    def step(self):
        """One training step on the current contents of the device buffers."""
        with _nvtx("ipr.dcgan.step"):
            self._step_or_replay()

    def _step_or_replay(self):
        if self.graph is not None:
            self.graph.replay()
            board = self.model.board
            if board is not None:
                board.touch()                       # the replay rewrote the loss slots behind the host's back
        else:
            self._step()

    def step_from_host(self, real_cpu, latent_cpu=None):
        """The call a user of the reference makes (experiments/image_generation.py:92-101): host tensors in,
        metrics dict (Python floats) out.  With ``device_latents`` the latent argument is not needed."""
        if self.graph_pinned is not None:
            # batches normally arrive IN the pinned buffers (no host copy); anything else is staged through them.  The
            # previous step's copies have completed: every call ends with the metrics read-back.
            if real_cpu.data_ptr() != self.real_host.data_ptr():
                self.real_host.copy_(real_cpu)
            if latent_cpu is not None and latent_cpu.data_ptr() != self.latent_host.data_ptr():
                self.latent_host.copy_(latent_cpu)
            with _nvtx("ipr.dcgan.step"):
                self.graph_pinned.replay()
                if self.model.board is not None:
                    self.model.board.touch()
            return self.model.get_metrics()
        self.set_inputs(real_cpu, latent_cpu)
        self.step()
        return self.model.get_metrics()


# ------------------------------------------------------------------------------------------ SRGAN / CycleGAN
# Data parallelism as for the DCGAN: one process per GPU, each trainer built with its PER-RANK batch and fed its
# ``dist.shard`` of the global batch; FlatAdam all-reduces the gradient arenas inside the captured graphs.
def _check_shard(host, static):
    """A shard of another size would be broadcast or refused by copy_ further down: say what is wrong instead."""
    if tuple(host.shape) != tuple(static.shape):
        raise ValueError("expected this rank's shard of shape %s, got %s" % (tuple(static.shape), tuple(host.shape)))


def _capture(fn, device, warmup=3, stream=None):
    """Warm ``fn`` up eagerly on a side stream, then capture it into a CUDA graph (weight packing included).
    Warm-up and capture use the SAME stream: autograd's AccumulateGrad nodes remember the stream they were created
    on, and a node from an uncaptured stream inside a capture is a capture-isolation error.
    -> (graph, library launches inside the captured region)"""
    s = stream if stream is not None else torch.cuda.Stream(device=device)
    s.wait_stream(torch.cuda.current_stream(device))
    with torch.cuda.stream(s):
        for _ in range(warmup):
            fn()
    torch.cuda.current_stream(device).wait_stream(s)
    torch.cuda.synchronize(device)
    engine.reset_caches()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s, capture_error_mode="thread_local"):
        before = _lib.launch_count()
        fn()
        launches = _lib.launch_count() - before
    torch.cuda.synchronize(device)
    return graph, launches


class ProtectedSRGANTrainer(object):
    """BASELINE config 3: IPR-SRGAN 24 -> 96 (SRResNet + Discriminator96 + VGG content loss, noise-patch trigger,
    pasted 48 x 48 watermark, SSIM loss, BatchNorm sign loss), GAN phase of experiments/image_super_resolution.py:84-113
    (``update_g`` then ``update_d`` on the same batch).  The eager step is ~1 400 short launches and host-bound; the
    whole step -- including the frozen VGG feature extractor, which stays a PyTorch module -- replays as ONE graph."""

    def __init__(self, batch, device, seed=1234, use_graph=True, pretrain=False):
        self.batch, self.device, self.use_graph, self.pretrain = batch, device, use_graph, pretrain
        import os
        os.environ.setdefault("IPR_VGG_RANDOM_INIT", "1")    # no network for pretrained VGG weights (outside the path)
        torch.manual_seed(seed)
        model = models.SRGAN(presets.srgan_model(), device=[device])
        model = models.BlackBoxWrapper(model, presets.srgan_blackbox())
        self.model = models.WhiteBoxWrapper(model, presets.whitebox("G"))
        self.low_res = torch.zeros(batch, 3, 24, 24, device=device)
        self.high_res = torch.zeros(batch, 3, 96, 96, device=device)
        self.graph, self.launches_per_step = None, None

    def _step(self):
        m = self.model
        m.update_g({"low_res": self.low_res, "high_res": self.high_res, "pretrain": self.pretrain})
        if not self.pretrain:
            m.update_d({"high_res": m.high_res, "super_res": m.super_res})

    def capture(self, warmup=3):
        if self.use_graph:
            self.graph, self.launches_per_step = _capture(self._step, self.device, warmup)
        else:
            for _ in range(warmup):
                before = _lib.launch_count()
                self._step()
                self.launches_per_step = _lib.launch_count() - before

    def step(self):
        with _nvtx("ipr.srgan.step"):
            if self.graph is not None:
                self.graph.replay()
            else:
                self._step()

    def step_from_host(self, low_res_cpu, high_res_cpu):
        """This rank's host batch in, metrics dict out (one step of experiments/image_super_resolution.py's training
        loop).  With several ranks the metrics are the global-batch values, the same dict on every rank."""
        _check_shard(low_res_cpu, self.low_res)
        _check_shard(high_res_cpu, self.high_res)
        self.low_res.copy_(low_res_cpu, non_blocking=True)
        self.high_res.copy_(high_res_cpu, non_blocking=True)
        self.step()
        return dist.reduce_metrics(self.model.get_metrics())


class ProtectedCycleGANTrainer(object):
    """BASELINE config 4: IPR-CycleGAN (two Resnet9Blocks generators, two PatchGAN discriminators, InstanceNorm sign
    loss on GB), one step of experiments/image_translation.py:90-112.  The image-history pools draw from the host RNG
    (models/util.py:5-35), so the step is TWO graphs -- the generator update and the discriminator update -- with the
    pool exchange running eagerly between them on static buffers.  The learning rate is a launch argument of the Adam
    kernel: when the schedulers change it (once per epoch) the graphs are re-captured."""

    def __init__(self, device, size=128, seed=1234, use_graph=True, batch=1):
        self.device, self.size, self.use_graph, self.batch = device, size, use_graph, batch
        # the seed also keeps the host RNG of all ranks in lockstep: the image pools draw from it (dist.pool_query)
        torch.manual_seed(seed)
        model = models.CycleGAN(presets.cyclegan_model(), device=[device])
        model = models.BlackBoxWrapper(model, presets.cyclegan_blackbox())
        self.model = models.WhiteBoxWrapper(model, presets.whitebox("GB"))
        self.inner = model.model
        shape = (batch, 3, size, size)
        self.real_A = torch.zeros(shape, device=device)
        self.real_B = torch.zeros(shape, device=device)
        self.pooled_A = torch.zeros(shape, device=device)
        self.pooled_B = torch.zeros(shape, device=device)
        # several ranks: the pools are queried with the global batch, gathered into these
        w = dist.world()
        self.gathered_A = torch.zeros((w * batch,) + shape[1:], device=device) if w > 1 else None
        self.gathered_B = torch.zeros((w * batch,) + shape[1:], device=device) if w > 1 else None
        self.graph_g = self.graph_d = None
        self.launches_per_step = None
        self._lr = None
        self._generated = None
        self.stream = torch.cuda.Stream(device=device)

    def _lrs(self):
        return (self.inner.optG.param_groups[0]["lr"], self.inner.optD.param_groups[0]["lr"])

    def _step_g(self):
        self.model.update_g({"real_A": self.real_A, "real_B": self.real_B})

    def _pool(self):
        m = self.inner
        # graph mode: the tensors the captured generator update writes (forward_d re-binds m.fake_A / m.fake_B to the
        # pooled images, and no Python runs during a replay to bind them back)
        fake_a, fake_b = self._generated if self._generated is not None else (m.fake_A, m.fake_B)
        self.pooled_A.copy_(dist.pool_query(m.poolA, fake_a, self.gathered_A))
        self.pooled_B.copy_(dist.pool_query(m.poolB, fake_b, self.gathered_B))

    def _step_d(self):
        self.model.update_d({"real_A": self.real_A, "real_B": self.real_B, "fake_A": self.pooled_A,
                             "fake_B": self.pooled_B, "pooled": True})

    def _eager(self):
        self._step_g()
        self._pool()
        self._step_d()

    def capture(self, warmup=3):
        s = self.stream
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            for _ in range(warmup):
                before = _lib.launch_count()
                self._eager()
                self.launches_per_step = _lib.launch_count() - before
        torch.cuda.current_stream(self.device).wait_stream(s)
        torch.cuda.synchronize(self.device)
        if self.use_graph:
            # nothing executes during a capture: eager and graph trainers have run the same number of steps afterwards
            self._generated = None
            self.graph_g, n_g = _capture(self._step_g, self.device, 0, stream=s)
            self._generated = (self.inner.fake_A, self.inner.fake_B)
            self.graph_d, n_d = _capture(self._step_d, self.device, 0, stream=s)
            self.launches_per_step = n_g + n_d
            self._lr = self._lrs()

    def step(self):
        if self.graph_g is None:
            return self._eager()
        # the schedulers moved the learning rate: capture it anew (the rate is the same on every rank, so all ranks
        # re-capture -- their collectives included -- in the same step)
        if self._lrs() != self._lr:
            self.capture(warmup=0)
        with _nvtx("ipr.cyclegan.step"):
            self.graph_g.replay()
            self._pool()
            self.graph_d.replay()

    def step_from_host(self, real_a_cpu, real_b_cpu):
        """This rank's host batch in, metrics dict out; with several ranks the global-batch values on every rank."""
        _check_shard(real_a_cpu, self.real_A)
        _check_shard(real_b_cpu, self.real_B)
        self.real_A.copy_(real_a_cpu, non_blocking=True)
        self.real_B.copy_(real_b_cpu, non_blocking=True)
        self.step()
        return dist.reduce_metrics(self.model.get_metrics())
