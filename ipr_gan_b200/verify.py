"""On-device watermark / signature verification sweeps (BASELINE config 5; the loop of
experiments/image_generation.py:185-223 and sign_flip.py:59-77 without the .cpu() hops and the per-image
Python loop).

Latent-input generators (DCGAN), ``verification_sweep``:

    z -> x = G(z);  zwm = fn_inp(z);  xwm = G(zwm);  ywm = fn_out(x)
    wm_x = postproc(apply_mask(xwm));  wm_y = postproc(apply_mask(ywm))          postproc = (clamp(-1,1)+1)/2
    q = ssim(wm_x, wm_y) per sample;  p = PDQ-hash matching p-value;  match = p < p_thres

Image-to-image generators (SRGAN's SRResNet, CycleGAN's GB), ``image_verification_sweep``: the same with an input
image in place of z (models/wrappers.py:48-51: the noise patch is pasted into the input), and the post-processing
chosen by ``fn_out.normalized``: (clamp(-1,1)+1)/2 for [-1, 1] outputs, clamp(0,1) for outputs in data range 1.
Its per-batch body is captured once into a CUDA graph and replayed.

All per-sample quantities stay on the GPU; one small all-reduce merges the per-rank sums when the sweep is sharded
over ranks (independent shards, no data-path collective).
"""
import torch

from . import dist, ops


_STAGING = {}


def _staging(*shape):
    """Pinned host buffer of one shape (page-locking 5 MB costs ~2 ms: done once per shape)."""
    buf = _STAGING.get(shape)
    if buf is None:
        buf = _STAGING[shape] = torch.empty(*shape).pin_memory()
    return buf


def _postproc(x):
    return (x.clamp(-1, 1) + 1.0) / 2.0


def rank_slice(n, rank, world):
    """[lo, hi) of the n sweep samples that rank ``rank`` of ``world`` evaluates: contiguous slices of ceil(n / world)
    samples, so the last ranks may get fewer (or none)."""
    per_rank = (n + world - 1) // world
    return min(n, rank * per_rank), min(n, (rank + 1) * per_rank)


def _window(fn_out):
    mod = fn_out.module if hasattr(fn_out, "module") else fn_out
    return mod, mod.config.size, mod.position


def _score(xwm, ywm, crop_bg, pos, size, postproc, p_thres, sums):
    """Crops through the opaque mask + post-processing, per-sample SSIM / p-value / Hamming count; the three sums
    (q, p, matches) accumulate into the float64 device vector ``sums``.  -> (q, p, r)"""
    wm_x = ops.crop_patch(xwm, crop_bg, pos, size, postproc=postproc)     # crop + post-processing in one launch
    wm_y = ops.crop_patch(ywm, crop_bg, pos, size, postproc=postproc)
    q = ops.ssim_per_sample(wm_x, wm_y)
    p, r = ops.matching_prob(wm_x, wm_y)
    sums[:3] += torch.stack([q.double().sum(), p.double().sum(), (p < p_thres).double().sum()])
    return q, p, r


def _finish(G, sums, n_local, keep, sign_model):
    """Sample count, the one all-reduce over ranks, the host read-back, WBOX and the per-sample tensors."""
    sums[3] += float(n_local)
    if dist.world() > 1:
        torch.distributed.all_reduce(sums)
    s = sums.tolist()
    out = {"Q_WM": s[0] / s[3], "P": s[1] / s[3], "MATCH": int(round(s[2])), "N": int(round(s[3]))}
    if sign_model is not None:
        wrong, total = sign_model.compute_ber_counts(G)
        out["WBOX"] = wrong / total
        out["WBOX_counts"] = (wrong, total)
    if keep is not None:
        out["per_sample"] = {k: torch.cat(v) for k, v in keep.items()}
    return out


@torch.no_grad()
def verification_sweep(G, fn_inp, fn_out, n_samples, batch=500, p_thres=0.01, seed=1234, sign_model=None,
                       return_per_sample=False):
    """G, fn_inp, fn_out: the (drop-in) generator and trigger modules on a CUDA device.  The watermark window is taken
    with ``opaque=True`` semantics like evaluate() does (a pure crop).  -> dict with Q_WM, P, MATCH, N (+ WBOX)."""
    dev = next(G.parameters()).device
    was_training = G.training
    G.eval()
    rank, world = dist.rank(), dist.world()
    lo, hi = rank_slice(n_samples, rank, world)
    gen = torch.Generator().manual_seed(seed + rank)
    _, size, pos = _window(fn_out)
    crop_bg = torch.zeros(1, 1, size, size, device=dev)             # evaluate() forces opaque=True for apply_mask
    sums = torch.zeros(4, device=dev, dtype=torch.float64)
    keep = {"q": [], "p": [], "r": []} if return_per_sample else None
    # latents: drawn batch by batch from the CPU generator (experiments/image_generation.py:191-196) straight into ONE
    # pinned buffer, so every copy is truly asynchronous and the host draws batch i+1 while the GPU works on batch i
    # (a pageable 1.3 MB source made each copy wait for the stream: ~1 ms of idle GPU per 2 500 samples)
    staged = _staging(max(hi - lo, 1), 128)
    i = lo
    while i < hi:
        b = min(batch, hi - i)
        z_host = staged[i - lo:i - lo + b]
        torch.randn(b, 128, generator=gen, out=z_host)
        z = z_host.to(dev, non_blocking=True)
        x = G(z)
        xwm = G(fn_inp(z))
        ywm = fn_out(x)
        q, p, r = _score(xwm, ywm, crop_bg, pos, size, True, p_thres, sums)
        if keep is not None:
            keep["q"].append(q), keep["p"].append(p), keep["r"].append(r)
        i += b
    out = _finish(G, sums, hi - lo, keep, sign_model)
    if was_training:
        G.train()
    return out


class _InputStager(object):
    """Copies batches of this rank's slice of a host tensor into device buffers.  A pageable source goes through one
    pinned buffer of two batch slots: the host fills slot j % 2 while the GPU still works on the previous batch, and
    only waits for the device copy out of that slot two batches ago.  A pinned or device source is copied directly."""

    def __init__(self, inputs, batch):
        self.inputs = inputs
        self.direct = inputs.is_cuda or inputs.is_pinned()
        if not self.direct:
            self.pinned = _staging(2, batch, *inputs.shape[1:])
            self.copied = [None, None]
        self.j = 0

    def copy_into(self, dst, lo, hi):
        src = self.inputs[lo:hi]
        if self.direct:
            dst.copy_(src, non_blocking=True)
            return dst
        slot = self.j % 2
        self.j += 1
        if self.copied[slot] is not None:
            self.copied[slot].synchronize()
        host = self.pinned[slot, :hi - lo]
        host.copy_(src)
        dst.copy_(host, non_blocking=True)
        self.copied[slot] = torch.cuda.Event()
        self.copied[slot].record()
        return dst


@torch.no_grad()
def image_verification_sweep(G, fn_inp, fn_out, inputs, batch=16, p_thres=0.05, sign_model=None,
                             return_per_sample=False, eager=False):
    """Verification of an image-to-image generator (SRGAN: ``G`` on low-res inputs; CycleGAN: ``GB`` on real_B images).

    G, fn_inp, fn_out: the (drop-in) generator and the checkpointed trigger modules on a CUDA device.  ``fn_inp`` is
    used as stored (never ``reset()``: its noise patch IS the trigger).  inputs: (N, C, h, w) float32 tensor of ALL N
    verification inputs (host memory; every rank evaluates its contiguous slice, see ``rank_slice``).  G runs in eval
    mode (BatchNorm: running statistics; InstanceNorm: per-image statistics); its training mode is restored after.

    Per batch:  x = G(inp);  Gxwm = G(fn_inp(inp));  ywm = fn_out(x);  crops of Gxwm and ywm through the opaque mask,
    post-processed according to ``fn_out.normalized``;  q = SSIM, p = pHash p-value, r = matching bits, match = p < p_thres.

    Every full batch replays ONE CUDA graph of that body over a static input buffer (the ragged last batch runs
    eagerly); the sums stay on the device and are read once.  ``eager=True`` runs every batch eagerly: a debugging
    switch (the results are bit-identical), not a performance option.  -> dict with Q_WM, P, MATCH, N (+ WBOX, WBOX_counts, per_sample)."""
    if not isinstance(inputs, torch.Tensor) or inputs.dim() != 4 or inputs.dtype != torch.float32:
        raise ValueError("inputs must be an (N, C, H, W) float32 tensor")
    if inputs.shape[0] < 1 or batch < 1:
        raise ValueError("need at least one input and a batch of at least one")
    dev = next(G.parameters()).device
    lo, hi = rank_slice(inputs.shape[0], dist.rank(), dist.world())
    mod, size, pos = _window(fn_out)
    postproc = ops.postproc_mode(mod.normalized)
    crop_bg = torch.zeros(1, 1, size, size, device=dev)             # evaluate() forces opaque=True for apply_mask
    sums = torch.zeros(4, device=dev, dtype=torch.float64)
    keep = {"q": [], "p": [], "r": []} if return_per_sample else None
    n_full = (hi - lo) // batch
    static_in = torch.empty(min(batch, max(hi - lo, 1)), *inputs.shape[1:], device=dev)
    stager = _InputStager(inputs, batch)

    def body(inp):
        x = G(inp)
        gxwm = G(fn_inp(inp))
        ywm = fn_out(x)
        return _score(gxwm, ywm, crop_bg, pos, size, postproc, p_thres, sums)

    def kept(qpr, clone):
        if keep is not None:
            for k, t in zip("qpr", qpr):
                keep[k].append(t.clone() if clone else t)

    was_training = G.training
    G.eval()
    try:
        i = lo
        if not eager and n_full > 0:
            from .trainer import _capture
            stager.copy_into(static_in, lo, lo + batch)
            outs = []
            graph, _ = _capture(lambda: outs.append(body(static_in)), dev, warmup=1)
            sums.zero_()                            # the warm-up batch accumulated; the capture itself ran nothing
            qpr = outs[-1]
            for _ in range(n_full):
                stager.copy_into(static_in, i, i + batch)
                graph.replay()
                kept(qpr, True)
                i += batch
        while i < hi:
            b = min(batch, hi - i)
            kept(body(stager.copy_into(static_in[:b], i, i + b)), False)
            i += b
        return _finish(G, sums, hi - lo, keep, sign_model)
    finally:
        if was_training:
            G.train()
