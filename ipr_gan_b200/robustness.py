"""Robustness sweeps of a protected generator, on the device: the removal attack (global magnitude pruning, the
reference's prune.py, SURVEY.md 2.1 row 34) and the ambiguity attack (a random share of the signature's gamma signs
flipped, sign_flip.py:59-77, SURVEY.md 3.3 / 8d), every level followed by the verification sweep of ``verify.py``.

Both perturbations write the generator's flat fp32 parameter arena (``flat.py``) in place with one kernel sequence
(csrc/prune.cu) and bump ``arena.version``, which is what makes the packed GEMM operands rebuild (``engine.PackSet``).
A sweep snapshots the arena once, restores it before every level and again at the end, so no level reloads the
experiment from disk and the model leaves the sweep as it entered it.

``torch.nn.utils.prune`` itself cannot be used on these networks: their forward never calls the child modules, so
the pruning pre-hook never runs.  The native forward refuses such a module (``engine.refuse_pruned``).
"""
import numbers
import weakref

import torch
import torch.nn as nn

from . import flat, ops, verify

AMOUNTS = (0.1, 0.2, 0.3, 0.4, 0.5, 0.6, 0.7, 0.8, 0.9)
PERCENTS = (10, 20, 30, 40, 50, 60, 70, 80, 90, 100)
_PRUNABLE = (nn.Conv2d, nn.ConvTranspose2d, nn.Linear)
_NORMS = (nn.BatchNorm2d, nn.InstanceNorm2d)
_TABLES = {}                    # (device, segments) -> device copy of the segment table
_SEGMENTS = weakref.WeakKeyDictionary()     # network -> (arena, its prunable segments)
_RESULT_KEYS = ("Q_WM", "P", "MATCH", "N", "WBOX", "WBOX_counts")


def _module(net):
    """A ``Replica``'s wrapped network, or the network itself."""
    inner = getattr(net, "module", None)
    return inner if isinstance(inner, nn.Module) else net


def _generator(net):
    import networks
    net = _module(net)
    if not isinstance(net, (networks.ConvGenerator, networks.SRResNet, networks.ResnetGenerator)):
        raise TypeError("expected a ConvGenerator32/64, SRResNet or ResnetGenerator (or a Replica of one), got %s"
                        % type(net).__name__)
    from .engine import refuse_pruned
    refuse_pruned(net)
    return net


def prunable_segments(net):
    """Arena segments ``[(offset, count), ...]`` (ascending offsets) of every Conv2d / ConvTranspose2d / Linear weight
    of one generator: what pruning may zero.  Biases, normalisation parameters, PReLU slopes, the arena's alignment
    padding and, for CycleGAN, the other generator's half of the shared arena are not in the list."""
    return _segments(_generator(net))[1]


def _segments(net):
    """-> (arena, segments), the list cached per network while its first parameter stays in the same valid arena
    (walking a 165-module SRResNet for its parameters alone costs ~0.2 ms of host time per call)."""
    arena = flat.arena_of(next(net.parameters()))
    hit = _SEGMENTS.get(net)
    if hit is not None and hit[0] is arena:
        return hit
    arena = flat.module_arena(net)
    segs = sorted((arena.offset_of(m.weight), m.weight.numel()) for m in net.modules() if isinstance(m, _PRUNABLE))
    _SEGMENTS[net] = (arena, segs)
    return arena, segs


def prune_count(amount, n):
    """Entries to prune out of n, as ``torch.nn.utils.prune`` counts them: an integer amount is the count, a float
    amount in [0, 1] the share, rounded with Python's round()."""
    if isinstance(amount, bool) or not isinstance(amount, numbers.Real):
        raise TypeError("amount must be an int or a float, got %r" % (amount,))
    if isinstance(amount, numbers.Integral):
        if not 0 <= amount <= n:
            raise ValueError("amount=%d entries outside [0, %d]" % (amount, n))
        return int(amount)
    if not 0.0 <= amount <= 1.0:
        raise ValueError("amount=%r outside [0, 1]" % (amount,))
    return int(round(amount * n))


def _segment_table(segs, device):
    key = (str(device), tuple(segs))
    t = _TABLES.get(key)
    if t is None:
        t = _TABLES[key] = torch.tensor(segs, dtype=torch.int64).to(device)
    return t


def prune_(net, amount):
    """Global magnitude pruning of one generator's conv / linear weights, in place on the device:
    ``torch.nn.utils.prune.global_unstructured(..., pruning_method=L1Unstructured, amount=amount)`` followed by
    ``prune.remove``, over the tensors of ``prunable_segments``.  Exactly k = round(amount * N) entries become w * 0;
    ties at the threshold magnitude go lowest arena offset first.  -> k

    Nothing is read back, so the call can be captured in a CUDA graph once it has run eagerly (the first call copies
    the segment table to the device); a replay does not bump ``arena.version`` -- the caller does."""
    net = _generator(net)
    arena, segs = _segments(net)
    n = sum(c for _, c in segs)
    k = prune_count(amount, n)
    ops.prune_magnitude_(arena.param, _segment_table(segs, arena.param.device), n, k)
    arena.version += 1
    return k


def _signature_gammas(net):
    return [m.weight for m in net.modules() if isinstance(m, _NORMS)]


def sign_flip_offsets(net, percent, generator):
    """Arena offsets of the gammas the sign flip negates in one generator: its normalisation gammas concatenated in
    ``named_modules()`` order (``tools.SignLossModel``'s order), one ``torch.randperm(n, generator=generator)``, and
    the first ``int(n * percent / 100)`` of it.  -> int64 CPU tensor"""
    net = _module(net)
    arena = flat.module_arena(net)
    flat_idx = torch.cat([torch.arange(g.numel(), dtype=torch.int64) + arena.offset_of(g) for g in _signature_gammas(net)])
    n = flat_idx.numel()
    perm = torch.randperm(n, generator=generator)
    return flat_idx[perm[:int(n * percent / 100)]]


def _generators(model):
    return [m for name, m in model._modules.items() if name.startswith("G")]


def flip_signs_(model, percent, generator):
    """The ambiguity attack's perturbation: for every ``G*`` network of the (wrapped) model, in ``_modules`` order,
    negate ``int(n * percent / 100)`` of its n normalisation gammas chosen by one ``torch.randperm(n)`` drawn from the
    CPU ``generator`` (``sign_flip_offsets``).  The reference tree is not at hand: this rounding and ordering are the
    definition used here for sign_flip.py:59-77 (SURVEY.md 3.3 / 8d).  One launch per generator.  -> entries flipped"""
    total = 0
    for g in _generators(model):
        net = _generator(g)
        idx = sign_flip_offsets(net, percent, generator)
        arena = flat.module_arena(net)
        ops.negate_indexed_(arena.param, idx.to(arena.param.device))
        arena.version += 1
        total += idx.numel()
    return total


def _sweep(model, sweep_args):
    """The verification sweep matching the target: latents for DCGAN (``verify.verification_sweep``, p_thres 0.01
    by default), images for SRGAN's G / CycleGAN's GB (``verify.image_verification_sweep`` with ``inputs=``, 0.05)."""
    import networks
    target = getattr(model, model.config.target)
    fn = verify.verification_sweep if isinstance(_module(target), networks.ConvGenerator) else \
        verify.image_verification_sweep
    return fn(target, model.fn_inp, model.fn_out, sign_model=model.loss_model, **sweep_args)


def _levels(model, arenas, levels, perturb, level_key, count_key, sweep_args):
    target = getattr(model, model.config.target)
    modes = [(m, m.training) for m in target.modules()]
    snaps = []
    for a in arenas:
        if all(a is not b for b, _ in snaps):
            snaps.append((a, a.param.clone()))

    def restore():
        for a, saved in snaps:
            a.param.copy_(saved)
            a.version += 1

    rows = []
    try:
        for level in levels:
            restore()
            count = perturb(level)
            res = _sweep(model, sweep_args)
            row = {level_key: level, count_key: count}
            row.update((k, res[k]) for k in _RESULT_KEYS if k in res)
            rows.append(row)
    finally:
        restore()
        for m, mode in modes:
            m.training = mode
    return rows


@torch.no_grad()
def prune_sweep(model, amounts=AMOUNTS, **sweep_args):
    """Removal attack: for each amount, the target generator (``model.config.target`` of the protection wrapper)
    pruned by ``prune_`` from its original weights, then verified.  ``sweep_args`` go to the verification sweep
    (``n_samples=`` / ``batch`` / ``seed`` for DCGAN, ``inputs=`` / ``batch`` for the image generators); every level
    sees the same latents or inputs.  Data-parallel: every rank prunes its identical replica identically and the
    sweep shards the samples as usual.  -> one dict per level: amount, pruned, Q_WM, P, MATCH, N (+ WBOX,
    WBOX_counts with a white-box wrapper).  The arena, BatchNorm running statistics and training modes are left as
    they were."""
    net = _generator(getattr(model, model.config.target))
    return _levels(model, [flat.module_arena(net)], amounts, lambda a: prune_(net, a), "amount", "pruned", sweep_args)


@torch.no_grad()
def sign_flip_sweep(model, percents=PERCENTS, seed=0, **sweep_args):
    """Ambiguity attack: for each percent, ``flip_signs_`` on the original weights with a CPU generator seeded with
    ``seed`` afresh for every level (a level's flips depend on (seed, percent) only, and a larger share flips a
    superset), then the verification sweep of the target as in ``prune_sweep``.  -> one dict per level: percent,
    flipped (over all G* networks), Q_WM, P, MATCH, N (+ WBOX, WBOX_counts)."""
    arenas = [flat.module_arena(_generator(g)) for g in _generators(model)]

    def perturb(p):
        return flip_signs_(model, p, torch.Generator().manual_seed(seed))
    return _levels(model, arenas, percents, perturb, "percent", "flipped", sweep_args)
