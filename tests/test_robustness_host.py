"""CPU: host side of the robustness attacks -- the prune / sign-flip entry points' declarations and argument checks,
the pruning segments of each generator family, the NumPy statement of the pruning kernel's contract against
torch.nn.utils.prune, the sign-flip draw, and the native forward's refusal of torch.nn.utils.prune modules."""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.utils.prune as tprune

from tests import prune_ref

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _nets():
    import networks
    return {"G32": networks.ConvGenerator32, "G64": networks.ConvGenerator64, "SRResNet": networks.SRResNet,
            "Resnet9": networks.Resnet9Blocks}


# ---------------------------------------------------------------------------------------------- C ABI
def test_entry_points_declared_and_exported():
    from ipr_gan_b200 import _lib
    header = open(os.path.join(ROOT, "include", "ipr_b200.h")).read()
    for name in ("ipr_prune_workspace_bytes", "ipr_prune_magnitude_f32", "ipr_negate_indexed_f32"):
        assert name + "(" in header and name in _lib.SIGNATURES
        assert hasattr(ctypes.CDLL(_lib.LIB_PATH), name)
    assert "#define IPR_PRUNE_MAX_SEGMENTS 256" in header


def test_argument_checks_need_no_gpu():
    """Error codes come from the host before any launch (the fake pointers are never dereferenced); k = 0 and an
    empty index list launch nothing."""
    from ipr_gan_b200 import _lib
    lib = _lib.lib()
    ws_n = lib.ipr_prune_workspace_bytes(3802816)
    assert ws_n >= 3802816 // 1024 * 12 and lib.ipr_prune_workspace_bytes(0) == 0
    f = lib.ipr_prune_magnitude_f32
    p, ws = ctypes.c_void_p(4096), ctypes.c_void_p(1 << 20)
    assert f(None, p, 5, 100, 10, ws, ws_n, None) == -1
    assert f(p, None, 5, 100, 10, ws, ws_n, None) == -1
    assert f(p, p, 5, 100, 10, None, ws_n, None) == -1
    assert f(p, p, 0, 100, 10, ws, ws_n, None) == -2                  # no segment
    assert f(p, p, 5, 0, 0, ws, ws_n, None) == -2                     # no entry
    assert f(p, p, 5, 100, 101, ws, ws_n, None) == -2                 # k > N
    assert f(p, p, 5, 100, -1, ws, ws_n, None) == -2
    assert f(p, p, 257, 100, 10, ws, ws_n, None) == -3                # more segments than the kernels stage
    assert f(p, p, 5, 100, 10, ws, lib.ipr_prune_workspace_bytes(100) - 1, None) == -5
    assert f(p, p, 5, 100, 10, ctypes.c_void_p((1 << 20) + 16), ws_n, None) == -4
    assert f(p, ctypes.c_void_p(4100), 5, 100, 10, ws, ws_n, None) == -4
    assert f(p, p, 5, 100, 0, ws, ws_n, None) == 0                    # k = 0: nothing to do, no launch
    g = lib.ipr_negate_indexed_f32
    assert g(p, p, 0, None) == 0 and g(None, None, 0, None) == 0
    assert g(None, p, 4, None) == -1 and g(p, None, 4, None) == -1 and g(p, p, -1, None) == -2


def test_ops_refuse_cpu_tensors():
    from ipr_gan_b200 import ops
    with pytest.raises(ops.IprError):
        ops.prune_magnitude_(torch.zeros(16), torch.zeros(1, 2, dtype=torch.int64), 16, 4)
    with pytest.raises(ops.IprError):
        ops.negate_indexed_(torch.zeros(16), torch.zeros(2, dtype=torch.int64))


# ---------------------------------------------------------------------------------------------- segments
@pytest.mark.parametrize("name,n", [("G32", 3802816), ("G64", 6948544), ("SRResNet", 1542528), ("Resnet9", 11372928)])
def test_prunable_segments_cover_exactly_the_conv_linear_weights(name, n):
    from ipr_gan_b200 import flat, robustness
    torch.manual_seed(0)
    net = _nets()[name]()
    segs = robustness.prunable_segments(net)
    arena = flat.module_arena(net)
    weights = [m.weight for m in net.modules() if isinstance(m, (nn.Conv2d, nn.ConvTranspose2d, nn.Linear))]
    assert segs == sorted((arena.offset_of(w), w.numel()) for w in weights)
    assert sum(c for _, c in segs) == n
    covered = np.zeros(arena.numel, dtype=bool)
    for o, c in segs:
        assert not covered[o:o + c].any()
        covered[o:o + c] = True
    others = [p for p in net.parameters() if all(p is not w for w in weights)]
    assert others                                         # biases, BatchNorm / InstanceNorm gammas and betas, PReLU
    for p in others:
        o = arena.offset_of(p)
        assert not covered[o:o + p.numel()].any()
    assert covered.sum() == n                            # so no alignment padding either


def test_generator32_count_matches_the_parameter_budget():
    """3 811 904 parameters minus the fc bias (8 192) and the BatchNorm gammas / betas (896)."""
    net = _nets()["G32"]()
    from ipr_gan_b200 import robustness
    assert sum(p.numel() for p in net.parameters()) == 3811904
    assert sum(c for _, c in robustness.prunable_segments(net)) == 3811904 - 8192 - 896


def test_cyclegan_segments_are_gb_only_in_the_shared_arena():
    """optG's arena spans GA and GB (models/cyclegan.py): only the target's tensors are listed."""
    from ipr_gan_b200 import flat, robustness
    ga, gb = _nets()["Resnet9"](), _nets()["Resnet9"]()
    arena = flat.arena_for(list(ga.parameters()) + list(gb.parameters()))
    segs = robustness.prunable_segments(gb)
    assert flat.module_arena(gb) is arena
    ga_end = max(arena.offset_of(p) + p.numel() for p in ga.parameters())
    assert all(o >= ga_end for o, _ in segs)
    assert sum(c for _, c in segs) == 11372928


def test_non_generator_is_refused():
    from ipr_gan_b200 import robustness
    import networks
    with pytest.raises(TypeError):
        robustness.prunable_segments(networks.SNDiscriminator32())


def test_prune_count_follows_torch():
    from ipr_gan_b200 import robustness
    for n in (1, 7, 10, 3802816, 11372928):
        for a in (0.0, 0.1, 0.25, 0.5, 0.35, 0.9, 1.0, 0, 1, n):
            assert robustness.prune_count(a, n) == tprune._compute_nparams_toprune(a, n)
    for bad in (-0.1, 1.5):
        with pytest.raises(ValueError):
            robustness.prune_count(bad, 10)
    with pytest.raises(ValueError):
        robustness.prune_count(11, 10)
    with pytest.raises(TypeError):
        robustness.prune_count("0.5", 10)


# ---------------------------------------------------------------------------------------------- the contract
def _layers(seed):
    torch.manual_seed(seed)
    mods = [nn.Linear(40, 96), nn.Conv2d(8, 16, 3), nn.ConvTranspose2d(16, 5, 4), nn.Linear(7, 3)]
    return mods


def test_emulation_equals_global_unstructured_without_ties():
    from ipr_gan_b200 import flat
    mods = _layers(1)
    arena = flat.arena_for([p for m in mods for p in m.parameters()])      # biases in the arena, not in the segments
    weights = [m.weight for m in mods]
    segs = [(arena.offset_of(w), w.numel()) for w in weights]
    n = sum(c for _, c in segs)
    gen = torch.Generator().manual_seed(2)
    distinct = (torch.randperm(n, generator=gen) + 1).float() * 1e-4 * (torch.randint(0, 2, (n,), generator=gen) * 2 - 1)
    with torch.no_grad():                                                  # distinct magnitudes, random signs
        for (o, c) in segs:
            arena.param[o:o + c] = distinct[:c]
            distinct = distinct[c:]
    base = arena.param.detach().numpy().copy()
    w = base[prune_ref.segment_index(segs)]
    assert np.unique(np.abs(w)).size == w.size                            # tie-free
    n = w.size
    for amount in (0.0, 0.1, 0.37, 0.5, 0.9, 1.0):
        k = tprune._compute_nparams_toprune(amount, n)
        got = prune_ref.prune_emulate(base, segs, k)
        clones = [nn.Module() for _ in weights]
        for c, wt in zip(clones, weights):
            c.weight = nn.Parameter(wt.detach().clone())
        tprune.global_unstructured([(c, "weight") for c in clones], pruning_method=tprune.L1Unstructured, amount=amount)
        want = base.copy()
        for c, (o, cnt) in zip(clones, segs):
            want[o:o + cnt] = c.weight.detach().reshape(-1).numpy()
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), amount
        assert int((prune_ref.prune_mask(w, k)).sum()) == k


def _tie_heavy(seed, n=6000):
    rng = np.random.default_rng(seed)
    vals = np.array([0.0, -0.0, 0.5, -0.5, 1.0, -1.0, 2.0, np.inf, -np.inf, np.nan, 1e-30, -1e-30], dtype=np.float32)
    arena = vals[rng.integers(0, vals.size, n)]
    arena[rng.integers(0, n, 40)] = rng.standard_normal(40).astype(np.float32)
    nan2 = np.array([0x7fc00001, 0xffc00000, 0x7f800001], dtype=np.uint32).view(np.float32)   # other NaN payloads
    arena[rng.integers(0, n, 3)] = nan2
    segs = [(0, 37), (40, 1000), (1044, 3), (1048, 2500), (3600, 2400)]     # gaps between the segments
    return arena, segs


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_emulation_on_tie_heavy_arenas(seed):
    arena, segs = _tie_heavy(seed)
    idx = prune_ref.segment_index(segs)
    outside = np.setdiff1d(np.arange(arena.size), idx)
    n = idx.size
    keys = prune_ref.magnitude_keys(arena[idx])
    order = np.argsort(keys, kind="stable")                 # smallest key first, lowest index first among ties
    for k in sorted({0, 1, 2, 37, n // 3, n // 2, n - 4, n - 1, n} | set(range(0, n, 397))):
        got = prune_ref.prune_emulate(arena, segs, k)
        m = prune_ref.prune_mask(arena[idx], k)
        assert int(m.sum()) == k
        want_m = np.zeros(n, dtype=bool)
        want_m[order[:k]] = True
        assert np.array_equal(m, want_m), k
        assert np.array_equal(got[outside].view(np.uint32), arena[outside].view(np.uint32))
        w = arena[idx]
        with np.errstate(invalid="ignore"):
            want = np.where(m, w * np.float32(0), w)
        assert np.array_equal(got[idx].view(np.uint32), want.view(np.uint32))
        neg = m & (w < 0) & np.isfinite(w)
        assert np.all(np.signbit(got[idx][neg])) and np.all(got[idx][neg] == 0)        # -w * 0 = -0.0
        if k == n:
            assert np.all((got[idx] == 0) | np.isnan(got[idx]))                          # inf * 0 and NaN * 0: NaN
        if k == 0:
            assert np.array_equal(got.view(np.uint32), arena.view(np.uint32))
    # +-0 share the key 0 and every NaN payload sits above +inf
    assert prune_ref.magnitude_keys(np.float32([-0.0]))[0] == prune_ref.magnitude_keys(np.float32([0.0]))[0] == 0
    nan_keys = prune_ref.magnitude_keys(np.array([0x7fc00001, 0xffc00000, 0x7f800001], dtype=np.uint32).view(np.float32))
    assert np.all(nan_keys == 0x7fffffff) and np.all(nan_keys > prune_ref.magnitude_keys(np.float32([np.inf])))


# ---------------------------------------------------------------------------------------------- sign flip draw
@pytest.mark.parametrize("name,n", [("G32", 448), ("SRResNet", 2112), ("Resnet9", 5248)])
def test_sign_flip_draw(name, n):
    from ipr_gan_b200 import flat, robustness
    net = _nets()[name]()
    arena = flat.module_arena(net)
    gammas = [m.weight for m in net.modules() if isinstance(m, (nn.BatchNorm2d, nn.InstanceNorm2d))]
    assert sum(g.numel() for g in gammas) == n
    gamma_offsets = np.concatenate([np.arange(g.numel()) + arena.offset_of(g) for g in gammas])
    for p in (10, 25, 50, 100):
        off = robustness.sign_flip_offsets(net, p, torch.Generator().manual_seed(5))
        assert off.dtype == torch.int64 and off.numel() == int(n * p / 100)
        perm = torch.randperm(n, generator=torch.Generator().manual_seed(5))
        assert np.array_equal(off.numpy(), gamma_offsets[perm[:int(n * p / 100)].numpy()])
        assert np.unique(off.numpy()).size == off.numel() and np.isin(off.numpy(), gamma_offsets).all()
    assert set(robustness.sign_flip_offsets(net, 100, torch.Generator().manual_seed(1)).tolist()) == set(gamma_offsets.tolist())
    assert robustness.sign_flip_offsets(net, 10, torch.Generator().manual_seed(0)).numel() == int(n * 10 / 100)


# ---------------------------------------------------------------------------------------------- refusal
@pytest.mark.parametrize("name", ["G32", "SRResNet"])
def test_torch_pruned_network_is_refused(name):
    from ipr_gan_b200 import engine, ops
    import networks
    net = _nets()[name]()
    engine.refuse_pruned(net)                                  # a clean network passes (and its dicts are cached)
    conv = next(m for m in net.modules() if isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)))
    tprune.l1_unstructured(conv, "weight", amount=0.3)
    with pytest.raises(ops.IprError, match="robustness.prune_"):
        engine.refuse_pruned(net)
    tprune.remove(conv, "weight")
    engine.refuse_pruned(net)
    engine.refuse_pruned(networks.SNDiscriminator32())         # spectral norm's weight_orig has no mask: not pruning


def test_segments_follow_a_new_arena():
    """The cached segment list of a network is rebuilt when an optimizer re-lays its parameters into a shared arena."""
    from ipr_gan_b200 import flat, robustness
    ga, gb = _nets()["Resnet9"](), _nets()["Resnet9"]()
    alone = robustness.prunable_segments(gb)
    shared = flat.arena_for(list(ga.parameters()) + list(gb.parameters()))
    again = robustness.prunable_segments(gb)
    assert again != alone and again == sorted((shared.offset_of(m.weight), m.weight.numel()) for m in gb.modules()
                                              if isinstance(m, (nn.Conv2d, nn.ConvTranspose2d, nn.Linear)))
