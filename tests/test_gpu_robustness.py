"""GPU: the robustness attacks on the device -- global magnitude pruning (csrc/prune.cu) against its NumPy contract
and torch.nn.utils.prune, graph capture, the prune / sign-flip sweeps against plain sweeps of a model whose weights
were perturbed with stock torch ops and loaded with load_state_dict, restoration after a sweep, the refusal of
torch.nn.utils.prune modules, and a two-rank sweep against one rank."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch
import torch.nn as nn
import torch.nn.utils.prune as tprune

from tests import prune_ref

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
AMOUNTS = (0.0, 0.1, 0.5, 0.9, 1.0)
_PRUNABLE = (nn.Conv2d, nn.ConvTranspose2d, nn.Linear)


def _net(name, dev):
    """The generator to prune and its arena; Resnet9 GB shares one arena with a GA, as under CycleGAN's optG."""
    import networks
    from ipr_gan_b200 import flat
    torch.manual_seed(11)
    if name == "Resnet9 GB":
        ga, gb = networks.Resnet9Blocks().to(dev), networks.Resnet9Blocks().to(dev)
        return gb, flat.arena_for(list(ga.parameters()) + list(gb.parameters()))
    net = {"G32": networks.ConvGenerator32, "G64": networks.ConvGenerator64, "SRResNet": networks.SRResNet}[name]()
    net = net.to(dev)
    return net, flat.module_arena(net)


@pytest.mark.parametrize("name", ["G32", "G64", "SRResNet", "Resnet9 GB"])
def test_prune_kernel_against_contract_and_torch(name):
    from ipr_gan_b200 import robustness
    dev = torch.device("cuda", 0)
    net, arena = _net(name, dev)
    segs = robustness.prunable_segments(net)
    idx = prune_ref.segment_index(segs)
    outside = np.setdiff1d(np.arange(arena.numel), idx)
    base = arena.param.clone()
    base_np = base.cpu().numpy()
    keys = prune_ref.magnitude_keys(base_np[idx])
    weights = [m.weight for m in net.modules() if isinstance(m, _PRUNABLE)]
    for amount in AMOUNTS:
        arena.param.copy_(base)
        k = robustness.prune_(net, amount)
        assert k == tprune._compute_nparams_toprune(amount, idx.size)
        got = arena.param.cpu().numpy()
        want = prune_ref.prune_emulate(base_np, segs, k)
        assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), amount          # the contract, bit for bit
        assert np.array_equal(got[outside].view(np.uint32), base_np[outside].view(np.uint32))
        # torch.nn.utils.prune on GPU copies of the same weights: weight_orig * weight_mask
        clones = []
        for w in weights:
            c = nn.Module()
            c.weight = nn.Parameter(base[arena.offset_of(w):arena.offset_of(w) + w.numel()].view(w.shape).clone())
            clones.append(c)
        tprune.global_unstructured([(c, "weight") for c in clones], pruning_method=tprune.L1Unstructured, amount=amount)
        ref = base_np.copy()
        for c, w in zip(clones, weights):
            o = arena.offset_of(w)
            ref[o:o + w.numel()] = c.weight.detach().reshape(-1).cpu().numpy()
        differ = np.flatnonzero(got.view(np.uint32) != ref.view(np.uint32))
        if k:
            T, _ = prune_ref.radix_threshold(keys, k)
            pos = np.searchsorted(idx, differ)                                  # idx ascends: segments ascend
            assert np.array_equal(idx[np.minimum(pos, idx.size - 1)], differ)
            assert np.all(keys[pos] == T), amount                               # only ties at the threshold differ
        torch_zeroed = int(sum((c.weight_mask == 0).sum().item() for c in clones))
        assert torch_zeroed == k
        mask = prune_ref.prune_mask(base_np[idx], k)
        assert int(mask.sum()) == k
    arena.param.copy_(base)


def test_prune_graph_equals_eager():
    from ipr_gan_b200 import robustness
    dev = torch.device("cuda", 0)
    net, arena = _net("SRResNet", dev)
    base = arena.param.clone()
    robustness.prune_(net, 0.5)                          # eager first: the segment table goes to the device
    eager = arena.param.clone()
    arena.param.copy_(base)
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    g = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(g, stream=s):
            robustness.prune_(net, 0.5)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(2):
        arena.param.copy_(base)
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(arena.param.view(torch.int32), eager.view(torch.int32))
    arena.param.copy_(base)


def test_negate_indexed():
    from ipr_gan_b200 import ops
    x = torch.randn(1000, device="cuda")
    x[3] = 0.0
    idx = torch.tensor([3, 5, 999, 0], dtype=torch.int64)
    want = x.clone()
    want[idx] = -want[idx]
    ops.negate_indexed_(x, idx.cuda())
    assert torch.equal(x.view(torch.int32), want.view(torch.int32))


# ---------------------------------------------------------------------------------------------- sweeps
def _dcgan(dev):
    import models
    from configs import presets
    torch.manual_seed(3)
    m = models.DCGAN(presets.dcgan_model(), device=[dev])
    m = models.BlackBoxWrapper(m, presets.dcgan_blackbox())
    return models.WhiteBoxWrapper(m, presets.dcgan_whitebox())


def _srgan(dev):
    import models
    from configs import presets
    os.environ["IPR_VGG_RANDOM_INIT"] = "1"
    torch.manual_seed(4)
    m = models.SRGAN(presets.srgan_model(), device=[dev])
    m = models.BlackBoxWrapper(m, presets.srgan_blackbox())
    return models.WhiteBoxWrapper(m, presets.whitebox("G"))


def _cyclegan(dev):
    import models
    from configs import presets
    torch.manual_seed(5)
    m = models.CycleGAN(presets.cyclegan_model(), device=[dev])
    m = models.BlackBoxWrapper(m, presets.cyclegan_blackbox())
    return models.WhiteBoxWrapper(m, presets.whitebox("GB"))


_FAMILIES = {"dcgan": (_dcgan, 448), "srgan": (_srgan, 2112), "cyclegan": (_cyclegan, 5248)}


def _sweep_args(family):
    if family == "dcgan":
        return {"n_samples": 48, "batch": 24}
    shape = (6, 3, 24, 24) if family == "srgan" else (3, 3, 256, 256)
    inputs = torch.rand(*shape, generator=torch.Generator().manual_seed(9))
    return {"inputs": inputs if family == "srgan" else inputs * 2 - 1, "batch": 2}


def _plain_sweep(model, args):
    from ipr_gan_b200 import verify
    import networks
    target = getattr(model, model.config.target)
    fn = verify.verification_sweep if isinstance(target.module, networks.ConvGenerator) else \
        verify.image_verification_sweep
    return fn(target, model.fn_inp, model.fn_out, sign_model=model.loss_model, **args)


def _torch_pruned_state(net, amount):
    """The target's state_dict with its conv / linear weights pruned by stock torch ops: a stable sort of |w| over all
    of them, the first round(amount * N) multiplied by 0 (lowest index first among equal magnitudes)."""
    sd = {k: v.clone() for k, v in net.state_dict().items()}
    names = [n + ".weight" for n, m in net.named_modules() if isinstance(m, _PRUNABLE)]
    from ipr_gan_b200 import flat
    arena = flat.module_arena(net)
    params = dict(net.named_parameters())
    names.sort(key=lambda n: arena.offset_of(params[n]))                 # arena order
    flat_w = torch.cat([sd[n].reshape(-1) for n in names])
    k = tprune._compute_nparams_toprune(amount, flat_w.numel())
    order = torch.sort(flat_w.abs(), stable=True).indices[:k]
    mask = torch.ones_like(flat_w)
    mask[order] = 0
    flat_w = flat_w * mask
    o = 0
    for n in names:
        c = sd[n].numel()
        sd[n] = flat_w[o:o + c].view_as(sd[n])
        o += c
    return sd


def _torch_flipped_states(model, percent, seed):
    gen = torch.Generator().manual_seed(seed)
    out = {}
    for name, g in model._modules.items():
        if not name.startswith("G"):
            continue
        net = g.module
        sd = {k: v.clone() for k, v in net.state_dict().items()}
        keys = [n + ".weight" for n, m in net.named_modules() if isinstance(m, (nn.BatchNorm2d, nn.InstanceNorm2d))]
        flat_g = torch.cat([sd[k].reshape(-1) for k in keys])
        n = flat_g.numel()
        sel = torch.randperm(n, generator=gen)[:int(n * percent / 100)]
        flat_g[sel.to(flat_g.device)] *= -1
        o = 0
        for k in keys:
            c = sd[k].numel()
            sd[k] = flat_g[o:o + c].view_as(sd[k])
            o += c
        out[name] = sd
    return out


def _same(a, b):
    for k in ("Q_WM", "P", "MATCH", "N", "WBOX_counts"):
        assert a[k] == b[k], (k, a[k], b[k])


@pytest.mark.parametrize("family", ["dcgan", "srgan", "cyclegan"])
def test_sweeps_equal_plain_sweeps_of_torch_perturbed_models(family):
    from ipr_gan_b200 import robustness
    dev = torch.device("cuda", 0)
    build, n_gamma = _FAMILIES[family]
    model = build(dev)
    fresh = build(dev)
    fresh.load_state_dict(model.state_dict())
    args = _sweep_args(family)
    target = getattr(model, model.config.target)
    net = target.module
    from ipr_gan_b200 import flat
    arena = flat.module_arena(net)
    before = arena.param.clone()
    bn = {k: v.clone() for k, v in net.state_dict().items() if "running" in k or "num_batches" in k}
    x_in = torch.randn(4, 128, device=dev) if family == "dcgan" else args["inputs"][:2].to(dev)
    target.eval()
    with torch.no_grad():
        out_before = target(x_in).clone()
    target.train()

    plain = _plain_sweep(model, args)
    amounts = (0.0, 0.5, 0.9)
    rows = robustness.prune_sweep(model, amounts, **args)
    _same(rows[0], plain)                                                       # level 0 = unperturbed sweep
    ftarget = getattr(fresh, fresh.config.target)
    for row, amount in zip(rows, amounts):
        assert row["amount"] == amount
        ftarget.module.load_state_dict(_torch_pruned_state(net, amount))
        _same(row, _plain_sweep(fresh, args))
        assert row["pruned"] == tprune._compute_nparams_toprune(amount, sum(
            c for _, c in robustness.prunable_segments(net)))

    percents = (10, 100)
    rows = robustness.sign_flip_sweep(model, percents, seed=7, **args)
    for row, p in zip(rows, percents):
        states = _torch_flipped_states(model, p, 7)
        for name, sd in states.items():
            getattr(fresh, name).module.load_state_dict(sd)
        _same(row, _plain_sweep(fresh, args))
        assert row["WBOX_counts"] == (int(n_gamma * p / 100), n_gamma)
        assert row["flipped"] == len(states) * int(n_gamma * p / 100)
    assert rows[-1]["WBOX"] == 1.0

    # the model leaves the sweeps as it entered them
    assert torch.equal(arena.param.view(torch.int32), before.view(torch.int32))
    for k, v in net.state_dict().items():
        if k in bn:
            assert torch.equal(v, bn[k]), k
    assert target.training and all(m.training for m in net.modules())
    target.eval()
    with torch.no_grad():
        assert torch.equal(target(x_in).view(torch.int32), out_before.view(torch.int32))
    target.train()
    _same(_plain_sweep(model, args), plain)


@pytest.mark.parametrize("name", ["G32", "SRResNet"])
def test_torch_pruned_generator_raises_on_forward(name):
    from ipr_gan_b200 import ops
    dev = torch.device("cuda", 0)
    net, _ = _net(name, dev)
    x = torch.randn(2, 128, device=dev) if name == "G32" else torch.rand(2, 3, 24, 24, device=dev)
    with torch.no_grad():
        net(x)                                                  # plans built before pruning: would run unpruned
    conv = next(m for m in net.modules() if isinstance(m, _PRUNABLE))
    tprune.l1_unstructured(conv, "weight", amount=0.5)
    with pytest.raises(ops.IprError, match="robustness.prune_"):
        with torch.no_grad():
            net(x)


def test_two_rank_sweep_equals_one_rank():
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from ipr_gan_b200 import robustness
    model = _srgan(torch.device("cuda", 0))
    inputs = torch.rand(13, 3, 24, 24, generator=torch.Generator().manual_seed(11))
    one = robustness.prune_sweep(model, (0.0, 0.5), inputs=inputs, batch=4)
    port = 29500 + (os.getpid() % 400) + 3
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "robustness_worker.py")]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    lines = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
    assert r.returncode == 0 and lines, r.stdout[-3000:] + r.stderr[-3000:]
    two = json.loads(lines[-1][7:])
    assert len(two) == len(one)
    for a, b in zip(one, two):
        assert a["N"] == b["N"] == 13 and a["MATCH"] == b["MATCH"] and a["pruned"] == b["pruned"]
        assert list(a["WBOX_counts"]) == list(b["WBOX_counts"])
        assert abs(a["P"] - b["P"]) <= 1e-12 * max(1.0, abs(a["P"]))
        assert abs(a["Q_WM"] - b["Q_WM"]) <= 1e-12 * max(1.0, abs(a["Q_WM"]))
