"""GPU: the re-training attacks (robustness.finetune_attack / overwrite_attack) on the three protected families --
captured replays against the eager step, fine-tuning against plain training of the inner model, the first row
against a plain verification sweep, current weights in eager forwards after replays, the overwritten signature and
checkpoint keys, and the re-capture of a trainer's step when its learning rate changes."""
import pytest
import torch

pytestmark = pytest.mark.gpu
KINDS = ("dcgan", "srgan", "cyclegan")
ATTACKER = "OVERWRITTEN"


@pytest.fixture(scope="module")
def attacker_mark(tmp_path_factory):
    """The attacker's watermark: the project's synthetic mark, mirrored."""
    from PIL import Image
    from ipr_gan_b200.assets import make_watermark
    path = str(tmp_path_factory.mktemp("mark") / "attacker.png")
    make_watermark.make().transpose(Image.Transpose.FLIP_LEFT_RIGHT).save(path)
    return path


def _trainer(kind, use_graph):
    """A trainer of the family after two protected steps (its Adam state, statistics and pools are non-trivial)."""
    from ipr_gan_b200 import trainer as T
    dev = torch.device("cuda", 0)
    tr = {"dcgan": lambda: T.ProtectedDCGANTrainer(16, dev, use_graph=use_graph),
          "srgan": lambda: T.ProtectedSRGANTrainer(2, dev, use_graph=use_graph),
          "cyclegan": lambda: T.ProtectedCycleGANTrainer(dev, 64, use_graph=use_graph)}[kind]()
    b = _batches(kind, 99)(0)
    static = {"dcgan": lambda: (tr.real, tr.latent), "srgan": lambda: (tr.low_res, tr.high_res),
              "cyclegan": lambda: (tr.real_A, tr.real_B)}[kind]()
    for dst, src in zip(static, b):
        dst.copy_(src)
    tr.capture(warmup=2)
    return tr


def _batches(kind, seed):
    def draw(i):
        g = torch.Generator().manual_seed(seed * 1000 + i)
        if kind == "dcgan":
            return torch.randn(16, 3, 32, 32, generator=g).clamp(-1, 1), torch.randn(16, 128, generator=g)
        if kind == "srgan":
            return torch.rand(2, 3, 24, 24, generator=g), torch.rand(2, 3, 96, 96, generator=g)
        return torch.rand(1, 3, 64, 64, generator=g) * 2 - 1, torch.rand(1, 3, 64, 64, generator=g) * 2 - 1
    return draw


def _sweep_args(kind):
    g = torch.Generator().manual_seed(7)
    if kind == "dcgan":
        return {"n_samples": 48, "batch": 16}
    if kind == "srgan":
        return {"inputs": torch.rand(3, 3, 24, 24, generator=g), "batch": 2}
    return {"inputs": torch.rand(3, 3, 64, 64, generator=g) * 2 - 1, "batch": 2}


def _attacker_cfgs(kind, mark):
    from configs import presets
    if kind == "dcgan":
        return presets.dcgan_blackbox(watermark=mark), presets.dcgan_whitebox(string=ATTACKER)
    if kind == "srgan":
        return presets.srgan_blackbox(watermark=mark), presets.whitebox("G", string=ATTACKER)
    return presets.cyclegan_blackbox(watermark=mark), presets.whitebox("GB", string=ATTACKER)


def _inner(model):
    from models.core import Wrapper
    while isinstance(model, Wrapper):
        model = model.model
    return model


def _nets(model):
    m = _inner(model)
    return [m.GA, m.GB, m.DA, m.DB] if hasattr(m, "GA") else [m.G, m.D]


def _state(model):
    """Every parameter and buffer of the trained networks and the Adam moments / step counters, as device copies."""
    m = _inner(model)
    out = [t.detach().clone() for n in _nets(model) for t in list(n.parameters()) + list(n.buffers())]
    for opt in (m.optG, m.optD):
        out += [opt._m.clone(), opt._v.clone(), opt._step.clone()]
    return out


def _attack(kind, which, use_graph, mark, steps=3, eval_every=2):
    tr = _trainer(kind, use_graph)
    torch.manual_seed(21)                  # the attacker's noise-patch trigger and CycleGAN's pool draws: alike in both arms
    from ipr_gan_b200 import robustness
    args = (_batches(kind, 5), steps, eval_every)
    if which == "finetune":
        rows = robustness.finetune_attack(tr, *args, **_sweep_args(kind))
    else:
        rows = robustness.overwrite_attack(tr, *_attacker_cfgs(kind, mark), *args, **_sweep_args(kind))
    torch.cuda.synchronize()
    return tr, rows


def _rows_close(ra, rb, tol):
    assert [r["step"] for r in ra] == [r["step"] for r in rb]
    for a, b in zip(ra, rb):
        assert a.keys() == b.keys()
        for who in a:
            if who == "step" or a[who] is None:
                assert a[who] == b[who]
                continue
            for k, v in a[who].items():
                w = b[who][k]
                if tol == 0 or not isinstance(v, float):
                    assert v == w, (a["step"], who, k, v, w)
                else:
                    assert abs(v - w) <= tol * max(1.0, abs(v)), (a["step"], who, k, v, w)


@pytest.mark.parametrize("which", ["finetune", "overwrite"])
@pytest.mark.parametrize("kind", KINDS)
def test_attack_graph_equals_eager(kind, which, attacker_mark):
    """The attack through captured replays against the same attack with use_graph=False: metrics, result rows, every
    parameter / buffer of G and D and the Adam moments.  DCGAN and CycleGAN run on this library alone and agree bit
    for bit.  SRGAN's content loss goes through the frozen PyTorch VGG, for which cuDNN picks its algorithms anew
    under capture: its trajectories separate in the last bits (the bound of test_gpu_srgan_cyclegan's replay test)."""
    det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        tr_e, rows_e = _attack(kind, which, False, attacker_mark)
        tr_g, rows_g = _attack(kind, which, True, attacker_mark)
    finally:
        torch.backends.cudnn.deterministic = det
    assert [r["step"] for r in rows_g] == [0, 2, 3] and rows_g[0]["metrics"] is None
    assert ("attacker" in rows_g[0]) == (which == "overwrite")
    tol, ptol = (5e-3, 1e-3) if kind == "srgan" else (0, 0)
    _rows_close(rows_e, rows_g, tol)
    for a, b in zip(_state(tr_e.model), _state(tr_g.model)):
        if ptol == 0:
            assert torch.equal(a, b), float((a - b).abs().max())
        else:
            assert float((a - b).abs().max()) <= ptol * max(1.0, float(a.abs().max()))


def _plain(kind, dev):
    import models
    from configs import presets
    if kind == "dcgan":
        return models.DCGAN(presets.dcgan_model(32), device=[dev])
    if kind == "srgan":
        return models.SRGAN(presets.srgan_model(), device=[dev])
    return models.CycleGAN(presets.cyclegan_model(), device=[dev])


def _plain_step(kind, m, batch, dev):
    a, b = (t.to(dev) for t in batch)
    if kind == "dcgan":
        m.update_d({"real_sample": a, "latent": b})
        m.update_g({"fake_sample": m.fake_sample})
    elif kind == "srgan":
        m.update_g({"low_res": a, "high_res": b, "pretrain": False})
        m.update_d({"high_res": m.high_res, "super_res": m.super_res})
    else:
        m.update_g({"real_A": a, "real_B": b})
        m.update_d({"real_A": m.real_A, "real_B": m.real_B, "fake_A": m.fake_A.detach(), "fake_B": m.fake_B.detach()})


def _keys_state(model):
    return [t.detach().clone() for part in (model.fn_inp, model.fn_out, model.loss_model)
            for t in part.state_dict().values()]


@pytest.mark.parametrize("kind", KINDS)
def test_finetune_equals_plain_training(kind):
    """Fine-tuning is the inner model's plain GAN step at lr x lr_scale: the unwrapped inner model, loaded with the
    same state and given the scaled rates explicitly, stepped on the same batches (CycleGAN: the host RNG seeded alike
    for the pools), ends bit-identical.  The first row equals a plain verification sweep of the untouched model, and
    the owner's key buffers leave the attack bit-identical.  DCGAN attacks through graph replays (bit-identical to its
    eager step); SRGAN and CycleGAN through their eager steps, so the comparison stays exact."""
    from ipr_gan_b200 import robustness, verify
    dev = torch.device("cuda", 0)
    det = torch.backends.cudnn.deterministic
    torch.backends.cudnn.deterministic = True
    try:
        tr = _trainer(kind, use_graph=(kind == "dcgan"))
        model = tr.model
        plain = _plain(kind, dev)
        plain.load_state_dict(model.state_dict())
        if kind == "srgan":
            plain.V.load_state_dict(_inner(model).V.state_dict())      # the frozen VGG is not in the checkpoint
        lrs = [0.1 * opt.param_groups[0]["lr"] for opt in (model.optG, model.optD)]
        for opt, lr in zip((plain.optG, plain.optD), lrs):
            opt.param_groups[0]["lr"] = lr
        args = _sweep_args(kind)
        target = getattr(model, model.config.target)
        fn = verify.verification_sweep if kind == "dcgan" else verify.image_verification_sweep
        sweep0 = fn(target, model.fn_inp, model.fn_out, sign_model=model.loss_model, **args)
        keys0 = _keys_state(model)
        draw = _batches(kind, 8)
        torch.manual_seed(33)
        rows = robustness.finetune_attack(tr, draw, 3, 3, **args)
        torch.manual_seed(33)
        for i in range(3):
            _plain_step(kind, plain, draw(i), dev)
        torch.cuda.synchronize()
    finally:
        torch.backends.cudnn.deterministic = det
    assert [opt.param_groups[0]["lr"] for opt in (model.optG, model.optD)] == lrs
    assert rows[0]["owner"] == {k: sweep0[k] for k in robustness._RESULT_KEYS}
    for a, b in zip(_state(model), _state(plain)):
        assert torch.equal(a, b), float((a - b).abs().max())
    assert all(torch.equal(a, b) for a, b in zip(keys0, _keys_state(model)))
    assert model is tr.model and tr.inhibit


@pytest.mark.parametrize("kind", KINDS)
def test_no_stale_weights_after_replays(kind):
    """After captured attack replays, the trainer's generator in an eager forward and in a sweep row computes what a
    fresh stack strict-loaded with the attacked state_dict computes (the replays bump the arenas' versions, so the
    eager forward re-packs its bf16 operands)."""
    from ipr_gan_b200 import robustness
    dev = torch.device("cuda", 0)
    tr = _trainer(kind, use_graph=True)
    args = _sweep_args(kind)
    rows = robustness.finetune_attack(tr, _batches(kind, 3), 3, 3, **args)
    fresh = _trainer(kind, use_graph=False)
    fresh.model.load_state_dict(tr.model.state_dict(), strict=True)
    name = tr.model.config.target
    g = torch.Generator().manual_seed(4)
    x = torch.randn(8, 128, generator=g) if kind == "dcgan" else args["inputs"][:2]
    outs = []
    for model in (tr.model, fresh.model):
        G = getattr(model, name)
        G.eval()
        with torch.no_grad():
            outs.append(G(x.to(dev)).clone())
        G.train()
    assert torch.equal(outs[0], outs[1]), float((outs[0] - outs[1]).abs().max())
    want = robustness._sweep(fresh.model, args)
    assert rows[-1]["owner"] == {k: want[k] for k in robustness._RESULT_KEYS}


@pytest.mark.parametrize("kind", KINDS)
def test_overwrite_signature_and_checkpoint(kind, attacker_mark):
    """Step 0 of an overwriting attack: the owner's WBOX_counts are exactly the signature positions where the two
    strings' bit streams disagree, the attacker's WBOX is 0.  Afterwards the checkpoint carries the attacker's fn_inp /
    fn_out / sign buffers and strict-loads into a fresh stack built with the attacker's configs."""
    import models
    from ipr_gan_b200 import robustness
    tr, rows = _attack(kind, "overwrite", True, attacker_mark, steps=2, eval_every=1)
    target = _inner(tr.model)
    name = tr.model.config.target
    widths = [g.numel() for g in robustness._signature_gammas(robustness._module(getattr(target, name)))]
    wrong = sum(robustness.sign_disagreements(widths, "EXAMPLE A", ATTACKER))
    assert wrong > 0
    assert rows[0]["owner"]["WBOX_counts"] == (wrong, sum(widths))
    assert rows[0]["attacker"]["WBOX"] == 0 and rows[0]["attacker"]["WBOX_counts"] == (0, sum(widths))
    assert [r["step"] for r in rows] == [0, 1, 2] and all(r["metrics"] is not None for r in rows[1:])
    sd = tr.model.state_dict()
    attacker = tr.model
    for key, part in (("fn_inp", attacker.fn_inp), ("fn_out", attacker.fn_out), ("sign", attacker.loss_model)):
        got = part.state_dict()
        assert sd[key].keys() == got.keys() and all(torch.equal(sd[key][k], got[k]) for k in got)
    assert any(not torch.equal(a, b) for a, b in zip(sd["sign"].values(), _owner_signs(kind)))
    bb, wb = _attacker_cfgs(kind, attacker_mark)
    fresh = models.WhiteBoxWrapper(models.BlackBoxWrapper(_plain(kind, torch.device("cuda", 0)), bb), wb)
    fresh.load_state_dict(sd, strict=True)
    for key in ("fn_inp", "fn_out", "sign"):
        f = fresh._modules[key].state_dict()
        assert all(torch.equal(f[k], sd[key][k]) for k in f)


def _owner_signs(kind):
    """The owner's sign buffers of a fresh trainer of the family (the signature string decides them)."""
    tr = _trainer(kind, use_graph=False)
    return list(tr.model.loss_model.state_dict().values())


@pytest.mark.parametrize("kind", KINDS)
def test_learning_rate_change_recaptures(kind):
    """The rate is a launch argument frozen into a captured step: after it changes the trainer captures anew.  At rate
    0 Adam leaves every parameter exactly where it is, which a replay of the old graph would not."""
    tr = _trainer(kind, use_graph=True)
    old = tr.graph if kind != "cyclegan" else tr.graph_g
    m = _inner(tr.model)
    for opt in (m.optG, m.optD):
        opt.param_groups[0]["lr"] = 0.0
    before = [p.detach().clone() for n in _nets(tr.model) for p in n.parameters()]
    tr.step_from_host(*_batches(kind, 6)(0))
    torch.cuda.synchronize()
    assert (tr.graph if kind != "cyclegan" else tr.graph_g) is not old
    after = [p.detach().clone() for n in _nets(tr.model) for p in n.parameters()]
    assert all(torch.equal(a, b) for a, b in zip(before, after))
