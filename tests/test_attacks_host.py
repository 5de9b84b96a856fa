"""CPU: host side of the re-training attacks (robustness.finetune_attack / overwrite_attack) -- argument refusals
that leave the model untouched, the verification schedule, and the count of signature positions on which two
signature strings disagree."""
import math
import types

import pytest
import torch


def _stack():
    """A protected DCGAN stack on the CPU, in a stand-in for a trainer (the refusals come before any step)."""
    import models
    from configs import presets
    torch.manual_seed(3)
    m = models.DCGAN(presets.dcgan_model(32), device=[torch.device("cpu")])
    m = models.BlackBoxWrapper(m, presets.dcgan_blackbox())
    m = models.WhiteBoxWrapper(m, presets.dcgan_whitebox())
    return types.SimpleNamespace(model=m, inhibit=False)


def _snapshot(tr):
    m = tr.model
    sd = {(k, n): t.clone() for k, part in m.state_dict().items() if k not in ("optG", "optD")
          for n, t in part.items()}
    lrs = (m.optG.param_groups[0]["lr"], m.optD.param_groups[0]["lr"])
    return m, dict(m._modules), sd, lrs, tr.inhibit


def _same(a, b):
    assert a[0] is b[0]
    assert a[1].keys() == b[1].keys() and all(a[1][k] is b[1][k] for k in a[1])
    assert a[2].keys() == b[2].keys() and all(torch.equal(a[2][k], b[2][k]) for k in a[2])
    assert a[3] == b[3] and a[4] == b[4]


def _batches(i):
    raise AssertionError("a refused attack must not ask for a batch")


@pytest.mark.parametrize("kw", [dict(steps=-1), dict(steps=2.0), dict(steps=True), dict(eval_every=0),
                                dict(eval_every=-3), dict(eval_every=1.5), dict(lr_scale=0.0), dict(lr_scale=-0.1),
                                dict(lr_scale=math.nan), dict(lr_scale=math.inf), dict(lr_scale="0.1")])
def test_refusals_leave_the_model_untouched(kw):
    from configs import presets
    from ipr_gan_b200 import robustness
    args = dict(steps=4, eval_every=2, lr_scale=0.1)
    args.update(kw)
    tr = _stack()
    before = _snapshot(tr)
    with pytest.raises(ValueError):
        robustness.finetune_attack(tr, _batches, args["steps"], args["eval_every"], lr_scale=args["lr_scale"],
                                   n_samples=8)
    _same(before, _snapshot(tr))
    with pytest.raises(ValueError):
        robustness.overwrite_attack(tr, presets.dcgan_blackbox(), presets.dcgan_whitebox(string="OTHER"), _batches,
                                    args["steps"], args["eval_every"], lr_scale=args["lr_scale"], n_samples=8)
    _same(before, _snapshot(tr))


def test_attacker_configs_must_target_the_protected_network():
    from configs import presets
    from ipr_gan_b200 import robustness
    tr = _stack()
    before = _snapshot(tr)
    for bb, wb in ((presets.cyclegan_blackbox(), presets.dcgan_whitebox(string="OTHER")),
                   (presets.dcgan_blackbox(), presets.whitebox("GB", string="OTHER"))):
        with pytest.raises(ValueError, match="target"):
            robustness.overwrite_attack(tr, bb, wb, _batches, 4, 2, n_samples=8)
        _same(before, _snapshot(tr))


@pytest.mark.parametrize("steps,k,want", [(0, 1, [0]), (0, 5, [0]), (1, 1, [0, 1]), (6, 2, [0, 2, 4, 6]),
                                          (7, 3, [0, 3, 6, 7]), (2, 5, [0, 2]), (5, 5, [0, 5]),
                                          (10, 4, [0, 4, 8, 10])])
def test_evaluation_schedule(steps, k, want):
    from ipr_gan_b200 import robustness
    assert robustness.attack_schedule(steps, k) == want


def test_sign_disagreements_hand_computed():
    """'EXAMPLE A' + TAB is an 80-bit period (SURVEY.md 8a A6); 'A' = 0x41 = 01000001 and 'B' = 0x42 = 01000010
    differ in the last two bits of character 8, stream bits 70 and 71 of every period.  'C' = 0x43 differs from 'A'
    in bit 70 only.  One stream runs across all layers."""
    from ipr_gan_b200 import robustness
    f = robustness.sign_disagreements
    assert f([80], "EXAMPLE A", "EXAMPLE A") == [0]
    assert f([80], "EXAMPLE A", "EXAMPLE B") == [2]
    assert f([70], "EXAMPLE A", "EXAMPLE B") == [0]
    assert f([71], "EXAMPLE A", "EXAMPLE B") == [1]
    assert f([64, 16, 160], "EXAMPLE A", "EXAMPLE B") == [0, 2, 4]
    assert f([71, 9], "EXAMPLE A", "EXAMPLE C") == [1, 0]
    # ConvGenerator32's BatchNorm widths: stream bits 0-255 (three periods + 16 bits), 256-383 (bits 310, 311), 384-447
    assert f([256, 128, 64], "EXAMPLE A", "EXAMPLE B") == [6, 2, 2]
    # a one-character string has a 16-bit period: 'A' (0x41), TAB against TAB, TAB
    assert f([16, 16], "A", "\t") == [bin(0x41 ^ 0x09).count("1")] * 2
    with pytest.raises(ValueError):
        f([8], None, "A")


def test_sign_disagreements_match_the_signs_the_stack_writes():
    """The helper against the sign buffers two SignLossModels write for the ConvGenerator32's three BatchNorms."""
    from configs import presets
    from ipr_gan_b200 import robustness
    from tools.signature import SignLossModel
    tr = _stack()
    G = tr.model.G
    widths = [m.weight.numel() for m in G.modules() if isinstance(m, torch.nn.BatchNorm2d)]
    owner = tr.model.loss_model
    other = SignLossModel(G, presets.dcgan_whitebox(string="ATTACKER'S OWN"))
    want = [int((getattr(owner, k) != getattr(other, k)).sum()) for k, _ in owner.named_buffers()]
    assert robustness.sign_disagreements(widths, "EXAMPLE A", "ATTACKER'S OWN") == want
    assert sum(want) > 0
