"""CPU: the 64 x 64 IPR-DCGAN configuration (the reference's CUB-200 configs: mg = md = 8, 32 x 32 watermark) --
the drop-in networks carry the reference's parameters and buffers, and the trainer takes the image and watermark
sizes while keeping its 32 x 32 defaults."""
import inspect

import torch


def _shapes(m):
    return [(k, tuple(v.shape)) for k, v in m.state_dict().items()]


def test_networks64_state_dict_matches_oracle():
    import networks
    from oracle import ipr_oracle as orc
    torch.manual_seed(0)
    G, D = networks.ConvGenerator64(), networks.SNDiscriminator64()
    Go, Do = orc.make_generator(8), orc.make_discriminator(8)
    assert _shapes(G) == _shapes(Go)
    assert _shapes(D) == _shapes(Do)
    assert G.mg == 8 and D.md == 8
    assert dict(_shapes(G))["fc.0.weight"] == (512 * 8 * 8, 128)
    # each side loads the other's state, values included
    Go.load_state_dict(G.state_dict())
    Do.load_state_dict(D.state_dict())
    torch.manual_seed(1)
    G2, D2 = networks.ConvGenerator64(), networks.SNDiscriminator64()
    G2.load_state_dict(Go.state_dict())
    D2.load_state_dict(Do.state_dict())
    for a, b in ((G, G2), (D, D2)):
        sa, sb = a.state_dict(), b.state_dict()
        assert all(torch.equal(sa[k], sb[k]) for k in sa)


def test_trainer_64x64_options_keep_32x32_defaults():
    from ipr_gan_b200.trainer import ProtectedDCGANTrainer
    params = inspect.signature(ProtectedDCGANTrainer).parameters
    assert params["size"].default == 32 and params["wm_size"].default == 16
