"""GPU: the banded one-launch 3-channel layer (csrc/tapfold.cu, ipr_tapfold3_band_f32) is bit-identical to the tap
GEMM + col2im3 path it replaces at 64 x 64 and at shapes with a partial last band, an uneven band count and W = 128,
and to the whole-image kernel where that one covers the shape."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _two_launch(a, pack, tanh_out, sigma=None):
    from ipr_gan_b200 import dense, engine
    plan = dense.Plan("linear", 64, 32)
    t9, _ = plan.run(a, pack, epi=dense.EPI_LINEAR_F32, sigma=sigma, n_valid=32)
    return engine.col2im3(t9, tanh_out)


def _inputs(B, H, W, seed):
    from ipr_gan_b200 import engine
    torch.manual_seed(seed)
    a = torch.randn(B, H, W, 64, device="cuda").to(torch.bfloat16)
    pack = engine._tap27_rows_layout(torch.randn(64, 3, 3, 3, device="cuda") * 0.1).to(torch.bfloat16)
    return a, pack


@pytest.mark.parametrize("B", [1, 5, 64, 512])
@pytest.mark.parametrize("tanh_out,with_sigma", [(True, False), (False, True), (False, False), (True, True)])
def test_band_fold_equals_gemm_plus_col2im3_64(B, tanh_out, with_sigma):
    from ipr_gan_b200 import engine
    a, pack = _inputs(B, 64, 64, B)
    sigma = torch.tensor([2.37], device="cuda") if with_sigma else None
    got = engine.tapfold3_band(a, pack, tanh_out, sigma=sigma)
    assert got is not None and got.shape == (B, 3, 64, 64)
    assert torch.equal(got, _two_launch(a, pack, tanh_out, sigma))


@pytest.mark.parametrize("B,H,W", [
    (7, 48, 64),        # 12-row bands: 4 an image, no partial band
    (9, 40, 32),        # 24-row bands: a partial last band of 16 rows
    (3, 128, 128),      # W = 128: 6-row bands, 22 an image (the last has 2 rows)
    (64, 64, 64),       # 6 bands an image (the last has 4 rows)
])
def test_band_fold_other_shapes(B, H, W):
    from ipr_gan_b200 import engine
    a, pack = _inputs(B, H, W, H * W + B)
    sigma = torch.tensor([0.73], device="cuda")
    for tanh_out, s in ((True, None), (False, sigma)):
        got = engine.tapfold3_band(a, pack, tanh_out, sigma=s)
        assert got is not None and got.shape == (B, 3, H, W)
        assert torch.equal(got, _two_launch(a, pack, tanh_out, s))


@pytest.mark.parametrize("B", [1, 64, 300])
def test_band_fold_equals_whole_image_fold_32(B):
    """At 32 x 32 the banded kernel folds two bands (24 + 8 rows) where the whole-image kernel folds the image."""
    from ipr_gan_b200 import engine
    a, pack = _inputs(B, 32, 32, 100 + B)
    got = engine.tapfold3_band(a, pack, True)
    whole = engine.tapfold3(a, pack, True)
    assert got is not None and whole is not None
    assert torch.equal(got, whole)
    assert torch.equal(got, _two_launch(a, pack, True))


def test_generator_and_discriminator_use_the_band_fold(monkeypatch):
    """At 64 x 64, G's last layer and D's input gradient run through the banded kernel (the whole-image one declines)."""
    import networks
    from ipr_gan_b200 import engine
    calls = []
    band = engine.tapfold3_band

    def counted(*args, **kw):
        out = band(*args, **kw)
        calls.append(out is not None)
        return out
    monkeypatch.setattr(engine, "tapfold3_band", counted)
    torch.manual_seed(0)
    G, D = networks.ConvGenerator64().cuda(), networks.SNDiscriminator64().cuda()
    x = G(torch.randn(4, 128, device="cuda"))
    D(x).sum().backward()
    torch.cuda.synchronize()
    assert x.shape == (4, 3, 64, 64) and calls == [True, True]
