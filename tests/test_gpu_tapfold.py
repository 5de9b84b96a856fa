"""GPU: the one-launch 3-channel layer (csrc/tapfold.cu) is bit-identical to the tap GEMM + col2im3 path it replaces,
both as a kernel and inside the protected training step (IPR_NO_TAPFOLD=1 selects the two-launch path)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _two_launch(a, pack, tanh_out, sigma=None):
    from ipr_gan_b200 import dense, engine
    plan = dense.Plan("linear", 64, 32)
    t9, _ = plan.run(a, pack, epi=dense.EPI_LINEAR_F32, sigma=sigma, n_valid=32)
    return engine.col2im3(t9, tanh_out)


@pytest.mark.parametrize("B", [1, 5, 64, 512])
@pytest.mark.parametrize("tanh_out,with_sigma", [(True, False), (False, True), (False, False), (True, True)])
def test_tapfold_equals_gemm_plus_col2im3(B, tanh_out, with_sigma):
    from ipr_gan_b200 import engine
    torch.manual_seed(B)
    a = torch.randn(B, 32, 32, 64, device="cuda").to(torch.bfloat16)
    w = torch.randn(64, 3, 3, 3, device="cuda") * 0.1
    pack = engine._tap27_rows_layout(w).to(torch.bfloat16)
    sigma = torch.tensor([2.37], device="cuda") if with_sigma else None
    got = engine.tapfold3(a, pack, tanh_out, sigma=sigma)
    assert got is not None and got.shape == (B, 3, 32, 32)
    want = _two_launch(a, pack, tanh_out, sigma)
    assert torch.equal(got, want)


@pytest.mark.parametrize("H,W", [(16, 16), (8, 128), (64, 16)])
def test_tapfold_other_supported_shapes(H, W):
    from ipr_gan_b200 import engine
    torch.manual_seed(H * W)
    a = torch.randn(7, H, W, 64, device="cuda").to(torch.bfloat16)
    pack = engine._tap27_rows_layout(torch.randn(64, 3, 3, 3, device="cuda") * 0.1).to(torch.bfloat16)
    got = engine.tapfold3(a, pack, True)
    assert got is not None
    assert torch.equal(got, _two_launch(a, pack, True))


def test_tapfold_unsupported_shape_returns_none():
    from ipr_gan_b200 import engine
    a = torch.zeros(2, 64, 64, 64, device="cuda", dtype=torch.bfloat16)        # 4096 pixels: more than one CTA holds
    pack = torch.zeros(1, 32, 64, device="cuda", dtype=torch.bfloat16)
    assert engine.tapfold3(a, pack, True) is None


@pytest.mark.parametrize("B,use_graph", [(64, False), (64, True), (512, True)])
def test_protected_step_identical_with_and_without_tapfold(monkeypatch, B, use_graph):
    from ipr_gan_b200.trainer import ProtectedDCGANTrainer
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(B)
    warm = (torch.randn(B, 3, 32, 32, generator=g).clamp(-1, 1), torch.randn(B, 128, generator=g))
    batches = [(torch.randn(B, 3, 32, 32, generator=g).clamp(-1, 1), torch.randn(B, 128, generator=g)) for _ in range(3)]

    def run(off):
        monkeypatch.setenv("IPR_NO_TAPFOLD", "1" if off else "0")
        tr = ProtectedDCGANTrainer(B, dev, use_graph=use_graph)
        tr.set_inputs(*warm)
        tr.capture(warmup=3)
        out = [tr.step_from_host(real, z) for real, z in batches]
        torch.cuda.synchronize()
        params = [p.detach().clone() for p in list(tr.model.G.parameters()) + list(tr.model.D.parameters())]
        bufs = [b.detach().clone() for b in list(tr.model.G.buffers()) + list(tr.model.D.buffers())]
        return out, params, bufs

    m0, p0, b0 = run(True)
    m1, p1, b1 = run(False)
    assert m0 == m1, (m0, m1)
    assert all(torch.equal(x, y) for x, y in zip(p0, p1))
    assert all(torch.equal(x, y) for x, y in zip(b0, b1))
