"""GPU: the 64 x 64 IPR-DCGAN (the reference's CUB-200 configs: ConvGenerator64 / SNDiscriminator64, mg = md = 8,
a 32 x 32 watermark) against the CPU oracle, with the method and tolerances of tests/test_gpu_dcgan.py: networks,
the protected step, graph replay, the banded 3-channel fold against the two-launch path, and the verification sweep."""
import copy

import numpy as np
import pytest
import torch

from tests.test_gpu_dcgan import GRAD_TOL, _nchw_masks, rel

pytestmark = pytest.mark.gpu

SIZE, WM = 64, 32


def _synth_step_inputs(batch, seed):
    """oracle.synth_step_inputs' recipe (SURVEY.md section 8d) at 64 x 64: real = randn.clamp(-1, 1), z = randn."""
    g = torch.Generator().manual_seed(seed)
    real = torch.randn(batch, 3, SIZE, SIZE, generator=g).clamp(-1, 1)
    return real, torch.randn(batch, 128, generator=g)


def _pair(seed=0):
    import networks
    from oracle import ipr_oracle as orc
    torch.manual_seed(seed)
    G, D = networks.ConvGenerator64(), networks.SNDiscriminator64()
    Go, Do = orc.make_generator(8), orc.make_discriminator(8)
    Go.load_state_dict(G.state_dict())
    Do.load_state_dict(D.state_dict())
    return G.cuda(), D.cuda(), Go, Do


@pytest.mark.parametrize("B", [1, 5, 64])
def test_generator64_forward_backward(B):
    from ipr_gan_b200 import engine
    from oracle import ipr_oracle as orc
    G, _, Go, _ = _pair()
    z = torch.randn(B, 128)
    Gs = copy.deepcopy(Go)
    engine.CAPTURE_ACTS = []
    try:
        out = G(z.cuda())
        (_, acts), = engine.CAPTURE_ACTS
    finally:
        engine.CAPTURE_ACTS = None
    ref = Go(z)
    sim = orc.gen_forward_sim_bf16(Gs, z, masks=_nchw_masks(acts))
    assert out.shape == (B, 3, SIZE, SIZE) and rel(out, ref) < 2e-2 and rel(out, sim) < 1e-2
    g = torch.randn_like(ref)
    out.backward(g.cuda())
    sim.backward(g)
    for (n, p), (_, r) in zip(G.named_parameters(), Gs.named_parameters()):
        assert rel(p.grad, r.grad) < GRAD_TOL, (n, rel(p.grad, r.grad))
    for (n, b), (_, c) in zip(G.named_buffers(), Go.named_buffers()):      # running statistics updated alike
        assert rel(b.float(), c.float()) < 2e-2, n
    G.eval(); Go.eval()
    with torch.no_grad():
        assert rel(G(z.cuda()), Go(z)) < 2e-2


@pytest.mark.parametrize("B", [1, 5, 64])
def test_discriminator64_forward_backward(B):
    from ipr_gan_b200 import engine
    from oracle import ipr_oracle as orc
    _, D, _, Do = _pair(1)
    x = torch.randn(B, 3, SIZE, SIZE).clamp(-1, 1)
    xg = x.clone().cuda().requires_grad_(True)
    xo = x.clone().requires_grad_(True)
    Ds = copy.deepcopy(Do)
    xs = x.clone().requires_grad_(True)
    engine.CAPTURE_ACTS = []
    try:
        out = D(xg)
        (_, acts), = engine.CAPTURE_ACTS
    finally:
        engine.CAPTURE_ACTS = None
    ref, sim = Do(xo), orc.dis_forward_sim_bf16(Ds, xs, masks=_nchw_masks(acts))
    assert out.shape == (B,) and rel(out, ref) < 2e-2 and rel(out, sim) < 1e-2
    w = torch.randn(B)
    (out * w.cuda()).sum().backward()
    (sim * w).sum().backward()
    assert rel(xg.grad, xs.grad) < GRAD_TOL, rel(xg.grad, xs.grad)
    for (n, p), (_, r) in zip(D.named_parameters(), Ds.named_parameters()):
        assert rel(p.grad, r.grad) < GRAD_TOL, (n, rel(p.grad, r.grad))
    for (n, b), (_, c) in zip(D.named_buffers(), Do.named_buffers()):      # power-iteration state advanced alike
        assert rel(b, c) < 1e-3, n


@pytest.mark.parametrize("B", [16, 64])
def test_protected_step64_vs_oracle(watermark_path, B):
    """update_d + update_g at 64 x 64 with a 32 x 32 watermark through the drop-in API vs the oracle step."""
    import models
    from configs import presets
    from oracle import ipr_oracle as orc
    torch.manual_seed(1234)
    model = models.DCGAN(presets.dcgan_model(SIZE), device=[torch.device("cuda", 0)])
    Go, Do = orc.make_generator(8), orc.make_discriminator(8)
    Go.load_state_dict(model.G.module.state_dict())
    Do.load_state_dict(model.D.module.state_dict())
    model = models.BlackBoxWrapper(model, presets.dcgan_blackbox(wm_size=WM))
    model = models.WhiteBoxWrapper(model, presets.dcgan_whitebox())
    fg, bg = orc.load_watermark(watermark_path, WM, True, True)
    ref = orc.DCGANStepOracle(Go, Do, orc.transform_dist, lambda y: orc.paste_patch(y, fg, bg, "tl", WM))
    for step in range(2):
        real, z = _synth_step_inputs(B, 1234 + step)
        model.update_d({"real_sample": real, "latent": z})
        model.update_g({"fake_sample": model.fake_sample})
        ref.step(real, z)
        got, want = model.get_metrics(), ref.metrics()
        assert sorted(got) == sorted(want)
        for k in want:
            assert abs(got[k] - want[k]) <= 2e-2 * max(1.0, abs(want[k])), (step, k, got[k], want[k])
        assert torch.equal(model.ywm.cpu(), orc.paste_patch(model.fake_sample.detach().cpu(), fg, bg, "tl", WM))
        assert torch.allclose(model.xwm.cpu(), ref.xwm, rtol=1e-4, atol=1e-6)
        tol = 2e-2 if step == 0 else 1e-1
        assert rel(model.fake_sample, ref.fake) < tol and rel(model.Gxwm, ref.Gxwm) < tol
    for (n, p), (_, q) in zip(model.G.module.named_parameters(), Go.named_parameters()):
        assert float((p.detach().cpu() - q.detach()).abs().max()) <= 2.0e-3, n
        if p.dim() > 1:
            assert rel(p, q) < 2e-2, n
    assert model.loss_model.compute_ber_counts(model.G) == (0, 448)


def _run_trainer(B, use_graph, seed, steps=3):
    from ipr_gan_b200.trainer import ProtectedDCGANTrainer
    dev = torch.device("cuda", 0)
    g = torch.Generator().manual_seed(seed)
    warm = (torch.randn(B, 3, SIZE, SIZE, generator=g).clamp(-1, 1), torch.randn(B, 128, generator=g))
    batches = [(torch.randn(B, 3, SIZE, SIZE, generator=g).clamp(-1, 1), torch.randn(B, 128, generator=g))
               for _ in range(steps)]
    tr = ProtectedDCGANTrainer(B, dev, use_graph=use_graph, size=SIZE, wm_size=WM)
    tr.set_inputs(*warm)
    tr.capture(warmup=3)
    assert (tr.graph is not None) == use_graph
    out = [tr.step_from_host(real, z) for real, z in batches]
    torch.cuda.synchronize()
    params = [p.detach().clone() for p in list(tr.model.G.parameters()) + list(tr.model.D.parameters())]
    bufs = [b.detach().clone() for b in list(tr.model.G.buffers()) + list(tr.model.D.buffers())]
    return out, params, bufs


def test_graph_replay_equals_eager64():
    m_e, p_e, b_e = _run_trainer(64, False, 11)
    m_g, p_g, b_g = _run_trainer(64, True, 11)
    assert m_e == m_g, (m_e, m_g)
    assert all(torch.equal(a, b) for a, b in zip(p_e, p_g))
    assert all(torch.equal(a, b) for a, b in zip(b_e, b_g))
    assert len({tuple(sorted(m.items())) for m in m_g}) == 3          # the replays really consumed the new inputs


@pytest.mark.parametrize("B,use_graph", [(64, False), (64, True), (512, True)])
def test_protected_step64_identical_with_and_without_band_fold(monkeypatch, B, use_graph):
    from ipr_gan_b200 import engine
    band = engine.tapfold3_band
    used = []

    def counted(*args, **kw):
        out = band(*args, **kw)
        used.append(out is not None)
        return out
    monkeypatch.setattr(engine, "tapfold3_band", counted)

    def run(off):
        monkeypatch.setenv("IPR_NO_TAPFOLD", "1" if off else "0")
        del used[:]
        res = _run_trainer(B, use_graph, B)
        assert used and all(u != off for u in used)        # the arm took the path it names
        return res

    m0, p0, b0 = run(True)
    m1, p1, b1 = run(False)
    assert m0 == m1, (m0, m1)
    assert all(torch.equal(x, y) for x, y in zip(p0, p1))
    assert all(torch.equal(x, y) for x, y in zip(b0, b1))


def test_verification_sweep64_matches_oracle():
    """The sweep on the 64 x 64 generator scores 32 x 32 watermark crops (no bicubic step before pHash)."""
    import models
    from configs import presets
    from ipr_gan_b200 import verify
    from oracle import ipr_oracle as orc
    torch.manual_seed(3)
    dev = torch.device("cuda", 0)
    model = models.DCGAN(presets.dcgan_model(SIZE), device=[dev])
    model = models.BlackBoxWrapper(model, presets.dcgan_blackbox(wm_size=WM))
    model = models.WhiteBoxWrapper(model, presets.dcgan_whitebox())
    G = model.G
    res = verify.verification_sweep(G, model.fn_inp, model.fn_out, n_samples=96, batch=40, p_thres=0.01,
                                    sign_model=model.loss_model, return_per_sample=True)
    assert res["N"] == 96 and res["WBOX_counts"] == (0, 448)
    gen = torch.Generator().manual_seed(1234)
    G.eval()
    qs, ps, rs = [], [], []
    with torch.no_grad():
        for b in (40, 40, 16):
            z = torch.randn(b, 128, generator=gen).to(dev)
            x = G(z)
            xwm, ywm = G(model.fn_inp(z)), model.fn_out(x)
            assert xwm.shape[-1] == SIZE
            cx = ((xwm[..., :WM, :WM].clamp(-1, 1) + 1) / 2).cpu()
            cy = ((ywm[..., :WM, :WM].clamp(-1, 1) + 1) / 2).cpu()
            qs.append(orc.ssim_per_sample(cx, cy))
            p, r = orc.matching_prob(cx, cy)
            ps.append(p), rs.append(torch.from_numpy(r))
    q, p, r = torch.cat(qs), torch.cat(ps), torch.cat(rs)
    per = res["per_sample"]
    assert np.array_equal(per["r"].cpu().numpy(), r.numpy())                 # Hamming agreement count: bit-exact
    assert np.array_equal(per["p"].cpu().numpy(), p.numpy())                 # p-values: bit-exact
    assert torch.allclose(per["q"].cpu(), q, rtol=1e-4, atol=1e-6)           # per-sample SSIM: 1e-4
    assert res["MATCH"] == int((p < 0.01).sum())
    with torch.no_grad():
        G.module.convs[0][1].weight[:44] *= -1
    res2 = verify.verification_sweep(G, model.fn_inp, model.fn_out, n_samples=8, batch=8, sign_model=model.loss_model)
    assert res2["WBOX_counts"] == (44, 448)
