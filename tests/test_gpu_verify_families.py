"""GPU: the on-device verification sweep of the image-to-image families -- protected SRGAN (config 3 shapes: 24 -> 96,
noise patch 12, watermark 48, normalized=False) and CycleGAN's GB (256 x 256, noise patch 64, watermark 64,
normalized=True) -- against the oracle's CPU evaluation of the same generator outputs; the clamp(0, 1) crop kernel;
graph replay against the eager sweep; and a two-rank sweep against one rank."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SEED = 1234


def _bits(t):
    return t.detach().cpu().contiguous().numpy().view(np.uint32)


def _srgan(dev):
    import models
    from configs import presets
    os.environ["IPR_VGG_RANDOM_INIT"] = "1"
    torch.manual_seed(SEED)
    m = models.SRGAN(presets.srgan_model(), device=[dev])
    m = models.BlackBoxWrapper(m, presets.srgan_blackbox())
    return models.WhiteBoxWrapper(m, presets.whitebox("G"))


def _cyclegan(dev):
    import models
    from configs import presets
    torch.manual_seed(SEED)
    m = models.CycleGAN(presets.cyclegan_model(), device=[dev])
    m = models.BlackBoxWrapper(m, presets.cyclegan_blackbox())
    return models.WhiteBoxWrapper(m, presets.whitebox("GB"))


@pytest.fixture(scope="module")
def srgan():
    dev = torch.device("cuda", 0)
    model = _srgan(dev)
    inputs = torch.rand(40, 3, 24, 24, generator=torch.Generator().manual_seed(7))
    return model, inputs


def _oracle_check(res, G, fn_inp, fn_out, inputs, splits, post, p_thres):
    """Regenerate the sweep's crops through the modules (same batch splits) and score them with the CPU oracle."""
    from oracle import ipr_oracle as orc
    dev = next(G.parameters()).device
    from ipr_gan_b200 import ops
    mod = fn_out.module
    s = mod.config.size
    G.eval()
    qs, ps, rs = [], [], []
    i = 0
    with torch.no_grad():
        for b in splits:
            inp = inputs[i:i + b].to(dev)
            i += b
            x = G(inp)
            gxwm, ywm = G(fn_inp(inp)), fn_out(x)
            r0, c0 = ops.window_origin(mod.position, s, x.shape[2], x.shape[3])
            cx, cy = (post(t[..., r0:r0 + s, c0:c0 + s]).cpu() for t in (gxwm, ywm))
            qs.append(orc.ssim_per_sample(cx, cy))
            p, r = orc.matching_prob(cx, cy)
            ps.append(p), rs.append(torch.from_numpy(r))
    G.train()
    q, p, r = torch.cat(qs), torch.cat(ps), torch.cat(rs)
    per = res["per_sample"]
    assert res["N"] == inputs.shape[0] == per["q"].numel()
    assert np.array_equal(per["r"].cpu().numpy(), r.numpy())                 # matching bits: bit-exact
    assert np.array_equal(per["p"].cpu().numpy(), p.numpy())                 # p-values: bit-exact
    assert torch.allclose(per["q"].cpu(), q, rtol=1e-4, atol=1e-6)           # per-sample SSIM: 1e-4
    assert res["MATCH"] == int((p < p_thres).sum())
    assert abs(res["P"] - float(p.double().mean())) < 1e-9 and abs(res["Q_WM"] - float(q.double().mean())) < 1e-5
    # the per-sample values the sweep returned add up to its sums
    pp, qq = per["p"].cpu().double(), per["q"].cpu().double()
    assert res["MATCH"] == int((per["p"].cpu() < p_thres).sum())
    assert abs(res["P"] - float(pp.mean())) < 1e-12 and abs(res["Q_WM"] - float(qq.mean())) < 1e-12


def test_srgan_sweep_matches_oracle(srgan):
    from ipr_gan_b200 import verify
    model, inputs = srgan
    G = model.G
    fg = model.fn_inp.module.fg.clone()
    assert G.training
    res = verify.image_verification_sweep(G, model.fn_inp, model.fn_out, inputs, batch=16,
                                          sign_model=model.loss_model, return_per_sample=True)
    assert G.training                                                        # training mode restored
    assert torch.equal(model.fn_inp.module.fg, fg)                          # the trigger is never re-drawn
    assert res["WBOX_counts"] == (0, 2112)
    _oracle_check(res, G, model.fn_inp, model.fn_out, inputs, (16, 16, 8), lambda t: t.clamp(0, 1), 0.05)
    # sign flip of 10 % of one BatchNorm layer's gammas: the white-box count is exactly the flipped bits
    bn = next(m for m in G.module.modules() if isinstance(m, torch.nn.BatchNorm2d))
    k = bn.weight.numel() // 10
    with torch.no_grad():
        bn.weight[:k] *= -1
    try:
        res2 = verify.image_verification_sweep(G, model.fn_inp, model.fn_out, inputs[:8], batch=8,
                                               sign_model=model.loss_model)
        assert res2["WBOX_counts"] == (k, 2112) and res2["N"] == 8
    finally:
        with torch.no_grad():
            bn.weight[:k] *= -1


def test_cyclegan_gb_sweep_matches_oracle():
    from ipr_gan_b200 import verify
    model = _cyclegan(torch.device("cuda", 0))
    inputs = torch.rand(5, 3, 256, 256, generator=torch.Generator().manual_seed(8)) * 2 - 1
    res = verify.image_verification_sweep(model.GB, model.fn_inp, model.fn_out, inputs, batch=2,
                                          sign_model=model.loss_model, return_per_sample=True)
    assert res["WBOX_counts"] == (0, 5248)
    _oracle_check(res, model.GB, model.fn_inp, model.fn_out, inputs, (2, 2, 1),
                  lambda t: (t.clamp(-1, 1) + 1) / 2, 0.05)


def test_crop_clamp01_bit_exact():
    """clamp(0, 1) post-processing of the crop, one launch: bit-identical to apply_mask followed by torch.clamp, special
    values included, at every window position; the (clamp(-1, 1) + 1) / 2 mode is unchanged."""
    from ipr_gan_b200 import ops
    torch.manual_seed(3)
    x = torch.randn(9, 3, 32, 32) * 1.5
    specials = torch.tensor([float("nan"), float("inf"), -float("inf"), -0.0, 0.0, 1.0, -1.0, 0.5, 1.0000001, -1e-30])
    for r0, left in ((0, True), (0, False), (31, True), (31, False)):   # inside every window below, at each corner
        x[1, 1, r0, :10] = specials if left else x[1, 1, r0, :10]
        x[1, 1, r0, 22:] = x[1, 1, r0, 22:] if left else specials.flip(0)
    xc = x.cuda()
    for pos in ("tl", "tr", "bl", "br"):
        for s in (16, 5):
            r0, c0 = ops.window_origin(pos, s, 32, 32)
            for bg in (torch.zeros(1, 1, s, s), (torch.rand(1, 1, s, s) > 0.5).float()):
                crop = ops.crop_patch(xc, bg.cuda(), pos, s)
                got = ops.crop_patch(xc, bg.cuda(), pos, s, postproc="unit")
                assert np.array_equal(_bits(got), _bits(crop.clamp(0, 1)))       # GPU torch.clamp
                assert np.array_equal(_bits(got), _bits(crop.cpu().clamp(0, 1)))  # CPU torch.clamp
                signed = ops.crop_patch(xc, bg.cuda(), pos, s, postproc="signed")
                assert np.array_equal(_bits(signed), _bits(ops.crop_patch(xc, bg.cuda(), pos, s, postproc=True)))
                want = (crop.cpu().clamp(-1, 1) + 1.0) / 2.0
                assert torch.equal(torch.nan_to_num(signed.cpu(), nan=7.0), torch.nan_to_num(want, nan=7.0))
            # an opaque window is a pure crop: the values of x[..., window].clamp(0, 1) (the crop's 0 + 1 * x maps
            # -0 to +0, hence a value comparison with NaN positions matched separately)
            got = ops.crop_patch(xc, torch.zeros(1, 1, s, s, device="cuda"), pos, s, postproc="unit").cpu()
            want = x[..., r0:r0 + s, c0:c0 + s].clamp(0, 1)
            assert torch.equal(got.isnan(), want.isnan())
            assert torch.equal(torch.nan_to_num(got, nan=7.0), torch.nan_to_num(want, nan=7.0))


def test_graph_sweep_equals_eager(srgan):
    from ipr_gan_b200 import verify
    model, inputs = srgan
    runs = [verify.image_verification_sweep(model.G, model.fn_inp, model.fn_out, inputs, batch=16,
                                            return_per_sample=True, eager=e) for e in (False, True, False)]
    for other in runs[1:]:
        for k in ("q", "p", "r"):
            assert np.array_equal(_bits(runs[0]["per_sample"][k]), _bits(other["per_sample"][k])), k
        for k in ("Q_WM", "P", "MATCH", "N"):
            assert runs[0][k] == other[k], k


def test_two_rank_sweep_equals_one_rank(srgan):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    from ipr_gan_b200 import verify
    model, _ = srgan
    n = 37
    inputs = torch.rand(n, 3, 24, 24, generator=torch.Generator().manual_seed(11))
    one = verify.image_verification_sweep(model.G, model.fn_inp, model.fn_out, inputs, batch=8)
    port = 29500 + (os.getpid() % 400) + 1
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "verify_families_worker.py"), str(n), "8"]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    lines = [l for l in r.stdout.splitlines() if l.startswith("RESULT ")]
    assert r.returncode == 0 and lines, r.stdout[-3000:] + r.stderr[-3000:]
    two = json.loads(lines[-1][7:])
    assert two["world"] == 2 and two["N"] == one["N"] == n
    assert two["MATCH"] == one["MATCH"]
    assert abs(two["P"] - one["P"]) <= 1e-12 * max(1.0, abs(one["P"]))
    assert abs(two["Q_WM"] - one["Q_WM"]) <= 1e-12 * max(1.0, abs(one["Q_WM"]))
