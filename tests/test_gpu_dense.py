"""GPU: the tcgen05 tap-GEMM (csrc/gemm_tc.cu) against fp32 PyTorch convolutions of the same
bf16-rounded operands.  Tolerance: bf16 operands, fp32 accumulate -> the result is exact up to the bf16
rounding of the OUTPUT (rel 2^-8) plus accumulation-order noise; north_star budget for bf16 convs is 2e-2."""
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def bf(x):
    return x.to(torch.bfloat16).float()


def nhwc(x):
    return x.permute(0, 2, 3, 1).contiguous().to(torch.bfloat16)


def close(got, want, tol=1e-2):
    scale = want.abs().max().item() + 1e-6
    err = (got.float() - want).abs().max().item()
    assert err <= tol * scale, (err, scale)


@pytest.mark.parametrize("B,C,O,H", [(8, 64, 128, 16), (4, 128, 256, 8), (16, 256, 512, 4), (3, 64, 64, 32)])
def test_conv3_forward_bias_lrelu(B, C, O, H):
    from ipr_gan_b200 import dense
    torch.manual_seed(B + C)
    x = torch.randn(B, C, H, H, device="cuda")
    w = torch.randn(O, C, 3, 3, device="cuda") * 0.05
    b = torch.randn(O, device="cuda")
    sigma = torch.tensor(1.7, device="cuda")
    plan = dense.Plan("conv3", C, O)
    out, _ = plan.run(nhwc(x), plan.pack(w), epi=dense.EPI_BIAS_LRELU, slope=0.1, sigma=sigma, bias=b)
    want = F.leaky_relu(F.conv2d(bf(x), bf(w), padding=1) / 1.7 + b.view(1, -1, 1, 1), 0.1)
    close(out.permute(0, 3, 1, 2), want)


@pytest.mark.parametrize("B,C,O,H", [(8, 64, 64, 32), (4, 128, 128, 16), (16, 256, 256, 8)])
def test_conv4s2_forward(B, C, O, H):
    from ipr_gan_b200 import dense
    torch.manual_seed(B + C)
    x = torch.randn(B, C, H, H, device="cuda")
    w = torch.randn(O, C, 4, 4, device="cuda") * 0.05
    plan = dense.Plan("conv4s2", C, O)
    out, _ = plan.run(nhwc(x), plan.pack(w))
    close(out.permute(0, 3, 1, 2), F.conv2d(bf(x), bf(w), stride=2, padding=1))


@pytest.mark.parametrize("B,C,O,H", [(8, 512, 256, 4), (4, 256, 128, 8), (2, 128, 64, 16)])
def test_convT4s2_forward_with_stats(B, C, O, H):
    from ipr_gan_b200 import dense
    torch.manual_seed(B + C)
    x = torch.randn(B, C, H, H, device="cuda")
    w = torch.randn(C, O, 4, 4, device="cuda") * 0.05
    plan = dense.Plan("convT4s2", C, O)
    out, stats = plan.run(nhwc(x), plan.pack(w), want_stats=True)
    want = F.conv_transpose2d(bf(x), bf(w), stride=2, padding=1)
    close(out.permute(0, 3, 1, 2), want)
    s = stats.sum(0)
    close(s[0], want.sum((0, 2, 3)), tol=2e-3)
    close(s[1], (want * want).sum((0, 2, 3)), tol=2e-3)


@pytest.mark.parametrize("epi", ["linear", "mask"])
def test_short_main_loop_stats(epi):
    """Statistics of a one-k-block layer with one N block and at least 4 tiles per SM: the launch runs a variant whose
    per-CTA statistics rows must match what ipr_tapgemm_stats_rows allocated.  The stats tensor is handed the block of
    a freed NaN-filled tensor, so a row the kernel does not write turns the sums into NaN."""
    from ipr_gan_b200 import dense
    torch.manual_seed(5)
    B, C, O, H = 512, 64, 128, 16
    x = torch.randn(B, H, H, C, device="cuda")
    w = torch.randn(O, C, device="cuda") * 0.05
    plan = dense.Plan("linear", C, O)
    wp = plan.pack(w)
    kw = dict(want_stats=True)
    if epi == "mask":
        mask = torch.randn(B, H, H, O, device="cuda").to(torch.bfloat16)
        kw.update(epi=dense.EPI_MASK, slope=0.1, mask=mask)
    a = x.to(torch.bfloat16)
    out, stats = plan.run(a, wp, **kw)
    shape = stats.shape
    del out, stats
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.full(shape, float("nan"), device="cuda")          # freed at once: its block goes back to the cache
    out, stats = plan.run(a, wp, **kw)
    want = (bf(x) @ bf(w).t()).view(B, H, H, O)
    if epi == "mask":
        want = want * torch.where(mask.float() > 0, 1.0, 0.1)
    close(out.float(), want)
    s = stats.sum(0)
    close(s[0], want.sum((0, 1, 2)), tol=2e-3)
    if epi == "linear":
        close(s[1], (want * want).sum((0, 1, 2)), tol=2e-3)


def test_convT3_tanh_nchw():
    from ipr_gan_b200 import dense
    torch.manual_seed(1)
    x = torch.randn(8, 64, 32, 32, device="cuda")
    w = torch.randn(64, 3, 3, 3, device="cuda") * 0.05
    plan = dense.Plan("convT3", 64, 3, n_pad=16)
    out, _ = plan.run(nhwc(x), plan.pack(w), epi=dense.EPI_TANH_NCHW, n_valid=3)
    assert out.shape == (8, 3, 32, 32) and out.dtype == torch.float32
    close(out, torch.tanh(F.conv_transpose2d(bf(x), bf(w), stride=1, padding=1)), tol=2e-3)


def test_linear_relu_and_batch_tail():
    from ipr_gan_b200 import dense
    torch.manual_seed(2)
    for B in (8, 64, 200):
        z = torch.randn(B, 128, device="cuda")
        w = torch.randn(8192, 128, device="cuda") * 0.05
        b = torch.randn(8192, device="cuda")
        plan = dense.Plan("linear", 128, 8192)
        a = z.to(torch.bfloat16).view(B, 1, 1, 128)
        out, _ = plan.run(a, plan.pack(w), epi=dense.EPI_BIAS_LRELU, slope=0.0, bias=b)
        close(out.view(B, 8192), F.relu(bf(z) @ bf(w).t() + b))


@pytest.mark.parametrize("kind,B,C,O,H", [("conv3_dgrad", 8, 128, 64, 16), ("conv4s2_dgrad", 8, 128, 128, 8),
                                          ("convT4s2_dgrad", 4, 128, 256, 16)])
def test_data_gradients(kind, B, C, O, H):
    """dgrad plans: A = dY (C channels), result = dX (O channels), checked against autograd."""
    from ipr_gan_b200 import dense
    torch.manual_seed(3)
    plan = dense.Plan(kind, C, O)
    if kind == "conv3_dgrad":
        w = torch.randn(C, O, 3, 3, device="cuda") * 0.05            # conv weight (out=C, in=O)
        x = torch.randn(B, O, H, H, device="cuda", requires_grad=True)
        y = F.conv2d(x, bf(w), padding=1)
    elif kind == "conv4s2_dgrad":
        w = torch.randn(C, O, 4, 4, device="cuda") * 0.05
        x = torch.randn(B, O, 2 * H, 2 * H, device="cuda", requires_grad=True)
        y = F.conv2d(x, bf(w), stride=2, padding=1)
    else:
        w = torch.randn(O, C, 4, 4, device="cuda") * 0.05            # convT weight (in=O, out=C)
        x = torch.randn(B, O, H // 2, H // 2, device="cuda", requires_grad=True)
        y = F.conv_transpose2d(x, bf(w), stride=2, padding=1)
    dy = torch.randn_like(y)
    y.backward(bf(dy))
    mask = torch.randn(B, x.shape[2], x.shape[3], O, device="cuda").to(torch.bfloat16)
    out, _ = plan.run(nhwc(dy), plan.pack(w), epi=dense.EPI_MASK, slope=0.1, mask=mask)
    want = x.grad * torch.where(mask.float() > 0, 1.0, 0.1).permute(0, 3, 1, 2)
    close(out.permute(0, 3, 1, 2), want)


@pytest.mark.parametrize("kind,B,C,O,H", [("conv3", 8, 64, 128, 16), ("conv3", 4, 256, 512, 4), ("conv4s2", 8, 64, 64, 32),
                                          ("conv4s2", 16, 256, 256, 8), ("convT4s2", 8, 512, 256, 4),
                                          ("convT4s2", 4, 128, 64, 16), ("linear", 200, 128, 8192, 1)])
def test_weight_gradients(kind, B, C, O, H):
    """tcgen05 wgrad (MN-major operands, split-K) against autograd of the fp32 op on bf16-rounded operands."""
    from ipr_gan_b200 import dense
    torch.manual_seed(4)
    if kind == "linear":
        w = (torch.randn(O, C, device="cuda") * 0.05).requires_grad_(True)
        x = torch.randn(B, C, device="cuda")
        y = bf(x) @ w.t()
        xa = x.to(torch.bfloat16).view(B, 1, 1, C)
    else:
        ksz = 3 if kind == "conv3" else 4
        if kind == "convT4s2":
            w = (torch.randn(C, O, ksz, ksz, device="cuda") * 0.05).requires_grad_(True)
            x = torch.randn(B, C, H, H, device="cuda")
            y = F.conv_transpose2d(bf(x), w, stride=2, padding=1)
        else:
            w = (torch.randn(O, C, ksz, ksz, device="cuda") * 0.05).requires_grad_(True)
            x = torch.randn(B, C, H, H, device="cuda")
            y = F.conv2d(bf(x), w, stride=1 if kind == "conv3" else 2, padding=1)
        xa = nhwc(x)
    dy = torch.randn_like(y)
    y.backward(bf(dy))
    plan = dense.Plan(kind, C, O)
    wg = dense.WGradPlan(plan, tuple(w.shape))
    dya = dy.to(torch.bfloat16).view(B, 1, 1, O) if kind == "linear" else nhwc(dy)
    grad = torch.full_like(w, 7.0).detach()
    wg.run(dya, xa, grad)
    close(grad, w.grad, tol=5e-3)
    wg.run(dya, xa, grad, accumulate=True, scale=0.5, splits=3)
    close(grad, 1.5 * w.grad, tol=5e-3)


@pytest.mark.parametrize("B,H", [(8, 32), (3, 32), (5, 16)])
def test_tap_expanded_three_channel_layers(B, H):
    """The 3-channel ends: one plain GEMM to 27 (tap, channel) columns + col2im3 fold, against
    ConvTranspose2d(64,3,3,1,1)+Tanh (generator) and the input gradient of Conv2d(3,64,3,1,1) (discriminator)."""
    from ipr_gan_b200 import dense, engine
    torch.manual_seed(B * H)
    plan = dense.Plan("linear", 64, 32)
    a = torch.randn(B, 64, H, H, device="cuda")
    # generator: weight (I=64, O=3, kh, kw)
    wt = torch.randn(64, 3, 3, 3, device="cuda") * 0.1
    t9, _ = plan.run(nhwc(a), engine._tap27_rows_layout(wt).to(torch.bfloat16), epi=dense.EPI_LINEAR_F32, n_valid=32)
    got = engine.col2im3(t9, True)
    want = torch.tanh(F.conv_transpose2d(bf(a), bf(wt), stride=1, padding=1))
    assert got.shape == (B, 3, H, H)
    close(got, want, tol=2e-3)
    # discriminator: weight (O=64, C=3, kh, kw), dy has 64 channels; dx = conv_transpose2d(dy, W) / sigma
    wc = torch.randn(64, 3, 3, 3, device="cuda") * 0.1
    sigma = torch.tensor(2.5, device="cuda")
    t9, _ = plan.run(nhwc(a), engine._tap27_rows_layout(wc).to(torch.bfloat16), epi=dense.EPI_LINEAR_F32, sigma=sigma,
                     n_valid=32)
    got = engine.col2im3(t9, False)
    want = F.conv_transpose2d(bf(a), bf(wc), stride=1, padding=1) / 2.5
    close(got, want, tol=2e-3)


# Batch 512 is the shape bench.py times (BASELINE config 2): every persistent CTA walks many tiles, the TMEM accumulator
# double-buffers, the TMA ring wraps many times.  The small-batch cases above never reach those code paths.
@pytest.mark.parametrize("fn,args", [
    ("test_conv3_forward_bias_lrelu", (512, 64, 128, 16)), ("test_conv3_forward_bias_lrelu", (512, 256, 512, 4)),
    ("test_conv4s2_forward", (512, 64, 64, 32)), ("test_conv4s2_forward", (512, 256, 256, 8)),
    ("test_convT4s2_forward_with_stats", (512, 512, 256, 4)), ("test_convT4s2_forward_with_stats", (512, 128, 64, 16)),
    ("test_data_gradients", ("conv3_dgrad", 512, 128, 64, 16)), ("test_data_gradients", ("conv4s2_dgrad", 512, 64, 64, 16)),
    ("test_data_gradients", ("convT4s2_dgrad", 512, 128, 256, 16)),
    ("test_weight_gradients", ("conv3", 512, 64, 128, 16)), ("test_weight_gradients", ("conv4s2", 512, 64, 64, 32)),
    ("test_weight_gradients", ("convT4s2", 512, 512, 256, 4)), ("test_weight_gradients", ("convT4s2", 512, 128, 64, 16)),
    ("test_weight_gradients", ("linear", 512, 128, 8192, 1)),
    ("test_tap_expanded_three_channel_layers", (512, 32)),
])
def test_batch_512_shapes(fn, args):
    globals()[fn](*args)
