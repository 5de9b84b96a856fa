"""CPU: the float64 references of tests/seq_kernel_refs.py against the kernels' contract as
tests/test_seqnet_host_logic.py emulates it (patch matrix, adjoint gather) and against stock torch
(nn.BatchNorm2d / nn.InstanceNorm2d + PReLU / LeakyReLU / ReLU autograd), and -- on the seeded inputs of
tests/test_gpu_seq_kernels.py -- every plausible wrong kernel (a ``variant=`` mutant of a reference) rejected by
the check the GPU test applies."""
import zlib

import pytest
import torch
import torch.nn as nn
import torch.nn.functional as F

from tests import seq_kernel_refs as R
from tests.test_seqnet_host_logic import CASES, emulate_col2im, emulate_im2col


def rejected(got, want, tol):
    return R.max_excess(got, want, tol) > 0


def case(cid):
    return next(c for c in R.net_cases() if c["id"] == cid)


def norm_case(cid, sms=148):
    return next(c for c in R.norm_cases() + R.norm_edges(sms) if c["id"] == cid)


def seed(cid, tag):
    """The GPU test's seed of an input (tests/test_gpu_seq_kernels.py uses the same function)."""
    return zlib.crc32(("%s/%s" % (cid, tag)).encode())


# ============================================================================================== patch matrix
@pytest.mark.parametrize("name,make,reflect,size", CASES, ids=[c[0] for c in CASES])
def test_patch_refs_equal_the_emulation(name, make, reflect, size):
    from ipr_gan_b200 import seqnet
    torch.manual_seed(0)
    b = seqnet.Block(make().double(), reflect)
    n, h, w = 2, size, size + 1
    oh, ow = b.out_hw(h, w)
    x = torch.randn(n, h, w, b.cin_p, dtype=torch.float64)
    assert torch.equal(R.im2col_ref(x, b, oh, ow), emulate_im2col(x, b, oh, ow))
    dcol = torch.randn(n * oh * ow, b.kp, dtype=torch.float64)
    addend = torch.randn(n, h, w, b.cin_p, dtype=torch.float64)
    want = emulate_col2im(dcol, b, (n, h, w, b.cin_p), oh, ow)
    assert torch.allclose(R.col2im_ref(dcol, b, (n, h, w, b.cin_p), oh, ow), want, rtol=1e-14, atol=1e-13)
    assert torch.allclose(R.col2im_ref(dcol, b, (n, h, w, b.cin_p), oh, ow, addend), want + addend, rtol=1e-14,
                          atol=1e-13)


def test_case_list_covers_the_issue_shapes():
    cs = R.net_cases()
    kps = {c["block"].kp for c in cs}
    assert {96, 416, 672, 18432} <= kps
    ms = {c["shape"][0] * c["ohw"][0] * c["ohw"][1] for c in cs}
    assert {16, 225, 196, 576} <= ms
    assert any(c["block"].reflect and c["block"].pad == 3 and c["block"].cin_p == 8 and c["dgrad"] for c in cs)
    assert any(c["block"].up == 2 for c in cs) and any(c["block"].stride == 2 and c["block"].k == 4 for c in cs)
    assert len({c["id"] for c in cs}) == len(cs)
    # every first block whose input gradient a training step uses: the discriminators' (D(G(z))) and Resnet9Blocks'
    first = {c["net"]: c for c in cs if c["i"] == 0 and "-odd" not in c["id"]}
    assert [n for n in first if first[n]["dgrad"]] == ["Discriminator96", "Resnet9Blocks", "ConvDiscriminator"]
    cd0 = first["ConvDiscriminator"]["block"]
    assert (cd0.k, cd0.stride, cd0.cin_p, cd0.kp) == (4, 2, 8, 128)


@pytest.mark.parametrize("integer", [True, False])
def test_im2col_clamp_rejected(integer):
    c = case("Resnet9Blocks-odd-b0")
    x, _, _, _ = R.conv_inputs(c, integer, seed(c["id"], "conv%d" % integer))
    want = R.im2col_ref(x, c["block"], *c["ohw"])
    assert not torch.equal(R.im2col_ref(x, c["block"], *c["ohw"], variant="clamp"), want)   # compared bit for bit


@pytest.mark.parametrize("cid,variant", [("Resnet9Blocks-odd-b0", "no_mirror"), ("Resnet9Blocks-odd-b3", "no_mirror"),
                                         ("Resnet9Blocks-odd-b21", "no_output_padding")])
def test_col2im_mutants_rejected(cid, variant):
    c = case(cid)
    b, (n, h, w, cp), (oh, ow) = c["block"], c["shape"], c["ohw"]
    M = n * oh * ow
    for integer in (True, False):
        dcol = R.dcol_inputs(M, b.kp, integer, seed(cid, "dcol%d" % integer))
        want = R.col2im_ref(dcol, b, (n, h, w, cp), oh, ow)
        mut = R.col2im_ref(dcol, b, (n, h, w, cp), oh, ow, variant=variant)
        if integer:
            assert not torch.equal(mut.to(torch.bfloat16), want.to(torch.bfloat16))
        else:
            assert rejected(mut, want, R.col2im_bound(dcol, b, (n, h, w, cp), oh, ow))


# ============================================================================================== GEMMs
def _gemm_operands(c, integer):
    b = c["block"]
    x, wt, bias, dy = R.conv_inputs(c, integer, seed(c["id"], "conv%d" % integer))
    col = R.im2col_ref(x, b, *c["ohw"])
    wp = b.fwd_layout(wt)[0].to(torch.bfloat16)
    return col, wp, (R.padded_bias(b, bias) if bias is not None else None), dy, wt


@pytest.mark.parametrize("cid,variant", [("SRResNet-odd-b0", "drop_last_k_chunk"), ("Resnet9Blocks-odd-b0", "drop_last_k_chunk"),
                                         ("ConvDiscriminator-b3", "drop_last_row"), ("ConvDiscriminator-b3", "drop_m_tail"),
                                         ("ConvDiscriminator-b4", "drop_m_tail"), ("Resnet9Blocks-odd-b1", "drop_last_row")])
def test_gemm_mutants_rejected(cid, variant):
    c = case(cid)
    for integer in (True, False):
        col, wp, bias, _, _ = _gemm_operands(c, integer)
        want = R.gemm_ref(col, wp, bias)
        mut = R.gemm_ref(col, wp, bias, variant=variant)
        if integer:
            assert not torch.equal(mut.to(torch.bfloat16), want.to(torch.bfloat16))
        else:
            assert rejected(mut, want, R.gemm_bound(col, wp, want))


@pytest.mark.parametrize("cid", ["ConvDiscriminator-b3", "SRResNet-odd-b1", "Discriminator96-b7"])
def test_wgrad_dropped_last_split_rejected(cid):
    c = case(cid)
    b = c["block"]
    off, s_n, row_map = b.wgrad_tables()
    wshape = tuple(b.conv.weight.shape)
    M = c["shape"][0] * c["ohw"][0] * c["ohw"][1]
    lo, hi = R.split_rows(M, 2, 1)
    assert hi > lo
    for integer in (True, False):
        col, _, _, dy, _ = _gemm_operands(c, integer)
        old = R.wgrad_old(wshape, integer, seed(cid, "old"))
        want, tol = R.wgrad_ref(dy, col, wshape, row_map, off, s_n, old, True, 0.5)
        mut, _ = R.wgrad_ref(dy, col, wshape, row_map, off, s_n, old, True, 0.5, drop_rows=(lo, hi))
        if integer:
            assert not torch.equal(mut.float(), want.float())
        else:
            assert rejected(mut, want, tol)


def test_wgrad_ref_is_autograd():
    c = case("Resnet9Blocks-odd-b21")                          # transposed: flipped, swapped scatter
    b = c["block"]
    n, h, w, cp = c["shape"]
    x, wt, _, dy = R.conv_inputs(c, False, 5)
    weight = wt.double().clone().requires_grad_(True)
    xin = x.double()[..., :b.cin].permute(0, 3, 1, 2)
    out = F.conv_transpose2d(xin, weight, stride=b.t_stride, padding=b.t_pad, output_padding=b.out_pad)
    oh, ow = c["ohw"]
    out.backward(dy.double()[:, :b.cout].view(n, oh, ow, b.cout).permute(0, 3, 1, 2))
    off, s_n, row_map = b.wgrad_tables()
    got, _ = R.wgrad_ref(dy, R.im2col_ref(x, b, oh, ow), tuple(weight.shape), row_map, off, s_n)
    assert torch.allclose(got, weight.grad, rtol=1e-10, atol=1e-10)


def test_empty_last_split():
    for t in (1, 2, 5, 36, 144, 2304):
        s = R.empty_last_split(t)
        per = -(-t // s)
        assert (s - 1) * per >= t and (s - 2) * per < t


# ============================================================================================== norms
def _module(c, p):
    C = c["C"]
    m = nn.BatchNorm2d(C) if c["bn"] else nn.InstanceNorm2d(C, affine=c["affine"])
    m = m.double()
    m.eps = R.r32(m.eps)
    m.momentum = R.r32(0.1)
    if c["affine"]:
        with torch.no_grad():
            m.weight.copy_(p["gamma"])
            m.bias.copy_(p["beta"])
    if c["bn"]:
        with torch.no_grad():
            m.running_mean.copy_(p["running_mean"])
            m.running_var.copy_(p["running_var"])
    return m


def _act_module(c, p):
    if c["act"] == R.ACT_PRELU:
        a = nn.PReLU().double()
        with torch.no_grad():
            a.weight.copy_(p["slope"])
        return a
    return {R.ACT_NONE: nn.Identity(), R.ACT_RELU: nn.ReLU(), R.ACT_LRELU: nn.LeakyReLU(c["slope"]),
            R.ACT_TANH: nn.Tanh()}[c["act"]]


@pytest.mark.parametrize("cid", ["Discriminator96-b7", "SRResNet-odd-b1", "Resnet9Blocks-odd-b0", "ConvDiscriminator-b3",
                                 "edge-C24-in-lrelu", "edge-in-tanh", "edge-bn-prelu-residual"])
def test_norm_refs_are_torch_modules(cid):
    c = norm_case(cid)
    x, dy, res, p = R.norm_inputs(c, seed(cid, "norm"))
    G, rows, C = c["groups"], c["rows"], c["C"]
    m, a = _module(c, p), _act_module(c, p)
    X = x.double().view(G, rows, C).permute(0, 2, 1).unsqueeze(-1).clone().requires_grad_(True)   # (N, C, rows, 1)
    Xin = X.permute(3, 1, 2, 0).reshape(1, C, rows, 1) if c["bn"] else X        # BatchNorm: one image of rows pixels
    R_ = res.double().view(G, rows, C).permute(0, 2, 1).unsqueeze(-1) if c["residual"] else 0
    y = a(m.train()(Xin))
    y = (y if not c["bn"] else y.view(C, rows).t().reshape(1, rows, C).permute(0, 2, 1).unsqueeze(-1)) + R_
    slope = float(p["slope"]) if c["act"] == R.ACT_PRELU else c["slope"]
    st, _ = R.norm_stats_ref(x, G, rows, p["gamma"] if c["affine"] else None, p["beta"] if c["affine"] else None,
                             1e-5, 0.1, p["running_mean"] if c["bn"] else None, p["running_var"] if c["bn"] else None)
    yw, _ = R.norm_act_ref(x, G, rows, st["scale"], st["shift"], c["act"], slope, res if c["residual"] else None)
    got = y.squeeze(-1).permute(0, 2, 1).reshape(G * rows, C)
    assert torch.allclose(yw, got, rtol=1e-10, atol=1e-10)
    if c["bn"]:
        assert torch.allclose(st["running_mean"], m.running_mean, rtol=1e-12, atol=1e-14)
        assert torch.allclose(st["running_var"], m.running_var, rtol=1e-12, atol=1e-14)
        assert int(m.num_batches_tracked) == 1                  # the kernel adds one per launch (checked on the GPU)
    # backward
    y.squeeze(-1).permute(0, 2, 1).reshape(G * rows, C).backward(dy.double())
    acc = 1
    old = {k: p[k] for k in ("dgamma_old", "dbeta_old", "dslope_old")}
    bw, _ = R.norm_bwd_ref(dy, x, G, rows, p["gamma"] if c["affine"] else None, st["scale"], st["shift"], 1e-5,
                           c["act"], slope, 1, None, 0.0, 0.0, old["dgamma_old"], old["dbeta_old"], old["dslope_old"],
                           acc, want_dslope=c["act"] == R.ACT_PRELU)
    gx = X.grad.squeeze(-1).permute(0, 2, 1).reshape(G * rows, C)
    assert torch.allclose(bw["dx"], gx, rtol=1e-9, atol=1e-11)
    if c["affine"]:
        assert torch.allclose(bw["dgamma"] - old["dgamma_old"].double(), m.weight.grad, rtol=1e-9, atol=1e-10)
        assert torch.allclose(bw["dbeta"] - old["dbeta_old"].double(), m.bias.grad, rtol=1e-9, atol=1e-10)
    if c["act"] == R.ACT_PRELU:
        assert abs(float(bw["dslope"]) - float(old["dslope_old"]) - float(a.weight.grad)) < 1e-9


def test_norm_bwd_without_norm_is_activation_gradient():
    c = norm_case("SRResNet-odd-b0")
    x, dy, _, p = R.norm_inputs(c, seed(c["id"], "norm"))
    X = x.double().clone().requires_grad_(True)
    F.prelu(X, p["slope"].double()).backward(dy.double())
    bw, _ = R.norm_bwd_ref(dy, x, 1, c["rows"], None, None, None, 1e-5, R.ACT_PRELU, float(p["slope"]), has_norm=0)
    assert torch.equal(bw["dx"], X.grad)


def _norm_run_refs(c, variant=None, acc=1):
    """The references the GPU test evaluates (here with float64 statistics standing in for the kernel's scale /
    shift) for a case and one of its backward launches."""
    x, dy, res, p = R.norm_inputs(c, seed(c["id"], "norm"), c.get("mean", 0.4), c.get("std", 1.3))
    G, rows = c["groups"], c["rows"]
    gamma = p["gamma"] if c["affine"] else None
    st, stt = R.norm_stats_ref(x, G, rows, gamma, p["beta"] if c["affine"] else None, 1e-5, 0.1,
                               p["running_mean"] if c["bn"] else None, p["running_var"] if c["bn"] else None,
                               variant=variant)
    slope = float(p["slope"]) if c["act"] == R.ACT_PRELU else c["slope"]
    yw, yt = R.norm_act_ref(x, G, rows, st["scale"].float(), st["shift"].float(), c["act"], slope,
                            res if c["residual"] else None, variant=variant)
    bw, bt = R.norm_bwd_ref(dy, x, G, rows, gamma, st["scale"].float(), st["shift"].float(), 1e-5, c["act"], slope,
                            c["has_norm"], p["sign"] if c["affine"] else None, 0.1, 0.5, p["dgamma_old"], p["dbeta_old"],
                            p["dslope_old"], acc, want_dslope=c["act"] == R.ACT_PRELU, variant=variant)
    return (st, stt), (yw, yt), (bw, bt)


@pytest.mark.parametrize("cid,variant,key", [
    ("Resnet9Blocks-odd-b0", "pooled", "mean"), ("Resnet9Blocks-odd-b1", "pooled", "rstd"),
    ("edge-C24-in-lrelu", "pooled", "shift"),
    ("Discriminator96-b7", "biased_running_var", "running_var"), ("SRResNet-odd-b1", "biased_running_var", "running_var"),
    ("edge-bn-prelu-residual", "residual_first", "y"),
    ("SRResNet-odd-b1", "slope_all", "dslope"), ("edge-rows20-bn-prelu", "slope_all", "dslope"),
    ("SRResNet-odd-b0", "slope_all", "dslope"),
    ("Discriminator96-b7", "sign_without_1_over_C", "dgamma"), ("Resnet9Blocks-odd-b0", "sign_without_1_over_C", "dgamma"),
    ("Discriminator96-b7", "no_B_mean", "dx"), ("Resnet9Blocks-odd-b1", "no_B_mean", "dx"),
    ("ConvDiscriminator-b3", "no_B_mean", "dx"),
    ("Discriminator96-b7", "accumulate_ignored", "dgamma"), ("Resnet9Blocks-odd-b0", "accumulate_ignored", "dbeta"),
    ("SRResNet-odd-b0", "accumulate_ignored", "dslope"),
])
def test_norm_mutants_rejected(cid, variant, key):
    c = norm_case(cid)
    (st, stt), (yw, yt), (bw, bt) = _norm_run_refs(c)
    (ms, _), (my, _), (mb, _) = _norm_run_refs(c, variant)
    if key == "y":
        assert rejected(my, yw, yt)
    elif key in st:
        assert rejected(ms[key], st[key], stt[key])
    else:
        assert rejected(mb[key], bw[key], bt[key])


def test_norm_bounds_are_small():
    """The statistics' bounds stay far below what a wrong kernel changes (here: a relative 1e-4 of the values)."""
    for cid in ("Discriminator96-b1", "Resnet9Blocks-odd-b0", "edge-C2048-bn-relu"):
        (st, stt), (yw, yt), (bw, bt) = _norm_run_refs(norm_case(cid))
        for k in ("rstd", "scale"):
            assert float((stt[k] / st[k].abs()).max()) < 1e-4, (cid, k)
        assert float((bt["dx"] - R.bf16_ulp(bw["dx"])).max()) < 1e-3 * float(bw["dx"].abs().max()), cid
