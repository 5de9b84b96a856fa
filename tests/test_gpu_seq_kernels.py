"""GPU: the SRGAN / CycleGAN layer kernels (csrc/layers.cu) and the single-tap GEMM plans seqnet.py builds on the
tcgen05 GEMM and weight-gradient kernels, each called as seqnet.py calls it, against the float64 references of
tests/seq_kernel_refs.py, at every layer shape of SRResNet / Discriminator96 (16 x 3 x 24 x 24, D at 96 x 96),
Resnet9Blocks / ConvDiscriminator (1 x 3 x 128 x 128) and of the generators at 3 x 3 x 20 x 22.

Copies (im2col, layout changes, pixel shuffle) are bit-exact.  Sums are bit-exact on integer-valued operands in
{-2..2}, where every partial sum stays below 2^20 so that fp32 adds exactly in any order and split; on real operands
each element stays within a bound derived from the kernel's fp32 arithmetic.  Every launch runs twice and must give
bit-identical results.  Output buffers carry sentinel rows or guard floats that must survive.  The bounded checks
print their largest error / bound ratio ("ratio <family> <value>")."""
import ctypes
import zlib

import pytest
import torch
import torch.nn.functional as F

from tests import seq_kernel_refs as R

pytestmark = pytest.mark.gpu

U = R.U32
SENT_BF16 = -7.25                   # sentinel rows after M (exact in bf16)
NAN = float("nan")                  # every output element a launch must write starts as NaN (or the sentinel)
GUARD = 123.5


def _lib():
    from ipr_gan_b200._lib import lib
    return lib()


def _check(rc, what):
    from ipr_gan_b200._lib import check
    check(rc, what)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _st():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def seed(cid, tag):
    return zlib.crc32(("%s/%s" % (cid, tag)).encode())


def bits_equal(a, b):
    return a.shape == b.shape and torch.equal(a.reshape(-1).view(torch.uint8), b.reshape(-1).view(torch.uint8))


def within(got, want, tol, what):
    """Elementwise |got - want| <= tol; prints the largest ratio error / bound."""
    err = (R.d64(got).to(want.device) - want).abs()
    tol = torch.as_tensor(tol, dtype=torch.float64, device=want.device).expand_as(err)
    zero = torch.where(err > 0, float("inf"), 0.0)
    ratio = float(torch.where(tol > 0, err / tol.clamp_min(1e-300), zero).max()) if err.numel() else 0.0
    print("ratio %s %.4g" % (what.split(" ")[0], ratio))
    ex = float((err - tol).max())
    assert ex <= 0, "%s: exceeds its bound by %.3g (ratio %.3g)" % (what, ex, ratio)


def exact(got, want, what):
    """got (bf16 / fp32) equals the float64 ``want`` rounded once (RNE) to got's dtype."""
    w = want.to(got.dtype) if got.dtype == torch.float32 else want.float().to(got.dtype)
    assert bits_equal(got, w), "%s: %d elements differ" % (what, int((got.double() != w.double()).sum()))


CASES = R.net_cases()
IDS = [c["id"] for c in CASES]


def _case(request_id):
    return next(c for c in CASES if c["id"] == request_id)


# ============================================================================================== patch matrix
def _im2col(x, b, oh, ow):
    n, h, w, c = x.shape
    M = n * oh * ow
    buf = torch.full((M + 3, b.kp), SENT_BF16, device="cuda", dtype=torch.bfloat16)
    _check(_lib().ipr_im2col_nhwc_bf16(_p(x), _p(buf), n, h, w, c, oh, ow, b.k, b.stride, b.pad, b.up, b.reflect, b.kp,
                                       _st()), "ipr_im2col_nhwc_bf16")
    return buf


@pytest.mark.parametrize("cid", IDS)
def test_im2col(cid):
    c = _case(cid)
    b, (oh, ow) = c["block"], c["ohw"]
    for integer in (True, False):
        x, _, _, _ = R.conv_inputs(c, integer, seed(cid, "conv%d" % integer))
        x = x.cuda()
        bufs = [_im2col(x, b, oh, ow) for _ in range(2)]
        torch.cuda.synchronize()
        assert bits_equal(bufs[0], bufs[1])
        M = x.shape[0] * oh * ow
        assert bool((bufs[0][M:] == SENT_BF16).all()), "rows past M written"
        exact(bufs[0][:M], R.im2col_ref(x, b, oh, ow), "im2col")


@pytest.mark.parametrize("cid", [c["id"] for c in CASES if c["dgrad"]])
def test_col2im(cid):
    c = _case(cid)
    b, shape, (oh, ow) = c["block"], c["shape"], c["ohw"]
    n, h, w, cp = shape
    M = n * oh * ow
    for integer in (True, False):
        dcol = R.dcol_inputs(M, b.kp, integer, seed(cid, "dcol%d" % integer)).cuda()
        gen = torch.Generator().manual_seed(seed(cid, "addend"))
        addend = (R.int_bf16(shape, gen) if integer else torch.randn(shape, generator=gen).to(torch.bfloat16)).cuda()
        for add in (None, addend):
            outs = []
            for _ in range(2):
                dx = torch.full(shape, NAN, device="cuda", dtype=torch.bfloat16)
                _check(_lib().ipr_col2im_nhwc_bf16(_p(dcol), _p(dx), _p(add), n, h, w, cp, oh, ow, b.k, b.stride, b.pad,
                                                   b.up, b.reflect, b.kp, _st()), "ipr_col2im_nhwc_bf16")
                outs.append(dx)
            torch.cuda.synchronize()
            assert bits_equal(outs[0], outs[1])
            want = R.col2im_ref(dcol, b, shape, oh, ow, add)
            if integer:
                exact(outs[0], want, "col2im integer addend=%s" % (add is not None))
            else:
                within(outs[0], want, R.col2im_bound(dcol, b, shape, oh, ow, add), "col2im addend=%s" % (add is not None))


# ============================================================================================== GEMMs
def _run_twice(fn):
    a, b = fn(), fn()
    torch.cuda.synchronize()
    assert bits_equal(a, b), "two launches differ"
    return a


@pytest.mark.parametrize("cid", IDS)
def test_gemms(cid):
    """Forward (EPI_BIAS_LRELU at slope 1 / EPI_LINEAR_F32 for a final layer), data gradient (EPI_LINEAR) and weight
    gradient (split-K + element-major reduce through the block's row_map / col_off) of one block, with the plans,
    weight layouts and bias vector as seqnet.NetPlans builds them."""
    from ipr_gan_b200 import dense
    c = _case(cid)
    b, (n, h, w, cp), (oh, ow) = c["block"], c["shape"], c["ohw"]
    M = n * oh * ow
    wshape = tuple(b.conv.weight.shape)
    fwd_plan = dense.Plan("linear", b.kp, b.n_p)
    dg_plan = dense.Plan("linear", b.n_p, (b.kp + 15) // 16 * 16)
    off, s_n, row_map = b.wgrad_tables()
    wg_plan = dense.WGradPlan(dense.Plan("linear", b.kp, b.n_p), wshape, row_perm=row_map, col_off=off, s_n=s_n)
    total_kb = -(-M // 64)
    split_set = [1, 2, None, R.empty_last_split(total_kb)]
    for integer in (True, False):
        x, wt, bias, dy = R.conv_inputs(c, integer, seed(cid, "conv%d" % integer))
        x, dy = x.cuda(), dy.cuda()
        col = _im2col(x, b, oh, ow)[:M]
        wp = b.fwd_layout(wt).to(torch.bfloat16).cuda()
        bias_p = R.padded_bias(b, bias).cuda() if (bias is not None and not b.final) else None
        # ---- forward, into a view of a larger buffer whose rows past M hold sentinels
        f32 = b.final
        big = torch.full((M + 130, b.n_p), SENT_BF16, device="cuda", dtype=torch.float32 if f32 else torch.bfloat16)

        def fwd():
            big.fill_(SENT_BF16)                    # a column or row the launch does not write keeps the sentinel
            out = big[:M].view(M, 1, 1, b.n_p)
            if f32:
                fwd_plan.run(col.view(M, 1, 1, b.kp), wp, epi=dense.EPI_LINEAR_F32, n_valid=b.n_p, out=out)
            else:
                fwd_plan.run(col.view(M, 1, 1, b.kp), wp, epi=dense.EPI_BIAS_LRELU, slope=1.0, bias=bias_p,
                             n_valid=b.n_p, out=out)
            return big.clone()

        got = _run_twice(fwd)
        assert bool((got[M:] == SENT_BF16).all()), "forward wrote rows past M"
        y = got[:M]
        assert bool((y[:, b.cout:] == 0).all()), "padding output channels not zero"
        want = R.gemm_ref(col, wp[0], bias_p)
        if integer:
            exact(y, want, "forward")
        else:
            within(y, want, R.gemm_bound(col, wp[0], want, bf16_out=not f32), "gemm-forward %s" % cid)
        # ---- data gradient
        if c["dgrad"]:
            dwp = b.dgrad_layout(wt).to(torch.bfloat16).cuda()                     # [1][kp][n_p]
            dbig = torch.full((M + 130, dg_plan.cout), SENT_BF16, device="cuda", dtype=torch.bfloat16)

            def dgrad():
                dbig.fill_(SENT_BF16)
                dg_plan.run(dy.view(M, 1, 1, b.n_p), dwp, out=dbig[:M].view(M, 1, 1, dg_plan.cout))
                return dbig.clone()

            got = _run_twice(dgrad)
            assert bool((got[M:] == SENT_BF16).all()), "data gradient wrote rows past M"
            want = R.gemm_ref(dy, dwp[0])
            if integer:
                exact(got[:M], want, "data gradient")
            else:
                within(got[:M], want, R.gemm_bound(dy, dwp[0], want), "gemm-dgrad %s" % cid)
        # ---- weight gradient: accumulate=True, scale=0.5 over old values; guard floats after the gradient
        old = R.wgrad_old(wshape, integer, seed(cid, "old"))
        want, tol = R.wgrad_ref(dy, col, wshape, row_map, off, s_n, old.cuda(), True, 0.5)
        numel = old.numel()
        for splits in sorted(set(split_set), key=lambda s: -1 if s is None else s):
            if splits is not None and splits > 4 * total_kb + 1:
                continue

            def wgrad():
                buf = torch.full((numel + 64,), GUARD, device="cuda")
                buf[:numel] = old.view(-1).cuda()
                wg_plan.run(dy.view(M, 1, 1, b.n_p), col.view(M, 1, 1, b.kp), buf[:numel].view(wshape), accumulate=True,
                            scale=0.5, splits=splits)
                return buf

            buf = _run_twice(wgrad)
            assert bool((buf[numel:] == GUARD).all()), "guard floats after grad written"
            g = buf[:numel].view(wshape)
            if integer:
                exact(g, want, "weight gradient splits=%s" % splits)
            else:
                within(g, want, tol, "gemm-wgrad %s splits=%s" % (cid, splits))

        # ---- weight gradient without accumulate into a NaN-filled gradient: every element is written
        def wgrad_overwrite():
            buf = torch.full((numel + 64,), GUARD, device="cuda")
            buf[:numel] = NAN
            wg_plan.run(dy.view(M, 1, 1, b.n_p), col.view(M, 1, 1, b.kp), buf[:numel].view(wshape), scale=0.5)
            return buf

        buf = _run_twice(wgrad_overwrite)
        assert bool((buf[numel:] == GUARD).all()), "guard floats after grad written"
        want, tol = R.wgrad_ref(dy, col, wshape, row_map, off, s_n, None, False, 0.5)
        if integer:
            exact(buf[:numel].view(wshape), want, "weight gradient accumulate=False")
        else:
            within(buf[:numel].view(wshape), want, tol, "gemm-wgrad %s accumulate=False" % cid)


# ============================================================================================== norms
def _norm_run(c, x, res, p, sc_in=None, sh_in=None):
    G, rows, C = c["groups"], c["rows"], c["C"]
    dev = "cuda"
    gamma = p["gamma"] if c["affine"] else None
    beta = p["beta"] if c["affine"] else None
    rm = p["running_mean"].clone() if (c["bn"] and c["has_norm"] == 1) else None
    rv = p["running_var"].clone() if (c["bn"] and c["has_norm"] == 1) else None
    nbt = torch.zeros((), dtype=torch.int64, device=dev) if rm is not None else None
    if c["has_norm"] == 2:
        scale, shift = sc_in.clone(), sh_in.clone()
        mean = rstd = None
    elif c["has_norm"] == 0:
        scale = shift = mean = rstd = None
    else:
        scale, shift, mean, rstd = (torch.full((G, C), NAN, device=dev) for _ in range(4))
    nbytes = _lib().ipr_norm_workspace_bytes(G, C)
    ws = torch.empty(nbytes // 4, device=dev)
    y = torch.full((G * rows, C), NAN, device=dev, dtype=torch.bfloat16)
    slope_ptr = p["slope"] if c["act"] == R.ACT_PRELU else None
    _check(_lib().ipr_norm_fwd_bf16(_p(x), _p(y), _p(res if c["residual"] else None), G, rows, C, c["has_norm"], 1e-5, 0.1,
                                    _p(gamma), _p(beta), _p(rm), _p(rv), _p(nbt), _p(scale), _p(shift), _p(mean), _p(rstd),
                                    c["act"], float(c["slope"]), _p(slope_ptr), _p(ws), nbytes, _st()), "ipr_norm_fwd_bf16")
    return {"y": y, "scale": scale, "shift": shift, "mean": mean, "rstd": rstd, "running_mean": rm, "running_var": rv,
            "nbt": nbt}


def _norm_bwd(c, dy, x, f, p, acc, mixed):
    G, rows, C = c["groups"], c["rows"], c["C"]
    affine = c["affine"]
    dg = p["dgamma_old"].clone() if affine else None
    db = p["dbeta_old"].clone() if affine else None
    prelu = c["act"] == R.ACT_PRELU
    dsl = (torch.zeros(1, device="cuda") if mixed else p["dslope_old"].clone()) if prelu else None
    nbytes = _lib().ipr_norm_workspace_bytes(G, C)
    ws = torch.empty(nbytes // 4, device="cuda")
    dx = torch.full_like(x, NAN)
    norm = c["has_norm"] == 1
    _check(_lib().ipr_norm_bwd_bf16(_p(dy), _p(x), _p(dx), G, rows, C, int(norm), _p(p["gamma"] if affine else None),
                                    _p(f["scale"] if norm else None), _p(f["shift"] if norm else None),
                                    _p(f["mean"] if norm else None), _p(f["rstd"] if norm else None), _p(dg), _p(db), acc,
                                    _p(p["sign"] if affine else None), 0.1, 0.5, c["act"], float(c["slope"]),
                                    _p(p["slope"] if prelu else None), _p(dsl), _p(ws), nbytes, _st()), "ipr_norm_bwd_bf16")
    return {"dx": dx, "dgamma": dg, "dbeta": db, "dslope": dsl}


def _norm_cases():
    return R.norm_cases() + R.norm_edges(sms() if torch.cuda.is_available() else 148)


@pytest.mark.parametrize("cid", [c["id"] for c in _norm_cases()])
def test_norm_fwd_bwd(cid):
    c = next(c for c in _norm_cases() if c["id"] == cid)
    G, rows, C = c["groups"], c["rows"], c["C"]
    x, dy, res, p = R.norm_inputs(c, seed(cid, "norm"), c.get("mean", 0.4), c.get("std", 1.3))
    x, dy, res = x.cuda(), dy.cuda(), res.cuda()
    p = {k: v.cuda() for k, v in p.items()}
    slope = float(p["slope"]) if c["act"] == R.ACT_PRELU else c["slope"]
    sc_in = sh_in = None
    if c["has_norm"] == 2:
        gen = torch.Generator().manual_seed(seed(cid, "eval"))
        sc_in = (torch.rand(1, C, generator=gen) + 0.5).cuda()
        sh_in = torch.randn(1, C, generator=gen).cuda()
    runs = [_norm_run(c, x, res, p, sc_in, sh_in) for _ in range(2)]
    torch.cuda.synchronize()
    for k, v in runs[0].items():
        if v is not None:
            assert bits_equal(v, runs[1][k]), k
    f = runs[0]
    if c["has_norm"] == 1:
        st, tol = R.norm_stats_ref(x, G, rows, p["gamma"] if c["affine"] else None, p["beta"] if c["affine"] else None,
                                   1e-5, 0.1, p["running_mean"] if c["bn"] else None,
                                   p["running_var"] if c["bn"] else None, sms=sms())
        for k in ("mean", "rstd", "scale", "shift") + (("running_mean", "running_var") if c["bn"] else ()):
            within(f[k], st[k], tol[k], "norm-stats-%s %s" % (k, cid))
        if c["bn"]:
            assert int(f["nbt"]) == 1
        if c.get("mean", 0.4) > 10:
            # what PyTorch's own InstanceNorm makes of the same bf16 input, next to the kernel
            X = x.float().view(G, rows, C)
            tv = torch.var(X, 1, unbiased=False)
            ref_r = st["rstd"]
            print("mean/std=100: rstd rel err kernel %.3g, torch fp32 variance %.3g" % (
                float(((R.d64(f["rstd"]) - ref_r).abs() / ref_r).max()),
                float(((1 / torch.sqrt(tv.double() + R.r32(1e-5)) - ref_r).abs() / ref_r).max())))
    scale = f["scale"] if c["has_norm"] else None
    yw, yt = R.norm_act_ref(x, G, rows, scale, f["shift"] if c["has_norm"] else None, c["act"], slope,
                            res if c["residual"] else None)
    within(f["y"], yw, yt, "norm-apply %s" % cid)
    if c["has_norm"] == 2:
        return                                    # eval mode has no backward on the training path
    for acc, mixed in ((0, False), (1, False), (1, True)):
        if mixed and c["act"] != R.ACT_PRELU:
            continue
        outs = [_norm_bwd(c, dy, x, f, p, acc, mixed) for _ in range(2)]
        torch.cuda.synchronize()
        for k, v in outs[0].items():
            if v is not None:
                assert bits_equal(v, outs[1][k]), k
        o = outs[0]
        dslope_old = torch.zeros(1, device="cuda") if mixed else p["dslope_old"]
        bw, bt = R.norm_bwd_ref(dy, x, G, rows, p["gamma"] if c["affine"] else None, f["scale"], f["shift"], 1e-5,
                                c["act"], slope, c["has_norm"], p["sign"] if c["affine"] else None, 0.1, 0.5,
                                p["dgamma_old"], p["dbeta_old"], dslope_old, acc, want_dslope=c["act"] == R.ACT_PRELU,
                                sms=sms())
        for k in bw:
            within(o[k].view(-1) if k == "dslope" else o[k], bw[k].to(o[k].device).view(-1) if k == "dslope" else bw[k],
                   bt[k].to(o[k].device).view(-1) if k == "dslope" else bt[k],
                   "norm-bwd-%s %s acc=%d mixed=%d" % (k, cid, acc, mixed))


# ============================================================================================== layout kernels
LAYOUT_SHAPES = [(16, 3, 96, 96, 16), (16, 3, 24, 24, 8), (1, 3, 128, 128, 8), (1, 3, 128, 128, 16), (3, 3, 20, 22, 8),
                 (3, 3, 20, 24, 16), (2, 64, 5, 7, 64)]


@pytest.mark.parametrize("n,c,h,w,cp", LAYOUT_SHAPES)
def test_nchw_to_nhwc(n, c, h, w, cp):
    gen = torch.Generator().manual_seed(n * 1000 + c * 100 + h + cp)
    x = (torch.randn(n, c, h, w, generator=gen) * 3).cuda()
    t = torch.tanh(torch.randn(n, c, h, w, generator=gen) * 2).cuda()
    for tanh_out in (None, t):
        def run():
            y = torch.full((n, h, w, cp), SENT_BF16, device="cuda", dtype=torch.bfloat16)
            _check(_lib().ipr_nchw_to_nhwc_bf16(_p(x), _p(tanh_out), _p(y), n, c, h, w, cp, _st()), "ipr_nchw_to_nhwc_bf16")
            return y
        y = _run_twice(run)
        assert bool((y[..., c:] == 0).all()), "padding channels not zero"
        if tanh_out is None:
            assert bits_equal(y[..., :c], x.permute(0, 2, 3, 1).to(torch.bfloat16))
        else:
            X, T = R.d64(x), R.d64(t)
            want = (X * (1 - T * T)).permute(0, 2, 3, 1)
            # 1 - t^2 (two roundings, or one under FMA contraction), the product, then bf16
            within(y[..., :c], want, R.bf16_ulp(want) + 4 * U * X.abs().permute(0, 2, 3, 1) * (1 + T * T).permute(0, 2, 3, 1),
                   "nchw_to_nhwc-tanh")


@pytest.mark.parametrize("n,c,h,w,ld", [(16, 3, 96, 96, 16), (1, 3, 128, 128, 16), (3, 3, 20, 24, 16), (2, 5, 7, 9, 8)])
def test_finish_nchw(n, c, h, w, ld):
    gen = torch.Generator().manual_seed(n + c + h + w + ld)
    t = (torch.randn(n * h * w, ld, generator=gen) * 2).cuda()
    bias = torch.randn(c, generator=gen).cuda()
    for b_, tanh_out in ((bias, 0), (None, 0), (bias, 1)):
        def run():
            out = torch.full((n, c, h, w), NAN, device="cuda")
            _check(_lib().ipr_finish_nchw_f32(_p(t), _p(b_), _p(out), n, c, h, w, ld, tanh_out, _st()), "ipr_finish_nchw_f32")
            return out
        out = _run_twice(run)
        v = t.view(n, h, w, ld)[..., :c].permute(0, 3, 1, 2)
        if b_ is not None:
            v = v + b_.view(1, -1, 1, 1)                    # one fp32 add, as the kernel's
        if not tanh_out:
            assert bits_equal(out, v.contiguous())
        else:
            want = torch.tanh(R.d64(v))
            within(out, want, 4 * U * want.abs() + 2 ** -126, "finish_nchw-tanh")


@pytest.mark.parametrize("n,h,w,c", [(16, 24, 24, 64), (16, 48, 48, 64), (3, 20, 22, 64), (3, 40, 44, 64), (2, 3, 5, 8)])
def test_pixel_shuffle2(n, h, w, c):
    gen = torch.Generator().manual_seed(n * h * w + c)
    x = torch.randn(n, h, w, 4 * c, generator=gen).to(torch.bfloat16).cuda()

    def run(src, inverse, shape):
        y = torch.full(shape, NAN, device="cuda", dtype=torch.bfloat16)
        _check(_lib().ipr_pixel_shuffle2_nhwc_bf16(_p(src), _p(y), n, h, w, c, inverse, _st()), "ipr_pixel_shuffle2_nhwc_bf16")
        return y

    y = _run_twice(lambda: run(x, 0, (n, 2 * h, 2 * w, c)))
    assert bits_equal(y, F.pixel_shuffle(x.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1).contiguous())
    z = torch.randn(n, 2 * h, 2 * w, c, generator=gen).to(torch.bfloat16).cuda()
    back = _run_twice(lambda: run(z, 1, (n, h, w, 4 * c)))
    assert bits_equal(back, F.pixel_unshuffle(z.permute(0, 3, 1, 2), 2).permute(0, 2, 3, 1).contiguous())


@pytest.mark.parametrize("numel", [8, 16 * 24 * 24 * 64, 3 * 20 * 22 * 64 + 8, 1 * 32 * 32 * 256])
def test_add_bf16(numel):
    gen = torch.Generator().manual_seed(numel)
    a = torch.randn(numel, generator=gen).to(torch.bfloat16).cuda()
    b = (torch.randn(numel, generator=gen) * 0.01).to(torch.bfloat16).cuda()

    def run():
        out = torch.full_like(a, NAN)
        _check(_lib().ipr_add_bf16(_p(a), _p(b), _p(out), numel, _st()), "ipr_add_bf16")
        return out
    assert bits_equal(_run_twice(run), (a.float() + b.float()).to(torch.bfloat16))
