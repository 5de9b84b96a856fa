"""CPU: the float64 references of tests/step_kernel_refs.py against stock torch where one exists (torch.optim.Adam,
torch.nn.utils.spectral_norm, autograd, F.unfold), the Philox4x32-10 port against the Random123 known-answer vectors,
and -- on the seeded inputs of tests/test_gpu_step_kernels.py -- every plausible wrong kernel (a ``variant=`` mutant of
a reference) rejected by the bound the GPU test applies."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from tests import step_kernel_refs as R

U = R.U32


def rejected(got, want, tol):
    """A mutant's result is caught: some element lies outside the bound."""
    return R.max_excess(got, want, tol) > 0


# ============================================================================================== Adam
@pytest.mark.parametrize("wd", [0.0, 1e-2])
def test_adam_ref_is_torch_adam(wd):
    p0, grads = R.adam_grads(1023, 5, seed=1023)
    ref = R.adam_ref(p0, grads, R.ADAM_LR, R.ADAM_BETAS, 1e-8, wd)
    p = torch.nn.Parameter(p0.double().clone())
    # the hyper-parameters as the kernel receives them (fp32)
    opt = torch.optim.Adam([p], lr=R.r32(R.ADAM_LR), betas=tuple(R.r32(b) for b in R.ADAM_BETAS), eps=R.r32(1e-8),
                           weight_decay=R.r32(wd), foreach=False)
    for g, want in zip(grads, ref):
        p.grad = g.double()
        opt.step()
        st = opt.state[p]
        assert torch.allclose(p.detach(), want["p"], rtol=1e-13, atol=1e-15)
        assert torch.allclose(st["exp_avg"], want["m"], rtol=1e-12, atol=1e-300)
        assert torch.allclose(st["exp_avg_sq"], want["v"], rtol=1e-12, atol=1e-300)


def test_adam_ref_resume_is_torch_adam():
    p0, grads = R.adam_grads(64, 4, seed=9)
    p = torch.nn.Parameter(p0.double().clone())
    opt = torch.optim.Adam([p], lr=R.r32(R.ADAM_LR), betas=tuple(R.r32(b) for b in R.ADAM_BETAS), eps=R.r32(1e-8),
                           foreach=False)
    for g in grads[:3]:
        p.grad = g.double()
        opt.step()
    st = opt.state[p]
    want = R.adam_ref(p.detach().clone(), grads[3:], R.ADAM_LR, R.ADAM_BETAS, 1e-8, 0.0, m0=st["exp_avg"].clone(),
                      v0=st["exp_avg_sq"].clone(), step0=3)[0]
    p.grad = grads[3].double()
    opt.step()
    assert torch.allclose(p.detach(), want["p"], rtol=1e-13, atol=1e-15)


@pytest.mark.parametrize("variant,n,wd,gs", [("no_bias_correction", 1023, 0.0, 1.0), ("eps_in_sqrt", 1023, 0.0, 1.0),
                                             ("scale_after_wd", 4099, 1e-2, 0.5), ("step_off_by_one", 1023, 0.0, 1.0),
                                             ("step_off_by_one", 4099, 1e-2, 0.5)])
def test_adam_mutants_rejected(variant, n, wd, gs):
    p0, grads = R.adam_grads(n, 5, seed=n)                  # test_adam_c_abi_against_float64_adam's inputs
    ref = R.adam_ref(p0, grads, R.ADAM_LR, R.ADAM_BETAS, 1e-8, wd, gs)
    mut = R.adam_ref(p0, grads, R.ADAM_LR, R.ADAM_BETAS, 1e-8, wd, gs, variant=variant)
    assert rejected(mut[0]["p"], ref[0]["p"], ref[0]["tp"])          # caught at the first step already


def test_adam_bounds_are_small():
    """The parameter bound stays a small fraction of one update (it must not hide wrong arithmetic)."""
    p0, grads = R.adam_grads(4099, 5, seed=4099)
    ref = R.adam_ref(p0, grads, R.ADAM_LR, R.ADAM_BETAS, 1e-8, 0.0)
    assert float(ref[-1]["tp"].max()) < 1e-3 * R.ADAM_LR + 16 * U * float(ref[-1]["p"].abs().max())


# ============================================================================================== spectral norm
def _torch_sn(W, u, v, training):
    lin = torch.nn.Linear(W.shape[1], W.shape[0], bias=False).double()
    lin = torch.nn.utils.spectral_norm(lin, eps=R.SN_EPS)
    with torch.no_grad():
        lin.weight_orig.copy_(W)
        lin.weight_u.copy_(u)
        lin.weight_v.copy_(v)
    lin.train(training)
    fn = next(h for h in lin._forward_pre_hooks.values() if type(h).__name__ == "SpectralNorm")
    with torch.no_grad():
        w_sn = fn.compute_weight(lin, do_power_iteration=training)
    return lin.weight_u.clone(), lin.weight_v.clone(), w_sn


@pytest.mark.parametrize("update", [1, 0])
def test_sn_power_ref_is_torch_spectral_norm(update):
    dims = [(33, 27), (1, 257), (64, 1024)]
    ws, us, vs = R.sn_inputs(dims, seed=len(dims))
    for W, u, v in zip(ws, us, vs):
        want = R.sn_power_ref(W, u, v, update)
        tu, tv, w_sn = _torch_sn(W.double(), u.double(), v.double(), bool(update))
        assert torch.allclose(want["u"], tu, rtol=1e-12, atol=1e-14)
        assert torch.allclose(want["v"], tv, rtol=1e-12, atol=1e-14)
        assert torch.allclose(W.double() / want["sigma"], w_sn, rtol=1e-12, atol=1e-14)


def test_sn_grad_ref_is_autograd():
    dims = [(33, 27), (7, 5), (64, 1024)]
    ws, us, vs = R.sn_inputs(dims, seed=3)
    G, _ = R.sn_grad_inputs(ws, seed=8)
    for W, u, v, g in zip(ws, us, vs, G):
        sig = float(u.double() @ (W.double() @ v.double()))
        want, _ = R.sn_grad_ref(W, u, v, sig, g)
        assert torch.allclose(want, R.sn_autograd_check(W, u, v, g), rtol=1e-10, atol=1e-12)


def _sn_synth_state():
    from tests.test_gpu_step_kernels import SN_SYNTH
    return SN_SYNTH, R.sn_inputs(SN_SYNTH, seed=len(SN_SYNTH))      # test_sn_power_iteration's synthetic inputs


@pytest.mark.parametrize("variant,key", [("u_not_updated", "u"), ("v_not_normalized", "v")])
def test_sn_power_mutants_rejected(variant, key):
    dims, (ws, us, vs) = _sn_synth_state()
    caught = 0
    for W, u, v in zip(ws, us, vs):
        ref = R.sn_power_ref(W, u, v, 1)
        mut = R.sn_power_ref(W, u, v, 1, variant=variant)
        caught += rejected(mut[key], ref[key], ref["t" + key])
    assert caught == len(dims) - (key == "u") * sum(r == 1 for r, _ in dims)     # a 1-row layer's u is +-1 either way


@pytest.mark.parametrize("variant", ["no_projection", "sigma_squared"])
def test_sn_grad_mutants_rejected(variant):
    from tests.test_gpu_step_kernels import SN_SYNTH
    ws, us, vs = R.sn_inputs(SN_SYNTH, seed=7)                     # test_sn_weight_grad's synthetic inputs
    G, _ = R.sn_grad_inputs(ws, seed=8)
    for W, u, v, g in zip(ws, us, vs, G):
        sig = R.r32(float(u.double() @ (W.double() @ v.double())))
        ref, tol = R.sn_grad_ref(W, u, v, sig, g)
        mut, _ = R.sn_grad_ref(W, u, v, sig, g, variant=variant)
        assert rejected(mut, ref, tol), tuple(W.shape)


# ============================================================================================== loss seeds
def test_hinge_ref_is_autograd():
    real, fake = R.hinge_inputs(1025, seed=1025)
    r, f = real.double().requires_grad_(True), fake.double().requires_grad_(True)
    (F.relu(1 - r).mean() + F.relu(1 + f).mean()).backward()
    losses, dr, df, _ = R.hinge_ref(real, fake, 1.0)
    assert torch.allclose(dr, r.grad, rtol=2 * U, atol=0) and torch.allclose(df, f.grad, rtol=2 * U, atol=0)
    assert bool((dr[real == 1] == 0).all()) and bool((df[fake == -1] == 0).all())   # margin 0: relu'(0) = 0 in torch
    assert abs(float(losses[0]) - float((F.relu(1 - r).mean() + F.relu(1 + f).mean()).detach())) < 1e-12


@pytest.mark.parametrize("B", [1, 5, 1025])
def test_hinge_mutants_rejected(B):
    real, fake = R.hinge_inputs(B, seed=B)
    losses, dr, df, tol = R.hinge_ref(real, fake, 0.37)
    _, mr, mf, _ = R.hinge_ref(real, fake, 0.37, variant="grad_at_zero_margin")
    assert not torch.equal(mr, dr) or not torch.equal(mf, df)       # the gradients are compared bit for bit
    ml, _, _, _ = R.hinge_ref(real, fake, 0.37, variant="unscaled")
    assert rejected(ml, losses, tol)


@pytest.mark.parametrize("kind", R.POINTWISE_KINDS)
@pytest.mark.parametrize("const", [None, "const"])
def test_pointwise_ref_is_autograd(kind, const):
    target = None if const is None else (1.0 if kind == "bce_logits" else 0.25)
    x, y = R.pointwise_inputs(kind, 4099, target, seed=4099)
    loss, dx, _, _ = R.pointwise_ref(kind, x, y, 0.7)
    xd = x.double().requires_grad_(True)
    yd = y.double() if isinstance(y, torch.Tensor) else torch.full_like(xd, R.r32(y))
    fn = {"mse": F.mse_loss, "l1": F.l1_loss, "bce_logits": F.binary_cross_entropy_with_logits}[kind]
    want = fn(xd, yd) * 0.7
    want.backward()
    assert abs(loss - float(want)) <= 1e-12 * max(1.0, abs(float(want)))
    assert torch.allclose(dx, xd.grad, rtol=2 * U, atol=0)
    if kind == "l1":
        assert bool((dx[::4] == 0).all())              # d == 0: sign(0) = 0


@pytest.mark.parametrize("kind,variant", [("l1", "sign_at_tie"), ("mse", "no_factor_two"),
                                          ("bce_logits", "sigmoid_of_minus_x"), ("mse", "sum_not_mean")])
@pytest.mark.parametrize("const", [None, "const"])
def test_pointwise_mutants_rejected(kind, variant, const):
    target = None if const is None else (1.0 if kind == "bce_logits" else 0.25)
    for n in (1, 4099):                                              # as test_pointwise_loss draws them
        x, y = R.pointwise_inputs(kind, n, target, seed=n)
        loss, dx, tl, tdx = R.pointwise_ref(kind, x, y, 0.7)
        ml, mdx, _, _ = R.pointwise_ref(kind, x, y, 0.7, variant=variant)
        if variant == "sum_not_mean":
            assert n == 1 or abs(ml - loss) > tl                    # (sum and mean agree for one element)
        elif kind == "l1":
            assert not torch.equal(mdx, dx)                          # compared bit for bit
        else:
            assert rejected(mdx, dx, tdx)


# ============================================================================================== Philox / randn
@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    got = R.philox4x32_10([np.array([c], np.uint64) for c in ctr], key)
    assert [int(w[0]) for w in got] == list(want)


def test_u01_open_interval_and_float32_steps():
    x = np.array([0, 255, 256, 0xFFFFFFFF, 0x80000000], np.uint64)
    u = R.u01_f32(x)
    assert u.dtype == np.float32
    assert u[0] == u[1] == np.float32(0.5 / 16777216.0)        # the low 8 bits are dropped
    assert u[0] > 0 and u[3] <= 1.0
    assert u[4] == np.float32(0.5 + 0.5 / 16777216.0)


def test_randn_ref_is_standard_normal():
    z, tol, nxt = R.randn_ref(1 << 16, 0x123456789ABCDEF0, 0)
    assert nxt == 1 << 14
    assert abs(float(z.mean())) < 0.02 and abs(float(z.var()) - 1) < 0.02
    assert float(tol.max()) < 1e-5


@pytest.mark.parametrize("n", [1, 3, 5, 128 * 512])
def test_randn_mutants_rejected(n):
    seed = 0x123456789ABCDEF0                                     # test_randn_against_philox_box_muller's inputs
    want, tol, nxt = R.randn_ref(n, seed, 0)
    swapped, _, _ = R.randn_ref(n, seed, 0, variant="swap_sin_cos")
    assert rejected(swapped, want, tol)
    _, _, mut_next = R.randn_ref(n, seed, 0, variant="counter_by_n")
    second, tol2, _ = R.randn_ref(n, seed, nxt)
    wrong_second, _, _ = R.randn_ref(n, seed, mut_next)
    assert mut_next != nxt or n < 4
    if mut_next != nxt:
        assert rejected(wrong_second, second, tol2)


# ============================================================================================== column sums
@pytest.mark.parametrize("rows,ncols,stride", [(7, 40, 72), (1000, 64, 64)])
def test_colsum_mutant_rejected(rows, ncols, stride):
    g = torch.Generator().manual_seed(rows * 7 + ncols)             # test_colsum_partials' inputs
    x = torch.randn(rows, stride, generator=g)
    old = torch.randn(ncols, generator=g) * 50
    want, tol = R.colsum_ref(x, ncols, old, 1, 0.75, depth=rows / 8 + 9)
    assert torch.allclose(want, old.double() + 0.75 * x.double()[:, :ncols].sum(0))
    mut, _ = R.colsum_ref(x, ncols, old, 1, 0.75, depth=rows / 8 + 9, variant="accumulate_ignored")
    assert rejected(mut, want, tol)


# ============================================================================================== BatchNorm
def test_bn_finalize_ref_is_batchnorm():
    x, _, p = R.bn_inputs(24, 333, seed=24 * 7919 + 333)
    bn = torch.nn.BatchNorm1d(24).double()
    with torch.no_grad():
        bn.weight.copy_(p["gamma"])
        bn.bias.copy_(p["beta"])
        bn.running_mean.copy_(p["running_mean"])
        bn.running_var.copy_(p["running_var"])
    bn.momentum = R.r32(0.1)
    bn.eps = R.r32(1e-5)
    X = x.double()
    y = bn.train()(X)
    part = torch.stack([X.sum(0), (X * X).sum(0)]).view(1, 2, -1)
    want, _ = R.bn_finalize_ref(part, 333, p["gamma"], p["beta"], 1e-5, 0.1, p["running_mean"], p["running_var"])
    assert torch.allclose(X * want["scale"] + want["shift"], y, rtol=1e-10, atol=1e-10)
    assert torch.allclose(want["running_mean"], bn.running_mean, rtol=1e-10, atol=1e-12)
    assert torch.allclose(want["running_var"], bn.running_var, rtol=1e-10, atol=1e-12)


@pytest.mark.parametrize("C,rows", [(256, 64), (64, 5 * 1024), (24, 333)])
def test_bn_mutants_rejected(C, rows):
    x, dy, p = R.bn_inputs(C, rows, seed=C * 7919 + rows)          # test_batchnorm_finalize_apply_backward's inputs
    stats = R.bn_stats_partials(x, 4)
    args = (stats, rows, p["gamma"], p["beta"], 1e-5, 0.1, p["running_mean"], p["running_var"])
    want, tol = R.bn_finalize_ref(*args)
    mut, _ = R.bn_finalize_ref(*args, variant="biased_running_var")
    assert rejected(mut["running_var"], want["running_var"], tol["running_var"])
    scale, shift = want["scale"].float(), want["shift"].float()
    mean, rstd = want["mean"], want["rstd"]
    del mean, rstd
    bw = R.bn_bwd_ref(dy, x, scale, shift, p["gamma"], p["beta"], 1e-5, rows, p["sign"], 0.1, 0.5,
                      p["dgamma_old"], p["dbeta_old"], 0)
    mw = R.bn_bwd_ref(dy, x, scale, shift, p["gamma"], p["beta"], 1e-5, rows, p["sign"], 0.1, 0.5,
                      p["dgamma_old"], p["dbeta_old"], 0, variant="sign_without_1_over_C")
    assert rejected(mw[1], bw[1], bw[4])


def test_bn_bwd_ref_without_mask_is_plain_batchnorm_backward():
    x, dy, p = R.bn_inputs(8, 1000, seed=8 * 7919 + 1000)
    big = torch.full((8,), 1e30)
    dx, dg, db, _, _, _ = R.bn_bwd_ref(dy, x, torch.zeros(8), big, p["gamma"], p["beta"], 1e-5, 1000)
    X, G = x.double(), dy.double()
    mu, var = X.mean(0), X.var(0, unbiased=False)
    rs = 1 / torch.sqrt(var + R.r32(1e-5))
    xh = (X - mu) * rs
    want = p["gamma"].double() * rs / 1000 * (1000 * G - G.sum(0) - xh * (G * xh).sum(0))
    assert torch.allclose(dx, want, rtol=1e-9, atol=1e-12)
    assert torch.allclose(dg, (G * xh).sum(0)) and torch.allclose(db, G.sum(0))


# ============================================================================================== final GEMV
def test_dfc_refs_are_autograd():
    a, w, dlogit, perm, dw_old = R.dfc_inputs(5, 8192, seed=8192 + 5)
    pre = a.double().clone().requires_grad_(True)
    wd = w.double().clone().requires_grad_(True)
    logits = F.leaky_relu(pre, 0.1) @ wd / 1.7 + 0.3          # a >= 0 or a < 0: lrelu' is 1 or slope, as at a
    logits.backward(dlogit.double())
    want, _ = R.dfc_fwd_ref(a, w, torch.tensor(1.7), torch.tensor(0.3))
    d, _ = R.dfc_bwd_data_ref(a, w, torch.tensor(1.7), dlogit, 0.1)
    assert torch.allclose(d * torch.where(a.double() > 0, 1.0, 1.0), pre.grad, rtol=1e-7, atol=1e-12)
    dw, _, _, _ = R.dfc_bwd_weight_ref(F.leaky_relu(a.double(), 0.1), dlogit, dw_old, 0)
    assert torch.allclose(dw / 1.7, wd.grad, rtol=1e-10, atol=1e-12)
    assert torch.allclose(want, F.leaky_relu(a.double(), 0.1) @ w.double() / 1.7 + 0.3 + (a.double() @ w.double() -
                          F.leaky_relu(a.double(), 0.1) @ w.double()) / 1.7)


@pytest.mark.parametrize("B,K", [(1, 8192), (512, 32768)])
def test_dfc_mutant_rejected(B, K):
    a, w, dlogit, perm, dw_old = R.dfc_inputs(B, K, seed=K + B)     # test_dfc_forward_backward's inputs
    want, tol, _, _ = R.dfc_bwd_weight_ref(a, dlogit, dw_old, 1, perm)
    mut, _, _, _ = R.dfc_bwd_weight_ref(a, dlogit, dw_old, 1, perm, variant="accumulate_ignored")
    assert rejected(mut, want, tol)


# ============================================================================================== im2col3 / col2im3
def test_im2col3_ref_is_unfold():
    x = torch.randn(2, 3, 9, 33)
    got = R.im2col3_ref(x)
    cols = F.unfold(x.double(), 3, padding=1).view(2, 3, 3, 3, 9, 33)       # (b, c, kh, kw, h, w)
    want = torch.zeros(2, 9, 33, 32, dtype=torch.float64)
    want[..., :27] = cols.permute(0, 4, 5, 2, 3, 1).reshape(2, 9, 33, 27)   # k = (kh*3+kw)*3 + c
    assert torch.equal(got, want)


def test_col2im3_ref_is_conv_transpose():
    """Folding taps T = a W (per pixel) in col2im3's order is conv_transpose2d(a, W, padding=1)."""
    torch.manual_seed(0)
    a = torch.randn(2, 64, 9, 13, dtype=torch.float64)
    W = torch.randn(64, 3, 3, 3, dtype=torch.float64)
    T = torch.zeros(2, 9, 13, 32, dtype=torch.float64)
    T[..., :27] = torch.einsum("bkhw,kcij->bhwijc", a, W).reshape(2, 9, 13, 27)
    got = R.col2im3_ref_f32(T, False).double()
    want = F.conv_transpose2d(a, W, padding=1)
    assert torch.allclose(got, want, rtol=1e-4, atol=1e-4)


def test_adam_moment_bound_covers_fp32_weight_decay_roundings():
    """With weight decay, g*s and wd*p can nearly cancel; the kernel rounds one or both products before the add (or
    fuses one of them into it), so exp_avg's error scales with |g s| + |wd p|, not with |g'|.  Every such fp32
    evaluation order of the first step stays within the bound the GPU test applies."""
    p0, grads = R.adam_grads(4099, 1, seed=4099)
    g, p = grads[0].numpy(), p0.numpy()
    wd, gs = np.float32(1e-2), np.float32(0.5)
    g[:64] = -(wd * p[:64]).astype(np.float32) / gs * (1 + np.linspace(-1e-3, 1e-3, 64)).astype(np.float32)
    want = R.adam_ref(torch.from_numpy(p), [torch.from_numpy(g)], R.ADAM_LR, R.ADAM_BETAS, 1e-8, 1e-2, 0.5)[0]
    f64 = np.float64
    gsp, wdp = (g * gs).astype(np.float32), (wd * p).astype(np.float32)
    orders = [(gsp + wdp).astype(np.float32),                                   # both products rounded
              (g.astype(f64) * f64(gs) + wdp.astype(f64)).astype(np.float32),   # fma(g, s, fl(wd p))
              (wd.astype(f64) * p.astype(f64) + gsp.astype(f64)).astype(np.float32)]   # fma(wd, p, fl(g s))
    for gk in orders:
        m = (np.float32(0.5) * gk).astype(np.float32)
        assert R.max_excess(torch.from_numpy(m), want["m"], want["tm"]) <= 0
