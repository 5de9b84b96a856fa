"""Float64 restatements of the contracts of the training step's non-GEMM kernels (csrc/optim.cu, sn.cu, step_misc.cu,
nn_misc.cu), written from the reference semantics (torch.optim.Adam, torch.nn.utils.spectral_norm, the hinge / pointwise
losses, Random123's Philox4x32-10, BatchNorm) rather than from the kernels.  Every function takes the fp32 / bf16 values
the kernel sees and returns float64 results, plus -- where a GPU test needs one -- an elementwise error bound derived from
the kernel's fp32 arithmetic.

Also here: the seeded inputs of tests/test_gpu_step_kernels.py, so that tests/test_step_kernels_host.py can show on the
very same numbers that each bound rejects plausible wrong kernels (the ``variant=`` mutants)."""
import math

import numpy as np
import torch
import torch.nn.functional as F

U32 = 2.0 ** -24            # unit roundoff of fp32 (round to nearest)
f32 = np.float32


def r32(x):
    """A Python / float64 value rounded to the fp32 the kernel receives (ctypes c_float arguments)."""
    return float(f32(x))


def d64(t):
    """float64 copy on the tensor's own device (the large references run on the GPU in float64)."""
    return t.detach().to(torch.float64)


def sum_bound(abs_sum, depth):
    """Error bound of an fp32 sum whose longest chain of dependent additions is ``depth``: depth * u * sum |terms|
    (Higham's gamma_depth, to first order)."""
    return 1.01 * depth * U32 * abs_sum


def block_sum_depth(serial):
    """Longest addition chain of a per-thread serial loop of ``serial`` steps followed by ``ipr_block_sum`` (a warp
    butterfly of 5 levels, then one over at most 32 warp results: 5 more)."""
    return serial + 10


def bf16_ulp(x):
    """Spacing of bf16 numbers at |x| (8 significant bits); 0 where x == 0."""
    x = torch.as_tensor(x, dtype=torch.float64).abs()
    e = torch.floor(torch.log2(torch.where(x > 0, x, torch.ones_like(x))))
    return torch.where(x > 0, torch.exp2(e - 7), torch.zeros_like(x))


def max_excess(got, want, tol):
    """max over elements of |got - want| - tol (<= 0: every element within its bound)."""
    return float((d64(got) - d64(want)).abs().sub(torch.as_tensor(tol, dtype=torch.float64)).max())


# ================================================================================================ Adam
ADAM_LR, ADAM_BETAS = 2e-4, (0.5, 0.999)          # the reference DCGAN's optimiser settings


def adam_grads(n, steps, seed):
    """Parameters and a gradient sequence: gradient magnitudes spread over 10^-7 .. 1 so that eps matters for some
    elements (it decides between sqrt(v) + eps and sqrt(v + eps))."""
    g = torch.Generator().manual_seed(seed)
    p = torch.randn(n, generator=g)
    mag = torch.pow(10.0, -7.0 * torch.rand(n, generator=g))
    grads = [torch.randn(n, generator=g) * mag for _ in range(steps)]
    return p, grads


def adam_ref(p0, grads, lr, betas, eps, wd, grad_scale=1.0, variant=None, m0=None, v0=None, step0=0):
    """torch.optim.Adam (L2 weight decay, no amsgrad) in float64 with the fp32 hyper-parameters the kernel receives.
    ``m0`` / ``v0`` / ``step0``: a resumed state.  -> list over steps of dicts p / m / v and the error bounds
    tp / tm / tv of the fp32 kernel.

    Bounds (elementwise, carried from step to step and doubled when reported):
      g' = g*s + wd*p: the kernel may round g*s and wd*p before the add (or fuse either into it), so its error is
         e_g = 2 u (|g s| + |wd p|), relative to the terms, not to g' (they can cancel), plus wd times p's own error;
      m = b1 m + (1-b1) g': e_m <- b1 e_m + (1-b1) e_g + 3 u (b1 |m| + (1-b1) |g'|)  (three roundings);
      v = b2 v + (1-b2) g' g': e_v <- b2 e_v + (1-b2) (2 |g'| e_g + e_g^2) + 4 u (b2 v + (1-b2) g'^2);
      p: its own rounding (u |p|), the update's relative error from the fp32 scalars -- step_size (1 - b1^t cancels:
         u / (1-b1)), 1/sqrt(1 - b2^t) (u / (1-b2)), sqrt, fma, the product and the approximate divide (2 ulp):
         (8 + 1/(1-b1) + 1/(1-b2)) u -- plus half of v's relative error (through sqrt), plus step_size e_m / den."""
    lr, b1, b2, eps, wd, gs = (r32(x) for x in (lr, betas[0], betas[1], eps, wd, grad_scale))
    p = d64(p0).clone()
    m = torch.zeros_like(p) if m0 is None else d64(m0).clone()
    v = torch.zeros_like(p) if v0 is None else d64(v0).clone()
    em = torch.zeros_like(p)
    ev = torch.zeros_like(p)
    tp = torch.zeros_like(p)
    rel = (8 + 1 / (1 - b1) + 1 / (1 - b2)) * U32
    out = []
    for k, g in enumerate(grads, start=1):
        g = d64(g)
        t = step0 + k + (1 if variant == "step_off_by_one" else 0)
        gp = (g + wd * p) * gs if variant == "scale_after_wd" else g * gs + wd * p
        eg = 2 * U32 * ((g * gs).abs() + (wd * p).abs()) + wd * tp
        em = b1 * em + (1 - b1) * eg + 3 * U32 * (b1 * m.abs() + (1 - b1) * gp.abs())
        ev = b2 * ev + (1 - b2) * (2 * gp.abs() * eg + eg * eg) + 4 * U32 * (b2 * v + (1 - b2) * gp * gp)
        m = b1 * m + (1 - b1) * gp
        v = b2 * v + (1 - b2) * gp * gp
        bc1, bc2 = 1 - b1 ** t, 1 - b2 ** t
        if variant == "no_bias_correction":
            bc1 = bc2 = 1.0
        if variant == "eps_in_sqrt":
            den = (v / bc2 + eps).sqrt()
        else:
            den = v.sqrt() / math.sqrt(bc2) + eps
        step_size = lr / bc1
        upd = step_size * m / den
        p = p - upd
        rel_v = torch.where(v > 0, ev / v.clamp_min(1e-300), torch.zeros_like(v))
        tp = tp + U32 * p.abs() + (rel + 0.5 * rel_v) * upd.abs() + step_size * em / den
        out.append({"p": p.clone(), "m": m.clone(), "v": v.clone(), "tp": 2 * tp, "tm": 2 * em, "tv": 2 * ev})
    return out


# ================================================================================================ spectral norm
SN_EPS = 1e-12


def sn_power_ref(w, u, v, update, eps=SN_EPS, variant=None):
    """torch.nn.utils.spectral_norm's power iteration (one step, ``_power_method``) on W = w.view(rows, -1), then
    sigma = u . (W v); update=False leaves u, v and evaluates sigma only.  -> dict u, v, sigma and bounds tu, tv, ts.

    Bounds: t = W^T u is a sum over rows in chunks of 32 plus a serial sum of the chunks (depth rows/32 + 32): error
    <= gamma |W|^T |u|; v = t / ||t|| adds |v| (gamma_norm + 3 u).  s = W v is a 256-thread block dot product (depth
    cols/256 + 14) of W with the already perturbed v: |W| (gamma |v| + dv); u = s / ||s|| and sigma = ||s|| likewise."""
    W = d64(w).reshape(d64(w).shape[0], -1)
    rows, cols = W.shape
    u0, v0 = d64(u), d64(v)
    Wa = W.abs()
    g_t = sum_bound(1.0, rows / 32 + 32 + 4)
    g_s = sum_bound(1.0, block_sum_depth(cols / 256 + 4) + 4)
    g_n = sum_bound(1.0, block_sum_depth(max(rows, cols) / 1024 + 1) + 4)
    if update:
        t = W.t() @ u0
        vn = t / max(float(t.norm()), eps)
        dv = g_t * (Wa.t() @ u0.abs()) / max(float(t.norm()), eps) + vn.abs() * (g_n + 3 * U32)
        if variant == "v_not_normalized":
            vn = t
        s = W @ vn
        ds = g_s * (Wa @ vn.abs()) + Wa @ dv
        sn = max(float(s.norm()), eps)
        un = s / sn
        if variant == "u_not_updated":
            un = u0.clone()
        sigma = float(un @ s)
        rel_n = float(ds.norm()) / sn + g_n + 3 * U32
        du = ds / sn + un.abs() * rel_n
        dsig = sigma * rel_n + float(ds.norm())
        return {"u": un, "v": vn, "sigma": sigma, "tu": 2 * du, "tv": 2 * dv, "ts": 2 * dsig}
    s = W @ v0
    ds = g_s * (Wa @ v0.abs())
    sigma = float(u0 @ s)
    dsig = sum_bound(float((u0 * s).abs().sum()), block_sum_depth(rows / 1024 + 1)) + float(u0.abs() @ ds)
    return {"u": u0, "v": v0, "sigma": sigma, "tu": torch.zeros_like(u0), "tv": torch.zeros_like(v0), "ts": 2 * dsig}


def sn_grad_ref(w, u, v, sigma32, gw, variant=None):
    """d/dW of <G, W / sigma(W)>, sigma(W) = u . (W v) with u, v detached, by float64 autograd; G = ``gw`` is the
    gradient with respect to the normalised weight.  The kernel receives sigma as the fp32 ``sigma32``; the reference
    evaluates the same expression at that sigma, so their difference is the kernel's rounding alone.

    Bound: <G, W> is a 256-thread partial per 4096 elements (depth 16 + 10), then a block sum over the partials
    (depth parts/256 + 10): gamma sum|G W|; each element then rounds coef = dot / sigma, coef*u*v, the difference and
    the product by 1/sigma: 6 u (|G| + |coef u v|) / sigma, plus |u v| dcoef / sigma; doubled."""
    W = d64(w).reshape(d64(w).shape[0], -1)
    u0, v0, G = d64(u), d64(v), d64(gw).reshape(W.shape)
    # autograd of W / sigma(W) is (G - <G,W>/s u v^T) / s at s = sigma(W) (sn_autograd_check pins this on the host);
    # here s is the fp32 sigma the kernel is given
    dot = float((G * W).sum())
    uvt = torch.outer(u0, v0)
    ref = (G - dot / sigma32 * uvt) / sigma32
    if variant == "no_projection":
        ref = G / sigma32
    elif variant == "sigma_squared":
        ref = (G - dot / sigma32 ** 2 * uvt) / sigma32
    n = W.numel()
    parts = (n + 4095) // 4096
    ddot = sum_bound(float((G * W).abs().sum()), 26 + block_sum_depth(parts / 256 + 1))
    coef = abs(dot / sigma32)
    tol = 2 * (6 * U32 * (G.abs() + coef * uvt.abs()) / abs(sigma32) + uvt.abs() * (ddot / abs(sigma32)) / abs(sigma32))
    return ref, tol


def sn_autograd_check(w, u, v, gw):
    """Float64 autograd of W / sigma(W) (u, v detached) at the float64 sigma: used on the host to pin sn_grad_ref."""
    W = d64(w).reshape(d64(w).shape[0], -1).clone().requires_grad_(True)
    u0, v0 = d64(u), d64(v)
    (d64(gw).reshape(W.shape) * (W / (u0 @ (W @ v0)))).sum().backward()
    return W.grad


# ================================================================================================ loss seeds
def hinge_ref(real, fake, loss_scale, variant=None):
    """relu(1 - real).mean() + relu(1 + fake).mean(), each scaled; gradients of the unscaled loss, as the kernel writes
    them: -1/B and +1/B in fp32 (one rounding), 0 where the margin is <= 0 (torch's relu'(0) = 0).
    -> (losses [D, R, F], d_real, d_fake, loss tolerance)."""
    r, f = d64(real), d64(fake)
    B = r.numel()
    inv = float(f32(1) / f32(B))
    mr, mf = 1 - r, 1 + f
    pos_r = (mr >= 0) if variant == "grad_at_zero_margin" else (mr > 0)
    pos_f = (mf >= 0) if variant == "grad_at_zero_margin" else (mf > 0)
    dr = torch.where(pos_r, torch.full_like(r, -inv), torch.zeros_like(r))
    df = torch.where(pos_f, torch.full_like(f, inv), torch.zeros_like(f))
    lr = F.relu(mr).sum() / B * loss_scale
    lf = F.relu(mf).sum() / B * loss_scale
    if variant == "unscaled":
        lr, lf = lr / loss_scale, lf / loss_scale
    # serial loop over batch / 1024 per thread + block sum; the margin (1 -/+ x) rounds once per term; then * inv
    # (itself rounded), * loss_scale (rounded to fp32) and (for LossD) the add: 5 u of the result
    dep = block_sum_depth(-(-B // 1024)) + 1
    tr = sum_bound(float(F.relu(mr).sum()) / B * abs(loss_scale), dep) + 5 * U32 * abs(float(lr))
    tf = sum_bound(float(F.relu(mf).sum()) / B * abs(loss_scale), dep) + 5 * U32 * abs(float(lf))
    losses = torch.tensor([float(lr + lf), float(lr), float(lf)], dtype=torch.float64)
    tol = torch.tensor([tr + tf + U32 * abs(float(lr + lf)), tr, tf], dtype=torch.float64)
    return losses, dr, df, tol


def gen_adv_ref(logits, loss_scale):
    """-mean(logits) * loss_scale, gradient -1/B (fp32, one rounding).  -> (loss, dlogits, tolerance)."""
    x = d64(logits)
    B = x.numel()
    inv = float(f32(1) / f32(B))
    loss = -float(x.sum()) / B * loss_scale
    tol = sum_bound(float(x.abs().sum()) / B * abs(loss_scale), block_sum_depth(-(-B // 1024))) + 5 * U32 * abs(loss)
    return loss, torch.full_like(x, -inv), tol


def hinge_inputs(B, seed):
    """Logits around the margins, including exact +-1 (a margin of exactly 0) on both sides."""
    g = torch.Generator().manual_seed(seed)
    real = torch.randn(B, generator=g) * 1.5
    fake = torch.randn(B, generator=g) * 1.5
    real[::3] = 1.0
    fake[1::3] = -1.0
    real[2::7] = -1.0
    fake[::5] = 1.0
    return real, fake


POINTWISE_KINDS = ("mse", "l1", "bce_logits")


def pointwise_inputs(kind, n, const_target, seed):
    """x (and a tensor target of the same shape unless ``const_target`` is a number); l1 gets exact ties (d == 0),
    bce gets logits up to |x| = 100 and targets in [0, 1]."""
    g = torch.Generator().manual_seed(seed)
    if kind == "bce_logits":
        x = torch.randn(n, generator=g) * 8
        x[::11] = 100.0
        x[1::11] = -100.0
        y = const_target if const_target is not None else torch.rand(n, generator=g)
    else:
        x = torch.randn(n, generator=g)
        y = const_target if const_target is not None else torch.randn(n, generator=g)
        if kind == "l1":
            if const_target is None:
                y[::4] = x[::4]
            else:
                x[::4] = float(const_target)
    return x, y


def pointwise_ref(kind, x, y, weight, variant=None):
    """weight * F.<loss>(x, y) (mean) and its float64 autograd gradient.  -> (loss, dx, loss tol, dx tol).

    Kernel arithmetic: per element d = x - t (one rounding) and l, g from it; gscale = weight / n (one rounding, and
    weight itself is rounded to fp32); dx = g * gscale.  mse: d rounds, 2 d is exact, the product rounds: 5 u |dx|.  l1: sign(d) is exact, so dx is
    +-fp32(weight / n) or 0: a single rounding, 1 u |dx| (bit-exact against the same fp32 division).  bce: sigmoid through
    expf (2 ulp), 1 + e, 1 / (.), minus t (cancellation: u (|sigmoid| + |t|)), times gscale: 8 u (|sigmoid| + |t|) gscale.
    Loss: grid-stride loop (<= 2 SMs CTAs) then a 1-CTA finalize: depth n/256 + 30 over sum |l_i|; each l_i itself is
    off by 4 u (|x| + |x t| + 1) for bce (three terms that cancel), 2 u l_i otherwise; times weight / n."""
    xd = d64(x).clone().requires_grad_(True)
    n = xd.numel()
    yd = d64(y) if isinstance(y, torch.Tensor) else torch.full_like(xd, float(f32(y)))
    if kind == "mse":
        per = (xd - yd) ** 2
    elif kind == "l1":
        per = (xd - yd).abs()
    else:
        per = F.binary_cross_entropy_with_logits(xd, yd, reduction="none")
    loss = per.mean() * weight
    loss.backward()
    loss = loss.detach()
    dx = xd.grad.detach()
    x0 = xd.detach()
    gscale = float(f32(weight) / f32(n))
    if kind == "l1":
        dx = torch.sign(x0 - yd) * gscale       # the fp32 weight / n the kernel scales by (autograd: within 1 u of it)
        if variant == "sign_at_tie":
            dx = torch.where(x0 == yd, torch.full_like(dx, gscale), dx)
        tdx = torch.zeros_like(dx)
    elif kind == "mse":
        if variant == "no_factor_two":
            dx = dx / 2
        tdx = 5 * U32 * dx.abs()
    else:
        if variant == "sigmoid_of_minus_x":
            dx = (torch.sigmoid(-x0) - yd) * weight / n
        tdx = 8 * U32 * (torch.sigmoid(x0) + yd.abs()) * abs(gscale) + 3 * U32 * dx.abs()
    per = per.detach()
    err_l = 4 * U32 * (x0.abs() + (x0 * yd).abs() + 1) if kind == "bce_logits" else 2 * U32 * per
    lsum = float(per.sum())
    tl = (sum_bound(lsum, n / 256 + 30) + float(err_l.sum())) * abs(weight) / n + 4 * U32 * abs(float(loss))
    if variant == "sum_not_mean":
        loss = loss * n
    return float(loss), dx, tl, tdx


# ================================================================================================ Philox / randn
PHILOX_M0, PHILOX_M1 = 0xD2511F53, 0xCD9E8D57
PHILOX_W0, PHILOX_W1 = 0x9E3779B9, 0xBB67AE85
_M32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(ctr, key):
    """Random123 Philox4x32-10 on numpy arrays: ctr (4, N) uint32-valued, key (2,) -> (4, N) uint64 holding uint32."""
    c = [np.asarray(x, np.uint64) & _M32 for x in ctr]
    k0, k1 = np.uint64(key[0]) & _M32, np.uint64(key[1]) & _M32
    for _ in range(10):
        p0 = np.uint64(PHILOX_M0) * c[0]
        p1 = np.uint64(PHILOX_M1) * c[2]
        hi0, lo0 = p0 >> np.uint64(32), p0 & _M32
        hi1, lo1 = p1 >> np.uint64(32), p1 & _M32
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
        k0 = (k0 + np.uint64(PHILOX_W0)) & _M32
        k1 = (k1 + np.uint64(PHILOX_W1)) & _M32
    return np.stack(c)


def u01_f32(x):
    """((float)(x >> 8) + 0.5f) * 2^-24 in exact float32 steps: in (0, 1]."""
    hi = (np.asarray(x, np.uint64) >> np.uint64(8)).astype(f32)
    return ((hi + f32(0.5)) * f32(1.0 / 16777216.0)).astype(f32)


TWO_PI_F32 = f32(6.28318530717958647692)


def randn_ref(n, seed, base, variant=None):
    """The n draws of one ipr_randn_f32 launch whose counter reads ``base``: quad q uses Philox4x32-10 of counter
    (base + q) = (lo, hi, 0, 0) under key (seed lo, seed hi); its words (0, 1) and (2, 3) become two Box-Muller pairs
    r cos, r sin with r = sqrt(-2 log u01(w0)), angle = fp32(2 pi * u01(w1)).  -> (float64 draws, bound, next counter).

    Bound: logf (1 ulp) then sqrtf: r is within 2 u; sincosf is within 2 ulp (<= 2^-23 absolute, |value| <= 1); the
    product rounds once: |draw - ref| <= r (2^-23 + 3 u) < 8 u r."""
    quads = (n + 3) // 4
    q = np.arange(quads, dtype=np.uint64) + np.uint64(base)
    zero = np.zeros(quads, np.uint64)
    words = philox4x32_10([q & _M32, q >> np.uint64(32), zero, zero], (seed & 0xFFFFFFFF, seed >> 32))
    out = np.empty((quads, 4), np.float64)
    rr = np.empty((quads, 4), np.float64)
    for h in range(2):
        r = np.sqrt(-2.0 * np.log(u01_f32(words[2 * h]).astype(np.float64)))
        ang = (TWO_PI_F32 * u01_f32(words[2 * h + 1])).astype(f32).astype(np.float64)
        cs, sn = np.cos(ang), np.sin(ang)
        if variant == "swap_sin_cos":
            cs, sn = sn, cs
        out[:, 2 * h], out[:, 2 * h + 1] = r * cs, r * sn
        rr[:, 2 * h] = rr[:, 2 * h + 1] = r
    step = n if variant == "counter_by_n" else quads
    return torch.from_numpy(out.reshape(-1)[:n].copy()), torch.from_numpy(8 * U32 * rr.reshape(-1)[:n]), base + step


# ================================================================================================ column sums
def colsum_ref(x2d, ncols, out_old, accumulate, scale, out_index=None, depth=None, variant=None):
    """out[c] (+)= scale * sum_r x[r][c] (column c lands at out[out_index[c]]).  -> (out, tol).
    Bound: the kernel's longest addition chain ``depth`` over sum |x| (fp32 stages; double stages add nothing), then
    the float conversion, * scale and the accumulating add: 3 u of the terms."""
    X = d64(x2d)[:, :ncols]
    s = X.sum(0) * scale
    a = X.abs().sum(0) * abs(scale)
    out = d64(out_old).clone()
    tol = torch.zeros_like(out)
    idx = torch.arange(ncols, device=X.device) if out_index is None else out_index.long().to(X.device)
    acc = accumulate and variant != "accumulate_ignored"
    new = out[idx] + s if acc else s
    tol[idx] = sum_bound(a, depth) + 3 * U32 * (a + out[idx].abs() * (1 if accumulate else 0))
    out[idx] = new
    return out, tol


# ================================================================================================ BatchNorm
def bn_finalize_ref(partial, count, gamma, beta, eps, momentum, run_mean, run_var, variant=None):
    """BatchNorm's training-mode statistics from fp32 column partials [rows][2][C] (sums, sums of squares) summed in
    float64: mean, biased variance (normalisation), unbiased variance (running_var), scale = gamma*rstd,
    shift = beta - mean*scale.  -> dict of float64 results and tolerances.

    The kernel works in double up to rstd, then rounds mean and rstd once each (1 u); scale rounds g*rstd (1 u);
    shift = beta - mean*g*rstd is 3 roundings of terms of size |beta| and |mean g rstd|; the running buffers mix two
    fp32 terms with up to 4 roundings."""
    P = d64(partial).reshape(d64(partial).shape[0], 2, -1).sum(0)
    mean = P[0] / count
    var = (P[1] / count - mean * mean).clamp_min(0)
    if variant == "biased_running_var":
        unb = var
    else:
        unb = var * count / (count - 1) if count > 1 else var
    rstd = 1 / torch.sqrt(var + r32(eps))
    g, b = d64(gamma), d64(beta)
    m = r32(momentum)
    rm, rv = d64(run_mean), d64(run_var)
    res = {"mean": mean, "rstd": rstd, "scale": g * rstd, "shift": b - mean * g * rstd,
           "running_mean": (1 - m) * rm + m * mean, "running_var": (1 - m) * rv + m * unb}
    tol = {"mean": 2 * U32 * mean.abs(), "rstd": 2 * U32 * rstd, "scale": 4 * U32 * (g * rstd).abs(),
           "shift": 6 * U32 * (b.abs() + (mean * g * rstd).abs()),
           "running_mean": 6 * U32 * ((1 - m) * rm.abs() + m * mean.abs()),
           "running_var": 6 * U32 * ((1 - m) * rv.abs() + m * unb.abs())}
    return res, tol


def bn_stats_partials(x2d, groups):
    """fp32 column partials [groups][2][C] of a bf16 [rows][C] tensor (float64 sums, rounded once): what a GEMM
    epilogue hands to the finalisation."""
    X = d64(x2d)
    out = []
    for chunk in torch.tensor_split(X, groups, dim=0):
        out.append(torch.stack([chunk.sum(0), (chunk * chunk).sum(0)]))
    return torch.stack(out).float()


def bn_apply_ref(x2d, scale, shift):
    """relu(x * scale + shift) with the kernel's fp32 scale / shift; the sign of the fp32 fmaf equals the sign of the
    exact value, so the mask is exact.  Output within one bf16 ulp (rounding via fp32 or float64 differs only at ties)."""
    y = (d64(x2d) * d64(scale) + d64(shift)).clamp_min(0)
    return y, bf16_ulp(y)


def bn_bwd_ref(dy, xraw, scale, shift, gamma, beta, eps, rows, sign=None, gamma0=0.0, sign_scale=0.0,
               dgamma_old=None, dbeta_old=None, accumulate=0, variant=None):
    """Backward of relu(BatchNorm_train(x)) by float64 autograd of F.batch_norm, the ReLU mask being the kernel's
    (x * scale + shift > 0, exact in float64 with the fp32 scale / shift), plus the white-box sign-loss term
    d/dgamma of sign_scale * mean_c relu(gamma0 - gamma_c sign_c) in dgamma.  -> (dx, dgamma, dbeta, tolerances)."""
    X = d64(xraw).clone().requires_grad_(True)
    g = d64(gamma).clone().requires_grad_(True)
    b = d64(beta).clone().requires_grad_(True)
    C = X.shape[1]
    mask = (d64(xraw) * d64(scale) + d64(shift)) > 0
    y = F.batch_norm(X, None, None, g, b, training=True, eps=r32(eps))
    (y * (d64(dy) * mask)).sum().backward()
    dx, dgam, dbet = X.grad, g.grad, b.grad
    if sign is not None:
        sv = d64(sign)
        act = (r32(gamma0) - d64(gamma) * sv) > 0
        per_c = 1.0 if variant == "sign_without_1_over_C" else 1.0 / C
        term = torch.where(act, -sv * r32(sign_scale) * per_c, torch.zeros_like(sv))
        dgam = dgam + term
    if accumulate:
        dgam = dgam + d64(dgamma_old)
        dbet = dbet + d64(dbeta_old)
    # tolerances.  Sums: per-thread serial rows / (CTAs * row lanes) plus the row lanes in shared memory (<= 256):
    # depth rows/8 + 260 bounds both; the mean / rstd the kernel uses are fp32 roundings of statistics computed from fp32
    # partials: relative 8 u E[x^2] / var, which moves xhat, the coefficients and dgamma alike.
    Xd = d64(xraw)
    gm = d64(dy) * mask
    mu = Xd.mean(0)
    var = Xd.var(0, unbiased=False)
    xh = (Xd - mu) / torch.sqrt(var + r32(eps))
    rel_stat = 8 * U32 * ((Xd * Xd).mean(0) + r32(eps)) / (var + r32(eps))
    dep = rows / 8 + 260
    t_dbeta = sum_bound(gm.abs().sum(0), dep) + U32 * dbet.abs()
    t_dgam = sum_bound((gm * xh).abs().sum(0), dep + 4) + rel_stat * (gm * xh).abs().sum(0) * 4 + 2 * U32 * dgam.abs()
    if sign is not None:                          # (sign * scale) / C and the add: 3 u of the term
        t_dgam = t_dgam + 3 * U32 * term.abs()
    gamma_d, rstd = d64(gamma), 1 / torch.sqrt(var + r32(eps))
    a = gamma_d * rstd
    bco = -gamma_d * rstd * rstd * (gm * xh).sum(0) / rows
    dco = -a * gm.sum(0) / rows - bco * mu
    terms = (a * gm).abs() + (bco * Xd).abs() + dco.abs()
    # dx = a g + b x + d in fp32: 4 roundings of these terms and the statistics' relative error in every term; the
    # column sums enter through d (a dbeta / M) and b (a rstd dgamma_bn / M, times x - mean); then one bf16 rounding
    d_sx = sum_bound((gm * xh).abs().sum(0), dep) + rel_stat * (gm * xh).abs().sum(0)
    t_dx = bf16_ulp(dx) + (8 * U32 + 2 * rel_stat) * terms + a.abs() * (sum_bound(gm.abs().sum(0), dep) + d_sx * xh.abs()) / rows
    if accumulate:
        t_dgam = t_dgam + U32 * (dgam.abs() + d64(dgamma_old).abs())
        t_dbeta = t_dbeta + U32 * (dbet.abs() + d64(dbeta_old).abs())
    return dx, dgam, dbet, t_dx, t_dgam, t_dbeta


# ================================================================================================ final GEMV
def dfc_fwd_ref(a, w, sigma, bias):
    """logits[b] = a[b] . w / sigma + bias (bf16 activations, fp32 weights).  -> (logits, tol).
    Bound: per thread K/2048 iterations of 8 products and 8 adds, then the block sum: depth K/256 + 20 over
    sum |a w|; / sigma and + bias round twice more."""
    A, W = d64(a), d64(w)
    s = 1.0 if sigma is None else float(sigma)
    bb = 0.0 if bias is None else float(bias)
    out = A @ W / s + bb
    K = A.shape[1]
    tol = sum_bound((A.abs() @ W.abs()) / abs(s), K / 256 + 20) + 3 * U32 * ((A @ W).abs() / abs(s) + abs(bb))
    return out, tol


def dfc_bwd_data_ref(a, w, sigma, dlogit, slope):
    """da[b,k] = dlogit[b] / sigma * w[k] * lrelu'(a[b,k]) (the mask from the stored post-activation: a > 0 <=>
    pre-activation > 0).  fp32 1/sigma, dlogit * inv, * w, * slope: 4 roundings, then bf16: within one bf16 ulp."""
    A = d64(a)
    s = 1.0 if sigma is None else float(sigma)
    d = d64(dlogit).view(-1, 1) / s * d64(w).view(1, -1) * torch.where(A > 0, 1.0, r32(slope))
    return d, bf16_ulp(d) + 6 * U32 * d.abs()


def dfc_bwd_weight_ref(a, dlogit, dw_old, accumulate, dw_index=None, dbias_old=None, variant=None):
    """dw[o(k)] (+)= sum_b dlogit[b] a[b,k]; dbias += sum_b dlogit[b] (always accumulating).
    Bounds: depth batch/8 + 8 over sum |dlogit a|, batch/32 + 5 for the bias; the accumulating add rounds once more."""
    A, dl = d64(a), d64(dlogit)
    B, K = A.shape
    s = dl @ A
    t = sum_bound(dl.abs() @ A.abs(), B / 8 + 8) + U32 * s.abs()
    idx = torch.arange(K, device=A.device) if dw_index is None else dw_index.long().to(A.device)
    dw = d64(dw_old).clone()
    tol = torch.zeros_like(dw)
    acc = accumulate and variant != "accumulate_ignored"
    dw[idx] = dw[idx] + s if acc else s
    tol[idx] = t + (U32 * (dw[idx].abs()) if accumulate else 0)
    db = db_t = None
    if dbias_old is not None:
        db = float(d64(dbias_old).sum()) + float(dl.sum())
        db_t = sum_bound(float(dl.abs().sum()), B / 32 + 5) + U32 * (abs(db) + abs(float(d64(dbias_old).sum())))
    return dw, tol, db, db_t


# ================================================================================================ 3-channel im2col / col2im
def im2col3_ref(x, t=None):
    """(B, 3, H, W) fp32 (times 1 - t^2 when the tanh output t is given) -> (B, H, W, 32) float64, column
    (kh*3+kw)*3 + c = x[b, c, h+kh-1, w+kw-1] (0 outside), columns 27..31 zero."""
    X = d64(x)
    if t is not None:
        T = d64(t)
        X = X * (1 - T * T)
    B, C, H, W = X.shape
    P = F.pad(X, (1, 1, 1, 1))
    out = torch.zeros(B, H, W, 32, dtype=torch.float64, device=X.device)
    for kh in range(3):
        for kw in range(3):
            for c in range(3):
                out[..., (kh * 3 + kw) * 3 + c] = P[:, c, kh:kh + H, kw:kw + W]
    return out


def col2im3_ref_f32(t, tanh_out):
    """out[b][c][h][w] = sum over kh (outer), kw (inner) of T[b, h+1-kh, w+1-kw][(kh*3+kw)*3 + c], summed in float32
    from 0 in that order (out-of-image taps add 0): the kernel's documented order, so bit-exact without tanh."""
    T = t.detach().cpu().numpy().astype(f32)
    B, H, W, _ = T.shape
    P = np.zeros((B, H + 2, W + 2, T.shape[3]), f32)
    P[:, 1:H + 1, 1:W + 1] = T
    acc = np.zeros((B, 3, H, W), f32)
    for kh in range(3):
        for kw in range(3):
            for c in range(3):
                # source pixel (h+1-kh, w+1-kw) sits at padded (h+2-kh, w+2-kw)
                acc[:, c] = (acc[:, c] + P[:, 2 - kh:2 - kh + H, 2 - kw:2 - kw + W, (kh * 3 + kw) * 3 + c]).astype(f32)
    out = torch.from_numpy(acc)
    return torch.tanh(out.double()) if tanh_out else out


# ================================================================================================ seeded inputs
def sn_inputs(dims, seed):
    """Per layer (rows, cols): W ~ N(0, 1/cols), unit-norm random u and v (CPU, fp32)."""
    g = torch.Generator().manual_seed(seed)
    ws, us, vs = [], [], []
    for r, c in dims:
        ws.append(torch.randn(r, c, generator=g) / math.sqrt(c))
        u, v = torch.randn(r, generator=g), torch.randn(c, generator=g)
        us.append(u / u.norm())
        vs.append(v / v.norm())
    return ws, us, vs


def sn_grad_inputs(ws, seed):
    """Upstream gradients correlated with W (so the projection term <G, W>/sigma u v^T is not lost in the noise),
    and the grad_out destinations."""
    g = torch.Generator().manual_seed(seed)
    G = [torch.randn(w.shape, generator=g) * 0.1 + 3.0 * w.detach().cpu() for w in ws]
    base = [torch.randn(w.shape, generator=g) for w in ws]
    return G, base


def bn_inputs(C, rows, seed):
    """bf16 pre-activations (mean 0.4, std 1.3) and upstream gradients, BatchNorm parameters and running buffers,
    sign vector and old gradient slots (CPU)."""
    g = torch.Generator().manual_seed(seed)
    x = (torch.randn(rows, C, generator=g) * 1.3 + 0.4).to(torch.bfloat16)
    dy = torch.randn(rows, C, generator=g).to(torch.bfloat16)
    p = {"gamma": torch.randn(C, generator=g), "beta": torch.randn(C, generator=g) * 0.5,
         "running_mean": torch.randn(C, generator=g), "running_var": torch.rand(C, generator=g) + 0.5,
         "sign": torch.where(torch.rand(C, generator=g) < 0.5, -1.0, 1.0),
         "dgamma_old": torch.randn(C, generator=g), "dbeta_old": torch.randn(C, generator=g)}
    return x, dy, p


def dfc_inputs(B, K, seed):
    """bf16 LeakyReLU(0.1) activations with exact zeros, fp32 weight row, upstream gradients, a feature permutation,
    old dw (CPU)."""
    g = torch.Generator().manual_seed(seed)
    a = F.leaky_relu(torch.randn(B, K, generator=g), 0.1).to(torch.bfloat16)
    a.view(-1)[::97] = 0
    w = torch.randn(K, generator=g) / math.sqrt(K)
    dlogit = torch.randn(B, generator=g)
    perm = torch.randperm(K, generator=g).to(torch.int32)
    dw_old = torch.randn(K, generator=g)
    return a, w, dlogit, perm, dw_old
