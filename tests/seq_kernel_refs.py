"""Float64 restatements of the contracts of the SRGAN / CycleGAN layer kernels (csrc/layers.cu) and of the single-tap
"linear" GEMM plans seqnet.py drives through csrc/gemm_tc.cu and csrc/wgrad_tc.cu, written from the operations they
stand for (convolution by patch matrix, BatchNorm / InstanceNorm + activation, their autograd) rather than from the
kernels.  Every function takes the values the kernel sees and returns float64 results plus, where a GPU test needs
one, an elementwise bound derived from the kernel's fp32 arithmetic.  The helpers and the BatchNorm bound reasoning
are those of tests/step_kernel_refs.py.

Also here: the seeded inputs of tests/test_gpu_seq_kernels.py and the case list derived from the four networks, so
that tests/test_seq_kernels_host.py can show on the very same numbers that each bound rejects plausible wrong kernels
(the ``variant=`` mutants)."""
import math

import torch
import torch.nn as nn
import torch.nn.functional as F

from tests.step_kernel_refs import U32, bf16_ulp, d64, max_excess, r32, sum_bound  # noqa: F401 (re-exported)

ACT_NONE, ACT_RELU, ACT_LRELU, ACT_PRELU, ACT_TANH = 0, 1, 2, 3, 4     # csrc/layers.cu


# ================================================================================================ cases
NET_SHAPES = [("SRResNet", (16, 3, 24, 24)), ("Discriminator96", (16, 3, 96, 96)),
              ("Resnet9Blocks", (1, 3, 128, 128)), ("ConvDiscriminator", (1, 3, 128, 128))]
ODD_SHAPE = (3, 3, 20, 22)          # tests/test_gpu_seqnet.py's layer-stack input; walked through the two generators
ODD_NETS = ("SRResNet", "Resnet9Blocks")


def _geom(b):
    return (b.k, b.stride, b.pad, b.up, b.reflect, b.cin_p, b.n_p, b.kp, b.transposed, getattr(b, "out_pad", 0))


def _walk():
    """(network, block index, Block, input NHWC shape, output grid, at the odd shape) for every block of the four
    networks at their benchmark shapes and of the two generators at the odd shape, walked with ``Block.out_hw``."""
    import networks
    from ipr_gan_b200 import seqnet
    runs = [(n, s) for n, s in NET_SHAPES] + [(n, ODD_SHAPE) for n in ODD_NETS]
    for name, shape in runs:
        n, _, h, w = shape
        torch.manual_seed(0)
        for i, b in enumerate(seqnet.lower(getattr(networks, name)())):
            oh, ow = b.out_hw(h, w)
            yield name, i, b, (n, h, w, b.cin_p), (oh, ow), shape == ODD_SHAPE
            h, w = (2 * oh, 2 * ow) if b.shuffle else (oh, ow)


_CACHE = {}


def net_cases():
    """Every convolution of the walk, deduplicated by (block geometry, input shape): dicts of the network, block
    index, Block, input NHWC shape, output grid and whether the networks need the block's data gradient: every block
    but SRResNet's first, whose input is the low-resolution image.  A discriminator's first block feeds the
    generator's gradient (D(G(z)) in the generator step), Resnet9Blocks' first block the cycle loss (G_B(G_A(x)))."""
    if "net" not in _CACHE:
        out, seen = [], set()
        for name, i, b, shape, ohw, odd in _walk():
            key = (_geom(b), shape)
            if key not in seen:
                seen.add(key)
                out.append({"net": name, "i": i, "block": b, "shape": shape, "ohw": ohw,
                            "dgrad": i > 0 or name != "SRResNet",
                            "id": "%s%s-b%d" % (name, "-odd" if odd else "", i)})
        _CACHE["net"] = out
    return _CACHE["net"]


def norm_cases():
    """Every normalisation / activation launch of the walk, deduplicated: dicts of groups, rows, channels, has_norm,
    affine, BatchNorm or not, activation, slope, residual wired or not."""
    if "norm" not in _CACHE:
        out, seen = [], set()
        for name, i, b, shape, ohw, odd in _walk():
            if b.final:
                continue
            nm = b.norm
            inst = isinstance(nm, nn.InstanceNorm2d)
            n, M = shape[0], shape[0] * ohw[0] * ohw[1]
            groups, rows = (n, M // n) if inst else (1, M)
            d = {"groups": groups, "rows": rows, "C": b.n_p, "has_norm": int(nm is not None),
                 "affine": nm is not None and nm.weight is not None, "bn": isinstance(nm, nn.BatchNorm2d),
                 "act": b.act, "slope": b.slope, "residual": b.residual is not None}
            key = tuple(sorted(d.items()))
            if key not in seen:
                seen.add(key)
                d["id"] = "%s%s-b%d" % (name, "-odd" if odd else "", i)
                out.append(d)
        _CACHE["norm"] = out
    return _CACHE["norm"]


def norm_edges(sms):
    """Norm launches the networks do not reach: one slab (rows < 32), rows not a multiple of the row lanes (C = 24:
    85 lanes), more InstanceNorm groups than 4 x SMs (norm_slabs falls back to one slab), C = 8 / 2048 (256 / 1 row
    lanes), a residual behind an activation, Tanh, the eval-mode path (caller's scale / shift), mean / std = 100 with
    more groups than 2 x SMs, so that one slab per group leaves every thread 64 rows to add in fp32 (the one-pass
    E[x^2] - mean^2 at its worst)."""
    base = {"has_norm": 1, "affine": True, "bn": False, "slope": 0.0, "residual": False}
    edges = [("rows20-bn-prelu", dict(groups=1, rows=20, C=64, bn=True, act=ACT_PRELU)),
             ("C24-in-lrelu", dict(groups=2, rows=333, C=24, act=ACT_LRELU, slope=0.2)),
             ("groups>4sms-C8", dict(groups=4 * sms + 3, rows=200, C=8, act=ACT_RELU)),
             ("C2048-bn-relu", dict(groups=1, rows=96, C=2048, bn=True, act=ACT_RELU)),
             ("bn-prelu-residual", dict(groups=1, rows=1000, C=24, bn=True, act=ACT_PRELU, residual=True)),
             ("in-tanh", dict(groups=2, rows=300, C=16, act=ACT_TANH)),
             ("eval-lrelu-residual", dict(groups=1, rows=500, C=32, bn=True, has_norm=2, act=ACT_LRELU, slope=0.2,
                                          residual=True)),
             ("in-mean100", dict(groups=2 * sms + 1, rows=2048, C=64, act=ACT_RELU, mean=100.0, std=1.0))]
    out = []
    for name, kw in edges:
        d = dict(base)
        d.update(kw)
        d["id"] = "edge-" + name
        out.append(d)
    return out


# ================================================================================================ patch matrix
def padded_input(x, b, oh, ow, variant=None):
    """(n, h, w, c) NHWC -> (n, c, (oh-1)*stride + k, (ow-1)*stride + k) float64: the virtual input every output pixel
    reads through its k x k window -- reflection border (``F.pad`` 'reflect'), or zero insertion by ``up`` (transposed
    convolution run as a direct one) and a zero border; the bottom / right edge extended with zeros or cut to what the
    output grid reads (output padding of a transposed convolution)."""
    X = x.to(torch.float64).permute(0, 3, 1, 2)                     # (not detached: col2im_ref differentiates this)
    hv, wv = (oh - 1) * b.stride + b.k, (ow - 1) * b.stride + b.k
    if b.reflect:
        P = F.pad(X, (b.pad,) * 4, mode="replicate" if variant == "clamp" else "reflect")
        return P[:, :, :hv, :wv]
    if b.up > 1:
        n, c, h, w = X.shape
        Z = X.new_zeros(n, c, (h - 1) * b.up + 1, (w - 1) * b.up + 1)
        Z[:, :, ::b.up, ::b.up] = X
        X = Z
    return F.pad(X, (b.pad, wv - b.pad - X.shape[3], b.pad, hv - b.pad - X.shape[2]))


def im2col_ref(x, b, oh, ow, variant=None):
    """Patch matrix [(n, oy, ox)][kp] in float64: column (ky*k + kx)*c + ch holds the virtual input at
    (oy*stride + ky, ox*stride + kx), columns past k*k*c are zero.  ``variant='clamp'``: a border that repeats the
    edge pixel instead of mirroring."""
    P = padded_input(x, b, oh, ow, variant)
    n, c = P.shape[:2]
    cols = F.unfold(P, b.k, stride=b.stride)                        # (n, c*k*k, L), row ch*k*k + ky*k + kx
    cols = cols.view(n, c, b.k * b.k, oh * ow).permute(0, 3, 2, 1).reshape(n * oh * ow, b.k * b.k * c)
    return F.pad(cols, (0, b.kp - cols.shape[1]))


def col2im_ref(dcol, b, shape, oh, ow, addend=None, variant=None):
    """The adjoint of ``im2col_ref`` (its vector-Jacobian product in float64) applied to ``dcol`` [M][kp], plus
    ``addend``.  Variants: 'no_mirror' (a reflection border whose mirrored reads get no gradient), 'no_output_padding'
    (the last output row and column of a transposed convolution dropped)."""
    D = d64(dcol)
    x = torch.zeros(shape, dtype=torch.float64, device=D.device, requires_grad=True)
    blk = b
    if variant == "no_mirror":
        blk = _Geom(b, reflect=0)
    elif variant == "no_output_padding":
        D = D.view(shape[0], oh, ow, -1).clone()
        D[:, -1] = 0
        D[:, :, -1] = 0
        D = D.view(-1, D.shape[-1])
    with torch.enable_grad():
        col = im2col_ref(x, blk, oh, ow)
        (dx,) = torch.autograd.grad(col, x, D)
    return dx + d64(addend) if addend is not None else dx


class _Geom(object):
    """A Block's geometry with some fields replaced (for the mutants)."""

    def __init__(self, b, **kw):
        for name in ("k", "stride", "pad", "up", "reflect", "kp"):
            setattr(self, name, kw.get(name, getattr(b, name)))


def col2im_bound(dcol, b, shape, oh, ow, addend=None):
    """Elementwise bound of the kernel's fp32 gather (at most k*k taps per mirror candidate, up to 2 x 2 candidates,
    plus the addend) rounded once to bf16."""
    mag = col2im_ref(d64(dcol).abs(), b, shape, oh, ow, None if addend is None else d64(addend).abs())
    ref = col2im_ref(dcol, b, shape, oh, ow, addend)
    return bf16_ulp(ref) + sum_bound(mag, b.k * b.k * (4 if b.reflect else 1) + 1)


# ================================================================================================ GEMMs
def gemm_depth(k):
    """Longest chain of fp32 additions of a tcgen05 product over k: one add per 16-wide MMA step, plus the epilogue.
    Measured on a B200 (1000 W power limit) over every case of tests/test_gpu_seq_kernels.py: the largest error / bound
    ratio is 0.04 for the fp32 weight gradient and 0.5 for the bf16 outputs (their final rounding dominates)."""
    return k / 16 + 32


def gemm_ref(a, w, bias=None, variant=None):
    """a [M][K] x w [N][K]^T (+ bias[N]) in float64.  Variants: 'drop_last_k_chunk' (columns 64*floor(K/64) .. K
    ignored: a lost TMA chunk), 'drop_last_row' (the last M row not computed), 'drop_m_tail' (rows past the last full
    128-row tile not computed)."""
    A, W = d64(a), d64(w)
    if variant == "drop_last_k_chunk":
        k0 = (A.shape[1] - 1) // 64 * 64
        A = A.clone()
        A[:, k0:] = 0
    out = A @ W.t()
    if bias is not None:
        out = out + d64(bias)
    if variant == "drop_last_row":
        out[-1] = 0
    elif variant == "drop_m_tail":
        out[(out.shape[0] - 1) // 128 * 128:] = 0
    return out


def gemm_bound(a, w, ref, bf16_out=True):
    """bf16 output: one bf16 ulp of the result (the fp32 value rounded once) plus the fp32 accumulation."""
    t = sum_bound(d64(a).abs() @ d64(w).abs().t(), gemm_depth(a.shape[1]))
    return t + (bf16_ulp(ref) if bf16_out else U32 * ref.abs())


def wgrad_ref(dy, col, weight_shape, row_map, col_off, s_n, grad_old=None, accumulate=False, scale=1.0, drop_rows=None):
    """grad[row_map[n]*s_n + col_off[k]] (+)= scale * sum_m dy[m][n] col[m][k] in float64 (row_map / col_off = -1:
    padding).  ``drop_rows=(lo, hi)``: the mutant whose reduction loses the pixel rows lo..hi (one split's k-blocks).
    -> (grad, bound).  Bound: the reduction over M pixels (depth M/16 + 32) plus the split sum, the scale and the add."""
    Y, X = d64(dy), d64(col)
    if drop_rows is not None:
        Y = Y.clone()
        Y[drop_rows[0]:drop_rows[1]] = 0
    G = Y.t() @ X
    T = sum_bound(Y.abs().t() @ X.abs(), gemm_depth(Y.shape[0]) + 64)
    rm = row_map.long().to(G.device)
    off = col_off.reshape(-1).long().to(G.device)
    rows, cols = (rm >= 0).nonzero()[:, 0], (off >= 0).nonzero()[:, 0]
    dst = (rm[rows].view(-1, 1) * s_n + off[cols].view(1, -1)).reshape(-1)
    out = torch.zeros(math.prod(weight_shape), dtype=torch.float64, device=G.device)
    tol = torch.zeros_like(out)
    out[dst] = G[rows][:, cols].reshape(-1) * scale
    tol[dst] = T[rows][:, cols].reshape(-1) * abs(scale)
    if accumulate:
        old = d64(grad_old).reshape(-1).to(G.device)
        out = out + old
        tol = tol + U32 * (out.abs() + old.abs())
    else:
        tol = tol + U32 * out.abs()
    return out.view(weight_shape), tol.view(weight_shape)


def empty_last_split(total_kb):
    """A split count that leaves the last split of the weight-gradient GEMM without k-blocks (kb_per_split =
    ceil(total / splits) and (splits - 1) * kb_per_split >= total), or None."""
    for s in range(2, 4 * total_kb + 2):
        if (s - 1) * (-(-total_kb // s)) >= total_kb:
            return s
    return None


def split_rows(m, splits, s):
    """Pixel rows of the single-tap weight gradient covered by split ``s`` (64-row k-blocks)."""
    total_kb = -(-m // 64)
    per = -(-total_kb // splits)
    return min(m, s * per * 64), min(m, (s + 1) * per * 64)


# ================================================================================================ norms
def norm_layout(rows, groups, C, sms):
    """csrc/layers.cu's launch geometry of the statistics / backward reduction: (slabs, row lanes per CTA, rows one
    thread adds serially).  Its fp32 addition chain is serial + row lanes long."""
    c_vec = C // 8
    threads = 256 if c_vec <= 256 else c_vec
    ry_n = threads // c_vec
    s = max(1, rows // 32)
    s = min(s, max(1, (4 * sms) // groups), 256)
    return s, ry_n, -(-rows // (s * ry_n))


def _act(v, act, slope):
    if act == ACT_RELU:
        return v.clamp_min(0)
    if act in (ACT_LRELU, ACT_PRELU):
        return torch.where(v > 0, v, v * slope)
    if act == ACT_TANH:
        return torch.tanh(v)
    return v


def _act_grad(v, act, slope):
    if act == ACT_RELU:
        return (v > 0).double()
    if act in (ACT_LRELU, ACT_PRELU):
        return torch.where(v > 0, torch.ones_like(v), torch.full_like(v, slope))
    if act == ACT_TANH:
        return 1 - torch.tanh(v) ** 2
    return torch.ones_like(v)


def norm_stats_ref(x, groups, rows, gamma, beta, eps, momentum, running_mean=None, running_var=None, sms=148,
                   variant=None):
    """Training-mode statistics per (group, channel) of x [groups*rows][C] (groups = 1: BatchNorm; the batch:
    InstanceNorm): mean, biased variance, rstd, scale = gamma*rstd, shift = beta - mean*scale, and the running
    buffers (BatchNorm only; unbiased variance).  -> (dict, tolerances).  Variants: 'pooled' (InstanceNorm statistics
    over the whole batch), 'biased_running_var'.

    Bound: the kernel adds x and x^2 in fp32 per thread and row lane (depth D = serial + lanes), the slabs in double;
    mean = S1/n has error D u E|x|, and the one-pass variance E[x^2] - mean^2 carries the error of the sum of squares
    and of mean^2: (D + 2) u (E[x^2] + 2 |mean| E|x|) -- relative rel_var to var + eps.  rstd moves by rel_var / 2 (plus
    its own rounding), scale and shift by that and their own roundings (as in bn_finalize_ref)."""
    X = d64(x).view(groups, rows, -1)
    C = X.shape[2]
    Xs = X.reshape(1, groups * rows, C) if variant == "pooled" else X
    mean = Xs.mean(1).expand(groups, C)
    ex2 = (Xs * Xs).mean(1).expand(groups, C)
    eab = Xs.abs().mean(1).expand(groups, C)
    var = (Xs.var(1, unbiased=False)).expand(groups, C)
    e = r32(eps)
    rstd = 1 / torch.sqrt(var + e)
    g = d64(gamma).view(1, C) if gamma is not None else torch.ones(1, C, dtype=torch.float64, device=X.device)
    bt = d64(beta).view(1, C) if beta is not None else torch.zeros(1, C, dtype=torch.float64, device=X.device)
    res = {"mean": mean, "rstd": rstd, "scale": g * rstd, "shift": bt - mean * g * rstd}
    _, _, serial = norm_layout(rows, groups, C, sms)
    _, ry_n, _ = norm_layout(rows, groups, C, sms)
    D = serial + ry_n
    t_mean = sum_bound(eab, D) + U32 * mean.abs()
    rel_var = sum_bound(ex2 + 2 * mean.abs() * eab, D + 2) / (var + e)
    tol = {"mean": 2 * t_mean, "rstd": 2 * rstd * (0.5 * rel_var + 3 * U32),
           "scale": 2 * (g * rstd).abs() * (0.5 * rel_var + 5 * U32),
           "shift": 2 * ((g * rstd).abs() * t_mean + (mean * g * rstd).abs() * (0.5 * rel_var + 5 * U32) +
                         2 * U32 * bt.abs())}
    if running_mean is not None:
        n = rows * groups
        m = r32(momentum)
        unb = var[0] if variant == "biased_running_var" else var[0] * n / (n - 1)
        rm, rv = d64(running_mean), d64(running_var)
        res["running_mean"] = (1 - m) * rm + m * mean[0]
        res["running_var"] = (1 - m) * rv + m * unb
        tol["running_mean"] = 6 * U32 * ((1 - m) * rm.abs() + m * mean[0].abs()) + 2 * m * t_mean[0]
        tol["running_var"] = 6 * U32 * ((1 - m) * rv.abs() + m * unb.abs()) + 2 * m * unb.abs() * rel_var[0]
    return res, tol


def norm_act_ref(x, groups, rows, scale, shift, act, slope, residual=None, variant=None):
    """y = act(x * scale + shift) + residual with the kernel's fp32 scale / shift (None: no normalisation); the
    pre-activation is one fmaf, so its sign -- the activation's branch -- is exact.  -> (y, bound).
    ``variant='residual_first'``: the residual added before the activation.
    Bound: fmaf, the slope product or tanhf (2 ulp), the residual add: 4 u of the terms, then one bf16 rounding."""
    X = d64(x).view(groups, rows, -1)
    pre = X if scale is None else X * d64(scale).view(groups, 1, -1) + d64(shift).view(groups, 1, -1)
    R = d64(residual).view(groups, rows, -1) if residual is not None else None
    if variant == "residual_first" and R is not None:
        y = _act(pre + R, act, slope)
    else:
        y = _act(pre, act, slope)
        if R is not None:
            y = y + R
    t = 4 * U32 * (pre.abs() + (R.abs() if R is not None else 0))
    y = y.view(groups * rows, -1)
    return y, bf16_ulp(y) + t.view(groups * rows, -1)


def norm_bwd_ref(dy, x, groups, rows, gamma, scale, shift, eps, act, slope, has_norm=1, sign=None, gamma0=0.0,
                 sign_scale=0.0, dgamma_old=None, dbeta_old=None, dslope_old=None, accumulate=0, want_dslope=False,
                 sms=148, variant=None):
    """Backward of act(BatchNorm / InstanceNorm_train(x)) by float64 autograd of F.batch_norm / F.instance_norm, the
    activation's branch taken at the kernel's own pre-activation fmaf(x, scale, shift) (exact in float64), plus:
    the PReLU slope gradient sum dy*pre over pre <= 0 (all groups), dgamma / dbeta summed over the groups with the
    white-box sign-loss term -sign*scale/C where gamma0 - gamma*sign > 0, and ``accumulate``.
    -> (dict dx, dgamma, dbeta, dslope; dict of bounds).

    Variants: 'slope_all' (the slope gradient also sums pre > 0), 'sign_without_1_over_C', 'no_B_mean' (the dx
    constant without its -B*mean part), 'accumulate_ignored'.

    Bounds follow bn_bwd_ref: the kernel's column sums are fp32 per thread and row lane (depth D = serial + lanes,
    then double); its mean / rstd are fp32 roundings of statistics from fp32 sums, off by rel_stat relative (the
    one-pass variance, see norm_stats_ref), which moves xhat, the coefficients and dgamma alike."""
    X = d64(x).view(groups, rows, -1)
    C = X.shape[2]
    G = d64(dy).view(groups, rows, -1)
    pre = X * d64(scale).view(groups, 1, C) + d64(shift).view(groups, 1, C) if has_norm else X
    ag = _act_grad(pre, act, slope)
    gm = G * ag
    out, tol = {}, {}
    _, ry_n, serial = norm_layout(rows, groups, C, sms)
    D = serial + ry_n
    if want_dslope:
        sel = torch.ones_like(pre, dtype=torch.bool) if variant == "slope_all" else pre <= 0
        s = float((G * pre)[sel].sum())
        mag = float((G * pre).abs()[pre <= 0].sum())
        old = float(d64(dslope_old)) if (accumulate and variant != "accumulate_ignored") else 0.0
        out["dslope"] = torch.tensor(s + old, dtype=torch.float64)
        # per-thread fp32 sums (D), the double sum of the partials cast to fp32 per thread and a block sum (10)
        tol["dslope"] = torch.tensor(sum_bound(mag, D + 12) + U32 * (abs(s) + 2 * abs(old)), dtype=torch.float64)
    if not has_norm:
        dx = gm.reshape(groups * rows, C)
        out["dx"] = dx
        tol["dx"] = bf16_ulp(dx) + 2 * U32 * dx.abs() + (4 * U32 * G.abs() * (pre.abs() + 1)).view_as(dx) * (act == ACT_TANH)
        return out, tol
    Xg = X.clone().requires_grad_(True)
    g = d64(gamma).clone().requires_grad_(True) if gamma is not None else None
    bta = torch.zeros(C, dtype=torch.float64, device=X.device, requires_grad=True) if gamma is not None else None
    with torch.enable_grad():
        if groups == 1:
            y = F.batch_norm(Xg.view(rows, C), None, None, g, bta, training=True, eps=r32(eps)).view(1, rows, C)
        else:
            y = F.instance_norm(Xg.permute(0, 2, 1).unsqueeze(-1), weight=g, bias=bta, eps=r32(eps))
            y = y.squeeze(-1).permute(0, 2, 1)
        (y * gm).sum().backward()
    dx = Xg.grad
    mu = X.mean(1, keepdim=True)
    var = X.var(1, unbiased=False, keepdim=True)
    e = r32(eps)
    rs = 1 / torch.sqrt(var + e)
    xh = (X - mu) * rs
    gam = d64(gamma).view(1, 1, C) if gamma is not None else torch.ones(1, 1, C, dtype=torch.float64, device=X.device)
    a = gam * rs
    sx = (gm * xh).sum(1, keepdim=True)
    bco = -gam * rs * rs * sx / rows
    if variant == "no_B_mean":
        dx = dx + bco * mu
    eab = X.abs().mean(1, keepdim=True)
    rel_stat = sum_bound((X * X).mean(1, keepdim=True) + 2 * mu.abs() * eab, D + 2) / (var + e) + 8 * U32
    terms = (a * gm).abs() + (bco * X).abs() + (a * gm.sum(1, keepdim=True) / rows).abs() + (bco * mu).abs()
    d_sx = sum_bound((gm * xh).abs().sum(1, keepdim=True), D) + rel_stat * (gm * xh).abs().sum(1, keepdim=True)
    t_dx = bf16_ulp(dx) + (8 * U32 + 2 * rel_stat) * terms + \
        a.abs() * (sum_bound(gm.abs().sum(1, keepdim=True), D) + d_sx * xh.abs()) / rows
    if act == ACT_TANH:                                # tanhf of the fp32 pre-activation: its derivative within 4 u (|pre| + 1)
        t_dx = t_dx + a.abs() * 3 * (4 * U32 * G.abs() * (pre.abs() + 1))
    out["dx"] = dx.reshape(groups * rows, C)
    tol["dx"] = t_dx.reshape(groups * rows, C)
    if gamma is not None:
        dg, db = g.grad.clone(), bta.grad.clone()
        t_dg = sum_bound((gm * xh).abs().sum((0, 1)), D + groups + 4) + 4 * (rel_stat * (gm * xh).abs()).sum((0, 1)) + \
            2 * U32 * dg.abs()
        t_db = sum_bound(gm.abs().sum((0, 1)), D + groups) + U32 * db.abs()
        if sign is not None:
            sv = d64(sign)
            on = (r32(gamma0) - d64(gamma) * sv) > 0
            per_c = 1.0 if variant == "sign_without_1_over_C" else 1.0 / C
            term = torch.where(on, -sv * r32(sign_scale) * per_c, torch.zeros_like(sv))
            dg = dg + term
            t_dg = t_dg + 3 * U32 * term.abs()
        if accumulate and variant != "accumulate_ignored":
            dg = dg + d64(dgamma_old)
            db = db + d64(dbeta_old)
        if accumulate:
            t_dg = t_dg + U32 * (dg.abs() + d64(dgamma_old).abs())
            t_db = t_db + U32 * (db.abs() + d64(dbeta_old).abs())
        out["dgamma"], out["dbeta"], tol["dgamma"], tol["dbeta"] = dg, db, t_dg, t_db
    return out, tol


# ================================================================================================ seeded inputs
def int_bf16(shape, gen, lo=-2, hi=2):
    """Integer-valued bf16 in {lo, ..., hi}: products and partial sums of the GEMMs below stay exact in fp32."""
    return torch.randint(lo, hi + 1, shape, generator=gen).to(torch.bfloat16)


def conv_inputs(case, integer, seed):
    """Layer input x (NHWC bf16, zero padding channels), the weight in the parameter's own layout (fp32), bias (fp32,
    None if the conv has none), upstream gradient dy0 [M][n_p] (bf16, zero padding channels) -- integer-valued in
    {-2..2} (biases in {-8..8}) or real-valued -- on the CPU."""
    b = case["block"]
    n, h, w, cp = case["shape"]
    oh, ow = case["ohw"]
    gen = torch.Generator().manual_seed(seed)
    wshape = tuple(b.conv.weight.shape)
    if integer:
        x = int_bf16((n, h, w, cp), gen)
        wt = int_bf16(wshape, gen).float()
        bias = torch.randint(-8, 9, (b.cout,), generator=gen).float()
        dy = int_bf16((n * oh * ow, b.n_p), gen)
    else:
        x = (torch.randn(n, h, w, cp, generator=gen) * 1.3 + 0.2).to(torch.bfloat16)
        wt = torch.randn(wshape, generator=gen) / math.sqrt(b.k * b.k * b.cin)
        bias = torch.randn(b.cout, generator=gen) * 0.1
        dy = torch.randn(n * oh * ow, b.n_p, generator=gen).to(torch.bfloat16)
    x[..., b.cin:] = 0
    dy[:, b.cout:] = 0
    return x, wt, (bias if b.conv.bias is not None else None), dy


def padded_bias(b, bias):
    """The bias as the packed fp32 vector the GEMM reads: zeros in the padding channels (engine.PackSet's gather of
    ``Block.bias_layout``'s source indices, -1 = zero)."""
    bl = b.bias_layout(torch.arange(b.cout, dtype=torch.float32))
    return torch.where(bl >= 0, bias[bl.clamp_min(0).long()], torch.zeros(()))


def wgrad_old(wshape, integer, seed):
    """The gradient the weight-gradient GEMM accumulates into: integers in {-8..8} (exact sums) or real values."""
    gen = torch.Generator().manual_seed(seed)
    return torch.randint(-8, 9, wshape, generator=gen).float() if integer else torch.randn(wshape, generator=gen)


def dcol_inputs(M, kp, integer, seed):
    gen = torch.Generator().manual_seed(seed)
    if integer:
        return int_bf16((M, kp), gen)
    return torch.randn(M, kp, generator=gen).to(torch.bfloat16)


def norm_inputs(case, seed, mean=0.4, std=1.3):
    """x, dy, residual [groups*rows][C] (bf16) and per-channel parameters, running buffers, sign vector, old gradient
    slots, PReLU slope (CPU)."""
    gen = torch.Generator().manual_seed(seed)
    n, C = case["groups"] * case["rows"], case["C"]
    x = (torch.randn(n, C, generator=gen) * std + mean).to(torch.bfloat16)
    dy = torch.randn(n, C, generator=gen).to(torch.bfloat16)
    res = torch.randn(n, C, generator=gen).to(torch.bfloat16)
    p = {"gamma": torch.randn(C, generator=gen) * 0.3 + 1.0, "beta": torch.randn(C, generator=gen) * 0.5,
         "running_mean": torch.randn(C, generator=gen), "running_var": torch.rand(C, generator=gen) + 0.5,
         "sign": torch.where(torch.rand(C, generator=gen) < 0.5, -1.0, 1.0),
         "dgamma_old": torch.randn(C, generator=gen), "dbeta_old": torch.randn(C, generator=gen),
         "slope": torch.rand(1, generator=gen) * 0.3 + 0.1, "dslope_old": torch.randn(1, generator=gen)}
    return x, dy, res, p
