"""Tensor-level entry points over the C ABI (device memory and streams come from PyTorch; the
arithmetic does not).  Every function enqueues on ``torch.cuda.current_stream()`` and never
synchronises, so all of them can be captured into CUDA graphs.

No CPU fallback: a non-CUDA tensor raises ``IprError``.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import IprError, SignLayer, check, lib

_POS = {"t": 0, "l": 0}


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _req(t, name, dtype=torch.float32):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise IprError("%s must be a CUDA tensor: the IPR-GAN hot path has no CPU fallback" % name)
    if t.dtype != dtype:
        raise IprError("%s must be %s, got %s" % (name, dtype, t.dtype))
    return t if t.is_contiguous() else t.contiguous()


def _p(t):
    return ctypes.c_void_p(t.data_ptr())


def window_origin(position, size, height, width):
    """Top-left corner of the trigger window for 'tl' | 'tr' | 'bl' | 'br'
    (tools/paste_watermark.py:40-43: 't'/'l' -> [0, s), 'b'/'r' -> [-s, end))."""
    v, h = position
    return (0 if v == "t" else height - size), (0 if h == "l" else width - size)


# ------------------------------------------------------------------------------ triggers
def paste_patch(x, fg, bg, position, size):
    x = _req(x, "x")
    fg = _req(fg, "fg")
    bg = _req(bg, "bg")
    B, C, H, W = x.shape
    r0, c0 = window_origin(position, size, H, W)
    y = torch.empty_like(x)
    check(lib().ipr_paste_patch_f32(_p(x), _p(y), _p(fg), _p(bg), B, C, H, W, size, r0, c0, _stream()),
          "ipr_paste_patch_f32")
    return y


def trigger_pair(x, fg, bg, position, size, z):
    """ywm = paste(x) and xwm = TransformDist(z) in one launch."""
    x = _req(x, "x")
    z = _req(z, "z")
    fg = _req(fg, "fg")
    bg = _req(bg, "bg")
    B, C, H, W = x.shape
    r0, c0 = window_origin(position, size, H, W)
    y = torch.empty_like(x)
    xwm = torch.empty_like(z)
    check(lib().ipr_trigger_pair_f32(_p(x), _p(y), _p(fg), _p(bg), B, C, H, W, size, r0, c0,
                                     _p(z), _p(xwm), z.numel(), _stream()), "ipr_trigger_pair_f32")
    return xwm, y


_CROP_FNS = {False: "ipr_crop_patch_f32", True: "ipr_crop_postproc_f32", "signed": "ipr_crop_postproc_f32",
             "unit": "ipr_crop_clamp01_f32"}


def postproc_mode(normalized):
    """The evaluation loop's post-processing for a trigger's ``normalized`` flag: 'signed' maps [-1, 1] outputs to
    [0, 1] with (clamp(-1, 1) + 1) / 2, 'unit' clamps outputs that are already in data range 1 to [0, 1]."""
    return "signed" if normalized else "unit"


def crop_patch(x, bg, position, size, postproc=False):
    """apply_mask's crop, optionally followed in the same launch by the evaluation loop's post-processing:
    ``postproc`` False: none; True or 'signed': (clamp(-1, 1) + 1) / 2; 'unit': clamp(0, 1) (see postproc_mode)."""
    if postproc not in _CROP_FNS:
        raise IprError("crop_patch: postproc must be False, True, 'signed' or 'unit', got %r" % (postproc,))
    x = _req(x, "x")
    bg = _req(bg, "bg")
    B, C, H, W = x.shape
    r0, c0 = window_origin(position, size, H, W)
    out = torch.empty(B, C, size, size, device=x.device, dtype=x.dtype)
    name = _CROP_FNS[postproc]
    check(getattr(lib(), name)(_p(x), _p(out), _p(bg), B, C, H, W, size, r0, c0, _stream()), name)
    return out


def bitmask_scatter(z, mask, constant):
    z = _req(z, "z")
    mask = _req(mask, "mask", torch.int64)
    B, D = z.shape
    out = torch.empty_like(z)
    check(lib().ipr_bitmask_scatter_f32(_p(z), _p(out), _p(mask), B, D, mask.numel(), float(constant), _stream()),
          "ipr_bitmask_scatter_f32")
    return out


def transform_dist(z):
    z = _req(z, "z")
    out = torch.empty_like(z)
    if z.numel():
        check(lib().ipr_transform_dist_f32(_p(z), _p(out), z.numel(), _stream()), "ipr_transform_dist_f32")
    return out


def transform_var(z, a, w):
    z = _req(z, "z")
    a = _req(a, "a")
    w = _req(w, "w")
    B, D = z.shape
    out = torch.empty_like(z)
    check(lib().ipr_transform_var_f32(_p(z), _p(out), _p(a), _p(w), B, D, _stream()), "ipr_transform_var_f32")
    return out


# ------------------------------------------------------------------------------ SSIM
def _ssim_ws(x):
    B, C, H, W = x.shape
    nbytes = lib().ipr_ssim_workspace_bytes(B, C, H, W)
    return torch.empty(max(1, (nbytes + 3) // 4), device=x.device, dtype=torch.float32), nbytes


def ssim_loss_fwd_bwd(x, y, normalized, grad_scale=1.0, need_grad=True, loss_out=None, loss_scale=1.0):
    """-> (loss 0-dim, dx or None):  loss = 1 - SSIM,  dx = grad_scale * dloss/dx.  ``loss_out``: an existing
    1-element fp32 CUDA view to write the loss into (a metrics slot)."""
    x = _req(x, "x")
    y = _req(y, "y")
    if x.shape != y.shape or x.dim() != 4:
        raise IprError("ssim: x and y must be (N, C, H, W) tensors of the same shape")
    B, C, H, W = x.shape
    ws, nbytes = _ssim_ws(x)
    loss = torch.empty((), device=x.device, dtype=torch.float32) if loss_out is None else loss_out
    dx = torch.empty_like(x) if need_grad else None
    check(lib().ipr_ssim_fwd_bwd_f32(_p(x), _p(y), _p(dx) if need_grad else None, _p(loss), _p(ws), nbytes,
                                     B, C, H, W, int(bool(normalized)), float(grad_scale), float(loss_scale), _stream()),
          "ipr_ssim_fwd_bwd_f32")
    return loss, dx


def ssim_per_sample(x, y):
    x = _req(x, "x")
    y = _req(y, "y")
    if x.shape != y.shape or x.dim() != 4:
        raise IprError("ssim: x and y must be (N, C, H, W) tensors of the same shape")
    B, C, H, W = x.shape
    ws, nbytes = _ssim_ws(x)
    out = torch.empty(B, device=x.device, dtype=torch.float32)
    check(lib().ipr_ssim_per_sample_f32(_p(x), _p(y), _p(out), _p(ws), nbytes, B, C, H, W, _stream()),
          "ipr_ssim_per_sample_f32")
    return out


# ------------------------------------------------------------------------------ signature
def _sign_table(gammas, signs, grads):
    n = len(gammas)
    if n == 0 or n > _lib.SIGN_MAX_LAYERS:
        raise IprError("sign: between 1 and %d layers per call" % _lib.SIGN_MAX_LAYERS)
    arr = (SignLayer * n)()
    keep = []
    for i in range(n):
        g = _req(gammas[i], "gamma")
        s = _req(signs[i], "sign")
        if g.data_ptr() != gammas[i].data_ptr():
            raise IprError("sign: gamma vectors must be contiguous")
        if g.numel() != s.numel():
            raise IprError("sign: gamma / sign length mismatch")
        keep.append(s)
        arr[i].gamma = g.data_ptr()
        arr[i].sign = s.data_ptr()
        arr[i].grad = grads[i].data_ptr() if grads is not None else None
        arr[i].n = g.numel()
    return arr, keep


def sign_loss_fwd_bwd(gammas, signs, gamma_0, grad_scale=1.0, grads=None, accumulate=False, need_grad=True,
                      loss_out=None, loss_scale=1.0):
    """-> (loss 0-dim, grads list).  ``grads`` (optional) are destinations to write / accumulate into;
    ``need_grad=False`` evaluates the loss only (its gradient then rides in the normalisation layers' backward);
    ``loss_out``: an existing 1-element view to write the loss into (single-call signatures only)."""
    if grads is None and need_grad:
        grads = [torch.empty_like(g) for g in gammas]
    total = 0
    loss = torch.empty((), device=gammas[0].device, dtype=torch.float32)
    if loss_out is not None and len(gammas) <= _lib.SIGN_MAX_LAYERS:
        loss = loss_out
    part = loss
    for lo in range(0, len(gammas), _lib.SIGN_MAX_LAYERS):
        hi = lo + _lib.SIGN_MAX_LAYERS
        arr, _keep = _sign_table(gammas[lo:hi], signs[lo:hi], grads[lo:hi] if grads is not None else None)
        if lo > 0:
            part = torch.empty((), device=gammas[0].device, dtype=torch.float32)
        check(lib().ipr_sign_loss_fwd_bwd_f32(arr, len(arr), float(gamma_0), float(grad_scale),
                                              int(bool(accumulate)), float(loss_scale), _p(part), _stream()),
              "ipr_sign_loss_fwd_bwd_f32")
        total = part if lo == 0 else total + part
    return total, grads


def sign_ber_counts(gammas, signs):
    """-> int32 tensor [wrong, total] on the device."""
    dev = gammas[0].device
    out = torch.zeros(2, device=dev, dtype=torch.int32)
    for lo in range(0, len(gammas), _lib.SIGN_MAX_LAYERS):
        hi = lo + _lib.SIGN_MAX_LAYERS
        arr, _keep = _sign_table(gammas[lo:hi], signs[lo:hi], None)
        part = torch.empty(2, device=dev, dtype=torch.int32)
        check(lib().ipr_sign_ber_i32(arr, len(arr), _p(part), _stream()), "ipr_sign_ber_i32")
        out = out + part
    return out


# ------------------------------------------------------------------------------ step scalars
def hinge_d_loss(real_logits, fake_logits, slots, loss_scale=1.0):
    """models/dcgan.py:31-35 in one launch: slots[0:3] <- (LossD, LossR, LossF); -> (dLossD/dreal, dLossD/dfake)."""
    r = _req(real_logits, "real_logits")
    f = _req(fake_logits, "fake_logits")
    if r.numel() != f.numel():
        raise IprError("hinge loss: real / fake batch mismatch")
    dr, df = torch.empty_like(r), torch.empty_like(f)
    check(lib().ipr_hinge_d_loss_f32(_p(r), _p(f), r.numel(), float(loss_scale), _p(slots), _p(dr), _p(df), _stream()),
          "ipr_hinge_d_loss_f32")
    return dr, df


def gen_adv_loss(logits, slot, loss_scale=1.0):
    """models/dcgan.py:37-40: slot[0] <- -mean(logits); -> d/dlogits (= -1/B)."""
    l = _req(logits, "logits")
    d = torch.empty_like(l)
    check(lib().ipr_gen_adv_loss_f32(_p(l), l.numel(), float(loss_scale), _p(slot), _p(d), _stream()),
          "ipr_gen_adv_loss_f32")
    return d


_LOSS_KINDS = {"mse": 0, "l1": 1, "bce_logits": 2}


def pointwise_loss(kind, x, target, weight=1.0, need_grad=True):
    """-> (weight * loss 0-dim, weight * dloss/dx or None) in one pass (csrc/step_misc.cu).  ``target``: a tensor of
    x's shape, or a Python number (the reference's ones_like / zeros_like targets)."""
    x = _req(x, "x")
    const = not isinstance(target, torch.Tensor)
    y = None if const else _req(target, "target")
    if y is not None and y.numel() != x.numel():
        raise IprError("pointwise loss: target shape mismatch")
    loss = torch.empty((), device=x.device, dtype=torch.float32)
    dx = torch.empty_like(x) if need_grad else None
    nbytes = lib().ipr_pointwise_loss_workspace_bytes()
    ws = torch.empty(nbytes // 4, device=x.device, dtype=torch.float32)
    check(lib().ipr_pointwise_loss_f32(_p(x), _p(y) if y is not None else None, float(target) if const else 0.0, x.numel(),
                                       _LOSS_KINDS[kind], float(weight), _p(loss), _p(dx) if need_grad else None, _p(ws),
                                       nbytes, _stream()), "ipr_pointwise_loss_f32")
    return loss, dx


class DeviceNormal(object):
    """Standard-normal draws made on the device (Philox4x32-10 keyed by ``seed``; the stream position lives in
    device memory and advances with every launch, so a captured CUDA graph draws fresh latents on every replay)."""

    def __init__(self, device, seed):
        self.seed = int(seed) & ((1 << 64) - 1)
        self.counter = torch.zeros(1, device=device, dtype=torch.int64)
        self.ticket = torch.zeros(1, device=device, dtype=torch.int32)

    def fill_(self, out):
        out = _req(out, "out")
        check(lib().ipr_randn_f32(_p(out), out.numel(), self.seed, _p(self.counter), _p(self.ticket), _stream()),
              "ipr_randn_f32")
        return out


# ------------------------------------------------------------------------------ verification
_DCT_CACHE = {}
_PTABLE_CACHE = {}


def pdq_dct_matrix(device):
    key = str(device)
    if key not in _DCT_CACHE:
        host = np.zeros((16, 64), dtype=np.float32)
        lib().ipr_pdq_dct_matrix_host(host.ctypes.data_as(ctypes.c_void_p))
        _DCT_CACHE[key] = torch.from_numpy(host).to(device)
    return _DCT_CACHE[key]


def pvalue_table_host(nbits=256):
    """1 - Binom(n, 1/2).cdf(r - 1) for r = 0..n, float64 -> float32: the same scipy call the
    reference makes per sample (tools/phash_pvalue.py:36), tabulated once."""
    from scipy.stats import binom
    r = np.arange(nbits + 1)
    return (1 - binom(n=nbits, p=0.5).cdf(r - 1)).astype(np.float32)


def pvalue_table(device):
    key = str(device)
    if key not in _PTABLE_CACHE:
        _PTABLE_CACHE[key] = torch.from_numpy(pvalue_table_host()).to(device)
    return _PTABLE_CACHE[key]


def bicubic_resize(x, hout, wout):
    x = _req(x, "x")
    B, C, H, W = x.shape
    out = torch.empty(B, C, hout, wout, device=x.device, dtype=x.dtype)
    check(lib().ipr_bicubic_resize_f32(_p(x), _p(out), B * C, H, W, hout, wout, _stream()),
          "ipr_bicubic_resize_f32")
    return out


def pdq_hash(img, want_coeffs=False):
    """img (B, 3, H, W) fp32 in [0, 1] -> (B, 8) int32 words (256-bit hashes)."""
    img = _req(img, "img")
    B, C, H, W = img.shape
    if C != 3:
        raise IprError("pdq_hash expects RGB images (B, 3, H, W)")
    h = torch.empty(B, 8, device=img.device, dtype=torch.int32)
    coeffs = torch.empty(B, 256, device=img.device, dtype=torch.float32) if want_coeffs else None
    check(lib().ipr_pdq_hash_f32(_p(img), _p(h), _p(coeffs) if want_coeffs else None,
                                 _p(pdq_dct_matrix(img.device)), B, H, W, _stream()), "ipr_pdq_hash_f32")
    return (h, coeffs) if want_coeffs else h


def hash_pvalue(hx, hy):
    """-> (p fp32 (B,), r int32 (B,))"""
    hx = _req(hx, "hx", torch.int32)
    hy = _req(hy, "hy", torch.int32)
    B = hx.shape[0]
    p = torch.empty(B, device=hx.device, dtype=torch.float32)
    r = torch.empty(B, device=hx.device, dtype=torch.int32)
    check(lib().ipr_hash_pvalue(_p(hx), _p(hy), _p(pvalue_table(hx.device)), _p(p), _p(r), B, _stream()),
          "ipr_hash_pvalue")
    return p, r


def matching_prob(img1, img2, min_size=32):
    """Device-side twin of tools.compute_matching_prob (tools/phash_pvalue.py:19-38):
    -> (p (B,), r (B,)) on the device."""
    x = _req(img1, "img1")
    y = _req(img2, "img2")
    k = min(x.shape[2:])
    if k < min_size:
        h = int(x.shape[2] * min_size / k)
        w = int(x.shape[3] * min_size / k)
        x = bicubic_resize(x, h, w)
        y = bicubic_resize(y, h, w)
    return hash_pvalue(pdq_hash(x), pdq_hash(y))


def unpack_hash_bits(h):
    """(B, 8) int32 words -> (B, 256) uint8 bits, bit k = 16*i + j of the DCT block (host helper for tests)."""
    words = h.detach().cpu().numpy().astype(np.uint32)
    return ((words[:, :, None] >> np.arange(32, dtype=np.uint32)[None, None, :]) & 1).reshape(words.shape[0], 256).astype(np.uint8)


# ------------------------------------------------------------------------------ robustness attacks
def prune_magnitude_(arena, segments, n_total, k):
    """Global magnitude pruning in place (csrc/prune.cu): zero the k entries of smallest |w| over the ``segments`` of
    the flat fp32 ``arena`` (ties: lowest index first).  segments: (S, 2) int64 CUDA tensor of ascending, disjoint
    (offset, count) rows whose counts sum to ``n_total``.  Nothing is read back: graph-capturable."""
    if not isinstance(arena, torch.Tensor) or not arena.is_cuda or arena.dtype != torch.float32 or not arena.is_contiguous():
        raise IprError("arena must be a contiguous float32 CUDA tensor (it is pruned in place)")
    segments = _req(segments, "segments", torch.int64)
    if segments.dim() != 2 or segments.shape[1] != 2 or segments.device != arena.device:
        raise IprError("segments must be an (S, 2) int64 tensor on the arena's device")
    nbytes = lib().ipr_prune_workspace_bytes(int(n_total))
    ws = torch.empty(max(1, nbytes), device=arena.device, dtype=torch.uint8)
    check(lib().ipr_prune_magnitude_f32(_p(arena), _p(segments), segments.shape[0], int(n_total), int(k), _p(ws), nbytes,
                                        _stream()), "ipr_prune_magnitude_f32")
    return arena


def negate_indexed_(arena, index):
    """arena[index] = -arena[index] in one launch (distinct int64 CUDA indices)."""
    if not isinstance(arena, torch.Tensor) or not arena.is_cuda or arena.dtype != torch.float32 or not arena.is_contiguous():
        raise IprError("arena must be a contiguous float32 CUDA tensor (it is changed in place)")
    index = _req(index, "index", torch.int64)
    if index.device != arena.device:
        raise IprError("index must be on the arena's device")
    check(lib().ipr_negate_indexed_f32(_p(arena), _p(index), index.numel(), _stream()), "ipr_negate_indexed_f32")
    return arena
