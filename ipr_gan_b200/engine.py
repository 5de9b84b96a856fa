"""Whole-network autograd nodes for the DCGAN generator / discriminator over the library's kernels.

``generator_forward(module, z)`` and ``discriminator_forward(module, x)`` are what the drop-in
``networks.ConvGenerator`` / ``networks.SNDiscriminator`` call on CUDA.  The module tree only holds
the parameters and buffers (reference ``state_dict`` format); the arithmetic runs here:

  generator      Linear+ReLU -> 3 x [ConvT k4s2 -> BatchNorm(batch stats) -> ReLU] -> ConvT k3s1 -> Tanh
                 (networks/conv_generator.py:13-27)
  discriminator  7 x [spectral-norm Conv + LeakyReLU(0.1)] -> spectral-norm Linear(8192 -> 1)
                 (networks/sn_discriminator.py:8-25)

Activations are NHWC bf16 between layers, fp32 NCHW at the module boundary; master weights fp32.
Every dense contraction (forward, data gradient, weight gradient) is a tcgen05 tap GEMM
(``dense.Plan`` / ``dense.WGradPlan``); normalisation, patch gathering and the final GEMV are the
kernels of csrc/nn_misc.cu.  Nothing here synchronises or allocates outside PyTorch's caching
allocator, so a whole training step can be captured in one CUDA graph.
"""
import ctypes

import os

import torch

from . import dense, flat
from ._lib import SnLayer
from ._lib import check, lib

BN_EPS_DEFAULT = 1e-5

# Test hook: when set to a list, every generator / discriminator forward appends the bf16 activations it stored
# (NHWC), so a parity test can hand the engine's own ReLU / LeakyReLU masks to the oracle (tests/test_gpu_dcgan.py).
CAPTURE_ACTS = None


def _st():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


# ----------------------------------------------------------------------------------------- kernel wrappers
def im2col3(x, tanh_out=None):
    B, C, H, W = x.shape
    assert C == 3 and x.dtype == torch.float32 and x.is_contiguous()
    out = torch.empty(B, H, W, 32, device=x.device, dtype=torch.bfloat16)
    check(lib().ipr_im2col3_bf16(_p(x), _p(tanh_out), _p(out), B, H, W, _st()), "ipr_im2col3_bf16")
    return out


def col2im3(t, tanh_out):
    """t: (B, H, W, ld) fp32 tap-expanded GEMM output -> (B, 3, H, W) fp32 (see csrc/nn_misc.cu: col2im3_kernel)."""
    B, H, W, ld = t.shape
    assert t.dtype == torch.float32 and t.is_contiguous()
    out = torch.empty(B, 3, H, W, device=t.device, dtype=torch.float32)
    check(lib().ipr_col2im3_f32(_p(t), _p(out), B, H, W, ld, int(bool(tanh_out)), _st()), "ipr_col2im3_f32")
    return out


IPR_E_UNSUPPORTED = -3


def tapfold3(a, b_packed, tanh_out, sigma=None):
    """The 3-output-channel 3x3 layer in one launch (csrc/tapfold.cu): a (B, H, W, 64) bf16 NHWC, b_packed the
    [1][32][64] ``_tap27_rows_layout`` pack -> (B, 3, H, W) fp32, bit-identical to ``col2im3`` of the tap GEMM.
    Returns None where the kernel does not cover the shape, or with IPR_NO_TAPFOLD=1 (A/B runs); the caller then
    runs the tap GEMM + ``col2im3``."""
    if os.environ.get("IPR_NO_TAPFOLD", "0") != "0":
        return None
    B, H, W, C = a.shape
    assert C == 64 and a.dtype == torch.bfloat16 and a.is_contiguous() and b_packed.dtype == torch.bfloat16
    out = torch.empty(B, 3, H, W, device=a.device, dtype=torch.float32)
    ev = dense._prof_begin()
    rc = lib().ipr_tapfold3_f32(_p(a), _p(b_packed), _p(sigma), _p(out), B, H, W, int(bool(tanh_out)), _st())
    if rc == IPR_E_UNSUPPORTED:
        return None
    check(rc, "ipr_tapfold3_f32")
    # the tap GEMM's useful flops (27 of 32 columns); the fold's adds are not counted
    dense._prof_end("tapfold:3ch", 2.0 * B * H * W * 64 * 27, ev, B * H * W * 128.0 + b_packed.numel() * 2)
    return out


def tapfold3_band(a, b_packed, tanh_out, sigma=None):
    """``tapfold3`` for images larger than one CTA stages (the 64 x 64 networks): the kernel folds bands of output
    rows, recomputing the GEMM-aligned sub-tile above and below each band for its halo rows, with the same results.
    Returns None where the kernel does not cover the shape, or with IPR_NO_TAPFOLD=1; the caller then runs the tap
    GEMM + ``col2im3``."""
    if os.environ.get("IPR_NO_TAPFOLD", "0") != "0":
        return None
    B, H, W, C = a.shape
    assert C == 64 and a.dtype == torch.bfloat16 and a.is_contiguous() and b_packed.dtype == torch.bfloat16
    out = torch.empty(B, 3, H, W, device=a.device, dtype=torch.float32)
    ev = dense._prof_begin()
    rc = lib().ipr_tapfold3_band_f32(_p(a), _p(b_packed), _p(sigma), _p(out), B, H, W, int(bool(tanh_out)), _st())
    if rc == IPR_E_UNSUPPORTED:
        return None
    check(rc, "ipr_tapfold3_band_f32")
    # counted as tapfold3 counts: the sub-tiles a band re-reads for its halo rows (a third more A at 64 x 64) are not
    dense._prof_end("tapfold:3ch", 2.0 * B * H * W * 64 * 27, ev, B * H * W * 128.0 + b_packed.numel() * 2)
    return out


def _fold3(a, b_packed, tanh_out, sigma=None):
    """The 3-output-channel 3x3 layer as one launch where a kernel covers the shape: whole images, then bands.
    None: the caller runs the tap GEMM + ``col2im3``."""
    out = tapfold3(a, b_packed, tanh_out, sigma=sigma)
    return out if out is not None else tapfold3_band(a, b_packed, tanh_out, sigma=sigma)


def colsum_partials(partial, out=None, accumulate=False, scale=1.0, ncols=None):
    """partial: [rows][row_stride] fp32 -> out[ncols] = column sums of the first ``ncols`` columns (fixed order)."""
    rows, stride = partial.shape[0], partial.numel() // partial.shape[0]
    ncols = stride if ncols is None else ncols
    if out is None:
        out = torch.empty(ncols, device=partial.device, dtype=torch.float32)
    nbytes = lib().ipr_colsum_workspace_bytes(ncols)
    ws = torch.empty(nbytes // 4, device=partial.device, dtype=torch.float32)
    check(lib().ipr_colsum_partials_f32(_p(partial), rows, ncols, stride, _p(out), int(bool(accumulate)), float(scale),
                                        _p(ws), nbytes, _st()), "ipr_colsum_partials_f32")
    return out


def colsum_bf16(x2d, out=None, accumulate=False, scale=1.0, out_index=None):
    """x2d: [rows][C] bf16 -> out[C] fp32 (column c lands at out[out_index[c]] when an int32 index is given;
    accumulate: False / True / 2 = atomic add)."""
    rows, C = x2d.shape
    if out is None:
        out = torch.empty(C, device=x2d.device, dtype=torch.float32)
    nbytes = lib().ipr_colsum_workspace_bytes(C)
    ws = torch.empty(nbytes // 4, device=x2d.device, dtype=torch.float32)
    check(lib().ipr_colsum_bf16(_p(x2d), rows, C, _p(out), int(accumulate), float(scale), _p(out_index), _p(ws), nbytes,
                                _st()), "ipr_colsum_bf16")
    return out


def bn_finalize(stats, count, bn, update_running):
    C = bn.num_features
    dev = stats.device
    if stats.shape[0] > 8:
        stats = colsum_partials(stats).view(1, 2, C)
    scale = torch.empty(C, device=dev)
    shift = torch.empty(C, device=dev)
    mean = torch.empty(C, device=dev)
    rstd = torch.empty(C, device=dev)
    momentum = bn.momentum if bn.momentum is not None else 0.1
    rm = bn.running_mean if update_running else None
    rv = bn.running_var if update_running else None
    nbt = bn.num_batches_tracked if update_running else None
    check(lib().ipr_bn_finalize_f32(_p(stats), stats.shape[0], C, float(count), float(bn.eps), float(momentum),
                                    _p(bn.weight.detach()), _p(bn.bias.detach()), _p(rm), _p(rv), _p(nbt),
                                    _p(scale), _p(shift), _p(mean), _p(rstd), _st()), "ipr_bn_finalize_f32")
    return scale, shift, mean, rstd


def bn_apply_relu(x, scale, shift):
    y = torch.empty_like(x)
    C = x.shape[-1]
    check(lib().ipr_bn_apply_relu_bf16(_p(x), _p(y), _p(scale), _p(shift), x.numel() // C, C, _st()),
          "ipr_bn_apply_relu_bf16")
    return y


def bn_relu_bwd(dy, xraw, scale, shift, gamma, mean, rstd, dgamma, dbeta, accumulate, sign=None, gamma0=0.0,
                sign_scale=0.0):
    C = dy.shape[-1]
    nbytes = lib().ipr_bn_bwd_workspace_bytes(C)
    ws = torch.empty(nbytes // 4, device=dy.device, dtype=torch.float32)
    dx = torch.empty_like(dy)
    check(lib().ipr_bn_relu_bwd_bf16(_p(dy), _p(xraw), _p(scale), _p(shift), _p(gamma), _p(mean), _p(rstd), _p(dx), _p(dgamma),
                                     _p(dbeta), int(accumulate), _p(sign), float(gamma0), float(sign_scale),
                                     _p(ws), nbytes, dy.numel() // C, C, _st()), "ipr_bn_relu_bwd_bf16")
    return dx


def dfc_fwd(a, w, sigma, bias):
    B, K = a.shape
    logits = torch.empty(B, device=a.device, dtype=torch.float32)
    check(lib().ipr_dfc_fwd_bf16(_p(a), _p(w), _p(sigma), _p(bias), _p(logits), B, K, _st()), "ipr_dfc_fwd_bf16")
    return logits


def dfc_bwd(a, w, sigma, dlogit, want_dw, slope, dw_index=None, dbias=None):
    """-> (da, dw).  dw_index (int32) scatters dw from the activation's feature order into the parameter's own order;
    dbias (a 1-element fp32 view) receives += sum(dlogit)."""
    B, K = a.shape
    da = torch.empty_like(a)
    dw = torch.empty(K, device=a.device, dtype=torch.float32) if want_dw else None
    check(lib().ipr_dfc_bwd_bf16(_p(a), _p(w), _p(sigma), _p(dlogit), _p(da), _p(dw), 0, float(slope), B, K,
                                 _p(dw_index) if want_dw else None, _p(dbias) if want_dw else None, _st()),
          "ipr_dfc_bwd_bf16")
    return da, dw


# ----------------------------------------------------------------------------------------- plan caches
def _ev_record(stream):
    """Event marking 'shared state updated on `stream`' (+ whether it was recorded inside a graph capture: captured
    events only mean something inside that capture, eager ones only outside)."""
    ev = torch.cuda.Event()
    ev.record(stream)
    return ev, stream, torch.cuda.is_current_stream_capturing()


def _ev_wait(rec, stream):
    if rec is not None and rec[1] != stream and rec[2] == torch.cuda.is_current_stream_capturing():
        stream.wait_event(rec[0])


class PackSet(object):
    """Every bf16 GEMM operand layout of one network, rebuilt from the network's fp32 parameter arena by ONE
    gather launch (csrc/optim.cu) whenever the masters changed."""

    def __init__(self, module, specs, specs_f32=()):
        # the arena the parameters already live in (an optimizer may have built one spanning several networks, e.g.
        # CycleGAN's optG over both generators), else one for this network alone
        params = list(module.parameters())
        arena = flat.arena_of(params[0])
        if arena is None or any(flat.arena_of(p) is not arena for p in params):
            arena = flat.arena_for(params)
        self.arena = arena
        dev = self.arena.param.device
        # fp32 side table: permuted fp32 copies (Linear bias in NHWC feature order, the final GEMV row), same launch
        parts32, self.slices32, off32 = [], {}, 0
        for key, param, layout_fn in specs_f32:
            o = self.arena.offset_of(param)
            src = (torch.arange(param.numel(), dtype=torch.float64) + o).view(param.shape)
            idx = layout_fn(src).reshape(-1).to(torch.int32)
            pad = (-idx.numel()) % 4
            self.slices32[key] = (off32, idx.numel())
            parts32.append(torch.cat([idx, torch.full((pad,), -1, dtype=torch.int32)]) if pad else idx)
            off32 += idx.numel() + pad
        self.index32 = torch.cat(parts32).to(dev) if parts32 else None
        self.buf32 = torch.empty(off32, device=dev, dtype=torch.float32) if parts32 else None
        parts, self.slices, off = [], {}, 0
        for key, param, layout_fn in specs:
            o = self.arena.offset_of(param)
            src = (torch.arange(param.numel(), dtype=torch.float64) + (o + 1)).view(param.shape)   # 0 = padding
            lay = layout_fn(src)
            idx = (lay.reshape(-1).to(torch.int64) - 1).to(torch.int32)
            n = idx.numel()
            pad = (-n) % 8
            if pad:
                idx = torch.cat([idx, torch.full((pad,), -1, dtype=torch.int32)])
            self.slices[key] = (off, n, tuple(lay.shape))
            parts.append(idx)
            off += n + pad
        self.index = torch.cat(parts).to(dev)
        self.buf = torch.empty(off, device=dev, dtype=torch.bfloat16)
        self.stamp = None
        self.event = None

    def refresh(self):
        # Parameters are views of the arena with their OWN version counters (flat.py: ``p.data = view``), so an
        # in-place write to one of them (load_state_dict, a stock torch optimizer, ``w[idx] = 0``) never shows in
        # ``arena.param._version``: stamp every parameter.  Writes through ``p.data`` bypass version counting
        # altogether -- callers that do that (sign_flip.py:74 does, before its first forward) call
        # ``engine.reset_caches()`` afterwards.
        stamp = (self.arena.version, self.arena.param._version) + tuple(p._version for p in self.arena.params)
        cur = torch.cuda.current_stream(self.buf.device)
        if stamp != self.stamp:
            check(lib().ipr_gather_pack_bf16(_p(self.arena.param), _p(self.index), _p(self.buf), self.buf.numel(),
                                             _p(self.index32), _p(self.buf32),
                                             self.buf32.numel() if self.buf32 is not None else 0, _st()),
                  "ipr_gather_pack_bf16")
            self.stamp = stamp
            self.event = _ev_record(cur)            # other streams (concurrent D(real) / D(fake) passes) wait for the pack
        else:
            _ev_wait(self.event, cur)

    def stale(self):
        return (self.arena.version, self.arena.param._version) + tuple(p._version for p in self.arena.params) != self.stamp

    def refresh_early(self, device):
        """Re-pack on a side stream NOW (if the masters changed), so that the gather overlaps whatever the caller
        enqueues next on its own stream; every later ``get`` waits for the recorded event.  Used by the discriminator,
        whose forward starts with the spectral-norm power iteration (fp32 masters only, ~40 us) right after Adam."""
        if not _USE_SIDE or not self.stale():
            return
        cur = torch.cuda.current_stream(device)
        key = ("pack", device.index if device.index is not None else torch.cuda.current_device())
        if key not in _SIDE_STREAMS:
            _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
        side = _SIDE_STREAMS[key]
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            self.refresh()

    def get(self, key):
        self.refresh()
        off, n, shape = self.slices[key]
        return self.buf[off:off + n].view(shape)

    def get32(self, key):
        self.refresh()
        off, n = self.slices32[key]
        return self.buf32[off:off + n]

    def clear(self):
        self.stamp = None
        self.event = None


_ALL_PACKS = []


_SN_EVENTS = {}                # id(DisPlans) -> event after the latest power iteration (orders SN state across streams)


def reset_caches():
    """Mark every packed-weight set stale (call before CUDA-graph capture so packing is part of the graph)."""
    for p in _ALL_PACKS:
        p.clear()
    _SN_EVENTS.clear()


def aux_stream(device):
    """Second compute stream of a device: models run independent network passes (D(real) next to G -> D(fake)) on
    it; inside a CUDA-graph capture the fork/join become graph branches."""
    key = ("aux", device.index if device.index is not None else torch.cuda.current_device())
    if key not in _SIDE_STREAMS:
        _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
    return _SIDE_STREAMS[key]


def concurrent_passes():
    return _USE_SIDE and os.environ.get("IPR_CONCURRENT_PASSES", "1") != "0"


def _col_off_patch27(n_is_first):
    """Column table for the 3-channel im2col layers: k = (kh*3+kw)*3 + c  ->  offset inside a (., 3, 3, 3) weight row."""
    off = torch.full((1, 32), -1, dtype=torch.int32)
    for kh in range(3):
        for kw in range(3):
            for c in range(3):
                off[0, (kh * 3 + kw) * 3 + c] = c * 9 + kh * 3 + kw
    return off


def _patch27_layout(w):
    """(n, 3, 3, 3)-shaped weight -> [1][64][32]: row n, column k = (kh*3+kw)*3 + c (conv: c = in channel of an
    (O, 3, kh, kw) weight; convT: c = out channel of an (I, 3, kh, kw) weight); columns 27..31 are zero."""
    m = torch.zeros(1, 64, 32, device=w.device, dtype=w.dtype)
    m[0, :, :27] = w.permute(0, 2, 3, 1).reshape(64, 27)
    return m


def _tap27_rows_layout(w):
    """(64, 3, 3, 3)-shaped weight whose first dimension is the contraction (ConvT (I, 3, kh, kw): I; Conv (O, 3, kh,
    kw) in its input gradient: O) -> [1][32][64]: row (kh*3+kw)*3 + c, column k; rows 27..31 are zero."""
    m = torch.zeros(1, 32, 64, device=w.device, dtype=w.dtype)
    m[0, :27] = w.permute(2, 3, 1, 0).reshape(27, 64)
    return m


class GenPlans(object):
    def __deepcopy__(self, memo):       # plans hold device buffers and events: a copied module builds its own
        return None

    def __init__(self, module):
        mg = module.mg
        self.mg = mg
        feat = 512 * mg * mg
        # NHWC position n' = hw*512 + c  <->  reference feature f = c*mg*mg + hw
        hw = torch.arange(mg * mg).view(-1, 1)
        c = torch.arange(512).view(1, -1)
        self.perm = (c * (mg * mg) + hw).reshape(-1)                    # perm[n'] = f
        self.fc = dense.Plan("linear", module.z_dim, feat)
        self.fc_wg = dense.WGradPlan(self.fc, (feat, module.z_dim), row_perm=self.perm)
        chans = (512, 256, 128, 64)
        self.ct = [dense.Plan("convT4s2", ci, co) for ci, co in zip(chans[:-1], chans[1:])]
        self.ct_dg = [dense.Plan("convT4s2_dgrad", co, ci) for ci, co in zip(chans[:-1], chans[1:])]
        self.ct_wg = [dense.WGradPlan(p, (p.cin, p.cout, 4, 4)) for p in self.ct]
        self.last = dense.Plan("linear", 64, 32)                       # tap-expanded last layer, folded by col2im3
        self.last.n_valid_flops = 27
        self.last_dg = dense.Plan("linear", 32, 64)                    # d(a3) = patches(dY) x W'  (patches stored 32 wide)
        self.last_wg = dense.WGradPlan(dense.Plan("linear", 32, 64), (64, 3, 3, 3), col_off=_col_off_patch27(True),
                                       s_n=27)
        self.last_dg.k_valid_override = 27            # flop accounting: 27 of the 64 patch columns carry data
        self.last_wg.k_valid_override = 27
        self._perm_dev = {}
        cv = module.convs
        perm = self.perm
        specs = [("fc", module.fc[0].weight, lambda w: self.fc.pack_layout(w, perm))]
        for i in range(3):
            specs.append(("ct%d" % i, cv[i][0].weight, self.ct[i].pack_layout))
            specs.append(("ct%d_dg" % i, cv[i][0].weight, self.ct_dg[i].pack_layout))
        specs.append(("ct3", cv[3].weight, _tap27_rows_layout))
        specs.append(("ct3_dg", cv[3].weight, _patch27_layout))
        self.packs = PackSet(module, specs, [("fcb", module.fc[0].bias, lambda b: b[perm])])
        _ALL_PACKS.append(self.packs)

    def perm_on(self, device):
        """int32 table: NHWC feature n' -> reference feature (scatter index of the kernels)"""
        key = str(device)
        if key not in self._perm_dev:
            self._perm_dev[key] = self.perm.to(device=device, dtype=torch.int32)
        return self._perm_dev[key]


class DisPlans(object):
    def __deepcopy__(self, memo):
        return None

    def __init__(self, module):
        md = module.md
        self.md = md
        specs = [("conv4s2", 64, 64), ("conv3", 64, 128), ("conv4s2", 128, 128), ("conv3", 128, 256),
                 ("conv4s2", 256, 256), ("conv3", 256, 512)]
        self.first = dense.Plan("linear", 32, 64)                      # patches(x) x W1  (patches stored 32 wide)
        self.first_wg = dense.WGradPlan(dense.Plan("linear", 32, 64), (64, 3, 3, 3), col_off=_col_off_patch27(False),
                                        s_n=27)
        self.first_dg = dense.Plan("linear", 64, 32)                   # tap-expanded input gradient, folded by col2im3
        self.first_dg.n_valid_flops = 27
        self.first.k_valid_override = 27
        self.first_wg.k_valid_override = 27
        self.conv = [dense.Plan(k, ci, co) for k, ci, co in specs]
        self.conv_dg = [dense.Plan(k + "_dgrad", co, ci) for k, ci, co in specs]
        self.conv_wg = [dense.WGradPlan(p, (p.cout, p.cin, 3 if p.kind == "conv3" else 4, 3 if p.kind == "conv3" else 4))
                        for p in self.conv]
        hw = torch.arange(md * md).view(-1, 1)
        c = torch.arange(512).view(1, -1)
        self.perm = (c * (md * md) + hw).reshape(-1)                    # NHWC feature n' -> reference feature
        self._perm_dev = {}
        layers = _sn_layers(module)
        pk = [("c0", layers[0].weight_orig, _patch27_layout), ("c0_dg", layers[0].weight_orig, _tap27_rows_layout)]
        for i in range(6):
            pk.append(("c%d" % (i + 1), layers[i + 1].weight_orig, self.conv[i].pack_layout))
            pk.append(("c%d_dg" % (i + 1), layers[i + 1].weight_orig, self.conv_dg[i].pack_layout))
        dperm = self.perm
        self.packs = PackSet(module, pk, [("w8", layers[7].weight_orig, lambda w: w.reshape(-1)[dperm])])
        _ALL_PACKS.append(self.packs)
        # power-iteration vectors of all layers in ONE buffer (the module's weight_u / weight_v become views), so a
        # forward snapshots them with a single copy; per-layer scratch slices for the batched SN kernels
        dev = layers[0].weight_orig.device
        sizes = []
        for l in layers:
            sizes += [l.weight_u.numel(), l.weight_v.numel()]
        self.uv = torch.empty(sum(sizes), device=dev, dtype=torch.float32)
        self.uv_off, off = [], 0
        with torch.no_grad():
            for l in layers:
                nu, nv = l.weight_u.numel(), l.weight_v.numel()
                self.uv[off:off + nu].copy_(l.weight_u)
                self.uv[off + nu:off + nu + nv].copy_(l.weight_v)
                l._buffers["weight_u"] = self.uv[off:off + nu]
                l._buffers["weight_v"] = self.uv[off + nu:off + nu + nv]
                self.uv_off.append((off, off + nu))
                off += nu + nv
        self.dims = [(l.weight_orig.shape[0], l.weight_orig.numel() // l.weight_orig.shape[0]) for l in layers]
        self.scr_off, off = [], 0
        for r, c2 in self.dims:
            self.scr_off.append(off)
            off += int(lib().ipr_sn_scratch_floats(r, c2))
        self.scratch_floats = off

    def uv_valid(self, layers):
        base = self.uv.data_ptr()
        return all(l.weight_u.data_ptr() == base + 4 * o[0] for l, o in zip(layers, self.uv_off))

    def perm_on(self, device):
        key = str(device)
        if key not in self._perm_dev:
            self._perm_dev[key] = self.perm.to(device=device, dtype=torch.int32)
        return self._perm_dev[key]

    def sn_table(self, layers, uv, sigma, grads=None, grad_outs=None, snap=None):
        arr = (SnLayer * 8)()
        for i, l in enumerate(layers):
            if snap is not None:
                arr[i].u_snap = snap.data_ptr() + 4 * self.uv_off[i][0]
                arr[i].v_snap = snap.data_ptr() + 4 * self.uv_off[i][1]
            arr[i].grad_out = grad_outs[i].data_ptr() if grad_outs is not None and grad_outs[i] is not None else None
            arr[i].w = l.weight_orig.data_ptr()
            arr[i].u = uv.data_ptr() + 4 * self.uv_off[i][0]
            arr[i].v = uv.data_ptr() + 4 * self.uv_off[i][1]
            arr[i].sigma = sigma.data_ptr() + 4 * i
            arr[i].grad = grads[i].data_ptr() if grads is not None else None
            arr[i].rows, arr[i].cols = self.dims[i]
            arr[i].scratch_off = self.scr_off[i]
        return arr


_SIDE_STREAMS = {}
_USE_SIDE = os.environ.get("IPR_SIDE_STREAM", "1") != "0"


N_SIDE = max(1, int(os.environ.get("IPR_SIDE_STREAMS", "4")))


class _Fork(object):
    """Runs the weight-gradient GEMMs (and their split-K reductions / bias column sums) of a backward pass on side
    streams so that they overlap the data-gradient chain.  Works the same eagerly and under stream capture (the waits
    become graph edges).  Tensors handed to a side stream are kept alive until ``join`` so the caching allocator cannot
    recycle them while that stream still reads them.

    There are ``N_SIDE`` side streams per device and every piece of work carries a ``key`` (its layer): work of one
    layer always lands on the same stream, so accumulations into that layer's slice of the gradient arena stay ordered
    -- also between two passes that back-propagate concurrently (D(real) / D(fake), adversarial / trigger pass) --
    while different layers proceed in parallel.  With ONE side stream the ~24 weight-gradient GEMMs and their ~24
    reductions of a step formed the longest dependency chain of the captured graph at 64 samples per GPU
    (scripts/graph_critical_path.py: 0.8 of 1.58 ms)."""

    def __init__(self, device):
        self.enabled = _USE_SIDE
        if not self.enabled:
            return
        self.main = torch.cuda.current_stream(device)
        d = device.index if device.index is not None else torch.cuda.current_device()
        self.sides = []
        for k in range(N_SIDE):
            key = d if k == 0 else ("side", d, k)
            if key not in _SIDE_STREAMS:
                _SIDE_STREAMS[key] = torch.cuda.Stream(device=device)
            self.sides.append(_SIDE_STREAMS[key])
        self.keep = []
        self.used = set()

    def run(self, fn, *tensors, key=0):
        if not self.enabled:
            return fn()
        k = key % len(self.sides)
        side = self.sides[k]
        side.wait_stream(self.main)                 # everything enqueued so far happens-before the side work
        with torch.cuda.stream(side):
            r = fn()
        self.keep.extend(tensors)
        self.used.add(k)
        return r

    def run_after_all(self, fn, *tensors):
        """Work that consumes the results of every side stream (the spectral-norm weight-gradient transform)."""
        if not self.enabled:
            return fn()
        first = self.sides[0]
        for k in sorted(self.used):
            if k != 0:
                first.wait_stream(self.sides[k])
        return self.run(fn, *tensors, key=0)

    def join(self):
        if self.enabled and self.used:
            for k in sorted(self.used):
                self.main.wait_stream(self.sides[k])
            self.keep = []
            self.used = set()


def _grad_dst(param):
    """Where a weight gradient goes: straight into the parameter's ``.grad`` arena view (accumulating, nothing is
    returned to autograd -- saves one add kernel and one temporary per parameter) or, without an arena, a fresh tensor
    that autograd accumulates itself.  -> (destination, accumulate, value returned from backward)"""
    g = param.grad
    if g is not None and g.is_contiguous() and flat.arena_of(param) is not None:
        return g, True, None
    t = torch.empty_like(param)
    return t, False, t


def _mark_dirty(module):
    """A backward pass wrote into the network's gradient arena: the next optimizer.zero_grad() has work to do."""
    a = flat.arena_of(next(module.parameters()))
    if a is not None:
        a.clean = False


def _plans(module, cls):
    p = getattr(module, "_ipr_plans", None)
    if p is not None:
        first = next(module.parameters())
        if p.packs.arena is not flat.arena_of(first) or (cls is DisPlans and not p.uv_valid(_sn_layers(module))):
            p = None                                # parameters / buffers were re-created (e.g. .to(device)): rebuild
    if p is None:
        p = cls(module)
        object.__setattr__(module, "_ipr_plans", p)
    return p


# ----------------------------------------------------------------------------------------- generator
class _GeneratorFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, z, fc_w, fc_b, w1, g1, b1, w2, g2, b2, w3, g3, b3, w4):
        if z.requires_grad:
            raise RuntimeError("ConvGenerator: a latent that requires grad is not on the IPR-GAN path (the node "
                               "returns no gradient for z); detach it")
        P = _plans(module, GenPlans)
        B = z.shape[0]
        mg = P.mg
        bns = [module.convs[i][1] for i in range(3)]
        # latents -> bf16 through the library's layout kernel (a (B, z, 1, 1) image is already "NHWC"): the captured
        # step then holds no ATen kernel at all
        zc = z.detach().contiguous()
        if zc.shape[1] % 8 == 0:
            a0 = torch.empty(B, 1, 1, zc.shape[1], device=zc.device, dtype=torch.bfloat16)
            check(lib().ipr_nchw_to_nhwc_bf16(_p(zc), None, _p(a0), B, zc.shape[1], 1, 1, zc.shape[1], _st()),
                  "ipr_nchw_to_nhwc_bf16")
        else:
            a0 = zc.to(torch.bfloat16).view(B, 1, 1, -1)
        h, _ = P.fc.run(a0, P.packs.get("fc"), epi=dense.EPI_BIAS_LRELU, slope=0.0, bias=P.packs.get32("fcb"))
        acts = [h.view(B, mg, mg, 512)]
        raws, means, rstds, scales, shifts = [], [], [], [], []
        ctx.eval_stats = False
        for i in range(3):
            bn = bns[i]
            # torch's rule (nn.BatchNorm2d.forward): batch statistics in training mode, or when there are no running
            # buffers at all.  DisableBatchNormStats (models/util.py:55-69) only clears ``track_running_stats`` -- the
            # buffers stay, so an eval-mode generator keeps using them; in training mode it stops them being updated.
            batch_stats = bn.training or (bn.running_mean is None and bn.running_var is None)
            if batch_stats:
                raw, stats = P.ct[i].run(acts[-1], P.packs.get("ct%d" % i), want_stats=True)
                count = raw.numel() // raw.shape[-1]
                update = bn.training and bn.track_running_stats
                scale, shift, mean, rstd = bn_finalize(stats, count, bn, update)
                acts.append(bn_apply_relu(raw, scale, shift))
            else:
                # eval: running statistics are known before the layer runs, so normalisation + ReLU ride in the GEMM
                # epilogue (relu(acc * scale[c] + shift[c])): no raw tensor, no second pass (the verification sweep
                # spent 17 % of its time in those passes)
                rstd = torch.rsqrt(bn.running_var + bn.eps)
                mean = bn.running_mean
                scale = (bn.weight.detach() * rstd).contiguous()
                shift = (bn.bias.detach() - mean * scale).contiguous()
                ctx.eval_stats = True
                raw, _ = P.ct[i].run(acts[-1], P.packs.get("ct%d" % i), epi=dense.EPI_BIAS_LRELU, slope=0.0, bias=shift,
                                     scale=scale)
                acts.append(raw)
            raws.append(raw)
            means.append(mean)
            rstds.append(rstd)
            scales.append(scale)
            shifts.append(shift)
        out = _fold3(acts[-1], P.packs.get("ct3"), True)
        if out is None:
            t9, _ = P.last.run(acts[-1], P.packs.get("ct3"), epi=dense.EPI_LINEAR_F32, n_valid=32)
            out = col2im3(t9, True)
        if CAPTURE_ACTS is not None:
            CAPTURE_ACTS.append(("G", list(acts)))
        ctx.module = module
        ctx.save_for_backward(a0, out, fc_w, w1, w2, w3, w4, g1, g2, g3, *acts, *raws, *means, *rstds, *scales, *shifts)
        return out

    @staticmethod
    def backward(ctx, dout):
        module = ctx.module
        P = _plans(module, GenPlans)
        sv = ctx.saved_tensors
        a0, out, fc_w, w1, w2, w3, w4, g1, g2, g3 = sv[:10]
        acts, raws, means, rstds = sv[10:14], sv[14:17], sv[17:20], sv[20:23]
        scales, shifts = sv[23:26], sv[26:29]
        cts, gammas = (w1, w2, w3), (g1, g2, g3)
        if ctx.eval_stats:
            raise RuntimeError("generator backward in eval mode (running statistics) is not on the training path")
        B = a0.shape[0]
        dev = a0.device
        # last layer: Tanh' fused into the patch gather, then one GEMM for d(a3) and one for dW4
        col = im2col3(dout.contiguous(), out)
        mod_c = module.convs
        fork = _Fork(dev)
        dw4, acc4, ret4 = _grad_dst(mod_c[3].weight)
        fork.run(lambda: P.last_wg.run(acts[3], col, dw4, accumulate=acc4), col, dw4, key=0)
        d_act, _ = P.last_dg.run(col, P.packs.get("ct3_dg"))
        dws, dgs, dbs = [None] * 3, [None] * 3, [None] * 3
        sign_hook = getattr(module, "_ipr_sign_hook", None)
        for i in (2, 1, 0):
            dg_t, acc_g, dgs[i] = _grad_dst(mod_c[i][1].weight)
            db_t, acc_b, dbs[i] = _grad_dst(mod_c[i][1].bias)
            if acc_g != acc_b:                       # one kernel writes both: keep them in the same mode
                dg_t = dgs[i] = torch.empty_like(gammas[i])
                db_t = dbs[i] = torch.empty_like(gammas[i])
                acc_g = False
            sg, g0, sc = (None, 0.0, 0.0)
            if sign_hook is not None:
                # white-box sign loss (tools/sign_model.py:42-49): d/dgamma rides in this layer's BatchNorm backward.
                # The hook hands each layer's sign vector out ONCE per armed step, so of the two generator passes
                # (G(z), G(trigger)) exactly one adds it.
                sg, g0, sc = sign_hook(i)
            # two generator passes may backpropagate on different streams: gamma / beta gradients are added
            # atomically (two contributions onto a zeroed slot: order-independent, hence still deterministic)
            dx = bn_relu_bwd(d_act, raws[i], scales[i], shifts[i], gammas[i], means[i], rstds[i], dg_t, db_t,
                             2 if acc_g else 0, sg, g0, sc)
            dw_t, acc_w, dws[i] = _grad_dst(mod_c[i][0].weight)
            fork.run(lambda i=i, dx=dx, dw_t=dw_t, acc_w=acc_w: P.ct_wg[i].run(dx, acts[i], dw_t, accumulate=acc_w), dx, dw_t,
                     key=1 + i)
            wd = P.packs.get("ct%d_dg" % i)
            if i > 0:
                d_act, _ = P.ct_dg[i].run(dx, wd)
            else:  # into the Linear's ReLU
                d_act, _ = P.ct_dg[i].run(dx, wd, epi=dense.EPI_MASK, slope=0.0, mask=acts[0])
        dh = d_act.view(B, 1, 1, -1)
        dfc_t, acc_fc, dfc_w = _grad_dst(module.fc[0].weight)
        fork.run(lambda: P.fc_wg.run(dh, a0, dfc_t, accumulate=acc_fc), dh, dfc_t, key=4)
        perm = P.perm_on(dev)
        db_t, acc_fb, dfc_b = _grad_dst(module.fc[0].bias)
        colsum_bf16(dh.view(B, -1), out=db_t, accumulate=2 if acc_fb else 0, out_index=perm)
        fork.join()
        _mark_dirty(module)
        return (None, None, dfc_w, dfc_b, dws[0], dgs[0], dbs[0], dws[1], dgs[1], dbs[1], dws[2], dgs[2], dbs[2], ret4)


def generator_forward(module, z):
    z = z.to(device=module.fc[0].weight.device, dtype=torch.float32)
    c = module.convs
    return _GeneratorFn.apply(module, z, module.fc[0].weight, module.fc[0].bias,
                              c[0][0].weight, c[0][1].weight, c[0][1].bias,
                              c[1][0].weight, c[1][1].weight, c[1][1].bias,
                              c[2][0].weight, c[2][1].weight, c[2][1].bias, c[3].weight)


# ----------------------------------------------------------------------------------------- discriminator
def _sn_layers(module):
    net = module.net
    return [net[0][0], net[0][2], net[1][0], net[1][2], net[2][0], net[2][2], net[3], net[6]]


class _DiscriminatorFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, module, param_grads, x, *params):
        P = _plans(module, DisPlans)
        layers = _sn_layers(module)
        ws, bs = params[0::2], params[1::2]
        B = x.shape[0]
        dev = x.device
        # spectral norm: one batched power iteration (training) / sigma evaluation (eval) for all 8 layers, in place
        # on the module's weight_u / weight_v buffers, then ONE copy snapshots the vectors for backward
        sigma = torch.empty(8, device=dev, dtype=torch.float32)
        scratch = torch.empty(P.scratch_floats, device=dev, dtype=torch.float32)
        cur = torch.cuda.current_stream(dev)
        P.packs.refresh_early(dev)                 # bf16 operand packing next to the power iteration below
        _ev_wait(_SN_EVENTS.get(id(P)), cur)       # a pass on another stream advanced u/v: keep the reference's order
        uv = torch.empty_like(P.uv)                # this forward's copy of u / v, written by the same kernels
        check(lib().ipr_sn_power_iter_f32(P.sn_table(layers, P.uv, sigma, snap=uv), 8, int(module.training), 1e-12,
                                          _p(scratch), _st()), "ipr_sn_power_iter_f32")
        _SN_EVENTS[id(P)] = _ev_record(cur)
        sig = [sigma[i:i + 1] for i in range(8)]
        # D(fake.detach()) and D(generated) see the same image in one step: when the model asks for it
        # (``module._ipr_keep_col``, set by dropin/models/dcgan.py around D(fake)) the patch matrix is handed over on the
        # tensor object itself, so its lifetime is the image's lifetime.  Never stashed implicitly: a persistent input
        # buffer (the trainer's static ``real`` tensor) would otherwise carry a patch matrix of an OLD batch into a
        # CUDA-graph capture, where the version check below cannot see the replay-time copies.
        stash = getattr(x, "_ipr_col", None)
        if stash is not None and stash[1] == x._version and stash[0].shape[0] == B and stash[0].device == dev:
            col = stash[0]
        else:
            col = im2col3(x.detach().contiguous())
            if getattr(module, "_ipr_keep_col", False):
                try:
                    x._ipr_col = (col, x._version)     # an in-place edit of the image bumps _version and voids it
                except Exception:
                    pass
        a, _ = P.first.run(col, P.packs.get("c0"), epi=dense.EPI_BIAS_LRELU, slope=0.1, sigma=sig[0], bias=bs[0].detach())
        acts = [a]
        for i, plan in enumerate(P.conv):
            a, _ = plan.run(acts[-1], P.packs.get("c%d" % (i + 1)), epi=dense.EPI_BIAS_LRELU, slope=0.1, sigma=sig[i + 1],
                            bias=bs[i + 1].detach())
            acts.append(a)
        w8 = P.packs.get32("w8")
        logits = dfc_fwd(acts[-1].view(B, -1), w8, sig[7], bs[7].detach())
        if CAPTURE_ACTS is not None:
            CAPTURE_ACTS.append(("D", list(acts)))
        ctx.module, ctx.param_grads = module, param_grads
        ctx.x_needs_grad = x.requires_grad
        ctx.save_for_backward(col, w8, sigma, uv, *ws, *acts)
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        module = ctx.module
        P = _plans(module, DisPlans)
        layers = _sn_layers(module)
        sv = ctx.saved_tensors
        col, w8, sigma, uv = sv[:4]
        ws, acts = sv[4:12], sv[12:19]
        sig = [sigma[i:i + 1] for i in range(8)]
        want = ctx.param_grads
        B = col.shape[0]
        dev = col.device
        dlogits = dlogits.contiguous().float()
        gW, gB = [None] * 8, [None] * 8
        gW_ret = {}
        a7 = acts[-1].view(B, -1)
        db8 = None
        if want:
            db8, acc8, gB[7] = _grad_dst(layers[7].bias)
            if not acc8:
                db8.zero_()
        dy, dw8 = dfc_bwd(a7, w8, sig[7], dlogits, want, 0.1, dw_index=P.perm_on(dev), dbias=db8)
        if want:
            gW[7] = dw8.view(1, -1)
        dy = dy.view(acts[-1].shape)
        fork = _Fork(dev)
        if want:
            dst, acc, gB[6] = _grad_dst(layers[6].bias)
            fork.run(lambda dy=dy, dst=dst, acc=acc: colsum_bf16(dy.view(-1, dy.shape[-1]), out=dst, accumulate=acc), dy, dst,
                     key=0)
        for i in range(5, -1, -1):                 # conv layers 7..2 (index i+1 in the layer list)
            li = i + 1
            if want:
                gW[li] = torch.empty_like(ws[li])
                fork.run(lambda i=i, dy=dy, g=gW[li]: P.conv_wg[i].run(dy, acts[i], g), dy, key=1 + i)
            # the data-gradient GEMM's epilogue also yields the column sums of its output = the bias gradient below
            dy, st = P.conv_dg[i].run(dy, P.packs.get("c%d_dg" % li), epi=dense.EPI_MASK, slope=0.1, mask=acts[i],
                                      sigma=sig[li], want_stats=want)
            if want:
                dst, acc, gB[i] = _grad_dst(layers[i].bias)
                fork.run(lambda st=st, dst=dst, acc=acc, n=dy.shape[-1]: colsum_partials(st, out=dst, accumulate=acc, ncols=n),
                         st, dst, key=2 + i)
        dx = None
        if ctx.x_needs_grad:
            dx = _fold3(dy, P.packs.get("c0_dg"), False, sigma=sig[0])
            if dx is None:
                t9, _ = P.first_dg.run(dy, P.packs.get("c0_dg"), epi=dense.EPI_LINEAR_F32, sigma=sig[0], n_valid=32)
                dx = col2im3(t9, False)
        if want:
            gW[0] = torch.empty_like(ws[0])
            fork.run(lambda: P.first_wg.run(dy, col, gW[0]), dy, key=0)
            # gradients so far are w.r.t. W / sigma: one batched kernel pair turns them into d/dW_orig.  It accumulates
            # into the gradient arena, so it runs on the shared side stream: two passes backpropagating concurrently on
            # different streams (D(real), D(fake)) then never race on the arena.
            outs = []
            for i, l in enumerate(layers):
                dst, acc, ret = _grad_dst(l.weight_orig)
                outs.append(dst if acc else None)
                if acc:
                    gW_ret[i] = None

            def _sn_grad():
                scratch = torch.empty(P.scratch_floats, device=dev, dtype=torch.float32)
                check(lib().ipr_sn_weight_grad_f32(P.sn_table(layers, uv, sigma, gW, outs), 8, _p(scratch), _st()),
                      "ipr_sn_weight_grad_f32")
                return scratch
            keep = fork.run_after_all(_sn_grad, *[g for g in gW if g is not None])
            fork.join()
            _mark_dirty(module)
        grads = []
        for i in range(8):
            grads += [gW_ret[i] if (want and i in gW_ret) else gW[i], gB[i]]
        return (None, None, dx, *grads)


def discriminator_forward(module, x):
    layers = _sn_layers(module)
    x = x.to(device=layers[0].weight_orig.device, dtype=torch.float32)
    params = []
    for l in layers:
        params += [l.weight_orig, l.bias]
    want = not getattr(module, "_ipr_skip_param_grads", False)
    return _DiscriminatorFn.apply(module, want, x, *params)


# ----------------------------------------------------------------------------------------- smoke
def smoke_step(orc):
    """One tiny generator/discriminator forward+backward on cuda:0 against the oracle's fp32 networks
    (bf16 tolerance 2e-2 of the tensor scale)."""
    import networks
    torch.manual_seed(7)
    G = networks.ConvGenerator32().cuda()
    D = networks.SNDiscriminator32().cuda()
    Go, Do = orc.make_generator(), orc.make_discriminator()
    Go.load_state_dict(G.state_dict())
    Do.load_state_dict(D.state_dict())
    z = torch.randn(8, 128)
    fake = generator_forward(G, z.cuda())
    logits = discriminator_forward(D, fake)
    (-logits.mean()).backward()
    fo = Go(z)
    lo = Do(fo)
    (-lo.mean()).backward()

    def rel(a, b):
        a, b = a.detach().cpu().float(), b.detach().float()
        return float((a - b).norm() / (b.norm() + 1e-12))

    assert rel(fake, fo) < 2e-2, rel(fake, fo)
    assert rel(logits, lo) < 6e-2, rel(logits, lo)      # two chained bf16 networks
