"""Dense-layer plans over the tap-GEMM kernel (csrc/gemm_tc.cu): how each convolution / transposed
convolution / linear layer of the DCGAN networks, and each of their data gradients, is expressed as
taps (shifted TMA boxes) + a packed bf16 weight matrix.

Activations are NHWC bf16 inside the engine; weights stay fp32 masters in the reference's layouts
(Conv2d: (O, I, kh, kw); ConvTranspose2d: (I, O, kh, kw); Linear: (O, I)) and are re-packed to bf16
"[phase][n][tap*C + c]" matrices after every optimizer step.
"""
import ctypes

import torch

from ._lib import MAX_PHASES, MAX_TAPS, TapGemm, WGrad, check, lib  # noqa: F401 (MAX_* and the structs re-exported)

# When set to a list, every GEMM launch appends (kind, algorithmic_flops, start_event, end_event): bench.py uses
# it for the live tensor-roofline measurement (CUDA events on the launching stream).
PROFILE = None
PROFILE_DETAIL = False         # scripts/gemm_detail.py: append the layer shape to the kind label


def _prof_begin():
    if PROFILE is None:
        return None
    ev = torch.cuda.Event(enable_timing=True)
    ev.record()
    return ev


def _prof_end(kind, flops, start, l2_bytes=0.0):
    if start is None:
        return
    ev = torch.cuda.Event(enable_timing=True)
    ev.record()
    PROFILE.append((kind, flops, start, ev))
    if PROFILE_L2 is not None:
        PROFILE_L2.append((kind, l2_bytes))


# Same order as PROFILE: (kind, bytes the launch's TMA loads pull through L2 into shared memory) -- the operand stream
# that bounds the low-arithmetic-intensity tiles (every tile re-reads its A box per tap and its B block per k-block).
PROFILE_L2 = None
EPI_LINEAR, EPI_BIAS_LRELU, EPI_MASK, EPI_TANH_NCHW, EPI_LINEAR_F32, EPI_LINEAR_NCHW = 0, 1, 2, 3, 4, 5


# stride-2, k=4, pad=1: kernel row kh reads input row 2*o + kh - 1 = 2*(o + d) + parity
_S2 = {0: (1, -1), 1: (0, 0), 2: (1, 0), 3: (0, 1)}          # kh -> (parity, d)
# k4 s2 p1 transposed conv: output row 2*q + r gathers kernel rows kh at input row q + d
_T2 = {0: ((1, 0), (3, -1)), 1: ((0, 1), (2, 0))}             # r -> ((kh, d), (kh, d))


def pick_block_n(n):
    for bn in (256, 128, 64, 32, 16):
        if n % bn == 0:
            return bn
    raise ValueError("N must be a multiple of 16, got %d" % n)


class Plan(object):
    """Static description of one tap-GEMM layer: tap tables, phases, output mapping, weight packer."""

    def __init__(self, kind, cin, cout, n_pad=None):
        self.kind, self.cin, self.cout = kind, cin, cout
        self.n_total = n_pad or cout
        self.block_n = pick_block_n(self.n_total)
        self.a_parity, self.n_phases = 0, 1
        self.out_s, self.out_o = 1, [(0, 0)] * 4
        k = kind
        if k in ("conv3", "conv3_dgrad", "convT3"):
            # conv3: in row = o + kh - 1; the other two: in row = o + 1 - kh
            flip = k != "conv3"
            self.taps = [[(0, (1 - kh) if flip else (kh - 1), (1 - kw) if flip else (kw - 1), kh, kw)
                          for kh in range(3) for kw in range(3)]]
        elif k in ("conv4s2", "convT4s2_dgrad"):
            self.a_parity = 1
            self.taps = [[(2 * _S2[kh][0] + _S2[kw][0], _S2[kh][1], _S2[kw][1], kh, kw)
                          for kh in range(4) for kw in range(4)]]
        elif k in ("convT4s2", "conv4s2_dgrad"):
            self.n_phases, self.out_s = 4, 2
            self.taps, self.out_o = [], []
            for rh in range(2):
                for rw in range(2):
                    self.taps.append([(0, dh, dw, kh, kw) for (kh, dh) in _T2[rh] for (kw, dw) in _T2[rw]])
                    self.out_o.append((rh, rw))
        elif k == "linear":
            self.taps = [[(0, 0, 0, 0, 0)]]
        else:
            raise ValueError(kind)
        self.n_taps = len(self.taps[0])

    # weight (reference layout) -> [phase][n_total][taps*cin] in the SAME dtype (zeros where padded); works on
    # index tensors too, which is how the gather tables of engine.PackSet are derived
    def pack_layout(self, w, perm=None):
        k = self.kind
        if k == "linear":
            m = w if perm is None else w[perm]
            mats = [m]                                               # (N, K)
        else:
            mats = []
            for taps in self.taps:
                cols = []
                for (_, _, _, kh, kw) in taps:
                    if k in ("conv3", "conv4s2"):                    # Conv2d weight (O, I, kh, kw): n = O, c = I
                        cols.append(w[:, :, kh, kw])
                    elif k in ("conv3_dgrad", "conv4s2_dgrad"):      # n = I, c = O
                        cols.append(w[:, :, kh, kw].t())
                    elif k in ("convT3", "convT4s2"):                # ConvT weight (I, O, kh, kw): n = O, c = I
                        cols.append(w[:, :, kh, kw].t())
                    else:                                            # convT4s2_dgrad: n = I, c = O
                        cols.append(w[:, :, kh, kw])
                mats.append(torch.cat(cols, dim=1))
        out = torch.zeros(self.n_phases, self.n_total, mats[0].shape[1], device=w.device, dtype=w.dtype)
        for i, m in enumerate(mats):
            out[i, :m.shape[0]] = m
        return out.contiguous()

    def pack(self, w, perm=None):
        return self.pack_layout(w, perm).to(torch.bfloat16)

    def out_hw(self, a_h, a_w):
        if self.kind in ("conv4s2", "convT4s2_dgrad"):
            return a_h // 2, a_w // 2
        if self.kind in ("convT4s2", "conv4s2_dgrad"):
            return a_h * 2, a_w * 2
        return a_h, a_w

    def run(self, a, b_packed, epi=EPI_LINEAR, slope=0.0, sigma=None, bias=None, mask=None, out=None,
            want_stats=False, n_valid=None, out_nchw_c=None, scale=None):
        """a: (N, H, W, C) bf16 NHWC.  Returns (out, stats or None)."""
        L = lib()
        assert a.dtype == torch.bfloat16 and a.is_cuda and a.is_contiguous() and a.dim() == 4
        N, H, W, C = a.shape
        assert C == self.cin, (C, self.cin)
        oh, ow = self.out_hw(H, W)
        # static part of the descriptor (tap tables, phases, strides) is filled once per plan and copied: the per-call
        # Python cost of the eager paths is dominated by ctypes field stores (up to 200 for a 16-tap layer)
        tmpl = getattr(self, "_tmpl", None)
        if tmpl is None:
            tmpl = TapGemm()
            tmpl.a_parity = self.a_parity
            tmpl.n_total, tmpl.n_phases, tmpl.n_taps = self.n_total, self.n_phases, self.n_taps
            for ph, taps in enumerate(self.taps):
                for t, (mp, dh, dw, _, _) in enumerate(taps):
                    tmpl.tap_map[ph][t], tmpl.tap_dh[ph][t], tmpl.tap_dw[ph][t] = mp, dh, dw
                tmpl.out_oh[ph], tmpl.out_ow[ph] = self.out_o[ph]
            tmpl.out_sh = tmpl.out_sw = self.out_s
            self._tmpl = tmpl
        d = TapGemm.from_buffer_copy(tmpl)
        d.a, d.a_n, d.a_h, d.a_w, d.a_c = a.data_ptr(), N, H, W, C
        d.q_h, d.q_w = (H // 2, W // 2) if self.a_parity else (H, W)
        # tile width: the kernel is paced by TMA row requests (128 A rows + BLOCK_N B rows per k-block and tile) and runs
        # one persistent CTA per SM, so pick the N tile that minimises  waves(tiles / SMs) * (128 + BLOCK_N)
        m_pix = N * ((H // 2) * (W // 2) if self.a_parity else H * W)
        m_tiles = (m_pix + 127) // 128
        block_n, best = self.block_n, None
        cache = self.__dict__.setdefault("_bn_cache", {})
        bn = self.block_n if (m_tiles, C) not in cache else 0
        if bn == 0:
            block_n = cache[(m_tiles, C)]
        while bn >= 16:
            if self.n_total % bn == 0:
                tiles = m_tiles * (self.n_total // bn) * self.n_phases
                b_all = self.n_phases * self.n_taps * C * bn * 2
                resident = bn == self.n_total and b_all <= 132 * 1024 and tiles >= 2 * _sm_count()   # weights stay in smem
                cost = -(-tiles // _sm_count()) * (128 + (0 if resident else bn)) * (1.0 if bn >= 64 else 1.5)
                if best is None or cost < best:
                    best, block_n = cost, bn
            bn //= 2
        cache[(m_tiles, C)] = block_n
        d.b, d.block_n = b_packed.data_ptr(), block_n
        d.epi_mode, d.slope = epi, float(slope)
        d.sigma = sigma.data_ptr() if sigma is not None else None
        d.bias = bias.data_ptr() if bias is not None else None
        d.mask = mask.data_ptr() if mask is not None else None
        d.scale = scale.data_ptr() if scale is not None else None
        assert scale is None or epi == EPI_BIAS_LRELU
        nv = n_valid or self.cout
        if out is None:
            if epi in (EPI_TANH_NCHW, EPI_LINEAR_NCHW):
                out = torch.empty(N, nv, oh, ow, device=a.device, dtype=torch.float32)
            elif epi == EPI_LINEAR_F32:
                out = torch.empty(N, oh, ow, nv, device=a.device, dtype=torch.float32)
            else:
                out = torch.empty(N, oh, ow, nv, device=a.device, dtype=torch.bfloat16)
        d.out, d.out_h, d.out_w = out.data_ptr(), oh, ow
        d.out_c = out.shape[1] if epi in (EPI_TANH_NCHW, EPI_LINEAR_NCHW) else out.shape[3]
        d.n_valid = nv
        stats = None
        if want_stats:
            rows = L.ipr_tapgemm_stats_rows(ctypes.byref(d))
            if rows < 0:
                check(rows, "ipr_tapgemm_stats_rows")
            stats = torch.empty(rows, 2, self.n_total, device=a.device, dtype=torch.float32)
            d.stats = stats.data_ptr()
        ev = _prof_begin()
        check(L.ipr_tapgemm_bf16(ctypes.byref(d), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)),
              "ipr_tapgemm_bf16(%s)" % self.kind)
        label = "tapgemm:" + self.kind
        if PROFILE_DETAIL:
            label += " %d->%d rows=%d taps=%dx%d bn=%d epi=%d" % (C, self.cout, m_pix, self.n_phases, self.n_taps, block_n, epi)
        l2 = 0.0
        if ev is not None:
            tiles = m_tiles * (self.n_total // block_n) * self.n_phases
            cw = min(64, C) * 2                                               # bytes of one operand row inside a k-block
            kb = self.n_taps * ((C + 63) // 64)
            b_all = self.n_phases * self.n_taps * C * block_n * 2
            resident = block_n == self.n_total and b_all <= 132 * 1024 and tiles >= 2 * _sm_count()
            l2 = tiles * kb * 128 * cw + (min(tiles, _sm_count()) * b_all if resident else tiles * kb * block_n * cw)
        _prof_end(label, 2.0 * N * d.q_h * d.q_w * self.n_phases * self.n_taps * self.k_valid() *
                  getattr(self, "n_valid_flops", nv), ev, l2)
        return out, stats

    def k_valid(self):
        """Channels per tap that carry data (the 3-channel patch layers pad 27 -> 64)."""
        return getattr(self, "k_valid_override", self.cin)


_SM_COUNT_CACHE = []


def _sm_count():
    """SMs of the current device (148 on B200), as the C side's ipr_sm_count() sees them; 148 without a device
    (host-logic tests of the planning code)."""
    if not _SM_COUNT_CACHE:
        n = 148
        if torch.cuda.is_available():
            n = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
        _SM_COUNT_CACHE.append(n)
    return _SM_COUNT_CACHE[0]


# Weight matrices with at least this many (row, input channel) pairs reduce their split-K partials destination-major
# (ipr_wgrad_reduce_taps_f32); smaller ones, with many splits and few threads, are faster element-major.
_REDUCE_TAPS_MIN = 32768


class WGradPlan(object):
    """Weight gradient of the layer described by a forward Plan (conv3 / conv4s2 / convT4s2 / linear).

    ``y`` is the gradient w.r.t. the layer output (NHWC bf16), ``x`` the layer input (NHWC bf16); the result
    is written into ``grad`` which has the parameter's own fp32 layout."""

    def __init__(self, fwd, weight_shape, row_perm=None, col_off=None, s_n=None):
        self.fwd = fwd
        k = fwd.kind
        assert k in ("conv3", "conv4s2", "convT4s2", "linear"), k
        self.y_parity = 1 if k == "convT4s2" else 0
        self.x_parity = fwd.a_parity
        self.n_phases, self.n_taps = fwd.n_phases, fwd.n_taps
        self.rows = fwd.cout                      # rows of dW in GEMM layout (n)
        self.x_c = fwd.cin
        self.k_total = self.n_taps * self.x_c
        self.row_perm = row_perm
        self._plain = col_off is None and k != "linear"
        if col_off is None:
            col_off = torch.full((self.n_phases, self.k_total), -1, dtype=torch.int32)
            if k == "linear":
                col_off[0] = torch.arange(self.k_total, dtype=torch.int32)
                s_n = weight_shape[1]
            else:
                ksz = weight_shape[-1]
                c = torch.arange(self.x_c, dtype=torch.int32)
                for ph, taps in enumerate(fwd.taps):
                    for t, (_, _, _, kh, kw) in enumerate(taps):
                        if k == "convT4s2":        # (I, O, kh, kw): n = O (stride k*k), c = I (stride O*k*k)
                            col_off[ph, t * self.x_c:(t + 1) * self.x_c] = c * (weight_shape[1] * ksz * ksz) + kh * ksz + kw
                        else:                      # (O, I, kh, kw): n = O (stride I*k*k), c = I (stride k*k)
                            col_off[ph, t * self.x_c:(t + 1) * self.x_c] = c * (ksz * ksz) + kh * ksz + kw
                s_n = ksz * ksz if k == "convT4s2" else weight_shape[1] * ksz * ksz
        self.s_n = int(s_n)
        self.dst_off_host = col_off.reshape(-1).to(torch.int32).contiguous()   # [phase * k_total + k] -> offset in a row
        self._dev = {}
        # plain conv / convT weights: destination-major reduction (contiguous writes), tap j = kh*ksz + kw <- (phase, tap)
        self.tap_of = None
        if self._plain:
            ksz = weight_shape[-1]
            kk = ksz * ksz
            tap_of = [-1] * kk
            for ph, taps in enumerate(fwd.taps):
                for t, (_, _, _, kh, kw) in enumerate(taps):
                    tap_of[kh * ksz + kw] = ph * self.n_taps + t
            if kk == self.n_phases * self.n_taps and min(tap_of) >= 0 and row_perm is None and \
                    self.rows * self.x_c >= _REDUCE_TAPS_MIN:
                self.tap_of = (ctypes.c_int32 * kk)(*tap_of)
                self.kk = kk
                if k == "convT4s2":
                    self.s_n_t, self.s_c_t = kk, weight_shape[1] * kk
                else:
                    self.s_n_t, self.s_c_t = weight_shape[1] * kk, kk

    def _tables(self, device):
        key = str(device)
        if key not in self._dev:
            rp = self.row_perm.to(device=device, dtype=torch.int32).contiguous() if self.row_perm is not None else None
            self._dev[key] = (self.dst_off_host.to(device), rp)
        return self._dev[key]

    def run(self, y, x, grad, accumulate=False, scale=1.0, splits=None):
        L = lib()
        assert y.dtype == torch.bfloat16 and x.dtype == torch.bfloat16 and y.is_contiguous() and x.is_contiguous()
        assert grad.dtype == torch.float32 and grad.is_contiguous()
        N, xh, xw, xc = x.shape
        assert xc == self.x_c and y.shape[3] == self.rows, (x.shape, y.shape, self.x_c, self.rows)
        tmpl = getattr(self, "_tmpl", None)
        if tmpl is None:                             # static part of the descriptor, filled once (see Plan.run)
            tmpl = WGrad()
            tmpl.y_parity, tmpl.x_parity = self.y_parity, self.x_parity
            tmpl.n_phases, tmpl.n_taps = self.n_phases, self.n_taps
            for ph, taps in enumerate(self.fwd.taps):
                for t, (mp, dh, dw, _, _) in enumerate(taps):
                    tmpl.tap_map[ph][t], tmpl.tap_dh[ph][t], tmpl.tap_dw[ph][t] = mp, dh, dw
                tmpl.y_map[ph] = (2 * self.fwd.out_o[ph][0] + self.fwd.out_o[ph][1]) if self.y_parity else 0
            self._tmpl = tmpl
        d = WGrad.from_buffer_copy(tmpl)
        d.y, d.y_c = y.data_ptr(), y.shape[3]
        d.x, d.x_c = x.data_ptr(), xc
        d.n_imgs = N
        d.q_h, d.q_w = (xh // 2, xw // 2) if self.x_parity else (xh, xw)
        kblocks = L.ipr_wgrad_total_kblocks(ctypes.byref(d))
        if kblocks < 0:
            check(kblocks, "ipr_wgrad_total_kblocks")
        if splits is None:
            tiles = L.ipr_wgrad_tiles(ctypes.byref(d))
            # one CTA per SM (about 200 KB of smem stages): never exceed one wave, a second partial wave doubles the time
            splits = max(1, min(kblocks // 4 if kblocks >= 8 else 1, _sm_count() // tiles))
        d.splits = splits
        nbytes = L.ipr_wgrad_workspace_bytes(ctypes.byref(d))
        ws = torch.empty(nbytes // 4, device=x.device, dtype=torch.float32)
        d.workspace = ws.data_ptr()
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        ev = _prof_begin()
        check(L.ipr_wgrad_bf16(ctypes.byref(d), st), "ipr_wgrad_bf16(%s)" % self.fwd.kind)
        label = "wgrad:" + self.fwd.kind
        if PROFILE_DETAIL:
            label += " %d->%d rows=%d taps=%dx%d splits=%d" % (xc, self.rows, N * d.q_h * d.q_w, self.n_phases, self.n_taps, splits)
        l2 = 0.0
        if ev is not None:
            tiles = L.ipr_wgrad_tiles(ctypes.byref(d))
            m_blks = max(1, (self.rows + 127) // 128)
            n_units = self.n_taps * ((xc + 63) // 64)
            # per 64-pixel k-block: two 8 KB Y boxes per CTA tile, one 8 KB X box per (tap, 64-channel) unit and M block
            l2 = float(self.n_phases) * kblocks * 8192.0 * (2 * tiles + n_units * m_blks)
        _prof_end(label, 2.0 * N * d.q_h * d.q_w * self.n_phases * self.n_taps *
                  getattr(self, "k_valid_override", xc) * getattr(self, "rows_valid_override", self.rows), ev, l2)
        if self.tap_of is not None:
            check(L.ipr_wgrad_reduce_taps_f32(ws.data_ptr(), splits, self.n_phases, self.rows, self.n_taps, self.x_c,
                                              self.tap_of, self.kk, self.s_n_t, self.s_c_t, grad.data_ptr(),
                                              int(bool(accumulate)), float(scale), st), "ipr_wgrad_reduce_taps_f32")
            return grad
        dst_off, row_map = self._tables(x.device)
        check(L.ipr_wgrad_reduce_f32(ws.data_ptr(), splits, self.n_phases, self.rows, self.k_total,
                                     dst_off.data_ptr(),
                                     row_map.data_ptr() if row_map is not None else None,
                                     self.s_n, grad.data_ptr(), int(bool(accumulate)), float(scale), st),
              "ipr_wgrad_reduce_f32")
        return grad
