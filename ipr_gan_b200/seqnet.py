"""Native execution of the SRGAN / CycleGAN network families (SURVEY.md K17):

  SRResNet          networks/sr_resnet.py:3-44        Discriminator96    networks/discriminator_96.py:3-35
  ResnetGenerator   networks/resnet_generator.py:3-59 ConvDiscriminator  networks/conv_discriminator.py:3-21

The module tree (same ``state_dict`` as the reference) is *lowered* once into a list of blocks

    [ReflectionPad] Conv2d | ConvTranspose2d  ->  [BatchNorm2d | InstanceNorm2d]  ->  [PixelShuffle(2)]
                                             ->  [ReLU | LeakyReLU | PReLU | Tanh]  ->  [+ skip]

and the whole network runs as ONE autograd node over the library's kernels: every convolution is a patch matrix
(``ipr_im2col_nhwc_bf16``: any kernel size / stride / zero or reflection border / transposed) times the packed bf16
weight on the tcgen05 GEMM, its data gradient the GEMM with the transposed weight folded back by the adjoint gather,
its weight gradient the tcgen05 weight-gradient GEMM over the same patch matrix; normalisation + activation
(+ residual) forward and backward are the kernels of csrc/layers.cu, with the white-box sign-loss gradient added
inside the normalisation backward.  NHWC bf16 inside, NCHW fp32 at the module boundary; no PyTorch-op path.
"""
import ctypes

import torch
import torch.nn as nn

from . import dense, engine, flat
from ._lib import check, lib

ACT_NONE, ACT_RELU, ACT_LRELU, ACT_PRELU, ACT_TANH = 0, 1, 2, 3, 4

CAPTURE = None         # test hook: a list that receives every block's (raw conv output, activation output), NHWC bf16


def _up(v, m):
    return (v + m - 1) // m * m


def _p(t):
    return ctypes.c_void_p(t.data_ptr()) if t is not None else None


def _st():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


# ----------------------------------------------------------------------------------------- lowering
class Block(object):
    """One convolution with what follows it up to the next convolution."""

    def __init__(self, conv, reflect):
        self.conv = conv
        self.transposed = isinstance(conv, nn.ConvTranspose2d)
        k, s, p = conv.kernel_size[0], conv.stride[0], conv.padding[0]
        assert conv.kernel_size[0] == conv.kernel_size[1] and conv.stride[0] == conv.stride[1] and conv.groups == 1
        assert conv.dilation[0] == 1 and conv.padding[0] == conv.padding[1]
        self.k = k
        if self.transposed:
            assert not reflect
            self.stride, self.up, self.pad, self.reflect = 1, s, k - 1 - p, 0
            self.out_pad, self.t_stride, self.t_pad = conv.output_padding[0], s, p
            self.cin, self.cout = conv.in_channels, conv.out_channels
        else:
            assert not (reflect and p), "reflection padding in front of a zero-padded convolution"
            self.stride, self.up, self.pad, self.reflect = s, 1, (reflect or p), int(bool(reflect))
            self.cin, self.cout = conv.in_channels, conv.out_channels
        self.cin_p, self.n_p = _up(self.cin, 8), _up(self.cout, 16)
        # 32: the weight-gradient GEMM's epilogue stores 32-column chunks (a narrower row would spill into the next one)
        self.kp = _up(k * k * self.cin_p, 32)
        self.norm = None
        self.shuffle = False
        self.act, self.slope, self.prelu = ACT_NONE, 0.0, None
        self.residual = None            # index of the tensor added to this block's output
        self.final = False

    def out_hw(self, h, w):
        if self.transposed:
            f = lambda v: (v - 1) * self.t_stride - 2 * self.t_pad + self.k + self.out_pad
        else:
            f = lambda v: (v + 2 * self.pad - self.k) // self.stride + 1
        return f(h), f(w)

    # ---- weight layouts (work on index tensors too: engine.PackSet derives its gather tables from them)
    def _okkc(self, w):
        """weight -> (O, k, k, cin_p) as a DIRECT convolution sees it (transposed conv: swapped and flipped)"""
        if self.transposed:
            w = w.flip(2, 3).permute(1, 2, 3, 0)
        else:
            w = w.permute(0, 2, 3, 1)
        out = torch.zeros(self.cout, self.k, self.k, self.cin_p, dtype=w.dtype)
        out[..., :self.cin] = w
        return out

    def fwd_layout(self, w):
        m = torch.zeros(1, self.n_p, self.kp, dtype=w.dtype)
        m[0, :self.cout, :self.k * self.k * self.cin_p] = self._okkc(w).reshape(self.cout, -1)
        return m

    def dgrad_layout(self, w):
        return self.fwd_layout(w).transpose(1, 2).contiguous()            # [1][kp][n_p]

    def bias_layout(self, b):
        return torch.cat([b, torch.full((self.n_p - self.cout,), -1.0, dtype=b.dtype)])

    def wgrad_tables(self):
        """-> (col_off [1][kp], s_n, row_map [n_p]) scattering the GEMM-layout gradient into the parameter's own layout"""
        k, kk = self.k, self.k * self.k
        off = torch.full((1, self.kp), -1, dtype=torch.int32)
        c = torch.arange(self.cin, dtype=torch.int32)
        for ky in range(k):
            for kx in range(k):
                base = (ky * k + kx) * self.cin_p
                if self.transposed:      # (I, O, kh, kw): row o stride kk, channel stride O*kk, taps flipped
                    off[0, base:base + self.cin] = c * (self.cout * kk) + (k - 1 - ky) * k + (k - 1 - kx)
                else:                    # (O, I, kh, kw): row o stride I*kk, channel stride kk
                    off[0, base:base + self.cin] = c * kk + ky * k + kx
        s_n = kk if self.transposed else self.cin * kk
        row_map = torch.full((self.n_p,), -1, dtype=torch.int32)
        row_map[:self.cout] = torch.arange(self.cout, dtype=torch.int32)
        return off, s_n, row_map


def lower(net):
    """Module tree -> list of Blocks (execution order).  Tensor i is the input of block i; tensor i+1 its output."""
    blocks, state = [], {"reflect": 0}

    def walk(m):
        if isinstance(m, nn.ReflectionPad2d):
            pad = m.padding
            assert len(set(pad)) == 1
            state["reflect"] = int(pad[0])
        elif isinstance(m, (nn.Conv2d, nn.ConvTranspose2d)):
            blocks.append(Block(m, state["reflect"]))
            state["reflect"] = 0
        elif isinstance(m, (nn.BatchNorm2d, nn.InstanceNorm2d)):
            assert blocks[-1].norm is None and blocks[-1].act == ACT_NONE and not blocks[-1].shuffle
            blocks[-1].norm = m
        elif isinstance(m, nn.PixelShuffle):
            assert m.upscale_factor == 2 and blocks[-1].act == ACT_NONE and blocks[-1].norm is None
            blocks[-1].shuffle = True
        elif isinstance(m, nn.PReLU):
            assert m.weight.numel() == 1 and blocks[-1].act == ACT_NONE
            blocks[-1].act, blocks[-1].prelu = ACT_PRELU, m
        elif isinstance(m, nn.LeakyReLU):
            assert blocks[-1].act == ACT_NONE
            blocks[-1].act, blocks[-1].slope = ACT_LRELU, float(m.negative_slope)
        elif isinstance(m, nn.ReLU):
            assert blocks[-1].act == ACT_NONE
            blocks[-1].act = ACT_RELU
        elif isinstance(m, nn.Tanh):
            assert blocks[-1].act == ACT_NONE
            blocks[-1].act = ACT_TANH
        elif hasattr(m, "block") and isinstance(m.block, nn.Module) and len(list(m.children())) == 1:
            # x + block(x)   (networks/sr_resnet.py:31-37, networks/resnet_generator.py:40-53)
            source = len(blocks)                      # tensor index of the skip's input
            walk(m.block)
            last = blocks[-1]
            assert last.residual is None and last.act == ACT_NONE and not last.shuffle and len(blocks) > source
            last.residual = source
        elif isinstance(m, nn.Sequential):
            for child in m.children():
                walk(child)
        else:
            raise NotImplementedError("seqnet: no lowering for %s" % type(m).__name__)

    walk(net)
    assert blocks and state["reflect"] == 0
    assert blocks[-1].norm is None and not blocks[-1].shuffle and blocks[-1].residual is None
    blocks[-1].final = True
    return blocks


# ----------------------------------------------------------------------------------------- plans
class NetPlans(object):
    def __deepcopy__(self, memo):       # plans hold device buffers and events: a copied module builds its own
        return None

    def __init__(self, net):
        self.blocks = lower(net)
        self.params = list(net.parameters())
        self.index = {id(p): i for i, p in enumerate(self.params)}
        specs, specs32 = [], []
        for i, b in enumerate(self.blocks):
            specs.append(("w%d" % i, b.conv.weight, b.fwd_layout))
            specs.append(("d%d" % i, b.conv.weight, b.dgrad_layout))
            if b.conv.bias is not None:
                specs32.append(("b%d" % i, b.conv.bias, b.bias_layout))
            b.fwd_plan = dense.Plan("linear", b.kp, b.n_p)
            b.dg_plan = dense.Plan("linear", b.n_p, _up(b.kp, 16))
            off, s_n, row_map = b.wgrad_tables()
            b.wg_plan = dense.WGradPlan(dense.Plan("linear", b.kp, b.n_p), tuple(b.conv.weight.shape), row_perm=row_map,
                                        col_off=off, s_n=s_n)
        self.packs = engine.PackSet(net, specs, specs32)
        engine._ALL_PACKS.append(self.packs)
        norms = [m for m in net.modules() if isinstance(m, (nn.BatchNorm2d, nn.InstanceNorm2d))]
        self.norm_index = {id(m): i for i, m in enumerate(norms)}


def _plans(net):
    p = getattr(net, "_ipr_seq_plans", None)
    if p is not None and p.packs.arena is not flat.arena_of(next(net.parameters())):
        p = None                                     # parameters were re-created (e.g. .to(device)): rebuild
    if p is None:
        p = NetPlans(net)
        object.__setattr__(net, "_ipr_seq_plans", p)
    return p


# ----------------------------------------------------------------------------------------- kernel wrappers
def _im2col(x, b, oh, ow):
    n, h, w, c = x.shape
    col = torch.empty(n * oh * ow, b.kp, device=x.device, dtype=torch.bfloat16)
    check(lib().ipr_im2col_nhwc_bf16(_p(x), _p(col), n, h, w, c, oh, ow, b.k, b.stride, b.pad, b.up, b.reflect, b.kp, _st()),
          "ipr_im2col_nhwc_bf16")
    return col


def _col2im(dcol, b, shape, oh, ow, addend):
    n, h, w, c = shape
    dx = torch.empty(shape, device=dcol.device, dtype=torch.bfloat16)
    check(lib().ipr_col2im_nhwc_bf16(_p(dcol), _p(dx), _p(addend), n, h, w, c, oh, ow, b.k, b.stride, b.pad, b.up,
                                     b.reflect, b.kp, _st()), "ipr_col2im_nhwc_bf16")
    return dx


def _norm_ws(groups, c, dev):
    nbytes = lib().ipr_norm_workspace_bytes(groups, c)
    return torch.empty(nbytes // 4, device=dev, dtype=torch.float32), nbytes


def _shuffle(x, inverse):
    if not inverse:
        n, h, w, c4 = x.shape
        y = torch.empty(n, 2 * h, 2 * w, c4 // 4, device=x.device, dtype=x.dtype)
        check(lib().ipr_pixel_shuffle2_nhwc_bf16(_p(x), _p(y), n, h, w, c4 // 4, 0, _st()), "ipr_pixel_shuffle2_nhwc_bf16")
    else:
        n, h2, w2, c = x.shape
        y = torch.empty(n, h2 // 2, w2 // 2, c * 4, device=x.device, dtype=x.dtype)
        check(lib().ipr_pixel_shuffle2_nhwc_bf16(_p(x), _p(y), n, h2 // 2, w2 // 2, c, 1, _st()),
              "ipr_pixel_shuffle2_nhwc_bf16")
    return y


def _add(a, b):
    out = torch.empty_like(a)
    check(lib().ipr_add_bf16(_p(a), _p(b), _p(out), a.numel(), _st()), "ipr_add_bf16")
    return out


# ----------------------------------------------------------------------------------------- the autograd node
class _SeqFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, net, x, *params):
        P = _plans(net)
        dev = x.device
        N, C, H, W = x.shape
        b0 = P.blocks[0]
        assert C == b0.cin, (C, b0.cin)
        t = torch.empty(N, H, W, b0.cin_p, device=dev, dtype=torch.bfloat16)
        check(lib().ipr_nchw_to_nhwc_bf16(_p(x.detach().contiguous()), None, _p(t), N, C, H, W, b0.cin_p, _st()),
              "ipr_nchw_to_nhwc_bf16")
        tensors, tape, out = [t], [], None
        for i, b in enumerate(P.blocks):
            xin = tensors[-1]
            n, h, w, c = xin.shape
            assert c == b.cin_p, (i, c, b.cin_p)
            oh, ow = b.out_hw(h, w)
            col = _im2col(xin, b, oh, ow)
            M = n * oh * ow
            a = col.view(M, 1, 1, b.kp)
            rec = {"col": col, "in_shape": (n, h, w, c), "ohw": (oh, ow)}
            if b.final:
                t32, _ = b.fwd_plan.run(a, P.packs.get("w%d" % i), epi=dense.EPI_LINEAR_F32, n_valid=b.n_p)
                out = torch.empty(n, b.cout, oh, ow, device=dev, dtype=torch.float32)
                bias = P.packs.get32("b%d" % i) if b.conv.bias is not None else None
                check(lib().ipr_finish_nchw_f32(_p(t32), _p(bias), _p(out), n, b.cout, oh, ow, b.n_p,
                                                int(b.act == ACT_TANH), _st()), "ipr_finish_nchw_f32")
                assert b.act in (ACT_NONE, ACT_TANH)
                tape.append(rec)
                break
            bias = P.packs.get32("b%d" % i) if b.conv.bias is not None else None
            y0, _ = b.fwd_plan.run(a, P.packs.get("w%d" % i), epi=dense.EPI_BIAS_LRELU, slope=1.0, bias=bias,
                                   n_valid=b.n_p)
            y0 = y0.view(n, oh, ow, b.n_p)
            groups, rows, has_norm = 1, M, 0
            scale = shift = mean = rstd = None
            nm = b.norm
            rm = rv = nbt = gamma = beta = None
            eps, mom = 1e-5, 0.1
            if nm is not None:
                inst = isinstance(nm, nn.InstanceNorm2d)
                groups, rows = (n, oh * ow) if inst else (1, M)
                gamma = nm.weight.detach() if nm.weight is not None else None
                beta = nm.bias.detach() if nm.bias is not None else None
                eps = nm.eps
                mom = nm.momentum if nm.momentum is not None else 0.1
                batch_stats = inst or nm.training or (nm.running_mean is None and nm.running_var is None)
                if batch_stats:
                    has_norm = 1
                    scale, shift, mean, rstd = (torch.empty(groups, b.n_p, device=dev) for _ in range(4))
                    if not inst and nm.training and nm.track_running_stats and nm.running_mean is not None:
                        rm, rv, nbt = nm.running_mean, nm.running_var, nm.num_batches_tracked
                else:                        # eval-mode BatchNorm: running statistics (not a training path)
                    has_norm = 2
                    r = torch.rsqrt(nm.running_var + nm.eps)
                    scale = ((gamma if gamma is not None else 1.0) * r).view(1, -1).contiguous()
                    shift = ((beta if beta is not None else 0.0) - nm.running_mean * scale.view(-1)).view(1, -1).contiguous()
                    mean, rstd = nm.running_mean.view(1, -1).contiguous(), r.view(1, -1).contiguous()
            res = tensors[b.residual] if b.residual is not None else None
            z = torch.empty_like(y0)
            ws, nbytes = _norm_ws(groups, b.n_p, dev)
            slope_ptr = b.prelu.weight.detach() if b.prelu is not None else None
            check(lib().ipr_norm_fwd_bf16(_p(y0), _p(z), _p(res), groups, rows, b.n_p, has_norm, float(eps), float(mom),
                                          _p(gamma), _p(beta), _p(rm), _p(rv), _p(nbt), _p(scale), _p(shift), _p(mean),
                                          _p(rstd), b.act, float(b.slope), _p(slope_ptr), _p(ws), nbytes, _st()),
                  "ipr_norm_fwd_bf16")
            if CAPTURE is not None:
                CAPTURE.append((y0, z))               # z before PixelShuffle: its sign pattern is the activation mask
            if b.shuffle:
                z = _shuffle(z, False)
            rec.update(y0=y0, groups=groups, rows=rows, has_norm=has_norm, scale=scale, shift=shift, mean=mean, rstd=rstd)
            tape.append(rec)
            tensors.append(z)
        ctx.net, ctx.tape, ctx.out = net, tape, out
        ctx.x_needs_grad = x.requires_grad
        ctx.skip_params = bool(getattr(net, "_ipr_skip_param_grads", False))
        ctx.in_shape = (N, C, H, W)
        return out

    @staticmethod
    def backward(ctx, dout):
        net, tape = ctx.net, ctx.tape
        P = _plans(net)
        dev = dout.device
        grads = [None] * len(P.params)
        hook = getattr(net, "_ipr_sign_hook", None)
        # a pass whose parameter gradients are never used (a discriminator inside a generator step): data gradient only
        skip_params = ctx.skip_params

        def give(param, value_fn):
            """Weight-type gradient: accumulate into the bound ``.grad`` view when there is one, else return a tensor."""
            dst, acc, ret = engine._grad_dst(param)
            value_fn(dst, acc)
            if ret is not None:
                grads[P.index[id(param)]] = ret

        # weight / bias gradients (GEMM, split-K reduction, column sums) are off the data-gradient chain: they run on
        # the engine's keyed side streams (same block -> same stream, so accumulations of one parameter stay ordered
        # across passes) and rejoin before the node returns
        fork = engine._Fork(dev)
        pending = {}                                  # tensor index -> gradient arriving over a skip connection
        dz = None
        for i in range(len(P.blocks) - 1, -1, -1):
            b, rec = P.blocks[i], tape[i]
            n, h, w, c = rec["in_shape"]
            oh, ow = rec["ohw"]
            M = n * oh * ow
            if b.final:
                dy0 = torch.empty(n, oh, ow, b.n_p, device=dev, dtype=torch.bfloat16)
                check(lib().ipr_nchw_to_nhwc_bf16(_p(dout.contiguous().float()), _p(ctx.out) if b.act == ACT_TANH else None,
                                                  _p(dy0), n, b.cout, oh, ow, b.n_p, _st()), "ipr_nchw_to_nhwc_bf16")
            else:
                if b.residual is not None:            # the skip source receives the same gradient
                    r = b.residual
                    pending[r] = dz if r not in pending else _add(pending[r], dz)
                if b.shuffle:
                    dz = _shuffle(dz, True)
                nm = b.norm
                y0 = rec["y0"]
                dy0 = torch.empty_like(y0)
                ws, nbytes = _norm_ws(rec["groups"], b.n_p, dev)
                gamma = nm.weight.detach() if (nm is not None and nm.weight is not None) else None
                if rec["has_norm"] == 2:
                    raise RuntimeError("seqnet: backward through eval-mode BatchNorm is not on the training path")
                # parameter gradients of this launch land in fresh buffers and are handed over below
                if skip_params:
                    gamma_g = None
                else:
                    gamma_g = gamma
                # gamma / beta gradients go straight into the parameters' bound ``.grad`` views (the kernel accumulates)
                # when both have one; otherwise into fresh buffers that are handed to autograd below
                dg = db = None
                direct = False
                if gamma_g is not None:
                    dst_g, acc_g, _ = engine._grad_dst(nm.weight)
                    dst_b, acc_b, _ = engine._grad_dst(nm.bias)
                    direct = acc_g and acc_b
                    dg, db = (dst_g, dst_b) if direct else (torch.empty_like(gamma), torch.empty_like(gamma))
                sg, g0, sc = (None, 0.0, 0.0)
                if hook is not None and gamma_g is not None:
                    # white-box sign loss (tools/sign_model.py:42-49): d/dgamma is added inside this launch, once per
                    # armed step and layer (models/protect.py: _SignHook)
                    sg, g0, sc = hook(P.norm_index[id(nm)])
                slope_ptr = b.prelu.weight.detach() if b.prelu is not None else None
                dsl, dsl_direct = None, False
                if slope_ptr is not None and not skip_params:
                    dst_s, acc_s, _ = engine._grad_dst(b.prelu.weight)
                    # one accumulate flag per launch: the slope gradient shares it with gamma / beta
                    dsl_direct = acc_s and (direct or gamma_g is None)
                    dsl = dst_s if dsl_direct else torch.empty_like(slope_ptr)
                accumulate = 1 if (direct or (gamma_g is None and dsl_direct)) else 0
                if accumulate and dsl is not None and not dsl_direct:
                    dsl.zero_()                       # (mixed case: the launch accumulates, this buffer is fresh)
                check(lib().ipr_norm_bwd_bf16(_p(dz), _p(y0), _p(dy0), rec["groups"], rec["rows"], b.n_p,
                                              rec["has_norm"], _p(gamma), _p(rec["scale"]), _p(rec["shift"]),
                                              _p(rec["mean"]), _p(rec["rstd"]), _p(dg), _p(db), accumulate, _p(sg),
                                              float(g0), float(sc), b.act, float(b.slope), _p(slope_ptr), _p(dsl), _p(ws),
                                              nbytes, _st()), "ipr_norm_bwd_bf16")
                if gamma_g is not None and not direct:
                    give(nm.weight, lambda dst, acc, v=dg: dst.add_(v) if acc else dst.copy_(v))
                    give(nm.bias, lambda dst, acc, v=db: dst.add_(v) if acc else dst.copy_(v))
                if dsl is not None and not dsl_direct:
                    give(b.prelu.weight, lambda dst, acc, v=dsl: dst.add_(v) if acc else dst.copy_(v))
            dy2 = dy0.view(M, 1, 1, b.n_p)
            # bias and weight gradients
            if skip_params:
                pass
            elif b.conv.bias is not None:
                def _bias(dst, acc, dy2=dy2, b=b):
                    if b.n_p == b.cout:               # no channel padding: the column sums land in the gradient itself
                        engine.colsum_bf16(dy2.view(M, b.n_p), out=dst, accumulate=acc)
                        return
                    full = engine.colsum_bf16(dy2.view(M, b.n_p))
                    if acc:
                        dst.add_(full[:b.cout])
                    else:
                        dst.copy_(full[:b.cout])
                give(b.conv.bias, lambda dst, acc, f=_bias, dy0=dy0, i=i: fork.run(lambda: f(dst, acc), dy0, dst, key=i + 1))
            if not skip_params:
                give(b.conv.weight,
                     lambda dst, acc, dy2=dy2, rec=rec, b=b, dy0=dy0, i=i: fork.run(
                         lambda: b.wg_plan.run(dy2, rec["col"].view(M, 1, 1, b.kp), dst, accumulate=acc),
                         dy0, rec["col"], dst, key=i))
            # data gradient
            need_dx = i > 0 or ctx.x_needs_grad
            if need_dx:
                dcol, _ = b.dg_plan.run(dy2, P.packs.get("d%d" % i))
                dz = _col2im(dcol.view(M, b.dg_plan.cout), b, rec["in_shape"], oh, ow, pending.pop(i, None))
            else:
                dz = None
        dx = None
        if ctx.x_needs_grad:
            N, C, H, W = ctx.in_shape
            dx = dz.float()[..., :C].permute(0, 3, 1, 2).contiguous()
        fork.join()
        ctx.tape = None
        return (None, dx, *grads)


def forward(net, x):
    """What the drop-in modules' ``forward`` calls on CUDA."""
    engine.refuse_pruned(net)
    x = x.to(device=next(net.parameters()).device, dtype=torch.float32)
    return _SeqFn.apply(net, x, *list(net.parameters()))
