"""GPU: the training step's non-GEMM kernels, each called through its C ABI or thin wrapper, against the float64
references of tests/step_kernel_refs.py: Adam (optim.cu), the bf16 re-pack (optim.cu), spectral norm (sn.cu), the loss
seeds and device RNG (step_misc.cu), column sums, BatchNorm, the final GEMV, im2col3 / col2im3 (nn_misc.cu).

Every comparison is elementwise against a bound derived from the kernel's arithmetic (see the reference functions) or
bit-exact where the contract is a copy, a single rounding or a sum order the reference reproduces.  Every kernel runs
twice and must give bit-identical results (fixed-order reductions).  Sizes that must cross a loop or branch boundary
are derived from the SM count the library itself uses."""
import ctypes

import pytest
import torch
import torch.nn.functional as F

from tests import step_kernel_refs as R

pytestmark = pytest.mark.gpu

U = R.U32


def _lib():
    from ipr_gan_b200._lib import lib
    return lib()


def _check(rc, what):
    from ipr_gan_b200._lib import check
    check(rc, what)


def _p(t, off=0):
    return ctypes.c_void_p(t.data_ptr() + 4 * off) if t is not None else None


def _st():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def within(got, want, tol, what=""):
    ex = R.max_excess(got.to(want.device), want, tol)
    assert ex <= 0, "%s: exceeds its bound by %.3g" % (what, ex)


def bits_equal(a, b):
    return a.shape == b.shape and torch.equal(a.reshape(-1).view(torch.uint8), b.reshape(-1).view(torch.uint8))


# ============================================================================================== Adam
ADAM_PAIR = 8 * 256                 # adam_flat_kernel: SMs * 8 CTAs of 256 threads; paired float4 loop above that


def adam_size(spec):
    if isinstance(spec, int):
        return spec
    s = sms() * ADAM_PAIR
    return 4 * s + 3 if spec == "pair-" else 4 * (s + 1) + 1     # n/4 == stride (no pair) / stride + 1 (one pair)


def _adam_run(p0, grads, lr, betas, eps, wd, gs, zero_grad=1):
    """The C ABI over a gradient sequence; buffers carry 8 guard floats after the n elements."""
    n = p0.numel()
    GUARD = 8
    p = torch.full((n + GUARD,), 7.0, device="cuda")
    g = torch.full((n + GUARD,), 5.0, device="cuda")
    m = torch.full((n + GUARD,), 3.0, device="cuda")
    v = torch.full((n + GUARD,), 2.0, device="cuda")
    m[:n] = 0
    v[:n] = 0
    p[:n] = p0.cuda()
    step = torch.zeros((), device="cuda")
    ticket = torch.zeros(1, device="cuda", dtype=torch.int32)
    states = []
    for gr in grads:
        g[:n] = gr.cuda()
        _check(_lib().ipr_adam_flat_f32(_p(p), _p(g), _p(m), _p(v), n, lr, betas[0], betas[1], eps, wd, gs, zero_grad,
                                        _p(step), _p(ticket), _st()), "ipr_adam_flat_f32")
        states.append((p[:n].clone(), m[:n].clone(), v[:n].clone(), g.clone()))
    torch.cuda.synchronize()
    for t, want in ((p, 7.0), (m, 3.0), (v, 2.0), (g, 5.0)):
        assert torch.all(t[n:] == want), "guard floats after the arena were written"
    assert float(step) == len(grads) and int(ticket) == 0
    return states


@pytest.mark.parametrize("spec,wd,gs", [(1, 0.0, 1.0), (3, 0.0, 1.0), (4, 0.0, 1.0), (5, 1e-2, 1.0), (1023, 0.0, 1.0),
                                        (4099, 1e-2, 0.5), (4099, 0.0, 0.5), ("pair-", 0.0, 1.0), ("pair-", 1e-2, 0.5),
                                        ("pair+", 0.0, 1.0), ("pair+", 1e-2, 0.5)])
def test_adam_c_abi_against_float64_adam(spec, wd, gs):
    n = adam_size(spec)
    p0, grads = R.adam_grads(n, 5, seed=n)
    args = (R.ADAM_LR, R.ADAM_BETAS, 1e-8, wd, gs)
    a = _adam_run(p0, grads, *args)
    b = _adam_run(p0, grads, *args)
    ref = R.adam_ref(p0.cuda(), [x.cuda() for x in grads], *args)         # float64 on the device
    for k, ((p, m, v, g), (p2, m2, v2, _), want) in enumerate(zip(a, b, ref)):
        assert bits_equal(p, p2) and bits_equal(m, m2) and bits_equal(v, v2), k
        # zero_grad=1 clears exactly the n gradient floats (the guards are checked in _adam_run)
        assert torch.all(g[:n] == 0)
        within(m, want["m"].cuda(), want["tm"].cuda(), "exp_avg step %d" % (k + 1))
        within(v, want["v"].cuda(), want["tv"].cuda(), "exp_avg_sq step %d" % (k + 1))
        within(p, want["p"].cuda(), want["tp"].cuda(), "param step %d" % (k + 1))


def test_adam_graph_replays_equal_eager_launches():
    """The device step counter and the arrival ticket: N replays of one captured launch == N eager launches, bit for
    bit, with a grid of the full SMs * 8 CTAs; step ends at N and the ticket back at 0."""
    n = adam_size("pair+") + 4 * 1000
    p0, (g0,) = R.adam_grads(n, 1, seed=3)
    N = 6

    def bufs():
        return (p0.cuda(), g0.cuda(), torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda"),
                torch.zeros((), device="cuda"), torch.zeros(1, device="cuda", dtype=torch.int32))

    def launch(b):
        p, g, m, v, step, ticket = b
        _check(_lib().ipr_adam_flat_f32(_p(p), _p(g), _p(m), _p(v), n, 2e-4, 0.5, 0.999, 1e-8, 0.0, 1.0, 0,
                                        _p(step), _p(ticket), _st()), "ipr_adam_flat_f32")

    eager = bufs()
    for _ in range(N):
        launch(eager)
    cap = bufs()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            launch(cap)
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(N):
        graph.replay()
    torch.cuda.synchronize()
    for a, b in zip(eager, cap):
        assert bits_equal(a, b)
    assert float(cap[4]) == N and int(cap[5]) == 0


def _net(kind, size):
    import networks
    torch.manual_seed(11 if kind == "G" else 12)
    name = {"G": "ConvGenerator", "D": "SNDiscriminator"}[kind] + str(size)
    return getattr(networks, name)().cuda()


@pytest.mark.parametrize("kind,size,wd", [("G", 32, 0.0), ("D", 32, 0.0), ("G", 64, 0.0), ("D", 64, 1e-3)])
def test_flat_adam_real_arenas(kind, size, wd):
    """FlatAdam over the real parameter arenas of both configurations (every tensor 16-byte aligned inside the arena,
    zero padding between them), five steps with the reference's lr / betas."""
    from ipr_gan_b200.optim import FlatAdam
    net = _net(kind, size)
    opt = FlatAdam(net.parameters(), lr=R.ADAM_LR, betas=R.ADAM_BETAS, weight_decay=wd)
    arena = opt.arena
    p0 = arena.param.detach().clone()
    _, grads = R.adam_grads(arena.numel, 5, seed=arena.numel)
    grads = [x.cuda() for x in grads]
    ref = R.adam_ref(p0, grads, R.ADAM_LR, R.ADAM_BETAS, 1e-8, wd)              # float64 on the device
    for k, (gr, want) in enumerate(zip(grads, ref)):
        arena.grad.copy_(gr)
        arena.clean = False
        opt.step()
        within(opt._m, want["m"].cuda(), want["tm"].cuda(), "exp_avg step %d" % (k + 1))
        within(opt._v, want["v"].cuda(), want["tv"].cuda(), "exp_avg_sq step %d" % (k + 1))
        within(arena.param, want["p"].cuda(), want["tp"].cuda(), "param step %d" % (k + 1))
        assert torch.all(arena.grad == 0)
    assert float(opt._step) == 5


def test_flat_adam_resumes_from_stock_adam_state():
    """A stock torch.optim.Adam state (three steps taken on the CPU) loaded into FlatAdam: the next step continues the
    stock optimiser's trajectory (moments and step count), not a fresh one."""
    from ipr_gan_b200.optim import FlatAdam
    torch.manual_seed(5)
    cpu = torch.nn.Sequential(torch.nn.Linear(37, 13), torch.nn.Linear(13, 5))
    stock = torch.optim.Adam(cpu.parameters(), lr=R.ADAM_LR, betas=R.ADAM_BETAS, foreach=False)
    g = torch.Generator().manual_seed(6)
    for _ in range(3):
        for q in cpu.parameters():
            q.grad = torch.randn(q.shape, generator=g) * 1e-2
        stock.step()
    gpu = torch.nn.Sequential(torch.nn.Linear(37, 13), torch.nn.Linear(13, 5)).cuda()
    gpu.load_state_dict(cpu.state_dict())
    opt = FlatAdam(gpu.parameters(), lr=R.ADAM_LR, betas=R.ADAM_BETAS)
    opt.load_state_dict(stock.state_dict())
    last = [torch.randn(q.shape, generator=g) * 1e-2 for q in cpu.parameters()]
    for q, gl in zip(gpu.parameters(), last):
        q.grad.copy_(gl.cuda())
    opt.arena.clean = False
    opt.step()
    for q, qc, gl in zip(gpu.parameters(), cpu.parameters(), last):
        st = stock.state[qc]
        want = R.adam_ref(qc.detach().reshape(-1), [gl.reshape(-1)], R.ADAM_LR, R.ADAM_BETAS, 1e-8, 0.0,
                          m0=st["exp_avg"].reshape(-1), v0=st["exp_avg_sq"].reshape(-1), step0=3)[0]
        within(q.detach().reshape(-1), want["p"].cuda(), want["tp"].cuda() + 3 * U * want["p"].abs().cuda(), "param")
    assert float(opt._step) == 4


# ============================================================================================== gather_pack
GATHER_PAIR = 8 * 256               # gather_pack_kernel: SMs * 8 CTAs; paired 8-element groups above that


def _pack_specs(net, kind):
    """The (key, parameter, layout) lists GenPlans / DisPlans build their PackSet from (engine.py)."""
    from ipr_gan_b200 import engine
    P = engine._plans(net, engine.GenPlans if kind == "G" else engine.DisPlans)
    if kind == "G":
        cv = net.convs
        specs = [("fc", net.fc[0].weight, lambda w: P.fc.pack_layout(w, P.perm.to(w.device)))]
        for i in range(3):
            specs.append(("ct%d" % i, cv[i][0].weight, P.ct[i].pack_layout))
            specs.append(("ct%d_dg" % i, cv[i][0].weight, P.ct_dg[i].pack_layout))
        specs.append(("ct3", cv[3].weight, engine._tap27_rows_layout))
        specs.append(("ct3_dg", cv[3].weight, engine._patch27_layout))
        specs32 = [("fcb", net.fc[0].bias, lambda b: b[P.perm.to(b.device)])]
    else:
        layers = engine._sn_layers(net)
        specs = [("c0", layers[0].weight_orig, engine._patch27_layout),
                 ("c0_dg", layers[0].weight_orig, engine._tap27_rows_layout)]
        for i in range(6):
            specs.append(("c%d" % (i + 1), layers[i + 1].weight_orig, P.conv[i].pack_layout))
            specs.append(("c%d_dg" % (i + 1), layers[i + 1].weight_orig, P.conv_dg[i].pack_layout))
        specs32 = [("w8", layers[7].weight_orig, lambda w: w.reshape(-1)[P.perm.to(w.device)])]
    return P, specs, specs32


@pytest.mark.parametrize("kind,size", [("G", 32), ("D", 32), ("G", 64), ("D", 64)])
def test_packset_bit_exact_against_layouts(kind, size):
    net = _net(kind, size)
    with torch.no_grad():
        for q in net.parameters():              # weights that straddle bf16 rounding boundaries everywhere
            q.copy_(torch.randn_like(q))
    P, specs, specs32 = _pack_specs(net, kind)
    packs = P.packs
    assert set(packs.slices) == {k for k, _, _ in specs}
    runs = []
    for _ in range(2):
        packs.clear()
        packs.refresh()
        torch.cuda.synchronize()
        runs.append((packs.buf.clone(), packs.buf32.clone()))
    assert bits_equal(runs[0][0], runs[1][0]) and bits_equal(runs[0][1], runs[1][1])
    for key, param, fn in specs:
        off, n, shape = packs.slices[key]
        want = fn(param.detach()).to(torch.bfloat16).reshape(-1)
        assert bits_equal(packs.buf[off:off + n], want), key
        pad_end = off + n + (-n) % 8
        assert torch.all(packs.buf[off + n:pad_end].float() == 0), key
    for key, param, fn in specs32:
        off, n = packs.slices32[key]
        assert bits_equal(packs.buf32[off:off + n], fn(param.detach()).reshape(-1).float()), key


@pytest.mark.parametrize("spec", ["pair-", "pair+"])
def test_gather_pack_synthetic_table(spec):
    """An index table with -1 (zero) entries across the paired-loop threshold, plus an odd-sized fp32 side table."""
    groups = sms() * GATHER_PAIR + (0 if spec == "pair-" else 3)
    n, n32 = 8 * groups, 1001
    g = torch.Generator().manual_seed(groups)
    src = torch.randn(300007, generator=g)
    idx = torch.randint(-1, src.numel(), (n,), generator=g, dtype=torch.int32)
    idx[torch.rand(n, generator=g) < 0.1] = -1
    idx32 = torch.randint(-1, src.numel(), (n32,), generator=g, dtype=torch.int32)
    want = torch.where(idx >= 0, src[idx.clamp_min(0).long()], torch.zeros(())).to(torch.bfloat16)
    want32 = torch.where(idx32 >= 0, src[idx32.clamp_min(0).long()], torch.zeros(()))
    s, i, i32 = src.cuda(), idx.cuda(), idx32.cuda()
    outs = []
    for _ in range(2):
        dst = torch.full((n,), 3.0, device="cuda", dtype=torch.bfloat16)
        dst32 = torch.full((n32 + 4,), 3.0, device="cuda")
        _check(_lib().ipr_gather_pack_bf16(_p(s), _p(i), _p(dst), n, _p(i32), _p(dst32), n32, _st()),
               "ipr_gather_pack_bf16")
        outs.append((dst, dst32))
    torch.cuda.synchronize()
    assert bits_equal(outs[0][0], outs[1][0]) and bits_equal(outs[0][1], outs[1][1])
    assert bits_equal(outs[0][0].cpu(), want)
    assert bits_equal(outs[0][1][:n32].cpu(), want32) and torch.all(outs[0][1][n32:] == 3.0)


# ============================================================================================== spectral norm
SN_SYNTH = [(1, 27), (33, 27), (33, 257), (1, 257), (7, 5), (64, 27), (5, 4097), (33, 256), (65, 1024), (1100, 8),
            (3, 2049), (2, 6), (128, 576), (31, 33), (9, 4096), (1, 8192)]
SN_OFFSET_LAYER = 14                # its w starts one float past a 16-byte boundary: the scalar branches


class _SnSet(object):
    """Layers for the batched SN kernels: weights, u, v, sigma, snapshots and per-layer scratch slices."""

    def __init__(self, dims, seed, weights=None, offset_layer=None):
        from ipr_gan_b200._lib import SnLayer
        ws, us, vs = R.sn_inputs(dims, seed)
        if weights is not None:
            ws = [w.detach().reshape(r, c) for w, (r, c) in zip(weights, dims)]
        self.dims = dims
        self.w, self.wbuf = [], []
        for i, (r, c) in enumerate(dims):
            off = 1 if i == offset_layer else 0
            buf = torch.empty(r * c + 4, device="cuda")
            buf[off:off + r * c] = ws[i].reshape(-1).cuda()
            self.wbuf.append((buf, off))
            self.w.append(buf[off:off + r * c].view(r, c))
        self.u = [u.cuda() for u in us]
        self.v = [v.cuda() for v in vs]
        self.sigma = torch.zeros(len(dims), device="cuda")
        self.usnap = [torch.full_like(u, 9.0) for u in self.u]
        self.vsnap = [torch.full_like(v, 9.0) for v in self.v]
        offs, tot = [], 0
        for r, c in dims:
            offs.append(tot)
            tot += int(_lib().ipr_sn_scratch_floats(r, c))
        self.scratch = torch.empty(tot, device="cuda")
        self.offs = offs
        self.SnLayer = SnLayer

    def table(self, grads=None, grad_outs=None):
        arr = (self.SnLayer * len(self.dims))()
        for i, (r, c) in enumerate(self.dims):
            buf, off = self.wbuf[i]
            arr[i].w = buf.data_ptr() + 4 * off
            arr[i].u, arr[i].v = self.u[i].data_ptr(), self.v[i].data_ptr()
            arr[i].sigma = self.sigma.data_ptr() + 4 * i
            arr[i].grad = grads[i].data_ptr() if grads is not None else None
            arr[i].grad_out = grad_outs[i].data_ptr() if grad_outs is not None else None
            arr[i].rows, arr[i].cols = r, c
            arr[i].scratch_off = self.offs[i]
            arr[i].u_snap, arr[i].v_snap = self.usnap[i].data_ptr(), self.vsnap[i].data_ptr()
        return arr

    def power(self, update):
        _check(_lib().ipr_sn_power_iter_f32(self.table(), len(self.dims), int(update), R.SN_EPS, _p(self.scratch), _st()),
               "ipr_sn_power_iter_f32")
        torch.cuda.synchronize()


def _sn_dims(source):
    if source == "synthetic":
        return SN_SYNTH, None, SN_OFFSET_LAYER
    from ipr_gan_b200 import engine
    D = _net("D", int(source[1:]))
    ws = [l.weight_orig for l in engine._sn_layers(D)]
    return [(w.shape[0], w.numel() // w.shape[0]) for w in ws], ws, None


@pytest.mark.parametrize("source", ["D32", "D64", "synthetic"])
@pytest.mark.parametrize("update", [1, 0])
def test_sn_power_iteration(source, update):
    dims, ws, offl = _sn_dims(source)
    assert len(dims) <= 16
    results = []
    for _ in range(2):
        S = _SnSet(dims, seed=len(dims), weights=ws, offset_layer=offl)
        u0, v0 = [u.clone() for u in S.u], [v.clone() for v in S.v]
        S.power(update)
        results.append(S)
    A, B = results
    assert bits_equal(A.sigma, B.sigma)
    for i in range(len(dims)):
        assert bits_equal(A.u[i], B.u[i]) and bits_equal(A.v[i], B.v[i])
        want = R.sn_power_ref(A.w[i], u0[i], v0[i], update)
        within(A.u[i], want["u"], want["tu"], "u of layer %d %s" % (i, dims[i]))
        within(A.v[i], want["v"], want["tv"], "v of layer %d %s" % (i, dims[i]))
        within(A.sigma[i:i + 1], torch.tensor([want["sigma"]], device="cuda", dtype=torch.float64),
               want["ts"], "sigma of layer %d %s" % (i, dims[i]))
        if not update:
            assert bits_equal(A.u[i], u0[i]) and bits_equal(A.v[i], v0[i])
        # the snapshots equal the vectors the launch left behind
        assert bits_equal(A.usnap[i], A.u[i]) and bits_equal(A.vsnap[i], A.v[i])


@pytest.mark.parametrize("source", ["D32", "D64", "synthetic"])
def test_sn_weight_grad(source):
    dims, ws, offl = _sn_dims(source)
    S = _SnSet(dims, seed=7, weights=ws, offset_layer=offl)
    G, base = R.sn_grad_inputs(S.w, seed=8)
    G, base = [x.cuda() for x in G], [x.cuda() for x in base]
    for i in range(len(dims)):
        S.sigma[i] = float(S.u[i].double() @ (S.w[i].double() @ S.v[i].double()))
    sig32 = S.sigma.cpu().tolist()
    # in place
    outs = []
    for _ in range(2):
        grads = [x.clone() for x in G]
        _check(_lib().ipr_sn_weight_grad_f32(S.table(grads=grads), len(dims), _p(S.scratch), _st()),
               "ipr_sn_weight_grad_f32")
        outs.append(grads)
    # added into grad_out (grad itself left as it was)
    grads = [x.clone() for x in G]
    gouts = [x.clone() for x in base]
    _check(_lib().ipr_sn_weight_grad_f32(S.table(grads=grads, grad_outs=gouts), len(dims), _p(S.scratch), _st()),
           "ipr_sn_weight_grad_f32")
    torch.cuda.synchronize()
    for i in range(len(dims)):
        assert bits_equal(outs[0][i], outs[1][i])
        want, tol = R.sn_grad_ref(S.w[i], S.u[i], S.v[i], sig32[i], G[i])
        within(outs[0][i], want, tol, "dW of layer %d %s" % (i, dims[i]))
        assert bits_equal(grads[i], G[i])
        within(gouts[i], want + base[i].double(), tol + U * (want.abs() + base[i].double().abs()),
               "grad_out of layer %d %s" % (i, dims[i]))


# ============================================================================================== loss seeds
@pytest.mark.parametrize("B", [1, 5, 512, 1025, 4097])
@pytest.mark.parametrize("loss_scale", [1.0, 0.37])
def test_hinge_d_loss(B, loss_scale):
    from ipr_gan_b200 import ops
    real, fake = R.hinge_inputs(B, seed=B)
    runs = []
    for _ in range(2):
        slots = torch.full((4,), 9.0, device="cuda")
        dr, df = ops.hinge_d_loss(real.cuda(), fake.cuda(), slots, loss_scale=loss_scale)
        runs.append((slots.clone(), dr, df))
    torch.cuda.synchronize()
    (slots, dr, df), (slots2, dr2, df2) = runs
    assert bits_equal(slots, slots2) and bits_equal(dr, dr2) and bits_equal(df, df2)
    losses, wr, wf, tol = R.hinge_ref(real, fake, loss_scale)
    assert bits_equal(dr.cpu(), wr.float()) and bits_equal(df.cpu(), wf.float())
    within(slots[:3], losses.cuda(), tol.cuda(), "hinge losses")
    assert float(slots[3]) == 9.0


@pytest.mark.parametrize("B", [1, 5, 512, 1025, 4097])
def test_gen_adv_loss(B):
    from ipr_gan_b200 import ops
    logits, _ = R.hinge_inputs(B, seed=B + 1)
    runs = []
    for _ in range(2):
        slot = torch.full((2,), 9.0, device="cuda")
        d = ops.gen_adv_loss(logits.cuda(), slot, loss_scale=0.37)
        runs.append((slot.clone(), d))
    torch.cuda.synchronize()
    assert bits_equal(runs[0][0], runs[1][0]) and bits_equal(runs[0][1], runs[1][1])
    loss, dl, tol = R.gen_adv_ref(logits, 0.37)
    assert bits_equal(runs[0][1].cpu(), dl.float())
    assert abs(float(runs[0][0][0]) - loss) <= tol and float(runs[0][0][1]) == 9.0


def pointwise_size(spec):
    return spec if isinstance(spec, int) else 2 * sms() * 1024 * 2 + 7       # several grid strides per thread


@pytest.mark.parametrize("kind", R.POINTWISE_KINDS)
@pytest.mark.parametrize("spec", [1, "grid"])
@pytest.mark.parametrize("const", [None, "const"])
def test_pointwise_loss(kind, spec, const):
    from ipr_gan_b200 import ops
    n = pointwise_size(spec)
    target = None if const is None else (1.0 if kind == "bce_logits" else 0.25)
    x, y = R.pointwise_inputs(kind, n, target, seed=n)
    yd = y.cuda() if isinstance(y, torch.Tensor) else y
    runs = [ops.pointwise_loss(kind, x.cuda(), yd, weight=0.7) for _ in range(2)]
    torch.cuda.synchronize()
    assert bits_equal(runs[0][0], runs[1][0]) and bits_equal(runs[0][1], runs[1][1])
    loss, dx, tl, tdx = R.pointwise_ref(kind, x, y, 0.7)
    assert abs(float(runs[0][0]) - loss) <= tl, (float(runs[0][0]), loss, tl)
    if kind == "l1":
        assert bits_equal(runs[0][1].cpu(), dx.float())
    else:
        within(runs[0][1], dx.cuda(), tdx.cuda(), kind + " gradient")


# ============================================================================================== randn
SEED = 0x123456789ABCDEF0


@pytest.mark.parametrize("n", [1, 3, 5, 128 * 512])
@pytest.mark.parametrize("offset", [0, 1])
def test_randn_against_philox_box_muller(n, offset):
    from ipr_gan_b200 import ops
    fills = []
    for _ in range(2):                                  # a second generator of the same seed draws the same numbers
        gen = ops.DeviceNormal("cuda", SEED)
        buf = torch.full((n + 8,), 9.0, device="cuda")
        base = 0
        for k in range(3):                              # consecutive fills continue the stream
            out = buf[offset:offset + n]
            gen.fill_(out)
            torch.cuda.synchronize()
            want, tol, nxt = R.randn_ref(n, SEED, base)
            within(out, want.cuda(), tol.cuda(), "draws of fill %d" % k)
            assert int(gen.counter) == nxt and int(gen.ticket) == 0
            base = nxt
            assert torch.all(buf[:offset] == 9.0) and torch.all(buf[offset + n:] == 9.0)
            fills.append(out.clone())
    assert all(bits_equal(a, b) for a, b in zip(fills[:3], fills[3:]))
    if n >= 64:                                         # another seed: another stream
        other = ops.DeviceNormal("cuda", SEED + 1).fill_(torch.empty(n, device="cuda"))
        assert float((other - fills[0]).abs().mean()) > 0.5


def test_randn_graph_replays_equal_eager_fills():
    from ipr_gan_b200 import ops
    n, N = 128 * 512 + 3, 4
    eager = ops.DeviceNormal("cuda", SEED)
    outs = []
    for _ in range(N):
        outs.append(eager.fill_(torch.empty(n, device="cuda")).clone())
    cap = ops.DeviceNormal("cuda", SEED)
    static = torch.empty(n, device="cuda")
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            cap.fill_(static)
    torch.cuda.current_stream().wait_stream(s)
    for k in range(N):
        graph.replay()
        torch.cuda.synchronize()
        assert bits_equal(static, outs[k]), k
    assert int(cap.counter) == int(eager.counter) == N * ((n + 3) // 4) and int(cap.ticket) == 0


# ============================================================================================== column sums
def _colsum_partials_call(x, rows, ncols, stride, out, acc, scale):
    nbytes = _lib().ipr_colsum_workspace_bytes(ncols)
    ws = torch.empty(nbytes // 4, device="cuda")
    _check(_lib().ipr_colsum_partials_f32(_p(x), rows, ncols, stride, _p(out), acc, scale, _p(ws), nbytes, _st()),
           "ipr_colsum_partials_f32")


@pytest.mark.parametrize("rows", [1, 7, 256, 257, 1000, 5000])
@pytest.mark.parametrize("ncols,stride", [(64, 64), (40, 40), (1000, 1000), (40, 72), (200, 256)])
def test_colsum_partials(rows, ncols, stride):
    """One launch up to 256 rows, two above; row_stride > ncols (statistics of a wider tile); ncols % 32 != 0."""
    g = torch.Generator().manual_seed(rows * 7 + ncols)
    x = torch.randn(rows, stride, generator=g).cuda()
    old = (torch.randn(ncols, generator=g) * 50).cuda()
    for acc in (0, 1, 2):
        outs = []
        for _ in range(2):
            out = old.clone()
            _colsum_partials_call(x, rows, ncols, stride, out, acc, 0.75)
            outs.append(out)
        torch.cuda.synchronize()
        assert bits_equal(outs[0], outs[1])
        want, tol = R.colsum_ref(x, ncols, old, acc, 0.75, depth=rows / 8 + 9)
        within(outs[0], want, tol, "accumulate=%d" % acc)


def colsum_bf16_rows(spec, C):
    return spec if isinstance(spec, int) else max(4099, (1 << 20) // C)


@pytest.mark.parametrize("C", [8, 24, 64, 512, 4096])
@pytest.mark.parametrize("spec", [1, 5, 63, 64, "large"])
@pytest.mark.parametrize("indexed", [False, True])
def test_colsum_bf16(C, spec, indexed):
    """c_vec a power of two or not (C = 24), and C > 2048 (column groups capped at 256 vectors); fewer rows than the
    64 row slabs, exactly 64, and many."""
    from ipr_gan_b200 import engine
    rows = colsum_bf16_rows(spec, C)
    g = torch.Generator().manual_seed(rows + C)
    x = torch.randn(rows, C, generator=g).to(torch.bfloat16).cuda()
    idx = torch.randperm(C + 5, generator=g)[:C].to(torch.int32).cuda() if indexed else None
    old = (torch.randn(C + 5, generator=g) * 50).cuda()
    for acc in (0, 1, 2):
        outs = []
        for _ in range(2):
            out = old.clone()
            engine.colsum_bf16(x, out=out, accumulate=acc, scale=0.75, out_index=idx)
            outs.append(out)
        torch.cuda.synchronize()
        assert bits_equal(outs[0], outs[1])
        want, tol = R.colsum_ref(x, C, old, acc, 0.75, out_index=idx if indexed else None,
                                 depth=-(-rows // min(rows, 64)) + 260)
        within(outs[0], want, tol, "accumulate=%d" % acc)


# ============================================================================================== BatchNorm
def _bn_shapes():
    shapes = []
    for mg in (4, 8):                        # ConvGenerator32 / 64: BN after convT 512->256, 256->128, 128->64
        for B in (1, 5, 64, 512):
            for C, hw in ((256, 2 * mg), (128, 4 * mg), (64, 8 * mg)):
                shapes.append((C, B * hw * hw))
    return sorted(set(shapes)) + [(8, 1000), (24, 333), (2048, 96)]


@pytest.mark.parametrize("C,rows", _bn_shapes())
def test_batchnorm_finalize_apply_backward(C, rows):
    from ipr_gan_b200 import engine
    dev = "cuda"
    x, dy, prm = R.bn_inputs(C, rows, seed=C * 7919 + rows)
    x, dy = x.to(dev), dy.to(dev)
    prm = {k: t.to(dev) for k, t in prm.items()}
    bn = torch.nn.BatchNorm2d(C).to(dev)
    with torch.no_grad():
        for name in ("weight", "bias", "running_mean", "running_var"):
            getattr(bn, name).copy_(prm["gamma" if name == "weight" else "beta" if name == "bias" else name])
    rm0, rv0 = bn.running_mean.clone(), bn.running_var.clone()
    stats = R.bn_stats_partials(x, 4)
    fin = []
    for _ in range(2):
        bn.running_mean.copy_(rm0)
        bn.running_var.copy_(rv0)
        fin.append([t.clone() for t in engine.bn_finalize(stats, rows, bn, True)] +
                   [bn.running_mean.clone(), bn.running_var.clone()])
    torch.cuda.synchronize()
    assert all(bits_equal(a, b) for a, b in zip(*fin))
    assert int(bn.num_batches_tracked) == 2
    scale, shift, mean, rstd, rm, rv = fin[0]
    want, tol = R.bn_finalize_ref(stats, rows, bn.weight, bn.bias, bn.eps, bn.momentum, rm0, rv0)
    for name, got in (("mean", mean), ("rstd", rstd), ("scale", scale), ("shift", shift), ("running_mean", rm),
                      ("running_var", rv)):
        within(got, want[name], tol[name], name)
    # the statistics against F.batch_norm's own on the bf16 tensor: the partials were rounded to fp32 once
    X = x.double()
    ex2 = (X * X).mean(0)
    var = X.var(0, unbiased=False)
    within(mean, X.mean(0), 2 * U * X.abs().mean(0) + 2 * U * X.mean(0).abs(), "mean vs batch_norm")
    within(rstd, 1 / torch.sqrt(var + bn.eps), (8 * U * (ex2 + bn.eps) / (var + bn.eps)) / torch.sqrt(var + bn.eps),
           "rstd vs batch_norm")
    # forward: relu(x * scale + shift)
    ys = [engine.bn_apply_relu(x, scale, shift) for _ in range(2)]
    torch.cuda.synchronize()
    assert bits_equal(ys[0], ys[1])
    yw, yt = R.bn_apply_ref(x, scale, shift)
    within(ys[0], yw, yt, "bn_apply_relu")
    # backward, with the sign-loss term, for accumulate = 0, 1, 2
    sign, dg_old, db_old = prm["sign"], prm["dgamma_old"], prm["dbeta_old"]
    gamma = bn.weight.detach()
    for acc in (0, 1, 2):
        use_sign = acc != 1
        outs = []
        for _ in range(2):
            dgam, dbet = dg_old.clone(), db_old.clone()
            dx = engine.bn_relu_bwd(dy, x, scale, shift, gamma, mean, rstd, dgam, dbet, acc,
                                    sign if use_sign else None, 0.1, 0.5)
            outs.append((dx, dgam, dbet))
        torch.cuda.synchronize()
        assert all(bits_equal(a, b) for a, b in zip(*outs))
        dx, dgam, dbet = outs[0]
        wdx, wdg, wdb, tdx, tdg, tdb = R.bn_bwd_ref(dy, x, scale, shift, gamma, bn.bias, bn.eps, rows,
                                                    sign if use_sign else None, 0.1, 0.5, dg_old, db_old, acc)
        within(dx, wdx, tdx, "dx (accumulate=%d)" % acc)
        within(dgam, wdg, tdg, "dgamma (accumulate=%d)" % acc)
        within(dbet, wdb, tdb, "dbeta (accumulate=%d)" % acc)


# ============================================================================================== final GEMV
@pytest.mark.parametrize("K", [8192, 32768])
@pytest.mark.parametrize("B", [1, 5, 512])
@pytest.mark.parametrize("affine", [True, False])
def test_dfc_forward_backward(K, B, affine):
    dev = "cuda"
    a, w, dlogit, perm, dw_old = (t.to(dev) for t in R.dfc_inputs(B, K, seed=K + B))
    sigma = torch.tensor([1.7], device=dev) if affine else None
    bias = torch.tensor([0.3], device=dev) if affine else None
    fw = []
    for _ in range(2):
        logits = torch.empty(B, device=dev)
        _check(_lib().ipr_dfc_fwd_bf16(_p(a), _p(w), _p(sigma), _p(bias), _p(logits), B, K, _st()), "ipr_dfc_fwd_bf16")
        fw.append(logits)
    torch.cuda.synchronize()
    assert bits_equal(fw[0], fw[1])
    want, tol = R.dfc_fwd_ref(a, w, sigma, bias)
    within(fw[0], want, tol, "logits")
    db_old = torch.tensor([0.25], device=dev)
    for acc, index in ((0, None), (1, perm), (0, perm)):
        outs = []
        for _ in range(2):
            da = torch.empty_like(a)
            dw, db = dw_old.clone(), db_old.clone()
            _check(_lib().ipr_dfc_bwd_bf16(_p(a), _p(w), _p(sigma), _p(dlogit), _p(da), _p(dw), acc, 0.1, B, K,
                                           _p(index), _p(db), _st()), "ipr_dfc_bwd_bf16")
            outs.append((da, dw, db))
        torch.cuda.synchronize()
        assert all(bits_equal(x, y) for x, y in zip(*outs))
        da, dw, db = outs[0]
        wda, tda = R.dfc_bwd_data_ref(a, w, sigma, dlogit, 0.1)
        within(da, wda, tda, "da")
        wdw, tdw, wdb, tdb = R.dfc_bwd_weight_ref(a, dlogit, dw_old, acc, index, db_old)
        within(dw, wdw, tdw, "dw (accumulate=%d, index=%s)" % (acc, index is not None))
        assert abs(float(db) - wdb) <= tdb


# ============================================================================================== im2col3 / col2im3
@pytest.mark.parametrize("B,H,W", [(1, 5, 7), (2, 9, 33), (3, 17, 40), (1, 32, 32), (2, 64, 48)])
def test_im2col3(B, H, W):
    from ipr_gan_b200 import engine
    g = torch.Generator(device="cuda").manual_seed(B * H * W)
    x = torch.randn(B, 3, H, W, device="cuda", generator=g)
    t = torch.tanh(torch.randn(B, 3, H, W, device="cuda", generator=g))
    plain = [engine.im2col3(x) for _ in range(2)]
    fused = [engine.im2col3(x, t) for _ in range(2)]
    torch.cuda.synchronize()
    assert bits_equal(plain[0], plain[1]) and bits_equal(fused[0], fused[1])
    # a copy and one bf16 rounding: bit-exact
    assert bits_equal(plain[0], R.im2col3_ref(x).to(torch.bfloat16))
    # x (1 - t^2): up to three fp32 roundings, then bf16
    want = R.im2col3_ref(x, t)
    within(fused[0], want, R.bf16_ulp(want) + 4 * U * R.im2col3_ref(x).abs(), "im2col3 with tanh'")


@pytest.mark.parametrize("B,H,W,ld", [(1, 5, 7, 32), (2, 9, 33, 36), (3, 17, 40, 32), (1, 32, 32, 28), (2, 64, 48, 32)])
@pytest.mark.parametrize("tanh_out", [False, True])
def test_col2im3(B, H, W, ld, tanh_out):
    from ipr_gan_b200 import engine
    g = torch.Generator(device="cuda").manual_seed(B * H * W + ld)
    t = torch.randn(B, H, W, ld, device="cuda", generator=g)
    outs = [engine.col2im3(t, tanh_out) for _ in range(2)]
    torch.cuda.synchronize()
    assert bits_equal(outs[0], outs[1])
    want = R.col2im3_ref_f32(t, tanh_out)
    if tanh_out:                                   # the tap sums are exact; tanhf is within 2 ulp
        within(outs[0], want.cuda(), 6 * U * want.abs().cuda() + 2 ** -149, "col2im3 tanh")
    else:
        assert bits_equal(outs[0].cpu(), want)
