"""Flat fp32 arenas for a network's parameters and gradients.

``arena_for(params)`` re-points every parameter's ``.data`` (and ``.grad``) into one contiguous buffer, each
tensor 16-byte aligned.  That is what lets (a) Adam update a whole network in one launch, (b) all bf16 GEMM
operand layouts be rebuilt from the masters by one gather launch, and (c) data-parallel training all-reduce a
network's gradients with a single NCCL call on one buffer.  ``state_dict`` keys / shapes are untouched.
"""
import torch

_BY_PARAM = {}          # id(param) -> Arena


class Arena(object):
    def __init__(self, params):
        params = [p for p in params]
        assert params and all(p.dtype == torch.float32 for p in params)
        dev = params[0].device
        assert all(p.device == dev for p in params)
        self.params = params
        self.offsets = []
        off = 0
        for p in params:
            self.offsets.append(off)
            off += (p.numel() + 3) // 4 * 4                      # keep every tensor 16-byte aligned
        self.numel = max(off, 4)
        self.param = torch.zeros(self.numel, device=dev, dtype=torch.float32)
        self.grad = torch.zeros(self.numel, device=dev, dtype=torch.float32)
        self.version = 0                                          # bumped by whoever rewrites the masters
        # ``clean``: gradient arena known to be all zeros.  Only honoured when ``track_clean`` is set by an owner that
        # controls every writer (the native DCGAN step: all gradients arrive through engine.py, which flags the arena
        # dirty, and FlatAdam clears it as it consumes it); otherwise zero_grad() always clears.
        self.clean = True
        self.track_clean = False
        self.slots = None                                         # 4 floats riding behind/before the gradients
        self.reduce_view = self.grad                              # what a data-parallel all-reduce covers
        with torch.no_grad():
            for p, o in zip(params, self.offsets):
                n = p.numel()
                self.param[o:o + n].copy_(p.data.reshape(-1))
                p.data = self.param[o:o + n].view(p.shape)
                p.grad = self.grad[o:o + n].view(p.shape)
                _BY_PARAM[id(p)] = self
        self.index = {id(p): o for p, o in zip(params, self.offsets)}

    def valid(self):
        base, end = self.param.data_ptr(), self.param.data_ptr() + self.numel * 4
        return all(base <= p.data_ptr() < end for p in self.params)

    def offset_of(self, p):
        return self.index[id(p)]

    def bind_grads(self):
        """(Re-)attach ``.grad`` views (after something set them to None)."""
        for p, o in zip(self.params, self.offsets):
            if p.grad is None or p.grad.data_ptr() != self.grad.data_ptr() + o * 4:
                p.grad = self.grad[o:o + p.numel()].view(p.shape)

    def zero_grad(self):
        if not (self.track_clean and self.clean):   # FlatAdam clears the arena as it consumes it: usually nothing to do
            self.grad.zero_()
            self.clean = True
        self.bind_grads()

    def _rebind(self, grad):
        with torch.no_grad():
            grad.copy_(self.grad)
        self.grad = grad
        for p, o in zip(self.params, self.offsets):
            p.grad = self.grad[o:o + p.numel()].view(p.shape)


def share_gradient_buffer(first, second):
    """Lay two networks' gradient arenas out as ONE allocation  [first.grad | first.slots | second.slots | second.grad].

    Each network's data-parallel all-reduce then covers its gradients AND its four metric slots in a single
    contiguous call (the per-rank loss sums ride along, as SURVEY.md 8e asks), and the eight slots together form
    one contiguous "board" that ``get_metrics()`` fetches with a single copy.  -> the board view."""
    dev = first.grad.device
    n1, n2 = first.numel, second.numel
    buf = torch.zeros(n1 + 8 + n2, device=dev, dtype=torch.float32)
    first._rebind(buf[:n1])
    second._rebind(buf[n1 + 8:])
    first.slots, second.slots = buf[n1:n1 + 4], buf[n1 + 4:n1 + 8]
    first.reduce_view, second.reduce_view = buf[:n1 + 4], buf[n1 + 4:]
    return buf[n1:n1 + 8]


def arena_for(params):
    """The arena holding exactly these parameters (created on first use)."""
    params = list(params)
    hit = _BY_PARAM.get(id(params[0]))
    if hit is not None and hit.valid() and len(hit.params) == len(params) and all(a is b for a, b in zip(hit.params, params)):
        return hit
    return Arena(params)


def module_arena(module):
    """The arena a network's parameters live in (an optimizer may have built one spanning several networks, e.g.
    CycleGAN's optG over both generators), else one for this network alone."""
    params = list(module.parameters())
    arena = arena_of(params[0])                 # validates the arena once; the lookups below are then O(1) each
    if arena is None or any(_BY_PARAM.get(id(p)) is not arena for p in params):
        arena = arena_for(params)
    return arena


def arena_of(param):
    hit = _BY_PARAM.get(id(param))
    return hit if hit is not None and hit.valid() else None
