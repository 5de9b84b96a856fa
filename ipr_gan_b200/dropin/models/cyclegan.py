"""CycleGAN step behind the reference's interface (models/cyclegan.py:10-164): generators GA (A->B) and GB (B->A),
PatchGAN discriminators DA / DB, LSGAN + cycle + identity losses, image-history pools, linearly decaying learning
rate; ``_modules`` = GA, GB, DA, DB, optG, optD, schG, schD, poolA, poolB.

Native step: the four networks run on ``ipr_gan_b200.seqnet``; the loss terms are rows of a table
(name, kind, prediction, target, weight) evaluated by ``ops.pointwise_loss`` -- one launch per term giving the value
and the gradient that seeds the backward pass (``models.core.Seeds``)."""
from itertools import chain

import torch
import torch.nn as nn
from torch import optim

import networks
from models.core import Model, Seeds
from models.srgan import make_optimizer
from models.util import Replica


class ImagePool(nn.Module):
    """History of generated images as registered buffers, so that it is part of the checkpoint (models/util.py:5-35).
    While filling up, images pass through and are stored; once full, each incoming image is exchanged with a random
    stored one with probability 1/2 (the CPU RNG draws ``rand`` then ``randperm``, in that order)."""

    def __init__(self, pool_size):
        super().__init__()
        self.pool_size = pool_size
        if pool_size > 0:
            self.register_buffer("images", torch.tensor([]))
            self.register_buffer("counts", torch.zeros([]))

    def load_state_dict(self, state, *args, **kwargs):
        self.images = torch.empty_like(state["images"])           # the stored history decides the buffer's shape
        return super().load_state_dict(state, *args, **kwargs)

    def forward(self, images):
        images = images.detach()
        if self.pool_size <= 0:
            return images
        n = images.size(0)
        if self.counts < self.pool_size:
            self.images = torch.cat([self.images.to(images.device), images])[:self.pool_size]
            self.counts += n
            return images
        take = torch.rand(n) > 0.5
        where = torch.randperm(self.pool_size)[:n][take]
        out = images.clone()
        out[take] = self.images[where]
        self.images[where] = images[take]
        return out


class CycleGAN(Model):
    seeded = True                        # wrappers add (tensor, gradient) seeds instead of loss-graph terms

    def __init__(self, config, device=[torch.device("cpu"), ]):
        super().__init__()
        self.device = device
        ids = [d.index for d in device]
        for name, key in (("GA", config.G), ("GB", config.G), ("DA", config.D), ("DB", config.D)):
            net = Replica(getattr(networks, key)().to(device[0]), device_ids=ids)
            net.train()
            setattr(self, name, net)
        self.poolA, self.poolB = ImagePool(config.pool_size), ImagePool(config.pool_size)
        self.lambda_A, self.lambda_B, self.lambda_idt = config.lambda_A, config.lambda_B, config.lambda_idt
        self.optG = make_optimizer(config, list(chain(self.GA.parameters(), self.GB.parameters())), device[0])
        self.optD = make_optimizer(config, list(chain(self.DA.parameters(), self.DB.parameters())), device[0])
        half = config.epoch // 2

        def decay(epoch):                                   # models/cyclegan.py:52-59
            return 1.0 - max(0, epoch - half) / half
        self.schedulerG = optim.lr_scheduler.LambdaLR(self.optG, lr_lambda=decay)
        self.schedulerD = optim.lr_scheduler.LambdaLR(self.optD, lr_lambda=decay)
        self._modules.update(GA=self.GA, GB=self.GB, DA=self.DA, DB=self.DB, optG=self.optG, optD=self.optD,
                             schG=self.schedulerG, schD=self.schedulerD, poolA=self.poolA, poolB=self.poolB)
        self.g_seeds = Seeds()
        self._scalars = {}               # metric name -> (0-dim device tensor, factor applied on the host)

    def _terms(self, rows, seeds):
        """rows: (metric name, kind, prediction, target, gradient weight, reported = value * factor)"""
        from ipr_gan_b200 import ops
        for name, kind, pred, target, weight, report in rows:
            value, grad = ops.pointwise_loss(kind, pred, target, weight)
            self._scalars[name] = (value, report)
            seeds.add(pred, grad)

    # ---- two streams, one per direction
    def _pair_streams(self):
        """(main, aux) when the two translation directions may run concurrently, else None.  Every pass of GA and DA
        is issued on the main stream, every pass of GB and DB on the aux stream -- forward and, through autograd,
        backward -- so that all gradient accumulations of one network stay ordered on ONE stream while the two
        directions overlap (at batch 1 a 32 x 32 feature map is 8-32 GEMM tiles on 148 SMs).  Tensors crossing over
        (fake_B -> GB, fake_A -> GA) are ordered by stream waits, which become graph edges under capture."""
        dev = self.device[0]
        if dev.type != "cuda":
            return None
        from ipr_gan_b200 import engine
        if not engine.concurrent_passes():
            return None
        main, aux = torch.cuda.current_stream(dev), engine.aux_stream(dev)
        for net in (self.GB, self.DB):
            object.__setattr__(net, "_ipr_pass_stream", aux)      # models/protect.py runs a trigger pass of GB there
        return main, aux

    # ---- generator step (models/cyclegan.py:91-105, 122-143)
    def forward_g(self, data):
        self.real_A, self.real_B = data["real_A"], data["real_B"]
        for d in (self.DA, self.DB):                       # only dD/d(image) is used in this step
            d.module._ipr_skip_param_grads = True
        try:
            st = self._pair_streams()
            if st is None:
                self.fake_B, self.fake_A = self.GA(self.real_A), self.GB(self.real_B)
                self.rec_A, self.rec_B = self.GB(self.fake_B), self.GA(self.fake_A)
                self.idt_A, self.idt_B = self.GA(self.real_B), self.GB(self.real_A)
                self.GA_logits, self.GB_logits = self.DA(self.fake_B), self.DB(self.fake_A)
            else:
                main, aux = st
                dev = self.device[0]
                self.real_A = self.real_A.to(dev, non_blocking=True)
                self.real_B = self.real_B.to(dev, non_blocking=True)
                aux.wait_stream(main)                      # the inputs exist
                self.fake_B = self.GA(self.real_A)
                with torch.cuda.stream(aux):
                    self.fake_A = self.GB(self.real_B)
                ev_b, ev_a = torch.cuda.Event(), torch.cuda.Event()
                ev_b.record(main)                          # fake_B ready (main), fake_A ready (aux)
                ev_a.record(aux)
                aux.wait_event(ev_b)
                main.wait_event(ev_a)
                with torch.cuda.stream(aux):
                    self.rec_A = self.GB(self.fake_B)
                    self.idt_B = self.GB(self.real_A)
                    self.GB_logits = self.DB(self.fake_A)
                self.rec_B = self.GA(self.fake_A)
                self.idt_A = self.GA(self.real_B)
                self.GA_logits = self.DA(self.fake_B)
                main.wait_stream(aux)
                for t in (self.fake_A, self.rec_A, self.idt_B, self.GB_logits):
                    t.record_stream(main)
                self.fake_B.record_stream(aux)
        finally:
            for d in (self.DA, self.DB):
                d.module._ipr_skip_param_grads = False

    def compute_g_loss(self):
        dev = self.rec_A.device
        self.real_A = self.real_A.to(dev, non_blocking=True)
        self.real_B = self.real_B.to(dev, non_blocking=True)
        la, lb, li = self.lambda_A, self.lambda_B, self.lambda_idt
        self.g_seeds = Seeds()
        rows = [("G/A", "mse", self.GA_logits, 1.0, 1.0, 1.0), ("G/B", "mse", self.GB_logits, 1.0, 1.0, 1.0),
                ("G/CycA", "l1", self.rec_A, self.real_A, la, 1.0), ("G/CycB", "l1", self.rec_B, self.real_B, lb, 1.0)]
        if li > 0:
            # the identity terms enter the total with lambda_idt but are reported without it (models/cyclegan.py:135-141)
            rows += [("G/IdtA", "l1", self.idt_A, self.real_B, lb * li, 1.0 / li),
                     ("G/IdtB", "l1", self.idt_B, self.real_A, la * li, 1.0 / li)]
        self._terms(rows, self.g_seeds)
        total = None
        for name, *_ in rows:
            v = self._scalars[name][0]
            total = v if total is None else total + v
        self.LossG = total                                  # the weighted sum that is minimised
        self.LossGA, self.LossGB = self._scalars["G/A"][0], self._scalars["G/B"][0]

    def backward_g(self, extra=None):
        self.optG.zero_grad()
        self.g_seeds.backward()

    def update_g(self, data, update=True):
        self.forward_g(data)
        self.compute_g_loss()
        if update:
            self.backward_g()
            self.optG.step()

    # ---- discriminator step (models/cyclegan.py:107-120, 145-164)
    def forward_d(self, data):
        self.real_A, self.real_B = data["real_A"], data["real_B"]
        if data.get("pooled", False):      # the caller already exchanged the images with the history pools
            self.fake_A, self.fake_B = data["fake_A"], data["fake_B"]      # (trainer.ProtectedCycleGANTrainer)
        else:                              # several ranks: the pools see the gathered global batch
            from ipr_gan_b200 import dist
            self.fake_A, self.fake_B = dist.pool_query(self.poolA, data["fake_A"]), dist.pool_query(self.poolB, data["fake_B"])
        st = self._pair_streams()
        if st is None:
            self.RA_logits, self.FA_logits = self.DB(self.real_A), self.DB(self.fake_A.detach())
            self.RB_logits, self.FB_logits = self.DA(self.real_B), self.DA(self.fake_B.detach())
            return
        main, aux = st
        dev = self.device[0]
        self.real_A, self.real_B = self.real_A.to(dev, non_blocking=True), self.real_B.to(dev, non_blocking=True)
        fa, fb = self.fake_A.detach().to(dev, non_blocking=True), self.fake_B.detach().to(dev, non_blocking=True)
        aux.wait_stream(main)
        with torch.cuda.stream(aux):                       # DB on its stream, DA on the main stream
            self.RA_logits, self.FA_logits = self.DB(self.real_A), self.DB(fa)
        self.RB_logits, self.FB_logits = self.DA(self.real_B), self.DA(fb)
        main.wait_stream(aux)
        for t in (self.RA_logits, self.FA_logits):
            t.record_stream(main)
        for t in (self.real_A, fa):
            t.record_stream(aux)

    def compute_d_loss(self):
        self._d_seeds = Seeds()
        # each discriminator minimises half the sum of its two terms; the terms are reported un-halved
        self._terms([("D/RealA", "mse", self.RB_logits, 1.0, 0.5, 2.0), ("D/FakeA", "mse", self.FB_logits, 0.0, 0.5, 2.0),
                     ("D/RealB", "mse", self.RA_logits, 1.0, 0.5, 2.0), ("D/FakeB", "mse", self.FA_logits, 0.0, 0.5, 2.0)],
                    self._d_seeds)

    def update_d(self, data):
        self.forward_d(data)
        self.compute_d_loss()
        self.optD.zero_grad()
        self._d_seeds.backward()
        self.optD.step()

    def update_lr(self):
        self.schedulerG.step()
        self.schedulerD.step()

    def get_metrics(self):
        names = sorted(self._scalars)
        vals = torch.stack([self._scalars[n][0] for n in names]).tolist()          # one device-to-host copy
        m = {n: v * self._scalars[n][1] for n, v in zip(names, vals)}
        idt_a, idt_b = m.get("G/IdtA", 0.0), m.get("G/IdtB", 0.0)
        return {"G/A": m["G/A"], "G/B": m["G/B"], "G/CycA": m["G/CycA"], "G/CycB": m["G/CycB"], "G/IdtA": idt_a,
                "G/IdtB": idt_b, "G/Sum": m["G/A"] + m["G/B"] + m["G/CycA"] + m["G/CycB"] + self.lambda_idt * (idt_a + idt_b),
                "D/RealA": m["D/RealA"], "D/FakeA": m["D/FakeA"], "D/SumA": 0.5 * (m["D/RealA"] + m["D/FakeA"]),
                "D/RealB": m["D/RealB"], "D/FakeB": m["D/FakeB"], "D/SumB": 0.5 * (m["D/RealB"] + m["D/FakeB"]),
                "LR": self.optG.param_groups[0]["lr"]}
