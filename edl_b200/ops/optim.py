"""Flat-buffer fused optimizers (csrc/optim.cu) + LR schedules.

``FlatSGDMomentum`` is the B200 counterpart of the reference's ``Momentum(lr, 0.9, L2Decay(1e-4))``
(example/distill/resnet/train_with_fleet.py:106-122) and its AMP master-weight helpers
(example/distill/resnet/utils/fp16_utils.py:86-129): one kernel per dtype group updates fp32 master
weights + momentum and writes the bf16 model copy.  The learning rate lives in a device scalar so a
captured CUDA graph can be replayed while the host-side schedule (reference:
utils/learning_rate.py:39-95 cosine/piecewise with warm-up) only updates that scalar.

``FlatLARS`` / ``FlatLAMB`` (csrc/optim_layerwise.cu) are the large-batch rules, Paddle's
``LarsMomentumOptimizer`` / ``LambOptimizer``: per-tensor norms over the flat buffers by a two-pass segmented
reduction, bitwise deterministic, with ``polynomial_decay_with_warmup`` as the schedule of the LARS recipes.
"""
from __future__ import annotations

import math
from typing import Optional

import torch


class _FlatOptimizerBase:
    def __init__(self, flat, lr: float):
        self.flat = flat
        dev = flat.device
        self.lr = float(lr)
        self.lr_t = torch.full((1,), float(lr), dtype=torch.float32, device=dev)
        self.grad_scale_t: Optional[torch.Tensor] = None  # device scalar multiplied into grads
        self.found_inf_t: Optional[torch.Tensor] = None   # device int flag: skip step when != 0
        self._found_inf_is_comm_error = False
        self.skip_dtype = None    # set by ElasticDataParallel.attach_optimizer: dtype -> "already updated this step"

    def set_lr(self, lr: float):
        self.lr = float(lr)
        self.lr_t.fill_(self.lr)

    def set_grad_scale(self, t: Optional[torch.Tensor]):
        self.grad_scale_t = t

    def set_found_inf(self, t: Optional[torch.Tensor], comm_error: bool = False):
        """``comm_error``: the flag is the fabric's error word (in-place elastic guard), not a gradient overflow
        flag -- the per-bucket fused optimizer may then still be used (its kernel checks the word itself)."""
        self.found_inf_t = t
        self._found_inf_is_comm_error = bool(comm_error) and t is not None

    def found_inf_is_comm_error(self) -> bool:
        return self.found_inf_t is None or self._found_inf_is_comm_error

    def zero_grad(self):
        self.flat.zero_grad()


class FlatSGDMomentum(_FlatOptimizerBase):
    def __init__(self, flat, lr=0.1, momentum=0.9, weight_decay=1e-4, nesterov=False,
                 decay_filter=None):
        super().__init__(flat, lr)
        self.momentum, self.weight_decay, self.nesterov = momentum, weight_decay, nesterov
        self.state = {}
        for dt, g in flat.groups.items():
            st = {"mom": torch.zeros(g.numel, dtype=torch.float32, device=flat.device), "wd_mask": None}
            if decay_filter is not None:
                mask = torch.zeros(g.numel, dtype=torch.float32, device=flat.device)
                for e in g.entries:
                    if decay_filter(e.name, e.param):
                        mask[e.offset:e.offset + e.numel] = 1.0
                st["wd_mask"] = mask
            self.state[dt] = st

    @torch.no_grad()
    def step(self):
        from . import native, count_launch

        for dt, g in self.flat.groups.items():
            if self.skip_dtype is not None and self.skip_dtype(dt):
                continue                 # updated bucket by bucket by the data-parallel engine (parallel/ddp.py)
            st = self.state[dt]
            master = g.master if g.master is not None else g.param
            lp = g.param if g.master is not None else None
            if g.param.is_cuda:
                native().sgd_momentum(lp, master, st["mom"], g.grad, st["wd_mask"], self.lr_t,
                                      self.grad_scale_t, self.found_inf_t, self.momentum,
                                      self.weight_decay, self.nesterov)
                count_launch()
            else:
                if self.found_inf_t is not None and int(self.found_inf_t.item()) != 0:
                    continue
                grad = g.grad.float()
                if self.grad_scale_t is not None:
                    grad = grad * self.grad_scale_t
                wd = self.weight_decay if st["wd_mask"] is None else self.weight_decay * st["wd_mask"]
                grad = grad + wd * master
                st["mom"].mul_(self.momentum).add_(grad)
                upd = grad + self.momentum * st["mom"] if self.nesterov else st["mom"]
                master.add_(upd * (-self.lr_t))
                if lp is not None:
                    lp.copy_(master.to(lp.dtype))

    def state_dict(self):
        return {
            "lr": self.lr,
            "momentum": {str(dt): st["mom"] for dt, st in self.state.items()},
            "master": {str(dt): (g.master if g.master is not None else g.param)
                       for dt, g in self.flat.groups.items()},
        }

    def load_state_dict(self, sd):
        self.set_lr(sd["lr"])
        for dt, st in self.state.items():
            st["mom"].copy_(sd["momentum"][str(dt)])
        for dt, g in self.flat.groups.items():
            src = sd["master"][str(dt)]
            if g.master is not None:
                g.master.copy_(src)
                g.param.copy_(src.to(g.param.dtype))
            else:
                g.param.copy_(src)


class FlatAdam(_FlatOptimizerBase):
    """Adam / AdamW on flat buffers (CTR-DNN uses Adam 1e-4, example/ctr/ctr/train.py:234; the NLP
    distill students use AdamW, example/distill/nlp/model.py:35-51)."""

    def __init__(self, flat, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.0,
                 decoupled=False):
        super().__init__(flat, lr)
        self.betas, self.eps, self.weight_decay, self.decoupled = betas, eps, weight_decay, decoupled
        self.step_t = torch.zeros(1, dtype=torch.float32, device=flat.device)
        self.state = {dt: {"m": torch.zeros(g.numel, dtype=torch.float32, device=flat.device),
                           "v": torch.zeros(g.numel, dtype=torch.float32, device=flat.device)}
                      for dt, g in flat.groups.items()}

    @torch.no_grad()
    def step(self):
        from . import native, count_launch

        # bias correction counts APPLIED steps only: a step skipped by found_inf (loss-scaling overflow, broken
        # collective) must not advance it -- decided on the device, no host round trip
        if self.found_inf_t is not None:
            if not self.step_t.is_cuda and int(self.found_inf_t.item()) != 0:
                return
            self.step_t += (self.found_inf_t.view(-1)[:1] == 0).to(self.step_t.dtype)
        else:
            self.step_t += 1
        for dt, g in self.flat.groups.items():
            st = self.state[dt]
            master = g.master if g.master is not None else g.param
            lp = g.param if g.master is not None else None
            if g.param.is_cuda:
                native().adam_step(lp, master, st["m"], st["v"], g.grad, self.lr_t,
                                   self.grad_scale_t, self.found_inf_t, self.step_t, self.betas[0],
                                   self.betas[1], self.eps, self.weight_decay, self.decoupled)
                count_launch()
            else:
                grad = g.grad.float()
                if self.grad_scale_t is not None:
                    grad = grad * self.grad_scale_t
                if not self.decoupled:
                    grad = grad + self.weight_decay * master
                b1, b2 = self.betas
                st["m"].mul_(b1).add_(grad, alpha=1 - b1)
                st["v"].mul_(b2).addcmul_(grad, grad, value=1 - b2)
                t = float(self.step_t.item())
                mhat = st["m"] / (1 - b1 ** t)
                vhat = st["v"] / (1 - b2 ** t)
                if self.decoupled:
                    master.mul_(1 - self.lr * self.weight_decay)
                master.add_(-self.lr * mhat / (vhat.sqrt() + self.eps))
                if lp is not None:
                    lp.copy_(master.to(lp.dtype))

    def state_dict(self):
        return {"lr": self.lr, "step": self.step_t,
                "m": {str(dt): st["m"] for dt, st in self.state.items()},
                "v": {str(dt): st["v"] for dt, st in self.state.items()},
                "master": {str(dt): (g.master if g.master is not None else g.param)
                           for dt, g in self.flat.groups.items()}}

    def load_state_dict(self, sd):
        self.set_lr(sd["lr"])
        self.step_t.copy_(sd["step"])
        for dt, st in self.state.items():
            st["m"].copy_(sd["m"][str(dt)])
            st["v"].copy_(sd["v"][str(dt)])
        for dt, g in self.flat.groups.items():
            src = sd["master"][str(dt)]
            if g.master is not None:
                g.master.copy_(src)
                g.param.copy_(src.to(g.param.dtype))
            else:
                g.param.copy_(src)


CHUNK_ELEMS = 8192   # elements per chunk of the layer-wise optimizers' chunk tables (one CTA each)


class _LayerwiseOptimizerBase(_FlatOptimizerBase):
    """Shared plumbing of the optimizers whose update depends on per-tensor norms (LARS, LAMB).

    On CUDA every update is two launches over a chunk table (csrc/optim_layerwise.cu): chunks of at most
    ``CHUNK_ELEMS`` elements that never straddle two tensors, each with its tensor's chunk range and decay flag.
    Tables are built on the host and uploaded once: one per dtype group for ``step()``, and one per bucket when
    the data-parallel engine applies the optimizer bucket by bucket (``plan_ranges`` / ``step_range``).  They
    live outside ``self.state``, which holds optimizer tensors only."""

    def __init__(self, flat, lr, exclude=None):
        super().__init__(flat, lr)
        # per dtype group: decay flag of every entry (False = excluded from weight decay / the trust ratio's wd)
        self._decay = {dt: [exclude is None or not exclude(e.name, e.param) for e in g.entries]
                       for dt, g in flat.groups.items()}
        self._tables = {}          # (dtype, start, numel) -> (int64 [n, 5] chunk table, fp32 [n, 2] partials)
        self._range_keys = set()   # the bucket tables of the current plan
        if flat.device.type == "cuda":
            for dt, g in flat.groups.items():
                self._table(dt, 0, g.numel)

    # ---------------------------------------------------------------- chunk tables
    def _entries_in(self, dt, start, numel):
        """(index, entry) of the group's entries lying inside [start, start + numel)."""
        end = start + numel
        for i, e in enumerate(self.flat.groups[dt].entries):
            if e.offset >= start and e.offset + e.numel <= end:
                yield i, e
            elif e.offset < end and e.offset + e.numel > start:
                raise ValueError("range [%d, %d) cuts tensor %s: per-tensor norms need whole tensors"
                                 % (start, end, e.name))

    def _table(self, dt, start, numel):
        key = (dt, int(start), int(numel))
        hit = self._tables.get(key)
        if hit is not None:
            return hit
        if torch.cuda.is_current_stream_capturing():
            raise RuntimeError("chunk table for %s [%d, +%d) requested inside a CUDA-graph capture: plan it first "
                               "(plan_ranges)" % key)
        rows = []
        decay = self._decay[dt]
        for i, e in self._entries_in(dt, start, numel):
            first = len(rows)
            count = -(-e.numel // CHUNK_ELEMS)
            for c in range(count):
                lo = c * CHUNK_ELEMS
                rows.append((e.offset - start + lo, min(CHUNK_ELEMS, e.numel - lo), first, count, int(decay[i])))
        table = torch.tensor(rows, dtype=torch.int64).view(-1, 5).to(self.flat.device)
        partials = torch.zeros(max(1, len(rows)), 2, dtype=torch.float32, device=self.flat.device)
        self._tables[key] = (table, partials)
        return self._tables[key]

    def plan_ranges(self, ranges):
        """Build (once, outside any capture) the chunk tables of the ranges ``step_range`` will be called with --
        the engine's bucket plan; tables of a previous plan are dropped."""
        keys = {(dt, int(s), int(n)) for dt, s, n in ranges}
        for k in self._range_keys - keys:
            if k[1:] != (0, self.flat.groups[k[0]].numel):
                self._tables.pop(k, None)
        self._range_keys = keys
        if self.flat.device.type == "cuda":
            for k in keys:
                self._table(*k)

    # ---------------------------------------------------------------- stepping
    def _found_inf_set(self) -> bool:
        """CPU path only: the host may look at the flag."""
        return self.found_inf_t is not None and int(self.found_inf_t.view(-1)[0].item()) != 0

    def _grad_scale(self) -> float:
        return 1.0 if self.grad_scale_t is None else float(self.grad_scale_t.view(-1)[0].item())

    def _windows(self, dt, start, numel):
        g = self.flat.groups[dt]
        lo, hi = start, start + numel
        master = g.master if g.master is not None else g.param
        lp = g.param[lo:hi] if g.master is not None else None
        return g, master[lo:hi], lp, g.grad[lo:hi]

    @torch.no_grad()
    def step_range(self, dtype, start: int, numel: int):
        """Apply this step's update to the whole tensors inside [start, start + numel) of the dtype group (one
        bucket of the data-parallel engine).  Does not advance step counters: ``step()`` does, once per step."""
        self._apply(dtype, int(start), int(numel))

    @torch.no_grad()
    def step(self):
        for dt, g in self.flat.groups.items():
            if self.skip_dtype is not None and self.skip_dtype(dt):
                continue                 # updated bucket by bucket by the data-parallel engine (parallel/ddp.py)
            self._apply(dt, 0, g.numel)
        self._advance()

    def _advance(self):
        pass

    def _entry_views(self, dt, start, numel, *bufs):
        """CPU path: per-entry windows of the group's flat buffers (master, model copy, grad, state...)."""
        g = self.flat.groups[dt]
        master = g.master if g.master is not None else g.param
        for i, e in self._entries_in(dt, start, numel):
            sl = slice(e.offset, e.offset + e.numel)
            yield (self._decay[dt][i], master[sl], g.param[sl] if g.master is not None else None, g.grad[sl],
                   *[b[sl] for b in bufs])


class FlatLARS(_LayerwiseOptimizerBase):
    """LARS (layer-wise adaptive rate scaling, You et al. 2017) in Paddle's ``LarsMomentumOptimizer`` form, on the
    flat buffers.  Per tensor, with ``g = grad * grad_scale`` and ``wd = 0`` for tensors ``exclude(name, param)``
    selects (the MLPerf recipe: BatchNorm scale / shift and biases)::

        local_lr = lr * lars_coeff * |w| / (|g| + wd * |w| + epsilon)   if wd > 0 and |w| > 0 and |g| > 0, else lr
        v = momentum * v + local_lr * (g + wd * w);   w = w - v

    For large-batch elastic jobs: the global batch grows with the world size (``scaled_lr``), and plain momentum
    SGD loses accuracy beyond a few thousand images per step."""

    def __init__(self, flat, lr, momentum=0.9, lars_coeff=0.001, lars_weight_decay=5e-4, epsilon=0.0,
                 exclude=None):
        self.momentum, self.lars_coeff = float(momentum), float(lars_coeff)
        self.lars_weight_decay, self.epsilon = float(lars_weight_decay), float(epsilon)
        super().__init__(flat, lr, exclude)
        self.state = {dt: {"mom": torch.zeros(g.numel, dtype=torch.float32, device=flat.device)}
                      for dt, g in flat.groups.items()}

    def _apply(self, dt, start, numel):
        from . import native, count_launch

        g, master, lp, grad = self._windows(dt, start, numel)
        mom = self.state[dt]["mom"]
        if g.param.is_cuda:
            table, partials = self._table(dt, start, numel)
            if table.shape[0] == 0:
                return
            native().lars_step(lp, master, mom[start:start + numel], grad, table, partials, self.lr_t,
                               self.grad_scale_t, self.found_inf_t, self.momentum, self.lars_coeff,
                               self.lars_weight_decay, self.epsilon)
            count_launch(2)
            return
        if self._found_inf_set():
            return
        lr, gs = float(self.lr_t.view(-1)[0].item()), self._grad_scale()
        for decay, w, p, gr, v in self._entry_views(dt, start, numel, mom):
            wd = self.lars_weight_decay if decay else 0.0
            gf = gr.float() * gs
            wn, gn = float(w.norm()), float(gf.norm())
            local_lr = lr * self.lars_coeff * wn / (gn + wd * wn + self.epsilon) if wd > 0 and wn > 0 and gn > 0 else lr
            v.mul_(self.momentum).add_(gf.add(w, alpha=wd), alpha=local_lr)
            w.sub_(v)
            if p is not None:
                p.copy_(w.to(p.dtype))

    def state_dict(self):
        return {
            "lr": self.lr,
            "momentum": {str(dt): st["mom"] for dt, st in self.state.items()},
            "master": {str(dt): (g.master if g.master is not None else g.param)
                       for dt, g in self.flat.groups.items()},
        }

    def load_state_dict(self, sd):
        self.set_lr(sd["lr"])
        for dt, st in self.state.items():
            st["mom"].copy_(sd["momentum"][str(dt)])
        _load_masters(self.flat, sd["master"])


class FlatLAMB(_LayerwiseOptimizerBase):
    """LAMB (You et al. 2019) in Paddle's ``LambOptimizer`` form, on the flat buffers.  Per tensor, with
    ``g = grad * grad_scale``, ``t`` = applied steps including this one and ``wd = 0`` for excluded tensors::

        m = b1 * m + (1 - b1) * g;   v = b2 * v + (1 - b2) * g^2
        r = (m / (1 - b1^t)) / (sqrt(v / (1 - b2^t)) + eps) + wd * w
        w = w - lr * (|w| / |r| if both > 0 else 1) * r

    The step counter lives on the device and advances only on applied steps (``found_inf`` == 0), as in
    ``FlatAdam``."""

    def __init__(self, flat, lr, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.01, exclude=None):
        self.betas, self.eps, self.weight_decay = (float(betas[0]), float(betas[1])), float(eps), float(weight_decay)
        super().__init__(flat, lr, exclude)
        self.step_t = torch.zeros(1, dtype=torch.float32, device=flat.device)   # applied steps so far
        self.state = {dt: {"m": torch.zeros(g.numel, dtype=torch.float32, device=flat.device),
                           "v": torch.zeros(g.numel, dtype=torch.float32, device=flat.device)}
                      for dt, g in flat.groups.items()}

    def _apply(self, dt, start, numel):
        from . import native, count_launch

        g, master, lp, grad = self._windows(dt, start, numel)
        st = self.state[dt]
        b1, b2 = self.betas
        if g.param.is_cuda:
            table, partials = self._table(dt, start, numel)
            if table.shape[0] == 0:
                return
            # the kernels use step_t + 1: the counter itself advances in _advance(), after every range of the step
            native().lamb_step(lp, master, st["m"][start:start + numel], st["v"][start:start + numel], grad, table,
                               partials, self.lr_t, self.grad_scale_t, self.found_inf_t, self.step_t, b1, b2,
                               self.eps, self.weight_decay)
            count_launch(2)
            return
        if self._found_inf_set():
            return
        lr, gs = float(self.lr_t.view(-1)[0].item()), self._grad_scale()
        t = float(self.step_t.item()) + 1.0
        bc1, bc2 = 1.0 - b1 ** t, 1.0 - b2 ** t
        for decay, w, p, gr, m, v in self._entry_views(dt, start, numel, st["m"], st["v"]):
            wd = self.weight_decay if decay else 0.0
            gf = gr.float() * gs
            m.mul_(b1).add_(gf, alpha=1 - b1)
            v.mul_(b2).addcmul_(gf, gf, value=1 - b2)
            r = (m / bc1) / ((v / bc2).sqrt() + self.eps) + wd * w
            wn, rn = float(w.norm()), float(r.norm())
            trust = wn / rn if wn > 0 and rn > 0 else 1.0
            w.add_(r, alpha=-lr * trust)
            if p is not None:
                p.copy_(w.to(p.dtype))

    def _advance(self):
        if self.found_inf_t is None:
            self.step_t += 1
        elif self.step_t.is_cuda:
            self.step_t += (self.found_inf_t.view(-1)[:1] == 0).to(self.step_t.dtype)
        elif not self._found_inf_set():
            self.step_t += 1

    def state_dict(self):
        return {"lr": self.lr, "step": self.step_t,
                "m": {str(dt): st["m"] for dt, st in self.state.items()},
                "v": {str(dt): st["v"] for dt, st in self.state.items()},
                "master": {str(dt): (g.master if g.master is not None else g.param)
                           for dt, g in self.flat.groups.items()}}

    def load_state_dict(self, sd):
        self.set_lr(sd["lr"])
        self.step_t.copy_(sd["step"])
        for dt, st in self.state.items():
            st["m"].copy_(sd["m"][str(dt)])
            st["v"].copy_(sd["v"][str(dt)])
        _load_masters(self.flat, sd["master"])


def _load_masters(flat, masters):
    for dt, g in flat.groups.items():
        src = masters[str(dt)]
        if g.master is not None:
            g.master.copy_(src)
            g.param.copy_(src.to(g.param.dtype))
        else:
            g.param.copy_(src)


# ---------------------------------------------------------------------------------------------
# LR schedules (host side; the result is written into the optimizer's device scalar)

def cosine_decay_with_warmup(step: int, base_lr: float, steps_per_epoch: int, epochs: int,
                             warmup_epochs: int = 5) -> float:
    """Linear warm-up then per-epoch cosine decay (reference utils/learning_rate.py:39-60)."""
    warm = warmup_epochs * steps_per_epoch
    if step < warm:
        return base_lr * step / max(warm, 1)
    epoch = step // max(steps_per_epoch, 1)
    return base_lr * 0.5 * (math.cos((epoch - warmup_epochs) * math.pi / max(epochs - warmup_epochs, 1)) + 1)


def piecewise_decay_with_warmup(step: int, base_lr: float, steps_per_epoch: int, boundaries_epochs,
                                gamma: float = 0.1, warmup_epochs: int = 5) -> float:
    """Step decay at epoch boundaries with linear warm-up (reference utils/learning_rate.py:62-95)."""
    warm = warmup_epochs * steps_per_epoch
    if step < warm:
        return base_lr * step / max(warm, 1)
    epoch = step // max(steps_per_epoch, 1)
    k = sum(1 for b in boundaries_epochs if epoch >= b)
    return base_lr * (gamma ** k)


def scaled_lr(lr: float, batch_per_trainer: int, num_trainers: int, ref_batch: int = 256) -> float:
    """``base_lr = lr * (batch * num_trainers) / 256`` -- the reference's world-size LR rescale
    (example/collective/resnet50/train_with_fleet.py:129-141)."""
    return lr * (batch_per_trainer * num_trainers) / ref_batch


def polynomial_decay_with_warmup(step: int, base_lr: float, steps_per_epoch: int, epochs: int, warmup_epochs: int,
                                 power: float = 2.0, end_lr: float = 0.0) -> float:
    """Linear warm-up, then ``(base_lr - end_lr) * (1 - progress) ** power + end_lr`` per step until the end of
    ``epochs`` -- the schedule of the LARS large-batch ResNet-50 recipes (MLPerf: power 2)."""
    warm = warmup_epochs * steps_per_epoch
    if step < warm:
        return base_lr * step / max(warm, 1)
    total = epochs * steps_per_epoch
    frac = min(1.0, (step - warm) / max(total - warm, 1))
    return (base_lr - end_lr) * (1.0 - frac) ** power + end_lr
