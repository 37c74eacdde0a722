"""Fused clip_grad_norm_ + AdamW over the engine's flat arenas, plus the reference's optimizer/scheduler factories.

Reference: src/train_utils.py:49-63 (get_optimizer / get_scheduler), transformers-3.0.2 AdamW
(src/transformer/optimization.py:168-267), torch.nn.utils.clip_grad_norm_ (src/multimodal_train.py:361-362).
"""
import ctypes as C
import math

import torch

from . import _lib, ops
from .engine import ALIGN


class FusedAdamW:
    """param_groups: [{'params': [Parameter...], 'weight_decay': float}, ...] exactly as the reference builds them.
    Parameters that appear in no group are never updated (this is how quirk Q1 manifests in the reference).  A frozen parameter
    (requires_grad=False when the engine's last forward ran) is skipped as torch / transformers AdamW skip a None grad: no update,
    no weight decay, moments unchanged.  The step count is shared, so a parameter of the groups whose trainability changes after
    the first step raises ValueError."""

    def __init__(self, engine, param_groups, lr=1e-5, betas=(0.9, 0.999), eps=1e-6, weight_decay=0.0, correct_bias=True,
                 max_grad_norm=None):
        self.engine = engine
        self.lr, self.betas, self.eps, self.correct_bias = lr, betas, eps, correct_bias
        self.max_grad_norm = max_grad_norm
        self.param_groups = [dict(g) for g in param_groups]
        for g in self.param_groups:
            g.setdefault("lr", lr)
        dev = engine.device
        n = engine.numel
        self.m = torch.zeros(n, device=dev)
        self.v = torch.zeros(n, device=dev)
        self.partial = torch.zeros(148 * 8, device=dev)
        self.sumsq = torch.zeros(1, device=dev)
        flags = torch.zeros(n // ALIGN, dtype=torch.uint8)
        by_id = {id(p): name for name, p in engine.params.items()}
        wds = set()
        self._names = []
        for g in self.param_groups:
            wd = float(g.get("weight_decay", weight_decay))
            for p in g["params"]:
                name = by_id.get(id(p))
                if name is None:
                    raise KeyError("parameter is not managed by the engine")
                lo = engine.offsets[name] // ALIGN
                hi = lo + (math.prod(engine.shapes[name]) + ALIGN - 1) // ALIGN
                flags[lo:hi] = 1 | (2 if wd > 0 else 0)
                self._names.append(name)
                if wd > 0:
                    wds.add(wd)
        if len(wds) > 1:
            raise ValueError("one non-zero weight_decay value supported")
        self.weight_decay = wds.pop() if wds else 0.0
        self._group_flags = flags
        self._trainable = None                # the engine's trainable set the device flags were computed for
        self.step_count = 0
        self._sync_flags()

    def _sync_flags(self):
        """Clear the update flags of frozen parameters (recomputed when the engine's trainable set changes)."""
        eng = self.engine
        t = eng.trainable
        if t == self._trainable:
            return
        if self._trainable is not None and self.step_count > 0:
            changed = sorted(n for n in self._names if (n in t) != (n in self._trainable))
            if changed:
                raise ValueError("requires_grad of %s changed after the first step; the fused optimizer keeps one step count for "
                                 "all its parameters (build a new optimizer, or use a torch optimizer)" % changed[:3])
        flags = self._group_flags.clone()
        for name in self._names:
            if name not in t:
                lo = eng.offsets[name] // ALIGN
                flags[lo:lo + (math.prod(eng.shapes[name]) + ALIGN - 1) // ALIGN] = 0
        self.flags = flags.to(eng.device)
        self._trainable = t

    def zero_grad(self, set_to_none=True):
        for p in self.engine.params.values():
            if set_to_none:
                p.grad = None
            elif p.grad is not None:
                p.grad.zero_()

    def step(self, lr=None):
        eng = self.engine
        if lr is None:
            lrs = {g["lr"] for g in self.param_groups if g["params"]}
            if len(lrs) > 1:
                raise ValueError("parameter groups with different learning rates are not supported by the fused step")
            lr = lrs.pop() if lrs else self.lr
        self._sync_flags()
        self.step_count += 1
        b1, b2 = self.betas
        step_size = lr
        if self.correct_bias:
            step_size = lr * math.sqrt(1.0 - b2 ** self.step_count) / (1.0 - b1 ** self.step_count)
        lib = _lib.lib()
        s = ops._stream()
        sumsq = None
        if self.max_grad_norm is not None:
            ops.check(lib.mmsum_grad_sumsq(ops._ptr(eng.G32), C.c_int64(eng.numel), ops._ptr(self.partial), self.partial.numel(),
                                           ops._ptr(self.sumsq), s), "mmsum_grad_sumsq", 2)
            sumsq = self.sumsq
        ops.check(lib.mmsum_adamw_step(ops._ptr(eng.W32), ops._ptr(eng.W16), ops._ptr(eng.G32), ops._ptr(self.m), ops._ptr(self.v),
                                       ops._ptr(self.flags), C.c_int64(eng.numel), C.c_float(lr), C.c_float(b1), C.c_float(b2),
                                       C.c_float(self.eps), C.c_float(self.weight_decay), C.c_float(step_size), ops._ptr(sumsq),
                                       C.c_float(self.max_grad_norm or 0.0), s), "mmsum_adamw_step")
        eng.mark_w16_fresh()                  # W16 was refreshed by the kernel itself

    def grad_norm(self):
        return self.sumsq.sqrt()

    # -- checkpoint interchange (src/train_utils.py:97 saves optimizer.state_dict() into training_state.bin) ---------------
    def state_dict(self):
        """torch.optim-style dict with transformers-AdamW state names (`step`, `exp_avg`, `exp_avg_sq`), so the reference's
        own AdamW can `load_state_dict` it when built over the same parameter groups."""
        eng = self.engine
        by_id = {id(p): name for name, p in eng.params.items()}
        state, groups, idx = {}, [], 0
        for g in self.param_groups:
            ids = []
            for p in g["params"]:
                name = by_id[id(p)]
                o, n = eng.offsets[name], math.prod(eng.shapes[name])
                if self.step_count > 0 and name in self._trainable:      # a frozen parameter was never updated: no state
                    state[idx] = {"step": self.step_count, "exp_avg": self.m[o:o + n].view(eng.shapes[name]).detach().cpu().clone(),
                                  "exp_avg_sq": self.v[o:o + n].view(eng.shapes[name]).detach().cpu().clone()}
                ids.append(idx)
                idx += 1
            groups.append({"lr": g["lr"], "betas": self.betas, "eps": self.eps, "weight_decay": float(g.get("weight_decay", 0.0)),
                           "correct_bias": self.correct_bias, "params": ids})
        return {"state": state, "param_groups": groups}

    def load_state_dict(self, sd):
        eng = self.engine
        by_id = {id(p): name for name, p in eng.params.items()}
        idx = 0
        steps = set()
        for g, gs in zip(self.param_groups, sd["param_groups"]):
            g["lr"] = gs["lr"]
            for p in g["params"]:
                st = sd["state"].get(idx)
                if st is not None:
                    name = by_id[id(p)]
                    o, n = eng.offsets[name], math.prod(eng.shapes[name])
                    self.m[o:o + n].copy_(st["exp_avg"].reshape(-1))
                    self.v[o:o + n].copy_(st["exp_avg_sq"].reshape(-1))
                    steps.add(int(st["step"]))
                idx += 1
        if len(steps) > 1:
            raise ValueError("per-parameter step counts differ; the fused optimizer keeps one")
        self.step_count = steps.pop() if steps else 0


class LinearWarmupSchedule:
    """`get_linear_schedule_with_warmup(optimizer, num_warmup_steps, num_training_steps)` (src/transformer/optimization.py:70-97,
    a torch LambdaLR): `step()` after every optimizer step sets lr = base_lr * lambda(step) in every parameter group.
    As LambdaLR does, construction performs the step-0 update (lr = 0 when there is a warm-up)."""

    def __init__(self, optimizer, num_warmup_steps, num_training_steps, last_epoch=-1):
        self.optimizer = optimizer
        self.num_warmup_steps, self.num_training_steps = num_warmup_steps, num_training_steps
        self.base_lrs = [g["lr"] for g in optimizer.param_groups]
        self.last_epoch = last_epoch
        self.step()

    def lr_lambda(self, current_step):
        if current_step < self.num_warmup_steps:
            return float(current_step) / float(max(1, self.num_warmup_steps))
        return max(0.0, float(self.num_training_steps - current_step) / float(max(1, self.num_training_steps - self.num_warmup_steps)))

    def step(self):
        self.last_epoch += 1
        for g, base in zip(self.optimizer.param_groups, self.base_lrs):
            g["lr"] = base * self.lr_lambda(self.last_epoch)

    def get_last_lr(self):
        return [g["lr"] for g in self.optimizer.param_groups]

    def state_dict(self):
        return {"base_lrs": list(self.base_lrs), "last_epoch": self.last_epoch, "_step_count": self.last_epoch + 1,
                "_last_lr": self.get_last_lr()}

    def load_state_dict(self, sd):
        self.base_lrs, self.last_epoch = list(sd["base_lrs"]), sd["last_epoch"]
        for g, base in zip(self.optimizer.param_groups, self.base_lrs):
            g["lr"] = base * self.lr_lambda(self.last_epoch)


def get_optimizer(engine, lr, no_decay, named_parameters, special_condition=None, max_grad_norm=None):
    """src/train_utils.py:49-57, statement for statement — including quirk Q1: when `named_parameters` is a generator
    (as `model.named_parameters()` is), the second comprehension finds it exhausted and the no-decay group is empty."""
    if special_condition is None:
        special_condition = lambda n: True  # noqa: E731
    groups = [
        {"params": [p for n, p in named_parameters if special_condition(n) and (not any(nd in n for nd in no_decay))],
         "weight_decay": 0.01},
        {"params": [p for n, p in named_parameters if special_condition(n) and (any(nd in n for nd in no_decay))],
         "weight_decay": 0.0},
    ]
    return FusedAdamW(engine, groups, lr=lr, max_grad_norm=max_grad_norm)


def get_scheduler(args, t_epoch, optimizer):
    """src/train_utils.py:59-63."""
    t_total = t_epoch * args.num_epochs
    warmup_step = int(t_total * args.warmup_ratio)
    return LinearWarmupSchedule(optimizer, num_warmup_steps=warmup_step, num_training_steps=t_total)


def linear_schedule_with_warmup(base_lr, num_warmup_steps, num_training_steps):
    """get_linear_schedule_with_warmup (src/transformer/optimization.py:70-97) as a step -> lr function."""
    def lr_at(step):
        if step < num_warmup_steps:
            return base_lr * float(step) / float(max(1, num_warmup_steps))
        return base_lr * max(0.0, float(num_training_steps - step) / float(max(1, num_training_steps - num_warmup_steps)))
    return lr_at
