"""Fused AdamW over the flat parameter buffer, with the reference's exact update rule
(optim/adamw.py:80-104) and parameter grouping (optim/misc.py:14-50): eps 1e-6 added to
sqrt(v), bias-corrected step size, decoupled weight decay applied after the Adam update with
the un-corrected lr, no decay for names containing 'bias' / 'LayerNorm.*'.

The reference launches ~10 pointwise kernels for each of ~208 tensors per step; here the flat
layout (decayed parameters first, see params.py) needs TWO launches, and the same kernel refreshes
the bf16 working copy so the next forward skips its cast pass. With `lr_mul != 1` (the fine-tuning
heads, e.g. train_videoQA.py) the reference's four groups are kept: each is a short list of
contiguous flat ranges, one launch per range.
"""
import math

import torch

from . import ops
from .params import FlatParams, is_no_decay


class FusedAdamW:
    def __init__(self, flat, lr=1e-4, betas=(0.9, 0.98), eps=1e-6, weight_decay=0.01,
                 correct_bias=True, lr_mul=1.0):
        assert isinstance(flat, FlatParams) and flat.flat is not None, \
            "call flat_of(model, device) (or run one forward) before building the optimizer"
        self.flat = flat
        self._generation = flat.generation
        self.correct_bias = correct_bias
        self.eps = eps
        self.betas = betas
        split = flat.no_decay_start
        # `param_groups` keeps the reference loops working:
        #     for g in optimizer.param_groups: g['lr'] = lr_this_step   (train_vcmr.py:245-247)
        #     param_groups[0, 1]['lr'] = lr * lr_mul; [2, 3]['lr'] = lr (train_videoQA.py:186-192)
        if float(lr_mul) == 1.0:
            self.param_groups = [
                {"lr": lr, "weight_decay": weight_decay, "ranges": [(0, split)]},
                {"lr": lr, "weight_decay": 0.0, "ranges": [(split, flat.total)]},
            ]
        else:
            self.param_groups = [
                {"lr": lr * lr_mul, "weight_decay": weight_decay, "ranges": []},
                {"lr": lr * lr_mul, "weight_decay": 0.0, "ranges": []},
                {"lr": lr, "weight_decay": weight_decay, "ranges": []},
                {"lr": lr, "weight_decay": 0.0, "ranges": []},
            ]
            for grp, a, b in _group_ranges(flat):
                self.param_groups[grp]["ranges"].append((a, b))
        self.exp_avg = torch.zeros_like(flat.flat)
        self.exp_avg_sq = torch.zeros_like(flat.flat)
        self.step_count = 0
        flat.ensure_flat_grads()

    def zero_grad(self, set_to_none=False):
        self.flat.ensure_flat_grads().zero_()

    def grad_norm(self):
        g = self.flat.ensure_flat_grads()
        acc = torch.zeros(1, dtype=torch.float32, device=g.device)
        ops.sumsq(g, acc)
        return acc.sqrt()

    def clip_grad_norm_(self, max_norm):
        """Global-norm clip folded into the update (train_vcmr.py:258-259): returns the norm and
        remembers the scale for the next step()."""
        total = float(self.grad_norm().item())
        self._grad_scale = min(1.0, max_norm / (total + 1e-6))
        return total

    def clip_grad_norm_device_(self, max_norm):
        """Global-norm clip (train_vcmr.py:258-259) with no device->host read: the sum of squares
        stays on the device and the next step()'s AdamW kernels scale the gradients by
        min(1, max_norm / (norm + 1e-6)) themselves. Returns the device scalar (sum of squares)."""
        g = self.flat.ensure_flat_grads()
        if getattr(self, "_sumsq", None) is None:
            self._sumsq = torch.zeros(1, dtype=torch.float32, device=g.device)
        self._sumsq.zero_()
        ops.sumsq(g, self._sumsq)
        self._clip = float(max_norm)
        return self._sumsq

    def step(self):
        if self.flat.generation != self._generation or self.exp_avg.numel() != self.flat.total:
            raise RuntimeError("the parameters were re-flattened (a module was replaced or moved) "
                               "after this optimizer was built: its moment buffers and ranges no "
                               "longer describe the flat buffer; rebuild the optimizer")
        self.step_count += 1
        t = self.step_count
        b1, b2 = self.betas
        g = self.flat.ensure_flat_grads()
        scale = getattr(self, "_grad_scale", 1.0)
        self._grad_scale = 1.0
        clip = getattr(self, "_clip", None)
        self._clip = None
        for grp in self.param_groups:
            lr = grp["lr"]
            step_size = lr
            if self.correct_bias:
                step_size = lr * math.sqrt(1.0 - b2 ** t) / (1.0 - b1 ** t)
            for a, b in grp["ranges"]:
                if b <= a:
                    continue
                ops.adamw_step(self.flat.flat[a:b], g[a:b], self.exp_avg[a:b],
                               self.exp_avg_sq[a:b], self.flat.mirror[a:b], step_size=step_size,
                               beta1=b1, beta2=b2, eps=self.eps, lr_wd=lr * grp["weight_decay"],
                               grad_scale=scale,
                               clip_sumsq=self._sumsq if clip is not None else None,
                               clip_max_norm=clip or 0.0)
        # masters changed in place through a flat view: the mirror is already fresh
        self.flat.dirty = False
        self.flat._version_sum = sum(p._version for _, p, _, _ in self.flat._probe)

    def state_dict(self):
        return {"step": self.step_count, "exp_avg": self.exp_avg, "exp_avg_sq": self.exp_avg_sq,
                "param_groups": [{k: v for k, v in g.items()} for g in self.param_groups]}

    def load_state_dict(self, sd):
        self.step_count = sd["step"]
        self.exp_avg.copy_(sd["exp_avg"])
        self.exp_avg_sq.copy_(sd["exp_avg_sq"])
        for g, s in zip(self.param_groups, sd["param_groups"]):
            g["lr"], g["weight_decay"] = s["lr"], s["weight_decay"]


def _group_ranges(flat):
    """(group, start, end) per maximal run of flat entries in one of the reference's four groups
    (optim/misc.py:14-37): 0 top-level decay, 1 top-level no-decay, 2 v_encoder decay,
    3 v_encoder no-decay. A run reaches to the next entry's offset (alignment padding included)."""
    runs = []
    ends = [off for _, _, off, _ in flat.entries[1:]] + [flat.total]
    for (name, _, off, _), end in zip(flat.entries, ends):
        grp = 2 * ("v_encoder" in name) + is_no_decay(name)
        if runs and runs[-1][0] == grp and runs[-1][2] == off:
            runs[-1][2] = end
        else:
            runs.append([grp, off, end])
    return [tuple(r) for r in runs]


def build_optimizer(model, opts, device=None):
    """optim/misc.py:14-50 for optim == 'adamw' on the flat layout. With lr_mul == 1 the
    reference's four groups share one learning rate and collapse to TWO flat ranges (decay,
    no-decay). With lr_mul != 1 `param_groups` are the reference's four groups in its order (top
    level x lr_mul decay / no-decay, v_encoder decay / no-decay), which its fine-tuning loops index
    (train_videoQA.py:186-192). Refused: optimizers other than AdamW, frozen parameters."""
    from .params import flat_of
    if getattr(opts, "optim", "adamw") != "adamw":
        raise ValueError(f"hero_b200.build_optimizer implements 'adamw' only (got {opts.optim!r}); "
                         "use the reference's torch optimizer for adam / adamax")
    frozen = [n for n, p in model.named_parameters() if not p.requires_grad]
    if frozen:
        raise ValueError(f"frozen parameters ({frozen[:3]}...) are not supported by the flat "
                         "optimizer: every element of the flat buffer is updated")
    device = device or next(model.parameters()).device
    flat = flat_of(model, device)
    return FusedAdamW(flat, lr=opts.learning_rate, betas=tuple(opts.betas),
                      weight_decay=opts.weight_decay, lr_mul=float(getattr(opts, "lr_mul", 1.0)))
