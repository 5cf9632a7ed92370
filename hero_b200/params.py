"""Flat parameter storage: fp32 masters as views of one buffer + a bf16 working mirror.

The reference keeps ~208 separate tensors and pays a pack/all-reduce/unpack copy for its gradient
exchange (utils/distributed.py:19-46) plus ~10 kernels per tensor in AdamW (optim/adamw.py:80-104).
Here every nn.Parameter of a module tree becomes a VIEW into one contiguous fp32 buffer (state_dict
keys and shapes unchanged, `load_state_dict` copies in place), ordered so that each layer's
query/key/value weights (and biases) are adjacent: the fused QKV GEMM reads them as one
[3H, H] matrix without any concatenation. A same-layout bf16 mirror feeds the tensor-core
kernels and is refreshed by ONE cast kernel when the masters changed.
"""
import re

import weakref

import torch

from . import ops

_ALIGN = 64  # elements; keeps every view 128-byte aligned in bf16 (TMA needs 16 B)


def _ordered_named_params(module):
    named = list(module.named_parameters())   # de-duplicated (tied weights appear once)
    by_name = dict(named)
    out, placed = [], set()
    for name, p in named:
        if name in placed:
            continue
        m = re.match(r"(.*attention\.self\.)query\.weight$", name)
        if m:
            base = m.group(1)
            group = [base + s for s in ("query.weight", "key.weight", "value.weight",
                                        "query.bias", "key.bias", "value.bias")]
            if all(g in by_name for g in group):
                for g in group:
                    out.append((g, by_name[g]))
                    placed.add(g)
                continue
        out.append((name, p))
        placed.add(name)
    # decayed parameters first, then the no-decay set of optim/misc.py:22 (names containing
    # 'bias' / 'LayerNorm.bias' / 'LayerNorm.weight'): the fused AdamW then needs two launches.
    # Inside each group, the parameters whose gradients only become final at the very end of
    # backward (the cross-modal embeddings: word / position / type tables, frame projection) go
    # last, so "everything that is final once the transformer stacks are differentiated" is one
    # contiguous range per group (distributed.FlatGradExchange reduces it during the embedding
    # backward). Stable sort keeps q/k/v weights (and q/k/v biases) adjacent.
    out.sort(key=lambda np_: (is_no_decay(np_[0]), is_late_grad(np_[0])))
    return out


NO_DECAY = ("bias", "LayerNorm.bias", "LayerNorm.weight")


def is_no_decay(name):
    return any(nd in name for nd in NO_DECAY)


LATE_GRAD = ("f_encoder.embeddings.", "f_encoder.img_embeddings.")


def is_late_grad(name):
    """Parameters differentiated by the LAST backward node (functional._CrossModalEmbed)."""
    return any(t in name for t in LATE_GRAD)


# Every live FlatParams; any torch optimizer step marks their bf16 mirrors stale (global post-step
# hook). The reference's optimizers update `p.data` in place (optim/adamw.py:94-104), which does
# not bump `p._version`, so the version probe in `ensure` alone would miss them.
_LIVE = weakref.WeakSet()
_HOOK = []


def _after_optimizer_step(optimizer, args, kwargs):
    for fp in list(_LIVE):
        fp.mark_dirty()


def _install_optimizer_hook():
    if not _HOOK:
        from torch.optim.optimizer import register_optimizer_step_post_hook
        _HOOK.append(register_optimizer_step_post_hook(_after_optimizer_step))


class FlatParams:
    def __init__(self, module):
        self.module = module
        self.flat = None
        self.mirror = None
        self.entries = []            # (name, param, offset, numel)
        self._by_id = {}
        self.dirty = True
        self._version_sum = -1
        self.grad_flat = None
        self._stale = False
        self._probe = []
        self._hooked = False
        self.generation = 0          # bumped by every re-flatten (optimizers / exchanges check it)
        _LIVE.add(self)
        _install_optimizer_hook()

    # ------------------------------------------------------------------ layout
    def _needs_flatten(self, device):
        """O(1) check: parameters that were moved (.to / .cuda) or replaced (pad_vocab, new
        modules) no longer point into the flat buffer. Structural edits that keep the sampled
        parameters in place must call `invalidate()`."""
        if self.flat is None or self.flat.device != device or self._stale:
            return True
        base = self.flat.data_ptr()
        for _, p, off, n in self._probe:
            if p.data_ptr() != base + off * 4:
                return True
        return False

    def invalidate(self):
        self._stale = True

    def ensure(self, device):
        """(Re)build the flat buffers if parameters were moved / replaced; refresh the mirror when
        the masters may have changed (after a backward, after load_state_dict, or when one of the
        probed parameters reports a new version)."""
        device = torch.device(device)
        if self._needs_flatten(device):
            named = _ordered_named_params(self.module)
            offs, total = [], 0
            for _, p in named:
                offs.append(total)
                total += (p.numel() + _ALIGN - 1) // _ALIGN * _ALIGN
            flat = torch.zeros(total, dtype=torch.float32, device=device)
            self.entries, self._by_id = [], {}
            with torch.no_grad():
                for (name, p), off in zip(named, offs):
                    view = flat[off:off + p.numel()].view(p.shape)
                    view.copy_(p.data.to(device=device, dtype=torch.float32))
                    p.data = view
                    self.entries.append((name, p, off, p.numel()))
                    self._by_id[id(p)] = (off, p.numel())
            self.flat = flat
            self.total = total
            # first element of the no-decay block (== total when every parameter decays)
            self.no_decay_start = next((off for (name, _), off in zip(named, offs)
                                        if is_no_decay(name)), total)
            # [early, late) split of each group: gradients in the "early" ranges are final when
            # the last transformer stack has been differentiated
            self.late_start_decay = next((off for (name, _), off in zip(named, offs)
                                          if not is_no_decay(name) and is_late_grad(name)),
                                         self.no_decay_start)
            self.late_start_no_decay = next((off for (name, _), off in zip(named, offs)
                                             if is_no_decay(name) and is_late_grad(name)), total)
            self.mirror = torch.empty(total, dtype=torch.bfloat16, device=device)
            self.grad_flat = None
            self.dirty = True
            self._stale = False
            self.generation += 1
            # every submodule resolves to THIS manager (modules swapped in after the first flatten,
            # e.g. HeroModel.load_partial_pretrained replacing f_encoder, must not build a private
            # one and pull their parameters out of the shared buffer)
            for m in self.module.modules():
                m.__dict__["_hero_flat"] = self
            k = max(1, len(self.entries) // 8)
            self._probe = self.entries[::k] + self.entries[-1:]
            if not self._hooked:
                self.module.register_load_state_dict_post_hook(
                    lambda module, incompatible: self.mark_dirty())
                self._hooked = True
        vs = 0
        for _, p, _, _ in self._probe:
            vs += p._version
        if self.dirty or vs != self._version_sum:
            ops.cast_bf16(self.flat, self.mirror)
            self.dirty = False
            self._version_sum = vs
        return self

    def mark_dirty(self):
        """The fp32 masters changed: refresh the bf16 mirror before the next forward. Called
        automatically after every `torch.optim.Optimizer.step()` and `load_state_dict`; call it by
        hand after editing weights through `p.data` outside an optimizer."""
        self.dirty = True

    def early_ranges(self):
        """Flat ranges whose gradients are final before the cross-modal embedding backward."""
        return [(0, self.late_start_decay), (self.no_decay_start, self.late_start_no_decay)]

    def late_ranges(self):
        return [(self.late_start_decay, self.no_decay_start),
                (self.late_start_no_decay, self.total)]

    # ------------------------------------------------------------------ views
    def bf16(self, p):
        off, n = self._by_id[id(p)]
        return self.mirror[off:off + n].view(p.shape)

    def bf16_span(self, first, count, shape):
        """bf16 view starting at parameter `first` spanning `count` elements (fused QKV)."""
        off, _ = self._by_id[id(first)]
        return self.mirror[off:off + count].view(shape)

    def f32_span(self, first, count, shape):
        off, _ = self._by_id[id(first)]
        return self.flat[off:off + count].view(shape)

    def contiguous_after(self, a, b):
        """True if parameter b starts right where a ends (no alignment gap)."""
        oa, na = self._by_id[id(a)]
        ob, _ = self._by_id[id(b)]
        return oa + na == ob

    # ------------------------------------------------------------------ flat gradients
    def ensure_flat_grads(self):
        """Point every p.grad at a view of one flat fp32 buffer (absent grads are zeros), so the
        data-parallel all-reduce and the fused AdamW run on ONE tensor with no pack/unpack."""
        if self.grad_flat is None:
            self.grad_flat = torch.zeros_like(self.flat)
        for _, p, off, n in self.entries:
            want = self.grad_flat[off:off + n].view(p.shape)
            if p.grad is None:
                want.zero_()      # "absent grads are zeros": never resurrect a stale gradient
                p.grad = want
            elif p.grad.data_ptr() != want.data_ptr():
                with torch.no_grad():
                    want.copy_(p.grad)
                p.grad = want
        return self.grad_flat

    def zero_grads_async(self):
        """`optimizer.zero_grad()` for the flat gradient buffer without a bubble in the compute
        stream: the 0.4 GB memset runs on a side stream, ordered after everything already
        enqueued on the current stream (the previous step's exchange / optimizer), beside the
        forward pass, which never touches gradients. Call `wait_grads_zeroed()` before the first
        kernel that writes a gradient (i.e. before backward)."""
        g = self.ensure_flat_grads()
        if not g.is_cuda:
            g.zero_()
            return
        if self.__dict__.get("_zero_stream") is None:
            self._zero_stream = torch.cuda.Stream(g.device)
            self._zero_start = torch.cuda.Event()
            self._zero_done = torch.cuda.Event()
        cur = torch.cuda.current_stream(g.device)
        self._zero_start.record(cur)
        self._zero_stream.wait_event(self._zero_start)
        with torch.cuda.stream(self._zero_stream):
            g.zero_()
            self._zero_done.record(self._zero_stream)
        self._zero_pending = True

    def wait_grads_zeroed(self):
        if self.__dict__.get("_zero_pending"):
            torch.cuda.current_stream(self.grad_flat.device).wait_event(self._zero_done)
            self._zero_pending = False


def flat_of(module, device):
    """The FlatParams owning `module`'s parameters: the one installed by the outermost hero_b200
    module that has run a forward, else a private one."""
    fp = module.__dict__.get("_hero_flat")
    if fp is not None and fp.module is not module and not fp._stale:
        # stamped by an outer manager: still part of its tree? (a module that was swapped out of
        # the tree, or swapped in without invalidate(), must not keep using a stale stamp)
        first = next(module.parameters(), None)
        if first is not None and id(first) not in fp._by_id:
            fp.invalidate()
    if fp is None:
        fp = FlatParams(module)
        for m in module.modules():
            m.__dict__["_hero_flat"] = fp
    return fp.ensure(device)
