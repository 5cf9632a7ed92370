"""Data-parallel plumbing: the function names of the reference's utils/distributed.py on top of
torch.distributed (NCCL over NVLink 5 / NVSwitch on the B200 box, gloo in CPU tests) instead of
Horovod.

Semantics kept from the reference (SURVEY.md Appendix D.8):
  * `all_reduce_and_rescale_tensors(tensors, denom)`: Horovod's `allreduce_` AVERAGES, so the
    result is mean-over-ranks / denom (utils/distributed.py:19-46).
  * `broadcast_tensors(tensors, root)` (utils/distributed.py:103-151), `all_gather_list`,
    `any_broadcast` (utils/distributed.py:182-212).
  * `VsmAllgather`: forward all-gather, backward = own slice of the incoming gradient with no
    reduction (model/pretrain.py:427-447).
What changes is the mechanism: when the gradients already live in one flat buffer
(`FlatParams.ensure_flat_grads`) the exchange is ONE in-place `all_reduce(AVG)` on that buffer —
no pack / unpack copies; otherwise tensors are coalesced once. One process per GPU, launched by
torchrun-style environment variables.
"""
import os
import pickle

import torch
import torch.distributed as dist


def init(backend=None):
    """Join the job described by RANK / WORLD_SIZE / MASTER_ADDR / MASTER_PORT (torchrun).
    Returns (rank, world_size, local_rank); a no-op single-process job when unset."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1 and not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
            dist.init_process_group(backend, rank=rank, world_size=world,
                                    device_id=torch.device("cuda", local_rank))
        else:
            dist.init_process_group(backend, rank=rank, world_size=world)
    return rank, world, local_rank


def size():
    return dist.get_world_size() if dist.is_initialized() else 1


def rank():
    return dist.get_rank() if dist.is_initialized() else 0


def _avg_inplace(buf):
    if size() == 1:
        return
    if dist.get_backend() == "nccl":
        dist.all_reduce(buf, op=dist.ReduceOp.AVG)     # ncclAvg: in-switch (NVLS) capable
    else:
        dist.all_reduce(buf, op=dist.ReduceOp.SUM)
        buf.div_(size())


def all_reduce_flat(buf, rescale_denom=1.0):
    """Mean over ranks of a flat gradient buffer, in place."""
    _avg_inplace(buf)
    if rescale_denom != 1.0:
        buf.div_(rescale_denom)
    return buf


class FlatGradExchange:
    """The gradient exchange of `all_reduce_and_rescale_tensors` (utils/distributed.py:19-46) on the
    flat gradient buffer of a FlatParams: mean over ranks, in place, no pack / unpack.

    wire="bf16" (default): ranges are cast into a persistent bf16 staging buffer, all-reduced there
    and cast back — half the NVLink bytes of an fp32 exchange (the reference exchanged fp16
    gradients under apex O2, train_vcmr.py:234-239); every rank ends with bit-identical fp32
    values (they are the same bf16 numbers). wire="fp32": in-place ncclAllReduce(AVG).

    overlap=True: the flat buffer keeps the cross-modal embedding tables (41 % of the bytes, final
    only when backward ends) at the end of each parameter group (params.is_late_grad). Call
    `prepare()` before the forward of a step that will be exchanged: when the embedding backward —
    the last node of the graph — begins, the exchange of everything else is enqueued on a side
    stream and runs beside it; `all_reduce()` after backward then reduces only the embedding
    ranges and joins. Without `prepare()` (or if the graph differentiates the stacks in an unusual
    order) `all_reduce()` reduces the whole buffer, as before."""

    def __init__(self, flat, wire="bf16", overlap=True):
        assert wire in ("bf16", "fp32")
        self.flat, self.wire, self.overlap = flat, wire, overlap
        g = flat.ensure_flat_grads()
        self.stage = (torch.empty(g.numel(), dtype=torch.bfloat16, device=g.device)
                      if wire == "bf16" else None)
        self.comm_stream = torch.cuda.Stream(g.device) if (overlap and g.is_cuda) else None
        self._armed = False
        self._early_done = None
        self._n_fwd = self._n_bwd = 0

    def describe(self):
        how = ("stack / head gradients all-reduced on a side stream during the embedding "
               "backward, embedding tables after backward" if self.overlap and self.comm_stream
               else "one all-reduce of the flat gradient buffer after backward")
        return f"NCCL all-reduce(AVG), {self.wire} on the wire; {how}"

    # ---- reduction of flat ranges on the current stream ----------------------------------------
    def _reduce_ranges(self, g, ranges):
        for a, b in ranges:
            if b <= a:
                continue
            if self.stage is None:
                _avg_inplace(g[a:b])
            else:
                self.stage[a:b].copy_(g[a:b])
                _avg_inplace(self.stage[a:b])
                g[a:b].copy_(self.stage[a:b])

    # ---- hook protocol (functional.EXCHANGE_HOOK) ------------------------------------------------
    def prepare(self):
        """The gradients of the forward/backward that follows will be exchanged."""
        from . import functional
        self._armed = bool(self.overlap and self.comm_stream is not None and size() > 1)
        self._early_done = None
        self._n_fwd = self._n_bwd = 0
        functional.EXCHANGE_HOOK[0] = self if self._armed else None

    def stack_forward(self):
        self._n_fwd += 1

    def stack_backward(self):
        self._n_bwd += 1

    def embedding_backward_begins(self):
        if not self._armed or self._early_done is not None:
            return
        if self._n_fwd == 0 or self._n_bwd != self._n_fwd:
            return          # some stack is still to be differentiated: leave it to all_reduce()
        g = self.flat.grad_flat
        cur = torch.cuda.current_stream(g.device)
        ready = torch.cuda.Event()
        ready.record(cur)
        self.comm_stream.wait_event(ready)
        with torch.cuda.stream(self.comm_stream):
            self._reduce_ranges(g, self.flat.early_ranges())
            done = torch.cuda.Event()
            done.record(self.comm_stream)
        self._early_done = done

    def all_reduce(self, rescale_denom=1.0):
        from . import functional
        g = self.flat.ensure_flat_grads()
        if size() > 1:
            if self._early_done is not None:
                self._reduce_ranges(g, self.flat.late_ranges())
                torch.cuda.current_stream(g.device).wait_event(self._early_done)
            else:
                self._reduce_ranges(g, [(0, g.numel())])
        self._early_done = None
        self._armed = False
        functional.EXCHANGE_HOOK[0] = None
        if rescale_denom != 1.0:
            g.div_(rescale_denom)
        return g

    def ranks_agree(self):
        """True iff every rank holds a bit-identical gradient buffer (collective call)."""
        g = self.flat.ensure_flat_grads()
        bits = g.view(torch.int32).to(torch.int64)
        digest = torch.stack([bits.sum(), (bits * (torch.arange(bits.numel(), device=g.device) % 8191
                                                   + 1)).sum()])
        if size() == 1:
            return True
        all_d = [torch.empty_like(digest) for _ in range(size())]
        dist.all_gather(all_d, digest)
        return all(bool((d == all_d[0]).all()) for d in all_d)

    def self_check(self):
        """Known-answer test of the exchange on this job's ranks and transport: rank r fills the
        buffer with (r + 1) * base, base a fixed pattern of multiples of 1/16 (exact in bf16);
        afterwards every rank must hold base * (W + 1) / 2 and all ranks must hold bit-identical
        buffers. With the bf16 wire the partial sums of W > 4 ranks are no longer all exact in
        bf16 (e.g. 21 * 13/16): the bound is one rounding (2^-9 relative) per addition plus the
        final one. Leaves the buffer zeroed."""
        g = self.flat.ensure_flat_grads()
        W, r = size(), rank()
        base = ((torch.arange(g.numel(), device=g.device) % 31) - 15).float() / 16.0
        g.copy_(base * (r + 1))
        self.all_reduce()
        want = base * ((W + 1) / 2.0)
        tol = (max(2.0 ** -7, (W + 1) * 2.0 ** -9) if self.stage is not None else 2.0 ** -20)
        err = float(((g - want).abs() - tol * want.abs()).max().item())
        same = self.ranks_agree()
        g.zero_()
        if err > 1e-6 or not same:
            raise RuntimeError(f"gradient all-reduce self-check failed on rank {r}: max excess "
                               f"error {err:.3e}, ranks bit-identical: {same}")
        return f"ok (mean of rank patterns reproduced on {W} ranks, bit-identical across ranks)"


def all_reduce_and_rescale_tensors(tensors, rescale_denom):
    """utils/distributed.py:19-46. Tensors that are consecutive views of one storage are reduced
    in place as a single message; anything else is coalesced once."""
    tensors = list(tensors)
    if not tensors:
        return
    flat = _as_single_view(tensors)
    if flat is not None:
        all_reduce_flat(flat, float(rescale_denom))
        return
    buf = torch.cat([t.reshape(-1) for t in tensors])
    all_reduce_flat(buf, float(rescale_denom))
    off = 0
    for t in tensors:
        n = t.numel()
        t.view(-1).copy_(buf[off:off + n])
        off += n


def _as_single_view(tensors):
    """If the tensors tile one contiguous region of a single storage (gaps allowed only as the
    alignment padding of FlatParams, which holds zeros), return that region as one tensor."""
    t0 = tensors[0]
    if not all(t.is_contiguous() and t.dtype == t0.dtype and t.device == t0.device and
               t.untyped_storage().data_ptr() == t0.untyped_storage().data_ptr()
               for t in tensors):
        return None
    es = t0.element_size()
    lo = min(t.data_ptr() for t in tensors)
    hi = max(t.data_ptr() + t.numel() * es for t in tensors)
    covered = sum(t.numel() for t in tensors)
    total = (hi - lo) // es
    if total > covered + 64 * len(tensors):     # more than alignment slack: not one region
        return None
    base = t0.untyped_storage().data_ptr()
    out = torch.empty(0, dtype=t0.dtype, device=t0.device)
    out.set_(t0.untyped_storage(), (lo - base) // es, (total,), (1,))
    return out


def broadcast_tensors(tensors, root_rank, buffer_size=None):
    """utils/distributed.py:103-151: every rank ends with root's values."""
    if size() == 1:
        return
    tensors = list(tensors)
    flat = _as_single_view(tensors) if tensors else None
    if flat is not None:
        dist.broadcast(flat, root_rank)
        return
    for t in tensors:
        dist.broadcast(t, root_rank)


def all_gather_list(data):
    """utils/distributed.py:182-198: gather arbitrary picklable data from all ranks. Stays off the
    GPU critical path (object collectives), unlike the reference's byte-tensor + .item() version."""
    if size() == 1:
        return [pickle.loads(pickle.dumps(data))]
    out = [None] * size()
    dist.all_gather_object(out, data)
    return out


def any_broadcast(data, root_rank):
    """utils/distributed.py:201-212."""
    if size() == 1:
        return pickle.loads(pickle.dumps(data))
    box = [data if rank() == root_rank else None]
    dist.broadcast_object_list(box, src=root_rank)
    return box[0]


def overlapped_exchange(flat, transport="none", **kw):
    """The gradient-exchange schedule selected by a training loop's `transport` option. Only
    None / "none" remains: the caller exchanges the gradients with FlatGradExchange (or
    `all_reduce_flat`) after or beside backward, and None is returned. Other keyword arguments
    (options of the removed schedule below) are ignored.

    A bucketed schedule that sent per-layer buckets during backward ("p2p": peer copies over
    symmetric memory, "nccl": a communicator capped in CTAs) was removed after losing to it on
    B200 / NVSwitch, 430 MB of fp32 gradients, 6.4-6.5 ms of compute per step, ms per step:
      N = 2: bucketed 7.23-7.34 device-resident but 7.96 end to end (its ~100 extra host-side
             enqueues per step double the host time of a step), all-reduce after backward 7.32;
      N = 4: bucketed 8.23, all-reduce after backward 7.65 - every bucket costs 2 (N-1) copies and
             signals per rank, and NCCL's all-reduce grows by only 0.3 ms from N = 2 to N = 4.
    It hid its exchanges completely, but the 41 % of the bytes that become final only when
    backward ends stay exposed either way (DESIGN.md §5)."""
    if transport in (None, "none"):
        return None
    raise ValueError(f"gradient exchange transport {transport!r}: the bucketed schedule was "
                     "removed (measured slower than the default exchange, DESIGN.md §5); "
                     "use 'none'")


class VsmAllgather(torch.autograd.Function):
    """model/pretrain.py:427-447: all-gather along dim 0 in rank order (ranks may contribute
    different row counts, as hvd.allgather allows); the backward hands each rank the slice of the
    gradient that corresponds to its own rows (no reduction)."""

    @staticmethod
    def forward(ctx, tensor, name=None, equal_counts=False):
        ctx.span = (0, tensor.shape[0])
        if size() == 1:
            return tensor
        tensor = tensor.contiguous()
        if equal_counts:
            # every rank contributes tensor.shape[0] rows (stated by the caller): one collective
            # into a preallocated block, nothing read back to the host
            n0 = tensor.shape[0]
            out = torch.empty((n0 * size(),) + tuple(tensor.shape[1:]), dtype=tensor.dtype,
                              device=tensor.device)
            dist.all_gather_into_tensor(out, tensor)
            ctx.span = (rank() * n0, (rank() + 1) * n0)
            return out
        n = torch.tensor([tensor.shape[0]], dtype=torch.int64, device=tensor.device)
        counts = [torch.zeros_like(n) for _ in range(size())]
        dist.all_gather(counts, n)
        counts = [int(c.item()) for c in counts]
        rest = tuple(tensor.shape[1:])
        if len(set(counts)) == 1:
            out = torch.empty((sum(counts),) + rest, dtype=tensor.dtype, device=tensor.device)
            dist.all_gather_into_tensor(out, tensor)
        else:
            mx = max(counts)
            padded = tensor.new_zeros((mx,) + rest)
            padded[:tensor.shape[0]] = tensor
            parts = [torch.empty_like(padded) for _ in range(size())]
            dist.all_gather(parts, padded)
            out = torch.cat([p[:c] for p, c in zip(parts, counts)], 0)
        start = sum(counts[:rank()])
        ctx.span = (start, start + counts[rank()])
        return out

    @staticmethod
    def backward(ctx, grad_output):
        a, b = ctx.span
        return grad_output[a:b], None, None


vsm_allgather = VsmAllgather.apply
